"""OpenVLA-OFT with two cameras and proprioception (the LIBERO checkpoints' form) on the full-size 7B shape.

Random-init Llama-2-7B-shaped decoder with 640 positions (`long_forward`, built layer by layer as tools/openvla_oft.py
does), full-depth DINOv2-L + SigLIP-so400m towers, the projector, a random-init L1-regression head and proprio
projector at OFT's widths.  Prompt: BOS + 34 instruction tokens (+ OFT's 29871), so a two-camera sequence is
1 + 2 x 256 + 1 + 35 + 56 + 1 = 606 positions, and the one-camera sequence of tools/openvla_oft.py (BOS + 23 tokens) is
338.  At batch 1 and 32, CUDA events around 30 interleaved calls (p50) of
  libero_chunk        `OftPolicy.predict_action_chunk_from_pixels`, two cameras + proprio: 8 actions x 7 per sequence;
  one_camera_chunk    the one-camera policy on the same towers, decoder and head (338 positions);
  vision_two_cameras  the towers + projector on both cameras ([2B, 6, 224, 224]);
  forward_rows        the decoder pass at 606 positions;
  proprio_projector   the proprio projector on B rows.
Also the in-graph attention time per layer (option "trace"): the streamed kernel at 606 keys, and both kernels on
sequences of 338 and 384 positions (the resident one at max_len = the length; the streamed one at max_len 385, which
selects it, with the same sequences: one more 16..64-row query tile per head of pad rows).  The card's name and power
limit are read in the same run.

    python tools/openvla_oft_cameras.py --out profiles/openvla_oft_cameras.json
"""

from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from blurr_b200 import openvla  # noqa: E402
from openvla_oft import attention_trace, build_decoder, card, time_cases  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_oft_cameras.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_oft_cameras.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "steps": args.steps,
              "model": "OpenVLA-7B shape, random init: DINOv2-L/14 reg4 + SigLIP-so400m/14 (full depth), projector, "
                       "Llama-2-7B-shaped decoder (640 positions, long_forward), L1-regression head 28672 -> 4096 -> 7 "
                       "(2 blocks), proprio projector 8 -> 4096 -> 4096"}
    oft = openvla.oft_libero_config()
    one_cfg = openvla.OftConfig()
    dec = build_decoder(openvla.openvla_oft_7b_config(oft), dev, 32)
    g = torch.Generator(device=dev).manual_seed(args.seed)
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(), dev, max_batch=64, seed=100)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(), dev, max_batch=64, seed=101)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=64 * 256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    fused = openvla.FusedVisionBackbone(dino, sig, proj)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, dev, max_batch=32, seed=7)
    pp = openvla.ProprioProjector.synthetic(oft.proprio_dim, 4096, dev, max_rows=32, seed=8)
    pres = [openvla.ImagePreprocessor(480, 640, device=dev), openvla.ImagePreprocessor(256, 256, device=dev)]
    libero = openvla.OftPolicy(pres, fused, dec, head, oft, proprio_projector=pp)
    one = openvla.OftPolicy(pres[0], fused, dec, head, one_cfg)
    q01, q99 = np.full(7, -1.0), np.full(7, 1.0)
    pq01, pq99 = np.full(8, -1.0), np.full(8, 1.0)

    def check():
        dec.check()
        head.check()

    def prompt(B, n):
        ids = torch.randint(3, 32000, (B, n), device=dev, generator=g)
        ids[:, 0] = 1
        ids[:, -1] = torch.where(ids[:, -1] == oft.empty_token, 3, ids[:, -1])
        return ids

    for B in (1, 32):
        px2 = (torch.rand((B, 12, 224, 224), device=dev, generator=g) * 2 - 1).to(torch.bfloat16)
        px1 = px2[:, :6].contiguous()
        ids2, ids1 = prompt(B, 35), prompt(B, 24)
        raw = np.random.default_rng(B).uniform(-1, 1, size=(B, 8))
        state = libero.proprio_state(raw, pq01, pq99)
        patch = libero.patch_embeds(px2, state)
        lay = openvla.oft_prompt_layout(ids2, n_patches=patch.shape[1], cfg=oft)
        x = openvla.build_oft_embeds(dec, lay, patch, oft.stop_token)
        px_cams = px2.reshape(2 * B, 6, 224, 224)
        cases = {
            "libero_chunk": lambda: libero.predict_action_chunk_from_pixels(px2, ids2, q01, q99, proprio=raw, proprio_q01=pq01,
                                                                            proprio_q99=pq99),
            "one_camera_chunk": lambda: one.predict_action_chunk_from_pixels(px1, ids1, q01, q99),
            "vision_two_cameras": lambda: fused.forward(px_cams[:, :3], px_cams[:, 3:]),
            "forward_rows": lambda: dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows),
            "proprio_projector": lambda: pp.forward(state),
        }
        t = time_cases(cases, args.steps, args.warmup, check)
        act = libero.predict_action_chunk_from_pixels(px2, ids2, q01, q99, proprio=raw, proprio_q01=pq01, proprio_q99=pq99)
        assert act.shape == (B, oft.chunk, oft.action_dim) and bool(torch.isfinite(act).all())
        dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
        lc = t["libero_chunk"]["ms_p50"]
        result[f"batch{B}"] = {
            "libero_sequence_positions": int(lay.max_len), "one_camera_sequence_positions": 1 + 256 + 24 + 57,
            "timings_ms": t, "launches": {"forward_rows": dec.last_launch_count},
            "libero_actions_per_s": B * oft.chunk / (lc / 1e3),
        }
        print(f"batch {B}: two cameras + proprio {lc:.3f} ms ({lay.max_len} positions), one camera "
              f"{t['one_camera_chunk']['ms_p50']:.3f} ms; vision {t['vision_two_cameras']['ms_p50']:.3f}, forward_rows "
              f"{t['forward_rows']['ms_p50']:.3f}, proprio {t['proprio_projector']['ms_p50']:.3f} ms")

    trace = {}
    for B in (1, 32):
        xt = (torch.randn((B, 606, 4096), device=dev, generator=g) * 0.5).to(torch.bfloat16)
        lens = np.full(B, 606, np.int32)
        trace[f"batch{B}_len606_streamed"] = attention_trace(
            dec, "mha_block_prefill", lambda: dec.forward_rows(xt, lens, lens - 57, lens - 58, 56))
        for L in (338, 384):
            l = np.full(B, L, np.int32)
            trace[f"batch{B}_len{L}_resident"] = attention_trace(
                dec, "mha_block_prefill", lambda: dec.forward_rows(xt[:, :L], l, l - 57, l - 58, 56))
            trace[f"batch{B}_len{L}_streamed_max_len385"] = attention_trace(
                dec, "mha_block_prefill", lambda: dec.forward_rows(xt[:, :385], l, l - 57, l - 58, 56))
    result["attention_in_graph"] = trace
    for k, v in trace.items():
        print(f"{k}: {v['us_per_layer_mean']:.2f} us per layer")
    check()
    result["card_after"] = card()
    for m in (*pres, dino, sig, proj, dec, head, pp):
        m.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
