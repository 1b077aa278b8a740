"""OpenVLA-OFT, the ALOHA form (three FiLM cameras, 14-D proprioception, chunks of 25 x 14) on the full-size 7B shape.

Random-init Llama-2-7B-shaped decoder with 1280 positions (`long_forward = 2`, built as tools/openvla_oft.py does),
full-depth DINOv2-L + SigLIP-so400m FiLM towers, the projector, a random-init L1-regression head 57 344 -> 4096 -> 14
and proprio projector 14 -> 4096 -> 4096.  BOS + 20 instruction tokens (+ 29871), so a sequence is
769 + 22 + 350 + 1 = 1142 positions.  At batch 1 and 32, CUDA events around 30 interleaved calls (p50, min-max) of
  aloha_chunk      `predict_action_chunk_from_pixels`: 25 actions of 14 values per sequence;
  vision           the FiLM towers + projector on the three images of each sequence;
  language_vector  `film_language_embedding`;
  forward_rows     the decoder pass over the assembled rows;
  head             the action head on its 350 rows per sequence.
Then the in-graph attention time per layer (option "trace") at that length, and the head's wide LayerNorm alone
(`torch.profiler`, graph replays of the head).  The card's name and power limit are read in the same run.

    python tools/openvla_oft_aloha.py --out profiles/openvla_oft_aloha.json
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


def kernel_profile(fn, name, reps=20):
    """Device time of the kernels whose name contains `name` over `reps` calls of `fn`, from torch.profiler."""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    times = sorted(e.time_range.elapsed_us() for e in prof.events()
                   if e.device_type == torch.autograd.DeviceType.CUDA and name in e.name)
    if not times:
        return {"kernel": name, "captured": 0}
    return {"kernel": name, "captured": len(times), "us_p50": times[len(times) // 2], "us_min": times[0], "us_max": times[-1]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_oft_aloha.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_oft_aloha.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    oft = openvla.oft_aloha_config()
    result = {"card": card(), "steps": args.steps,
              "model": "OpenVLA-7B shape, random init: DINOv2-L/14 reg4 + SigLIP-so400m/14 FiLM towers (full depth), "
                       "projector, Llama-2-7B-shaped decoder (1280 positions, long_forward 2), L1-regression head "
                       "57344 -> 4096 -> 14 (2 blocks), proprio projector 14 -> 4096 -> 4096; three cameras, chunks of 25 x 14"}
    dec = build_decoder(openvla.openvla_oft_7b_config(oft), dev, 32)
    g = torch.Generator(device=dev).manual_seed(args.seed)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=96 * 256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    d, s = openvla.dinov2_large_reg4_config(), openvla.siglip_so400m_config()
    d.film_dim = s.film_dim = 4096
    dino = openvla.VitEncoder.synthetic(d, dev, max_batch=96, seed=100)
    sig = openvla.VitEncoder.synthetic(s, dev, max_batch=96, seed=101)
    fused = openvla.FusedVisionBackbone(dino, sig, proj)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, dev, max_batch=32, seed=7)
    pp = openvla.ProprioProjector.synthetic(oft.proprio_dim, 4096, dev, max_rows=32, seed=8)
    pres = [openvla.ImagePreprocessor(480, 640, device=dev) for _ in range(3)]
    pol = openvla.OftPolicy(pres, fused, dec, head, oft, proprio_projector=pp)
    amin, amax = np.full(14, -1.0), np.full(14, 1.0)          # BOUNDS statistics (min / max)
    pmin, pmax = np.full(14, -1.0), np.full(14, 1.0)

    def check():
        dec.check()
        head.check()

    def prompt(B, n):
        ids = torch.randint(3, 32000, (B, n), device=dev, generator=g)
        ids[:, 0] = 1
        ids[:, -1] = torch.where(ids[:, -1] == oft.empty_token, 3, ids[:, -1])
        return ids

    trace = {}
    for B in (1, 32):
        px = (torch.rand((B, 18, 224, 224), device=dev, generator=g) * 2 - 1).to(torch.bfloat16)
        ids = prompt(B, 21)
        raw = np.random.default_rng(B).uniform(-1, 1, size=(B, 14))
        lay = openvla.oft_prompt_layout(ids, n_patches=3 * 256 + 1, cfg=oft)
        cond = openvla.film_language_embedding(dec, lay)
        state = pol.proprio_state(raw, pmin, pmax)
        px3 = px.reshape(3 * B, 6, 224, 224)
        x = openvla.build_oft_embeds(dec, lay, pol.patch_embeds(px, state, cond))
        rows = dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
        kw = dict(proprio=raw, proprio_q01=pmin, proprio_q99=pmax)
        cases = {
            "aloha_chunk": lambda: pol.predict_action_chunk_from_pixels(px, ids, amin, amax, **kw),
            "vision": lambda: fused.forward(px3[:, :3], px3[:, 3:], film_cond=cond, images_per_cond=3),
            "language_vector": lambda: openvla.film_language_embedding(dec, lay),
            "forward_rows": lambda: dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows),
            "head": lambda: head.forward(rows),
        }
        t = time_cases(cases, args.steps, args.warmup, check)
        out = cases["aloha_chunk"]()
        assert out.shape == (B, 25, 14) and bool(torch.isfinite(out).all())
        dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
        fr_launches = dec.last_launch_count
        head.forward(rows)
        result[f"batch{B}"] = {
            "seq_len": int(lay.max_len), "timings_ms": t, "forward_rows_kernels": fr_launches,
            "head_kernels": head.last_launch_count,
            "head_wide_layernorm": kernel_profile(lambda: head.forward(rows), "act_wide_layernorm"),
        }
        trace[f"batch{B}_len{lay.max_len}_streamed"] = attention_trace(
            dec, "mha_block_prefill", lambda: dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows))
        p50 = {k: v["ms_p50"] for k, v in t.items()}
        print(f"batch {B} ({lay.max_len} positions): " + ", ".join(f"{k} {v:.3f}" for k, v in p50.items()) + " ms")
        print(f"batch {B}: head wide LayerNorm {result[f'batch{B}']['head_wide_layernorm']}")
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
