"""OpenVLA-OFT's parallel decoding against OpenVLA's autoregressive decode, on the full-size 7B shape.

Random-init Llama-2-7B-shaped decoder (built layer by layer, as `bench.py --workload openvla` does, with OFT's 384
positions), full-depth DINOv2-L + SigLIP-so400m towers, the projector and a random-init L1-regression head at OFT's widths
(4096 x 7 -> 4096 -> 7, two blocks).  At batch 1 and 32, CUDA events around 30 interleaved calls (p50) of
  oft_chunk        `OftPolicy.predict_action_chunk_from_pixels`: 8 actions x 7 values per sequence per call;
  openvla_action   `OpenVlaPolicy.predict_action_from_pixels` with the same decoder and towers: 1 action x 7 values;
and per OFT stage (vision towers + projector, `forward_rows`, head).  Prompts: BOS + 23 instruction tokens (+ OFT's
29871), so OpenVLA's prompt is 280 positions and OFT's sequence 338.  Also the in-graph timeline of the new attention
mode (MODE 3) against the causal prefill attention (MODE 2) at the same length (319 rows, the most MODE 2 takes with one
new token), and MODE 3 at OFT's length.  The card's name and power limit are read in the same run.

    python tools/openvla_oft.py --out profiles/openvla_oft.json
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from blurr_b200 import capi, openvla  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def build_decoder(cfg, dev, max_batch):
    dec = openvla.LlamaDecoder(cfg, dev, max_batch=max_batch)
    one = openvla.LlamaShapedConfig(**{**cfg.__dict__, "num_layers": 1})
    for l in range(cfg.num_layers):
        sd = openvla.synthetic_llama_state_dict(one, dev, seed=l)
        for k, v in sd.items():
            if k.startswith("model.layers.0."):
                dec.set_weight(k.replace("model.layers.0.", f"model.layers.{l}."), v)
            elif l == 0:
                dec.set_weight(k, v)
        del sd
    cos, sin = openvla.rope_tables(openvla.default_inv_freq(cfg.head_dim, cfg.rope_theta, dev), cfg.max_positions)
    torch.cuda.synchronize()
    capi.check(dec.lib.blurr_llm_set_rope_table(dec.handle, C.c_void_p(cos.data_ptr()), C.c_void_p(sin.data_ptr()),
                                                cfg.max_positions))
    capi.check(dec.lib.blurr_llm_finalize(dec.handle))
    return dec


def time_cases(cases, steps, warmup, check):
    """cases: name -> zero-argument callable.  Interleaved: one call of each case per round; p50 of CUDA events."""
    for _ in range(warmup):
        for fn in cases.values():
            fn()
    torch.cuda.synchronize()
    check()
    lat = {k: [] for k in cases}
    for _ in range(steps):
        for k, fn in cases.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            lat[k].append((a, b))
    torch.cuda.synchronize()
    check()
    out = {}
    for k, evs in lat.items():
        t = sorted(a.elapsed_time(b) for a, b in evs)
        out[k] = {"ms_p50": t[len(t) // 2], "ms_min": t[0], "ms_max": t[-1]}
    return out


def attention_trace(dec, label, fn, reps=5):
    """Mean per-layer time (us, in-graph %globaltimer: first CTA past its dependency wait -> last CTA done) of the
    attention kernels whose label is `label`, over `reps` graph replays."""
    dec.set_option("trace", 1)
    fn()                                              # capture the traced graph
    per_call = []
    for _ in range(reps):
        fn()
        torch.cuda.synchronize()
        us = []
        for line in dec.trace_report().splitlines():
            f = line.split()
            if line.startswith("#") or len(f) < 5 or f[4] != label:
                continue
            start, waited, end = float(f[1]), float(f[2]), float(f[3])
            us.append(end - max(start, waited))
        per_call.append(float(np.mean(us)))
    dec.set_option("trace", 0)
    return {"us_per_layer_mean": float(np.mean(per_call)), "us_per_layer_min": float(np.min(per_call)), "layers": len(us)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_oft.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_oft.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "steps": args.steps,
              "model": "OpenVLA-7B shape, random init: DINOv2-L/14 reg4 + SigLIP-so400m/14 (full depth), projector, "
                       "Llama-2-7B-shaped decoder (384 positions), L1-regression head 28672 -> 4096 -> 7 (2 blocks)"}
    oft = openvla.OftConfig()
    dec = build_decoder(openvla.openvla_oft_7b_config(oft), dev, 32)
    g = torch.Generator(device=dev).manual_seed(args.seed)
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(), dev, max_batch=32, seed=100)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(), dev, max_batch=32, seed=101)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=32 * 256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    fused = openvla.FusedVisionBackbone(dino, sig, proj)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, dev, max_batch=32, seed=7)
    pre = openvla.ImagePreprocessor(480, 640, device=dev)
    oft_pol = openvla.OftPolicy(pre, fused, dec, head, oft)
    vla_pol = openvla.OpenVlaPolicy(pre, fused, dec)
    q01, q99 = np.full(7, -1.0), np.full(7, 1.0)

    def check():
        dec.check()
        head.check()

    for B in (1, 32):
        px = (torch.rand((B, 6, 224, 224), device=dev, generator=g) * 2 - 1).to(torch.bfloat16)
        ids = torch.randint(3, 32000, (B, 24), device=dev, generator=g)
        ids[:, 0] = 1
        ids[:, -1] = torch.where(ids[:, -1] == oft.empty_token, 3, ids[:, -1])
        lay = openvla.oft_prompt_layout(ids, n_patches=256, cfg=oft)
        patch = fused.forward(px[:, :3], px[:, 3:])
        x = openvla.build_oft_embeds(dec, lay, patch, oft.stop_token)
        rows = dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
        cases = {
            "oft_chunk": lambda: oft_pol.predict_action_chunk_from_pixels(px, ids, q01, q99),
            "openvla_action": lambda: vla_pol.predict_action_from_pixels(px, ids, q01, q99),
            "vision": lambda: fused.forward(px[:, :3], px[:, 3:]),
            "forward_rows": lambda: dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows),
            "head": lambda: head.forward(rows),
        }
        t = time_cases(cases, args.steps, args.warmup, check)
        dec.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
        fr_launches = dec.last_launch_count
        head.forward(rows)
        act = oft_pol.predict_action_chunk_from_pixels(px, ids, q01, q99)
        assert act.shape == (B, oft.chunk, oft.action_dim) and bool(torch.isfinite(act).all())
        oc, oa = t["oft_chunk"]["ms_p50"], t["openvla_action"]["ms_p50"]
        result[f"batch{B}"] = {
            "oft_sequence_positions": int(lay.max_len), "openvla_prompt_positions": 1 + 256 + 23,
            "timings_ms": t,
            "launches": {"forward_rows": fr_launches, "head": head.last_launch_count},
            "oft_actions_per_s": B * oft.chunk / (oc / 1e3),
            "oft_action_values_per_s": B * oft.chunk * oft.action_dim / (oc / 1e3),
            "openvla_actions_per_s": B / (oa / 1e3),
            "openvla_action_values_per_s": B * oft.action_dim / (oa / 1e3),
            "note": "one OFT call yields chunk=8 actions of 7 values per sequence; one OpenVLA call yields 1 action of 7",
        }
        print(f"batch {B}: OFT chunk {oc:.3f} ms ({B * oft.chunk / (oc / 1e3):.1f} actions/s), OpenVLA action {oa:.3f} ms "
              f"({B / (oa / 1e3):.1f} actions/s); vision {t['vision']['ms_p50']:.3f}, forward_rows "
              f"{t['forward_rows']['ms_p50']:.3f}, head {t['head']['ms_p50']:.3f} ms")

    # attention: MODE 3 (block-bidirectional) against MODE 2 (causal prefill) at the same length, in the graph
    trace = {}
    for B in (1, 32):
        T = 319
        xt = (torch.randn((B, T, 4096), device=dev, generator=g) * 0.5).to(torch.bfloat16)
        lens = np.full(B, T, np.int32)
        a0 = lens - 57
        trace[f"batch{B}_len319_mode2_causal_prefill"] = attention_trace(dec, "mha_prefill", lambda: dec.generate(xt, 1))
        trace[f"batch{B}_len319_mode3_block"] = attention_trace(
            dec, "mha_block_prefill", lambda: dec.forward_rows(xt, lens, a0, a0 - 1, 56))
        trace[f"batch{B}_len319_mode3_block_at_len"] = attention_trace(
            dec, "mha_block_prefill", lambda: dec.forward_rows(xt, lens, lens, lens - 56, 56))
        T2 = 338
        x2 = (torch.randn((B, T2, 4096), device=dev, generator=g) * 0.5).to(torch.bfloat16)
        l2 = np.full(B, T2, np.int32)
        trace[f"batch{B}_len338_mode3_block"] = attention_trace(
            dec, "mha_block_prefill", lambda: dec.forward_rows(x2, l2, l2 - 57, l2 - 58, 56))
    result["attention_in_graph"] = trace
    for k, v in trace.items():
        print(f"{k}: {v['us_per_layer_mean']:.2f} us per layer")
    check()
    result["card_after"] = card()
    for m in (pre, dino, sig, proj, dec, head):
        m.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
