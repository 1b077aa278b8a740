"""Sampled decoding on the OpenVLA-7B-shaped decoder: what `do_sample=True` costs against greedy decoding.

Full-size random-init Llama-2-7B-shaped decoder (built layer by layer, as tools/openvla_ragged.py builds it), prompts of
1 + 256 + 24 = 281 positions, 7 tokens.  Measured in one run, on the card named in the output:
  generate       p50 of interleaved calls (CUDA events) at batch 1 and 32: greedy, sampled with T = 0.7, top_k = 50,
                 top_p = 0.9, and sampled with top_k = 0, top_p = 0.9 (the widest kept set);
  predict_action batch 1, full-depth DINOv2 + SigLIP towers and projector from prepared pixels to actions
                 (`OpenVlaPolicy.predict_action_from_pixels`), greedy against `do_sample=True` (HF defaults);
  in-graph       option "trace": the sampler's own time (first CTA past its dependency wait -> last CTA done) per step,
                 and for greedy and sampled calls alike the gap from the lm_head GEMM's end to the next step's first
                 traced kernel (logits epilogue + argmax or sampler + embedding), whose difference is the sampler's cost
                 over argmax inside the graph.

    python tools/openvla_sampling.py --out profiles/openvla_sampling.json
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from blurr_b200 import openvla  # noqa: E402
from openvla_ragged import build_decoder, card, time_cases  # noqa: E402

N_NEW, PROMPT = 7, 281
SAMPLED = {"sampled_k50_p0.9": dict(do_sample=True, temperature=0.7, top_k=50, top_p=0.9),
           "sampled_k0_p0.9": dict(do_sample=True, temperature=0.7, top_k=0, top_p=0.9)}


def parse_trace(report: str):
    rows = []
    for line in report.splitlines():
        if line.startswith("#") or not line.strip():
            continue
        idx, start, waited, end, label = line.split(None, 4)
        rows.append((float(start), float(waited), float(end), label))
    return rows


def trace_stats(dec, x, kw, lm_head_n: int):
    dec.set_option("trace", 1)
    dec.generate(x, N_NEW, **kw)                        # capture
    dec.generate(x, N_NEW, **kw)
    rows = parse_trace(dec.trace_report())
    dec.set_option("trace", 0)
    sampler = [e - w for s, w, e, lab in rows if lab == "sample_rows"]
    heads = [i for i, r in enumerate(rows) if r[3].startswith("gemm[") and f" N{lm_head_n} " in r[3]]
    tails = []
    for i in heads:                                     # -> the next step's input-norm consumer (the next traced kernel
        nxt = [r for r in rows[i + 1:] if r[3].startswith("consumer")]      # of a greedy call, after the sampler's)
        if nxt:
            tails.append(nxt[0][0] - rows[i][2])
    out = {"head_tail_gap_us": {"per_step": tails, "p50": float(np.median(tails)) if tails else None}}
    if sampler:
        out["sample_rows_us"] = {"per_step": sampler, "p50": float(np.median(sampler)), "max": max(sampler)}
    return out


def build_policy(dev, dec):
    g = torch.Generator(device=dev).manual_seed(1)
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(), dev, max_batch=1, seed=100)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(), dev, max_batch=1, seed=101)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    pre = openvla.ImagePreprocessor(224, 224, device=dev)
    return openvla.OpenVlaPolicy(pre, openvla.FusedVisionBackbone(dino, sig, proj), dec), (pre, dino, sig, proj)


def time_host(cases, steps, warmup):
    """cases: name -> callable that ends in a host synchronisation (predict_action returns host actions)."""
    for _ in range(warmup):
        for fn in cases.values():
            fn()
    lat = {k: [] for k in cases}
    for _ in range(steps):
        for k, fn in cases.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            lat[k].append((time.perf_counter() - t0) * 1e3)
    return {k: {"ms_p50": float(np.median(v)), "ms_min": min(v), "ms_max": max(v)} for k, v in lat.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_sampling.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_sampling.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "model": f"Llama-2-7B-shaped decoder, random init, {PROMPT}-position prompts, {N_NEW} tokens",
              "steps": args.steps}
    cfg, dec = build_decoder(dev, 32)
    g = torch.Generator(device=dev).manual_seed(0)
    gen = {}
    for B in (1, 32):
        x = (torch.randn((B, PROMPT, cfg.hidden), device=dev, generator=g) * 0.5).to(torch.bfloat16)
        cases = {"greedy": lambda x=x: dec.generate(x, N_NEW)}
        for name, kw in SAMPLED.items():
            cases[name] = lambda x=x, kw=kw: dec.generate(x, N_NEW, seed=list(range(B)), **kw)
        t = time_cases(dec, cases, args.steps, args.warmup)
        launches = {}
        for name, fn in cases.items():
            fn()
            launches[name] = dec.last_launch_count
        for name in SAMPLED:
            t[name]["over_greedy_ms"] = t[name]["ms_p50"] - t["greedy"]["ms_p50"]
            t[name]["over_greedy_pct"] = 100.0 * t[name]["over_greedy_ms"] / t["greedy"]["ms_p50"]
        t["launches"] = launches
        lm_n = (cfg.vocab + 127) // 128 * 128
        t["in_graph"] = {"greedy": trace_stats(dec, x, {}, lm_n)}
        for name, kw in SAMPLED.items():
            t["in_graph"][name] = trace_stats(dec, x, dict(seed=list(range(B)), **kw), lm_n)
        dec.check()
        gen[f"batch{B}"] = t
    result["generate"] = gen

    pol, parts = build_policy(dev, dec)
    px = (torch.rand((1, 6, 224, 224), device=dev, generator=g) * 2 - 1).to(torch.bfloat16)
    ids = torch.randint(3, 32000, (1, 25), device=dev, generator=g)
    ids[0, 0] = 1
    q01, q99 = np.full(7, -1.0), np.full(7, 1.0)
    pa = time_host({"greedy": lambda: pol.predict_action_from_pixels(px, ids, q01, q99),
                    "do_sample": lambda: pol.predict_action_from_pixels(px, ids, q01, q99, do_sample=True, seed=0)},
                   args.steps, args.warmup)
    pa["do_sample"]["over_greedy_pct"] = 100.0 * (pa["do_sample"]["ms_p50"] - pa["greedy"]["ms_p50"]) / pa["greedy"]["ms_p50"]
    result["predict_action_batch1"] = pa
    dec.check()
    result["card_after"] = card()
    for m in parts:
        m.close()
    dec.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))
    for bs, t in gen.items():
        for name in ("greedy", *SAMPLED):
            ig = t["in_graph"][name]
            extra = f", sample_rows p50 {ig['sample_rows_us']['p50']:.1f} us" if "sample_rows_us" in ig else ""
            print(f"{bs} {name:18s}: generate(7) p50 {t[name]['ms_p50']:.3f} ms, head tail gap p50 "
                  f"{ig['head_tail_gap_us']['p50']:.1f} us{extra}")
    print(f"predict_action batch 1: greedy {pa['greedy']['ms_p50']:.3f} ms, do_sample {pa['do_sample']['ms_p50']:.3f} ms "
          f"({pa['do_sample']['over_greedy_pct']:+.2f} %)")


if __name__ == "__main__":
    main()
