"""Prompts of different lengths on the OpenVLA-7B-shaped decoder: what a ragged batch costs against equal lengths.

Full-size random-init Llama-2-7B-shaped decoder (built layer by layer, as `bench.py --workload openvla` does), 7 greedy
tokens.  At batch 32, `generate` p50 (CUDA events over back-to-back calls, cases interleaved) for
  equal_281      every prompt 1 + 256 + 24 = 281 positions (the benchmark's shape);
  ragged         seeded lengths over 270..300 (256 patches + BOS + 13..43 text tokens), padded to their maximum;
  equal_max      every prompt at that maximum;
each for 7 tokens and for 1 token (prefill + first token), so that the decode time per token is their difference / 6.
At batch 1: the ragged call (`prompt_lens=[281]`) against the plain call at 281.  Also: the share of ragged rows whose
7 token ids equal a batch-1 run of that row alone.  The card's name and power limit are read in the same run.

    python tools/openvla_ragged.py --out profiles/openvla_ragged.json
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


def build_decoder(dev, max_batch):
    cfg = openvla.openvla_7b_config()
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
    return cfg, dec


def time_cases(dec, cases, steps, warmup):
    """cases: name -> zero-argument callable.  Interleaved: one call of each case per round."""
    for _ in range(warmup):
        for fn in cases.values():
            fn()
    torch.cuda.synchronize()
    dec.check()
    lat = {k: [] for k in cases}
    for _ in range(steps):
        for k, fn in cases.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            lat[k].append((a, b))
    torch.cuda.synchronize()
    dec.check()
    out = {}
    for k, evs in lat.items():
        t = sorted(a.elapsed_time(b) for a, b in evs)
        out[k] = {"ms_p50": t[len(t) // 2], "ms_min": t[0], "ms_max": t[-1]}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_ragged.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_ragged.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "model": "Llama-2-7B-shaped decoder, random init, 7 greedy tokens", "steps": args.steps}
    cfg, dec = build_decoder(dev, 32)
    n_new, base = 7, 281
    g = torch.Generator(device=dev).manual_seed(args.seed)
    lens = np.random.default_rng(args.seed).integers(1 + 256 + 13, 1 + 256 + 43 + 1, size=32).astype(np.int32)
    T = int(lens.max())
    x_base = (torch.randn((32, base, cfg.hidden), device=dev, generator=g) * 0.5).to(torch.bfloat16)
    x_max = (torch.randn((32, T, cfg.hidden), device=dev, generator=g) * 0.5).to(torch.bfloat16)
    result["batch32_lengths"] = {"min": int(lens.min()), "max": T, "mean": float(lens.mean()), "values": lens.tolist()}

    cases = {}
    for n in (n_new, 1):
        cases[f"equal_281_n{n}"] = lambda n=n: dec.generate(x_base, n)
        cases[f"ragged_n{n}"] = lambda n=n: dec.generate(x_max, n, prompt_lens=lens)
        cases[f"equal_max_n{n}"] = lambda n=n: dec.generate(x_max, n)
    t32 = time_cases(dec, cases, args.steps, args.warmup)
    b32 = {}
    for name in ("equal_281", "ragged", "equal_max"):
        full, one = t32[f"{name}_n{n_new}"], t32[f"{name}_n1"]
        b32[name] = {"generate_7": full, "generate_1": one,
                     "decode_ms_per_token_p50": (full["ms_p50"] - one["ms_p50"]) / (n_new - 1)}
    result["batch32"] = b32

    # rows of the ragged batch against batch-1 runs of each row alone
    ids_r = dec.generate(x_max, n_new, prompt_lens=lens)
    same = 0
    for b in range(32):
        same += int(torch.equal(dec.generate(x_max[b:b + 1, :int(lens[b])].contiguous(), n_new)[0], ids_r[b]))
    dec.check()
    result["batch32_rows_equal_to_batch1"] = {"rows": same, "of": 32, "share": same / 32}

    x1 = x_base[:1].contiguous()
    cases1 = {}
    for n in (n_new, 1):
        cases1[f"equal_281_n{n}"] = lambda n=n: dec.generate(x1, n)
        cases1[f"ragged_281_n{n}"] = lambda n=n: dec.generate(x1, n, prompt_lens=[base])
    t1 = time_cases(dec, cases1, args.steps, args.warmup)
    b1 = {}
    for name in ("equal_281", "ragged_281"):
        full, one = t1[f"{name}_n{n_new}"], t1[f"{name}_n1"]
        b1[name] = {"generate_7": full, "generate_1": one,
                    "decode_ms_per_token_p50": (full["ms_p50"] - one["ms_p50"]) / (n_new - 1)}
    result["batch1"] = b1
    assert torch.equal(dec.generate(x1, n_new, prompt_lens=[base]), dec.generate(x1, n_new))
    result["card_after"] = card()
    dec.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "batch32_rows_equal_to_batch1")}))
    for bs, d in (("32", b32), ("1", b1)):
        for k, v in d.items():
            print(f"batch {bs} {k:10s}: generate(7) p50 {v['generate_7']['ms_p50']:.3f} ms, "
                  f"decode/token {v['decode_ms_per_token_p50']:.3f} ms")


if __name__ == "__main__":
    main()
