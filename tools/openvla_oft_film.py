"""OpenVLA-OFT with FiLM language conditioning of the vision towers (the paper's "OFT+" form) on the full-size 7B shape.

Random-init Llama-2-7B-shaped decoder with 640 positions (built as tools/openvla_oft.py does), full-depth DINOv2-L +
SigLIP-so400m towers twice - plain, and FiLM towers with the same other weights plus 4096 -> hidden FiLM Linears per
block - the projector, a random-init L1-regression head and proprio projector.  Prompts as in tools/openvla_oft.py and
tools/openvla_oft_cameras.py: one camera at 338 positions, two cameras + proprio at 606.  At batch 1 and 32, CUDA events
around 30 interleaved calls (p50) of
  film_one_camera_chunk / one_camera_chunk   the one-camera policy with and without FiLM (same decoder and head);
  film_libero_chunk / libero_chunk           the two-camera + proprio policy with and without FiLM;
  vision_film / vision                        the towers + projector on one camera, with and without FiLM;
  language_vector                             `film_language_embedding` (embedding rows + the per-sequence mean).
The conditioning GEMM of each tower alone comes from a separate `torch.profiler` run of eager (no CUDA graph) tower
calls: the kernel right after the im2col, reported as weight bytes / time.  The card's name and power limit are read in
the same run.

    python tools/openvla_oft_film.py --out profiles/openvla_oft_film.json
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
from openvla_oft import build_decoder, card, time_cases  # noqa: E402


def film_gemm_profile(enc, px, cond, reps=20):
    """Device time of the conditioning GEMM (the kernel after the im2col of each eager call), from torch.profiler."""
    enc.set_option("use_cuda_graph", 0)
    enc.forward(px, film_cond=cond)
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(reps):
            enc.forward(px, film_cond=cond)
        torch.cuda.synchronize()
    enc.set_option("use_cuda_graph", 1)
    kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name),
                  key=lambda e: e.time_range.start)
    times, names = [], set()
    for i, e in enumerate(kern[:-1]):
        if "im2col" in e.name:
            times.append(kern[i + 1].time_range.elapsed_us())
            names.add(kern[i + 1].name[:80])
    assert len(times) >= reps // 2, (len(times), reps)         # the profiler may miss the first call's events
    times.sort()
    weight_bytes = enc.cfg.num_layers * 2 * enc.cfg.hidden * enc.cfg.film_dim * 2
    us = times[len(times) // 2]
    return {"kernel": sorted(names), "us_p50": us, "us_min": times[0], "weight_bytes": weight_bytes,
            "tb_per_s_p50": weight_bytes / (us * 1e-6) / 1e12}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/openvla_oft_film.json")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_oft_film.py measures on a CUDA device (B200); there is no CPU path")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "steps": args.steps,
              "model": "OpenVLA-7B shape, random init: DINOv2-L/14 reg4 + SigLIP-so400m/14 (full depth; plain and FiLM "
                       "4096 -> hidden per block), projector, Llama-2-7B-shaped decoder (640 positions, long_forward), "
                       "L1-regression head 28672 -> 4096 -> 7 (2 blocks), proprio projector 8 -> 4096 -> 4096"}
    oft = openvla.oft_libero_config()
    dec = build_decoder(openvla.openvla_oft_7b_config(oft), dev, 32)
    g = torch.Generator(device=dev).manual_seed(args.seed)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=64 * 256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    towers, fused = {}, {}
    for film_dim in (0, 4096):
        d, s = openvla.dinov2_large_reg4_config(), openvla.siglip_so400m_config()
        d.film_dim = s.film_dim = film_dim
        towers[film_dim] = (openvla.VitEncoder.synthetic(d, dev, max_batch=64, seed=100),
                            openvla.VitEncoder.synthetic(s, dev, max_batch=64, seed=101))
        fused[film_dim] = openvla.FusedVisionBackbone(*towers[film_dim], proj)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, dev, max_batch=32, seed=7)
    pp = openvla.ProprioProjector.synthetic(oft.proprio_dim, 4096, dev, max_rows=32, seed=8)
    pres = [openvla.ImagePreprocessor(480, 640, device=dev), openvla.ImagePreprocessor(256, 256, device=dev)]
    pol = {}
    for film in (False, True):
        o2 = openvla.OftConfig(**{**oft.__dict__, "use_film": film})
        o1 = openvla.OftConfig(use_film=film)
        fb = fused[4096 if film else 0]
        pol[("libero", film)] = openvla.OftPolicy(pres, fb, dec, head, o2, proprio_projector=pp)
        pol[("one", film)] = openvla.OftPolicy(pres[0], fb, dec, head, o1)
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
        lay1 = openvla.oft_prompt_layout(ids1, n_patches=256, cfg=pol[("one", True)].cfg)
        cond = openvla.film_language_embedding(dec, lay1)
        kw = dict(proprio=raw, proprio_q01=pq01, proprio_q99=pq99)
        cases = {
            "film_one_camera_chunk": lambda: pol[("one", True)].predict_action_chunk_from_pixels(px1, ids1, q01, q99),
            "one_camera_chunk": lambda: pol[("one", False)].predict_action_chunk_from_pixels(px1, ids1, q01, q99),
            "film_libero_chunk": lambda: pol[("libero", True)].predict_action_chunk_from_pixels(px2, ids2, q01, q99, **kw),
            "libero_chunk": lambda: pol[("libero", False)].predict_action_chunk_from_pixels(px2, ids2, q01, q99, **kw),
            "vision_film": lambda: fused[4096].forward(px1[:, :3], px1[:, 3:], film_cond=cond),
            "vision": lambda: fused[0].forward(px1[:, :3], px1[:, 3:]),
            "language_vector": lambda: openvla.film_language_embedding(dec, lay1),
        }
        t = time_cases(cases, args.steps, args.warmup, check)
        for k in ("film_one_camera_chunk", "film_libero_chunk"):
            out = cases[k]()
            assert out.shape == (B, oft.chunk, oft.action_dim) and bool(torch.isfinite(out).all())
        p50 = {k: v["ms_p50"] for k, v in t.items()}
        result[f"batch{B}"] = {
            "timings_ms": t,
            "film_cost_ms": {"one_camera_chunk": p50["film_one_camera_chunk"] - p50["one_camera_chunk"],
                             "libero_chunk": p50["film_libero_chunk"] - p50["libero_chunk"],
                             "vision": p50["vision_film"] - p50["vision"]},
            "conditioning_gemm": {name: film_gemm_profile(enc, px1[:, :3] if name == "dinov2" else px1[:, 3:], cond)
                                  for name, enc in zip(("dinov2", "siglip"), towers[4096])},
        }
        print(f"batch {B}: " + ", ".join(f"{k} {v:.3f}" for k, v in p50.items()) + " ms")
        print(f"batch {B}: FiLM cost {result[f'batch{B}']['film_cost_ms']}")
        print(f"batch {B}: conditioning GEMMs {result[f'batch{B}']['conditioning_gemm']}")
    check()
    result["card_after"] = card()
    for m in (*pres, *towers[0], *towers[4096], proj, dec, head, pp):
        m.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
