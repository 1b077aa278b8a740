"""OpenVLA from camera frames on one GPU: what the device-side image preprocessing costs and saves.

Writes one JSON file with
  * kernel:  the preprocessing kernel alone, 480x640 uint8 -> 2 x 224^2 bf16 (DINOv2 + SigLIP normalisations), batch
             1 and 32: CUDA events around 200 back-to-back launches (per-launch mean), and the kernel's own device
             time from torch.profiler in a separate pass.  The frames (0.9 MB each) stay in L2 across launches.
  * predict_action p50 on the full-size random-init model (DINOv2-L/14 reg4 + SigLIP-so400m towers, the 3-layer
             projector, the 32-layer Llama-2-7B-shaped decoder, as bench.py's openvla leg builds it), batch 1:
             (a) from a device-resident uint8 frame, (b) from prepared bf16 pixel values, (c) from a host uint8
             frame (pageable, copied to the device inside the call).  Each call ends with the token ids on the host.
             The three are measured interleaved, call by call.
  * host:    the PIL + torchvision pipeline of OpenVLA's processor per 480x640 frame on this machine's CPU, for
             comparison (no GPU involved).
with the card name and power limit read in the same run.

    python tools/openvla_frames.py --out profiles/openvla_frames.json
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from blurr_b200 import openvla  # noqa: E402

H, W = 480, 640


def card() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True,
                           timeout=30)
        return {"nvidia_smi": q.stdout.strip(), "torch_device_name": torch.cuda.get_device_name(0)}
    except Exception as e:  # noqa: BLE001 - recorded, not fatal
        return {"nvidia_smi_error": repr(e), "torch_device_name": torch.cuda.get_device_name(0)}


def torchvision_pixels(img: np.ndarray) -> torch.Tensor:
    import torchvision.transforms.functional as TVF
    from PIL import Image
    pil = Image.fromarray(img)
    outs = []
    for m, s in ((openvla.DINOV2_MEAN, openvla.DINOV2_STD), (openvla.SIGLIP_MEAN, openvla.SIGLIP_STD)):
        x = TVF.center_crop(TVF.resize(pil, 224, interpolation=TVF.InterpolationMode.BICUBIC), 224)
        outs.append(TVF.normalize(TVF.to_tensor(x), m, s))
    return torch.vstack(outs).to(torch.bfloat16)


def time_kernel(pre: openvla.ImagePreprocessor, batch: int, dev, launches: int = 200, repeats: int = 5) -> dict:
    g = torch.Generator(device=dev).manual_seed(batch)
    frames = torch.randint(0, 256, (batch, H, W, 3), device=dev, dtype=torch.uint8, generator=g)
    out = torch.empty((batch, 6, 224, 224), device=dev, dtype=torch.bfloat16)
    for _ in range(20):
        pre(frames, out=out)
    torch.cuda.synchronize()
    per_launch = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            pre(frames, out=out)
        e1.record()
        torch.cuda.synchronize()
        per_launch.append(e0.elapsed_time(e1) / launches)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(launches):
            pre(frames, out=out)
        torch.cuda.synchronize()
    dev_us = [e.device_time for e in prof.events() if "resize_bicubic_crop_normalize" in e.name]
    bytes_in, bytes_out = frames.numel(), out.numel() * 2
    ms = statistics.median(per_launch)
    return {"batch": batch, "launches_per_window": launches, "events_ms_per_launch": per_launch, "events_ms_per_launch_median": ms,
            "profiler_kernel_us_p50": statistics.median(dev_us) if dev_us else None, "profiler_kernel_count": len(dev_us),
            "bytes_in": bytes_in, "bytes_out": bytes_out,
            "achieved_gbps_events": (bytes_in + bytes_out) / ms / 1e6,
            "achieved_gbps_kernel": (bytes_in + bytes_out) / (statistics.median(dev_us) * 1e3) if dev_us else None,
            "l2": "frames stay L2-resident across launches (<= 29.5 MB)"}


def build_policy(dev) -> tuple:
    """The full-size random-init model of bench.py's openvla leg (batch 1)."""
    cfg = openvla.openvla_7b_config()
    dec = openvla.LlamaDecoder(cfg, dev, max_batch=1)
    one = openvla.LlamaShapedConfig(**{**cfg.__dict__, "num_layers": 1})
    for layer in range(cfg.num_layers):
        sd = openvla.synthetic_llama_state_dict(one, dev, seed=layer)
        for k, v in sd.items():
            if k.startswith("model.layers.0."):
                dec.set_weight(k.replace("model.layers.0.", f"model.layers.{layer}."), v)
            elif layer == 0:
                dec.set_weight(k, v)
        del sd
    import ctypes as C
    from blurr_b200 import capi
    cos, sin = openvla.rope_tables(openvla.default_inv_freq(cfg.head_dim, cfg.rope_theta, dev), cfg.max_positions)
    torch.cuda.synchronize()
    capi.check(dec.lib.blurr_llm_set_rope_table(dec.handle, C.c_void_p(cos.data_ptr()), C.c_void_p(sin.data_ptr()),
                                                cfg.max_positions))
    capi.check(dec.lib.blurr_llm_finalize(dec.handle))
    g = torch.Generator(device=dev).manual_seed(0)
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(), dev, max_batch=1, seed=100)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(), dev, max_batch=1, seed=101)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    pre = openvla.ImagePreprocessor(H, W, device=dev)
    return openvla.OpenVlaPolicy(pre, openvla.FusedVisionBackbone(dino, sig, proj), dec), (dino, sig, proj, dec, pre)


def time_predict_action(policy, dev, iters: int, warmup: int) -> dict:
    rng = np.random.default_rng(0)
    frame_host = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    frame_dev = torch.as_tensor(frame_host).to(dev)
    px = policy.pixel_values(frame_dev)
    ids = torch.tensor([[1] + list(rng.integers(3, 32000, 24))], device=dev)
    q01, q99 = -np.ones(7), np.ones(7)
    calls = {
        "device_frame": lambda: policy.predict_action(frame_dev, ids, q01, q99),
        "prepared_pixels": lambda: policy.predict_action_from_pixels(px, ids, q01, q99),
        "host_frame": lambda: policy.predict_action(frame_host, ids, q01, q99),
    }
    same = [torch.equal(calls["device_frame"](), calls["prepared_pixels"]()),
            torch.equal(calls["host_frame"](), calls["prepared_pixels"]())]
    times = {k: [] for k in calls}
    for i in range(warmup + iters):
        for name, fn in calls.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()                                      # ends in a device -> host copy of the token ids
            dt = (time.perf_counter() - t0) * 1e3
            if i >= warmup:
                times[name].append(dt)
    res = {name: {"ms_p50": statistics.median(t), "ms_mean": statistics.fmean(t), "ms_min": min(t), "n": len(t)}
           for name, t in times.items()}
    res["device_frame_minus_prepared_pixels_ms_p50"] = res["device_frame"]["ms_p50"] - res["prepared_pixels"]["ms_p50"]
    res["same_actions_from_all_three"] = all(same)
    return res


def time_host_pipeline(n: int = 100) -> dict:
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    for _ in range(5):
        torchvision_pixels(img)
    t = []
    for _ in range(n):
        t0 = time.perf_counter()
        torchvision_pixels(img)
        t.append((time.perf_counter() - t0) * 1e3)
    import PIL
    import torchvision
    return {"ms_p50": statistics.median(t), "ms_min": min(t), "n": n, "torch_threads": torch.get_num_threads(),
            "cpu_count": os.cpu_count(), "pillow": PIL.__version__, "torchvision": torchvision.__version__,
            "note": "PIL bicubic resize + center crop + to_tensor + 2 x normalize + vstack + bf16, one 480x640 frame; "
                    "the copy of the result to the GPU is not included"}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--iters", type=int, default=30, help="timed predict_action calls per variant")
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("openvla_frames.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"card": card(), "frame": [H, W, 3], "output": [6, 224, 224]}
    pre = openvla.ImagePreprocessor(H, W, device=dev)
    img = np.random.default_rng(2).integers(0, 256, (H, W, 3), dtype=np.uint8)
    result["bit_exact_vs_torchvision"] = torch.equal(pre(torch.as_tensor(img).to(dev))[0].cpu().view(torch.int16),
                                                     torchvision_pixels(img).view(torch.int16))
    result["kernel"] = [time_kernel(pre, b, dev) for b in (1, 32)]
    pre.close()
    result["host_pipeline"] = time_host_pipeline()
    policy, parts = build_policy(dev)
    result["predict_action_bs1"] = time_predict_action(policy, dev, args.iters, args.warmup)
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w", encoding="utf-8") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))
    for p in parts:
        p.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
