#!/usr/bin/env python3
"""Benchmark of the Pi-0 Bridge control step (BASELINE.json metric), one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path

A *step* is one control step: one `PiZeroInference.forward` (= `infer_action`, reference
`src/model/vla/pizero.py:473-547`) per episode, producing a chunk of `horizon_steps` = 4 actions.

BASELINE.json's metric has two halves, and every line carries both measurements:
  * `latency`  — configs[1]: Bridge, bf16, ONE episode per GPU, 1 flow step (`--preset blurr`), a fresh image + proprio
                 every control step of a 50-step episode; p50 latency per control step.
  * `batched`  — configs[3]: 64 episodes per GPU, episode-sharded (weights replicated, no data-path collective, one NCCL
                 all_gather of the final actions); actions/s over all GPUs.
Which one is the line's headline (`value`, `ms_per_step`, `config.workload`, `e2e`, `clocks`) is `--workload`:
  auto (default) = `latency` for a single-GPU run on a single-GPU box (the driver's BENCH run), `batched` whenever the run
  is a point of the 1/2/4/8-GPU scaling curve: N > 1, or N = 1 on a box that shows more than one GPU (so that every point
  of the curve, N = 1 included, is the bs=64/GPU workload the metric names and v_N / (N v_1) compares like with like).
The other measurement is still taken and reported under its own key (`latency_bs1` / `batched`).

For N > 1 the batched leg also deals the ranks contiguous 64-episode blocks of ONE seeded global batch
(`blurr_b200.dist.infer_sharded`), gathers the actions over NCCL, and rank 0 recomputes every block locally:
`actions_equal_across_gpus` = `torch.equal` of the two.

`e2e` = the headline workload through the public call with all input tensors copied from pinned host memory and the
actions read back every step (what `src/agent/eval.py:207-218,239` does).  The line also carries the roofline of the
dominant kernel, the whole-step roofline and the CPU baseline (`cpu_baseline`; N = 1 only).
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALG_WEIGHT_BYTES_STEP = 5_793_957_358          # SURVEY.md §8(d): bf16 weights one bs=1, S=1 step depends on
ALG_FLOPS_STEP = 1.2373e12                     # SURVEY.md §8(d), per sample
HORIZON = 4


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed steps of every leg except the batched leg of the latency workload (--batched-steps)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=["auto", "latency", "batched", "openvla"], default="auto",
                    help="headline measurement (see the module docstring)")
    ap.add_argument("--batch", type=int, default=1, help="episodes per GPU of the latency measurement")
    ap.add_argument("--batched", type=int, default=64, help="episodes per GPU of the batched measurement (0 = skip)")
    ap.add_argument("--batched-steps", type=int, default=0, help="timed steps of the batched leg when it is not the headline (0 = 10); --steps times it when it is")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-raw-frames", action="store_true", help="skip the e2e leg that starts from raw camera frames")
    ap.add_argument("--flow-steps", type=int, default=1, help="num_inference_steps (1 = --preset blurr)")
    ap.add_argument("--robot", choices=["bridge", "fractal"], default="bridge", help="config family (BASELINE.json configs[2]: fractal)")
    ap.add_argument("--ring", type=int, default=50, help="distinct pre-staged control-step inputs (one episode)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each timed leg returned as DIR/<name>.npy; with N > 1 GPUs "
                         "rank 0 writes its own episodes (its shard of the batched leg)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batched_steps < 0:
        ap.error("--batched-steps must not be negative")
    return args


def dump_outputs(out_dir, arrays):
    """Save each output as float32 (float64 for integer ids, exact) .npy so that two builds can be compared output
    for output; every input of the run is seeded, so the same arguments give the same inputs."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        t = t.double() if not t.is_floating_point() else t.float()
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.lines = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.lines.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def mark(self):
        """Start of the timed region: only samples taken after this call are reported."""
        self.first = len(self.lines)

    def count(self):
        return len(self.lines) - getattr(self, "first", 0)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines[getattr(self, "first", 0):]:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(args):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def pct(xs, q):
    xs = sorted(xs)
    if not xs:
        return None
    i = min(len(xs) - 1, max(0, int(round(q * (len(xs) - 1)))))
    return xs[i]


def make_ring(cfg, batch, n, device, seed, pinned=False):
    """`n` control-step input sets: same instruction (input_ids / masks / positions), a fresh image,
    proprio and flow noise per step."""
    import torch
    from blurr_b200 import synth
    base = synth.synthetic_inputs(cfg, batch, seed=seed, dtype=torch.bfloat16, vary_text=batch > 1)
    ring = []
    g = torch.Generator().manual_seed(seed + 17)
    for _ in range(n):
        d = dict(base)
        img = torch.randint(0, 256, base["pixel_values"].shape, dtype=torch.uint8, generator=g)
        d["pixel_values"] = synth.process_images(img).to(torch.bfloat16)
        d["proprios"] = (torch.rand(base["proprios"].shape, generator=g) * 2 - 1).to(torch.bfloat16)
        d["noise"] = torch.randn(base["noise"].shape, generator=g).to(torch.bfloat16)
        keys = list(synth.CALL_KEYS) + ["noise"]
        if pinned:
            ring.append({k: d[k].contiguous().pin_memory() for k in keys})
        else:
            ring.append({k: d[k].to(device) for k in keys})
    return ring


class Ctx:
    """What every leg needs: the model, the process group, timing helpers."""

    def __init__(self, args):
        import torch
        from blurr_b200 import synth
        from blurr_b200.config import bridge_config, fractal_config
        from blurr_b200.pizero import PiZeroInference
        self.args = args
        self.world, self.rank, self.local = dist_setup(args)
        self.dev = torch.device("cuda", self.local)
        torch.cuda.set_device(self.dev)
        self.peaks = measured_peaks()
        self.cfg = fractal_config(args.flow_steps) if args.robot == "fractal" else bridge_config(args.flow_steps)
        sd = synth.random_state_dict_on_device(self.cfg, self.dev, seed=0)     # identical replicas on every rank
        self.model = PiZeroInference.from_state_dict(self.cfg, sd, device=self.dev)
        del sd
        self.model.set_engine_options(reserve_batch=max(args.batch, args.batched))
        self.outputs = {}           # leg name -> actions of its last timed step (--dump-outputs)

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x: float) -> float:
        import torch
        if self.world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step(self, r):
        from blurr_b200 import synth
        return self.model(**{k: r[k] for k in synth.CALL_KEYS}, noise=r["noise"])


def timed_device_loop(ctx, ring, K, W, sample_clocks, name):
    """W warm-up + K timed steps on device-resident inputs: CUDA events on the launching stream, barrier +
    synchronize on both sides, max over ranks.  Returns (total_ms, per-step latencies, launches per step, clocks);
    the actions of the last timed step go to `ctx.outputs[name + "_actions"]`."""
    import torch
    model, dev = ctx.model, ctx.dev
    clocks = None
    with torch.inference_mode():
        sampler = ClockSampler(ctx.local) if sample_clocks else None
        if sampler:
            sampler.start()                 # nvidia-smi needs a few 100 ms to come up: start before warm-up
        for i in range(W):
            ctx.step(ring[i % len(ring)])
        model._engine.check()
        launches = model.last_launch_count
        ctx.barrier()
        if sampler:
            sampler.mark()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        evs[0].record()
        for i in range(K):
            actions = ctx.step(ring[i % len(ring)])
            evs[i + 1].record()
        ctx.barrier()
        ctx.outputs[name + "_actions"] = actions
        if sampler:
            # a short timed region ends before nvidia-smi has sampled it a few times: keep the same load
            # running (untimed) until there are enough samples of the clocks under this workload
            tail_steps, t_tail = 0, time.perf_counter()
            while sampler.proc is not None and sampler.count() < 6 and time.perf_counter() - t_tail < 3.0:
                ctx.step(ring[tail_steps % len(ring)])
                tail_steps += 1
                if tail_steps % 8 == 0:
                    torch.cuda.synchronize(dev)
            torch.cuda.synchronize(dev)
            clocks = sampler.stop()
            clocks["untimed_tail_steps"] = tail_steps
        model._engine.check()       # device-side flags (pipeline time-outs, bad token ids): results are invalid if set
    total_ms = ctx.max_over_ranks(evs[0].elapsed_time(evs[K]))
    lat = [evs[i].elapsed_time(evs[i + 1]) for i in range(K)]
    return total_ms, lat, int(launches), clocks


def timed_e2e_loop(ctx, hring, K, W, B):
    """The same steps through the public call from pinned host memory: H2D of all inputs and D2H of the actions
    inside the timed region (wall clock between synchronised points, max over ranks)."""
    import torch
    from blurr_b200 import synth
    dev = ctx.dev
    h2d = sum(t.numel() * t.element_size() for t in hring[0].values())
    host_out = torch.empty((B, HORIZON, ctx.cfg.action_dim), dtype=torch.float32).pin_memory()
    with torch.inference_mode():
        def e2e_step(r):
            d = {k: v.to(dev, non_blocking=True) for k, v in r.items()}
            a = ctx.model(**{k: d[k] for k in synth.CALL_KEYS}, noise=d["noise"])
            host_out.copy_(a.float(), non_blocking=False)        # `actions.float().cpu()` (eval.py:239)
            return a
        for i in range(W):
            e2e_step(hring[i % len(hring)])
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(K):
            e2e_step(hring[i % len(hring)])
        torch.cuda.synchronize(dev)
        e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
        ctx.barrier()
        ctx.model._engine.check()
    d2h = host_out.numel() * host_out.element_size()
    return {"value": ctx.world * B * HORIZON * K / e2e_s, "unit": "actions/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3 / K}, host_out


def leg_latency(ctx, K, W, headline):
    """configs[1]: one episode per GPU, p50 latency per control step."""
    args, cfg, world, rank = ctx.args, ctx.cfg, ctx.world, ctx.rank
    B = args.batch
    ring = make_ring(cfg, B, min(args.ring, max(K, 1)), ctx.dev, seed=1234 + rank)
    total_ms, lat, launches, clocks = timed_device_loop(ctx, ring, K, W, sample_clocks=headline, name="latency")
    wl = "bridge_bs1_blurr_preset_50step_episode (BASELINE.json configs[1])"
    if args.robot == "fractal" or args.flow_steps != 1:
        wl = f"{args.robot}_bs1_{args.flow_steps}_flow_steps (BASELINE.json configs[2])"
    res = {"workload": wl, "episodes_per_gpu": B,
           "steps": K, "warmup": W, "value": world * B * HORIZON * K / (total_ms / 1e3), "unit": "actions/s",
           "ms_per_step": total_ms / K, "gpu_launches_per_step": launches,
           "latency_ms": {"p50": pct(lat, 0.5), "p90": pct(lat, 0.9), "mean": statistics.fmean(lat), "min": min(lat),
                          "note": "per control step at this rank, CUDA events, device-resident inputs"},
           "clocks": clocks}
    if B == 1 and args.flow_steps == 1:
        t_hbm = ALG_WEIGHT_BYTES_STEP / (ctx.peaks["hbm_gbs"] * 1e9) * 1e3
        res["step_roofline"] = {
            "hbm_time_ms": t_hbm, "tensor_time_ms": ALG_FLOPS_STEP / (ctx.peaks["bf16_tflops"] * 1e12) * 1e3,
            "frac_of_hbm_roofline": t_hbm / pct(lat, 0.5), "target_frac": 1 / 1.5, "target_p50_ms": 1.5 * t_hbm,
            "alg_bytes_per_step": ALG_WEIGHT_BYTES_STEP, "peaks": ctx.peaks["source"]}
    if headline and B == 1 and args.flow_steps == 1:
        res["stages"] = stage_breakdown(ctx, ring)
    if headline or world == 1:
        hring = make_ring(cfg, B, min(8, len(ring)), ctx.dev, seed=4321 + rank, pinned=True)
        res["e2e"], host_out = timed_e2e_loop(ctx, hring, K, W, B)
        if not args.no_raw_frames:
            res["e2e_raw_frames"] = leg_raw_frames(ctx, K, W, B, host_out)
    return res


# SURVEY.md 8(d): per-stage floors of one bs=1, S=1 control step (weights bytes / FLOPs of each stage)
STAGE_ALG = {"siglip+projector": (0.830e9, 220.2e9), "gemma_prefill": (3.746e9, 1013.9e9),
             "proprio+action_experts": (0.589e9 + 0.629e9, 3.3e9)}


def stage_breakdown(ctx, ring, n=30):
    """Time of each stage run ALONE under the real launch regime (engine option `stage_mask`: the step with only that
    stage's kernels; results are meaningless, timings are not) beside its HBM / tensor floor.  The stages of a full step
    overlap (the experts run on side streams under the prefill), so the parts do not add up to the step."""
    import torch
    eng, dev, peaks = ctx.model._engine, ctx.dev, ctx.peaks
    out = {}
    try:
        for name, mask in (("siglip+projector", 1), ("gemma_prefill", 2), ("proprio+action_experts", 4)):
            eng.set_option("stage_mask", mask)
            with torch.inference_mode():
                for i in range(4):
                    ctx.step(ring[i % len(ring)])
                torch.cuda.synchronize(dev)
                ts = []
                for i in range(n):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); ctx.step(ring[i % len(ring)]); b.record()
                    torch.cuda.synchronize(dev)
                    ts.append(a.elapsed_time(b))
            by, fl = STAGE_ALG[name]
            t_hbm = by / (peaks["hbm_gbs"] * 1e9) * 1e3
            t_tc = fl / (peaks["bf16_tflops"] * 1e12) * 1e3
            ms = statistics.median(ts)
            out[name] = {"ms": ms, "hbm_floor_ms": t_hbm, "tensor_floor_ms": t_tc, "frac_of_floor": max(t_hbm, t_tc) / ms}
    finally:
        eng.set_option("stage_mask", 7)
    out["note"] = ("each stage alone (stage_mask), p50 of %d launches incl. the input staging kernels; floors = SURVEY.md 8(d) "
                   "bytes / measured copy bandwidth and FLOPs / measured burst bf16" % n)
    return out


def leg_raw_frames(ctx, K, W, B, host_out):
    """e2e from RAW observations (SURVEY.md 8(f) row 1): 480x640x3 uint8 camera frames + raw float64 proprio in pinned
    host memory; per step: H2D of the raw observation, device-side cv2-equivalent Lanczos resize + normalise + proprio
    normalise, the model graph, D2H of the actions.  Beside it: what the reference does on the host CPU for the same
    step (cv2 resize + VLAProcessor + mask / position building), timed on this box."""
    import torch
    from blurr_b200 import synth
    from blurr_b200.episode import Episode
    cfg, dev, rank, world = ctx.cfg, ctx.dev, ctx.rank, ctx.world
    dim = int(cfg.proprio_dim)      # 7 (Bridge) or 8 (Fractal)
    stats = {"p01": ([0.17, -0.21, -0.04, -3.1, -0.5, -1.2, 0.0, -0.3])[:dim], "p99": ([0.45, 0.24, 0.28, 3.1, 0.6, 1.3, 1.0, 0.3])[:dim]}
    base = synth.synthetic_inputs(cfg, B, seed=99 + rank, dtype=torch.bfloat16, vary_text=B > 1)
    ep = Episode(ctx.model, base["input_ids"], base["attention_mask"], (480, 640), stats, "bound")
    g = torch.Generator().manual_seed(5 + rank)
    frames = [torch.randint(0, 256, (B, 480, 640, 3), dtype=torch.uint8, generator=g).pin_memory() for _ in range(4)]
    props = [(torch.rand((B, dim), generator=g, dtype=torch.float64) * 0.4).pin_memory() for _ in range(4)]
    noise = base["noise"].to(dev)
    with torch.inference_mode():
        def raw_step(i):
            a = ep.step(frames[i % 4], props[i % 4], noise=noise)
            host_out.copy_(a.float(), non_blocking=False)
        for i in range(W):
            raw_step(i)
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(K):
            raw_step(i)
        torch.cuda.synchronize(dev)
        raw_s = ctx.max_over_ranks(time.perf_counter() - t0)
        ctx.barrier()
    ep.close()
    raw = {"value": world * B * HORIZON * K / raw_s, "unit": "actions/s", "ms_per_step": raw_s * 1e3 / K,
           "h2d_bytes_per_step": B * (480 * 640 * 3 + dim * 8), "d2h_bytes_per_step": host_out.numel() * host_out.element_size(),
           "observation": f"480x640x3 uint8 frame + {dim} float64 proprio per episode, pinned host memory",
           "device_ops": "cv2.INTER_LANCZOS4-equivalent resize + VLAProcessor normalise + bf16 cast + normalize_bound (bit-exact)"}
    if rank == 0 and world == 1:
        raw["reference_host_preprocess"] = reference_host_preprocess_ms(cfg, base, B)
    return raw


def global_batch(cfg, episodes_per_gpu, world, seed):
    """ONE seeded batch of `episodes_per_gpu * world` episodes (distinct images, per-episode instruction lengths),
    identical on every rank; rank r owns the contiguous block r (blurr_b200.dist.shard_inputs)."""
    import torch
    from blurr_b200 import synth
    return synth.synthetic_inputs(cfg, episodes_per_gpu * world, seed=seed, dtype=torch.bfloat16, vary_text=True)


def leg_batched(ctx, K, W, headline):
    """configs[3]: 64 episodes per GPU, episode-sharded; actions/s over all GPUs, fraction of the bf16 tensor roofline,
    and for N > 1 the cross-GPU equality check of SURVEY.md 8(d) config 4."""
    import torch
    from blurr_b200 import dist as bdist
    from blurr_b200 import synth
    args, cfg, world, rank, dev = ctx.args, ctx.cfg, ctx.world, ctx.rank, ctx.dev
    Bb = args.batched
    keys = list(synth.CALL_KEYS) + ["noise"]
    # two input sets per rank (2 x 30 MB on the device): this rank's blocks of two seeded global batches
    ring = []
    for s in range(2):
        glob = global_batch(cfg, Bb, world, seed=7000 + s)
        local = bdist.shard_inputs({k: glob[k] for k in keys}, world, rank)
        ring.append({k: v.to(dev) for k, v in local.items()})
        if s == 0:
            check_inputs = glob
    total_ms, lat, launches, clocks = timed_device_loop(ctx, ring, K, W, sample_clocks=headline, name="batched")
    value = world * Bb * HORIZON * K / (total_ms / 1e3)
    flops = ALG_FLOPS_STEP * Bb * K / (total_ms / 1e3) / 1e12          # per GPU
    res = {"workload": "bridge_bs64_per_gpu_episode_sharded (BASELINE.json configs[3])", "episodes_per_gpu": Bb,
           "steps": K, "warmup": W, "value": value, "actions_per_sec": value, "unit": "actions/s",
           "ms_per_step": total_ms / K, "gpu_launches_per_step": launches, "clocks": clocks,
           "latency_ms": {"p50": pct(lat, 0.5), "p90": pct(lat, 0.9), "mean": statistics.fmean(lat), "min": min(lat),
                          "note": "per 64-episode control step at this rank"},
           "tensor_roofline": {"bound": "tensor", "achieved": flops, "peak": ctx.peaks["bf16_tflops_sustained"],
                               "unit": "TFLOP/s", "frac": flops / ctx.peaks["bf16_tflops_sustained"],
                               "note": "algorithmic FLOPs per GPU / step time, of " + ctx.peaks["source"] + " sustained cuBLAS bf16"}}
    if headline:
        hring = []
        for r in ring:
            hring.append({k: v.cpu().contiguous().pin_memory() for k, v in r.items()})
        res["e2e"], _ = timed_e2e_loop(ctx, hring, K, W, Bb)
    # ---- cross-GPU equality: the gathered actions of the sharded run == the same blocks computed on ONE GPU ----
    if world > 1:
        with torch.inference_mode():
            dev_inputs = {k: check_inputs[k].to(dev) for k in keys}
            step_fn = lambda **kw: ctx.model(**{k: kw[k] for k in synth.CALL_KEYS}, noise=kw["noise"])
            gathered = bdist.infer_sharded(step_fn, dev_inputs)                 # NCCL all_gather, every rank gets all blocks
            ctx.model._engine.check()
            equal = None
            if rank == 0:
                blocks = []
                for r in range(world):                                          # one 64-episode block at a time, on this GPU
                    blk = bdist.shard_inputs(dev_inputs, world, r)
                    blocks.append(step_fn(**blk).clone())
                ctx.model._engine.check()
                equal = bool(torch.equal(torch.cat(blocks, 0), gathered))
            ctx.barrier()
        res["actions_equal_across_gpus"] = equal
        res["equality_check"] = (f"{world} x {Bb} episodes of one seeded global batch: NCCL-gathered actions of the sharded run vs "
                                 "the same blocks run one at a time on rank 0 (equal per-GPU batch size), torch.equal")
    return res


def run_ours(args):
    import torch
    if args.workload == "openvla":
        return run_openvla(args)
    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    visible = torch.cuda.device_count()
    workload = args.workload
    if workload == "auto":
        workload = "latency" if (world == 1 and visible == 1) or args.batched <= 0 else "batched"
    K, W = args.steps, max(args.warmup, 3)

    # The dominant kernel alone, before anything else has run on this GPU: measured after a 64-episode step the same
    # launches take 47-52 us instead of 38 (tools/roofline_state_probe.py: it follows the big engine's presence and
    # disappears when that engine is released), which made this number bimodal from run to run.
    roof = dominant_kernel_roofline(ctx.dev, ctx.peaks) if (rank == 0 and not args.no_roofline) else None

    legs = {}
    if workload == "latency":
        legs["latency"] = leg_latency(ctx, K, W, headline=True)
        if args.batched > 0:
            legs["batched"] = leg_batched(ctx, args.batched_steps or 10, 3, headline=False)
        head = legs["latency"]
    else:
        legs["batched"] = leg_batched(ctx, K, W, headline=True)
        legs["latency"] = leg_latency(ctx, K, W, headline=False)
        head = legs["batched"]

    line = {
        "metric": "pi0_bridge_actions_per_sec", "value": head["value"], "unit": "actions/s",
        "n_gpus": world, "steps": head["steps"], "warmup": head["warmup"], "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (random-init weights, random uint8 images, random proprio, injected flow noise)",
        "config": {"workload": head["workload"], "episodes_per_gpu": head["episodes_per_gpu"],
                   "flow_steps": args.flow_steps, "actions_per_step": HORIZON,
                   "parallelism": f"episode-sharded x{world}, weights replicated",
                   "workload_rule": f"--workload {args.workload}: visible GPUs {visible}, N {world} -> {workload}",
                   "l2": "inputs larger than L2: each step streams 5.79 GB of weights (L2 is 126 MB)",
                   "cuda_graph": True},
        "latency_ms": legs["latency"]["latency_ms"],
        "e2e": head.get("e2e"),
        "gpu_launches": head["gpu_launches_per_step"] * head["steps"],
        "gpu_launches_per_step": head["gpu_launches_per_step"],
        "clocks": head["clocks"],
        "latency_bs1": {k: v for k, v in legs["latency"].items() if k != "clocks" or workload != "latency"},
    }
    if "step_roofline" in legs["latency"]:
        line["step_roofline"] = legs["latency"]["step_roofline"]
    if "stages" in legs["latency"]:
        line["stages"] = legs["latency"]["stages"]
    if "e2e_raw_frames" in legs["latency"]:
        line["e2e_raw_frames"] = legs["latency"]["e2e_raw_frames"]
    if "batched" in legs:
        line["batched"] = {k: v for k, v in legs["batched"].items() if k != "clocks" or workload != "batched"}
        if "actions_equal_across_gpus" in legs["batched"]:
            line["actions_equal_across_gpus"] = legs["batched"]["actions_equal_across_gpus"]
    # ---------------- roofline of the dominant kernel (rank 0) ----------------
    if roof is not None:
        line["roofline"] = roof
    # ---------------- CPU baseline (rank 0, N = 1) ----------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(ctx.cfg, ctx.model, warm=1, timed=2)
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ctx.outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def run_openvla(args):
    """BASELINE.json configs[4]: OpenVLA-7B-shaped 7-token greedy action decode with a KV cache, batch 1 and 32 -
    the Llama-2-7B-shaped language model behind include/blurr_llm.h on random-init weights and random projected patch
    embeddings (the vision backbone is not part of this leg).  One "step" = one predict_action's language-model work:
    prefill of 1 + 256 + 24 prompt positions, then 7 greedy tokens.  Prints its own JSON line (metric
    openvla7b_shaped_action_chunks_per_sec)."""
    import torch
    from blurr_b200 import openvla
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    peaks = measured_peaks()
    cfg = openvla.openvla_7b_config()
    prompt, n_new = 1 + 256 + 24, 7
    K, W = args.steps, max(args.warmup, 3)
    dec = openvla.LlamaDecoder(cfg, dev, max_batch=32)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    # weights layer by layer: the 13.5 GB state_dict never exists twice
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
    import ctypes as C
    from blurr_b200 import capi
    capi.check(dec.lib.blurr_llm_set_rope_table(dec.handle, C.c_void_p(cos.data_ptr()), C.c_void_p(sin.data_ptr()), cfg.max_positions))
    capi.check(dec.lib.blurr_llm_finalize(dec.handle))
    hbm = peaks["hbm_gbs"]
    # vision side: full-depth DINOv2-L/14 (reg4) + SigLIP-so400m/14 towers (second-to-last block) and the 3-layer projector
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(), dev, max_batch=32, seed=100)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(), dev, max_batch=32, seed=101)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], dev, max_rows=32 * 256)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=dev, generator=g) * 0.02).to(torch.bfloat16),
                       torch.zeros(n_out, device=dev, dtype=torch.bfloat16))
    fused = openvla.FusedVisionBackbone(dino, sig, proj)
    n_text = prompt - 1 - 256
    out, outputs = {}, {}
    for B in (1, 32):
        ring = [(torch.randn((B, prompt, cfg.hidden), device=dev, generator=g) * 0.5).to(torch.bfloat16) for _ in range(4)]
        host = [r.cpu().pin_memory() for r in ring]
        res = {}
        # vision towers + projector alone
        px = (torch.rand((B, 3, 224, 224), device=dev, generator=g) * 2 - 1).to(torch.bfloat16)
        ids_prompt = torch.randint(3, cfg.vocab - 100, (B, 1 + n_text), device=dev, generator=g)
        for _ in range(W):
            fused.forward(px, px)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        evs[0].record()
        for i in range(K):
            fused.forward(px, px)
            evs[i + 1].record()
        torch.cuda.synchronize()
        lat = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(K))
        res["vision_towers_and_projector"] = {"ms_p50": lat[len(lat) // 2], "launches": dino.last_launch_count + sig.last_launch_count + 4}

        def full_step():
            patch = fused.forward(px, px)
            return dec.generate(openvla.build_prompt_embeds(dec, ids_prompt, patch), n_new)
        for _ in range(W):
            full_step()
        dec.check()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        evs[0].record()
        for i in range(K):
            full_step()
            evs[i + 1].record()
        torch.cuda.synchronize()
        dec.check()
        lat = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(K))
        res["predict_action_full"] = {"ms_p50": lat[len(lat) // 2], "ms_mean": evs[0].elapsed_time(evs[K]) / K,
                                      "note": "pixels -> DINOv2 + SigLIP -> projector -> [BOS] + 256 patches + prompt tokens -> 7 greedy tokens"}
        for label, n in (("prefill_plus_1", 1), ("predict_action", n_new)):
            for i in range(W):
                dec.generate(ring[i % 4], n)
            dec.check()
            sampler = ClockSampler(0) if (label == "predict_action" and B == 1) else None
            if sampler:
                sampler.start()
                t0 = time.perf_counter()
                while sampler.count() < 3 and time.perf_counter() - t0 < 3.0:
                    dec.generate(ring[0], n)
                    torch.cuda.synchronize()
                sampler.mark()
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
            evs[0].record()
            for i in range(K):
                ids = dec.generate(ring[i % 4], n)
                evs[i + 1].record()
            torch.cuda.synchronize()
            dec.check()
            outputs[f"bs{B}_{label}_token_ids"] = ids
            lat = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(K))
            res[label] = {"ms_p50": lat[len(lat) // 2], "ms_mean": evs[0].elapsed_time(evs[K]) / K, "launches": dec.last_launch_count}
            if sampler:
                res["clocks"] = sampler.stop()
        # end to end: pinned host prompt embeddings -> device -> generate -> token ids on the host
        ids_host = torch.empty((B, n_new), dtype=torch.int64).pin_memory()
        stage = torch.empty_like(ring[0])
        t_e2e = []
        for i in range(W + K):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            stage.copy_(host[i % 4], non_blocking=True)
            ids = dec.generate(stage, n_new)
            ids_host.copy_(ids, non_blocking=True)
            torch.cuda.synchronize()
            if i >= W:
                t_e2e.append((time.perf_counter() - t0) * 1e3)
        t_e2e.sort()
        per_tok = (res["predict_action"]["ms_mean"] - res["prefill_plus_1"]["ms_mean"]) / (n_new - 1)
        wb = dec.weight_bytes_per_token
        res.update({
            "batch": B, "prompt_positions": prompt, "new_tokens": n_new,
            "decode_ms_per_token": per_tok,
            "decode_weight_stream": {"bytes_per_token": wb, "achieved_gbps": wb / per_tok / 1e6, "peak_gbps": hbm,
                                     "frac": wb / per_tok / 1e6 / hbm, "hbm_floor_ms": wb / hbm / 1e6},
            "action_chunks_per_sec": B * 1e3 / res["predict_action"]["ms_mean"],
            "action_chunks_per_sec_full_model": B * 1e3 / res["predict_action_full"]["ms_mean"],
            "e2e": {"ms_p50": t_e2e[len(t_e2e) // 2], "action_chunks_per_sec": B * 1e3 / (sum(t_e2e) / len(t_e2e)),
                    "h2d_bytes_per_step": stage.numel() * 2, "d2h_bytes_per_step": ids_host.numel() * 8},
        })
        out[f"bs{B}"] = res
    head = out["bs1"]
    line = {
        "metric": "openvla7b_shaped_action_chunks_per_sec", "value": head["action_chunks_per_sec"], "unit": "action chunks/s",
        "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": head["predict_action"]["ms_mean"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (random-init Llama-2-7B-shaped weights, random projected patch embeddings)",
        "config": {"workload": "openvla7b_shaped_bs1_7_token_decode (BASELINE.json configs[4]; headline value = language model, "
                               "openvla.bs*.predict_action_full = with the DINOv2 + SigLIP towers and the projector)",
                   "prompt_positions": prompt, "new_tokens": n_new, "layers": cfg.num_layers, "hidden": cfg.hidden,
                   "l2": "inputs larger than L2: every token streams 13.2 GB of weights", "cuda_graph": True},
        "e2e": {"value": head["e2e"]["action_chunks_per_sec"], "unit": "action chunks/s",
                "h2d_bytes_per_step": head["e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": head["e2e"]["d2h_bytes_per_step"]},
        "gpu_launches": head["predict_action"]["launches"] * K, "gpu_launches_per_step": head["predict_action"]["launches"],
        "clocks": head.get("clocks"),
        "roofline": {"bound": "hbm", "achieved": head["decode_weight_stream"]["achieved_gbps"], "peak": hbm, "unit": "GB/s",
                     "frac": head["decode_weight_stream"]["frac"], "traffic": None,
                     "kernel": "one decode step (all weight-streaming GEMMs of a token)", "peak_source": peaks["source"]},
        "parity": "pinned against transformers 5.5 LlamaForCausalLM (tests/test_gpu_llm.py); unpinned against the reference's remote code",
        "openvla": out,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    dec.close()
    return 0


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the
    committed `ncu --set full` capture (profiles/ncu_gateup_traffic.json); None when there is none."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_gateup_traffic.json")
    try:
        with open(path) as f:
            return float(json.load(f)["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        return None


def reference_host_preprocess_ms(cfg, base, batch):
    """The per-step host work of the reference's control loop (env_adapter/simpler.py:52-98 and
    agent/eval.py:170-183) on this box's CPU: cv2 Lanczos resize (the oracle's restatement when cv2 is
    missing), VLAProcessor normalisation, normalize_bound, mask / position building, casts to bf16."""
    import numpy as np
    import torch
    from blurr_b200 import masks
    from oracle import preprocess_oracle as P
    try:
        import cv2
        resize = lambda im: cv2.resize(im, (224, 224), interpolation=cv2.INTER_LANCZOS4)
        kind = "cv2 " + cv2.__version__
    except ImportError:
        resize = lambda im: P.resize_lanczos4_u8(im, 224, 224)
        kind = "oracle restatement (cv2 not importable)"
    rng = np.random.default_rng(0)
    frames = rng.integers(0, 256, (batch, 480, 640, 3), dtype=np.uint8)
    stats = {"p01": [0.17, -0.21, -0.04, -3.1, -0.5, -1.2, 0.0], "p99": [0.45, 0.24, 0.28, 3.1, 0.6, 1.3, 1.0]}
    n_it = cfg["max_image_text_tokens"]

    def one():
        for b in range(batch):
            small = resize(frames[b])
            px = P.process_images(torch.as_tensor(small, dtype=torch.uint8).permute(2, 0, 1)[None]).to(torch.bfloat16)
            P.preprocess_proprio(rng.normal(0.2, 0.2, 7), stats, "bound")
        cm, *_ = masks.build_causal_mask_and_position_ids(base["attention_mask"], torch.bfloat16, n_it, cfg["cond_steps"],
                                                          cfg["horizon_steps"])
        masks.split_full_mask_into_submasks(cm, n_it, cfg["cond_steps"], cfg["horizon_steps"])
        return px
    for _ in range(3):
        one()
    t0 = time.perf_counter()
    n = 20
    for _ in range(n):
        one()
    return {"ms_per_step": (time.perf_counter() - t0) * 1e3 / n, "resize": kind,
            "note": "host CPU time the reference spends per control step before the model call; not part of its model-only latency"}


def dominant_kernel_roofline(dev, peaks):
    """The Gemma gate/up GEMM + GeGLU (32768 x 2048 weights, 276 tokens): 46 % of the step's bytes.
    Times the kernel through its C-ABI operator entry point on 4 rotating weight buffers (537 MB
    > L2) with CUDA events on the launching stream."""
    import ctypes as C
    import torch
    from blurr_b200 import capi
    lib = capi.load_library()
    N, Kd, T = 32768, 2048, 276
    nbuf, iters = 4, 40
    # fresh device memory for the weight ring: blocks carved out of the caching allocator's recycled segments (the legs
    # before this one free several GB) made this measurement bimodal from run to run (38 vs 47 us per launch)
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()
    Wall = torch.empty((nbuf, N, Kd), device=dev, dtype=torch.bfloat16).uniform_(-0.02, 0.02)
    Ws = [Wall[i] for i in range(nbuf)]
    X = torch.randn((T, Kd), device=dev, dtype=torch.bfloat16)
    out = torch.empty((T, N // 2), device=dev, dtype=torch.bfloat16)
    stream = torch.cuda.current_stream(dev)
    sp = C.c_void_p(stream.cuda_stream)

    def launch(i):
        # ldw = 0: tile-packed weights, the layout the engine streams (random values: no packing pass needed)
        return lib.blurr_op_gemm_async(sp, C.c_void_p(Ws[i % nbuf].data_ptr()), N, Kd, 0, C.c_void_p(X.data_ptr()), T, Kd,
                                 capi.EPI_GEGLU, 1, None, C.c_void_p(out.data_ptr()), N // 2, None)
    for i in range(nbuf):
        capi.check(launch(i))
    torch.cuda.synchronize(dev)
    # (a) back to back, one event pair around `iters` launches on the launching stream: the average launch duration in
    #     the regime the step runs in (successive kernels overlap their set-up through programmatic dependent launch)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(stream)
    for i in range(iters):
        capi.check(launch(i))
    e.record(stream)
    torch.cuda.synchronize(dev)
    ms = s.elapsed_time(e) / iters
    # (b) isolated launches (synchronise in between): includes the full launch latency of a cluster kernel
    times = []
    for i in range(10):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        capi.check(launch(i))
        e.record(stream)
        torch.cuda.synchronize(dev)
        times.append(s.elapsed_time(e))
    alg_bytes = N * Kd * 2
    achieved = alg_bytes / (ms / 1e3) / 1e9
    return {"bound": "hbm", "kernel": "gemm_tcp2_kernel<EPI_GEGLU> (Gemma gate/up, 276 tokens, persistent CTA pairs)",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": ncu_traffic_bytes(), "alg_bytes_per_launch": alg_bytes, "ms_per_launch": ms,
            "ms_isolated_launch_median": statistics.median(times), "launches_timed": iters,
            "note": "algorithmic bytes = the 32768x2048 bf16 weight tile stream; peak = " + peaks["source"] + " copy bandwidth"}


def cpu_baseline(cfg, model, warm=1, timed=2, state_dict=None):
    """The reference's CPU path on the box's host cores: fp32, bs=1, full-size model (BASELINE.json configs[0]) —
    the unmodified reference when reachable (`kind: "reference"`, see run_reference), else the oracle port."""
    import torch
    from blurr_b200 import synth
    from oracle import pi0_oracle as O
    from oracle import ref_harness
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if state_dict is None:
        state_dict = {k: v.detach().to("cpu", torch.float32) for k, v in model.state_dict().items()}
    inp = synth.synthetic_inputs(cfg, 1, dtype=torch.float32)
    kind = "port"
    call = lambda: O.infer_action(state_dict, cfg, **synth.call_args(inp), noise=inp["noise"])
    if ref_harness.reference_available():
        try:
            ref = ref_harness.load_reference_model(cfg, state_dict, torch.float32)
            def call():
                with ref_harness.patched_randn(inp["noise"]):
                    return ref(**{k: (v.clone() if k == "pixel_values" else v) for k, v in synth.call_args(inp).items()})
            kind = "reference"
        except Exception as exc:
            print(f"reference import failed ({type(exc).__name__}: {exc}); timing the port", file=sys.stderr)
    ts = []
    with torch.inference_mode():
        for i in range(warm + timed):
            t0 = time.perf_counter()
            call()
            dt = time.perf_counter() - t0
            if i >= warm:
                ts.append(dt)
    sec = statistics.median(ts)
    return {"value": HORIZON / sec, "unit": "actions/s", "cores": cores, "kind": kind,
            "ms_per_step": sec * 1e3,
            "sample": f"{timed} full-size Bridge control steps (bs=1, fp32, 1 flow step) after {warm} warm-up; "
                      f"torch {torch.__version__} with {torch.get_num_threads()} threads"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, rank 0 only.
    When the unmodified reference is reachable (`/root/reference` in the build container, the copy that
    `__graft_entry__.build()` ships in the git-ignored `baseline/_ref/` on the GPU box) it is the thing timed
    (`kind: "reference"`): `PiZeroInference` imported through `oracle/ref_harness.py`, called exactly like
    `scripts/benchmark_pi0.py:238-242`.  Otherwise its pinned restatement, the oracle (`kind: "port"`).
    fp32 on all host cores, bs=1, the same synthetic inputs every step, mean over the timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from blurr_b200 import synth
    from blurr_b200.config import bridge_config
    from oracle import pi0_oracle as O
    from oracle import ref_harness
    cfg = bridge_config(args.flow_steps)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synth.synthetic_state_dict(cfg, 0, torch.float32)
    inp = synth.synthetic_inputs(cfg, 1, dtype=torch.float32)
    kind = "port"
    call = lambda: O.infer_action(sd, cfg, **synth.call_args(inp), noise=inp["noise"])
    if ref_harness.reference_available():
        try:
            model = ref_harness.load_reference_model(cfg, sd, torch.float32)
            def call():
                with ref_harness.patched_randn(inp["noise"]):
                    return model(**{k: (v.clone() if k == "pixel_values" else v) for k, v in synth.call_args(inp).items()})
            kind = "reference"
        except Exception as exc:       # a broken shipped copy must not take the arm down: fall back to the port
            print(f"reference import failed ({type(exc).__name__}: {exc}); timing the port", file=sys.stderr)
    W = max(1, min(args.warmup, 2))
    ts = []
    with torch.inference_mode():
        for _ in range(W):
            call()
        for _ in range(args.steps):
            t0 = time.perf_counter()
            actions = call()
            ts.append(time.perf_counter() - t0)
    sec = statistics.fmean(ts)
    value = HORIZON / sec
    what = ("the unmodified reference PiZeroInference (" + ref_harness.REF_ROOT + ")") if kind == "reference" else \
        "the oracle port of the reference's op sequence (reference tree not reachable)"
    sample = (f"{what}: {len(ts)} full-size Bridge control steps (bs=1, fp32, {args.flow_steps} flow "
              f"step, identical inputs every step, mean) after {W} warm-up; torch {torch.__version__}, "
              f"{cores} threads")
    line = {
        "impl": "reference", "metric": "pi0_bridge_actions_per_sec", "value": value, "unit": "actions/s",
        "n_gpus": args.gpus, "steps": len(ts), "warmup": W, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "bridge_bs1_blurr_preset_50step_episode (BASELINE.json configs[0]: the reference's CPU-runnable case)",
                   "episodes_per_gpu": 1, "flow_steps": args.flow_steps, "actions_per_step": HORIZON,
                   "parallelism": "host CPU, rank 0 only",
                   "differs_from_gpu_arm": "fp32 instead of bf16, at most 2 warm-up steps, one episode whatever the GPU arm's batch"},
        "cpu_baseline": {"value": value, "unit": "actions/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "actions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"reference_actions": actions})
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
