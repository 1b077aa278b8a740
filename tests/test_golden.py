"""Golden vectors produced by the real reference (tests/golden/make_golden.py, build container):
  * CPU (-m "not gpu"): the oracle reproduces them bit-for-bit from the same recipe — this is the
    oracle's pin on machines without the reference source;
  * GPU (-m gpu): the CUDA path against the reference's own CPU results (different device, so the
    tolerance is the reference's bf16-vs-fp32 noise floor, not 1 ulp)."""

import os

import pytest
import torch

from blurr_b200 import synth
from blurr_b200.config import bridge_config, fractal_config, shrink_config
from oracle import pi0_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "pi0_reference_golden.pt")
GOLDEN_FULL = os.path.join(HERE, "golden", "pi0_reference_golden_full.pt")
# How the CPU run that made pi0_reference_golden.pt summed: ATen's kernel set and its intra-op thread count.  The
# thread count sets how CPU GEMMs and reductions split their sums, so fp32 / bf16 bits follow it as much as the torch
# build; the oracle runs with the same count, and the bits are only comparable on the same kernel set.
GOLDEN_CPU_CAPABILITY = "AVX512"
GOLDEN_THREADS = 8

CASES = {
    "shrunk_bridge_s1": lambda: shrink_config(bridge_config(1), 2, 3),
    "shrunk_bridge_s1_stress": lambda: shrink_config(bridge_config(1), 2, 3),
    "shrunk_fractal_s10": lambda: shrink_config(fractal_config(10), 2, 3),
    "full_bridge_s1": lambda: bridge_config(1),
    "full_fractal_s10": lambda: fractal_config(10),
}


def _load(path):
    return torch.load(path, map_location="cpu", weights_only=False)


@pytest.mark.parametrize("name", ["shrunk_bridge_s1", "shrunk_bridge_s1_stress", "shrunk_fractal_s10"])
@pytest.mark.parametrize("tag,dtype", [("fp32", torch.float32), ("bf16", torch.bfloat16)])
def test_oracle_reproduces_reference_golden(name, tag, dtype):
    blob = _load(GOLDEN)
    g = blob[name]
    cfg = CASES[name]()
    cfg.final_action_clip_value = None
    sd = synth.synthetic_state_dict(cfg, 0, torch.float32, stress=g["stress"])
    sd = {k: v.to(dtype) for k, v in sd.items()}
    inp = synth.synthetic_inputs(cfg, g["batch"], dtype=dtype, vary_text=g["vary_text"])
    taps = {}
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        with torch.inference_mode():
            got = O.infer_action(sd, cfg, **synth.call_args(inp), noise=inp["noise"],
                                 tap=lambda n, t: taps.__setitem__(n, t.detach().float()[..., :4, :8].clone()))
    finally:
        torch.set_num_threads(threads)
    if blob["torch"] == torch.__version__ and torch.backends.cpu.get_cpu_capability() == GOLDEN_CPU_CAPABILITY:
        assert torch.equal(got.float(), g[f"actions_{tag}"])
        for n, t in g[f"taps_{tag}"].items():
            assert torch.equal(taps[n], t), n
    else:   # another torch build or CPU kernel set may order reductions differently
        assert (got.float() - g[f"actions_{tag}"]).abs().max().item() <= (1e-4 if tag == "fp32" else 5e-2)
        tol = 1e-4 if tag == "fp32" else 2e-2     # bf16: a few ulps of each activation
        for n, t in g[f"taps_{tag}"].items():
            assert torch.allclose(taps[n], t, rtol=tol, atol=tol), n


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["shrunk_bridge_s1", "shrunk_fractal_s10", "full_bridge_s1", "full_fractal_s10"])
def test_cuda_path_vs_reference_cpu_golden(name):
    from blurr_b200.pizero import PiZeroInference

    path = GOLDEN_FULL if name.startswith("full") else GOLDEN
    if not os.path.isfile(path):
        pytest.skip(f"{os.path.basename(path)} not generated")
    g = _load(path)[name]
    cfg = CASES[name]()
    cfg.final_action_clip_value = None
    sd = synth.synthetic_state_dict(cfg, 0, torch.bfloat16, stress=g["stress"])
    model = PiZeroInference.from_state_dict(cfg, sd, device="cuda")
    del sd
    inp = synth.synthetic_inputs(cfg, g["batch"], dtype=torch.bfloat16, vary_text=g["vary_text"], device="cuda")
    with torch.inference_mode():
        got = model(**synth.call_args(inp), noise=inp["noise"]).float().cpu()
    model._engine.check()
    ref16, ref32 = g["actions_bf16"], g["actions_fp32"]
    e_ours = (got - ref32).abs().max().item()
    e_ref = (ref16 - ref32).abs().max().item()
    e_pair = (got - ref16).abs().max().item()
    clamped = (got.clamp(-1, 1) - ref16.clamp(-1, 1)).abs().max().item()
    print(f"{name}: ours vs ref-fp32 {e_ours:.3e} | ref-bf16(CPU) vs ref-fp32 {e_ref:.3e} | ours vs ref-bf16(CPU) "
          f"{e_pair:.3e} (clamped {clamped:.3e})")
    # the fp32 reference is the tie-breaker: our bf16 error must not exceed the reference's own
    # bf16 error by more than ~one bf16 ulp of the un-clamped range (|a| < 4 -> 1.6e-2)
    assert e_ours <= e_ref + 1.6e-2
    assert clamped <= 1e-2          # north_star tolerance (clamped actions), here against the reference's CPU bf16 run
    model.release_engine()
