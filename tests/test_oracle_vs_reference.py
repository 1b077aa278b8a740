"""Pins the oracle (`oracle/pi0_oracle.py`) against the *unmodified reference*, imported from the source tree
that `oracle/ref_harness.py` finds (`BLURR_REF_ROOT`); skipped without it — the committed golden vectors in
tests/golden/ carry the infer_action part of the check to other machines."""

import pytest
import torch

from blurr_b200 import synth
from blurr_b200.config import bridge_config, fractal_config, shrink_config
from oracle import pi0_oracle as O
from oracle import ref_harness

pytestmark = pytest.mark.skipif(not ref_harness.reference_available(),
                                reason="reference source not found (set BLURR_REF_ROOT)")


def _ref_model(cfg, sd, dtype):
    return ref_harness.load_reference_model(cfg, sd, dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("steps,fractal", [(1, False), (3, True)])
def test_infer_action_bit_identical(dtype, steps, fractal):
    base = fractal_config(steps) if fractal else bridge_config(steps)
    cfg = shrink_config(base, 2, 2)
    cfg.final_action_clip_value = None
    sd = synth.synthetic_state_dict(cfg, 0, torch.float32)
    model = _ref_model(cfg, sd, dtype)
    sd_t = model.state_dict()
    inp = synth.synthetic_inputs(cfg, 2, dtype=dtype, vary_text=True)
    ref_taps, or_taps = {}, {}
    handles = ref_harness.install_taps(model, lambda n, t: ref_taps.__setitem__(n, t.detach().clone()))
    with torch.inference_mode():
        with ref_harness.patched_randn(inp["noise"]):
            a_ref = model(**{k: (v.clone() if k == "pixel_values" else v) for k, v in synth.call_args(inp).items()})
        a_or = O.infer_action(sd_t, cfg, **synth.call_args(inp), noise=inp["noise"],
                              tap=lambda n, t: or_taps.__setitem__(n, t.detach().clone()))
    for h in handles:
        h.remove()
    assert torch.equal(a_ref, a_or)
    for name, t in ref_taps.items():
        assert torch.equal(t, or_taps[name]), name


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode,clip,cache_fp", [("int8", None, False), ("int8", 1.0, False), ("int8_cached", 0.75, True)])
def test_int8_fake_quant_mode_bit_identical(dtype, mode, clip, cache_fp):
    """`enable_action_quantization` (pizero.py:274-321, int8_linear.py) on the unmodified reference against the oracle's
    restatement (weights de-quantised up front, inputs of the swapped Linears clamped)."""
    cfg = shrink_config(bridge_config(2), 2, 2)
    cfg.action_quantization = dict(mode=mode, activation_clip=clip, cache_fp_weight=cache_fp, fp_dtype="bfloat16")
    sd = synth.synthetic_state_dict(cfg, 0, torch.float32)
    model = _ref_model(cfg, sd, dtype)
    sd_t = {k: v.clone() for k, v in model.state_dict().items()}
    model.enable_action_quantization()
    assert model._action_quant_enabled
    inp = synth.synthetic_inputs(cfg, 2, dtype=dtype, vary_text=True)
    with torch.inference_mode():
        with ref_harness.patched_randn(inp["noise"]):
            a_ref = model(**{k: (v.clone() if k == "pixel_values" else v) for k, v in synth.call_args(inp).items()})
        sd_q = O.quantize_state_dict_int8(sd_t, cache_fp_weight=cache_fp, fp_dtype=torch.bfloat16)
        with O.int8_fake_quant(clip):
            a_or = O.infer_action(sd_q, cfg, **synth.call_args(inp), noise=inp["noise"])
        a_plain = O.infer_action(sd_t, cfg, **synth.call_args(inp), noise=inp["noise"])
    assert torch.equal(a_ref, a_or)
    assert not torch.equal(a_or, a_plain)          # the mode really changes the arithmetic


def test_infer_action_naive_bit_identical_and_self_consistent():
    cfg = shrink_config(bridge_config(2), 2, 2)
    sd = synth.synthetic_state_dict(cfg, 0, torch.float32)
    model = _ref_model(cfg, sd, torch.float32)
    inp = synth.synthetic_inputs(cfg, 2, dtype=torch.float32, vary_text=True)
    with torch.inference_mode():
        with ref_harness.patched_randn(inp["noise"]):
            n_ref = model.infer_action_naive(inp["input_ids"], inp["pixel_values"], inp["causal_mask"],
                                             inp["vlm_position_ids"], inp["proprio_position_ids"],
                                             inp["action_position_ids"], inp["proprios"])
        n_or = O.infer_action_naive(model.state_dict(), cfg, inp["input_ids"], inp["pixel_values"],
                                    inp["causal_mask"], inp["vlm_position_ids"], inp["proprio_position_ids"],
                                    inp["action_position_ids"], inp["proprios"], noise=inp["noise"])
        c_or = O.infer_action(model.state_dict(), cfg, **synth.call_args(inp), noise=inp["noise"])
    assert torch.equal(n_ref, n_or)
    # the one relation the reference itself asserts (agent/eval.py:213-214): exact in fp32
    assert (n_or - c_or).abs().max().item() < 1e-5


def test_masks_and_positions_bit_identical():
    cfg = shrink_config(bridge_config(1), 1, 1)
    pz = ref_harness.import_reference()
    with torch.device("meta"):
        model = pz.PiZeroInference(cfg, use_ddp=False)
    inp = synth.synthetic_inputs(cfg, 4, vary_text=True)
    for dtype in (torch.float32, torch.bfloat16):
        ref = model.build_causal_mask_and_position_ids(inp["attention_mask"], dtype)
        mine = O.build_causal_mask_and_position_ids(cfg, inp["attention_mask"], dtype)
        for a, b in zip(ref, mine):
            assert torch.equal(a, b)
        for a, b in zip(model.split_full_mask_into_submasks(ref[0]), O.split_full_mask_into_submasks(cfg, mine[0])):
            assert torch.equal(a, b)


def test_default_init_matches_reference_under_same_seed():
    """The host mirror draws the reference's default-init weights (same module order)."""
    from blurr_b200.pizero import PiZeroInference

    cfg = shrink_config(bridge_config(1), 1, 1)
    torch.manual_seed(0)
    mine = PiZeroInference(cfg)
    ref = ref_harness.build_reference_model(cfg, seed=0)
    sd_r, sd_m = ref.state_dict(), mine.state_dict()
    assert list(sd_r.keys()) == list(sd_m.keys())
    for k in sd_r:
        assert torch.equal(sd_r[k], sd_m[k]), k
