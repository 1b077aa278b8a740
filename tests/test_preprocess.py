"""Observation preprocessing (SURVEY.md §8(f) row 1).

CPU (-m "not gpu"): the oracle against cv2 itself where cv2 imports, against the committed golden
digests (cv2 + the reference's process_images), against the reference module when the reference source is found
(oracle/ref_harness.py); the C library's OpenCV tables against the oracle's.
GPU (-m gpu): the CUDA kernels through the C ABI against the oracle (bit-exact: integer resize, fp32
normalise, bf16 cast, float64 proprio), and `Episode.step` against the manual eval.py sequence."""

import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from blurr_b200 import capi
from oracle import preprocess_oracle as P
from oracle import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "preprocess_golden.json")))["cases"]
REF = ref_harness.OPZ_ROOT
BRIDGE_STATS = {"p01": [0.17, -0.21, -0.04, -3.1, -0.5, -1.2, 0.0], "p99": [0.45, 0.24, 0.28, 3.1, 0.6, 1.3, 1.0],
                "mean": [0.3, 0.0, 0.1, 0.0, 0.0, 0.1, 0.6], "std": [0.06, 0.09, 0.07, 1.9, 0.2, 0.5, 0.4]}


def _frame(seed, h, w, kind):
    from make_preprocess_golden_frames import frame
    return frame(seed, h, w, kind)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("case", GOLD, ids=lambda c: f"{c['h']}x{c['w']}-{c['kind']}")
def test_oracle_reproduces_golden_digests(case):
    img = _frame(case["seed"], case["h"], case["w"], case["kind"])
    small = P.resize_lanczos4_u8(img, 224, 224)
    assert small[::37, ::41].reshape(-1).tolist() == case["resized_samples"]
    assert hashlib.sha256(small.tobytes()).hexdigest() == case["resized_sha256"]
    if "pixel_values_bf16_sha256" in case:
        px = P.preprocess_frame(img)
        assert hashlib.sha256(px.view(torch.int16).numpy().tobytes()).hexdigest() == case["pixel_values_bf16_sha256"]


def test_oracle_matches_cv2_bit_for_bit():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    for (h, w, dh, dw) in [(480, 640, 224, 224), (225, 223, 224, 224), (96, 96, 224, 224), (37, 53, 16, 24),
                           (300, 200, 112, 150), (1080, 1920, 224, 224)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        ref = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LANCZOS4)
        assert np.array_equal(P.resize_lanczos4_u8(img, dh, dw), ref), (h, w, dh, dw)


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference not mounted")
def test_oracle_matches_reference_processor_and_normalisers():
    sys.path.insert(0, REF)
    from src.agent.env_adapter.base import BaseEnvAdapter
    from src.model.vla.processing import IMAGENET_STANDARD_MEAN, IMAGENET_STANDARD_STD, process_images
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (2, 3, 224, 224), dtype=torch.uint8, generator=g)
    ref = process_images(img, rescale_factor=1 / 255.0, image_mean=IMAGENET_STANDARD_MEAN, image_std=IMAGENET_STANDARD_STD)
    assert torch.equal(P.process_images(img), ref)
    adapter = BaseEnvAdapter()
    raw = np.random.default_rng(0).normal(0.2, 0.4, (5, 7))
    lo, hi = np.array(BRIDGE_STATS["p01"]), np.array(BRIDGE_STATS["p99"])
    assert np.array_equal(P.normalize_bound(raw, lo, hi), adapter.normalize_bound(raw, lo, hi, clip_min=-1, clip_max=1))
    m, s = np.array(BRIDGE_STATS["mean"]), np.array(BRIDGE_STATS["std"])
    assert np.array_equal(P.normalize_gaussian(raw, m, s), adapter.normalize_gaussian(raw, m, s))


@pytest.mark.parametrize("src,dst", [(640, 224), (480, 224), (224, 224), (1280, 224), (517, 224), (53, 24), (100, 300),
                                     (1920, 224), (225, 224)])
def test_library_tables_equal_opencv_tables(src, dst):
    """The C++ table builder (host code of the library, no GPU needed) against the oracle's tables."""
    import ctypes as C
    lib = capi.load_library()
    ofs = np.zeros(dst, np.int32)
    alpha = np.zeros((dst, 8), np.int16)
    capi.check(lib.blurr_preproc_build_tables(src, dst, ofs.ctypes.data_as(C.POINTER(C.c_int32)),
                                              alpha.ctypes.data_as(C.POINTER(C.c_int16))))
    o_ofs, o_alpha = P.lanczos4_tables(src, dst)
    assert np.array_equal(ofs, o_ofs) and np.array_equal(alpha, o_alpha)
    assert (alpha.astype(np.int64).sum(1) - 2048).__abs__().max() <= 4        # weights sum to ~1.0 in Q11


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(480, 640), (512, 640), (224, 224), (333, 517), (96, 96), (720, 1280)])
def test_gpu_frame_preprocessing_bit_exact(h, w):
    from blurr_b200.episode import FramePreprocessor
    pre = FramePreprocessor(h, w, (224, 224), "cuda:0")
    xo, xa, yo, ya = pre.tables()
    oxo, oxa = P.lanczos4_tables(w, 224)
    oyo, oya = P.lanczos4_tables(h, 224)
    assert np.array_equal(xo, oxo) and np.array_equal(xa, oxa) and np.array_equal(yo, oyo) and np.array_equal(ya, oya)
    rng = np.random.default_rng(h * 7 + w)
    frames = np.stack([rng.integers(0, 256, (h, w, 3), dtype=np.uint8), _frame(3, h, w, "smooth")])
    px, small = pre(torch.as_tensor(frames).cuda(), return_resized=True)
    torch.cuda.synchronize()
    for b in range(2):
        ref_small = P.resize_lanczos4_u8(frames[b], 224, 224)
        assert np.array_equal(small[b].cpu().numpy(), ref_small)
        ref_px = P.preprocess_frame(frames[b])
        assert torch.equal(px[b:b + 1].cpu().view(torch.int16), ref_px.view(torch.int16))
    pre.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bound", "gaussian"])
def test_gpu_proprio_normalisation_bit_exact(kind):
    from blurr_b200.episode import normalize_proprio
    rng = np.random.default_rng(3)
    raw = rng.normal(0.2, 0.6, (9, 7))
    raw[0, 0] = 10.0; raw[1, 1] = -10.0          # clipped by "bound"
    keys = ("p01", "p99") if kind == "bound" else ("mean", "std")
    lo = torch.as_tensor(np.array(BRIDGE_STATS[keys[0]])).cuda()
    hi = torch.as_tensor(np.array(BRIDGE_STATS[keys[1]])).cuda()
    got = normalize_proprio(torch.as_tensor(raw).cuda(), lo, hi, kind)
    torch.cuda.synchronize()
    ref = torch.cat([P.preprocess_proprio(raw[i], BRIDGE_STATS, kind)[0] for i in range(raw.shape[0])])
    assert torch.equal(got.cpu().view(torch.int16), ref.view(torch.int16))


@pytest.mark.gpu
def test_episode_step_equals_manual_eval_sequence():
    """Episode.step (device preprocessing, cached masks) == the reference's per-step sequence done by hand
    with the oracle's preprocessing and the same model: bit-identical actions."""
    from blurr_b200 import synth
    from blurr_b200.config import bridge_config, shrink_config
    from blurr_b200.episode import Episode
    from blurr_b200.pizero import PiZeroInference
    cfg = shrink_config(bridge_config(1), 2, 3)
    sd = synth.synthetic_state_dict(cfg, 0, torch.bfloat16)
    model = PiZeroInference.from_state_dict(cfg, sd, device="cuda:0")
    inp = synth.synthetic_inputs(cfg, 1, dtype=torch.bfloat16)
    ep = Episode(model, inp["input_ids"], inp["attention_mask"], (480, 640), BRIDGE_STATS, "bound")
    rng = np.random.default_rng(11)
    for step in range(3):
        frame = _frame(20 + step, 480, 640, "smooth")
        raw = rng.normal(0.2, 0.3, 7)
        noise = inp["noise"].cuda()
        got = ep.step(frame, raw, noise=noise)
        px = P.preprocess_frame(frame).cuda()
        prop = P.preprocess_proprio(raw, BRIDGE_STATS, "bound").cuda()
        cm, vp, pp, ap = model.build_causal_mask_and_position_ids(inp["attention_mask"], dtype=torch.bfloat16)
        m1, m2 = model.split_full_mask_into_submasks(cm)
        with torch.inference_mode():
            ref = model(inp["input_ids"].cuda(), px, m1.cuda(), m2.cuda(), vp.cuda(), pp.cuda(), ap.cuda(), prop, noise=noise)
        assert torch.equal(got, ref), step
    ep.close()
    model.release_engine()
