"""Action post-processing (SURVEY.md §8(f) row 4), CPU only: de-normalisers against the reference's own
BaseEnvAdapter (when the reference source is found, see oracle/ref_harness.py) and fixed numbers; euler -> axis-angle BIT-EXACT against the
reference's vendored transforms3d functions (src/utils/geometry.py:261-291) - directly when the reference is mounted,
and through tests/golden/postprocess_golden.json (generated from it by make_postprocess_golden.py) everywhere - plus
scipy's rotation vectors as an independent check; gripper logic against simpler.py:181-186,221-252."""

import os
import sys

import numpy as np
import pytest

from blurr_b200 import postprocess as PP
from oracle import ref_harness

REF = ref_harness.OPZ_ROOT
STATS = {"p01": [-0.03, -0.04, -0.03, -0.08, -0.09, -0.2, 0.0], "p99": [0.03, 0.04, 0.03, 0.08, 0.09, 0.2, 1.0],
         "mean": [0.0, 0.001, -0.002, 0.0, 0.01, 0.0, 0.6], "std": [0.01, 0.013, 0.012, 0.03, 0.03, 0.08, 0.5]}


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference not mounted")
def test_denormalisers_match_reference_adapter():
    sys.path.insert(0, REF)
    from src.agent.env_adapter.base import BaseEnvAdapter
    ad = BaseEnvAdapter()
    x = np.random.default_rng(0).uniform(-1.2, 1.2, (4, 6)).astype(np.float32)
    lo, hi = np.array(STATS["p01"])[:-1], np.array(STATS["p99"])[:-1]
    assert np.array_equal(PP.denormalize_bound(x, lo, hi, clip_min=-1, clip_max=1), ad.denormalize_bound(x, lo, hi, clip_min=-1, clip_max=1))
    m, s = np.array(STATS["mean"])[:-1], np.array(STATS["std"])[:-1]
    assert np.array_equal(PP.denormalize_gaussian(x, m, s), ad.denormalize_gaussian(x, m, s))


def test_denormalize_bound_fixed_numbers():
    lo, hi = np.array([0.0, -2.0]), np.array([1.0, 2.0])
    out = PP.denormalize_bound(np.array([[-1.0, -1.0], [0.0, 0.0], [1.0, 1.0], [0.5, -0.5]]), lo, hi)
    assert np.allclose(out, [[0.0, -2.0], [0.5, 0.0], [1.0, 2.0], [0.75, -1.0]], atol=0)


def test_euler_to_axis_angle_matches_scipy_rotation_vectors():
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(1)
    for rpy in np.concatenate([rng.uniform(-3.0, 3.0, (200, 3)), np.zeros((1, 3)), [[1e-9, 0, 0], [0, np.pi / 2, 0]]]):
        ax, ang = PP.euler2axangle(*rpy)
        ref = Rotation.from_euler("xyz", rpy).as_rotvec()          # extrinsic xyz == static 'sxyz'
        got = ax * ang
        # same rotation; transforms3d keeps the angle in [0, 2*pi), scipy in [0, pi]; 2*acos(w) loses angles
        # below ~1e-8 (w rounds to 1), which is the package's behaviour, hence the tolerance
        assert np.allclose(Rotation.from_rotvec(got).as_matrix(), Rotation.from_rotvec(ref).as_matrix(), atol=2e-8)
        assert abs(np.linalg.norm(ax) - 1.0) < 1e-12 and 0.0 <= ang <= 2 * np.pi
    assert PP.euler2axangle(0.0, 0.0, 0.0)[1] == 0.0


def test_euler_to_axis_angle_bit_exact_with_reference_golden():
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "postprocess_golden.json")) as f:
        cases = json.load(f)["cases"]
    assert len(cases) >= 100
    for c in cases:
        rpy = [float.fromhex(v) for v in c["rpy"]]
        ax, ang = PP.euler2axangle(*rpy)
        want_ang = float.fromhex(c["angle"])
        assert [float(v) for v in ax] == [float.fromhex(v) for v in c["axis"]], (rpy, ax)
        assert ang == want_ang or (np.isnan(ang) and np.isnan(want_ang)), (rpy, ang)


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference not mounted")
def test_euler_to_axis_angle_bit_exact_with_reference_geometry():
    sys.path.insert(0, REF)
    from src.utils.geometry import euler2axangle as ref_euler2axangle
    rng = np.random.default_rng(7)
    for rpy in np.concatenate([rng.uniform(-3.2, 3.2, (500, 3)), rng.uniform(-0.1, 0.1, (200, 3)), np.zeros((1, 3))]):
        ax, ang = PP.euler2axangle(*rpy)
        rax, rang = ref_euler2axangle(*rpy)
        assert np.array_equal(ax, rax) and ang == rang, rpy


def _reference_adapters():
    """The reference's adapter classes, imported unmodified; `simpler_env` (absent here, only used by the
    observation side) is stubbed, and the constructors (tokenizer download) are bypassed."""
    import types
    sys.path.insert(0, REF)
    if "simpler_env" not in sys.modules:
        pkg = types.ModuleType("simpler_env")
        for name in ("simpler_env.utils", "simpler_env.utils.env", "simpler_env.utils.env.observation_utils"):
            sys.modules[name] = types.ModuleType(name)
        sys.modules["simpler_env"] = pkg
        sys.modules["simpler_env.utils.env.observation_utils"].get_image_from_maniskill2_obs_dict = lambda *a, **k: None
    from src.agent.env_adapter.simpler import BridgeSimplerAdapter, EDRSimplerAdapter
    return BridgeSimplerAdapter, EDRSimplerAdapter


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference not mounted")
@pytest.mark.parametrize("kind,norm", [("bridge", "bound"), ("fractal", "bound"), ("fractal", "gaussian")])
def test_postprocess_matches_reference_adapters(kind, norm):
    """Whole `postprocess` (simpler.py:100-141) incl. the sticky gripper state machine over 40 control steps of
    4-action chunks: bit-exact with the reference's adapter objects."""
    Bridge, EDR = _reference_adapters()
    cls = Bridge if kind == "bridge" else EDR
    ref = cls.__new__(cls)
    ref.action_normalization_type = norm
    ref.dataset_statistics = {"action": STATS}
    if kind == "fractal":
        ref.sticky_gripper_num_repeat = 15
        ref.reset()
    ours = PP.ActionPostprocessor(STATS, kind, action_normalization_type=norm)
    rng = np.random.default_rng(3)
    for step in range(40):
        chunk = rng.uniform(-1.0, 1.0, (4, 7)).astype(np.float32)
        chunk[:, -1] = rng.uniform(0.0, 1.0, 4) if step % 3 else rng.choice([0.0, 1.0], 4)
        a, b = ours.postprocess(chunk), ref.postprocess(chunk)
        assert a.dtype == b.dtype and np.array_equal(a, b), (kind, norm, step)


def test_bridge_and_fractal_gripper_rules():
    bridge = PP.ActionPostprocessor(STATS, "bridge")
    assert [bridge.postprocess_gripper(a) for a in (0.0, 0.5, 0.51, 1.0)] == [-1.0, -1.0, 1.0, 1.0]
    fr = PP.ActionPostprocessor(STATS, "fractal", sticky_gripper_num_repeat=3)
    # open command (1.0 -> relative -1) latches for 3 calls, then releases
    seq = [fr.postprocess_gripper(a) for a in (1.0, 0.5, 0.5, 0.5, 0.0)]
    assert seq == [-1.0, -1.0, -1.0, -0.0, 1.0]
    fr.reset()
    assert fr.sticky_action_is_on is False and fr.gripper_action_repeat == 0


def test_postprocess_chunk_layout():
    pp = PP.ActionPostprocessor(STATS, "bridge")
    actions = np.array([[0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.9], [1.0, -1.0, 0.5, 0.2, -0.3, 0.1, 0.1]], dtype=np.float32)
    out = pp.postprocess(actions)
    assert out.shape == (2, 7) and out.dtype == np.float64
    assert np.allclose(out[0], [0, 0, 0, 0, 0, 0, 1.0])            # mid-range -> zero motion, gripper open
    assert np.allclose(out[1, :3], [0.03, -0.04, 0.015]) and out[1, 6] == -1.0
    from scipy.spatial.transform import Rotation
    rpy = np.array([0.2 * 0.08, -0.3 * 0.09, 0.1 * 0.2])
    assert np.allclose(out[1, 3:6], Rotation.from_euler("xyz", rpy).as_rotvec(), atol=1e-9)
