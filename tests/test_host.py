"""Host-side logic on CPU: config handling, mask builders, state_dict contract, C-ABI library
loading and symbol table, loud failure without a GPU."""

import ctypes
import os
import re

import pytest
import torch

from blurr_b200 import capi, masks, synth
from blurr_b200.config import (AttrDict, bridge_config, fractal_config, load_yaml_config, merge,
                               shrink_config)
from blurr_b200.pizero import PiZeroInference, sinusoidal_time_table
from oracle import pi0_oracle as O
from oracle import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = capi.load_library()
    assert lib.blurr_abi_version() == capi.ABI_VERSION
    declared = set()
    for name in ("blurr_pi0.h", "blurr_llm.h", "blurr_vit.h"):
        header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", name)).read(), flags=re.S)
        declared |= set(re.findall(r"\b(blurr_[a-z0-9_]+)\s*\(", header))
    declared -= {"blurr_status", "blurr_dtype"}
    assert declared == set(capi.DECLARED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_config_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "blurr_pi0.h")).read()
    body = header[header.index("typedef struct blurr_pi0_config {"):header.index("} blurr_pi0_config;")]
    fields = re.findall(r"^\s+(?:int32_t|int64_t|float)\s+([a-z_0-9]+);", body, flags=re.M)
    assert fields == [f[0] for f in capi.Pi0ConfigC._fields_]
    body = header[header.index("typedef struct blurr_pi0_inputs {"):header.index("} blurr_pi0_inputs;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"([a-z_0-9]+)(?:\[4\])?\s*[;,]", body)
    assert [f[0] for f in capi.Pi0InputsC._fields_] == names


def test_llm_config_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "blurr_llm.h")).read()
    body = header[header.index("typedef struct blurr_llm_config {"):header.index("} blurr_llm_config;")]
    fields = re.findall(r"^\s+(?:int32_t|int64_t|float)\s+([a-z_0-9]+);", body, flags=re.M)
    assert fields == [f[0] for f in capi.LlmConfigC._fields_]


def test_vit_config_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "blurr_vit.h")).read()
    body = header[header.index("typedef struct blurr_vit_config {"):header.index("} blurr_vit_config;")]
    fields = re.findall(r"^\s+(?:int32_t|int64_t|float)\s+([a-z_0-9]+);", body, flags=re.M)
    assert fields == [f[0] for f in capi.VitConfigC._fields_]


def test_llm_create_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from blurr_b200 import openvla
    with pytest.raises(capi.BlurrError, match="no CUDA device"):
        openvla.LlamaDecoder(openvla.openvla_7b_config(), "cuda:0")


def test_openvla_action_detokenizer_and_rope_tables():
    """`predict_action`'s tail (bins on [-1, 1], q01/q99 de-normalisation) and the RoPE tables against transformers'
    LlamaRotaryEmbedding on CPU."""
    import numpy as np
    from blurr_b200 import openvla
    d = openvla.ActionDetokenizer(vocab_size=32000, n_bins=256)
    ids = np.array([31999, 31998, 31745, 31744, 31000, 5])
    centers = (np.linspace(-1, 1, 256)[:-1] + np.linspace(-1, 1, 256)[1:]) / 2
    assert np.array_equal(d.normalized(ids), centers[[0, 1, 254, 254, 254, 254]])
    q01, q99 = np.array([-0.5, 0.0]), np.array([0.5, 2.0])
    out = d.actions(np.array([31999, 31745]), q01, q99, mask=np.array([True, False]))
    assert np.allclose(out, [0.5 * (centers[0] + 1) * 1.0 - 0.5, centers[254]])
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding
    rot = LlamaRotaryEmbedding(LlamaConfig(hidden_size=256, num_attention_heads=2, head_dim=128, rope_theta=10000.0))
    assert torch.equal(rot.inv_freq, openvla.default_inv_freq(128, 10000.0, "cpu"))
    x = torch.zeros((1, 40, 256), dtype=torch.bfloat16)
    cos, sin = rot(x, torch.arange(40)[None, :])
    c2, s2 = openvla.rope_tables(rot.inv_freq, 40)
    assert torch.equal(cos[0, :, :64].float(), c2) and torch.equal(sin[0, :, :64].float(), s2)
    assert torch.equal(cos[0, :, 64:], cos[0, :, :64])


def test_openvla_shape_configs():
    """The OpenVLA-7B-shaped defaults: tower depths minus one (second-to-last block), concatenated width 2176, Llama-2-7B."""
    from blurr_b200 import openvla
    d, s_, l = openvla.dinov2_large_reg4_config(), openvla.siglip_so400m_config(), openvla.openvla_7b_config()
    assert (d.num_layers, d.hidden, d.num_heads, d.mlp_dim, d.num_prefix_tokens, d.use_layerscale, d.gelu_erf) == (23, 1024, 16, 4096, 5, True, True)
    assert (s_.num_layers, s_.hidden, s_.num_heads, s_.mlp_dim, s_.num_prefix_tokens, s_.use_layerscale, s_.gelu_erf) == (26, 1152, 16, 4304, 0, False, False)
    assert d.hidden + s_.hidden == 2176
    assert (l.num_layers, l.hidden, l.num_heads, l.head_dim, l.intermediate, l.vocab) == (32, 4096, 32, 128, 11008, 32064)
    assert 1 + 256 + 24 + 7 <= l.max_positions <= 320
    # weight bytes one decode step streams: 32 x (qkv + o + gate/up + down) + the padded lm_head
    per_layer = (3 * 4096 * 4096 + 4096 * 4096 + 2 * 11008 * 4096 + 4096 * 11008) * 2
    assert abs(32 * per_layer + 32128 * 4096 * 2 - 13215203328) == 0


def test_create_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = capi.load_library()
    cfg = shrink_config(bridge_config(1), 1, 1)
    model = PiZeroInference.from_state_dict(cfg, synth.synthetic_state_dict(cfg, 0, torch.bfloat16))
    h = ctypes.c_void_p()
    rc = lib.blurr_pi0_create(ctypes.byref(model._config_c()), 0, 1, ctypes.byref(h))
    assert rc < 0 and b"CUDA" in lib.blurr_last_error()
    inp = synth.synthetic_inputs(cfg, 1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        model(**synth.call_args(inp))


def test_invalid_config_rejected():
    lib = capi.load_library()
    cfg = shrink_config(bridge_config(1), 1, 1)
    model = PiZeroInference.from_state_dict(cfg, synth.synthetic_state_dict(cfg, 0, torch.bfloat16))
    c = model._config_c()
    c.head_dim = 128
    h = ctypes.c_void_p()
    assert lib.blurr_pi0_create(ctypes.byref(c), 0, 1, ctypes.byref(h)) == -1
    assert b"head_dim" in lib.blurr_last_error()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_mask_builder_matches_oracle(dtype):
    cfg = bridge_config(1)
    am = torch.zeros(5, 276, dtype=torch.long)
    for b, n in enumerate([276, 268, 257, 256, 1]):      # full, typical, BOS only, image only, degenerate
        am[b, :n] = 1
    got = masks.build_causal_mask_and_position_ids(am, dtype, 276, 1, 4)
    want = O.build_causal_mask_and_position_ids(cfg, am, dtype)
    for a, b in zip(got, want):
        assert a.dtype == b.dtype and torch.equal(a, b)
    assert int((got[0][1] == 0).sum()) == 268 * 268 + 5 * 268 + 1 + 4 * 5   # SURVEY.md appendix F
    g1, g2 = masks.split_full_mask_into_submasks(got[0], 276, 1, 4)
    w1, w2 = O.split_full_mask_into_submasks(cfg, want[0])
    assert g1.shape == (5, 1, 277, 277) and g2.shape == (5, 1, 4, 281)
    assert torch.equal(g1, w1) and torch.equal(g2, w2)
    assert g1.data_ptr() == got[0].data_ptr()            # views, like the reference


def test_state_dict_contract():
    cfg = bridge_config(1)
    spec = synth.state_dict_spec(cfg)
    assert len(spec) == 938                               # SURVEY.md appendix C
    total = sum(int(torch.Size(s).numel()) for _, s, _, _ in spec)
    assert total == 3_549_565_687
    with torch.device("meta"):
        model = PiZeroInference(cfg)
    sd = model.state_dict()
    assert set(sd.keys()) == {k for k, _, _, _ in spec}
    for k, shape, _, _ in spec:
        assert tuple(sd[k].shape) == tuple(shape), k
    f = synth.state_dict_spec(fractal_config(10))
    assert dict((k, s) for k, s, _, _ in f)["proprio_encoder.weight"] == (1024, 8)


def test_time_table_matches_oracle_and_bf16_accumulation():
    for steps in (1, 10):
        cfg = bridge_config(steps)
        for dtype in (torch.float32, torch.bfloat16):
            got = sinusoidal_time_table(steps, 1024, 10000.0, "cpu", dtype)
            want = O.time_cond_table(cfg, dtype)
            assert torch.equal(got, want)
    one = sinusoidal_time_table(1, 1024, 10000.0, "cpu", torch.bfloat16)
    assert torch.equal(one[0, :512], torch.zeros(512, dtype=torch.bfloat16))     # t = 0: [0.., 1..]
    assert torch.equal(one[0, 512:], torch.ones(512, dtype=torch.bfloat16))


def test_config_helpers(tmp_path):
    cfg = bridge_config(10)
    assert cfg.mixture.vlm.hidden_size == 2048 and cfg.get("missing", 3) == 3
    assert cfg.joint.config.mixture.action.cache is False
    m = merge(cfg.joint.config, cfg.joint.config.mixture.action)      # joint_model.py:328-330
    assert m.hidden_size == 1024 and m.num_hidden_layers == 18
    y = tmp_path / "c.yaml"
    y.write_text("a: 3\nb: ${a}\nmixture:\n  vlm:\n    h: ${b}\nname: x_${a}\nn: ${eval:'2 * 5'}\n")
    loaded = load_yaml_config(str(y))
    assert loaded.b == 3 and loaded.mixture.vlm.h == 3 and loaded.name == "x_3" and loaded.n == 10
    ref_yaml = os.path.join(ref_harness.OPZ_ROOT, "config", "eval", "bridge.yaml")
    if os.path.isfile(ref_yaml):
        ref_cfg = load_yaml_config(ref_yaml)
        for key in ("num_inference_steps", "final_action_clip_value", "cond_steps", "horizon_steps", "action_dim",
                    "proprio_dim", "max_image_text_tokens", "image_token_index", "vocab_size", "pad_token_id",
                    "time_max_period"):
            assert ref_cfg[key] == cfg[key], key
        assert ref_cfg.vision.config == cfg.vision.config
        assert ref_cfg.joint.config.mixture == cfg.joint.config.mixture
        for key in ("num_hidden_layers", "num_attention_heads", "num_key_value_heads", "head_dim", "rms_norm_eps"):
            assert ref_cfg.joint.config[key] == cfg.joint.config[key]
        step1 = load_yaml_config(ref_yaml.replace("bridge.yaml", "bridge_step1.yaml"))
        assert step1.num_inference_steps == 1
        fr = load_yaml_config(ref_yaml.replace("bridge.yaml", "fractal_coke.yaml"))
        assert fr.proprio_dim == fractal_config().proprio_dim and fr.act_steps == 2


def test_synthetic_inputs_layout():
    cfg = bridge_config(1)
    inp = synth.synthetic_inputs(cfg, 3, vary_text=True)
    ids = inp["input_ids"]
    assert ids.shape == (3, 276) and (ids[:, :256] == 257152).all() and (ids[:, 256] == 2).all()
    cnt = inp["attention_mask"].sum(1)
    for b in range(3):
        assert ids[b, cnt[b] - 1] == 108 and (ids[b, cnt[b]:] == 0).all()
    assert inp["pixel_values"].abs().max() <= 1.0
    base = synth.synthetic_inputs(cfg, 1)
    assert base["attention_mask"].sum().item() == 268
    assert base["input_ids"][0, 257:267].tolist() == [179378, 5125, 195997, 211369, 93264, 178254, 3810, 17301,
                                                      14683, 160681]   # SURVEY.md appendix F


@pytest.mark.parametrize("N,K,T,band", [(32768, 2048, 17664, 0), (32768, 2048, 4416, 0), (2048, 16384, 17664, 0),
                                        (3456, 1152, 16384, 0), (4352, 1152, 16384, 5), (4096, 1152, 2100, 3),
                                        (1152, 4352, 16384, 2), (40960, 128, 1500, 7), (256, 64, 1025, 1)])
def test_pair_raster_visits_every_tile_once_in_bands(N, K, T, band):
    """The raster order of the batched GEMM's persistent CTA pairs (csrc/gemm_body.cuh pair_tile_coords, the
    function the kernel runs, exposed host-side through blurr_op_pair_raster): every (weight tile pair, token
    tile) exactly once; a band's weight tile pairs sweep all token tiles before the next band starts; inside a
    band the weight index runs fastest.  Automatic banding only when one wave of pairs cannot hold every weight
    tile pair (gate/up: 128 pairs of tiles, 74 CTA pairs -> bands of 32 MB of weights)."""
    import ctypes as C
    import numpy as np
    lib = capi.load_library()
    gxp, gy = (N // 128 + 1) // 2, (T + 255) // 256
    order = np.full((gxp * gy, 2), -1, np.int32)
    b, p = C.c_int(), C.c_int()
    try:
        capi.check(lib.blurr_set_global_option(b"gemm_pair_band", band))
        tiles = lib.blurr_op_pair_raster(N, K, T, C.byref(b), C.byref(p), order.ctypes.data_as(C.POINTER(C.c_int32)), len(order))
    finally:
        capi.check(lib.blurr_set_global_option(b"gemm_pair_band", 0))
    assert tiles == gxp * gy and p.value == min(tiles, 74)
    if band:
        assert b.value == min(band, gxp)
    elif gxp <= p.value:
        assert b.value == gxp
    else:
        assert b.value == max(4, min(gxp, (32 << 20) // (2 * 128 * K * 2)))
    assert sorted(map(tuple, order.tolist())) == [(x, y) for x in range(gxp) for y in range(gy)]
    bands = order[:, 0] // b.value
    assert (np.diff(bands) >= 0).all()                                   # bands in order, never revisited
    for bi in np.unique(bands):
        sub = order[bands == bi]
        w = min(b.value, gxp - bi * b.value)
        assert len(sub) == w * gy
        assert (sub[:, 0] == bi * b.value + np.arange(len(sub)) % w).all()   # weight index fastest
        assert (sub[:, 1] == np.arange(len(sub)) // w).all()                 # token tiles ascending


def test_pair_raster_rejects_bad_shapes():
    lib = capi.load_library()
    assert lib.blurr_op_pair_raster(100, 64, 2048, None, None, None, 0) < 0
    assert lib.blurr_op_pair_raster(128, 64, 0, None, None, None, 0) < 0
