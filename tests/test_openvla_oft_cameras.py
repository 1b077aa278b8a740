"""OpenVLA-OFT with a wrist camera and proprioception (the LIBERO checkpoints): `blurr_llm_forward_rows` past 384
positions (the streamed-K/V block attention, handles created with `long_forward`), `ProprioProjector`,
`normalize_proprio`, and `OftPolicy` with two cameras and the proprio row.  The specification is
oracle/openvla_oft_oracle.py and oracle/openvla_oft_cameras_oracle.py.

CPU (-m "not gpu"): the layout with 2 x 256 patches + 1 proprio row for every prompt form, `normalize_proprio` on hand
cases, the oracle projector against the same arithmetic in functional ops, the oracle's patch assembly order, and the
decoder config's ctypes field and ABI version.
GPU (-m gpu): forward_rows past 384 keys against transformers' `LlamaModel` (eager, the oracle's 4-D mask) run on each
sequence alone, with fp32 as the tie-breaker; the streamed kernel against the resident one (bitwise); pads, other
sequences and graph replays past 384 (bitwise); rejected calls; the proprio projector against the oracle module; the
two-camera policy on a shrunk stack."""

import copy
import os
import re

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla
from llama_helpers import Q01, Q99, hf_llama, instructions
from oracle import openvla_oft_cameras_oracle as OC
from oracle import openvla_oft_oracle as O

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_LIBERO = 2 * 256 + 1


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _padded(rows, left: bool, pad_id: int = 7):
    S = max(r.numel() for r in rows)
    ids = torch.full((len(rows), S), pad_id, dtype=torch.int64)
    mask = torch.zeros((len(rows), S), dtype=torch.int64)
    for b, r in enumerate(rows):
        sl = slice(S - r.numel(), S) if left else slice(0, r.numel())
        ids[b, sl] = r
        mask[b, sl] = 1
    return ids, mask


def _check_layout(lay, rows, P):
    for b, r in enumerate(rows):
        ids, a0, n, row0 = O.prompt_layout(r.tolist(), P, 8, 7)
        assert lay.text_lens[b] == len(ids) and lay.ids[b, :len(ids)].tolist() == ids
        assert (lay.block_starts[b], lay.seq_lens[b], lay.row_starts[b]) == (a0, n, row0)
    assert lay.max_len == int(lay.seq_lens.max()) and lay.n_rows == 56


def test_libero_layout_with_two_images_and_the_proprio_row():
    cfg = openvla.oft_libero_config()
    assert (cfg.num_images, cfg.use_proprio, cfg.proprio_dim, cfg.chunk, cfg.action_dim, cfg.max_positions) == (2, True, 8, 8, 7, 640)
    rows = instructions([34, 12, 40], 0)
    lay = openvla.oft_prompt_layout(rows, n_patches=P_LIBERO, cfg=cfg)
    assert lay.block_starts.tolist() == [513 + 35, 513 + 13, 513 + 41]
    assert lay.seq_lens.tolist() == [a + 57 for a in lay.block_starts.tolist()]
    assert lay.row_starts.tolist() == [a - 1 for a in lay.block_starts.tolist()] and lay.max_len == 611
    _check_layout(lay, rows, P_LIBERO)
    for left in (True, False):
        p, m = _padded(rows, left)
        lay2 = openvla.oft_prompt_layout(p, attention_mask=m, n_patches=P_LIBERO, cfg=cfg)
        assert torch.equal(lay2.ids, lay.ids) and np.array_equal(lay2.seq_lens, lay.seq_lens)
        assert np.array_equal(lay2.block_starts, lay.block_starts) and np.array_equal(lay2.row_starts, lay.row_starts)
    eq = torch.stack(instructions([30, 30], 1))
    lay3 = openvla.oft_prompt_layout(eq, n_patches=P_LIBERO, cfg=cfg)
    assert lay3.seq_lens.tolist() == [513 + 31 + 57] * 2
    _check_layout(lay3, list(eq), P_LIBERO)
    # 513 + 70 (69 tokens + 29871) + 56 + 1 = 640 fits; one more token does not
    assert openvla.oft_prompt_layout(instructions([69], 2), n_patches=P_LIBERO, cfg=cfg).max_len == 640
    with pytest.raises(ValueError, match="max_positions"):
        openvla.oft_prompt_layout(instructions([70], 2), n_patches=P_LIBERO, cfg=cfg)


def test_normalize_proprio_hand_cases():
    q01, q99 = np.array([-1.0, 0.0, 2.0, 5.0]), np.array([1.0, 4.0, 2.0, 7.0])
    x = np.array([[0.5, 1.0, 2.0, 9.0],
                  [-3.0, 4.0, 1.0, 6.0]])
    got = openvla.normalize_proprio(x, q01, q99)
    assert got.dtype == np.float64 and np.array_equal(got, OC.normalize_proprio(x, q01, q99))
    assert got[0, 0] == 2 * 1.5 / (2 + 1e-8) - 1                 # inside the range
    assert got[0, 1] == 2 * 1.0 / (4 + 1e-8) - 1
    assert got[0, 3] == 1.0 and got[1, 0] == -1.0               # beyond q99 / q01: clipped
    assert got[1, 1] == 2 * 4.0 / (4 + 1e-8) - 1                # exactly q99: just under 1
    assert got[0, 2] == -1.0 and got[1, 2] == -1.0               # q01 == q99: 2 * (x - q) / 1e-8 - 1, clipped
    mask = np.array([True, False, True, False])
    m = openvla.normalize_proprio(x, q01, q99, mask)
    assert np.array_equal(m, OC.normalize_proprio(x, q01, q99, mask))
    assert m[0, 1] == 1.0 and m[1, 1] == 1.0 and m[1, 3] == 1.0  # masked dims pass through, then the clip
    assert np.array_equal(openvla.normalize_proprio(np.array([0.25, 0.5, 2.0, 5.5]), q01, q99, mask)[[1, 3]], [0.5, 1.0])
    assert np.array_equal(openvla.normalize_proprio(torch.tensor(x), q01, q99), got)


def test_oracle_proprio_projector_is_the_functional_stack_and_has_oft_keys():
    torch.manual_seed(0)
    proj = OC.ProprioProjector(llm_dim=64, proprio_dim=8)
    sd = proj.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {"fc1.weight": (64, 8), "fc1.bias": (64,), "fc2.weight": (64, 64),
                                                           "fc2.bias": (64,)}
    x = torch.randn(5, 8)
    F = torch.nn.functional
    ref = F.linear(F.gelu(F.linear(x, sd["fc1.weight"], sd["fc1.bias"])), sd["fc2.weight"], sd["fc2.bias"])
    assert torch.equal(proj(x), ref)


def test_oracle_patch_assembly_order():
    B, H = 2, 4
    cams = [torch.full((B, 256, H), float(i + 1)) for i in range(2)]
    state = torch.full((B, H), 9.0)
    rows = OC.assemble_patches(cams, state)
    assert rows.shape == (B, 513, H)
    assert (rows[:, :256] == 1).all() and (rows[:, 256:512] == 2).all() and (rows[:, 512] == 9).all()
    assert torch.equal(OC.assemble_patches(cams), rows[:, :512])


def test_llm_config_has_long_forward_and_abi_version_3():
    assert [f[0] for f in capi.LlmConfigC._fields_][-1] == "long_forward"
    header = open(os.path.join(ROOT, "include", "blurr_llm.h")).read()
    assert re.search(r"#define BLURR_LLM_ABI_VERSION (\d+)", header).group(1) == str(capi.LLM_ABI_VERSION) == "3"
    assert openvla.openvla_oft_7b_config(openvla.oft_libero_config()).long_forward
    assert openvla.openvla_oft_7b_config(openvla.oft_libero_config()).max_positions == 640
    assert not openvla.openvla_oft_7b_config().long_forward and not openvla.LlamaShapedConfig().long_forward


# ---------------------------------------------------------------------------------------------------------------------
# GPU: forward_rows past 384 keys against transformers
# ---------------------------------------------------------------------------------------------------------------------
def _check_against_fp32(name, got, ref16, ref32):
    e_ours = (got.float() - ref32).abs()
    e_ref = (ref16.float() - ref32).abs()
    rms = ref32.pow(2).mean().sqrt().item()
    print(f"{name}: vs fp32 ours max {e_ours.max().item():.3e} mean {e_ours.mean().item():.3e} | transformers bf16 max "
          f"{e_ref.max().item():.3e} mean {e_ref.mean().item():.3e} (ref rms {rms:.3f})")
    assert e_ours.mean().item() <= 1.5 * e_ref.mean().item() + 1e-4 * rms
    assert e_ours.max().item() <= 2.5 * e_ref.max().item() + 1e-2 * rms


def _long_cfg(hidden, heads, hd, inter, layers, T, vocab=320):
    return openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                     intermediate=inter, vocab=vocab, max_positions=T, rms_eps=1e-6, long_forward=T > 384)


LONG_CASES = [
    # hidden, heads, head_dim, inter, layers, lens, block sizes (len - a0; 0: a0 = len), stress
    pytest.param(256, 2, 128, 512, 2, [610], [57], True, id="b1-610"),
    pytest.param(256, 2, 128, 512, 2, [300, 500, 637], [57, 57, 57], True, id="ragged-straddling-384"),
    pytest.param(256, 2, 128, 512, 1, [1024, 700], [57, 200], True, id="cap-1024"),
    pytest.param(512, 8, 64, 1024, 2, [700, 450, 390], [57, 30, 12], True, id="hd64"),
    pytest.param(512, 4, 128, 1408, 2, [520, 450], [0, 0], False, id="causal-block-at-len"),
    pytest.param(512, 4, 128, 1408, 2, [600, 480], [520, 300], True, id="wide-bidirectional-block"),
    pytest.param(4096, 32, 128, 11008, 2, list(np.random.default_rng(4).integers(590, 641, size=32)), [57] * 32, False,
                 id="llama2-7b-widths-b32-libero-lengths"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,heads,hd,inter,layers,lens,blocks,stress", LONG_CASES)
def test_forward_rows_past_384_matches_transformers_per_sequence(hidden, heads, hd, inter, layers, lens, blocks, stress):
    lens = np.asarray(lens, dtype=np.int32)
    blk = (lens - np.asarray(blocks, dtype=np.int32)).astype(np.int32)
    B, T = len(lens), int(lens.max())
    n_rows = int(min(blocks)) if min(blocks) > 0 else 6
    row0 = (blk - 1 if min(blocks) > 0 else lens - n_rows).astype(np.int32)
    cfg = _long_cfg(hidden, heads, hd, inter, layers, T)
    model = hf_llama(cfg, 0, qk_scale=6.0 if stress else 1.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, model.state_dict(), DEV, max_batch=B,
                                               inv_freq=model.model.rotary_emb.inv_freq.detach().float())
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn((B, T, hidden), device=DEV, generator=g) * (1.0 if stress else 0.3)).to(torch.bfloat16)
    got = dec.forward_rows(x, lens, blk, row0, n_rows)
    dec.check()
    assert got.shape == (B, n_rows, hidden)
    m16 = model.model
    m32 = copy.deepcopy(m16).float()
    ours, r16, r32 = [], [], []
    for b in range(B):
        L = int(lens[b])
        with torch.inference_mode():
            h16 = m16(inputs_embeds=x[b:b + 1, :L], attention_mask=O.additive_mask(L, int(blk[b]), L, torch.bfloat16).to(DEV)).last_hidden_state
            h32 = m32(inputs_embeds=x[b:b + 1, :L].float(),
                      attention_mask=O.additive_mask(L, int(blk[b]), L, torch.float32).to(DEV)).last_hidden_state
        sl = slice(int(row0[b]), int(row0[b]) + n_rows)
        ours.append(got[b]); r16.append(h16[0, sl]); r32.append(h32[0, sl])
    _check_against_fp32(f"forward_rows B={B} lens {lens.min()}..{lens.max()}", torch.stack(ours), torch.stack(r16), torch.stack(r32))
    dec.close()


def _synthetic(B, T, hidden=256, heads=2, hd=128):
    cfg = _long_cfg(hidden, heads, hd, 2 * hidden, 2, T, vocab=300)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    with torch.no_grad():
        for k, v in sd.items():
            if "q_proj" in k or "k_proj" in k:
                v.mul_(8.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV, max_batch=B)
    g = torch.Generator(device=DEV).manual_seed(7)
    return dec, (torch.randn((B, T, hidden), device=DEV, generator=g) * 0.5).to(torch.bfloat16)


@pytest.mark.gpu
@pytest.mark.parametrize("hd", [128, 64])
@pytest.mark.parametrize("L,block", [(384, 57), (350, 57), (301, 301), (200, 150)])
def test_streamed_attention_equals_resident_attention(L, block, hd):
    # one sequence of <= 384 positions: max_len 384 takes attn_block_kernel, max_len 448 attn_block_stream_kernel (pad
    # rows behind the sequence); both row counts take the GEMMs' store epilogue, whose per-row result does not depend on M
    dec, x = _synthetic(1, 448, hidden=512 if hd == 64 else 256, heads=8 if hd == 64 else 2, hd=hd)
    lens, blk, row0 = np.array([L], np.int32), np.array([L - block if block < L else L], np.int32), np.array([0], np.int32)
    resident = dec.forward_rows(x[:, :384], lens, blk, row0, L)
    streamed = dec.forward_rows(x, lens, blk, row0, L)
    dec.check()
    assert torch.equal(streamed, resident)
    dec.close()


def _vectors(B, T, n_rows, seed):
    r = np.random.default_rng(seed)
    lens = r.integers(n_rows + 2, T + 1, size=B).astype(np.int32)
    lens[0] = T
    blk = np.array([r.integers(n_rows + 1, L + 1) for L in lens], dtype=np.int32)
    row0 = np.array([r.integers(0, L - n_rows + 1) for L in lens], dtype=np.int32)
    return lens, blk, row0


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,hd", [(3, 600, 128), (4, 1024, 64), (2, 449, 128)])
def test_forward_rows_past_384_pads_other_sequences_and_graph_replay(B, T, hd):
    dec, x = _synthetic(B, T, hidden=512 if hd == 64 else 256, heads=8 if hd == 64 else 2, hd=hd)
    n_rows = 3
    lens, blk, row0 = _vectors(B, T, n_rows, 11)
    pad = torch.arange(T, device=DEV)[None, :, None] >= torch.as_tensor(lens, device=DEV)[:, None, None]
    zero = x.masked_fill(pad, 0.0)
    ref = dec.forward_rows(zero, lens, blk, row0, n_rows)
    launches = dec.last_launch_count
    for fill in (float("nan"), 1e30, -1e30):
        assert torch.equal(dec.forward_rows(x.masked_fill(pad, fill), lens, blk, row0, n_rows), ref), fill
    g = torch.Generator(device=DEV).manual_seed(99)
    other = (torch.randn(x.shape, device=DEV, generator=g) * 0.5).to(torch.bfloat16)
    for b in (0, B - 1):
        y = other.clone()
        y[b] = zero[b]
        assert torch.equal(dec.forward_rows(y, lens, blk, row0, n_rows)[b], ref[b]), b
    lens2, blk2, row2 = _vectors(B, T, 2, 12)
    got = dec.forward_rows(x, lens2, blk2, row2, 2)
    assert dec.last_launch_count == launches
    dec.set_option("use_cuda_graph", 0)
    eager = dec.forward_rows(x, lens2, blk2, row2, 2)
    assert dec.last_launch_count == launches
    dec.check()
    assert torch.equal(got, eager)
    dec.close()


@pytest.mark.gpu
def test_rejected_long_calls_leave_the_handle_working():
    import ctypes as C
    dec, x = _synthetic(2, 1024)
    lens, blk, row0 = np.array([1024, 700], np.int32), np.array([968, 650], np.int32), np.array([967, 0], np.int32)
    ok = dec.forward_rows(x, lens, blk, row0, 56)
    small = dict(num_layers=1, hidden=256, num_heads=2, num_kv_heads=2, head_dim=128, intermediate=512, vocab=300)
    for bad in (dict(max_positions=1025, long_forward=True), dict(max_positions=640, long_forward=2),
                dict(max_positions=385, long_forward=False)):
        with pytest.raises(capi.BlurrError):
            openvla.LlamaDecoder(openvla.LlamaShapedConfig(**small, **bad), DEV)
    # max_len past max_positions on a long handle
    d640 = openvla.LlamaDecoder(openvla.LlamaShapedConfig(**small, max_positions=640, long_forward=True), DEV)
    d640.close()
    lib, stream = dec.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    arr = [(C.c_int32 * 2)(*([20] * 2)) for _ in range(3)]
    out = torch.empty((2, 5, 256), device=DEV, dtype=torch.bfloat16)
    big = torch.zeros((2, 1025, 256), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(capi.BlurrError):
        capi.check(lib.blurr_llm_forward_rows(dec.handle, stream, 2, 1025, C.c_void_p(big.data_ptr()), *arr, 5, C.c_void_p(out.data_ptr())))
    with pytest.raises(capi.BlurrError):
        dec.forward_rows(x, np.array([1024, 1025], np.int32), blk, row0, 56)
    # generate on a 1024-position handle still stops at 320
    y = torch.zeros((1, 300, 256), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(capi.BlurrError, match="320"):
        dec.generate(y, 21)
    assert dec.generate(y, 20).shape == (1, 20)
    assert torch.equal(dec.forward_rows(x, lens, blk, row0, 56), ok)
    dec.check()
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the proprio projector against the oracle module
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 32])
def test_proprio_projector_matches_the_oracle_module(rows):
    torch.manual_seed(0)
    ref16 = OC.ProprioProjector(4096, 8).to(DEV, torch.bfloat16).eval()
    proj = openvla.ProprioProjector.from_state_dict({"proprio_projector." + k: v for k, v in ref16.state_dict().items()}, DEV,
                                                    max_rows=32, prefix="proprio_projector.")
    g = np.random.default_rng(rows)
    raw = g.uniform(-2, 2, size=(rows, 8))
    state = torch.from_numpy(OC.normalize_proprio(raw, -np.ones(8), np.ones(8)).astype(np.float32)).to(DEV, torch.bfloat16)
    got = proj.forward(state)
    assert got.shape == (rows, 4096) and got.dtype == torch.bfloat16
    with torch.inference_mode():
        r16 = ref16(state)
        r32 = copy.deepcopy(ref16).float()(state.float())
    _check_against_fp32(f"proprio projector rows {rows}", got, r16, r32)
    with pytest.raises(ValueError):
        proj.forward(state[:, :7])
    proj.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the two-camera, proprio policy on a shrunk stack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def libero_policy():
    B = 4
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(depth=3), DEV, max_batch=2 * B, seed=3)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(depth=3), DEV, max_batch=2 * B, seed=4)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=2 * B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    backbone = openvla.FusedVisionBackbone(dino, sig, proj)
    oft = openvla.oft_libero_config()
    cfg = openvla.openvla_oft_7b_config(oft)
    cfg.num_layers = 2
    dec = openvla.LlamaDecoder.from_state_dict(cfg, openvla.synthetic_llama_state_dict(cfg, DEV, 0), DEV, max_batch=B)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, DEV, max_batch=B, seed=6)
    pp = openvla.ProprioProjector.synthetic(8, 4096, DEV, max_rows=B, seed=8)
    cam = torch.device("cuda", torch.cuda.current_device())        # the frames' device, index included
    pres = [openvla.ImagePreprocessor(480, 640, device=cam), openvla.ImagePreprocessor(256, 256, device=cam)]
    pol = openvla.OftPolicy(pres, backbone, dec, head, oft, proprio_projector=pp)
    frames = [torch.randint(0, 256, (B, 480, 640, 3), device=DEV, dtype=torch.uint8, generator=g),
              torch.randint(0, 256, (B, 256, 256, 3), device=DEV, dtype=torch.uint8, generator=g)]
    yield pol, frames
    torch.cuda.synchronize()
    dec.check()
    head.check()
    for m in (*pres, dino, sig, proj, dec, head, pp):
        m.close()


MASK = np.array([True] * 6 + [False])
PQ01, PQ99 = np.linspace(-1.0, 0.0, 8), np.linspace(0.5, 2.0, 8)


def _raw_state(B, seed):
    return np.random.default_rng(seed).uniform(-1.5, 2.5, size=(B, 8))


@pytest.mark.gpu
def test_libero_policy_pixels_camera_order_and_proprio_row(libero_policy):
    pol, frames = libero_policy
    px = pol.pixel_values(frames)
    assert px.shape == (4, 12, 224, 224)
    assert torch.equal(px[:, :6], pol.preprocessors[0](frames[0])) and torch.equal(px[:, 6:], pol.preprocessors[1](frames[1]))
    state = pol.proprio_state(_raw_state(4, 0), PQ01, PQ99)
    assert torch.equal(state, torch.from_numpy(OC.normalize_proprio(_raw_state(4, 0), PQ01, PQ99).astype(np.float32))
                       .to(DEV, torch.bfloat16))
    rows = pol.patch_embeds(px, state)
    assert rows.shape == (4, 513, 4096)
    swapped = pol.patch_embeds(torch.cat([px[:, 6:], px[:, :6]], dim=1), state)
    assert torch.equal(swapped[:, :256], rows[:, 256:512]) and torch.equal(swapped[:, 256:512], rows[:, :256])
    assert torch.equal(rows[:, 512], pol.proprio_projector.forward(state))


@pytest.mark.gpu
def test_libero_policy_chunk_is_the_hand_composition_and_rows_match_batch_one(libero_policy):
    pol, frames = libero_policy
    rows = instructions([34, 12, 40, 25], 0)
    raw = _raw_state(4, 1)
    act, norm = pol.predict_action_chunk(frames, rows, Q01, Q99, MASK, return_normalized=True, proprio=raw, proprio_q01=PQ01,
                                         proprio_q99=PQ99)
    assert act.shape == (4, 8, 7) and act.dtype == torch.float64
    # backbone -> projector -> build_oft_embeds -> forward_rows -> head -> denormalize_chunk
    px = pol.pixel_values(frames)
    patches = pol.backbone.forward(px.reshape(8, 6, 224, 224)[:, :3], px.reshape(8, 6, 224, 224)[:, 3:]).reshape(4, 512, 4096)
    state = torch.from_numpy(openvla.normalize_proprio(raw, PQ01, PQ99).astype(np.float32)).to(DEV, torch.bfloat16)
    p = OC.assemble_patches([patches[:, :256], patches[:, 256:]], pol.proprio_projector.forward(state))
    lay = openvla.oft_prompt_layout(rows, n_patches=513, cfg=pol.cfg)
    x = openvla.build_oft_embeds(pol.decoder, lay, p)
    h = pol.decoder.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
    n2 = pol.head.forward(h)
    assert torch.equal(norm, n2)
    assert np.array_equal(act.numpy(), openvla.denormalize_chunk(n2.cpu().numpy(), Q01, Q99, MASK))
    for left in (True, False):
        ids, m = _padded(rows, left)
        assert torch.equal(pol.predict_action_chunk(frames, ids.to(DEV), Q01, Q99, MASK, attention_mask=m, proprio=raw,
                                                    proprio_q01=PQ01, proprio_q99=PQ99), act)
    scale = norm.abs().max().item()
    for b, r in enumerate(rows):
        _, n1 = pol.predict_action_chunk([f[b] for f in frames], r[None].to(DEV), Q01, Q99, MASK, return_normalized=True,
                                         proprio=raw[b], proprio_q01=PQ01, proprio_q99=PQ99)
        d = (n1[0] - norm[b]).abs().max().item()
        print(f"row {b}: batch-1 vs batch-4 max_abs {d:.3e} (scale {scale:.3e})")
        assert d <= 0.05 * scale + 1e-2, (b, d, scale)


@pytest.mark.gpu
def test_libero_policy_rejects_bad_inputs(libero_policy):
    pol, frames = libero_policy
    rows = instructions([10, 10, 10, 10], 2)
    raw = _raw_state(4, 2)
    kw = dict(proprio=raw, proprio_q01=PQ01, proprio_q99=PQ99)
    with pytest.raises(ValueError, match="camera"):
        pol.predict_action_chunk(frames[:1], rows, Q01, Q99, **kw)
    with pytest.raises(ValueError, match="camera"):
        pol.predict_action_chunk(frames[0], rows, Q01, Q99, **kw)
    with pytest.raises(ValueError, match="proprio"):
        pol.predict_action_chunk(frames, rows, Q01, Q99)
    with pytest.raises(ValueError, match="proprio"):
        pol.predict_action_chunk(frames, rows, Q01, Q99, proprio=raw[:, :7], proprio_q01=PQ01[:7], proprio_q99=PQ99[:7])
    with pytest.raises(ValueError, match="positions"):
        pol.predict_action_chunk(frames, instructions([80] * 4, 3), Q01, Q99, **kw)
    with pytest.raises(ValueError):
        openvla.OftPolicy(pol.preprocessors[:1], pol.backbone, pol.decoder, pol.head, pol.cfg, pol.proprio_projector)
    with pytest.raises(ValueError):
        openvla.OftPolicy(pol.preprocessors, pol.backbone, pol.decoder, pol.head, pol.cfg)


@pytest.mark.gpu
def test_one_camera_config_keeps_its_actions(libero_policy):
    pol, frames = libero_policy
    oft1 = openvla.OftConfig()
    one = openvla.OftPolicy(pol.preprocessors[0], pol.backbone, pol.decoder, pol.head, oft1)
    rows = instructions([14, 3, 25, 9], 4)
    got = one.predict_action_chunk(frames[0], rows, Q01, Q99, MASK)
    # the one-camera composition as it stood before cameras and proprio existed
    px = pol.preprocessors[0](frames[0])
    patch = pol.backbone.forward(px[:, :3], px[:, 3:])
    lay = openvla.oft_prompt_layout(rows, None, patch.shape[1], oft1)
    x = openvla.build_oft_embeds(pol.decoder, lay, patch, oft1.stop_token)
    h = pol.decoder.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)
    assert np.array_equal(got.numpy(), openvla.denormalize_chunk(pol.head.forward(h).cpu().numpy(), Q01, Q99, MASK))
    with pytest.raises(ValueError, match="use_proprio"):
        one.predict_action_chunk(frames[0], rows, Q01, Q99, proprio=_raw_state(4, 0), proprio_q01=PQ01, proprio_q99=PQ99)
