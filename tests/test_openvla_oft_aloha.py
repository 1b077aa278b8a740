"""OpenVLA-OFT, the ALOHA form (three FiLM cameras, 14-D proprioception, chunks of 25 x 14): `blurr_llm_forward_rows`
past 1024 positions (handles created with `long_forward = 2`, the streamed block attention up to 2048 keys with its tile
halved past 1152), the action head on rows of 14 x 4096 = 57 344 columns (the shared-memory LayerNorm), and `OftPolicy`
with `oft_aloha_config()`.  The specification is oracle/openvla_oft_oracle.py, oracle/openvla_oft_cameras_oracle.py and
oracle/openvla_oft_film_oracle.py.

CPU (-m "not gpu"): the layout with 3 x 256 patches + 1 proprio row and 350 slots for every prompt form and its
1280-position limit, FiLM's averaged rows on it, the preset and the decoder config it gives, the oracle head's keys and
shapes at 25 x 14, `normalize_proprio` with ALOHA's min / max statistics, and the head header's width limit.
GPU (-m gpu): forward_rows past 1024 keys against transformers' `LlamaModel` (eager, the oracle's 4-D mask) run on each
sequence alone, with fp32 as the tie-breaker; the tile fallback and the 1024 boundary bit for bit; pads, other sequences
and graph replays past 1024 (bitwise); rejected calls; the head at ALOHA's width against the oracle module; the ALOHA
policy on a shrunk stack."""

import copy
import os
import re

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla
from llama_helpers import hf_llama, instructions
from oracle import openvla_oft_cameras_oracle as OC
from oracle import openvla_oft_film_oracle as OF
from oracle import openvla_oft_oracle as O

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_ALOHA = 3 * 256 + 1


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


def _check_layout(lay, rows):
    for b, r in enumerate(rows):
        ids, a0, n, row0 = O.prompt_layout(r.tolist(), P_ALOHA, 25, 14)
        assert lay.text_lens[b] == len(ids) and lay.ids[b, :len(ids)].tolist() == ids
        assert (lay.block_starts[b], lay.seq_lens[b], lay.row_starts[b]) == (a0, n, row0)
    assert lay.max_len == int(lay.seq_lens.max()) and lay.n_rows == 350


def test_aloha_preset_and_layout_with_three_images_and_the_proprio_row():
    cfg = openvla.oft_aloha_config()
    assert (cfg.num_images, cfg.use_proprio, cfg.proprio_dim, cfg.chunk, cfg.action_dim, cfg.use_film, cfg.max_positions) == \
        (3, True, 14, 25, 14, True, 1280)
    rows = instructions([20, 12, 31], 0)
    lay = openvla.oft_prompt_layout(rows, n_patches=P_ALOHA, cfg=cfg)
    assert lay.block_starts.tolist() == [769 + 21, 769 + 13, 769 + 32]
    assert lay.seq_lens.tolist() == [a + 351 for a in lay.block_starts.tolist()]
    assert lay.row_starts.tolist() == [a - 1 for a in lay.block_starts.tolist()] and lay.max_len == 1152
    _check_layout(lay, rows)
    for left in (True, False):
        p, m = _padded(rows, left)
        lay2 = openvla.oft_prompt_layout(p, attention_mask=m, n_patches=P_ALOHA, cfg=cfg)
        assert torch.equal(lay2.ids, lay.ids) and np.array_equal(lay2.seq_lens, lay.seq_lens)
        assert np.array_equal(lay2.block_starts, lay.block_starts) and np.array_equal(lay2.row_starts, lay.row_starts)
    eq = torch.stack(instructions([25, 25], 1))
    lay3 = openvla.oft_prompt_layout(eq, n_patches=P_ALOHA, cfg=cfg)
    assert lay3.seq_lens.tolist() == [769 + 26 + 351] * 2
    _check_layout(lay3, list(eq))
    # 769 + 160 (159 tokens + 29871) + 350 + 1 = 1280 fits; one more token does not
    assert openvla.oft_prompt_layout(instructions([159], 2), n_patches=P_ALOHA, cfg=cfg).max_len == 1280
    with pytest.raises(ValueError, match="max_positions"):
        openvla.oft_prompt_layout(instructions([160], 2), n_patches=P_ALOHA, cfg=cfg)


def test_film_language_rows_on_the_aloha_layout():
    cfg = openvla.oft_aloha_config()
    rows = instructions([20, 12, 31], 3)
    for form in ("list", "left", "right"):
        if form == "list":
            lay = openvla.oft_prompt_layout(rows, n_patches=P_ALOHA, cfg=cfg)
        else:
            p, m = _padded(rows, form == "left")
            lay = openvla.oft_prompt_layout(p, attention_mask=m, n_patches=P_ALOHA, cfg=cfg)
        got = openvla.film_language_rows(lay)
        for b, r in enumerate(rows):
            prompt = O.prompt_layout(r.tolist(), P_ALOHA, 25, 14)[0]
            # BOS, the instruction, 29871 and the stop token: no slot placeholder and no pad
            assert got[b].tolist() == OF.language_rows(prompt, 350) == prompt + [2], (form, b)


def test_decoder_config_long_forward_by_position_count():
    aloha = openvla.openvla_oft_7b_config(openvla.oft_aloha_config())
    assert aloha.long_forward == 2 and aloha.max_positions == 1280
    assert openvla.openvla_oft_7b_config(openvla.oft_libero_config()).long_forward == 1
    assert openvla.openvla_oft_7b_config().long_forward == 0 and openvla.LlamaShapedConfig().long_forward == 0
    assert openvla.openvla_oft_7b_config(openvla.OftConfig(max_positions=1024)).long_forward == 1
    assert openvla.openvla_oft_7b_config(openvla.OftConfig(max_positions=1025)).long_forward == 2


def test_oracle_head_at_25_by_14_has_oft_keys_and_shapes():
    with torch.device("meta"):
        head = O.L1RegressionActionHead(input_dim=4096, hidden_dim=4096, action_dim=14, chunk=25)
    W, H = 14 * 4096, 4096
    expect = {"model.layer_norm1.weight": (W,), "model.layer_norm1.bias": (W,), "model.fc1.weight": (H, W),
              "model.fc1.bias": (H,), "model.layer_norm2.weight": (H,), "model.layer_norm2.bias": (H,),
              "model.fc2.weight": (14, H), "model.fc2.bias": (14,)}
    for i in range(2):
        p = f"model.mlp_resnet_blocks.{i}.ffn."
        expect.update({p + "0.weight": (H,), p + "0.bias": (H,), p + "1.weight": (H, H), p + "1.bias": (H,)})
    assert {k: tuple(v.shape) for k, v in head.state_dict().items()} == expect


def test_normalize_proprio_with_min_max_statistics():
    # ALOHA's BOUNDS rule is the BOUNDS_Q99 arithmetic with min / max in place of q01 / q99
    lo = np.array([-1.0, 0.0, 2.0, 5.0, -0.5, 0.0, 0.0] * 2)
    hi = np.array([1.0, 4.0, 2.0, 7.0, 0.5, 1.0, 0.1] * 2)
    x = np.array([[0.5, 1.0, 2.0, 9.0, -0.5, 1.0, 0.05] * 2,
                  [-3.0, 4.0, 1.0, 6.0, 0.0, 0.0, 0.2] * 2])
    got = openvla.normalize_proprio(x, lo, hi)
    assert got.shape == (2, 14) and got.dtype == np.float64 and np.array_equal(got, OC.normalize_proprio(x, lo, hi))
    for c in (0, 7):
        assert got[0, c] == 2 * 1.5 / (2 + 1e-8) - 1                  # inside the range
        assert got[0, c + 3] == 1.0 and got[1, c] == -1.0              # beyond max / min: clipped
        assert got[1, c + 1] == 2 * 4.0 / (4 + 1e-8) - 1               # exactly the max: just under 1
        assert got[0, c + 2] == -1.0                                   # min == max: clipped
        assert got[0, c + 4] == -1.0 and got[1, c + 4] == 2 * 0.5 / (1 + 1e-8) - 1
        assert got[0, c + 6] == 2 * 0.05 / (0.1 + 1e-8) - 1
    mask = np.array([True, False] * 7)
    assert np.array_equal(openvla.normalize_proprio(x, lo, hi, mask), OC.normalize_proprio(x, lo, hi, mask))


def test_head_header_states_the_65536_column_limit():
    header = open(os.path.join(ROOT, "include", "blurr_act_head.h")).read()
    assert re.search(r"D \* H is a multiple of 64 and at most 65536", header)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: forward_rows past 1024 keys against transformers
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
    lf = 0 if T <= 384 else 1 if T <= 1024 else 2
    return openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                     intermediate=inter, vocab=vocab, max_positions=T, rms_eps=1e-6, long_forward=lf)


LONGER_CASES = [
    # hidden, heads, head_dim, inter, layers, lens, block sizes (len - a0; 0: a0 = len), stress
    pytest.param(256, 2, 128, 512, 2, [1141], [351], True, id="b1-aloha-1141"),
    pytest.param(256, 2, 128, 512, 2, [900, 1150, 1153, 1300], [351, 351, 351, 351], True, id="ragged-straddling-1024-1152"),
    pytest.param(256, 2, 128, 512, 1, [2048, 1500], [351, 200], True, id="cap-2048"),
    pytest.param(512, 8, 64, 1024, 2, [1800, 1100, 1030], [351, 30, 12], True, id="hd64"),
    pytest.param(512, 4, 128, 1408, 2, [1200, 1090], [0, 0], False, id="causal-block-at-len"),
    pytest.param(512, 4, 128, 1408, 2, [1250, 1100], [1000, 700], True, id="wide-bidirectional-block"),
    pytest.param(4096, 32, 128, 11008, 2, list(np.random.default_rng(5).integers(1130, 1281, size=32)), [351] * 32, False,
                 id="llama2-7b-widths-b32-aloha-lengths"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,heads,hd,inter,layers,lens,blocks,stress", LONGER_CASES)
def test_forward_rows_past_1024_matches_transformers_per_sequence(hidden, heads, hd, inter, layers, lens, blocks, stress):
    lens = np.asarray(lens, dtype=np.int32)
    blk = (lens - np.asarray(blocks, dtype=np.int32)).astype(np.int32)
    B, T = len(lens), int(lens.max())
    n_rows = int(min(blocks)) if min(blocks) > 0 else 6
    row0 = (blk - 1 if min(blocks) > 0 else lens - n_rows).astype(np.int32)
    cfg = _long_cfg(hidden, heads, hd, inter, layers, T)
    assert cfg.long_forward == 2
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
def test_tile_fallback_and_the_1024_boundary_are_bitwise_invisible():
    # 5 sequences x 4 heads: at 1152 keys the streamed kernel runs 64-row tiles; at max_len 1216 they no longer fit the
    # shared-memory limit and the launcher halves them to 32.  Pad rows behind each sequence change nothing a real row sees.
    dec, x = _synthetic(5, 1216, hidden=512, heads=4)
    lens = np.array([1152, 1100, 1030, 1150, 1141], np.int32)
    blk = np.array([801, 749, 930, 1150, 790], np.int32)           # the fourth: a0 = len (causal)
    row0 = np.zeros(5, np.int32)
    bm64 = dec.forward_rows(x[:, :1152], lens, blk, row0, 1030)
    bm32 = dec.forward_rows(x, lens, blk, row0, 1030)
    assert torch.equal(bm64, bm32)
    # across 1024: the same sequences at max_len 1024 and 1088
    lens2 = np.array([1024, 1000, 700, 1023, 990], np.int32)
    blk2 = np.array([673, 649, 600, 1023, 933], np.int32)
    a = dec.forward_rows(x[:, :1024], lens2, blk2, row0, 700)
    b = dec.forward_rows(x[:, :1088], lens2, blk2, row0, 700)
    dec.check()
    assert torch.equal(a, b)
    dec.close()


def _vectors(B, T, n_rows, seed):
    r = np.random.default_rng(seed)
    lens = r.integers(1025, T + 1, size=B).astype(np.int32)
    lens[0] = T
    blk = np.array([r.integers(n_rows + 1, L + 1) for L in lens], dtype=np.int32)
    row0 = np.array([r.integers(0, L - n_rows + 1) for L in lens], dtype=np.int32)
    return lens, blk, row0


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,hd", [(3, 1300, 128), (4, 2048, 64)])
def test_forward_rows_past_1024_pads_other_sequences_and_graph_replay(B, T, hd):
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
def test_rejected_longer_calls_leave_the_handle_working():
    import ctypes as C
    dec, x = _synthetic(2, 2048)
    lens, blk, row0 = np.array([2048, 1100], np.int32), np.array([1697, 700], np.int32), np.array([1696, 0], np.int32)
    ok = dec.forward_rows(x, lens, blk, row0, 351)
    small = dict(num_layers=1, hidden=256, num_heads=2, num_kv_heads=2, head_dim=128, intermediate=512, vocab=300)
    with pytest.raises(capi.BlurrError, match="1025..2048"):
        openvla.LlamaDecoder(openvla.LlamaShapedConfig(**small, max_positions=2049, long_forward=2), DEV)
    with pytest.raises(capi.BlurrError, match="long_forward = 1"):
        openvla.LlamaDecoder(openvla.LlamaShapedConfig(**small, max_positions=1024, long_forward=2), DEV)
    for bad in (dict(max_positions=1280, long_forward=3), dict(max_positions=1280, long_forward=1),
                dict(max_positions=1280, long_forward=-1)):
        with pytest.raises(capi.BlurrError):
            openvla.LlamaDecoder(openvla.LlamaShapedConfig(**small, **bad), DEV)
    lib, stream = dec.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    arr = [(C.c_int32 * 2)(*([20] * 2)) for _ in range(3)]
    out = torch.empty((2, 5, 256), device=DEV, dtype=torch.bfloat16)
    big = torch.zeros((2, 2049, 256), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(capi.BlurrError, match="max_positions"):          # max_len past max_positions
        capi.check(lib.blurr_llm_forward_rows(dec.handle, stream, 2, 2049, C.c_void_p(big.data_ptr()), *arr, 5, C.c_void_p(out.data_ptr())))
    # generate on a 2048-position handle still stops at 320
    y = torch.zeros((1, 300, 256), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(capi.BlurrError, match="320"):
        dec.generate(y, 21)
    assert dec.generate(y, 20).shape == (1, 20)
    assert torch.equal(dec.forward_rows(x, lens, blk, row0, 351), ok)
    dec.check()
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the head at ALOHA's width (57 344 -> 4096 -> 14) against the oracle module
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def aloha_head():
    cfg = openvla.oft_aloha_config()
    torch.manual_seed(0)
    with torch.device(DEV):
        ref = O.L1RegressionActionHead(input_dim=4096, hidden_dim=cfg.head_hidden_dim, action_dim=cfg.action_dim, chunk=cfg.chunk)
    with torch.no_grad():                               # LayerNorms away from their init of 1 / 0
        for name, p in ref.named_parameters():
            if "layer_norm" in name or "ffn.0" in name:
                p.copy_((1.0 if name.endswith("weight") else 0.0) + 0.1 * torch.randn_like(p))
    ref16 = ref.to(torch.bfloat16).eval()
    head = openvla.L1RegressionHead.from_state_dict(cfg, ref16.state_dict(), 4096, DEV, max_batch=32)
    yield cfg, ref16, head
    head.close()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 32])           # 25 rows (split-K partials) and 800 rows (store epilogue)
def test_aloha_head_matches_the_oracle_module(aloha_head, batch):
    cfg, ref16, head = aloha_head
    g = torch.Generator(device=DEV).manual_seed(batch)
    rows = torch.randn((batch, cfg.chunk * cfg.action_dim, 4096), device=DEV, generator=g).to(torch.bfloat16)
    got = head.forward(rows)
    head.check()
    assert got.shape == (batch, 25, 14) and got.dtype == torch.float32
    with torch.inference_mode():
        r16 = ref16.predict_action(rows)
        r32 = copy.deepcopy(ref16).float().predict_action(rows.float())
    assert torch.equal(got, got.to(torch.bfloat16).float())
    _check_against_fp32(f"aloha head batch {batch}", got, r16, r32)
    launches = head.last_launch_count
    assert torch.equal(head.forward(rows), got) and head.last_launch_count == launches == 9


@pytest.mark.gpu
def test_head_width_limit_is_65536_columns():
    wide = openvla.L1RegressionHead(openvla.OftConfig(chunk=1, action_dim=16), 4096, DEV)      # 65 536 columns
    wide.close()
    with pytest.raises(capi.BlurrError, match="65536"):
        openvla.L1RegressionHead(openvla.OftConfig(chunk=1, action_dim=17), 4096, DEV)
    with pytest.raises(capi.BlurrError, match="65536"):
        openvla.L1RegressionHead(openvla.OftConfig(chunk=1, action_dim=16), 4160, DEV)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the ALOHA policy (three FiLM cameras + 14-D proprio) on a shrunk stack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def aloha_policy():
    B = 4
    d, s = openvla.dinov2_large_reg4_config(depth=3), openvla.siglip_so400m_config(depth=3)
    d.film_dim = s.film_dim = 4096
    dino = openvla.VitEncoder.synthetic(d, DEV, max_batch=3 * B, seed=3)
    sig = openvla.VitEncoder.synthetic(s, DEV, max_batch=3 * B, seed=4)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=3 * B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    backbone = openvla.FusedVisionBackbone(dino, sig, proj)
    oft = openvla.oft_aloha_config()
    cfg = openvla.openvla_oft_7b_config(oft)
    cfg.num_layers = 2
    dec = openvla.LlamaDecoder.from_state_dict(cfg, openvla.synthetic_llama_state_dict(cfg, DEV, 0), DEV, max_batch=B)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, DEV, max_batch=B, seed=6)
    pp = openvla.ProprioProjector.synthetic(14, 4096, DEV, max_rows=B, seed=8)
    cam = torch.device("cuda", torch.cuda.current_device())
    sizes = [(480, 640), (256, 256), (240, 320)]                    # top, left wrist, right wrist
    pres = [openvla.ImagePreprocessor(h, w, device=cam) for h, w in sizes]
    pol = openvla.OftPolicy(pres, backbone, dec, head, oft, proprio_projector=pp)
    frames = [torch.randint(0, 256, (B, h, w, 3), device=DEV, dtype=torch.uint8, generator=g) for h, w in sizes]
    yield pol, frames
    torch.cuda.synchronize()
    dec.check()
    head.check()
    for m in (*pres, dino, sig, proj, dec, head, pp):
        m.close()


# BOUNDS statistics: the dataset's min / max go where the LIBERO form passes q01 / q99
AMIN, AMAX = np.linspace(-1.0, -0.2, 14), np.linspace(0.3, 1.5, 14)
AMASK = np.array(([True] * 6 + [False]) * 2)
PMIN, PMAX = np.linspace(-2.0, -0.5, 14), np.linspace(0.5, 2.5, 14)
RAW = np.random.default_rng(1).uniform(-2.5, 3.0, size=(4, 14))


def _oracle_language(dec, lay):
    out = []
    for b in range(lay.ids.shape[0]):
        ids, mask = OF.oft_input_ids(lay.ids[b, :int(lay.text_lens[b])].tolist(), lay.n_rows)
        emb = dec.embed(torch.tensor(ids))[None]
        out.append(OF.language_embedding(emb, torch.tensor(mask, device=emb.device)[None]))
    return torch.cat(out)


@pytest.mark.gpu
def test_aloha_policy_is_the_hand_composition_and_rows_match_batch_one(aloha_policy):
    pol, frames = aloha_policy
    rows = instructions([20, 12, 31, 25], 0)
    kw = dict(proprio=RAW, proprio_q01=PMIN, proprio_q99=PMAX)
    act, norm = pol.predict_action_chunk(frames, rows, AMIN, AMAX, AMASK, return_normalized=True, **kw)
    assert act.shape == (4, 25, 14) and act.dtype == torch.float64 and norm.shape == (4, 25, 14)
    # oracle mean -> towers -> projector -> proprio row -> forward_rows -> head
    lay = openvla.oft_prompt_layout(rows, n_patches=P_ALOHA, cfg=pol.cfg)
    assert 1141 <= lay.max_len <= 1152
    lang = _oracle_language(pol.decoder, lay)
    px = pol.pixel_values(frames)
    assert px.shape == (4, 18, 224, 224)
    for i in range(3):
        assert torch.equal(px[:, 6 * i:6 * i + 6], pol.preprocessors[i](frames[i]))
    px3 = px.reshape(12, 6, 224, 224)
    patches = pol.backbone.forward(px3[:, :3], px3[:, 3:], film_cond=lang, images_per_cond=3).reshape(4, 768, 4096)
    state = torch.from_numpy(OC.normalize_proprio(RAW, PMIN, PMAX).astype(np.float32)).to(DEV, torch.bfloat16)
    p = OC.assemble_patches([patches[:, 256 * i:256 * i + 256] for i in range(3)], pol.proprio_projector.forward(state))
    x = openvla.build_oft_embeds(pol.decoder, lay, p)
    n2 = pol.head.forward(pol.decoder.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows))
    assert torch.equal(norm, n2)
    assert np.array_equal(act.numpy(), openvla.denormalize_chunk(n2.cpu().numpy(), AMIN, AMAX, AMASK))
    scale = norm.abs().max().item()
    for b, r in enumerate(rows):
        _, n1 = pol.predict_action_chunk([f[b] for f in frames], r[None].to(DEV), AMIN, AMAX, AMASK, return_normalized=True,
                                         proprio=RAW[b], proprio_q01=PMIN, proprio_q99=PMAX)
        d = (n1[0] - norm[b]).abs().max().item()
        print(f"row {b}: batch-1 vs batch-4 max_abs {d:.3e} (scale {scale:.3e})")
        assert d <= 0.05 * scale + 1e-2, (b, d, scale)


@pytest.mark.gpu
def test_aloha_policy_camera_permutation_permutes_the_patch_blocks(aloha_policy):
    pol, frames = aloha_policy
    lay = openvla.oft_prompt_layout(instructions([20] * 4, 1), n_patches=P_ALOHA, cfg=pol.cfg)
    cond = openvla.film_language_embedding(pol.decoder, lay)
    px = pol.pixel_values(frames)
    state = pol.proprio_state(RAW, PMIN, PMAX)
    rows = pol.patch_embeds(px, state, cond)
    assert rows.shape == (4, 769, 4096)
    perm = (2, 0, 1)
    moved = pol.patch_embeds(torch.cat([px[:, 6 * i:6 * i + 6] for i in perm], dim=1), state, cond)
    for j, i in enumerate(perm):
        assert torch.equal(moved[:, 256 * j:256 * j + 256], rows[:, 256 * i:256 * i + 256]), (j, i)
    assert torch.equal(moved[:, 768], rows[:, 768]) and torch.equal(rows[:, 768], pol.proprio_projector.forward(state))


@pytest.mark.gpu
def test_aloha_policy_rejects_bad_inputs(aloha_policy):
    pol, frames = aloha_policy
    rows = instructions([10, 10, 10, 10], 2)
    kw = dict(proprio=RAW, proprio_q01=PMIN, proprio_q99=PMAX)
    with pytest.raises(ValueError, match="3 per-camera"):
        pol.predict_action_chunk(frames[:2], rows, AMIN, AMAX, **kw)
    with pytest.raises(ValueError, match=r"proprio must be \[B, 14\]"):
        pol.predict_action_chunk(frames, rows, AMIN, AMAX, proprio=RAW[:, :8], proprio_q01=PMIN[:8], proprio_q99=PMAX[:8])
    with pytest.raises(ValueError, match="positions"):
        pol.predict_action_chunk(frames, instructions([170] * 4, 3), AMIN, AMAX, **kw)
    with pytest.raises(ValueError, match="2 preprocessors for 3 cameras"):
        openvla.OftPolicy(pol.preprocessors[:2], pol.backbone, pol.decoder, pol.head, pol.cfg, pol.proprio_projector)
