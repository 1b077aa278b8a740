"""OpenVLA-OFT's parallel decoding of action chunks: `blurr_llm_forward_rows` (OFT's block-bidirectional prefill and the
final-normed action rows), the L1-regression head (`include/blurr_act_head.h`), `oft_prompt_layout` and
`OftPolicy.predict_action_chunk`.  The specification is oracle/openvla_oft_oracle.py.

CPU (-m "not gpu"): the prompt layout for every prompt form, the oracle's mask against the hand-written rule and
transformers' own causal mask, the oracle head against the same module stack and its state_dict keys, the chunk
de-normalisation, the head config's ctypes layout and the head's symbol table.
GPU (-m gpu): forward_rows against transformers' `LlamaModel` (eager, the oracle's 4-D mask) run on each sequence alone,
with fp32 as the tie-breaker (the bar of tests/test_gpu_vit.py); forward_rows tied to generate's prefill; pads, other
sequences and graph replays; rejected calls; the head against the oracle module; the policy on a shrunk stack."""

import copy
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla
from llama_helpers import Q01, Q99, hf_llama, instructions
from oracle import openvla_oft_oracle as O

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _check_layout(lay, rows, P=256, K=8, D=7):
    for b, r in enumerate(rows):
        ids, a0, n, row0 = O.prompt_layout(r.tolist(), P, K, D)
        assert lay.text_lens[b] == len(ids) and lay.ids[b, :len(ids)].tolist() == ids and not lay.ids[b, len(ids):].any()
        assert (lay.block_starts[b], lay.seq_lens[b], lay.row_starts[b]) == (a0, n, row0)
    assert lay.max_len == int(lay.seq_lens.max()) and lay.n_rows == K * D


def test_oft_prompt_layout_forms_and_the_empty_token_rule():
    rows = instructions([5, 9, 3], 0)
    rows[1][-1] = O.EMPTY_TOKEN                               # already ends in 29871: nothing appended
    lay = openvla.oft_prompt_layout(rows)
    assert lay.text_lens.tolist() == [6, 9, 4]
    assert lay.block_starts.tolist() == [262, 265, 260] and lay.seq_lens.tolist() == [319, 322, 317]
    assert lay.row_starts.tolist() == [261, 264, 259] and lay.max_len == 322
    _check_layout(lay, rows)
    for left in (True, False):
        p, m = _padded(rows, left)
        lay2 = openvla.oft_prompt_layout(p, attention_mask=m)
        assert torch.equal(lay2.ids, lay.ids) and torch.equal(lay2.text_lens, lay.text_lens)
        assert np.array_equal(lay2.seq_lens, lay.seq_lens) and np.array_equal(lay2.block_starts, lay.block_starts)
    # equal prompts as a [B, S] tensor; rows that differ in their last id become ragged after the rule
    eq = torch.stack(instructions([7, 7], 1))
    eq[1, -1] = O.EMPTY_TOKEN
    lay3 = openvla.oft_prompt_layout(eq, n_patches=16)
    assert lay3.text_lens.tolist() == [8, 7]
    _check_layout(lay3, list(eq), P=16)
    # the causal variant: the block starts at len
    causal = openvla.oft_prompt_layout(rows, cfg=openvla.OftConfig(bidirectional_actions=False))
    assert np.array_equal(causal.block_starts, causal.seq_lens) and np.array_equal(causal.row_starts, lay.row_starts)


def test_oft_prompt_layout_rejects_sequences_past_max_positions():
    # 256 + 70 + 1 (29871) + 56 + 1 = 384 fits; one more token does not
    assert openvla.oft_prompt_layout(instructions([70], 2)).max_len == 384
    with pytest.raises(ValueError, match="max_positions"):
        openvla.oft_prompt_layout(instructions([71], 2))
    with pytest.raises(ValueError, match="max_positions"):
        openvla.oft_prompt_layout(instructions([5], 2), cfg=openvla.OftConfig(max_positions=300))
    with pytest.raises(ValueError):
        openvla.oft_prompt_layout([torch.tensor([1]), torch.tensor([], dtype=torch.int64)])


def test_oracle_mask_is_the_rule():
    L, n, a0 = 9, 8, 5                                        # one pad row at the end
    m = O.additive_mask(n, a0, L, torch.float32)[0, 0]
    lo = torch.finfo(torch.float32).min
    for p in range(L):
        for k in range(L):
            ok = k < n and (k <= p or (p >= a0 and a0 <= k < n))
            assert m[p, k].item() == (0.0 if ok else lo), (p, k)
    # a0 = len: the causal mask
    assert torch.equal(O.allowed(n, n, n), torch.ones(n, n, dtype=torch.bool).tril())


def test_oracle_mask_with_block_at_len_equals_transformers_causal_mask():
    from transformers import LlamaConfig, LlamaModel
    hc = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=2,
                     head_dim=32, vocab_size=50, max_position_embeddings=64, attn_implementation="eager")
    torch.manual_seed(0)
    model = LlamaModel(hc).eval()
    x = torch.randn(1, 12, 64)
    with torch.no_grad():
        ref = model(inputs_embeds=x).last_hidden_state
        causal = model(inputs_embeds=x, attention_mask=O.additive_mask(12, 12, dtype=torch.float32)).last_hidden_state
        bidir = model(inputs_embeds=x, attention_mask=O.additive_mask(12, 7, dtype=torch.float32)).last_hidden_state
    assert torch.equal(causal, ref)
    assert torch.equal(bidir[:, :7], ref[:, :7]) and not torch.allclose(bidir[:, 7:], ref[:, 7:])


def test_oracle_head_is_the_module_stack_and_has_oft_keys():
    torch.manual_seed(0)
    head = O.L1RegressionActionHead(input_dim=32, hidden_dim=48, action_dim=3, chunk=4)
    keys = set(head.state_dict())
    expect = {"model.layer_norm1.weight", "model.layer_norm1.bias", "model.fc1.weight", "model.fc1.bias",
              "model.layer_norm2.weight", "model.layer_norm2.bias", "model.fc2.weight", "model.fc2.bias"}
    for i in range(2):
        expect |= {f"model.mlp_resnet_blocks.{i}.ffn.{j}.{w}" for j in (0, 1) for w in ("weight", "bias")}
    assert keys == expect
    sd = head.state_dict()
    x = torch.randn(2, 12, 32)
    y = head.predict_action(x)
    assert y.shape == (2, 4, 3)
    # the same stack written out with functional ops
    h = x.reshape(2, 4, 96)
    ln = torch.nn.functional.layer_norm
    h = torch.relu(torch.nn.functional.linear(ln(h, (96,), sd["model.layer_norm1.weight"], sd["model.layer_norm1.bias"]),
                                              sd["model.fc1.weight"], sd["model.fc1.bias"]))
    for i in range(2):
        p = f"model.mlp_resnet_blocks.{i}.ffn."
        h = h + torch.relu(torch.nn.functional.linear(ln(h, (48,), sd[p + "0.weight"], sd[p + "0.bias"]), sd[p + "1.weight"], sd[p + "1.bias"]))
    h = torch.nn.functional.linear(ln(h, (48,), sd["model.layer_norm2.weight"], sd["model.layer_norm2.bias"]), sd["model.fc2.weight"],
                                   sd["model.fc2.bias"])
    assert torch.equal(y, h)
    # the product's synthetic weights carry the same keys and shapes
    syn = openvla.synthetic_act_head_state_dict(openvla.OftConfig(chunk=4, action_dim=3, head_hidden_dim=48), 32, "cpu")
    assert {k: tuple(v.shape) for k, v in syn.items()} == {k: tuple(v.shape) for k, v in sd.items()}


def test_chunk_denormalisation_is_the_detokenizer_formula_per_step():
    det = openvla.ActionDetokenizer()
    g = np.random.default_rng(0)
    tokens = g.integers(31744, 32000, size=(3, 8, 7))
    norm = det.normalized(tokens)
    q01 = np.stack([Q01 * (1 + b) for b in range(3)])
    q99 = np.stack([Q99 * (1 + 2 * b) for b in range(3)])
    mask = np.stack([np.ones(7, bool), np.array([True] * 6 + [False]), np.zeros(7, bool)])
    for stats in ((Q01, Q99, mask[1]), (q01, q99, mask), (Q01, Q99, None)):
        got = openvla.denormalize_chunk(norm, *stats)
        assert got.dtype == np.float64 and got.shape == (3, 8, 7)
        assert np.array_equal(got, O.denormalize_chunk(norm, *stats))
        for k in range(8):
            assert np.array_equal(got[:, k], det.actions(tokens[:, k], *stats))


def test_act_head_config_ctypes_layout_and_symbols():
    assert C.sizeof(capi.ActHeadConfigC) == 28 and capi.ActHeadConfigC.ln_eps.offset == 24
    assert [f[0] for f in capi.ActHeadConfigC._fields_] == ["abi_version", "input_dim", "action_dim", "chunk", "hidden_dim",
                                                          "num_blocks", "ln_eps"]
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "blurr_act_head.h")).read(), flags=re.S)
    assert set(re.findall(r"\b(blurr_[a-z0-9_]+)\s*\(", header)) == set(capi.ACT_HEAD_SYMBOLS)
    assert re.search(r"#define BLURR_ACT_HEAD_ABI_VERSION (\d+)", header).group(1) == str(capi.ACT_HEAD_ABI_VERSION)
    lib = capi.load_library()
    for name in capi.ACT_HEAD_SYMBOLS:
        assert hasattr(lib, name), name


# ---------------------------------------------------------------------------------------------------------------------
# GPU: forward_rows against transformers
# ---------------------------------------------------------------------------------------------------------------------
def _check_against_fp32(name, got, ref16, ref32):
    e_ours = (got.float() - ref32).abs()
    e_ref = (ref16.float() - ref32).abs()
    rms = ref32.pow(2).mean().sqrt().item()
    print(f"{name}: vs fp32 ours max {e_ours.max().item():.3e} mean {e_ours.mean().item():.3e} | transformers bf16 max "
          f"{e_ref.max().item():.3e} mean {e_ref.mean().item():.3e} (ref rms {rms:.3f})")
    assert e_ours.mean().item() <= 1.5 * e_ref.mean().item() + 1e-4 * rms
    assert e_ours.max().item() <= 2.5 * e_ref.max().item() + 1e-2 * rms


ROWS_CASES = [
    # hidden, heads, head_dim, inter, layers, lens, block sizes (len - a0), stress
    pytest.param(256, 2, 128, 512, 2, [12, 9], [5, 4], False, id="few-rows"),                       # 24 rows
    pytest.param(512, 4, 128, 1408, 2, [60, 41, 52], [9, 9, 12], True, id="mid-rows-stressed"),      # 180 rows
    pytest.param(512, 8, 64, 1024, 2, [100, 77, 91, 64], [20, 9, 33, 12], True, id="many-rows-hd64-stressed"),
    pytest.param(512, 4, 128, 1408, 2, [100, 97, 80], [0, 0, 0], True, id="causal-block-at-len"),
    pytest.param(256, 2, 128, 512, 1, [384, 350], [57, 57], True, id="sixth-key-block-384"),
    pytest.param(4096, 32, 128, 11008, 1, list(np.random.default_rng(3).integers(326, 341, size=32)), [57] * 32, False,
                 id="llama2-7b-widths-b32-oft-lengths"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,heads,hd,inter,layers,lens,blocks,stress", ROWS_CASES)
def test_forward_rows_matches_transformers_per_sequence(hidden, heads, hd, inter, layers, lens, blocks, stress):
    lens = np.asarray(lens, dtype=np.int32)
    blk = (lens - np.asarray(blocks, dtype=np.int32)).astype(np.int32)
    B, T = len(lens), int(lens.max())
    n_rows = int(min(blocks)) if min(blocks) > 0 else 6
    row0 = (blk - 1 if min(blocks) > 0 else lens - n_rows).astype(np.int32)
    cfg = openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=inter, vocab=320, max_positions=max(T, 8), rms_eps=1e-6)
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
            mask16 = O.additive_mask(L, int(blk[b]), L, torch.bfloat16).to(DEV)
            h16 = m16(inputs_embeds=x[b:b + 1, :L], attention_mask=mask16).last_hidden_state
            mask32 = O.additive_mask(L, int(blk[b]), L, torch.float32).to(DEV)
            h32 = m32(inputs_embeds=x[b:b + 1, :L].float(), attention_mask=mask32).last_hidden_state
        sl = slice(int(row0[b]), int(row0[b]) + n_rows)
        ours.append(got[b]); r16.append(h16[0, sl]); r32.append(h32[0, sl])
    _check_against_fp32(f"forward_rows B={B} lens {lens.min()}..{lens.max()}", torch.stack(ours), torch.stack(r16), torch.stack(r32))
    dec.close()


@pytest.mark.gpu
def test_forward_rows_last_row_is_generates_prefill():
    cfg = openvla.LlamaShapedConfig(num_layers=2, hidden=512, num_heads=4, num_kv_heads=4, head_dim=128, intermediate=1408,
                                    vocab=1064, max_positions=64)
    model = hf_llama(cfg, 0, qk_scale=6.0, head_scale=4.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, model.state_dict(), DEV, max_batch=3,
                                               inv_freq=model.model.rotary_emb.inv_freq.detach().float())
    lens = np.array([37, 20, 29], dtype=np.int32)
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn((3, 37, 512), device=DEV, generator=g)).to(torch.bfloat16)
    rows = dec.forward_rows(x, lens, lens, lens - 1, 1)
    logits = rows[:, 0] @ model.lm_head.weight.T
    ids, ref = dec.generate(x, 1, return_logits=True, prompt_lens=lens)
    dec.check()
    for b in range(3):
        scale = ref[b, 0].float().abs().max().item()
        d = (logits[b].float() - ref[b, 0].float()).abs().max().item()
        assert d <= 0.03 * scale + 1e-3, (b, d, scale)
        a = int(logits[b].float().argmax())
        if a != int(ids[b, 0]):
            top2 = ref[b, 0].float().topk(2).values
            assert (top2[0] - top2[1]).item() <= 2 * d + 2 ** -7 * scale
    dec.close()


def _synthetic(B, T, hidden=256, heads=2, hd=128, max_positions=384):
    cfg = openvla.LlamaShapedConfig(num_layers=2, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=2 * hidden, vocab=300, max_positions=max_positions)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    with torch.no_grad():
        for k, v in sd.items():
            if "q_proj" in k or "k_proj" in k:
                v.mul_(8.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV, max_batch=B)
    g = torch.Generator(device=DEV).manual_seed(7)
    return dec, (torch.randn((B, T, hidden), device=DEV, generator=g) * 0.5).to(torch.bfloat16)


def _vectors(B, T, n_rows, seed):
    r = np.random.default_rng(seed)
    lens = r.integers(n_rows + 2, T + 1, size=B).astype(np.int32)
    lens[0] = T
    blk = np.array([r.integers(n_rows + 1, L + 1) for L in lens], dtype=np.int32)
    row0 = np.array([r.integers(0, L - n_rows + 1) for L in lens], dtype=np.int32)
    return lens, blk, row0


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,hd", [(4, 8, 128), (3, 70, 128), (32, 12, 64), (2, 384, 128)])
def test_forward_rows_pads_other_sequences_and_graph_replay(B, T, hd):
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
    # the same graph replayed with other lengths, starts and row counts equals an eager run
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
def test_rejected_forward_rows_calls_leave_the_handle_working():
    B, T = 3, 40
    dec, x = _synthetic(B, T)
    lens, blk, row0 = np.array([40, 30, 20], np.int32), np.array([30, 30, 1], np.int32), np.array([29, 0, 15], np.int32)
    ok = dec.forward_rows(x, lens, blk, row0, 5)
    bad = [
        (np.array([0, 30, 20]), blk, row0, 5),         # a zero length
        (np.array([41, 30, 20]), blk, row0, 5),        # a length past max_len
        (lens, np.array([0, 30, 1]), row0, 5),          # a block start of 0
        (lens, np.array([30, 31, 1]), row0, 5),         # a block start past the length
        (lens, blk, np.array([36, 0, 15]), 5),          # rows run past the length
        (lens, blk, np.array([-1, 0, 15]), 5),          # a negative row start
        (lens, blk, row0, 0),                           # no rows
    ]
    for args in bad:
        with pytest.raises(capi.BlurrError):
            dec.forward_rows(x, *args)
    with pytest.raises(ValueError):
        dec.forward_rows(x, lens[:2], blk, row0, 5)
    lib, stream = dec.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty((4, 5, 256), device=DEV, dtype=torch.bfloat16)
    arr = [(C.c_int32 * 4)(*([20] * 4)) for _ in range(3)]
    for batch in (0, B + 1):
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_llm_forward_rows(dec.handle, stream, batch, T, C.c_void_p(x.data_ptr()), *arr, 5, C.c_void_p(out.data_ptr())))
    with pytest.raises(capi.BlurrError):                              # max_len past max_positions
        capi.check(lib.blurr_llm_forward_rows(dec.handle, stream, 1, 385, C.c_void_p(x.data_ptr()), *arr, 5, C.c_void_p(out.data_ptr())))
    # generate on a 384-position handle still stops at 320 (its decode kernels' limit)
    y = torch.zeros((1, 300, 256), device=DEV, dtype=torch.bfloat16)
    with pytest.raises(capi.BlurrError, match="320"):
        dec.generate(y, 21)
    assert dec.generate(y, 20).shape == (1, 20)
    # max_positions 385 at create
    with pytest.raises(capi.BlurrError):
        openvla.LlamaDecoder(openvla.LlamaShapedConfig(num_layers=1, hidden=256, num_heads=2, num_kv_heads=2, head_dim=128,
                                                       intermediate=512, vocab=300, max_positions=385), DEV)
    assert torch.equal(dec.forward_rows(x, lens, blk, row0, 5), ok)
    dec.check()
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the head against the oracle module
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def oft_head():
    cfg = openvla.OftConfig()
    torch.manual_seed(0)
    ref = O.L1RegressionActionHead(input_dim=4096, hidden_dim=cfg.head_hidden_dim, action_dim=cfg.action_dim, chunk=cfg.chunk)
    with torch.no_grad():                               # LayerNorms away from their init of 1 / 0
        for name, p in ref.named_parameters():
            if "layer_norm" in name or "ffn.0" in name:
                p.copy_((1.0 if name.endswith("weight") else 0.0) + 0.1 * torch.randn_like(p))
    ref16 = ref.to(DEV, torch.bfloat16).eval()
    head = openvla.L1RegressionHead.from_state_dict(cfg, ref16.state_dict(), 4096, DEV, max_batch=32)
    yield cfg, ref16, head
    head.close()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 32])           # 8 rows (split-K partials) and 256 rows (store epilogue)
def test_head_matches_the_oracle_module(oft_head, batch):
    cfg, ref16, head = oft_head
    g = torch.Generator(device=DEV).manual_seed(batch)
    rows = torch.randn((batch, cfg.chunk * cfg.action_dim, 4096), device=DEV, generator=g).to(torch.bfloat16)
    got = head.forward(rows)
    head.check()
    assert got.shape == (batch, cfg.chunk, cfg.action_dim) and got.dtype == torch.float32
    with torch.inference_mode():
        r16 = ref16.predict_action(rows)
        r32 = copy.deepcopy(ref16).float().predict_action(rows.float())
    assert torch.equal(got, got.to(torch.bfloat16).float())             # the module's bf16 values, widened
    _check_against_fp32(f"head batch {batch}", got, r16, r32)
    launches = head.last_launch_count
    assert torch.equal(head.forward(rows), got) and head.last_launch_count == launches == 9


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the policy on a shrunk stack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def oft_policy():
    B = 4
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(depth=3), DEV, max_batch=B, seed=3)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(depth=3), DEV, max_batch=B, seed=4)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    backbone = openvla.FusedVisionBackbone(dino, sig, proj)
    oft = openvla.OftConfig()
    cfg = openvla.openvla_oft_7b_config(oft)
    cfg.num_layers = 2
    dec = openvla.LlamaDecoder.from_state_dict(cfg, openvla.synthetic_llama_state_dict(cfg, DEV, 0), DEV, max_batch=B)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, DEV, max_batch=B, seed=6)
    pre = openvla.ImagePreprocessor(480, 640, device=DEV)
    pol = openvla.OftPolicy(pre, backbone, dec, head, oft)
    px = (torch.rand((B, 6, 224, 224), device=DEV, generator=g) * 2 - 1).to(torch.bfloat16)
    yield pol, px
    torch.cuda.synchronize()
    dec.check()
    head.check()
    for m in (pre, dino, sig, proj, dec, head):
        m.close()


MASK = np.array([True] * 6 + [False])


@pytest.mark.gpu
def test_policy_chunk_shape_prompt_forms_and_rows_against_batch_one(oft_policy):
    pol, px = oft_policy
    rows = instructions([14, 3, 25, 9], 0)
    act, norm = pol.predict_action_chunk_from_pixels(px, rows, Q01, Q99, MASK, return_normalized=True)
    assert act.shape == (4, 8, 7) and act.dtype == torch.float64 and norm.shape == (4, 8, 7)
    assert np.array_equal(act.numpy(), openvla.denormalize_chunk(norm.cpu().numpy(), Q01, Q99, MASK))
    for left in (True, False):
        p, m = _padded(rows, left)
        a2 = pol.predict_action_chunk_from_pixels(px, p.to(DEV), Q01, Q99, MASK, attention_mask=m)
        assert torch.equal(a2, act)
    scale = norm.abs().max().item()
    for b, r in enumerate(rows):
        _, n1 = pol.predict_action_chunk_from_pixels(px[b:b + 1], r[None].to(DEV), Q01, Q99, MASK, return_normalized=True)
        d = (n1[0] - norm[b]).abs().max().item()
        print(f"row {b}: batch-1 vs batch-4 max_abs {d:.3e} (scale {scale:.3e})")
        assert d <= 0.05 * scale + 1e-2, (b, d, scale)
    # equal prompts as a tensor
    eq = instructions([17] * 4, 1)
    assert torch.equal(pol.predict_action_chunk_from_pixels(px, torch.stack(eq).to(DEV), Q01, Q99),
                       pol.predict_action_chunk_from_pixels(px, eq, Q01, Q99))


@pytest.mark.gpu
def test_policy_causal_variant_is_the_causal_restatement(oft_policy):
    pol, px = oft_policy
    rows = instructions([10, 22, 5, 16], 3)
    causal = openvla.OftPolicy(pol.preprocessor, pol.backbone, pol.decoder, pol.head,
                               openvla.OftConfig(bidirectional_actions=False))
    got = causal.predict_action_chunk_from_pixels(px, rows, Q01, Q99)
    patch = pol.backbone.forward(px[:, :3], px[:, 3:])
    lay = openvla.oft_prompt_layout(rows, n_patches=256)
    x = openvla.build_oft_embeds(pol.decoder, lay, patch)
    h = pol.decoder.forward_rows(x, lay.seq_lens, lay.seq_lens, lay.row_starts, lay.n_rows)       # block start = len: causal
    expect = openvla.denormalize_chunk(pol.head.forward(h).cpu().numpy(), Q01, Q99)
    assert np.array_equal(got.numpy(), expect)
    assert not torch.equal(got, pol.predict_action_chunk_from_pixels(px, rows, Q01, Q99))
    # the embeddings: prompt rows, zeroed slots, the stop row, zeros after
    for b in range(4):
        a0, n = int(lay.block_starts[b]), int(lay.seq_lens[b])
        assert not x[b, a0:a0 + 56].any() and not x[b, n:].any()
        assert torch.equal(x[b, a0 + 56], pol.decoder.embed(torch.tensor([2], device=DEV))[0])
