"""Prompts of different lengths in one batch on the OpenVLA path (`LlamaDecoder.generate(..., prompt_lens=...)`,
`blurr_llm_generate_ragged`, `ragged_prompt_ids`, `build_prompt_embeds_ragged`, `OpenVlaPolicy.predict_action` with a
list or an `attention_mask`).

Layout: sequence b's prompt is rows 0 .. len_b - 1 of its T_max rows, pads after; its token i is generated at position
len_b + i.  So every sequence must get what the model gives for that sequence alone.

CPU (-m "not gpu"): the three prompt forms normalise to the same ids and lengths; malformed masks and empty rows raise.
GPU (-m gpu): every sequence of a ragged batch against transformers' `LlamaForCausalLM` (eager) run on that sequence
alone, in every regime the engine switches on (tolerance and near-tie rule of tests/test_gpu_llm.py); bitwise: equal
lengths through `prompt_lens` == the plain call, pad contents never matter, other sequences never matter, a graph
replay with new lengths == an eager run; rejected calls; the policy's prompt forms, per-row statistics and rows against
batch-1 calls."""

import ctypes as C

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla

DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: prompt normalisation
# ---------------------------------------------------------------------------------------------------------------------
def _prompts():
    g = torch.Generator().manual_seed(0)
    rows = []
    for n in (5, 1, 9, 3):
        r = torch.randint(3, 32000, (n,), generator=g)
        r[0] = 1
        rows.append(r)
    return rows


def _padded(rows, left: bool):
    S = max(r.numel() for r in rows)
    ids = torch.full((len(rows), S), 7, dtype=torch.int64)          # pad id 7: must not leak into the result
    mask = torch.zeros((len(rows), S), dtype=torch.int64)
    for b, r in enumerate(rows):
        sl = slice(S - r.numel(), S) if left else slice(0, r.numel())
        ids[b, sl] = r
        mask[b, sl] = 1
    return ids, mask


def test_ragged_prompt_ids_forms_agree():
    rows = _prompts()
    ids, lens = openvla.ragged_prompt_ids(rows)
    assert lens.tolist() == [5, 1, 9, 3] and ids.shape == (4, 9) and ids.dtype == torch.int64
    for b, r in enumerate(rows):
        assert torch.equal(ids[b, :r.numel()], r) and not ids[b, r.numel():].any()
    for left in (True, False):
        p, m = _padded(rows, left)
        ids2, lens2 = openvla.ragged_prompt_ids(p, attention_mask=m)
        assert torch.equal(ids2, ids) and torch.equal(lens2, lens)
        ids3, lens3 = openvla.ragged_prompt_ids(p, attention_mask=m.bool())
        assert torch.equal(ids3, ids) and torch.equal(lens3, lens)
    # a [B, S] tensor without a mask: every row is S tokens
    full = torch.stack([torch.arange(1, 6), torch.arange(11, 16)])
    ids4, lens4 = openvla.ragged_prompt_ids(full)
    assert torch.equal(ids4, full) and lens4.tolist() == [5, 5]


@pytest.mark.parametrize("mask", [
    [[1, 0, 1, 1], [1, 1, 1, 1]],          # a gap
    [[0, 1, 1, 0], [1, 1, 0, 1]],          # a gap in the second row
    [[1, 1, 1, 1], [0, 0, 0, 0]],          # an empty row
    [[1, 1, 2, 1], [1, 1, 1, 1]],          # not a 0/1 mask
    [[1, 1, 1], [1, 1, 1]],                # wrong shape
])
def test_ragged_prompt_ids_rejects_malformed_masks(mask):
    ids = torch.arange(8).reshape(2, 4)
    with pytest.raises(ValueError):
        openvla.ragged_prompt_ids(ids, attention_mask=torch.tensor(mask))


def test_ragged_prompt_ids_rejects_empty_rows():
    with pytest.raises(ValueError):
        openvla.ragged_prompt_ids([torch.tensor([1, 2, 3]), torch.tensor([], dtype=torch.int64)])
    with pytest.raises(ValueError):
        openvla.ragged_prompt_ids([])
    with pytest.raises(ValueError):
        openvla.ragged_prompt_ids([torch.tensor([[1, 2]])])
    with pytest.raises(ValueError):
        openvla.ragged_prompt_ids([torch.tensor([1, 2])], attention_mask=torch.ones(1, 2))


def test_actions_take_per_row_statistics():
    det = openvla.ActionDetokenizer()
    tokens = np.array([[31900, 31800, 31744, 31990, 31872, 31850, 31999],
                       [31950, 31760, 31999, 31745, 31800, 31901, 31744]])
    q01 = np.array([[-1.0] * 7, [-0.1, -0.2, -0.3, -0.4, -0.5, -0.6, 0.0]])
    q99 = np.array([[1.0] * 7, [0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 2.0]])
    mask = np.array([[True] * 7, [True] * 6 + [False]])
    got = det.actions(tokens, q01, q99, mask)
    for b in range(2):
        assert np.array_equal(got[b], det.actions(tokens[b:b + 1], q01[b], q99[b], mask[b])[0])
    norm = det.normalized(tokens)
    assert np.array_equal(got[0], norm[0])                              # q01 = -1, q99 = 1: the identity
    assert got[1, 6] == norm[1, 6]                                      # masked out: stays normalised


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the decoder against transformers, sequence by sequence
# ---------------------------------------------------------------------------------------------------------------------
def _hf_model(cfg: openvla.LlamaShapedConfig, seed: int, stress: bool):
    from transformers import LlamaConfig, LlamaForCausalLM
    hc = LlamaConfig(hidden_size=cfg.hidden, intermediate_size=cfg.intermediate, num_hidden_layers=cfg.num_layers,
                     num_attention_heads=cfg.num_heads, num_key_value_heads=cfg.num_kv_heads, head_dim=cfg.head_dim,
                     vocab_size=cfg.vocab, max_position_embeddings=2048, rms_norm_eps=cfg.rms_eps, rope_theta=cfg.rope_theta,
                     attn_implementation="eager", tie_word_embeddings=False)
    torch.manual_seed(seed)
    model = LlamaForCausalLM(hc).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "layernorm" in name or name.endswith("norm.weight"):
                p.copy_(1.0 + 0.2 * torch.randn_like(p))                 # norms away from their init of 1
            elif stress and ("q_proj" in name or "k_proj" in name):
                p.mul_(6.0)                                              # peaked attention: RoPE and the mask matter
            elif stress and ("embed_tokens" in name or "lm_head" in name):
                p.mul_(4.0)
    return model.to(torch.bfloat16).to(DEV)


@torch.inference_mode()
def _hf_greedy(model, inputs_embeds, n_new):
    out = model(inputs_embeds=inputs_embeds, use_cache=True)
    past = out.past_key_values
    logits, ids = [], []
    last = out.logits[:, -1, :]
    for i in range(n_new):
        logits.append(last)
        tok = last.float().argmax(dim=-1)
        ids.append(tok)
        if i + 1 < n_new:
            out = model(input_ids=tok[:, None], past_key_values=past, use_cache=True)
            past = out.past_key_values
            last = out.logits[:, -1, :]
    return torch.stack(ids, dim=1), torch.stack(logits, dim=1)


def _lens(batch, lo, hi, seed):
    return np.random.default_rng(seed).integers(lo, hi + 1, size=batch).astype(np.int32)


RAGGED_CASES = [
    # hidden, heads, head_dim, inter, layers, vocab, lengths, stress
    pytest.param(256, 2, 128, 512, 2, 1000, [8, 1, 5, 3], False, id="few-token-with-one-token-prompt"),   # 32 rows
    pytest.param(256, 2, 128, 512, 1, 300, [1, 2], False, id="few-token-lengths-1-2"),
    pytest.param(512, 4, 128, 1408, 3, 1064, [37, 20, 29], True, id="mid-stressed"),                       # 111 rows
    pytest.param(512, 8, 64, 1024, 1, 300, _lens(32, 2, 6, 1), False, id="fused-decode-hd64-32x8"),     # 256 CTAs
    pytest.param(1280, 10, 128, 2560, 2, 1000, _lens(32, 5, 40, 2), False, id="loop-decode-32x10"),
    pytest.param(4096, 32, 128, 11008, 1, 32064, _lens(32, 270, 291, 3), False, id="llama2-7b-widths-b32"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,heads,hd,inter,layers,vocab,lens,stress", RAGGED_CASES)
def test_ragged_generate_matches_transformers_per_sequence(hidden, heads, hd, inter, layers, vocab, lens, stress):
    n_new = 7
    lens = np.asarray(lens, dtype=np.int32)
    B, T = len(lens), int(lens.max())
    cfg = openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=inter, vocab=vocab, max_positions=T + n_new + 1, rms_eps=1e-6)
    model = _hf_model(cfg, 0, stress)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, model.state_dict(), DEV, max_batch=B,
                                               inv_freq=model.model.rotary_emb.inv_freq.detach().float())
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn((B, T, hidden), device=DEV, generator=g) * (1.0 if stress else 0.3)).to(torch.bfloat16)
    ids, logits = dec.generate(x, n_new, return_logits=True, prompt_lens=lens)
    dec.check()
    assert torch.equal(dec.generate(x, n_new, prompt_lens=lens), ids)          # graph replay, no logits
    first_equal, worst = 0, 0.0
    for b in range(B):
        ref_ids, ref_logits = _hf_greedy(model, x[b:b + 1, :lens[b]], n_new)
        scale = ref_logits.float().abs().max().item()
        for i in range(n_new):
            d = (logits[b, i].float() - ref_logits[0, i].float()).abs().max().item()
            worst = max(worst, d / scale)
            assert d <= 0.03 * scale + 1e-3, (b, int(lens[b]), i, d, scale)
            if ids[b, i] != ref_ids[0, i]:
                top2 = ref_logits[0, i].float().topk(2).values
                assert (top2[0] - top2[1]).item() <= 2 * d + 2 ** -7 * scale, (b, i, top2, d)
                break                                  # the sequences diverged on a tie: later steps see other tokens
        first_equal += int(ids[b, 0] == ref_ids[0, 0])
    print(f"ragged B={B} lengths {lens.min()}..{lens.max()}: logits max_abs/largest {worst:.3e}, "
          f"first token equal in {first_equal}/{B}")
    assert first_equal >= 0.5 * B
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: bitwise properties (synthetic weights)
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = {
    # hidden, heads, head_dim, inter, layers, vocab, batch, T_max
    "few": (256, 2, 128, 512, 2, 1000, 4, 8),
    "mid": (512, 4, 128, 1408, 2, 1064, 3, 37),
    "b32": (1280, 10, 128, 2560, 2, 1000, 32, 12),
    "b32-fused": (512, 8, 64, 1024, 1, 300, 32, 6),
}


def _decoder(name, n_new=7):
    hidden, heads, hd, inter, layers, vocab, B, T = SHAPES[name]
    cfg = openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=inter, vocab=vocab, max_positions=T + n_new + 1)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    with torch.no_grad():
        for k, v in sd.items():
            if "q_proj" in k or "k_proj" in k:
                v.mul_(8.0)                                              # peaked attention
            if k.startswith("lm_head"):
                v.mul_(4.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV, max_batch=B)
    g = torch.Generator(device=DEV).manual_seed(7)
    x = (torch.randn((B, T, hidden), device=DEV, generator=g) * 0.5).to(torch.bfloat16)
    return dec, x


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "mid", "b32", "b32-fused"])
def test_equal_lengths_through_prompt_lens_are_bitwise_the_plain_call(name):
    dec, x = _decoder(name)
    B, T = x.shape[:2]
    ids0, lg0 = dec.generate(x, 7, return_logits=True)
    ids1, lg1 = dec.generate(x, 7, return_logits=True, prompt_lens=[T] * B)
    dec.check()
    assert torch.equal(ids0, ids1) and torch.equal(lg0, lg1)
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "mid", "b32", "b32-fused"])
def test_pad_rows_and_other_sequences_never_matter(name):
    dec, x = _decoder(name)
    B, T = x.shape[:2]
    lens = _lens(B, 1, T, 11)
    lens[0] = T
    pad = torch.arange(T, device=DEV)[None, :, None] >= torch.as_tensor(lens, device=DEV)[:, None, None]
    zero = x.masked_fill(pad, 0.0)
    ids0, lg0 = dec.generate(zero, 7, return_logits=True, prompt_lens=lens)
    for fill in (float("nan"), 1e30, -1e30):
        ids1, lg1 = dec.generate(x.masked_fill(pad, fill), 7, return_logits=True, prompt_lens=lens)
        assert torch.equal(ids1, ids0) and torch.equal(lg1, lg0), fill
    # other sequences' contents: sequence b's outputs are unchanged
    g = torch.Generator(device=DEV).manual_seed(99)
    other = (torch.randn(x.shape, device=DEV, generator=g) * 0.5).to(torch.bfloat16)
    for b in (0, B - 1):
        y = other.clone()
        y[b] = zero[b]
        ids2, lg2 = dec.generate(y, 7, return_logits=True, prompt_lens=lens)
        assert torch.equal(ids2[b], ids0[b]) and torch.equal(lg2[b], lg0[b]), b
    dec.check()
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "b32", "b32-fused"])
def test_graph_replay_with_new_lengths_equals_eager(name):
    dec, x = _decoder(name)
    B, T = x.shape[:2]
    lens_a, lens_b = _lens(B, 1, T, 21), _lens(B, 1, T, 22)
    dec.generate(x, 7, prompt_lens=lens_a)                   # captures the (B, T, 7) ragged graph
    launches = dec.last_launch_count
    ids_g, lg_g = dec.generate(x, 7, return_logits=True, prompt_lens=lens_b)
    ids_g2 = dec.generate(x, 7, prompt_lens=lens_b)
    assert dec.last_launch_count == launches                 # same graph, replayed with other lengths
    dec.set_option("use_cuda_graph", 0)
    ids_e, lg_e = dec.generate(x, 7, return_logits=True, prompt_lens=lens_b)
    assert dec.last_launch_count == launches
    dec.check()
    assert torch.equal(ids_g, ids_e) and torch.equal(lg_g, lg_e) and torch.equal(ids_g2, ids_e)
    dec.close()


@pytest.mark.gpu
def test_rejected_ragged_calls_leave_the_handle_working():
    dec, x = _decoder("few")
    B, T = x.shape[:2]
    ok = dec.generate(x, 7, prompt_lens=[T] * B)
    bad = [
        [0] + [T] * (B - 1),                                  # a zero length
        [T + 1] + [T] * (B - 1),                              # above max_prompt_len
        [-3] * B,
    ]
    for lens in bad:
        with pytest.raises(capi.BlurrError):
            dec.generate(x, 7, prompt_lens=lens)
    with pytest.raises(capi.BlurrError):                      # max_prompt_len + n_new > max_positions
        dec.generate(x, 9, prompt_lens=[T] * B)
    with pytest.raises(ValueError):                           # one length per sequence
        dec.generate(x, 7, prompt_lens=[T] * (B - 1))
    lib, stream = dec.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty((B, 7), device=DEV, dtype=torch.int64)
    lens = (C.c_int32 * B)(*([T] * B))
    with pytest.raises(capi.BlurrError):                      # null prompt_lens
        capi.check(lib.blurr_llm_generate_ragged(dec.handle, stream, B, T, C.c_void_p(x.data_ptr()), None, 7,
                                                 C.c_void_p(out.data_ptr()), None))
    for batch in (0, B + 1):                                  # batch out of range
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_llm_generate_ragged(dec.handle, stream, batch, T, C.c_void_p(x.data_ptr()), lens, 7,
                                                     C.c_void_p(out.data_ptr()), None))
    assert torch.equal(dec.generate(x, 7, prompt_lens=[T] * B), ok)
    dec.check()
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the policy
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def policy():
    """Shrunk towers (depth 3) and a 2-layer 4096-wide decoder, as in tests/test_openvla_preprocess.py."""
    B = 4
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(depth=3), DEV, max_batch=B, seed=3)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(depth=3), DEV, max_batch=B, seed=4)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    backbone = openvla.FusedVisionBackbone(dino, sig, proj)
    cfg = openvla.LlamaShapedConfig(num_layers=2)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    with torch.no_grad():
        sd["lm_head.weight"].mul_(8.0)                       # spread the logits: fewer near-ties between rows
    dec = openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV, max_batch=B)
    pre = openvla.ImagePreprocessor(480, 640, device=DEV)
    pol = openvla.OpenVlaPolicy(pre, backbone, dec)
    px = (torch.rand((B, 6, 224, 224), device=DEV, generator=g) * 2 - 1).to(torch.bfloat16)
    yield pol, px
    torch.cuda.synchronize()
    dec.check()
    for m in (pre, dino, sig, proj, dec):
        m.close()


def _instructions(lengths, seed):
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in lengths:
        r = torch.randint(3, 32000, (n,), generator=g)
        r[0] = 1
        rows.append(r)
    return rows


Q01 = np.array([-0.03, -0.04, -0.02, -0.1, -0.1, -0.2, 0.0])
Q99 = np.array([0.03, 0.04, 0.03, 0.1, 0.1, 0.2, 1.0])
MASK = np.array([True] * 6 + [False])


@pytest.mark.gpu
def test_policy_prompt_forms_agree_and_rows_match_batch_one(policy):
    pol, px = policy
    rows = _instructions([14, 3, 25, 9], 0)
    act, ids = pol.predict_action_from_pixels(px, rows, Q01, Q99, MASK, return_token_ids=True)
    assert act.shape == (4, 7) and ids.shape == (4, 7)
    for left in (True, False):
        p, m = _padded(rows, left)
        a2, i2 = pol.predict_action_from_pixels(px, p.to(DEV), Q01, Q99, MASK, return_token_ids=True, attention_mask=m)
        assert torch.equal(i2, ids) and torch.equal(a2, act)
    dec = pol.decoder
    patch = pol.backbone.forward(px[:, :3], px[:, 3:])
    text, text_lens = openvla.ragged_prompt_ids(rows)
    x, lens = openvla.build_prompt_embeds_ragged(dec, text.to(DEV), text_lens, patch)
    assert lens.tolist() == [256 + n for n in (14, 3, 25, 9)] and x.shape[1] == 256 + 25
    ids_r, lg_r = dec.generate(x, 7, return_logits=True, prompt_lens=lens)
    assert torch.equal(ids_r, ids)
    same = 0
    for b, r in enumerate(rows):
        a1, i1 = pol.predict_action_from_pixels(px[b:b + 1], r[None].to(DEV), Q01, Q99, MASK, return_token_ids=True)
        if torch.equal(i1[0], ids[b]):
            assert torch.equal(a1[0], act[b])
            same += 1
            continue
        # batch 1 and the ragged batch run their GEMMs on other row counts (other split-K plans, other summation
        # orders): a different token only where the batch-1 logits are a near-tie within that noise
        _, lg1 = dec.generate(openvla.build_prompt_embeds(dec, r[None].to(DEV), patch[b:b + 1]), 7, return_logits=True)
        scale = lg1.float().abs().max().item()
        for i in range(7):
            d = (lg_r[b, i].float() - lg1[0, i].float()).abs().max().item()
            assert d <= 0.03 * scale + 1e-3, (b, i, d, scale)
            if ids[b, i] != i1[0, i]:
                top2 = lg1[0, i].float().topk(2).values
                assert (top2[0] - top2[1]).item() <= 2 * d + 2 ** -7 * scale, (b, i, top2, d)
                break
    print(f"policy: {same}/4 rows equal a batch-1 call")
    assert same >= 2


@pytest.mark.gpu
def test_policy_equal_length_list_is_bitwise_the_tensor_call(policy):
    pol, px = policy
    rows = _instructions([17] * 4, 1)
    a0, i0 = pol.predict_action_from_pixels(px, torch.stack(rows).to(DEV), Q01, Q99, MASK, return_token_ids=True)
    a1, i1 = pol.predict_action_from_pixels(px, rows, Q01, Q99, MASK, return_token_ids=True)
    assert torch.equal(i0, i1) and torch.equal(a0, a1)


@pytest.mark.gpu
def test_policy_per_row_statistics(policy):
    pol, px = policy
    rows = _instructions([6, 11, 2, 20], 2)
    q01 = np.stack([Q01 * (1 + b) for b in range(4)])
    q99 = np.stack([Q99 * (1 + 2 * b) for b in range(4)])
    mask = np.stack([MASK, ~MASK, MASK, np.ones(7, bool)])
    act, ids = pol.predict_action_from_pixels(px, rows, q01, q99, mask, return_token_ids=True)
    det = pol.detokenizer
    tok = ids.cpu().numpy()
    for b in range(4):
        expect = det.actions(tok[b:b + 1], q01[b], q99[b], mask[b])[0]
        assert np.array_equal(act[b].numpy(), expect)
    act_shared = pol.predict_action_from_pixels(px, rows, Q01, Q99, MASK)
    assert np.array_equal(act_shared[0].numpy(), act[0].numpy()) and not np.array_equal(act_shared[1].numpy(), act[1].numpy())
