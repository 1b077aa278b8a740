"""Sampled decoding on the OpenVLA path (`LlamaDecoder.generate(..., do_sample=True)`, `LlamaDecoder.sample`,
`blurr_llm_generate` with `params`, `blurr_llm_sample`, `OpenVlaPolicy.predict_action(..., do_sample=True)`).

The reference semantics are transformers' `generate(do_sample=True)`: fp32 logits -> Temperature -> TopK -> TopP warpers
-> softmax -> one draw; oracle/openvla_sampling_oracle.py restates them with the kernel's Philox draw.

Error bound of a draw (the oracle's "boundary" flag): the kernel's masses are CUDA `expf` (within 2 ulp, relative
2^-22) of the same fp32 difference s - s_max, rounded to 2^-shift units (shift = 63 - bit_length(vocab)).  A prefix mass
and the target u * Z each differ from the float64 oracle by at most 2^-22 * Z plus half a unit per token, so a draw whose
target lies within 2 * 2^-22 * Z + (n_kept + 2) * 2^-shift of a prefix boundary (or of p * Z at the top-p cut) may
legitimately pick the neighbour.  Against HF's top-p a separate margin applies: HF's fp32 cumsum runs in its own order,
so tokens whose mass ahead lies within 1e-5 * Z of p * Z count as either kept or removed.

CPU (-m "not gpu"): Philox known answers, the oracle's warpers against transformers' on CPU tensors, the ctypes struct
against the header, Python argument checks.
GPU (-m gpu): the operator against HF and the oracle (kept set, probabilities, ids, non-finite rows), the draw
distribution (chi-square), sampled generate end to end in every decode regime (ids against the oracle on the returned
logits, the logits against transformers with teacher forcing), bitwise properties, rejected calls, the policy."""

import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla
from llama_helpers import Q01, Q99, hf_llama, instructions, small_policy, synthetic_decoder
from oracle import openvla_sampling_oracle as orc

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HF_MARGIN = 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("counter,key,expect", [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(counter, key, expect):
    assert orc.philox4x32_10(counter, key).tolist() == expect


def test_uniform24_is_word0_of_the_step_counter():
    seeds = np.array([0, 1, 2 ** 40 + 5, 2 ** 64 - 1], dtype=np.uint64)
    u = orc.uniform24(seeds, 3)
    for s, v in zip(seeds.tolist(), u.tolist()):
        w = orc.philox4x32_10([3, 0, 0, 0], [s & 0xFFFFFFFF, s >> 32])
        assert v == int(w[0]) >> 8 and 0 <= v < 2 ** 24


def _hf_warped(scores: torch.Tensor, T: float, k: int, p: float) -> torch.Tensor:
    from transformers.generation.logits_process import TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper
    s = scores.float()[None]
    ids = torch.zeros((1, 1), dtype=torch.long, device=s.device)
    if T != 1.0:
        s = TemperatureLogitsWarper(T)(ids, s)
    if k != 0:
        s = TopKLogitsWarper(top_k=k, min_tokens_to_keep=1)(ids, s)
    if p < 1.0:
        s = TopPLogitsWarper(top_p=p, min_tokens_to_keep=1)(ids, s)
    return torch.softmax(s, dim=-1)[0]


def _rows(vocab: int, seed: int):
    """Hand-made bf16 logits rows (fp32 tensors holding bf16 values): random, peaked, flat, ties at a top-k threshold and
    at the max, a -inf run, NaN entries."""
    g = torch.Generator().manual_seed(seed)
    r = {}
    r["random"] = torch.randn(vocab, generator=g) * 2.0
    pk = torch.randn(vocab, generator=g)
    pk[torch.randint(0, vocab, (3,), generator=g)] = torch.tensor([9.0, 7.5, 7.0])
    r["peaked"] = pk
    r["flat"] = torch.randn(vocab, generator=g) * 0.05
    r["ties"] = torch.randint(-6, 3, (vocab,), generator=g).float() * 0.5        # few levels: ties at every threshold
    tm = torch.randn(vocab, generator=g)
    tm[[3, 17, vocab - 2]] = 6.0                                                   # a tied maximum
    r["tied-max"] = tm
    ni = torch.randn(vocab, generator=g) * 1.5
    ni[vocab // 4: vocab // 2] = -float("inf")
    r["neg-inf-run"] = ni
    nn = torch.randn(vocab, generator=g) * 1.5
    nn[torch.randint(0, vocab, (vocab // 20,), generator=g)] = float("nan")
    r["nan-entries"] = nn
    return {k: v.to(torch.bfloat16).float() for k, v in r.items()}


@pytest.mark.parametrize("T", [0.25, 0.5, 1.0, 2.0])         # powers of two: x / T == x * (1 / T) exactly
def test_oracle_warpers_equal_transformers_on_cpu(T):
    vocab = 700
    checked = 0
    for name, row in _rows(vocab, 1).items():
        clean = torch.where(row.isnan(), torch.tensor(-float("inf")), row)
        for k in (0, 1, 50, vocab + 5):
            for p in (0.0, 0.5, 0.9, 1.0):
                hf = _hf_warped(clean, T, k, p) > 0
                w = orc.warp(row.numpy(), T, k, p, hf_margin=HF_MARGIN)
                # "kept" in HF's sense is a positive probability; a kept token whose exp underflows has none
                ours = w["kept"] & (w["mass"] > 0)
                if p == 1.0:
                    assert np.array_equal(ours, hf.numpy()), (name, k, p)
                else:
                    diff = ours != hf.numpy()
                    assert not (diff & ~w["ambiguous"]).any(), (name, k, p, np.nonzero(diff)[0][:8])
                checked += 1
    assert checked == 7 * 16


def test_ctypes_struct_matches_the_header():
    with open(os.path.join(ROOT, "include", "blurr_llm.h"), encoding="utf-8") as f:
        hdr = f.read()
    body = re.search(r"typedef struct blurr_llm_sampling \{(.*?)\} blurr_llm_sampling;", hdr, re.S).group(1)
    fields = re.findall(r"(\w+)\s+(\w+);", body)
    assert fields == [("uint64_t", "seed"), ("float", "temperature"), ("int32_t", "top_k"), ("float", "top_p")]
    assert [n for n, _ in capi.LlmSamplingC._fields_] == [n for _, n in fields]
    m = re.search(r"static_assert\(sizeof\(blurr_llm_sampling\) == (\d+) && offsetof\(blurr_llm_sampling, temperature\) == (\d+) &&"
                  r"\s*offsetof\(blurr_llm_sampling, top_k\) == (\d+) && offsetof\(blurr_llm_sampling, top_p\) == (\d+)", hdr)
    size, o_t, o_k, o_p = map(int, m.groups())
    assert C.sizeof(capi.LlmSamplingC) == size == 24
    assert capi.LlmSamplingC.seed.offset == 0
    assert (capi.LlmSamplingC.temperature.offset, capi.LlmSamplingC.top_k.offset, capi.LlmSamplingC.top_p.offset) == (o_t, o_k, o_p)


@pytest.mark.parametrize("kw", [
    dict(temperature=0.0), dict(temperature=-1.0), dict(temperature=float("nan")), dict(temperature=float("inf")),
    dict(top_k=-1), dict(top_k=2.5), dict(top_p=-0.1), dict(top_p=1.5), dict(top_p=float("nan")),
    dict(temperature=[1.0, 1.0]), dict(top_k=[50] * 4), dict(seed=[1, 2]), dict(seed=[-1, 0, 0]),
    dict(seed=[2 ** 64, 0, 0]), dict(seed=1.5),
])
def test_sampling_arguments_are_checked(kw):
    with pytest.raises(ValueError):
        openvla.sampling_params(3, **kw)


def test_sampling_params_defaults_and_seeds():
    torch.manual_seed(123)
    a = openvla.sampling_params(3)
    torch.manual_seed(123)
    b = openvla.sampling_params(3)
    assert [r.seed for r in a] == [r.seed for r in b] and all(0 <= r.seed < 2 ** 63 for r in a)
    assert [(r.temperature, r.top_k, r.top_p) for r in a] == [(1.0, 50, 1.0)] * 3
    c = openvla.sampling_params(3, temperature=[0.5, 1.0, 2.0], top_k=0, top_p=0.9, seed=10)
    assert [r.seed for r in c] == [10, 11, 12] and [r.temperature for r in c] == [0.5, 1.0, 2.0]
    assert [r.seed for r in openvla.sampling_params(2, seed=[2 ** 64 - 1, 0])] == [2 ** 64 - 1, 0]


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the operator
# ---------------------------------------------------------------------------------------------------------------------
def _bare_decoder(vocab: int, max_batch: int):
    """A handle without weights: blurr_llm_sample works before finalize."""
    cfg = openvla.LlamaShapedConfig(num_layers=1, hidden=128, num_heads=1, num_kv_heads=1, head_dim=128, intermediate=128,
                                    vocab=vocab, max_positions=16)
    return openvla.LlamaDecoder(cfg, DEV, max_batch=max_batch)


@pytest.mark.gpu
@pytest.mark.parametrize("vocab", [1003, 32064])
def test_operator_matches_transformers_and_the_oracle(vocab):
    rows = _rows(vocab, 2)
    names = list(rows)
    x = torch.stack([rows[n] for n in names]).to(torch.bfloat16)
    ld = (vocab + 127) // 128 * 128
    buf = torch.full((len(names), ld), float("nan"), dtype=torch.bfloat16, device=DEV)     # columns past vocab: ignored
    buf[:, :vocab] = x.to(DEV)
    dec = _bare_decoder(vocab, len(names))
    n_draws = n_flag = 0
    worst = 0.0
    for T in (0.25, 0.7, 1.0, 1.3):
        for k in (0, 1, 50, vocab + 1):
            for p in (0.0, 0.5, 0.9, 1.0):
                seeds = [1000 * len(names) * n_draws + b for b in range(len(names))]
                step = n_draws % 5
                ids, probs = dec.sample(buf, temperature=T, top_k=k, top_p=p, seed=seeds, step=step, return_probs=True)
                ids, probs = ids.cpu().numpy(), probs.cpu().numpy()
                for b, name in enumerate(names):
                    row = rows[name]
                    clean = torch.where(row.isnan(), torch.tensor(-float("inf")), row)
                    hf = _hf_warped(clean.to(DEV), T, k, p).cpu().numpy()
                    w = orc.warp(row.numpy(), T, k, p, hf_margin=HF_MARGIN)
                    ours = probs[b] > 0
                    if p == 1.0:
                        assert np.array_equal(ours, hf > 0), (name, T, k, p)
                    else:
                        diff = ours != (hf > 0)
                        assert not (diff & ~w["ambiguous"]).any(), (name, T, k, p, np.nonzero(diff)[0][:8])
                    d = np.abs(probs[b] - w["probs"]).max()
                    worst = max(worst, d)
                    assert d <= 1e-6, (name, T, k, p, d)
                    if np.array_equal(ours, hf > 0):
                        assert np.abs(probs[b] - hf).max() <= 1e-6, (name, T, k, p)
                    want, boundary = orc.draw(row.numpy(), T, k, p, seeds[b], step)
                    n_draws += 1
                    n_flag += boundary
                    if not boundary:
                        assert ids[b] == want, (name, T, k, p, ids[b], want)
                    assert w["kept"][ids[b]] and w["mass"][ids[b]] > 0, (name, T, k, p)
    dec.check()
    print(f"operator vocab {vocab}: {n_draws} draws, {n_flag} flagged as boundary, probs max |diff| {worst:.2e}")
    dec.close()


@pytest.mark.gpu
def test_non_finite_rows_take_the_argmax_and_raise_once():
    vocab = 1000
    g = torch.Generator().manual_seed(3)
    base = torch.randn(vocab, generator=g)
    rows = []
    r = torch.full((vocab,), -float("inf")); rows.append((r, 0))                  # all -inf: argmax 0
    r = torch.full((vocab,), float("nan")); rows.append((r, 0))                   # all NaN
    r = base.clone(); r[[40, 700]] = float("inf"); rows.append((r, 40))           # +inf logits: the first one
    r = base.clone(); r[123] = 3.0e38; rows.append((r, 123))                      # T = 0.25: the scaled score overflows
    r = base.clone(); r[::2] = float("nan"); r[1::2] = -float("inf"); rows.append((r, 1))   # NaN and -inf only
    x = torch.stack([v for v, _ in rows]).to(torch.bfloat16).to(DEV)
    dec = _bare_decoder(vocab, len(rows))
    dec.check()
    ids, probs = dec.sample(x, temperature=0.25, top_k=50, top_p=0.9, seed=5, return_probs=True)
    assert ids.tolist() == [i for _, i in rows]
    assert not probs.any()
    with pytest.raises(capi.BlurrError, match="sampling"):
        dec.check()
    dec.check()                                                                    # cleared
    ok = torch.randn((2, vocab), device=DEV).to(torch.bfloat16)
    dec.sample(ok, seed=1)
    dec.check()
    dec.close()


def _chi2_pvalue(counts: np.ndarray, probs: np.ndarray) -> float:
    from scipy.stats import chi2
    n = counts.sum()
    expected = probs * n
    order = np.argsort(expected)
    obs, exp = [], []
    acc_o = acc_e = 0.0
    for i in order:                                   # merge bins (smallest first) until each expects >= 5
        acc_o += counts[i]
        acc_e += expected[i]
        if acc_e >= 5.0:
            obs.append(acc_o); exp.append(acc_e)
            acc_o = acc_e = 0.0
    if acc_e > 0 and exp:
        obs[-1] += acc_o; exp[-1] += acc_e
    obs, exp = np.array(obs), np.array(exp)
    stat = ((obs - exp) ** 2 / exp).sum()
    return float(chi2.sf(stat, len(obs) - 1))


@pytest.mark.gpu
@pytest.mark.parametrize("T,k,p", [(0.7, 50, 0.9), (0.7, 0, 0.95)])
@pytest.mark.parametrize("kind", ["peaked", "flat"])
def test_draw_distribution_chi_square(kind, T, k, p):
    vocab, B = 1000, 32
    row = _rows(vocab, 4)[kind]
    w = orc.warp(row.numpy(), T, k, p)
    x = row.to(torch.bfloat16).to(DEV)[None].expand(B, vocab).contiguous()
    dec = _bare_decoder(vocab, B)
    n = 1 << 18
    ids = []
    for s0 in range(0, n, B):
        ids.append(dec.sample(x, temperature=T, top_k=k, top_p=p, seed=list(range(s0, s0 + B))))
    ids = torch.cat(ids).cpu().numpy()
    dec.check()
    dec.close()
    assert w["kept"][ids].all()
    counts = np.bincount(ids, minlength=vocab).astype(np.float64)
    kept = w["kept"]
    pv = _chi2_pvalue(counts[kept], w["probs"][kept])
    print(f"chi-square {kind} T={T} k={k} p={p}: {int(kept.sum())} kept tokens, p-value {pv:.4f}")
    assert pv > 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# GPU: sampled generate end to end
# ---------------------------------------------------------------------------------------------------------------------
GEN_CASES = [
    # hidden, heads, head_dim, inter, layers, vocab, lengths
    pytest.param(256, 2, 128, 512, 2, 1000, [8, 1, 5, 3], id="few-token"),
    pytest.param(512, 4, 128, 1408, 2, 1064, [37, 20, 29], id="mid"),
    pytest.param(512, 8, 64, 1024, 1, 300, [2, 3, 4, 5, 6, 6, 5, 4] * 4, id="fused-decode-32x8"),
    pytest.param(1280, 10, 128, 2560, 1, 1000, [5 + (7 * b) % 30 for b in range(32)], id="loop-decode-32x10"),
]
PARAMS = [(0.7, 50, 0.9), (1.3, 0, 0.95), (1.0, 50, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,heads,hd,inter,layers,vocab,lens", GEN_CASES)
def test_sampled_generate_against_the_oracle_and_transformers(hidden, heads, hd, inter, layers, vocab, lens):
    n_new = 7
    lens = np.asarray(lens, dtype=np.int32)
    B, T = len(lens), int(lens.max())
    cfg = openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=inter, vocab=vocab, max_positions=T + n_new + 1, rms_eps=1e-6)
    model = hf_llama(cfg, 0, head_scale=4.0)                # logits spread over a few units: peaked and flat rows
    dec = openvla.LlamaDecoder.from_state_dict(cfg, model.state_dict(), DEV, max_batch=B,
                                               inv_freq=model.model.rotary_emb.inv_freq.detach().float())
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn((B, T, hidden), device=DEV, generator=g) * 0.3).to(torch.bfloat16)
    flags = {True: [0, 0], False: [0, 0]}                 # top_k == 50: [draws, flagged]
    worst = 0.0
    for ragged in (False, True):
        for ci, (temp, k, p) in enumerate(PARAMS):
            seeds = [7919 * ci + 31 * b + (1 << 40) * ragged for b in range(B)]
            kw = dict(do_sample=True, temperature=temp, top_k=k, top_p=p, seed=seeds)
            if ragged:
                ids, logits = dec.generate(x, n_new, return_logits=True, prompt_lens=lens, **kw)
            else:
                ids, logits = dec.generate(x, n_new, return_logits=True, **kw)
            dec.check()
            ids_c, lg = ids.cpu().numpy(), logits.float().cpu().numpy()
            for b in range(B):
                for i in range(n_new):
                    want, boundary = orc.draw(lg[b, i], temp, k, p, seeds[b], i)
                    f = flags[k == 50]
                    f[0] += 1
                    f[1] += boundary
                    if not boundary:
                        assert ids_c[b, i] == want, (ragged, temp, k, p, b, i, ids_c[b, i], want)
            # the sampled token is what the next step was fed: transformers on prompt + ids, teacher-forced
            with torch.inference_mode():
                for b in range(B):
                    L = int(lens[b]) if ragged else T
                    emb = model.model.embed_tokens(ids[b:b + 1, :n_new - 1])
                    full = torch.cat([x[b:b + 1, :L], emb], dim=1)
                    ref = model(inputs_embeds=full).logits[0, L - 1:L - 1 + n_new].float()
                    scale = ref.abs().max().item()
                    d = (logits[b].float() - ref).abs().max().item()
                    worst = max(worst, d / scale)
                    assert d <= 0.03 * scale + 1e-3, (ragged, b, d, scale)
    total = flags[True][0] + flags[False][0]
    flagged = flags[True][1] + flags[False][1]
    print(f"sampled generate B={B}: {total} draws, {flagged} boundary ({100.0 * flagged / total:.3f} %), "
          f"top_k=50 {flags[True][1]}/{flags[True][0]}; teacher-forced logits max_abs/largest {worst:.3e}")
    assert flagged <= 0.05 * total
    assert flags[True][1] <= 0.001 * flags[True][0]
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "b32", "b32-fused"])
def test_sampled_graph_replay_equals_eager_and_repeats(name):
    dec, x = synthetic_decoder(name)
    B, T = x.shape[:2]
    greedy = dec.generate(x, 7)
    greedy_launches = dec.last_launch_count
    a = dec.generate(x, 7, do_sample=True, temperature=0.7, top_k=50, top_p=0.9, seed=1)      # captures the graph
    launches = dec.last_launch_count
    assert launches == greedy_launches
    assert torch.equal(dec.generate(x, 7, do_sample=True, temperature=0.7, top_k=50, top_p=0.9, seed=1), a)
    kw = dict(do_sample=True, temperature=[1.3] * (B - 1) + [0.5], top_k=[0] * B, top_p=0.95, seed=[99 + 3 * b for b in range(B)])
    ids_g, lg_g = dec.generate(x, 7, return_logits=True, **kw)
    assert dec.last_launch_count == launches
    lens = [max(1, T - b % 3) for b in range(B)]
    ids_gr = dec.generate(x, 7, prompt_lens=lens, **kw)
    dec.set_option("use_cuda_graph", 0)
    ids_e, lg_e = dec.generate(x, 7, return_logits=True, **kw)
    assert dec.last_launch_count == launches
    assert torch.equal(ids_g, ids_e) and torch.equal(lg_g, lg_e)
    assert torch.equal(dec.generate(x, 7, prompt_lens=lens, **kw), ids_gr)
    assert torch.equal(dec.generate(x, 7), greedy)
    dec.check()
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "mid", "b32-fused"])
def test_a_rows_ids_depend_only_on_its_prompt_and_seed(name):
    dec, x = synthetic_decoder(name)
    B, T = x.shape[:2]
    seeds = [1000 + b for b in range(B)]
    kw = dict(do_sample=True, temperature=1.0, top_k=0, top_p=0.95)
    ids0, lg0 = dec.generate(x, 7, return_logits=True, seed=seeds, **kw)
    # batch slot: the batch reversed, seeds with it
    ids1, lg1 = dec.generate(x.flip(0).contiguous(), 7, return_logits=True, seed=seeds[::-1], **kw)
    assert torch.equal(lg1.flip(0), lg0) and torch.equal(ids1.flip(0), ids0)
    # other rows' contents and seeds
    g = torch.Generator(device=DEV).manual_seed(5)
    other = (torch.randn(x.shape, device=DEV, generator=g) * 0.5).to(torch.bfloat16)
    for b in (0, B - 1):
        y = other.clone()
        y[b] = x[b]
        s = [77 + 5 * j for j in range(B)]
        s[b] = seeds[b]
        ids2 = dec.generate(y, 7, seed=s, **kw)
        assert torch.equal(ids2[b], ids0[b]), b
    # pad contents of a ragged batch
    lens = [T] + [max(1, T - 1 - b % 4) for b in range(1, B)]
    pad = torch.arange(T, device=DEV)[None, :, None] >= torch.as_tensor(lens, device=DEV)[:, None, None]
    ids3 = dec.generate(x.masked_fill(pad, 0.0), 7, prompt_lens=lens, seed=seeds, **kw)
    for fill in (float("nan"), 1e30):
        assert torch.equal(dec.generate(x.masked_fill(pad, fill), 7, prompt_lens=lens, seed=seeds, **kw), ids3), fill
    dec.check()
    dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["few", "mid", "b32", "b32-fused"])
def test_top_k_one_is_greedy(name):
    dec, x = synthetic_decoder(name)
    ids_g, lg = dec.generate(x, 7, return_logits=True)
    ids_s = dec.generate(x, 7, do_sample=True, top_k=1, temperature=0.8, top_p=0.5, seed=3)
    for b in range(x.shape[0]):
        for i in range(7):
            if ids_s[b, i] != ids_g[b, i]:
                row = lg[b, i].float()
                assert row[ids_s[b, i]] == row.max() and row[ids_g[b, i]] == row.max(), (b, i)    # a tied maximum
                break
    dec.check()
    dec.close()


@pytest.mark.gpu
def test_rejected_sampled_calls_and_null_params():
    dec, x = synthetic_decoder("few")
    B, T = x.shape[:2]
    ok = dec.generate(x, 7, do_sample=True, seed=4)
    lib, stream = dec.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty((B, 7), device=DEV, dtype=torch.int64)

    def params(**kw):
        arr = openvla.sampling_params(B, seed=4)
        for r in arr:
            for key, v in kw.items():
                setattr(r, key, v)
        return arr

    bad = [dict(temperature=0.0), dict(temperature=-2.0), dict(temperature=float("nan")), dict(temperature=float("inf")),
           dict(top_k=-1), dict(top_p=-0.5), dict(top_p=1.01), dict(top_p=float("nan"))]
    for kw in bad:
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_llm_generate(dec.handle, stream, B, T, C.c_void_p(x.data_ptr()), None, params(**kw), 7,
                                              C.c_void_p(out.data_ptr()), None))
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_llm_sample(dec.handle, stream, C.c_void_p(x.data_ptr()), B, dec.cfg.vocab, params(**kw), 0,
                                            C.c_void_p(out.data_ptr()), None))
    good = params()
    # NULL params: the greedy call
    capi.check(lib.blurr_llm_generate(dec.handle, stream, B, T, C.c_void_p(x.data_ptr()), None, None, 7, C.c_void_p(out.data_ptr()),
                                      None))
    assert torch.equal(out, dec.generate(x, 7))
    lens = (C.c_int32 * B)(*([0] + [T] * (B - 1)))
    with pytest.raises(capi.BlurrError):                                        # a zero prompt length
        capi.check(lib.blurr_llm_generate(dec.handle, stream, B, T, C.c_void_p(x.data_ptr()), lens, good, 7,
                                          C.c_void_p(out.data_ptr()), None))
    for batch in (0, B + 1):
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_llm_generate(dec.handle, stream, batch, T, C.c_void_p(x.data_ptr()), None, good, 7,
                                              C.c_void_p(out.data_ptr()), None))
    with pytest.raises(capi.BlurrError):                                        # max_prompt_len + n_new > max_positions
        dec.generate(x, 9, do_sample=True, seed=4)
    with pytest.raises(capi.BlurrError):                                        # rows > max_batch
        dec.sample(torch.zeros((B + 1, dec.cfg.vocab), device=DEV, dtype=torch.bfloat16), seed=1)
    with pytest.raises(ValueError):
        dec.generate(x, 7, do_sample=True, top_p=2.0)
    with pytest.raises(ValueError):
        dec.generate(x, 7, do_sample=True, seed=[1] * (B + 1))
    assert torch.equal(dec.generate(x, 7, do_sample=True, seed=4), ok)
    dec.check()
    dec.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the policy
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def policy():
    yield from small_policy()


@pytest.mark.gpu
def test_policy_sampling_is_repeatable_and_composes(policy):
    pol, px = policy
    dec = pol.decoder
    rows = instructions([12, 12, 12, 12], 0)
    ids_t = torch.stack(rows).to(DEV)
    kw = dict(do_sample=True, temperature=0.7, top_k=50, top_p=0.9, seed=11)
    a1, i1 = pol.predict_action_from_pixels(px, ids_t, Q01, Q99, return_token_ids=True, **kw)
    a2, i2 = pol.predict_action_from_pixels(px, ids_t, Q01, Q99, return_token_ids=True, **kw)
    assert torch.equal(i1, i2) and torch.equal(a1, a2)
    patch = pol.backbone.forward(px[:, :3], px[:, 3:])
    x = openvla.build_prompt_embeds(dec, ids_t, patch)
    assert torch.equal(dec.generate(x, 7, **kw), i1)
    # the three prompt forms agree (equal lengths: list and tensor are one computation)
    a3, i3 = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True, **kw)
    assert torch.equal(i3, i1) and torch.equal(a3, a1)
    mask = torch.ones(ids_t.shape, dtype=torch.int64)
    a4, i4 = pol.predict_action_from_pixels(px, ids_t, Q01, Q99, return_token_ids=True, attention_mask=mask, **kw)
    assert torch.equal(i4, i1) and torch.equal(a4, a1)
    # frames in, through predict_action (a preprocessor on the frames' own device index)
    frames = torch.randint(0, 256, (4, 480, 640, 3), dtype=torch.uint8, device=DEV)
    pre = openvla.ImagePreprocessor(480, 640, device=frames.device)
    pol_f = openvla.OpenVlaPolicy(pre, pol.backbone, dec)
    f1 = pol_f.predict_action(frames, rows, Q01, Q99, return_token_ids=True, **kw)[1]
    assert torch.equal(pol_f.predict_action(frames, rows, Q01, Q99, return_token_ids=True, **kw)[1], f1)
    assert torch.equal(pol_f.predict_action_from_pixels(pol_f.pixel_values(frames), rows, Q01, Q99, return_token_ids=True, **kw)[1], f1)
    pre.close()
    # seed=None: torch's default generator
    torch.manual_seed(17)
    n1 = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True, do_sample=True)[1]
    torch.manual_seed(17)
    n2 = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True, do_sample=True)[1]
    assert torch.equal(n1, n2)


@pytest.mark.gpu
def test_policy_top_k_one_is_greedy_and_default_top_k_is_50(policy):
    pol, px = policy
    dec = pol.decoder
    rows = instructions([14, 3, 25, 9], 1)
    a_g, i_g = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True)
    a_1, i_1 = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True, do_sample=True, top_k=1, seed=2)
    assert torch.equal(i_1, i_g) and torch.equal(a_1, a_g)
    # do_sample with no top_k: HF's default 50, against the oracle on the logits of the same call
    seeds = [40 + b for b in range(4)]
    _, i_d = pol.predict_action_from_pixels(px, rows, Q01, Q99, return_token_ids=True, do_sample=True, seed=seeds)
    patch = pol.backbone.forward(px[:, :3], px[:, 3:])
    text, text_lens = openvla.ragged_prompt_ids(rows)
    x, lens = openvla.build_prompt_embeds_ragged(dec, text.to(DEV), text_lens, patch)
    ids, lg = dec.generate(x, 7, return_logits=True, prompt_lens=lens, do_sample=True, seed=seeds)
    assert torch.equal(ids, i_d)
    lg = lg.float().cpu().numpy()
    flagged = 0
    for b in range(4):
        for i in range(7):
            want50, f50 = orc.draw(lg[b, i], 1.0, 50, 1.0, seeds[b], i)
            flagged += f50
            if not f50:
                assert ids[b, i].item() == want50, (b, i)
    assert flagged <= 1
