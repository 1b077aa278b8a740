"""Llama-shaped decoder (SURVEY.md §8(f) row 3, include/blurr_llm.h) against transformers' `LlamaForCausalLM` with
eager attention - the class OpenVLA's remote code instantiates for its language model - on the same bf16 weights and
prompt embeddings: the logits every generated token is chosen from, and the greedy tokens themselves.  The reference's
own OpenVLA code is not vendored (parity against it is unpinned, DESIGN.md); transformers 5.5 is a library of this image.

Tolerance: both sides are bf16 pipelines with fp32 accumulation whose GEMMs sum in different orders, so logits agree to
a few bf16 ulps of the largest logit; a greedy token may only differ where the HF run's own top-2 margin is inside that
noise (then the sequences legitimately diverge and the comparison stops there)."""

import numpy as np
import pytest
import torch

from blurr_b200 import openvla
from llama_helpers import hf_greedy, hf_llama

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _inv_freq(model):
    return model.model.rotary_emb.inv_freq.detach().float()


CASES = [
    # hidden, heads, head_dim, inter, layers, vocab, batch, prompt, stress
    (256, 2, 128, 512, 2, 1000, 1, 20, False),        # prefill on the few-token path too
    (512, 4, 128, 1408, 3, 1064, 3, 37, True),        # 111 prompt rows: bf16 hand-off path; vocab not a tile multiple
    (512, 4, 128, 1408, 2, 1064, 1, 281, True),       # OpenVLA's prompt length: the 257..288-row CTA-pair GEMMs
    (256, 4, 64, 704, 2, 520, 4, 64, False),          # head_dim 64
    (1280, 10, 128, 2560, 2, 1000, 32, 12, False),    # 32 sequences x 10 heads: the many-CTA decode attention + separate RoPE
    (1280, 10, 128, 2560, 1, 1000, 31, 59, False),    # odd sizes: 59 + i keys, 31 sequences
    (256, 2, 128, 512, 1, 300, 5, 1, False),          # a one-token prompt
    (512, 8, 64, 1024, 1, 300, 32, 3, False),         # head_dim 64, 256 decode CTAs (fused RoPE path at its upper edge)
    (4096, 32, 128, 11008, 2, 32064, 2, 40, False),   # Llama-2-7B's real widths (4096-column consumer, 172-tile gate/up, padded vocab)
    (4096, 32, 128, 11008, 1, 32064, 32, 9, False),   # ... at 32 sequences: 288 prompt rows (the widest chunked split-K case)
]


@pytest.mark.parametrize("hidden,heads,hd,inter,layers,vocab,batch,prompt,stress", CASES)
def test_generate_matches_transformers_llama(hidden, heads, hd, inter, layers, vocab, batch, prompt, stress):
    n_new = 7
    cfg = openvla.LlamaShapedConfig(num_layers=layers, hidden=hidden, num_heads=heads, num_kv_heads=heads, head_dim=hd,
                                    intermediate=inter, vocab=vocab, max_positions=prompt + n_new + 1, rms_eps=1e-6)
    model = hf_llama(cfg, 0, qk_scale=6.0 if stress else 1.0, head_scale=4.0 if stress else 1.0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, model.state_dict(), DEV, max_batch=batch, inv_freq=_inv_freq(model))
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    x = (torch.randn((batch, prompt, hidden), device=DEV, generator=g) * (1.0 if stress else 0.3)).to(torch.bfloat16)
    ref_ids, ref_logits = hf_greedy(model, x, n_new)
    ids, logits = dec.generate(x, n_new, return_logits=True)
    dec.check()
    ids2 = dec.generate(x, n_new)                      # graph replay, no logits
    dec.check()
    assert torch.equal(ids, ids2)
    assert dec.last_launch_count > 0
    scale = ref_logits.float().abs().max().item()
    worst = 0.0
    for b in range(batch):
        for i in range(n_new):
            d = (logits[b, i].float() - ref_logits[b, i].float()).abs().max().item()
            worst = max(worst, d)
            assert d <= 0.03 * scale + 1e-3, (b, i, d, scale)
            if ids[b, i] != ref_ids[b, i]:
                top2 = ref_logits[b, i].float().topk(2).values
                assert (top2[0] - top2[1]).item() <= 2 * d + 2 ** -7 * scale, (b, i, top2, d)
                break                                  # the sequences diverged on a tie: later steps see other tokens
    same = (ids == ref_ids).float().mean().item()
    print(f"hidden {hidden} heads {heads}x{hd} layers {layers} batch {batch} prompt {prompt}: logits max_abs {worst:.3e} "
          f"(largest logit {scale:.2f}); {same * 100:.0f}% of greedy tokens equal; launches {dec.last_launch_count}")
    # sequences that hit a top-2 near-tie (checked above) legitimately continue with other tokens, so the share of equal
    # tokens is reported, not bounded; the first token of most sequences must agree
    assert (ids[:, 0] == ref_ids[:, 0]).float().mean().item() >= 0.5
    dec.close()


def test_embed_and_prompt_assembly():
    cfg = openvla.LlamaShapedConfig(num_layers=1, hidden=256, num_heads=2, num_kv_heads=2, head_dim=128, intermediate=512,
                                    vocab=300, max_positions=64)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV)
    ids = torch.tensor([[1, 7, 299, 0]], device=DEV)
    rows = dec.embed(ids)
    assert torch.equal(rows, sd["model.embed_tokens.weight"][ids])
    patches = torch.randn((1, 5, 256), device=DEV).to(torch.bfloat16)
    x = openvla.build_prompt_embeds(dec, ids, patches)
    assert x.shape == (1, 9, 256) and torch.equal(x[:, 1:6], patches) and torch.equal(x[:, 0], rows[:, 0])
    out = dec.generate(x, 7)
    dec.check()
    assert out.shape == (1, 7) and int(out.min()) >= 0 and int(out.max()) < 300
    with pytest.raises(Exception):
        dec.generate(torch.zeros((1, 60, 256), device=DEV, dtype=torch.bfloat16), 7)      # 67 > max_positions
    dec.close()


def test_missing_weight_is_an_error():
    cfg = openvla.LlamaShapedConfig(num_layers=1, hidden=256, num_heads=2, num_kv_heads=2, head_dim=128, intermediate=512,
                                    vocab=300, max_positions=64)
    sd = openvla.synthetic_llama_state_dict(cfg, DEV, 0)
    del sd["model.layers.0.mlp.up_proj.weight"]
    with pytest.raises(Exception, match="missing"):
        openvla.LlamaDecoder.from_state_dict(cfg, sd, DEV)
