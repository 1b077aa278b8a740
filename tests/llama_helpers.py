"""Shared scaffolding of the Llama-shaped decoder tests: the transformers reference model and its greedy decode,
synthetic decoders at the shapes the engine switches on, prompt instructions, and a shrunk OpenVLA policy."""

from __future__ import annotations

import numpy as np
import torch

from blurr_b200 import openvla

DEV = "cuda"


def hf_llama(cfg: openvla.LlamaShapedConfig, seed: int, qk_scale: float = 1.0, head_scale: float = 1.0):
    """transformers' `LlamaForCausalLM` (eager attention) of `cfg`'s shape, bf16 on the device, from `torch.manual_seed(seed)`.
    The norms are redrawn away from their init of 1; q/k projections are scaled by `qk_scale` (peaked attention: RoPE and
    the mask matter) and embed_tokens / lm_head by `head_scale` (logits spread over a few units)."""
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
            elif "q_proj" in name or "k_proj" in name:
                p.mul_(qk_scale)
            elif "embed_tokens" in name or "lm_head" in name:
                p.mul_(head_scale)
    return model.to(torch.bfloat16).to(DEV)


@torch.inference_mode()
def hf_greedy(model, inputs_embeds, n_new):
    """transformers' greedy decode with a KV cache: ids [B, n_new] and the logits each was chosen from [B, n_new, vocab]."""
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


SHAPES = {
    # hidden, heads, head_dim, inter, layers, vocab, batch, T_max
    "few": (256, 2, 128, 512, 2, 1000, 4, 8),
    "mid": (512, 4, 128, 1408, 2, 1064, 3, 37),
    "b32": (1280, 10, 128, 2560, 2, 1000, 32, 12),
    "b32-fused": (512, 8, 64, 1024, 1, 300, 32, 6),
}


def synthetic_decoder(name, n_new=7):
    """A decoder of shape SHAPES[name] on synthetic weights (peaked attention, spread logits) with room for `n_new`
    tokens, and bf16 prompt embeddings [batch, T_max, hidden]."""
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


def instructions(lengths, seed):
    """One random instruction of each length: BOS, then token ids in 3..31999."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for n in lengths:
        r = torch.randint(3, 32000, (n,), generator=g)
        r[0] = 1
        rows.append(r)
    return rows


Q01 = np.array([-0.03, -0.04, -0.02, -0.1, -0.1, -0.2, 0.0])
Q99 = np.array([0.03, 0.04, 0.03, 0.1, 0.1, 0.2, 1.0])


def small_policy():
    """Yields (policy, pixels [4, 6, 224, 224]): shrunk towers (depth 3) and a 2-layer 4096-wide decoder; closes them after."""
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
