"""Host-side restatement of FiLM, OpenVLA-OFT's language conditioning of the vision towers (the paper's "OFT+" form).
The rest of OFT is restated in `oracle/openvla_oft_oracle.py` and `oracle/openvla_oft_cameras_oracle.py`.  OFT's own
code (`modeling_prismatic.py` and its FiLM wrappers in the OFT repository) is neither vendored nor downloadable, so this
file is the specification the engine is tested against; parity with the released checkpoints' code is unpinned.

- Language vector.  OFT embeds its whole input ids (prompt, action placeholders, stop token) and drops the positions its
  action mask marks: `language_embeddings = input_embeddings[~all_actions_mask].reshape(B, -1, D)`, then
  `language_embeddings.mean(dim=1)` in bf16 (fp32 sum, one rounding).  The mask is taken to cover the action
  placeholders only, as OFT's action mask is publicly described, so the averaged rows are BOS, the instruction, the
  29871 empty token and the stop token.  A batch of prompts of different lengths is averaged per sequence: pads are
  never averaged.
- Per block and tower: `gamma = scale(avg)`, `beta = shift(avg)`, each `nn.Linear(llm_dim -> vision_dim)` with bias.
- Inside each block that runs (OpenVLA reads the second-to-last block, so the first `depth - 1`):
    x = x + LS1(attn(LN1(x)))        (DINOv2 has LayerScale, SigLIP does not)
    x = x * (1 + gamma) + beta       (every row, cls and register tokens included; bf16 as torch runs it)
    x = x + LS2(MLP(LN2(x)))
  Both towers are conditioned.  With n cameras, the images of sequence b (rows b·n .. b·n + n - 1 of the towers'
  batch) all use sequence b's gamma and beta.
"""

from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
from torch import nn

from oracle.openvla_oft_oracle import STOP_TOKEN

ACTION_PLACEHOLDER = 31743          # any id: the placeholders' embeddings are never averaged


class FiLM(nn.Module):
    """One block's FiLM pair, OFT's `scale` / `shift` naming."""

    def __init__(self, llm_dim: int, vision_dim: int):
        super().__init__()
        self.scale = nn.Linear(llm_dim, vision_dim)
        self.shift = nn.Linear(llm_dim, vision_dim)


def film_modules(n_blocks: int, llm_dim: int, vision_dim: int) -> nn.ModuleList:
    return nn.ModuleList(FiLM(llm_dim, vision_dim) for _ in range(n_blocks))


def oft_input_ids(prompt_ids: Sequence[int], n_slots: int, stop: int = STOP_TOKEN) -> Tuple[List[int], List[bool]]:
    """OFT's input ids after the prompt (29871 already appended) and its action mask: prompt, `n_slots` placeholders,
    stop.  The mask marks the placeholders only."""
    ids = list(prompt_ids) + [ACTION_PLACEHOLDER] * n_slots + [stop]
    mask = [False] * len(prompt_ids) + [True] * n_slots + [False]
    return ids, mask


def language_rows(prompt_ids: Sequence[int], n_slots: int, stop: int = STOP_TOKEN) -> List[int]:
    """The ids whose embeddings are averaged: OFT's input ids where the action mask is False."""
    ids, mask = oft_input_ids(prompt_ids, n_slots, stop)
    return [i for i, m in zip(ids, mask) if not m]


def language_embedding(input_embeddings: torch.Tensor, action_mask: torch.Tensor) -> torch.Tensor:
    """`input_embeddings[~mask].reshape(B, -1, D).mean(dim=1)`: [B, L, D] and a bool mask [B, L] with the same count of
    unmasked rows per sequence -> [B, D]."""
    B, _, D = input_embeddings.shape
    return input_embeddings[~action_mask].reshape(B, -1, D).mean(dim=1)


def _is_siglip(layer: nn.Module) -> bool:
    return hasattr(layer, "self_attn")


def film_block(layer: nn.Module, x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor) -> torch.Tensor:
    """One FiLMed block over transformers' own submodules: a `Dinov2WithRegistersLayer` or a `SiglipEncoderLayer`.
    x [N, T, H]; gamma / beta [N, H] (one row per image)."""
    if _is_siglip(layer):
        h, _ = layer.self_attn(hidden_states=layer.layer_norm1(x), attention_mask=None)
        x = x + h
    else:
        x = layer.layer_scale1(layer.attention(layer.norm1(x))) + x
    x = x * (1 + gamma[:, None]) + beta[:, None]
    if _is_siglip(layer):
        return x + layer.mlp(layer.layer_norm2(x))
    return layer.layer_scale2(layer.mlp(layer.norm2(x))) + x


def film_tower(model: nn.Module, pixel_values: torch.Tensor, films: nn.ModuleList, language: torch.Tensor,
               images_per_cond: int = 1) -> torch.Tensor:
    """Patch-token features of the second-to-last block of a transformers `Dinov2WithRegistersModel` or
    `SiglipVisionModel`, every block FiLMed.  pixel_values [N, 3, 224, 224] with N = B * images_per_cond; language
    [B, llm_dim]; films: one `FiLM` per block that runs (depth - 1)."""
    if hasattr(model, "vision_model"):
        x = model.vision_model.embeddings(pixel_values)
        layers, prefix = model.vision_model.encoder.layers, 0
    else:
        x = model.embeddings(pixel_values)
        layers, prefix = model.encoder.layer, 1 + model.config.num_register_tokens
    assert len(films) == len(layers) - 1
    for layer, f in zip(layers, films):
        gamma = f.scale(language).repeat_interleave(images_per_cond, dim=0)
        beta = f.shift(language).repeat_interleave(images_per_cond, dim=0)
        x = film_block(layer, x, gamma, beta)
    return x[:, prefix:]
