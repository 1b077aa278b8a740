"""Host-side restatement of OpenVLA-OFT's `predict_action` (Kim, Finn, Liang 2025, "Fine-Tuning VLAs: Optimizing Speed
and Success"): parallel decoding of an action chunk with an L1-regression head.  OFT's own code (`modeling_prismatic.py`
of the OFT repository, `action_heads.py`) is neither vendored nor downloadable, so this file is the specification the
engine is tested against; parity with the released checkpoints' code is unpinned.

What OFT's `predict_action` computes, restated:

- Prompt ids.  If the last prompt id is not 29871 (the empty token after "Out:"), append 29871.  Call the resulting
  length `S` (it includes BOS).  Then append `K·D` placeholder ids and the stop id 2.  Placeholder embeddings are
  zeroed; the stop token keeps its embedding.
- Multimodal sequence.  `[BOS] + P patch embeddings + ids[1:S] + K·D zero rows + embed(2)`, so
  `len = P + S + K·D + 1`.  The first action slot is at position `a0 = P + S`.
- Attention rule.  A query at position `p` sees key `k` iff `k ≤ p`, or `p ≥ a0` and `a0 ≤ k < len`.  This is causal
  over the prompt and bidirectional inside the action block plus the stop token.  Pads beyond `len` are never seen.
  Setting `a0 = len` gives plain causal attention through the same rule.
- Hidden rows.  Take `LlamaModel.last_hidden_state`, which is after the final RMSNorm: what transformers 4.x's
  `hidden_states[-1]` returned for OFT.  Use rows `[a0 - 1, a0 - 1 + K·D)`: the row before each action slot, as in
  training, where hidden `t` pairs with label `t + 1`.
- Head (`L1RegressionActionHead` -> `MLPResNet(num_blocks=2, input_dim=D·H, hidden_dim=H, output_dim=D)`).  Reshape the
  rows `[B, K·D, H]` to `[B·K, D·H]`; this is a view, with no copy.  Then:
    `LayerNorm(D·H)` -> `Linear(D·H->H)` -> ReLU;
    2 x `x + ReLU(Linear(H->H)(LayerNorm(H)(x)))`;
    `LayerNorm(H)` -> `Linear(H->D)`.
  Everything is in bf16 as torch runs it: LayerNorm in fp32 internally with bf16 out (eps 1e-5), Linear as
  bf16(acc + bias), ReLU and the residual add in bf16.  The output is `[B, K, D]`.
- De-normalisation.  `ActionDetokenizer`'s q01 / q99 / mask formula (`0.5·(a+1)·(q99−q01)+q01` where mask), applied
  to every step of the chunk.
"""

from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import torch
from torch import nn

EMPTY_TOKEN = 29871
STOP_TOKEN = 2


def prompt_layout(prompt: Sequence[int], n_patches: int, chunk: int = 8, action_dim: int = 7) -> Tuple[List[int], int, int, int]:
    """One prompt (ids starting with BOS) -> (text ids with 29871 appended if missing, a0, len, row_start)."""
    ids = [int(t) for t in prompt]
    if ids[-1] != EMPTY_TOKEN:
        ids.append(EMPTY_TOKEN)
    a0 = n_patches + len(ids)
    return ids, a0, a0 + chunk * action_dim + 1, a0 - 1


def allowed(seq_len: int, a0: int, max_len: int) -> torch.Tensor:
    """bool [max_len, max_len]: query p sees key k iff k < seq_len and (k <= p, or p >= a0 and a0 <= k)."""
    p = torch.arange(max_len)[:, None]
    k = torch.arange(max_len)[None, :]
    return (k < seq_len) & ((k <= p) | ((p >= a0) & (k >= a0)))


def additive_mask(seq_len: int, a0: int, max_len: int = None, dtype=torch.bfloat16) -> torch.Tensor:
    """The rule as the 4-D additive mask [1, 1, L, L] that transformers' `LlamaModel(attn_implementation="eager")`
    takes as-is: 0 where allowed, finfo(dtype).min elsewhere."""
    L = seq_len if max_len is None else max_len
    m = torch.full((L, L), torch.finfo(dtype).min, dtype=dtype)
    m[allowed(seq_len, a0, L)] = 0
    return m[None, None]


@torch.inference_mode()
def llama_action_rows(model, embeds: torch.Tensor, a0: int, n_rows: int) -> torch.Tensor:
    """`LlamaModel(inputs_embeds=embeds [1, len, H], attention_mask=the rule).last_hidden_state` rows a0 - 1 .. + n_rows."""
    L = embeds.shape[1]
    mask = additive_mask(L, a0, L, embeds.dtype).to(embeds.device)
    out = model(inputs_embeds=embeds, attention_mask=mask, use_cache=False)
    return out.last_hidden_state[:, a0 - 1:a0 - 1 + n_rows]


class MLPResNetBlock(nn.Module):
    """OFT's `MLPResNetBlock`: x + ReLU(Linear(LayerNorm(x)))."""

    def __init__(self, dim: int):
        super().__init__()
        self.dim = dim
        self.ffn = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, dim), nn.ReLU())

    def forward(self, x):
        return x + self.ffn(x)


class MLPResNet(nn.Module):
    """OFT's `MLPResNet`."""

    def __init__(self, num_blocks: int, input_dim: int, hidden_dim: int, output_dim: int):
        super().__init__()
        self.layer_norm1 = nn.LayerNorm(input_dim)
        self.fc1 = nn.Linear(input_dim, hidden_dim)
        self.relu = nn.ReLU()
        self.mlp_resnet_blocks = nn.ModuleList([MLPResNetBlock(hidden_dim) for _ in range(num_blocks)])
        self.layer_norm2 = nn.LayerNorm(hidden_dim)
        self.fc2 = nn.Linear(hidden_dim, output_dim)

    def forward(self, x):
        x = self.relu(self.fc1(self.layer_norm1(x)))
        for block in self.mlp_resnet_blocks:
            x = block(x)
        return self.fc2(self.layer_norm2(x))


class L1RegressionActionHead(nn.Module):
    """OFT's `L1RegressionActionHead`: rows [B, K·D, H] -> actions [B, K, D]."""

    def __init__(self, input_dim: int = 4096, hidden_dim: int = 4096, action_dim: int = 7, chunk: int = 8, num_blocks: int = 2):
        super().__init__()
        self.action_dim, self.chunk = action_dim, chunk
        self.model = MLPResNet(num_blocks=num_blocks, input_dim=input_dim * action_dim, hidden_dim=hidden_dim, output_dim=action_dim)

    def predict_action(self, actions_hidden_states: torch.Tensor) -> torch.Tensor:
        B = actions_hidden_states.shape[0]
        return self.model(actions_hidden_states.reshape(B, self.chunk, -1))


def denormalize_chunk(norm: np.ndarray, q01, q99, mask=None) -> np.ndarray:
    """norm [B, K, D] -> actions [B, K, D] in float64; q01 / q99 / mask are [D] or [B, D] and apply to every step."""
    norm = np.asarray(norm, dtype=np.float64)
    q01, q99 = np.asarray(q01, dtype=np.float64), np.asarray(q99, dtype=np.float64)
    mask = np.ones(q01.shape, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    if q01.ndim == 2:
        q01, q99 = q01[:, None], q99[:, None]
    if mask.ndim == 2:
        mask = mask[:, None]
    return np.where(mask, 0.5 * (norm + 1) * (q99 - q01) + q01, norm)
