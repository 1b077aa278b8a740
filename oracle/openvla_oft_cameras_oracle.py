"""Host-side restatement of what OpenVLA-OFT's LIBERO checkpoints add to `predict_action`: a wrist camera and the robot
state (proprioception).  The rest of OFT (prompt layout, attention rule, head, de-normalisation) is restated in
`oracle/openvla_oft_oracle.py`.  OFT's own code (`modeling_prismatic.py`, `projectors.py` of the OFT repository) is
neither vendored nor downloadable, so this file is the specification the engine is tested against; parity with the
released checkpoints' code is unpinned.

- Cameras.  The pixel values stack the cameras along channels, 6 per camera (DINOv2's 3 first), third-person image
  first.  Each image goes through the towers and the projector on its own; the patch rows are concatenated in camera
  order (`torch.cat(all_patches, dim=1)`), so image i's 256 patches sit at rows `256·i …` after BOS.
- Proprioception.  The raw state is normalised with the dataset's BOUNDS_Q99 statistics,
  `clip(where(mask, 2·(x − q01)/(q99 − q01 + 1e-8) − 1, x), −1, 1)`, taken to the model as `torch.Tensor(x)` (fp32)
  then bf16, and projected by `ProprioProjector`: `fc1 (D_p -> H)` -> exact GELU -> `fc2 (H -> H)`.  The one projected
  row is appended after all patch rows, so `P = 256·n + 1` in `openvla_oft_oracle.prompt_layout`.
"""

from __future__ import annotations

from typing import Sequence

import numpy as np
import torch
from torch import nn


def normalize_proprio(state, q01, q99, mask=None) -> np.ndarray:
    """OFT's BOUNDS_Q99 `normalize_proprio`, in float64."""
    x = np.asarray(state, dtype=np.float64)
    lo, hi = np.asarray(q01, dtype=np.float64), np.asarray(q99, dtype=np.float64)
    mask = np.ones(lo.shape, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    return np.clip(np.where(mask, 2 * (x - lo) / (hi - lo + 1e-8) - 1, x), a_min=-1.0, a_max=1.0)


class ProprioProjector(nn.Module):
    """OFT's `ProprioProjector(llm_dim, proprio_dim)`: fc1 -> GELU (exact) -> fc2."""

    def __init__(self, llm_dim: int = 4096, proprio_dim: int = 8):
        super().__init__()
        self.fc1 = nn.Linear(proprio_dim, llm_dim, bias=True)
        self.fc2 = nn.Linear(llm_dim, llm_dim, bias=True)
        self.act_fn1 = nn.GELU()

    def forward(self, proprio: torch.Tensor) -> torch.Tensor:
        return self.fc2(self.act_fn1(self.fc1(proprio)))


def assemble_patches(image_patches: Sequence[torch.Tensor], proprio_features: torch.Tensor = None) -> torch.Tensor:
    """Projected patches of each camera [B, 256, H] (camera order) and the projected state [B, H] or None -> the rows
    between BOS and the prompt [B, 256·n (+ 1), H]."""
    rows = torch.cat(list(image_patches), dim=1)
    if proprio_features is None:
        return rows
    return torch.cat([rows, proprio_features[:, None].to(rows.dtype)], dim=1)
