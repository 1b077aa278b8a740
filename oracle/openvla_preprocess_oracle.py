"""CPU restatement of OpenVLA's image preprocessing: the `PrismaticImageProcessor` step that turns a uint8 camera
frame into the fused backbone's 6-channel `pixel_values`.  TEST INFRASTRUCTURE ONLY: imported by tests/ and
tools/, never by the product path.

OpenVLA's remote code is not vendored here, so parity is pinned to the libraries that processor calls:
  * resize      — `TVF.resize(pil_image, size, BICUBIC)` = Pillow `Image.resize((w, h), Image.BICUBIC)` with
                  `reducing_gap=None`.  Pillow's algorithm (libImaging/Resample.c): `precompute_coeffs` in double
                  with the bicubic filter (a = -0.5, support 2), window clipped at the borders and renormalised,
                  `normalize_coeffs_8bpc` to int32 with PRECISION_BITS = 22, then a horizontal pass and a vertical
                  pass, each run only when its dimension changes, each rounding to uint8.  Pillow does not expose
                  its tables; this module restates them so that the library's C++ table builder has something to
                  be compared with (tests/test_openvla_preprocess.py also pins this module against Pillow itself).
  * output size — torchvision `_compute_resized_output_size`: an int `size` becomes the shorter side and the
                  longer side is `int(size * long / short)`; an `(h, w)` tuple is taken as is ("resize-naive").
  * center crop — `TVF.center_crop`: offsets `int(round((H - crop) / 2.0))` (Python's round-half-to-even).
  * normalise   — `TVF.to_tensor` (fp32 `v / 255`) then `TVF.normalize` (`(x - mean) / std` in fp32), per tower;
                  the towers are stacked channel-wise (DINOv2 first) and cast to bf16.
"""

from __future__ import annotations

import math
from typing import Sequence, Tuple, Union

import numpy as np
import torch

PRECISION_BITS = 22
DINOV2_MEAN, DINOV2_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
SIGLIP_MEAN, SIGLIP_STD = (0.5, 0.5, 0.5), (0.5, 0.5, 0.5)


def bicubic_filter(x: float) -> float:
    """Resample.c `bicubic_filter` with a = -0.5."""
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def coefficients(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray]:
    """Resample.c `precompute_coeffs` + `normalize_coeffs_8bpc` for one axis: bounds int32 [out, 2] = (xmin, count)
    and weights int32 [out, ksize] (zero past `count`)."""
    scale = float(in_size) / out_size
    filterscale = max(scale, 1.0)
    support = 2.0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), np.int32)
    weights = np.zeros((out_size, ksize), np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        k = [bicubic_filter((x + xmin - center + 0.5) * ss) for x in range(xmax)]
        ww = 0.0
        for w in k:
            ww += w
        if ww != 0.0:
            k = [w / ww for w in k]
        for x, w in enumerate(k):
            weights[xx, x] = int(-0.5 + w * (1 << PRECISION_BITS)) if w < 0 else int(0.5 + w * (1 << PRECISION_BITS))
        bounds[xx] = (xmin, xmax)
    return bounds, weights


def _pass(x: np.ndarray, bounds: np.ndarray, weights: np.ndarray, axis: int) -> np.ndarray:
    """One integer pass along `axis` of an int64 HWC array: sum of taps from 1 << 21, >> 22, clipped to uint8."""
    n = x.shape[axis]
    idx = np.minimum(bounds[:, :1] + np.arange(weights.shape[1])[None], n - 1)      # taps past `count` weigh 0
    taps = np.take(x, idx, axis=axis)                                                # axis -> (out, ksize)
    w = weights.astype(np.int64)
    acc = np.einsum("okwc,ok->owc", taps, w) if axis == 0 else np.einsum("hokc,ok->hoc", taps, w)
    return np.clip((acc + (1 << (PRECISION_BITS - 1))) >> PRECISION_BITS, 0, 255)


def resize_bicubic_u8(img: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """uint8 [H][W][3] -> uint8 [out_h][out_w][3], bit-exact `Image.resize((out_w, out_h), Image.BICUBIC)`."""
    assert img.dtype == np.uint8 and img.ndim == 3
    h, w, _ = img.shape
    x = img.astype(np.int64)
    if out_w != w:
        x = _pass(x, *coefficients(w, out_w), axis=1)
    if out_h != h:
        x = _pass(x, *coefficients(h, out_h), axis=0)
    return x.astype(np.uint8)


def resize_geometry(h: int, w: int, size: Union[int, Sequence[int]] = 224,
                    crop: Union[int, Sequence[int]] = 224) -> Tuple[int, int, int, int]:
    """torchvision's output-size and center-crop rules: (resize_h, resize_w, crop_top, crop_left)."""
    if isinstance(size, int):
        short, long = (w, h) if w <= h else (h, w)
        new_short, new_long = size, int(size * long / short)
        rw, rh = (new_short, new_long) if w <= h else (new_long, new_short)
    else:
        rh, rw = int(size[0]), int(size[1])
    ch, cw = (crop, crop) if isinstance(crop, int) else (int(crop[0]), int(crop[1]))
    return rh, rw, int(round((rh - ch) / 2.0)), int(round((rw - cw) / 2.0))


def preprocess(frame: np.ndarray, size=224, crop=224, means=(DINOV2_MEAN, SIGLIP_MEAN),
               stds=(DINOV2_STD, SIGLIP_STD)) -> Tuple[torch.Tensor, np.ndarray]:
    """uint8 HWC frame -> (bf16 pixel_values [3 * len(means), crop_h, crop_w], the cropped uint8 resize)."""
    rh, rw, top, left = resize_geometry(frame.shape[0], frame.shape[1], size, crop)
    ch, cw = (crop, crop) if isinstance(crop, int) else crop
    small = resize_bicubic_u8(frame, rh, rw)[top:top + ch, left:left + cw]
    x = torch.from_numpy(np.ascontiguousarray(small)).permute(2, 0, 1).float() / 255
    outs = []
    for m, s in zip(means, stds):
        mean = torch.tensor(m, dtype=torch.float32)[:, None, None]
        std = torch.tensor(s, dtype=torch.float32)[:, None, None]
        outs.append((x - mean) / std)
    return torch.cat(outs).to(torch.bfloat16), small
