"""Host restatement of the sampled decoding of `blurr_llm_generate_sampled` / `blurr_llm_sample` (test-only).

HF semantics (transformers 5.5 `generation/utils.py` `_sample`, `generation/logits_process.py`): the last logits row is
cast to fp32, then `TemperatureLogitsWarper` (T != 1), `TopKLogitsWarper` (k != 0), `TopPLogitsWarper` (p < 1) with
min_tokens_to_keep = 1, softmax, one draw.  The rules restated here:
  * temperature: `scores / T` on CUDA is a multiplication by the fp32 reciprocal `1.0f / (float)T`;
  * top-k: keep every score >= the k-th largest (repeats counted); k >= vocab keeps all;
  * top-p (on the top-k survivors): a token is kept iff the mass strictly ahead of it in (score, index) descending order
    is < p * Z, and the first token always (torch's stable ascending sort removes the lower index of equal scores first);
  * draw: u = (x >> 8) * 2^-24 with x word 0 of Philox4x32-10(counter = (step, 0, 0, 0), key = (seed lo, seed hi));
    target = u * Z_kept; the chosen token is the first index whose inclusive prefix mass is > target.
NaN logits are never kept (they count as -inf); a row without a finite positive mass is the kernel's argmax fallback.

The kernel's masses are `expf(fp32(s - s_max))` rounded to fixed point with 2^shift units (shift = 63 - bit_length(vocab)).
CUDA's expf is within 2 ulp (relative 2^-22), so every prefix mass and the target u * Z differ from the float64 values
here by at most 2^-22 * Z each, plus half a unit per summed token.  `draw` flags a draw as "boundary" when the target,
or p * Z at the top-p cut, lies within that bound of a prefix-mass boundary: there the kernel may legitimately choose the
neighbour.
"""

from __future__ import annotations

import numpy as np

PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
EXPF_REL = 2.0 ** -22                 # CUDA expf: maximum error 2 ulp


def philox4x32_10(counter, key) -> np.ndarray:
    """Philox4x32-10 (Salmon et al., SC'11).  counter uint32 [..., 4], key uint32 [..., 2] -> uint32 [..., 4]."""
    c = np.asarray(counter, dtype=np.uint64) & 0xFFFFFFFF
    k = np.asarray(key, dtype=np.uint64) & 0xFFFFFFFF
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    k0, k1 = k[..., 0], k[..., 1]
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * c0
        p1 = np.uint64(PHILOX_M1) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & mask, p1 & mask, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & mask, p0 & mask
        k0, k1 = (k0 + np.uint64(PHILOX_W0)) & mask, (k1 + np.uint64(PHILOX_W1)) & mask
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def uniform24(seeds, step: int) -> np.ndarray:
    """x >> 8 (an int in [0, 2^24)) of every 64-bit seed at `step`: u = that * 2^-24."""
    s = np.atleast_1d(np.asarray(seeds, dtype=np.uint64))
    key = np.stack([s & np.uint64(0xFFFFFFFF), s >> np.uint64(32)], axis=-1)
    ctr = np.zeros(s.shape + (4,), dtype=np.uint64)
    ctr[..., 0] = step
    return (philox4x32_10(ctr, key)[..., 0] >> np.uint32(8)).astype(np.int64)


def scaled_scores(logits, temperature: float) -> np.ndarray:
    """fp32 scores * fp32(1 / fp32(T)), NaN -> -inf."""
    x = np.asarray(logits, dtype=np.float32)
    inv = np.float32(1.0) / np.float32(temperature)
    s = (x * inv).astype(np.float32)
    return np.where(np.isnan(s), np.float32(-np.inf), s)


def fixed_point_shift(vocab: int) -> int:
    return 63 - int(vocab).bit_length()


def warp(logits, temperature: float, top_k: int, top_p: float, hf_margin: float = 0.0) -> dict:
    """The kept set of one row after the three warpers, and its probabilities (float64).

    Returns dict(kept bool [V], probs float64 [V] (0 outside the kept set), mass float64 [V] (exp(fp32(s - s_max)) of
    the kept tokens), z (kept mass), ahead float64 [V] (mass ahead in the top-p order, NaN off the top-k set),
    z_topk, ambiguous bool [V] (top-p: |ahead - p Z| <= hf_margin * Z, or a member of a group of equal scores the cut
    splits: HF may keep either way), finite (False:
    no finite positive mass, the argmax fallback))."""
    s = scaled_scores(logits, temperature)
    V = s.shape[0]
    idx = np.arange(V)
    m = s.max()
    out = dict(kept=np.zeros(V, bool), probs=np.zeros(V), mass=np.zeros(V), z=0.0, ahead=np.full(V, np.nan), z_topk=0.0,
               ambiguous=np.zeros(V, bool), finite=bool(np.isfinite(m)))
    if not out["finite"]:
        return out
    keep = np.ones(V, bool)
    if 0 < top_k < V:
        thr = np.sort(s)[::-1][top_k - 1]
        keep = s >= thr
    e = np.exp((s - m).astype(np.float32).astype(np.float64))
    e = np.where(keep, e, 0.0)
    z = e.sum()
    out["z_topk"] = z
    if top_p < 1.0:
        cand = idx[keep]
        order = cand[np.lexsort((-cand, -s[cand].astype(np.float64)))]      # score descending, index descending
        ahead = np.concatenate([[0.0], np.cumsum(e[order])[:-1]])
        pz = float(np.float64(np.float32(top_p)) * z)
        kp = ahead < pz
        kp[0] = True
        out["ahead"][order] = ahead
        out["ambiguous"][order] = np.abs(ahead - pz) <= hf_margin * z
        out["ambiguous"][order[0]] = False
        keep2 = np.zeros(V, bool)
        keep2[order[kp]] = True
        # TopPLogitsWarper sorts with torch.sort(stable=False): which members of a group of equal scores that straddles
        # the cut it keeps is unspecified (the kernel keeps the higher indices, as a stable sort would)
        for v in np.unique(s[cand]):
            grp = cand[s[cand] == v]
            if keep2[grp].any() and not keep2[grp].all():
                out["ambiguous"][grp] = True
        keep = keep2
        e = np.where(keep, e, 0.0)
    out["kept"] = keep
    out["mass"] = e
    out["z"] = e.sum()
    out["probs"] = e / out["z"]
    return out


def draw(logits, temperature: float, top_k: int, top_p: float, seed: int, step: int, vocab=None):
    """(token id, boundary flag) of one row; the argmax fallback (flag False) for a row without finite positive mass."""
    x = np.asarray(logits, dtype=np.float32)
    w = warp(x, temperature, top_k, top_p)
    if not w["finite"]:
        v = np.where(np.isnan(x), -np.inf, x)
        return int(np.argmax(v)) if not np.all(np.isnan(x)) else 0, False
    V = x.shape[0] if vocab is None else vocab
    z = w["z"]
    n_kept = int(w["kept"].sum())
    eps = 2.0 * EXPF_REL * w["z_topk"] + (n_kept + 2) * 2.0 ** -fixed_point_shift(V)
    u = uniform24([seed], step)[0] * 2.0 ** -24
    target = u * z
    prefix = np.cumsum(w["mass"])
    i = int(np.searchsorted(prefix, target, side="right"))
    i = min(i, x.shape[0] - 1)
    lo = prefix[i - 1] if i > 0 else 0.0
    boundary = (target - lo) <= eps or (prefix[i] - target) <= eps
    # a zero-mass token right after the chosen boundary cannot be chosen; tokens of mass < eps around it can
    if top_p < 1.0:
        pz = float(np.float64(np.float32(top_p)) * w["z_topk"])
        a = w["ahead"]
        a = a[~np.isnan(a) & (a > 0)]                   # the first token (nothing ahead) is kept exactly
        near = np.abs(a - pz) <= eps
        boundary = boundary or bool(near.any())
    return i, bool(boundary)
