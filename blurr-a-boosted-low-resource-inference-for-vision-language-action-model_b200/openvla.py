"""OpenVLA-7B-shaped path (SURVEY.md §8(f) row 3, BASELINE.json configs[4]), from the camera frame to the actions.

The reference has no source for this model — `scripts/benchmark_hf_vla.py:100-109` loads `openvla/openvla-7b` with
`trust_remote_code=True` and times `model.predict_action(**inputs, unnorm_key=..., do_sample=False)` (:141-197).
That call (public Prismatic/OpenVLA architecture) runs the fused SigLIP+DINOv2 backbone and the MLP projector, builds
`[BOS] + 256 patch embeddings + prompt tokens`, and lets a `LlamaForCausalLM` generate `action_dim` = 7 tokens greedily
with a KV cache; each token is mapped to one of 256 uniform bins on [-1, 1] and de-normalised with q01/q99.

Built here, all on the device:
  * `ImagePreprocessor` — the processor's bicubic resize, center crop and the two per-tower normalisations
    (csrc/preprocess.cu behind include/blurr_vit.h), bit-exact against Pillow + torchvision;
  * `VitEncoder` x 2 + `MlpProjector` = `FusedVisionBackbone` — DINOv2 and SigLIP towers and the projector
    (csrc/vit_engine.cu behind include/blurr_vit.h);
  * `LlamaDecoder` — the Llama-2-7B-shaped decoder (csrc/llm_engine.cu behind include/blurr_llm.h): prefill of the
    multimodal prompt embeddings + greedy decode, or sampled decode (`do_sample=True` with HF's `temperature`, `top_k`,
    `top_p`; defaults 1.0 / 50 / 1.0 as in `generate`) drawn on the device inside the same CUDA graph, Philox-seeded
    per row so that a row's tokens depend only on its seed;
  * `ActionDetokenizer` (host) and `OpenVlaPolicy`, which chains them: `predict_action(frames, input_ids, q01, q99)`.
A batch may carry instructions of different lengths (`input_ids` as a list, or `[B, S]` with a tokenizer's
`attention_mask`): `ragged_prompt_ids` packs them, `build_prompt_embeds_ragged` lays out `[BOS] + patches + text_b` with
pad rows behind it, and `LlamaDecoder.generate(..., prompt_lens=...)` generates every sequence at its own positions, so
each row gets what it would get alone.
`predict_action(..., do_sample=True, temperature=, top_k=, top_p=, seed=)` samples the action tokens for every prompt
form.  Not built: tokenisation of the instruction (the caller passes `input_ids`).  PARITY: the towers are pinned against
transformers (tests/test_gpu_vit.py), the decoder against `LlamaForCausalLM` with eager attention
(tests/test_gpu_llm.py), the preprocessing against Pillow + torchvision (tests/test_openvla_preprocess.py); against
the reference's remote code all of it is UNPINNED (not vendored, not downloadable)."""

from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import capi


@dataclass
class LlamaShapedConfig:
    num_layers: int = 32
    hidden: int = 4096
    num_heads: int = 32
    num_kv_heads: int = 32
    head_dim: int = 128
    intermediate: int = 11008
    vocab: int = 32064            # Llama-2's 32000 padded to a multiple of 64 (OpenVLA adds <PAD>)
    max_positions: int = 320      # 1 + 256 patches + prompt + 7 action tokens fits
    rms_eps: float = 1e-6
    rope_theta: float = 10000.0
    long_forward: int = 0         # max_positions: 0 up to 384, 1 up to 1024 (True means 1), 2 in 1025..2048, for
                                  # forward_rows; generate stops at 320 on every handle


def openvla_7b_config() -> LlamaShapedConfig:
    return LlamaShapedConfig()


def rope_tables(inv_freq: torch.Tensor, n_pos: int, dtype: torch.dtype = torch.bfloat16) -> Tuple[torch.Tensor, torch.Tensor]:
    """cos / sin of `LlamaRotaryEmbedding.forward` (modeling_llama.py) for positions 0..n_pos-1, first half of the head
    dim: fp32 angle `inv_freq.float() * position`, cos/sin cast to the activation dtype.  `inv_freq` is the module's own
    buffer (a model cast with `.to(bfloat16)` carries a bf16-rounded one)."""
    pos = torch.arange(n_pos, device=inv_freq.device, dtype=torch.float32)
    freqs = pos[:, None] * inv_freq.float()[None, :]
    return freqs.cos().to(dtype).float().contiguous(), freqs.sin().to(dtype).float().contiguous()


def default_inv_freq(head_dim: int, theta: float, device) -> torch.Tensor:
    """`ROPE_INIT_FUNCTIONS['default']`: 1 / theta^(2i / d), computed in fp32 on int64 indices."""
    return 1.0 / (theta ** (torch.arange(0, head_dim, 2, dtype=torch.int64, device=device).float() / head_dim))


def _per_row(value, rows: int, name: str) -> list:
    if isinstance(value, torch.Tensor):
        value = value.detach().cpu().tolist()
    elif isinstance(value, np.ndarray):
        value = value.tolist()
    if isinstance(value, (list, tuple)):
        if len(value) != rows:
            raise ValueError(f"{name} must be a scalar or hold one value per row ({rows}), got {len(value)}")
        return list(value)
    return [value] * rows


def sampling_params(rows: int, temperature=1.0, top_k=50, top_p=1.0, seed=None) -> "C.Array":
    """`blurr_llm_sampling[rows]` for `rows` sequences; each argument is a scalar or one value per row.  Checks HF's
    rules (temperature finite and > 0, top_k an int >= 0, top_p in [0, 1]) and raises ValueError.  `seed`: None draws
    one 63-bit seed per row from torch's default CPU generator (so `torch.manual_seed` makes a run repeatable); an int
    `s` gives row b the seed s + b; a sequence gives each row its own seed (ints in [0, 2^64))."""
    temps = [float(t) for t in _per_row(temperature, rows, "temperature")]
    ks = _per_row(top_k, rows, "top_k")
    ps = [float(p) for p in _per_row(top_p, rows, "top_p")]
    if seed is None:
        seeds = torch.randint(0, 2 ** 63 - 1, (rows,), dtype=torch.int64).tolist()
    elif isinstance(seed, (int, np.integer)) and not isinstance(seed, bool):
        seeds = [int(seed) + b for b in range(rows)]
    else:
        seeds = _per_row(seed, rows, "seed")
    for t in temps:
        if not math.isfinite(t) or t <= 0.0:
            raise ValueError(f"temperature must be finite and > 0, got {t}")
    for k in ks:
        if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 0 or k > 2 ** 31 - 1:
            raise ValueError(f"top_k must be an int >= 0, got {k!r}")
    for p in ps:
        if not math.isfinite(p) or p < 0.0 or p > 1.0:
            raise ValueError(f"top_p must be in [0, 1], got {p}")
    for sd in seeds:
        if isinstance(sd, bool) or not isinstance(sd, (int, np.integer)) or not 0 <= int(sd) < 2 ** 64:
            raise ValueError(f"seeds must be ints in [0, 2^64), got {sd!r}")
    arr = (capi.LlmSamplingC * rows)()
    for b in range(rows):
        arr[b] = capi.LlmSamplingC(int(seeds[b]), temps[b], int(ks[b]), ps[b])
    return arr


class LlamaDecoder:
    """Greedy or sampled generation of a Llama-shaped decoder on one B200 through `include/blurr_llm.h`."""

    def __init__(self, cfg: LlamaShapedConfig, device, max_batch: int = 1):
        self.lib = capi.load_library()
        self.cfg = cfg
        self.device = torch.device(device)
        self.max_batch = max_batch
        self.handle = C.c_void_p()
        c = capi.LlmConfigC(capi.LLM_ABI_VERSION, cfg.num_layers, cfg.hidden, cfg.num_heads, cfg.num_kv_heads, cfg.head_dim,
                            cfg.intermediate, cfg.vocab, cfg.max_positions, cfg.rms_eps, int(cfg.long_forward))
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        capi.check(self.lib.blurr_llm_create(C.byref(c), index, max_batch, C.byref(self.handle)))

    @classmethod
    def from_state_dict(cls, cfg: LlamaShapedConfig, state_dict: Dict[str, torch.Tensor], device, max_batch: int = 1,
                        inv_freq: Optional[torch.Tensor] = None, prefix: str = "") -> "LlamaDecoder":
        """`state_dict`: keys of transformers' LlamaForCausalLM (optionally under `prefix`, e.g. "language_model.")."""
        self = cls(cfg, device, max_batch)
        try:
            torch.cuda.current_stream(self.device).synchronize()
            for key, t in state_dict.items():
                if prefix and not key.startswith(prefix):
                    continue
                name = key[len(prefix):]
                if name.endswith("rotary_emb.inv_freq"):
                    continue
                self.set_weight(name, t)
            if inv_freq is None:
                inv_freq = default_inv_freq(cfg.head_dim, cfg.rope_theta, self.device)
            cos, sin = rope_tables(inv_freq.to(self.device), cfg.max_positions)
            torch.cuda.current_stream(self.device).synchronize()
            capi.check(self.lib.blurr_llm_set_rope_table(self.handle, C.c_void_p(cos.data_ptr()), C.c_void_p(sin.data_ptr()),
                                                         cfg.max_positions))
            capi.check(self.lib.blurr_llm_finalize(self.handle))
        except Exception:
            self.close()
            raise
        return self

    def set_weight(self, name: str, tensor: torch.Tensor):
        t = tensor.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        torch.cuda.current_stream(self.device).synchronize()
        shape = (C.c_int64 * t.dim())(*t.shape)
        capi.check(self.lib.blurr_llm_set_weight(self.handle, name.encode(), C.c_void_p(t.data_ptr()), shape, t.dim()))

    def embed(self, ids: torch.Tensor) -> torch.Tensor:
        ids = ids.to(device=self.device, dtype=torch.int64).contiguous()
        out = torch.empty((*ids.shape, self.cfg.hidden), device=self.device, dtype=torch.bfloat16)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        capi.check(self.lib.blurr_llm_embed(self.handle, C.c_void_p(stream), C.c_void_p(ids.data_ptr()), ids.numel(),
                                            C.c_void_p(out.data_ptr())))
        return out

    def generate(self, inputs_embeds: torch.Tensor, n_new: int, return_logits: bool = False, prompt_lens=None,
                 do_sample: bool = False, temperature=1.0, top_k=50, top_p=1.0, seed=None):
        """inputs_embeds: bf16 [B, T, hidden] on the device -> int64 [B, n_new] (and bf16 logits [B, n_new, vocab]).

        `prompt_lens` (B ints, 1..T): prompts of different lengths.  Sequence b's prompt is rows 0 .. prompt_lens[b] - 1
        of `inputs_embeds[b]`; the rows after it are padding and never influence any output.  Its token i is generated
        at position prompt_lens[b] + i, so each sequence gets what it would get alone.  One CUDA graph per
        (B, T, n_new) serves every length vector.  None: every sequence is T rows long.

        `do_sample`: draw every token as HF's `generate(do_sample=True, temperature=, top_k=, top_p=)` does instead of
        taking the argmax (see `sampling_params` for the arguments and seeds).  Token i of row b depends only on the
        row's logits, its seed and i; one CUDA graph serves every seed and parameter vector."""
        if inputs_embeds.dim() != 3 or inputs_embeds.shape[2] != self.cfg.hidden:
            raise ValueError(f"inputs_embeds must be [B, T, {self.cfg.hidden}]")
        if inputs_embeds.dtype != torch.bfloat16 or inputs_embeds.device.type != "cuda":
            raise ValueError("inputs_embeds must be a bf16 CUDA tensor")
        x = inputs_embeds.contiguous()
        B, T = x.shape[0], x.shape[1]
        ids = torch.empty((B, n_new), device=self.device, dtype=torch.int64)
        logits = torch.empty((B, n_new, self.cfg.vocab), device=self.device, dtype=torch.bfloat16) if return_logits else None
        stream = torch.cuda.current_stream(self.device).cuda_stream
        out_logits = C.c_void_p(logits.data_ptr()) if logits is not None else None
        params = sampling_params(B, temperature, top_k, top_p, seed) if do_sample else None
        lens_p = None
        if prompt_lens is not None:
            lens = np.ascontiguousarray(torch.as_tensor(prompt_lens).cpu().numpy(), dtype=np.int32)
            if lens.shape != (B,):
                raise ValueError(f"prompt_lens must hold one length per sequence ({B}), got shape {lens.shape}")
            lens_p = lens.ctypes.data_as(C.POINTER(C.c_int32))
        capi.check(self.lib.blurr_llm_generate(self.handle, C.c_void_p(stream), B, T, C.c_void_p(x.data_ptr()), lens_p, params,
                                               n_new, C.c_void_p(ids.data_ptr()), out_logits))
        return (ids, logits) if return_logits else ids

    def forward_rows(self, inputs_embeds: torch.Tensor, seq_lens, block_starts, row_starts, n_rows: int) -> torch.Tensor:
        """One forward pass without lm_head (OpenVLA-OFT's parallel decoding): inputs_embeds bf16 [B, T, hidden] on the
        device, one int per sequence in `seq_lens` (1..T), `block_starts` (1..seq_lens[b]) and `row_starts` (0..
        seq_lens[b] - n_rows) -> bf16 [B, n_rows, hidden]: rows row_starts[b] .. + n_rows - 1 of sequence b after the
        final RMSNorm.  Query p of sequence b sees key k iff k < seq_lens[b] and (k <= p, or p >= block_starts[b] and
        k >= block_starts[b]); block_starts[b] = seq_lens[b] is plain causal attention.  Rows past seq_lens[b] are pads
        and never influence any output.  One CUDA graph per (B, T) serves every vector of lengths and starts."""
        if inputs_embeds.dim() != 3 or inputs_embeds.shape[2] != self.cfg.hidden:
            raise ValueError(f"inputs_embeds must be [B, T, {self.cfg.hidden}]")
        if inputs_embeds.dtype != torch.bfloat16 or inputs_embeds.device.type != "cuda":
            raise ValueError("inputs_embeds must be a bf16 CUDA tensor")
        x = inputs_embeds.contiguous()
        B, T = x.shape[0], x.shape[1]
        arrs = []
        for name, v in (("seq_lens", seq_lens), ("block_starts", block_starts), ("row_starts", row_starts)):
            a = np.ascontiguousarray(torch.as_tensor(v).cpu().numpy(), dtype=np.int32)
            if a.shape != (B,):
                raise ValueError(f"{name} must hold one value per sequence ({B}), got shape {a.shape}")
            arrs.append(a)
        out = torch.empty((B, int(n_rows), self.cfg.hidden), device=self.device, dtype=torch.bfloat16)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        ptrs = [a.ctypes.data_as(C.POINTER(C.c_int32)) for a in arrs]
        capi.check(self.lib.blurr_llm_forward_rows(self.handle, C.c_void_p(stream), B, T, C.c_void_p(x.data_ptr()), *ptrs, int(n_rows),
                                                   C.c_void_p(out.data_ptr())))
        return out

    def sample(self, logits: torch.Tensor, temperature=1.0, top_k=50, top_p=1.0, seed=None, step: int = 0,
               return_probs: bool = False):
        """The device sampler alone: bf16 logits [rows, ld >= vocab] on the device (rows <= max_batch; the first vocab
        columns are used) -> int64 ids [rows] (and fp32 [rows, vocab]: the probability each token was drawn with, 0
        outside the kept set).  `step` is the Philox counter: `generate` draws its token i with step i."""
        if logits.dim() != 2 or logits.dtype != torch.bfloat16 or logits.device.type != "cuda" or logits.stride(1) != 1:
            raise ValueError("logits must be a bf16 CUDA tensor [rows, ld] with contiguous rows")
        rows = logits.shape[0]
        params = sampling_params(rows, temperature, top_k, top_p, seed)
        ids = torch.empty(rows, device=self.device, dtype=torch.int64)
        probs = torch.empty((rows, self.cfg.vocab), device=self.device, dtype=torch.float32) if return_probs else None
        stream = torch.cuda.current_stream(self.device).cuda_stream
        capi.check(self.lib.blurr_llm_sample(self.handle, C.c_void_p(stream), C.c_void_p(logits.data_ptr()), rows, logits.stride(0),
                                             params, int(step), C.c_void_p(ids.data_ptr()),
                                             C.c_void_p(probs.data_ptr()) if probs is not None else None))
        return (ids, probs) if return_probs else ids

    def check(self):
        capi.check(self.lib.blurr_llm_check(self.handle, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def set_option(self, name: str, value: int):
        capi.check(self.lib.blurr_llm_set_option(self.handle, name.encode(), int(value)))

    def trace_report(self) -> str:
        buf = C.create_string_buffer(1 << 20)
        capi.check(self.lib.blurr_llm_trace_report(self.handle, buf, len(buf)))
        return buf.value.decode()

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.blurr_llm_last_launch_count(self.handle))

    @property
    def weight_bytes_per_token(self) -> int:
        return int(self.lib.blurr_llm_weight_bytes_per_token(self.handle))

    def close(self):
        if self.handle:
            self.lib.blurr_llm_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def denormalize_actions(norm: np.ndarray, q01, q99, mask=None) -> np.ndarray:
    """OpenVLA's de-normalisation: `0.5 * (a + 1) * (q99 - q01) + q01` where `mask`, `a` elsewhere, in float64.  q01 / q99
    / mask broadcast against `norm` from the right.  OFT's BOUNDS statistics (ALOHA) go in as min / max in place of
    q01 / q99.  No `+ 1e-8` is added to the range; whether OFT's own un-normalisation adds one is unpinned."""
    q01, q99 = np.asarray(q01, dtype=np.float64), np.asarray(q99, dtype=np.float64)
    mask = np.ones_like(q01, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    return np.where(mask, 0.5 * (norm + 1) * (q99 - q01) + q01, norm)


def denormalize_chunk(norm: np.ndarray, q01, q99, mask=None) -> np.ndarray:
    """`denormalize_actions` on a chunk: norm [B, K, D] -> float64 [B, K, D]; q01 / q99 / mask are [D] (one dataset) or
    [B, D] (one dataset's statistics per row), the same for every step of the chunk."""
    q01, q99 = np.asarray(q01, dtype=np.float64), np.asarray(q99, dtype=np.float64)
    m = None if mask is None else np.asarray(mask, dtype=bool)
    if q01.ndim == 2:
        q01, q99 = q01[:, None, :], q99[:, None, :]
    if m is not None and m.ndim == 2:
        m = m[:, None, :]
    return denormalize_actions(np.asarray(norm, dtype=np.float64), q01, q99, m)


class ActionDetokenizer:
    """OpenVLA's `predict_action` tail (public modeling_prismatic.py): the last `action_dim` generated ids ->
    `vocab_size - id` -> bin index -> bin centre on [-1, 1] -> de-normalised with the dataset's q01 / q99 where `mask`.
    q01 / q99 / mask are `[action_dim]` (one dataset for the batch) or `[B, action_dim]` (one dataset's statistics per
    row); they broadcast against the `[B, action_dim]` ids."""

    def __init__(self, vocab_size: int = 32000, n_bins: int = 256):
        self.vocab_size = vocab_size
        bins = np.linspace(-1.0, 1.0, n_bins)
        self.bin_centers = (bins[:-1] + bins[1:]) / 2.0

    def normalized(self, token_ids: np.ndarray) -> np.ndarray:
        discretized = self.vocab_size - np.asarray(token_ids, dtype=np.int64)
        discretized = np.clip(discretized - 1, a_min=0, a_max=self.bin_centers.shape[0] - 1)
        return self.bin_centers[discretized]

    def actions(self, token_ids: np.ndarray, q01: np.ndarray, q99: np.ndarray, mask: Optional[np.ndarray] = None) -> np.ndarray:
        return denormalize_actions(self.normalized(token_ids), q01, q99, mask)


def build_prompt_embeds(decoder: LlamaDecoder, input_ids: torch.Tensor, patch_embeds: torch.Tensor) -> torch.Tensor:
    """Prismatic's multimodal prompt: `[BOS] + projected patch embeddings + the remaining prompt tokens`.
    input_ids [B, S] (first column BOS), patch_embeds bf16 [B, P, hidden] -> bf16 [B, 1 + P + S - 1, hidden]."""
    tok = decoder.embed(input_ids)
    return torch.cat([tok[:, :1], patch_embeds.to(tok.dtype), tok[:, 1:]], dim=1).contiguous()


def ragged_prompt_ids(input_ids, attention_mask: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Prompts of different lengths -> (ids int64 [B, S_max], lengths int64 [B]): row b holds its S_b tokens in columns
    0 .. S_b - 1 and pad id 0 after them.  `input_ids` is either a list of 1-D id tensors (each starting with BOS) or
    `[B, S]` with an `attention_mask` whose ones form one contiguous run per row, left- or right-padded (a HF tokenizer's
    padded batch).  Raises ValueError for an empty row or a mask with a gap.  Runs on the host; the ids keep the
    device of the input."""
    if isinstance(input_ids, (list, tuple)):
        if attention_mask is not None:
            raise ValueError("attention_mask goes with a [B, S] input_ids tensor, not with a list")
        if len(input_ids) == 0:
            raise ValueError("input_ids is an empty list")
        rows = [torch.as_tensor(r) for r in input_ids]
        if any(r.dim() != 1 for r in rows):
            raise ValueError("every prompt in the list must be a 1-D id tensor")
        lens = torch.tensor([r.numel() for r in rows], dtype=torch.int64)
        if int(lens.min()) < 1:
            raise ValueError("empty prompt in input_ids")
        ids = torch.zeros((len(rows), int(lens.max())), dtype=torch.int64, device=rows[0].device)
        for b, r in enumerate(rows):
            ids[b, :r.numel()] = r.to(device=ids.device, dtype=torch.int64)
        return ids, lens
    ids = torch.as_tensor(input_ids)
    if ids.dim() != 2:
        raise ValueError("input_ids must be a list of 1-D tensors or a [B, S] tensor")
    if attention_mask is None:
        if ids.shape[1] < 1:
            raise ValueError("empty prompt in input_ids")
        return ids.to(torch.int64), torch.full((ids.shape[0],), ids.shape[1], dtype=torch.int64)
    m = torch.as_tensor(attention_mask).to("cpu")
    if tuple(m.shape) != tuple(ids.shape):
        raise ValueError(f"attention_mask shape {tuple(m.shape)} != input_ids shape {tuple(ids.shape)}")
    if ((m != 0) & (m != 1)).any():
        raise ValueError("attention_mask must hold only 0 and 1")
    m = m.bool()
    lens = m.sum(dim=1).to(torch.int64)
    if int(lens.min()) < 1:
        raise ValueError("empty prompt in input_ids (a row of attention_mask has no ones)")
    first = m.to(torch.int64).argmax(dim=1)
    col = torch.arange(ids.shape[1], dtype=torch.int64)
    run = (col[None] >= first[:, None]) & (col[None] < (first + lens)[:, None])
    if not torch.equal(run, m):
        raise ValueError("every row of attention_mask must be one contiguous run of ones (left or right padding)")
    S = int(lens.max())
    src = (first[:, None] + col[None, :S]).clamp(max=ids.shape[1] - 1)
    keep = col[None, :S] < lens[:, None]
    out = torch.where(keep, ids.to("cpu", torch.int64).gather(1, src), torch.zeros((), dtype=torch.int64))
    return out.to(ids.device), lens


def build_prompt_embeds_ragged(decoder: LlamaDecoder, input_ids: torch.Tensor, text_lens, patch_embeds: torch.Tensor
                               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """`build_prompt_embeds` for prompts of different lengths.  input_ids [B, S_max] with row b's S_b tokens first (as
    `ragged_prompt_ids` returns them, first column BOS), text_lens [B], patch_embeds bf16 [B, P, hidden] ->
    (bf16 [B, 1 + P + S_max - 1, hidden], int64 prompt lengths 1 + P + (S_b - 1) [B] on the host).  Row b is
    `[BOS] + patches + text_b`, followed by pad rows, the layout `LlamaDecoder.generate(..., prompt_lens=...)` takes."""
    lens = torch.as_tensor(text_lens, dtype=torch.int64).cpu()
    if lens.shape != (input_ids.shape[0],) or int(lens.min()) < 1 or int(lens.max()) > input_ids.shape[1]:
        raise ValueError("text_lens must hold one length in 1..S_max per row of input_ids")
    return build_prompt_embeds(decoder, input_ids, patch_embeds), lens + patch_embeds.shape[1]


def synthetic_llama_state_dict(cfg: LlamaShapedConfig, device, seed: int = 0, dtype=torch.bfloat16) -> Dict[str, torch.Tensor]:
    """Random-init weights with transformers' key names and init scale (normal std 0.02; norms at 1), generated on the
    device layer by layer (13.5 GB for the 7B shape)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    QW, KVW = cfg.num_heads * cfg.head_dim, cfg.num_kv_heads * cfg.head_dim

    def w(rows, cols):
        return (torch.randn((rows, cols), device=device, dtype=torch.float32, generator=g) * 0.02).to(dtype)

    sd = {"model.embed_tokens.weight": w(cfg.vocab, cfg.hidden)}
    for l in range(cfg.num_layers):
        p = f"model.layers.{l}."
        sd[p + "self_attn.q_proj.weight"] = w(QW, cfg.hidden)
        sd[p + "self_attn.k_proj.weight"] = w(KVW, cfg.hidden)
        sd[p + "self_attn.v_proj.weight"] = w(KVW, cfg.hidden)
        sd[p + "self_attn.o_proj.weight"] = w(cfg.hidden, QW)
        sd[p + "mlp.gate_proj.weight"] = w(cfg.intermediate, cfg.hidden)
        sd[p + "mlp.up_proj.weight"] = w(cfg.intermediate, cfg.hidden)
        sd[p + "mlp.down_proj.weight"] = w(cfg.hidden, cfg.intermediate)
        sd[p + "input_layernorm.weight"] = torch.ones(cfg.hidden, device=device, dtype=dtype)
        sd[p + "post_attention_layernorm.weight"] = torch.ones(cfg.hidden, device=device, dtype=dtype)
    sd["model.norm.weight"] = torch.ones(cfg.hidden, device=device, dtype=dtype)
    sd["lm_head.weight"] = w(cfg.vocab, cfg.hidden)
    return sd


# ---------------------------------------------------------------------------------------------------------------------
# Vision side: generic ViT towers + projector (include/blurr_vit.h)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class VitShapedConfig:
    num_layers: int            # blocks to RUN (OpenVLA takes the second-to-last block's output: depth - 1)
    hidden: int
    num_heads: int
    mlp_dim: int
    num_prefix_tokens: int = 0
    use_layerscale: bool = False
    gelu_erf: bool = False
    image_size: int = 224
    patch_size: int = 14
    ln_eps: float = 1e-6
    film_dim: int = 0          # > 0: FiLM-conditioned blocks (OpenVLA-OFT's language conditioning), conditioning width


def dinov2_large_reg4_config(depth: int = 24) -> VitShapedConfig:
    """`vit_large_patch14_reg4_dinov2` at 224 px: 24 blocks, 1024 wide, cls + 4 registers, LayerScale, exact GELU."""
    return VitShapedConfig(num_layers=depth - 1, hidden=1024, num_heads=16, mlp_dim=4096, num_prefix_tokens=5,
                           use_layerscale=True, gelu_erf=True)


def siglip_so400m_config(depth: int = 27) -> VitShapedConfig:
    """`vit_so400m_patch14_siglip_224`: 27 blocks, 1152 wide, no prefix tokens, tanh GELU."""
    return VitShapedConfig(num_layers=depth - 1, hidden=1152, num_heads=16, mlp_dim=4304)


class VitEncoder:
    """One ViT tower on one B200 through `include/blurr_vit.h`; `forward` returns the patch-token features."""

    def __init__(self, cfg: VitShapedConfig, device, max_batch: int = 1):
        self.lib = capi.load_library()
        self.cfg = cfg
        self.device = torch.device(device)
        self.max_batch = max_batch
        self.handle = C.c_void_p()
        c = capi.VitConfigC(capi.VIT_ABI_VERSION, cfg.num_layers, cfg.hidden, cfg.num_heads, cfg.mlp_dim, cfg.image_size,
                            cfg.patch_size, cfg.num_prefix_tokens, int(cfg.use_layerscale), int(cfg.gelu_erf), cfg.ln_eps,
                            cfg.film_dim)
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        capi.check(self.lib.blurr_vit_create(C.byref(c), index, max_batch, C.byref(self.handle)))
        self.n_patches = (cfg.image_size // cfg.patch_size) ** 2

    def set_weight(self, key: str, tensor: torch.Tensor):
        t = tensor.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        torch.cuda.current_stream(self.device).synchronize()
        shape = (C.c_int64 * t.dim())(*t.shape)
        capi.check(self.lib.blurr_vit_set_weight(self.handle, key.encode(), C.c_void_p(t.data_ptr()), shape, t.dim()))

    def finalize(self):
        capi.check(self.lib.blurr_vit_finalize(self.handle))

    def set_option(self, name: str, value: int):
        capi.check(self.lib.blurr_vit_set_option(self.handle, name.encode(), int(value)))

    def _set_films(self, films: Optional[Dict[str, torch.Tensor]]):
        """FiLM Linears from a state dict keyed like OFT's per-block pairs: "N.scale.weight|bias", "N.shift.weight|bias"."""
        for l in range(self.cfg.num_layers if films is not None else 0):
            for name in ("scale", "shift"):
                self.set_weight(f"layers.{l}.film_{name}.weight", films[f"{l}.{name}.weight"])
                self.set_weight(f"layers.{l}.film_{name}.bias", films[f"{l}.{name}.bias"])

    @classmethod
    def from_hf_dinov2(cls, model, device, max_batch: int = 1, num_layers: Optional[int] = None,
                       films: Optional[Dict[str, torch.Tensor]] = None) -> "VitEncoder":
        """From a transformers `Dinov2WithRegistersModel` (image_size 224 so that its position embeddings are native).
        `films`: FiLM weights ("N.scale.weight" [hidden, film_dim], ...) for a FiLM tower."""
        hc = model.config
        depth = hc.num_hidden_layers
        cfg = VitShapedConfig(num_layers=num_layers or depth - 1, hidden=hc.hidden_size, num_heads=hc.num_attention_heads,
                              mlp_dim=int(hc.hidden_size * hc.mlp_ratio), num_prefix_tokens=1 + hc.num_register_tokens,
                              use_layerscale=True, gelu_erf=True, image_size=hc.image_size, patch_size=hc.patch_size,
                              ln_eps=hc.layer_norm_eps, film_dim=films["0.scale.weight"].shape[1] if films else 0)
        self = cls(cfg, device, max_batch)
        sd = {k: v.to(torch.bfloat16) for k, v in model.state_dict().items()}
        e = "embeddings."
        self.set_weight("patch.weight", sd[e + "patch_embeddings.projection.weight"].flatten(1))
        self.set_weight("patch.bias", sd[e + "patch_embeddings.projection.bias"])
        pos = sd[e + "position_embeddings"][0]
        self.set_weight("pos", pos[1:])
        prefix = torch.cat([sd[e + "cls_token"][0] + pos[:1], sd[e + "register_tokens"][0]], dim=0)     # bf16 add, like HF
        self.set_weight("prefix", prefix)
        for l in range(cfg.num_layers):
            p, q = f"encoder.layer.{l}.", f"layers.{l}."
            for a, b in (("norm1", "ln1"), ("norm2", "ln2"), ("mlp.fc1", "fc1"), ("mlp.fc2", "fc2"),
                         ("attention.attention.query", "q"), ("attention.attention.key", "k"),
                         ("attention.attention.value", "v"), ("attention.output.dense", "o")):
                self.set_weight(q + b + ".weight", sd[p + a + ".weight"])
                self.set_weight(q + b + ".bias", sd[p + a + ".bias"])
            self.set_weight(q + "ls1", sd[p + "layer_scale1.lambda1"])
            self.set_weight(q + "ls2", sd[p + "layer_scale2.lambda1"])
        self._set_films(films)
        self.finalize()
        return self

    @classmethod
    def from_hf_siglip(cls, model, device, max_batch: int = 1, num_layers: Optional[int] = None,
                       films: Optional[Dict[str, torch.Tensor]] = None) -> "VitEncoder":
        """From a transformers `SiglipVisionModel` (`films` as in `from_hf_dinov2`)."""
        hc = model.config
        cfg = VitShapedConfig(num_layers=num_layers or hc.num_hidden_layers - 1, hidden=hc.hidden_size,
                              num_heads=hc.num_attention_heads, mlp_dim=hc.intermediate_size, image_size=hc.image_size,
                              patch_size=hc.patch_size, ln_eps=hc.layer_norm_eps,
                              film_dim=films["0.scale.weight"].shape[1] if films else 0)
        self = cls(cfg, device, max_batch)
        sd = {k: v.to(torch.bfloat16) for k, v in model.state_dict().items()}
        e = "vision_model.embeddings."
        self.set_weight("patch.weight", sd[e + "patch_embedding.weight"].flatten(1))
        self.set_weight("patch.bias", sd[e + "patch_embedding.bias"])
        self.set_weight("pos", sd[e + "position_embedding.weight"])
        for l in range(cfg.num_layers):
            p, q = f"vision_model.encoder.layers.{l}.", f"layers.{l}."
            for a, b in (("layer_norm1", "ln1"), ("layer_norm2", "ln2"), ("mlp.fc1", "fc1"), ("mlp.fc2", "fc2"),
                         ("self_attn.q_proj", "q"), ("self_attn.k_proj", "k"), ("self_attn.v_proj", "v"),
                         ("self_attn.out_proj", "o")):
                self.set_weight(q + b + ".weight", sd[p + a + ".weight"])
                self.set_weight(q + b + ".bias", sd[p + a + ".bias"])
        self._set_films(films)
        self.finalize()
        return self

    @classmethod
    def synthetic(cls, cfg: VitShapedConfig, device, max_batch: int = 1, seed: int = 0) -> "VitEncoder":
        """Random-init tower of the given shape (benchmarks).  With `film_dim` the FiLM Linears are drawn after every other
        weight, so a FiLM tower shares its other weights with the plain tower of the same seed."""
        self = cls(cfg, device, max_batch)
        g = torch.Generator(device=device)
        g.manual_seed(seed)
        H = cfg.hidden

        def w(*shape, std=0.02):
            return (torch.randn(shape, device=device, generator=g) * std).to(torch.bfloat16)

        self.set_weight("patch.weight", w(H, 3 * cfg.patch_size ** 2))
        self.set_weight("patch.bias", w(H))
        self.set_weight("pos", w(self.n_patches, H))
        if cfg.num_prefix_tokens:
            self.set_weight("prefix", w(cfg.num_prefix_tokens, H))
        ones = torch.ones(H, device=device, dtype=torch.bfloat16)
        for l in range(cfg.num_layers):
            q = f"layers.{l}."
            for name, (n, k) in (("q", (H, H)), ("k", (H, H)), ("v", (H, H)), ("o", (H, H)), ("fc1", (cfg.mlp_dim, H)),
                                 ("fc2", (H, cfg.mlp_dim))):
                self.set_weight(q + name + ".weight", w(n, k))
                self.set_weight(q + name + ".bias", w(n))
            for name in ("ln1", "ln2"):
                self.set_weight(q + name + ".weight", ones)
                self.set_weight(q + name + ".bias", torch.zeros_like(ones))
            if cfg.use_layerscale:
                self.set_weight(q + "ls1", ones)
                self.set_weight(q + "ls2", ones)
        for l in range(cfg.num_layers if cfg.film_dim else 0):
            for name in ("film_scale", "film_shift"):
                self.set_weight(f"layers.{l}.{name}.weight", w(H, cfg.film_dim))
                self.set_weight(f"layers.{l}.{name}.bias", w(H))
        self.finalize()
        return self

    def forward(self, pixel_values: torch.Tensor, out: Optional[torch.Tensor] = None, film_cond: Optional[torch.Tensor] = None,
                images_per_cond: int = 1) -> torch.Tensor:
        """pixel_values bf16 [B, 3, 224, 224] -> bf16 [B, n_patches, hidden] (or the first `hidden` columns of `out`).
        FiLM towers (`cfg.film_dim` > 0) need `film_cond`, bf16 [B / images_per_cond, film_dim] on the device: image i
        is conditioned on row i // images_per_cond."""
        if pixel_values.dtype != torch.bfloat16 or pixel_values.device.type != "cuda" or pixel_values.dim() != 4:
            raise ValueError("pixel_values must be a bf16 CUDA tensor [B, 3, H, W]")
        B = pixel_values.shape[0]
        film = self.cfg.film_dim > 0
        if film != (film_cond is not None):
            raise ValueError("film_cond is required by a FiLM tower (film_dim > 0) and rejected by any other")
        if film and (film_cond.dtype != torch.bfloat16 or film_cond.device.type != "cuda" or film_cond.dim() != 2
                     or film_cond.shape[1] != self.cfg.film_dim or film_cond.stride(1) != 1
                     or images_per_cond < 1 or film_cond.shape[0] * images_per_cond != B):
            raise ValueError(f"film_cond must be a bf16 CUDA tensor [B / images_per_cond, {self.cfg.film_dim}] with "
                             f"contiguous rows (B = {B}, images_per_cond = {images_per_cond})")
        if out is None:
            out = torch.empty((B, self.n_patches, self.cfg.hidden), device=self.device, dtype=torch.bfloat16)
        if out.stride(-1) != 1 or out.stride(0) != self.n_patches * out.stride(1):
            raise ValueError("out must be [B, n_patches, >= hidden] with contiguous rows")
        strides = (C.c_int64 * 4)(*pixel_values.stride())
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if film:
            capi.check(self.lib.blurr_vit_forward_film(self.handle, C.c_void_p(stream), B, C.c_void_p(pixel_values.data_ptr()),
                                                       strides, C.c_void_p(film_cond.data_ptr()), film_cond.stride(0),
                                                       images_per_cond, C.c_void_p(out.data_ptr()), out.stride(1)))
        else:
            capi.check(self.lib.blurr_vit_forward(self.handle, C.c_void_p(stream), B, C.c_void_p(pixel_values.data_ptr()),
                                                  strides, C.c_void_p(out.data_ptr()), out.stride(1)))
        return out

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.blurr_vit_last_launch_count(self.handle))

    def close(self):
        if self.handle:
            self.lib.blurr_vit_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MlpProjector:
    """OpenVLA's fused-backbone projector: Linear -> GELU -> Linear -> GELU -> Linear (exact GELU), `include/blurr_vit.h`."""

    def __init__(self, dims, device, max_rows: int):
        self.lib = capi.load_library()
        self.dims = list(dims)
        self.device = torch.device(device)
        self.handle = C.c_void_p()
        arr = (C.c_int32 * len(self.dims))(*self.dims)
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        capi.check(self.lib.blurr_mlp_create(arr, len(self.dims) - 1, index, max_rows, C.byref(self.handle)))

    def set_layer(self, i: int, weight: torch.Tensor, bias: torch.Tensor):
        w = weight.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        b = bias.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        assert tuple(w.shape) == (self.dims[i + 1], self.dims[i]) and tuple(b.shape) == (self.dims[i + 1],)
        torch.cuda.current_stream(self.device).synchronize()
        capi.check(self.lib.blurr_mlp_set_weight(self.handle, i, C.c_void_p(w.data_ptr()), C.c_void_p(b.data_ptr())))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x bf16 [..., dims[0]] contiguous -> bf16 [..., dims[-1]]."""
        x2 = x.reshape(-1, self.dims[0])
        if not x2.is_contiguous() or x2.dtype != torch.bfloat16:
            raise ValueError("x must be contiguous bf16")
        y = torch.empty((x2.shape[0], self.dims[-1]), device=self.device, dtype=torch.bfloat16)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        capi.check(self.lib.blurr_mlp_forward(self.handle, C.c_void_p(stream), x2.shape[0], C.c_void_p(x2.data_ptr()),
                                              self.dims[0], C.c_void_p(y.data_ptr()), self.dims[-1]))
        return y.reshape(*x.shape[:-1], self.dims[-1])

    def close(self):
        if self.handle:
            self.lib.blurr_mlp_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FusedVisionBackbone:
    """DINOv2 + SigLIP towers on the same image, patch features concatenated (DINOv2 first, as in Prismatic's
    `dinosiglip` backbone) and projected to the language model's width."""

    def __init__(self, dino: VitEncoder, siglip: VitEncoder, projector: MlpProjector, concurrent: bool = True):
        self.dino, self.siglip, self.projector = dino, siglip, projector
        self.width = dino.cfg.hidden + siglip.cfg.hidden
        # the two towers are independent chains of small, latency-bound kernels: run them side by side on two streams
        self._side = torch.cuda.Stream(device=dino.device) if concurrent else None

    def forward(self, pixel_values_dino: torch.Tensor, pixel_values_siglip: torch.Tensor, film_cond: Optional[torch.Tensor] = None,
                images_per_cond: int = 1) -> torch.Tensor:
        """`film_cond` (FiLM towers only): bf16 [B / images_per_cond, film_dim], given to both towers."""
        B = pixel_values_dino.shape[0]
        feats = torch.empty((B, self.dino.n_patches, self.width), device=pixel_values_dino.device, dtype=torch.bfloat16)
        sig_out = feats[:, :, self.dino.cfg.hidden:]
        if self._side is None:
            self.dino.forward(pixel_values_dino, out=feats, film_cond=film_cond, images_per_cond=images_per_cond)
            self.siglip.forward(pixel_values_siglip, out=sig_out, film_cond=film_cond, images_per_cond=images_per_cond)
        else:
            cur = torch.cuda.current_stream(self.dino.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self.siglip.forward(pixel_values_siglip, out=sig_out, film_cond=film_cond, images_per_cond=images_per_cond)
            self.dino.forward(pixel_values_dino, out=feats, film_cond=film_cond, images_per_cond=images_per_cond)
            cur.wait_stream(self._side)
            pixel_values_siglip.record_stream(self._side)
            feats.record_stream(self._side)
            if film_cond is not None:
                film_cond.record_stream(self._side)
        return self.projector.forward(feats)


# ---------------------------------------------------------------------------------------------------------------------
# Image preprocessing (include/blurr_vit.h: blurr_vla_preproc_*) and the whole policy
# ---------------------------------------------------------------------------------------------------------------------
DINOV2_MEAN, DINOV2_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)     # ImageNet, timm's DINOv2 data config
SIGLIP_MEAN, SIGLIP_STD = (0.5, 0.5, 0.5), (0.5, 0.5, 0.5)


def resize_geometry(h: int, w: int, size: Union[int, Sequence[int]] = 224,
                    crop: Union[int, Sequence[int]] = 224) -> Tuple[int, int, int, int]:
    """(resize_h, resize_w, crop_top, crop_left) of `TVF.center_crop(TVF.resize(img, size), crop)` on an h x w image.
    An int `size` becomes the shorter side, the longer one `int(size * long / short)`; an `(h, w)` tuple is the exact
    output shape (OpenVLA's "resize-naive").  Crop offsets are `int(round((H - crop) / 2.0))`, half to even."""
    if isinstance(size, int):
        short, long = (w, h) if w <= h else (h, w)
        new_short, new_long = size, int(size * long / short)
        rw, rh = (new_short, new_long) if w <= h else (new_long, new_short)
    else:
        rh, rw = int(size[0]), int(size[1])
    ch, cw = (crop, crop) if isinstance(crop, int) else (int(crop[0]), int(crop[1]))
    if ch > rh or cw > rw:
        raise ValueError(f"crop {(ch, cw)} is larger than the resized image {(rh, rw)} (torchvision would pad: not supported)")
    return rh, rw, int(round((rh - ch) / 2.0)), int(round((rw - cw) / 2.0))


def pillow_bicubic_coefficients(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray]:
    """Pillow's bicubic tables for one axis, from the library's host-side builder: bounds int32 [out, 2] = (first
    source index, tap count) and weights int32 [out, ksize] in Q22."""
    lib = capi.load_library()
    ksize = capi.check(lib.blurr_vla_preproc_build_coeffs(in_size, out_size, None, None, 0))
    bounds = np.zeros((out_size, 2), np.int32)
    weights = np.zeros((out_size, ksize), np.int32)
    capi.check(lib.blurr_vla_preproc_build_coeffs(in_size, out_size, bounds.ctypes.data_as(C.POINTER(C.c_int32)),
                                                  weights.ctypes.data_as(C.POINTER(C.c_int32)), ksize))
    return bounds, weights


class ImagePreprocessor:
    """OpenVLA's `PrismaticImageProcessor` for one frame geometry, on the device: Pillow bicubic resize, center crop,
    and one `to_tensor` + `normalize` per tower, stacked channel-wise ([DINOv2 RGB, SigLIP RGB]) in bf16."""

    def __init__(self, src_h: int, src_w: int, size: Union[int, Sequence[int]] = 224, crop: Union[int, Sequence[int]] = 224,
                 means: Sequence[Sequence[float]] = (DINOV2_MEAN, SIGLIP_MEAN),
                 stds: Sequence[Sequence[float]] = (DINOV2_STD, SIGLIP_STD), device="cuda:0"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("ImagePreprocessor runs on a CUDA device only (no CPU fallback)")
        if len(means) != len(stds) or any(len(m) != 3 for m in means) or any(len(s) != 3 for s in stds):
            raise ValueError("means and stds must be equally many RGB triples")
        self.src_h, self.src_w = int(src_h), int(src_w)
        self.resize_h, self.resize_w, self.crop_top, self.crop_left = resize_geometry(self.src_h, self.src_w, size, crop)
        self.crop_h, self.crop_w = (crop, crop) if isinstance(crop, int) else (int(crop[0]), int(crop[1]))
        self.n_norms = len(means)
        mean = (C.c_float * (3 * self.n_norms))(*[float(v) for m in means for v in m])
        std = (C.c_float * (3 * self.n_norms))(*[float(v) for s in stds for v in s])
        self.lib = capi.load_library()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        handle = C.c_void_p()
        capi.check(self.lib.blurr_vla_preproc_create(index, self.src_h, self.src_w, self.resize_h, self.resize_w,
                                                     self.crop_top, self.crop_left, self.crop_h, self.crop_w, self.n_norms,
                                                     mean, std, C.byref(handle)))
        self.handle = handle

    def coefficients(self):
        """((x_bounds, x_weights), (y_bounds, y_weights)): Pillow's tables for the whole resize of each axis.  An axis
        whose size does not change is not resampled (Pillow skips that pass), whatever its table says."""
        return (pillow_bicubic_coefficients(self.src_w, self.resize_w), pillow_bicubic_coefficients(self.src_h, self.resize_h))

    def __call__(self, frames_u8: torch.Tensor, out: Optional[torch.Tensor] = None, return_resized: bool = False):
        """frames_u8: CUDA uint8 [H, W, 3] or [B, H, W, 3]; rows and frames may be strided.  Returns bf16 pixel_values
        [B, 3 * n_norms, crop_h, crop_w]; with `return_resized` also the cropped uint8 resize [B, crop_h, crop_w, 3]."""
        if frames_u8.dtype != torch.uint8 or frames_u8.device != self.device:
            raise ValueError("frames must be uint8 tensors on the preprocessor's device")
        if frames_u8.dim() == 3:
            frames_u8 = frames_u8[None]
        if frames_u8.dim() != 4 or tuple(frames_u8.shape[1:]) != (self.src_h, self.src_w, 3):
            raise ValueError(f"frame geometry {tuple(frames_u8.shape)} != [B, {self.src_h}, {self.src_w}, 3]")
        if frames_u8.stride(3) != 1 or frames_u8.stride(2) != 3:
            frames_u8 = frames_u8.contiguous()
        B = frames_u8.shape[0]
        shape = (B, 3 * self.n_norms, self.crop_h, self.crop_w)
        if out is None:
            out = torch.empty(shape, device=self.device, dtype=torch.bfloat16)
        elif tuple(out.shape) != shape or out.dtype != torch.bfloat16 or out.device != self.device or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous bf16 tensor {shape} on the preprocessor's device")
        resized = (torch.empty((B, self.crop_h, self.crop_w, 3), device=self.device, dtype=torch.uint8)
                   if return_resized else None)
        capi.check(self.lib.blurr_vla_preproc_frame(
            self.handle, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream), C.c_void_p(frames_u8.data_ptr()),
            frames_u8.stride(1), B, frames_u8.stride(0), C.c_void_p(out.data_ptr()),
            C.c_void_p(resized.data_ptr()) if resized is not None else None))
        return (out, resized) if return_resized else out

    def close(self):
        if getattr(self, "handle", None):
            self.lib.blurr_vla_preproc_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OpenVlaPolicy:
    """OpenVLA's `predict_action` from raw camera frames: device preprocessing -> DINOv2 + SigLIP towers (fed the two
    halves of one 6-channel pixel tensor as strided views) -> projector -> `[BOS] + patches + prompt` -> greedy or
    sampled decode of `action_dim` tokens -> de-tokenised, de-normalised actions."""

    def __init__(self, preprocessor: ImagePreprocessor, backbone: FusedVisionBackbone, decoder: LlamaDecoder,
                 detokenizer: Optional[ActionDetokenizer] = None, action_dim: int = 7):
        if preprocessor.n_norms != 2:
            raise ValueError("the fused backbone needs two normalisations (DINOv2's, then SigLIP's)")
        if (preprocessor.crop_h, preprocessor.crop_w) != (backbone.dino.cfg.image_size,) * 2:
            raise ValueError("the preprocessor's crop must match the towers' image size")
        self.preprocessor, self.backbone, self.decoder = preprocessor, backbone, decoder
        self.detokenizer = detokenizer if detokenizer is not None else ActionDetokenizer()
        self.action_dim = action_dim

    def pixel_values(self, frames) -> torch.Tensor:
        """uint8 frame(s) [H, W, 3] / [B, H, W, 3], on the device or on the host (copied over as they are) ->
        bf16 [B, 6, 224, 224]."""
        f = torch.as_tensor(frames)
        if f.dim() == 3:
            f = f[None]
        if not f.is_cuda:
            f = f.to(self.preprocessor.device)
        return self.preprocessor(f)

    def predict_action_from_pixels(self, pixel_values: torch.Tensor, input_ids, q01, q99, mask=None,
                                   return_token_ids: bool = False, attention_mask: Optional[torch.Tensor] = None,
                                   do_sample: bool = False, temperature=1.0, top_k=50, top_p=1.0, seed=None):
        """The same as `predict_action`, from prepared bf16 pixel values [B, 6, 224, 224]."""
        patch = self.backbone.forward(pixel_values[:, :3], pixel_values[:, 3:])
        sample = dict(do_sample=True, temperature=temperature, top_k=top_k, top_p=top_p, seed=seed) if do_sample else {}
        if isinstance(input_ids, (list, tuple)) or attention_mask is not None:
            text, text_lens = ragged_prompt_ids(input_ids, attention_mask)
            x, lens = build_prompt_embeds_ragged(self.decoder, text.to(self.decoder.device), text_lens, patch)
            ids = self.decoder.generate(x, self.action_dim, prompt_lens=lens, **sample)
        else:
            ids = self.decoder.generate(build_prompt_embeds(self.decoder, input_ids, patch), self.action_dim, **sample)
        tokens = ids.cpu().numpy()
        actions = torch.from_numpy(self.detokenizer.actions(tokens[:, -self.action_dim:], q01, q99, mask))
        return (actions, ids) if return_token_ids else actions

    def predict_action(self, frames, input_ids, q01, q99, mask=None, return_token_ids: bool = False,
                       attention_mask: Optional[torch.Tensor] = None, do_sample: bool = False, temperature=1.0, top_k=50,
                       top_p=1.0, seed=None):
        """frames: uint8 [H, W, 3] or [B, H, W, 3] RGB.  input_ids: [B, S] (first column BOS), every row S tokens; or
        instructions of different lengths, as a list of B 1-D id tensors (each starting with BOS) or as [B, S] with a
        tokenizer's left- or right-padded `attention_mask` (see `ragged_prompt_ids`).  `mask` is the action mask of
        the de-normalisation, not a prompt mask.  q01 / q99 / mask: [action_dim], or [B, action_dim] for one dataset's
        statistics per row.  Returns float64 actions [B, action_dim] on the host (and the int64 token ids
        [B, action_dim] on the device with `return_token_ids`).  `do_sample=True` draws the action tokens with HF's
        `temperature`, `top_k` (default 50, as `generate` has it) and `top_p` instead of decoding greedily; `seed` as in
        `sampling_params` (None: drawn from torch's default generator)."""
        return self.predict_action_from_pixels(self.pixel_values(frames), input_ids, q01, q99, mask, return_token_ids,
                                               attention_mask, do_sample, temperature, top_k, top_p, seed)


# ---------------------------------------------------------------------------------------------------------------------
# OpenVLA-OFT: parallel decoding of action chunks (include/blurr_llm.h blurr_llm_forward_rows, include/blurr_act_head.h)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class OftConfig:
    """OpenVLA-OFT's action chunking (Kim, Finn, Liang 2025): `chunk` actions of `action_dim` dimensions per call, one
    empty action slot per value.  `bidirectional_actions`: the slots (and the stop token) attend to each other, as the
    paper describes; False gives plain causal attention.  The head is `MLPResNet(head_num_blocks, action_dim * hidden,
    head_hidden_dim, action_dim)`; `max_positions` is the decoder's (1 + patches + prompt + 56 slots + stop).
    `num_images` cameras (third-person first, then the wrist camera; ALOHA: top, left wrist, right wrist) give 256
    patch rows each; `use_proprio` appends
    one projected row of the `proprio_dim`-wide robot state after them.  `use_film`: the towers are FiLM-conditioned on
    the averaged instruction embedding (`film_language_embedding`), OFT's "OFT+" form."""
    chunk: int = 8
    action_dim: int = 7
    bidirectional_actions: bool = True
    head_hidden_dim: int = 4096
    head_num_blocks: int = 2
    head_ln_eps: float = 1e-5
    max_positions: int = 384
    empty_token: int = 29871          # Llama-2's empty token after "Out:"
    stop_token: int = 2               # </s>
    num_images: int = 1
    use_proprio: bool = False
    proprio_dim: int = 8
    use_film: bool = False


def oft_libero_config() -> OftConfig:
    """OFT's LIBERO checkpoints: third-person and wrist cameras, 8-D proprioception, chunks of 8 x 7.  A sequence is
    1 + 513 + prompt + 56 + 1 positions (about 605 with LIBERO's instructions); the decoder holds 640."""
    return OftConfig(num_images=2, use_proprio=True, proprio_dim=8, chunk=8, action_dim=7, max_positions=640)


def oft_aloha_config() -> OftConfig:
    """OFT's bimanual ALOHA checkpoints (OFT+): three cameras in the order top, left wrist, right wrist, 14-D
    proprioception, chunks of 25 x 14 and FiLM.  P = 3 * 256 + 1 = 769 rows precede the prompt and 25 * 14 = 350 empty
    slots and the stop token follow it, so a sequence is 769 + S + 350 + 1 = 1120 + S positions (S: the prompt with BOS
    and 29871; about 1140-1150 with OpenVLA's template).  The decoder holds 1280, which allows S <= 160.  ALOHA
    normalises with OFT's BOUNDS statistics (min / max): pass them where the LIBERO form passes q01 / q99."""
    return OftConfig(num_images=3, use_proprio=True, proprio_dim=14, chunk=25, action_dim=14, use_film=True, max_positions=1280)


def openvla_oft_7b_config(oft: Optional[OftConfig] = None) -> LlamaShapedConfig:
    """The OpenVLA-7B decoder with room for OFT's sequence (`oft.max_positions`, 384 by default; `openvla_7b_config`
    keeps 320).  `long_forward` is 0 up to 384 positions, 1 up to 1024 and 2 beyond."""
    n = (oft or OftConfig()).max_positions
    return LlamaShapedConfig(max_positions=n, long_forward=0 if n <= 384 else 1 if n <= 1024 else 2)


def normalize_proprio(state, q01, q99, mask=None) -> np.ndarray:
    """OFT's BOUNDS_Q99 normalisation of the robot state, on the host in float64:
    `clip(where(mask, 2 * (x - q01) / (q99 - q01 + 1e-8) - 1, x), -1, 1)`.  state [B, D] (or [D]); q01 / q99 / mask
    [D] or [B, D].  OFT's BOUNDS rule (ALOHA) is the same arithmetic on the dataset's min / max: pass them as q01 / q99."""
    x = np.asarray(state.detach().cpu() if isinstance(state, torch.Tensor) else state, dtype=np.float64)
    lo, hi = np.asarray(q01, dtype=np.float64), np.asarray(q99, dtype=np.float64)
    m = np.ones(lo.shape, dtype=bool) if mask is None else np.asarray(mask, dtype=bool)
    return np.clip(np.where(m, 2 * (x - lo) / (hi - lo + 1e-8) - 1, x), -1.0, 1.0)


@dataclass
class OftLayout:
    """Host-side layout of one OFT batch.  Sequence b is `[BOS] + P patches + ids[b, 1:text_lens[b]] + chunk * action_dim
    zero rows + embed(stop)`, pads after it up to `max_len`."""
    ids: torch.Tensor                  # int64 [B, S_max] on the host: row b's text_lens[b] tokens (29871 appended), pad id 0 after
    text_lens: torch.Tensor            # int64 [B]: S_b, BOS included
    seq_lens: np.ndarray               # int32 [B]: P + S_b + chunk * action_dim + 1
    block_starts: np.ndarray           # int32 [B]: a0 = P + S_b (seq_lens with bidirectional_actions=False)
    row_starts: np.ndarray             # int32 [B]: P + S_b - 1, the row before each action slot
    max_len: int
    n_rows: int                        # chunk * action_dim


def oft_prompt_layout(input_ids, attention_mask: Optional[torch.Tensor] = None, n_patches: int = 256,
                      cfg: Optional[OftConfig] = None) -> OftLayout:
    """OFT's `predict_action` prompt for the three forms `ragged_prompt_ids` accepts ([B, S], a list of 1-D id tensors, or
    [B, S] with a left- or right-padded `attention_mask`): a row whose last id is not `empty_token` (29871) gets it
    appended; then the action slots, the stop token and the attention block follow.  Raises ValueError when a sequence
    would need more than `cfg.max_positions` positions."""
    cfg = cfg or OftConfig()
    ids, lens = ragged_prompt_ids(input_ids, attention_mask)
    ids, lens = ids.cpu(), lens.clone()
    last = ids.gather(1, (lens - 1)[:, None])[:, 0]
    add = last != cfg.empty_token
    S = int((lens + add.to(torch.int64)).max())
    out = torch.zeros((ids.shape[0], S), dtype=torch.int64)
    out[:, :ids.shape[1]] = ids[:, :S]
    rows = torch.arange(ids.shape[0])
    out[rows[add], lens[add]] = cfg.empty_token
    lens = lens + add.to(torch.int64)
    n_rows = cfg.chunk * cfg.action_dim
    a0 = (lens + n_patches).numpy().astype(np.int32)
    seq = a0 + n_rows + 1
    max_len = int(seq.max())
    if max_len > cfg.max_positions:
        raise ValueError(f"an OFT sequence needs {max_len} positions (patches {n_patches} + prompt {int(lens.max())} + "
                         f"{n_rows} action slots + stop), more than max_positions = {cfg.max_positions}")
    blk = a0.copy() if cfg.bidirectional_actions else seq.copy()
    return OftLayout(ids=out, text_lens=lens, seq_lens=seq, block_starts=blk,
                     row_starts=(a0 - 1).astype(np.int32), max_len=max_len, n_rows=n_rows)


def build_oft_embeds(decoder: LlamaDecoder, layout: OftLayout, patch_embeds: torch.Tensor, stop_token: int = 2) -> torch.Tensor:
    """bf16 [B, layout.max_len, hidden]: the prompt rows of `build_prompt_embeds` / `build_prompt_embeds_ragged`, then
    chunk * action_dim zeroed slots and the stop token's embedding; zeros after it."""
    x, _ = build_prompt_embeds_ragged(decoder, layout.ids.to(decoder.device), layout.text_lens, patch_embeds)
    B, L, H = x.shape[0], layout.max_len, x.shape[2]
    full = torch.zeros((B, L, H), device=x.device, dtype=x.dtype)
    full[:, :x.shape[1]] = x
    pos = torch.arange(L, device=x.device)[None, :]
    a0 = torch.as_tensor(layout.row_starts + 1, device=x.device, dtype=torch.int64)[:, None]
    stop_row = decoder.embed(torch.tensor([stop_token], device=x.device))[0]
    full = torch.where((pos < a0)[..., None], full, torch.zeros((), device=x.device, dtype=x.dtype))
    return torch.where((pos == a0 + layout.n_rows)[..., None], stop_row, full).contiguous()


def film_language_rows(layout: OftLayout, stop_token: int = 2) -> List[torch.Tensor]:
    """The token ids whose embeddings FiLM averages, one int64 tensor per sequence: `ids[b, :text_lens[b]]` (BOS, the
    instruction, the appended 29871) and the stop token.  OFT embeds its whole input and drops the positions its action
    mask marks; that mask is taken to cover the action placeholders only, so the stop token stays - a restatement choice
    (OFT's own code is not available here, DESIGN.md 10).  The action slots and the pads are never averaged, so a sequence
    of a ragged batch gets what it gets alone.  Everything that needs these rows calls this function."""
    stop = torch.tensor([stop_token], dtype=torch.int64)
    return [torch.cat([layout.ids[b, :int(layout.text_lens[b])], stop]) for b in range(layout.ids.shape[0])]


def film_language_embedding(decoder: LlamaDecoder, layout: OftLayout, stop_token: int = 2) -> torch.Tensor:
    """FiLM's language vector, bf16 [B, hidden] on the decoder's device: the mean of the embeddings of
    `film_language_rows`, per sequence, as OFT's `language_embeddings.mean(dim=1)` (fp32 sum, one bf16 rounding)."""
    return torch.cat([decoder.embed(r)[None].mean(dim=1) for r in film_language_rows(layout, stop_token)]).contiguous()


class L1RegressionHead:
    """OpenVLA-OFT's `L1RegressionActionHead` on one B200 through `include/blurr_act_head.h`: the decoder's action rows
    [B, chunk * action_dim, hidden] -> normalised actions fp32 [B, chunk, action_dim] (the module's bf16 output)."""

    def __init__(self, cfg: OftConfig, input_dim: int, device, max_batch: int = 1):
        self.lib = capi.load_library()
        self.cfg, self.input_dim = cfg, int(input_dim)
        self.device = torch.device(device)
        self.max_batch = max_batch
        self.handle = C.c_void_p()
        c = capi.ActHeadConfigC(capi.ACT_HEAD_ABI_VERSION, self.input_dim, cfg.action_dim, cfg.chunk, cfg.head_hidden_dim,
                                cfg.head_num_blocks, cfg.head_ln_eps)
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        capi.check(self.lib.blurr_act_head_create(C.byref(c), index, max_batch, C.byref(self.handle)))

    @classmethod
    def from_state_dict(cls, cfg: OftConfig, state_dict: Dict[str, torch.Tensor], input_dim: int, device, max_batch: int = 1,
                        prefix: str = "") -> "L1RegressionHead":
        """`state_dict`: keys of OFT's `L1RegressionActionHead.state_dict()` ("model.fc1.weight", ...), optionally under
        `prefix`."""
        self = cls(cfg, input_dim, device, max_batch)
        try:
            for key, t in state_dict.items():
                if prefix and not key.startswith(prefix):
                    continue
                self.set_weight(key[len(prefix):], t)
            capi.check(self.lib.blurr_act_head_finalize(self.handle))
        except Exception:
            self.close()
            raise
        return self

    @classmethod
    def synthetic(cls, cfg: OftConfig, input_dim: int, device, max_batch: int = 1, seed: int = 0) -> "L1RegressionHead":
        """Random-init head with nn.Linear's default init (uniform, bound 1 / sqrt(fan_in)) and LayerNorms at 1 / 0,
        generated on the device (0.25 GB at OFT's widths)."""
        return cls.from_state_dict(cfg, synthetic_act_head_state_dict(cfg, input_dim, device, seed), input_dim, device, max_batch)

    def set_weight(self, name: str, tensor: torch.Tensor):
        t = tensor.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        torch.cuda.current_stream(self.device).synchronize()
        shape = (C.c_int64 * t.dim())(*t.shape)
        capi.check(self.lib.blurr_act_head_set_weight(self.handle, name.encode(), C.c_void_p(t.data_ptr()), shape, t.dim()))

    def forward(self, hidden_rows: torch.Tensor) -> torch.Tensor:
        """hidden_rows bf16 [B, chunk * action_dim, input_dim] on the device -> fp32 [B, chunk, action_dim]."""
        K, D = self.cfg.chunk, self.cfg.action_dim
        if hidden_rows.dim() != 3 or tuple(hidden_rows.shape[1:]) != (K * D, self.input_dim):
            raise ValueError(f"hidden_rows must be [B, {K * D}, {self.input_dim}]")
        if hidden_rows.dtype != torch.bfloat16 or hidden_rows.device.type != "cuda":
            raise ValueError("hidden_rows must be a bf16 CUDA tensor")
        x = hidden_rows.contiguous()
        B = x.shape[0]
        out = torch.empty((B, K, D), device=self.device, dtype=torch.float32)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        capi.check(self.lib.blurr_act_head_forward(self.handle, C.c_void_p(stream), B, C.c_void_p(x.data_ptr()),
                                                   C.c_void_p(out.data_ptr())))
        return out

    def check(self):
        capi.check(self.lib.blurr_act_head_check(self.handle, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.blurr_act_head_last_launch_count(self.handle))

    def close(self):
        if self.handle:
            self.lib.blurr_act_head_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def synthetic_act_head_state_dict(cfg: OftConfig, input_dim: int, device, seed: int = 0,
                                  dtype=torch.bfloat16) -> Dict[str, torch.Tensor]:
    """Random-init weights of `L1RegressionActionHead` with its state_dict keys, nn.Linear's default init."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    H, W, D = cfg.head_hidden_dim, cfg.action_dim * input_dim, cfg.action_dim

    def u(shape, fan_in):
        return ((torch.rand(shape, device=device, generator=g) * 2 - 1) / math.sqrt(fan_in)).to(dtype)

    sd = {"model.layer_norm1.weight": torch.ones(W, device=device, dtype=dtype),
          "model.layer_norm1.bias": torch.zeros(W, device=device, dtype=dtype),
          "model.fc1.weight": u((H, W), W), "model.fc1.bias": u((H,), W)}
    for i in range(cfg.head_num_blocks):
        p = f"model.mlp_resnet_blocks.{i}.ffn."
        sd[p + "0.weight"] = torch.ones(H, device=device, dtype=dtype)
        sd[p + "0.bias"] = torch.zeros(H, device=device, dtype=dtype)
        sd[p + "1.weight"] = u((H, H), H)
        sd[p + "1.bias"] = u((H,), H)
    sd["model.layer_norm2.weight"] = torch.ones(H, device=device, dtype=dtype)
    sd["model.layer_norm2.bias"] = torch.zeros(H, device=device, dtype=dtype)
    sd["model.fc2.weight"] = u((D, H), H)
    sd["model.fc2.bias"] = u((D,), H)
    return sd


class ProprioProjector:
    """OpenVLA-OFT's `ProprioProjector`: `fc1 (proprio_dim -> hidden) -> GELU (exact) -> fc2 (hidden -> hidden)`, on
    the `MlpProjector` engine.  That engine takes inputs 64 columns wide, so the state is zero-padded to 64 columns and
    fc1's weight to [hidden, 64]; the padded products are exact zeros, so the result is fc1's."""

    K_PAD = 64

    def __init__(self, proprio_dim: int, hidden: int, device, max_rows: int = 1):
        if not 1 <= proprio_dim <= self.K_PAD:
            raise ValueError(f"proprio_dim must be in 1..{self.K_PAD}")
        self.proprio_dim, self.hidden = int(proprio_dim), int(hidden)
        self.device = torch.device(device)
        self.mlp = MlpProjector([self.K_PAD, self.hidden, self.hidden], device, max_rows)

    @classmethod
    def from_state_dict(cls, state_dict: Dict[str, torch.Tensor], device, max_rows: int = 1, prefix: str = "") -> "ProprioProjector":
        """`state_dict`: keys of OFT's `ProprioProjector.state_dict()` ("fc1.weight", "fc1.bias", "fc2.weight",
        "fc2.bias"), optionally under `prefix`."""
        sd = {k[len(prefix):]: v for k, v in state_dict.items() if k.startswith(prefix)}
        missing = {"fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias"} - set(sd)
        if missing:
            raise ValueError(f"ProprioProjector.from_state_dict: missing {sorted(missing)}")
        hidden, dim = sd["fc1.weight"].shape
        self = cls(dim, hidden, device, max_rows)
        try:
            w1 = torch.zeros((hidden, cls.K_PAD), device=self.device, dtype=torch.bfloat16)
            w1[:, :dim] = sd["fc1.weight"].to(device=self.device, dtype=torch.bfloat16)
            self.mlp.set_layer(0, w1, sd["fc1.bias"])
            self.mlp.set_layer(1, sd["fc2.weight"], sd["fc2.bias"])
        except Exception:
            self.close()
            raise
        return self

    @classmethod
    def synthetic(cls, proprio_dim: int, hidden: int, device, max_rows: int = 1, seed: int = 0) -> "ProprioProjector":
        """Random-init projector with nn.Linear's default init (uniform, bound 1 / sqrt(fan_in))."""
        g = torch.Generator(device=device)
        g.manual_seed(seed)

        def u(shape, fan_in):
            return ((torch.rand(shape, device=device, generator=g) * 2 - 1) / math.sqrt(fan_in)).to(torch.bfloat16)

        sd = {"fc1.weight": u((hidden, proprio_dim), proprio_dim), "fc1.bias": u((hidden,), proprio_dim),
              "fc2.weight": u((hidden, hidden), hidden), "fc2.bias": u((hidden,), hidden)}
        return cls.from_state_dict(sd, device, max_rows)

    def forward(self, state: torch.Tensor) -> torch.Tensor:
        """state [B, proprio_dim] (already normalised; cast to bf16 on the device) -> bf16 [B, hidden]."""
        if state.dim() != 2 or state.shape[1] != self.proprio_dim:
            raise ValueError(f"state must be [B, {self.proprio_dim}]")
        x = torch.zeros((state.shape[0], self.K_PAD), device=self.device, dtype=torch.bfloat16)
        x[:, :self.proprio_dim] = state.to(device=self.device, dtype=torch.bfloat16)
        return self.mlp.forward(x)

    def close(self):
        self.mlp.close()


class OftPolicy:
    """OpenVLA-OFT's `predict_action` with parallel decoding: device preprocessing of each camera -> DINOv2 + SigLIP
    towers -> projector (-> the proprio projector) -> `[BOS] + patches (+ proprio row) + prompt + empty action slots +
    stop` -> one decoder pass (`forward_rows`) -> the L1-regression head -> a whole chunk of de-normalised actions.  No
    decode loop: one call yields `chunk` actions.  `preprocessor` is one `ImagePreprocessor` per camera (a single one
    for one camera); the towers need max_batch >= B * num_images."""

    def __init__(self, preprocessor, backbone: FusedVisionBackbone, decoder: LlamaDecoder,
                 head: L1RegressionHead, cfg: Optional[OftConfig] = None, proprio_projector: Optional[ProprioProjector] = None):
        cfg = cfg or head.cfg
        pres = list(preprocessor) if isinstance(preprocessor, (list, tuple)) else [preprocessor]
        if len(pres) != cfg.num_images:
            raise ValueError(f"{len(pres)} preprocessors for {cfg.num_images} cameras")
        for p in pres:
            if p.n_norms != 2:
                raise ValueError("the fused backbone needs two normalisations (DINOv2's, then SigLIP's)")
        if (head.cfg.chunk, head.cfg.action_dim) != (cfg.chunk, cfg.action_dim) or head.input_dim != decoder.cfg.hidden:
            raise ValueError("the head's chunk, action_dim and input width must match the config and the decoder")
        if cfg.use_proprio and (proprio_projector is None or proprio_projector.proprio_dim != cfg.proprio_dim
                                or proprio_projector.hidden != decoder.cfg.hidden):
            raise ValueError("use_proprio needs a ProprioProjector of proprio_dim columns and the decoder's width")
        film_dims = (backbone.dino.cfg.film_dim, backbone.siglip.cfg.film_dim)
        if film_dims != ((decoder.cfg.hidden,) * 2 if cfg.use_film else (0, 0)):
            raise ValueError(f"use_film = {cfg.use_film} needs towers with film_dim = "
                             f"{decoder.cfg.hidden if cfg.use_film else 0} (the decoder's width with FiLM, 0 without); "
                             f"they have {film_dims}")
        self.preprocessors, self.preprocessor = pres, pres[0]
        self.backbone, self.decoder, self.head, self.cfg = backbone, decoder, head, cfg
        self.proprio_projector = proprio_projector if cfg.use_proprio else None

    def pixel_values(self, frames) -> torch.Tensor:
        """uint8 frame(s) [H, W, 3] / [B, H, W, 3] (one camera), or a sequence of num_images such batches (one per
        camera, in the config's order) -> bf16 [B, 6 * num_images, 224, 224]: each camera's `OpenVlaPolicy.pixel_values`
        stacked along channels."""
        n = self.cfg.num_images
        per_cam = [frames] if n == 1 else list(frames) if isinstance(frames, (list, tuple)) else None
        if per_cam is None or len(per_cam) != n:
            raise ValueError(f"frames must be a sequence of {n} per-camera uint8 batches")
        out = []
        for pre, fr in zip(self.preprocessors, per_cam):
            f = torch.as_tensor(fr)
            if f.dim() == 3:
                f = f[None]
            if not f.is_cuda:
                f = f.to(pre.device)
            out.append(pre(f))
        if len({o.shape[0] for o in out}) != 1:
            raise ValueError("every camera needs the same batch size")
        return out[0] if n == 1 else torch.cat(out, dim=1)

    def patch_embeds(self, pixel_values: torch.Tensor, proprio_state: Optional[torch.Tensor] = None,
                     film_cond: Optional[torch.Tensor] = None) -> torch.Tensor:
        """bf16 pixel values [B, 6 * num_images, 224, 224] (and the normalised state [B, proprio_dim]) -> the rows
        between BOS and the prompt, bf16 [B, 256 * num_images (+ 1), hidden]: image i's patches at rows 256 i ..
        (OFT's `torch.cat(all_patches, dim=1)`), then the projected state.  With `use_film`, `film_cond` is the language
        vector [B, hidden] every camera of a sequence is conditioned on."""
        n = self.cfg.num_images
        if pixel_values.dim() != 4 or pixel_values.shape[1] != 6 * n:
            raise ValueError(f"pixel_values must be [B, {6 * n}, H, W] ({n} camera(s) of 6 channels)")
        B = pixel_values.shape[0]
        px = pixel_values if n == 1 else pixel_values.reshape(B * n, 6, *pixel_values.shape[2:])
        if self.cfg.use_film and film_cond is None:
            raise ValueError("use_film needs the language vector (film_language_embedding)")
        patch = self.backbone.forward(px[:, :3], px[:, 3:], film_cond if self.cfg.use_film else None, images_per_cond=n)
        if n > 1:
            patch = patch.reshape(B, n * patch.shape[1], patch.shape[2])
        if self.proprio_projector is None:
            return patch
        if proprio_state is None or proprio_state.dim() != 2 or tuple(proprio_state.shape) != (B, self.cfg.proprio_dim):
            raise ValueError(f"use_proprio needs a proprio state [{B}, {self.cfg.proprio_dim}]")
        row = self.proprio_projector.forward(proprio_state)
        return torch.cat([patch, row[:, None].to(patch.dtype)], dim=1)

    def action_rows(self, pixel_values: torch.Tensor, input_ids, attention_mask: Optional[torch.Tensor] = None,
                    proprio_state: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The decoder's final-normed rows in front of the action slots, bf16 [B, chunk * action_dim, hidden].  The layout
        comes first: with `use_film` the towers need the language vector it defines."""
        P = self.backbone.dino.n_patches * self.cfg.num_images + (1 if self.cfg.use_proprio else 0)
        lay = oft_prompt_layout(input_ids, attention_mask, P, self.cfg)
        if lay.max_len > self.decoder.cfg.max_positions:
            raise ValueError(f"an OFT sequence needs {lay.max_len} positions; the decoder holds {self.decoder.cfg.max_positions}")
        cond = film_language_embedding(self.decoder, lay, self.cfg.stop_token) if self.cfg.use_film else None
        if cond is not None and cond.shape[0] != pixel_values.shape[0]:
            raise ValueError("input_ids must hold one prompt per sequence of pixel_values")
        patch = self.patch_embeds(pixel_values, proprio_state, cond)
        x = build_oft_embeds(self.decoder, lay, patch, self.cfg.stop_token)
        return self.decoder.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows)

    def proprio_state(self, proprio, proprio_q01, proprio_q99, proprio_mask=None) -> Optional[torch.Tensor]:
        """The raw robot state [B, proprio_dim] -> `normalize_proprio` on the host -> float32 -> bf16 on the device, as
        OFT's `torch.Tensor(proprio).to(bfloat16)` (None when the config has no proprio)."""
        if not self.cfg.use_proprio:
            if proprio is not None:
                raise ValueError("proprio given, but the config has use_proprio = False")
            return None
        if proprio is None or proprio_q01 is None or proprio_q99 is None:
            raise ValueError("use_proprio needs proprio, proprio_q01 and proprio_q99")
        p = np.asarray(proprio.detach().cpu() if isinstance(proprio, torch.Tensor) else proprio, dtype=np.float64)
        if p.ndim == 1:
            p = p[None]
        if p.ndim != 2 or p.shape[1] != self.cfg.proprio_dim:
            raise ValueError(f"proprio must be [B, {self.cfg.proprio_dim}], got shape {p.shape}")
        x = normalize_proprio(p, proprio_q01, proprio_q99, proprio_mask)
        return torch.from_numpy(x.astype(np.float32)).to(device=self.decoder.device, dtype=torch.bfloat16)

    def predict_action_chunk_from_pixels(self, pixel_values: torch.Tensor, input_ids, q01, q99, mask=None,
                                         attention_mask: Optional[torch.Tensor] = None, return_normalized: bool = False,
                                         proprio=None, proprio_q01=None, proprio_q99=None, proprio_mask=None):
        """The same as `predict_action_chunk`, from prepared bf16 pixel values [B, 6 * num_images, 224, 224]."""
        state = self.proprio_state(proprio, proprio_q01, proprio_q99, proprio_mask)
        if state is not None and state.shape[0] != pixel_values.shape[0]:
            raise ValueError("proprio must hold one state per sequence")
        norm = self.head.forward(self.action_rows(pixel_values, input_ids, attention_mask, state))
        actions = torch.from_numpy(denormalize_chunk(norm.cpu().numpy(), q01, q99, mask))
        return (actions, norm) if return_normalized else actions

    def predict_action_chunk(self, frames, input_ids, q01, q99, mask=None, attention_mask: Optional[torch.Tensor] = None,
                             return_normalized: bool = False, proprio=None, proprio_q01=None, proprio_q99=None,
                             proprio_mask=None):
        """frames: uint8 [H, W, 3] or [B, H, W, 3] RGB for one camera; with num_images > 1 a sequence of such batches,
        one per camera (third-person first, then the wrist camera; ALOHA: top, left wrist, right wrist).  input_ids: [B, S] (first column BOS), a list of B
        1-D id tensors, or [B, S] with a left- or right-padded `attention_mask` (see `oft_prompt_layout`).  q01 / q99 /
        mask: [action_dim] or [B, action_dim], applied to every step of the chunk.  With `use_proprio`: `proprio` the
        raw state [B, proprio_dim] and its dataset's `proprio_q01` / `proprio_q99` (/ `proprio_mask`), normalised by
        `normalize_proprio`.  For ALOHA (BOUNDS statistics) pass the min / max in place of q01 / q99, for the actions
        and the state alike.  Returns float64 actions [B, chunk, action_dim] on the host (and, with
        `return_normalized`, the head's output fp32 [B, chunk, action_dim] on the device)."""
        return self.predict_action_chunk_from_pixels(self.pixel_values(frames), input_ids, q01, q99, mask, attention_mask,
                                                     return_normalized, proprio, proprio_q01, proprio_q99, proprio_mask)
