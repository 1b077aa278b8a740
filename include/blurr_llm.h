/*
 * blurr_llm.h - C ABI of the Llama-shaped decoder behind the OpenVLA-7B-shaped path (SURVEY.md 8(f) row 3,
 * BASELINE.json configs[4]: "OpenVLA-7B-shaped (SigLIP+DINOv2 fused encoder + Llama-2-7B) random-init, 7-token
 * autoregressive action decode with KV cache, batch 1 and 32").
 *
 * What it replaces.  The reference has no source for this model: `scripts/benchmark_hf_vla.py:100-109,141-197` loads
 * `openvla/openvla-7b` through `AutoModelForVision2Seq.from_pretrained(..., trust_remote_code=True)` and times
 * `model.predict_action(**inputs, unnorm_key=..., do_sample=False)` (:152).  That call runs the vision backbone and
 * projector, then `LlamaForCausalLM` greedy generation of `action_dim` tokens with a KV cache.  This library is the
 * language-model part: prefill of the multimodal prompt embeddings + N greedy decode steps, arithmetic as in
 * transformers' `LlamaForCausalLM` with eager attention (modeling_llama.py: LlamaRMSNorm, apply_rotary_pos_emb,
 * eager_attention_forward, LlamaMLP) - the class the remote code instantiates for its `language_model`.
 * PARITY: pinned against transformers 5.5.0 `LlamaForCausalLM` (a library present in this image, not reference source);
 * against the reference itself it is UNPINNED (the remote code is neither vendored nor downloadable), see DESIGN.md.
 *
 * blurr_llm_generate serves equal-length, ragged and sampled calls.  A batch may mix prompts of different lengths
 * (prompt_lens): each sequence's prompt sits at the front of its rows, pads behind it, and its tokens are generated at its
 * own positions, so each sequence gets what it would get alone; one CUDA graph per batch shape serves every vector of
 * lengths.
 *
 * Sampled decoding (params) draws each token as transformers' `generate(do_sample=True)` does: the fp32 logits go
 * through TemperatureLogitsWarper, TopKLogitsWarper and TopPLogitsWarper, then softmax and one draw.  The draw of
 * sequence b at step i uses Philox4x32-10 with key = params[b].seed and counter = (i, 0, 0, 0), so it depends on nothing
 * but the seed, the step and the logits; the result is bitwise repeatable.
 *
 * All pointers are device pointers unless stated.  Errors: negative blurr_status (blurr_pi0.h), message from
 * blurr_last_error().  One handle per GPU and per host thread.  Weights are bf16.
 */
#ifndef BLURR_LLM_H_
#define BLURR_LLM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct blurr_llm blurr_llm_t;

typedef struct blurr_llm_config {
    int32_t abi_version;          /* BLURR_LLM_ABI_VERSION */
    int32_t num_layers;           /* 32 */
    int32_t hidden;               /* 4096, multiple of 128 */
    int32_t num_heads;            /* 32 */
    int32_t num_kv_heads;         /* 32 (== num_heads: multi-head attention) */
    int32_t head_dim;             /* 128 (or 64) */
    int32_t intermediate;         /* 11008, multiple of 64 */
    int32_t vocab;                /* 32064 (rows of embed_tokens / lm_head) */
    int32_t max_positions;        /* KV-cache slots per sequence, <= 384, or <= 1024 with long_forward = 1, or 1025..2048
                                     with long_forward = 2 (generate: prompt + generated tokens <= 320 on every handle) */
    float rms_eps;                /* 1e-6 (OpenVLA) / 1e-5 (Llama-2) */
    int32_t long_forward;         /* 0: max_positions <= 384; 1: up to 1024 for blurr_llm_forward_rows (OFT's two-camera
                                     sequences); 2: 1025..2048 (OFT's three-camera ALOHA sequences); any other value is
                                     rejected */
} blurr_llm_config;
#define BLURR_LLM_ABI_VERSION 3

/* Per-sequence sampling parameters (HF names and rules):
 *   temperature  finite, > 0: scores * (1.0f / temperature) (ATen's fp32 reciprocal);
 *   top_k        >= 0; 0 = off, >= vocab = all; ties at the k-th largest score are all kept;
 *   top_p        in [0, 1]; 1 = off; keeps the smallest set of highest scores whose mass reaches top_p (always the top
 *                token; among equal scores at the cut the higher token ids are kept, as torch's stable sort does). */
typedef struct blurr_llm_sampling {
    uint64_t seed;
    float temperature;
    int32_t top_k;
    float top_p;
} blurr_llm_sampling;
#ifdef __cplusplus
static_assert(sizeof(blurr_llm_sampling) == 24 && offsetof(blurr_llm_sampling, temperature) == 8 &&
                  offsetof(blurr_llm_sampling, top_k) == 12 && offsetof(blurr_llm_sampling, top_p) == 16,
              "blurr_llm_sampling layout");
#else
_Static_assert(sizeof(blurr_llm_sampling) == 24 && offsetof(blurr_llm_sampling, temperature) == 8 &&
                   offsetof(blurr_llm_sampling, top_k) == 12 && offsetof(blurr_llm_sampling, top_p) == 16,
               "blurr_llm_sampling layout");
#endif

int blurr_llm_create(const blurr_llm_config* cfg, int device, int max_batch, blurr_llm_t** out);
void blurr_llm_destroy(blurr_llm_t* h);

/* `key`: a state_dict key of transformers' LlamaForCausalLM ("model.embed_tokens.weight",
 * "model.layers.N.self_attn.{q,k,v,o}_proj.weight", "model.layers.N.mlp.{gate,up,down}_proj.weight",
 * "model.layers.N.{input,post_attention}_layernorm.weight", "model.norm.weight", "lm_head.weight"); the tensor is copied
 * and repacked (fused QKV, interleaved gate/up, tile-packed), so the caller may free it afterwards. */
int blurr_llm_set_weight(blurr_llm_t* h, const char* key, const void* dev_ptr, const int64_t* shape, int ndim);
/* cos / sin of `LlamaRotaryEmbedding.forward` for positions 0..n_pos-1, first half of the head dim only
 * ([n_pos][head_dim / 2] float32, values already cast to bf16 and back - the caller computes them with the model's own
 * `inv_freq` buffer so that a `.to(bfloat16)`-rounded buffer is reproduced). */
int blurr_llm_set_rope_table(blurr_llm_t* h, const float* cos_dev, const float* sin_dev, int n_pos);
int blurr_llm_finalize(blurr_llm_t* h);

/* rows[i] = embed_tokens[ids[i]]  (bf16 [n][hidden]) */
int blurr_llm_embed(blurr_llm_t* h, void* cuda_stream, const int64_t* ids, int n, void* rows_out);

/* Generation.  inputs_embeds: bf16 [batch][max_prompt_len][hidden]; max_prompt_len + n_new <= min(max_positions, 320).
 * prompt_lens: HOST int32 [batch] or NULL.  NULL: every sequence is max_prompt_len rows, no padding.  Otherwise
 * 1 <= prompt_lens[b] <= max_prompt_len and sequence b's prompt is rows 0 .. prompt_lens[b] - 1; rows t >= prompt_lens[b]
 * are ignored (never influence any output: they are zeroed on the device before the prefill, which runs over all
 * max_prompt_len rows), and token i of sequence b is generated at position prompt_lens[b] + i, so each sequence gets what
 * it would get alone.  A non-NULL prompt_lens takes this ragged schedule even when every length is max_prompt_len.
 * params: HOST [batch] or NULL.  NULL: greedy argmax.  Otherwise each token is drawn with its sequence's parameters,
 * checked on the host; a row with no finite positive mass (all -inf / NaN, a +inf logit, or a scaled score that
 * overflows) takes the greedy argmax and sets a sticky error that blurr_llm_check reports.
 * Writes out_ids int64 [batch][n_new]; if out_logits != NULL also the raw bf16 logits each token was chosen from,
 * [batch][n_new][vocab] (n_new <= 16).  A bad argument returns BLURR_ERR_INVALID and the handle keeps working.
 * The whole call (prefill, n_new - 1 decode steps, argmax or draw) is replayed as one CUDA graph per
 * (batch, max_prompt_len, n_new, logits, ragged, sampled): lengths and parameters are uploaded before the launch and read
 * by the kernels at run time, so one graph serves every vector of them; a sampled call launches as many kernels as a
 * greedy one. */
int blurr_llm_generate(blurr_llm_t* h, void* cuda_stream, int batch, int max_prompt_len, const void* inputs_embeds,
                       const int32_t* prompt_lens, const blurr_llm_sampling* params, int n_new, int64_t* out_ids,
                       void* out_logits);
/* One forward pass without lm_head, for OpenVLA-OFT's parallel decoding: the final-normed hidden rows of each sequence.
 * inputs_embeds bf16 [batch][max_len][hidden]; seq_lens, block_starts, row_starts: HOST int32 [batch] with
 * 1 <= seq_lens[b] <= max_len <= max_positions, 1 <= block_starts[b] <= seq_lens[b], 0 <= row_starts[b] and
 * row_starts[b] + n_rows <= seq_lens[b].  Rows t >= seq_lens[b] are pads: zeroed on the device, they never influence any
 * output.  Attention: query p of sequence b sees key k iff k < seq_lens[b] and (k <= p, or p >= block_starts[b] and
 * k >= block_starts[b]): causal over the prompt, bidirectional inside the block [block_starts[b], seq_lens[b]);
 * block_starts[b] == seq_lens[b] is plain causal attention.  Positions (RoPE) are 0..max_len-1 for every sequence.
 * Writes out_hidden bf16 [batch][n_rows][hidden]: rows row_starts[b] .. + n_rows - 1 of sequence b after the final
 * RMSNorm (transformers' LlamaModel.last_hidden_state).  Accepts up to max_positions: 384, 1024 on a handle created
 * with long_forward = 1, or 2048 with long_forward = 2 (past 384 keys the attention streams K and V through shared memory
 * with the same arithmetic; blurr_llm_generate stops at 320).  The
 * pass is replayed as one CUDA graph per (batch, max_len) whatever the lengths, starts and n_rows; the row copy to
 * out_hidden is one more kernel after it.  A bad argument returns BLURR_ERR_INVALID and the handle keeps working. */
int blurr_llm_forward_rows(blurr_llm_t* h, void* cuda_stream, int batch, int max_len, const void* inputs_embeds,
                           const int32_t* seq_lens, const int32_t* block_starts, const int32_t* row_starts, int n_rows,
                           void* out_hidden);
/* The sampler alone, on caller-made logits (usable before blurr_llm_finalize): logits bf16 [rows][ld], first `vocab`
 * columns used, rows <= max_batch, ld >= vocab; params HOST [rows]; `step` is the Philox counter.  Writes out_ids int64
 * [rows]; out_probs (may be NULL) fp32 [rows][vocab]: the probability each token was drawn with, 0 outside the kept set. */
int blurr_llm_sample(blurr_llm_t* h, void* cuda_stream, const void* logits, int rows, int ld, const blurr_llm_sampling* params,
                     int step, int64_t* out_ids, float* out_probs);
/* Options: "use_cuda_graph" (default 1), "trace" (default 0: every kernel stamps %globaltimer, see blurr_llm_trace_report). */
int blurr_llm_set_option(blurr_llm_t* h, const char* name, int64_t value);
/* Synchronises the stream; reports and clears device-side sticky errors (token id outside the table, a sampled row with
 * no finite positive mass, expired pipeline wait). */
int blurr_llm_check(blurr_llm_t* h, void* cuda_stream);
/* Text timeline of the last generate call under option "trace": one line per kernel, microseconds. */
int blurr_llm_trace_report(blurr_llm_t* h, char* buf, size_t buf_bytes);
/* Kernels launched by the last blurr_llm_generate / blurr_llm_forward_rows call, and the weight bytes one decode step streams. */
int64_t blurr_llm_last_launch_count(const blurr_llm_t* h);
int64_t blurr_llm_weight_bytes_per_token(const blurr_llm_t* h);

#ifdef __cplusplus
}
#endif
#endif /* BLURR_LLM_H_ */
