// Launchers of the bandwidth-bound and attention kernels (norm_consumers.cu, attention.cu,
// misc_kernels.cu).  All launchers are asynchronous on `stream` and return cudaGetLastError().
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace blurr {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------
// norm_consumers.cu — finish a GEMM (split-K sum, bias, residual / position add) and apply
// the following normalisation in one pass over the row.
// ---------------------------------------------------------------------------
enum AddMode { ADD_NONE = 0, ADD_RESIDUAL = 1, ADD_POSEMB = 2 };
enum NormMode { NORM_NONE = 0, NORM_RMS_GEMMA = 1, NORM_LAYERNORM = 2, NORM_RMS_LLAMA = 3 };   // Llama: bf16(w * bf16(x * rstd))

struct ConsumerArgs {
    const float* partial;   // [splitk][T][ldp] fp32 or nullptr (then x = res)
    int splitk, T, N, ldp;
    const bf16* bias;       // [N] or nullptr
    int add_mode;
    const bf16* res;        // [T][ldr]
    int ldr;
    const bf16* pos;        // [pos_rows][N]
    int pos_rows;
    float out_scale;        // applied as bf16(x * out_scale) after bias (1.0f = none)
    bf16* x_out;            // [T][ldx] stream after the add (nullable)
    int ldx;
    int norm_mode;
    const bf16* norm_w;
    const bf16* norm_b;
    float eps;
    bf16* xn_out;           // [T][ldn] normalised output (nullable)
    int ldn;
    unsigned long long* trace;   // in-graph timeline slot (launch.cuh) or nullptr
    // alternative to `partial` (batched episodes, one K slice): the Linear output itself, bf16(acc + bias),
    // written by the GEMM's store epilogue - half the bytes of the fp32 partial and no bias pass here
    const bf16* lin;        // [T][ldl] or nullptr
    int ldl;
    const bf16* col_scale;  // [N] or nullptr: per-column scale applied as bf16(x * g) after the bias (DINOv2 LayerScale)
    // output row map (0 = identity): row t is written to row t + (t / row_group) * row_extra + row_offset of x_out / xn_out
    // (ViT prefix tokens: the 256 patch rows of sample b land behind that sample's cls / register rows)
    int row_group, row_extra, row_offset;
    // FiLM (non-null film_gamma; 1024 or 1152 columns only): after the residual add, row t becomes
    // bf16(bf16(x * bf16(1 + gamma[c])) + beta[c]) with c = t / film_rows, before x_out and the norm statistics
    const bf16* film_gamma;  // [n_cond][film_ld]
    const bf16* film_beta;   // [n_cond][film_ld]
    int film_ld, film_rows;
};
cudaError_t launch_consumer(cudaStream_t stream, const ConsumerArgs& a);

// Element-wise finish without a norm: out = act(bf16(sum + bias)) * scale
enum ActMode { ACT_NONE = 0, ACT_SILU = 1 };
// GemmCall::glu_act also selects the EPI_GELU flavour: 0 tanh approximation (SigLIP, Gemma), 2 exact erf (DINOv2, nn.GELU())
enum GeluKind { GELU_TANH = 0, GELU_ERF = 2 };
cudaError_t launch_bias_act(cudaStream_t stream, const float* partial, int splitk, int T, int N, int ldp,
                            const bf16* bias, int act, float scale, bf16* out, int ldo);

// RoPE + KV-cache append: finishes the fused QKV GEMM for one mixture.
struct RopeKvArgs {
    const float* partial;   // [splitk][T][ldp], columns: q (n_heads*256) | k (256) | v (256)
    int splitk, T, ldp;
    int n_heads;            // 8
    int tokens_per_sample;  // 276 / 1 / 4
    const int64_t* position_ids;   // [B][tokens_per_sample]
    const float* cos_table; // [n_pos][128]  (values already rounded to bf16)
    const float* sin_table;
    int n_pos;
    bf16* q_out;            // [T][n_heads*256] (nullable: last-layer vlm/proprio need no query)
    bf16* k_cache;          // layer base: [B][n_slots][256]
    bf16* v_cache;
    int n_slots, slot_base;
    unsigned long long* trace;
    const bf16* lin;        // alternative to `partial`: the bf16 q|k|v Linear output [T][ldl]
    int ldl;
};
cudaError_t launch_rope_kv(cudaStream_t stream, const RopeKvArgs& a);

// ---------------------------------------------------------------------------
// attention.cu
// ---------------------------------------------------------------------------
// Arguments of the tiled (mma.sync) attention body, shared by SigLIP and the joint prefill.
struct AttnMmaArgs {
    const bf16* q; int ldq; int q_col0; int q_per_sample;
    const bf16* k; int ldk; int k_col0; int kv_per_sample;
    const bf16* v; int ldv; int v_col0;
    bf16* out; int ldo; int o_col0;
    int hd;            // real head dim (72 / 256)
    int head_stride_q; // column step between query heads (hd)
    int head_stride_kv;// column step between kv heads (0 for MQA)
    int n_keys;
    float scale;       // SigLIP: head_dim^-0.5
    const bf16* mask; long long mask_bstride, mask_rstride; int q_row_offset;
    // MQA few-query mode (mqa_nq > 0): the tile's rows enumerate (head, query) pairs of one sample,
    // pair p -> head p / mqa_nq, query p % mqa_nq; all pairs share the sample's single K/V head.
    int mqa_nq, mqa_heads;
    unsigned long long* trace;
};

// SigLIP MHA (siglip.py:133-152): qkv [T][3*hidden] with head_dim 72, no mask.
cudaError_t launch_siglip_attention(cudaStream_t stream, const bf16* qkv, int ld_qkv, int batch, int seq,
                                    int n_heads, int hidden, bf16* out, int ld_out,
                                    unsigned long long* trace = nullptr);

// Gemma joint attention, many queries (prefill): soft-clamped, additive mask, MQA.
struct JointAttnArgs {
    const bf16* q;          // [B*q_per_sample][n_heads*256]
    int q_per_sample;       // rows of this query segment per sample
    int q_row_offset;       // row of the first query in the mask (0 vlm, 276 proprio, 0 action)
    const bf16* k_cache;    // [B][n_slots][256]
    const bf16* v_cache;
    int n_slots, n_keys;    // keys 0..n_keys-1 are attended
    const bf16* mask;       // additive mask element (b, row, col) at mask[b*mask_bstride + row*mask_rstride + col]
    int64_t mask_bstride, mask_rstride;
    int batch, n_heads;
    bf16* out;              // [B*q_per_sample][n_heads*256]
    unsigned long long* trace;
};
cudaError_t launch_joint_attention_prefill(cudaStream_t stream, const JointAttnArgs& a);
// attention_tc.cu: the same operator on tcgen05 for batched episodes (one CTA = 128 (head, query) pairs)
void attn_set_tc(int mode);                      // -1 automatic (batch >= 8), 0 never, 1 whenever the shape allows
bool attn_tc_applies(const JointAttnArgs& a);
void attn_set_tc_fewq(int mode);                 // few-query attention on the tcgen05 kernel: 1 on, 0 / -1 off (default: measured slower at batch 1)
bool attn_tc_fewq_applies(const JointAttnArgs& a);
void attn_set_prefill_stream(int on);           // prefill attention of <= 2 waves of 16-row tiles as the streaming kernel (default 1)
void attn_set_siglip_stream(int on);            // SigLIP attention of <= 2 waves of 32-row tiles as the streaming kernel (default 1)
void attn_set_fewq_stream(int on);              // few-query attention as the streaming kernel (default 1) vs the mma.sync tile kernel
int attn_take_timeout_flag();
int attn_set_cta_trace(void* dev_ptr);          // per-CTA timeline of the tcgen05 attention kernel (attention_tc.cu)
// The AttnMmaArgs the two launchers above build (the step kernel runs the same bodies as work items).
AttnMmaArgs make_siglip_attn_args(const bf16* qkv, int ld_qkv, int seq, int n_heads, int hidden, bf16* out,
                                  int ld_out);
AttnMmaArgs make_prefill_attn_args(const JointAttnArgs& a);
AttnMmaArgs make_fewq_attn_args(const JointAttnArgs& a);
static constexpr int kAttnTileRows = 16;     // query rows per attention work item of the step kernel
int attn_tile_rows(int rows, int heads, int batch, int max_rows);   // tile rows the launchers pick
// Few queries per sample (proprio: 1, action: 4): bandwidth kernel over the KV cache.
cudaError_t launch_joint_attention_fewq(cudaStream_t stream, const JointAttnArgs& a);

// ---------------------------------------------------------------------------
// misc_kernels.cu
// ---------------------------------------------------------------------------
// pixel_values [B][3][224][224] (arbitrary strides, bf16) -> patches [B*256][ldp] with column
// c*196 + kh*14 + kw (the flattened Conv2d weight order); columns >= 588 untouched (zero).
cudaError_t launch_im2col(cudaStream_t stream, const bf16* pixels, int64_t sb, int64_t sc, int64_t sh,
                          int64_t sw, int batch, bf16* patches, int ldp);

// Merge text embeddings and projected image features (pizero.py:452-470) and apply the
// `embeds *= sqrt(hidden)` of JointModel.forward (joint_model.py:358-365).
cudaError_t launch_embed_merge(cudaStream_t stream, const int64_t* input_ids, int batch, int seq,
                               const bf16* embed_table, int64_t vocab, const bf16* img_feat, int n_img,
                               int hidden, int64_t image_token, int64_t pad_token, float inv_div,
                               float normalizer, bf16* out, int* err_flag);

// y[t][col_off + n] = bf16(bf16(sum_k x[t][k] W[n][k] + b[n]) * scale), K <= 8 (proprio_encoder,
// action_encoder.linear_1); optionally fills y[t][0..time_cols) with time_cond (the torch.cat).
cudaError_t launch_small_k_linear(cudaStream_t stream, const bf16* x, int T, int K, const bf16* W,
                                  const bf16* b, int N, float scale, bf16* y, int ldy, int col_off,
                                  const bf16* time_row, int time_cols);

// action_decoder + Euler update (pizero.py:536-537): a = bf16(a + bf16(dt * bf16(dot + b)))
cudaError_t launch_action_tail(cudaStream_t stream, const bf16* xn, int T, int hidden, const bf16* W,
                               const bf16* b, int action_dim, float dt, bf16* action, bf16* velocity_tap);

cudaError_t launch_clamp_copy(cudaStream_t stream, const bf16* src, bf16* dst, int n, int do_clamp, float clip,
                              const int* flag0 = nullptr, const int* flag1 = nullptr, const int* flag2 = nullptr);
// device addresses of the sticky pipeline time-out words (gemm_tc.cu / attention_tc.cu), or nullptr
const int* gemm_timeout_flag_ptr();
const int* attn_timeout_flag_ptr();

cudaError_t launch_rope_table(cudaStream_t stream, const float* inv_freq, int n_pos, float* cos_t,
                              float* sin_t);

// ---------------------------------------------------------------------------
// Llama-shaped decoder (llm_engine.cu / llm_kernels.cu): the OpenVLA-7B-shaped path
// ---------------------------------------------------------------------------
struct MhaAttnArgs {
    const bf16* q;            // [B * q_per_sample][n_heads * head_dim]
    int q_per_sample, q_pos0; // query row r of a sequence sits at key position q_pos0 + r (causal)
    const bf16* k_cache;      // [B][n_slots][n_kv_heads * head_dim], token-major
    const bf16* v_cache;
    int n_slots, n_keys;
    int batch, n_heads, n_kv_heads, head_dim;
    float scale;              // head_dim ** -0.5
    bf16* out;                // [B * q_per_sample][n_heads * head_dim]
    unsigned long long* trace;
    // decode of prompts of different lengths (q_per_sample 1): non-null -> sequence b attends keys 0 .. seq_len[b] + len_off - 1
    // (n_keys is then the batch's largest count); nullptr -> every sequence attends n_keys keys
    const int* seq_len; int len_off;
};
struct RopeMhaArgs;
// OFT's block-bidirectional prefill (attention.cu, up to 1024 keys; K and V resident up to 384): q_per_sample == n_keys rows per sequence from position
// 0; sequence b's query p sees key k iff k < seq_len[b] and (k <= p, or p >= block_start[b] and k >= block_start[b]).
// a.seq_len and block_start are device arrays [batch], read at run time; block_start[b] == seq_len[b] is plain causal.
cudaError_t launch_mha_block_attention(cudaStream_t stream, const MhaAttnArgs& a, const int* block_start);
// decode steps of <= 2 waves of (sequence, head) CTAs can do the new token's RoPE + cache append themselves
bool mha_decode_fuses_rope(const MhaAttnArgs& a);
cudaError_t launch_mha_attention(cudaStream_t stream, const MhaAttnArgs& a, const RopeMhaArgs* fused_rope = nullptr);

// q/k/v projection output -> RoPE (HF apply_rotary_pos_emb, rotate_half over head_dim / 2) -> q buffer and KV cache
struct RopeMhaArgs {
    const float* partial; int splitk;   // fp32 split-K partials [splitk][T][ldp] ...
    const bf16* lin; int ldl;           // ... or the bf16 linear output
    int T, ldp;
    int n_heads, n_kv_heads, head_dim;  // columns: q heads | k heads | v heads
    int tokens_per_seq, pos0;           // token t -> sequence t / tokens_per_seq, position pos0 + t % tokens_per_seq
    const float* cos_table; const float* sin_table; int n_pos;   // [n_pos][head_dim / 2], values already rounded to bf16
    bf16* q_out;                        // [T][n_heads * head_dim]
    bf16* k_cache; bf16* v_cache; int n_slots;      // [B][n_slots][n_kv_heads * head_dim]
    unsigned long long* trace;
    // non-null: token t sits at position (and cache slot) seq_len[s] + len_off + t % tokens_per_seq instead (ragged decode)
    const int* seq_len; int len_off;
};
cudaError_t launch_rope_mha(cudaStream_t stream, const RopeMhaArgs& a);
// rows[i] = table[ids[i]] (token embedding); ids outside [0, vocab) set *err_flag and read row 0
cudaError_t launch_embed_rows(cudaStream_t stream, const int64_t* ids, int n, const bf16* table, long long vocab, int width,
                              bf16* out, int* err_flag);
// dst[b] = src[(b * rows_per_seq + row) ] (the last prompt position of every sequence); with `seq_len` the row of sequence b
// is seq_len[b] - 1 instead of `row`
cudaError_t launch_gather_rows(cudaStream_t stream, const bf16* src, int batch, int rows_per_seq, int row, int width, bf16* dst,
                               const int* seq_len = nullptr);
// dst[b][i] = src[b * rows_per_seq + row_start[b] + i] for i < n_rows (row_start: device [batch], read at run time)
cudaError_t launch_gather_row_block(cudaStream_t stream, const bf16* src, int batch, int rows_per_seq, const int* row_start, int n_rows,
                                    int width, bf16* dst);
// tile-packed weight (gemm_tc.h) <- src rows [rows][cols]; destination row = r * row_mul + row_off (llm_engine.cu)
cudaError_t launch_pack_rows(cudaStream_t stream, const bf16* src, int rows, int cols, bf16* dst, int row_mul, int row_off, int kb_total);
// K slices of a few-token split-K GEMM over `tiles` weight tiles: as few, as full waves of 148 CTAs as possible (llm_engine.cu)
int pick_splitk_waves(int tiles, int kb_total);
// x[b][t][:] = 0 for seq_len[b] <= t < rows_per_seq: the pad rows of a ragged prompt batch (device lengths, read at run time)
cudaError_t launch_zero_pad_rows(cudaStream_t stream, bf16* x, int batch, int rows_per_seq, int width, const int* seq_len);
// ids[b] = argmax over logits[b][0..vocab) (lowest index among equal maxima, like torch.argmax on CPU)
cudaError_t launch_argmax_rows(cudaStream_t stream, const bf16* logits, int batch, int ld, int vocab, int64_t* ids,
                               int64_t* ids_copy, int copy_stride);
// Per-row parameters of the sampler; the layout of `blurr_llm_sampling` (include/blurr_llm.h, checked in llm_engine.cu).
struct SampleParams {
    uint64_t seed;
    float temperature;      // > 0, finite
    int32_t top_k;          // 0: off
    float top_p;            // in [0, 1]; 1: off
};
// ids[b] = one draw from softmax(top-p(top-k(logits[b][0..vocab) * (1 / T)))), HF's warper order, with Philox4x32-10
// (key = seed, counter = (step, 0, 0, 0)).  probs != nullptr: probs[b][0..vocab) = the probability each token was drawn
// with (0 outside the kept set).  A row with no finite positive mass takes the greedy argmax and sets *err_flag |= 2.
cudaError_t launch_sample_rows(cudaStream_t stream, const bf16* logits, int batch, int ld, int vocab, const SampleParams* params,
                               int step, int64_t* ids, int64_t* ids_copy, int copy_stride, float* probs, int* err_flag,
                               unsigned long long* trace);
// few-token GLU from the split-K partials of a gate/up projection with interleaved rows; act: 0 tanh GELU, 1 SiLU
cudaError_t launch_glu_partial(cudaStream_t stream, const float* partial, int splitk, int T, int Nw, int act, bf16* out, int ldo,
                               unsigned long long* trace = nullptr);

// dst[(b * rows + r) * ldd + c] = src[(b * src_rows_per_sample + row0 + r) * lds + c]  (patch-token features of a ViT)
cudaError_t launch_copy_rows(cudaStream_t stream, const bf16* src, int batch, int src_rows_per_sample, int row0, int rows, int width,
                             int lds, bf16* dst, int ldd);

// argument bundles of the small single-purpose kernels (engine.cu builds them once per op)
struct EmbedMergeArgs {
    const int64_t* ids; int seq; const bf16* table; long long vocab; const bf16* img; int n_img, hidden;
    long long image_token, pad_token; float inv_div, normalizer; bf16* out; int* err_flag;
};
struct SmallKArgs {
    const bf16* x; int T, K; const bf16* W; const bf16* bias; int N; float scale; bf16* y; int ldy, col_off;
    const bf16* time_row; int time_cols;
};
struct ActionTailArgs { const bf16* xn; int T, hidden; const bf16* W; const bf16* bias; int action_dim; float dt; bf16* action; bf16* vel_tap; };
struct ClampArgs { const bf16* src; bf16* dst; int n, do_clamp; float clip; };

}  // namespace blurr
