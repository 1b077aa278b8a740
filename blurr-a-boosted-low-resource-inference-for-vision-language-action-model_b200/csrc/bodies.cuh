// Device bodies of every non-GEMM kernel of the control step, shared by the stand-alone
// `__global__` wrappers (norm_consumers.cu, attention.cu, misc_kernels.cu) and by the persistent
// step kernel (step_kernel.cu), which runs them as work items between grid barriers.
//
// Loads of data produced earlier in the step go through L2 (`__ldcg`, `cp.async.cg`): inside the
// persistent kernel other SMs wrote it during the same launch and L1 is not coherent.  Weights,
// masks and position ids are constant for the launch and use ordinary loads.
#pragma once

#include "common.cuh"
#include "kernels.h"

namespace blurr {

__device__ __forceinline__ bf16 ldcg_bf16(const bf16* p) {
    const unsigned short u = __ldcg(reinterpret_cast<const unsigned short*>(p));
    return *reinterpret_cast<const bf16*>(&u);
}
__device__ __forceinline__ bf16x8 ldcg_bf16x8(const bf16* p) {
    const uint4 u = __ldcg(reinterpret_cast<const uint4*>(p));
    bf16x8 r;
    r.u[0] = u.x; r.u[1] = u.y; r.u[2] = u.z; r.u[3] = u.w;
    return r;
}

// ===========================================================================
// GEMM consumers (split-K sum, bias, residual / position add, norms), RoPE + KV append
// ===========================================================================
static constexpr int kRowThreads = 256;

template <int THREADS = kRowThreads>
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();               // protect `red` from the previous use
    if (l == 0) red[w] = v;
    __syncthreads();
    float t = (l < (THREADS / 32)) ? red[l] : 0.f;
    t = warp_sum(t);
    return t;                      // every thread holds the total
}

// sum of the split-K slices of 4 consecutive columns; up to 8 independent 16-byte loads in flight (the
// consumers are latency-bound: one round trip to L2 per batch of loads; 8 measured better than 4 and than
// 16 predicated loads - same-box A/B 4.263 / 4.210 / 4.285 ms per step), accumulated in slice order
__device__ __forceinline__ float4 sum_slices(const float* __restrict__ base, size_t slice_stride, int splitk) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int z = 0;
    for (; z + 8 <= splitk; z += 8) {
        float4 p[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) p[i] = __ldcg(reinterpret_cast<const float4*>(base + (z + i) * slice_stride));
#pragma unroll
        for (int i = 0; i < 8; ++i) { acc.x += p[i].x; acc.y += p[i].y; acc.z += p[i].z; acc.w += p[i].w; }   // fixed order z = 0, 1, 2, ...
    }
    if (z + 4 <= splitk) {
        float4 p[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) p[i] = __ldcg(reinterpret_cast<const float4*>(base + (z + i) * slice_stride));
#pragma unroll
        for (int i = 0; i < 4; ++i) { acc.x += p[i].x; acc.y += p[i].y; acc.z += p[i].z; acc.w += p[i].w; }
        z += 4;
    }
    for (; z < splitk; ++z) {
        const float4 p = __ldcg(reinterpret_cast<const float4*>(base + z * slice_stride));
        acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
    }
    return acc;
}

__device__ __forceinline__ float4 load_bf16x4(const bf16* p) {
    const uint2 u = __ldcg(reinterpret_cast<const uint2*>(p));
    const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void store_bf16x4(bf16* p, float4 v) {
    uint2 u;
    u.x = pack_bf16x2(v.x, v.y);
    u.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
}

// One CTA per token row; each thread owns VPT groups of 4 consecutive columns in registers.
// THREADS x VPT >= N / 4; the stand-alone kernel picks an exact fit (SigLIP's 1152 columns: 288 threads x 1),
// the persistent step kernel always runs 256 threads.
// Inputs of one row that a streaming launch fetched ahead of time (bf16 hand-off mode only).
template <int VPT>
struct ConsumerRowIn { uint2 lin[VPT], add[VPT]; };
__device__ __forceinline__ float4 unpack_bf16x4(uint2 u) {
    const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
}
template <int VPT, int THREADS>
__device__ __forceinline__ void consumer_prefetch(const ConsumerArgs& a, const int t, ConsumerRowIn<VPT>& in) {
    const int nvec = a.N >> 2;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = threadIdx.x + i * THREADS;
        in.lin[i] = make_uint2(0u, 0u); in.add[i] = make_uint2(0u, 0u);
        if (v >= nvec) continue;
        const int n = v << 2;
        in.lin[i] = __ldcg(reinterpret_cast<const uint2*>(a.lin + static_cast<size_t>(t) * a.ldl + n));
        if (a.add_mode == ADD_RESIDUAL) in.add[i] = __ldcg(reinterpret_cast<const uint2*>(a.res + static_cast<size_t>(t) * a.ldr + n));
        else if (a.add_mode == ADD_POSEMB) in.add[i] = __ldcg(reinterpret_cast<const uint2*>(a.pos + static_cast<size_t>(t % a.pos_rows) * a.N + n));
    }
}

// FILM: the FiLM step of the ViT towers (ConsumerArgs::film_gamma) - a compile-time variant, so that the instantiations
// without it keep their code
template <int VPT, int THREADS = kRowThreads, bool PRELOADED = false, bool FILM = false>
__device__ __forceinline__ void consumer_body(const ConsumerArgs& a, const int t, const ConsumerRowIn<VPT>* pre = nullptr) {
    __shared__ float red[(THREADS + 31) / 32];
    const int nvec = a.N >> 2;
    const int to = a.row_group > 0 ? t + (t / a.row_group) * a.row_extra + a.row_offset : t;     // output row
    float4 x[VPT];
    float lsum = 0.f, lsq = 0.f;
    // Everything that does not depend on the partial sums is requested first - residual / position row, norm weights -
    // so the row costs one round trip to L2 plus the reduction instead of three dependent ones (the kernel is latency-bound).
    const bool want_norm = a.norm_mode != NORM_NONE && a.xn_out != nullptr;
    const bool from_res = a.partial == nullptr && a.lin == nullptr;
    uint2 pf_add[VPT], pf_w[VPT], pf_b[VPT];
    uint2 pf_fg[VPT], pf_fb[VPT];          // FiLM gamma / beta of the row's condition
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = threadIdx.x + i * THREADS;
        pf_add[i] = make_uint2(0u, 0u); pf_w[i] = make_uint2(0u, 0u); pf_b[i] = make_uint2(0u, 0u);
        if (v >= nvec) continue;
        const int n = v << 2;
        if constexpr (FILM) {
            const size_t c = static_cast<size_t>(t / a.film_rows) * a.film_ld + n;
            pf_fg[i] = __ldcg(reinterpret_cast<const uint2*>(a.film_gamma + c));
            pf_fb[i] = __ldcg(reinterpret_cast<const uint2*>(a.film_beta + c));
        }
        if (!PRELOADED || from_res) {
            if (from_res || a.add_mode == ADD_RESIDUAL) pf_add[i] = __ldcg(reinterpret_cast<const uint2*>(a.res + static_cast<size_t>(t) * a.ldr + n));
            else if (a.add_mode == ADD_POSEMB) pf_add[i] = __ldcg(reinterpret_cast<const uint2*>(a.pos + static_cast<size_t>(t % a.pos_rows) * a.N + n));
        }
        if (want_norm) {
            pf_w[i] = __ldcg(reinterpret_cast<const uint2*>(a.norm_w + n));
            if (a.norm_mode == NORM_LAYERNORM) pf_b[i] = __ldcg(reinterpret_cast<const uint2*>(a.norm_b + n));
        }
    }
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = threadIdx.x + i * THREADS;
        x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (v >= nvec) continue;
        const int n = v << 2;
        float4 val;
        if (a.partial != nullptr || a.lin != nullptr) {
            if (PRELOADED) {
                val = unpack_bf16x4(pre->lin[i]);
            } else if (a.lin != nullptr) {
                val = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + n);      // already bf16(acc + bias)
            } else {
                float4 acc = sum_slices(a.partial + static_cast<size_t>(t) * a.ldp + n,
                                        static_cast<size_t>(a.T) * a.ldp, a.splitk);
                if (a.bias != nullptr) {
                    const float4 b = load_bf16x4(a.bias + n);
                    acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
                }
                val = make_float4(bf16_round(acc.x), bf16_round(acc.y), bf16_round(acc.z), bf16_round(acc.w));
            }
            if (a.out_scale != 1.0f)
                val = make_float4(bf16_round(val.x * a.out_scale), bf16_round(val.y * a.out_scale),
                                  bf16_round(val.z * a.out_scale), bf16_round(val.w * a.out_scale));
            if (a.col_scale != nullptr) {
                const float4 gsc = load_bf16x4(a.col_scale + n);
                val = make_float4(bf16_round(val.x * gsc.x), bf16_round(val.y * gsc.y), bf16_round(val.z * gsc.z),
                                  bf16_round(val.w * gsc.w));
            }
            if (a.add_mode == ADD_RESIDUAL) {
                const float4 r = PRELOADED ? unpack_bf16x4(pre->add[i]) : unpack_bf16x4(pf_add[i]);
                val = make_float4(bf16_round(r.x + val.x), bf16_round(r.y + val.y), bf16_round(r.z + val.z),
                                  bf16_round(r.w + val.w));
            } else if (a.add_mode == ADD_POSEMB) {
                const float4 r = PRELOADED ? unpack_bf16x4(pre->add[i]) : unpack_bf16x4(pf_add[i]);
                val = make_float4(bf16_round(val.x + r.x), bf16_round(val.y + r.y), bf16_round(val.z + r.z),
                                  bf16_round(val.w + r.w));
            }
        } else {
            val = unpack_bf16x4(pf_add[i]);
        }
        if constexpr (FILM) {
            // torch's bf16 `x * (1 + gamma) + beta`: every operation rounded to bf16
            const float4 g = unpack_bf16x4(pf_fg[i]), be = unpack_bf16x4(pf_fb[i]);
            val = make_float4(bf16_round(bf16_round(val.x * bf16_round(1.0f + g.x)) + be.x),
                              bf16_round(bf16_round(val.y * bf16_round(1.0f + g.y)) + be.y),
                              bf16_round(bf16_round(val.z * bf16_round(1.0f + g.z)) + be.z),
                              bf16_round(bf16_round(val.w * bf16_round(1.0f + g.w)) + be.w));
        }
        if (a.x_out != nullptr) store_bf16x4(a.x_out + static_cast<size_t>(to) * a.ldx + n, val);
        x[i] = val;
        lsum += (val.x + val.y) + (val.z + val.w);
        lsq += (val.x * val.x + val.y * val.y) + (val.z * val.z + val.w * val.w);
    }
    if (a.norm_mode == NORM_NONE || a.xn_out == nullptr) return;

    if (a.norm_mode == NORM_RMS_GEMMA || a.norm_mode == NORM_RMS_LLAMA) {
        const float ms = block_sum<THREADS>(lsq, red) / static_cast<float>(a.N);
        const float r = rsqrtf(ms + a.eps);
        const bool llama = a.norm_mode == NORM_RMS_LLAMA;
#pragma unroll
        for (int i = 0; i < VPT; ++i) {
            const int v = threadIdx.x + i * THREADS;
            if (v >= nvec) continue;
            const int n = v << 2;
            const float4 w = unpack_bf16x4(pf_w[i]);
            // Gemma: (x * rstd) * (1 + w) in fp32, one rounding.  Llama (HF LlamaRMSNorm.forward): weight * (x * rstd).to(bf16)
            const float4 y = llama
                ? make_float4(w.x * bf16_round(x[i].x * r), w.y * bf16_round(x[i].y * r), w.z * bf16_round(x[i].z * r),
                              w.w * bf16_round(x[i].w * r))
                : make_float4((x[i].x * r) * (1.0f + w.x), (x[i].y * r) * (1.0f + w.y),
                              (x[i].z * r) * (1.0f + w.z), (x[i].w * r) * (1.0f + w.w));
            store_bf16x4(a.xn_out + static_cast<size_t>(to) * a.ldn + n, y);
        }
    } else {
        const float mean = block_sum<THREADS>(lsum, red) / static_cast<float>(a.N);
        float lvar = 0.f;
#pragma unroll
        for (int i = 0; i < VPT; ++i) {
            const int v = threadIdx.x + i * THREADS;
            if (v >= nvec) continue;
            const float dx = x[i].x - mean, dy = x[i].y - mean, dz = x[i].z - mean, dw = x[i].w - mean;
            lvar += (dx * dx + dy * dy) + (dz * dz + dw * dw);
        }
        const float var = block_sum<THREADS>(lvar, red) / static_cast<float>(a.N);
        const float rstd = rsqrtf(var + a.eps);
#pragma unroll
        for (int i = 0; i < VPT; ++i) {
            const int v = threadIdx.x + i * THREADS;
            if (v >= nvec) continue;
            const int n = v << 2;
            const float4 w = unpack_bf16x4(pf_w[i]), b = unpack_bf16x4(pf_b[i]);
            const float4 y = make_float4((x[i].x - mean) * rstd * w.x + b.x, (x[i].y - mean) * rstd * w.y + b.y,
                                         (x[i].z - mean) * rstd * w.z + b.z, (x[i].w - mean) * rstd * w.w + b.w);
            store_bf16x4(a.xn_out + static_cast<size_t>(to) * a.ldn + n, y);
        }
    }
}

__device__ __forceinline__ void bias_act_body(const float* partial, int splitk, int T, int N, int ldp,
                                              const bf16* bias, int act, float scale, bf16* out, int ldo,
                                              const int bx) {
    const int idx = bx * 256 + threadIdx.x;
    const int nvec = N >> 2;
    if (idx >= T * nvec) return;
    const int t = idx / nvec, n = (idx - t * nvec) << 2;
    float4 acc = sum_slices(partial + static_cast<size_t>(t) * ldp + n, static_cast<size_t>(T) * ldp, splitk);
    if (bias != nullptr) {
        const float4 b = load_bf16x4(bias + n);
        acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
    }
    float v[4] = {bf16_round(acc.x), bf16_round(acc.y), bf16_round(acc.z), bf16_round(acc.w)};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (act == ACT_SILU) v[i] = bf16_round(silu_f32(v[i]));
        if (scale != 1.0f) v[i] = bf16_round(v[i] * scale);
    }
    store_bf16x4(out + static_cast<size_t>(t) * ldo + n, make_float4(v[0], v[1], v[2], v[3]));
}

// One CTA per token.  Work items: for every rotated head (queries + the key head) 32 pairs of
// float4 column groups (dims [4j,4j+4) and [128+4j,128+4j+4): the rotate_half partners), plus 64
// plain float4 groups of the value head.
// The bf16 inputs and the position of one work item of one row, fetched ahead of time by the streaming launch.
struct RopeItemIn { uint2 x1, x2; long long pos; };
__device__ __forceinline__ void rope_prefetch(const RopeKvArgs& a, const int t, RopeItemIn& in) {
    const int b = t / a.tokens_per_sample, i = t - b * a.tokens_per_sample;
    in.pos = __ldcg(a.position_ids + static_cast<size_t>(b) * a.tokens_per_sample + i);
    const int n_rot = (a.n_heads + 1) * 32;
    const int it = threadIdx.x;
    in.x1 = make_uint2(0u, 0u); in.x2 = make_uint2(0u, 0u);
    if (it < n_rot) {
        const int h = it >> 5, j = (it & 31) << 2;
        if (h < a.n_heads && a.q_out == nullptr) return;
        in.x1 = __ldcg(reinterpret_cast<const uint2*>(a.lin + static_cast<size_t>(t) * a.ldl + h * 256 + j));
        in.x2 = __ldcg(reinterpret_cast<const uint2*>(a.lin + static_cast<size_t>(t) * a.ldl + h * 256 + 128 + j));
    } else if (it < n_rot + 64) {
        const int j = (it - n_rot) << 2;
        in.x1 = __ldcg(reinterpret_cast<const uint2*>(a.lin + static_cast<size_t>(t) * a.ldl + (a.n_heads + 1) * 256 + j));
    }
}

template <bool PRELOADED = false>
__device__ __forceinline__ void rope_kv_body(const RopeKvArgs& a, const int t, const RopeItemIn* pre = nullptr) {
    const int b = t / a.tokens_per_sample, i = t - b * a.tokens_per_sample;
    long long pos = PRELOADED ? pre->pos : __ldcg(a.position_ids + static_cast<size_t>(b) * a.tokens_per_sample + i);
    if (pos < 0) pos = 0;
    if (pos >= a.n_pos) pos = a.n_pos - 1;   // host validates the range; never read out of bounds
    const int slot = a.slot_base + i;
    const size_t cache_row = (static_cast<size_t>(b) * a.n_slots + slot) * 256;
    const float* prow = a.partial + static_cast<size_t>(t) * a.ldp;
    const size_t sstride = static_cast<size_t>(a.T) * a.ldp;
    const int n_rot = (a.n_heads + 1) * 32;
    const int n_items = n_rot + 64;
    for (int it = threadIdx.x; it < n_items; it += blockDim.x) {
        if (it < n_rot) {
            const int h = it >> 5, j = (it & 31) << 2;             // head, first dim of the group
            if (h < a.n_heads && a.q_out == nullptr) continue;
            float4 x1, x2;
            if (PRELOADED) {
                x1 = unpack_bf16x4(pre->x1);
                x2 = unpack_bf16x4(pre->x2);
            } else if (a.lin != nullptr) {
                x1 = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + h * 256 + j);
                x2 = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + h * 256 + 128 + j);
            } else {
                x1 = sum_slices(prow + h * 256 + j, sstride, a.splitk);
                x2 = sum_slices(prow + h * 256 + 128 + j, sstride, a.splitk);
            }
            const float4 cs = *reinterpret_cast<const float4*>(a.cos_table + pos * 128 + j);
            const float4 sn = *reinterpret_cast<const float4*>(a.sin_table + pos * 128 + j);
            float u1[4] = {bf16_round(x1.x), bf16_round(x1.y), bf16_round(x1.z), bf16_round(x1.w)};
            float u2[4] = {bf16_round(x2.x), bf16_round(x2.y), bf16_round(x2.z), bf16_round(x2.w)};
            const float c[4] = {cs.x, cs.y, cs.z, cs.w}, s[4] = {sn.x, sn.y, sn.z, sn.w};
            float y1[4], y2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                // x*cos + rotate_half(x)*sin, every op rounded to bf16 (utils.py:11-16)
                y1[e] = bf16_round(bf16_round(u1[e] * c[e]) + bf16_round(-u2[e] * s[e]));
                y2[e] = bf16_round(bf16_round(u2[e] * c[e]) + bf16_round(u1[e] * s[e]));
            }
            bf16* dst = (h < a.n_heads) ? a.q_out + static_cast<size_t>(t) * (a.n_heads * 256) + h * 256
                                        : a.k_cache + cache_row;
            store_bf16x4(dst + j, make_float4(y1[0], y1[1], y1[2], y1[3]));
            store_bf16x4(dst + 128 + j, make_float4(y2[0], y2[1], y2[2], y2[3]));
        } else {
            const int j = (it - n_rot) << 2;
            const float4 v = PRELOADED ? unpack_bf16x4(pre->x1)
                             : a.lin != nullptr ? load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + (a.n_heads + 1) * 256 + j)
                                                : sum_slices(prow + (a.n_heads + 1) * 256 + j, sstride, a.splitk);
            store_bf16x4(a.v_cache + cache_row + j,
                         make_float4(bf16_round(v.x), bf16_round(v.y), bf16_round(v.z), bf16_round(v.w)));
        }
    }
}


// ===========================================================================
// attention
// ===========================================================================
static constexpr int kAttnThreads = 256;   // 8 warps per attention tile
static constexpr int kBK = 64;             // keys per streamed block
static constexpr int kAttnMaxBlocks = 5;   // up to 320 keys resident in shared memory
static constexpr int kAttnMaxBlocksWide = 6;   // MODE 3 (block-bidirectional prefill): up to 384 keys

__device__ __forceinline__ void attn_bar_sync() { __syncthreads(); }

template <int N>
__device__ __forceinline__ void cp_async_wait_dyn(int pending) {
    // cp.async.wait_group needs an immediate: wait until at most `pending` groups are in flight
    if (pending <= 0) cp_async_wait<0>();
    else if (pending == 1) cp_async_wait<1>();
    else if (pending == 2) cp_async_wait<2>();
    else if (pending == 3) cp_async_wait<3>();
    else cp_async_wait<4>();
}

// dst: [nrows][LDS]; 16-byte chunks; rows >= nrows_valid and columns >= hd are zero-filled
template <int LDS, int CH>
__device__ __forceinline__ void load_rows_async(bf16* dst, const bf16* src, int ld, int row0, int nrows,
                                                int nrows_valid, int hd) {
    for (int idx = threadIdx.x; idx < nrows * CH; idx += kAttnThreads) {
        const int r = idx / CH, c = idx - r * CH;
        const bool valid = (row0 + r < nrows_valid) && (c * 8 < hd);
        const bf16* g = valid ? (src + static_cast<size_t>(row0 + r) * ld + c * 8) : src;
        cp_async_16(dst + r * LDS + c * 8, g, valid);
    }
}

// One tile = 16 query rows of one (sample, head); 4 warps split the keys (logits) / the head dim
// (output).  All K blocks are requested at once (one cp.async group per 64-key block) and consumed
// as they land; the V blocks are requested into the same buffers as soon as the logits are done, so
// their latency hides behind the softmax.
// MODE: 0 = logits * scale (SigLIP), 1 = Gemma chain (1/16, soft-clamp, additive mask), 2 = logits * scale with the
// causal mask computed from positions (Llama-style MHA: query row r sits at key position q_row_offset + r), 3 = MODE 2's
// logits with a per-sequence rule read from `seq_len[b]` / `block_start[b]` (OFT's action block): query p sees key k iff
// k < seq_len and (k <= p, or p >= block_start and k >= block_start).  MAXB: key blocks a row's softmax holds.
template <int HD_PAD, int BM, int MODE, int MAXB = kAttnMaxBlocks>
__device__ __forceinline__ void attn_mma_body(const AttnMmaArgs& a, uint8_t* smem_attn, const int qt, const int h,
                                              const int b, const int* seq_len = nullptr, const int* block_start = nullptr) {
    // BM query rows per tile: 16 at batch 1 (most tiles, least latency), 32/64 for batched episodes
    // (K/V of a head are re-read once per tile, so larger tiles cut the L2 -> SM traffic)
    constexpr int WR = BM / 16;                 // row groups
    constexpr int WC = (kAttnThreads / 32) / WR;   // column groups
    constexpr int KPW = kBK / WC;               // keys per warp per block
    constexpr int NT_S = KPW / 8;               // logit n-tiles per warp per block
    constexpr int NT_ALL = HD_PAD / 8;          // output n-tiles over the head dim
    constexpr int NT_PV = (NT_ALL + WC - 1) / WC;
    constexpr int NP_PV = (NT_PV + 1) / 2;
    constexpr int CH = HD_PAD / 8;              // 16-byte chunks per row that carry data
    constexpr int LDS_MIN = WC * NP_PV * 16 > HD_PAD ? WC * NP_PV * 16 : HD_PAD;
    constexpr int LDS = LDS_MIN + 8;            // smem row stride (elements), conflict-free for ldmatrix
    // causal (MODE 2): keys past the tile's last query position are masked for every row - never load them
    int n_keys_tile = MODE == 2 ? min(a.n_keys, a.q_row_offset + qt * BM + BM) : a.n_keys;
    int blk_len = 0, blk0 = 0;
    if constexpr (MODE == 3) {
        // keys past the sequence are never seen; a tile without a query in the action block needs the causal bound only
        blk_len = max(1, min(seq_len[b], a.n_keys));           // the host validates both; never read out of range
        blk0 = max(1, min(block_start[b], blk_len));
        const int last_q = a.q_row_offset + qt * BM + BM - 1;
        n_keys_tile = min(blk_len, last_q >= blk0 ? a.n_keys : last_q + 1);
    }
    const int nkb = (n_keys_tile + kBK - 1) / kBK;
    const int ldl = nkb * kBK + 8;              // logit row stride (elements)
    bf16* Qs = reinterpret_cast<bf16*>(smem_attn);
    bf16* KVs = Qs + BM * LDS;                  // nkb buffers of [64][LDS]
    bf16* Ls = KVs + nkb * kBK * LDS;           // [BM][ldl]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp % WR, wc = warp / WR;
    const int q_row0 = qt * BM;

    const bf16* qbase = a.q + static_cast<size_t>(b) * a.q_per_sample * a.ldq + a.q_col0 + h * a.head_stride_q;
    const bf16* kbase = a.k + static_cast<size_t>(b) * a.kv_per_sample * a.ldk + a.k_col0 + h * a.head_stride_kv;
    const bf16* vbase = a.v + static_cast<size_t>(b) * a.kv_per_sample * a.ldv + a.v_col0 + h * a.head_stride_kv;

    // query rows -> smem (zero-filled past the valid rows / head dim)
    const int n_rows_valid = a.mqa_nq > 0 ? a.mqa_heads * a.mqa_nq : a.q_per_sample;
    for (int idx = threadIdx.x; idx < BM * CH; idx += kAttnThreads) {
        const int r = idx / CH, c = idx - r * CH;
        const int row = q_row0 + r;
        const bool valid = (row < n_rows_valid) && (c * 8 < a.hd);
        const bf16* g = qbase;
        if (valid) {
            if (a.mqa_nq > 0)
                g = a.q + (static_cast<size_t>(b) * a.mqa_nq + row % a.mqa_nq) * a.ldq + (row / a.mqa_nq) * a.head_stride_q + c * 8;
            else
                g = qbase + static_cast<size_t>(row) * a.ldq + c * 8;
        }
        cp_async_16(Qs + r * LDS + c * 8, g, valid);
    }
    for (int kb = 0; kb < nkb; ++kb) {
        load_rows_async<LDS, CH>(KVs + kb * kBK * LDS, kbase, a.ldk, kb * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
    }

    // ---------------- phase S: logits = chain(Q K^T) -> Ls (bf16) ----------------
    for (int kb = 0; kb < nkb; ++kb) {
        const bf16* Kcur = KVs + kb * kBK * LDS;
        cp_async_wait_dyn<0>(nkb - 1 - kb);
        attn_bar_sync();

        float acc[NT_S][4];
#pragma unroll
        for (int i = 0; i < NT_S; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

#pragma unroll
        for (int kk = 0; kk < HD_PAD / 16; ++kk) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(Qs + (wr * 16 + (lane & 15)) * LDS + kk * 16 + (lane >> 4) * 8));
            if (NT_S == 1) {
                // one 8-key n-tile per warp: matrices (keys, dims k0..7) and (keys, dims k8..15)
                uint32_t bfr[2];
                const int key = wc * KPW + (lane & 7);
                ldmatrix_x2(bfr, smem_u32(Kcur + key * LDS + kk * 16 + ((lane >> 3) & 1) * 8));
                mma_bf16_16816(acc[0], af, bfr[0], bfr[1]);
            } else {
#pragma unroll
                for (int np = 0; np < NT_S / 2; ++np) {
                    uint32_t bfr[4];
                    const int mi = lane >> 3;
                    const int key = wc * KPW + np * 16 + (mi >> 1) * 8 + (lane & 7);
                    ldmatrix_x4(bfr, smem_u32(Kcur + key * LDS + kk * 16 + (mi & 1) * 8));
                    mma_bf16_16816(acc[np * 2 + 0], af, bfr[0], bfr[1]);
                    mma_bf16_16816(acc[np * 2 + (NT_S > 1 ? 1 : 0)], af, bfr[2], bfr[3]);
                }
            }
        }
        // epilogue of this key block: rounding chain, write bf16 logits
#pragma unroll
        for (int nt = 0; nt < NT_S; ++nt) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = wr * 16 + (lane >> 2) + half * 8;
                const int kcol = kb * kBK + wc * KPW + nt * 8 + (lane & 3) * 2;
                float s0 = bf16_round(acc[nt][half * 2 + 0]);
                float s1 = bf16_round(acc[nt][half * 2 + 1]);
                if (MODE == 1) {
                    s0 = s0 * 0.0625f;                           // / sqrt(256): exact, stays a bf16 value
                    s1 = s1 * 0.0625f;
                    const float inv50 = 1.0f / 50.0f;            // ATen: a * (1 / b) for a scalar divisor
                    s0 = bf16_round(s0 * inv50);
                    s1 = bf16_round(s1 * inv50);
                    s0 = bf16_round(tanhf(s0));
                    s1 = bf16_round(tanhf(s1));
                    s0 = bf16_round(s0 * 50.0f);
                    s1 = bf16_round(s1 * 50.0f);
                    const int qr = q_row0 + r;
                    if (qr < n_rows_valid) {
                        const int mr = a.mqa_nq > 0 ? qr % a.mqa_nq : qr;
                        const bf16* mrow = a.mask + static_cast<size_t>(b) * a.mask_bstride +
                                           static_cast<size_t>(a.q_row_offset + mr) * a.mask_rstride;
                        if (kcol < n_keys_tile) s0 = bf16_round(s0 + bf2f(mrow[kcol]));
                        if (kcol + 1 < n_keys_tile) s1 = bf16_round(s1 + bf2f(mrow[kcol + 1]));
                    }
                } else {
                    s0 = bf16_round(s0 * a.scale);
                    s1 = bf16_round(s1 * a.scale);
                    if (MODE == 2) {
                        // HF adds finfo.min above the diagonal; after the fp32 softmax that is a zero, like -inf here
                        const int qpos = a.q_row_offset + q_row0 + r;
                        if (kcol > qpos) s0 = -INFINITY;
                        if (kcol + 1 > qpos) s1 = -INFINITY;
                    }
                    if constexpr (MODE == 3) {
                        const int qpos = a.q_row_offset + q_row0 + r;
                        const bool in_blk = qpos >= blk0;
                        if (!(kcol < blk_len && (kcol <= qpos || (in_blk && kcol >= blk0)))) s0 = -INFINITY;
                        if (!(kcol + 1 < blk_len && (kcol + 1 <= qpos || (in_blk && kcol + 1 >= blk0)))) s1 = -INFINITY;
                    }
                }
                *reinterpret_cast<uint32_t*>(Ls + r * ldl + kcol) = pack_bf16x2(s0, s1);
            }
        }
    }
    attn_bar_sync();   // every warp is done with the K blocks; all logits are visible

    // V blocks into the same buffers; the softmax below runs while they arrive
    for (int kb = 0; kb < nkb; ++kb) {
        load_rows_async<LDS, CH>(KVs + kb * kBK * LDS, vbase, a.ldv, kb * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
    }

    // ---------------- softmax: fp32 over bf16 logits, result bf16 in place ----------------
    for (int rr = 0; rr < BM / 8; ++rr) {
        bf16* lrow = Ls + (warp * (BM / 8) + rr) * ldl;
        constexpr int PER_LANE = MAXB * kBK / 32;               // 10 logits per lane (12 at 384 keys)
        float x[PER_LANE];
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int c = lane + i * 32;
            x[i] = (c < n_keys_tile) ? bf2f(lrow[c]) : -INFINITY;
            m = fmaxf(m, x[i]);
        }
        m = warp_max(m);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int c = lane + i * 32;
            x[i] = (c < n_keys_tile) ? expf(x[i] - m) : 0.f;
            sum += x[i];
        }
        sum = warp_sum(sum);
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int c = lane + i * 32;
            if (c < nkb * kBK) lrow[c] = f2bf(x[i] / sum);
        }
    }

    // ---------------- phase PV ----------------
    float oacc[NP_PV * 2][4];
#pragma unroll
    for (int i = 0; i < NP_PV * 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) oacc[i][j] = 0.f;
    const int nt0 = wc * NT_PV;                 // first output n-tile of this warp

    for (int kb = 0; kb < nkb; ++kb) {
        const bf16* Vcur = KVs + kb * kBK * LDS;
        cp_async_wait_dyn<0>(nkb - 1 - kb);
        attn_bar_sync();                        // (kb == 0: also publishes the probabilities)
#pragma unroll
        for (int kk = 0; kk < kBK / 16; ++kk) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(Ls + (wr * 16 + (lane & 15)) * ldl + kb * kBK + kk * 16 + (lane >> 4) * 8));
#pragma unroll
            for (int np = 0; np < NP_PV; ++np) {
                if ((nt0 + np * 2) >= NT_ALL) continue;          // warp past the head dim
                uint32_t bfr[4];
                const int mi = lane >> 3;
                const int key = kk * 16 + (mi & 1) * 8 + (lane & 7);
                const int dim = (nt0 + np * 2) * 8 + (mi >> 1) * 8;
                ldmatrix_x4_trans(bfr, smem_u32(Vcur + key * LDS + dim));
                mma_bf16_16816(oacc[np * 2 + 0], af, bfr[0], bfr[1]);
                if (np * 2 + 1 < NT_PV && nt0 + np * 2 + 1 < NT_ALL)
                    mma_bf16_16816(oacc[np * 2 + 1], af, bfr[2], bfr[3]);
            }
        }
    }

    // ---------------- store ----------------
    bf16* obase = a.out + static_cast<size_t>(b) * a.q_per_sample * a.ldo + a.o_col0 + h * a.head_stride_q;
#pragma unroll
    for (int nt = 0; nt < NT_PV; ++nt) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = q_row0 + wr * 16 + (lane >> 2) + half * 8;
            const int dim = (nt0 + nt) * 8 + (lane & 3) * 2;
            if (r < n_rows_valid && dim < a.hd) {
                bf16* dst = (a.mqa_nq > 0)
                    ? a.out + (static_cast<size_t>(b) * a.mqa_nq + r % a.mqa_nq) * a.ldo + (r / a.mqa_nq) * a.head_stride_q
                    : obase + static_cast<size_t>(r) * a.ldo;
                *reinterpret_cast<uint32_t*>(dst + dim) = pack_bf16x2(oacc[nt][half * 2 + 0], oacc[nt][half * 2 + 1]);
            }
        }
    }
    attn_bar_sync();   // shared memory is reused by the caller's next work item
}

template <int HD_PAD, int BM>
inline size_t attn_smem_bytes(int n_keys) {
    constexpr int WC = (kAttnThreads / 32) / (BM / 16);
    constexpr int NT_PV = (HD_PAD / 8 + WC - 1) / WC;
    constexpr int NP_PV = (NT_PV + 1) / 2;
    constexpr int LDS_MIN = WC * NP_PV * 16 > HD_PAD ? WC * NP_PV * 16 : HD_PAD;
    constexpr int LDS = LDS_MIN + 8;
    const int nkb = (n_keys + kBK - 1) / kBK;
    return static_cast<size_t>(BM + nkb * kBK) * LDS * 2 + static_cast<size_t>(BM) * (nkb * kBK + 8) * 2;
}

// ===========================================================================
// small kernels at the edges of the step
// ===========================================================================
__device__ __forceinline__ void im2col_body(const bf16* px, long long sb, long long sc, long long sh, long long sw,
                                            bf16* patches, int ldp, const int p, const int b) {
    // p: patch index within the image, row-major 16x16
    const int ph = p >> 4, pw = p & 15;
    bf16* dst = patches + (static_cast<size_t>(b) * 256 + p) * ldp;
    for (int idx = threadIdx.x; idx < 588; idx += blockDim.x) {
        const int c = idx / 196, rem = idx - c * 196;
        const int kh = rem / 14, kw = rem - kh * 14;
        dst[idx] = px[b * sb + c * sc + static_cast<long long>(ph * 14 + kh) * sh +
                      static_cast<long long>(pw * 14 + kw) * sw];
    }
}

__device__ __forceinline__ void embed_merge_body(const int64_t* ids, int seq, const bf16* table, long long vocab,
                                                 const bf16* img, int n_img, int hidden, long long image_token,
                                                 long long pad_token, float inv_div, float normalizer, bf16* out,
                                                 int* err_flag, const int pos, const int b) {
    __shared__ int s_rank;
    __syncthreads();                     // s_rank may still be in use by the previous work item
    const int64_t* row = ids + static_cast<size_t>(b) * seq;
    const long long id = __ldcg(row + pos);
    bf16* dst = out + (static_cast<size_t>(b) * seq + pos) * hidden;
    if (id == image_token) {
        if (threadIdx.x == 0) s_rank = 0;
        __syncthreads();
        int cnt = 0;
        for (int i = threadIdx.x; i < pos; i += blockDim.x) cnt += (__ldcg(row + i) == image_token) ? 1 : 0;
        cnt = static_cast<int>(warp_sum(static_cast<float>(cnt)));
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&s_rank, cnt);
        __syncthreads();
        const int rank = s_rank;
        if (rank >= n_img) {             // the reference would raise a shape error here
            if (threadIdx.x == 0) *err_flag = 1;
            return;
        }
        const bf16* src = img + (static_cast<size_t>(b) * n_img + rank) * hidden;
        for (int n = threadIdx.x; n < hidden; n += blockDim.x) {
            float x = bf16_round(bf2f(ldcg_bf16(src + n)) * inv_div);     // image_features / sqrt(hidden)
            x = bf16_round(x * normalizer);                   // embeds *= bf16(sqrt(hidden))
            dst[n] = f2bf(x);
        }
    } else if (id != pad_token) {
        if (id < 0 || id >= vocab) {
            if (threadIdx.x == 0) *err_flag = 2;
            return;
        }
        const bf16* src = table + static_cast<size_t>(id) * hidden;
        for (int n = threadIdx.x; n < hidden; n += blockDim.x)
            dst[n] = f2bf(bf16_round(bf2f(src[n]) * normalizer));
    } else {
        // torch.full(..., pad_token_id) rows, then *= normalizer
        const float x = bf16_round(bf16_round(static_cast<float>(pad_token)) * normalizer);
        for (int n = threadIdx.x; n < hidden; n += blockDim.x) dst[n] = f2bf(x);
    }
}

__device__ __forceinline__ void small_k_linear_body(const bf16* x, int T, int K, const bf16* W, const bf16* bias,
                                                    int N, float scale, bf16* y, int ldy, int col_off,
                                                    const bf16* time_row, int time_cols, const int bx, const int t) {
    const int n = bx * 256 + threadIdx.x;
    if (n < N) {
        float acc = 0.f;
        for (int k = 0; k < K; ++k) acc += bf2f(ldcg_bf16(x + t * K + k)) * bf2f(W[n * K + k]);
        acc += bf2f(bias[n]);
        float v = bf16_round(acc);
        if (scale != 1.0f) v = bf16_round(v * scale);
        y[static_cast<size_t>(t) * ldy + col_off + n] = f2bf(v);
    }
    if (time_row != nullptr && n < time_cols) y[static_cast<size_t>(t) * ldy + n] = time_row[n];
}

__device__ __forceinline__ void action_tail_body(const bf16* xn, int T, int hidden, const bf16* W, const bf16* bias,
                                                 int action_dim, float dt, bf16* action, bf16* vel_tap,
                                                 const int bx) {
    const int gw = (bx * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= T * action_dim) return;
    const int t = gw / action_dim, d = gw - t * action_dim;
    float acc = 0.f;
    for (int k = lane; k < hidden; k += 32)
        acc += bf2f(ldcg_bf16(xn + static_cast<size_t>(t) * hidden + k)) * bf2f(W[static_cast<size_t>(d) * hidden + k]);
    acc = warp_sum(acc);
    if (lane == 0) {
        const float vel = bf16_round(acc + bf2f(bias[d]));
        if (vel_tap != nullptr) vel_tap[gw] = f2bf(vel);
        const float step = bf16_round(dt * vel);                       // delta_t * action_vel
        action[gw] = f2bf(bf16_round(bf2f(ldcg_bf16(action + gw)) + step));        // action += ...
    }
}

__device__ __forceinline__ void clamp_copy_body(const bf16* src, bf16* dst, int n, int do_clamp, float clip,
                                                const int bx) {
    const int i = bx * 256 + threadIdx.x;
    if (i >= n) return;
    float v = bf2f(ldcg_bf16(src + i));
    if (do_clamp) v = (v < -clip) ? -clip : ((v > clip) ? clip : v);   // NaN propagates like torch.clamp
    dst[i] = f2bf(v);
}


}  // namespace blurr
