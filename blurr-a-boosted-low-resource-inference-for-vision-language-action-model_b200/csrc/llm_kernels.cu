// Small kernels of the Llama-shaped decoder (OpenVLA-7B-shaped path, SURVEY.md 8(f) row 3): RoPE + KV-cache append for
// multi-head attention, token embedding gather, last-row gather and greedy argmax.  All bandwidth-trivial (KB per call);
// written for few dependent launches: one CTA per token row, vectorised 8-byte accesses, warp-shuffle reductions.
#include "bodies.cuh"
#include "kernels.h"
#include "launch.cuh"

namespace blurr {

// HF Llama (modeling_llama.py apply_rotary_pos_emb / rotate_half): with d = head_dim, for j < d/2
//   y[j]       = bf16(bf16(x[j] * cos[j])       + bf16(-x[j + d/2] * sin[j]))
//   y[j + d/2] = bf16(bf16(x[j + d/2] * cos[j]) + bf16( x[j]       * sin[j]))
// (cos/sin are cat(freqs, freqs), cast to the activation dtype).  One thread per 4 rotation pairs.  Three CTAs per SM:
// left free, ptxas settles at 48 registers and spills loop invariants of the split-K sums to local memory.
__global__ void __launch_bounds__(256, 3) rope_mha_kernel(const RopeMhaArgs a) {
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    const int t = blockIdx.x;
    const int seq = t / a.tokens_per_seq, i = t - seq * a.tokens_per_seq;
    int pos = (a.seq_len != nullptr ? a.seq_len[seq] + a.len_off : a.pos0) + i;
    if (pos >= a.n_pos) pos = a.n_pos - 1;               // the host validates the range
    const int half = a.head_dim >> 1;
    const int gpr = half >> 2;                            // 4-wide groups per rotated head
    const int n_rot_heads = a.n_heads + a.n_kv_heads;
    const int n_rot = n_rot_heads * gpr;
    const int n_v = (a.n_kv_heads * a.head_dim) >> 2;
    const size_t sstride = static_cast<size_t>(a.T) * a.ldp;
    const size_t cache_row = (static_cast<size_t>(seq) * a.n_slots + pos) * (a.n_kv_heads * a.head_dim);
    for (int it = blockIdx.y * blockDim.x + threadIdx.x; it < n_rot + n_v; it += gridDim.y * blockDim.x) {
        if (it < n_rot) {
            const int h = it / gpr, j = (it - h * gpr) << 2;
            const int col = h * a.head_dim + j;           // q heads then k heads are contiguous in the projection
            float4 x1, x2;
            if (a.lin != nullptr) {
                x1 = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + col);
                x2 = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + col + half);
            } else {
                x1 = sum_slices(a.partial + static_cast<size_t>(t) * a.ldp + col, sstride, a.splitk);
                x2 = sum_slices(a.partial + static_cast<size_t>(t) * a.ldp + col + half, sstride, a.splitk);
            }
            const float4 cs = *reinterpret_cast<const float4*>(a.cos_table + static_cast<size_t>(pos) * half + j);
            const float4 sn = *reinterpret_cast<const float4*>(a.sin_table + static_cast<size_t>(pos) * half + j);
            const float u1[4] = {bf16_round(x1.x), bf16_round(x1.y), bf16_round(x1.z), bf16_round(x1.w)};
            const float u2[4] = {bf16_round(x2.x), bf16_round(x2.y), bf16_round(x2.z), bf16_round(x2.w)};
            const float c[4] = {cs.x, cs.y, cs.z, cs.w}, s[4] = {sn.x, sn.y, sn.z, sn.w};
            float y1[4], y2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                y1[e] = bf16_round(bf16_round(u1[e] * c[e]) + bf16_round(-u2[e] * s[e]));
                y2[e] = bf16_round(bf16_round(u2[e] * c[e]) + bf16_round(u1[e] * s[e]));
            }
            bf16* dst = (h < a.n_heads) ? a.q_out + static_cast<size_t>(t) * (a.n_heads * a.head_dim) + h * a.head_dim
                                        : a.k_cache + cache_row + (h - a.n_heads) * a.head_dim;
            store_bf16x4(dst + j, make_float4(y1[0], y1[1], y1[2], y1[3]));
            store_bf16x4(dst + half + j, make_float4(y2[0], y2[1], y2[2], y2[3]));
        } else {
            const int j = (it - n_rot) << 2;
            const int col = n_rot_heads * a.head_dim + j;
            const float4 v = a.lin != nullptr ? load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + col)
                                              : sum_slices(a.partial + static_cast<size_t>(t) * a.ldp + col, sstride, a.splitk);
            store_bf16x4(a.v_cache + cache_row + j,
                         make_float4(bf16_round(v.x), bf16_round(v.y), bf16_round(v.z), bf16_round(v.w)));
        }
    }
    trace_stamp(a.trace, 2);
}

// Decode attention: ONE query row per (sequence, head) against that head's cached keys - pure K/V streaming (2 * n_keys *
// head_dim * 2 bytes per CTA), so no tensor cores: a group of HD / 8 lanes owns one key (16-byte loads, 4 keys in flight
// per group), scores and probabilities live in shared memory, the P.V sum is reduced across groups at the end.
// Rounding chain of HF eager attention: bf16(q.k) * scale -> bf16, fp32 softmax -> bf16, fp32 accumulate -> bf16.
// FUSED: the kernel also does the RoPE + cache append of its own head for the step's new token (rope_mha_kernel's work for
// one (sequence, head): with multi-head attention nothing a CTA needs lives in another head), so a decode step has one
// kernel less per layer: q, k, v of the new token come from the q/k/v GEMM's split-K partials, the new K/V row is written
// to the cache and used from shared memory as key n - 1.
// RAGGED: prompts of different lengths - the key count (and with FUSED the new token's position / cache slot) comes from
// the device length array per sequence.  A template parameter, not a runtime test, so that the equal-length kernels keep
// their register allocation (the FUSED head_dim-128 kernel sits at ~242 of 255 registers).
template <int HD, bool FUSED, bool RAGGED>
__global__ void __launch_bounds__(256, 1) mha_decode_kernel(const MhaAttnArgs a, const RopeMhaArgs r) {
    constexpr int LPK = HD / 8;                 // lanes per key
    constexpr int GROUPS = 256 / LPK;           // keys in flight per pass
    __shared__ float sc[320];
    __shared__ float red[8];
    __shared__ float part[GROUPS][HD + 4];
    __shared__ float raw[3][HD];
    __shared__ __align__(16) bf16 qkv_s[3][HD];
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    const int h = blockIdx.x, b = blockIdx.y;
    const int width = a.n_heads * HD;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int group = threadIdx.x / LPK, gl = threadIdx.x % LPK;
    const size_t row0 = static_cast<size_t>(b) * a.n_slots;
    const bf16* kbase = a.k_cache + row0 * width + h * HD + gl * 8;
    const bf16* vbase = a.v_cache + row0 * width + h * HD + gl * 8;
    const int n = RAGGED ? a.seq_len[b] + a.len_off : a.n_keys;
    const int nload = FUSED ? n - 1 : n;        // FUSED: key n - 1 is the token this step appends
    // every K and V row of this group is requested up front (<= 320 / GROUPS keys per group, 16 bytes each per lane): the
    // kernel is two HBM round trips long instead of one per 4 keys (measured 15 -> 4 us per layer at one sequence)
    constexpr int KPG = 320 / GROUPS;
    uint4 kr[KPG], vr[KPG];
#pragma unroll
    for (int u = 0; u < KPG; ++u) {
        const int k = group + u * GROUPS;
        kr[u] = k < nload ? __ldcg(reinterpret_cast<const uint4*>(kbase + static_cast<size_t>(k) * width)) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < KPG; ++u) {
        const int k = group + u * GROUPS;
        vr[u] = k < nload ? __ldcg(reinterpret_cast<const uint4*>(vbase + static_cast<size_t>(k) * width)) : make_uint4(0u, 0u, 0u, 0u);
    }
    uint4 qraw;
    if (FUSED) {
        // q / k / v of the new token: sum the K slices, round to bf16 (the Linear's output), rotate q and k
        const int half = HD >> 1;
        const size_t sstride = static_cast<size_t>(r.T) * r.ldp;
        for (int i = threadIdx.x; i < 3 * HD; i += 256) {
            const int which = i / HD, d = i - which * HD;
            const int col = (which == 0 ? 0 : which == 1 ? r.n_heads * HD : (r.n_heads + r.n_kv_heads) * HD) + h * HD + d;
            const float* src = r.partial + static_cast<size_t>(b) * r.ldp + col;
            float acc = 0.f;
            for (int z = 0; z < r.splitk; ++z) acc += __ldcg(src + z * sstride);
            raw[which][d] = bf16_round(acc);
        }
        __syncthreads();
        int pos = RAGGED ? r.seq_len[b] + r.len_off : r.pos0;
        if (pos >= r.n_pos) pos = r.n_pos - 1;
        const size_t cache_row = (row0 + pos) * width + h * HD;
        for (int i = threadIdx.x; i < 2 * half + HD; i += 256) {
            if (i < 2 * half) {                               // rotation pair j of q (i < half) or k
                const int which = i / half, j = i - which * half;
                const float c = r.cos_table[static_cast<size_t>(pos) * half + j], sn = r.sin_table[static_cast<size_t>(pos) * half + j];
                const float x1 = raw[which][j], x2 = raw[which][j + half];
                const float y1 = bf16_round(bf16_round(x1 * c) + bf16_round(-x2 * sn));
                const float y2 = bf16_round(bf16_round(x2 * c) + bf16_round(x1 * sn));
                qkv_s[which][j] = f2bf(y1);
                qkv_s[which][j + half] = f2bf(y2);
                if (which == 1) { r.k_cache[cache_row + j] = f2bf(y1); r.k_cache[cache_row + j + half] = f2bf(y2); }
            } else {
                const int d = i - 2 * half;
                const bf16 v = f2bf(raw[2][d]);
                qkv_s[2][d] = v;
                r.v_cache[cache_row + d] = v;
            }
        }
        __syncthreads();
        qraw = *reinterpret_cast<const uint4*>(&qkv_s[0][gl * 8]);
#pragma unroll
        for (int u = 0; u < KPG; ++u)
            if (group + u * GROUPS == n - 1) {
                kr[u] = *reinterpret_cast<const uint4*>(&qkv_s[1][gl * 8]);
                vr[u] = *reinterpret_cast<const uint4*>(&qkv_s[2][gl * 8]);
            }
    } else {
        qraw = *reinterpret_cast<const uint4*>(a.q + static_cast<size_t>(b) * width + h * HD + gl * 8);
    }
    float q[8];
    {
        const uint32_t w[4] = {qraw.x, qraw.y, qraw.z, qraw.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) { q[2 * e] = __uint_as_float(w[e] << 16); q[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u); }
    }
    // ---- scores ----
#pragma unroll
    for (int u = 0; u < KPG; ++u) {
        const uint32_t w[4] = {kr[u].x, kr[u].y, kr[u].z, kr[u].w};
        float d = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            d = fmaf(q[2 * e], __uint_as_float(w[e] << 16), d);
            d = fmaf(q[2 * e + 1], __uint_as_float(w[e] & 0xffff0000u), d);
        }
#pragma unroll
        for (int o = LPK / 2; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        const int k = group + u * GROUPS;
        if (gl == 0 && k < n) sc[k] = bf16_round(bf16_round(d) * a.scale);
    }
    __syncthreads();
    // ---- softmax (fp32) -> bf16 probabilities ----
    float m = -INFINITY;
    for (int k = threadIdx.x; k < n; k += 256) m = fmaxf(m, sc[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float sum = 0.f;
    for (int k = threadIdx.x; k < n; k += 256) { const float e = expf(sc[k] - m); sc[k] = e; sum += e; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) red[warp] = sum;
    __syncthreads();
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[w];
    for (int k = threadIdx.x; k < n; k += 256) sc[k] = bf16_round(sc[k] / sum);
    __syncthreads();
    // ---- O = P V ----
    float o8[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) o8[e] = 0.f;
#pragma unroll
    for (int u = 0; u < KPG; ++u) {
        const int k = group + u * GROUPS;
        const float p = k < n ? sc[k] : 0.f;
        const uint32_t w[4] = {vr[u].x, vr[u].y, vr[u].z, vr[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            o8[2 * e] = fmaf(p, __uint_as_float(w[e] << 16), o8[2 * e]);
            o8[2 * e + 1] = fmaf(p, __uint_as_float(w[e] & 0xffff0000u), o8[2 * e + 1]);
        }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) part[group][gl * 8 + e] = o8[e];
    __syncthreads();
    for (int d = threadIdx.x; d < HD; d += 256) {
        float acc = 0.f;
#pragma unroll 4
        for (int g = 0; g < GROUPS; ++g) acc += part[g][d];
        a.out[static_cast<size_t>(b) * width + h * HD + d] = f2bf(acc);
    }
    trace_stamp(a.trace, 2);
}

// Many sequences (grid > 2 CTAs per SM): the same kernel with 4 keys in flight per group and ~60 registers, so that
// several CTAs share an SM and hide each other's round trips (measured at 32 sequences: 4.75 vs 5.34 ms per token).
template <int HD, bool RAGGED>
__global__ void __launch_bounds__(256) mha_decode_loop_kernel(const MhaAttnArgs a) {
    constexpr int LPK = HD / 8;                 // lanes per key
    constexpr int GROUPS = 256 / LPK;           // keys in flight per pass
    __shared__ float sc[320];
    __shared__ float red[8];
    __shared__ float part[GROUPS][HD + 4];
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    const int h = blockIdx.x, b = blockIdx.y;
    const int width = a.n_heads * HD;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int group = threadIdx.x / LPK, gl = threadIdx.x % LPK;
    const bf16* qp = a.q + static_cast<size_t>(b) * width + h * HD + gl * 8;
    const uint4 qraw = *reinterpret_cast<const uint4*>(qp);
    float q[8];
    {
        const uint32_t w[4] = {qraw.x, qraw.y, qraw.z, qraw.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) { q[2 * e] = __uint_as_float(w[e] << 16); q[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u); }
    }
    const size_t row0 = static_cast<size_t>(b) * a.n_slots;
    const bf16* kbase = a.k_cache + row0 * width + h * HD + gl * 8;
    const bf16* vbase = a.v_cache + row0 * width + h * HD + gl * 8;
    const int n = RAGGED ? a.seq_len[b] + a.len_off : a.n_keys;
    // ---- scores ----
    for (int kfirst = 0; kfirst < n; kfirst += 4 * GROUPS) {      // warp-uniform trip count: the groups of a warp shuffle together
        const int k0 = kfirst + group;
        uint4 kr[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * GROUPS;
            kr[u] = k < n ? __ldcg(reinterpret_cast<const uint4*>(kbase + static_cast<size_t>(k) * width)) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t w[4] = {kr[u].x, kr[u].y, kr[u].z, kr[u].w};
            float d = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                d = fmaf(q[2 * e], __uint_as_float(w[e] << 16), d);
                d = fmaf(q[2 * e + 1], __uint_as_float(w[e] & 0xffff0000u), d);
            }
#pragma unroll
            for (int o = LPK / 2; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
            const int k = k0 + u * GROUPS;
            if (gl == 0 && k < n) sc[k] = bf16_round(bf16_round(d) * a.scale);
        }
    }
    __syncthreads();
    // ---- softmax (fp32) -> bf16 probabilities ----
    float m = -INFINITY;
    for (int k = threadIdx.x; k < n; k += 256) m = fmaxf(m, sc[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float sum = 0.f;
    for (int k = threadIdx.x; k < n; k += 256) { const float e = expf(sc[k] - m); sc[k] = e; sum += e; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) red[warp] = sum;
    __syncthreads();
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[w];
    for (int k = threadIdx.x; k < n; k += 256) sc[k] = bf16_round(sc[k] / sum);
    __syncthreads();
    // ---- O = P V ----
    float o8[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) o8[e] = 0.f;
    for (int kfirst = 0; kfirst < n; kfirst += 4 * GROUPS) {      // warp-uniform trip count: the groups of a warp shuffle together
        const int k0 = kfirst + group;
        uint4 vr[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * GROUPS;
            vr[u] = k < n ? __ldcg(reinterpret_cast<const uint4*>(vbase + static_cast<size_t>(k) * width)) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * GROUPS;
            const float p = k < n ? sc[k] : 0.f;
            const uint32_t w[4] = {vr[u].x, vr[u].y, vr[u].z, vr[u].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                o8[2 * e] = fmaf(p, __uint_as_float(w[e] << 16), o8[2 * e]);
                o8[2 * e + 1] = fmaf(p, __uint_as_float(w[e] & 0xffff0000u), o8[2 * e + 1]);
            }
        }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) part[group][gl * 8 + e] = o8[e];
    __syncthreads();
    for (int d = threadIdx.x; d < HD; d += 256) {
        float acc = 0.f;
#pragma unroll 4
        for (int g = 0; g < GROUPS; ++g) acc += part[g][d];
        a.out[static_cast<size_t>(b) * width + h * HD + d] = f2bf(acc);
    }
    trace_stamp(a.trace, 2);
}

bool mha_decode_fuses_rope(const MhaAttnArgs& a) {
    return a.q_per_sample == 1 && a.n_heads * a.batch <= 2 * 148 && (a.head_dim == 128 || a.head_dim == 64);
}

template <int HD, bool RAGGED>
static cudaError_t launch_mha_decode_hd(cudaStream_t stream, const MhaAttnArgs& a, const RopeMhaArgs* rope, bool wide) {
    const dim3 grid(a.n_heads, a.batch);
    if (rope != nullptr) return launch_kernel(mha_decode_kernel<HD, true, RAGGED>, grid, dim3(256), 0, stream, a, *rope);
    const RopeMhaArgs none{};
    return wide ? launch_kernel(mha_decode_kernel<HD, false, RAGGED>, grid, dim3(256), 0, stream, a, none)
                : launch_kernel(mha_decode_loop_kernel<HD, RAGGED>, grid, dim3(256), 0, stream, a);
}

// `rope` != nullptr (only when mha_decode_fuses_rope): the kernel also rotates / appends this step's token (no rope_mha launch).
// a.seq_len != nullptr selects the ragged kernels; a fused `rope` must then carry the same lengths.
cudaError_t launch_mha_decode(cudaStream_t stream, const MhaAttnArgs& a, const RopeMhaArgs* rope) {
    if (a.q_per_sample != 1 || a.n_keys > 320 || a.n_kv_heads != a.n_heads) return cudaErrorInvalidValue;
    const bool wide = a.n_heads * a.batch <= 2 * 148;       // few CTAs: every load of a CTA in flight at once
    const bool ragged = a.seq_len != nullptr;
    if (rope != nullptr) {
        if (!mha_decode_fuses_rope(a) || rope->lin != nullptr || rope->tokens_per_seq != 1) return cudaErrorInvalidValue;
        if ((rope->seq_len != nullptr) != ragged) return cudaErrorInvalidValue;
    }
    if (a.head_dim == 128)
        return ragged ? launch_mha_decode_hd<128, true>(stream, a, rope, wide) : launch_mha_decode_hd<128, false>(stream, a, rope, wide);
    if (a.head_dim == 64)
        return ragged ? launch_mha_decode_hd<64, true>(stream, a, rope, wide) : launch_mha_decode_hd<64, false>(stream, a, rope, wide);
    return cudaErrorInvalidValue;
}

cudaError_t launch_rope_mha(cudaStream_t stream, const RopeMhaArgs& a) {
    if ((a.head_dim & 7) || a.T <= 0) return cudaErrorInvalidValue;
    // one work item (4 rotation pairs / 4 value columns, all K slices) per thread: a decode step's single row still
    // spreads over ~10 CTAs instead of looping in one (measured 19 -> 5 us per layer at one sequence)
    const int items = (a.n_heads + a.n_kv_heads) * (a.head_dim >> 3) + ((a.n_kv_heads * a.head_dim) >> 2);
    int gy = (items + 255) / 256;
    if (a.T * gy > 148 * 8) gy = (148 * 8 + a.T - 1) / a.T;      // prefill: enough rows already
    if (gy < 1) gy = 1;
    return launch_kernel(rope_mha_kernel, dim3(a.T, gy), dim3(256), 0, stream, a);
}

__global__ void __launch_bounds__(256) embed_rows_kernel(const int64_t* ids, int n, const bf16* table, long long vocab,
                                                         int width, bf16* out, int* err_flag) {
    pdl_wait();
    pdl_trigger();
    const int r = blockIdx.x;
    long long id = ids[r];
    if (id < 0 || id >= vocab) { if (threadIdx.x == 0 && err_flag) atomicExch(err_flag, 1); id = 0; }
    const uint4* src = reinterpret_cast<const uint4*>(table + static_cast<size_t>(id) * width);
    uint4* dst = reinterpret_cast<uint4*>(out + static_cast<size_t>(r) * width);
    for (int i = threadIdx.x; i < width / 8; i += blockDim.x) dst[i] = src[i];
}

cudaError_t launch_embed_rows(cudaStream_t stream, const int64_t* ids, int n, const bf16* table, long long vocab, int width,
                              bf16* out, int* err_flag) {
    if (width & 7) return cudaErrorInvalidValue;
    return launch_kernel(embed_rows_kernel, dim3(n), dim3(256), 0, stream, ids, n, table, vocab, width, out, err_flag);
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const bf16* src, int rows_per_seq, int row, int width, bf16* dst,
                                                          const int* seq_len) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.x;
    if (seq_len != nullptr) row = seq_len[b] - 1;
    const uint4* s = reinterpret_cast<const uint4*>(src + (static_cast<size_t>(b) * rows_per_seq + row) * width);
    uint4* d = reinterpret_cast<uint4*>(dst + static_cast<size_t>(b) * width);
    for (int i = threadIdx.x; i < width / 8; i += blockDim.x) d[i] = s[i];
}

cudaError_t launch_gather_rows(cudaStream_t stream, const bf16* src, int batch, int rows_per_seq, int row, int width, bf16* dst,
                               const int* seq_len) {
    if (width & 7) return cudaErrorInvalidValue;
    return launch_kernel(gather_rows_kernel, dim3(batch), dim3(256), 0, stream, src, rows_per_seq, row, width, dst, seq_len);
}

// Pad rows of a ragged prompt batch -> 0 before prefill.  The prefill attention multiplies whole key blocks by P, and a
// masked key's P = 0 still turns a NaN / Inf value into NaN; with zero inputs every pad row stays a finite function of
// its sequence's real rows, so nothing the caller left in the pads reaches a real row.  One CTA column per sequence.
__global__ void __launch_bounds__(256) zero_pad_rows_kernel(bf16* x, int rows_per_seq, int width, const int* seq_len) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.x;
    int len = seq_len[b];
    len = len < 0 ? 0 : (len > rows_per_seq ? rows_per_seq : len);      // the host validates the range
    const size_t n = static_cast<size_t>(rows_per_seq - len) * (width >> 3);
    uint4* p = reinterpret_cast<uint4*>(x + (static_cast<size_t>(b) * rows_per_seq + len) * width);
    for (size_t i = static_cast<size_t>(blockIdx.y) * blockDim.x + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.y) * blockDim.x)
        p[i] = make_uint4(0u, 0u, 0u, 0u);
}

cudaError_t launch_zero_pad_rows(cudaStream_t stream, bf16* x, int batch, int rows_per_seq, int width, const int* seq_len) {
    if ((width & 7) || seq_len == nullptr) return cudaErrorInvalidValue;
    return launch_kernel(zero_pad_rows_kernel, dim3(batch, 4), dim3(256), 0, stream, x, rows_per_seq, width, seq_len);
}

// One CTA per sequence.  Greedy decoding compares the bf16 logits as fp32 (HF casts the last row to fp32 first); the
// lowest index wins among equal maxima.
__global__ void __launch_bounds__(1024) argmax_rows_kernel(const bf16* logits, int ld, int vocab, int64_t* ids, int64_t* ids_copy,
                                                           int copy_stride) {
    pdl_wait();
    pdl_trigger();
    __shared__ float s_val[32];
    __shared__ int s_idx[32];
    const int b = blockIdx.x;
    const bf16* row = logits + static_cast<size_t>(b) * ld;
    float best = -INFINITY;
    int best_i = 0x7fffffff;
    const bool vec = ((reinterpret_cast<uintptr_t>(row) & 15) == 0);
    const int nvec = vec ? (vocab >> 3) : 0;
    for (int c = threadIdx.x; c < nvec; c += blockDim.x) {
        const uint4 q = __ldcg(reinterpret_cast<const uint4*>(row) + c);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float v = __uint_as_float((e & 1) ? (w[e >> 1] & 0xffff0000u) : (w[e >> 1] << 16));
            const int i = c * 8 + e;
            if (v != v) continue;                               // NaN never wins
            if (v > best || (v == best && i < best_i)) { best = v; best_i = i; }
        }
    }
    for (int i = nvec * 8 + threadIdx.x; i < vocab; i += blockDim.x) {
        const float v = bf2f(row[i]);
        if (v != v) continue;
        if (v > best || (v == best && i < best_i)) { best = v; best_i = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_val[warp] = best; s_idx[warp] = best_i; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        best = lane < nw ? s_val[lane] : -INFINITY;
        best_i = lane < nw ? s_idx[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
            if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
        }
        if (lane == 0) {
            const int64_t id = best_i == 0x7fffffff ? 0 : best_i;
            ids[b] = id;
            if (ids_copy != nullptr) ids_copy[static_cast<size_t>(b) * copy_stride] = id;
        }
    }
}

cudaError_t launch_argmax_rows(cudaStream_t stream, const bf16* logits, int batch, int ld, int vocab, int64_t* ids,
                               int64_t* ids_copy, int copy_stride) {
    return launch_kernel(argmax_rows_kernel, dim3(batch), dim3(1024), 0, stream, logits, ld, vocab, ids, ids_copy, copy_stride);
}

// GLU over split-K partials of a few-token gate/up projection whose weight rows alternate gate_j, up_j (the layout of
// the EPI_GEGLU epilogue): out[t][j] = bf16(bf16(act(bf16(gate_j))) * bf16(up_j)).  8 partial columns -> 4 outputs per thread.
__global__ void __launch_bounds__(256) glu_partial_kernel(const float* partial, int splitk, int T, int Nw, int act, bf16* out,
                                                          int ldo, unsigned long long* trace) {
    trace_stamp(trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(trace, 1);
    const int per_row = Nw >> 3;
    const int idx = blockIdx.x * 256 + threadIdx.x;
    if (idx >= T * per_row) { trace_stamp(trace, 2); return; }
    const int t = idx / per_row, c = (idx - t * per_row) << 3;
    const size_t sstride = static_cast<size_t>(T) * Nw;
    const float4 a = sum_slices(partial + static_cast<size_t>(t) * Nw + c, sstride, splitk);
    const float4 b = sum_slices(partial + static_cast<size_t>(t) * Nw + c + 4, sstride, splitk);
    const float g[4] = {bf16_round(a.x), bf16_round(a.z), bf16_round(b.x), bf16_round(b.z)};
    const float u[4] = {bf16_round(a.y), bf16_round(a.w), bf16_round(b.y), bf16_round(b.w)};
    store_bf16x4(out + static_cast<size_t>(t) * ldo + (c >> 1),
                 make_float4(bf16_round(glu_act_f32(g[0], act)) * u[0], bf16_round(glu_act_f32(g[1], act)) * u[1],
                             bf16_round(glu_act_f32(g[2], act)) * u[2], bf16_round(glu_act_f32(g[3], act)) * u[3]));
    trace_stamp(trace, 2);
}

cudaError_t launch_glu_partial(cudaStream_t stream, const float* partial, int splitk, int T, int Nw, int act, bf16* out, int ldo,
                               unsigned long long* trace) {
    if (Nw & 7) return cudaErrorInvalidValue;
    const int total = T * (Nw >> 3);
    return launch_kernel(glu_partial_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, partial, splitk, T, Nw, act, out, ldo,
                         trace);
}

}  // namespace blurr
