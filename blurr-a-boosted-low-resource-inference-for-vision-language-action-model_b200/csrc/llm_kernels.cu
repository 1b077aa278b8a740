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
    if (id < 0 || id >= vocab) { if (threadIdx.x == 0 && err_flag) atomicOr(err_flag, 1); id = 0; }
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

// OFT's action rows: a block of n_rows consecutive rows per sequence, starting where the device array says.  One CTA per
// (sequence, row), 16-byte copies.
__global__ void __launch_bounds__(256) gather_row_block_kernel(const bf16* src, int rows_per_seq, const int* row_start, int width,
                                                               bf16* dst) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.y, i = blockIdx.x;
    const int row = row_start[b] + i;           // the host validates row_start[b] + n_rows <= rows_per_seq
    const uint4* s = reinterpret_cast<const uint4*>(src + (static_cast<size_t>(b) * rows_per_seq + row) * width);
    uint4* d = reinterpret_cast<uint4*>(dst + (static_cast<size_t>(b) * gridDim.x + i) * width);
    for (int j = threadIdx.x; j < width / 8; j += blockDim.x) d[j] = s[j];
}

cudaError_t launch_gather_row_block(cudaStream_t stream, const bf16* src, int batch, int rows_per_seq, const int* row_start, int n_rows,
                                    int width, bf16* dst) {
    if ((width & 7) || row_start == nullptr || n_rows < 1 || batch < 1) return cudaErrorInvalidValue;
    return launch_kernel(gather_row_block_kernel, dim3(n_rows, batch), dim3(256), 0, stream, src, rows_per_seq, row_start, width, dst);
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

// ---- sampled decoding (HF `_sample`: fp32 scores, Temperature -> TopK -> TopP warpers, softmax, one draw) ----
// One CTA per row, deterministic: no float atomics, nothing that depends on scheduling.  For T > 0 the scaled score
// __fmul_rn(logit, 1 / T) is monotone in the bf16 logit, so the top-k threshold and the top-p cut are found by two
// 8-bit radix passes over a 16-bit key of the bf16 bits with exact integer counts; masses are exp(s - s_max) rounded
// to 64-bit fixed point (2^shift per unit, vocab * 2^shift < 2^63), so every histogram and prefix sum is an integer sum
// whose value does not depend on the order of the atomics.  The row is read from L2 once per pass (at most six passes).
namespace {

constexpr int kSampleThreads = 1024;

struct SampleShared {
    unsigned cnt_hi[256], cnt_lo[256], cnt_cut[256];
    unsigned long long mass_hi[256], mass_cut[256];
    unsigned long long scan[32];
    unsigned long long best, z, total, above, z_kept, target;
    unsigned above_cnt, n_group, n_keep;
    int bin, thr_key, cut_key, found;
};

// bf16 bits -> 16-bit key whose unsigned order is the float order; -0 -> +0 (HF counts them as one score); NaN -> -1
__device__ __forceinline__ int sample_key(uint32_t b) {
    b &= 0xffffu;
    if ((b & 0x7fffu) > 0x7f80u) return -1;
    if (b == 0x8000u) b = 0u;
    return static_cast<int>((b & 0x8000u) ? (~b & 0xffffu) : (b | 0x8000u));
}

__device__ __forceinline__ float key_logit(int key) {
    const uint32_t b = (key & 0x8000) ? (key & 0x7fff) : (~key & 0xffff);
    return __uint_as_float(b << 16);
}

// keys of columns 8c .. 8c + 7 (-1 past the end of the row)
__device__ __forceinline__ void load_keys8(const bf16* row, int vocab, bool vec, int c, int (&k)[8]) {
    const int i0 = c * 8;
    if (vec && i0 + 8 <= vocab) {
        const uint4 q = __ldcg(reinterpret_cast<const uint4*>(row) + c);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) k[e] = sample_key((e & 1) ? (w[e >> 1] >> 16) : w[e >> 1]);
    } else {
        const unsigned short* r = reinterpret_cast<const unsigned short*>(row);
#pragma unroll
        for (int e = 0; e < 8; ++e) k[e] = i0 + e < vocab ? sample_key(__ldcg(r + i0 + e)) : -1;
    }
}

// Philox4x32-10 (Salmon et al., SC'11; Random123's constants), counter (step, 0, 0, 0), key (seed lo, seed hi): word 0
__device__ __forceinline__ uint32_t philox_word0(uint64_t seed, uint32_t step) {
    uint32_t c0 = step, c1 = 0u, c2 = 0u, c3 = 0u;
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

// Warp 0, lane l: bins 8l .. 8l + 7 of a 256-bin histogram; above[e] = base + the sum of every bin above bin 8l + e
template <typename T>
__device__ __forceinline__ void bins_above(const T* h, T base, int lane, T (&v)[8], T (&above)[8]) {
    T sum = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) { v[e] = h[8 * lane + e]; sum += v[e]; }
    T incl = sum;                                         // over lanes >= lane
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T x = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += x;
    }
    T run = base + incl - sum;
#pragma unroll
    for (int e = 7; e >= 0; --e) { above[e] = run; run += v[e]; }
}

// Warp 0: the largest bin j with above[j] + v[j] >= k (where the k-th largest key lies); `above` of it -> *above_out
__device__ __forceinline__ int bin_of_kth(const unsigned* h, unsigned base, unsigned k, int lane, unsigned* above_out) {
    unsigned v[8], above[8];
    bins_above<unsigned>(h, base, lane, v, above);
    int cand = -1;
#pragma unroll
    for (int e = 0; e < 8; ++e) if (above[e] + v[e] >= k) cand = 8 * lane + e;
    const int bin = __reduce_max_sync(0xffffffffu, cand);
#pragma unroll
    for (int e = 0; e < 8; ++e) if (8 * lane + e == bin) *above_out = above[e];
    return bin;
}

// Warp 0: the smallest bin j whose mass above it is < target (the lowest bin top-p keeps anything of)
__device__ __forceinline__ int bin_of_cut(const unsigned long long* h, unsigned long long base, unsigned long long target, int lane,
                                          unsigned long long* above_out) {
    unsigned long long v[8], above[8];
    bins_above<unsigned long long>(h, base, lane, v, above);
    int cand = 0x7fffffff;
#pragma unroll
    for (int e = 7; e >= 0; --e) if (above[e] < target) cand = 8 * lane + e;
    const int bin = __reduce_min_sync(0xffffffffu, cand);
#pragma unroll
    for (int e = 0; e < 8; ++e) if (8 * lane + e == bin) *above_out = above[e];
    return bin;
}

// The first column i (index order) with  sum_{j <= i} w(key_j, j) > target, or -1.  Called by the whole CTA.
template <class W>
__device__ int select_first(const bf16* row, int vocab, bool vec, const W& w, unsigned long long target, SampleShared& sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nchunk = (vocab + 7) >> 3;
    unsigned long long base = 0;
    if (threadIdx.x == 0) sh.found = -1;
    for (int r0 = 0; r0 < nchunk; r0 += kSampleThreads) {
        const int c = r0 + static_cast<int>(threadIdx.x);
        int k[8];
        if (c < nchunk) {
            load_keys8(row, vocab, vec, c, k);
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) k[e] = -1;
        }
        unsigned long long wv[8], local = 0;
#pragma unroll
        for (int e = 0; e < 8; ++e) { wv[e] = k[e] >= 0 ? w(k[e], c * 8 + e) : 0ull; local += wv[e]; }
        unsigned long long incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long x = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += x;
        }
        if (lane == 31) sh.scan[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long v = sh.scan[lane];
            unsigned long long s = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long x = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += x;
            }
            sh.scan[lane] = s - v;                        // exclusive prefix of warp `lane`
            if (lane == 31) sh.total = s;
        }
        __syncthreads();
        const unsigned long long excl = base + sh.scan[warp] + incl - local;
        if (local > 0 && excl <= target && target - excl < local) {
            unsigned long long acc = excl;
            int found = -1;
#pragma unroll
            for (int e = 0; e < 8; ++e) { acc += wv[e]; if (found < 0 && acc > target) found = c * 8 + e; }
            sh.found = found;
        }
        base += sh.total;
        __syncthreads();
        if (sh.found >= 0) break;
    }
    const int f = sh.found;
    __syncthreads();                                      // the caller may reuse `sh`
    return f;
}

}  // namespace

__global__ void __launch_bounds__(kSampleThreads) sample_rows_kernel(const bf16* logits, int ld, int vocab, const SampleParams* params,
                                                                     int step, int64_t* ids, int64_t* ids_copy, int copy_stride,
                                                                     float* probs, int* err_flag, unsigned long long* trace) {
    __shared__ SampleShared sh;
    trace_stamp(trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(trace, 1);
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bf16* row = logits + static_cast<size_t>(b) * ld;
    const bool vec = (reinterpret_cast<uintptr_t>(row) & 15) == 0;
    const int nchunk = (vocab + 7) >> 3;
    const SampleParams prm = params[b];
    const float inv_t = 1.0f / prm.temperature;          // ATen's `scores / T`: a multiplication by the fp32 reciprocal
    const int shift = 63 - (32 - __clz(vocab));           // vocab * 2^shift < 2^63: the kept mass fits 63 bits
    const float unit = __uint_as_float(static_cast<uint32_t>(127 + shift) << 23);      // 2^shift
    for (int i = threadIdx.x; i < 256; i += kSampleThreads) {
        sh.cnt_hi[i] = sh.cnt_lo[i] = sh.cnt_cut[i] = 0u;
        sh.mass_hi[i] = sh.mass_cut[i] = 0ull;
    }
    if (threadIdx.x == 0) { sh.best = 0ull; sh.z = 0ull; }
    __syncthreads();

    // ---- pass 1: the largest key (lowest column among equal ones: the greedy token) and the count of each high byte ----
    {
        unsigned long long best = 0ull;
        int run_bin = -1;
        unsigned run_n = 0u;
        for (int c = threadIdx.x; c < nchunk; c += kSampleThreads) {
            int k[8];
            load_keys8(row, vocab, vec, c, k);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (k[e] < 0) continue;
                const unsigned long long packed = (static_cast<unsigned long long>(k[e] + 1) << 32) | static_cast<uint32_t>(~(c * 8 + e));
                best = packed > best ? packed : best;
                const int bin = k[e] >> 8;                // adjacent logits mostly share it: one atomic per run
                if (bin != run_bin) {
                    if (run_n) atomicAdd(&sh.cnt_hi[run_bin], run_n);
                    run_bin = bin; run_n = 0u;
                }
                ++run_n;
            }
        }
        if (run_n) atomicAdd(&sh.cnt_hi[run_bin], run_n);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long x = __shfl_xor_sync(0xffffffffu, best, o);
            best = x > best ? x : best;
        }
        if (lane == 0) atomicMax(&sh.best, best);
    }
    __syncthreads();
    const int key_max = static_cast<int>(sh.best >> 32) - 1;
    const int idx_max = key_max < 0 ? 0 : static_cast<int>(~static_cast<uint32_t>(sh.best));
    const float s_max = key_max < 0 ? __int_as_float(0x7fc00000) : __fmul_rn(key_logit(key_max), inv_t);
    if (!isfinite(s_max)) {
        // all NaN / -inf, a +inf logit, or a scaled score that overflows: softmax is undefined -> the greedy token
        if (threadIdx.x == 0) {
            ids[b] = idx_max;
            if (ids_copy != nullptr) ids_copy[static_cast<size_t>(b) * copy_stride] = idx_max;
            if (err_flag != nullptr) atomicOr(err_flag, 2);
        }
        if (probs != nullptr)
            for (int i = threadIdx.x; i < vocab; i += kSampleThreads) probs[static_cast<size_t>(b) * vocab + i] = 0.f;
        trace_stamp(trace, 2);
        return;
    }
    auto mass_of = [&](float s) { return __float2ull_rn(expf(__fsub_rn(s, s_max)) * unit); };

    // ---- top-k: the k-th largest key, counting repeats (pass 2: low bytes inside its high byte) ----
    if (warp == 0) {
        unsigned v[8], above[8];
        bins_above<unsigned>(sh.cnt_hi, 0u, lane, v, above);
        const unsigned n_valid = __shfl_sync(0xffffffffu, above[0] + v[0], 0);
        const unsigned k = static_cast<unsigned>(prm.top_k);
        int bin = -1;
        unsigned ab = 0u;
        if (prm.top_k > 0 && k < n_valid) bin = bin_of_kth(sh.cnt_hi, 0u, k, lane, &ab);
        if (bin >= 0 && (lane == (bin >> 3))) sh.above_cnt = ab;
        if (lane == 0) sh.bin = bin;
    }
    __syncthreads();
    int thr_key = -1;
    if (sh.bin >= 0) {
        const int bin = sh.bin;
        for (int c = threadIdx.x; c < nchunk; c += kSampleThreads) {
            int k[8];
            load_keys8(row, vocab, vec, c, k);
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (k[e] >= 0 && (k[e] >> 8) == bin) atomicAdd(&sh.cnt_lo[k[e] & 255], 1u);
        }
        __syncthreads();
        if (warp == 0) {
            unsigned ab = 0u;
            const int lo = bin_of_kth(sh.cnt_lo, sh.above_cnt, static_cast<unsigned>(prm.top_k), lane, &ab);
            if (lane == 0) sh.thr_key = (bin << 8) | lo;
        }
        __syncthreads();
        thr_key = sh.thr_key;
    }
    // every score >= the k-th largest survives (ties at the threshold included; the scaled threshold also admits keys
    // that scale to the same fp32 value)
    const float s_thr = thr_key < 0 ? -INFINITY : __fmul_rn(key_logit(thr_key), inv_t);

    // ---- pass 3: the mass Z of the top-k set, and (top-p) the mass of each high byte ----
    const bool top_p = prm.top_p < 1.0f;
    {
        unsigned long long z = 0ull, run_m = 0ull;
        int run_bin = -1;
        for (int c = threadIdx.x; c < nchunk; c += kSampleThreads) {
            int k[8];
            load_keys8(row, vocab, vec, c, k);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (k[e] < 0) continue;
                const float s = __fmul_rn(key_logit(k[e]), inv_t);
                if (!(s >= s_thr)) continue;
                const unsigned long long m = mass_of(s);
                z += m;
                if (top_p) {
                    const int bin = k[e] >> 8;
                    if (bin != run_bin) {
                        if (run_m) atomicAdd(&sh.mass_hi[run_bin], run_m);
                        run_bin = bin; run_m = 0ull;
                    }
                    run_m += m;
                }
            }
        }
        if (run_m) atomicAdd(&sh.mass_hi[run_bin], run_m);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
        if (lane == 0) atomicAdd(&sh.z, z);
    }
    __syncthreads();

    // ---- top-p: HF keeps a token iff the mass strictly ahead of it in (score, column) descending order is < p * Z, and
    // always the first one.  The cut group (one key) is found by radix over the masses (pass 4); inside it the columns
    // are kept from the highest down (torch's stable ascending sort removes the lower columns first) ----
    int cut_key = -1, idx_cut = 0;
    unsigned long long z_kept = sh.z;
    if (top_p) {
        if (warp == 0) {
            const unsigned long long target = static_cast<unsigned long long>(ceil(static_cast<double>(prm.top_p) * static_cast<double>(z_kept)));
            int bin = key_max >> 8;                       // p * Z rounds to 0: only the first token
            unsigned long long ab = 0ull;
            if (target > 0ull) bin = bin_of_cut(sh.mass_hi, 0ull, target, lane, &ab);
            if (target > 0ull && lane == (bin >> 3)) sh.above = ab;
            if (lane == 0) { sh.bin = bin; sh.target = target; }
        }
        __syncthreads();
        const int bin = sh.bin;
        for (int c = threadIdx.x; c < nchunk; c += kSampleThreads) {
            int k[8];
            load_keys8(row, vocab, vec, c, k);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (k[e] < 0 || (k[e] >> 8) != bin) continue;
                const float s = __fmul_rn(key_logit(k[e]), inv_t);
                if (!(s >= s_thr)) continue;
                atomicAdd(&sh.mass_cut[k[e] & 255], mass_of(s));
                atomicAdd(&sh.cnt_cut[k[e] & 255], 1u);
            }
        }
        __syncthreads();
        if (warp == 0) {
            const unsigned long long target = sh.target;
            int lo = key_max & 255;
            unsigned long long ab = 0ull;
            if (target > 0ull) lo = bin_of_cut(sh.mass_cut, sh.above, target, lane, &ab);
            if (target > 0ull && lane == (lo >> 3)) sh.above = ab;
            __syncwarp();
            if (lane == 0) {
                const int cut = (bin << 8) | lo;
                const unsigned long long above = target > 0ull ? sh.above : 0ull;
                const unsigned long long m = mass_of(__fmul_rn(key_logit(cut), inv_t));
                const unsigned g = sh.cnt_cut[lo];
                unsigned keep = 1u;
                if (target > 0ull) {                      // columns r = 0, 1, .. of the group have above + r * m ahead
                    const unsigned long long r = m == 0ull ? g : (target - above + m - 1ull) / m;
                    keep = r < g ? static_cast<unsigned>(r) : g;
                }
                sh.cut_key = cut; sh.n_group = g; sh.n_keep = keep;
                sh.z_kept = above + keep * m;
            }
        }
        __syncthreads();
        cut_key = sh.cut_key;
        z_kept = sh.z_kept;
        const unsigned g = sh.n_group, keep = sh.n_keep;
        if (keep < g) {                                   // pass 5: the first kept column of the cut group
            const auto member = [cut_key](int k, int) { return k == cut_key ? 1ull : 0ull; };
            idx_cut = select_first(row, vocab, vec, member, static_cast<unsigned long long>(g - keep), sh);
        }
    }

    // ---- pass 6: the draw, an inverse CDF over the kept set in column order: target = floor(u * Z_kept), u = x / 2^24 ----
    const uint32_t x = philox_word0(prm.seed, static_cast<uint32_t>(step));
    const unsigned long long target = __umul64hi(z_kept, static_cast<unsigned long long>(x >> 8) << 40);
    const auto kept = [&](int k, int i, float s) { return s >= s_thr && k >= cut_key && (k != cut_key || i >= idx_cut); };
    const auto kept_mass = [&](int k, int i) -> unsigned long long {
        const float s = __fmul_rn(key_logit(k), inv_t);
        return kept(k, i, s) ? mass_of(s) : 0ull;
    };
    int id = select_first(row, vocab, vec, kept_mass, target, sh);
    if (id < 0) id = idx_max;                             // unreachable: the kept mass z_kept > target
    if (threadIdx.x == 0) {
        ids[b] = id;
        if (ids_copy != nullptr) ids_copy[static_cast<size_t>(b) * copy_stride] = id;
    }
    if (probs != nullptr) {
        const float zf = static_cast<float>(static_cast<double>(z_kept) * exp2(-static_cast<double>(shift)));
        const unsigned short* r16 = reinterpret_cast<const unsigned short*>(row);
        for (int i = threadIdx.x; i < vocab; i += kSampleThreads) {
            const int k = sample_key(__ldcg(r16 + i));
            const float s = k >= 0 ? __fmul_rn(key_logit(k), inv_t) : 0.f;
            float p = 0.f;                                // (a kept token whose fixed-point mass rounds to 0 is never drawn)
            if (k >= 0 && kept(k, i, s)) p = expf(__fsub_rn(s, s_max)) / zf;
            probs[static_cast<size_t>(b) * vocab + i] = p;
        }
    }
    trace_stamp(trace, 2);
}

cudaError_t launch_sample_rows(cudaStream_t stream, const bf16* logits, int batch, int ld, int vocab, const SampleParams* params,
                               int step, int64_t* ids, int64_t* ids_copy, int copy_stride, float* probs, int* err_flag,
                               unsigned long long* trace) {
    if (batch < 1 || vocab < 1 || ld < vocab || params == nullptr || ids == nullptr) return cudaErrorInvalidValue;
    return launch_kernel(sample_rows_kernel, dim3(batch), dim3(kSampleThreads), 0, stream, logits, ld, vocab, params, step, ids,
                         ids_copy, copy_stride, probs, err_flag, trace);
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
