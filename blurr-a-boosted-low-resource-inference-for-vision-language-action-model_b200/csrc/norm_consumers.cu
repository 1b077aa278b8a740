// Stand-alone launches of the GEMM consumers (bodies in bodies.cuh): deterministic split-K
// reduction + bias + residual/position add + norm, and RoPE + KV-cache append.  HBM/L2-bandwidth-
// bound row kernels: one CTA per token row, 16-byte loads, warp-shuffle + shared-memory reductions.
//
// Rounding points follow the reference exactly (SURVEY.md Appendix A):
//   linear output  -> bf16(acc + bias)                              (nn.Linear)
//   residual       -> bf16(res + x)                                 (siglip.py:228,236; joint_model.py:79-81,126-128)
//   GemmaRMSNorm   -> bf16((x * rsqrt(mean(x^2) + eps)) * (1 + w))  (paligemma/modules.py:13-21)
//   LayerNorm      -> bf16((x - mean) * rstd * w + b)               (nn.LayerNorm, eps 1e-6)
//   RoPE           -> bf16(bf16(x*cos) + bf16(rot(x)*sin))          (utils.py:11-16), K cached post-RoPE
#include "bodies.cuh"
#include "launch.cuh"

namespace blurr {

template <int VPT, int THREADS, bool FILM = false>
__global__ void __launch_bounds__(THREADS) consumer_kernel(const ConsumerArgs a) {
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();     // only now: a successor that is resident earlier just holds SM resources while it waits (measured)
    trace_stamp(a.trace, 1);
    consumer_body<VPT, THREADS, false, FILM>(a, blockIdx.x);
    trace_stamp(a.trace, 2);
}

// Batched episodes, bf16 hand-off mode: a fixed grid streams the rows, every CTA fetching the inputs of its next
// row before it reduces the current one (the one-row-per-CTA launch is latency-bound: 1.7-2.4 TB/s at 64 episodes).
template <int VPT, int THREADS, bool FILM = false>
__global__ void __launch_bounds__(THREADS) consumer_stream_kernel(const ConsumerArgs a) {
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    int t = blockIdx.x;
    ConsumerRowIn<VPT> cur, nxt;
    if (t < a.T) consumer_prefetch<VPT, THREADS>(a, t, cur);
    for (; t < a.T; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < a.T) consumer_prefetch<VPT, THREADS>(a, tn, nxt);
        consumer_body<VPT, THREADS, true, FILM>(a, t, &cur);
        cur = nxt;
    }
    trace_stamp(a.trace, 2);
}

static constexpr int kStreamMinRows = 2048;

// FiLM consumers: the ViT towers' widths (DINOv2-L 1024, SigLIP-so400m 1152 columns) in the three regimes the towers
// reach - split-K partials (<= 288 rows), the bf16 hand-off, and the streaming launch from kStreamMinRows rows
static cudaError_t launch_film_consumer(cudaStream_t stream, const ConsumerArgs& a) {
    if ((a.N != 4 * 256 && a.N != 4 * 288) || (a.ldp & 3) || (a.film_ld & 3) || a.film_rows < 1) return cudaErrorInvalidValue;
    const bool wide = a.N == 4 * 288;
    if (a.lin != nullptr && a.T >= kStreamMinRows && a.partial == nullptr) {
        const int grid = 148 * 6;
        if (wide) return launch_kernel(consumer_stream_kernel<1, 288, true>, dim3(grid), dim3(288), 0, stream, a);
        return launch_kernel(consumer_stream_kernel<1, kRowThreads, true>, dim3(grid), dim3(kRowThreads), 0, stream, a);
    }
    if (wide) return launch_kernel(consumer_kernel<1, 288, true>, dim3(a.T), dim3(288), 0, stream, a);
    return launch_kernel(consumer_kernel<1, kRowThreads, true>, dim3(a.T), dim3(kRowThreads), 0, stream, a);
}

cudaError_t launch_consumer(cudaStream_t stream, const ConsumerArgs& a) {
    if (a.film_gamma != nullptr) return launch_film_consumer(stream, a);
    if (a.lin != nullptr && a.T >= kStreamMinRows && !(a.N & 3) && a.partial == nullptr) {
        const int grid = 148 * 6;
        if (a.N == 4 * 288) return launch_kernel(consumer_stream_kernel<1, 288>, dim3(grid), dim3(288), 0, stream, a);
        if (a.N == 4 * 512) return launch_kernel(consumer_stream_kernel<2, kRowThreads>, dim3(grid), dim3(kRowThreads), 0, stream, a);
        if (a.N == 4 * 256) return launch_kernel(consumer_stream_kernel<1, kRowThreads>, dim3(grid), dim3(kRowThreads), 0, stream, a);
    }
    if ((a.N & 3) || a.N > 2 * 4 * 512 || (a.ldp & 3)) return cudaErrorInvalidValue;
    if (a.N > 2 * 4 * kRowThreads)      // Llama-2-7B's 4096 columns: two 4-column groups per thread on 512 threads
        return launch_kernel(consumer_kernel<2, 512>, dim3(a.T), dim3(512), 0, stream, a);
    // exact fits: every thread owns the same number of 4-column groups (1152 columns on 256 threads left 7/8 of
    // the CTA idle in the second pass and cost an occupancy-limiting 46 registers)
    if (a.N == 4 * 288) return launch_kernel(consumer_kernel<1, 288>, dim3(a.T), dim3(288), 0, stream, a);
    if (a.N <= 4 * kRowThreads)
        return launch_kernel(consumer_kernel<1, kRowThreads>, dim3(a.T), dim3(kRowThreads), 0, stream, a);
    // Gemma's 2048 columns: one 4-column group per thread on 512 threads, so that all of a row's split-K loads go out
    // in two round trips to L2 instead of four (the kernel is latency-bound)
    if (a.N == 4 * 512) return launch_kernel(consumer_kernel<1, 512>, dim3(a.T), dim3(512), 0, stream, a);
    return launch_kernel(consumer_kernel<2, kRowThreads>, dim3(a.T), dim3(kRowThreads), 0, stream, a);
}

__global__ void __launch_bounds__(256) bias_act_kernel(const float* partial, int splitk, int T, int N, int ldp,
                                                       const bf16* bias, int act, float scale, bf16* out, int ldo) {
    pdl_wait();
    pdl_trigger();     // only now: a successor that is resident earlier just holds SM resources while it waits (measured)
    bias_act_body(partial, splitk, T, N, ldp, bias, act, scale, out, ldo, blockIdx.x);
}

cudaError_t launch_bias_act(cudaStream_t stream, const float* partial, int splitk, int T, int N, int ldp,
                            const bf16* bias, int act, float scale, bf16* out, int ldo) {
    if ((N & 3) || (ldp & 3)) return cudaErrorInvalidValue;
    const int total = T * (N >> 2);
    return launch_kernel(bias_act_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, partial, splitk, T, N,
                         ldp, bias, act, scale, out, ldo);
}

__global__ void __launch_bounds__(384) rope_kv_kernel(const RopeKvArgs a) {
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();     // only now: a successor that is resident earlier just holds SM resources while it waits (measured)
    trace_stamp(a.trace, 1);
    rope_kv_body<false>(a, blockIdx.x);
    trace_stamp(a.trace, 2);
}

// Batched episodes, bf16 hand-off mode: fixed grid, one work item per thread, next row's inputs fetched early.
__global__ void __launch_bounds__(384) rope_kv_stream_kernel(const RopeKvArgs a) {
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    int t = blockIdx.x;
    RopeItemIn cur, nxt;
    if (t < a.T) rope_prefetch(a, t, cur);
    for (; t < a.T; t += gridDim.x) {
        const int tn = t + gridDim.x;
        if (tn < a.T) rope_prefetch(a, tn, nxt);
        rope_kv_body<true>(a, t, &cur);
        cur = nxt;
    }
    trace_stamp(a.trace, 2);
}

cudaError_t launch_rope_kv(cudaStream_t stream, const RopeKvArgs& a) {
    if (a.ldp & 3) return cudaErrorInvalidValue;
    if (a.lin != nullptr && a.T >= kStreamMinRows) {
        const int items = (a.n_heads + 1) * 32 + 64;
        if (items <= 384)
            return launch_kernel(rope_kv_stream_kernel, dim3(148 * 5), dim3((items + 31) / 32 * 32), 0, stream, a);
    }
    // one work item (4 rotated pairs or 4 value columns) per thread: (n_heads + 1) * 32 + 64 items per token
    const int items = (a.n_heads + 1) * 32 + 64;
    const int threads = items <= 384 ? (items + 31) / 32 * 32 : 256;
    return launch_kernel(rope_kv_kernel, dim3(a.T), dim3(threads), 0, stream, a);
}

__global__ void rope_table_kernel(const float* __restrict__ inv_freq, int n_pos, float* __restrict__ cos_t,
                                  float* __restrict__ sin_t) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_pos * 128) return;
    const int pos = idx >> 7, j = idx & 127;
    // GemmaRotaryEmbedding.forward (paligemma/modules.py:47-67): fp32 angle, cos/sin -> model dtype
    const float angle = __fmul_rn(inv_freq[j], static_cast<float>(pos));
    cos_t[idx] = bf16_round(cosf(angle));
    sin_t[idx] = bf16_round(sinf(angle));
}

cudaError_t launch_rope_table(cudaStream_t stream, const float* inv_freq, int n_pos, float* cos_t,
                              float* sin_t) {
    const int total = n_pos * 128;
    rope_table_kernel<<<(total + 255) / 256, 256, 0, stream>>>(inv_freq, n_pos, cos_t, sin_t);
    return cudaGetLastError();
}

}  // namespace blurr
