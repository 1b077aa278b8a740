// Attention kernels of the Pi-0 path.
//
//  * attn_mma_kernel<HD_PAD, BM, GEMMA>: "full-row" attention, BM query rows per CTA (16 at batch 1,
//    32/64 for batched episodes), for the many-query cases
//      - SigLIP MHA, 16 heads x 256 tokens x head_dim 72 (siglip.py:133-152), no mask;
//      - Gemma joint-attention prefill, 8 query heads sharing one KV head (MQA), 276 query rows
//        x 277 keys x head_dim 256 with tanh soft-clamp and additive block mask
//        (joint_model.py:273-288).
//    The tiles are tiny (<= 64 x 320 logits), so they run on warp-level mma.sync (bf16, fp32
//    accumulate) with ldmatrix-fed fragments; the whole logit row is kept in shared memory so
//    the softmax is the reference's exact two-pass fp32 softmax over bf16-rounded logits.
//  * few-query mode of the same kernel: 1 (proprio) or 4 (action) query rows per sample over the
//    KV cache (joint_model.py:164-170 "append_non_active"); the (head, query) pairs of a sample
//    form the tile rows, so the sample's single K/V head is read once for all 8 query heads.
//
// Rounding points (SURVEY.md Appendix A.2/A.6): QK^T -> bf16; every scale / tanh / mask op
// -> bf16; softmax in fp32 -> bf16; PV -> bf16.  Divisions by Python scalars are done as the
// ATen CUDA kernels do them (multiplication by the fp32 reciprocal).
#include "bodies.cuh"
#include "launch.cuh"

#include <string>

namespace blurr {

template <int HD_PAD, int BM, int GEMMA>
__global__ void __launch_bounds__(kAttnThreads) attn_mma_kernel(const AttnMmaArgs a) {
    extern __shared__ __align__(16) uint8_t smem_attn[];
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();     // only now: a successor that is resident earlier just holds SM resources while it waits (measured)
    trace_stamp(a.trace, 1);
    attn_mma_body<HD_PAD, BM, GEMMA>(a, smem_attn, blockIdx.x, blockIdx.y, blockIdx.z);
    trace_stamp(a.trace, 2);
}

AttnMmaArgs make_siglip_attn_args(const bf16* qkv, int ld_qkv, int seq, int n_heads, int hidden, bf16* out,
                                  int ld_out) {
    AttnMmaArgs a{};
    a.trace = nullptr;
    const int hd = hidden / n_heads;           // 72
    a.q = qkv; a.ldq = ld_qkv; a.q_col0 = 0; a.q_per_sample = seq;
    a.k = qkv; a.ldk = ld_qkv; a.k_col0 = hidden; a.kv_per_sample = seq;
    a.v = qkv; a.ldv = ld_qkv; a.v_col0 = 2 * hidden;
    a.out = out; a.ldo = ld_out; a.o_col0 = 0;
    a.hd = hd; a.head_stride_q = hd; a.head_stride_kv = hd; a.n_keys = seq;
    // Python: head_dim ** -0.5 evaluated in double, then used as an fp32 scalar operand
    a.scale = static_cast<float>(pow(static_cast<double>(hd), -0.5));
    a.mask = nullptr;
    return a;
}

AttnMmaArgs make_prefill_attn_args(const JointAttnArgs& j) {
    AttnMmaArgs a{};
    a.q = j.q; a.ldq = j.n_heads * 256; a.q_col0 = 0; a.q_per_sample = j.q_per_sample;
    a.k = j.k_cache; a.ldk = 256; a.k_col0 = 0; a.kv_per_sample = j.n_slots;
    a.v = j.v_cache; a.ldv = 256; a.v_col0 = 0;
    a.out = j.out; a.ldo = j.n_heads * 256; a.o_col0 = 0;
    a.hd = 256; a.head_stride_q = 256; a.head_stride_kv = 0; a.n_keys = j.n_keys;
    a.scale = 0.f;
    a.mask = j.mask; a.mask_bstride = j.mask_bstride; a.mask_rstride = j.mask_rstride;
    a.q_row_offset = j.q_row_offset;
    a.trace = j.trace;
    return a;
}

// Few queries per sample (proprio: 1, action: 4): the (head, query) pairs of a sample form the rows of
// the same tensor-core tile kernel — all 8 query heads share the sample's single K/V head (MQA), so
// K and V are read once per 16 pairs instead of once per head.
AttnMmaArgs make_fewq_attn_args(const JointAttnArgs& j) {
    AttnMmaArgs a = make_prefill_attn_args(j);
    a.head_stride_q = 256;
    a.mqa_nq = j.q_per_sample;
    a.mqa_heads = j.n_heads;
    return a;
}

static constexpr size_t kAttnSmemMax = 215 * 1024;

template <int HD_PAD, int BM, int GEMMA>
static cudaError_t launch_attn(cudaStream_t stream, const AttnMmaArgs& a, int rows, int heads, int batch) {
    const size_t smem = attn_smem_bytes<HD_PAD, BM>(a.n_keys);
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(attn_mma_kernel<HD_PAD, BM, GEMMA>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kAttnSmemMax));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    if (smem > kAttnSmemMax) return cudaErrorInvalidValue;
    dim3 grid((rows + BM - 1) / BM, heads, batch);
    return launch_kernel(attn_mma_kernel<HD_PAD, BM, GEMMA>, grid, dim3(kAttnThreads), smem, stream, a);
}

// rows per tile: 16 while that already gives every SM a couple of tiles, larger tiles beyond
int attn_tile_rows(int rows, int heads, int batch, int max_rows) {
    const long tiles16 = static_cast<long>((rows + 15) / 16) * heads * batch;
    if (tiles16 <= 2 * 148 || max_rows <= 16) return 16;
    const long tiles32 = static_cast<long>((rows + 31) / 32) * heads * batch;
    if (tiles32 <= 4 * 148 || max_rows <= 32) return 32;
    return 64;
}

bool attn_tc_siglip_applies(int batch, int seq, int n_heads, int hidden);
cudaError_t launch_siglip_attention_tc(cudaStream_t stream, const bf16* qkv, int ld_qkv, int batch, int seq, int n_heads,
                                       int hidden, bf16* out, int ld_out, unsigned long long* trace);

static bool siglip_stream_applies(const AttnMmaArgs& a, int seq, int n_heads, int batch);
static cudaError_t launch_siglip_stream(cudaStream_t stream, const AttnMmaArgs& a, int seq, int n_heads, int batch);

cudaError_t launch_siglip_attention(cudaStream_t stream, const bf16* qkv, int ld_qkv, int batch, int seq,
                                    int n_heads, int hidden, bf16* out, int ld_out, unsigned long long* trace) {
    const int hd = hidden / n_heads;
    if (hd > 80 || seq > kAttnMaxBlocks * kBK) return cudaErrorInvalidValue;
    {
        AttnMmaArgs sa = make_siglip_attn_args(qkv, ld_qkv, seq, n_heads, hidden, out, ld_out);
        sa.trace = trace;
        if (siglip_stream_applies(sa, seq, n_heads, batch)) return launch_siglip_stream(stream, sa, seq, n_heads, batch);
    }
    if (attn_tc_siglip_applies(batch, seq, n_heads, hidden))
        return launch_siglip_attention_tc(stream, qkv, ld_qkv, batch, seq, n_heads, hidden, out, ld_out, trace);
    AttnMmaArgs a = make_siglip_attn_args(qkv, ld_qkv, seq, n_heads, hidden, out, ld_out);
    a.trace = trace;
    switch (attn_tile_rows(seq, n_heads, batch, 64)) {
        case 16: return launch_attn<80, 16, false>(stream, a, seq, n_heads, batch);
        case 32: return launch_attn<80, 32, false>(stream, a, seq, n_heads, batch);
        default: return launch_attn<80, 64, false>(stream, a, seq, n_heads, batch);
    }
}

cudaError_t launch_joint_attention_prefill_tc(cudaStream_t stream, const JointAttnArgs& j, std::string* err);

static bool prefill_stream_applies(const JointAttnArgs& j);
static cudaError_t launch_prefill_stream(cudaStream_t stream, const JointAttnArgs& j);

cudaError_t launch_joint_attention_prefill(cudaStream_t stream, const JointAttnArgs& j) {
    if (j.n_keys > kAttnMaxBlocks * kBK) return cudaErrorInvalidValue;
    if (prefill_stream_applies(j)) return launch_prefill_stream(stream, j);      // one or two episodes: streaming kernel
    if (attn_tc_applies(j)) {
        std::string err;
        return launch_joint_attention_prefill_tc(stream, j, &err);
    }
    AttnMmaArgs a = make_prefill_attn_args(j);
    if (attn_tile_rows(j.q_per_sample, j.n_heads, j.batch, 32) == 16)
        return launch_attn<256, 16, true>(stream, a, j.q_per_sample, j.n_heads, j.batch);
    return launch_attn<256, 32, true>(stream, a, j.q_per_sample, j.n_heads, j.batch);
}


// ---------------------------------------------------------------------------------------------
// Few-query joint attention as a streaming kernel (the experts: 1 proprio / 4 action queries per sample, 8 query heads
// over ONE shared K/V head, <= 288 keys).  The tile kernel above spends its time in dependent phases (K blocks, logits,
// V blocks into the same buffers, P.V): ~13 us for 0.6 MFLOP.  Here a CTA owns 8 (head, query) rows of one sample and
// requests everything it will read at once:
//  * K straight from global into mma.sync B fragments (no shared memory): the dot product does not care in which order
//    the 256 dims are summed, so k-steps 2t / 2t+1 of lane (g, c) are DEFINED as dims 32t + 8c .. + 7 - one 16-byte load
//    per lane per t for the key row g of its 8-key tile, and the same permutation for the query row's A fragments;
//  * all of V into shared memory with cp.async (read back with ldmatrix.trans for P.V).
// 18 warps x 2 key tiles x 8 keys = 288 keys.  Same rounding chain as attn_mma_body<256, ., 1> (joint_model.py:246-288):
// bf16(q.k) / 16 -> bf16(/50) -> bf16(tanh) -> bf16(*50) -> bf16(+ mask) -> fp32 softmax -> bf16 -> P.V in fp32.
// ---------------------------------------------------------------------------------------------
static constexpr int kFqWarps = 18;
static constexpr int kFqThreads = kFqWarps * 32;
static constexpr int kFqMaxKeys = kFqWarps * 16;                 // 288
static constexpr int kFqRows = 8;
static constexpr int kFqLdV = 256 + 8;                           // V row stride in shared memory (elements): conflict-free ldmatrix
static constexpr int kFqLdP = kFqMaxKeys + 8;
static constexpr size_t kFqSmem = static_cast<size_t>(kFqMaxKeys) * kFqLdV * 2 + kFqRows * kFqLdP * 4 + kFqRows * kFqLdP * 2;

__global__ void __launch_bounds__(kFqThreads, 1) fewq_stream_kernel(const JointAttnArgs j) {
    extern __shared__ __align__(16) uint8_t fq_smem[];
    bf16* v_s = reinterpret_cast<bf16*>(fq_smem);                                                   // [288][264]
    float* sc = reinterpret_cast<float*>(fq_smem + static_cast<size_t>(kFqMaxKeys) * kFqLdV * 2);   // [8][296] logits
    bf16* p_s = reinterpret_cast<bf16*>(sc + kFqRows * kFqLdP);                                     // [8][296] probabilities
    trace_stamp(j.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(j.trace, 1);
    const int b = blockIdx.y, tile = blockIdx.x;
    const int nq = j.q_per_sample, rows_total = j.n_heads * nq, n = j.n_keys;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, c = lane & 3;
    const bf16* kb = j.k_cache + static_cast<size_t>(b) * j.n_slots * 256;
    const bf16* vb = j.v_cache + static_cast<size_t>(b) * j.n_slots * 256;
    // ---- everything this CTA reads, requested up front ----
    for (int i = threadIdx.x; i < kFqMaxKeys * 32; i += kFqThreads) {
        const int key = i >> 5, ch = i & 31;
        const bool valid = key < n;                           // rows past n_keys are zero-filled (their probabilities are 0)
        cp_async_16(v_s + key * kFqLdV + ch * 8, valid ? vb + static_cast<size_t>(key) * 256 + ch * 8 : vb, valid);
    }
    cp_async_commit();
    uint4 kr[2][8];
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        const int key = (warp * 2 + t2) * 8 + g;
#pragma unroll
        for (int t = 0; t < 8; ++t)
            kr[t2][t] = key < n ? __ldcg(reinterpret_cast<const uint4*>(kb + static_cast<size_t>(key) * 256 + 32 * t + 8 * c))
                                : make_uint4(0u, 0u, 0u, 0u);
    }
    // row g of this tile -> (head, query)
    const int p = tile * kFqRows + g;
    const bool row_valid = p < rows_total;
    const int head = row_valid ? p / nq : 0, qi = row_valid ? p - head * nq : 0;
    const bf16* qrow = j.q + (static_cast<size_t>(b) * nq + qi) * (j.n_heads * 256) + head * 256;
    uint4 qr[8];
#pragma unroll
    for (int t = 0; t < 8; ++t)
        qr[t] = row_valid ? *reinterpret_cast<const uint4*>(qrow + 32 * t + 8 * c) : make_uint4(0u, 0u, 0u, 0u);
    // ---- logits: 2 key tiles x 16 k-steps of m16n8k16 (rows 8..15 of A are zero) ----
    const bf16* mrow = row_valid ? j.mask + static_cast<size_t>(b) * j.mask_bstride +
                                       static_cast<size_t>(j.q_row_offset + qi) * j.mask_rstride
                                 : nullptr;
    // the additive mask values of this lane's logits, requested with everything else (not after the MMAs)
    float mk[2][2];
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int k = (warp * 2 + t2) * 8 + 2 * c + e;
            mk[t2][e] = (mrow != nullptr && k < n) ? bf2f(mrow[k]) : 0.f;
        }
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const uint32_t a0[4] = {qr[t].x, 0u, qr[t].y, 0u};
            mma_bf16_16816(acc, a0, kr[t2][t].x, kr[t2][t].y);
            const uint32_t a1[4] = {qr[t].z, 0u, qr[t].w, 0u};
            mma_bf16_16816(acc, a1, kr[t2][t].z, kr[t2][t].w);
        }
        // acc[0], acc[1]: row g, keys key0 + 2c, + 1
        const int key0 = (warp * 2 + t2) * 8 + 2 * c;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int k = key0 + e;
            float s0 = bf16_round(acc[e]) * 0.0625f;          // / sqrt(256): exact
            s0 = bf16_round(s0 * (1.0f / 50.0f));
            s0 = bf16_round(tanhf(s0));
            s0 = bf16_round(s0 * 50.0f);
            if (mrow != nullptr && k < n) s0 = bf16_round(s0 + mk[t2][e]);
            sc[g * kFqLdP + k] = s0;
        }
    }
    __syncthreads();
    // ---- softmax: fp32 over the bf16 logits, probabilities rounded to bf16 ----
    if (warp < kFqRows) {
        const float* row = sc + warp * kFqLdP;
        constexpr int PER_LANE = kFqMaxKeys / 32;            // 9
        float x[PER_LANE];
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? row[col] : -INFINITY;
            m = fmaxf(m, x[i]);
        }
        m = warp_max(m);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? expf(x[i] - m) : 0.f;
            sum += x[i];
        }
        sum = warp_sum(sum);
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) p_s[warp * kFqLdP + lane + i * 32] = f2bf(x[i] / sum);
    }
    cp_async_wait<0>();
    __syncthreads();
    // ---- O = P V: warps 0..15 own 16 output dims each ----
    if (warp < 16) {
        float oacc[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int e = 0; e < 4; ++e) oacc[i][e] = 0.f;
        const int dim0 = warp * 16;
#pragma unroll 3
        for (int ks = 0; ks < kFqMaxKeys / 16; ++ks) {
            uint32_t pa[2];
            // lanes 0..7: rows of the (keys ks*16 .. +7) matrix, lanes 8..15: the (+8 .. +15) matrix
            ldmatrix_x2(pa, smem_u32(p_s + (lane & 7) * kFqLdP + ks * 16 + ((lane >> 3) & 1) * 8));
            const uint32_t af[4] = {pa[0], 0u, pa[1], 0u};
            uint32_t bfr[4];
            const int mi = lane >> 3;
            const int key = ks * 16 + (mi & 1) * 8 + (lane & 7);
            const int dim = dim0 + (mi >> 1) * 8;
            ldmatrix_x4_trans(bfr, smem_u32(v_s + key * kFqLdV + dim));
            mma_bf16_16816(oacc[0], af, bfr[0], bfr[1]);
            mma_bf16_16816(oacc[1], af, bfr[2], bfr[3]);
        }
        if (row_valid) {
            bf16* orow = j.out + (static_cast<size_t>(b) * nq + qi) * (j.n_heads * 256) + head * 256 + dim0 + 2 * c;
            *reinterpret_cast<uint32_t*>(orow) = pack_bf16x2(oacc[0][0], oacc[0][1]);
            *reinterpret_cast<uint32_t*>(orow + 8) = pack_bf16x2(oacc[1][0], oacc[1][1]);
        }
    }
    trace_stamp(j.trace, 2);
}

// The same streaming design for the PREFILL at one or two episodes (276 queries x 8 heads = 2208 rows per sample): a CTA owns
// 16 rows = 2 queries x 8 heads (all heads share the K/V head, and rows of one query share a mask row), so 138 CTAs cover
// a sample in ONE wave, each reading the sample's K (registers) and V (shared memory) once from L2 - 40 MB of L2 traffic
// per layer, fine for a couple of samples, absurd for 64 (those keep the tcgen05 kernel, which reads K/V once per 128
// rows).  A fragments come from a shared-memory copy of the 16 query rows whose columns are stored in the permuted order
// of the K fragments (see fewq_stream_kernel), so a plain ldmatrix yields matching k indices.
static constexpr int kPsRows = 16;
static constexpr int kPsLdQ = 256 + 8;
static constexpr size_t kPsSmem = static_cast<size_t>(kFqMaxKeys) * kFqLdV * 2 + kPsRows * kPsLdQ * 2 + kPsRows * kFqLdP * 4 +
                                  kPsRows * kFqLdP * 2;

__global__ void __launch_bounds__(kFqThreads, 1) prefill_stream_kernel(const JointAttnArgs j) {
    extern __shared__ __align__(16) uint8_t ps_smem[];
    bf16* v_s = reinterpret_cast<bf16*>(ps_smem);                                                   // [288][264]
    bf16* q_s = v_s + static_cast<size_t>(kFqMaxKeys) * kFqLdV;                                     // [16][264], permuted columns
    float* sc = reinterpret_cast<float*>(q_s + kPsRows * kPsLdQ);                                   // [16][296]
    bf16* p_s = reinterpret_cast<bf16*>(sc + kPsRows * kFqLdP);                                     // [16][296]
    trace_stamp(j.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(j.trace, 1);
    const int b = blockIdx.y, tile = blockIdx.x;
    const int qps = j.q_per_sample, nh = j.n_heads, rows_total = nh * qps, n = j.n_keys;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, c = lane & 3;
    const bf16* kb = j.k_cache + static_cast<size_t>(b) * j.n_slots * 256;
    const bf16* vb = j.v_cache + static_cast<size_t>(b) * j.n_slots * 256;
    for (int i = threadIdx.x; i < kFqMaxKeys * 32; i += kFqThreads) {
        const int key = i >> 5, ch = i & 31;
        const bool valid = key < n;
        cp_async_16(v_s + key * kFqLdV + ch * 8, valid ? vb + static_cast<size_t>(key) * 256 + ch * 8 : vb, valid);
    }
    cp_async_commit();
    uint4 kr[2][8];
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        const int key = (warp * 2 + t2) * 8 + g;
#pragma unroll
        for (int t = 0; t < 8; ++t)
            kr[t2][t] = key < n ? __ldcg(reinterpret_cast<const uint4*>(kb + static_cast<size_t>(key) * 256 + 32 * t + 8 * c))
                                : make_uint4(0u, 0u, 0u, 0u);
    }
    // rows g and g + 8 of this tile
    const bf16* mrow[2];
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const int p = tile * kPsRows + g + hh * 8;
        mrow[hh] = p < rows_total ? j.mask + static_cast<size_t>(b) * j.mask_bstride +
                                        static_cast<size_t>(j.q_row_offset + p / nh) * j.mask_rstride
                                  : nullptr;
    }
    float mk[2][2][2];                 // [key tile][row half][key]: requested before the MMAs
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = (warp * 2 + t2) * 8 + 2 * c + e;
                mk[t2][hh][e] = (mrow[hh] != nullptr && k < n) ? bf2f(mrow[hh][k]) : 0.f;
            }
    // query rows -> shared memory, dims (d, d + 1) of row r stored at the column the K fragments use for them
    for (int i = threadIdx.x; i < kPsRows * 128; i += kFqThreads) {
        const int r = i >> 7, d = (i & 127) << 1;
        const int p = tile * kPsRows + r;
        uint32_t val = 0u;
        if (p < rows_total) {
            const int query = p / nh, head = p - query * nh;
            val = *reinterpret_cast<const uint32_t*>(j.q + (static_cast<size_t>(b) * qps + query) * (nh * 256) + head * 256 + d);
        }
        const int t = d >> 5, rr = d & 31, cc = rr >> 3, o = rr & 7;
        const int col = (2 * t + (o >> 2)) * 16 + 2 * cc + ((o & 2) ? 8 : 0);
        *reinterpret_cast<uint32_t*>(q_s + r * kPsLdQ + col) = val;
    }
    __syncthreads();
#pragma unroll
    for (int t2 = 0; t2 < 2; ++t2) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 16; ++ks) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(q_s + (lane & 15) * kPsLdQ + ks * 16 + (lane >> 4) * 8));
            const uint4 kk = kr[t2][ks >> 1];
            if (ks & 1) mma_bf16_16816(acc, af, kk.z, kk.w);
            else mma_bf16_16816(acc, af, kk.x, kk.y);
        }
        const int key0 = (warp * 2 + t2) * 8 + 2 * c;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = key0 + e;
                float s0 = bf16_round(acc[hh * 2 + e]) * 0.0625f;
                s0 = bf16_round(s0 * (1.0f / 50.0f));
                s0 = bf16_round(tanhf(s0));
                s0 = bf16_round(s0 * 50.0f);
                if (mrow[hh] != nullptr && k < n) s0 = bf16_round(s0 + mk[t2][hh][e]);
                sc[(g + hh * 8) * kFqLdP + k] = s0;
            }
        }
    }
    __syncthreads();
    if (warp < kPsRows) {
        const float* row = sc + warp * kFqLdP;
        constexpr int PER_LANE = kFqMaxKeys / 32;
        float x[PER_LANE];
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? row[col] : -INFINITY;
            m = fmaxf(m, x[i]);
        }
        m = warp_max(m);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? expf(x[i] - m) : 0.f;
            sum += x[i];
        }
        sum = warp_sum(sum);
#pragma unroll
        for (int i = 0; i < PER_LANE; ++i) p_s[warp * kFqLdP + lane + i * 32] = f2bf(x[i] / sum);
    }
    cp_async_wait<0>();
    __syncthreads();
    if (warp < 16) {
        float oacc[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int e = 0; e < 4; ++e) oacc[i][e] = 0.f;
        const int dim0 = warp * 16;
#pragma unroll 3
        for (int ks = 0; ks < kFqMaxKeys / 16; ++ks) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(p_s + (lane & 15) * kFqLdP + ks * 16 + (lane >> 4) * 8));
            uint32_t bfr[4];
            const int mi = lane >> 3;
            const int key = ks * 16 + (mi & 1) * 8 + (lane & 7);
            const int dim = dim0 + (mi >> 1) * 8;
            ldmatrix_x4_trans(bfr, smem_u32(v_s + key * kFqLdV + dim));
            mma_bf16_16816(oacc[0], af, bfr[0], bfr[1]);
            mma_bf16_16816(oacc[1], af, bfr[2], bfr[3]);
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int p = tile * kPsRows + g + hh * 8;
            if (p >= rows_total) continue;
            const int query = p / nh, head = p - query * nh;
            bf16* orow = j.out + (static_cast<size_t>(b) * qps + query) * (nh * 256) + head * 256 + dim0 + 2 * c;
            *reinterpret_cast<uint32_t*>(orow) = pack_bf16x2(oacc[0][hh * 2], oacc[0][hh * 2 + 1]);
            *reinterpret_cast<uint32_t*>(orow + 8) = pack_bf16x2(oacc[1][hh * 2], oacc[1][hh * 2 + 1]);
        }
    }
    trace_stamp(j.trace, 2);
}

static int g_prefill_stream = 1;
void attn_set_prefill_stream(int on) { g_prefill_stream = on; }
static bool prefill_stream_applies(const JointAttnArgs& j) {
    if (!g_prefill_stream || j.n_keys > kFqMaxKeys || j.mask == nullptr) return false;
    const long tiles = (static_cast<long>(j.n_heads) * j.q_per_sample + kPsRows - 1) / kPsRows;
    return tiles * j.batch <= 2 * 148;          // every CTA re-reads the sample's K/V from L2: only worth it within two waves
}
static cudaError_t launch_prefill_stream(cudaStream_t stream, const JointAttnArgs& j) {
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(prefill_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kPsSmem));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    const int rows = j.n_heads * j.q_per_sample;
    return launch_kernel(prefill_stream_kernel, dim3((rows + kPsRows - 1) / kPsRows, j.batch), dim3(kFqThreads), kPsSmem, stream, j);
}

// SigLIP self-attention (siglip.py:133-152) at one or two images, the same streaming design: a CTA owns 32 query rows of
// one head (8 tiles x 16 heads = 128 CTAs per image: one wave), its 8 warps take 32 keys each straight into permuted
// B fragments (head_dim 72 = dims 0..63 in two 16-byte steps + one more that only lane column 0 fills), V (256 x 72) goes
// to shared memory with cp.async, the logits are bf16(bf16(q.k) * scale), fp32 softmax, bf16 P, P.V by mma.sync.
static constexpr int kSsThreads = 256;
static constexpr int kSsRows = 32;
static constexpr int kSsKeys = 256;
static constexpr int kSsLdV = 96 + 8;         // up to 96 head dims
static constexpr int kSsLdQ = 96 + 8;
static constexpr int kSsLdP = kSsKeys + 8;
static constexpr size_t kSsSmem = static_cast<size_t>(kSsKeys) * kSsLdV * 2 + kSsRows * kSsLdQ * 2 + kSsRows * kSsLdP * 4 + kSsRows * kSsLdP * 2;

__global__ void __launch_bounds__(kSsThreads) siglip_stream_kernel(const AttnMmaArgs a) {
    extern __shared__ __align__(16) uint8_t ss_smem[];
    bf16* v_s = reinterpret_cast<bf16*>(ss_smem);                                    // [256][104]
    bf16* q_s = v_s + kSsKeys * kSsLdV;                                              // [32][104], permuted columns
    float* sc = reinterpret_cast<float*>(q_s + kSsRows * kSsLdQ);                    // [32][264]
    bf16* p_s = reinterpret_cast<bf16*>(sc + kSsRows * kSsLdP);                      // [32][264]
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    const int tile = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int n = a.n_keys, hd = a.hd, rows_total = a.q_per_sample;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, c = lane & 3;
    const bf16* qbase = a.q + static_cast<size_t>(b) * a.q_per_sample * a.ldq + a.q_col0 + h * a.head_stride_q;
    const bf16* kbase = a.k + static_cast<size_t>(b) * a.kv_per_sample * a.ldk + a.k_col0 + h * a.head_stride_kv;
    const bf16* vbase = a.v + static_cast<size_t>(b) * a.kv_per_sample * a.ldv + a.v_col0 + h * a.head_stride_kv;
    const int vch = hd >> 3;                                   // 16-byte chunks per V row (9)
    for (int i = threadIdx.x; i < kSsKeys * 12; i += kSsThreads) {
        const int key = i / 12, ch = i - key * 12;
        const bool valid = key < n && ch < vch;                // the rest is zero-filled: padded dims / keys contribute 0
        cp_async_16(v_s + key * kSsLdV + ch * 8, valid ? vbase + static_cast<size_t>(key) * a.ldv + ch * 8 : vbase, valid);
    }
    cp_async_commit();
    uint4 kr[4][3];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        const int key = warp * 32 + nt * 8 + g;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const int d = 32 * t + 8 * c;
            kr[nt][t] = (key < n && d < hd) ? __ldcg(reinterpret_cast<const uint4*>(kbase + static_cast<size_t>(key) * a.ldk + d))
                                            : make_uint4(0u, 0u, 0u, 0u);
        }
    }
    for (int i = threadIdx.x; i < kSsRows * 48; i += kSsThreads) {
        const int r = i / 48, d = (i - r * 48) << 1;
        const int row = tile * kSsRows + r;
        uint32_t val = 0u;
        if (row < rows_total && d < hd) val = *reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(row) * a.ldq + d);
        const int t = d >> 5, rr = d & 31, cc = rr >> 3, o = rr & 7;
        const int col = (2 * t + (o >> 2)) * 16 + 2 * cc + ((o & 2) ? 8 : 0);
        *reinterpret_cast<uint32_t*>(q_s + r * kSsLdQ + col) = val;
    }
    __syncthreads();
    // ---- logits: 2 row tiles x 4 key tiles x 6 k-steps ----
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        uint32_t af[6][4];
#pragma unroll
        for (int ks = 0; ks < 6; ++ks)
            ldmatrix_x4(af[ks], smem_u32(q_s + (mt * 16 + (lane & 15)) * kSsLdQ + ks * 16 + (lane >> 4) * 8));
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int ks = 0; ks < 6; ++ks) {
                const uint4 kk = kr[nt][ks >> 1];
                if (ks & 1) mma_bf16_16816(acc, af[ks], kk.z, kk.w);
                else mma_bf16_16816(acc, af[ks], kk.x, kk.y);
            }
            const int key0 = warp * 32 + nt * 8 + 2 * c;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    sc[(mt * 16 + g + hh * 8) * kSsLdP + key0 + e] = bf16_round(bf16_round(acc[hh * 2 + e]) * a.scale);
        }
    }
    __syncthreads();
    // ---- softmax: 4 rows per warp ----
    for (int rr = 0; rr < kSsRows / 8; ++rr) {
        const int r = warp * (kSsRows / 8) + rr;
        const float* row = sc + r * kSsLdP;
        float x[kSsKeys / 32];
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < kSsKeys / 32; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? row[col] : -INFINITY;
            m = fmaxf(m, x[i]);
        }
        m = warp_max(m);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < kSsKeys / 32; ++i) {
            const int col = lane + i * 32;
            x[i] = col < n ? expf(x[i] - m) : 0.f;
            sum += x[i];
        }
        sum = warp_sum(sum);
#pragma unroll
        for (int i = 0; i < kSsKeys / 32; ++i) p_s[r * kSsLdP + lane + i * 32] = f2bf(x[i] / sum);
    }
    cp_async_wait<0>();
    __syncthreads();
    // ---- O = P V: warp -> row tile (warp & 1), output 8-dim tiles (warp >> 1) + 4 i ----
    {
        const int mt = warp & 1;
        const int n_tiles = (hd + 7) >> 3;
        float oacc[3][4];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int e = 0; e < 4; ++e) oacc[i][e] = 0.f;
#pragma unroll 4
        for (int ks = 0; ks < kSsKeys / 16; ++ks) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(p_s + (mt * 16 + (lane & 15)) * kSsLdP + ks * 16 + (lane >> 4) * 8));
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int nt = (warp >> 1) + 4 * i;
                if (nt >= n_tiles) continue;                       // warp-uniform
                uint32_t bfr[2];
                // x2.trans: lanes 0..7 -> keys ks*16 .. +7, lanes 8..15 -> keys +8 .. +15 of dim tile nt
                ldmatrix_x2_trans(bfr, smem_u32(v_s + (ks * 16 + (lane & 15)) * kSsLdV + nt * 8));
                mma_bf16_16816(oacc[i], af, bfr[0], bfr[1]);
            }
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int nt = (warp >> 1) + 4 * i;
            if (nt >= n_tiles) continue;
            const int dim = nt * 8 + 2 * c;
            if (dim >= hd) continue;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int row = tile * kSsRows + mt * 16 + g + hh * 8;
                if (row >= rows_total) continue;
                bf16* dst = a.out + static_cast<size_t>(b) * a.q_per_sample * a.ldo + static_cast<size_t>(row) * a.ldo + a.o_col0 +
                            h * a.head_stride_q + dim;
                *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(oacc[i][hh * 2], oacc[i][hh * 2 + 1]);
            }
        }
    }
    trace_stamp(a.trace, 2);
}

static int g_siglip_stream = 1;
void attn_set_siglip_stream(int on) { g_siglip_stream = on; }
static bool siglip_stream_applies(const AttnMmaArgs& a, int seq, int n_heads, int batch) {
    if (!g_siglip_stream || seq > kSsKeys || a.hd > 96 || (a.hd & 7)) return false;
    return static_cast<long>((seq + kSsRows - 1) / kSsRows) * n_heads * batch <= 2 * 148;
}
static cudaError_t launch_siglip_stream(cudaStream_t stream, const AttnMmaArgs& a, int seq, int n_heads, int batch) {
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(siglip_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSsSmem));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    return launch_kernel(siglip_stream_kernel, dim3((seq + kSsRows - 1) / kSsRows, n_heads, batch), dim3(kSsThreads), kSsSmem, stream, a);
}

static int g_fewq_stream = 1;
void attn_set_fewq_stream(int on) { g_fewq_stream = on; }

static cudaError_t launch_fewq_stream(cudaStream_t stream, const JointAttnArgs& j) {
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(fewq_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFqSmem));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    const int rows = j.n_heads * j.q_per_sample;
    return launch_kernel(fewq_stream_kernel, dim3((rows + kFqRows - 1) / kFqRows, j.batch), dim3(kFqThreads), kFqSmem, stream, j);
}

cudaError_t launch_joint_attention_fewq(cudaStream_t stream, const JointAttnArgs& j) {
    if (g_fewq_stream && j.n_keys <= kFqMaxKeys && j.mask != nullptr) return launch_fewq_stream(stream, j);
    if (j.n_keys > kAttnMaxBlocks * kBK) return cudaErrorInvalidValue;
    if (attn_tc_fewq_applies(j)) {
        std::string err;
        return launch_joint_attention_prefill_tc(stream, j, &err);
    }
    AttnMmaArgs a = make_fewq_attn_args(j);
    const int pairs = j.n_heads * j.q_per_sample;
    if (attn_tile_rows(pairs, 1, j.batch, 32) == 16) return launch_attn<256, 16, true>(stream, a, pairs, 1, j.batch);
    return launch_attn<256, 32, true>(stream, a, pairs, 1, j.batch);
}

// Llama-style multi-head attention over a token-major KV cache (llm_engine.cu): head_dim 128 (or 64), one K/V head per
// query head, causal by position.  Prefill (many query rows) and decode (one row per sequence) share the kernel.
cudaError_t launch_mha_decode(cudaStream_t stream, const MhaAttnArgs& a, const RopeMhaArgs* rope);     // llm_kernels.cu

cudaError_t launch_mha_attention(cudaStream_t stream, const MhaAttnArgs& m, const RopeMhaArgs* fused_rope) {
    if (m.n_keys > kAttnMaxBlocks * kBK || m.n_kv_heads != m.n_heads) return cudaErrorInvalidValue;
    if (m.q_per_sample == 1) return launch_mha_decode(stream, m, fused_rope);       // decode: K/V streaming, no tensor cores
    if (fused_rope != nullptr) return cudaErrorInvalidValue;
    AttnMmaArgs a{};
    const int width = m.n_heads * m.head_dim;
    a.q = m.q; a.ldq = width; a.q_col0 = 0; a.q_per_sample = m.q_per_sample;
    a.k = m.k_cache; a.ldk = width; a.k_col0 = 0; a.kv_per_sample = m.n_slots;
    a.v = m.v_cache; a.ldv = width; a.v_col0 = 0;
    a.out = m.out; a.ldo = width; a.o_col0 = 0;
    a.hd = m.head_dim; a.head_stride_q = m.head_dim; a.head_stride_kv = m.head_dim; a.n_keys = m.n_keys;
    a.scale = m.scale; a.mask = nullptr; a.q_row_offset = m.q_pos0; a.trace = m.trace;
    const int bm = attn_tile_rows(m.q_per_sample, m.n_heads, m.batch, 64);
    if (m.head_dim == 128) {
        if (bm == 16) return launch_attn<128, 16, 2>(stream, a, m.q_per_sample, m.n_heads, m.batch);
        if (bm == 32) return launch_attn<128, 32, 2>(stream, a, m.q_per_sample, m.n_heads, m.batch);
        return launch_attn<128, 64, 2>(stream, a, m.q_per_sample, m.n_heads, m.batch);
    }
    if (m.head_dim == 64) {
        if (bm == 16) return launch_attn<64, 16, 2>(stream, a, m.q_per_sample, m.n_heads, m.batch);
        return launch_attn<64, 32, 2>(stream, a, m.q_per_sample, m.n_heads, m.batch);
    }
    return cudaErrorInvalidValue;
}

// OFT's prefill (llm_engine.cu blurr_llm_forward_rows): causal over the prompt, bidirectional inside the action block,
// per-sequence lengths and block starts read at run time, up to 384 keys resident.  A kernel of its own so that MODE 2's
// instantiations above keep their code.
template <int HD_PAD, int BM>
__global__ void __launch_bounds__(kAttnThreads) attn_block_kernel(const AttnMmaArgs a, const int* seq_len, const int* block_start) {
    extern __shared__ __align__(16) uint8_t smem_attn[];
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    attn_mma_body<HD_PAD, BM, 3, kAttnMaxBlocksWide>(a, smem_attn, blockIdx.x, blockIdx.y, blockIdx.z, seq_len, block_start);
    trace_stamp(a.trace, 2);
}

template <int HD_PAD, int BM>
static cudaError_t launch_attn_block(cudaStream_t stream, const AttnMmaArgs& a, const int* seq_len, const int* block_start, int rows,
                                     int heads, int batch) {
    const size_t smem = attn_smem_bytes<HD_PAD, BM>(a.n_keys);      // 168 KB at head_dim 128, BM 64, 384 keys
    static bool attr = false;
    if (!attr) {
        int dev = 0, optin = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return e;
        if (static_cast<size_t>(optin) < kAttnSmemMax) return cudaErrorInvalidConfiguration;
        e = cudaFuncSetAttribute(attn_block_kernel<HD_PAD, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kAttnSmemMax));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    if (smem > kAttnSmemMax) return cudaErrorInvalidValue;
    dim3 grid((rows + BM - 1) / BM, heads, batch);
    return launch_kernel(attn_block_kernel<HD_PAD, BM>, grid, dim3(kAttnThreads), smem, stream, a, seq_len, block_start);
}

// The same rule past 384 keys: K and V stream through a ring of kAttnStreamStages 64-key buffers instead of staying
// resident, while the bf16 logits of the tile's whole key range stay in shared memory.  The rounding chain, the fp32
// softmax over the whole row (lane striding c = lane + 32 i, the same summation order) and the key-block order of P.V
// are attn_mma_body's, so a row's output equals the resident kernel's for any key count both can hold.  The softmax
// reads the row from shared memory on each pass instead of holding up to 32 logits per lane in registers; expf is
// recomputed on the last pass, which gives the same value.
static constexpr int kAttnStreamStages = 3;
static constexpr int kAttnStreamMaxBlocks = 32;     // 2048 keys (BM 32 at head_dim 128 past 1152 keys, see below)

template <int HD_PAD, int BM>
__device__ __forceinline__ void attn_block_stream_body(const AttnMmaArgs& a, uint8_t* smem_attn, const int qt, const int h,
                                                       const int b, const int* seq_len, const int* block_start) {
    constexpr int S = kAttnStreamStages;
    constexpr int WR = BM / 16;
    constexpr int WC = (kAttnThreads / 32) / WR;
    constexpr int KPW = kBK / WC;
    constexpr int NT_S = KPW / 8;
    constexpr int NT_ALL = HD_PAD / 8;
    constexpr int NT_PV = (NT_ALL + WC - 1) / WC;
    constexpr int NP_PV = (NT_PV + 1) / 2;
    constexpr int CH = HD_PAD / 8;
    constexpr int LDS_MIN = WC * NP_PV * 16 > HD_PAD ? WC * NP_PV * 16 : HD_PAD;
    constexpr int LDS = LDS_MIN + 8;
    const int blk_len = max(1, min(seq_len[b], a.n_keys));            // the host validates both; never read out of range
    const int blk0 = max(1, min(block_start[b], blk_len));
    const int last_q = a.q_row_offset + qt * BM + BM - 1;
    const int n_keys_tile = min(blk_len, last_q >= blk0 ? a.n_keys : last_q + 1);
    const int nkb = (n_keys_tile + kBK - 1) / kBK;
    const int ldl = nkb * kBK + 8;
    bf16* Qs = reinterpret_cast<bf16*>(smem_attn);
    bf16* ring = Qs + BM * LDS;                 // S buffers of [64][LDS]
    bf16* Ls = ring + S * kBK * LDS;            // [BM][ldl]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp % WR, wc = warp / WR;
    const int q_row0 = qt * BM;
    const int n_rows_valid = a.q_per_sample;
    const bf16* qbase = a.q + static_cast<size_t>(b) * a.q_per_sample * a.ldq + a.q_col0 + h * a.head_stride_q;
    const bf16* kbase = a.k + static_cast<size_t>(b) * a.kv_per_sample * a.ldk + a.k_col0 + h * a.head_stride_kv;
    const bf16* vbase = a.v + static_cast<size_t>(b) * a.kv_per_sample * a.ldv + a.v_col0 + h * a.head_stride_kv;

    for (int idx = threadIdx.x; idx < BM * CH; idx += kAttnThreads) {
        const int r = idx / CH, c = idx - r * CH;
        const int row = q_row0 + r;
        const bool valid = (row < n_rows_valid) && (c * 8 < a.hd);
        cp_async_16(Qs + r * LDS + c * 8, valid ? qbase + static_cast<size_t>(row) * a.ldq + c * 8 : qbase, valid);
    }
    // one cp.async group per key block (empty past the last one); block kb lives in buffer kb % S.  S - 1 blocks are in
    // flight ahead of the one being consumed; a buffer is refilled after the barrier that ends every warp's use of it.
    for (int kb = 0; kb < S - 1; ++kb) {
        if (kb < nkb) load_rows_async<LDS, CH>(ring + kb * kBK * LDS, kbase, a.ldk, kb * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
    }

    // ---------------- phase S: logits = chain(Q K^T) -> Ls (bf16) ----------------
    for (int kb = 0; kb < nkb; ++kb) {
        cp_async_wait<S - 2>();
        attn_bar_sync();
        if (kb + S - 1 < nkb)
            load_rows_async<LDS, CH>(ring + ((kb + S - 1) % S) * kBK * LDS, kbase, a.ldk, (kb + S - 1) * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
        const bf16* Kcur = ring + (kb % S) * kBK * LDS;

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
#pragma unroll
        for (int nt = 0; nt < NT_S; ++nt) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = wr * 16 + (lane >> 2) + half * 8;
                const int kcol = kb * kBK + wc * KPW + nt * 8 + (lane & 3) * 2;
                float s0 = bf16_round(acc[nt][half * 2 + 0]);
                float s1 = bf16_round(acc[nt][half * 2 + 1]);
                s0 = bf16_round(s0 * a.scale);
                s1 = bf16_round(s1 * a.scale);
                const int qpos = a.q_row_offset + q_row0 + r;
                const bool in_blk = qpos >= blk0;
                if (!(kcol < blk_len && (kcol <= qpos || (in_blk && kcol >= blk0)))) s0 = -INFINITY;
                if (!(kcol + 1 < blk_len && (kcol + 1 <= qpos || (in_blk && kcol + 1 >= blk0)))) s1 = -INFINITY;
                *reinterpret_cast<uint32_t*>(Ls + r * ldl + kcol) = pack_bf16x2(s0, s1);
            }
        }
    }
    attn_bar_sync();   // every warp is done with the K buffers; all logits are visible

    for (int kb = 0; kb < S - 1; ++kb) {
        if (kb < nkb) load_rows_async<LDS, CH>(ring + kb * kBK * LDS, vbase, a.ldv, kb * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
    }

    // ---------------- softmax: fp32 over bf16 logits, result bf16 in place ----------------
    const int n_it = (n_keys_tile + 31) / 32;
    for (int rr = 0; rr < BM / 8; ++rr) {
        bf16* lrow = Ls + (warp * (BM / 8) + rr) * ldl;
        float m = -INFINITY;
        for (int i = 0; i < n_it; ++i) {
            const int c = lane + i * 32;
            m = fmaxf(m, (c < n_keys_tile) ? bf2f(lrow[c]) : -INFINITY);
        }
        m = warp_max(m);
        float sum = 0.f;
        for (int i = 0; i < n_it; ++i) {
            const int c = lane + i * 32;
            sum += (c < n_keys_tile) ? expf(bf2f(lrow[c]) - m) : 0.f;
        }
        sum = warp_sum(sum);
        for (int i = 0; i < nkb * (kBK / 32); ++i) {
            const int c = lane + i * 32;
            const float x = (c < n_keys_tile) ? expf(bf2f(lrow[c]) - m) : 0.f;
            lrow[c] = f2bf(x / sum);
        }
    }

    // ---------------- phase PV ----------------
    float oacc[NP_PV * 2][4];
#pragma unroll
    for (int i = 0; i < NP_PV * 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) oacc[i][j] = 0.f;
    const int nt0 = wc * NT_PV;
    for (int kb = 0; kb < nkb; ++kb) {
        cp_async_wait<S - 2>();
        attn_bar_sync();                        // (kb == 0: also publishes the probabilities)
        if (kb + S - 1 < nkb)
            load_rows_async<LDS, CH>(ring + ((kb + S - 1) % S) * kBK * LDS, vbase, a.ldv, (kb + S - 1) * kBK, kBK, n_keys_tile, a.hd);
        cp_async_commit();
        const bf16* Vcur = ring + (kb % S) * kBK * LDS;
#pragma unroll
        for (int kk = 0; kk < kBK / 16; ++kk) {
            uint32_t af[4];
            ldmatrix_x4(af, smem_u32(Ls + (wr * 16 + (lane & 15)) * ldl + kb * kBK + kk * 16 + (lane >> 4) * 8));
#pragma unroll
            for (int np = 0; np < NP_PV; ++np) {
                if ((nt0 + np * 2) >= NT_ALL) continue;
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
    cp_async_wait<0>();

    bf16* obase = a.out + static_cast<size_t>(b) * a.q_per_sample * a.ldo + a.o_col0 + h * a.head_stride_q;
#pragma unroll
    for (int nt = 0; nt < NT_PV; ++nt) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = q_row0 + wr * 16 + (lane >> 2) + half * 8;
            const int dim = (nt0 + nt) * 8 + (lane & 3) * 2;
            if (r < n_rows_valid && dim < a.hd)
                *reinterpret_cast<uint32_t*>(obase + static_cast<size_t>(r) * a.ldo + dim) =
                    pack_bf16x2(oacc[nt][half * 2 + 0], oacc[nt][half * 2 + 1]);
        }
    }
}

template <int HD_PAD, int BM>
inline size_t attn_stream_smem_bytes(int n_keys) {
    constexpr int WC = (kAttnThreads / 32) / (BM / 16);
    constexpr int NT_PV = (HD_PAD / 8 + WC - 1) / WC;
    constexpr int NP_PV = (NT_PV + 1) / 2;
    constexpr int LDS_MIN = WC * NP_PV * 16 > HD_PAD ? WC * NP_PV * 16 : HD_PAD;
    constexpr int LDS = LDS_MIN + 8;
    const int nkb = (n_keys + kBK - 1) / kBK;
    return static_cast<size_t>(BM + kAttnStreamStages * kBK) * LDS * 2 + static_cast<size_t>(BM) * (nkb * kBK + 8) * 2;
}

template <int HD_PAD, int BM>
__global__ void __launch_bounds__(kAttnThreads) attn_block_stream_kernel(const AttnMmaArgs a, const int* seq_len, const int* block_start) {
    extern __shared__ __align__(16) uint8_t smem_attn[];
    trace_stamp(a.trace, 0);
    pdl_wait();
    pdl_trigger();
    trace_stamp(a.trace, 1);
    attn_block_stream_body<HD_PAD, BM>(a, smem_attn, blockIdx.x, blockIdx.y, blockIdx.z, seq_len, block_start);
    trace_stamp(a.trace, 2);
}

template <int HD_PAD, int BM>
static cudaError_t launch_attn_block_stream(cudaStream_t stream, const AttnMmaArgs& a, const int* seq_len, const int* block_start,
                                            int rows, int heads, int batch) {
    const size_t smem = attn_stream_smem_bytes<HD_PAD, BM>(a.n_keys);     // 197 KB at head_dim 128, BM 64, 1024 keys
    static bool attr = false;
    if (!attr) {
        int dev = 0, optin = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return e;
        if (static_cast<size_t>(optin) < kAttnSmemMax) return cudaErrorInvalidConfiguration;
        e = cudaFuncSetAttribute(attn_block_stream_kernel<HD_PAD, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kAttnSmemMax));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    if (smem > kAttnSmemMax) return cudaErrorInvalidValue;
    dim3 grid((rows + BM - 1) / BM, heads, batch);
    return launch_kernel(attn_block_stream_kernel<HD_PAD, BM>, grid, dim3(kAttnThreads), smem, stream, a, seq_len, block_start);
}

template <int HD_PAD, int BM>
static cudaError_t launch_block_rule(bool stream_kv, cudaStream_t stream, const AttnMmaArgs& a, const int* seq_len,
                                     const int* block_start, const MhaAttnArgs& m) {
    return stream_kv ? launch_attn_block_stream<HD_PAD, BM>(stream, a, seq_len, block_start, m.q_per_sample, m.n_heads, m.batch)
                     : launch_attn_block<HD_PAD, BM>(stream, a, seq_len, block_start, m.q_per_sample, m.n_heads, m.batch);
}

// The streamed kernel's logits grow with the key count (BM x n_keys bf16), so past 1152 keys at head_dim 128 a 64-row tile
// no longer fits the opt-in limit: the tile is halved until it does (BM 32 holds 2048 keys at either head_dim).  A row's
// output does not depend on BM (its own rounding chain, lane-strided softmax and key-block order of P.V), so this changes
// speed only; up to 1152 keys BM is what attn_tile_rows picks.
static int attn_stream_fit_rows(int hd, int bm, int n_keys) {
    if (hd == 64) return bm > 32 ? 32 : bm;                         // head_dim 64 runs at most BM 32: 2048 keys fit
    if (bm == 64 && attn_stream_smem_bytes<128, 64>(n_keys) > kAttnSmemMax) bm = 32;
    if (bm == 32 && attn_stream_smem_bytes<128, 32>(n_keys) > kAttnSmemMax) bm = 16;
    return bm;
}

// Up to 384 keys every key block of a head stays resident in shared memory (attn_block_kernel); past that, up to 2048,
// K and V stream through a ring (attn_block_stream_kernel).
cudaError_t launch_mha_block_attention(cudaStream_t stream, const MhaAttnArgs& m, const int* block_start) {
    if (m.n_keys > kAttnStreamMaxBlocks * kBK || m.n_kv_heads != m.n_heads || m.q_pos0 != 0 ||
        m.n_keys != m.q_per_sample || m.seq_len == nullptr || block_start == nullptr)
        return cudaErrorInvalidValue;
    AttnMmaArgs a{};
    const int width = m.n_heads * m.head_dim;
    a.q = m.q; a.ldq = width; a.q_col0 = 0; a.q_per_sample = m.q_per_sample;
    a.k = m.k_cache; a.ldk = width; a.k_col0 = 0; a.kv_per_sample = m.n_slots;
    a.v = m.v_cache; a.ldv = width; a.v_col0 = 0;
    a.out = m.out; a.ldo = width; a.o_col0 = 0;
    a.hd = m.head_dim; a.head_stride_q = m.head_dim; a.head_stride_kv = m.head_dim; a.n_keys = m.n_keys;
    a.scale = m.scale; a.mask = nullptr; a.q_row_offset = 0; a.trace = m.trace;
    int bm = attn_tile_rows(m.q_per_sample, m.n_heads, m.batch, 64);
    const int* L = m.seq_len;
    const bool sk = m.n_keys > kAttnMaxBlocksWide * kBK;
    if (sk) bm = attn_stream_fit_rows(m.head_dim, bm, m.n_keys);
    if (m.head_dim == 128) {
        if (bm == 16) return launch_block_rule<128, 16>(sk, stream, a, L, block_start, m);
        if (bm == 32) return launch_block_rule<128, 32>(sk, stream, a, L, block_start, m);
        return launch_block_rule<128, 64>(sk, stream, a, L, block_start, m);
    }
    if (m.head_dim == 64) {
        if (bm == 16) return launch_block_rule<64, 16>(sk, stream, a, L, block_start, m);
        return launch_block_rule<64, 32>(sk, stream, a, L, block_start, m);
    }
    return cudaErrorInvalidValue;
}

}  // namespace blurr
