// OpenVLA-OFT's L1-regression action head behind include/blurr_act_head.h: MLPResNet over the decoder's action rows
// (R = batch * chunk rows of D * H = 28672 columns at OFT's widths).  The Linears run on the tcgen05 GEMM (gemm_tc.cu) on
// tile-packed weights, as the decoder runs its own: split-K fp32 partials at few rows (8 at batch 1: fc1 alone streams
// 235 MB of weights), the bf16 store epilogue beyond.  Around them three kernels of this file: a LayerNorm over the wide
// input rows, a consumer that fuses split-K reduce + bias + ReLU (+ residual) + the next LayerNorm, and the last bias
// with the fp32 output.  The decoder's consumer_kernel stays as it is (no ReLU, rows of at most 8192 columns).
#include "blurr_act_head.h"
#include "blurr_pi0.h"

#include "bodies.cuh"
#include "gemm_tc.h"
#include "kernels.h"
#include "launch.cuh"

#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

namespace blurr {
int record_error(int code, const std::string& msg);      // engine.cu: sets blurr_last_error()
}
using namespace blurr;

static int fail(int code, const std::string& msg) { return record_error(code, msg); }
#define HEAD_CUDA_TRY(expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return fail(BLURR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

namespace {

constexpr int kFewRows = 32;              // at most this many rows: split-K partials (weight streaming), as the decoder
constexpr int kWideThreads = 512;
constexpr int kWideVpt = 16;              // 4-column groups per thread: rows of up to 512 * 16 * 4 = 32768 columns
constexpr int kWideSmemMaxCols = 65536;   // act_wide_layernorm_smem_kernel: the bf16 row in 128 KB of shared memory
constexpr int kActThreads = 512;
constexpr int kActVpt = 2;                // rows of up to 4096 columns

// nn.LayerNorm over one wide row (OFT: D * H = 28672 columns) in fp32, the row resident in registers; bf16 out
__global__ void __launch_bounds__(kWideThreads) act_wide_layernorm_kernel(const bf16* __restrict__ x, int N, const bf16* __restrict__ w,
                                                                          const bf16* __restrict__ bias, float eps, bf16* __restrict__ y) {
    __shared__ float red[kWideThreads / 32];
    pdl_wait();
    pdl_trigger();
    const size_t row = static_cast<size_t>(blockIdx.x) * N;
    const int nvec = N >> 2;
    float4 v[kWideVpt];
    float lsum = 0.f;
#pragma unroll
    for (int i = 0; i < kWideVpt; ++i) {
        const int g = threadIdx.x + i * kWideThreads;
        v[i] = g < nvec ? load_bf16x4(x + row + g * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        lsum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
    const float mean = block_sum<kWideThreads>(lsum, red) / static_cast<float>(N);
    float lvar = 0.f;
#pragma unroll
    for (int i = 0; i < kWideVpt; ++i) {
        if (threadIdx.x + i * kWideThreads >= nvec) continue;
        const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
        lvar += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = rsqrtf(block_sum<kWideThreads>(lvar, red) / static_cast<float>(N) + eps);
#pragma unroll
    for (int i = 0; i < kWideVpt; ++i) {
        const int g = threadIdx.x + i * kWideThreads;
        if (g >= nvec) continue;
        const float4 ww = load_bf16x4(w + g * 4), bb = load_bf16x4(bias + g * 4);
        store_bf16x4(y + row + g * 4, make_float4((v[i].x - mean) * rstd * ww.x + bb.x, (v[i].y - mean) * rstd * ww.y + bb.y,
                                                  (v[i].z - mean) * rstd * ww.z + bb.z, (v[i].w - mean) * rstd * ww.w + bb.w));
    }
}

// The same LayerNorm for rows past the register kernel's 32768 columns (ALOHA: 14 * 4096 = 57344), the bf16 row staged in
// dynamic shared memory (N * 2 bytes) instead of registers.  Thread striding (g = tid + 512 i), the per-thread summation
// order and the block reductions are act_wide_layernorm_kernel's, so a row both kernels could take gets the same result.
__global__ void __launch_bounds__(kWideThreads) act_wide_layernorm_smem_kernel(const bf16* __restrict__ x, int N,
                                                                               const bf16* __restrict__ w,
                                                                               const bf16* __restrict__ bias, float eps,
                                                                               bf16* __restrict__ y) {
    extern __shared__ __align__(16) uint2 xs[];     // [N / 4]: four bf16 per entry
    __shared__ float red[kWideThreads / 32];
    pdl_wait();
    pdl_trigger();
    const size_t row = static_cast<size_t>(blockIdx.x) * N;
    const int nvec = N >> 2;
    float lsum = 0.f;
    for (int g = threadIdx.x; g < nvec; g += kWideThreads) {
        const uint2 u = __ldcg(reinterpret_cast<const uint2*>(x + row + g * 4));
        xs[g] = u;
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
        lsum += (a.x + a.y) + (b.x + b.y);
    }
    const float mean = block_sum<kWideThreads>(lsum, red) / static_cast<float>(N);
    float lvar = 0.f;
    for (int g = threadIdx.x; g < nvec; g += kWideThreads) {        // each thread reads back only what it wrote
        const uint2 u = xs[g];
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
        const float dx = a.x - mean, dy = a.y - mean, dz = b.x - mean, dw = b.y - mean;
        lvar += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = rsqrtf(block_sum<kWideThreads>(lvar, red) / static_cast<float>(N) + eps);
    for (int g = threadIdx.x; g < nvec; g += kWideThreads) {
        const uint2 u = xs[g];
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
        const float4 ww = load_bf16x4(w + g * 4), bb = load_bf16x4(bias + g * 4);
        store_bf16x4(y + row + g * 4, make_float4((a.x - mean) * rstd * ww.x + bb.x, (a.y - mean) * rstd * ww.y + bb.y,
                                                  (b.x - mean) * rstd * ww.z + bb.z, (b.y - mean) * rstd * ww.w + bb.w));
    }
}

struct ActConsumerArgs {
    const float* partial; int splitk, T, N, ldp;     // split-K partials [splitk][T][ldp] ...
    const bf16* lin; int ldl;                        // ... or the bf16 Linear output (bias included)
    const bf16* bias;                                // [N] (partials only)
    const bf16* res;                                 // [T][N] residual or nullptr
    bf16* x_out;                                     // [T][N]: bf16(res + relu(linear)) (may alias res)
    const bf16* ln_w; const bf16* ln_b; float eps;
    bf16* xn_out;                                    // [T][N]: LayerNorm(x_out)
};

// One CTA per row: x = [res +] ReLU(bf16(sum of slices + bias)), every op rounded to bf16 as torch does it; then the next
// LayerNorm in fp32 from the row held in registers
__global__ void __launch_bounds__(kActThreads, 1) act_consumer_kernel(const ActConsumerArgs a) {
    __shared__ float red[kActThreads / 32];
    pdl_wait();
    pdl_trigger();
    const int t = blockIdx.x, nvec = a.N >> 2;
    float4 x[kActVpt];
    float lsum = 0.f;
#pragma unroll
    for (int i = 0; i < kActVpt; ++i) {
        const int g = threadIdx.x + i * kActThreads;
        x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g >= nvec) continue;
        const int n = g << 2;
        float4 v;
        if (a.partial != nullptr) {
            float4 acc = sum_slices(a.partial + static_cast<size_t>(t) * a.ldp + n, static_cast<size_t>(a.T) * a.ldp, a.splitk);
            const float4 b = load_bf16x4(a.bias + n);
            v = make_float4(bf16_round(acc.x + b.x), bf16_round(acc.y + b.y), bf16_round(acc.z + b.z), bf16_round(acc.w + b.w));
        } else {
            v = load_bf16x4(a.lin + static_cast<size_t>(t) * a.ldl + n);
        }
        // ReLU (NaN stays NaN, as torch.relu)
        v = make_float4(v.x < 0.f ? 0.f : v.x, v.y < 0.f ? 0.f : v.y, v.z < 0.f ? 0.f : v.z, v.w < 0.f ? 0.f : v.w);
        if (a.res != nullptr) {
            const float4 r = load_bf16x4(a.res + static_cast<size_t>(t) * a.N + n);
            v = make_float4(bf16_round(v.x + r.x), bf16_round(v.y + r.y), bf16_round(v.z + r.z), bf16_round(v.w + r.w));
        }
        store_bf16x4(a.x_out + static_cast<size_t>(t) * a.N + n, v);
        x[i] = v;
        lsum += (v.x + v.y) + (v.z + v.w);
    }
    const float mean = block_sum<kActThreads>(lsum, red) / static_cast<float>(a.N);
    float lvar = 0.f;
#pragma unroll
    for (int i = 0; i < kActVpt; ++i) {
        if (threadIdx.x + i * kActThreads >= nvec) continue;
        const float dx = x[i].x - mean, dy = x[i].y - mean, dz = x[i].z - mean, dw = x[i].w - mean;
        lvar += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = rsqrtf(block_sum<kActThreads>(lvar, red) / static_cast<float>(a.N) + a.eps);
#pragma unroll
    for (int i = 0; i < kActVpt; ++i) {
        const int g = threadIdx.x + i * kActThreads;
        if (g >= nvec) continue;
        const int n = g << 2;
        const float4 w = load_bf16x4(a.ln_w + n), b = load_bf16x4(a.ln_b + n);
        store_bf16x4(a.xn_out + static_cast<size_t>(t) * a.N + n,
                     make_float4((x[i].x - mean) * rstd * w.x + b.x, (x[i].y - mean) * rstd * w.y + b.y,
                                 (x[i].z - mean) * rstd * w.z + b.z, (x[i].w - mean) * rstd * w.w + b.w));
    }
}

// out[t][d] = fp32(bf16(fc2 output)) for d < D: the slices summed in order + bias, or the store epilogue's bf16
__global__ void __launch_bounds__(256) act_out_kernel(const float* partial, int splitk, int T, int ldp, const bf16* lin,
                                                      const bf16* bias, int D, float* out) {
    pdl_wait();
    pdl_trigger();
    const int idx = blockIdx.x * 256 + threadIdx.x;
    if (idx >= T * D) return;
    const int t = idx / D, d = idx - t * D;
    float v;
    if (partial != nullptr) {
        float acc = 0.f;
        for (int z = 0; z < splitk; ++z) acc += __ldcg(partial + (static_cast<size_t>(z) * T + t) * ldp + d);
        v = bf16_round(acc + bf2f(bias[d]));
    } else {
        v = bf2f(ldcg_bf16(lin + static_cast<size_t>(t) * ldp + d));
    }
    out[idx] = v;
}

struct HeadLin { bf16* w = nullptr; bf16* bias = nullptr; int N = 0, Nw = 0, K = 0; };

}  // namespace

struct blurr_act_head {
    blurr_act_head_config cfg{};
    int device = 0, max_batch = 1, max_rows = 0;
    std::vector<void*> allocs;
    bf16 *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
    std::vector<bf16*> blk_ln_w, blk_ln_b;
    HeadLin fc1, fc2;
    std::vector<HeadLin> blk;
    bf16 *IN = nullptr, *XN1 = nullptr, *X = nullptr, *XN = nullptr, *LIN = nullptr;
    float *OUT = nullptr, *ws = nullptr;
    size_t ws_floats = 0;
    std::set<std::string> seen;
    size_t expected_keys = 0;
    bool finalized = false;
    int64_t launches = 0;
    struct GraphEntry { cudaGraph_t graph; cudaGraphExec_t exec; int64_t launches; };
    std::map<int, GraphEntry> graphs;            // by batch
};

static void* dalloc(blurr_act_head* h, size_t bytes) {
    void* p = nullptr;
    if (bytes == 0) bytes = 16;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, bytes);
    h->allocs.push_back(p);
    return p;
}

static void drop_graphs(blurr_act_head* h) {
    for (auto& kv : h->graphs) { cudaGraphExecDestroy(kv.second.exec); cudaGraphDestroy(kv.second.graph); }
    h->graphs.clear();
}

extern "C" void blurr_act_head_destroy(blurr_act_head_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    drop_graphs(h);
    for (void* p : h->allocs) cudaFree(p);
    gemm_forget_tensor_maps();
    delete h;
}

extern "C" int blurr_act_head_create(const blurr_act_head_config* cfg, int device, int max_batch, blurr_act_head_t** out) {
    if (!cfg || !out || max_batch < 1) return fail(BLURR_ERR_INVALID, "blurr_act_head_create: bad arguments");
    const blurr_act_head_config& c = *cfg;
    if (c.abi_version != BLURR_ACT_HEAD_ABI_VERSION) return fail(BLURR_ERR_INVALID, "blurr_act_head_config abi_version mismatch");
    if (c.input_dim < 1 || c.action_dim < 1 || c.chunk < 1 || c.num_blocks < 0 || !(c.ln_eps > 0.0f))
        return fail(BLURR_ERR_INVALID, "blurr_act_head_create: input_dim, action_dim, chunk >= 1, num_blocks >= 0, ln_eps > 0");
    const int64_t wide = static_cast<int64_t>(c.action_dim) * c.input_dim;
    if (wide % 64 || wide > kWideSmemMaxCols)
        return fail(BLURR_ERR_INVALID, "action_dim * input_dim must be a multiple of 64 and at most 65536 (one LayerNorm row in "
                                       "shared memory)");
    if (c.hidden_dim < 128 || c.hidden_dim % 128 || c.hidden_dim > 4 * kActThreads * kActVpt)
        return fail(BLURR_ERR_INVALID, "hidden_dim must be a multiple of 128 and at most 4096");
    if (static_cast<int64_t>(max_batch) * c.chunk > 4096) return fail(BLURR_ERR_INVALID, "max_batch * chunk must be at most 4096 rows");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BLURR_ERR_CUDA, "no CUDA device: the B200 path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BLURR_ERR_INVALID, "bad device index");
    cudaDeviceProp prop{};
    HEAD_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(BLURR_ERR_CUDA, "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + ": this library is built for sm_100a only");
    HEAD_CUDA_TRY(cudaSetDevice(device));
    if (wide > 4 * kWideThreads * kWideVpt)
        HEAD_CUDA_TRY(cudaFuncSetAttribute(act_wide_layernorm_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           kWideSmemMaxCols * 2));
    auto* h = new blurr_act_head();
    h->cfg = c; h->device = device; h->max_batch = max_batch; h->max_rows = max_batch * c.chunk;
    const size_t R = h->max_rows, W = static_cast<size_t>(wide), H = c.hidden_dim;
    auto bufb = [&](size_t elems) { return static_cast<bf16*>(dalloc(h, elems * 2)); };
    auto lin = [&](HeadLin& L, int N, int K) {
        L.N = N; L.Nw = (N + 127) / 128 * 128; L.K = K;
        L.w = bufb(static_cast<size_t>(L.Nw) * K); L.bias = bufb(L.Nw);        // rows / bias past N stay zero
        return L.w != nullptr && L.bias != nullptr;
    };
    bool ok = lin(h->fc1, c.hidden_dim, static_cast<int>(wide)) && lin(h->fc2, c.action_dim, c.hidden_dim);
    h->blk.resize(c.num_blocks);
    for (auto& L : h->blk) ok &= lin(L, c.hidden_dim, c.hidden_dim);
    h->ln1_w = bufb(W); h->ln1_b = bufb(W); h->ln2_w = bufb(H); h->ln2_b = bufb(H);
    ok &= h->ln1_w && h->ln1_b && h->ln2_w && h->ln2_b;
    for (int i = 0; i < c.num_blocks; ++i) {
        h->blk_ln_w.push_back(bufb(H)); h->blk_ln_b.push_back(bufb(H));
        ok &= h->blk_ln_w.back() && h->blk_ln_b.back();
    }
    h->IN = bufb(R * W); h->XN1 = bufb(R * W); h->X = bufb(R * H); h->XN = bufb(R * H); h->LIN = bufb(R * H);
    h->OUT = static_cast<float*>(dalloc(h, R * c.action_dim * 4));
    h->ws_floats = 16 * static_cast<size_t>(kFewRows) * H;
    h->ws = static_cast<float*>(dalloc(h, h->ws_floats * 4));
    ok &= h->IN && h->XN1 && h->X && h->XN && h->LIN && h->OUT && h->ws;
    if (!ok) { blurr_act_head_destroy(h); return fail(BLURR_ERR_CUDA, "blurr_act_head_create: device allocation failed"); }
    h->expected_keys = 8 + 4 * static_cast<size_t>(c.num_blocks);
    *out = h;
    return 0;
}

extern "C" int blurr_act_head_set_weight(blurr_act_head_t* h, const char* key_c, const void* dev_ptr, const int64_t* shape, int ndim) {
    if (!h || !key_c || !dev_ptr || !shape) return fail(BLURR_ERR_INVALID, "blurr_act_head_set_weight: null argument");
    HEAD_CUDA_TRY(cudaSetDevice(h->device));
    const auto& c = h->cfg;
    const std::string key(key_c);
    const bf16* src = static_cast<const bf16*>(dev_ptr);
    const int wide = c.action_dim * c.input_dim;
    auto bad = [&]() { return fail(BLURR_ERR_INVALID, "unexpected shape for " + key); };
    auto vec = [&](bf16* dst, int n) -> int {
        if (ndim != 1 || shape[0] != n) return bad();
        HEAD_CUDA_TRY(cudaMemcpy(dst, src, static_cast<size_t>(n) * 2, cudaMemcpyDeviceToDevice));
        return 0;
    };
    auto linear = [&](HeadLin& L, const std::string& what) -> int {
        if (what == "weight") {
            if (ndim != 2 || shape[0] != L.N || shape[1] != L.K) return bad();
            const cudaError_t e = launch_pack_rows(nullptr, src, L.N, L.K, L.w, 1, 0, L.K / 64);
            return e == cudaSuccess ? 0 : fail(BLURR_ERR_CUDA, std::string("weight repack: ") + cudaGetErrorString(e));
        }
        if (what == "bias") return vec(L.bias, L.N);
        return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    };
    auto norm = [&](bf16* w, bf16* b, int n, const std::string& what) -> int {
        if (what == "weight") return vec(w, n);
        if (what == "bias") return vec(b, n);
        return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    };
    const size_t dot = key.rfind('.');
    if (key.rfind("model.", 0) != 0 || dot == std::string::npos || dot < 6) return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    const std::string mod = key.substr(6, dot - 6), what = key.substr(dot + 1);
    int rc = 0;
    if (mod == "layer_norm1") rc = norm(h->ln1_w, h->ln1_b, wide, what);
    else if (mod == "fc1") rc = linear(h->fc1, what);
    else if (mod == "layer_norm2") rc = norm(h->ln2_w, h->ln2_b, c.hidden_dim, what);
    else if (mod == "fc2") rc = linear(h->fc2, what);
    else if (mod.rfind("mlp_resnet_blocks.", 0) == 0) {
        const std::string rest = mod.substr(18);
        const size_t d2 = rest.find('.');
        if (d2 == std::string::npos || d2 == 0 || rest.find_first_not_of("0123456789") != d2)
            return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
        const int i = atoi(rest.substr(0, d2).c_str());
        if (i < 0 || i >= c.num_blocks) return fail(BLURR_ERR_INVALID, "block index out of range in " + key);
        const std::string sub = rest.substr(d2 + 1);
        if (sub == "ffn.0") rc = norm(h->blk_ln_w[i], h->blk_ln_b[i], c.hidden_dim, what);
        else if (sub == "ffn.1") rc = linear(h->blk[i], what);
        else return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    } else {
        return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    }
    if (rc) return rc;
    h->seen.insert(key);
    h->finalized = false;
    return 0;
}

extern "C" int blurr_act_head_finalize(blurr_act_head_t* h) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_act_head_finalize: null handle");
    if (h->seen.size() != h->expected_keys)
        return fail(BLURR_ERR_STATE, "blurr_act_head_finalize: " + std::to_string(h->expected_keys - h->seen.size()) + " state_dict keys missing");
    HEAD_CUDA_TRY(cudaSetDevice(h->device));
    HEAD_CUDA_TRY(cudaDeviceSynchronize());
    drop_graphs(h);
    h->finalized = true;
    return 0;
}

namespace {

struct HeadRun {
    blurr_act_head* h;
    cudaStream_t st;
    int rc = 0;

    void launched(cudaError_t e, const char* what) {
        ++h->launches;
        if (e != cudaSuccess && !rc) rc = fail(BLURR_ERR_CUDA, std::string(what) + " launch failed: " + cudaGetErrorString(e));
    }
    // Y = X W^T over R rows: few rows -> fp32 split-K partials in ws (returns the slice count), else bf16(acc + bias) in LIN
    int gemm(const HeadLin& L, const bf16* X, int R) {
        if (rc) return 0;
        const bool few = R <= kFewRows;
        GemmCall c{};
        c.W = L.w; c.Nw = L.Nw; c.K = L.K; c.ldw = L.K; c.w_packed = 1;
        c.X = X; c.T = R; c.ldx = L.K;
        c.splitk = 1; c.glu_act = 1; c.w_static = 1;
        if (few) {
            c.epi = EPI_PARTIAL;
            c.splitk = pick_splitk_waves(L.Nw / 128, (L.K + 63) / 64);
            c.partial = h->ws;
        } else {
            c.epi = EPI_STORE;
            c.bias = L.bias; c.out = h->LIN; c.ldo = L.Nw;
        }
        std::string err;
        const int s = gemm_launch(st, c, &err);
        ++h->launches;
        if (s < 0) { rc = fail(BLURR_ERR_CUDA, err); return 0; }
        return few ? s : 0;
    }
    void consumer(const HeadLin& L, int splitk, int R, const bf16* res, const bf16* ln_w, const bf16* ln_b) {
        if (rc) return;
        ActConsumerArgs a{};
        a.T = R; a.N = L.N; a.ldp = L.Nw;
        if (splitk > 0) { a.partial = h->ws; a.splitk = splitk; a.bias = L.bias; }
        else { a.lin = h->LIN; a.ldl = L.Nw; }
        a.res = res; a.x_out = h->X; a.ln_w = ln_w; a.ln_b = ln_b; a.eps = h->cfg.ln_eps; a.xn_out = h->XN;
        launched(launch_kernel(act_consumer_kernel, dim3(R), dim3(kActThreads), 0, st, a), "act_consumer");
    }
};

void run_head(HeadRun& R, int rows) {
    blurr_act_head* h = R.h;
    const auto& c = h->cfg;
    const int wide = c.action_dim * c.input_dim, nb = c.num_blocks;
    // by width only: rows up to 32768 columns keep the register kernel
    const bool in_regs = wide <= 4 * kWideThreads * kWideVpt;
    R.launched(launch_kernel(in_regs ? act_wide_layernorm_kernel : act_wide_layernorm_smem_kernel, dim3(rows), dim3(kWideThreads),
                             in_regs ? 0 : static_cast<size_t>(wide) * 2, R.st, static_cast<const bf16*>(h->IN), wide,
                             static_cast<const bf16*>(h->ln1_w), static_cast<const bf16*>(h->ln1_b), c.ln_eps, h->XN1),
               "act_wide_layernorm");
    int s = R.gemm(h->fc1, h->XN1, rows);
    R.consumer(h->fc1, s, rows, nullptr, nb > 0 ? h->blk_ln_w[0] : h->ln2_w, nb > 0 ? h->blk_ln_b[0] : h->ln2_b);
    for (int i = 0; i < nb; ++i) {
        s = R.gemm(h->blk[i], h->XN, rows);
        R.consumer(h->blk[i], s, rows, h->X, i + 1 < nb ? h->blk_ln_w[i + 1] : h->ln2_w, i + 1 < nb ? h->blk_ln_b[i + 1] : h->ln2_b);
    }
    s = R.gemm(h->fc2, h->XN, rows);
    if (R.rc) return;
    const int total = rows * c.action_dim;
    R.launched(launch_kernel(act_out_kernel, dim3((total + 255) / 256), dim3(256), 0, R.st, static_cast<const float*>(s > 0 ? h->ws : nullptr),
                             s, rows, h->fc2.Nw, static_cast<const bf16*>(h->LIN), static_cast<const bf16*>(h->fc2.bias), c.action_dim,
                             h->OUT),
               "act_out");
}

}  // namespace

extern "C" int blurr_act_head_forward(blurr_act_head_t* h, void* cuda_stream, int batch, const void* hidden_rows, float* out) {
    const char* fn = "blurr_act_head_forward";
    if (!h || !hidden_rows || !out) return fail(BLURR_ERR_INVALID, std::string(fn) + ": null argument");
    if (!h->finalized) return fail(BLURR_ERR_STATE, std::string(fn) + ": call blurr_act_head_finalize first");
    if (batch < 1 || batch > h->max_batch) return fail(BLURR_ERR_INVALID, std::string(fn) + ": batch out of range");
    const auto& c = h->cfg;
    const int rows = batch * c.chunk;
    HEAD_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    HEAD_CUDA_TRY(cudaMemcpyAsync(h->IN, hidden_rows, static_cast<size_t>(rows) * c.action_dim * c.input_dim * 2, cudaMemcpyDeviceToDevice, st));
    h->launches = 0;
    auto it = h->graphs.find(batch);
    if (it == h->graphs.end()) {
        HeadRun R{h, st};
        run_head(R, rows);                              // warm run: attribute setup, tensor maps
        if (R.rc) return R.rc;
        HEAD_CUDA_TRY(cudaStreamSynchronize(st));
        h->launches = 0;
        cudaStream_t cs;
        HEAD_CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        HeadRun C{h, cs};
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) { cudaStreamDestroy(cs); return fail(BLURR_ERR_CUDA, "graph capture begin failed"); }
        run_head(C, rows);
        cudaGraph_t g = nullptr;
        e = cudaStreamEndCapture(cs, &g);
        cudaStreamDestroy(cs);
        if (C.rc) { if (g) cudaGraphDestroy(g); return C.rc; }
        if (e != cudaSuccess || !g) return fail(BLURR_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(e));
        cudaGraphExec_t ex = nullptr;
        e = cudaGraphInstantiate(&ex, g, 0);
        if (e != cudaSuccess) { cudaGraphDestroy(g); return fail(BLURR_ERR_CUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(e)); }
        it = h->graphs.emplace(batch, blurr_act_head::GraphEntry{g, ex, h->launches}).first;
    }
    HEAD_CUDA_TRY(cudaGraphLaunch(it->second.exec, st));
    h->launches = it->second.launches;
    HEAD_CUDA_TRY(cudaMemcpyAsync(out, h->OUT, static_cast<size_t>(rows) * c.action_dim * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int blurr_act_head_check(blurr_act_head_t* h, void* cuda_stream) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_act_head_check: null handle");
    HEAD_CUDA_TRY(cudaSetDevice(h->device));
    HEAD_CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(cuda_stream)));
    if (gemm_take_timeout_flag() > 0) return fail(BLURR_ERR_CUDA, "a bounded pipeline wait expired inside a GEMM kernel");
    return 0;
}

extern "C" int64_t blurr_act_head_last_launch_count(const blurr_act_head_t* h) { return h ? h->launches : 0; }
