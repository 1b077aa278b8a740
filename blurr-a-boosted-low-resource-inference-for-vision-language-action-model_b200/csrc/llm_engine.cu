// Llama-shaped decoder engine behind include/blurr_llm.h: the language-model half of the OpenVLA-7B-shaped path
// (SURVEY.md 8(f) row 3).  Prefill of the prompt embeddings + greedy decode with a KV cache, arithmetic as in
// transformers' LlamaForCausalLM (eager attention).  It is a second client of the kernels the Pi-0 engine uses: the
// tcgen05 GEMM family (gemm_tc.cu; SwiGLU = the GLU epilogue with a SiLU gate), the split-K consumers (RMSNorm in its
// Llama form), the mma.sync attention body at head_dim 128 with a positional causal mask, plus the small kernels of
// llm_kernels.cu.  One decode step streams every weight once (13.5 GB for Llama-2-7B): a pure HBM weight-streaming
// workload, which is what the few-token persistent GEMM was built for.
#include "blurr_llm.h"
#include "blurr_pi0.h"

#include "common.cuh"
#include "gemm_tc.h"
#include "kernels.h"
#include "launch.cuh"

#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <tuple>
#include <vector>

namespace blurr {
int record_error(int code, const std::string& msg);      // engine.cu: sets blurr_last_error()
const int* gemm_timeout_flag_ptr();
const int* attn_timeout_flag_ptr();
int gemm_take_timeout_flag();
int attn_take_timeout_flag();
}
using namespace blurr;

// the device array the sampler reads is the host ABI struct, byte for byte
static_assert(sizeof(blurr_llm_sampling) == sizeof(SampleParams) && offsetof(blurr_llm_sampling, seed) == offsetof(SampleParams, seed) &&
                  offsetof(blurr_llm_sampling, temperature) == offsetof(SampleParams, temperature) &&
                  offsetof(blurr_llm_sampling, top_k) == offsetof(SampleParams, top_k) &&
                  offsetof(blurr_llm_sampling, top_p) == offsetof(SampleParams, top_p),
              "blurr_llm_sampling and SampleParams must share one layout");

static int fail(int code, const std::string& msg) { return record_error(code, msg); }
#define LLM_CUDA_TRY(expr)                                                                       \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return fail(BLURR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

namespace {

constexpr int kSMs = 148;
constexpr int kTraceMax = 4096;
constexpr int kMaxKeptLogits = 16;    // generated tokens whose logits blurr_llm_generate can return
constexpr int kMidTokens = 288;       // up to here o / down run as chunked split-K (plan_mid_tokens)
constexpr int kFewTokens = 32;        // at most this many token rows: split-K partials + consumers (weight streaming)
constexpr int kGenerateMaxPositions = 320;     // generate's decode kernels hold a sequence's logits in sc[320]
constexpr int kForwardMaxPositions = 384;      // long_forward 0: attn_block_kernel keeps every key block resident (6 x 64)
constexpr int kLongForwardMaxPositions = 1024; // long_forward 1: attn_block_stream_kernel streams K/V (16 x 64 keys)
constexpr int kLongerForwardMaxPositions = 2048;   // long_forward 2 (1025..2048): the same kernel, 32 x 64 keys (BM <= 32 past 1152)

struct Lin { bf16* w = nullptr; int Nw = 0, K = 0; };
struct Layer { Lin qkv, o, gu, down; bf16 *in_ln = nullptr, *post_ln = nullptr; };

// dst (tile-packed [Nw/128][K/64][128][64], gemm_tc.h) <- src rows [rows][cols]; destination row = r * row_mul + row_off
__global__ void llm_pack_rows_kernel(const bf16* __restrict__ src, int rows, int cols, bf16* __restrict__ dst, int row_mul,
                                     int row_off, int kb_total) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<size_t>(rows) * cols) return;
    const int r = static_cast<int>(idx / cols), c = static_cast<int>(idx - static_cast<size_t>(r) * cols);
    const int dr = r * row_mul + row_off;
    dst[((static_cast<size_t>(dr / 128) * kb_total + c / 64) * 128 + dr % 128) * 64 + c % 64] = src[idx];
}

}  // namespace

namespace blurr {
cudaError_t launch_pack_rows(cudaStream_t stream, const bf16* src, int rows, int cols, bf16* dst, int row_mul, int row_off, int kb_total) {
    const size_t total = static_cast<size_t>(rows) * cols;
    llm_pack_rows_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(src, rows, cols, dst, row_mul, row_off, kb_total);
    return cudaGetLastError();
}
}  // namespace blurr

struct blurr_llm {
    blurr_llm_config cfg{};
    int device = 0, max_batch = 1;
    std::vector<void*> allocs;
    bf16* embed = nullptr;
    std::vector<Layer> layers;
    bf16* final_norm = nullptr;
    Lin lm_head;
    float *cos_t = nullptr, *sin_t = nullptr;
    int n_pos = 0;
    bf16 *IN = nullptr, *X = nullptr, *XN = nullptr, *Q = nullptr, *AO = nullptr, *HM = nullptr, *LIN = nullptr;
    bf16 *LAST = nullptr, *LOGITS = nullptr, *LOGITS_ALL = nullptr;
    float* ws = nullptr;
    size_t ws_floats = 0;
    bf16 *kcache = nullptr, *vcache = nullptr;
    int64_t *ids = nullptr, *out_ids = nullptr;
    int* d_err = nullptr;
    // per-row inputs the captured kernels read at replay, so one graph serves every vector of them: the prompt lengths of
    // a ragged call or sequence lengths of forward_rows (d_lens), forward_rows' block and row starts (d_blk, d_row0: the
    // same allocation) and the sampling parameters of a sampled call (d_sampling).  h_stage is their pinned staging copy
    // ([max_batch] parameters, then [max_batch] each of lengths, block starts, row starts), reused once `staged` says the
    // last upload has left it.
    int *d_lens = nullptr, *d_blk = nullptr, *d_row0 = nullptr;
    SampleParams* d_sampling = nullptr;
    unsigned char* h_stage = nullptr;
    cudaEvent_t staged = nullptr;
    std::set<std::string> seen;
    size_t expected_keys = 0;
    bool finalized = false, use_graph = true;
    int64_t launches = 0, weight_bytes = 0;
    struct GraphEntry { cudaGraph_t graph; cudaGraphExec_t exec; int64_t launches; };
    // (batch, prompt_len, n_new, logits, ragged, sampled, forward_rows); forward_rows: (batch, max_len, 0, 0, 0, 0, 1)
    std::map<std::tuple<int, int, int, int, int, int, int>, GraphEntry> graphs;
    // in-graph timeline (option "trace"): every kernel stamps %globaltimer at entry / after its dependency wait / at exit
    bool trace = false;
    unsigned long long* trace_buf = nullptr;
    std::vector<std::string> trace_labels;
};

static void* dalloc(blurr_llm* h, size_t bytes) {
    void* p = nullptr;
    if (bytes == 0) bytes = 16;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, bytes);
    h->allocs.push_back(p);
    return p;
}

static void drop_graphs(blurr_llm* h) {
    for (auto& kv : h->graphs) { cudaGraphExecDestroy(kv.second.exec); cudaGraphDestroy(kv.second.graph); }
    h->graphs.clear();
}

extern "C" void blurr_llm_destroy(blurr_llm_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    drop_graphs(h);
    for (void* p : h->allocs) cudaFree(p);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->staged) cudaEventDestroy(h->staged);
    gemm_forget_tensor_maps();
    delete h;
}

extern "C" int blurr_llm_create(const blurr_llm_config* cfg, int device, int max_batch, blurr_llm_t** out) {
    if (!cfg || !out || max_batch < 1) return fail(BLURR_ERR_INVALID, "blurr_llm_create: bad arguments");
    const blurr_llm_config& c = *cfg;
    if (c.abi_version != BLURR_LLM_ABI_VERSION) return fail(BLURR_ERR_INVALID, "blurr_llm_config abi_version mismatch");
    if (c.num_layers < 1 || c.hidden % 128 || c.intermediate % 64 || c.hidden < 128 || c.vocab < 1)
        return fail(BLURR_ERR_INVALID, "hidden must be a multiple of 128, intermediate of 64");
    if (c.num_kv_heads != c.num_heads || (c.head_dim != 128 && c.head_dim != 64))
        return fail(BLURR_ERR_INVALID, "the attention kernel is built for multi-head attention with head_dim 128 or 64");
    if ((c.num_heads * c.head_dim) % 128 || c.hidden > 4096 * 2)
        return fail(BLURR_ERR_INVALID, "num_heads * head_dim must be a multiple of 128; hidden <= 8192");
    if (c.hidden > 4096) return fail(BLURR_ERR_INVALID, "the RMSNorm consumer covers rows of up to 4096 columns");
    if (c.long_forward < 0 || c.long_forward > 2) return fail(BLURR_ERR_INVALID, "long_forward must be 0, 1 or 2");
    if (c.long_forward == 2) {
        if (c.max_positions <= kLongForwardMaxPositions || c.max_positions > kLongerForwardMaxPositions)
            return fail(BLURR_ERR_INVALID, "max_positions must be in 1025..2048 with long_forward = 2 (up to 1024: long_forward = 1)");
    } else if (c.max_positions < 2 || c.max_positions > (c.long_forward ? kLongForwardMaxPositions : kForwardMaxPositions)) {
        return fail(BLURR_ERR_INVALID, c.long_forward ? "max_positions must be in 2..1024 with long_forward"
                                                      : "max_positions must be in 2..384 (1024 with long_forward = 1)");
    }
    if (max_batch > kFewTokens) return fail(BLURR_ERR_INVALID, "max_batch <= 32 (one decode step is a few-token GEMM)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BLURR_ERR_CUDA, "no CUDA device: the B200 path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BLURR_ERR_INVALID, "bad device index");
    cudaDeviceProp prop{};
    LLM_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(BLURR_ERR_CUDA, "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + ": this library is built for sm_100a only");
    LLM_CUDA_TRY(cudaSetDevice(device));
    auto* h = new blurr_llm();
    h->cfg = c; h->device = device; h->max_batch = max_batch;
    const int QW = c.num_heads * c.head_dim, KVW = c.num_kv_heads * c.head_dim;
    const size_t Tmax = static_cast<size_t>(max_batch) * c.max_positions;
    auto bufb = [&](size_t elems) { return static_cast<bf16*>(dalloc(h, elems * 2)); };
    auto lin = [&](Lin& L, int Nw, int K) { L.Nw = (Nw + 127) / 128 * 128; L.K = K; L.w = bufb(static_cast<size_t>(L.Nw) * K); return L.w != nullptr; };
    bool ok = true;
    h->embed = bufb(static_cast<size_t>(c.vocab) * c.hidden);
    h->layers.resize(c.num_layers);
    for (auto& L : h->layers) {
        ok &= lin(L.qkv, QW + 2 * KVW, c.hidden) && lin(L.o, c.hidden, QW) && lin(L.gu, 2 * c.intermediate, c.hidden) &&
              lin(L.down, c.hidden, c.intermediate);
        L.in_ln = bufb(c.hidden); L.post_ln = bufb(c.hidden);
        ok &= L.in_ln && L.post_ln;
        h->weight_bytes += 2ll * (static_cast<int64_t>(L.qkv.Nw) * L.qkv.K + static_cast<int64_t>(L.o.Nw) * L.o.K +
                                  static_cast<int64_t>(L.gu.Nw) * L.gu.K + static_cast<int64_t>(L.down.Nw) * L.down.K);
    }
    h->final_norm = bufb(c.hidden);
    ok &= lin(h->lm_head, c.vocab, c.hidden);
    h->weight_bytes += 2ll * h->lm_head.Nw * h->lm_head.K;
    h->IN = bufb(Tmax * c.hidden); h->X = bufb(Tmax * c.hidden); h->XN = bufb(Tmax * c.hidden);
    h->Q = bufb(Tmax * QW); h->AO = bufb(Tmax * QW); h->HM = bufb(Tmax * c.intermediate);
    size_t widest = static_cast<size_t>(QW + 2 * KVW);
    if (widest < static_cast<size_t>(c.hidden)) widest = c.hidden;
    h->LIN = bufb(Tmax * widest);
    h->LAST = bufb(static_cast<size_t>(max_batch) * c.hidden);
    h->LOGITS = bufb(static_cast<size_t>(max_batch) * h->lm_head.Nw);
    h->LOGITS_ALL = bufb(static_cast<size_t>(max_batch) * kMaxKeptLogits * c.vocab);
    size_t widest_nw = h->lm_head.Nw;
    if (widest_nw < static_cast<size_t>(2 * c.intermediate)) widest_nw = 2 * c.intermediate;
    h->ws_floats = 16 * static_cast<size_t>(kFewTokens) * widest_nw;
    if (h->ws_floats < 4 * static_cast<size_t>(kMidTokens) * c.hidden) h->ws_floats = 4 * static_cast<size_t>(kMidTokens) * c.hidden;
    h->ws = static_cast<float*>(dalloc(h, h->ws_floats * 4));
    const size_t cache = static_cast<size_t>(c.num_layers) * max_batch * c.max_positions * KVW;
    h->kcache = bufb(cache); h->vcache = bufb(cache);
    h->ids = static_cast<int64_t*>(dalloc(h, static_cast<size_t>(max_batch) * 8));
    h->out_ids = static_cast<int64_t*>(dalloc(h, static_cast<size_t>(max_batch) * c.max_positions * 8));
    h->d_err = static_cast<int*>(dalloc(h, 16));
    h->d_lens = static_cast<int*>(dalloc(h, static_cast<size_t>(max_batch) * 3 * 4));
    if (h->d_lens) { h->d_blk = h->d_lens + max_batch; h->d_row0 = h->d_lens + 2 * max_batch; }
    h->d_sampling = static_cast<SampleParams*>(dalloc(h, static_cast<size_t>(max_batch) * sizeof(SampleParams)));
    if (cudaMallocHost(&h->h_stage, static_cast<size_t>(max_batch) * (sizeof(SampleParams) + 3 * 4)) != cudaSuccess) h->h_stage = nullptr;
    if (cudaEventCreateWithFlags(&h->staged, cudaEventDisableTiming) != cudaSuccess) h->staged = nullptr;
    ok &= h->d_lens && h->d_sampling && h->h_stage && h->staged;
    ok &= h->embed && h->final_norm && h->IN && h->X && h->XN && h->Q && h->AO && h->HM && h->LIN && h->LAST && h->LOGITS &&
          h->LOGITS_ALL && h->ws && h->kcache && h->vcache && h->ids && h->out_ids && h->d_err;
    if (!ok) { blurr_llm_destroy(h); return fail(BLURR_ERR_CUDA, "blurr_llm_create: device allocation failed"); }
    h->expected_keys = 3 + static_cast<size_t>(c.num_layers) * 9;
    *out = h;
    return 0;
}

static int pack(const bf16* src, int rows, int cols, Lin& L, int row_mul, int row_off) {
    const cudaError_t e = launch_pack_rows(nullptr, src, rows, cols, L.w, row_mul, row_off, L.K / 64);
    return e == cudaSuccess ? 0 : fail(BLURR_ERR_CUDA, std::string("weight repack: ") + cudaGetErrorString(e));
}

extern "C" int blurr_llm_set_weight(blurr_llm_t* h, const char* key_c, const void* dev_ptr, const int64_t* shape, int ndim) {
    if (!h || !key_c || !dev_ptr || !shape) return fail(BLURR_ERR_INVALID, "blurr_llm_set_weight: null argument");
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    const auto& c = h->cfg;
    const std::string key(key_c);
    const bf16* src = static_cast<const bf16*>(dev_ptr);
    const int QW = c.num_heads * c.head_dim, KVW = c.num_kv_heads * c.head_dim;
    auto is2 = [&](int64_t r, int64_t k) { return ndim == 2 && shape[0] == r && shape[1] == k; };
    auto is1 = [&](int64_t n) { return ndim == 1 && shape[0] == n; };
    auto bad = [&]() { return fail(BLURR_ERR_INVALID, "unexpected shape for " + key); };
    auto vec = [&](bf16* dst) -> int {
        if (!is1(c.hidden)) return bad();
        LLM_CUDA_TRY(cudaMemcpy(dst, src, static_cast<size_t>(c.hidden) * 2, cudaMemcpyDeviceToDevice));
        return 0;
    };
    int rc = 0;
    if (key == "model.embed_tokens.weight") {
        if (!is2(c.vocab, c.hidden)) return bad();
        LLM_CUDA_TRY(cudaMemcpy(h->embed, src, static_cast<size_t>(c.vocab) * c.hidden * 2, cudaMemcpyDeviceToDevice));
    } else if (key == "model.norm.weight") {
        rc = vec(h->final_norm);
    } else if (key == "lm_head.weight") {
        if (!is2(c.vocab, c.hidden)) return bad();
        rc = pack(src, c.vocab, c.hidden, h->lm_head, 1, 0);
    } else if (key.rfind("model.layers.", 0) == 0) {
        const size_t dot = key.find('.', 13);
        if (dot == std::string::npos) return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
        const int l = atoi(key.substr(13, dot - 13).c_str());
        if (l < 0 || l >= c.num_layers) return fail(BLURR_ERR_INVALID, "layer index out of range in " + key);
        Layer& L = h->layers[l];
        const std::string rest = key.substr(dot + 1);
        if (rest == "self_attn.q_proj.weight") { if (!is2(QW, c.hidden)) return bad(); rc = pack(src, QW, c.hidden, L.qkv, 1, 0); }
        else if (rest == "self_attn.k_proj.weight") { if (!is2(KVW, c.hidden)) return bad(); rc = pack(src, KVW, c.hidden, L.qkv, 1, QW); }
        else if (rest == "self_attn.v_proj.weight") { if (!is2(KVW, c.hidden)) return bad(); rc = pack(src, KVW, c.hidden, L.qkv, 1, QW + KVW); }
        else if (rest == "self_attn.o_proj.weight") { if (!is2(c.hidden, QW)) return bad(); rc = pack(src, c.hidden, QW, L.o, 1, 0); }
        // gate_j / up_j alternate rows: the GLU epilogue pairs adjacent accumulator rows
        else if (rest == "mlp.gate_proj.weight") { if (!is2(c.intermediate, c.hidden)) return bad(); rc = pack(src, c.intermediate, c.hidden, L.gu, 2, 0); }
        else if (rest == "mlp.up_proj.weight") { if (!is2(c.intermediate, c.hidden)) return bad(); rc = pack(src, c.intermediate, c.hidden, L.gu, 2, 1); }
        else if (rest == "mlp.down_proj.weight") { if (!is2(c.hidden, c.intermediate)) return bad(); rc = pack(src, c.hidden, c.intermediate, L.down, 1, 0); }
        else if (rest == "input_layernorm.weight") rc = vec(L.in_ln);
        else if (rest == "post_attention_layernorm.weight") rc = vec(L.post_ln);
        else return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    } else {
        return fail(BLURR_ERR_INVALID, "unknown state_dict key " + key);
    }
    if (rc) return rc;
    h->seen.insert(key);
    h->finalized = false;
    return 0;
}

extern "C" int blurr_llm_set_rope_table(blurr_llm_t* h, const float* cos_dev, const float* sin_dev, int n_pos) {
    if (!h || !cos_dev || !sin_dev) return fail(BLURR_ERR_INVALID, "blurr_llm_set_rope_table: null argument");
    if (n_pos < h->cfg.max_positions) return fail(BLURR_ERR_INVALID, "rope table shorter than max_positions");
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    const size_t bytes = static_cast<size_t>(n_pos) * (h->cfg.head_dim / 2) * 4;
    if (!h->cos_t || h->n_pos != n_pos) {
        h->cos_t = static_cast<float*>(dalloc(h, bytes));
        h->sin_t = static_cast<float*>(dalloc(h, bytes));
        if (!h->cos_t || !h->sin_t) return fail(BLURR_ERR_CUDA, "rope table allocation failed");
        h->n_pos = n_pos;
    }
    LLM_CUDA_TRY(cudaMemcpy(h->cos_t, cos_dev, bytes, cudaMemcpyDeviceToDevice));
    LLM_CUDA_TRY(cudaMemcpy(h->sin_t, sin_dev, bytes, cudaMemcpyDeviceToDevice));
    return 0;
}

extern "C" int blurr_llm_finalize(blurr_llm_t* h) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_llm_finalize: null handle");
    if (h->seen.size() != h->expected_keys)
        return fail(BLURR_ERR_STATE, "blurr_llm_finalize: " + std::to_string(h->expected_keys - h->seen.size()) + " state_dict keys missing");
    if (!h->cos_t) return fail(BLURR_ERR_STATE, "blurr_llm_finalize: call blurr_llm_set_rope_table first");
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    LLM_CUDA_TRY(cudaDeviceSynchronize());
    drop_graphs(h);
    h->finalized = true;
    return 0;
}

// K slices of a few-token GEMM: tiles * S CTAs in as few, as full waves of 148 as possible (each slice >= 4 k-blocks)
int blurr::pick_splitk_waves(int tiles, int kb_total) {
    int best_s = 1;
    double best = 0.0;
    for (int s = 1; s <= 16; ++s) {
        if (s > 1 && kb_total / s < 4) break;
        const int ctas = tiles * s;
        const double eff = static_cast<double>(ctas) / (static_cast<double>((ctas + kSMs - 1) / kSMs) * kSMs);
        if (eff > best + 0.02) { best = eff; best_s = s; }
    }
    return best_s;
}

namespace {

struct Run {
    blurr_llm* h;
    cudaStream_t st;
    int rc = 0;

    unsigned long long* slot(const std::string& what) {
        if (!h->trace || !h->trace_buf || h->trace_labels.size() >= static_cast<size_t>(kTraceMax)) return nullptr;
        h->trace_labels.push_back(what);
        return h->trace_buf + (h->trace_labels.size() - 1) * 4;
    }
    void launched(cudaError_t e, const char* what) {
        ++h->launches;
        if (e != cudaSuccess && !rc) rc = fail(BLURR_ERR_CUDA, std::string(what) + " launch failed: " + cudaGetErrorString(e));
    }
    // Y = X W^T.  Few tokens: fp32 split-K partials in the workspace (returns the slice count); otherwise the bf16 linear
    // output in `out` (returns 0).  EPI_GEGLU: SwiGLU straight from the epilogue (out = HM).
    GemmCall make_call(const Lin& L, const bf16* X, int T, int epi, bf16* out, int ldo) const {
        GemmCall c{};
        c.W = L.w; c.Nw = L.Nw; c.K = L.K; c.ldw = L.K; c.w_packed = 1;
        c.X = X; c.T = T; c.ldx = L.K;
        c.epi = epi; c.splitk = 1; c.glu_act = 1; c.w_static = 1;
        c.out = out; c.ldo = ldo;
        if (epi == EPI_PARTIAL) {
            c.splitk = T <= kFewTokens ? pick_splitk_waves(L.Nw / 128, (L.K + 63) / 64)
                                       : gemm_plan_chunked_splitk(T, L.Nw, L.K, h->ws_floats, &c.bn_override);
            c.partial = h->ws;
        }
        return c;
    }
    int gemm(const Lin& L, const bf16* X, int T, int epi, bf16* out, int ldo) {
        if (rc) return 0;
        GemmCall c = make_call(L, X, T, epi, out, ldo);
        if (epi == EPI_PARTIAL && static_cast<size_t>(c.splitk) * T * L.Nw > h->ws_floats) {
            rc = fail(BLURR_ERR_STATE, "split-K workspace too small");
            return 0;
        }
        std::string err;
        char nm[96];
        snprintf(nm, sizeof nm, "gemm[epi%d T%d N%d K%d S%d]", epi, T, L.Nw, L.K, c.splitk);
        c.trace = slot(nm);
        const int s = gemm_launch(st, c, &err);
        ++h->launches;
        if (s < 0) { rc = fail(BLURR_ERR_CUDA, err); return 0; }
        return epi == EPI_PARTIAL ? s : 0;
    }
    // x = res + bf16(linear output); xn = LlamaRMSNorm(x) with `norm_w` (nullptr: no norm)
    void consumer(int splitk, const bf16* lin, int T, int N, int ldp, const bf16* res, bf16* x_out, const bf16* norm_w, bf16* xn_out) {
        if (rc) return;
        ConsumerArgs a{};
        a.T = T; a.N = N; a.ldp = ldp; a.splitk = splitk > 0 ? splitk : 1;
        if (splitk > 0) a.partial = h->ws;
        else if (lin != nullptr) { a.lin = lin; a.ldl = ldp; }
        a.add_mode = (splitk > 0 || lin != nullptr) ? ADD_RESIDUAL : ADD_NONE;
        a.res = res; a.ldr = N; a.out_scale = 1.0f;
        a.x_out = x_out; a.ldx = N;
        a.norm_mode = norm_w ? NORM_RMS_LLAMA : NORM_NONE; a.norm_w = norm_w; a.eps = h->cfg.rms_eps;
        a.xn_out = norm_w ? xn_out : nullptr; a.ldn = N;
        a.trace = slot("consumer[T" + std::to_string(T) + "]");
        launched(launch_consumer(st, a), "consumer");
    }

    // One decoder layer over B sequences x Tq new tokens at positions pos0..pos0+Tq-1 (modeling_llama.py LlamaDecoderLayer).
    // `lens` (decode of a ragged batch, Tq == 1): sequence b's token sits at position lens[b] + step - 1 instead and
    // attends lens[b] + step keys; pos0 is then the batch's largest position.
    // `blk` (forward_rows, pos0 == 0): the attention takes OFT's rule with lengths d_lens and block starts blk.
    void layer(int l, int B, int Tq, int pos0, const bf16* next_norm, const int* lens = nullptr, int step = 0, const int* blk = nullptr) {
        const auto& c = h->cfg;
        Layer& L = h->layers[l];
        const int T = B * Tq, QW = c.num_heads * c.head_dim, KVW = c.num_kv_heads * c.head_dim;
        const bool few = T <= kFewTokens;
        const bool part = few || T <= kMidTokens;       // o / down: few weight tiles, long K -> split-K partials + consumer
        const size_t cache_off = static_cast<size_t>(l) * h->max_batch * c.max_positions * KVW;
        // q/k/v projections + RoPE + cache append
        int s = gemm(L.qkv, h->XN, T, few ? EPI_PARTIAL : EPI_STORE, h->LIN, L.qkv.Nw);
        RopeMhaArgs r{};
        if (few) { r.partial = h->ws; r.splitk = s; } else { r.lin = h->LIN; r.ldl = L.qkv.Nw; r.splitk = 1; }
        r.T = T; r.ldp = L.qkv.Nw; r.n_heads = c.num_heads; r.n_kv_heads = c.num_kv_heads; r.head_dim = c.head_dim;
        r.tokens_per_seq = Tq; r.pos0 = pos0; r.cos_table = h->cos_t; r.sin_table = h->sin_t; r.n_pos = h->n_pos;
        r.q_out = h->Q; r.k_cache = h->kcache + cache_off; r.v_cache = h->vcache + cache_off; r.n_slots = c.max_positions;
        r.seq_len = lens; r.len_off = step - 1;
        // causal multi-head attention over the cache
        MhaAttnArgs m{};
        m.q = h->Q; m.q_per_sample = Tq; m.q_pos0 = pos0; m.k_cache = r.k_cache; m.v_cache = r.v_cache;
        m.n_slots = c.max_positions; m.n_keys = pos0 + Tq; m.batch = B; m.n_heads = c.num_heads; m.n_kv_heads = c.num_kv_heads;
        m.head_dim = c.head_dim; m.scale = static_cast<float>(std::pow(static_cast<double>(c.head_dim), -0.5)); m.out = h->AO;
        m.seq_len = lens; m.len_off = step;
        const bool fuse = blk == nullptr && few && Tq == 1 && mha_decode_fuses_rope(m);       // decode: RoPE + append inside the attention kernel
        if (!fuse) {
            r.trace = slot("rope_mha");
            if (!rc) launched(launch_rope_mha(st, r), "rope_mha");
        }
        if (blk != nullptr) {
            m.seq_len = h->d_lens; m.len_off = 0;
            m.trace = slot("mha_block_prefill");
            if (!rc) launched(launch_mha_block_attention(st, m, blk), "mha_block_attention");
        } else {
            m.trace = slot(Tq == 1 ? (fuse ? "rope+mha_decode" : "mha_decode") : "mha_prefill");
            if (!rc) launched(launch_mha_attention(st, m, fuse ? &r : nullptr), "mha_attention");
        }
        // o_proj + residual + post-attention norm
        s = gemm(L.o, h->AO, T, part ? EPI_PARTIAL : EPI_STORE, h->LIN, L.o.Nw);
        consumer(part ? s : 0, part ? nullptr : h->LIN, T, c.hidden, L.o.Nw, h->X, h->X, L.post_ln, h->XN);
        // SwiGLU MLP
        if (few) {
            s = gemm(L.gu, h->XN, T, EPI_PARTIAL, nullptr, 0);
            if (!rc) launched(launch_glu_partial(st, h->ws, s, T, L.gu.Nw, 1, h->HM, c.intermediate, slot("glu")), "glu");
        } else {
            gemm(L.gu, h->XN, T, EPI_GEGLU, h->HM, c.intermediate);
        }
        s = gemm(L.down, h->HM, T, part ? EPI_PARTIAL : EPI_STORE, h->LIN, L.down.Nw);
        consumer(part ? s : 0, part ? nullptr : h->LIN, T, c.hidden, L.down.Nw, h->X, h->X, next_norm, h->XN);
        (void)QW;
    }

    // final-normed rows [B][hidden] -> logits -> token `step` of every sequence: greedy, or (`sampled`) drawn with the
    // per-row parameters in d_sampling
    void head(const bf16* xn_rows, int B, int step, int n_new, bool keep_logits, bool sampled) {
        const auto& c = h->cfg;
        const int s = gemm(h->lm_head, xn_rows, B, EPI_PARTIAL, nullptr, 0);
        if (!rc) launched(launch_bias_act(st, h->ws, s, B, h->lm_head.Nw, h->lm_head.Nw, nullptr, ACT_NONE, 1.0f, h->LOGITS, h->lm_head.Nw), "logits");
        if (sampled) {
            unsigned long long* tr = slot("sample_rows");
            if (!rc) launched(launch_sample_rows(st, h->LOGITS, B, h->lm_head.Nw, c.vocab, h->d_sampling, step, h->ids, h->out_ids + step,
                                                 n_new, nullptr, h->d_err, tr), "sample_rows");
        } else if (!rc) {
            launched(launch_argmax_rows(st, h->LOGITS, B, h->lm_head.Nw, c.vocab, h->ids, h->out_ids + step, n_new), "argmax");
        }
        if (keep_logits && !rc) {
            const cudaError_t e = cudaMemcpy2DAsync(h->LOGITS_ALL + static_cast<size_t>(step) * c.vocab, static_cast<size_t>(n_new) * c.vocab * 2,
                                                    h->LOGITS, static_cast<size_t>(h->lm_head.Nw) * 2, static_cast<size_t>(c.vocab) * 2, B,
                                                    cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) rc = fail(BLURR_ERR_CUDA, std::string("logits copy: ") + cudaGetErrorString(e));
        }
    }
};

// `ragged`: sequence b's prompt is rows 0 .. d_lens[b] - 1 of its T rows; the rest are pads.  Prefill runs over all T rows
// unchanged (pads come after the real rows, so the causal mask hides them from every real query); the pads are zeroed
// first, the first token is read from row d_lens[b] - 1, and decode step i places sequence b's token at d_lens[b] + i - 1.
void reset_trace(Run& R) {
    blurr_llm* h = R.h;
    if (h->trace && h->trace_buf) {
        h->trace_labels.clear();
        if (cudaMemsetAsync(h->trace_buf, 0xFF, static_cast<size_t>(kTraceMax) * 4 * sizeof(unsigned long long), R.st) != cudaSuccess)
            R.rc = fail(BLURR_ERR_CUDA, "trace reset failed");
    }
}

void run_generate(Run& R, int B, int T, int n_new, bool keep_logits, bool ragged, bool sampled) {
    blurr_llm* h = R.h;
    const auto& c = h->cfg;
    const int L = c.num_layers;
    reset_trace(R);
    const int* lens = ragged ? h->d_lens : nullptr;
    if (ragged && !R.rc) R.launched(launch_zero_pad_rows(R.st, h->IN, B, T, c.hidden, lens), "zero_pad_rows");
    // ---- prefill: X <- inputs_embeds, XN <- input norm of layer 0 ----
    R.consumer(0, nullptr, B * T, c.hidden, c.hidden, h->IN, h->X, h->layers[0].in_ln, h->XN);
    for (int l = 0; l < L; ++l) R.layer(l, B, T, 0, l + 1 < L ? h->layers[l + 1].in_ln : h->final_norm);
    if (!R.rc) R.launched(launch_gather_rows(R.st, h->XN, B, T, T - 1, c.hidden, h->LAST, lens), "gather_last");
    R.head(h->LAST, B, 0, n_new, keep_logits, sampled);
    // ---- decode: one token per sequence per step ----
    for (int i = 1; i < n_new; ++i) {
        if (!R.rc) R.launched(launch_embed_rows(R.st, h->ids, B, h->embed, c.vocab, c.hidden, h->X, h->d_err), "embed");
        R.consumer(0, nullptr, B, c.hidden, c.hidden, h->X, nullptr, h->layers[0].in_ln, h->XN);
        for (int l = 0; l < L; ++l) R.layer(l, B, 1, T + i - 1, l + 1 < L ? h->layers[l + 1].in_ln : h->final_norm, lens, i);
        R.head(h->XN, B, i, n_new, keep_logits, sampled);
    }
}

// forward_rows: the prefill schedule over B x T rows with OFT's attention rule (lengths d_lens, block starts d_blk); pads
// are zeroed first, and XN ends as the final norm's output of every row.
void run_forward_rows(Run& R, int B, int T) {
    blurr_llm* h = R.h;
    const auto& c = h->cfg;
    const int L = c.num_layers;
    reset_trace(R);
    if (!R.rc) R.launched(launch_zero_pad_rows(R.st, h->IN, B, T, c.hidden, h->d_lens), "zero_pad_rows");
    R.consumer(0, nullptr, B * T, c.hidden, c.hidden, h->IN, h->X, h->layers[0].in_ln, h->XN);
    for (int l = 0; l < L; ++l) R.layer(l, B, T, 0, l + 1 < L ? h->layers[l + 1].in_ln : h->final_norm, nullptr, 0, h->d_blk);
}

using GraphKey = std::tuple<int, int, int, int, int, int, int>;

// Runs `body` on `st`: eagerly (option use_cuda_graph 0), or as the CUDA graph cached under `key`, captured on first use
// after one warm run (attribute setup, tensor maps).  h->launches ends as the launch count of one run.
template <typename Body>
int run_graph(blurr_llm* h, cudaStream_t st, const GraphKey& key, Body body) {
    h->launches = 0;
    Run R{h, st};
    if (!h->use_graph) {
        body(R);
        return R.rc;
    }
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
        body(R);
        if (R.rc) return R.rc;
        LLM_CUDA_TRY(cudaStreamSynchronize(st));
        h->launches = 0;
        cudaStream_t cs;
        LLM_CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        Run C{h, cs};
        cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) { cudaStreamDestroy(cs); return fail(BLURR_ERR_CUDA, "graph capture begin failed"); }
        body(C);
        cudaGraph_t g = nullptr;
        e = cudaStreamEndCapture(cs, &g);
        cudaStreamDestroy(cs);
        if (C.rc) { if (g) cudaGraphDestroy(g); return C.rc; }
        if (e != cudaSuccess || !g) return fail(BLURR_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(e));
        cudaGraphExec_t ex = nullptr;
        e = cudaGraphInstantiate(&ex, g, 0);
        if (e != cudaSuccess) { cudaGraphDestroy(g); return fail(BLURR_ERR_CUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(e)); }
        it = h->graphs.emplace(key, blurr_llm::GraphEntry{g, ex, h->launches}).first;
    }
    LLM_CUDA_TRY(cudaGraphLaunch(it->second.exec, st));
    h->launches = it->second.launches;
    return 0;
}

}  // namespace

extern "C" int blurr_llm_embed(blurr_llm_t* h, void* cuda_stream, const int64_t* ids, int n, void* rows_out) {
    if (!h || !ids || !rows_out || n < 1) return fail(BLURR_ERR_INVALID, "blurr_llm_embed: bad arguments");
    if (!h->seen.count("model.embed_tokens.weight")) return fail(BLURR_ERR_STATE, "blurr_llm_embed: embed_tokens not set");
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    LLM_CUDA_TRY(launch_embed_rows(static_cast<cudaStream_t>(cuda_stream), ids, n, h->embed, h->cfg.vocab, h->cfg.hidden,
                                   static_cast<bf16*>(rows_out), h->d_err));
    return 0;
}

// Uploads the per-row inputs a graph reads at replay (host arrays of `rows` entries, any may be null) through the pinned
// staging buffer, on `st` ahead of the launch: lengths -> d_lens, block starts -> d_blk, row starts -> d_row0.
static int stage_rows(blurr_llm_t* h, cudaStream_t st, int rows, const int32_t* lens, const blurr_llm_sampling* params,
                      const int32_t* blk = nullptr, const int32_t* row0 = nullptr) {
    if (!lens && !params && !blk && !row0) return 0;
    LLM_CUDA_TRY(cudaEventSynchronize(h->staged));              // the previous upload has read the staging buffer
    unsigned char* stage_params = h->h_stage;
    if (params) {
        memcpy(stage_params, params, static_cast<size_t>(rows) * sizeof(SampleParams));
        LLM_CUDA_TRY(cudaMemcpyAsync(h->d_sampling, stage_params, static_cast<size_t>(rows) * sizeof(SampleParams), cudaMemcpyHostToDevice, st));
    }
    const int32_t* src[3] = {lens, blk, row0};
    int* dst[3] = {h->d_lens, h->d_blk, h->d_row0};
    for (int i = 0; i < 3; ++i) {
        if (!src[i]) continue;
        unsigned char* stage = h->h_stage + static_cast<size_t>(h->max_batch) * (sizeof(SampleParams) + 4 * i);
        memcpy(stage, src[i], static_cast<size_t>(rows) * 4);
        LLM_CUDA_TRY(cudaMemcpyAsync(dst[i], stage, static_cast<size_t>(rows) * 4, cudaMemcpyHostToDevice, st));
    }
    LLM_CUDA_TRY(cudaEventRecord(h->staged, st));
    return 0;
}

// HF's checks of the warpers' arguments (TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper) on the host
static int check_sampling(const char* fn, const blurr_llm_sampling* params, int rows) {
    if (!params) return fail(BLURR_ERR_INVALID, std::string(fn) + ": params is null");
    for (int b = 0; b < rows; ++b) {
        const blurr_llm_sampling& p = params[b];
        const std::string at = std::string(fn) + ": params[" + std::to_string(b) + "].";
        if (!std::isfinite(p.temperature) || !(p.temperature > 0.0f))
            return fail(BLURR_ERR_INVALID, at + "temperature = " + std::to_string(p.temperature) + " must be finite and > 0");
        if (p.top_k < 0) return fail(BLURR_ERR_INVALID, at + "top_k = " + std::to_string(p.top_k) + " must be >= 0");
        if (!std::isfinite(p.top_p) || p.top_p < 0.0f || p.top_p > 1.0f)
            return fail(BLURR_ERR_INVALID, at + "top_p = " + std::to_string(p.top_p) + " must be in [0, 1]");
    }
    return 0;
}

// `prompt_lens` (host) selects the ragged schedule, even when every length is max_prompt_len; `params` (host) the sampler.
extern "C" int blurr_llm_generate(blurr_llm_t* h, void* cuda_stream, int batch, int max_prompt_len, const void* inputs_embeds,
                                  const int32_t* prompt_lens, const blurr_llm_sampling* params, int n_new, int64_t* out_ids,
                                  void* out_logits) {
    const char* fn = "blurr_llm_generate";
    if (!h || !inputs_embeds || !out_ids) return fail(BLURR_ERR_INVALID, std::string(fn) + ": null argument");
    if (!h->finalized) return fail(BLURR_ERR_STATE, std::string(fn) + ": call blurr_llm_finalize first");
    const auto& c = h->cfg;
    if (batch < 1 || batch > h->max_batch) return fail(BLURR_ERR_INVALID, std::string(fn) + ": batch out of range");
    if (max_prompt_len < 1 || n_new < 1 || max_prompt_len + n_new > c.max_positions)
        return fail(BLURR_ERR_INVALID, std::string(fn) + ": max_prompt_len + n_new exceeds max_positions");
    if (max_prompt_len + n_new > kGenerateMaxPositions)
        return fail(BLURR_ERR_INVALID, std::string(fn) + ": max_prompt_len + n_new exceeds 320 (the decode attention's limit)");
    if (prompt_lens)
        for (int b = 0; b < batch; ++b)
            if (prompt_lens[b] < 1 || prompt_lens[b] > max_prompt_len)
                return fail(BLURR_ERR_INVALID, std::string(fn) + ": prompt_lens[" + std::to_string(b) + "] = " +
                                                   std::to_string(prompt_lens[b]) + " is outside 1.." + std::to_string(max_prompt_len));
    if (out_logits != nullptr && n_new > kMaxKeptLogits)
        return fail(BLURR_ERR_INVALID, std::string(fn) + ": logits are kept for at most 16 new tokens");
    if (const int rc = params ? check_sampling(fn, params, batch) : 0) return rc;
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const bool keep = out_logits != nullptr;
    const bool ragged = prompt_lens != nullptr;
    const bool sampled = params != nullptr;
    LLM_CUDA_TRY(cudaMemcpyAsync(h->IN, inputs_embeds, static_cast<size_t>(batch) * max_prompt_len * c.hidden * 2, cudaMemcpyDeviceToDevice, st));
    if (const int rc = stage_rows(h, st, batch, prompt_lens, params)) return rc;
    const GraphKey key = std::make_tuple(batch, max_prompt_len, n_new, keep ? 1 : 0, ragged ? 1 : 0, sampled ? 1 : 0, 0);
    if (const int rc = run_graph(h, st, key, [&](Run& R) { run_generate(R, batch, max_prompt_len, n_new, keep, ragged, sampled); }))
        return rc;
    LLM_CUDA_TRY(cudaMemcpyAsync(out_ids, h->out_ids, static_cast<size_t>(batch) * n_new * 8, cudaMemcpyDeviceToDevice, st));
    if (keep)
        LLM_CUDA_TRY(cudaMemcpyAsync(out_logits, h->LOGITS_ALL, static_cast<size_t>(batch) * n_new * c.vocab * 2, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int blurr_llm_forward_rows(blurr_llm_t* h, void* cuda_stream, int batch, int max_len, const void* inputs_embeds,
                                      const int32_t* seq_lens, const int32_t* block_starts, const int32_t* row_starts, int n_rows,
                                      void* out_hidden) {
    const char* fn = "blurr_llm_forward_rows";
    if (!h || !inputs_embeds || !seq_lens || !block_starts || !row_starts || !out_hidden)
        return fail(BLURR_ERR_INVALID, std::string(fn) + ": null argument");
    if (!h->finalized) return fail(BLURR_ERR_STATE, std::string(fn) + ": call blurr_llm_finalize first");
    const auto& c = h->cfg;
    if (batch < 1 || batch > h->max_batch) return fail(BLURR_ERR_INVALID, std::string(fn) + ": batch out of range");
    if (max_len < 1 || max_len > c.max_positions)
        return fail(BLURR_ERR_INVALID, std::string(fn) + ": max_len must be in 1..max_positions (" + std::to_string(c.max_positions) + ")");
    if (n_rows < 1 || n_rows > max_len) return fail(BLURR_ERR_INVALID, std::string(fn) + ": n_rows must be in 1..max_len");
    for (int b = 0; b < batch; ++b) {
        const std::string at = std::string(fn) + ": sequence " + std::to_string(b) + ": ";
        if (seq_lens[b] < 1 || seq_lens[b] > max_len)
            return fail(BLURR_ERR_INVALID, at + "seq_lens = " + std::to_string(seq_lens[b]) + " is outside 1.." + std::to_string(max_len));
        if (block_starts[b] < 1 || block_starts[b] > seq_lens[b])
            return fail(BLURR_ERR_INVALID, at + "block_starts = " + std::to_string(block_starts[b]) + " is outside 1..seq_lens");
        if (row_starts[b] < 0 || row_starts[b] > seq_lens[b] - n_rows)
            return fail(BLURR_ERR_INVALID, at + "rows " + std::to_string(row_starts[b]) + " + " + std::to_string(n_rows) +
                                               " run past seq_lens = " + std::to_string(seq_lens[b]));
    }
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    LLM_CUDA_TRY(cudaMemcpyAsync(h->IN, inputs_embeds, static_cast<size_t>(batch) * max_len * c.hidden * 2, cudaMemcpyDeviceToDevice, st));
    if (const int rc = stage_rows(h, st, batch, seq_lens, nullptr, block_starts, row_starts)) return rc;
    // the graph ends at XN; the rows go straight to the caller's buffer, so one graph serves every n_rows and out_hidden
    const GraphKey key = std::make_tuple(batch, max_len, 0, 0, 0, 0, 1);
    if (const int rc = run_graph(h, st, key, [&](Run& R) { run_forward_rows(R, batch, max_len); })) return rc;
    LLM_CUDA_TRY(launch_gather_row_block(st, h->XN, batch, max_len, h->d_row0, n_rows, c.hidden, static_cast<bf16*>(out_hidden)));
    ++h->launches;
    return 0;
}

extern "C" int blurr_llm_sample(blurr_llm_t* h, void* cuda_stream, const void* logits, int rows, int ld, const blurr_llm_sampling* params,
                                int step, int64_t* out_ids, float* out_probs) {
    const char* fn = "blurr_llm_sample";
    if (!h || !logits || !out_ids) return fail(BLURR_ERR_INVALID, std::string(fn) + ": null argument");
    if (rows < 1 || rows > h->max_batch) return fail(BLURR_ERR_INVALID, std::string(fn) + ": rows out of range 1..max_batch");
    if (ld < h->cfg.vocab) return fail(BLURR_ERR_INVALID, std::string(fn) + ": ld < vocab");
    if (step < 0) return fail(BLURR_ERR_INVALID, std::string(fn) + ": step < 0");
    if (const int rc = check_sampling(fn, params, rows)) return rc;
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    if (const int rc = stage_rows(h, st, rows, nullptr, params)) return rc;
    LLM_CUDA_TRY(launch_sample_rows(st, static_cast<const bf16*>(logits), rows, ld, h->cfg.vocab, h->d_sampling, step, out_ids, nullptr, 0,
                                    out_probs, h->d_err, nullptr));
    return 0;
}

extern "C" int blurr_llm_set_option(blurr_llm_t* h, const char* name, int64_t value) {
    if (!h || !name) return fail(BLURR_ERR_INVALID, "blurr_llm_set_option: null argument");
    const std::string n(name);
    if (n == "use_cuda_graph") h->use_graph = value != 0;
    else if (n == "trace") {
        if (value != 0 && !h->trace_buf) {
            h->trace_buf = static_cast<unsigned long long*>(dalloc(h, static_cast<size_t>(kTraceMax) * 4 * sizeof(unsigned long long)));
            if (!h->trace_buf) return fail(BLURR_ERR_CUDA, "trace buffer allocation failed");
        }
        h->trace = value != 0;
        drop_graphs(h);
    }
    else return fail(BLURR_ERR_INVALID, "blurr_llm_set_option: unknown option " + n);
    return 0;
}

extern "C" int blurr_llm_check(blurr_llm_t* h, void* cuda_stream) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_llm_check: null handle");
    LLM_CUDA_TRY(cudaSetDevice(h->device));
    LLM_CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(cuda_stream)));
    int flag = 0;
    LLM_CUDA_TRY(cudaMemcpy(&flag, h->d_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        LLM_CUDA_TRY(cudaMemset(h->d_err, 0, sizeof(int)));
        if (flag & 1) return fail(BLURR_ERR_INPUT, "a generated token id fell outside the embedding table");
        return fail(BLURR_ERR_INPUT, "sampling: a logits row had no finite positive mass (all -inf / NaN, a +inf logit, or a scaled "
                                     "score that overflows); that row took the greedy argmax");
    }
    const int g = gemm_take_timeout_flag(), a = attn_take_timeout_flag();
    if (g > 0 || a > 0) return fail(BLURR_ERR_CUDA, "a bounded pipeline wait expired inside a GEMM / attention kernel");
    return 0;
}

extern "C" int blurr_llm_trace_report(blurr_llm_t* h, char* buf, size_t buf_bytes) {
    if (!h || !buf || buf_bytes == 0) return fail(BLURR_ERR_INVALID, "blurr_llm_trace_report: bad arguments");
    if (!h->trace || !h->trace_buf) return fail(BLURR_ERR_STATE, "blurr_llm_trace_report: option trace is off");
    LLM_CUDA_TRY(cudaDeviceSynchronize());
    const size_t n = h->trace_labels.size();
    std::vector<unsigned long long> host(n * 4);
    if (n) LLM_CUDA_TRY(cudaMemcpy(host.data(), h->trace_buf, n * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    unsigned long long t0 = ~0ull;
    for (size_t i = 0; i < n; ++i) if (host[i * 4] < t0) t0 = host[i * 4];
    std::string out = "# idx start_us waited_us end_us label   (globaltimer, relative to the first kernel start)\n";
    char line[256];
    for (size_t i = 0; i < n; ++i) {
        const unsigned long long s = host[i * 4], w = host[i * 4 + 1], e = ~host[i * 4 + 2];
        if (s == ~0ull) continue;
        snprintf(line, sizeof line, "%zu %.3f %.3f %.3f %s\n", i, (s - t0) * 1e-3, w == ~0ull ? -1.0 : (w - t0) * 1e-3, (e - t0) * 1e-3,
                 h->trace_labels[i].c_str());
        out += line;
    }
    if (out.size() + 1 > buf_bytes) return fail(BLURR_ERR_INVALID, "blurr_llm_trace_report: buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
    return 0;
}

extern "C" int64_t blurr_llm_last_launch_count(const blurr_llm_t* h) { return h ? h->launches : 0; }
extern "C" int64_t blurr_llm_weight_bytes_per_token(const blurr_llm_t* h) { return h ? h->weight_bytes : 0; }
