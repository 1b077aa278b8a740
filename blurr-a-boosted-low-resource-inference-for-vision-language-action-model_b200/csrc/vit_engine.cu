// Generic pre-LN ViT encoder + MLP projector behind include/blurr_vit.h: the vision side of the OpenVLA-7B-shaped path
// (SURVEY.md 8(f) row 3) - DINOv2 ViT-L/14 (cls + 4 register tokens, LayerScale, exact GELU) and SigLIP-so400m/14 towers,
// patch tokens of the second-to-last block, and the 3-layer GELU projector.  A third client of the Pi-0 kernels: the
// schedule is the one of the Pi-0 SigLIP tower (engine.cu run_vision) with three additions - prefix-token rows (the
// consumer's output row map), LayerScale (the consumer's per-column scale) and the erf GELU flavour of the GEMM epilogue.
// FiLM handles (film_dim > 0, OpenVLA-OFT's language conditioning) add one GEMM in front of the blocks - every block's
// gamma and beta from the caller's conditioning rows - and the FiLM variant of the out-projection's consumer.
#include "blurr_pi0.h"
#include "blurr_vit.h"

#include "common.cuh"
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
int record_error(int code, const std::string& msg);      // engine.cu
}
using namespace blurr;

static int fail(int code, const std::string& msg) { return record_error(code, msg); }
#define VIT_CUDA_TRY(expr)                                                                       \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return fail(BLURR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

namespace {

constexpr int kMidRows = 288;        // up to here split-K partials (chunked), above the bf16 hand-off

struct VLin { bf16* w = nullptr; bf16* bias = nullptr; int Nw = 0, K = 0, N = 0, Kreal = 0; };
struct VLayer { bf16 *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr, *ls1 = nullptr, *ls2 = nullptr; VLin qkv, o, fc1, fc2; };

__global__ void vit_pack_rows_kernel(const bf16* __restrict__ src, int rows, int cols, bf16* __restrict__ dst, int row_off, int kb_total) {
    const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<size_t>(rows) * cols) return;
    const int r = static_cast<int>(idx / cols), c = static_cast<int>(idx - static_cast<size_t>(r) * cols);
    const int dr = r + row_off;
    dst[((static_cast<size_t>(dr / 128) * kb_total + c / 64) * 128 + dr % 128) * 64 + c % 64] = src[idx];
}

template <typename H>
void* dalloc_in(H* h, size_t bytes) {
    void* p = nullptr;
    if (bytes == 0) bytes = 16;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, bytes);
    h->allocs.push_back(p);
    return p;
}

template <typename H>
bool alloc_lin(H* h, VLin& L, int N, int K) {
    L.N = N; L.Kreal = K;
    L.Nw = (N + 127) / 128 * 128;
    L.K = (K + 63) / 64 * 64;
    L.w = static_cast<bf16*>(dalloc_in(h, static_cast<size_t>(L.Nw) * L.K * 2));
    L.bias = static_cast<bf16*>(dalloc_in(h, static_cast<size_t>(L.Nw) * 2));
    return L.w && L.bias;
}

int pack_weight(const bf16* src, int rows, int cols, VLin& L, int row_off) {
    const size_t total = static_cast<size_t>(rows) * cols;
    vit_pack_rows_kernel<<<static_cast<unsigned>((total + 255) / 256), 256>>>(src, rows, cols, L.w, row_off, L.K / 64);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail(BLURR_ERR_CUDA, std::string("weight repack: ") + cudaGetErrorString(e));
}

// Shared launcher state of the two engines
struct Launcher {
    cudaStream_t st;
    float* ws;
    size_t ws_floats;
    bf16* lin;             // bf16 hand-off buffer [rows][widest Nw]
    int64_t* launches;
    int rc = 0;

    void launched(cudaError_t e, const char* what) {
        ++*launches;
        if (e != cudaSuccess && !rc) rc = fail(BLURR_ERR_CUDA, std::string(what) + " launch failed: " + cudaGetErrorString(e));
    }
    // returns the K slices of an EPI_PARTIAL launch, 0 for the other epilogues
    int gemm(const VLin& L, const bf16* X, int T, int epi, bf16* out, int ldo, int gelu_kind) {
        if (rc) return 0;
        GemmCall c{};
        c.W = L.w; c.Nw = L.Nw; c.K = L.K; c.ldw = L.K; c.w_packed = 1;
        c.X = X; c.T = T; c.ldx = L.K;
        c.epi = epi; c.splitk = 1; c.glu_act = gelu_kind; c.w_static = 1;
        c.bias = epi == EPI_PARTIAL ? nullptr : L.bias;
        c.out = out; c.ldo = ldo;
        if (epi == EPI_PARTIAL) {
            c.splitk = gemm_plan_chunked_splitk(T, L.Nw, L.K, ws_floats, &c.bn_override);
            c.partial = ws;
            if (static_cast<size_t>(c.splitk) * T * L.Nw > ws_floats) { rc = fail(BLURR_ERR_STATE, "split-K workspace too small"); return 0; }
        }
        std::string err;
        const int s = gemm_launch(st, c, &err);
        ++*launches;
        if (s < 0) { rc = fail(BLURR_ERR_CUDA, err); return 0; }
        return epi == EPI_PARTIAL ? s : 0;
    }
    // y = X W^T + b as split-K partials (<= 288 rows) or the bf16 linear output, then `fill` completes the consumer
    void linear_consumer(const VLin& L, const bf16* X, int T, ConsumerArgs a) {
        if (rc) return;
        a.T = T; a.N = L.N; a.ldp = L.Nw; a.out_scale = 1.0f;
        if (T <= kMidRows) {
            const int s = gemm(L, X, T, EPI_PARTIAL, nullptr, 0, 0);
            a.partial = ws; a.splitk = s; a.bias = L.bias;
        } else {
            gemm(L, X, T, EPI_STORE, lin, L.Nw, 0);
            a.lin = lin; a.ldl = L.Nw; a.splitk = 1; a.bias = nullptr;
        }
        if (!rc) launched(launch_consumer(st, a), "consumer");
    }
};

}  // namespace

struct blurr_vit {
    blurr_vit_config cfg{};
    int device = 0, max_batch = 1, n_patches = 0, seq = 0;
    std::vector<void*> allocs;
    VLin patch;
    bf16 *pos = nullptr, *prefix = nullptr;
    // FiLM: [layers * 2 * hidden][film_dim] tile-packed, block l's scale rows at 2 l hidden, its shift rows behind them;
    // cond [max_batch][film_dim] (the caller's rows, copied in before the graph), film_out [max_batch][film.Nw]
    VLin film;
    bf16 *cond = nullptr, *film_out = nullptr;
    std::vector<VLayer> layers;
    bf16 *patches = nullptr, *X = nullptr, *XN = nullptr, *QKV = nullptr, *AO = nullptr, *HM = nullptr, *LINB = nullptr;
    float* ws = nullptr;
    size_t ws_floats = 0;
    std::set<std::string> seen;
    size_t expected = 0;
    bool finalized = false, use_graph = true;
    int64_t launches = 0;
    // blocks between the patch im2col (reads the caller's pixels) and the final row copy (writes the caller's buffer)
    // only touch the handle's own buffers: one CUDA graph per (batch size, images per condition; 0 without FiLM)
    struct GraphEntry { cudaGraph_t graph; cudaGraphExec_t exec; int64_t launches; };
    std::map<std::pair<int, int>, GraphEntry> graphs;
};

extern "C" void blurr_vit_destroy(blurr_vit_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (auto& kv : h->graphs) { cudaGraphExecDestroy(kv.second.exec); cudaGraphDestroy(kv.second.graph); }
    for (void* p : h->allocs) cudaFree(p);
    gemm_forget_tensor_maps();
    delete h;
}

extern "C" int blurr_vit_create(const blurr_vit_config* cfg, int device, int max_batch, blurr_vit_t** out) {
    if (!cfg || !out || max_batch < 1) return fail(BLURR_ERR_INVALID, "blurr_vit_create: bad arguments");
    const blurr_vit_config& c = *cfg;
    if (c.abi_version != BLURR_VIT_ABI_VERSION) return fail(BLURR_ERR_INVALID, "blurr_vit_config abi_version mismatch");
    if (c.image_size != 224 || c.patch_size != 14) return fail(BLURR_ERR_INVALID, "the patch-embed kernel is built for 224x224 images, 14x14 patches");
    if (c.num_layers < 1 || c.hidden % 128 || c.hidden > 2048 || c.num_heads < 1 || c.hidden % c.num_heads)
        return fail(BLURR_ERR_INVALID, "hidden must be a multiple of 128 (<= 2048) and divisible by num_heads");
    const int hd = c.hidden / c.num_heads;
    if ((hd & 7) || hd > 80) return fail(BLURR_ERR_INVALID, "head_dim must be a multiple of 8 and <= 80");
    if (c.num_prefix_tokens < 0 || c.num_prefix_tokens > 16 || c.mlp_dim < 64) return fail(BLURR_ERR_INVALID, "bad prefix token count / mlp_dim");
    if (c.film_dim < 0 || c.film_dim % 64 || c.film_dim > 8192) return fail(BLURR_ERR_INVALID, "film_dim must be 0 or a multiple of 64 (<= 8192)");
    if (c.film_dim > 0 && c.hidden != 1024 && c.hidden != 1152)
        return fail(BLURR_ERR_INVALID, "FiLM towers must be 1024 (DINOv2-L) or 1152 (SigLIP-so400m) wide");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(BLURR_ERR_CUDA, "no CUDA device: the B200 path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BLURR_ERR_INVALID, "bad device index");
    cudaDeviceProp prop{};
    VIT_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(BLURR_ERR_CUDA, "this library is built for sm_100a only");
    VIT_CUDA_TRY(cudaSetDevice(device));
    auto* h = new blurr_vit();
    h->cfg = c; h->device = device; h->max_batch = max_batch;
    h->n_patches = (c.image_size / c.patch_size) * (c.image_size / c.patch_size);
    h->seq = h->n_patches + c.num_prefix_tokens;
    if (h->seq > 320) { delete h; return fail(BLURR_ERR_INVALID, "sequence longer than 320 tokens"); }
    const size_t T = static_cast<size_t>(max_batch) * h->seq, Tp = static_cast<size_t>(max_batch) * h->n_patches;
    const int H = c.hidden;
    auto bufb = [&](size_t elems) { return static_cast<bf16*>(dalloc_in(h, elems * 2)); };
    bool ok = alloc_lin(h, h->patch, H, 3 * c.patch_size * c.patch_size);
    h->pos = bufb(static_cast<size_t>(h->n_patches) * H);
    h->prefix = bufb(static_cast<size_t>(c.num_prefix_tokens > 0 ? c.num_prefix_tokens : 1) * H);
    h->layers.resize(c.num_layers);
    for (auto& L : h->layers) {
        ok &= alloc_lin(h, L.qkv, 3 * H, H) && alloc_lin(h, L.o, H, H) && alloc_lin(h, L.fc1, c.mlp_dim, H);
        ok &= alloc_lin(h, L.fc2, H, L.fc1.Nw);            // fc2 reads the padded fc1 output (pad columns are zero)
        L.ln1w = bufb(H); L.ln1b = bufb(H); L.ln2w = bufb(H); L.ln2b = bufb(H); L.ls1 = bufb(H); L.ls2 = bufb(H);
        ok &= L.ln1w && L.ln1b && L.ln2w && L.ln2b && L.ls1 && L.ls2;
    }
    if (c.film_dim > 0) {
        ok &= alloc_lin(h, h->film, c.num_layers * 2 * H, c.film_dim);
        h->cond = bufb(static_cast<size_t>(max_batch) * c.film_dim);
        h->film_out = bufb(static_cast<size_t>(max_batch) * h->film.Nw);
        ok &= h->cond && h->film_out;
    }
    const int mlp_pad = h->layers[0].fc1.Nw;
    h->patches = bufb(Tp * h->patch.K);
    h->X = bufb(T * H); h->XN = bufb(T * H); h->QKV = bufb(T * 3 * H); h->AO = bufb(T * H); h->HM = bufb(T * mlp_pad);
    h->LINB = bufb(T * static_cast<size_t>(3 * H > mlp_pad ? 3 * H : mlp_pad));
    h->ws_floats = 16 * static_cast<size_t>(kMidRows) * H;
    h->ws = static_cast<float*>(dalloc_in(h, h->ws_floats * 4));
    ok &= h->pos && h->prefix && h->patches && h->X && h->XN && h->QKV && h->AO && h->HM && h->LINB && h->ws;
    if (!ok) { blurr_vit_destroy(h); return fail(BLURR_ERR_CUDA, "blurr_vit_create: device allocation failed"); }
    h->expected = 3 + (c.num_prefix_tokens > 0 ? 1 : 0) +
                  static_cast<size_t>(c.num_layers) * (16 + (c.use_layerscale ? 2 : 0) + (c.film_dim > 0 ? 4 : 0));
    *out = h;
    return 0;
}

extern "C" int blurr_vit_set_weight(blurr_vit_t* h, const char* key_c, const void* dev_ptr, const int64_t* shape, int ndim) {
    if (!h || !key_c || !dev_ptr || !shape) return fail(BLURR_ERR_INVALID, "blurr_vit_set_weight: null argument");
    VIT_CUDA_TRY(cudaSetDevice(h->device));
    const auto& c = h->cfg;
    const int H = c.hidden;
    const std::string key(key_c);
    const bf16* src = static_cast<const bf16*>(dev_ptr);
    auto is2 = [&](int64_t r, int64_t k) { return ndim == 2 && shape[0] == r && shape[1] == k; };
    auto is1 = [&](int64_t n) { return ndim == 1 && shape[0] == n; };
    auto bad = [&]() { return fail(BLURR_ERR_INVALID, "unexpected shape for " + key); };
    auto copy = [&](bf16* dst, size_t n) -> int {
        VIT_CUDA_TRY(cudaMemcpy(dst, src, n * 2, cudaMemcpyDeviceToDevice));
        return 0;
    };
    auto mat = [&](VLin& L, int row_off, int rows) -> int {
        if (!is2(rows, L.Kreal)) return bad();
        return pack_weight(src, rows, L.Kreal, L, row_off);
    };
    int rc = 0;
    if (key == "patch.weight") rc = mat(h->patch, 0, H);
    else if (key == "patch.bias") { if (!is1(H)) return bad(); rc = copy(h->patch.bias, H); }
    else if (key == "pos") { if (!is2(h->n_patches, H)) return bad(); rc = copy(h->pos, static_cast<size_t>(h->n_patches) * H); }
    else if (key == "prefix") { if (!is2(c.num_prefix_tokens, H)) return bad(); rc = copy(h->prefix, static_cast<size_t>(c.num_prefix_tokens) * H); }
    else if (key.rfind("layers.", 0) == 0) {
        const size_t dot = key.find('.', 7);
        if (dot == std::string::npos) return fail(BLURR_ERR_INVALID, "unknown key " + key);
        const int l = atoi(key.substr(7, dot - 7).c_str());
        if (l < 0 || l >= c.num_layers) return fail(BLURR_ERR_INVALID, "layer index out of range in " + key);
        VLayer& L = h->layers[l];
        const std::string rest = key.substr(dot + 1);
        auto vec = [&](bf16* dst, int n) -> int { if (!is1(n)) return bad(); return copy(dst, n); };
        if (rest == "ln1.weight") rc = vec(L.ln1w, H);
        else if (rest == "ln1.bias") rc = vec(L.ln1b, H);
        else if (rest == "ln2.weight") rc = vec(L.ln2w, H);
        else if (rest == "ln2.bias") rc = vec(L.ln2b, H);
        else if (rest == "ls1") rc = vec(L.ls1, H);
        else if (rest == "ls2") rc = vec(L.ls2, H);
        else if (rest == "q.weight") rc = mat(L.qkv, 0, H);
        else if (rest == "k.weight") rc = mat(L.qkv, H, H);
        else if (rest == "v.weight") rc = mat(L.qkv, 2 * H, H);
        else if (rest == "q.bias") rc = vec(L.qkv.bias, H);
        else if (rest == "k.bias") rc = vec(L.qkv.bias + H, H);
        else if (rest == "v.bias") rc = vec(L.qkv.bias + 2 * H, H);
        else if (rest == "o.weight") rc = mat(L.o, 0, H);
        else if (rest == "o.bias") rc = vec(L.o.bias, H);
        else if (rest == "fc1.weight") rc = mat(L.fc1, 0, c.mlp_dim);
        else if (rest == "fc1.bias") rc = vec(L.fc1.bias, c.mlp_dim);
        else if (rest == "fc2.weight") {
            if (!is2(H, c.mlp_dim)) return bad();
            rc = pack_weight(src, H, c.mlp_dim, L.fc2, 0);          // K padded to fc1.Nw: the pad columns stay zero
        }
        else if (rest == "fc2.bias") rc = vec(L.fc2.bias, H);
        else if (c.film_dim > 0 && (rest == "film_scale.weight" || rest == "film_shift.weight"))
            rc = mat(h->film, (2 * l + (rest == "film_shift.weight" ? 1 : 0)) * H, H);
        else if (c.film_dim > 0 && (rest == "film_scale.bias" || rest == "film_shift.bias"))
            rc = vec(h->film.bias + static_cast<size_t>(2 * l + (rest == "film_shift.bias" ? 1 : 0)) * H, H);
        else return fail(BLURR_ERR_INVALID, "unknown key " + key);
    } else {
        return fail(BLURR_ERR_INVALID, "unknown key " + key);
    }
    if (rc) return rc;
    h->seen.insert(key);
    h->finalized = false;
    return 0;
}

extern "C" int blurr_vit_finalize(blurr_vit_t* h) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_vit_finalize: null handle");
    if (h->seen.size() != h->expected)
        return fail(BLURR_ERR_STATE, "blurr_vit_finalize: " + std::to_string(static_cast<long long>(h->expected) - static_cast<long long>(h->seen.size())) + " keys missing");
    VIT_CUDA_TRY(cudaSetDevice(h->device));
    VIT_CUDA_TRY(cudaDeviceSynchronize());
    h->finalized = true;
    return 0;
}

// patch GEMM .. last block, on the handle's own buffers (graph-capturable); FiLM handles: image i uses condition row
// i / images_per_cond of h->cond
static void vit_body(blurr_vit* h, Launcher& R, int batch, int images_per_cond) {
    const auto& c = h->cfg;
    cudaStream_t st = R.st;
    const int H = c.hidden, P = c.num_prefix_tokens, S = h->seq, NP = h->n_patches;
    const int T = batch * S, Tp = batch * NP;
    const int gelu = c.gelu_erf ? GELU_ERF : GELU_TANH;
    // every block's gamma | beta of every condition row at once: bf16(cond W^T + b), as nn.Linear
    if (c.film_dim > 0) R.gemm(h->film, h->cond, batch / images_per_cond, EPI_STORE, h->film_out, h->film.Nw, 0);
    {   // patch embedding + position embeddings -> the patch rows of X (behind each sample's prefix rows)
        ConsumerArgs a{};
        a.add_mode = ADD_POSEMB; a.pos = h->pos; a.pos_rows = NP;
        a.x_out = h->X; a.ldx = H; a.norm_mode = NORM_NONE;
        if (P > 0) { a.row_group = NP; a.row_extra = P; a.row_offset = P; }
        R.linear_consumer(h->patch, h->patches, Tp, a);
    }
    for (int b = 0; b < batch && P > 0 && !R.rc; ++b)
        if (cudaMemcpyAsync(h->X + static_cast<size_t>(b) * S * H, h->prefix, static_cast<size_t>(P) * H * 2, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            R.rc = fail(BLURR_ERR_CUDA, "prefix token copy failed");
    {   // LN1 of block 0 over every row
        ConsumerArgs a{};
        a.T = T; a.N = H; a.splitk = 1; a.add_mode = ADD_NONE; a.res = h->X; a.ldr = H; a.out_scale = 1.0f;
        a.norm_mode = NORM_LAYERNORM; a.norm_w = h->layers[0].ln1w; a.norm_b = h->layers[0].ln1b; a.eps = c.ln_eps;
        a.xn_out = h->XN; a.ldn = H;
        if (!R.rc) R.launched(launch_consumer(st, a), "consumer");
    }
    for (int l = 0; l < c.num_layers; ++l) {
        VLayer& L = h->layers[l];
        R.gemm(L.qkv, h->XN, T, EPI_STORE, h->QKV, 3 * H, 0);
        if (!R.rc) R.launched(launch_siglip_attention(st, h->QKV, 3 * H, batch, S, c.num_heads, H, h->AO, H, nullptr), "attention");
        {
            ConsumerArgs a{};
            a.add_mode = ADD_RESIDUAL; a.res = h->X; a.ldr = H; a.x_out = h->X; a.ldx = H;
            a.col_scale = c.use_layerscale ? L.ls1 : nullptr;
            a.norm_mode = NORM_LAYERNORM; a.norm_w = L.ln2w; a.norm_b = L.ln2b; a.eps = c.ln_eps; a.xn_out = h->XN; a.ldn = H;
            if (c.film_dim > 0) {       // x = x * (1 + gamma) + beta between the attention and the MLP residual
                a.film_gamma = h->film_out + static_cast<size_t>(2 * l) * H;
                a.film_beta = a.film_gamma + H;
                a.film_ld = h->film.Nw; a.film_rows = images_per_cond * S;
            }
            R.linear_consumer(L.o, h->AO, T, a);
        }
        R.gemm(L.fc1, h->XN, T, EPI_GELU, h->HM, L.fc1.Nw, gelu);
        {
            ConsumerArgs a{};
            a.add_mode = ADD_RESIDUAL; a.res = h->X; a.ldr = H; a.x_out = h->X; a.ldx = H;
            a.col_scale = c.use_layerscale ? L.ls2 : nullptr;
            const bool last = l + 1 == c.num_layers;
            a.norm_mode = last ? NORM_NONE : NORM_LAYERNORM;
            if (!last) { a.norm_w = h->layers[l + 1].ln1w; a.norm_b = h->layers[l + 1].ln1b; a.xn_out = h->XN; a.ldn = H; }
            a.eps = c.ln_eps;
            R.linear_consumer(L.fc2, h->HM, T, a);
        }
    }
}

// images_per_cond: 0 on handles without FiLM; cond is then unused
static int vit_forward(blurr_vit* h, void* cuda_stream, int batch, const void* pixel_values, const int64_t strides[4],
                       const void* cond, int cond_ld, int images_per_cond, void* out, int out_ld, const std::string& who) {
    if (!h || !pixel_values || !strides || !out) return fail(BLURR_ERR_INVALID, who + ": null argument");
    if (!h->finalized) return fail(BLURR_ERR_STATE, who + ": call blurr_vit_finalize first");
    if (batch < 1 || batch > h->max_batch) return fail(BLURR_ERR_INVALID, who + ": batch out of range");
    const auto& c = h->cfg;
    const int H = c.hidden, P = c.num_prefix_tokens, S = h->seq, NP = h->n_patches;
    if (out_ld < H || (out_ld & 7)) return fail(BLURR_ERR_INVALID, who + ": out_ld must be >= hidden and a multiple of 8");
    VIT_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    h->launches = 0;
    Launcher R{st, h->ws, h->ws_floats, h->LINB, &h->launches};
    if (images_per_cond > 0)        // the graph reads the handle's copy: one graph serves every condition
        VIT_CUDA_TRY(cudaMemcpy2DAsync(h->cond, static_cast<size_t>(c.film_dim) * 2, cond, static_cast<size_t>(cond_ld) * 2,
                                       static_cast<size_t>(c.film_dim) * 2, batch / images_per_cond, cudaMemcpyDeviceToDevice, st));
    R.launched(launch_im2col(st, static_cast<const bf16*>(pixel_values), strides[0], strides[1], strides[2], strides[3], batch,
                             h->patches, h->patch.K), "im2col");
    if (R.rc) return R.rc;
    if (!h->use_graph) {
        vit_body(h, R, batch, images_per_cond);
    } else {
        const std::pair<int, int> key(batch, images_per_cond);
        auto it = h->graphs.find(key);
        if (it == h->graphs.end()) {
            vit_body(h, R, batch, images_per_cond);                                   // warm run: attribute setup, tensor maps
            if (R.rc) return R.rc;
            VIT_CUDA_TRY(cudaStreamSynchronize(st));
            int64_t captured = 0;
            cudaStream_t cs;
            VIT_CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            Launcher C{cs, h->ws, h->ws_floats, h->LINB, &captured};
            cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
            if (e != cudaSuccess) { cudaStreamDestroy(cs); return fail(BLURR_ERR_CUDA, "graph capture begin failed"); }
            vit_body(h, C, batch, images_per_cond);
            cudaGraph_t g = nullptr;
            e = cudaStreamEndCapture(cs, &g);
            cudaStreamDestroy(cs);
            if (C.rc) { if (g) cudaGraphDestroy(g); return C.rc; }
            if (e != cudaSuccess || !g) return fail(BLURR_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(e));
            cudaGraphExec_t ex = nullptr;
            e = cudaGraphInstantiate(&ex, g, 0);
            if (e != cudaSuccess) { cudaGraphDestroy(g); return fail(BLURR_ERR_CUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(e)); }
            it = h->graphs.emplace(key, blurr_vit::GraphEntry{g, ex, captured}).first;
            h->launches = 1;                                         // the im2col of this call; the replay below adds the rest
        }
        VIT_CUDA_TRY(cudaGraphLaunch(it->second.exec, st));
        h->launches = 1 + it->second.launches;
    }
    if (!R.rc) R.launched(launch_copy_rows(st, h->X, batch, S, P, NP, H, H, static_cast<bf16*>(out), out_ld), "copy_rows");
    return R.rc;
}

extern "C" int blurr_vit_forward(blurr_vit_t* h, void* cuda_stream, int batch, const void* pixel_values, const int64_t strides[4],
                                 void* out, int out_ld) {
    if (h && h->cfg.film_dim > 0) return fail(BLURR_ERR_STATE, "blurr_vit_forward: a FiLM handle needs blurr_vit_forward_film");
    return vit_forward(h, cuda_stream, batch, pixel_values, strides, nullptr, 0, 0, out, out_ld, "blurr_vit_forward");
}

extern "C" int blurr_vit_forward_film(blurr_vit_t* h, void* cuda_stream, int batch, const void* pixel_values, const int64_t strides[4],
                                      const void* cond, int cond_ld, int images_per_cond, void* out, int out_ld) {
    if (!h) return fail(BLURR_ERR_INVALID, "blurr_vit_forward_film: null handle");
    if (h->cfg.film_dim == 0) return fail(BLURR_ERR_STATE, "blurr_vit_forward_film: the handle was created without FiLM (film_dim 0)");
    if (!cond) return fail(BLURR_ERR_INVALID, "blurr_vit_forward_film: null cond");
    if (cond_ld < h->cfg.film_dim) return fail(BLURR_ERR_INVALID, "blurr_vit_forward_film: cond_ld smaller than film_dim");
    if (images_per_cond < 1 || batch % images_per_cond)
        return fail(BLURR_ERR_INVALID, "blurr_vit_forward_film: images_per_cond must be >= 1 and divide batch");
    return vit_forward(h, cuda_stream, batch, pixel_values, strides, cond, cond_ld, images_per_cond, out, out_ld,
                       "blurr_vit_forward_film");
}

extern "C" int blurr_vit_set_option(blurr_vit_t* h, const char* name, int64_t value) {
    if (!h || !name) return fail(BLURR_ERR_INVALID, "blurr_vit_set_option: null argument");
    if (std::string(name) == "use_cuda_graph") h->use_graph = value != 0;
    else return fail(BLURR_ERR_INVALID, std::string("blurr_vit_set_option: unknown option ") + name);
    return 0;
}

extern "C" int64_t blurr_vit_last_launch_count(const blurr_vit_t* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------
// MLP projector
// ---------------------------------------------------------------------------
struct blurr_mlp {
    int device = 0, max_rows = 0;
    std::vector<void*> allocs;
    std::vector<VLin> layers;
    std::vector<bool> set;
    bf16 *A = nullptr, *B = nullptr;
    int widest = 0;
    int64_t launches = 0;
};

extern "C" void blurr_mlp_destroy(blurr_mlp_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (void* p : h->allocs) cudaFree(p);
    gemm_forget_tensor_maps();
    delete h;
}

extern "C" int blurr_mlp_create(const int32_t* dims, int n_layers, int device, int max_rows, blurr_mlp_t** out) {
    if (!dims || !out || n_layers < 1 || n_layers > 8 || max_rows < 1) return fail(BLURR_ERR_INVALID, "blurr_mlp_create: bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(BLURR_ERR_CUDA, "no CUDA device: the B200 path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BLURR_ERR_INVALID, "bad device index");
    VIT_CUDA_TRY(cudaSetDevice(device));
    auto* h = new blurr_mlp();
    h->device = device; h->max_rows = max_rows;
    h->layers.resize(n_layers);
    h->set.assign(n_layers, false);
    bool ok = true;
    int k_in = dims[0];
    for (int i = 0; i < n_layers; ++i) {
        if (dims[i + 1] < 1 || k_in < 1) { ok = false; break; }
        ok &= alloc_lin(h, h->layers[i], dims[i + 1], k_in);
        h->layers[i].Kreal = dims[i];           // columns of the caller's weight; K itself is the padded input width
        if (h->layers[i].Nw > h->widest) h->widest = h->layers[i].Nw;
        k_in = h->layers[i].Nw;                 // the next layer reads the padded output (pad columns are zero)
    }
    if (dims[0] % 64) ok = false;               // the caller's input rows are read as they are
    h->A = static_cast<bf16*>(dalloc_in(h, static_cast<size_t>(max_rows) * h->widest * 2));
    h->B = static_cast<bf16*>(dalloc_in(h, static_cast<size_t>(max_rows) * h->widest * 2));
    if (!ok || !h->A || !h->B) { blurr_mlp_destroy(h); return fail(BLURR_ERR_INVALID, "blurr_mlp_create: bad widths (dims[0] must be a multiple of 64) or allocation failure"); }
    *out = h;
    return 0;
}

extern "C" int blurr_mlp_set_weight(blurr_mlp_t* h, int layer, const void* weight_dev, const void* bias_dev) {
    if (!h || !weight_dev || layer < 0 || layer >= static_cast<int>(h->layers.size())) return fail(BLURR_ERR_INVALID, "blurr_mlp_set_weight: bad arguments");
    VIT_CUDA_TRY(cudaSetDevice(h->device));
    VLin& L = h->layers[layer];
    const int rc = pack_weight(static_cast<const bf16*>(weight_dev), L.N, L.Kreal, L, 0);
    if (rc) return rc;
    if (bias_dev) VIT_CUDA_TRY(cudaMemcpy(L.bias, bias_dev, static_cast<size_t>(L.N) * 2, cudaMemcpyDeviceToDevice));
    VIT_CUDA_TRY(cudaDeviceSynchronize());
    h->set[layer] = true;
    return 0;
}

extern "C" int blurr_mlp_forward(blurr_mlp_t* h, void* cuda_stream, int rows, const void* x, int ldx, void* y, int ldy) {
    if (!h || !x || !y || rows < 1 || rows > h->max_rows) return fail(BLURR_ERR_INVALID, "blurr_mlp_forward: bad arguments");
    for (bool s : h->set) if (!s) return fail(BLURR_ERR_STATE, "blurr_mlp_forward: a layer has no weights");
    if (ldx != h->layers[0].K) return fail(BLURR_ERR_INVALID, "blurr_mlp_forward: ldx must equal the input width");
    const int n = static_cast<int>(h->layers.size());
    if (ldy < h->layers[n - 1].N) return fail(BLURR_ERR_INVALID, "blurr_mlp_forward: ldy smaller than the output width");
    VIT_CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    h->launches = 0;
    Launcher R{st, nullptr, 0, nullptr, &h->launches};
    const bf16* in = static_cast<const bf16*>(x);
    for (int i = 0; i < n; ++i) {
        const bool last = i + 1 == n;
        bf16* outp = (i & 1) ? h->B : h->A;
        R.gemm(h->layers[i], in, rows, last ? EPI_STORE : EPI_GELU, outp, h->layers[i].Nw, GELU_ERF);
        in = outp;
    }
    if (!R.rc) R.launched(launch_copy_rows(st, in, 1, rows, 0, rows, h->layers[n - 1].N, h->layers[n - 1].Nw, static_cast<bf16*>(y), ldy), "copy_rows");
    return R.rc;
}
