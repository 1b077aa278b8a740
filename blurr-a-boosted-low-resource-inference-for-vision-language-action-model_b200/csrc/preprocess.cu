// Device-side observation preprocessing (SURVEY.md 8(f) row 1): the per-control-step host work the
// reference does between the simulator and the model, moved onto the GPU with bit-identical results.
//
//  * frame:   uint8 HWC camera frame -> cv2.resize(INTER_LANCZOS4) to the model resolution
//             (env_adapter/simpler.py:59-64) -> VLAProcessor rescale / normalise in fp32
//             (model/vla/processing.py:27-58,112-117) -> `.to(bfloat16)` (agent/eval.py:187), written
//             as the contiguous [3][h][w] pixel_values tensor the engine's patch loader reads.
//             The resize is OpenCV's 8-tap fixed-point Lanczos (modules/imgproc/src/resize.cpp:
//             interpolateLanczos4, INTER_RESIZE_COEF_BITS = 11, HResizeLanczos4 / VResizeLanczos4 with
//             FixedPtCast<int, uchar, 22>, replicated borders); the tables are built on the host at
//             create time with the same float / double operation order, the two integer passes run in
//             one kernel (one CTA per output row, the 8 source rows staged in shared memory).
//  * proprio: normalize_bound / normalize_gaussian in float64 (env_adapter/base.py:8-18,33-40),
//             float32 (simpler.py:93-95), then bfloat16 (eval.py:194).
//  * OpenVLA frame: uint8 HWC camera frame -> Pillow `Image.resize(BICUBIC)` (what torchvision's resize does to a
//             PIL image) -> center crop -> per-tower fp32 `to_tensor` / `normalize` -> bf16, written as the
//             [3 * n_norms][crop_h][crop_w] pixel_values of the fused DINOv2 + SigLIP backbone.  The resize is
//             Pillow's fixed-point resample (libImaging/Resample.c: precompute_coeffs in double,
//             normalize_coeffs_8bpc with PRECISION_BITS = 22, a horizontal then a vertical pass, each only when
//             its dimension changes, each rounding to uint8); only the cropped window is computed.
// All three kernels are pure bandwidth/latency work (a 640x480 frame is 0.9 MB): no tensor cores.
#include "blurr_pi0.h"
#include "blurr_vit.h"
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

namespace blurr {
int record_error(int code, const std::string& msg);      // engine.cu: sets blurr_last_error()
inline int fail(int code, const std::string& msg) { return record_error(code, msg); }
}
using blurr::bf16;

struct blurr_preproc {
    int device = 0;
    int src_h = 0, src_w = 0, dst_h = 0, dst_w = 0;
    int32_t *x_ofs = nullptr, *y_ofs = nullptr;      // device
    int16_t *x_alpha = nullptr, *y_alpha = nullptr;  // device, [dst][8]
    std::vector<int32_t> hx_ofs, hy_ofs;
    std::vector<int16_t> hx_alpha, hy_alpha;
};

namespace {

constexpr int kTaps = 8;
constexpr int kCoefBits = 11;

// resize.cpp interpolateLanczos4(float x, float* coeffs), operation for operation
void lanczos4_coeffs(float x, float* coeffs) {
    static const double s45 = 0.70710678118654752440084436210485;
    static const double cs[][2] = {{1, 0}, {-s45, -s45}, {0, 1}, {s45, -s45}, {-1, 0}, {s45, s45}, {0, -1}, {-s45, s45}};
    const double pi = 3.1415926535897932384626433832795;
    float sum = 0;
    const float x3 = x + 3;
    const double y0 = -static_cast<double>(x3) * pi * 0.25, s0 = std::sin(y0), c0 = std::cos(y0);
    for (int i = 0; i < kTaps; ++i) {
        const float y0_ = x3 - static_cast<float>(i);
        if (std::fabs(y0_) >= 1e-6f) {
            const double y = -static_cast<double>(y0_) * pi * 0.25;
            coeffs[i] = static_cast<float>((cs[i][0] * s0 + cs[i][1] * c0) / (y * y));
        } else {
            coeffs[i] = 1e30f;
        }
        sum += coeffs[i];
    }
    sum = 1.f / sum;
    for (int i = 0; i < kTaps; ++i) coeffs[i] *= sum;
}

void build_tables(int src, int dst, std::vector<int32_t>* ofs, std::vector<int16_t>* alpha) {
    const double inv_scale = static_cast<double>(dst) / src;
    const double scale = 1. / inv_scale;
    ofs->resize(dst);
    alpha->resize(static_cast<size_t>(dst) * kTaps);
    for (int d = 0; d < dst; ++d) {
        float f = static_cast<float>((d + 0.5) * scale - 0.5);
        const int s = static_cast<int>(std::floor(f));
        f -= static_cast<float>(s);
        float c[kTaps];
        lanczos4_coeffs(f, c);
        for (int k = 0; k < kTaps; ++k) {
            long v = std::lrintf(c[k] * static_cast<float>(1 << kCoefBits));     // saturate_cast<short>(float)
            v = v < -32768 ? -32768 : (v > 32767 ? 32767 : v);
            (*alpha)[static_cast<size_t>(d) * kTaps + k] = static_cast<int16_t>(v);
        }
        (*ofs)[d] = s;
    }
}

struct FrameArgs {
    const uint8_t* frame; long long row_stride, frame_stride;
    int src_h, src_w, dst_h, dst_w;
    const int32_t *x_ofs, *y_ofs;
    const int16_t *x_alpha, *y_alpha;
    bf16* pixel_values;       // [batch][3][dst_h][dst_w]
    uint8_t* resized;         // [batch][dst_h][dst_w][3] or nullptr
};

__global__ void __launch_bounds__(256) resize_lanczos4_normalize_kernel(const FrameArgs a) {
    extern __shared__ __align__(16) uint8_t rows[];          // [8][src_w * 3]
    const int dy = blockIdx.x, b = blockIdx.y;
    const int row_bytes = a.src_w * 3;
    const uint8_t* src = a.frame + static_cast<size_t>(b) * a.frame_stride;
    const int sy0 = a.y_ofs[dy] - (kTaps / 2 - 1);
    for (int k = 0; k < kTaps; ++k) {
        int sy = sy0 + k;
        sy = sy < 0 ? 0 : (sy >= a.src_h ? a.src_h - 1 : sy);            // replicated border
        const uint8_t* g = src + static_cast<size_t>(sy) * a.row_stride;
        uint8_t* s = rows + k * row_bytes;
        if (((reinterpret_cast<uintptr_t>(g) | static_cast<uintptr_t>(row_bytes) | reinterpret_cast<uintptr_t>(s)) & 3) == 0) {
            for (int i = threadIdx.x; i < row_bytes / 4; i += blockDim.x)
                reinterpret_cast<uint32_t*>(s)[i] = __ldg(reinterpret_cast<const uint32_t*>(g) + i);
        } else {
            for (int i = threadIdx.x; i < row_bytes; i += blockDim.x) s[i] = __ldg(g + i);
        }
    }
    __syncthreads();
    int beta[kTaps];
#pragma unroll
    for (int k = 0; k < kTaps; ++k) beta[k] = a.y_alpha[dy * kTaps + k];
    for (int dx = threadIdx.x; dx < a.dst_w; dx += blockDim.x) {
        int xi[kTaps], al[kTaps];
        const int sx0 = a.x_ofs[dx] - (kTaps / 2 - 1);
#pragma unroll
        for (int j = 0; j < kTaps; ++j) {
            int sx = sx0 + j;
            sx = sx < 0 ? 0 : (sx >= a.src_w ? a.src_w - 1 : sx);
            xi[j] = sx * 3;
            al[j] = a.x_alpha[dx * kTaps + j];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            int v = 0;                                   // cv2 accumulates both passes in int (WT = int)
#pragma unroll
            for (int k = 0; k < kTaps; ++k) {
                const uint8_t* r = rows + k * row_bytes + c;
                int h = 0;
#pragma unroll
                for (int j = 0; j < kTaps; ++j) h += static_cast<int>(r[xi[j]]) * al[j];
                v += h * beta[k];
            }
            v = (v + (1 << (2 * kCoefBits - 1))) >> (2 * kCoefBits);      // FixedPtCast<int, uchar, 22>
            v = v < 0 ? 0 : (v > 255 ? 255 : v);
            if (a.resized != nullptr)
                a.resized[((static_cast<size_t>(b) * a.dst_h + dy) * a.dst_w + dx) * 3 + c] = static_cast<uint8_t>(v);
            // processing.py: image * (1/255.0) -> (x - 0.5) / 0.5 in fp32 (one rounding per op), then bf16
            float f = __fmul_rn(static_cast<float>(v), static_cast<float>(1 / 255.0));
            f = __fdiv_rn(__fsub_rn(f, 0.5f), 0.5f);
            a.pixel_values[((static_cast<size_t>(b) * 3 + c) * a.dst_h + dy) * a.dst_w + dx] = __float2bfloat16_rn(f);
        }
    }
}

__global__ void normalize_proprio_kernel(const double* raw, const double* lo, const double* hi, int kind, int n,
                                         int dim, bf16* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * dim) return;
    const int d = i % dim;
    const double x = raw[i];
    double y;
    if (kind == 0) {
        // 2 * (data - min) / (max - min + eps) - 1, then clip to [-1, 1]  (base.py:17-18)
        const double num = __dmul_rn(2.0, __dsub_rn(x, lo[d]));
        const double den = __dadd_rn(__dsub_rn(hi[d], lo[d]), 1e-8);
        y = __dsub_rn(__ddiv_rn(num, den), 1.0);
        y = y < -1.0 ? -1.0 : (y > 1.0 ? 1.0 : y);
    } else {
        // (data - mean) / (std + eps)  (base.py:40)
        y = __ddiv_rn(__dsub_rn(x, lo[d]), __dadd_rn(hi[d], 1e-8));
    }
    out[i] = __float2bfloat16_rn(static_cast<float>(y));      // float64 -> float32 -> bf16, as the reference
}

// ------------------------------------------------------------------------------------------------------------------
// OpenVLA: Pillow bicubic resize + center crop + per-tower normalisation
// ------------------------------------------------------------------------------------------------------------------
constexpr int kPrecisionBits = 22;                 // Resample.c PRECISION_BITS
constexpr int kVlaMaxSize = 1 << 15;               // any side of the source or the resize
constexpr int kVlaMaxNorms = 2;
constexpr int kVlaBandRows = 8;                    // output rows per CTA (fewer when the staged rows would not fit)
constexpr int kVlaMaxSmem = 200 * 1024;
constexpr int kVlaThreads = 256;

// Resample.c bicubic_filter, a = -0.5
double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// Resample.c precompute_coeffs (box = the whole axis) + normalize_coeffs_8bpc, operation for operation in double.
// bounds: [out][2] = (first source index, tap count); weights: [out][ksize], zero past the tap count.  Returns ksize.
int pillow_bicubic_coeffs(int in_size, int out_size, std::vector<int32_t>* bounds, std::vector<int32_t>* weights) {
    const double scale = static_cast<double>(in_size) / out_size;
    const double filterscale = scale < 1.0 ? 1.0 : scale;
    const double support = 2.0 * filterscale;
    const int ksize = static_cast<int>(std::ceil(support)) * 2 + 1;
    bounds->assign(static_cast<size_t>(out_size) * 2, 0);
    weights->assign(static_cast<size_t>(out_size) * ksize, 0);
    std::vector<double> k(ksize);
    for (int xx = 0; xx < out_size; ++xx) {
        const double center = (xx + 0.5) * scale;
        const double ss = 1.0 / filterscale;
        int xmin = static_cast<int>(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = static_cast<int>(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        double ww = 0.0;
        for (int x = 0; x < xmax; ++x) {
            const double w = bicubic_filter((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; ++x) {
            if (ww != 0.0) k[x] /= ww;
            (*weights)[static_cast<size_t>(xx) * ksize + x] = k[x] < 0 ? static_cast<int32_t>(-0.5 + k[x] * (1 << kPrecisionBits))
                                                                       : static_cast<int32_t>(0.5 + k[x] * (1 << kPrecisionBits));
        }
        (*bounds)[2 * xx] = xmin;
        (*bounds)[2 * xx + 1] = xmax;
    }
    return ksize;
}

// The kernel's table for one axis: Pillow's coefficients for output indices [first, first + count) of an `in -> out`
// resize, or, when in == out (Pillow skips that pass), the identity: one tap of weight 1.0, which reproduces the
// source byte exactly ((v << 22) + (1 << 21)) >> 22 = v.
int axis_table(int in_size, int out_size, int first, int count, std::vector<int32_t>* bounds, std::vector<int32_t>* weights) {
    if (in_size == out_size) {
        bounds->resize(static_cast<size_t>(count) * 2);
        weights->assign(count, 1 << kPrecisionBits);
        for (int i = 0; i < count; ++i) { (*bounds)[2 * i] = first + i; (*bounds)[2 * i + 1] = 1; }
        return 1;
    }
    std::vector<int32_t> b, w;
    const int ksize = pillow_bicubic_coeffs(in_size, out_size, &b, &w);
    bounds->assign(b.begin() + 2 * static_cast<size_t>(first), b.begin() + 2 * static_cast<size_t>(first + count));
    weights->assign(w.begin() + static_cast<size_t>(first) * ksize, w.begin() + static_cast<size_t>(first + count) * ksize);
    return ksize;
}

struct VlaArgs {
    const uint8_t* frame; long long row_stride, frame_stride;
    int crop_h, crop_w, kx, ky, band_rows, n_norms;
    const int32_t *x_bounds, *x_weights, *y_bounds, *y_weights;    // crop-window slices of the two axis tables
    float mean[3 * kVlaMaxNorms], stdev[3 * kVlaMaxNorms];
    bf16* pixel_values;        // [batch][3 * n_norms][crop_h][crop_w]
    uint8_t* resized;          // [batch][crop_h][crop_w][3] or nullptr
};

__device__ __forceinline__ int clip8(int acc) {
    acc >>= kPrecisionBits;
    return acc < 0 ? 0 : (acc > 255 ? 255 : acc);
}

// One CTA = one band of output rows of one frame.  The horizontal pass runs over the source rows the band's vertical
// windows cover, for the crop's columns only, into shared memory as uint8 (Pillow rounds between the passes); the
// vertical pass then reads those rows.  Pillow accumulates in int32 from 1 << 21; the sums stay below 2^31 (255 times
// the absolute weight sum, at most ~1.2 * 2^22).
__global__ void __launch_bounds__(kVlaThreads) resize_bicubic_crop_normalize_kernel(const VlaArgs a) {
    extern __shared__ __align__(16) uint8_t hrows[];      // [span][crop_w * 3]
    const int b = blockIdx.y;
    const int r0 = blockIdx.x * a.band_rows;
    const int r1 = min(r0 + a.band_rows, a.crop_h);
    const int y0 = __ldg(a.y_bounds + 2 * r0);
    const int span = __ldg(a.y_bounds + 2 * (r1 - 1)) + __ldg(a.y_bounds + 2 * (r1 - 1) + 1) - y0;   // windows are monotonic
    const int row_bytes = a.crop_w * 3;
    const uint8_t* src = a.frame + static_cast<long long>(b) * a.frame_stride;
    for (int i = threadIdx.x; i < span * a.crop_w; i += blockDim.x) {
        const int j = i / a.crop_w, c = i - j * a.crop_w;
        const int xmin = __ldg(a.x_bounds + 2 * c), n = __ldg(a.x_bounds + 2 * c + 1);
        const int32_t* w = a.x_weights + static_cast<size_t>(c) * a.kx;
        const uint8_t* p = src + static_cast<long long>(y0 + j) * a.row_stride + xmin * 3;
        int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
        for (int k = 0; k < n; ++k) {
            const int wk = __ldg(w + k);
            s0 += static_cast<int>(__ldg(p + 3 * k)) * wk;
            s1 += static_cast<int>(__ldg(p + 3 * k + 1)) * wk;
            s2 += static_cast<int>(__ldg(p + 3 * k + 2)) * wk;
        }
        uint8_t* d = hrows + j * row_bytes + c * 3;
        d[0] = static_cast<uint8_t>(clip8(s0));
        d[1] = static_cast<uint8_t>(clip8(s1));
        d[2] = static_cast<uint8_t>(clip8(s2));
    }
    __syncthreads();
    const size_t plane = static_cast<size_t>(a.crop_h) * a.crop_w;
    for (int i = threadIdx.x; i < (r1 - r0) * a.crop_w; i += blockDim.x) {
        const int r = r0 + i / a.crop_w, c = i % a.crop_w;
        const int ymin = __ldg(a.y_bounds + 2 * r) - y0, n = __ldg(a.y_bounds + 2 * r + 1);
        const int32_t* w = a.y_weights + static_cast<size_t>(r) * a.ky;
        const uint8_t* p = hrows + ymin * row_bytes + c * 3;
        int s0 = 1 << (kPrecisionBits - 1), s1 = s0, s2 = s0;
        for (int k = 0; k < n; ++k) {
            const int wk = __ldg(w + k);
            s0 += static_cast<int>(p[k * row_bytes]) * wk;
            s1 += static_cast<int>(p[k * row_bytes + 1]) * wk;
            s2 += static_cast<int>(p[k * row_bytes + 2]) * wk;
        }
        const int v[3] = {clip8(s0), clip8(s1), clip8(s2)};
        if (a.resized != nullptr) {
            uint8_t* d = a.resized + ((static_cast<size_t>(b) * a.crop_h + r) * a.crop_w + c) * 3;
            d[0] = static_cast<uint8_t>(v[0]); d[1] = static_cast<uint8_t>(v[1]); d[2] = static_cast<uint8_t>(v[2]);
        }
        // TVF.to_tensor: fp32 v / 255 (a true division); TVF.normalize: (x - mean) / std in fp32; then .to(bfloat16)
        float f[3];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) f[ch] = __fdiv_rn(static_cast<float>(v[ch]), 255.0f);
        bf16* out = a.pixel_values + static_cast<size_t>(b) * 3 * a.n_norms * plane + static_cast<size_t>(r) * a.crop_w + c;
#pragma unroll
        for (int m = 0; m < kVlaMaxNorms; ++m) {
            if (m >= a.n_norms) break;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch)
                out[(3 * m + ch) * plane] = __float2bfloat16_rn(__fdiv_rn(__fsub_rn(f[ch], a.mean[3 * m + ch]), a.stdev[3 * m + ch]));
        }
    }
}

}  // namespace

struct blurr_vla_preproc {
    int device = 0;
    int src_h = 0, src_w = 0, crop_h = 0, crop_w = 0, n_norms = 0;
    int kx = 0, ky = 0, band_rows = 0, smem = 0;
    int32_t* tables = nullptr;                        // device: x_bounds | x_weights | y_bounds | y_weights
    size_t x_weights_at = 0, y_bounds_at = 0, y_weights_at = 0;
    float mean[3 * kVlaMaxNorms] = {}, stdev[3 * kVlaMaxNorms] = {};
};

extern "C" int blurr_preproc_create(int device, int src_h, int src_w, int dst_h, int dst_w, blurr_preproc_t** out) {
    if (!out) return blurr::fail(BLURR_ERR_INVALID, "preproc_create: null out");
    *out = nullptr;
    if (src_h < 1 || src_w < 1 || dst_h < 1 || dst_w < 1)
        return blurr::fail(BLURR_ERR_INVALID, "preproc_create: sizes must be positive");
    if (static_cast<long long>(src_w) * 3 * kTaps > 200 * 1024)
        return blurr::fail(BLURR_ERR_INVALID, "preproc_create: source rows too wide for the shared-memory stage");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0)
        return blurr::fail(BLURR_ERR_CUDA, "no CUDA device: the preprocessing path has no CPU fallback");
    if (device < 0 || device >= n_dev) return blurr::fail(BLURR_ERR_INVALID, "preproc_create: bad device index");
    if (cudaSetDevice(device) != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, "cudaSetDevice failed");
    blurr_preproc* p = new blurr_preproc();
    p->device = device; p->src_h = src_h; p->src_w = src_w; p->dst_h = dst_h; p->dst_w = dst_w;
    build_tables(src_w, dst_w, &p->hx_ofs, &p->hx_alpha);
    build_tables(src_h, dst_h, &p->hy_ofs, &p->hy_alpha);
    bool ok = cudaMalloc(&p->x_ofs, dst_w * sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&p->y_ofs, dst_h * sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&p->x_alpha, static_cast<size_t>(dst_w) * kTaps * sizeof(int16_t)) == cudaSuccess &&
              cudaMalloc(&p->y_alpha, static_cast<size_t>(dst_h) * kTaps * sizeof(int16_t)) == cudaSuccess;
    ok = ok && cudaMemcpy(p->x_ofs, p->hx_ofs.data(), dst_w * sizeof(int32_t), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(p->y_ofs, p->hy_ofs.data(), dst_h * sizeof(int32_t), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(p->x_alpha, p->hx_alpha.data(), p->hx_alpha.size() * sizeof(int16_t), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(p->y_alpha, p->hy_alpha.data(), p->hy_alpha.size() * sizeof(int16_t), cudaMemcpyHostToDevice) == cudaSuccess;
    const int smem = src_w * 3 * kTaps;
    if (ok && smem > 48 * 1024)
        ok = cudaFuncSetAttribute(resize_lanczos4_normalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess;
    if (!ok) {
        blurr_preproc_destroy(p);
        return blurr::fail(BLURR_ERR_CUDA, "preproc_create: device allocation failed");
    }
    *out = p;
    return 0;
}

extern "C" void blurr_preproc_destroy(blurr_preproc_t* p) {
    if (!p) return;
    cudaFree(p->x_ofs); cudaFree(p->y_ofs); cudaFree(p->x_alpha); cudaFree(p->y_alpha);
    delete p;
}

extern "C" int blurr_preproc_tables(const blurr_preproc_t* p, int32_t* x_ofs, int16_t* x_alpha, int32_t* y_ofs,
                                    int16_t* y_alpha) {
    if (!p || !x_ofs || !x_alpha || !y_ofs || !y_alpha) return blurr::fail(BLURR_ERR_INVALID, "preproc_tables: null argument");
    std::copy(p->hx_ofs.begin(), p->hx_ofs.end(), x_ofs);
    std::copy(p->hx_alpha.begin(), p->hx_alpha.end(), x_alpha);
    std::copy(p->hy_ofs.begin(), p->hy_ofs.end(), y_ofs);
    std::copy(p->hy_alpha.begin(), p->hy_alpha.end(), y_alpha);
    return 0;
}

extern "C" int blurr_preproc_build_tables(int src, int dst, int32_t* ofs, int16_t* alpha) {
    if (src < 1 || dst < 1 || !ofs || !alpha) return blurr::fail(BLURR_ERR_INVALID, "preproc_build_tables: bad argument");
    std::vector<int32_t> o;
    std::vector<int16_t> a;
    build_tables(src, dst, &o, &a);
    std::copy(o.begin(), o.end(), ofs);
    std::copy(a.begin(), a.end(), alpha);
    return 0;
}

extern "C" int blurr_preproc_frame(blurr_preproc_t* p, void* cuda_stream, const void* frame_u8, int64_t row_stride_bytes,
                                   int batch, int64_t frame_stride_bytes, void* pixel_values_bf16, void* resized_u8) {
    if (!p || !frame_u8 || !pixel_values_bf16) return blurr::fail(BLURR_ERR_INVALID, "preproc_frame: null argument");
    if (batch < 1 || row_stride_bytes < static_cast<int64_t>(p->src_w) * 3)
        return blurr::fail(BLURR_ERR_INVALID, "preproc_frame: bad batch or row stride");
    if (cudaSetDevice(p->device) != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, "cudaSetDevice failed");
    FrameArgs a{};
    a.frame = static_cast<const uint8_t*>(frame_u8); a.row_stride = row_stride_bytes; a.frame_stride = frame_stride_bytes;
    a.src_h = p->src_h; a.src_w = p->src_w; a.dst_h = p->dst_h; a.dst_w = p->dst_w;
    a.x_ofs = p->x_ofs; a.y_ofs = p->y_ofs; a.x_alpha = p->x_alpha; a.y_alpha = p->y_alpha;
    a.pixel_values = static_cast<bf16*>(pixel_values_bf16); a.resized = static_cast<uint8_t*>(resized_u8);
    const size_t smem = static_cast<size_t>(p->src_w) * 3 * kTaps;
    resize_lanczos4_normalize_kernel<<<dim3(p->dst_h, batch), 256, smem, static_cast<cudaStream_t>(cuda_stream)>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, std::string("preproc_frame launch failed: ") + cudaGetErrorString(e));
    return 0;
}

extern "C" int blurr_vla_preproc_build_coeffs(int in_size, int out_size, int32_t* bounds, int32_t* weights, int max_taps) {
    if (in_size < 1 || out_size < 1 || in_size > kVlaMaxSize || out_size > kVlaMaxSize)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_build_coeffs: sizes must be in 1..32768");
    std::vector<int32_t> b, w;
    const int ksize = pillow_bicubic_coeffs(in_size, out_size, &b, &w);
    if (bounds == nullptr && weights == nullptr) return ksize;              // query the tap count
    if (bounds == nullptr || weights == nullptr || max_taps < ksize)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_build_coeffs: null table or max_taps below the tap count");
    std::copy(b.begin(), b.end(), bounds);
    for (int o = 0; o < out_size; ++o)
        for (int k = 0; k < max_taps; ++k)
            weights[static_cast<size_t>(o) * max_taps + k] = k < ksize ? w[static_cast<size_t>(o) * ksize + k] : 0;
    return ksize;
}

extern "C" int blurr_vla_preproc_create(int device, int src_h, int src_w, int resize_h, int resize_w, int crop_top,
                                        int crop_left, int crop_h, int crop_w, int n_norms, const float* mean,
                                        const float* stdev, blurr_vla_preproc_t** out) {
    if (!out) return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: null out");
    *out = nullptr;
    for (int s : {src_h, src_w, resize_h, resize_w, crop_h, crop_w})
        if (s < 1 || s > kVlaMaxSize) return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: sizes must be in 1..32768");
    if (crop_top < 0 || crop_left < 0 || crop_top + crop_h > resize_h || crop_left + crop_w > resize_w)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: the crop lies outside the resized image");
    if (n_norms < 1 || n_norms > kVlaMaxNorms)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: n_norms must be 1 or 2");
    if (!mean || !stdev) return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: null mean or std");
    for (int i = 0; i < 3 * n_norms; ++i)
        if (!(stdev[i] != 0.0f) || !std::isfinite(stdev[i]) || !std::isfinite(mean[i]))
            return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: mean and std must be finite and std non-zero");
    std::vector<int32_t> xb, xw, yb, yw;
    const int kx = axis_table(src_w, resize_w, crop_left, crop_w, &xb, &xw);
    const int ky = axis_table(src_h, resize_h, crop_top, crop_h, &yb, &yw);
    // staged source rows of the widest band: the first row of its first window to the last row of its last window
    int band_rows = kVlaBandRows;
    long long smem = 0;
    for (; band_rows >= 1; band_rows /= 2) {
        long long span = 0;
        for (int r0 = 0; r0 < crop_h; r0 += band_rows) {
            const int r1 = std::min(r0 + band_rows, crop_h) - 1;
            span = std::max<long long>(span, yb[2 * r1] + yb[2 * r1 + 1] - yb[2 * r0]);
        }
        smem = span * crop_w * 3;
        if (smem <= kVlaMaxSmem) break;
    }
    if (band_rows < 1)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: one output row's source window is too large for shared memory");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0)
        return blurr::fail(BLURR_ERR_CUDA, "no CUDA device: the preprocessing path has no CPU fallback");
    if (device < 0 || device >= n_dev) return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_create: bad device index");
    if (cudaSetDevice(device) != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, "cudaSetDevice failed");
    blurr_vla_preproc* p = new blurr_vla_preproc();
    p->device = device; p->src_h = src_h; p->src_w = src_w; p->crop_h = crop_h; p->crop_w = crop_w; p->n_norms = n_norms;
    p->kx = kx; p->ky = ky; p->band_rows = band_rows; p->smem = static_cast<int>(smem);
    std::copy(mean, mean + 3 * n_norms, p->mean);
    std::copy(stdev, stdev + 3 * n_norms, p->stdev);
    std::vector<int32_t> all(xb);
    p->x_weights_at = all.size(); all.insert(all.end(), xw.begin(), xw.end());
    p->y_bounds_at = all.size(); all.insert(all.end(), yb.begin(), yb.end());
    p->y_weights_at = all.size(); all.insert(all.end(), yw.begin(), yw.end());
    bool ok = cudaMalloc(&p->tables, all.size() * sizeof(int32_t)) == cudaSuccess &&
              cudaMemcpy(p->tables, all.data(), all.size() * sizeof(int32_t), cudaMemcpyHostToDevice) == cudaSuccess;
    if (ok && smem > 48 * 1024)
        ok = cudaFuncSetAttribute(resize_bicubic_crop_normalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p->smem) == cudaSuccess;
    if (!ok) {
        blurr_vla_preproc_destroy(p);
        return blurr::fail(BLURR_ERR_CUDA, "vla_preproc_create: device allocation failed");
    }
    *out = p;
    return 0;
}

extern "C" void blurr_vla_preproc_destroy(blurr_vla_preproc_t* p) {
    if (!p) return;
    cudaFree(p->tables);
    delete p;
}

extern "C" int blurr_vla_preproc_frame(blurr_vla_preproc_t* p, void* cuda_stream, const void* frames_u8,
                                       int64_t row_stride_bytes, int batch, int64_t frame_stride_bytes,
                                       void* pixel_values_bf16, void* resized_u8) {
    if (!p || !frames_u8 || !pixel_values_bf16) return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_frame: null argument");
    if (batch < 1 || batch > 65535 || row_stride_bytes < static_cast<int64_t>(p->src_w) * 3)
        return blurr::fail(BLURR_ERR_INVALID, "vla_preproc_frame: batch must be in 1..65535 and the row stride >= 3 * width");
    if (cudaSetDevice(p->device) != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, "cudaSetDevice failed");
    VlaArgs a{};
    a.frame = static_cast<const uint8_t*>(frames_u8); a.row_stride = row_stride_bytes; a.frame_stride = frame_stride_bytes;
    a.crop_h = p->crop_h; a.crop_w = p->crop_w; a.kx = p->kx; a.ky = p->ky; a.band_rows = p->band_rows; a.n_norms = p->n_norms;
    a.x_bounds = p->tables; a.x_weights = p->tables + p->x_weights_at;
    a.y_bounds = p->tables + p->y_bounds_at; a.y_weights = p->tables + p->y_weights_at;
    std::copy(p->mean, p->mean + 3 * kVlaMaxNorms, a.mean);
    std::copy(p->stdev, p->stdev + 3 * kVlaMaxNorms, a.stdev);
    a.pixel_values = static_cast<bf16*>(pixel_values_bf16); a.resized = static_cast<uint8_t*>(resized_u8);
    const dim3 grid((p->crop_h + p->band_rows - 1) / p->band_rows, batch);
    resize_bicubic_crop_normalize_kernel<<<grid, kVlaThreads, p->smem, static_cast<cudaStream_t>(cuda_stream)>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, std::string("vla_preproc_frame launch failed: ") + cudaGetErrorString(e));
    return 0;
}

extern "C" int blurr_op_normalize_proprio(void* cuda_stream, const double* raw, const double* lo, const double* hi,
                                          int kind, int n, int dim, void* out_bf16) {
    if (!raw || !lo || !hi || !out_bf16 || n < 1 || dim < 1 || (kind != 0 && kind != 1))
        return blurr::fail(BLURR_ERR_INVALID, "normalize_proprio: bad argument");
    const int total = n * dim;
    normalize_proprio_kernel<<<(total + 127) / 128, 128, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        raw, lo, hi, kind, n, dim, static_cast<bf16*>(out_bf16));
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return blurr::fail(BLURR_ERR_CUDA, std::string("normalize_proprio launch failed: ") + cudaGetErrorString(e));
    return 0;
}
