/*
 * blurr_vit.h - C ABI of the generic pre-LN ViT encoder and of the MLP projector behind the OpenVLA-7B-shaped path's
 * vision side (SURVEY.md 8(f) row 3, BASELINE.json configs[4]: "SigLIP+DINOv2 fused encoder").
 *
 * What it replaces.  Inside `model.predict_action` (`scripts/benchmark_hf_vla.py:152`) OpenVLA's remote code runs two
 * ViTs on the same 224x224 image - DINOv2 ViT-L/14 with 4 register tokens and SigLIP-so400m/14 - takes the patch tokens of
 * each tower's second-to-last block, concatenates them along the feature dim (1024 + 1152) and feeds a 3-layer GELU MLP
 * projector (2176 -> 8704 -> 4096 -> 4096).  None of that code is in the reference tree (parity against it: unpinned);
 * the arithmetic here follows transformers 5.5 `Dinov2WithRegistersModel` / `SiglipVisionModel` with eager attention
 * (a library of this image), against which tests/test_gpu_vit.py pins it.
 *
 * One encoder handle = one tower: patch embedding (14x14 conv as im2col + GEMM), optional cls / register prefix tokens,
 * `num_layers` blocks of LN -> fused QKV -> attention -> out-proj (+ LayerScale) -> residual -> LN -> fc1 + GELU -> fc2
 * (+ LayerScale) -> residual; output = the patch-token rows after the last block that was built.  All on the kernels of
 * the Pi-0 SigLIP tower (tcgen05 GEMMs, LayerNorm consumers, the attention kernels of csrc/attention.cu).
 * Device pointers unless stated; errors as in blurr_pi0.h.  bf16 weights.
 *
 * FiLM (film_dim > 0): OpenVLA-OFT's language conditioning of the towers (its "OFT+" form).  Every block that runs becomes
 * x = x + LS1(attn(LN1(x)));  x = x * (1 + gamma) + beta;  x = x + LS2(MLP(LN2(x)))
 * with gamma = film_scale(cond), beta = film_shift(cond) (nn.Linear(film_dim -> hidden) each, per block) and every
 * operation rounded to bf16 as torch does; cls / register rows are conditioned too.  FiLM towers must be 1024 or 1152
 * wide.  One GEMM per call produces every block's gamma and beta before the first block.
 */
#ifndef BLURR_VIT_H_
#define BLURR_VIT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct blurr_vit blurr_vit_t;
typedef struct blurr_mlp blurr_mlp_t;

typedef struct blurr_vit_config {
    int32_t abi_version;          /* BLURR_VIT_ABI_VERSION */
    int32_t num_layers;           /* blocks to run (OpenVLA: depth - 1 of each tower) */
    int32_t hidden;               /* 1024 (DINOv2-L) / 1152 (SigLIP-so400m); multiple of 128 */
    int32_t num_heads;            /* 16; head_dim = hidden / num_heads must be a multiple of 8 and <= 80 */
    int32_t mlp_dim;              /* 4096 / 4304 */
    int32_t image_size;           /* 224 */
    int32_t patch_size;           /* 14 */
    int32_t num_prefix_tokens;    /* 5 = cls + 4 registers (DINOv2), 0 (SigLIP) */
    int32_t use_layerscale;       /* 1 (DINOv2) / 0 */
    int32_t gelu_erf;             /* 1: exact GELU (DINOv2), 0: tanh approximation (SigLIP) */
    float ln_eps;                 /* 1e-6 */
    int32_t film_dim;             /* 0: no FiLM; else the conditioning width (OpenVLA-OFT: 4096), multiple of 64, <= 8192 */
} blurr_vit_config;
#define BLURR_VIT_ABI_VERSION 2

int blurr_vit_create(const blurr_vit_config* cfg, int device, int max_batch, blurr_vit_t** out);
void blurr_vit_destroy(blurr_vit_t* h);
/* Keys: "patch.weight" [hidden][3*p*p] (conv weight flattened c,kh,kw), "patch.bias" [hidden], "pos" [n_patches][hidden]
 * (position embeddings of the patch tokens), "prefix" [num_prefix_tokens][hidden] (the prefix rows as they enter block 0:
 * cls + its position embedding, then the register tokens), and per block N: "layers.N.ln1.weight|bias",
 * "layers.N.q|k|v|o.weight|bias", "layers.N.ls1" [hidden], "layers.N.ln2.weight|bias", "layers.N.fc1|fc2.weight|bias",
 * "layers.N.ls2" [hidden]; with film_dim > 0 also "layers.N.film_scale.weight|bias" and "layers.N.film_shift.weight|bias"
 * ([hidden][film_dim], [hidden]).  Tensors are copied and repacked. */
int blurr_vit_set_weight(blurr_vit_t* h, const char* key, const void* dev_ptr, const int64_t* shape, int ndim);
int blurr_vit_finalize(blurr_vit_t* h);
/* pixel_values: bf16 [batch][3][image][image] with element strides (b, c, h, w).  Writes the patch-token features,
 * bf16 [batch * n_patches][out_ld], columns 0..hidden-1 of the rows starting at `out` (so two towers can fill the two
 * halves of one concatenated feature matrix).  BLURR_ERR_STATE on a FiLM handle. */
int blurr_vit_forward(blurr_vit_t* h, void* cuda_stream, int batch, const void* pixel_values, const int64_t strides[4],
                      void* out, int out_ld);
/* FiLM handles only (BLURR_ERR_STATE otherwise): blurr_vit_forward, with image i conditioned on row i / images_per_cond
 * of cond, bf16 [batch / images_per_cond][cond_ld] (cond_ld >= film_dim).  images_per_cond must divide batch.  cond is
 * copied into the handle before the blocks run, so one CUDA graph per (batch, images_per_cond) serves every condition. */
int blurr_vit_forward_film(blurr_vit_t* h, void* cuda_stream, int batch, const void* pixel_values, const int64_t strides[4],
                           const void* cond, int cond_ld, int images_per_cond, void* out, int out_ld);
/* Options: "use_cuda_graph" (default 1: the blocks replay as one CUDA graph per batch size and images_per_cond). */
int blurr_vit_set_option(blurr_vit_t* h, const char* name, int64_t value);
int64_t blurr_vit_last_launch_count(const blurr_vit_t* h);

/* Projector: y = W_n(... GELU(W_1 x + b_1) ...) + b_n, exact GELU between the layers (nn.GELU()). dims = n_layers + 1
 * widths, e.g. {2176, 8704, 4096, 4096}. */
int blurr_mlp_create(const int32_t* dims, int n_layers, int device, int max_rows, blurr_mlp_t** out);
void blurr_mlp_destroy(blurr_mlp_t* h);
int blurr_mlp_set_weight(blurr_mlp_t* h, int layer, const void* weight_dev, const void* bias_dev);   /* [out][in], [out] */
int blurr_mlp_forward(blurr_mlp_t* h, void* cuda_stream, int rows, const void* x, int ldx, void* y, int ldy);

/* Image preprocessing of OpenVLA's `PrismaticImageProcessor`, on the device: uint8 RGB frame -> Pillow
 * `Image.resize((resize_w, resize_h), BICUBIC)` (torchvision's resize of a PIL image) -> crop of crop_h x crop_w at
 * (crop_top, crop_left) -> for each of `n_norms` normalisations: fp32 v / 255, (x - mean) / std -> bf16.  Bit-exact
 * against Pillow + torchvision (tests/test_openvla_preprocess.py).  Only the cropped window is computed.
 * mean / std: host float[3 * n_norms], one RGB triple per normalisation (DINOv2's, then SigLIP's).  Sizes are 1..32768;
 * create rejects a crop outside the resize, n_norms outside 1..2, a zero std, and geometries whose source rows for one
 * output row do not fit in shared memory. */
typedef struct blurr_vla_preproc blurr_vla_preproc_t;
int blurr_vla_preproc_create(int device, int src_h, int src_w, int resize_h, int resize_w, int crop_top, int crop_left,
                             int crop_h, int crop_w, int n_norms, const float* mean, const float* std,
                             blurr_vla_preproc_t** out);
void blurr_vla_preproc_destroy(blurr_vla_preproc_t* h);
/* frames_u8: [batch] frames of src_h rows of src_w RGB pixels, `row_stride_bytes` (>= 3 * src_w) between rows and
 * `frame_stride_bytes` between frames.  pixel_values_bf16: [batch][3 * n_norms][crop_h][crop_w]; resized_u8 (or NULL):
 * [batch][crop_h][crop_w][3], the cropped uint8 resize.  Asynchronous on `cuda_stream`. */
int blurr_vla_preproc_frame(blurr_vla_preproc_t* h, void* cuda_stream, const void* frames_u8, int64_t row_stride_bytes,
                            int batch, int64_t frame_stride_bytes, void* pixel_values_bf16, void* resized_u8);
/* Host only, no device needed: Pillow's bicubic coefficients for one axis of an in_size -> out_size resize.
 * Returns ksize, the taps per output index, or a negative status.  With bounds and weights both NULL it only returns
 * ksize; otherwise bounds gets int32 [out_size][2] = (first source index, tap count) and weights int32
 * [out_size][max_taps] in Q22 (zero past the tap count), and max_taps must be >= ksize. */
int blurr_vla_preproc_build_coeffs(int in_size, int out_size, int32_t* bounds, int32_t* weights, int max_taps);

#ifdef __cplusplus
}
#endif
#endif /* BLURR_VIT_H_ */
