/*
 * blurr_act_head.h - C ABI of OpenVLA-OFT's L1-regression action head (Kim, Finn, Liang 2025, "Fine-Tuning VLAs:
 * Optimizing Speed and Success"): `L1RegressionActionHead` -> `MLPResNet(num_blocks, input_dim = D*H, hidden_dim,
 * output_dim = D)`, shipped beside the language model as a module and checkpoint of its own.
 *
 * The head maps the decoder's final-normed hidden rows of the K*D action slots of a sequence to a chunk of K continuous
 * actions of D dimensions.  Rows [batch*K*D][H] are viewed as [batch*K][D*H] (no copy), then:
 *   LayerNorm(D*H) -> Linear(D*H -> hidden) -> ReLU;
 *   num_blocks x: x = x + ReLU(Linear(hidden -> hidden)(LayerNorm(hidden)(x)));
 *   LayerNorm(hidden) -> Linear(hidden -> D).
 * Arithmetic as torch runs the bf16 module: LayerNorm in fp32 with bf16 output, Linear as bf16(acc + bias), ReLU and the
 * residual add in bf16.  The first LayerNorm keeps a row of up to 32768 columns in registers and a wider one (up to 65536,
 * ALOHA's 14 * 4096 = 57344) in shared memory, with the same summation order.  PARITY: pinned against a torch restatement of the module (oracle/openvla_oft_oracle.py); against
 * the OFT repository's code it is UNPINNED (neither vendored nor downloadable), see DESIGN.md.
 *
 * All pointers are device pointers.  Errors: negative blurr_status (blurr_pi0.h), message from blurr_last_error().
 * Weights are bf16.
 */
#ifndef BLURR_ACT_HEAD_H_
#define BLURR_ACT_HEAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct blurr_act_head blurr_act_head_t;

typedef struct blurr_act_head_config {
    int32_t abi_version;          /* BLURR_ACT_HEAD_ABI_VERSION */
    int32_t input_dim;            /* H: the decoder's hidden width, 4096 */
    int32_t action_dim;           /* D: 7 (14 for ALOHA); D * H is a multiple of 64 and at most 65536 */
    int32_t chunk;                /* K: actions per chunk, 8 (25 for ALOHA) */
    int32_t hidden_dim;           /* 4096, a multiple of 128, at most 4096 */
    int32_t num_blocks;           /* MLP-ResNet blocks, 2 */
    float ln_eps;                 /* nn.LayerNorm's 1e-5 */
} blurr_act_head_config;
#define BLURR_ACT_HEAD_ABI_VERSION 1
#ifdef __cplusplus
static_assert(sizeof(blurr_act_head_config) == 28 && offsetof(blurr_act_head_config, ln_eps) == 24, "blurr_act_head_config layout");
#else
_Static_assert(sizeof(blurr_act_head_config) == 28 && offsetof(blurr_act_head_config, ln_eps) == 24, "blurr_act_head_config layout");
#endif

/* max_batch: sequences per forward call (each gives `chunk` rows of D*H). */
int blurr_act_head_create(const blurr_act_head_config* cfg, int device, int max_batch, blurr_act_head_t** out);
void blurr_act_head_destroy(blurr_act_head_t* h);
/* `key`: a key of `L1RegressionActionHead.state_dict()`: "model.layer_norm1.{weight,bias}", "model.fc1.{weight,bias}",
 * "model.mlp_resnet_blocks.N.ffn.0.{weight,bias}" (LayerNorm), "model.mlp_resnet_blocks.N.ffn.1.{weight,bias}" (Linear),
 * "model.layer_norm2.{weight,bias}", "model.fc2.{weight,bias}".  The tensor is copied (Linear weights tile-packed), so
 * the caller may free it afterwards. */
int blurr_act_head_set_weight(blurr_act_head_t* h, const char* key, const void* dev_ptr, const int64_t* shape, int ndim);
int blurr_act_head_finalize(blurr_act_head_t* h);
/* hidden_rows bf16 [batch * chunk][action_dim * input_dim] (the decoder's [batch][chunk * action_dim][input_dim] rows);
 * writes out fp32 [batch][chunk][action_dim]: the head's bf16 output, widened.  Replayed as one CUDA graph per batch. */
int blurr_act_head_forward(blurr_act_head_t* h, void* cuda_stream, int batch, const void* hidden_rows, float* out);
/* Synchronises the stream and reports an expired pipeline wait inside a GEMM. */
int blurr_act_head_check(blurr_act_head_t* h, void* cuda_stream);
/* Kernels launched by the last forward call. */
int64_t blurr_act_head_last_launch_count(const blurr_act_head_t* h);

#ifdef __cplusplus
}
#endif
#endif /* BLURR_ACT_HEAD_H_ */
