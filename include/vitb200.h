/* vitb200.h -- C ABI of the Blackwell-native ViT forward path (drop-in boundary for staghado/vit.cpp).
 *
 * The reference exposes the forward path as C++ free functions in vit.h:
 *     bool vit_model_load(const std::string&, vit_model&)                       (reference vit.h:120, vit.cpp:308-712)
 *     int  vit_predict(const vit_model&, vit_state&, const image_f32,
 *                      const vit_params&, std::vector<std::pair<float,int>>&)   (reference vit.h:122, vit.cpp:1004-1075)
 * There is no plugin registry; the seam is the vit_predict function boundary (SURVEY.md 8b).  The entry points
 * below are what a binding at that seam needs: plain pointers and sizes, no C++ or torch types.  INTEGRATION.md
 * shows the vit.h-side shim (vit_predict re-implemented on top of this header) and the ctypes binding.
 *
 * Conventions (same as the reference, SURVEY.md 8b "Error convention"): functions return 0 on success and a
 * non-zero code on failure; a message is retrievable with vitb200_last_error(); nothing throws or aborts.
 * An engine is bound to ONE CUDA device and is thread-compatible (not thread-safe), like vit_state.
 */
#ifndef VITB200_H
#define VITB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vitb200_engine vitb200_engine;

/* Mirrors the POD part of vit_hparams (reference vit.h:20-37). */
typedef struct vitb200_hparams
{
    int32_t hidden_size;
    int32_t num_hidden_layers;
    int32_t num_attention_heads;
    int32_t num_classes;
    int32_t patch_size;
    int32_t img_size;
    int32_t ftype; /* the model file's ftype (reference vit.cpp:385-414): 0 f32, 1 f16, 2 q4_0, 3 q4_1, 6 q5_0, 7 q5_1, 8 q8_0.
                    * Informational: what counts is each tensor's own `type`.  f16 is the native path; every other format the
                    * reference loader accepts is converted to f16 once at upload (DESIGN.md section 3) */
    float eps;     /* layer-norm epsilon, 1e-6 in the reference (vit.h:29) */
} vitb200_hparams;

/* One host tensor, as found in vit_model::tensors (reference vit.h:88, names at vit.cpp:518-579).
 * `type` uses ggml's type ids for the formats the loader accepts: 0 = F32, 1 = F16, 2 = Q4_0, 3 = Q4_1, 6 = Q5_0, 7 = Q5_1,
 * 8 = Q8_0 (block layouts ggml-quants.h:11-47), plus 30 = BF16 for GGUF containers.  `ne` is ggml order (ne[0] fastest); entries
 * at index >= n_dims are ignored (treated as 1).  Shapes are checked against the reference's declarations (vit.cpp:510-574) and
 * names must be unique. */
typedef struct vitb200_tensor
{
    const char *name;
    const void *data;
    int32_t type;
    int32_t n_dims;
    int64_t ne[4];
} vitb200_tensor;

/* Create an engine from weights that already live in host memory (this is what a vit.h-side shim calls with
 * the contents of vit_model::tensors).  Weights are repacked and uploaded once; the host arena is not retained.
 * max_batch bounds the batch accepted by vitb200_forward*.  Replaces, per model, what the reference re-does per
 * image in vit_predict (graph build x2, ggml_allocr, thread pool; vit.cpp:1009-1036). */
int vitb200_create(const vitb200_hparams *hp, const vitb200_tensor *tensors, int n_tensors, int device, int max_batch,
                   vitb200_engine **out);

/* Same, reading the legacy-ggml model file the reference's vit_model_load parses (vit.cpp:308-712), or a true GGUF v2/v3
 * container with the same tensors (vit.cpp_b200/csrc/gguf_file.hpp). */
int vitb200_create_from_file(const char *path, int device, int max_batch, vitb200_engine **out);

/* The ViTSTR extension of the reference (extensions/vitstr.cpp): the same encoder on a 1-channel image -- the channel count
 * is taken from the patch kernel's shape [P, P, C, D] (vitstr.cpp:482; C = 3 in vit.cpp:515) -- whose classifier reads the
 * first `head_tokens` tokens of every image instead of token 0 (vitstr.cpp:864-903: 25 tokens -> LayerNorm -> head ->
 * soft-max per token).  head_tokens = 1 is vitb200_create / vitb200_create_from_file.  With head_tokens = n every per-image
 * output of vitb200_forward* becomes n consecutive rows: probs/logits float32[batch][n][num_classes], top-k [batch][n][k];
 * images are float32[batch][img][img][C]. */
int vitb200_create_ex(const vitb200_hparams *hp, const vitb200_tensor *tensors, int n_tensors, int device, int max_batch,
                      int head_tokens, vitb200_engine **out);
int vitb200_create_from_file_ex(const char *path, int device, int max_batch, int head_tokens, vitb200_engine **out);
int vitb200_in_chans(const vitb200_engine *e);    /* 3, or 1 for a ViTSTR model */
int vitb200_head_tokens(const vitb200_engine *e); /* classifier rows per image */

void vitb200_destroy(vitb200_engine *e);

int vitb200_get_hparams(const vitb200_engine *e, vitb200_hparams *out);

/* id2label entry of the model file (vit.cpp:356-371); NULL if absent or created from tensors. */
const char *vitb200_label(const vitb200_engine *e, int class_id);

/* Batched vit_predict with HOST buffers (host->device copy of the images and device->host copy of the results
 * are part of the call).  images: float32[batch][img][img][3], the image_f32 layout (vit.h:98-103).
 * Any output pointer may be NULL.  probs/logits: float32[batch][num_classes]; probs are the reference's
 * soft-maxed `state.prediction` (vit.cpp:931-933), logits the pre-softmax node (vit.cpp:928).
 * topk_idx/topk_prob: [batch][k], probabilities descending (the head of the reference's sorted
 * `predictions`, vit.cpp:1047-1057). */
int vitb200_forward(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, int32_t *topk_idx,
                    float *topk_prob, int k);

/* Pipelined form of vitb200_forward: returns as soon as the work is enqueued; the host->device copy of call i+1 overlaps the
 * kernels of call i (two input/output slots).  Host buffers (pinned memory for real overlap) must stay valid, and outputs
 * must not be read, until vitb200_sync() returns.  vitb200_forward == vitb200_forward_async + vitb200_sync. */
int vitb200_forward_async(vitb200_engine *e, const float *images, int batch, float *probs, float *logits,
                          int32_t *topk_idx, float *topk_prob, int k);
int vitb200_sync(vitb200_engine *e);

/* Data-parallel vitb200_forward over n_engines engines (one per GPU of the box, same model, weights replicated) from one host
 * thread: contiguous image shards, no collective (images are independent units).  batch may exceed one engine's max_batch
 * as long as every shard fits. */
int vitb200_forward_sharded(vitb200_engine *const *engines, int n_engines, const float *images, int batch, float *probs, float *logits,
                            int32_t *topk_idx, float *topk_prob, int k);
/* Pipelined form: returns once every shard is enqueued on its engine's two-slot pipeline (vitb200_forward_async), so the same host
 * thread can submit the next global batch while this one runs; buffers must stay valid until vitb200_sync_all() (== vitb200_sync
 * on every engine) returns.  vitb200_forward_sharded == this + vitb200_sync_all. */
int vitb200_forward_sharded_async(vitb200_engine *const *engines, int n_engines, const float *images, int batch, float *probs,
                                  float *logits, int32_t *topk_idx, float *topk_prob, int k);
int vitb200_sync_all(vitb200_engine *const *engines, int n_engines);

/* vit_image_preprocess + vit_predict fused on the GPU (reference vit.h:119, vit.cpp:130-305 + vit.cpp:1004): `images[b]` is the
 * interleaved RGB u8 image the reference's load_image_from_file produces (image_u8::data, vit.h:91-96), nx[b] x ny[b]
 * pixels, any size.  bilinear = 0 selects the reference's default bicubic path (hparams.interpolation, vit.h:30).  The resize,
 * the round-to-u8 and the mean/std normalisation run on the device and feed the forward pass directly; images_f32_out
 * (optional, host, [batch][img][img][3]) returns the pre-processed image_f32 batch.  probs/logits/top-k as vitb200_forward;
 * all of them NULL = preprocess only. */
int vitb200_forward_u8(vitb200_engine *e, const uint8_t *const *images, const int *nx, const int *ny, int batch, int bilinear,
                       float *images_f32_out, float *probs, float *logits, int32_t *topk_idx, float *topk_prob, int k);

/* Pipelined form (vitb200_forward_u8 == this + vitb200_sync, plus the optional f32 read-back): the images are packed into a pinned
 * staging buffer inside the call (so `images` may be reused as soon as it returns), ONE host-to-device copy per batch overlaps the
 * previous call's kernels, the pre-processed pixels go straight into the f16 patch matrix of the patch-embedding GEMM, and nothing
 * synchronises or allocates in steady state.  Output buffers must stay valid until vitb200_sync().  Shares its two pipeline slots
 * with vitb200_forward_async. */
int vitb200_forward_u8_async(vitb200_engine *e, const uint8_t *const *images, const int *nx, const int *ny, int batch, int bilinear,
                             float *probs, float *logits, int32_t *topk_idx, float *topk_prob, int k);

/* Same with DEVICE buffers on the engine's device, enqueued on `stream` (a cudaStream_t; NULL = the engine's own
 * stream) without synchronising: the caller owns ordering.  This is the resident-data path bench.py times. */
int vitb200_forward_device(vitb200_engine *e, const float *d_images, int batch, float *d_probs, float *d_logits,
                           int32_t *d_topk_idx, float *d_topk_prob, int k, void *stream);

/* Number of kernels this library launched during the most recent forward call. */
int vitb200_last_launch_count(const vitb200_engine *e);

/* Per-kernel device timing for roofline reporting: while enabled, CUDA-event pairs are recorded around every
 * launch of the tracked kernels on the stream the forward runs on.  kind: 0 patch GEMM, 1 qkv GEMM, 2 proj GEMM,
 * 3 fc1 GEMM, 4 fc2 GEMM, 5 head GEMM, 6 attention, 7 layernorm.  profile_read synchronises the device and returns
 * the summed duration, the launch count and the algorithmic FLOPs of one launch (0 for HBM-bound kernels). */
int vitb200_profile_enable(vitb200_engine *e, int on);
int vitb200_profile_read(vitb200_engine *e, int kind, double *ms_total, int *launches, double *flops_per_launch);

/* Opaque handles for timing on the engine's stream (bench.py passes its own stream instead, normally). */
void *vitb200_stream(vitb200_engine *e);

const char *vitb200_last_error(void);

/* ---- test / debug surface (used by tests/ only) -------------------------------------------------------- */

/* Intermediates of one forward of `batch` <= max_batch images, converted to float32 on the host.
 * Any pointer may be NULL.  Shapes per image (N = tokens, D = hidden): see oracle/vit_oracle.c vo_taps. */
typedef struct vitb200_taps
{
    int32_t layer;
    float *embed;    /* [batch][N][D]  */
    float *ln1;      /* [batch][N][D]  */
    float *qkv;      /* [batch][N][3D] */
    float *attn;     /* [batch][N][D]  */
    float *x1;       /* [batch][N][D]  */
    float *ln2;      /* [batch][N][D]  */
    float *h;        /* [batch][N][4D] */
    float *x2;       /* [batch][N][D]  */
    float *final_ln; /* [batch][D]     */
    float *x_final;  /* [batch][N][D]  */
} vitb200_taps;

int vitb200_forward_debug(vitb200_engine *e, const float *images, int batch, float *probs, float *logits,
                          const vitb200_taps *taps);

/* Stand-alone run of the tcgen05 GEMM kernel: out[M][N] = epilogue(A[M][K] (f16 bits) x W[N][K]^T (f16 bits)).
 * epilogue: 0 bias->f16, 1 bias+gelu->f16, 2 bias+resid->f32, 4 bias->f32, 6 bias->split precision (hi = f16(x), lo = f16(x - hi);
 * `out` receives hi + lo).  out is float32[M][N] on the host (f16 results widened).  resid may be NULL unless epilogue == 2. */
int vitb200_test_gemm(int device, int M, int N, int K, int epilogue, const uint16_t *A, const uint16_t *W,
                      const float *bias, const float *resid, float *out);

/* Stand-alone run of the block LayerNorm kernel the forward schedule uses (reference ggml_norm + ggml_mul + ggml_add, vit.cpp:808-812,
 * ggml.c:8959-9008): x float32 [rows][D] -> y float32 [rows][D] holding the f16 results (the next GEMM's A operand) widened. */
int vitb200_test_layernorm(int device, int rows, int D, const float *x, const float *w, const float *b, float eps, float *y);

/* Stand-alone run of the final soft-max + top-k (reference vit.cpp:931 + the sorted predictions of vit.cpp:1047-1057) through the
 * forward's own launcher: logits = float32 [R][ldl] (host), of which the first C columns of every row are read; probs = float32 [R][C]
 * with the reference's f16-exp semantics; idx / val = [R][k], probabilities descending, index ascending on ties, entries past C are
 * (-1, 0).  0 <= k <= 16 (the forward's limit); idx / val may be NULL when k == 0. */
int vitb200_test_softmax_topk(int device, int R, int C, int ldl, const float *logits, int k, float *probs, int32_t *idx, float *val);

/* Prototype of the reference's q8_0 x q8_0 linear layer on the INTEGER tensor cores (tcgen05.mma kind::i8, one K = 32 MMA per
 * q8_0 block; csrc/gemm_q8_tcgen05.cuh).  Replaces, for one layer, quantize_row_q8_0 (reference ggml-quants.c:702-790: the f32
 * activation rows x [M][K] are quantised on the device, bit for bit as the reference does) + ggml_vec_dot_q8_0_q8_0
 * (ggml-quants.c:3521+) + the bias add.  w_q8_0 is the tensor as stored in a q8_0 model file: [N][K/32] blocks of {f16 d; int8 q[32]}
 * (ggml-quants.h:42-46).  y = float32 [M][N]; xq (int8 [M][K]) and xd (float32 [M][K/32]) optionally receive the quantised
 * activations; with iters > 0 *ms_per_launch receives the CUDA-event time of one GEMM launch averaged over `iters` launches.
 * K % 128 == 0, N % 4 == 0.  Not part of the forward schedule (it is slower than the f16 tensor-core path, DESIGN.md section 3). */
int vitb200_test_gemm_q8(int device, int M, int N, int K, const float *x, const void *w_q8_0, const float *bias, float *y,
                         int8_t *xq, float *xd, int iters, float *ms_per_launch);

/* Stand-alone run of one attention kernel (head dim 64) over a fused QKV buffer: qkv = f16 bits [B*N][3*H*64] (what the qkv
 * GEMM leaves behind, reference vit.cpp:826-846), out = float32 [B*N][H*64] (the merged heads before proj, vit.cpp:860-866).
 * kernel: 0 = the engine's choice for N, 1 = mma.sync two-pass, 2 = tcgen05 single block (N <= 224), 3 = tcgen05 two sweeps
 * (224 < N <= 640). */
int vitb200_test_attention(int device, int kernel, int B, int N, int H, const uint16_t *qkv, float *out);

/* The tcgen05 single-block attention kernel (N <= 224) on split-precision operands, the way the engine runs it: every q, k, v value is
 * the sum of two f16 numbers, qkv_hi + qkv_lo (what the qkv GEMM's hi-lo epilogue leaves behind: hi = f16(x), lo = f16(x - hi)), so
 * the f16 tensor cores reproduce the reference's f32-operand attention mat-muls (vit.cpp:848,858). */
int vitb200_test_attention_hilo(int device, int B, int N, int H, const uint16_t *qkv_hi, const uint16_t *qkv_lo, float *out);

/* Host-only: the upload-time weight conversion of one quantised tensor, `n_blocks` ggml blocks of 32 weights
 * (type = ggml_type / file ftype: 2 q4_0, 3 q4_1, 6 q5_0, 7 q5_1, 8 q8_0; ggml-quants.h:11-47) -> f16 bits, exactly what
 * vitb200_create stores on the device.  Needs no GPU.  Follows dequantize_row_q* (ggml-quants.c:1074-1185). */
int vitb200_test_dequant(int type, const void *blocks, int64_t n_blocks, uint16_t *out_f16);

#ifdef __cplusplus
}
#endif
#endif /* VITB200_H */
