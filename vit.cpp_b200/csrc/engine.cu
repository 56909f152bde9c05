// engine.cu -- host side of the C ABI in include/vitb200.h: weight upload/repack, the static device arena,
// TMA descriptors, and the fixed kernel schedule that replaces the reference's per-image graph build +
// ggml_allocr + ggml_graph_compute thread pool (reference vit.cpp:1004-1075, ggml.c:15774-16039).
#include "../../include/vitb200.h"

#include "gemm_tcgen05.cuh"
#include "kernels.cuh"
#include "attention_tcgen05.cuh"
#include "attention_tcgen05_long.cuh"
#include "gemm_q8_tcgen05.cuh"
#include "gguf_file.hpp"
#include "preprocess.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <string>
#include <vector>

using namespace vitb200;

namespace {

thread_local std::string g_err;

int fail(const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    fprintf(stderr, "vitb200: %s\n", buf); // reference convention: message on stderr + non-zero return
    return 1;
}

#define CUDA_TRY(x)                                                                       \
    do                                                                                    \
    {                                                                                     \
        cudaError_t e_ = (x);                                                             \
        if (e_ != cudaSuccess)                                                            \
        {                                                                                 \
            (void)cudaGetLastError(); /* do not leave it for an unrelated later check */  \
            return fail("%s failed: %s", #x, cudaGetErrorString(e_));                     \
        }                                                                                 \
    } while (0)

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                        const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_tmapEncodeTiled tmap_encoder()
{
    static PFN_tmapEncodeTiled fn = nullptr;
    if (!fn)
    {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
    }
    return fn;
}

// 2-D f16 row-major tensor [rows][cols] with row pitch `pitch` elements, box = 64 columns x box_rows rows,
// SWIZZLE_128B (matches the UMMA K-major SWIZZLE_128B smem descriptor), out-of-bounds elements read as zero.
// 2-D f32 row-major tensor [rows][cols], box = 32 columns (128 B) x 32 rows, SWIZZLE_128B: the residual stream X as the
// residual epilogue loads and stores it (one 4-KB box per epilogue warp and 32-column chunk).
int make_tmap_f32_box32(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint64_t pitch)
{
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(f32) failed (%d)", (int)r);
    return 0;
}

// 3-D f16 view [images][tokens][cols] of a [images*tokens][cols] buffer, box = 64 columns x 32 tokens x 1 image, SWIZZLE_128B:
// the attention epilogue's store target -- token rows past `tokens` are clipped by the TMA unit instead of spilling into the
// next image.
int make_tmap_tokens3d(CUtensorMap *m, const void *ptr, uint64_t images, uint64_t tokens, uint64_t cols)
{
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[3] = {cols, tokens, images};
    cuuint64_t strides[2] = {cols * 2, tokens * cols * 2};
    cuuint32_t box[3] = {64, 32, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(3d) failed (%d)", (int)r);
    return 0;
}

// 3-D f16 view of a HEAD-MAJOR q / k / v buffer [planes][plane_rows][64] (planes = 3 x heads: q heads, then k heads, then v heads;
// plane_rows = the arena's token rows): dims {64, rows, planes}, box = 64 columns x box_rows rows x 1 plane, SWIZZLE_128B.  `rows` may be
// smaller than plane_rows (the qkv epilogue's store map of a batch: rows past the batch are clipped).
int make_tmap_heads3d(CUtensorMap *m, const void *ptr, uint64_t planes, uint64_t rows, uint64_t plane_rows, uint32_t box_rows)
{
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[3] = {64, rows, planes};
    cuuint64_t strides[2] = {128, plane_rows * 128};
    cuuint32_t box[3] = {64, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(heads3d) failed (%d) planes=%llu rows=%llu box_rows=%u", (int)r,
                                       (unsigned long long)planes, (unsigned long long)rows, box_rows);
    return 0;
}

int make_tmap(CUtensorMap *m, const void *ptr, uint64_t rows, uint64_t cols, uint64_t pitch, uint32_t box_rows)
{
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch * 2};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu pitch=%llu box_rows=%u", (int)r,
                                       (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)pitch, box_rows);
    return 0;
}

// generic 2-D row-major tensor map (the q8_0 prototype's int8 planes and f32 scale planes)
int make_tmap_2d(CUtensorMap *m, CUtensorMapDataType dt, size_t elem_bytes, const void *ptr, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                 uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle sw)
{
    PFN_tmapEncodeTiled enc = tmap_encoder();
    if (!enc) return fail("cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch_elems * elem_bytes};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, dt, 2, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(2d) failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows, (unsigned long long)cols);
    return 0;
}

struct Linear
{
    __half *w = nullptr; // [n_out][ld] f16, K contiguous (ggml ne0 = K)
    float *b = nullptr;  // [n_out]
    int n_out = 0, n_in = 0, ld = 0, bn = 256;
    CUtensorMap tm;  // box = 64 x (bn / cta_group) rows: the share of the W tile one CTA stages
};

struct Layer
{
    float *n1w = nullptr, *n1b = nullptr, *n2w = nullptr, *n2b = nullptr;
    Linear qkv, proj, fc1, fc2;
};

int pick_bn(int n_out) { return n_out >= 256 ? 256 : 128; }

} // namespace

struct vitb200_engine
{
    vitb200_hparams hp;
    int device = 0, max_batch = 0, num_sms = 148;
    int N = 0, NP = 0, G = 0, KP = 0, KPp = 0;
    int Cp = 0;           // num_classes rounded up to a multiple of 4: pitch of the internal logits rows (128-bit epilogue stores)
    float *d_sm_scratch = nullptr; // soft-max working rows in global memory, only when num_classes floats exceed shared memory
    int C = 3;            // input channels: 3 (vit.cpp) or 1 (ViTSTR extension, vitstr.cpp:713), taken from the patch kernel's shape
    int head_tokens = 1;  // tokens the classifier head reads per image: 1 (token 0, vit.cpp:910) or 25 (vitstr.cpp:864-903)
    cudaStream_t stream = nullptr;
    std::vector<void *> allocs;
    // weights
    float *cls = nullptr, *pos = nullptr, *norm_w = nullptr, *norm_b = nullptr;
    Linear patch, head;
    std::vector<Layer> layers;
    // activations (static arena, sized for max_batch)
    float *d_img = nullptr, *X = nullptr, *d_logits = nullptr, *d_probs = nullptr, *d_topk_val = nullptr;
    int32_t *d_topk_idx = nullptr;
    __half *A16 = nullptr, *QKV16 = nullptr, *H16 = nullptr, *CLS16 = nullptr, *PA = nullptr;
    __half *QKV16L = nullptr; // lo halves of q, k, v (x - f16(x), as f16): the tcgen05 attention's split-precision operands
    int *d_ln_count = nullptr; // fused LayerNorm: one completion counter per 32-row group of the residual stream (zero between launches)
    bool fused_ln = false;     // LayerNorm applied inside the proj / fc2 residual epilogues (VITB200_FUSED_LN=0: separate kernel)
    bool attn_hilo = false;   // qkv GEMM emits hi + lo and attention_tc_kernel runs the 3 + 2 term products (VITB200_ATTN_HILO=0: hi only)
    CUtensorMap tmQl, tmKVl;
    CUtensorMap tmA_D, tmA_H, tmA_P, tmA_C, tmQ, tmKV, tmAO, tmKV64;
    // maps of the tensors the GEMM epilogues WRITE with TMA, clipped to batch * N rows so that nothing past the batch is ever
    // stored (and, for the residual stream, loaded): X f32 (32 x 32 boxes), QKV hi / lo and the MLP hidden buffer f16 (64 x 32 boxes)
    struct BatchMaps { CUtensorMap X, QKVh, QKVl, H; };
    std::map<int, BatchMaps> batch_maps;
    bool attn_tc = false;      // tcgen05 single-block attention (N <= 224)
    bool attn_tc_long = false; // tcgen05 two-sweep attention (224 < N <= 640); anything longer uses the mma.sync two-pass kernel
    int max_k = 16;
    int launches = 0;
    int cta_group = 2; // CTAs per tcgen05.mma in the GEMMs (2 = CTA pairs; VITB200_CTA_GROUP=1 selects the 1-CTA kernels)
    std::map<int, std::string> labels;
    // host-buffer pipeline (vitb200_forward_async): 2 input/output slots, H2D on a copy stream overlapping the previous
    // call's kernels on the compute stream
    cudaStream_t copy_stream = nullptr;
    float *d_img_slot[2] = {nullptr, nullptr}, *d_probs_slot[2] = {nullptr, nullptr}, *d_logits_slot[2] = {nullptr, nullptr};
    float *d_topk_val_slot[2] = {nullptr, nullptr};
    int32_t *d_topk_idx_slot[2] = {nullptr, nullptr};
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    unsigned long long submits = 0;
    // GPU preprocessing (vitb200_forward_u8*): per pipeline slot a PINNED host staging buffer (the caller's images are packed into it,
    // followed by the per-image descriptors) and its device twin; grown only when a batch needs more than any batch before it
    uint8_t *h_u8[2] = {nullptr, nullptr}, *d_u8[2] = {nullptr, nullptr};
    size_t u8_cap[2] = {0, 0};
    // CUDA-graph cache for the kernel schedule of one forward, keyed by its arguments (launch-bound inner loop: ~90 kernels)
    struct GraphEntry { const void *img; int batch; void *probs, *logits, *tidx, *tval; int k; int state; int launches; cudaGraphExec_t exec; };
    std::vector<GraphEntry> graphs;
    bool use_graph = true;
    // optional per-kernel timing (bench.py roofline): CUDA event pairs around tracked launches
    bool profile = false;
    struct ProfRec { int kind; cudaEvent_t a, b; double flops; };
    std::vector<ProfRec> prof;
    std::vector<cudaEvent_t> event_pool;
};

namespace {

template <typename T>
int dev_alloc(vitb200_engine *e, T **p, size_t count)
{
    void *q = nullptr;
    CUDA_TRY(cudaMalloc(&q, count * sizeof(T) + 256));
    e->allocs.push_back(q);
    // activation rows past the current batch are read (and masked) by the attention tiles: they must never hold NaN bit patterns
    CUDA_TRY(cudaMemset(q, 0, count * sizeof(T) + 256));
    *p = reinterpret_cast<T *>(q);
    return 0;
}

const vitb200_tensor *find_tensor(const vitb200_tensor *t, int n, const std::string &name)
{
    for (int i = 0; i < n; ++i)
        if (t[i].name && name == t[i].name) return &t[i];
    return nullptr;
}

// the reference keeps tensors in a std::map keyed by name (vit.h:88), so a name can only occur once; a caller-built list with a
// repeated name is rejected instead of silently taking the first
int check_unique_names(const vitb200_tensor *t, int n)
{
    std::map<std::string, int> seen;
    for (int i = 0; i < n; ++i)
    {
        if (!t[i].name || !t[i].data) return fail("tensor %d has a null name or data pointer", i);
        if (t[i].n_dims < 1 || t[i].n_dims > 4) return fail("tensor '%s' has %d dimensions", t[i].name, t[i].n_dims);
        if (seen.count(t[i].name)) return fail("duplicate tensor '%s' in model", t[i].name);
        seen[t[i].name] = i;
    }
    return 0;
}

int64_t dim_of(const vitb200_tensor *t, int i) { return i < t->n_dims ? t->ne[i] : 1; }

// the reference loader's shape check (vit.cpp:633-641): all four ggml extents must match the tensor the model declares
int check_shape(const vitb200_tensor *x, const std::string &name, int64_t e0, int64_t e1, int64_t e2, int64_t e3)
{
    if (dim_of(x, 0) != e0 || dim_of(x, 1) != e1 || dim_of(x, 2) != e2 || dim_of(x, 3) != e3)
        return fail("tensor '%s' has wrong shape in model file: got [%lld, %lld, %lld, %lld], expected [%lld, %lld, %lld, %lld]", name.c_str(),
                    (long long)dim_of(x, 0), (long long)dim_of(x, 1), (long long)dim_of(x, 2), (long long)dim_of(x, 3),
                    (long long)e0, (long long)e1, (long long)e2, (long long)e3);
    return 0;
}

int64_t nelem(const vitb200_tensor *t)
{
    int64_t n = 1;
    for (int i = 0; i < t->n_dims && i < 4; ++i) n *= t->ne[i];
    return n;
}

// f32 tensor with the reference's declared extents {e0, e1, e2, e3} (vit.cpp:510-574); `padded` >= the element count allocates a
// zero-filled tail (the classifier bias when num_classes is not a multiple of 4)
int upload_f32(vitb200_engine *e, const vitb200_tensor *t, int n, const std::string &name, int64_t e0, int64_t e1, int64_t e2, int64_t e3,
               float **dst, int64_t padded = 0)
{
    const vitb200_tensor *x = find_tensor(t, n, name);
    if (!x) return fail("missing tensor '%s'", name.c_str());
    if (x->type != 0) return fail("tensor '%s' must be f32 (type %d)", name.c_str(), x->type);
    const int64_t expect = e0 * e1 * e2 * e3;
    if (nelem(x) != expect) return fail("tensor '%s' has wrong size in model file: got %lld, expected %lld", name.c_str(), (long long)nelem(x), (long long)expect);
    if (check_shape(x, name, e0, e1, e2, e3)) return 1;
    if (dev_alloc(e, dst, (size_t)(padded > expect ? padded : expect))) return 1;
    CUDA_TRY(cudaMemcpy(*dst, x->data, (size_t)expect * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

// IEEE f32 -> f16 round-to-nearest-even on the host (upload-time conversions only)
uint16_t host_f32_to_f16(float f) { const __half h = __float2half_rn(f); uint16_t u; memcpy(&u, &h, 2); return u; }
float host_f16_to_f32(uint16_t u) { __half h; memcpy(&h, &u, 2); return __half2float(h); }

// ggml block formats of 32 weights (ggml-quants.h:11-47), keyed by ggml_type / file ftype (vit.cpp:645-672).
size_t quant_block_bytes(int type)
{
    switch (type)
    {
    case 2: return 18; // q4_0 { f16 d; u8 qs[16] }
    case 3: return 20; // q4_1 { f16 d; f16 m; u8 qs[16] }
    case 6: return 22; // q5_0 { f16 d; u8 qh[4]; u8 qs[16] }
    case 7: return 24; // q5_1 { f16 d; f16 m; u8 qh[4]; u8 qs[16] }
    case 8: return 34; // q8_0 { f16 d; i8 qs[32] }
    default: return 0;
    }
}

// One block -> 32 floats, the arithmetic of ggml's dequantize_row_q* (ggml-quants.c:1074-1185): low nibbles are elements
// 0..15, high nibbles 16..31, the q5 formats take their fifth bit from qh; the *_1 formats add the block minimum m.
void dequant_block(int type, const uint8_t *blk, float *y)
{
    uint16_t du = 0, mu = 0;
    memcpy(&du, blk, 2);
    const float d = host_f16_to_f32(du);
    if (type == 8)
    {
        const int8_t *q = (const int8_t *)(blk + 2);
        for (int i = 0; i < 32; ++i) y[i] = d * (float)q[i];
        return;
    }
    const bool has_min = type == 3 || type == 7, five = type == 6 || type == 7;
    float m = 0.f;
    if (has_min) { memcpy(&mu, blk + 2, 2); m = host_f16_to_f32(mu); }
    const uint8_t *p = blk + (has_min ? 4 : 2);
    uint32_t qh = 0;
    if (five) { memcpy(&qh, p, 4); p += 4; }
    for (int j = 0; j < 16; ++j)
    {
        int x0 = p[j] & 0x0F, x1 = p[j] >> 4;
        if (five)
        {
            x0 |= (int)(((qh >> j) << 4) & 0x10);
            x1 |= (int)((qh >> (j + 12)) & 0x10);
        }
        if (has_min) { y[j] = (float)x0 * d + m; y[j + 16] = (float)x1 * d + m; }
        else
        {
            const int off = five ? 16 : 8;
            y[j] = (float)(x0 - off) * d; y[j + 16] = (float)(x1 - off) * d;
        }
    }
}

// Weight matrix [n_out][n_in] -> device f16, row pitch padded to ld (zero filled), + its TMA descriptor.
//   type 1 (F16): used as stored -- the reference's own operand (ggml.c:1200-1236).
//   type 8 (Q8_0, blocks of {f16 d; int8 q[32]}, ggml-quants.h:42-46): dequantised once to f16(d * q).  The reference
//          multiplies int8 x dynamically quantised int8 activations (ggml-quants.c:3521); this W8A16 form stays within the
//          q8_0 noise floor of that path (SURVEY.md 7.4: 1.6e-2 either way); an int8 tensor-core path is future work.
//   types 2/3/6/7 (Q4_0, Q4_1, Q5_0, Q5_1): same treatment -- dequantised once with ggml's dequantize_row arithmetic and
//          rounded to f16 (exact for q4_0/q5_0 whenever d*q is a normal f16: a 5-bit integer times an f16).  The reference
//          dots them against activations quantised on the fly to q8_0/q8_1 (ggml.c type traits vec_dot_type).
//   type 0 (F32): rounded once to f16 (the reference keeps f32 weights AND f32 activations, ggml.c:1163-1198).
//   type 30 (BF16, GGUF containers): widened to f32, then as type 0.
int upload_linear(vitb200_engine *e, const vitb200_tensor *t, int n, const std::string &wname, const std::string &bname,
                  int n_out, int n_in, int ld, Linear *L, int conv_p = 0)
{
    const vitb200_tensor *w = find_tensor(t, n, wname);
    if (!w) return fail("missing tensor '%s'", wname.c_str());
    if (w->type != 0 && w->type != 1 && w->type != 30 && quant_block_bytes(w->type) == 0)
        return fail("tensor '%s': weight type %d is not supported (f32, f16, bf16, q4_0, q4_1, q5_0, q5_1, q8_0 only)", wname.c_str(), w->type);
    if (nelem(w) != (int64_t)n_out * n_in) return fail("tensor '%s' has wrong size in model file: got %lld, expected %lld", wname.c_str(), (long long)nelem(w), (long long)n_out * n_in);
    if (conv_p > 0) { if (check_shape(w, wname, conv_p, conv_p, n_in / (conv_p * conv_p), n_out)) return 1; } // [P, P, C, D], vit.cpp:515
    else if (check_shape(w, wname, n_in, n_out, 1, 1)) return 1;                                             // [in, out], vit.cpp:531-543
    if (quant_block_bytes(w->type) && n_in % 32 != 0) return fail("tensor '%s': quantised rows must be a multiple of 32", wname.c_str());
    L->n_out = n_out; L->n_in = n_in; L->ld = ld; L->bn = pick_bn(n_out);
    if (dev_alloc(e, &L->w, (size_t)n_out * ld)) return 1;
    CUDA_TRY(cudaMemset(L->w, 0, (size_t)n_out * ld * sizeof(__half)));
    const void *src = w->data;
    std::vector<uint16_t> conv;
    if (w->type != 1)
    {
        conv.resize((size_t)n_out * n_in);
        if (w->type == 0)
        {
            // Rounded once to f16.  A bf16 checkpoint widened to f32 (the only way this container can carry bf16,
            // BASELINE.json configs[2]) converts EXACTLY for every weight with |w| >= 2^-14 (8-bit mantissa fits in 11).
            // Keeping such weights as bf16 is not an option: tcgen05.mma kind::f16 with a_format = f16 and b_format = bf16
            // raises "illegal instruction" on B200 (tried in round 1), and bf16 activations cost 5e-3 parity (SURVEY.md 7.4).
            const float *f = (const float *)w->data;
            for (size_t i = 0; i < conv.size(); ++i) conv[i] = host_f32_to_f16(f[i]);
        }
        else if (w->type == 30)
        {
            // BF16 tensors (GGUF containers only): widened to f32 (exact) and rounded to f16 like the f32 case above
            const uint16_t *h = (const uint16_t *)w->data;
            for (size_t i = 0; i < conv.size(); ++i)
            {
                const uint32_t u = (uint32_t)h[i] << 16;
                float f;
                memcpy(&f, &u, 4);
                conv[i] = host_f32_to_f16(f);
            }
        }
        else
        {
            const uint8_t *blk = (const uint8_t *)w->data;
            const size_t nb = conv.size() / 32, bs = quant_block_bytes(w->type);
            float y[32];
            for (size_t b = 0; b < nb; ++b)
            {
                dequant_block(w->type, blk + b * bs, y);
                for (int i = 0; i < 32; ++i) conv[b * 32 + i] = host_f32_to_f16(y[i]);
            }
        }
        src = conv.data();
    }
    CUDA_TRY(cudaMemcpy2D(L->w, (size_t)ld * 2, src, (size_t)n_in * 2, (size_t)n_in * 2, (size_t)n_out, cudaMemcpyHostToDevice));
    // conv bias is declared [1, 1, D] (vit.cpp:516), every other bias [n_out]; the tail up to a multiple of 4 stays zero
    if (conv_p > 0 ? upload_f32(e, t, n, bname, 1, 1, n_out, 1, &L->b) : upload_f32(e, t, n, bname, n_out, 1, 1, 1, &L->b, (n_out + 3) / 4 * 4)) return 1;
    return make_tmap(&L->tm, L->w, (uint64_t)n_out, (uint64_t)ld, (uint64_t)ld, (uint32_t)(L->bn / e->cta_group));
}

// dynamic shared memory the soft-max kernel may use for its working row (227 KB per CTA minus room for its static arrays); the
// launch needs the opt-in as soon as the row and those arrays exceed the 48 KB default
constexpr size_t kSoftmaxStaticSmem = 1024;
constexpr size_t kSoftmaxSmemMax = 232448 - kSoftmaxStaticSmem;

enum ProfKind { PK_PATCH = 0, PK_QKV, PK_PROJ, PK_FC1, PK_FC2, PK_HEAD, PK_ATTN, PK_LN, PK_COUNT };

struct ProfScope
{
    vitb200_engine *e;
    cudaStream_t s;
    cudaEvent_t b = nullptr;
    ProfScope(vitb200_engine *e_, int kind, double flops, cudaStream_t s_) : e(e_), s(s_)
    {
        if (!e || !e->profile) { e = nullptr; return; }
        cudaEvent_t a = nullptr;
        auto get = [&](cudaEvent_t *ev) {
            if (!e->event_pool.empty()) { *ev = e->event_pool.back(); e->event_pool.pop_back(); }
            else cudaEventCreate(ev);
        };
        get(&a);
        get(&b);
        cudaEventRecord(a, s);
        e->prof.push_back({kind, a, b, flops});
    }
    ~ProfScope()
    {
        if (e) cudaEventRecord(b, s);
    }
};

// L2 eviction hints on the big streamed-once transfers (profiles/microbench_r02.md: fc1 -4 %, LayerNorm -2 %, proj / fc2 -1 % at batch 256 --
// the 465 MB of q, k, v and the 310 MB MLP hidden buffer no longer push the LayerNorm output, which the next GEMM reads nine to twelve
// times, out of the 126 MB L2).  VITB200_L2HINT = bit mask, default 7: 1 = qkv / fc1 output stores evict_first, 2 = attention operand
// loads evict_first, 4 = LayerNorm input loads evict_first (8 = LayerNorm output stores evict_last: measured worse, off).
int l2_hint_mask()
{
    static const int m = getenv("VITB200_L2HINT") ? atoi(getenv("VITB200_L2HINT")) : 7;
    return m;
}

// Programmatic dependent launch for the per-layer kernels (GEMMs, attention, LayerNorm): each of them ends its prologue with
// griddepcontrol.launch_dependents + griddepcontrol.wait (ptx.cuh), so kernel k+1's barrier init / TMEM allocation / descriptor
// prefetch runs on the SMs kernel k has already left.  VITB200_PDL=0 launches them fully serialised.
bool pdl_enabled()
{
    static const bool on = !(getenv("VITB200_PDL") && atoi(getenv("VITB200_PDL")) == 0);
    return on;
}

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args &&...args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

template <int BN, int EPI, int CG, int DEEPK = 0>
int launch_gemm_t(vitb200_engine *e, const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmX, const CUtensorMap &tmO2, const GemmParams &p, cudaStream_t s, int num_sms)
{
    using Cfg = GemmCfg<BN, EPI == EPI_BIAS_RESID_F32, CG, EPI == EPI_PATCH_GATHER_F32, DEEPK != 0,
                        EPI == EPI_BIAS_F16 || EPI == EPI_BIAS_GELU_F16 || EPI == EPI_BIAS_F16_HILO>;
    auto kern = gemm_tcgen05_kernel<BN, EPI, DEEPK, CG>;
    // the opt-in to > 48 KB dynamic shared memory is per device (one engine per device, possibly several per process)
    static bool attr_set[64] = {};
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (!attr_set[dev & 63])
    {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_set[dev & 63] = true;
    }
    const int m_tiles = (p.M + GEMM_BM * CG - 1) / (GEMM_BM * CG), n_tiles = (p.N + BN - 1) / BN;
    const int tiles = m_tiles * n_tiles;
    const int max_groups = num_sms / CG;
    const int groups = tiles < max_groups ? tiles : max_groups;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(groups * CG));
    cfg.blockDim = dim3((unsigned)Cfg::kThreads);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmX, tmO2, p));
    if (e) e->launches++;
    return 0;
}

// tmB: box rows = bn / cg.  tmX: EPI_BIAS_RESID_F32 -- f32 [M][ldo] map of the residual/output; f16 epilogues -- f16 [M][ldo] map of the
// output (64 x 32 boxes) and tmO2 the lo tensor of EPI_BIAS_F16_HILO; ignored otherwise
int launch_gemm(vitb200_engine *e, int cg, int bn, int epi, const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmX, const CUtensorMap &tmO2, const GemmParams &p, cudaStream_t s, int num_sms)
{
#define VB_CASE(BN, EPI)                                                                                         \
    if (bn == BN && epi == EPI)                                                                                  \
        return cg == 2 ? launch_gemm_t<BN, EPI, 2>(e, tmA, tmB, tmX, tmO2, p, s, num_sms) : launch_gemm_t<BN, EPI, 1>(e, tmA, tmB, tmX, tmO2, p, s, num_sms);
    if (epi == EPI_PATCH_GATHER_F32) // CTA pairs only (the A producers fill three pipeline stages at a time)
    {
        if (cg != 2) return fail("gathered patch embedding needs cta_group 2");
        return bn == 256 ? launch_gemm_t<256, EPI_PATCH_GATHER_F32, 2>(e, tmA, tmB, tmX, tmO2, p, s, num_sms)
                         : launch_gemm_t<128, EPI_PATCH_GATHER_F32, 2>(e, tmA, tmB, tmX, tmO2, p, s, num_sms);
    }
    if (epi == EPI_BIAS_RESID_F32 && bn == 256 && cg == 2 && p.K >= 2048) // fc2: shallower residual ring, one more operand stage
        return launch_gemm_t<256, EPI_BIAS_RESID_F32, 2, 1>(e, tmA, tmB, tmX, tmO2, p, s, num_sms);
    VB_CASE(256, EPI_BIAS_F16) VB_CASE(128, EPI_BIAS_F16)
    VB_CASE(256, EPI_BIAS_F16_HILO) VB_CASE(128, EPI_BIAS_F16_HILO)
    VB_CASE(256, EPI_BIAS_GELU_F16) VB_CASE(128, EPI_BIAS_GELU_F16)
    VB_CASE(256, EPI_BIAS_RESID_F32) VB_CASE(128, EPI_BIAS_RESID_F32)
    VB_CASE(256, EPI_PATCH_F32) VB_CASE(128, EPI_PATCH_F32)
    VB_CASE(256, EPI_BIAS_F32) VB_CASE(128, EPI_BIAS_F32)
#undef VB_CASE
    return fail("no GEMM instantiation for bn=%d epilogue=%d", bn, epi);
}

int launch_patchify(vitb200_engine *e, const float *img, __half *A, int B, cudaStream_t s)
{
    const long long total = (long long)B * e->G * e->hp.patch_size * e->G;
    const int threads = 256;
    const int blocks = (int)((total + threads - 1) / threads);
    if (e->C == 1)
    {
        if (e->hp.patch_size != 16 && e->hp.patch_size != 8) return fail("1-channel input: patch size %d not supported (8, 16)", e->hp.patch_size);
        if (e->hp.patch_size == 16) patchify_f16_kernel<16, 1><<<blocks, threads, 0, s>>>(img, A, B, e->hp.img_size, e->G, e->KPp);
        else patchify_f16_kernel<8, 1><<<blocks, threads, 0, s>>>(img, A, B, e->hp.img_size, e->G, e->KPp);
        CUDA_TRY(cudaGetLastError());
        e->launches++;
        return 0;
    }
    switch (e->hp.patch_size)
    {
    case 16:
    {
        const int n_patches = B * e->G * e->G; // one warp per patch, grid-stride over a few waves
        const int wblocks = std::min((n_patches + 7) / 8, e->num_sms * 16);
        patchify16_warp_kernel<<<wblocks, 256, 0, s>>>(img, A, n_patches, e->hp.img_size, e->G, e->KPp);
        break;
    }
    case 14: patchify_f16_kernel<14><<<blocks, threads, 0, s>>>(img, A, B, e->hp.img_size, e->G, e->KPp); break;
    case 8: patchify_f16_kernel<8><<<blocks, threads, 0, s>>>(img, A, B, e->hp.img_size, e->G, e->KPp); break;
    case 32: patchify_f16_kernel<32><<<blocks, threads, 0, s>>>(img, A, B, e->hp.img_size, e->G, e->KPp); break;
    default: return fail("patch size %d not supported (8, 14, 16, 32)", e->hp.patch_size);
    }
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return 0;
}

int launch_layernorm(vitb200_engine *e, const float *x, size_t x_row_stride, const float *w, const float *b, __half *y, int rows, cudaStream_t s,
                     int rows_per_group = 0, size_t group_stride = 0)
{
    const int D = e->hp.hidden_size;
    // block LayerNorms (all rows consecutive): the persistent bulk-copy kernel; VITB200_LN_TMA=0 keeps the row-per-warp kernel
    static const bool ln_tma = !(getenv("VITB200_LN_TMA") && atoi(getenv("VITB200_LN_TMA")) == 0);
    // (two CTAs per SM must fit: with one, as for D = 1024, it is slower than the row-per-warp kernel -- 4.98 against 3.9 ms per ViT-L forward)
    if (ln_tma && rows_per_group <= 0 && x_row_stride == (size_t)D && D % 128 == 0 && 2 * (layernorm_tma_smem_bytes(D) + 1024) <= 233472 && rows >= 8)
    {
        const int smem = layernorm_tma_smem_bytes(D);
        const int nblk = (rows + LN_TMA_ROWS - 1) / LN_TMA_ROWS;
        const int grid = std::min(nblk, 2 * e->num_sms);
        auto launch = [&](auto kern) -> int {
            // per kernel instantiation (all of them share this lambda's type: index by D / 128) and per device (one engine per device,
            // possibly several per process)
            static bool attr_set[9][64] = {};
            int dev = 0;
            CUDA_TRY(cudaGetDevice(&dev));
            if (!attr_set[D / 128][dev & 63]) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); attr_set[D / 128][dev & 63] = true; }
            CUDA_TRY(launch_pdl(kern, dim3(grid), dim3(LN_TMA_THREADS), (size_t)smem, s, x, w, b, y, rows, e->hp.eps,
                                (unsigned long long)((l2_hint_mask() & 4) ? ptx::L2_EVICT_FIRST : 0), (unsigned long long)((l2_hint_mask() & 8) ? ptx::L2_EVICT_LAST : 0)));
            return 0;
        };
        int rc = 1;
        switch (D / 128)
        {
        case 1: rc = launch(layernorm_tma_kernel<1>); break;
        case 2: rc = launch(layernorm_tma_kernel<2>); break;
        case 3: rc = launch(layernorm_tma_kernel<3>); break;
        case 4: rc = launch(layernorm_tma_kernel<4>); break;
        case 5: rc = launch(layernorm_tma_kernel<5>); break;
        case 6: rc = launch(layernorm_tma_kernel<6>); break;
        case 7: rc = launch(layernorm_tma_kernel<7>); break;
        case 8: rc = launch(layernorm_tma_kernel<8>); break;
        }
        if (rc) return 1;
        CUDA_TRY(cudaGetLastError());
        e->launches++;
        return 0;
    }
    if (rows_per_group <= 0) rows_per_group = rows > 0 ? rows : 1; // one group: plain consecutive rows
    const int threads = 256, rows_per_block = threads / 32;
    const int blocks = (rows + rows_per_block - 1) / rows_per_block;
    if (D <= 4 * 128) CUDA_TRY(launch_pdl(layernorm_f16_kernel<4>, dim3(blocks), dim3(threads), 0, s, x, x_row_stride, rows_per_group, group_stride, w, b, y, rows, D, e->hp.eps));
    else if (D <= 8 * 128) CUDA_TRY(launch_pdl(layernorm_f16_kernel<8>, dim3(blocks), dim3(threads), 0, s, x, x_row_stride, rows_per_group, group_stride, w, b, y, rows, D, e->hp.eps));
    else if (D <= 16 * 128) CUDA_TRY(launch_pdl(layernorm_f16_kernel<16>, dim3(blocks), dim3(threads), 0, s, x, x_row_stride, rows_per_group, group_stride, w, b, y, rows, D, e->hp.eps));
    else return fail("hidden size %d not supported (max 2048)", D);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return 0;
}

template <int NW>
int launch_attention_t(vitb200_engine *e, int B, cudaStream_t s)
{
    const int N = e->N, D = e->hp.hidden_size, H = e->hp.num_attention_heads;
    const int Npad = (N + ATT_KC - 1) / ATT_KC * ATT_KC;
    const int smem = 2 * Npad * 128;
    auto kern = attention_kernel<NW>;
    static int smem_set[64] = {};
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (smem > smem_set[dev & 63])
    {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        smem_set[dev & 63] = smem;
    }
    kern<<<B * H, NW * 32, smem, s>>>(e->QKV16, (size_t)e->max_batch * N, e->A16, N, D, H, Npad, 1.0f / sqrtf((float)(D / H)));
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return 0;
}

int launch_attention_tc(vitb200_engine *e, int B, cudaStream_t s)
{
    AttnTcParams p{};
    p.N = e->N; p.D = e->hp.hidden_size; p.H = e->hp.num_attention_heads;
    p.n_problems = B * p.H;
    p.NKP = (e->N + 15) / 16 * 16;
    p.n_mtiles = (e->N + 127) / 128;
    p.kv_bytes = (p.NKP * 128 + 1023) / 1024 * 1024;
    p.scale = 1.0f / sqrtf((float)(p.D / p.H));
    p.hilo = e->attn_hilo ? 1 : 0;
    p.load_policy = (l2_hint_mask() & 2) ? ptx::L2_EVICT_FIRST : 0;
    p.reverse = !(getenv("VITB200_ATTN_REVERSE") && atoi(getenv("VITB200_ATTN_REVERSE")) == 0);
    const int smem = attention_tc_smem_bytes(p.kv_bytes);
    static int smem_set[64] = {};
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (smem > smem_set[dev & 63])
    {
        CUDA_TRY(cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        smem_set[dev & 63] = smem;
    }
    const int grid = p.n_problems < e->num_sms ? p.n_problems : e->num_sms;
    // dev knob: VITB200_ATTN_TRACE=<file> dumps the clock64 phase stamps of CTA 0 for the first launch of the process
    static int trace_state = 0; // 0 unknown, 1 armed, 2 done/off
    const char *trace_path = trace_state == 0 ? getenv("VITB200_ATTN_TRACE") : nullptr;
    if (trace_state == 0) trace_state = trace_path ? 1 : 2;
    long long *d_trace = nullptr;
    if (trace_state == 1)
    {
        CUDA_TRY(cudaMalloc(&d_trace, 16 * 32 * sizeof(long long)));
        CUDA_TRY(cudaMemset(d_trace, 0, 16 * 32 * sizeof(long long)));
        p.trace = d_trace;
    }
    CUDA_TRY(launch_pdl(attention_tc_kernel, dim3(grid), dim3(ATT_TC_THREADS), (size_t)smem, s, e->tmQ, e->tmKV,
                        e->attn_hilo ? e->tmQl : e->tmQ, e->attn_hilo ? e->tmKVl : e->tmKV, e->tmAO, p));
    CUDA_TRY(cudaGetLastError());
    if (d_trace)
    {
        std::vector<long long> h(16 * 32);
        CUDA_TRY(cudaStreamSynchronize(s));
        CUDA_TRY(cudaMemcpy(h.data(), d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(d_trace);
        if (FILE *f = fopen(getenv("VITB200_ATTN_TRACE"), "w"))
        {
            for (int i = 0; i < 16; ++i) { for (int j = 0; j < 32; ++j) fprintf(f, "%lld ", h[i * 32 + j]); fprintf(f, "\n"); }
            fclose(f);
        }
        trace_state = 2;
    }
    e->launches++;
    return 0;
}

int launch_attention_tc_long(vitb200_engine *e, int B, cudaStream_t s)
{
    AttnLongParams p{};
    p.N = e->N; p.D = e->hp.hidden_size; p.H = e->hp.num_attention_heads;
    p.n_problems = B * p.H;
    p.NKP = (e->N + 15) / 16 * 16;
    p.kv_rows = (p.NKP + 63) / 64 * 64;
    p.n_tiles = (e->N + 127) / 128;
    {
        const int chunks = (p.NKP + 31) / 32;    // 32-key chunks; a block holds at most 3 (96 TMEM columns)
        p.nb = (chunks + 2) / 3;
        if (p.nb < 2) p.nb = 2;                  // the sweep-B pipeline alternates between two buffers
    }
    p.scale = 1.0f / sqrtf((float)(p.D / p.H));
    p.load_policy = (l2_hint_mask() & 2) ? ptx::L2_EVICT_FIRST : 0;
    if (p.nb > ATT_LONG_MAX_BLOCKS || (p.NKP + 31) / 32 < p.nb)
        return fail("attention: %d tokens cannot be cut into 2..%d key blocks", e->N, ATT_LONG_MAX_BLOCKS);
    for (int j = 0; j < p.nb; ++j) p.key0[j] = att_long_block_key0(p.NKP, p.nb, j);
    p.key0[p.nb] = p.NKP;
    if (p.n_tiles < 2) return fail("two-sweep attention needs at least two query tiles (N > 128)");
    const int smem = attention_tc_long_smem_bytes(p.kv_rows);
    static int smem_set[64] = {};
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (smem > smem_set[dev & 63])
    {
        CUDA_TRY(cudaFuncSetAttribute(attention_tc_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        smem_set[dev & 63] = smem;
    }
    const int grid = p.n_problems < e->num_sms ? p.n_problems : e->num_sms;
    // dev knob: VITB200_ATTN_TRACE=<file> dumps the clock64 phase stamps of CTA 0 (first 16 query tiles) of the first launch of the process
    static int trace_state = 0; // 0 unknown, 1 armed, 2 done/off
    if (trace_state == 0) trace_state = getenv("VITB200_ATTN_TRACE") ? 1 : 2;
    long long *d_trace = nullptr;
    if (trace_state == 1)
    {
        CUDA_TRY(cudaMalloc(&d_trace, 16 * 32 * sizeof(long long)));
        CUDA_TRY(cudaMemset(d_trace, 0, 16 * 32 * sizeof(long long)));
        p.trace = d_trace;
    }
    CUDA_TRY(launch_pdl(attention_tc_long_kernel, dim3(grid), dim3(ATT_LONG_THREADS), (size_t)smem, s, e->tmQ, e->tmKV64, e->tmAO, p));
    if (d_trace)
    {
        std::vector<long long> h(16 * 32);
        CUDA_TRY(cudaStreamSynchronize(s));
        CUDA_TRY(cudaMemcpy(h.data(), d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(d_trace);
        if (FILE *f = fopen(getenv("VITB200_ATTN_TRACE"), "w"))
        {
            for (int i = 0; i < 16; ++i) { for (int j = 0; j < 32; ++j) fprintf(f, "%lld ", h[i * 32 + j]); fprintf(f, "\n"); }
            fclose(f);
        }
        trace_state = 2;
    }
    e->launches++;
    return 0;
}

int launch_attention(vitb200_engine *e, int B, cudaStream_t s)
{
    if (e->attn_tc) return launch_attention_tc(e, B, s);
    if (e->attn_tc_long) return launch_attention_tc_long(e, B, s);
    const int qtiles = (e->N + 15) / 16;
    if (qtiles <= 4) return launch_attention_t<4>(e, B, s);
    if (qtiles <= 14) return launch_attention_t<7>(e, B, s);
    return launch_attention_t<8>(e, B, s);
}

// floats of global scratch the soft-max needs for R rows of C classes: none while a row fits in shared memory
size_t softmax_scratch_floats(int R, int C) { return (size_t)C * sizeof(float) > kSoftmaxSmemMax ? (size_t)R * C : 0; }

// The soft-max / top-k launch of the forward (and of vitb200_test_softmax_topk): one CTA per row of lg ([R][ldl]); the working row
// lives in dynamic shared memory while C floats fit in kSoftmaxSmemMax, and otherwise in `scratch` (softmax_scratch_floats(R, C)
// floats; row r at scratch + r * C).
int launch_softmax_topk(const float *lg, int ldl, float *probs, int32_t *idx, float *val, int R, int C, int k, float *scratch, cudaStream_t s)
{
    const size_t row_bytes = (size_t)C * sizeof(float);
    const bool global_row = row_bytes > kSoftmaxSmemMax;
    if (global_row && !scratch) return fail("soft-max over %d classes needs a global scratch row", C);
    if (!global_row && row_bytes + kSoftmaxStaticSmem > 48 * 1024) // the static arrays count against the default too
    {
        static bool attr_set[64] = {}; // per device
        int dev = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        if (!attr_set[dev & 63])
        {
            CUDA_TRY(cudaFuncSetAttribute(softmax_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSoftmaxSmemMax));
            attr_set[dev & 63] = true;
        }
    }
    softmax_topk_kernel<<<R, 256, global_row ? 0 : row_bytes, s>>>(lg, ldl, probs, idx, val, C, k, global_row ? scratch : nullptr);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// D2H helpers for the debug taps
int tap_f32(float *dst, const float *src, size_t n, cudaStream_t s)
{
    if (!dst) return 0;
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaMemcpy(dst, src, n * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
}
int tap_f16(float *dst, const __half *src, size_t n, cudaStream_t s, const __half *lo = nullptr)
{
    if (!dst) return 0;
    CUDA_TRY(cudaStreamSynchronize(s));
    std::vector<__half> tmp(n);
    CUDA_TRY(cudaMemcpy(tmp.data(), src, n * sizeof(__half), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; ++i) dst[i] = __half2float(tmp[i]);
    if (lo) // split-precision tensor: value = hi + lo
    {
        CUDA_TRY(cudaMemcpy(tmp.data(), lo, n * sizeof(__half), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < n; ++i) dst[i] += __half2float(tmp[i]);
    }
    return 0;
}

// debug tap of the q | k | v activations in the reference's [tokens][3 D] order (the device buffers are head-major: [3 H][rows][64])
int tap_qkv(vitb200_engine *e, float *dst, int T, cudaStream_t s)
{
    if (!dst) return 0;
    const int D = e->hp.hidden_size, H = e->hp.num_attention_heads;
    const size_t plane_rows = (size_t)e->max_batch * e->N, n = (size_t)3 * H * plane_rows * 64;
    std::vector<float> tmp(n);
    if (tap_f16(tmp.data(), e->QKV16, n, s, e->attn_hilo ? e->QKV16L : nullptr)) return 1;
    for (int t = 0; t < T; ++t)
        for (int pl = 0; pl < 3 * H; ++pl)
            memcpy(dst + (size_t)t * 3 * D + (size_t)pl * 64, tmp.data() + ((size_t)pl * plane_rows + t) * 64, 64 * sizeof(float));
    return 0;
}

// The fixed kernel schedule == reference vit_encode_image (vit.cpp:718-941), batched over images.
int run_forward(vitb200_engine *e, const float *d_images, int B, float *d_probs, float *d_logits, int32_t *d_topk_idx,
                float *d_topk_val, int k, cudaStream_t s, const vitb200_taps *taps)
{
    if (B < 1 || B > e->max_batch) return fail("batch %d out of range (1..%d)", B, e->max_batch);
    if (k < 0 || k > e->max_k) return fail("k %d out of range (0..%d)", k, e->max_k);
    if (!d_images && taps) return fail("debug taps need the f32 image path");
    const int D = e->hp.hidden_size, N = e->N, T = B * N, C = e->hp.num_classes;
    e->launches = 0;
    __half *PA = e->PA;
    // the epilogues store whole boxes with TMA (and the residual epilogue read-modify-writes 32-row boxes of X): with maps of exactly T
    // rows the rows of the last M tile that lie past the batch are zero-filled on load and clipped on store
    auto bm = e->batch_maps.find(B);
    if (bm == e->batch_maps.end())
    {
        vitb200_engine::BatchMaps m;
        memset(&m, 0, sizeof(m));
        if (make_tmap_f32_box32(&m.X, e->X, (uint64_t)T, (uint64_t)D, (uint64_t)D) ||
            make_tmap_heads3d(&m.QKVh, e->QKV16, 3 * (uint64_t)e->hp.num_attention_heads, (uint64_t)T, (uint64_t)e->max_batch * N, 32) ||
            (e->QKV16L && make_tmap_heads3d(&m.QKVl, e->QKV16L, 3 * (uint64_t)e->hp.num_attention_heads, (uint64_t)T, (uint64_t)e->max_batch * N, 32)) ||
            make_tmap(&m.H, e->H16, (uint64_t)T, 4 * (uint64_t)D, 4 * (uint64_t)D, 32))
            return 1;
        bm = e->batch_maps.emplace(B, m).first;
    }
    const CUtensorMap &tmX = bm->second.X, &tmQKVh = bm->second.QKVh, &tmQKVl = bm->second.QKVl, &tmH = bm->second.H;

    // patch embedding (vit.cpp:772-797): the f16 patch matrix PA (im2col of a stride == kernel conv is a pure permutation,
    // ggml.c:11528-11608) is either already there (d_images == NULL: the u8 path's preprocess kernel wrote it) or written by
    // patchify (one warp per patch, coalesced); the TMA-fed GEMM adds conv bias + pos_embed and writes token rows.
    // VITB200_PATCH_GATHER=1 (P = 16, CTA pairs, 3 channels) selects the single-kernel variant whose A producers gather the f32
    // pixels straight into the operand tiles: no patch matrix, but its dependent 128-bit loads are L2-latency bound on an SM with no
    // L1 left (0.29 ms against 0.05 + 0.10 ms at batch 256, profiles/), so it is no longer the default.
    const bool patches_ready = d_images == nullptr;
    const bool fused_patch = !patches_ready && e->hp.patch_size == 16 && e->cta_group == 2 && e->C == 3 &&
                             getenv("VITB200_PATCH_GATHER") && atoi(getenv("VITB200_PATCH_GATHER")) == 1;
    {
        GemmParams p{};
        p.M = B * e->NP; p.N = D; p.K = e->KPp; p.bias = e->patch.b; p.out = e->X; p.ldo = D;
        p.pos = e->pos; p.np = e->NP; p.ntok = N;
        p.img = d_images; p.S = e->hp.img_size; p.G = e->G;
        ProfScope ps(e, PK_PATCH, 2.0 * p.M * p.N * e->KP, s);
        if (!patches_ready && !fused_patch && launch_patchify(e, d_images, PA, B, s)) return 1;
        {
            const int n = B * D, threads = 256;
            cls_rows_kernel<<<(n + threads - 1) / threads, threads, 0, s>>>(e->X, e->cls, e->pos, B, N, D);
            CUDA_TRY(cudaGetLastError());
            e->launches++;
        }
        if (launch_gemm(e, e->cta_group, e->patch.bn, fused_patch ? EPI_PATCH_GATHER_F32 : EPI_PATCH_F32, e->tmA_P, e->patch.tm, tmX, tmX, p, s, e->num_sms)) return 1;
    }
    if (taps && tap_f32(taps->embed, e->X, (size_t)T * D, s)) return 1;

    const int n_layers = e->hp.num_hidden_layers;
    for (int il = 0; il < n_layers; ++il)
    {
        const Layer &L = e->layers[il];
        const bool tap = taps && taps->layer == il;
        // LayerNorm 1 (vit.cpp:808-812): a kernel of its own only in front of the first block -- with fused_ln the fc2 epilogue of
        // the previous block has already left norm1(x) of this block in A16
        if (il == 0 || !e->fused_ln)
        {
            ProfScope ps(e, PK_LN, 0.0, s);
            if (launch_layernorm(e, e->X, (size_t)D, L.n1w, L.n1b, e->A16, T, s)) return 1;
            if (tap && tap_f16(taps->ln1, e->A16, (size_t)T * D, s)) return 1;
        }
        {
            GemmParams p{};
            p.M = T; p.N = 3 * D; p.K = D; p.bias = L.qkv.b; p.out = e->QKV16; p.out2 = e->QKV16L; p.ldo = 3 * D; p.headmajor = 1; p.store_policy = (l2_hint_mask() & 1) ? ptx::L2_EVICT_FIRST : 0;
            ProfScope ps(e, PK_QKV, 2.0 * p.M * p.N * p.K, s);
            if (launch_gemm(e, e->cta_group, L.qkv.bn, e->attn_hilo ? EPI_BIAS_F16_HILO : EPI_BIAS_F16, e->tmA_D, L.qkv.tm, tmQKVh, tmQKVl, p, s, e->num_sms)) return 1; // vit.cpp:820-821
        }
        if (tap && tap_qkv(e, taps->qkv, T, s)) return 1;
        {
            ProfScope ps(e, PK_ATTN, 4.0 * B * e->hp.num_attention_heads * (double)N * N * 64, s);
            if (launch_attention(e, B, s)) return 1; // vit.cpp:826-866
        }
        if (tap && tap_f16(taps->attn, e->A16, (size_t)T * D, s)) return 1;
        {
            // proj + residual (vit.cpp:868-873); fused: + LayerNorm 2 (vit.cpp:881-885) of each 32-row group as its last column tile
            // lands, written over the attention output in A16 (every tile that read those rows has finished its MMAs by then)
            GemmParams p{};
            p.M = T; p.N = D; p.K = D; p.bias = L.proj.b; p.out = e->X; p.ldo = D; p.resid = e->X;
            if (e->fused_ln) { p.ln_out = e->A16; p.ln_w = L.n2w; p.ln_b = L.n2b; p.ln_count = e->d_ln_count; p.ln_eps = e->hp.eps; p.ln_dbg = getenv("VITB200_LN_DBG") ? atoi(getenv("VITB200_LN_DBG")) : 0; }
            ProfScope ps(e, PK_PROJ, 2.0 * p.M * p.N * p.K, s);
            if (launch_gemm(e, e->cta_group, L.proj.bn, EPI_BIAS_RESID_F32, e->tmA_D, L.proj.tm, tmX, tmX, p, s, e->num_sms)) return 1;
        }
        if (tap && tap_f32(taps->x1, e->X, (size_t)T * D, s)) return 1;
        if (!e->fused_ln)
        {
            ProfScope ps(e, PK_LN, 0.0, s);
            if (launch_layernorm(e, e->X, (size_t)D, L.n2w, L.n2b, e->A16, T, s)) return 1; // vit.cpp:881-885
        }
        if (tap && tap_f16(taps->ln2, e->A16, (size_t)T * D, s)) return 1;
        {
            GemmParams p{};
            p.M = T; p.N = 4 * D; p.K = D; p.bias = L.fc1.b; p.out = e->H16; p.ldo = 4 * D; p.store_policy = (l2_hint_mask() & 1) ? ptx::L2_EVICT_FIRST : 0;
            ProfScope ps(e, PK_FC1, 2.0 * p.M * p.N * p.K, s);
            if (launch_gemm(e, e->cta_group, L.fc1.bn, EPI_BIAS_GELU_F16, e->tmA_D, L.fc1.tm, tmH, tmH, p, s, e->num_sms)) return 1; // vit.cpp:889-893
        }
        if (tap && tap_f16(taps->h, e->H16, (size_t)T * 4 * D, s)) return 1;
        {
            // fc2 + residual (vit.cpp:896-900); fused: + LayerNorm 1 of the NEXT block (the last block's output goes to the pooled
            // final LayerNorm instead)
            GemmParams p{};
            p.M = T; p.N = D; p.K = 4 * D; p.bias = L.fc2.b; p.out = e->X; p.ldo = D; p.resid = e->X;
            if (e->fused_ln && il + 1 < n_layers)
            {
                const Layer &Ln = e->layers[il + 1];
                p.ln_out = e->A16; p.ln_w = Ln.n1w; p.ln_b = Ln.n1b; p.ln_count = e->d_ln_count; p.ln_eps = e->hp.eps;
                p.ln_dbg = getenv("VITB200_LN_DBG") ? atoi(getenv("VITB200_LN_DBG")) : 0;
            }
            ProfScope ps(e, PK_FC2, 2.0 * p.M * p.N * p.K, s);
            if (launch_gemm(e, e->cta_group, L.fc2.bn, EPI_BIAS_RESID_F32, e->tmA_H, L.fc2.tm, tmX, tmX, p, s, e->num_sms)) return 1;
        }
        if (tap && tap_f32(taps->x2, e->X, (size_t)T * D, s)) return 1;
        if (e->fused_ln && taps && taps->layer == il + 1 && tap_f16(taps->ln1, e->A16, (size_t)T * D, s)) return 1; // norm1 of the next block
    }
    if (taps && tap_f32(taps->x_final, e->X, (size_t)T * D, s)) return 1;

    // pool (token 0; the first 25 tokens for ViTSTR, vitstr.cpp:864-883) + final LN + head + soft-max + top-k
    // (vit.cpp:910-933, 1047-1057); one row of the head GEMM / one soft-max per pooled token
    const int TH = e->head_tokens, R = B * TH;
    if (launch_layernorm(e, e->X, (size_t)D, e->norm_w, e->norm_b, e->CLS16, R, s, TH, (size_t)N * D)) return 1;
    if (taps && tap_f16(taps->final_ln, e->CLS16, (size_t)R * D, s)) return 1;
    // internal logits rows have pitch Cp (num_classes padded to 4; the padded W rows are TMA zero fill, the padded bias is 0);
    // a caller's dense [rows][num_classes] buffer is written directly when the two coincide, else through a 2-D copy
    const int Cp = e->Cp;
    float *lg = (d_logits && Cp == C) ? d_logits : e->d_logits;
    {
        GemmParams p{};
        p.M = R; p.N = Cp; p.K = D; p.bias = e->head.b; p.out = lg; p.ldo = Cp;
        ProfScope ps(e, PK_HEAD, 2.0 * p.M * C * p.K, s);
        if (launch_gemm(e, e->cta_group, e->head.bn, EPI_BIAS_F32, e->tmA_C, e->head.tm, tmX, tmX, p, s, e->num_sms)) return 1;
    }
    if (d_logits && lg != d_logits)
        CUDA_TRY(cudaMemcpy2DAsync(d_logits, (size_t)C * 4, lg, (size_t)Cp * 4, (size_t)C * 4, (size_t)R, cudaMemcpyDeviceToDevice, s));
    if (d_probs || (k > 0 && (d_topk_idx || d_topk_val)))
    {
        if (launch_softmax_topk(lg, Cp, d_probs, d_topk_idx, d_topk_val, R, C, k, e->d_sm_scratch, s)) return 1;
        e->launches++;
    }
    return 0;
}

// run_forward through a cached CUDA graph: the first call with a given argument set runs eagerly (also sets the kernels'
// function attributes), the second captures + instantiates, later ones replay.  Profiling / taps always run eagerly.
int run_forward_graphed(vitb200_engine *e, const float *d_images, int B, float *d_probs, float *d_logits, int32_t *d_topk_idx,
                        float *d_topk_val, int k, cudaStream_t s)
{
    // Graph replay pays off where the ~90 launches are a visible fraction of the step (small batches); at B = 256 every kernel
    // runs >= 80 us and eager launches stay ahead of the GPU (measured: no gain), so large batches launch eagerly.
    if (!e->use_graph || e->profile || (long long)B * e->N > 8192) return run_forward(e, d_images, B, d_probs, d_logits, d_topk_idx, d_topk_val, k, s, nullptr);
    vitb200_engine::GraphEntry *g = nullptr;
    for (auto &x : e->graphs)
        if (x.img == d_images && x.batch == B && x.probs == d_probs && x.logits == d_logits && x.tidx == d_topk_idx && x.tval == d_topk_val && x.k == k) { g = &x; break; }
    if (!g)
    {
        if (e->graphs.size() >= 16) { if (e->graphs.front().exec) cudaGraphExecDestroy(e->graphs.front().exec); e->graphs.erase(e->graphs.begin()); }
        e->graphs.push_back({d_images, B, d_probs, d_logits, d_topk_idx, d_topk_val, k, 0, 0, nullptr});
        g = &e->graphs.back();
    }
    if (g->state == 0)
    {
        if (run_forward(e, d_images, B, d_probs, d_logits, d_topk_idx, d_topk_val, k, s, nullptr)) return 1;
        g->state = 1;
        g->launches = e->launches;
        return 0;
    }
    if (g->state == 1)
    {
        cudaGraph_t graph = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        const int rc = run_forward(e, d_images, B, d_probs, d_logits, d_topk_idx, d_topk_val, k, s, nullptr);
        cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (rc != 0 || ce != cudaSuccess || !graph)
        {
            if (graph) cudaGraphDestroy(graph);
            (void)cudaGetLastError();
            g->state = 0;
            e->use_graph = false; // fall back to eager launches (same kernels, same results)
            return run_forward(e, d_images, B, d_probs, d_logits, d_topk_idx, d_topk_val, k, s, nullptr);
        }
        g->launches = e->launches;
        ce = cudaGraphInstantiate(&g->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { g->exec = nullptr; g->state = 0; e->use_graph = false; return fail("cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
        g->state = 2;
    }
    CUDA_TRY(cudaGraphLaunch(g->exec, s));
    e->launches = g->launches;
    return 0;
}

} // namespace

extern "C" {

const char *vitb200_last_error(void) { return g_err.c_str(); }

int vitb200_create(const vitb200_hparams *hp, const vitb200_tensor *t, int n, int device, int max_batch, vitb200_engine **out)
{
    return vitb200_create_ex(hp, t, n, device, max_batch, 1, out);
}

// The C ABI promises "non-zero return, never abort": nothing may unwind through an extern "C" frame.  Host-side allocations
// (std::vector staging buffers sized from a model file) can throw; every entry point that owns such code runs it through this.
#define VB_NOEXCEPT_BEGIN try {
#define VB_NOEXCEPT_END(cleanup)                                                                          \
    } catch (const std::exception &ex) { cleanup; return fail("%s: %s", __func__, ex.what()); }            \
    catch (...) { cleanup; return fail("%s: unknown exception", __func__); }

static int create_impl(const vitb200_hparams *hp, const vitb200_tensor *t, int n, int device, int max_batch, int head_tokens,
                       vitb200_engine *&e, vitb200_engine **out);

int vitb200_create_ex(const vitb200_hparams *hp, const vitb200_tensor *t, int n, int device, int max_batch, int head_tokens,
                      vitb200_engine **out)
{
    if (!hp || !t || !out) return fail("vitb200_create: null argument");
    *out = nullptr;
    vitb200_engine *e = nullptr;
    VB_NOEXCEPT_BEGIN
    return create_impl(hp, t, n, device, max_batch, head_tokens, e, out);
    VB_NOEXCEPT_END(if (e) vitb200_destroy(e))
}

static int create_impl(const vitb200_hparams *hp, const vitb200_tensor *t, int n, int device, int max_batch, int head_tokens,
                       vitb200_engine *&e, vitb200_engine **out)
{
    // hyper-parameter sanity first (no division by a field a corrupt file may have zeroed; no device needed to reject them)
    if (hp->hidden_size < 64 || hp->hidden_size > 8192 || hp->num_hidden_layers < 1 || hp->num_hidden_layers > 4096 ||
        hp->num_attention_heads < 1 || hp->num_attention_heads > 128 || hp->num_classes < 1 || hp->num_classes > (1 << 20) ||
        hp->patch_size < 1 || hp->patch_size > 64 || hp->img_size < hp->patch_size || hp->img_size > 4096 || n < 1)
        return fail("invalid hyper-parameters (hidden %d, layers %d, heads %d, classes %d, patch %d, img %d)", hp->hidden_size,
                    hp->num_hidden_layers, hp->num_attention_heads, hp->num_classes, hp->patch_size, hp->img_size);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("no CUDA device: the vit.cpp_b200 forward path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    if (hp->hidden_size % hp->num_attention_heads != 0 || hp->hidden_size / hp->num_attention_heads != 64)
        return fail("head dim %d not supported (64 only)", hp->num_attention_heads ? hp->hidden_size / hp->num_attention_heads : 0);
    if (hp->hidden_size % 64 != 0) return fail("hidden size %d must be a multiple of 64", hp->hidden_size);
    if (hp->img_size % hp->patch_size != 0) return fail("img_size %d not a multiple of patch_size %d", hp->img_size, hp->patch_size);
    if (max_batch < 1) return fail("max_batch must be >= 1");
    if (check_unique_names(t, n)) return 1;

    e = new vitb200_engine();
    e->hp = *hp;
    if (e->hp.eps <= 0.f) e->hp.eps = 1e-6f;
    e->device = device;
    e->max_batch = max_batch;
    e->num_sms = prop.multiProcessorCount;
    const int D = hp->hidden_size, P = hp->patch_size;
    e->G = hp->img_size / P;
    e->NP = e->G * e->G;
    e->N = e->NP + 1;
    {
        // input channels from the patch kernel [P, P, C, D] (vit.cpp:515; C = 1 in vitstr.cpp:482)
        const vitb200_tensor *pw = find_tensor(t, n, "patch_embed.proj.weight");
        const int64_t per_c = (int64_t)D * P * P;
        if (!pw || nelem(pw) % per_c != 0 || (nelem(pw) / per_c != 1 && nelem(pw) / per_c != 3))
        {
            delete e;
            e = nullptr;
            return fail("tensor 'patch_embed.proj.weight' is missing or is not a 1- or 3-channel %dx%d kernel", P, P);
        }
        e->C = (int)(nelem(pw) / per_c);
    }
    if (head_tokens < 1 || head_tokens > e->N) { const int ntok = e->N; delete e; e = nullptr; return fail("head_tokens %d out of range (1..%d)", head_tokens, ntok); }
    e->head_tokens = head_tokens;
    e->Cp = (hp->num_classes + 3) / 4 * 4;
    e->KP = e->C * P * P;
    e->KPp = (e->KP + 63) / 64 * 64;
    e->cta_group = (getenv("VITB200_CTA_GROUP") && atoi(getenv("VITB200_CTA_GROUP")) == 1) ? 1 : 2;
    e->use_graph = !(getenv("VITB200_GRAPH") && atoi(getenv("VITB200_GRAPH")) == 0);
    auto bail = [&](int) { vitb200_destroy(e); e = nullptr; return 1; };
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail("cudaStreamCreate failed"));

    // ---- weights (names: reference vit.cpp:518-579)
    if (upload_f32(e, t, n, "cls_token", D, 1, 1, 1, &e->cls)) return bail(1);
    if (upload_f32(e, t, n, "pos_embed", D, e->N, 1, 1, &e->pos)) return bail(1);
    if (upload_linear(e, t, n, "patch_embed.proj.weight", "patch_embed.proj.bias", D, e->KP, e->KPp, &e->patch, P)) return bail(1);
    e->layers.resize(hp->num_hidden_layers);
    for (int i = 0; i < hp->num_hidden_layers; ++i)
    {
        Layer &L = e->layers[i];
        const std::string p = "blocks." + std::to_string(i) + ".";
        if (upload_f32(e, t, n, p + "norm1.weight", D, 1, 1, 1, &L.n1w) || upload_f32(e, t, n, p + "norm1.bias", D, 1, 1, 1, &L.n1b) ||
            upload_f32(e, t, n, p + "norm2.weight", D, 1, 1, 1, &L.n2w) || upload_f32(e, t, n, p + "norm2.bias", D, 1, 1, 1, &L.n2b))
            return bail(1);
        if (upload_linear(e, t, n, p + "attn.qkv.weight", p + "attn.qkv.bias", 3 * D, D, D, &L.qkv) ||
            upload_linear(e, t, n, p + "attn.proj.weight", p + "attn.proj.bias", D, D, D, &L.proj) ||
            upload_linear(e, t, n, p + "mlp.fc1.weight", p + "mlp.fc1.bias", 4 * D, D, D, &L.fc1) ||
            upload_linear(e, t, n, p + "mlp.fc2.weight", p + "mlp.fc2.bias", D, 4 * D, 4 * D, &L.fc2))
            return bail(1);
    }
    if (upload_f32(e, t, n, "norm.weight", D, 1, 1, 1, &e->norm_w) || upload_f32(e, t, n, "norm.bias", D, 1, 1, 1, &e->norm_b)) return bail(1);
    if (upload_linear(e, t, n, "head.weight", "head.bias", hp->num_classes, D, D, &e->head)) return bail(1);

    // ---- activation arena
    const size_t B = (size_t)max_batch, T = B * e->N;
    const size_t h16 = T * 4 * D;
    // The patch matrix [B*NP][KPp] aliases the MLP hidden buffer (dead while the patch GEMM runs) when it fits and
    // has no K padding; otherwise it gets its own buffer whose zeroed padding columns are never written again.
    const size_t pa_elems = B * e->NP * e->KPp;
    const bool pa_alias = (e->KPp == e->KP) && pa_elems <= h16;
    const size_t R = B * (size_t)e->head_tokens;                        // classifier rows: pooled tokens of all images
    const size_t img_elems = (size_t)e->C * hp->img_size * hp->img_size; // per image
    if (dev_alloc(e, &e->d_img, B * img_elems) || dev_alloc(e, &e->X, T * D) ||
        dev_alloc(e, &e->A16, T * D) || dev_alloc(e, &e->QKV16, T * 3 * D) || dev_alloc(e, &e->H16, h16) ||
        dev_alloc(e, &e->CLS16, R * D) || dev_alloc(e, &e->d_logits, R * e->Cp) || dev_alloc(e, &e->d_logits_slot[0], R * hp->num_classes) ||
        dev_alloc(e, &e->d_probs, R * hp->num_classes) || dev_alloc(e, &e->d_topk_idx, R * e->max_k) ||
        dev_alloc(e, &e->d_topk_val, R * e->max_k))
        return bail(1);
    e->d_img_slot[0] = e->d_img; e->d_probs_slot[0] = e->d_probs;
    {
        // soft-max working rows in global memory when a row does not fit in shared memory (launch_softmax_topk)
        const size_t n_scratch = softmax_scratch_floats((int)R, hp->num_classes);
        if (n_scratch && dev_alloc(e, &e->d_sm_scratch, n_scratch)) return bail(1);
    }
    e->d_topk_idx_slot[0] = e->d_topk_idx; e->d_topk_val_slot[0] = e->d_topk_val;
    if (dev_alloc(e, &e->d_img_slot[1], B * img_elems) || dev_alloc(e, &e->d_probs_slot[1], R * hp->num_classes) ||
        dev_alloc(e, &e->d_logits_slot[1], R * hp->num_classes) || dev_alloc(e, &e->d_topk_idx_slot[1], R * e->max_k) ||
        dev_alloc(e, &e->d_topk_val_slot[1], R * e->max_k))
        return bail(1);
    if (cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail("cudaStreamCreate failed"));
    for (int i = 0; i < 2; ++i)
        if (cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&e->ev_done[i], cudaEventDisableTiming) != cudaSuccess)
            return bail(fail("cudaEventCreate failed"));
    {
        // Fused LayerNorm (residual epilogue + dedicated LayerNorm warps, gemm_tcgen05.cuh): bit-identical to the stand-alone kernel but
        // SLOWER on B200 at batch 256 (proj + LN 2.78 ms vs 1.15 + 0.60 ms per forward, DESIGN.md section 3), so it is opt-in
        // (VITB200_FUSED_LN=1).  It needs the whole row in N % 128 == 0 float4-per-lane form and w, b in shared memory.
        const bool want = getenv("VITB200_FUSED_LN") && atoi(getenv("VITB200_FUSED_LN")) == 1;
        e->fused_ln = want && D % 128 == 0 && D <= 1024;
        if (e->fused_ln && dev_alloc(e, &e->d_ln_count, (T + 255) / 256 * 8 + 8)) return bail(1);
    }
    if (pa_alias) e->PA = e->H16;
    else
    {
        if (dev_alloc(e, &e->PA, pa_elems)) return bail(1);
        if (cudaMemset(e->PA, 0, pa_elems * sizeof(__half)) != cudaSuccess) return bail(fail("cudaMemset failed"));
    }
    if (make_tmap(&e->tmA_D, e->A16, T, D, D, GEMM_BM) || make_tmap(&e->tmA_H, e->H16, T, 4 * (uint64_t)D, 4 * (uint64_t)D, GEMM_BM) ||
        make_tmap(&e->tmA_P, e->PA, B * e->NP, e->KPp, e->KPp, GEMM_BM) || make_tmap(&e->tmA_C, e->CLS16, R, D, D, GEMM_BM))
        return bail(1);
    {
        const char *force = getenv("VITB200_ATTENTION"); // bring-up knob: "mma" forces the warp-MMA kernel
        const bool force_mma = force && strcmp(force, "mma") == 0;
        e->attn_tc = e->N <= 224 && !force_mma;
        e->attn_tc_long = e->N > 224 && e->N <= ATT_LONG_MAX_KEYS && !force_mma;
        if (e->attn_tc_long)
        {
            if (make_tmap_heads3d(&e->tmQ, e->QKV16, 3 * (uint64_t)hp->num_attention_heads, T, T, 128) ||
                make_tmap_heads3d(&e->tmKV64, e->QKV16, 3 * (uint64_t)hp->num_attention_heads, T, T, 64) ||
                make_tmap_tokens3d(&e->tmAO, e->A16, (uint64_t)B, (uint64_t)e->N, (uint64_t)D))
                return bail(1);
        }
        if (e->attn_tc)
        {
            const int NKP = (e->N + 15) / 16 * 16;
            if (make_tmap_heads3d(&e->tmQ, e->QKV16, 3 * (uint64_t)hp->num_attention_heads, T, T, 128) ||
                make_tmap_heads3d(&e->tmKV, e->QKV16, 3 * (uint64_t)hp->num_attention_heads, T, T, (uint32_t)NKP) ||
                make_tmap_tokens3d(&e->tmAO, e->A16, (uint64_t)B, (uint64_t)e->N, (uint64_t)D))
                return bail(1);
            // split-precision q, k, v (reference: f32 operands, vit.cpp:848,858); VITB200_ATTN_HILO=0 keeps the f16-only operands
            e->attn_hilo = !(getenv("VITB200_ATTN_HILO") && atoi(getenv("VITB200_ATTN_HILO")) == 0);
            if (e->attn_hilo)
            {
                if (dev_alloc(e, &e->QKV16L, T * 3 * D) ||
                    make_tmap_heads3d(&e->tmQl, e->QKV16L, 3 * (uint64_t)hp->num_attention_heads, T, T, 128) ||
                    make_tmap_heads3d(&e->tmKVl, e->QKV16L, 3 * (uint64_t)hp->num_attention_heads, T, T, (uint32_t)NKP))
                    return bail(1);
            }
        }
    }
    if (cudaDeviceSynchronize() != cudaSuccess) return bail(fail("device sync after upload failed"));
    *out = e;
    e = nullptr; // ownership passed to the caller
    return 0;
}

void vitb200_destroy(vitb200_engine *e)
{
    if (!e) return;
    cudaSetDevice(e->device);
    for (void *p : e->allocs) cudaFree(p);
    for (auto &g : e->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    for (int i = 0; i < 2; ++i) { if (e->d_u8[i]) cudaFree(e->d_u8[i]); if (e->h_u8[i]) cudaFreeHost(e->h_u8[i]); }
    for (auto &r : e->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto ev : e->event_pool) cudaEventDestroy(ev);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    for (int i = 0; i < 2; ++i) { if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]); if (e->ev_done[i]) cudaEventDestroy(e->ev_done[i]); }
    delete e;
}

int vitb200_get_hparams(const vitb200_engine *e, vitb200_hparams *out)
{
    if (!e || !out) return fail("null argument");
    *out = e->hp;
    return 0;
}

const char *vitb200_label(const vitb200_engine *e, int class_id)
{
    if (!e) return nullptr;
    auto it = e->labels.find(class_id);
    return it == e->labels.end() ? nullptr : it->second.c_str();
}

int vitb200_last_launch_count(const vitb200_engine *e) { return e ? e->launches : 0; }
int vitb200_in_chans(const vitb200_engine *e) { return e ? e->C : 0; }
int vitb200_head_tokens(const vitb200_engine *e) { return e ? e->head_tokens : 0; }

int vitb200_profile_enable(vitb200_engine *e, int on)
{
    if (!e) return fail("null argument");
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaDeviceSynchronize());
    for (auto &r : e->prof) { e->event_pool.push_back(r.a); e->event_pool.push_back(r.b); }
    e->prof.clear();
    e->profile = on != 0;
    return 0;
}

int vitb200_profile_read(vitb200_engine *e, int kind, double *ms_total, int *launches, double *flops_per_launch)
{
    if (!e || !ms_total || !launches || !flops_per_launch) return fail("null argument");
    if (kind < 0 || kind >= PK_COUNT) return fail("profile kind %d out of range", kind);
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaDeviceSynchronize());
    double ms = 0.0, fl = 0.0;
    int n = 0;
    for (auto &r : e->prof)
    {
        if (r.kind != kind) continue;
        float t = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&t, r.a, r.b));
        ms += t; fl = r.flops; ++n;
    }
    *ms_total = ms; *launches = n; *flops_per_launch = fl;
    return 0;
}
static int test_attention_impl(int device, int kernel, int B, int N, int H, const uint16_t *qkv, const uint16_t *qkv_lo, float *out);

int vitb200_test_attention(int device, int kernel, int B, int N, int H, const uint16_t *qkv, float *out)
{
    VB_NOEXCEPT_BEGIN
    return test_attention_impl(device, kernel, B, N, H, qkv, nullptr, out);
    VB_NOEXCEPT_END((void)0)
}

int vitb200_test_attention_hilo(int device, int B, int N, int H, const uint16_t *qkv_hi, const uint16_t *qkv_lo, float *out)
{
    if (!qkv_lo) return fail("bad argument");
    VB_NOEXCEPT_BEGIN
    return test_attention_impl(device, 2, B, N, H, qkv_hi, qkv_lo, out);
    VB_NOEXCEPT_END((void)0)
}

static int test_attention_impl(int device, int kernel, int B, int N, int H, const uint16_t *qkv, const uint16_t *qkv_lo, float *out)
{
    if (!qkv || !out || B < 1 || N < 1 || H < 1) return fail("bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("no CUDA device: the vit.cpp_b200 forward path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    vitb200_engine *e = new vitb200_engine();
    e->device = device;
    auto bail = [&](int rc) { vitb200_destroy(e); return rc; };
    e->num_sms = prop.multiProcessorCount;
    e->N = N; e->hp.hidden_size = H * 64; e->hp.num_attention_heads = H; e->max_batch = B;
    const int D = H * 64;
    const uint64_t T = (uint64_t)B * N;
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail("stream creation failed"));
    if (dev_alloc(e, &e->QKV16, (size_t)T * 3 * D) || dev_alloc(e, &e->A16, (size_t)T * D)) return bail(1);
    // the kernels read the HEAD-MAJOR layout the qkv GEMM writes ([3 H][T][64]); the caller hands over the reference's [T][3 D]
    std::vector<uint16_t> hm((size_t)T * 3 * D);
    auto to_head_major = [&](const uint16_t *src) {
        for (uint64_t t = 0; t < T; ++t)
            for (int pl = 0; pl < 3 * H; ++pl)
                memcpy(&hm[((size_t)pl * T + t) * 64], src + (size_t)t * 3 * D + (size_t)pl * 64, 128);
    };
    to_head_major(qkv);
    if (cudaMemcpy(e->QKV16, hm.data(), (size_t)T * 3 * D * 2, cudaMemcpyHostToDevice) != cudaSuccess) return bail(fail("H2D failed"));
    if (qkv_lo)
    {
        if (N > 224) return bail(fail("split-precision attention needs N <= 224"));
        if (dev_alloc(e, &e->QKV16L, (size_t)T * 3 * D)) return bail(1);
        to_head_major(qkv_lo);
        if (cudaMemcpy(e->QKV16L, hm.data(), (size_t)T * 3 * D * 2, cudaMemcpyHostToDevice) != cudaSuccess) return bail(fail("H2D failed"));
        e->attn_hilo = true;
    }
    // cudaMemcpy from pageable memory may return before the DMA has landed, and the kernels below run on a NON-BLOCKING stream (no implicit
    // ordering with the legacy stream the copies used): wait for the device before launching
    if (cudaDeviceSynchronize() != cudaSuccess) return bail(fail("device sync after upload failed"));
    if (kernel == 0) kernel = N <= 224 ? 2 : (N <= ATT_LONG_MAX_KEYS ? 3 : 1);
    if (kernel == 2 && N > 224) return bail(fail("tcgen05 single-block attention needs N <= 224"));
    if (kernel == 3 && (N <= 128 || N > ATT_LONG_MAX_KEYS)) return bail(fail("tcgen05 two-sweep attention needs 128 < N <= %d", ATT_LONG_MAX_KEYS));
    e->attn_tc = kernel == 2;
    e->attn_tc_long = kernel == 3;
    if (kernel >= 2)
    {
        const int NKP = (N + 15) / 16 * 16;
        if (make_tmap_heads3d(&e->tmQ, e->QKV16, 3 * (uint64_t)H, T, T, 128) ||
            make_tmap_heads3d(&e->tmKV, e->QKV16, 3 * (uint64_t)H, T, T, (uint32_t)(NKP <= 224 ? NKP : 64)) ||
            make_tmap_heads3d(&e->tmKV64, e->QKV16, 3 * (uint64_t)H, T, T, 64) ||
            make_tmap_tokens3d(&e->tmAO, e->A16, (uint64_t)B, (uint64_t)N, (uint64_t)D))
            return bail(1);
        if (qkv_lo && (make_tmap_heads3d(&e->tmQl, e->QKV16L, 3 * (uint64_t)H, T, T, 128) ||
                       make_tmap_heads3d(&e->tmKVl, e->QKV16L, 3 * (uint64_t)H, T, T, (uint32_t)NKP)))
            return bail(1);
    }
    if (launch_attention(e, B, e->stream)) return bail(1);
    if (cudaStreamSynchronize(e->stream) != cudaSuccess) return bail(fail("attention kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    std::vector<__half> tmp((size_t)T * D);
    if (cudaMemcpy(tmp.data(), e->A16, tmp.size() * 2, cudaMemcpyDeviceToHost) != cudaSuccess) return bail(fail("D2H failed"));
    for (size_t i = 0; i < tmp.size(); ++i) out[i] = __half2float(tmp[i]);
    return bail(0);
}

int vitb200_test_dequant(int type, const void *blocks, int64_t n_blocks, uint16_t *out_f16)
{
    const size_t bs = quant_block_bytes(type);
    if (!bs) return fail("type %d is not a supported block format", type);
    if (!blocks || !out_f16 || n_blocks < 0) return fail("null argument");
    float y[32];
    for (int64_t b = 0; b < n_blocks; ++b)
    {
        dequant_block(type, (const uint8_t *)blocks + (size_t)b * bs, y);
        for (int i = 0; i < 32; ++i) out_f16[b * 32 + i] = host_f32_to_f16(y[i]);
    }
    return 0;
}

void *vitb200_stream(vitb200_engine *e) { return e ? (void *)e->stream : nullptr; }

int vitb200_forward_device(vitb200_engine *e, const float *d_images, int batch, float *d_probs, float *d_logits,
                           int32_t *d_topk_idx, float *d_topk_prob, int k, void *stream)
{
    if (!e || !d_images) return fail("null argument");
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
    if (batch < 1 || batch > e->max_batch) return fail("batch %d out of range (1..%d)", batch, e->max_batch);
    if (k < 0 || k > e->max_k) return fail("k %d out of range (0..%d)", k, e->max_k);
    return run_forward_graphed(e, d_images, batch, d_probs, d_logits, d_topk_idx, d_topk_prob, k, s);
}

// Enqueue one batched forward with HOST buffers.  Slot s = call parity: the H2D of this call runs on the copy stream and
// may overlap the kernels of the previous call (other slot); kernels + D2H run on the compute stream in call order.
static int forward_enqueue(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, int32_t *topk_idx,
                           float *topk_prob, int k, const vitb200_taps *taps)
{
    if (!e || !images) return fail("null argument");
    if (batch < 1 || batch > e->max_batch) return fail("batch %d out of range (1..%d)", batch, e->max_batch);
    if (k < 0 || k > e->max_k) return fail("k %d out of range (0..%d)", k, e->max_k); // before anything is enqueued
    CUDA_TRY(cudaSetDevice(e->device));
    const int sl = (int)(e->submits & 1);
    cudaStream_t s = e->stream, cs = e->copy_stream;
    const size_t img_elems = (size_t)e->C * e->hp.img_size * e->hp.img_size;
    const size_t rows = (size_t)batch * e->head_tokens; // classifier rows returned
    const int C = e->hp.num_classes;
    if (e->submits >= 2) CUDA_TRY(cudaStreamWaitEvent(cs, e->ev_done[sl], 0)); // slot's previous forward has consumed its inputs/outputs
    CUDA_TRY(cudaMemcpyAsync(e->d_img_slot[sl], images, (size_t)batch * img_elems * sizeof(float), cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaEventRecord(e->ev_h2d[sl], cs));
    CUDA_TRY(cudaStreamWaitEvent(s, e->ev_h2d[sl], 0));
    const bool want_topk = k > 0 && (topk_idx || topk_prob);
    float *dp = (probs || want_topk) ? e->d_probs_slot[sl] : nullptr;
    int32_t *di = want_topk ? e->d_topk_idx_slot[sl] : nullptr;
    float *dv = want_topk ? e->d_topk_val_slot[sl] : nullptr;
    const int kk = want_topk ? k : 0;
    if (taps ? run_forward(e, e->d_img_slot[sl], batch, dp, e->d_logits_slot[sl], di, dv, kk, s, taps)
             : run_forward_graphed(e, e->d_img_slot[sl], batch, dp, e->d_logits_slot[sl], di, dv, kk, s))
        return 1;
    if (probs) CUDA_TRY(cudaMemcpyAsync(probs, e->d_probs_slot[sl], rows * C * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (logits) CUDA_TRY(cudaMemcpyAsync(logits, e->d_logits_slot[sl], rows * C * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (want_topk && topk_idx) CUDA_TRY(cudaMemcpyAsync(topk_idx, e->d_topk_idx_slot[sl], rows * k * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (want_topk && topk_prob) CUDA_TRY(cudaMemcpyAsync(topk_prob, e->d_topk_val_slot[sl], rows * k * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaEventRecord(e->ev_done[sl], s));
    e->submits++;
    return 0;
}

int vitb200_forward_async(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, int32_t *topk_idx,
                          float *topk_prob, int k)
{
    return forward_enqueue(e, images, batch, probs, logits, topk_idx, topk_prob, k, nullptr);
}

int vitb200_sync(vitb200_engine *e)
{
    if (!e) return fail("null argument");
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaStreamSynchronize(e->copy_stream));
    CUDA_TRY(cudaStreamSynchronize(e->stream));
    return 0;
}

static int forward_host(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, int32_t *topk_idx,
                        float *topk_prob, int k, const vitb200_taps *taps)
{
    if (forward_enqueue(e, images, batch, probs, logits, topk_idx, topk_prob, k, taps)) return 1;
    return vitb200_sync(e);
}

// Data-parallel forward over several engines (one per GPU, weights replicated) driven from ONE host thread: image b goes to
// engine floor(b * n / batch)-style contiguous shards, every shard is enqueued with the non-blocking pipeline entry point, then
// all engines are synchronised.  No collective: shards are independent (SURVEY.md 8e).
static int forward_sharded_impl(vitb200_engine *const *engines, int n_engines, const float *images, int batch, float *probs, float *logits,
                                int32_t *topk_idx, float *topk_prob, int k, bool sync)
{
    if (!engines || n_engines < 1 || !images) return fail("null argument");
    const vitb200_engine *e0 = engines[0];
    if (!e0) return fail("null engine");
    if (k < 0 || k > e0->max_k) return fail("k %d out of range (0..%d)", k, e0->max_k);
    {
        // validate every shard before the first one is enqueued
        const int base0 = batch / n_engines, rem0 = batch % n_engines;
        for (int g = 0; g < n_engines; ++g)
        {
            const int cnt = base0 + (g < rem0 ? 1 : 0);
            if (cnt == 0) continue;
            if (!engines[g]) return fail("null engine %d", g);
            if (cnt > engines[g]->max_batch) return fail("shard %d: batch %d out of range (1..%d)", g, cnt, engines[g]->max_batch);
        }
    }
    const size_t img_elems = (size_t)e0->C * e0->hp.img_size * e0->hp.img_size;
    const size_t C = (size_t)e0->hp.num_classes * e0->head_tokens; // output floats per image
    const size_t kk = (size_t)k * e0->head_tokens;                 // top-k entries per image
    const int base = batch / n_engines, rem = batch % n_engines;
    int begin = 0;
    for (int g = 0; g < n_engines; ++g)
    {
        const int cnt = base + (g < rem ? 1 : 0);
        if (cnt == 0) continue;
        if (!engines[g]) return fail("null engine %d", g);
        if (engines[g]->hp.img_size != e0->hp.img_size || engines[g]->hp.num_classes != e0->hp.num_classes || engines[g]->head_tokens != e0->head_tokens ||
            engines[g]->C != e0->C)
            return fail("engine %d holds a different model", g);
        if (vitb200_forward_async(engines[g], images + (size_t)begin * img_elems, cnt, probs ? probs + (size_t)begin * C : nullptr,
                                  logits ? logits + (size_t)begin * C : nullptr, topk_idx ? topk_idx + (size_t)begin * kk : nullptr,
                                  topk_prob ? topk_prob + (size_t)begin * kk : nullptr, k))
        {
            // shards already enqueued are copying into the caller's buffers: drain them before reporting the failure
            const std::string first = g_err;
            for (int h = 0; h < g; ++h)
                if (engines[h]) (void)vitb200_sync(engines[h]);
            g_err = first;
            return 1;
        }
        begin += cnt;
    }
    if (!sync) return 0;
    int rc = 0;
    for (int g = 0; g < n_engines; ++g)
        if (engines[g] && vitb200_sync(engines[g])) rc = 1;
    return rc;
}

int vitb200_forward_sharded(vitb200_engine *const *engines, int n_engines, const float *images, int batch, float *probs, float *logits,
                            int32_t *topk_idx, float *topk_prob, int k)
{
    return forward_sharded_impl(engines, n_engines, images, batch, probs, logits, topk_idx, topk_prob, k, true);
}

// Pipelined form: every shard goes through its engine's two-slot vitb200_forward_async pipeline and the call returns; the host
// thread can enqueue the next global batch (other host buffers) while this one runs.  vitb200_sync_all() waits for everything.
int vitb200_forward_sharded_async(vitb200_engine *const *engines, int n_engines, const float *images, int batch, float *probs,
                                  float *logits, int32_t *topk_idx, float *topk_prob, int k)
{
    return forward_sharded_impl(engines, n_engines, images, batch, probs, logits, topk_idx, topk_prob, k, false);
}

int vitb200_sync_all(vitb200_engine *const *engines, int n_engines)
{
    if (!engines || n_engines < 1) return fail("null argument");
    int rc = 0;
    for (int g = 0; g < n_engines; ++g)
        if (engines[g] && vitb200_sync(engines[g])) rc = 1;
    return rc;
}

int vitb200_forward(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, int32_t *topk_idx,
                    float *topk_prob, int k)
{
    return forward_host(e, images, batch, probs, logits, topk_idx, topk_prob, k, nullptr);
}

int vitb200_forward_debug(vitb200_engine *e, const float *images, int batch, float *probs, float *logits, const vitb200_taps *taps)
{
    return forward_host(e, images, batch, probs, logits, nullptr, nullptr, 0, taps);
}

// vit_image_preprocess (reference vit.cpp:289-305) for a batch of u8 RGB images of arbitrary sizes, on the GPU, followed by the
// forward pass: the "images" of vitb200_forward never exist on the host, and (unless images_f32_out asks for them) not in HBM
// either -- the preprocess kernel writes the f16 patch matrix the patch-embedding GEMM reads.  Pipelined like
// vitb200_forward_async: the caller's images are packed into this slot's pinned staging buffer, ONE host-to-device copy on the copy
// stream overlaps the previous call's kernels, nothing synchronises on entry and nothing is allocated once the staging buffers
// have grown to the largest batch seen.
static int forward_u8_enqueue(vitb200_engine *e, const uint8_t *const *images, const int *nx, const int *ny, int batch, int bilinear,
                              float *images_f32_out, float *probs, float *logits, int32_t *topk_idx, float *topk_prob, int k)
{
    if (!e || !images || !nx || !ny) return fail("null argument");
    if (e->C != 3) return fail("vitb200_forward_u8 implements vit_image_preprocess (RGB, vit.cpp:289-305); this model takes %d-channel input", e->C);
    if (batch < 1 || batch > e->max_batch) return fail("batch %d out of range (1..%d)", batch, e->max_batch);
    if (k < 0 || k > e->max_k) return fail("k %d out of range (0..%d)", k, e->max_k);
    size_t total = 0;
    for (int b = 0; b < batch; ++b)
    {
        if (!images[b] || nx[b] < 1 || ny[b] < 1) return fail("image %d: bad pointer or size", b);
        total += ((size_t)nx[b] * ny[b] * 3 + 255) / 256 * 256;
    }
    const size_t table_off = total;
    total += (size_t)batch * sizeof(PreImage);
    CUDA_TRY(cudaSetDevice(e->device));
    const int sl = (int)(e->submits & 1);
    cudaStream_t s = e->stream, cs = e->copy_stream;
    // this slot's previous call (two submissions ago) must have consumed its staging buffer before the host overwrites it
    if (e->submits >= 2) CUDA_TRY(cudaEventSynchronize(e->ev_done[sl]));
    if (total > e->u8_cap[sl])
    {
        const size_t cap = total + total / 4;
        if (e->h_u8[sl]) cudaFreeHost(e->h_u8[sl]);
        if (e->d_u8[sl]) cudaFree(e->d_u8[sl]);
        e->h_u8[sl] = nullptr; e->d_u8[sl] = nullptr; e->u8_cap[sl] = 0;
        CUDA_TRY(cudaHostAlloc((void **)&e->h_u8[sl], cap, cudaHostAllocDefault));
        CUDA_TRY(cudaMalloc((void **)&e->d_u8[sl], cap));
        e->u8_cap[sl] = cap;
    }
    PreImage *table = reinterpret_cast<PreImage *>(e->h_u8[sl] + table_off);
    size_t off = 0;
    for (int b = 0; b < batch; ++b)
    {
        const size_t n = (size_t)nx[b] * ny[b] * 3;
        memcpy(e->h_u8[sl] + off, images[b], n);
        table[b].offset = off; table[b].nx = nx[b]; table[b].ny = ny[b];
        off += (n + 255) / 256 * 256;
    }
    CUDA_TRY(cudaMemcpyAsync(e->d_u8[sl], e->h_u8[sl], total, cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaEventRecord(e->ev_h2d[sl], cs));
    CUDA_TRY(cudaStreamWaitEvent(s, e->ev_h2d[sl], 0));
    const int S = e->hp.img_size;
    dim3 grid((unsigned)((S * S + 255) / 256), (unsigned)batch);
    float *d_f32 = images_f32_out ? e->d_img_slot[sl] : nullptr;
    preprocess_kernel<<<grid, 256, 0, s>>>(e->d_u8[sl], reinterpret_cast<const PreImage *>(e->d_u8[sl] + table_off), d_f32, S, bilinear ? 1 : 0,
                                           e->PA, e->hp.patch_size, e->KPp);
    CUDA_TRY(cudaGetLastError());
    const size_t img_elems = (size_t)3 * S * S;
    if (images_f32_out) CUDA_TRY(cudaMemcpyAsync(images_f32_out, d_f32, (size_t)batch * img_elems * sizeof(float), cudaMemcpyDeviceToHost, s));
    const bool want_topk = k > 0 && (topk_idx || topk_prob);
    const int C = e->hp.num_classes;
    if (probs || logits || want_topk)
    {
        float *dp = (probs || want_topk) ? e->d_probs_slot[sl] : nullptr;
        if (run_forward_graphed(e, nullptr, batch, dp, e->d_logits_slot[sl], want_topk ? e->d_topk_idx_slot[sl] : nullptr,
                                want_topk ? e->d_topk_val_slot[sl] : nullptr, want_topk ? k : 0, s))
            return 1;
        e->launches += 1; // the preprocess kernel
        const size_t rows = (size_t)batch * e->head_tokens;
        if (probs) CUDA_TRY(cudaMemcpyAsync(probs, e->d_probs_slot[sl], rows * C * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (logits) CUDA_TRY(cudaMemcpyAsync(logits, e->d_logits_slot[sl], rows * C * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (want_topk && topk_idx) CUDA_TRY(cudaMemcpyAsync(topk_idx, e->d_topk_idx_slot[sl], rows * k * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        if (want_topk && topk_prob) CUDA_TRY(cudaMemcpyAsync(topk_prob, e->d_topk_val_slot[sl], rows * k * sizeof(float), cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(cudaEventRecord(e->ev_done[sl], s));
    e->submits++;
    return 0;
}

int vitb200_forward_u8_async(vitb200_engine *e, const uint8_t *const *images, const int *nx, const int *ny, int batch, int bilinear,
                             float *probs, float *logits, int32_t *topk_idx, float *topk_prob, int k)
{
    VB_NOEXCEPT_BEGIN
    return forward_u8_enqueue(e, images, nx, ny, batch, bilinear, nullptr, probs, logits, topk_idx, topk_prob, k);
    VB_NOEXCEPT_END((void)0)
}

int vitb200_forward_u8(vitb200_engine *e, const uint8_t *const *images, const int *nx, const int *ny, int batch, int bilinear,
                       float *images_f32_out, float *probs, float *logits, int32_t *topk_idx, float *topk_prob, int k)
{
    VB_NOEXCEPT_BEGIN
    if (forward_u8_enqueue(e, images, nx, ny, batch, bilinear, images_f32_out, probs, logits, topk_idx, topk_prob, k)) return 1;
    return vitb200_sync(e);
    VB_NOEXCEPT_END((void)0)
}

int vitb200_test_gemm(int device, int M, int N, int K, int epilogue, const uint16_t *A, const uint16_t *W, const float *bias,
                      const float *resid, float *out)
{
    if (!A || !W || !bias || !out) return fail("null argument");
    if (K % 8 != 0) return fail("K must be a multiple of 8");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    __half *dA = nullptr, *dW = nullptr;
    float *dB = nullptr, *dR = nullptr;
    void *dO = nullptr;
    const bool f16out = epilogue == EPI_BIAS_F16 || epilogue == EPI_BIAS_GELU_F16 || epilogue == EPI_BIAS_F16_HILO;
    const size_t osz = (size_t)M * N * (f16out ? 2 : 4);
    void *dO2 = nullptr;
    int rc = 1;
    do
    {
        if (cudaMalloc(&dA, (size_t)M * K * 2) || cudaMalloc(&dW, (size_t)N * K * 2) || cudaMalloc(&dB, (size_t)N * 4) || cudaMalloc(&dO, osz)) { fail("cudaMalloc failed"); break; }
        cudaMemcpy(dA, A, (size_t)M * K * 2, cudaMemcpyHostToDevice);
        cudaMemcpy(dW, W, (size_t)N * K * 2, cudaMemcpyHostToDevice);
        cudaMemcpy(dB, bias, (size_t)N * 4, cudaMemcpyHostToDevice);
        cudaMemset(dO, 0, osz);
        if (epilogue == EPI_BIAS_F16_HILO)
        {
            if (cudaMalloc(&dO2, osz)) { fail("cudaMalloc failed"); break; }
            cudaMemset(dO2, 0, osz);
        }
        if (epilogue == EPI_BIAS_RESID_F32)
        {
            if (!resid) { fail("resid required"); break; }
            if (cudaMalloc(&dR, (size_t)M * N * 4)) { fail("cudaMalloc failed"); break; }
            cudaMemcpy(dR, resid, (size_t)M * N * 4, cudaMemcpyHostToDevice);
        }
        const int bn = pick_bn(N);
        const int cg = (getenv("VITB200_CTA_GROUP") && atoi(getenv("VITB200_CTA_GROUP")) == 1) ? 1 : 2;
        CUtensorMap tA, tB, tX, tO2;
        if (make_tmap(&tA, dA, M, K, K, GEMM_BM) || make_tmap(&tB, dW, N, K, K, bn / cg)) break;
        memset(&tX, 0, sizeof(tX));
        memset(&tO2, 0, sizeof(tO2));
        if (f16out && make_tmap(&tX, dO, M, N, N, 32)) break;            // the f16 epilogues store through TMA
        if (dO2 && make_tmap(&tO2, dO2, M, N, N, 32)) break;
        if (epilogue == EPI_BIAS_RESID_F32)
        {
            // the residual epilogue works in place on the f32 stream, like the engine uses it (X += ...)
            cudaMemcpy(dO, dR, (size_t)M * N * 4, cudaMemcpyDeviceToDevice);
            if (make_tmap_f32_box32(&tX, dO, M, N, N)) break;
        }
        GemmParams p{};
        p.M = M; p.N = N; p.K = K; p.bias = dB; p.out = dO; p.out2 = dO2; p.ldo = N; p.resid = (const float *)dO;
        if (launch_gemm(nullptr, cg, bn, epilogue, tA, tB, tX, tO2, p, 0, prop.multiProcessorCount)) break;
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { fail("GEMM kernel failed: %s", cudaGetErrorString(err)); break; }
        if (f16out)
        {
            std::vector<__half> tmp((size_t)M * N);
            cudaMemcpy(tmp.data(), dO, osz, cudaMemcpyDeviceToHost);
            for (size_t i = 0; i < tmp.size(); ++i) out[i] = __half2float(tmp[i]);
            if (dO2) // split-precision result: hi + lo (exact in f32: the two parts do not overlap)
            {
                cudaMemcpy(tmp.data(), dO2, osz, cudaMemcpyDeviceToHost);
                for (size_t i = 0; i < tmp.size(); ++i) out[i] += __half2float(tmp[i]);
            }
        }
        else
            cudaMemcpy(out, dO, osz, cudaMemcpyDeviceToHost);
        rc = 0;
    } while (0);
    cudaFree(dA); cudaFree(dW); cudaFree(dB); cudaFree(dO); cudaFree(dR); cudaFree(dO2);
    return rc;
}

// Stand-alone run of the block LayerNorm as the engine launches it (persistent bulk-copy kernel for hidden sizes that are a multiple of 128
// and >= 8 rows, the row-per-warp kernel otherwise): x [rows][D] f32 -> y [rows][D] (f16 results widened to f32).
int vitb200_test_layernorm(int device, int rows, int D, const float *x, const float *w, const float *b, float eps, float *y)
{
    if (!x || !w || !b || !y || rows < 1 || D < 4 || D % 4 != 0 || D > 2048) return fail("bad argument");
    VB_NOEXCEPT_BEGIN
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device: the vit.cpp_b200 forward path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    vitb200_engine e{};
    e.hp.hidden_size = D; e.hp.eps = eps; e.num_sms = prop.multiProcessorCount; e.device = device;
    float *dx = nullptr, *dw = nullptr, *db = nullptr;
    __half *dy = nullptr;
    int rc = 1;
    do
    {
        if (cudaMalloc(&dx, (size_t)rows * D * 4) || cudaMalloc(&dw, (size_t)D * 4) || cudaMalloc(&db, (size_t)D * 4) || cudaMalloc(&dy, (size_t)rows * D * 2)) { fail("cudaMalloc failed"); break; }
        cudaMemcpy(dx, x, (size_t)rows * D * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dw, w, (size_t)D * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(db, b, (size_t)D * 4, cudaMemcpyHostToDevice);
        cudaMemset(dy, 0xFF, (size_t)rows * D * 2);
        if (cudaDeviceSynchronize() != cudaSuccess) { fail("device sync failed"); break; }
        if (launch_layernorm(&e, dx, (size_t)D, dw, db, dy, rows, 0)) break;
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { fail("LayerNorm kernel failed: %s", cudaGetErrorString(err)); break; }
        std::vector<__half> tmp((size_t)rows * D);
        cudaMemcpy(tmp.data(), dy, tmp.size() * 2, cudaMemcpyDeviceToHost);
        for (size_t i = 0; i < tmp.size(); ++i) y[i] = __half2float(tmp[i]);
        rc = 0;
    } while (0);
    cudaFree(dx); cudaFree(dw); cudaFree(db); cudaFree(dy);
    return rc;
    VB_NOEXCEPT_END((void)0)
}

// Stand-alone run of the final soft-max + top-k through the forward's own launcher (launch_softmax_topk): logits [R][ldl] f32, of which
// the first C columns of every row are read -> probs [R][C], idx / val [R][k].
int vitb200_test_softmax_topk(int device, int R, int C, int ldl, const float *logits, int k, float *probs, int32_t *idx, float *val)
{
    if (!logits || !probs || R < 1 || C < 1 || ldl < C || k < 0 || k > 16 || (k > 0 && (!idx || !val))) return fail("bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device: the vit.cpp_b200 forward path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    float *dl = nullptr, *dp = nullptr, *dv = nullptr, *dscr = nullptr;
    int32_t *di = nullptr;
    const size_t n_scratch = softmax_scratch_floats(R, C);
    int rc = 1;
    do
    {
        if (cudaMalloc(&dl, (size_t)R * ldl * 4) || cudaMalloc(&dp, (size_t)R * C * 4) || cudaMalloc(&di, (size_t)R * (k ? k : 1) * 4) ||
            cudaMalloc(&dv, (size_t)R * (k ? k : 1) * 4) || (n_scratch && cudaMalloc(&dscr, n_scratch * 4))) { fail("cudaMalloc failed"); break; }
        if (cudaMemcpy(dl, logits, (size_t)R * ldl * 4, cudaMemcpyHostToDevice) != cudaSuccess) { fail("H2D failed"); break; }
        if (launch_softmax_topk(dl, ldl, dp, k ? di : nullptr, k ? dv : nullptr, R, C, k, dscr, 0)) break;
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { fail("soft-max kernel failed: %s", cudaGetErrorString(err)); break; }
        if (cudaMemcpy(probs, dp, (size_t)R * C * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
            (k && (cudaMemcpy(idx, di, (size_t)R * k * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
                   cudaMemcpy(val, dv, (size_t)R * k * 4, cudaMemcpyDeviceToHost) != cudaSuccess))) { fail("D2H failed"); break; }
        rc = 0;
    } while (0);
    cudaFree(dl); cudaFree(dp); cudaFree(di); cudaFree(dv); cudaFree(dscr);
    return rc;
}

// q8_0 linear layer on the integer tensor cores (gemm_q8_tcgen05.cuh; prototype for BASELINE.json configs[4]): x [M][K] f32 is
// quantised on the device exactly as the reference quantises activation rows, w is a q8_0 tensor in the model-file layout
// ([N][K/32] blocks of {f16 d; int8 q[32]}, ggml-quants.h:42-46).  Outputs: y [M][N] f32, and (optional) the quantised activations
// xq [M][K] int8, xd [M][K/32] f32.  iters > 0 additionally times `iters` back-to-back GEMM launches (CUDA events) into *ms_per_launch.
int vitb200_test_gemm_q8(int device, int M, int N, int K, const float *x, const void *w_q8_0, const float *bias, float *y,
                         int8_t *xq, float *xd, int iters, float *ms_per_launch)
{
    if (!x || !w_q8_0 || !bias || !y || M < 1 || N < 1 || K < 1) return fail("bad argument");
    if (K % Q8_BK != 0) return fail("K must be a multiple of %d", Q8_BK);
    if (N % 4 != 0) return fail("N must be a multiple of 4");
    VB_NOEXCEPT_BEGIN
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device: the vit.cpp_b200 forward path has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    const int KB = K / 32;
    // repack the 34-byte blocks: int8 plane [N][K] + transposed scale plane [K/32][N]
    std::vector<int8_t> wq((size_t)N * K);
    std::vector<float> wdT((size_t)KB * N);
    const uint8_t *blk = (const uint8_t *)w_q8_0;
    for (int n = 0; n < N; ++n)
        for (int b = 0; b < KB; ++b)
        {
            const uint8_t *src = blk + ((size_t)n * KB + b) * 34;
            uint16_t du;
            memcpy(&du, src, 2);
            wdT[(size_t)b * N + n] = host_f16_to_f32(du);
            memcpy(&wq[(size_t)n * K + (size_t)b * 32], src + 2, 32);
        }
    float *dX = nullptr, *dAd = nullptr, *dWd = nullptr, *dB = nullptr, *dY = nullptr;
    int8_t *dAq = nullptr, *dWq = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = 1;
    do
    {
        if (cudaMalloc(&dX, (size_t)M * K * 4) || cudaMalloc(&dAq, (size_t)M * K) || cudaMalloc(&dAd, (size_t)M * KB * 4) ||
            cudaMalloc(&dWq, (size_t)N * K) || cudaMalloc(&dWd, (size_t)KB * N * 4) || cudaMalloc(&dB, (size_t)N * 4) ||
            cudaMalloc(&dY, (size_t)M * N * 4)) { fail("cudaMalloc failed"); break; }
        cudaMemcpy(dX, x, (size_t)M * K * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dWq, wq.data(), wq.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(dWd, wdT.data(), wdT.size() * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(dB, bias, (size_t)N * 4, cudaMemcpyHostToDevice);
        cudaMemset(dY, 0, (size_t)M * N * 4);
        CUtensorMap tA, tW, tAd, tWd;
        if (make_tmap_2d(&tA, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, dAq, (uint64_t)M, (uint64_t)K, (uint64_t)K, Q8_BK, Q8_BM, CU_TENSOR_MAP_SWIZZLE_128B) ||
            make_tmap_2d(&tW, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, dWq, (uint64_t)N, (uint64_t)K, (uint64_t)K, Q8_BK, Q8_BN, CU_TENSOR_MAP_SWIZZLE_128B) ||
            make_tmap_2d(&tAd, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, dAd, (uint64_t)M, (uint64_t)KB, (uint64_t)KB, 4, Q8_BM, CU_TENSOR_MAP_SWIZZLE_NONE) ||
            make_tmap_2d(&tWd, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, dWd, (uint64_t)KB, (uint64_t)N, (uint64_t)N, Q8_BN, 4, CU_TENSOR_MAP_SWIZZLE_NONE))
            break;
        const long long n_blocks = (long long)M * KB;
        const int qthreads = 256;
        const long long qgrid = (n_blocks * 8 + qthreads - 1) / qthreads;
        quantize_q8_0_kernel<<<(unsigned)qgrid, qthreads>>>(dX, dAq, dAd, n_blocks);
        if (cudaGetLastError() != cudaSuccess) { fail("quantize launch failed"); break; }
        if (cudaFuncSetAttribute(gemm_q8_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Q8_SMEM_BYTES) != cudaSuccess) { fail("cudaFuncSetAttribute failed"); break; }
        Q8GemmParams p{};
        p.M = M; p.N = N; p.K = K; p.bias = dB; p.out = dY; p.ldo = N;
        const int tiles = ((M + Q8_BM - 1) / Q8_BM) * ((N + Q8_BN - 1) / Q8_BN);
        const int grid = tiles < prop.multiProcessorCount ? tiles : prop.multiProcessorCount;
        gemm_q8_tcgen05_kernel<<<grid, Q8_THREADS, Q8_SMEM_BYTES>>>(tA, tW, tAd, tWd, p);
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { fail("q8_0 GEMM kernel failed: %s", cudaGetErrorString(err)); break; }
        cudaMemcpy(y, dY, (size_t)M * N * 4, cudaMemcpyDeviceToHost);
        if (xq) cudaMemcpy(xq, dAq, (size_t)M * K, cudaMemcpyDeviceToHost);
        if (xd) cudaMemcpy(xd, dAd, (size_t)M * KB * 4, cudaMemcpyDeviceToHost);
        if (iters > 0 && ms_per_launch)
        {
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            cudaEventRecord(e0);
            for (int i = 0; i < iters; ++i) gemm_q8_tcgen05_kernel<<<grid, Q8_THREADS, Q8_SMEM_BYTES>>>(tA, tW, tAd, tWd, p);
            cudaEventRecord(e1);
            err = cudaDeviceSynchronize();
            if (err != cudaSuccess) { fail("q8_0 GEMM kernel failed: %s", cudaGetErrorString(err)); break; }
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            *ms_per_launch = ms / (float)iters;
        }
        rc = 0;
    } while (0);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(dX); cudaFree(dAq); cudaFree(dAd); cudaFree(dWq); cudaFree(dWd); cudaFree(dB); cudaFree(dY);
    return rc;
    VB_NOEXCEPT_END((void)0)
}

} // extern "C"

// ------------------------------------------------------------------------------------------------
// Legacy-ggml model file reader (the format reference vit_model_load parses, vit.cpp:308-712; written by
// convert-pth-to-ggml.py:105-158).  Validation mirrors the reference: magic, known tensor names, element
// counts; failures return non-zero with a message, never abort.

extern "C" int vitb200_create_from_file(const char *path, int device, int max_batch, vitb200_engine **out)
{
    return vitb200_create_from_file_ex(path, device, max_batch, 1, out);
}

extern "C" int vitb200_create_from_file_ex(const char *path, int device, int max_batch, int head_tokens, vitb200_engine **out)
{
    if (!path || !out) return fail("null argument");
    *out = nullptr;
    VB_NOEXCEPT_BEGIN
    std::ifstream fin(path, std::ios::binary);
    if (!fin) return fail("failed to open '%s'", path);
    fin.seekg(0, std::ios::end);
    const std::streamoff fend = fin.tellg();
    // a directory or an unseekable stream reports -1; model files beyond 64 GiB are not something this loader stages in host memory
    if (!fin || fend < 0) return fail("failed to read '%s' (not a regular file)", path);
    if ((unsigned long long)fend > (64ull << 30)) return fail("model file '%s' is too large (%lld bytes)", path, (long long)fend);
    const size_t fsize = (size_t)fend;
    fin.seekg(0);
    std::vector<char> buf(fsize);
    fin.read(buf.data(), (std::streamsize)fsize);
    if (!fin) return fail("failed to read '%s'", path);
    // a true GGUF container (SURVEY.md 8(f) rank 3) or the legacy-ggml file the reference itself reads; both parsers live in
    // gguf_file.hpp (plain host C++, fuzzed under ASan/UBSan by tests/cpp/gguf_fuzz.cpp) and fill the same structure
    GgufModel g;
    const bool is_gguf = fsize >= 4 && memcmp(buf.data(), "GGUF", 4) == 0;
    if (is_gguf)
    {
        if (!parse_gguf(buf.data(), fsize, g)) return fail("invalid GGUF file '%s': %s", path, g.error.c_str());
    }
    else if (!parse_legacy_ggml(buf.data(), fsize, g))
        return fail("invalid model file '%s' (%s)", path, g.error.c_str());
    vitb200_hparams hp{};
    auto i32 = [](int64_t v) { return (int32_t)(v < -1 ? -1 : (v > (1 << 30) ? (1 << 30) : v)); }; // out-of-range values stay out of range
    hp.hidden_size = i32(g.hidden_size); hp.num_hidden_layers = i32(g.num_hidden_layers);
    hp.num_attention_heads = i32(g.num_attention_heads); hp.num_classes = i32(g.num_classes);
    hp.patch_size = i32(g.patch_size); hp.img_size = i32(g.img_size); hp.ftype = i32(g.ftype); hp.eps = g.eps;
    if (hp.num_hidden_layers < 1 || hp.num_hidden_layers > 4096) return fail("invalid model file '%s' (num_hidden_layers %d)", path, hp.num_hidden_layers);
    const int expected = 4 + 12 * hp.num_hidden_layers + 4; // vit.cpp:697
    if ((int)g.tensors.size() != expected) return fail("model file has %d tensors, but %d tensors were expected", (int)g.tensors.size(), expected);
    std::vector<vitb200_tensor> ts(g.tensors.size());
    for (size_t i = 0; i < g.tensors.size(); ++i)
    {
        ts[i].name = g.tensors[i].name.c_str();
        ts[i].data = buf.data() + g.tensors[i].offset;
        ts[i].type = g.tensors[i].type;
        ts[i].n_dims = g.tensors[i].n_dims;
        for (int j = 0; j < 4; ++j) ts[i].ne[j] = g.tensors[i].ne[j];
    }
    const std::map<int, std::string> &labels = g.labels;
    int rc = vitb200_create_ex(&hp, ts.data(), (int)ts.size(), device, max_batch, head_tokens, out);
    if (rc == 0) (*out)->labels = labels;
    return rc;
    VB_NOEXCEPT_END(if (*out) { vitb200_destroy(*out); *out = nullptr; })
}
