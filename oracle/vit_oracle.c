/* oracle/vit_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain-C CPU restatement of the forward path of staghado/vit.cpp (reference @ a4841f6, ggml @
 * a5e4560): the node sequence emitted by vit_encode_image (reference vit.cpp:718-941) with the
 * arithmetic of the ggml CPU kernels it dispatches to (ggml.c / ggml-quants.c, x86 AVX2+FMA+F16C
 * build).  It exists so that tests/ can compare the CUDA path against something whose every
 * rounding point is written down, and so that per-layer intermediates ("taps") are available.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load it.
 *
 * Pinning: tests/test_oracle.py checks this file against oracle/_ref/libvitref.so (the unmodified
 * reference compiled from /root/reference) and against tests/golden/ fixtures that were generated
 * by that same reference build (tests/golden/make_golden.py).  The summation ORDER of every dot
 * product below reproduces the reference's AVX2 kernels (4 accumulators x 8 lanes, then the
 * GGML_F32x8_REDUCE tree), so on the same host/libm the logits agree bit for bit.
 *
 * Every function cites the reference lines it follows.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <pthread.h>

/* ---- tiny pthread parallel-for (this image's gcc ships without libgomp) ------------------ */
static int g_threads = 4;
typedef void (*pf_fn)(int begin, int end, void *ctx);
typedef struct { pf_fn fn; void *ctx; int begin, end; } pf_job;
static void *pf_tramp(void *p) { pf_job *j = (pf_job *)p; j->fn(j->begin, j->end, j->ctx); return NULL; }
static void par_for(int n, pf_fn fn, void *ctx) {
    int T = g_threads < 1 ? 1 : g_threads;
    if (T > n) T = n;
    if (T <= 1) { fn(0, n, ctx); return; }
    pthread_t th[64]; pf_job jobs[64];
    if (T > 64) T = 64;
    const int per = (n + T - 1) / T;
    for (int t = 0; t < T; ++t) {
        jobs[t].fn = fn; jobs[t].ctx = ctx; jobs[t].begin = t * per; jobs[t].end = (t + 1) * per < n ? (t + 1) * per : n;
        if (t > 0) pthread_create(&th[t], NULL, pf_tramp, &jobs[t]);
    }
    pf_tramp(&jobs[0]);
    for (int t = 1; t < T; ++t) pthread_join(th[t], NULL);
}

#define QK8_0 32

/* ---- f16 helpers ------------------------------------------------------------------------ */
/* ggml.c:315-332 ggml_fp32_to_fp16_row / GGML_FP32_TO_FP16: IEEE round-to-nearest-even (F16C). */
static inline float round_f16(float x) { return (float)(_Float16)x; }
static inline uint16_t f16_bits(float x) { _Float16 h = (_Float16)x; uint16_t u; memcpy(&u, &h, 2); return u; }
static inline float f16_from_bits(uint16_t u) { _Float16 h; memcpy(&h, &u, 2); return (float)h; }

/* ggml.c:2186-2201: 64K-entry f16 tables for GELU and exp, built with the host libm.
 * Stored here as the f32 value of the f16 table entry. */
static float g_tab_gelu[1 << 16];
static float g_tab_exp[1 << 16];
static int g_tab_init = 0;

/* ggml.c:1414-1424 ggml_gelu_f32 (tanh form, NOT erf); the reference build contracts 1 + A*x*x into one fma */
static inline float gelu_f32(float x) {
    const float GELU_COEF_A = 0.044715f;
    const float SQRT_2_OVER_PI = 0.79788456080286535587989211986876f;
    return 0.5f * x * (1.0f + tanhf(SQRT_2_OVER_PI * x * fmaf(GELU_COEF_A * x, x, 1.0f)));
}

static void init_tables(void) {
    if (g_tab_init) return;
    for (int i = 0; i < (1 << 16); ++i) {
        const float f = f16_from_bits((uint16_t)i);
        g_tab_gelu[i] = round_f16(gelu_f32(f)); /* ggml.c:2197 */
        g_tab_exp[i] = round_f16(expf(f));      /* ggml.c:2200 */
    }
    g_tab_init = 1;
}

/* ---- dot products (summation order of the AVX2 build) ----------------------------------- */
/* GGML_F32x8_REDUCE, ggml.c:776-791: sum[0]+=sum[2]; sum[1]+=sum[3]; sum[0]+=sum[1]; then
 * lo128+hi128, hadd, hadd. s[j*8+lane] is accumulator j, lane `lane`. */
static inline float reduce_4x8(const float *s) {
    float v[8], t0[4];
    for (int l = 0; l < 8; ++l) v[l] = (s[l] + s[16 + l]) + (s[8 + l] + s[24 + l]);
    for (int i = 0; i < 4; ++i) t0[i] = v[i] + v[i + 4];
    const float t1a = t0[0] + t0[1];
    const float t1b = t0[2] + t0[3];
    return t1a + t1b;
}

/* ggml.c:1163-1198 ggml_vec_dot_f32 and ggml.c:1200-1236 ggml_vec_dot_f16 (operands already
 * widened to f32 -- f16*f16 products are exact in f32, so vfmadd on widened values is the same
 * arithmetic).  `dbl_tail`: the f16 kernel accumulates leftovers in double; the f32 kernel adds
 * them in float, in order: gcc vectorises the multiplies of that loop 8 and then 4 at a time and
 * keeps the adds sequential, and its scalar epilogue for the last (n - np) % 4 terms is a fused
 * multiply-add (checked in the disassembly of the reference build, gcc 13, and pinned bit-for-bit
 * by tests/test_oracle.py). */
/* Experiment knob (tests/bench never set it): 0 = the reference's arithmetic (default, bit-exact);
 * 1 = same rounding points but dot products accumulated in double ("any other correct implementation");
 * 2 = 1 + q,k,v rounded to f16 before attention; 3 = 1 + only v rounded to f16; 4 = 1 + only q,k rounded to f16;
 * 5 = 1 + only q rounded; 6 = 1 + only k rounded; 7 = 1 + q,k,v replaced by hi + lo with hi = f16(x), lo = f16(x - hi) (what a
 * split-precision tensor-core attention sees); 8 = reference rounding points with every dot product accumulated in f32 in blocks
 * of 16 terms (each block summed exactly, then added to a running f32 sum: a tensor-core-like order).  Used to measure the parity noise floor between non-bit-identical
 * implementations and which attention operand's precision matters (DESIGN.md).
 * q8_0 models only: 9 = each q8_0 dot product replaced by sum_k f16(d_w q_w) * f16(d_x q_x) accumulated in double -- what an f16
 * tensor-core GEMM sees when the weights are dequantised once and the activations are quantised per 32-block exactly as the
 * reference does (quantize_row_q8_0) and then folded back to f16; 10 = the same with the activation factor d_x q_x kept exact
 * (a hi + lo f16 pair); 11 = dequantised f16 weights against plain f16-rounded activations, no activation quantisation (round 1's
 * engine).  The rest of the graph keeps the reference's rounding points. */
static int g_variant = 0;
void vo_set_variant(int v) { g_variant = v; }

static float dot_ggml(int n, const float *x, const float *y, int dbl_tail) {
    if (g_variant == 8) {
        float acc = 0.0f;
        for (int i = 0; i < n; i += 16) {
            double blk = 0.0;
            for (int j = i; j < n && j < i + 16; ++j) blk += (double)x[j] * (double)y[j];
            acc = (float)((double)acc + blk);
        }
        return acc;
    }
    if (g_variant) {
        double acc = 0.0;
        for (int i = 0; i < n; ++i) acc += (double)x[i] * (double)y[i];
        return (float)acc;
    }
    float s[32];
    for (int l = 0; l < 32; ++l) s[l] = 0.0f;
    const int np = n & ~31;
    for (int i = 0; i < np; i += 32)
        for (int l = 0; l < 32; ++l) s[l] = fmaf(x[i + l], y[i + l], s[l]);
    float r = reduce_4x8(s);
    if (dbl_tail) {
        double sd = (double)r;
        for (int i = np; i < n; ++i) sd += (double)(x[i] * y[i]);
        return (float)sd;
    }
    const int nf = n - ((n - np) & 3);
    for (int i = np; i < nf; ++i) r = r + x[i] * y[i];
    for (int i = nf; i < n; ++i) r = fmaf(x[i], y[i], r);
    return r;
}

/* ggml-quants.c:702-790 quantize_row_q8_0 (AVX2 branch): d = amax/127 stored as f16,
 * q = nearbyint(x * (127/amax)) (round-half-even). */
static void quantize_row_q8_0(const float *x, int n, float *d_out, int8_t *q_out) {
    const int nb = n / QK8_0;
    for (int b = 0; b < nb; ++b) {
        float amax = 0.0f;
        for (int i = 0; i < QK8_0; ++i) { const float a = fabsf(x[b * QK8_0 + i]); if (a > amax) amax = a; }
        const float d = amax / 127.f;
        d_out[b] = round_f16(d);
        const float id = (amax != 0.0f) ? 127.f / amax : 0.0f;
        for (int i = 0; i < QK8_0; ++i) q_out[b * QK8_0 + i] = (int8_t)nearbyintf(x[b * QK8_0 + i] * id);
    }
}

/* ggml-quants.c:3521+ ggml_vec_dot_q8_0_q8_0 (AVX2 branch): acc[lane] = fma(d_x*d_y, q[lane], acc),
 * q[lane] = sum of 4 consecutive int8 products; then hsum_float_8 (ggml-quants.c:67-73). */
static float dot_q8_0(int n, const float *dw, const int8_t *qw, const float *dx, const int8_t *qx) {
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const int nb = n / QK8_0;
    for (int b = 0; b < nb; ++b) {
        const float d = dw[b] * dx[b];
        for (int l = 0; l < 8; ++l) {
            int32_t q = 0;
            for (int k = 0; k < 4; ++k) q += (int32_t)qw[b * 32 + l * 4 + k] * (int32_t)qx[b * 32 + l * 4 + k];
            acc[l] = fmaf(d, (float)q, acc[l]);
        }
    }
    float r4[4];
    for (int i = 0; i < 4; ++i) r4[i] = acc[4 + i] + acc[i];
    const float a = r4[0] + r4[2];
    const float b = r4[1] + r4[3];
    return a + b;
}

/* ---- model --------------------------------------------------------------------------------- */
typedef struct {
    int type;        /* 0 f32, 1 f16, 8 q8_0 (how the reference stores / multiplies it) */
    int n_out, n_in; /* ggml ne1, ne0 */
    float *w;        /* [n_out][n_in] widened to f32 (types 0,1) */
    float *qd;       /* q8_0: [n_out][n_in/32] block scales (f16 value as f32) */
    int8_t *qs;      /* q8_0: [n_out][n_in] */
} vo_mat;

typedef struct {
    const float *norm1_w, *norm1_b, *qkv_b, *proj_b, *norm2_w, *norm2_b, *fc1_b, *fc2_b;
    vo_mat qkv, proj, fc1, fc2;
} vo_layer;

typedef struct {
    int hidden, layers, heads, classes, patch, img;
    int in_chans;    /* 3 (vit.cpp:747) or 1 (the ViTSTR extension, vitstr.cpp:713) */
    int head_tokens; /* tokens the classifier reads: 1 (token 0, vit.cpp:910) or 25 (vitstr.cpp:864-883) */
    float eps;
    const float *cls, *pos, *patch_b, *norm_w, *norm_b, *head_b;
    vo_mat patch_w, head;
    vo_layer *L;
} vo_model;

static void mat_init(vo_mat *m, const void *data, int type, int n_out, int n_in) {
    m->type = type; m->n_out = n_out; m->n_in = n_in; m->w = NULL; m->qd = NULL; m->qs = NULL;
    const size_t n = (size_t)n_out * n_in;
    if (type == 0) {
        m->w = (float *)malloc(n * sizeof(float));
        memcpy(m->w, data, n * sizeof(float));
    } else if (type == 1) {
        m->w = (float *)malloc(n * sizeof(float));
        const uint16_t *h = (const uint16_t *)data;
        for (size_t i = 0; i < n; ++i) m->w[i] = f16_from_bits(h[i]);
    } else { /* q8_0: ggml-quants.h:42-46 block_q8_0 { ggml_fp16_t d; int8_t qs[32]; } */
        const size_t nb = n / QK8_0;
        m->qd = (float *)malloc(nb * sizeof(float));
        m->qs = (int8_t *)malloc(n);
        const uint8_t *p = (const uint8_t *)data;
        for (size_t b = 0; b < nb; ++b) {
            uint16_t u; memcpy(&u, p + b * 34, 2);
            m->qd[b] = f16_from_bits(u);
            memcpy(m->qs + b * 32, p + b * 34 + 2, 32);
        }
    }
}
static void mat_free(vo_mat *m) { free(m->w); free(m->qd); free(m->qs); }

/* hp: hidden, layers, heads, classes, patch, img.  tensors/types: 4 + 12*layers + 4 entries in
 * timm state_dict order (see vit.cpp_b200/ggml_file.py tensor_specs; names at vit.cpp:518-579). */
void *vo_create_ex(const int32_t *hp, const void *const *tensors, const int32_t *types, int in_chans, int head_tokens);
void *vo_create(const int32_t *hp, const void *const *tensors, const int32_t *types) { return vo_create_ex(hp, tensors, types, 3, 1); }

/* The ViTSTR extension (extensions/vitstr.cpp/vitstr.cpp:684-916) builds the SAME graph with a 1-channel input tensor
 * (vitstr.cpp:713) and a classifier over the first 25 tokens (vitstr.cpp:864-903): in_chans = 1, head_tokens = 25. */
void *vo_create_ex(const int32_t *hp, const void *const *tensors, const int32_t *types, int in_chans, int head_tokens) {
    init_tables();
    vo_model *m = (vo_model *)calloc(1, sizeof(vo_model));
    m->hidden = hp[0]; m->layers = hp[1]; m->heads = hp[2]; m->classes = hp[3]; m->patch = hp[4]; m->img = hp[5];
    m->in_chans = in_chans; m->head_tokens = head_tokens;
    m->eps = 1e-6f; /* vit.h:29; the -e CLI flag never reaches the graph (vit.cpp:808) */
    const int D = m->hidden;
    int t = 0;
    m->cls = (const float *)tensors[t++];
    m->pos = (const float *)tensors[t++];
    mat_init(&m->patch_w, tensors[t], types[t], D, m->in_chans * m->patch * m->patch); t++;
    m->patch_b = (const float *)tensors[t++];
    m->L = (vo_layer *)calloc((size_t)m->layers, sizeof(vo_layer));
    for (int l = 0; l < m->layers; ++l) {
        vo_layer *L = &m->L[l];
        L->norm1_w = (const float *)tensors[t++];
        L->norm1_b = (const float *)tensors[t++];
        mat_init(&L->qkv, tensors[t], types[t], 3 * D, D); t++;
        L->qkv_b = (const float *)tensors[t++];
        mat_init(&L->proj, tensors[t], types[t], D, D); t++;
        L->proj_b = (const float *)tensors[t++];
        L->norm2_w = (const float *)tensors[t++];
        L->norm2_b = (const float *)tensors[t++];
        mat_init(&L->fc1, tensors[t], types[t], 4 * D, D); t++;
        L->fc1_b = (const float *)tensors[t++];
        mat_init(&L->fc2, tensors[t], types[t], D, 4 * D); t++;
        L->fc2_b = (const float *)tensors[t++];
    }
    m->norm_w = (const float *)tensors[t++];
    m->norm_b = (const float *)tensors[t++];
    mat_init(&m->head, tensors[t], types[t], m->classes, D); t++;
    m->head_b = (const float *)tensors[t++];
    return m;
}

void vo_destroy(void *mv) {
    vo_model *m = (vo_model *)mv;
    if (!m) return;
    mat_free(&m->patch_w); mat_free(&m->head);
    for (int l = 0; l < m->layers; ++l) { mat_free(&m->L[l].qkv); mat_free(&m->L[l].proj); mat_free(&m->L[l].fc1); mat_free(&m->L[l].fc2); }
    free(m->L); free(m);
}

/* ---- ops -------------------------------------------------------------------------------------- */
/* y[t][o] = W[o] . x[t] + b[o]  -- ggml_mul_mat + ggml_add_inplace (vit.cpp:820-821 etc.).
 * ggml.c:9493-9506: src1 (activations) is converted to the weight type's vec_dot_type first:
 * f16 weights -> f16 RNE activations; q8_0 weights -> dynamic q8_0 activations; f32 -> none. */
typedef struct { const vo_mat *W; const float *bias, *xa, *xd; const int8_t *xq; int T; float *y; } lin_ctx;
static void linear_rows(int o0, int o1, void *cv) {
    const lin_ctx *c = (const lin_ctx *)cv;
    const vo_mat *W = c->W;
    const int K = W->n_in, N = W->n_out, T = c->T;
    for (int o = o0; o < o1; ++o)
        for (int t = 0; t < T; ++t) {
            float v;
            if (W->type == 8 && g_variant >= 9) {
                const float *dw = W->qd + (size_t)o * (K / QK8_0), *dx = c->xd + (size_t)t * (K / QK8_0);
                const int8_t *qw = W->qs + (size_t)o * K, *qx = c->xq + (size_t)t * K;
                double acc = 0.0;
                for (int k = 0; k < K; ++k) {
                    const float wv = round_f16(dw[k / QK8_0] * (float)qw[k]);
                    float av = dx[k / QK8_0] * (float)qx[k];
                    if (g_variant == 9) av = round_f16(av);
                    if (g_variant == 11) av = round_f16(c->xa[(size_t)t * K + k]);
                    acc += (double)wv * (double)av;
                }
                v = (float)acc;
            } else if (W->type == 8)
                v = dot_q8_0(K, W->qd + (size_t)o * (K / QK8_0), W->qs + (size_t)o * K,
                             c->xd + (size_t)t * (K / QK8_0), c->xq + (size_t)t * K);
            else
                v = dot_ggml(K, W->w + (size_t)o * K, c->xa + (size_t)t * K, W->type == 1);
            c->y[(size_t)t * N + o] = c->bias ? v + c->bias[o] : v;
        }
}
static void linear(const vo_mat *W, const float *bias, const float *x, int T, float *y) {
    const int K = W->n_in, N = W->n_out;
    lin_ctx c = {W, bias, x, NULL, NULL, T, y};
    float *xd = NULL, *xr = NULL; int8_t *xq = NULL;
    if (W->type == 8) {
        xd = (float *)malloc((size_t)T * (K / QK8_0) * sizeof(float));
        xq = (int8_t *)malloc((size_t)T * K);
        for (int t = 0; t < T; ++t) quantize_row_q8_0(x + (size_t)t * K, K, xd + (size_t)t * (K / QK8_0), xq + (size_t)t * K);
        c.xd = xd; c.xq = xq;
    } else if (W->type == 1) {
        xr = (float *)malloc((size_t)T * K * sizeof(float));
        for (size_t i = 0; i < (size_t)T * K; ++i) xr[i] = round_f16(x[i]);
        c.xa = xr;
    }
    par_for(N, linear_rows, &c);
    free(xd); free(xq); free(xr);
}

/* ggml_norm (ggml.c:8959-9008) then ggml_mul by w (ggml.c:7583) then ggml_add_inplace b
 * (vit.cpp:808-812): double sums, biased variance, three separate f32 roundings. */
static void layernorm(const float *x, int T, int D, const float *w, const float *b, float eps, float *y) {
    for (int t = 0; t < T; ++t) {
        const float *xr = x + (size_t)t * D;
        float *yr = y + (size_t)t * D;
        double sum = 0.0;
        for (int i = 0; i < D; ++i) sum += (double)xr[i];
        const float mean = (float)(sum / D);
        double sum2 = 0.0;
        for (int i = 0; i < D; ++i) { const float v = xr[i] - mean; yr[i] = v; sum2 += (double)(v * v); }
        const float variance = (float)(sum2 / D);
        const float scale = 1.0f / sqrtf(variance + eps);
        for (int i = 0; i < D; ++i) {
            float v = yr[i] * scale;
            v = v * w[i];
            yr[i] = v + b[i];
        }
    }
}

/* ggml_compute_forward_soft_max_f32, ggml.c:10498-10567: true max, f16 exp table, double sum,
 * multiply by (float)(1/sum). */
static void softmax_row(float *p, int n) {
    float mx = -INFINITY;
    for (int i = 0; i < n; ++i) mx = p[i] > mx ? p[i] : mx;
    double sum = 0.0;
    for (int i = 0; i < n; ++i) {
        if (p[i] == -INFINITY) { p[i] = 0.0f; continue; }
        const float val = g_tab_exp[f16_bits(p[i] - mx)];
        sum += (double)val;
        p[i] = val;
    }
    const float inv = (float)(1.0 / sum);
    for (int i = 0; i < n; ++i) p[i] *= inv;
}

/* attention, all f32 (vit.cpp:826-866): q|k|v = qkv[t][0:D | D:2D | 2D:3D], head h = columns
 * h*hd..(h+1)*hd; S = K.Q (ggml_vec_dot_f32 over hd), x 1/sqrt(hd), softmax over keys, O = V^T.P */
typedef struct { const float *qkv; float *att; int N, D, hd; } att_ctx;
static void attention_heads(int h0, int h1, void *cv) {
    const att_ctx *c = (const att_ctx *)cv;
    const int N = c->N, D = c->D, hd = c->hd;
    float *s = (float *)malloc((size_t)N * sizeof(float));
    float *vt = (float *)malloc((size_t)hd * N * sizeof(float));
    const float scale = 1.0f / sqrtf((float)hd);
    for (int h = h0; h < h1; ++h) {
        for (int t = 0; t < N; ++t)
            for (int d = 0; d < hd; ++d) vt[(size_t)d * N + t] = c->qkv[(size_t)t * 3 * D + 2 * D + h * hd + d];
        for (int q = 0; q < N; ++q) {
            const float *qv = c->qkv + (size_t)q * 3 * D + h * hd;
            for (int k = 0; k < N; ++k) {
                const float *kv = c->qkv + (size_t)k * 3 * D + D + h * hd;
                s[k] = dot_ggml(hd, kv, qv, 0) * scale;                           /* vit.cpp:848-854 */
            }
            softmax_row(s, N);                                                    /* vit.cpp:856 */
            for (int d = 0; d < hd; ++d)
                c->att[(size_t)q * D + h * hd + d] = dot_ggml(N, vt + (size_t)d * N, s, 0); /* vit.cpp:858 */
        }
    }
    free(s); free(vt);
}

typedef struct {
    int layer;      /* which encoder block the per-layer taps refer to */
    float *embed;   /* [N][D]  tokens after cls concat + pos add (vit.cpp:797) */
    float *ln1;     /* [N][D]  LN1 output, f32 (vit.cpp:812) */
    float *qkv;     /* [N][3D] after bias (vit.cpp:821) */
    float *attn;    /* [N][D]  merged heads (vit.cpp:860-866) */
    float *x1;      /* [N][D]  after attention residual (vit.cpp:873) */
    float *ln2;     /* [N][D]  (vit.cpp:885) */
    float *h;       /* [N][4D] after GELU (vit.cpp:893) */
    float *x2;      /* [N][D]  block output (vit.cpp:900) */
    float *final_ln;/* [D]     (vit.cpp:919) */
    float *x_final; /* [N][D]  residual stream after the last block */
} vo_taps;

/* One forward pass of vit_encode_image (vit.cpp:718-941) on one HWC f32 image ([S][S][in_chans]).  logits_out / probs_out
 * hold head_tokens x classes values (one soft-max per pooled token). */
int vo_forward(void *mv, const float *img_hwc, float *logits_out, float *probs_out, const vo_taps *taps) {
    vo_model *m = (vo_model *)mv;
    const int D = m->hidden, H = m->heads, hd = D / H, P = m->patch, S = m->img, G = S / P, NP = G * G, N = NP + 1;
    const int CH = m->in_chans, KP = CH * P * P, TH = m->head_tokens;

    float *x = (float *)malloc((size_t)N * D * sizeof(float));
    float *cur = (float *)malloc((size_t)N * D * sizeof(float));
    float *qkv = (float *)malloc((size_t)N * 3 * D * sizeof(float));
    float *att = (float *)malloc((size_t)N * D * sizeof(float));
    float *hbuf = (float *)malloc((size_t)N * 4 * D * sizeof(float));
    float *tmp = (float *)malloc((size_t)N * D * sizeof(float));

    /* --- patch embedding: HWC->CHW copy (vit.cpp:759-768), im2col to f16 with K order
     * c*P*P + ky*P + kx (ggml.c:11597-11599), f16 x f16 mul_mat (ggml.c:5272-5277), + conv bias
     * (vit.cpp:773-775), cls concat (vit.cpp:794), + pos_embed (vit.cpp:797). */
    {
        float *col = (float *)malloc((size_t)NP * KP * sizeof(float));
        for (int py = 0; py < G; ++py)
            for (int px = 0; px < G; ++px)
                for (int c = 0; c < CH; ++c)
                    for (int ky = 0; ky < P; ++ky)
                        for (int kx = 0; kx < P; ++kx) {
                            const int iy = py * P + ky, ix = px * P + kx;
                            col[(size_t)(py * G + px) * KP + c * P * P + ky * P + kx] =
                                round_f16(img_hwc[((size_t)iy * S + ix) * CH + c]);
                        }
        linear(&m->patch_w, m->patch_b, col, NP, x + D); /* f16 x f16: rounding col again is a no-op */
        for (int p = 0; p < NP; ++p)
            for (int o = 0; o < D; ++o) x[(size_t)(1 + p) * D + o] += m->pos[(size_t)(1 + p) * D + o];
        for (int o = 0; o < D; ++o) x[o] = m->cls[o] + m->pos[o];
        free(col);
    }
    if (taps && taps->embed) memcpy(taps->embed, x, (size_t)N * D * sizeof(float));

    for (int il = 0; il < m->layers; ++il) {
        const vo_layer *L = &m->L[il];
        const int tap = taps && taps->layer == il;

        layernorm(x, N, D, L->norm1_w, L->norm1_b, m->eps, cur);                /* vit.cpp:808-812 */
        if (tap && taps->ln1) memcpy(taps->ln1, cur, (size_t)N * D * sizeof(float));
        linear(&L->qkv, L->qkv_b, cur, N, qkv);                                 /* vit.cpp:820-821 */
        if (g_variant == 2) for (size_t i = 0; i < (size_t)N * 3 * D; ++i) qkv[i] = round_f16(qkv[i]);
        if (g_variant == 7) for (size_t i = 0; i < (size_t)N * 3 * D; ++i) { const float hi = round_f16(qkv[i]); qkv[i] = hi + round_f16(qkv[i] - hi); }
        if (g_variant >= 3 && g_variant <= 6) {
            const int c0 = g_variant == 3 ? 2 * D : (g_variant == 6 ? D : 0);
            const int c1 = g_variant == 3 ? 3 * D : (g_variant == 5 ? D : 2 * D);
            for (int t = 0; t < N; ++t) for (int d = c0; d < c1; ++d) qkv[(size_t)t * 3 * D + d] = round_f16(qkv[(size_t)t * 3 * D + d]);
        }
        if (tap && taps->qkv) memcpy(taps->qkv, qkv, (size_t)N * 3 * D * sizeof(float));

        { att_ctx ac = {qkv, att, N, D, hd}; par_for(H, attention_heads, &ac); }
        if (tap && taps->attn) memcpy(taps->attn, att, (size_t)N * D * sizeof(float));

        linear(&L->proj, L->proj_b, att, N, tmp);                               /* vit.cpp:868-869 */
        for (size_t i = 0; i < (size_t)N * D; ++i) x[i] = tmp[i] + x[i];        /* vit.cpp:873 */
        if (tap && taps->x1) memcpy(taps->x1, x, (size_t)N * D * sizeof(float));

        layernorm(x, N, D, L->norm2_w, L->norm2_b, m->eps, cur);                /* vit.cpp:881-885 */
        if (tap && taps->ln2) memcpy(taps->ln2, cur, (size_t)N * D * sizeof(float));
        linear(&L->fc1, L->fc1_b, cur, N, hbuf);                                /* vit.cpp:889-890 */
        for (size_t i = 0; i < (size_t)N * 4 * D; ++i) hbuf[i] = g_tab_gelu[f16_bits(hbuf[i])]; /* vit.cpp:893, ggml.c:1434-1441 */
        if (tap && taps->h) memcpy(taps->h, hbuf, (size_t)N * 4 * D * sizeof(float));
        linear(&L->fc2, L->fc2_b, hbuf, N, tmp);                                /* vit.cpp:896-897 */
        for (size_t i = 0; i < (size_t)N * D; ++i) x[i] = tmp[i] + x[i];        /* vit.cpp:900 */
        if (tap && taps->x2) memcpy(taps->x2, x, (size_t)N * D * sizeof(float));
    }
    if (taps && taps->x_final) memcpy(taps->x_final, x, (size_t)N * D * sizeof(float));

    /* --- pool + head (vit.cpp:910-933): token 0 (the first TH tokens for ViTSTR, vitstr.cpp:864-903), LN, head linear,
     * f16-table softmax per token */
    float *cl = (float *)malloc((size_t)TH * D * sizeof(float));
    float *lg = (float *)malloc((size_t)TH * m->classes * sizeof(float));
    layernorm(x, TH, D, m->norm_w, m->norm_b, m->eps, cl);
    if (taps && taps->final_ln) memcpy(taps->final_ln, cl, (size_t)D * sizeof(float));
    linear(&m->head, m->head_b, cl, TH, lg);
    if (logits_out) memcpy(logits_out, lg, (size_t)TH * m->classes * sizeof(float));
    if (probs_out) {
        for (int t = 0; t < TH; ++t) softmax_row(lg + (size_t)t * m->classes, m->classes);
        memcpy(probs_out, lg, (size_t)TH * m->classes * sizeof(float));
    }
    free(cl); free(lg); free(x); free(cur); free(qkv); free(att); free(hbuf); free(tmp);
    return 0;
}

/* Stand-alone primitives, exported so tests can pin them one by one. */
void vo_round_f16(const float *x, float *y, int64_t n) { for (int64_t i = 0; i < n; ++i) y[i] = round_f16(x[i]); }
void vo_gelu_table(const float *x, float *y, int64_t n) { init_tables(); for (int64_t i = 0; i < n; ++i) y[i] = g_tab_gelu[f16_bits(x[i])]; }
void vo_exp_table(const float *x, float *y, int64_t n) { init_tables(); for (int64_t i = 0; i < n; ++i) y[i] = g_tab_exp[f16_bits(x[i])]; }
void vo_softmax_rows(float *p, int rows, int n) { init_tables(); for (int r = 0; r < rows; ++r) softmax_row(p + (size_t)r * n, n); }
void vo_layernorm(const float *x, int T, int D, const float *w, const float *b, float eps, float *y) { layernorm(x, T, D, w, b, eps, y); }
void vo_set_threads(int n) { g_threads = n; }
/* Test helper for the q8_0 GEMM prototype: ONE q8_0 linear layer, y[T][N] = W x + b, exactly as the reference evaluates it
 * (quantize_row_q8_0 on every activation row, then ggml_vec_dot_q8_0_q8_0 per output, ggml.c:9493-9506 + ggml-quants.c:702-790,
 * 3521+).  wblocks = the tensor as stored in the model file ([N][K/32] block_q8_0).  xd_out [T][K/32] / xq_out [T][K] (optional)
 * receive the quantised activations. */
void vo_linear_q8_0(int T, int N, int K, const void *wblocks, const float *bias, const float *x, float *y, float *xd_out, int8_t *xq_out) {
    vo_mat W;
    mat_init(&W, wblocks, 8, N, K);
    linear(&W, bias, x, T, y);
    if (xd_out && xq_out)
        for (int t = 0; t < T; ++t) quantize_row_q8_0(x + (size_t)t * K, K, xd_out + (size_t)t * (K / QK8_0), xq_out + (size_t)t * K);
    mat_free(&W);
}

