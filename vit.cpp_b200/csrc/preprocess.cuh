// preprocess.cuh -- vit_image_preprocess on the GPU (SURVEY.md 8(f) rank 1): u8 RGB image of any size -> bicubic (default) or
// bilinear resize to img_size^2 -> round to u8 -> (v - mean_c) / std_c -> image_f32 (HWC f32, vit.h:98-103), written straight
// into the engine's input buffer.  One thread per output pixel (three channels).
//
// The arithmetic reproduces the reference build operation for operation, including its quirks (reference vit.cpp:204-287):
//  * sampling position tx*j with NO half-pixel offset, clamp-to-edge taps, no anti-aliasing;
//  * cubic coefficients evaluated in DOUBLE (the literals -1.0/3, 1.0/6 promote the expression) and narrowed to float;
//  * the float polynomial a0 + a1 t + a2 t^2 + a3 t^3 with the fused multiply-adds gcc emits under -ffp-contract=fast
//    (checked in the disassembly of the reference build): fma(a1,t,a0); fma(a2*t,t,.); fma((a3*t)*t,t,.);
//  * the result is rounded to u8 (round half away from zero, clamped) BEFORE normalisation (vit.cpp:279-280);
//  * bilinear (vit.cpp:130-196) uses half-pixel centres: sx = fma(x+0.5, scale, -0.5), and each of its three lerps
//    u * (1 - t) + v * t is one fma(u, 1 - t, v * t), as in the reference build, for every channel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vitb200 {

struct PreImage
{
    size_t offset; // byte offset of this image's RGB data in the staging buffer
    int nx, ny;
};

__device__ __forceinline__ int pre_clipi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

__device__ __forceinline__ float pre_cubic(float p0, float p1, float p2, float p3, float t)
{
    const float d0 = p0 - p1, d2 = p2 - p1, d3 = p3 - p1, a0 = p1;
    const float a1 = (float)fma(-(1.0 / 6), (double)d3, fma(-1.0 / 3, (double)d0, (double)d2));
    const float a2 = (float)fma(1.0 / 2, (double)d0, (1.0 / 2) * (double)d2);
    const float a3 = (float)fma(1.0 / 6, (double)d3, fma(-(1.0 / 2), (double)d2, (-1.0 / 6) * (double)d0));
    float r = __fmaf_rn(a1, t, a0);
    r = __fmaf_rn(__fmul_rn(a2, t), t, r);
    r = __fmaf_rn(__fmul_rn(__fmul_rn(a3, t), t), t, r);
    return r;
}

// out (image_f32 batch, may be NULL) and/or patches (may be NULL): the f16 patch matrix the patch-embedding GEMM reads through TMA,
// row = (image, patch), k = c*P*P + ky*P + kx (ggml.c:11597-11599), row pitch ldk -- written directly so that the f32 image never
// exists in HBM on the u8 path (the reference rounds the pixels to f16 for the conv anyway, ggml.c:11599).
__global__ void preprocess_kernel(const uint8_t *__restrict__ staging, const PreImage *__restrict__ imgs, float *__restrict__ out,
                                  int S, int bilinear, __half *__restrict__ patches, int P, int ldk)
{
    const int b = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= S * S) return;
    const int i = idx / S, j = idx - i * S; // output row, column
    const PreImage im = imgs[b];
    const uint8_t *src = staging + im.offset;
    const int nx = im.nx, ny = im.ny;
    const float m3[3] = {123.675f, 116.280f, 103.530f}; // vit.cpp:233-234
    const float s3[3] = {58.395f, 57.120f, 57.375f};
    float px3[3];
    float *dst = px3;
    if (!bilinear)
    {
        const float tx = __fdiv_rn((float)nx, (float)S), ty = __fdiv_rn((float)ny, (float)S);
        const float fx = __fmul_rn(tx, (float)j), fy = __fmul_rn(ty, (float)i);
        const int x = (int)fx, y = (int)fy;
        const float dx = fx - (float)x, dy = fy - (float)y;
        const int xs[4] = {pre_clipi(x - 1, 0, nx - 1), pre_clipi(x, 0, nx - 1), pre_clipi(x + 1, 0, nx - 1), pre_clipi(x + 2, 0, nx - 1)};
#pragma unroll
        for (int k = 0; k < 3; ++k)
        {
            float C[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
            {
                const uint8_t *row = src + (size_t)pre_clipi(y - 1 + jj, 0, ny - 1) * nx * 3;
                C[jj] = pre_cubic((float)row[xs[0] * 3 + k], (float)row[xs[1] * 3 + k], (float)row[xs[2] * 3 + k], (float)row[xs[3] * 3 + k], dx);
            }
            const float Cc = pre_cubic(C[0], C[1], C[2], C[3], dy);
            const float v = fminf(fmaxf(roundf(Cc), 0.0f), 255.0f);
            dst[k] = __fdiv_rn((float)(uint8_t)v - m3[k], s3[k]);
        }
    }
    else
    {
        const float x_scale = __fdiv_rn((float)nx, (float)S), y_scale = __fdiv_rn((float)ny, (float)S);
        const float sx = __fmaf_rn((float)j + 0.5f, x_scale, -0.5f), sy = __fmaf_rn((float)i + 0.5f, y_scale, -0.5f);
        const int x0 = max(0, (int)floorf(sx)), y0 = max(0, (int)floorf(sy));
        const int x1 = min(x0 + 1, nx - 1), y1 = min(y0 + 1, ny - 1);
        const float dx = sx - (float)x0, dy = sy - (float)y0;
#pragma unroll
        for (int k = 0; k < 3; ++k)
        {
            const float v00 = src[3 * ((size_t)y0 * nx + x0) + k], v01 = src[3 * ((size_t)y0 * nx + x1) + k];
            const float v10 = src[3 * ((size_t)y1 * nx + x0) + k], v11 = src[3 * ((size_t)y1 * nx + x1) + k];
            const float v0 = __fmaf_rn(v00, 1.0f - dx, __fmul_rn(v01, dx));
            const float v1 = __fmaf_rn(v10, 1.0f - dx, __fmul_rn(v11, dx));
            const float v = __fmaf_rn(v0, 1.0f - dy, __fmul_rn(v1, dy));
            const float r = fminf(fmaxf(roundf(v), 0.0f), 255.0f);
            dst[k] = __fdiv_rn((float)(uint8_t)r - m3[k], s3[k]);
        }
    }
    if (out)
    {
        float *o = out + ((size_t)b * S * S + idx) * 3;
        o[0] = px3[0]; o[1] = px3[1]; o[2] = px3[2];
    }
    if (patches)
    {
        const int G = S / P, py = i / P, ky = i - py * P, pxi = j / P, kx = j - pxi * P;
        __half *row = patches + ((size_t)b * G * G + (size_t)py * G + pxi) * ldk + ky * P + kx;
#pragma unroll
        for (int k = 0; k < 3; ++k) row[k * P * P] = __float2half_rn(px3[k]);
    }
}

} // namespace vitb200
