// image_math.h -- per-pixel arithmetic of the image plumbing around the conv hot path (reference src/main.cpp:74-76,
// 135-146, 158-167, 171-172), shared by the device kernels (image.cu) and host checks.
//
// Every function restates one routine of host/imgproc.hpp with the same fp32 / fp64 operations in the same order, so the
// device path is bit-identical to the host path.  nvcc contracts a*b+c into FFMA / DFMA by default and the host code has no
// FMA, so all arithmetic goes through mul / add / sub below: __fmul_rn / __fadd_rn / __fsub_rn / __dmul_rn / __dadd_rn /
// __dsub_rn on the device (never contracted), plain operators on the host.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define W2X_HD __host__ __device__ __forceinline__
#else
#define W2X_HD inline
#endif

namespace w2x {
namespace img {

#ifdef __CUDA_ARCH__
W2X_HD float mul(float a, float b) { return __fmul_rn(a, b); }
W2X_HD float add(float a, float b) { return __fadd_rn(a, b); }
W2X_HD float sub(float a, float b) { return __fsub_rn(a, b); }
W2X_HD double mul(double a, double b) { return __dmul_rn(a, b); }
W2X_HD double add(double a, double b) { return __dadd_rn(a, b); }
W2X_HD double sub(double a, double b) { return __dsub_rn(a, b); }
W2X_HD uint32_t bits(float v) { return __float_as_uint(v); }
#else
W2X_HD float mul(float a, float b) { return a * b; }
W2X_HD float add(float a, float b) { return a + b; }
W2X_HD float sub(float a, float b) { return a - b; }
W2X_HD double mul(double a, double b) { return a * b; }
W2X_HD double add(double a, double b) { return a + b; }
W2X_HD double sub(double a, double b) { return a - b; }
W2X_HD uint32_t bits(float v) { uint32_t b; memcpy(&b, &v, 4); return b; }
#endif
W2X_HD int imin(int a, int b) { return a < b ? a : b; }
W2X_HD int imax(int a, int b) { return a > b ? a : b; }

// from_u8 + rgb2yuv: one 8-bit pixel (channel 0 is treated as "R", as the reference does with B,G,R data) -> Y, U, V
W2X_HD void bgr8_to_yuv(const uint8_t *px, float *Y, float *U, float *V) {
    const float a = (float)(1.0 / 255.0);
    const float c0 = mul((float)px[0], a), c1 = mul((float)px[1], a), c2 = mul((float)px[2], a);
    const float y = add(add(mul(c0, 0.299f), mul(c1, 0.587f)), mul(c2, 0.114f));
    *Y = y;
    *U = add(mul(sub(c2, y), 0.492f), 0.5f);
    *V = add(mul(sub(c0, y), 0.877f), 0.5f);
}

// to_u8_span: saturate first (NaN -> 0), then round half to even by adding 2^23
W2X_HD uint8_t to_u8(float x) {
    float v = mul(x, 255.0f);
    v = v > 0.f ? v : 0.f;
    v = v < 255.f ? v : 255.f;
    return (uint8_t)(bits(add(v, 8388608.0f)) & 0xFFu);
}

// yuv2rgb + to_u8: Y, U, V -> one 8-bit pixel (c0, c1, c2)
W2X_HD void yuv_to_bgr8(float Y, float U, float V, uint8_t *px) {
    const float c2 = add(Y, mul(sub(U, 0.5f), 2.032f));
    const float c1 = add(add(Y, mul(sub(V, 0.5f), -0.581f)), mul(sub(U, 0.5f), -0.395f));
    const float c0 = add(Y, mul(sub(V, 0.5f), 1.14f));
    px[0] = to_u8(c0);
    px[1] = to_u8(c1);
    px[2] = to_u8(c2);
}

// INTER_NEAREST source index: min(floor(d * scale), limit - 1), scale = src / dst in double
W2X_HD int nearest_index(int d, double scale, int limit) { return imin((int)floor(mul((double)d, scale)), limit - 1); }

// source coordinate of output d: fd = (d + 0.5) * scale - 0.5 in double, s = floor(fd), fraction rounded to float once
W2X_HD void source_coord(double scale, int d, int *s, float *f) {
    const double fd = sub(mul(add((double)d, 0.5), scale), 0.5);
    *s = (int)floor(fd);
    *f = (float)sub(fd, (double)*s);
}

// `coeffs` of resize(..., LINEAR)
W2X_HD void linear_coeffs(double scale, int d, int limit, int *idx, float *w) {
    int s;
    float f;
    source_coord(scale, d, &s, &f);
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= limit - 1) { f = 0.f; s = limit - 1; }
    idx[0] = s;
    idx[1] = imin(s + 1, limit - 1);
    w[0] = sub(1.f, f);
    w[1] = f;
}

// `coeffs` of resize(..., CUBIC), A = -0.75: w3 = ((1 - w0) - w1) - w2, taps clamped to the image
W2X_HD void cubic_coeffs(double scale, int d, int limit, int *idx, float *w) {
    int s;
    float f;
    source_coord(scale, d, &s, &f);
    const float A = -0.75f;
    const float f1 = add(f, 1.f), g = sub(1.f, f);
    w[0] = sub(mul(add(mul(sub(mul(A, f1), 5 * A), f1), 8 * A), f1), 4 * A);
    w[1] = add(mul(mul(sub(mul(A + 2, f), A + 3), f), f), 1.f);
    w[2] = add(mul(mul(sub(mul(A + 2, g), A + 3), g), g), 1.f);
    w[3] = sub(sub(sub(1.f, w[0]), w[1]), w[2]);
    for (int k = 0; k < 4; k++) idx[k] = imin(imax(s - 1 + k, 0), limit - 1);
}

// horizontal pass at one source row: ((0 + s0 w0) + s1 w1) + ...
template <int NTAP>
W2X_HD float hsum(const float *row, const int *xi, const float *xw) {
    float a = 0.f;
    for (int k = 0; k < NTAP; k++) a = add(a, mul(row[xi[k]], xw[k]));
    return a;
}

// one output pixel of resize(plane, LINEAR | CUBIC) = vertical pass over horizontal passes (the same values the two-pass
// host routine stores in its temporary rows): 4 taps ((r0 w0 + r1 w1) + r2 w2) + r3 w3, 2 taps r0 w0 + r1 w1
template <int NTAP>
W2X_HD float sample(const float *plane, long stride, const int *xi, const float *xw, const int *yi, const float *yw) {
    float r[NTAP];
    for (int k = 0; k < NTAP; k++) r[k] = hsum<NTAP>(plane + (long)yi[k] * stride, xi, xw);
    if (NTAP == 4) return add(add(add(mul(r[0], yw[0]), mul(r[1], yw[1])), mul(r[2], yw[2])), mul(r[NTAP - 1], yw[NTAP - 1]));
    return add(mul(r[0], yw[0]), mul(r[NTAP - 1], yw[NTAP - 1]));
}

}  // namespace img
}  // namespace w2x
