// image.cu -- the image plumbing around the conv hot path on the device: 8-bit B,G,R <-> planar fp32 Y, U, V and the
// nearest / bicubic / bilinear resizes of the reference's main.cpp (src/main.cpp:74-76, 135-146, 158-167, 171-172).
// Memory-bound elementwise and gather kernels, one thread per output pixel; the arithmetic is image_math.h, which keeps
// host/imgproc.hpp's operations and their order, so the results are bit-identical to the host path.
#include <cuda_runtime.h>

#include "image_math.h"
#include "kernels.h"

namespace w2x {
namespace {

constexpr int TX = 32, TY = 8;

dim3 grid_of(int w, int h) { return dim3((unsigned)((w + TX - 1) / TX), (unsigned)((h + TY - 1) / TY)); }

__global__ void __launch_bounds__(TX *TY) k_bgr8_to_yuv(const uint8_t *__restrict__ bgr, size_t stride, int w, int h,
                                                         float *__restrict__ Y, float *__restrict__ U, float *__restrict__ V) {
    const int x = blockIdx.x * TX + threadIdx.x, y = blockIdx.y * TY + threadIdx.y;
    if (x >= w || y >= h) return;
    const size_t o = (size_t)y * w + x;
    img::bgr8_to_yuv(bgr + (size_t)y * stride + (size_t)x * 3, Y + o, U + o, V + o);
}

__global__ void __launch_bounds__(TX *TY) k_yuv_to_bgr8(const float *__restrict__ Y, const float *__restrict__ U,
                                                         const float *__restrict__ V, int w, int h, uint8_t *__restrict__ bgr,
                                                         size_t stride) {
    const int x = blockIdx.x * TX + threadIdx.x, y = blockIdx.y * TY + threadIdx.y;
    if (x >= w || y >= h) return;
    const size_t o = (size_t)y * w + x;
    img::yuv_to_bgr8(Y[o], U[o], V[o], bgr + (size_t)y * stride + (size_t)x * 3);
}

__global__ void __launch_bounds__(TX *TY) k_resize_nearest(const float *__restrict__ src, int sw, int sh, float *__restrict__ dst,
                                                            int dw, int dh, double sx, double sy) {
    const int x = blockIdx.x * TX + threadIdx.x, y = blockIdx.y * TY + threadIdx.y;
    if (x >= dw || y >= dh) return;
    dst[(size_t)y * dw + x] = src[(size_t)img::nearest_index(y, sy, sh) * sw + img::nearest_index(x, sx, sw)];
}

// NTAP = 4: bicubic, NTAP = 2: bilinear; planes [0, n_planes) of src / dst share one geometry
template <int NTAP>
__global__ void __launch_bounds__(TX *TY) k_resize(ResizePlanes p, int n_planes, int sw, int sh, int dw, int dh, double sx, double sy) {
    const int x = blockIdx.x * TX + threadIdx.x, y = blockIdx.y * TY + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int xi[4], yi[4];
    float xw[4], yw[4];
    if (NTAP == 4) {
        img::cubic_coeffs(sx, x, sw, xi, xw);
        img::cubic_coeffs(sy, y, sh, yi, yw);
    } else {
        img::linear_coeffs(sx, x, sw, xi, xw);
        img::linear_coeffs(sy, y, sh, yi, yw);
    }
#pragma unroll
    for (int c = 0; c < 3; c++)   // unrolled: the plane pointers stay in registers
        if (c < n_planes) p.dst[c][(size_t)y * dw + x] = img::sample<NTAP>(p.src[c], sw, xi, xw, yi, yw);
}

}  // namespace

cudaError_t launch_bgr8_to_yuv(const uint8_t *bgr, size_t stride_bytes, int w, int h, float *Y, float *U, float *V, cudaStream_t s) {
    k_bgr8_to_yuv<<<grid_of(w, h), dim3(TX, TY), 0, s>>>(bgr, stride_bytes, w, h, Y, U, V);
    return cudaGetLastError();
}

cudaError_t launch_yuv_to_bgr8(const float *Y, const float *U, const float *V, int w, int h, uint8_t *bgr, size_t stride_bytes, cudaStream_t s) {
    k_yuv_to_bgr8<<<grid_of(w, h), dim3(TX, TY), 0, s>>>(Y, U, V, w, h, bgr, stride_bytes);
    return cudaGetLastError();
}

cudaError_t launch_resize_nearest(const float *src, int sw, int sh, float *dst, int dw, int dh, cudaStream_t s) {
    k_resize_nearest<<<grid_of(dw, dh), dim3(TX, TY), 0, s>>>(src, sw, sh, dst, dw, dh, (double)sw / dw, (double)sh / dh);
    return cudaGetLastError();
}

cudaError_t launch_resize(const ResizePlanes &p, int n_planes, int sw, int sh, int dw, int dh, bool cubic, cudaStream_t s) {
    const double sx = (double)sw / dw, sy = (double)sh / dh;   // scale = src / dst in double, as host/imgproc.hpp computes it
    if (cubic) k_resize<4><<<grid_of(dw, dh), dim3(TX, TY), 0, s>>>(p, n_planes, sw, sh, dw, dh, sx, sy);
    else k_resize<2><<<grid_of(dw, dh), dim3(TX, TY), 0, s>>>(p, n_planes, sw, sh, dw, dh, sx, sy);
    return cudaGetLastError();
}

}  // namespace w2x
