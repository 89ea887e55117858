// kernels.h -- launchers of every kernel in the library (device code lives in the .cu files).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace w2x {

// ---- kernels_fp32.cu --------------------------------------------------------------------------
cudaError_t launch_pad_replicate(const float *in, int w, int h, long in_stride_floats, int pad, int rows_above,
                                 int rows_below, float *out, cudaStream_t s);
// general form: horizontal pad pad_x, vertical pads pad_top / pad_bottom (row-band sessions)
// skip_top / skip_bottom: frame rows at the top / bottom that are NOT written (a neighbour GPU stores them)
cudaError_t launch_pad_replicate_xy(const float *in, int w, int h, long in_stride_floats, int pad_x, int pad_top,
                                    int pad_bottom, int rows_above, int rows_below, float *out, cudaStream_t s,
                                    int skip_top = 0, int skip_bottom = 0);
// Peer-memory halo exchange (engine_band.cu): ONE kernel copies up to 8 row segments into the neighbour GPUs' frames,
// publishes `value` in their flag words once every byte is visible system-wide, then waits until the neighbours have
// published the same value here.  Flag values only grow, so nothing is ever reset.
struct HaloXArgs {
    int n;                       // segments
    const char *src[8];
    char *dst[8];
    size_t bytes;                // per segment (multiple of 4)
    unsigned *counter;           // block-completion counter in this GPU's memory (self-resetting)
    unsigned *peer_flag[2];      // where to publish (nullptr = no neighbour on that side)
    const unsigned *my_flag[2];  // what to wait for
    unsigned value;
};
cudaError_t launch_halo_exchange(const HaloXArgs &a, cudaStream_t s);
cudaError_t launch_crop(const float *in, int w, int h, int pad, float *out, long out_stride_floats, cudaStream_t s);
cudaError_t launch_copy2d(const float *in, long in_stride_floats, float *out, long out_stride_floats, int w, int h,
                          cudaStream_t s);
cudaError_t launch_conv3x3_fp32(const float *in, float *out, const float *wgt, const float *bias, int Cin, int Cout,
                                int W, int H, cudaStream_t s);

// ---- image.cu: whole-image plumbing on dense planar fp32 Y, U, V planes (bit-identical to host/imgproc.hpp) -----------
// interleaved 8-bit B,G,R (row stride in bytes) <-> three dense w x h planes
cudaError_t launch_bgr8_to_yuv(const uint8_t *bgr, size_t stride_bytes, int w, int h, float *Y, float *U, float *V, cudaStream_t s);
cudaError_t launch_yuv_to_bgr8(const float *Y, const float *U, const float *V, int w, int h, uint8_t *bgr, size_t stride_bytes,
                               cudaStream_t s);
cudaError_t launch_resize_nearest(const float *src, int sw, int sh, float *dst, int dw, int dh, cudaStream_t s);
struct ResizePlanes { const float *src[3]; float *dst[3]; };
// bicubic (A = -0.75) or bilinear resize of n_planes (<= 3) dense planes of one geometry
cudaError_t launch_resize(const ResizePlanes &p, int n_planes, int sw, int sh, int dw, int dh, bool cubic, cudaStream_t s);

// ---- kernels_tc.cu ----------------------------------------------------------------------------
namespace tc {
constexpr int REGION = 16;          // a tile-set covers REGION x REGION output pixels (two 8x16 M-tiles)
constexpr int HALO = REGION + 2;    // staged input footprint per side
constexpr float ACT_SCALE = 16.0f;  // activations are stored as fp16 hi/lo of (value * ACT_SCALE)

// Activation frame between layers: 4 bytes per element (RECORD frame, see launch_tc_layer).
inline size_t act_bytes(int C, int Wp, int Hp) { return (size_t)Hp * Wp * C * 4; }

bool layer_supported(int cin, int cout);
size_t layer_smem_bytes(int cin, int cout);
// One-time per process: raise the dynamic shared memory limit of every instantiation.
cudaError_t init_kernels();

// First layer (Cin = 1): same-size 3x3 correlation with BORDER_REPLICATE (src/modelHandler.cpp:141-142) on the frame of pw x ph
// whose pixel (fy, fx) is the source plane's pixel (clamp(fy - pad_top), clamp(fx - pad_x)) -- i.e. cv::copyMakeBorder
// (src/convertRoutine.cpp:35,96) is folded into the loads; pad_x = pad_top = 0 with w x h = pw x ph reads an already padded ROI.
// rows_above / rows_below: real rows readable beyond the plane (row bands).  -> RECORD frame.
// `wgt` ([C][9]) and `bias` ((float)bias) are HOST pointers: they travel as kernel parameters.
struct FirstSource {
    const float *in;
    long stride_floats;
    int w, h, pad_x, pad_top, rows_above, rows_below;
};
cudaError_t launch_first(const FirstSource &src, int pw, int ph, const float *wgt /*[C][9]*/, const float *bias, int cout, __half *out,
                         cudaStream_t s, int f8 = 0, int out_y0 = 0, int out_rows = -1);
// tcgen05 layer: in/out NHWC frames (pw x ph); the tensor maps are built inside.
// `bias` is a HOST pointer to the layer's (float)bias values (they travel as kernel parameters).
// f8 = 0: "f16x3" frames [hi][lo], wpack = TcPack::bytes, wstrip = TcPack::strip;
// f8 = 1: frames [xh][xh8][xl8], wpack = TcPack::bytes8, wstrip = TcPack::strip8.
// wstrip (device copy of the row-strip image, nullptr if the layer has none) selects the row-strip kernel for the
// narrow layers (Cin, Cout <= 64, not fused); the choice depends on the layer shape only, never on the frame size.
cudaError_t launch_tc_layer(const __half *in, const void *wpack, const void *wstrip, const float *bias, __half *out,
                            int cin, int cout, int pw, int ph, float out_scale, int f8, int num_sms,
                            cudaStream_t s, unsigned long long *prof = nullptr, const float *last_w = nullptr,
                            float *partial = nullptr, int pair = 0, int out_y0 = 0, int out_rows = -1);
// Frames: every activation between layers is a RECORD frame [Hp][Wp][C/32][128 B] -- one 128-byte record per pixel per
// 32-channel block = {xh fp16 x32 | xh8 e4m3 x32 | xl8 e4m3 x32} (f8) or {hi fp16 x32 | lo fp16 x32} (f16x3): 4 bytes per
// element, one TMA box row per record (SWIZZLE_128B).
// out_y0 / out_rows (both launchers): only frame rows [out_y0, out_y0 + out_rows) are stored (-1 = the whole frame); a
// row-band session keeps its halo rows out of the window because its neighbours write them.
bool strip_supported(int cin, int cout);
// Fused last layer: launch_tc_layer(..., last_w = HOST pointer to [9][cout] fp32 tap-major, partial = [ph][pw][12] fp32) makes the
// tcgen05 layer emit per-pixel tap partials instead of activations; launch_last_gather sums the 3x3
// neighbourhood of partials, adds the bias, applies the leaky-ReLU and writes the cropped fp32 plane.
cudaError_t launch_last_gather(const float *partial, int pw, int ph, float bias, int crop, float *dst,
                               long dst_stride_floats, cudaStream_t s);
// general form: crop_x columns left/right, crop_top / crop_bottom rows
cudaError_t launch_last_gather_xy(const float *partial, int pw, int ph, float bias, int crop_x, int crop_top,
                                  int crop_bottom, float *dst, long dst_stride_floats, cudaStream_t s);
inline size_t partial_bytes(int Wp, int Hp) { return (size_t)Hp * Wp * 12 * sizeof(float); }
constexpr int PROF_WORDS = 16;      // per-CTA profile record (see tc_config.cuh PROF_*)
constexpr int PROF_MAX_CTAS = 256;
// Last layer (Cout = 1): NHWC hi/lo frame -> fp32 plane, interior only: out(y,x) for
// y in [crop, ph-crop), x in [crop, pw-crop) is written to dst[(y-crop)*stride + (x-crop)].
cudaError_t launch_last(const __half *in, int cin, int pw, int ph, const float *wgt /*[C][9]*/, float bias,
                        int crop, float *dst, long dst_stride_floats, cudaStream_t s, int f8 = 0);
// planar fp32 [C][h][w] -> NHWC hi/lo frame (h+2) x (w+2), replicate ring of 1 (for w2x_filter_layer)
cudaError_t launch_planar_to_nhwc(const float *in, int C, int w, int h, __half *out, cudaStream_t s, int f8 = 0);
// NHWC hi/lo frame (h+2) x (w+2) -> planar fp32 [C][h][w] (interior)
cudaError_t launch_nhwc_to_planar(const __half *in, int C, int w, int h, float *out, cudaStream_t s, int f8 = 0);

}  // namespace tc

}  // namespace w2x
