// engine_internal.h -- the GPU context, the row-band session and the helpers shared by engine.cu (plane driver, C ABI) and
// engine_band.cu (row-band sessions, peer-memory halo exchange, the one-process multi-GPU driver).  Not installed.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges cost a few nanoseconds when no tool is attached

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "kernels.h"
#include "w2x_internal.h"

namespace w2x {
namespace eng {

struct DevModel {                       // device-resident copy of one model
    std::vector<float *> w;             // per layer [Cout][Cin][9] fp32
    std::vector<float *> b;             // per layer [Cout] fp32  ((float)bias, src/modelHandler.cpp:147)
    std::vector<std::vector<float>> b_host;   // the same on the host (the tcgen05 kernels take them as kernel parameters)
    std::vector<uint16_t *> pack;       // per layer tcgen05 operand image (nullptr if not eligible)
    std::vector<uint8_t *> pack8;       // same for the "f8" flavour (fp16 main product + e4m3 corrections)
    std::vector<uint8_t *> strip, strip8;   // row-strip kernel images of the narrow layers (nullptr otherwise), both flavours
    std::vector<float> out_scale;       // 1 / (wscale * ACT_SCALE)
    std::vector<float> last_w_t;        // HOST: last layer's weights transposed to [9][Cin] (fused last layer, passed as kernel parameters)
};

struct TimedSpan { int layer; cudaEvent_t e0, e1; };

}  // namespace eng
}  // namespace w2x

struct w2x_ctx {
    int device = 0;
    int num_sms = 0;
    int cc_major = 0, cc_minor = 0;
    int engine = W2X_ENGINE_AUTO;
    int walk = W2X_WALK_FUSED;
    bool fuse_last = true;             // fold the N->1 last layer into the preceding tcgen05 layer's epilogue
    int precision = W2X_PRECISION_F16_F8X2;   // default; W2X_PRECISION=f16x3 in the environment or w2x_ctx_set_precision() selects the 3 x fp16 scheme
    int strip = 1;                     // 1 = run the narrow layers (Cin, Cout <= 64) on the row-strip kernel; w2x_debug_set_strip(0) = 16x16-tile kernel
    int pair = 1;                      // 1 = run the 128-wide layers on CTA pairs (cta_group::2); w2x_debug_set_pair(0) = single-CTA kernels
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    size_t scratch_limit = (size_t)16 << 30;
    w2x_log_fn log = nullptr;
    void *log_user = nullptr;
    bool log_muted = false;            // the reference's line sequence of the current call has already been emitted
    uint64_t launches = 0;
    bool timing = false;
    std::vector<w2x::eng::TimedSpan> spans;
    std::vector<cudaEvent_t> event_pool;
    std::vector<std::string> layer_kernel;
    std::map<uint64_t, w2x::eng::DevModel> models;
    // scratch
    void *buf[2] = {nullptr, nullptr};
    size_t buf_bytes[2] = {0, 0};
    float *pad_buf = nullptr;
    size_t pad_bytes = 0;
    float *io_buf[2] = {nullptr, nullptr};   // device staging for the host-buffer entry points
    size_t io_bytes[2] = {0, 0};
    bool tc_ready = false;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;   // host<->device copies of w2x_convert_plane overlap the compute stream
    cudaEvent_t ev_in[8] = {}, ev_done[8] = {};
    int host_bands = 0;                                   // 0 = automatic (up to 4 bands of >= 512 rows), 1 = no pipelining
    unsigned long long *prof_buf = nullptr;   // [16 layers][PROF_MAX_CTAS][PROF_WORDS], debug profile
    std::vector<w2x_image *> images;          // live w2x_image handles of this context (engine_image.cu)
};

// One rank's rows of a plane (w2x_band_*): every intermediate activation keeps only the band's rows plus one halo row per
// neighbour side; the halo rows are written by the neighbours (peer memory) or by the caller (w2x_band_halo segments).
struct w2x_band {
    w2x_ctx *ctx = nullptr;
    const w2x_model *model = nullptr;
    w2x::eng::DevModel *dm = nullptr;
    int width = 0, rows = 0, n = 0;
    bool up = false, down = false; // a neighbour GPU owns the rows above / below: one halo row, exchanged after every layer
    bool ov_up = false, ov_down = false;   // the n rows above / below are REAL input rows supplied with the band (recomputed overlap, no exchange)
    int pt = 0, pb = 0;            // frame rows above / below the band: 1 (neighbour halo) or n (image border: replicated; overlap: real rows)
    int pw = 0, hf = 0;            // frame width / height
    float *pad = nullptr;          // padded fp32 input frame
    __half *act[2] = {nullptr, nullptr};
    size_t act_bytes = 0;
    int cur = 0;                   // act[cur] holds the output of the last queued step
    int last_step = -1;
    // peer-memory exchange (w2x_band_connect* / w2x_band_exchange)
    unsigned *flags = nullptr;     // [0] "rows from the up neighbour have landed", [1] same from down, [4] block counter
    unsigned seq = 0;              // exchanges issued so far: the value the next one publishes / waits for is seq + 1
    struct Peer {
        float *pad = nullptr;
        char *act[2] = {nullptr, nullptr};
        unsigned *flags = nullptr;
        int hf = 0;
        bool ipc = false;          // mapped with cudaIpcOpenMemHandle (closed in w2x_band_destroy)
    } peer[2];                     // 0 = up, 1 = down
};

namespace w2x {
namespace eng {

#define CU_CHECK(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(W2X_ERR_CUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e__), __FILE__, __LINE__, \
                        cudaGetErrorString(e__));                                                   \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ---- helpers defined in engine.cu --------------------------------------------------------------------------------------
int ensure(void **p, size_t *have, size_t need);
int get_dev_model(w2x_ctx *ctx, const w2x_model *m, DevModel **out);
cudaEvent_t take_event(w2x_ctx *ctx);
void note_kernel(w2x_ctx *ctx, int layer, const char *name);
int ensure_tc(w2x_ctx *ctx);
int check_ctx(w2x_ctx *ctx);
int pick_engine(w2x_ctx *ctx, const w2x_model *m);
void emit_reference_progress(w2x_ctx *ctx, int w, int h, int n_layers, bool split);   // the reference's stdout lines of one convertWithModels call
bool layer_is_strip(const w2x_ctx *ctx, const w2x_model *m, const DevModel *dm, int li);   // does layer li run on the row-strip kernel?
// One tcgen05 layer `li` on frames of pw x ph: in -> out (or, fused with the last layer, -> per-pixel tap partials in `out`).
// Only frame rows [out_y0, out_y0 + out_rows) are stored (out_rows < 0: the whole frame).
int launch_layer_tc(w2x_ctx *ctx, const w2x_model *m, DevModel *dm, int li, const __half *in, __half *out, int pw, int ph,
                    bool fused, bool profile, int out_y0 = 0, int out_rows = -1);
// convertWithModels on device buffers (rows_above / rows_below: real neighbour rows available around the band)
int convert_device(w2x_ctx *ctx, const w2x_model *m, const float *d_in, int w, int h, size_t in_stride_bytes, int rows_above,
                   int rows_below, float *d_out, size_t out_stride_bytes, int block_splitting);

int tiles_enqueue_compute(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles, int n_tiles, int width, int height, size_t in_stride_bytes);
int tiles_enqueue_download(w2x_ctx *ctx, float *const *out_tiles, int n_tiles, int width, int height, size_t out_stride_bytes);

struct LogMute {   // silences the per-launch lines while a caller that already emitted the reference's sequence runs the layers
    w2x_ctx *ctx;
    bool prev;
    explicit LogMute(w2x_ctx *c, bool on) : ctx(c), prev(c->log_muted) { if (on) c->log_muted = true; }
    ~LogMute() { ctx->log_muted = prev; }
};

// engine_image.cu: w2x_ctx_destroy releases the device buffers of the context's images that are still alive
void release_images(w2x_ctx *ctx);

struct NvtxRange {    // a named range on the calling thread's timeline (nsys / ncu --nvtx), e.g. "w2x L3", "w2x halo exchange"
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

struct LayerTimer {   // brackets one layer launch with an NVTX range, and with events when timing is on
    w2x_ctx *ctx;
    TimedSpan span{};
    bool on;
    LayerTimer(w2x_ctx *c, int layer) : ctx(c), on(c->timing) {
        char name[24];
        snprintf(name, sizeof name, "w2x L%d", layer);
        nvtxRangePushA(name);
        if (on) {
            span.layer = layer;
            span.e0 = take_event(c);
            span.e1 = take_event(c);
            cudaEventRecord(span.e0, c->stream);
        }
    }
    ~LayerTimer() {
        if (on) {
            cudaEventRecord(span.e1, ctx->stream);
            ctx->spans.push_back(span);
        }
        nvtxRangePop();
    }
};

}  // namespace eng
}  // namespace w2x
