// engine.cu -- GPU context, plane driver and the compute half of the C ABI.
//
// The plane driver re-creates w2xc::convertWithModels (reference src/convertRoutine.cpp:21-51),
// convertWithModelsBasic (:53-82) and convertWithModelsBlockSplit (:84-169) on top of the layer
// kernels: replicate-pad by nModel, run the layers, crop nModel.  A plane the reference would
// block-split is by default processed whole (every output pixel still sees exactly the operands
// and the operation order it sees inside its reference block, so the result is bit-identical);
// W2X_WALK_BLOCKS walks the reference's blocks literally.
//
// There is no CPU fallback anywhere in this file: without an sm_100 device every compute entry
// point fails with W2X_ERR_NO_DEVICE.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "engine_internal.h"

using namespace w2x;

namespace w2x {
namespace eng {

int ensure(void **p, size_t *have, size_t need) {
    if (*have >= need) return W2X_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    cudaError_t e = cudaMalloc(p, need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(W2X_ERR_NOMEM, "cudaMalloc of %zu bytes failed (%s)", need, cudaGetErrorString(e));
    }
    *have = need;
    return W2X_OK;
}

int get_dev_model(w2x_ctx *ctx, const w2x_model *m, DevModel **out) {
    auto it = ctx->models.find(m->uid);
    if (it != ctx->models.end()) {
        *out = &it->second;
        return W2X_OK;
    }
    DevModel dm;
    const size_t n = m->layers.size();
    dm.w.assign(n, nullptr);
    dm.b.assign(n, nullptr);
    dm.pack.assign(n, nullptr);
    dm.pack8.assign(n, nullptr);
    dm.strip.assign(n, nullptr);
    dm.strip8.assign(n, nullptr);
    dm.out_scale.assign(n, 1.f);
    for (size_t i = 0; i < n; i++) {
        const Layer &L = m->layers[i];
        CU_CHECK(cudaMalloc(&dm.w[i], L.w.size() * sizeof(float)));
        CU_CHECK(cudaMemcpyAsync(dm.w[i], L.w.data(), L.w.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        std::vector<float> bf(L.b.size());
        for (size_t k = 0; k < bf.size(); k++) bf[k] = static_cast<float>(L.b[k]);
        dm.b_host.push_back(bf);
        CU_CHECK(cudaMalloc(&dm.b[i], bf.size() * sizeof(float)));
        CU_CHECK(cudaMemcpyAsync(dm.b[i], bf.data(), bf.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        CU_CHECK(cudaStreamSynchronize(ctx->stream));   // bf goes out of scope
        const TcPack &P = m->tc[i];
        if (!P.bytes.empty()) {
            CU_CHECK(cudaMalloc(&dm.pack[i], P.bytes.size() * 2));
            CU_CHECK(cudaMemcpyAsync(dm.pack[i], P.bytes.data(), P.bytes.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
            dm.out_scale[i] = 1.0f / (P.wscale * tc::ACT_SCALE);
            CU_CHECK(cudaMalloc(&dm.pack8[i], P.bytes8.size()));
            CU_CHECK(cudaMemcpyAsync(dm.pack8[i], P.bytes8.data(), P.bytes8.size(), cudaMemcpyHostToDevice, ctx->stream));
            if (!P.strip.empty()) {
                CU_CHECK(cudaMalloc(&dm.strip[i], P.strip.size()));
                CU_CHECK(cudaMemcpyAsync(dm.strip[i], P.strip.data(), P.strip.size(), cudaMemcpyHostToDevice, ctx->stream));
                CU_CHECK(cudaMalloc(&dm.strip8[i], P.strip8.size()));
                CU_CHECK(cudaMemcpyAsync(dm.strip8[i], P.strip8.data(), P.strip8.size(), cudaMemcpyHostToDevice, ctx->stream));
            }
        }
    }
    if (m->tc_eligible) {
        const Layer &L = m->layers.back();                // n_out == 1: w is [1][Cin][9]
        dm.last_w_t.assign((size_t)9 * L.n_in, 0.f);
        for (int c = 0; c < L.n_in; c++)
            for (int t = 0; t < 9; t++) dm.last_w_t[(size_t)t * L.n_in + c] = L.w[(size_t)c * 9 + t];
    }
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    auto res = ctx->models.emplace(m->uid, std::move(dm));
    *out = &res.first->second;
    return W2X_OK;
}

cudaEvent_t take_event(w2x_ctx *ctx) {
    if (!ctx->event_pool.empty()) {
        cudaEvent_t e = ctx->event_pool.back();
        ctx->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void note_kernel(w2x_ctx *ctx, int layer, const char *name) {
    if ((int)ctx->layer_kernel.size() <= layer) ctx->layer_kernel.resize((size_t)layer + 1);
    ctx->layer_kernel[(size_t)layer] = name;
}

void logf(w2x_ctx *ctx, const char *fmt, int a, int b = 0) {
    if (!ctx->log || ctx->log_muted) return;
    char line[128];
    snprintf(line, sizeof line, fmt, a, b);
    ctx->log(line, ctx->log_user);
}

// The progress lines the reference prints for one convertWithModels call (src/convertRoutine.cpp:67,133-134): per block
// "start process block (c,r) ..." + one "Iteration #k..." per layer when the plane is split, else just the iterations.
// The fused walk and the copy pipeline process the plane in other units, so they emit the reference's sequence up front.
void emit_reference_progress(w2x_ctx *ctx, int w, int h, int n_layers, bool split) {
    if (!ctx->log) return;
    int nb = 1;
    std::vector<int> tab;
    if (split) {
        const Config &cfg = config();
        nb = block_table(w, h, cfg.block_w, cfg.block_h, n_layers, nullptr, 0, nullptr, nullptr);
        if (nb < 1) return;
        tab.resize((size_t)nb * 8);
        block_table(w, h, cfg.block_w, cfg.block_h, n_layers, tab.data(), nb, nullptr, nullptr);
    }
    for (int i = 0; i < nb; i++) {
        if (split) logf(ctx, "start process block (%d,%d) ...", tab[(size_t)i * 8 + 1], tab[(size_t)i * 8]);
        for (int k = 1; k <= n_layers; k++) logf(ctx, "Iteration #%d...", k);
    }
}

int pick_engine(w2x_ctx *ctx, const w2x_model *m) {
    int e = ctx->engine;
    if (e == W2X_ENGINE_AUTO) e = m->tc_eligible ? W2X_ENGINE_TC : W2X_ENGINE_FP32;
    if (e == W2X_ENGINE_TC && !m->tc_eligible) {
        fail(W2X_ERR_UNSUPPORTED, "tcgen05 engine needs a 1->{32,64,128}...->1 layer chain");
        return -1;
    }
    return e;
}

int ensure_tc(w2x_ctx *ctx) {
    if (ctx->tc_ready) return W2X_OK;
    CU_CHECK(tc::init_kernels());
    ctx->tc_ready = true;
    return W2X_OK;
}

// Does layer li run on the row-strip kernel?  A property of the layer's shape and position only, never of the frame size,
// so every tiling of a plane picks the same kernels.
bool layer_is_strip(const w2x_ctx *ctx, const w2x_model *m, const DevModel *dm, int li) {
    const int n = (int)m->layers.size();
    if (li < 1 || li > n - 2 || !ctx->strip) return false;
    const Layer &L = m->layers[(size_t)li];
    const bool fused = ctx->fuse_last && n >= 3 && !dm->last_w_t.empty() && li == n - 2;
    return !fused && tc::strip_supported(L.n_in, L.n_out) && dm->strip[(size_t)li] != nullptr;
}

// One tcgen05 layer `li` on frames of pw x ph: in -> out (or, fused with the last layer, -> per-pixel tap partials in `out`).
int launch_layer_tc(w2x_ctx *ctx, const w2x_model *m, DevModel *dm, int li, const __half *in, __half *out, int pw, int ph,
                    bool fused, bool profile, int out_y0, int out_rows) {
    if (out_rows < 0) { out_y0 = 0; out_rows = ph; }
    const Layer &L = m->layers[(size_t)li];
    const int f8 = ctx->precision == W2X_PRECISION_F16_F8X2 ? 1 : 0;
    const bool strip = !fused && layer_is_strip(ctx, m, dm, li);
    {
        LayerTimer t(ctx, li);
        CU_CHECK(tc::launch_tc_layer(in, f8 ? (const void *)dm->pack8[(size_t)li] : (const void *)dm->pack[(size_t)li],
                                     strip ? (f8 ? (const void *)dm->strip8[(size_t)li] : (const void *)dm->strip[(size_t)li]) : nullptr,
                                     dm->b_host[(size_t)li].data(), out, L.n_in, L.n_out, pw, ph, dm->out_scale[(size_t)li], f8,
                                     ctx->num_sms, ctx->stream,
                                     profile && ctx->prof_buf ? ctx->prof_buf + (size_t)li * tc::PROF_MAX_CTAS * tc::PROF_WORDS : nullptr,
                                     fused ? dm->last_w_t.data() : nullptr, fused ? reinterpret_cast<float *>(out) : nullptr, ctx->pair,
                                     out_y0, out_rows));
    }
    note_kernel(ctx, li, f8 ? (fused ? "tcgen05_f16+f8x2+last" : strip ? "tcgen05_f16+f8x2_strip" : "tcgen05_f16+f8x2")
                            : (fused ? "tcgen05_f16x3+last" : strip ? "tcgen05_f16x3_strip" : "tcgen05_f16x3"));
    ctx->launches++;
    return W2X_OK;
}

// ---- convertWithModelsBasic on an already padded ROI ------------------------------------------
// src: pw x ph fp32 region (row stride src_stride floats) that already contains the n-pixel ring.
// dst: receives the (pw-2n) x (ph-2n) interior.
// n_tiles > 1 (tcgen05 engine with the fused last layer only): src holds n_tiles padded planes of pw x ph stacked vertically; the
// layers run ONCE on the (n_tiles * ph)-row frame -- the seams pollute only the rings that are cropped anyway -- and tile t's
// interior goes to dst + t * (ph - 2n) * dst_stride.
// direct (tcgen05 engine, one plane): the first layer reads the UNPADDED plane it describes and folds the replicate padding into
// its loads; src / src_stride are then unused.
int run_basic(w2x_ctx *ctx, const w2x_model *m, DevModel *dm, int engine, const float *src, long src_stride, int pw,
              int ph, float *dst, long dst_stride, int n_tiles = 1, const tc::FirstSource *direct = nullptr) {
    const int n = (int)m->layers.size();
    if (pw - 2 * n < 1 || ph - 2 * n < 1) return fail(W2X_ERR_ARG, "plane smaller than the model's receptive ring");
    const int tile_ph = ph;
    ph *= n_tiles;
    int maxc = 1;
    for (auto &L : m->layers) maxc = std::max(maxc, std::max(L.n_in, L.n_out));
    if (engine == W2X_ENGINE_FP32) {
        const size_t need = (size_t)maxc * pw * ph * sizeof(float);
        for (int i = 0; i < 2; i++) {
            int rc = ensure(&ctx->buf[i], &ctx->buf_bytes[i], need);
            if (rc) return rc;
        }
        float *cur = static_cast<float *>(ctx->buf[0]), *nxt = static_cast<float *>(ctx->buf[1]);
        CU_CHECK(launch_copy2d(src, src_stride, cur, pw, pw, ph, ctx->stream));   // ROI -> dense plane
        ctx->launches++;
        for (int li = 0; li < n; li++) {
            const Layer &L = m->layers[(size_t)li];
            logf(ctx, "Iteration #%d...", li + 1);                                 // src/convertRoutine.cpp:67
            {
                LayerTimer t(ctx, li);
                CU_CHECK(launch_conv3x3_fp32(cur, nxt, dm->w[(size_t)li], dm->b[(size_t)li], L.n_in, L.n_out, pw, ph,
                                             ctx->stream));
            }
            note_kernel(ctx, li, "fp32_direct");
            ctx->launches++;
            std::swap(cur, nxt);
        }
        CU_CHECK(launch_crop(cur, pw - 2 * n, ph - 2 * n, n, dst, dst_stride, ctx->stream));
        ctx->launches++;
        return W2X_OK;
    }
    // ---- tcgen05 engine ----
    const int f8 = ctx->precision == W2X_PRECISION_F16_F8X2 ? 1 : 0;
    int rc = ensure_tc(ctx);
    if (rc) return rc;
    const size_t need = tc::act_bytes(maxc, pw, ph);
    for (int i = 0; i < 2; i++) {
        rc = ensure(&ctx->buf[i], &ctx->buf_bytes[i], need);
        if (rc) return rc;
    }
    __half *cur = static_cast<__half *>(ctx->buf[0]), *nxt = static_cast<__half *>(ctx->buf[1]);
    {
        const Layer &L = m->layers[0];
        logf(ctx, "Iteration #%d...", 1);
        LayerTimer t(ctx, 0);
        const tc::FirstSource padded{src, src_stride, pw, ph, 0, 0, 0, 0};
        CU_CHECK(tc::launch_first(direct ? *direct : padded, pw, ph, L.w.data(), dm->b_host[0].data(), L.n_out, cur, ctx->stream, f8));
        note_kernel(ctx, 0, "first_1xN");
        ctx->launches++;
    }
    const bool fuse = ctx->fuse_last && n >= 3 && !dm->last_w_t.empty();
    for (int li = 1; li + 1 < n; li++) {
        logf(ctx, "Iteration #%d...", li + 1);
        rc = launch_layer_tc(ctx, m, dm, li, cur, nxt, pw, ph, fuse && li == n - 2, true);
        if (rc) return rc;
        std::swap(cur, nxt);
    }
    {
        const Layer &L = m->layers[(size_t)n - 1];
        logf(ctx, "Iteration #%d...", n);
        LayerTimer t(ctx, n - 1);
        if (fuse) {
            for (int t = 0; t < n_tiles; t++) {
                CU_CHECK(tc::launch_last_gather(reinterpret_cast<const float *>(cur) + (size_t)t * tile_ph * pw * 12, pw, tile_ph, static_cast<float>(L.b[0]), n,
                                                dst + (long)t * (tile_ph - 2 * n) * dst_stride, dst_stride, ctx->stream));
                if (t) ctx->launches++;
            }
            note_kernel(ctx, n - 1, "last_gather");
        } else {
            if (n_tiles != 1) return fail(W2X_ERR_UNSUPPORTED, "batched tiles need the fused last layer");
            CU_CHECK(tc::launch_last(cur, L.n_in, pw, ph, dm->w[(size_t)n - 1], static_cast<float>(L.b[0]), n, dst,
                                     dst_stride, ctx->stream, f8));
            note_kernel(ctx, n - 1, "last_Nx1");
        }
        ctx->launches++;
    }
    return W2X_OK;
}

// Whole plane (or row band) already available as a padded plane: cut it into horizontal bands that
// respect the scratch limit, each band re-reads n rows of context above and below.
// direct_in != nullptr (tcgen05 engine): no padded plane exists; the first layer reads d_in (rows_above / rows_below real rows
// beyond the plane) with the padding folded into its loads.
int run_padded_plane(w2x_ctx *ctx, const w2x_model *m, DevModel *dm, int engine, const float *padp, int w, int h,
                     float *dst, long dst_stride, const float *direct_in = nullptr, long in_stride = 0, int rows_above = 0, int rows_below = 0) {
    const int n = (int)m->layers.size();
    const int pw = w + 2 * n;
    int maxc = 1;
    for (auto &L : m->layers) maxc = std::max(maxc, std::max(L.n_in, L.n_out));
    const size_t per_row = (size_t)maxc * pw * 4;   // both engines: 4 bytes per activation element
    long max_rows = (long)(ctx->scratch_limit / per_row) - 2 * n;
    if (max_rows < 16) max_rows = 16;
    int band = (int)std::min<long>(h, max_rows);
    for (int y0 = 0; y0 < h; y0 += band) {
        const int bh = std::min(band, h - y0);
        int rc;
        if (direct_in) {
            const tc::FirstSource fs{direct_in + (long)y0 * in_stride, in_stride, w, bh, n, n, std::min(n, y0 + rows_above), std::min(n, h - y0 - bh + rows_below)};
            rc = run_basic(ctx, m, dm, engine, nullptr, 0, pw, bh + 2 * n, dst + (long)y0 * dst_stride, dst_stride, 1, &fs);
        } else {
            rc = run_basic(ctx, m, dm, engine, padp + (long)y0 * pw, pw, pw, bh + 2 * n, dst + (long)y0 * dst_stride, dst_stride);
        }
        if (rc) return rc;
    }
    return W2X_OK;
}

int check_ctx(w2x_ctx *ctx) {
    if (!ctx) return fail(W2X_ERR_ARG, "NULL context");
    return W2X_OK;
}

int convert_device(w2x_ctx *ctx, const w2x_model *m, const float *d_in, int w, int h, size_t in_stride_bytes,
                   int rows_above, int rows_below, float *d_out, size_t out_stride_bytes, int block_splitting) {
    if (!m || !d_in || !d_out || w < 1 || h < 1) return fail(W2X_ERR_ARG, "w2x_convert_plane: bad argument");
    if (in_stride_bytes % 4 || out_stride_bytes % 4 || in_stride_bytes < (size_t)w * 4 || out_stride_bytes < (size_t)w * 4)
        return fail(W2X_ERR_ARG, "w2x_convert_plane: row strides must be multiples of 4 bytes and >= width*4");
    if (m->layers.front().n_in != 1 || m->layers.back().n_out != 1)
        return fail(W2X_ERR_ARG, "w2x_convert_plane: model must map 1 plane to 1 plane");
    DeviceGuard g(ctx->device);
    NvtxRange nvtx("w2x convertWithModels");
    const int engine = pick_engine(ctx, m);
    if (engine < 0) return W2X_ERR_UNSUPPORTED;
    DevModel *dm = nullptr;
    int rc = get_dev_model(ctx, m, &dm);
    if (rc) return rc;
    const int n = (int)m->layers.size();
    const int pw = w + 2 * n, ph = h + 2 * n;
    const long ostride = (long)(out_stride_bytes / 4);
    const bool split = block_splitting && w2x_requires_splitting(w, h);
    if (engine == W2X_ENGINE_TC && !(split && ctx->walk == W2X_WALK_BLOCKS)) {
        // cv::copyMakeBorder (src/convertRoutine.cpp:35, :96) is folded into the first layer's loads: no padded copy of the plane
        if (split && !ctx->log_muted) emit_reference_progress(ctx, w, h, n, true);
        LogMute mute(ctx, split);
        return run_padded_plane(ctx, m, dm, engine, nullptr, w, h, d_out, ostride, d_in, (long)(in_stride_bytes / 4), rows_above, rows_below);
    }
    rc = ensure(reinterpret_cast<void **>(&ctx->pad_buf), &ctx->pad_bytes, (size_t)pw * ph * sizeof(float));
    if (rc) return rc;
    // cv::copyMakeBorder(in, temp, n, n, n, n, BORDER_REPLICATE)   (src/convertRoutine.cpp:35, :96)
    CU_CHECK(launch_pad_replicate(d_in, w, h, (long)(in_stride_bytes / 4), n, std::min(rows_above, n),
                                  std::min(rows_below, n), ctx->pad_buf, ctx->stream));
    ctx->launches++;
    if (split && ctx->walk == W2X_WALK_BLOCKS) {
        // the literal block walk of convertWithModelsBlockSplit (src/convertRoutine.cpp:114-165)
        const Config &cfg = config();
        int nb = block_table(w, h, cfg.block_w, cfg.block_h, n, nullptr, 0, nullptr, nullptr);
        if (nb < 0) return fail(W2X_ERR_ARG, "block size too small for a %d-layer model", n);
        std::vector<int> tab((size_t)nb * 8);
        block_table(w, h, cfg.block_w, cfg.block_h, n, tab.data(), nb, nullptr, nullptr);
        for (int i = 0; i < nb; i++) {
            const int *t = &tab[(size_t)i * 8];
            logf(ctx, "start process block (%d,%d) ...", t[1], t[0]);              // :133-134 prints (c,r)
            const int bw_i = t[5] - t[4], bh_i = t[3] - t[2];
            if (t[6] + bh_i - 2 * n > h || t[7] + bw_i - 2 * n > w)
                return fail(W2X_ERR_ARG, "block (%d,%d) does not fit the output plane (non-square block size?)", t[1], t[0]);
            rc = run_basic(ctx, m, dm, engine, ctx->pad_buf + (long)t[2] * pw + t[4], pw, bw_i, bh_i,
                           d_out + (long)t[6] * ostride + t[7], ostride);
            if (rc) return rc;
        }
        return W2X_OK;
    }
    if (split && !ctx->log_muted) emit_reference_progress(ctx, w, h, n, true);     // fused walk: the reference's per-block lines, up front
    LogMute mute(ctx, split);
    return run_padded_plane(ctx, m, dm, engine, ctx->pad_buf, w, h, d_out, ostride);
}

}  // namespace eng
}  // namespace w2x

using namespace w2x::eng;

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int w2x_ctx_create(int device, w2x_ctx **out_ctx) {
    if (!out_ctx) return fail(W2X_ERR_ARG, "w2x_ctx_create: NULL out pointer");
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(W2X_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(W2X_ERR_ARG, "w2x_ctx_create: device %d out of range [0,%d)", device, count);
    cudaDeviceProp prop;
    CU_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(W2X_ERR_NO_DEVICE, "device %d (%s) is sm_%d%d; this build carries sm_100a code only", device,
                    prop.name, prop.major, prop.minor);
    auto ctx = std::make_unique<w2x_ctx>();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    DeviceGuard g(device);
    CU_CHECK(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    if (const char *pe = std::getenv("W2X_PRECISION")) {
        if (!std::strcmp(pe, "f16x3")) ctx->precision = W2X_PRECISION_F16X3;
        else if (!std::strcmp(pe, "f16+f8x2") || !std::strcmp(pe, "f8")) ctx->precision = W2X_PRECISION_F16_F8X2;
    }
    CU_CHECK(cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking));
    CU_CHECK(cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) {
        CU_CHECK(cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming));
        CU_CHECK(cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming));
    }
    *out_ctx = ctx.release();
    return W2X_OK;
}

static void free_dev_model(DevModel &dm) {
    for (auto p : dm.w) cudaFree(p);
    for (auto p : dm.b) cudaFree(p);
    for (auto p : dm.pack) cudaFree(p);
    for (auto p : dm.pack8) cudaFree(p);
    for (auto p : dm.strip) cudaFree(p);
    for (auto p : dm.strip8) cudaFree(p);
}

// Drops the context's device copies of a model (weights, packed operands); call it before w2x_model_free in a long-lived
// context that cycles through many models.  The next conversion with the same model uploads it again.
int w2x_ctx_forget_model(w2x_ctx *ctx, const w2x_model *model) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!model) return fail(W2X_ERR_ARG, "w2x_ctx_forget_model: NULL model");
    auto it = ctx->models.find(model->uid);
    if (it == ctx->models.end()) return W2X_OK;
    DeviceGuard g(ctx->device);
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    free_dev_model(it->second);
    ctx->models.erase(it);
    return W2X_OK;
}

void w2x_ctx_destroy(w2x_ctx *ctx) {
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    release_images(ctx);
    for (auto &kv : ctx->models) free_dev_model(kv.second);
    for (int i = 0; i < 2; i++) {
        cudaFree(ctx->buf[i]);
        cudaFree(ctx->io_buf[i]);
    }
    cudaFree(ctx->pad_buf);
    cudaFree(ctx->prof_buf);
    for (auto &s : ctx->spans) { cudaEventDestroy(s.e0); cudaEventDestroy(s.e1); }
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    for (int i = 0; i < 8; i++) {
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
    }
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int w2x_ctx_set_engine(w2x_ctx *ctx, int engine) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (engine < W2X_ENGINE_AUTO || engine > W2X_ENGINE_TC) return fail(W2X_ERR_ARG, "unknown engine %d", engine);
    ctx->engine = engine;
    return W2X_OK;
}
int w2x_ctx_get_engine(const w2x_ctx *ctx) { return ctx ? ctx->engine : -1; }

int w2x_ctx_set_precision(w2x_ctx *ctx, int precision) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (precision != W2X_PRECISION_F16X3 && precision != W2X_PRECISION_F16_F8X2) return fail(W2X_ERR_ARG, "unknown precision mode %d", precision);
    ctx->precision = precision;
    return W2X_OK;
}
int w2x_ctx_get_precision(const w2x_ctx *ctx) { return ctx ? ctx->precision : -1; }

int w2x_ctx_set_stream(w2x_ctx *ctx, void *cuda_stream) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return W2X_OK;
}

int w2x_ctx_synchronize(w2x_ctx *ctx) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    DeviceGuard g(ctx->device);
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    return W2X_OK;
}

int w2x_ctx_set_log(w2x_ctx *ctx, w2x_log_fn fn, void *user) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->log = fn;
    ctx->log_user = user;
    return W2X_OK;
}

int w2x_ctx_set_block_walk(w2x_ctx *ctx, int mode) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (mode != W2X_WALK_FUSED && mode != W2X_WALK_BLOCKS) return fail(W2X_ERR_ARG, "unknown block walk mode %d", mode);
    ctx->walk = mode;
    return W2X_OK;
}

int w2x_ctx_set_scratch_limit(w2x_ctx *ctx, size_t bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->scratch_limit = bytes ? bytes : (size_t)16 << 30;
    return W2X_OK;
}

// Probe hooks (not part of the stable ABI): per-role wait/work cycle counters of the tcgen05 layer kernels.
W2X_API int w2x_debug_tc_profile_enable(w2x_ctx *ctx, int on) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    DeviceGuard g(ctx->device);
    const size_t bytes = (size_t)16 * tc::PROF_MAX_CTAS * tc::PROF_WORDS * sizeof(unsigned long long);
    if (on) {
        if (!ctx->prof_buf) CU_CHECK(cudaMalloc(&ctx->prof_buf, bytes));
        CU_CHECK(cudaMemsetAsync(ctx->prof_buf, 0, bytes, ctx->stream));
    } else if (ctx->prof_buf) {
        CU_CHECK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->prof_buf);
        ctx->prof_buf = nullptr;
    }
    return W2X_OK;
}
// out[PROF_WORDS]: counters of `layer` summed over CTAs; *n_ctas = CTAs that ran.
W2X_API int w2x_debug_tc_profile_read(w2x_ctx *ctx, int layer, unsigned long long *out, int *n_ctas) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!ctx->prof_buf || layer < 0 || layer >= 16 || !out) return fail(W2X_ERR_ARG, "profile not enabled or bad layer");
    DeviceGuard g(ctx->device);
    std::vector<unsigned long long> h((size_t)tc::PROF_MAX_CTAS * tc::PROF_WORDS);
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    CU_CHECK(cudaMemcpy(h.data(), ctx->prof_buf + (size_t)layer * h.size(), h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    int n = 0;
    for (int w = 0; w < tc::PROF_WORDS; w++) out[w] = 0;
    for (int c = 0; c < tc::PROF_MAX_CTAS; c++) {
        if (h[(size_t)c * tc::PROF_WORDS] == 0) continue;
        n++;
        for (int w = 0; w < tc::PROF_WORDS; w++) out[w] += h[(size_t)c * tc::PROF_WORDS + w];
    }
    if (n_ctas) *n_ctas = n;
    return W2X_OK;
}

// Probe switch (not part of the stable ABI): 1 = CTA-pair (cta_group::2) kernels for the 128-wide layers.
W2X_API int w2x_debug_set_pair(w2x_ctx *ctx, int on) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->pair = on != 0;
    return W2X_OK;
}

// Probe switch (not part of the stable ABI): 1 = row-strip kernel for the narrow layers (default), 0 = the 16x16-tile kernel.
W2X_API int w2x_debug_set_strip(w2x_ctx *ctx, int on) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->strip = on != 0;
    return W2X_OK;
}

// Probe switch (not part of the stable ABI): number of SMs the persistent tcgen05 kernels of this context occupy (0 = all).
W2X_API int w2x_debug_set_num_sms(w2x_ctx *ctx, int n) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    cudaDeviceProp prop;
    CU_CHECK(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->num_sms = n > 0 && n < prop.multiProcessorCount ? n : prop.multiProcessorCount;
    return W2X_OK;
}

// Probe switch (not part of the stable ABI): number of host-copy pipeline bands of w2x_convert_plane (0 auto, 1 off).
W2X_API int w2x_debug_set_host_bands(w2x_ctx *ctx, int bands) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->host_bands = bands < 0 ? 0 : bands;
    return W2X_OK;
}

// Probe switch (not part of the stable ABI): 1 = fold the last layer into the preceding tcgen05 layer (default), 0 = separate kernel.
W2X_API int w2x_debug_set_fuse_last(w2x_ctx *ctx, int on) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->fuse_last = on != 0;
    return W2X_OK;
}

int w2x_convert_plane_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in, int width, int height,
                             size_t in_stride_bytes, float *d_out, size_t out_stride_bytes, int block_splitting) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    return convert_device(ctx, model, d_in, width, height, in_stride_bytes, 0, 0, d_out, out_stride_bytes, block_splitting);
}

int w2x_convert_band_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in, int width, int band_height,
                            int rows_above, int rows_below, size_t in_stride_bytes, float *d_out, size_t out_stride_bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (rows_above < 0 || rows_below < 0) return fail(W2X_ERR_ARG, "w2x_convert_band_device: negative halo");
    if (model && ((rows_above && rows_above < (int)model->layers.size()) || (rows_below && rows_below < (int)model->layers.size())))
        return fail(W2X_ERR_ARG, "w2x_convert_band_device: a halo must be 0 (image border) or >= the layer count (%zu)",
                    model->layers.size());
    if (!d_in) return fail(W2X_ERR_ARG, "w2x_convert_band_device: NULL input");
    const float *band0 = d_in + (size_t)rows_above * (in_stride_bytes / 4);
    return convert_device(ctx, model, band0, width, band_height, in_stride_bytes, rows_above, rows_below, d_out,
                          out_stride_bytes, 0);
}

int w2x_convert_plane(w2x_ctx *ctx, const w2x_model *model, const float *in, int width, int height, size_t in_stride_bytes,
                      float *out, size_t out_stride_bytes, int block_splitting) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!in || !out || width < 1 || height < 1) return fail(W2X_ERR_ARG, "w2x_convert_plane: bad argument");
    if (in_stride_bytes < (size_t)width * 4 || out_stride_bytes < (size_t)width * 4)
        return fail(W2X_ERR_ARG, "w2x_convert_plane: row stride smaller than a row");
    DeviceGuard g(ctx->device);
    const size_t bytes = (size_t)width * height * sizeof(float);
    for (int i = 0; i < 2; i++) {
        int rc = ensure(reinterpret_cast<void **>(&ctx->io_buf[i]), &ctx->io_bytes[i], bytes);
        if (rc) return rc;
    }
    // Large planes are cut into row bands so that the upload of band i+1 and the download of band i-1 overlap the
    // layers of band i (copy engines + compute run concurrently); each band re-reads n real rows of context from its
    // neighbours, which keeps the result bit-identical to the single-pass path.
    const int n_model = model ? (int)model->layers.size() : 0;
    int nb = ctx->host_bands > 0 ? ctx->host_bands : std::min(4, height / 512);
    const bool literal_walk = block_splitting && ctx->walk == W2X_WALK_BLOCKS && w2x_requires_splitting(width, height);
    if (nb > 8) nb = 8;
    if (nb < 2 || literal_walk || !model || height / nb < 2 * n_model) {
        CU_CHECK(cudaMemcpy2DAsync(ctx->io_buf[0], (size_t)width * 4, in, in_stride_bytes, (size_t)width * 4, (size_t)height,
                                   cudaMemcpyHostToDevice, ctx->stream));
        int rc = convert_device(ctx, model, ctx->io_buf[0], width, height, (size_t)width * 4, 0, 0, ctx->io_buf[1],
                                (size_t)width * 4, block_splitting);
        if (rc) return rc;
        CU_CHECK(cudaMemcpy2DAsync(out, out_stride_bytes, ctx->io_buf[1], (size_t)width * 4, (size_t)width * 4, (size_t)height,
                                   cudaMemcpyDeviceToHost, ctx->stream));
        CU_CHECK(cudaStreamSynchronize(ctx->stream));
        return W2X_OK;
    }
    // the copy pipeline cuts the plane its own way: the reference's progress lines for this plane go out first
    emit_reference_progress(ctx, width, height, n_model, block_splitting && w2x_requires_splitting(width, height));
    LogMute mute(ctx, true);
    std::vector<int> r0((size_t)nb + 1);
    for (int i = 0; i <= nb; i++) r0[(size_t)i] = (int)((long)height * i / nb);
    for (int i = 0; i < nb; i++) {
        // upload i carries band i plus the n rows of context band i needs from band i+1, so that band i waits for ITS upload only
        const int y = i == 0 ? 0 : r0[(size_t)i] + n_model, y_end = i + 1 < nb ? r0[(size_t)i + 1] + n_model : height;
        CU_CHECK(cudaMemcpy2DAsync(ctx->io_buf[0] + (size_t)y * width, (size_t)width * 4, reinterpret_cast<const char *>(in) + (size_t)y * in_stride_bytes,
                                   in_stride_bytes, (size_t)width * 4, (size_t)(y_end - y), cudaMemcpyHostToDevice, ctx->copy_in));
        CU_CHECK(cudaEventRecord(ctx->ev_in[i], ctx->copy_in));
    }
    for (int i = 0; i < nb; i++) {
        const int y = r0[(size_t)i], rows = r0[(size_t)i + 1] - y;
        CU_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[i], 0));
        const int above = i > 0 ? n_model : 0, below = i + 1 < nb ? n_model : 0;
        int rc = convert_device(ctx, model, ctx->io_buf[0] + (size_t)y * width, width, rows, (size_t)width * 4, above, below,
                                ctx->io_buf[1] + (size_t)y * width, (size_t)width * 4, 0);
        if (rc) {   // uploads / downloads already queued still touch the caller's buffers and the staging: drain them first
            cudaStreamSynchronize(ctx->copy_in);
            cudaStreamSynchronize(ctx->stream);
            cudaStreamSynchronize(ctx->copy_out);
            return rc;
        }
        CU_CHECK(cudaEventRecord(ctx->ev_done[i], ctx->stream));
        CU_CHECK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[i], 0));
        CU_CHECK(cudaMemcpy2DAsync(reinterpret_cast<char *>(out) + (size_t)y * out_stride_bytes, out_stride_bytes, ctx->io_buf[1] + (size_t)y * width,
                                   (size_t)width * 4, (size_t)width * 4, (size_t)rows, cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    CU_CHECK(cudaStreamSynchronize(ctx->copy_out));
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    return W2X_OK;
}

int w2x_filter_layer_device(w2x_ctx *ctx, const w2x_model *model, int layer, const float *d_in, float *d_out, int width,
                            int height) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!model || layer < 0 || layer >= (int)model->layers.size() || !d_in || !d_out || width < 1 || height < 1)
        return fail(W2X_ERR_ARG, "w2x_filter_layer: bad argument");
    DeviceGuard g(ctx->device);
    DevModel *dm = nullptr;
    int rc = get_dev_model(ctx, model, &dm);
    if (rc) return rc;
    const Layer &L = model->layers[(size_t)layer];
    int engine = ctx->engine == W2X_ENGINE_AUTO ? W2X_ENGINE_FP32 : ctx->engine;
    if (engine == W2X_ENGINE_TC) {
        if (!tc::layer_supported(L.n_in, L.n_out))
            return fail(W2X_ERR_UNSUPPORTED, "tcgen05 engine does not support a %d->%d layer", L.n_in, L.n_out);
        rc = ensure_tc(ctx);
        if (rc) return rc;
        // Model::filter semantics (same size, BORDER_REPLICATE): stage a frame with a replicated ring
        // of one pixel, run the same-size tcgen05 layer on it, return the interior.
        const int pw = width + 2, ph = height + 2;
        rc = ensure(&ctx->buf[0], &ctx->buf_bytes[0], tc::act_bytes(L.n_in, pw, ph));
        if (rc) return rc;
        rc = ensure(&ctx->buf[1], &ctx->buf_bytes[1], tc::act_bytes(L.n_out, pw, ph));
        if (rc) return rc;
        __half *fin = static_cast<__half *>(ctx->buf[0]), *fout = static_cast<__half *>(ctx->buf[1]);
        const int f8 = ctx->precision == W2X_PRECISION_F16_F8X2 ? 1 : 0;
        CU_CHECK(tc::launch_planar_to_nhwc(d_in, L.n_in, width, height, fin, ctx->stream, f8));
        rc = launch_layer_tc(ctx, model, dm, layer, fin, fout, pw, ph, false, false);
        if (rc) return rc;
        CU_CHECK(tc::launch_nhwc_to_planar(fout, L.n_out, width, height, d_out, ctx->stream, f8));
        ctx->launches += 2;
        return W2X_OK;
    }
    {
        LayerTimer t(ctx, layer);
        CU_CHECK(launch_conv3x3_fp32(d_in, d_out, dm->w[(size_t)layer], dm->b[(size_t)layer], L.n_in, L.n_out, width, height,
                                     ctx->stream));
    }
    note_kernel(ctx, layer, "fp32_direct");
    ctx->launches++;
    return W2X_OK;
}

int w2x_filter_layer(w2x_ctx *ctx, const w2x_model *model, int layer, const float *const *in_planes, int n_in_planes,
                     float *const *out_planes, int n_out_planes, int width, int height, size_t in_stride_bytes,
                     size_t out_stride_bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!model || layer < 0 || layer >= (int)model->layers.size() || !in_planes || !out_planes || width < 1 || height < 1)
        return fail(W2X_ERR_ARG, "w2x_filter_layer: bad argument");
    const Layer &L = model->layers[(size_t)layer];
    if (n_in_planes != L.n_in)   // src/modelHandler.cpp:29-35
        return fail(W2X_ERR_ARG, "Error : Model-filter : \nnumber of input planes mismatch.\n%d,%d", n_in_planes, L.n_in);
    if (n_out_planes != L.n_out)
        return fail(W2X_ERR_ARG, "w2x_filter_layer: %d output planes supplied, layer produces %d", n_out_planes, L.n_out);
    if (in_stride_bytes < (size_t)width * 4 || out_stride_bytes < (size_t)width * 4)
        return fail(W2X_ERR_ARG, "w2x_filter_layer: row stride smaller than a row");
    DeviceGuard g(ctx->device);
    const size_t plane = (size_t)width * height * sizeof(float);
    int rc = ensure(reinterpret_cast<void **>(&ctx->io_buf[0]), &ctx->io_bytes[0], plane * (size_t)L.n_in);
    if (rc) return rc;
    rc = ensure(reinterpret_cast<void **>(&ctx->io_buf[1]), &ctx->io_bytes[1], plane * (size_t)L.n_out);
    if (rc) return rc;
    for (int i = 0; i < L.n_in; i++) {
        if (!in_planes[i]) return fail(W2X_ERR_ARG, "w2x_filter_layer: NULL input plane %d", i);
        CU_CHECK(cudaMemcpy2DAsync(reinterpret_cast<char *>(ctx->io_buf[0]) + plane * (size_t)i, (size_t)width * 4, in_planes[i],
                                   in_stride_bytes, (size_t)width * 4, (size_t)height, cudaMemcpyHostToDevice, ctx->stream));
    }
    rc = w2x_filter_layer_device(ctx, model, layer, ctx->io_buf[0], ctx->io_buf[1], width, height);
    if (rc) return rc;
    for (int i = 0; i < L.n_out; i++) {
        if (!out_planes[i]) return fail(W2X_ERR_ARG, "w2x_filter_layer: NULL output plane %d", i);
        CU_CHECK(cudaMemcpy2DAsync(out_planes[i], out_stride_bytes, reinterpret_cast<char *>(ctx->io_buf[1]) + plane * (size_t)i,
                                   (size_t)width * 4, (size_t)width * 4, (size_t)height, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    return W2X_OK;
}

// Page-locked host memory for planes: copies from / to it are truly asynchronous and run at the link rate (the reference's
// cv::Mat data is pageable; host/w2xc.hpp's Plane allocates through this).  Falls back to malloc without a device.
void *w2x_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (bytes == 0) bytes = 1;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) == cudaSuccess) return p;
    cudaGetLastError();
    return nullptr;
}
void w2x_host_free(void *p) {
    if (p && cudaFreeHost(p) != cudaSuccess) cudaGetLastError();
}

int w2x_ctx_launch_count(const w2x_ctx *ctx, uint64_t *n_launches) {
    if (!ctx || !n_launches) return fail(W2X_ERR_ARG, "w2x_ctx_launch_count: NULL argument");
    *n_launches = ctx->launches;
    return W2X_OK;
}

int w2x_ctx_set_timing(w2x_ctx *ctx, int enabled) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    ctx->timing = enabled != 0;
    return W2X_OK;
}

int w2x_ctx_layer_times(w2x_ctx *ctx, int max_layers, float *ms, int *launches, int *n_layers_out, int reset) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (max_layers < 0 || (max_layers > 0 && (!ms || !launches))) return fail(W2X_ERR_ARG, "w2x_ctx_layer_times: bad argument");
    DeviceGuard g(ctx->device);
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < max_layers; i++) { ms[i] = 0.f; launches[i] = 0; }
    int top = 0;
    for (auto &s : ctx->spans) {
        float t = 0.f;
        cudaEventElapsedTime(&t, s.e0, s.e1);
        if (s.layer >= 0 && s.layer < max_layers) { ms[s.layer] += t; launches[s.layer]++; }
        top = std::max(top, s.layer + 1);
    }
    if (n_layers_out) *n_layers_out = top;
    if (reset) {
        for (auto &s : ctx->spans) { ctx->event_pool.push_back(s.e0); ctx->event_pool.push_back(s.e1); }
        ctx->spans.clear();
    }
    return W2X_OK;
}

const char *w2x_ctx_layer_kernel_name(const w2x_ctx *ctx, int layer) {
    if (!ctx || layer < 0 || layer >= (int)ctx->layer_kernel.size()) return "";
    return ctx->layer_kernel[(size_t)layer].c_str();
}

}  // extern "C"

// ---- independent planes of one shape, one pass (the reference's block loop, src/convertRoutine.cpp:114-165) ------------------
namespace {
int convert_tiles_dev(w2x_ctx *ctx, const w2x_model *m, const float *d_in, float *d_out, int n_tiles, int w, int h) {
    if (!m || !d_in || !d_out || n_tiles < 1 || w < 1 || h < 1) return fail(W2X_ERR_ARG, "w2x_convert_tiles: bad argument");
    if (m->layers.front().n_in != 1 || m->layers.back().n_out != 1) return fail(W2X_ERR_ARG, "w2x_convert_tiles: model must map 1 plane to 1 plane");
    DeviceGuard g(ctx->device);
    const int engine = pick_engine(ctx, m);
    if (engine < 0) return W2X_ERR_UNSUPPORTED;
    DevModel *dm = nullptr;
    int rc = get_dev_model(ctx, m, &dm);
    if (rc) return rc;
    const int n = (int)m->layers.size();
    const int pw = w + 2 * n, ph = h + 2 * n;
    int maxc = 1;
    for (auto &L : m->layers) maxc = std::max(maxc, std::max(L.n_in, L.n_out));
    const bool batch = engine == W2X_ENGINE_TC && ctx->fuse_last && n >= 3 && !dm->last_w_t.empty();
    // tiles per pass: what the scratch limit allows (one frame of maxc channels, 4 bytes per element)
    const size_t per_tile = (size_t)maxc * pw * ph * 4;
    int group = batch ? (int)std::max<size_t>(1, std::min<size_t>((size_t)n_tiles, ctx->scratch_limit / per_tile)) : 1;
    rc = ensure(reinterpret_cast<void **>(&ctx->pad_buf), &ctx->pad_bytes, (size_t)group * pw * ph * sizeof(float));
    if (rc) return rc;
    for (int t0 = 0; t0 < n_tiles; t0 += group) {
        const int nt = std::min(group, n_tiles - t0);
        for (int t = 0; t < nt; t++) {   // cv::copyMakeBorder per tile (src/convertRoutine.cpp:35)
            CU_CHECK(launch_pad_replicate(d_in + (size_t)(t0 + t) * w * h, w, h, w, n, 0, 0, ctx->pad_buf + (size_t)t * pw * ph, ctx->stream));
            ctx->launches++;
        }
        rc = run_basic(ctx, m, dm, engine, ctx->pad_buf, pw, pw, ph, d_out + (size_t)t0 * w * h, w, nt);
        if (rc) return rc;
    }
    return W2X_OK;
}
}  // namespace

namespace w2x {
namespace eng {
// phase 1: uploads + the batched pass (results stay in the context's staging buffer); phase 2: downloads.  Split so that a
// multi-GPU driver can queue phase 1 everywhere before a download into pageable memory blocks its thread.
int tiles_enqueue_compute(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles, int n_tiles, int width, int height, size_t in_stride_bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!in_tiles || n_tiles < 1 || width < 1 || height < 1) return fail(W2X_ERR_ARG, "w2x_convert_tiles: bad argument");
    if (in_stride_bytes < (size_t)width * 4) return fail(W2X_ERR_ARG, "w2x_convert_tiles: row stride smaller than a row");
    DeviceGuard g(ctx->device);
    const size_t tile_bytes = (size_t)width * height * sizeof(float);
    for (int i = 0; i < 2; i++) {
        int rc = ensure(reinterpret_cast<void **>(&ctx->io_buf[i]), &ctx->io_bytes[i], tile_bytes * (size_t)n_tiles);
        if (rc) return rc;
    }
    for (int t = 0; t < n_tiles; t++) {
        if (!in_tiles[t]) return fail(W2X_ERR_ARG, "w2x_convert_tiles: NULL tile %d", t);
        CU_CHECK(cudaMemcpy2DAsync(reinterpret_cast<char *>(ctx->io_buf[0]) + tile_bytes * (size_t)t, (size_t)width * 4, in_tiles[t], in_stride_bytes,
                                   (size_t)width * 4, (size_t)height, cudaMemcpyHostToDevice, ctx->stream));
    }
    return convert_tiles_dev(ctx, model, ctx->io_buf[0], ctx->io_buf[1], n_tiles, width, height);
}

int tiles_enqueue_download(w2x_ctx *ctx, float *const *out_tiles, int n_tiles, int width, int height, size_t out_stride_bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (!out_tiles || out_stride_bytes < (size_t)width * 4) return fail(W2X_ERR_ARG, "w2x_convert_tiles: bad output argument");
    DeviceGuard g(ctx->device);
    const size_t tile_bytes = (size_t)width * height * sizeof(float);
    for (int t = 0; t < n_tiles; t++) {
        if (!out_tiles[t]) return fail(W2X_ERR_ARG, "w2x_convert_tiles: NULL tile %d", t);
        CU_CHECK(cudaMemcpy2DAsync(out_tiles[t], out_stride_bytes, reinterpret_cast<char *>(ctx->io_buf[1]) + tile_bytes * (size_t)t, (size_t)width * 4,
                                   (size_t)width * 4, (size_t)height, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return W2X_OK;
}
}  // namespace eng
}  // namespace w2x

extern "C" {

int w2x_convert_tiles_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in, float *d_out, int n_tiles, int width, int height) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    return convert_tiles_dev(ctx, model, d_in, d_out, n_tiles, width, height);
}

int w2x_convert_tiles_async(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles, float *const *out_tiles, int n_tiles,
                            int width, int height, size_t in_stride_bytes, size_t out_stride_bytes) {
    int rc = tiles_enqueue_compute(ctx, model, in_tiles, n_tiles, width, height, in_stride_bytes);
    if (rc) return rc;
    return tiles_enqueue_download(ctx, out_tiles, n_tiles, width, height, out_stride_bytes);
}

int w2x_convert_tiles(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles, float *const *out_tiles, int n_tiles,
                      int width, int height, size_t in_stride_bytes, size_t out_stride_bytes) {
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    // Larger batches run as up to four groups: the uploads of group g+1 and the downloads of group g-1 overlap the layers of
    // group g (copy engines + compute), as the row bands of w2x_convert_plane do.  Tiles are independent, so the grouping
    // does not change a bit of any of them.
    const int groups = n_tiles >= 8 ? std::min(4, n_tiles / 4) : 1;
    if (groups < 2) {
        int rc = w2x_convert_tiles_async(ctx, model, in_tiles, out_tiles, n_tiles, width, height, in_stride_bytes, out_stride_bytes);
        int rc2 = w2x_ctx_synchronize(ctx);
        return rc ? rc : rc2;
    }
    if (!in_tiles || !out_tiles || width < 1 || height < 1) return fail(W2X_ERR_ARG, "w2x_convert_tiles: bad argument");
    if (in_stride_bytes < (size_t)width * 4 || out_stride_bytes < (size_t)width * 4)
        return fail(W2X_ERR_ARG, "w2x_convert_tiles: row stride smaller than a row");
    for (int t = 0; t < n_tiles; t++)
        if (!in_tiles[t] || !out_tiles[t]) return fail(W2X_ERR_ARG, "w2x_convert_tiles: NULL tile %d", t);
    DeviceGuard g(ctx->device);
    const size_t tile_px = (size_t)width * height, tile_bytes = tile_px * sizeof(float);
    for (int i = 0; i < 2; i++) {
        int rc = ensure(reinterpret_cast<void **>(&ctx->io_buf[i]), &ctx->io_bytes[i], tile_bytes * (size_t)n_tiles);
        if (rc) return rc;
    }
    auto first = [&](int gi) { return (int)((long)n_tiles * gi / groups); };
    for (int gi = 0; gi < groups; gi++) {
        for (int t = first(gi); t < first(gi + 1); t++)
            CU_CHECK(cudaMemcpy2DAsync(ctx->io_buf[0] + tile_px * (size_t)t, (size_t)width * 4, in_tiles[t], in_stride_bytes, (size_t)width * 4,
                                       (size_t)height, cudaMemcpyHostToDevice, ctx->copy_in));
        CU_CHECK(cudaEventRecord(ctx->ev_in[gi], ctx->copy_in));
    }
    for (int gi = 0; gi < groups; gi++) {
        const int t0 = first(gi), nt = first(gi + 1) - t0;
        CU_CHECK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[gi], 0));
        int rc = convert_tiles_dev(ctx, model, ctx->io_buf[0] + tile_px * (size_t)t0, ctx->io_buf[1] + tile_px * (size_t)t0, nt, width, height);
        if (rc) {   // copies already queued still touch the caller's buffers and the staging: drain them first
            cudaStreamSynchronize(ctx->copy_in);
            cudaStreamSynchronize(ctx->stream);
            cudaStreamSynchronize(ctx->copy_out);
            return rc;
        }
        CU_CHECK(cudaEventRecord(ctx->ev_done[gi], ctx->stream));
        CU_CHECK(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[gi], 0));
        for (int t = t0; t < t0 + nt; t++)
            CU_CHECK(cudaMemcpy2DAsync(out_tiles[t], out_stride_bytes, ctx->io_buf[1] + tile_px * (size_t)t, (size_t)width * 4, (size_t)width * 4,
                                       (size_t)height, cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    CU_CHECK(cudaStreamSynchronize(ctx->copy_out));
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    return W2X_OK;
}

}  // extern "C"
