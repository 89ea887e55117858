// engine_image.cu -- w2x_image_*: whole images on the device (include/w2x_b200.h).
//
// What the reference's main.cpp does around its two convertWithModels calls (src/main.cpp:74-76, 82-100, 126-167, 171-172):
// the 8-bit image is uploaded once, kept as three dense fp32 planes Y, U, V on the context's device and downloaded once.
// The plumbing kernels live in image.cu; the conv passes are convert_device, exactly as w2x_convert_plane runs them.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>

#include "engine_internal.h"

using namespace w2x;
using namespace w2x::eng;

struct w2x_image {
    w2x_ctx *ctx = nullptr;        // nullptr once the context has been destroyed
    int width = 0, height = 0;
    float *plane[3] = {};          // Y, U, V: dense width x height
    size_t plane_bytes[3] = {};
    float *next[3] = {};           // the planes of the next phase (conv output, resize outputs); swapped with plane[]
    size_t next_bytes[3] = {};
    float *near = nullptr;         // nearest 2x of Y: the conv input of scale2x
    size_t near_bytes = 0;
    uint8_t *bgr = nullptr;        // staging of the host-pointer uploads / downloads
    size_t bgr_bytes = 0;
};

namespace {

void free_buffers(w2x_image *img) {
    for (int c = 0; c < 3; c++) {
        cudaFree(img->plane[c]);
        cudaFree(img->next[c]);
        img->plane[c] = img->next[c] = nullptr;
        img->plane_bytes[c] = img->next_bytes[c] = 0;
    }
    cudaFree(img->near);
    cudaFree(img->bgr);
    img->near = nullptr;
    img->bgr = nullptr;
    img->near_bytes = img->bgr_bytes = 0;
}

int check_image(const w2x_image *img, const char *fn) {
    if (!img) return fail(W2X_ERR_ARG, "%s: NULL image", fn);
    if (!img->ctx) return fail(W2X_ERR_ARG, "%s: the image's context has been destroyed", fn);
    return W2X_OK;
}

int check_pixels(const void *p, int width, int height, size_t stride_bytes, const char *fn) {
    if (!p) return fail(W2X_ERR_ARG, "%s: NULL pixel pointer", fn);
    if (width < 1 || height < 1) return fail(W2X_ERR_ARG, "%s: image size %dx%d, must be at least 1x1", fn, width, height);
    if (stride_bytes < (size_t)width * 3) return fail(W2X_ERR_ARG, "%s: row stride %zu bytes, a row is %zu", fn, stride_bytes, (size_t)width * 3);
    return W2X_OK;
}

int check_model(const w2x_model *m, const char *fn) {
    if (!m) return fail(W2X_ERR_ARG, "%s: NULL model", fn);
    if (m->layers.empty() || m->layers.front().n_in != 1 || m->layers.back().n_out != 1)
        return fail(W2X_ERR_ARG, "%s: model must map 1 plane to 1 plane", fn);
    return W2X_OK;
}

int ensure_next(w2x_image *img, int n_planes, size_t bytes) {
    for (int c = 0; c < n_planes; c++) {
        int rc = ensure(reinterpret_cast<void **>(&img->next[c]), &img->next_bytes[c], bytes);
        if (rc) return rc;
    }
    return W2X_OK;
}

void swap_next(w2x_image *img, int n_planes, int width, int height) {
    for (int c = 0; c < n_planes; c++) {
        std::swap(img->plane[c], img->next[c]);
        std::swap(img->plane_bytes[c], img->next_bytes[c]);
    }
    img->width = width;
    img->height = height;
}

// convertWithModels(src) -> dst on the context's stream, block_splitting = 1 (what the reference's main.cpp passes by
// default).  The reference's progress lines of one call go out first, as w2x_convert_plane emits them.
int convert(w2x_image *img, const w2x_model *m, const float *src, float *dst, int w, int h) {
    w2x_ctx *ctx = img->ctx;
    emit_reference_progress(ctx, w, h, (int)m->layers.size(), w2x_requires_splitting(w, h) != 0);
    LogMute mute(ctx, true);
    return convert_device(ctx, m, src, w, h, (size_t)w * 4, 0, 0, dst, (size_t)w * 4, 1);
}

int create(w2x_ctx *ctx, const uint8_t *bgr, bool host, int width, int height, size_t stride_bytes, w2x_image **out) {
    const char *fn = host ? "w2x_image_create" : "w2x_image_create_device";
    if (!out) return fail(W2X_ERR_ARG, "%s: NULL out pointer", fn);
    *out = nullptr;
    if (check_ctx(ctx)) return W2X_ERR_ARG;
    if (int rc = check_pixels(bgr, width, height, stride_bytes, fn)) return rc;
    DeviceGuard g(ctx->device);
    auto img = new w2x_image();
    img->ctx = ctx;
    ctx->images.push_back(img);
    auto bail = [&](int rc) {
        w2x_image_destroy(img);
        return rc;
    };
    const size_t bytes = (size_t)width * height * sizeof(float);
    for (int c = 0; c < 3; c++)
        if (int rc = ensure(reinterpret_cast<void **>(&img->plane[c]), &img->plane_bytes[c], bytes)) return bail(rc);
    size_t stride = stride_bytes;
    if (host) {
        const size_t row = (size_t)width * 3;
        if (int rc = ensure(reinterpret_cast<void **>(&img->bgr), &img->bgr_bytes, row * height)) return bail(rc);
        cudaError_t e = cudaMemcpy2DAsync(img->bgr, row, bgr, stride_bytes, row, (size_t)height, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) return bail(fail(W2X_ERR_CUDA, "%s: upload failed (%s)", fn, cudaGetErrorString(e)));
        bgr = img->bgr;
        stride = row;
    }
    img->width = width;
    img->height = height;
    cudaError_t e = launch_bgr8_to_yuv(bgr, stride, width, height, img->plane[0], img->plane[1], img->plane[2], ctx->stream);
    ctx->launches++;
    if (e == cudaSuccess && host) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return bail(fail(W2X_ERR_CUDA, "%s: %s", fn, cudaGetErrorString(e)));
    *out = img;
    return W2X_OK;
}

int download(w2x_image *img, uint8_t *bgr, bool host, size_t stride_bytes) {
    const char *fn = host ? "w2x_image_download" : "w2x_image_download_device";
    if (int rc = check_image(img, fn)) return rc;
    if (int rc = check_pixels(bgr, img->width, img->height, stride_bytes, fn)) return rc;
    w2x_ctx *ctx = img->ctx;
    DeviceGuard g(ctx->device);
    const size_t row = (size_t)img->width * 3;
    uint8_t *dst = bgr;
    if (host) {
        if (int rc = ensure(reinterpret_cast<void **>(&img->bgr), &img->bgr_bytes, row * img->height)) return rc;
        dst = img->bgr;
    }
    CU_CHECK(launch_yuv_to_bgr8(img->plane[0], img->plane[1], img->plane[2], img->width, img->height, dst, host ? row : stride_bytes,
                                ctx->stream));
    ctx->launches++;
    if (host) {
        CU_CHECK(cudaMemcpy2DAsync(bgr, stride_bytes, img->bgr, row, row, (size_t)img->height, cudaMemcpyDeviceToHost, ctx->stream));
        CU_CHECK(cudaStreamSynchronize(ctx->stream));
    }
    return W2X_OK;
}

}  // namespace

namespace w2x {
namespace eng {

void release_images(w2x_ctx *ctx) {
    for (w2x_image *img : ctx->images) {
        free_buffers(img);
        img->ctx = nullptr;
    }
    ctx->images.clear();
}

}  // namespace eng
}  // namespace w2x

extern "C" {

int w2x_image_create(w2x_ctx *ctx, const uint8_t *bgr, int width, int height, size_t stride_bytes, w2x_image **out) {
    return create(ctx, bgr, true, width, height, stride_bytes, out);
}

int w2x_image_create_device(w2x_ctx *ctx, const uint8_t *d_bgr, int width, int height, size_t stride_bytes, w2x_image **out) {
    return create(ctx, d_bgr, false, width, height, stride_bytes, out);
}

void w2x_image_destroy(w2x_image *img) {
    if (!img) return;
    if (w2x_ctx *ctx = img->ctx) {
        DeviceGuard g(ctx->device);
        cudaStreamSynchronize(ctx->stream);   // kernels still queued may read or write the buffers
        free_buffers(img);
        ctx->images.erase(std::remove(ctx->images.begin(), ctx->images.end(), img), ctx->images.end());
    }
    delete img;
}

int w2x_image_size(const w2x_image *img, int *width, int *height) {
    if (int rc = check_image(img, "w2x_image_size")) return rc;
    if (width) *width = img->width;
    if (height) *height = img->height;
    return W2X_OK;
}

int w2x_image_denoise(w2x_image *img, const w2x_model *model) {
    if (int rc = check_image(img, "w2x_image_denoise")) return rc;
    if (int rc = check_model(model, "w2x_image_denoise")) return rc;
    DeviceGuard g(img->ctx->device);
    const int w = img->width, h = img->height;
    if (int rc = ensure_next(img, 1, (size_t)w * h * sizeof(float))) return rc;
    if (int rc = convert(img, model, img->plane[0], img->next[0], w, h)) return rc;
    swap_next(img, 1, w, h);
    return W2X_OK;
}

int w2x_image_scale2x(w2x_image *img, const w2x_model *model) {
    if (int rc = check_image(img, "w2x_image_scale2x")) return rc;
    if (int rc = check_model(model, "w2x_image_scale2x")) return rc;
    const int w = img->width, h = img->height;
    if (w > INT_MAX / 2 || h > INT_MAX / 2) return fail(W2X_ERR_ARG, "w2x_image_scale2x: %dx%d image too large to double", w, h);
    w2x_ctx *ctx = img->ctx;
    DeviceGuard g(ctx->device);
    const int w2 = 2 * w, h2 = 2 * h;
    const size_t bytes = (size_t)w2 * h2 * sizeof(float);
    if (int rc = ensure_next(img, 3, bytes)) return rc;
    if (int rc = ensure(reinterpret_cast<void **>(&img->near), &img->near_bytes, bytes)) return rc;
    // resize(INTER_NEAREST) + split, only the Y plane is used (src/main.cpp:135-139)
    CU_CHECK(launch_resize_nearest(img->plane[0], w, h, img->near, w2, h2, ctx->stream));
    ctx->launches++;
    // resize(INTER_CUBIC) (:144); its channel 0 is overwritten by the conv output (:148-154), so only U and V are computed
    const ResizePlanes uv{{img->plane[1], img->plane[2], nullptr}, {img->next[1], img->next[2], nullptr}};
    CU_CHECK(launch_resize(uv, 2, w, h, w2, h2, true, ctx->stream));
    ctx->launches++;
    if (int rc = convert(img, model, img->near, img->next[0], w2, h2)) return rc;
    swap_next(img, 3, w2, h2);
    return W2X_OK;
}

int w2x_image_resize_linear(w2x_image *img, int width, int height) {
    if (int rc = check_image(img, "w2x_image_resize_linear")) return rc;
    if (width < 1 || height < 1) return fail(W2X_ERR_ARG, "w2x_image_resize_linear: target size %dx%d, must be at least 1x1", width, height);
    w2x_ctx *ctx = img->ctx;
    DeviceGuard g(ctx->device);
    if (int rc = ensure_next(img, 3, (size_t)width * height * sizeof(float))) return rc;
    const ResizePlanes yuv{{img->plane[0], img->plane[1], img->plane[2]}, {img->next[0], img->next[1], img->next[2]}};
    CU_CHECK(launch_resize(yuv, 3, img->width, img->height, width, height, false, ctx->stream));
    ctx->launches++;
    swap_next(img, 3, width, height);
    return W2X_OK;
}

int w2x_image_download(w2x_image *img, uint8_t *bgr, size_t stride_bytes) { return download(img, bgr, true, stride_bytes); }

int w2x_image_download_device(w2x_image *img, uint8_t *d_bgr, size_t stride_bytes) { return download(img, d_bgr, false, stride_bytes); }

int w2x_image_planes(w2x_image *img, float *y, float *u, float *v, size_t stride_bytes) {
    if (int rc = check_image(img, "w2x_image_planes")) return rc;
    if (!y || !u || !v) return fail(W2X_ERR_ARG, "w2x_image_planes: NULL plane pointer");
    const size_t row = (size_t)img->width * sizeof(float);
    if (stride_bytes < row) return fail(W2X_ERR_ARG, "w2x_image_planes: row stride %zu bytes, a row is %zu", stride_bytes, row);
    w2x_ctx *ctx = img->ctx;
    DeviceGuard g(ctx->device);
    float *dst[3] = {y, u, v};
    for (int c = 0; c < 3; c++)
        CU_CHECK(cudaMemcpy2DAsync(dst[c], stride_bytes, img->plane[c], row, row, (size_t)img->height, cudaMemcpyDeviceToHost, ctx->stream));
    CU_CHECK(cudaStreamSynchronize(ctx->stream));
    return W2X_OK;
}

}  // extern "C"
