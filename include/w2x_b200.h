/*
 * w2x_b200.h -- C ABI of the B200-native convolution hot path of waifu2x-converter-cpp.
 *
 * This is the drop-in boundary.  The reference (WL-Amigo/waifu2x-converter-cpp, C++11) has no
 * plugin/FFI layer; the functions its CLI calls for this path are the ones replaced here.  Every
 * entry point cites the reference interface it stands in for (paths relative to the reference
 * repository root).  Plain C types only: no OpenCV, no torch, no C++ in the signatures.
 *
 * Conventions
 *   - every function that can fail returns an int status (W2X_OK == 0); the reference's `bool`
 *     results and its std::exit(-1) paths (src/modelHandler.hpp:57,69, src/convertRoutine.cpp:69)
 *     both become non-zero statuses -- the library never calls exit();
 *   - w2x_last_error() returns the message the reference would have written to std::cerr
 *     (thread-local, valid until the next failing call on the same thread);
 *   - planes are fp32 (CV_32FC1), row-major, described by (pointer, width, height,
 *     row stride in BYTES) so a strided ROI (src/convertRoutine.cpp:116-131) can be passed as is;
 *   - there is NO CPU fallback: the compute entry points fail with W2X_ERR_NO_DEVICE when no
 *     sm_100 device is present.
 */
#ifndef W2X_B200_H_
#define W2X_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define W2X_API __attribute__((visibility("default")))
#else
#define W2X_API
#endif

/* ---- status codes ------------------------------------------------------------------------- */
#define W2X_OK 0
#define W2X_ERR_ARG 1          /* bad argument (NULL, non-positive size, plane-count mismatch) */
#define W2X_ERR_IO 2           /* "Error : couldn't open <file>"  (src/modelHandler.cpp:176-179) */
#define W2X_ERR_PARSE 3        /* "Error : PicoJSON Error : ..."  (src/modelHandler.cpp:183-187) */
#define W2X_ERR_MODEL 4        /* malformed model: non-square kernel (src/modelHandler.hpp:52-58),
                                  wrong types/shapes, layer chain mismatch, unsupported kernel size */
#define W2X_ERR_CUDA 5         /* a CUDA runtime/driver call failed */
#define W2X_ERR_NO_DEVICE 6    /* no CUDA device / not an sm_100 part: no CPU fallback exists */
#define W2X_ERR_UNSUPPORTED 7  /* layer shape not supported by the requested engine */
#define W2X_ERR_NOMEM 8

typedef struct w2x_model w2x_model; /* a loaded model = std::vector<std::unique_ptr<w2xc::Model>> */
typedef struct w2x_ctx w2x_ctx;     /* one GPU + stream + scratch buffers */

W2X_API const char *w2x_last_error(void);
W2X_API const char *w2x_version(void); /* "1.0.0-b200.<n>" ; the reference CLI is 1.0.0 (src/main.cpp:26) */

/* ---- model container ---------------------------------------------------------------------- */
/* Replaces w2xc::modelUtility::generateModelFromJSON(fileName, models)
 * (src/modelHandler.hpp:104-105, src/modelHandler.cpp:170-197) together with the Model
 * constructor and loadModelFromJSONObject (src/modelHandler.hpp:48-71, src/modelHandler.cpp:74-115):
 * same file format (array of {nInputPlane,nOutputPlane,kW,kH,weight[o][i][ky][kx],bias[o]}),
 * numbers parsed strtod-exactly, weights rounded double->float, biases kept double. */
W2X_API int w2x_model_load_json(const char *path, w2x_model **out_model);
/* Same container built from memory (what a binding that already holds the parsed arrays calls).
 * weights[l] is [n_out][n_in][3][3] fp32, biases[l] is [n_out] fp64. */
W2X_API int w2x_model_create(int n_layers, const int *n_in, const int *n_out,
                             const float *const *weights, const double *const *biases,
                             w2x_model **out_model);
W2X_API void w2x_model_free(w2x_model *model);
/* models.size() as used at src/convertRoutine.cpp:33,93 (nModel = pad width = 7). */
W2X_API int w2x_model_layer_count(const w2x_model *model);
/* Model::getNInputPlanes / getNOutputPlanes (src/modelHandler.hpp:81-82) + kernelSize. */
W2X_API int w2x_model_layer_dims(const w2x_model *model, int layer, int *n_in, int *n_out, int *k);
/* Read-only views of the stored parameters (the reference's printWeightMatrix/printBiases
 * debugging hooks, src/modelHandler.hpp:77-78). */
W2X_API int w2x_model_layer_params(const w2x_model *model, int layer, const float **weights,
                                   const double **biases);

/* ---- process-wide configuration: w2xc::modelUtility (src/modelHandler.hpp:92-113) ----------- */
W2X_API int w2x_set_jobs(int n_job);               /* setNumberOfJobs: <1 -> W2X_ERR_ARG. Parsed and
                                                      stored for drop-in compatibility; the GPU path
                                                      has no use for it. */
W2X_API int w2x_get_jobs(void);                     /* default 4 */
W2X_API int w2x_set_block_size(int width, int height);   /* setBlockSize */
W2X_API int w2x_set_block_size_exp2_square(int exp);     /* setBlockSizeExp2Square */
W2X_API void w2x_get_block_size(int *width, int *height); /* default 512 x 512 */

/* ---- block geometry of convertWithModelsBlockSplit (src/convertRoutine.cpp:84-169) ----------- */
/* The split decision of src/convertRoutine.cpp:25-26 (int arithmetic, current block size). */
W2X_API int w2x_requires_splitting(int width, int height);
/* Fills 8 ints per block in the reference's processing order (r outer, c inner):
 *   { r, c, in_y0, in_y1, in_x0, in_x1, out_y0, out_x0 }
 * in_* index the pad-n_model plane, out_* the output plane.  Returns the number of blocks, or a
 * negative status.  table may be NULL (count only); capacity counts blocks. */
W2X_API int w2x_block_table(int width, int height, int n_model, int *table, int capacity,
                            int *split_cols, int *split_rows);

/* ---- context ------------------------------------------------------------------------------ */
#define W2X_ENGINE_AUTO 0  /* tcgen05 path when the model shape allows, else fp32 */
#define W2X_ENGINE_FP32 1  /* hand-written fp32 CUDA-core direct convolution (reference op order) */
#define W2X_ENGINE_TC 2    /* hand-written tcgen05/TMA implicit-GEMM, 2-term fp16 split, fp32 accum */

W2X_API int w2x_ctx_create(int device, w2x_ctx **out_ctx);
W2X_API void w2x_ctx_destroy(w2x_ctx *ctx);
/* A context caches device copies of every model it has converted with; this drops one model's copies
 * (call before w2x_model_free when a long-lived context cycles through many models). */
W2X_API int w2x_ctx_forget_model(w2x_ctx *ctx, const w2x_model *model);
W2X_API int w2x_ctx_set_engine(w2x_ctx *ctx, int engine);
W2X_API int w2x_ctx_get_engine(const w2x_ctx *ctx);
/* Arithmetic of the tcgen05 engine (both keep fp32 accumulators and meet the 1e-4 gate of BASELINE.json):
 *   W2X_PRECISION_F16X3     x*w = xh*wh + xl*wh + xh*wl, three fp16 tensor-core products
 *                           (measured <= 8e-6 max-abs against the reference CPU path on white noise)
 *   W2X_PRECISION_F16_F8X2  (default) the two correction products run on e4m3 copies of the operands at twice
 *                           the tensor rate: 2.0 instead of 3.0 pass-equivalents; measured <= 2.9e-5 max-abs on
 *                           white noise, <= 7e-6 on a smooth image (profiles/r01_parity_report.txt)
 * The environment variable W2X_PRECISION=f16x3|f8 sets the initial value of new contexts. */
#define W2X_PRECISION_F16X3 0
#define W2X_PRECISION_F16_F8X2 1
W2X_API int w2x_ctx_set_precision(w2x_ctx *ctx, int precision);
W2X_API int w2x_ctx_get_precision(const w2x_ctx *ctx);
/* Run on a caller-owned CUDA stream (cudaStream_t passed as void*); NULL = the ctx's own stream. */
W2X_API int w2x_ctx_set_stream(w2x_ctx *ctx, void *cuda_stream);
/* Block until everything queued by this context has finished. */
W2X_API int w2x_ctx_synchronize(w2x_ctx *ctx);
/* Progress lines exactly as the reference prints them to std::cout
 * ("Iteration #k..." src/convertRoutine.cpp:67, "start process block (c,r) ..." :133-134).
 * NULL disables (default). */
typedef void (*w2x_log_fn)(const char *line, void *user);
W2X_API int w2x_ctx_set_log(w2x_ctx *ctx, w2x_log_fn fn, void *user);
/* W2X_WALK_FUSED (default): a plane that the reference would block-split is processed in one pass
 * of whole-plane kernels (results are bit-identical to the block walk because every output pixel
 * sees the same operands in the same order).  W2X_WALK_BLOCKS: walk the reference's blocks one by
 * one in its order -- kept for fidelity tests and for the per-block progress lines. */
#define W2X_WALK_FUSED 0
#define W2X_WALK_BLOCKS 1
W2X_API int w2x_ctx_set_block_walk(w2x_ctx *ctx, int mode);
/* Upper bound in bytes for ONE activation scratch buffer (two are kept); larger planes are
 * processed in horizontal bands with a 7-row recompute halo.  0 = default (16 GiB). */
W2X_API int w2x_ctx_set_scratch_limit(w2x_ctx *ctx, size_t bytes);

/* Page-locked host memory for planes handed to the host-buffer entry points (optional: any host pointer works, pinned
 * ones make the copies asynchronous and link-rate).  NULL when no device / out of memory: fall back to malloc. */
W2X_API void *w2x_host_alloc(size_t bytes);
W2X_API void w2x_host_free(void *p);

/* ---- the hot path ------------------------------------------------------------------------- */
/* Replaces bool w2xc::convertWithModels(cv::Mat& in, cv::Mat& out, models, bool blockSplitting)
 * (src/convertRoutine.hpp:25-28, src/convertRoutine.cpp:21-51): out = crop_n(L_{n-1}(...L_0(
 * replicate_pad_n(in)))) with every layer = 3x3 correlation + bias + leaky-ReLU(0.1).
 * HOST buffers; host->device and device->host copies happen inside the call; synchronous.
 * in and out must not overlap (the reference's callers deep-copy first, src/main.cpp:94,140). */
W2X_API int w2x_convert_plane(w2x_ctx *ctx, const w2x_model *model, const float *in, int width,
                              int height, size_t in_stride_bytes, float *out,
                              size_t out_stride_bytes, int block_splitting);
/* Same, DEVICE buffers, asynchronous on the context's stream. */
W2X_API int w2x_convert_plane_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in,
                                     int width, int height, size_t in_stride_bytes, float *d_out,
                                     size_t out_stride_bytes, int block_splitting);
/* Replaces bool Model::filter(std::vector<cv::Mat>& in, std::vector<cv::Mat>& out)
 * (src/modelHandler.hpp:87-88, src/modelHandler.cpp:26-72,117-159): one layer, same-size output,
 * BORDER_REPLICATE.  n_in_planes must equal the layer's nInputPlane (mismatch -> W2X_ERR_ARG with
 * the reference's "number of input planes mismatch." message).  HOST plane pointers. */
W2X_API int w2x_filter_layer(w2x_ctx *ctx, const w2x_model *model, int layer,
                             const float *const *in_planes, int n_in_planes,
                             float *const *out_planes, int n_out_planes, int width, int height,
                             size_t in_stride_bytes, size_t out_stride_bytes);
/* Same on dense planar DEVICE tensors: d_in [n_in][h][w], d_out [n_out][h][w]; asynchronous. */
W2X_API int w2x_filter_layer_device(w2x_ctx *ctx, const w2x_model *model, int layer,
                                    const float *d_in, float *d_out, int width, int height);

/* ---- whole images on the device ----------------------------------------------------------- */
/* What the reference's main.cpp does around its two convertWithModels calls with OpenCV, on the GPU: an 8-bit image is
 * uploaded once, kept as three fp32 planes (Y, U, V) through every phase and downloaded once as 8-bit pixels.  Every result
 * is bit-identical to the host plumbing (host/imgproc.hpp): same fp32/fp64 operations in the same order, no contraction.
 * Pixels are interleaved 8-bit B,G,R (as imread loads them; channel 0 is treated as "R" like the reference does), rows
 * `stride_bytes` apart (>= width*3).  An image belongs to one context: every operation queues on the context's stream
 * (w2x_ctx_set_stream included); the calls that take HOST pointers are synchronous, the others are asynchronous.
 * Destroy images before their context; w2x_ctx_destroy releases the device memory of images still alive, after which
 * every call on them fails with W2X_ERR_ARG and w2x_image_destroy only frees the handle.  No CPU fallback: without a
 * context every call fails with W2X_ERR_ARG. */
typedef struct w2x_image w2x_image; /* Y, U, V fp32 planes on the context's device */
/* imread + convertTo(CV_32F, 1/255) + cvtColor(RGB2YUV)   (src/main.cpp:74-76) */
W2X_API int w2x_image_create(w2x_ctx *ctx, const uint8_t *bgr, int width, int height, size_t stride_bytes,
                             w2x_image **out);
/* Same from DEVICE pixels, asynchronous: d_bgr must stay valid until the context's stream has passed this call. */
W2X_API int w2x_image_create_device(w2x_ctx *ctx, const uint8_t *d_bgr, int width, int height, size_t stride_bytes,
                                    w2x_image **out);
W2X_API void w2x_image_destroy(w2x_image *img);
W2X_API int w2x_image_size(const w2x_image *img, int *width, int *height);
/* Noise reduction phase (src/main.cpp:82-100): Y <- convertWithModels(Y), block_splitting = 1 */
W2X_API int w2x_image_denoise(w2x_image *img, const w2x_model *model);
/* One 2x scaling iteration (src/main.cpp:126-156): Y <- convertWithModels(nearest 2x of Y), U, V <- bicubic 2x */
W2X_API int w2x_image_scale2x(w2x_image *img, const w2x_model *model);
/* The shrink of non-power-of-two ratios (src/main.cpp:158-167): bilinear resize of all three planes */
W2X_API int w2x_image_resize_linear(w2x_image *img, int width, int height);
/* cvtColor(YUV2RGB) + convertTo(CV_8U, 255)   (src/main.cpp:171-172), to HOST pixels; synchronous */
W2X_API int w2x_image_download(w2x_image *img, uint8_t *bgr, size_t stride_bytes);
/* Same to DEVICE pixels, asynchronous */
W2X_API int w2x_image_download_device(w2x_image *img, uint8_t *d_bgr, size_t stride_bytes);
/* The fp32 planes to HOST memory (tests, callers that want float output); synchronous */
W2X_API int w2x_image_planes(w2x_image *img, float *y, float *u, float *v, size_t stride_bytes);

/* ---- multi-GPU row-band mode (one process per GPU; the caller moves the halo rows) ----------- */
/* A plane of `height` rows is cut into contiguous bands, one per rank.  Each rank calls
 * w2x_band_begin with ITS band of the input plus up to n_layers rows of real neighbour data
 * above and below (rows_above/rows_below; 0 at the image border, where the library replicates
 * like src/convertRoutine.cpp:35,96).  This is the zero-exchange ("input halo, recompute")
 * variant: one call per rank, no collective on the data path.  d_in points at the first halo row
 * (i.e. band row -rows_above); d_out receives band_height rows. */
W2X_API int w2x_convert_band_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in,
                                    int width, int band_height, int rows_above, int rows_below,
                                    size_t in_stride_bytes, float *d_out, size_t out_stride_bytes);

/* ---- multi-GPU row-band mode with a halo exchange BETWEEN LAYERS ------------------------------ */
/* The variant BASELINE.json's north_star names: each GPU keeps only its own rows (+1 halo row per
 * neighbour side) of every intermediate activation and trades ONE boundary row with each neighbour
 * after every layer.  A session is one GPU's band; all calls are asynchronous on the context's stream.
 *
 * Exchange inside the library (the product path): the neighbours' frames are peer-mapped and
 * w2x_band_exchange stores the boundary rows straight into them over NVLink -- one small kernel per
 * layer (rows, a flag in the receiver's memory, wait for the neighbours' flags); no host round trip.
 *     w2x_band_connect_local(band, up, down)        neighbours in the same process (cudaDeviceEnablePeerAccess), or
 *     w2x_band_export(band, blob) + w2x_band_connect(band, up_blob, down_blob)   between processes (CUDA IPC):
 *                                                   every rank exports, the blobs travel over any host channel
 *     w2x_band_run(band, d_in, stride, d_out, stride)   one pass: own rows in -> own rows out
 *         = w2x_band_load_rows; w2x_band_exchange(-1); { w2x_band_step(k); w2x_band_exchange(k) } k = 0..n-2; w2x_band_finish
 * Every rank of a group must run the same sequence of exchanges (they are numbered).
 *
 * Exchange by the caller (cross-check path; ncclSend/ncclRecv, torch.distributed P2P):
 *     w2x_band_load(band, d_in, stride)            input: band rows + 1 real row per neighbour side
 *     for k in 0 .. n-2:  w2x_band_step(band, k);  w2x_band_halo(band, k, ...) -> move the segments
 *     w2x_band_finish(band, d_out, stride)
 * Step n-2 is the tcgen05 layer with the last layer folded into its epilogue; its rows are per-pixel tap
 * partials instead of activations.  Requires the tcgen05 engine.  The layer kernels never store a band's
 * halo rows, so a neighbour's row may arrive at any time after the previous exchange. */
typedef struct w2x_band w2x_band;
/* What lies beyond a band's first / last row: */
#define W2X_EDGE_BORDER 0      /* the image border: replicate (src/convertRoutine.cpp:35,96) */
#define W2X_EDGE_NEIGHBOUR 1   /* another GPU's band: one halo row, exchanged after every layer */
#define W2X_EDGE_OVERLAP 2     /* n_layers real input rows supplied with the band and recomputed (no exchange): the seam
                                  between two sub-bands of ONE GPU (w2x_slab_*), input read through w2x_band_load_rows */
W2X_API int w2x_band_create(w2x_ctx *ctx, const w2x_model *model, int width, int band_rows,
                            int up_edge, int down_edge, w2x_band **out_band);
W2X_API void w2x_band_destroy(w2x_band *band);
W2X_API int w2x_band_load(w2x_band *band, const float *d_in, size_t in_stride_bytes);
W2X_API int w2x_band_load_rows(w2x_band *band, const float *d_in_own_rows, size_t in_stride_bytes);
W2X_API int w2x_band_step(w2x_band *band, int step);
/* Segments to move after `step` was queued: n_segments (<= 4) contiguous device ranges of
 * seg_bytes each per direction; send_* hold this rank's boundary row, recv_* its halo row.
 * Pointers for a missing neighbour are NULL.  Arrays must have room for 4 entries. */
W2X_API int w2x_band_halo(w2x_band *band, int step, int *n_segments, void **send_up, void **recv_up,
                          void **send_down, void **recv_down, size_t *seg_bytes);
W2X_API int w2x_band_finish(w2x_band *band, float *d_out, size_t out_stride_bytes);
#define W2X_BAND_BLOB_BYTES 320
W2X_API int w2x_band_export(w2x_band *band, void *blob /* W2X_BAND_BLOB_BYTES */);
W2X_API int w2x_band_connect(w2x_band *band, const void *up_blob, const void *down_blob);
W2X_API int w2x_band_connect_local(w2x_band *band, w2x_band *up, w2x_band *down);
W2X_API int w2x_band_exchange(w2x_band *band, int step /* -1 after w2x_band_load_rows */);
W2X_API int w2x_band_run(w2x_band *band, const float *d_in_own_rows, size_t in_stride_bytes, float *d_out,
                         size_t out_stride_bytes);

/* ---- one GPU's slab of a multi-GPU plane, HOST buffers ------------------------------------------------ */
/* What a rank of a multi-process job (or one GPU of w2x_multi_*) owns of the plane: rows in pinned host memory go in,
 * rows come out.  The slab is cut into sub-bands so that uploads, layers and downloads overlap; seams inside the slab are
 * W2X_EDGE_OVERLAP (recomputed, local data), its outer edges exchange a halo row per layer with the neighbour slab.
 * order: 0 = walk the sub-bands top -> bottom, 1 = bottom -> top; neighbouring slabs must alternate (rank parity) so that
 * both sides of a boundary are in flight at the same time.  n_sub = 0: automatic.  Blobs are 2 * W2X_BAND_BLOB_BYTES. */
typedef struct w2x_slab w2x_slab;
W2X_API int w2x_slab_create(w2x_ctx *ctx, const w2x_model *model, int width, int rows, int has_up_neighbour,
                            int has_down_neighbour, int order, int n_sub, w2x_slab **out_slab);
W2X_API void w2x_slab_destroy(w2x_slab *slab);
W2X_API int w2x_slab_export(w2x_slab *slab, void *blob /* 2 * W2X_BAND_BLOB_BYTES */);
W2X_API int w2x_slab_connect(w2x_slab *slab, const void *up_blob, const void *down_blob);
W2X_API int w2x_slab_connect_local(w2x_slab *slab, w2x_slab *up, w2x_slab *down);
W2X_API int w2x_slab_convert(w2x_slab *slab, const float *in_rows, size_t in_stride_bytes, float *out_rows,
                             size_t out_stride_bytes);
W2X_API int w2x_slab_convert_async(w2x_slab *slab, const float *in_rows, size_t in_stride_bytes, float *out_rows,
                                   size_t out_stride_bytes);
W2X_API int w2x_slab_synchronize(w2x_slab *slab);

/* ---- independent planes of one shape in one pass ---------------------------------------------- */
/* The reference's block loop (src/convertRoutine.cpp:114-165) and BASELINE config 5 (64 x 512x512 tiles):
 * n_tiles planes, each converted exactly like w2x_convert_plane(block_splitting = 0) would -- bit-identical --
 * but stacked into ONE frame so that every layer is one launch for the whole batch.  HOST pointers; batches of
 * eight tiles and more are cut into up to four such frames so that uploads, layers and downloads overlap. */
W2X_API int w2x_convert_tiles(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles,
                              float *const *out_tiles, int n_tiles, int width, int height,
                              size_t in_stride_bytes, size_t out_stride_bytes);
/* Same, returns once everything is queued (pinned host memory makes it truly asynchronous);
 * w2x_ctx_synchronize completes it. */
W2X_API int w2x_convert_tiles_async(w2x_ctx *ctx, const w2x_model *model, const float *const *in_tiles,
                                    float *const *out_tiles, int n_tiles, int width, int height,
                                    size_t in_stride_bytes, size_t out_stride_bytes);
/* Same on dense DEVICE batches d_in [n_tiles][height][width] -> d_out; asynchronous. */
W2X_API int w2x_convert_tiles_device(w2x_ctx *ctx, const w2x_model *model, const float *d_in, float *d_out,
                                     int n_tiles, int width, int height);

/* ---- one process, N GPUs ---------------------------------------------------------------------- */
/* The sibling of the reference's -j (src/main.cpp:58-60, modelUtility::setNumberOfJobs): N contexts driven by
 * one host thread.  w2x_multi_convert_plane = w2x_convert_plane with the plane cut into N row bands and the
 * per-layer halo exchange above between them (bit-identical to one GPU); planes too small to cut run on the
 * first GPU.  w2x_multi_convert_tiles = w2x_convert_tiles with tile t on GPU t mod N (no exchange).
 * devices == NULL means 0 .. n_devices-1. */
typedef struct w2x_multi w2x_multi;
W2X_API int w2x_multi_create(const int *devices, int n_devices, w2x_multi **out);
W2X_API void w2x_multi_destroy(w2x_multi *multi);
W2X_API int w2x_multi_device_count(const w2x_multi *multi);
W2X_API w2x_ctx *w2x_multi_ctx(w2x_multi *multi, int index);   /* the i-th GPU's context (settings, timing) */
W2X_API int w2x_multi_set_precision(w2x_multi *multi, int precision);
W2X_API int w2x_multi_set_log(w2x_multi *multi, w2x_log_fn fn, void *user);
W2X_API int w2x_multi_convert_plane(w2x_multi *multi, const w2x_model *model, const float *in, int width,
                                    int height, size_t in_stride_bytes, float *out, size_t out_stride_bytes,
                                    int block_splitting);
W2X_API int w2x_multi_convert_tiles(w2x_multi *multi, const w2x_model *model, const float *const *in_tiles,
                                    float *const *out_tiles, int n_tiles, int width, int height,
                                    size_t in_stride_bytes, size_t out_stride_bytes);

/* ---- instrumentation ---------------------------------------------------------------------- */
/* Number of kernels of THIS library launched by the context so far. */
W2X_API int w2x_ctx_launch_count(const w2x_ctx *ctx, uint64_t *n_launches);
/* When enabled, every layer kernel launched by convert_* is bracketed by CUDA events on the
 * launching stream; w2x_ctx_layer_times returns, per layer, the summed milliseconds and launch
 * count since the last reset (synchronises the stream). */
W2X_API int w2x_ctx_set_timing(w2x_ctx *ctx, int enabled);
W2X_API int w2x_ctx_layer_times(w2x_ctx *ctx, int max_layers, float *ms, int *launches,
                                int *n_layers_out, int reset);
/* Name of the kernel family the last convert call used for `layer` ("fp32_direct",
 * "tcgen05_f16x3", "first_1xN", "last_Nx1"). */
W2X_API const char *w2x_ctx_layer_kernel_name(const w2x_ctx *ctx, int layer);

#ifdef __cplusplus
}
#endif
#endif /* W2X_B200_H_ */
