// w2xc.hpp -- the reference's C++ interface for the conv hot path, re-created above the C ABI.
//
// Same namespace, class and function names, argument meaning and error behaviour as the reference
// (WL-Amigo/waifu2x-converter-cpp):
//   w2xc::Model                         src/modelHandler.hpp:24-90
//   w2xc::modelUtility                  src/modelHandler.hpp:92-113
//   w2xc::convertWithModels             src/convertRoutine.hpp:25-28
// so code shaped like the reference's main.cpp compiles against it with `Plane` in place of a
// CV_32FC1 cv::Mat (this image has no OpenCV C++; when it is available define W2X_WITH_OPENCV and
// the cv::Mat overloads at the bottom are enabled).  All arithmetic happens in libw2x_b200.so on
// the GPU; nothing here computes.
#ifndef W2XC_HPP_
#define W2XC_HPP_

#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>
#include <future>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "w2x_b200.h"

#ifdef W2X_WITH_OPENCV
#include <opencv2/core.hpp>
#endif

namespace w2xc {

// A CV_32FC1 matrix stand-in: fp32, row-major, possibly a strided view (like a cv::Mat ROI).  Storage is page-locked
// (w2x_host_alloc) when a device is present, so the host<->device copies inside convertWithModels run at the link rate and
// overlap the layers; plain calloc otherwise.
struct Plane {
    int width = 0, height = 0;
    size_t stride_bytes = 0;
    float *data = nullptr;
    std::shared_ptr<void> owner;   // empty for views

    Plane() {}
    Plane(int w, int h) { create(w, h); }
    void create(int w, int h) {
        const size_t bytes = (size_t)w * h * sizeof(float);
        void *p = bytes >= (size_t)(1 << 20) ? w2x_host_alloc(bytes) : nullptr;   // small planes are not worth a page-locked allocation
        if (p) {
            std::memset(p, 0, bytes);                                         // cv::Mat::zeros
            owner = std::shared_ptr<void>(p, w2x_host_free);
        } else {
            p = std::calloc(bytes ? bytes : 1, 1);
            owner = std::shared_ptr<void>(p, std::free);
        }
        width = w; height = h; stride_bytes = (size_t)w * sizeof(float); data = static_cast<float *>(p);
    }
    bool empty() const { return data == nullptr; }
    float &at(int y, int x) { return *reinterpret_cast<float *>(reinterpret_cast<char *>(data) + (size_t)y * stride_bytes + (size_t)x * 4); }
    const float &at(int y, int x) const { return *reinterpret_cast<const float *>(reinterpret_cast<const char *>(data) + (size_t)y * stride_bytes + (size_t)x * 4); }
    Plane roi(int x0, int y0, int w, int h) const {                          // cv::Mat::operator()(Range, Range)
        Plane p; p.width = w; p.height = h; p.stride_bytes = stride_bytes; p.owner = owner;
        p.data = const_cast<float *>(&at(y0, x0));
        return p;
    }
    Plane clone() const {                                                   // cv::Mat::copyTo / clone
        Plane p(width, height);
        for (int y = 0; y < height; y++) std::memcpy(&p.at(y, 0), &at(y, 0), (size_t)width * sizeof(float));
        return p;
    }
};

// Process-wide GPU runtime shared by Model::filter and convertWithModels (the reference keeps its process-wide state in
// the modelUtility singleton as well).  The number of GPUs is the sibling of the reference's -j (src/main.cpp:58-60):
// gpuRuntime::setNumberOfGpus(n) before the first conversion, or W2X_GPUS=n in the environment; planes are then cut into n
// row bands with a per-layer halo exchange between the GPUs (bit-identical to one GPU).  W2X_DEVICE picks the first device.
class gpuRuntime {
public:
    static bool setNumberOfGpus(int n) {
        if (n < 1 || created()) return false;
        requested() = n;
        return true;
    }
    // nullptr if the runtime could not be created; the reason is printed ONCE, by the first caller that needs the context (not by
    // whichever thread happened to construct the runtime: a front end may create it in the background, see host/main.cpp)
    static w2x_ctx *context() {
        gpuRuntime &rt = instance();
        if (!rt.ctx_ && !rt.error_.empty()) {
            static std::once_flag once;
            std::call_once(once, [&] { std::cerr << ("Error : " + rt.error_ + "\n") << std::flush; });
        }
        return rt.ctx_;
    }
    static void warmup() { (void)instance(); }                // create the runtime (CUDA context) now, silently
    static w2x_multi *multi() { return instance().multi_; }   // nullptr with one GPU
    // the number of GPUs the runtime is (or will be) created with, without creating it
    static int numberOfGpus() {
        const char *ng = std::getenv("W2X_GPUS");
        return requested() > 0 ? requested() : (ng ? std::atoi(ng) : 1);
    }
private:
    static int &requested() { static int n = 0; return n; }
    static bool &created() { static bool c = false; return c; }
    static gpuRuntime &instance() { static gpuRuntime rt; return rt; }
    w2x_ctx *ctx_ = nullptr;
    w2x_multi *multi_ = nullptr;
    std::string error_;
    gpuRuntime() {
        created() = true;
        const char *dev = std::getenv("W2X_DEVICE");
        const int first = dev ? std::atoi(dev) : 0;
        const int n = numberOfGpus();
        if (n > 1) {
            std::vector<int> ids;
            for (int i = 0; i < n; i++) ids.push_back(first + i);
            if (w2x_multi_create(ids.data(), n, &multi_) != W2X_OK) {
                error_ = w2x_last_error();
                multi_ = nullptr;
                return;
            }
            ctx_ = w2x_multi_ctx(multi_, 0);
        } else if (w2x_ctx_create(first, &ctx_) != W2X_OK) {
            error_ = w2x_last_error();
            ctx_ = nullptr;
        }
    }
    ~gpuRuntime() {
        if (multi_) w2x_multi_destroy(multi_);
        else w2x_ctx_destroy(ctx_);
    }
};

class modelUtility;

// One layer of a loaded model file.  The reference constructs a Model per JSON object
// (src/modelHandler.hpp:48-71); here a Model is a (shared model file, layer index) pair.
class Model {
    std::shared_ptr<w2x_model> file_;
    int layer_ = 0;
    friend class modelUtility;
    friend class DeviceImage;
    friend bool convertWithModels(Plane &, Plane &, std::vector<std::unique_ptr<Model>> &, bool);
    Model(std::shared_ptr<w2x_model> f, int layer) : file_(std::move(f)), layer_(layer) {}
    // the model file of `models`, which must be its layers in order (as generateModelFromJSON produces them); nullptr + message if not
    static w2x_model *fileOf(std::vector<std::unique_ptr<Model>> &models) {
        for (size_t i = 0; i < models.size(); i++)
            if (models[i]->file_ != models[0]->file_ || models[i]->layer_ != (int)i ||
                (int)models.size() != w2x_model_layer_count(models[0]->file_.get())) {
                std::cerr << "Error : convertWithModels : models must be the layers of one model file, in order." << std::endl;
                return nullptr;
            }
        return models.empty() ? nullptr : models[0]->file_.get();
    }

public:
    int getNInputPlanes() { int a = 0; w2x_model_layer_dims(file_.get(), layer_, &a, nullptr, nullptr); return a; }
    int getNOutputPlanes() { int b = 0; w2x_model_layer_dims(file_.get(), layer_, nullptr, &b, nullptr); return b; }

    void printWeightMatrix() {
        const float *w; int ni, no, k;
        w2x_model_layer_dims(file_.get(), layer_, &ni, &no, &k);
        w2x_model_layer_params(file_.get(), layer_, &w, nullptr);
        for (int m = 0; m < ni * no; m++) {
            std::cout << "[";
            for (int r = 0; r < k; r++) {
                for (int c = 0; c < k; c++) std::cout << w[(m * k + r) * k + c] << (c + 1 < k ? ", " : "");
                std::cout << (r + 1 < k ? ";\n " : "]");
            }
            std::cout << std::endl;
        }
    }
    void printBiases() {
        const double *b; int no;
        w2x_model_layer_dims(file_.get(), layer_, nullptr, &no, nullptr);
        w2x_model_layer_params(file_.get(), layer_, nullptr, &b);
        for (int i = 0; i < no; i++) std::cout << b[i] << std::endl;
    }

    // bool Model::filter(std::vector<cv::Mat>& inputPlanes, std::vector<cv::Mat>& outputPlanes)
    // (src/modelHandler.cpp:26-72): same-size output planes, BORDER_REPLICATE; a plane-count
    // mismatch prints the reference's message and returns false.
    bool filter(std::vector<Plane> &inputPlanes, std::vector<Plane> &outputPlanes) {
        w2x_ctx *ctx = gpuRuntime::context();
        if (!ctx) return false;
        if ((int)inputPlanes.size() != getNInputPlanes()) {
            std::cerr << "Error : Model-filter : \nnumber of input planes mismatch." << std::endl;
            std::cerr << inputPlanes.size() << "," << getNInputPlanes() << std::endl;
            return false;
        }
        const int w = inputPlanes[0].width, h = inputPlanes[0].height;
        outputPlanes.clear();
        for (int i = 0; i < getNOutputPlanes(); i++) outputPlanes.push_back(Plane(w, h));
        std::vector<const float *> in;
        std::vector<float *> out;
        for (auto &p : inputPlanes) {
            if (p.width != w || p.height != h || p.stride_bytes != inputPlanes[0].stride_bytes) return false;
            in.push_back(p.data);
        }
        for (auto &p : outputPlanes) out.push_back(p.data);
        int rc = w2x_filter_layer(ctx, file_.get(), layer_, in.data(), (int)in.size(), out.data(), (int)out.size(), w, h,
                                  inputPlanes[0].stride_bytes, outputPlanes[0].stride_bytes);
        if (rc != W2X_OK) {
            std::cerr << w2x_last_error() << std::endl;
            return false;
        }
        return true;
    }
#ifdef W2X_WITH_OPENCV
    bool filter(std::vector<cv::Mat> &inputPlanes, std::vector<cv::Mat> &outputPlanes);   // the reference's signature, defined below
#endif
};

class modelUtility {
    modelUtility() {}

public:
    // static bool generateModelFromJSON(const std::string& fileName, std::vector<std::unique_ptr<Model>>& models)
    // (src/modelHandler.cpp:170-197): appends one Model per layer; false + message on failure.
    static bool generateModelFromJSON(const std::string &fileName, std::vector<std::unique_ptr<Model>> &models) {
        w2x_model *m = take_prefetched(fileName);
        if (!m && w2x_model_load_json(fileName.c_str(), &m) != W2X_OK) {
            std::cerr << w2x_last_error() << std::endl;
            return false;
        }
        std::shared_ptr<w2x_model> sp(m, w2x_model_free);
        for (int i = 0; i < w2x_model_layer_count(m); i++) models.push_back(std::unique_ptr<Model>(new Model(sp, i)));
        return true;
    }
    // Not in the reference: start reading + parsing a model file on a background thread (a 5.5 MB JSON file costs ~60 ms); a later
    // generateModelFromJSON(fileName, ...) of the same name takes the result.  Silent: if the background load failed, the
    // foreground call loads again and reports the failure exactly as it always did.
    static void prefetchModelFromJSON(const std::string &fileName) {
        std::lock_guard<std::mutex> lock(prefetch_mutex());
        if (prefetched().count(fileName)) return;
        prefetched()[fileName] = std::async(std::launch::async, [fileName]() -> w2x_model * {
            w2x_model *m = nullptr;
            return w2x_model_load_json(fileName.c_str(), &m) == W2X_OK ? m : nullptr;
        });
    }
    static modelUtility &getInstance() {
        static modelUtility inst;
        return inst;
    }

private:
    static std::mutex &prefetch_mutex() { static std::mutex mu; return mu; }
    static std::map<std::string, std::future<w2x_model *>> &prefetched() {
        struct Holder {
            std::map<std::string, std::future<w2x_model *>> map;
            ~Holder() { for (auto &kv : map) if (kv.second.valid()) if (w2x_model *m = kv.second.get()) w2x_model_free(m); }   // never collected
        };
        static Holder h;
        return h.map;
    }
    static w2x_model *take_prefetched(const std::string &fileName) {
        std::future<w2x_model *> f;
        {
            std::lock_guard<std::mutex> lock(prefetch_mutex());
            auto it = prefetched().find(fileName);
            if (it == prefetched().end()) return nullptr;
            f = std::move(it->second);
            prefetched().erase(it);
        }
        return f.valid() ? f.get() : nullptr;
    }

public:
    bool setNumberOfJobs(int setNJob) { return w2x_set_jobs(setNJob) == W2X_OK; }
    int getNumberOfJobs() { return w2x_get_jobs(); }
    bool setBlockSize(int width, int height) { return w2x_set_block_size(width, height) == W2X_OK; }
    bool setBlockSizeExp2Square(int exp) { return w2x_set_block_size_exp2_square(exp) == W2X_OK; }
    void getBlockSize(int &width, int &height) { w2x_get_block_size(&width, &height); }
};

// bool convertWithModels(cv::Mat& inputPlane, cv::Mat& outputPlane, models, bool blockSplitting = true)
// (src/convertRoutine.cpp:21-51).  `models` must be the layers of ONE model file in order, as
// generateModelFromJSON produces them.  outputPlane is (re)allocated like the reference does.
inline bool convertWithModels(Plane &inputPlane, Plane &outputPlane, std::vector<std::unique_ptr<Model>> &models,
                              bool blockSplitting = true) {
    w2x_ctx *ctx = gpuRuntime::context();
    if (!ctx || models.empty() || inputPlane.empty() || !Model::fileOf(models)) return false;
    if (outputPlane.data == inputPlane.data || outputPlane.width != inputPlane.width || outputPlane.height != inputPlane.height)
        outputPlane.create(inputPlane.width, inputPlane.height);
    static struct Printer {
        static void line(const char *l, void *) { std::cout << l << std::endl; }
    } printer;
    (void)printer;
    w2x_ctx_set_log(ctx, &Printer::line, nullptr);   // "Iteration #k..." / "start process block (c,r) ..."
    int rc;
    if (w2x_multi *mg = gpuRuntime::multi())
        rc = w2x_multi_convert_plane(mg, models[0]->file_.get(), inputPlane.data, inputPlane.width, inputPlane.height, inputPlane.stride_bytes,
                                     outputPlane.data, outputPlane.stride_bytes, blockSplitting ? 1 : 0);
    else
        rc = w2x_convert_plane(ctx, models[0]->file_.get(), inputPlane.data, inputPlane.width, inputPlane.height,
                               inputPlane.stride_bytes, outputPlane.data, outputPlane.stride_bytes, blockSplitting ? 1 : 0);
    if (rc != W2X_OK) {
        std::cerr << w2x_last_error() << std::endl;
        return false;
    }
    return true;
}

// Not in the reference: a whole image on the GPU (w2x_image_*), for the single-GPU runtime.  What the reference's main.cpp
// does with cv::Mat around its convertWithModels calls (src/main.cpp:74-76, 82-100, 126-167, 171-172) happens on the device,
// bit-identical to the host plumbing: upload 8-bit B,G,R once, denoise / scale2x / resizeLinear, download once.  Every
// method returns once the work has finished; on failure it prints w2x_last_error() and returns false.
class DeviceImage {
    w2x_image *img_ = nullptr;
    static bool report() {
        std::cerr << w2x_last_error() << std::endl;
        return false;
    }
    bool finish(int rc) { return rc == W2X_OK && w2x_ctx_synchronize(gpuRuntime::context()) == W2X_OK ? true : report(); }
    bool convert(std::vector<std::unique_ptr<Model>> &models, int (*fn)(w2x_image *, const w2x_model *)) {
        w2x_ctx *ctx = gpuRuntime::context();
        w2x_model *m = Model::fileOf(models);
        if (!ctx || !img_ || !m) return false;
        static struct Printer {
            static void line(const char *l, void *) { std::cout << l << std::endl; }
        } printer;
        (void)printer;
        w2x_ctx_set_log(ctx, &Printer::line, nullptr);   // "Iteration #k..." / "start process block (c,r) ...", as convertWithModels
        return finish(fn(img_, m));
    }

public:
    DeviceImage() {}
    DeviceImage(const DeviceImage &) = delete;
    DeviceImage &operator=(const DeviceImage &) = delete;
    ~DeviceImage() { w2x_image_destroy(img_); }
    // 8-bit B,G,R pixels, rows stride_bytes apart (0 = width * 3), on the runtime's single-GPU context
    bool create(const uint8_t *bgr, int width, int height, size_t stride_bytes = 0) {
        w2x_ctx *ctx = gpuRuntime::context();
        if (!ctx) return false;
        w2x_image_destroy(img_);
        img_ = nullptr;
        return w2x_image_create(ctx, bgr, width, height, stride_bytes ? stride_bytes : (size_t)width * 3, &img_) == W2X_OK ? true : report();
    }
    bool denoise(std::vector<std::unique_ptr<Model>> &models) { return convert(models, w2x_image_denoise); }
    bool scale2x(std::vector<std::unique_ptr<Model>> &models) { return convert(models, w2x_image_scale2x); }
    bool resizeLinear(int width, int height) { return img_ && finish(w2x_image_resize_linear(img_, width, height)); }
    bool download(uint8_t *bgr) { return img_ && (w2x_image_download(img_, bgr, (size_t)width() * 3) == W2X_OK ? true : report()); }
    int width() const { int w = 0; w2x_image_size(img_, &w, nullptr); return w; }
    int height() const { int h = 0; w2x_image_size(img_, nullptr, &h); return h; }
};

#ifdef W2X_WITH_OPENCV
// The reference's own signatures (src/modelHandler.hpp:87-88, src/convertRoutine.hpp:25-28) on cv::Mat: CV_32FC1 planes are
// viewed in place (no copy), outputs are allocated like the reference does (cv::Mat::zeros).
inline Plane viewOf(cv::Mat &m) {
    CV_Assert(m.type() == CV_32FC1);
    Plane p; p.width = m.cols; p.height = m.rows; p.stride_bytes = m.step; p.data = m.ptr<float>();
    return p;
}
inline bool convertWithModels(cv::Mat &inputPlane, cv::Mat &outputPlane, std::vector<std::unique_ptr<Model>> &models,
                              bool blockSplitting = true) {
    cv::Mat out = cv::Mat::zeros(inputPlane.size(), CV_32FC1);
    Plane in = viewOf(inputPlane), o = viewOf(out);
    bool ok = convertWithModels(in, o, models, blockSplitting);
    outputPlane = out;
    return ok;
}
// bool Model::filter(std::vector<cv::Mat>& inputPlanes, std::vector<cv::Mat>& outputPlanes)  (call site: src/test.cpp:76)
inline bool Model::filter(std::vector<cv::Mat> &inputPlanes, std::vector<cv::Mat> &outputPlanes) {
    Model &model = *this;
    std::vector<Plane> in, out;
    for (auto &m : inputPlanes) {
        if (!inputPlanes.empty() && m.step != inputPlanes[0].step) m = m.clone();   // one row stride for all planes (dense after clone)
        in.push_back(viewOf(m));
    }
    if (!model.filter(in, out)) return false;
    outputPlanes.clear();
    for (auto &p : out) {
        cv::Mat m = cv::Mat::zeros(cv::Size(p.width, p.height), CV_32FC1);
        for (int y = 0; y < p.height; y++) std::memcpy(m.ptr<float>(y), &p.at(y, 0), (size_t)p.width * sizeof(float));
        outputPlanes.push_back(m);
    }
    return true;
}
#endif

}  // namespace w2xc
#endif  // W2XC_HPP_
