// main.cpp -- drop-in command line of waifu2x-converter-cpp (reference src/main.cpp) on top of the GPU hot path.
// Same flags, defaults, progress messages, output naming and exit codes; the two convertWithModels calls
// (src/main.cpp:96,148) go to libw2x_b200.so through host/w2xc.hpp, everything around them is restated from
// src/main.cpp line by line with host/imgproc.hpp + host/imageio.hpp standing in for OpenCV.  With one GPU the colour and
// resize steps run on the device instead (w2xc::DeviceImage), bit-identical to imgproc.hpp.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "imageio.hpp"
#include "imgproc.hpp"
#include "w2xc.hpp"

namespace {

// ---- a TCLAP-shaped parser: ValueArg flags only, ' ' delimiter, --help / --version / -- (reference src/main.cpp:26-71) ----
struct Arg {
    std::string flag, name, desc, type;
    bool required;
    std::string def;
    std::vector<std::string> allowed;
    std::string value;
    bool set = false;
    bool hidden = false;   // accepted, but not part of the reference's flag surface: left out of --help and the usage lines
};

struct CmdLine {
    std::string prog, message = "waifu2x reimplementation using OpenCV", version = "1.0.0";
    std::vector<Arg> args;

    Arg &add(const char *flag, const char *name, const char *desc, bool req, const char *def, const char *type,
             std::vector<std::string> allowed = {}) {
        Arg a; a.flag = flag; a.name = name; a.desc = desc; a.required = req; a.def = def; a.type = type; a.allowed = allowed; a.value = def;
        args.push_back(a);
        return args.back();
    }
    std::string id(const Arg &a) const { return (a.flag.empty() ? "" : "-" + a.flag + " ") + "(--" + a.name + ")"; }
    std::string shortid(const Arg &a) const {
        std::string t = a.allowed.empty() ? a.type : "";
        for (size_t i = 0; i < a.allowed.size(); i++) t += (i ? "|" : "") + a.allowed[i];
        std::string s = (a.flag.empty() ? "--" + a.name : "-" + a.flag) + " <" + t + ">";
        return a.required ? s : "[" + s + "]";
    }
    void brief(std::ostream &os) const {
        os << "Brief USAGE: \n   " << prog << " ";
        for (auto it = args.rbegin(); it != args.rend(); ++it)
            if (!it->hidden) os << " " << shortid(*it);
        os << " [--] [--version] [-h]\n\nFor complete USAGE and HELP type: \n   " << prog << " --help\n\n";
    }
    [[noreturn]] void parse_error(const std::string &argid, const std::string &text) const {
        std::cerr << "PARSE ERROR: " << argid << "\n             " << text << "\n\n";
        brief(std::cerr);
        std::exit(1);   // TCLAP StdOutput::failure -> exit(1)
    }
    void usage() const {
        std::cout << "\nUSAGE: \n\n   " << prog << " ";
        for (auto it = args.rbegin(); it != args.rend(); ++it)
            if (!it->hidden) std::cout << " " << shortid(*it);
        std::cout << " [--] [--version] [-h]\n\n\nWhere: \n\n";
        for (auto it = args.rbegin(); it != args.rend(); ++it) {
            if (it->hidden) continue;
            std::string t = it->allowed.empty() ? it->type : "";
            for (size_t i = 0; i < it->allowed.size(); i++) t += (i ? "|" : "") + it->allowed[i];
            std::cout << "   " << (it->flag.empty() ? "" : "-" + it->flag + " <" + t + ">,  ") << "--" << it->name << " <" << t << ">\n     "
                      << (it->required ? "(required)  " : "") << it->desc << "\n\n";
        }
        std::cout << "   --,  --ignore_rest\n     Ignores the rest of the labeled arguments following this flag.\n\n"
                     "   --version\n     Displays version information and exits.\n\n"
                     "   -h,  --help\n     Displays usage information and exits.\n\n\n   " << message << "\n\n";
    }
    void parse(int argc, char **argv) {
        prog = argv[0];
        size_t slash = prog.find_last_of('/');
        if (slash != std::string::npos) prog = prog.substr(slash + 1);
        for (int i = 1; i < argc; i++) {
            std::string tok = argv[i];
            if (tok == "--" || tok == "--ignore_rest") break;
            if (tok == "-h" || tok == "--help") { usage(); std::exit(0); }
            if (tok == "--version") { std::cout << "\n" << prog << "  version: " << version << "\n\n"; std::exit(0); }
            Arg *hit = nullptr;
            for (auto &a : args)
                if ((tok.rfind("--", 0) == 0 && tok.substr(2) == a.name) || (!a.flag.empty() && tok == "-" + a.flag)) hit = &a;
            if (!hit) parse_error("Argument: " + tok, "Couldn't find match for argument");
            if (hit->set) parse_error("Argument: " + id(*hit), "Argument already set!");
            if (i + 1 >= argc) parse_error("Argument: " + id(*hit), "Missing a value for this argument!");
            hit->value = argv[++i];
            hit->set = true;
            if (hit->type == "integer" || hit->type == "double") {
                char *end = nullptr;
                if (hit->type == "integer") std::strtol(hit->value.c_str(), &end, 10); else std::strtod(hit->value.c_str(), &end);
                if (end == hit->value.c_str() || *end) parse_error("Argument: " + id(*hit), "Couldn't read argument value from string '" + hit->value + "'");
            }
            if (!hit->allowed.empty()) {
                bool ok = false;
                for (auto &v : hit->allowed) ok = ok || v == hit->value;
                if (!ok) {
                    std::string c;
                    for (size_t k = 0; k < hit->allowed.size(); k++) c += (k ? "|" : "") + hit->allowed[k];
                    parse_error("Argument: " + id(*hit), "Value '" + hit->value + "' does not meet constraint: " + c);
                }
            }
        }
        for (auto &a : args)
            if (a.required && !a.set) parse_error(" ", "Required argument missing: " + a.name);   // TCLAP: CmdLineParseException with argId " "
    }
    const std::string &get(const char *name) const {
        for (auto &a : args) if (a.name == name) return a.value;
        static std::string empty;
        return empty;
    }
};

w2xc::Plane plane_of(const w2ximg::Image3f &im, int c) {              // cv::split, one channel
    w2xc::Plane p(im.width, im.height);
    w2ximg::get_channel(im, c, p.data, p.stride_bytes / 4);
    return p;
}
// channel c of cv::resize(im, Size(dw, dh), 0, 0, INTER_NEAREST) (src/main.cpp:135-139: resize, then split, then only [0] is used)
w2xc::Plane plane_of_nearest(const w2ximg::Image3f &im, int c, int dw, int dh) {
    w2xc::Plane p(dw, dh);
    w2ximg::resize_nearest_channel(im, c, dw, dh, p.data, p.stride_bytes / 4);
    return p;
}

}  // namespace

int main(int argc, char **argv) {
    CmdLine cmd;
    cmd.add("i", "input_file", "path to input image file (you should input full path)", true, "", "string");
    cmd.add("o", "output_file", "path to output image file (you should input full path)", false, "(auto)", "string");
    cmd.add("m", "mode", "image processing mode", false, "noise_scale", "string", {"noise", "scale", "noise_scale"});
    cmd.add("", "noise_level", "noise reduction level", false, "1", "integer", {"1", "2"});
    cmd.add("", "scale_ratio", "custom scale ratio", false, "2.0", "double");
    cmd.add("", "model_dir", "path to custom model directory (don't append last / )", false, "models", "string");
    cmd.add("j", "jobs", "number of threads launching at the same time", false, "4", "integer");
    // the sibling of -j for this implementation (src/main.cpp:58-60 is where the reference declares -j): planes are cut into
    // this many row bands, one per GPU, halo rows exchanged between the GPUs after every layer; W2X_GPUS does the same
    cmd.add("", "gpus", "number of GPUs the conversion is spread over", false, "1", "integer").hidden = true;
    cmd.parse(argc, argv);
    if (std::atoi(cmd.get("gpus").c_str()) > 1) w2xc::gpuRuntime::setNumberOfGpus(std::atoi(cmd.get("gpus").c_str()));
    // CUDA context creation (~0.2 s) overlaps image decoding, colour conversion and model parsing; joined before the first conversion
    std::thread gpu_warmup([] { w2xc::gpuRuntime::warmup(); });
    // every way out of main below joins it first: std::exit runs the static destructors, and the runtime must not still be under construction
    auto leave = [&](int code) {
        if (gpu_warmup.joinable()) gpu_warmup.join();
        std::exit(code);
    };
    const bool timing = std::getenv("W2X_CLI_TIMING") != nullptr;   // stage times (ms) as one JSON line on stderr
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_start = now();
    double t_conv = 0.0, t_ctx_wait = 0.0;
    auto wait_for_gpu = [&] {                      // the part of the CUDA context creation the host work before it did not hide
        const double t0 = now();
        if (gpu_warmup.joinable()) gpu_warmup.join();
        t_ctx_wait += now() - t0;
    };

    const std::string mode = cmd.get("mode"), inputFile = cmd.get("input_file"), modelDir = cmd.get("model_dir");
    const int nrLevel = std::atoi(cmd.get("noise_level").c_str());
    // the model files this run will ask for are read and parsed in the background while the image is decoded (silently: failures are
    // reported where the reference reports them, by the generateModelFromJSON calls below)
    if (mode == "noise" || mode == "noise_scale") w2xc::modelUtility::prefetchModelFromJSON(modelDir + "/noise" + std::to_string(nrLevel) + "_model.json");
    if (mode == "scale" || mode == "noise_scale") w2xc::modelUtility::prefetchModelFromJSON(modelDir + "/scale2.0x_model.json");
    const double scaleRatio = std::strtod(cmd.get("scale_ratio").c_str(), nullptr);

    // load image file (src/main.cpp:74-76)
    std::string ioerr;
    w2xio::Image8 in8 = w2xio::imread(inputFile, &ioerr);
    if (in8.empty()) {
        std::cerr << "Error : couldn't read image " << inputFile << " (" << ioerr << ")" << std::endl;
        leave(-1);
    }
    const double t_read = now();
    // The image runs on one of two paths, picked at the first convertWithModels call site (after that phase's model file has
    // loaded, so that every message and exit code stays where the reference has it):
    //   device: one GPU -- w2xc::DeviceImage keeps Y, U, V on the GPU from the upload to the download (bit-identical);
    //   host:   --gpus > 1 (w2x_multi_convert_plane takes host planes), no device, or no conversion at all --
    //           host/imgproc.hpp around convertWithModels, as below.
    // W2X_CLI_HOST_PLUMBING=1 forces the host path (A/B measurements, the bit-identity tests).
    w2ximg::Image3f image;
    bool image_ready = false;
    auto host_image = [&]() -> w2ximg::Image3f & {                                        // :75-76, deferred to first use
        if (!image_ready) {
            image = w2ximg::from_u8(in8.bgr.data(), in8.width, in8.height);
            w2ximg::rgb2yuv(image);
            image_ready = true;
        }
        return image;
    };
    w2xc::DeviceImage dev;
    bool on_device = false, path_chosen = false;
    // sets on_device on the first call; *failed = the upload of the device path failed (reported like a failed conversion)
    auto choose_path = [&](bool *failed) {
        *failed = false;
        if (path_chosen) return;
        path_chosen = true;
        if (std::getenv("W2X_CLI_HOST_PLUMBING") || w2xc::gpuRuntime::numberOfGpus() > 1) return;
        wait_for_gpu();
        if (!w2xc::gpuRuntime::context() || w2xc::gpuRuntime::multi()) return;                // no device: the host path fails as today
        on_device = true;
        *failed = !dev.create(in8.bgr.data(), in8.width, in8.height);
    };

    w2xc::modelUtility::getInstance().setNumberOfJobs(std::atoi(cmd.get("jobs").c_str()));   // :79
    // (-j bounds the reference's filter threads; here it bounds the host image plumbing's row workers, the GPU does the filtering)

    // ===== Noise Reduction Phase ===== (:82-100)
    if (mode == "noise" || mode == "noise_scale") {
        std::string modelFileName = modelDir + "/noise" + std::to_string(nrLevel) + "_model.json";
        std::vector<std::unique_ptr<w2xc::Model>> models;
        if (!w2xc::modelUtility::generateModelFromJSON(modelFileName, models)) leave(-1);
        bool failed;
        choose_path(&failed);
        if (failed) leave(-1);
        if (on_device) {
            const double t0 = now();
            if (!dev.denoise(models)) leave(-1);
            t_conv += now() - t0;
        } else {
            w2xc::Plane imageY = plane_of(host_image(), 0), out;
            wait_for_gpu();
            const double t0 = now();
            // The reference ignores the return value here (:96) because a failing layer has already ended the process inside
            // convertWithModelsBasic (src/convertRoutine.cpp:69: std::exit(-1)).  The library never exits, so the same outcome
            // is produced here: no device, out of memory or a CUDA error must not write the un-denoised image with exit code 0.
            if (!w2xc::convertWithModels(imageY, out, models) || out.empty()) leave(-1);
            t_conv += now() - t0;
            w2ximg::set_channel(image, 0, out.data, out.stride_bytes / 4);
        }
    }

    // ===== scaling phase ===== (:104-169)
    if (mode == "scale" || mode == "noise_scale") {
        int iterTimesTwiceScaling = static_cast<int>(std::ceil(std::log2(scaleRatio)));
        double shrinkRatio = 0.0;
        if (static_cast<int>(scaleRatio) != std::pow(2, iterTimesTwiceScaling))
            shrinkRatio = scaleRatio / std::pow(2.0, static_cast<double>(iterTimesTwiceScaling));
        std::string modelFileName = modelDir + "/scale2.0x_model.json";
        std::vector<std::unique_ptr<w2xc::Model>> models;
        if (!w2xc::modelUtility::generateModelFromJSON(modelFileName, models)) leave(-1);
        std::cout << "start scaling" << std::endl;
        for (int nIteration = 0; nIteration < iterTimesTwiceScaling; nIteration++) {
            std::cout << "#" << std::to_string(nIteration + 1) << " 2x scaling..." << std::endl;
            bool failed;
            choose_path(&failed);
            if (on_device) {
                const double t0 = now();
                if (failed || !dev.scale2x(models)) {                                       // nearest + bicubic + conv + merge, :135-155
                    std::cerr << "w2xc::convertWithModels : something error has occured.\nstop." << std::endl;
                    leave(1);
                }
                t_conv += now() - t0;
                continue;
            }
            w2ximg::Image3f &im = host_image();
            const int w2 = im.width * 2, h2 = im.height * 2;
            w2xc::Plane imageY = plane_of_nearest(im, 0, w2, h2), out;                    // :135-139 (only the Y plane of the nearest image is used)
            w2ximg::Image3f bicubic = w2ximg::resize(im, w2, h2, w2ximg::CUBIC);         // :144
            wait_for_gpu();
            const double t0 = now();
            if (!w2xc::convertWithModels(imageY, out, models)) {
                std::cerr << "w2xc::convertWithModels : something error has occured.\nstop." << std::endl;
                leave(1);
            }
            t_conv += now() - t0;
            w2ximg::set_channel(bicubic, 0, out.data, out.stride_bytes / 4);              // merge, :154
            image = std::move(bicubic);
        }
        if (shrinkRatio != 0.0) {                                                           // :158-167
            const int cw = on_device ? dev.width() : host_image().width, ch = on_device ? dev.height() : image.height;
            int lw = static_cast<int>(static_cast<double>(cw * shrinkRatio));
            int lh = static_cast<int>(static_cast<double>(ch * shrinkRatio));
            if (on_device) {
                if (!dev.resizeLinear(lw, lh)) leave(-1);
            } else {
                image = w2ximg::resize(image, lw, lh, w2ximg::LINEAR);
            }
        }
    }

    std::vector<uint8_t> out8;
    int out_w, out_h;
    if (on_device) {                                                                        // :171-172 on the GPU, one download
        out_w = dev.width();
        out_h = dev.height();
        out8.resize((size_t)out_w * out_h * 3);
        if (!dev.download(out8.data())) leave(-1);
    } else {
        w2ximg::yuv2rgb(host_image());                                                      // :171
        out8 = w2ximg::to_u8(image);                                                        // :172
        out_w = image.width;
        out_h = image.height;
    }
    std::string outputFileName = cmd.get("output_file");
    if (outputFileName == "(auto)") {                                                       // :173-189
        outputFileName = inputFile;
        size_t tailDot = outputFileName.find_last_of('.');
        if (tailDot != std::string::npos) outputFileName.erase(tailDot, outputFileName.length());
        outputFileName = outputFileName + "(" + mode + ")";
        if (mode.find("noise") != mode.npos) outputFileName = outputFileName + "(Level" + std::to_string(nrLevel) + ")";
        if (mode.find("scale") != mode.npos) outputFileName = outputFileName + "(x" + std::to_string(scaleRatio) + ")";
        outputFileName += ".png";
    }
    const double t_write0 = now();
    if (!w2xio::imwrite(outputFileName, out8.data(), out_w, out_h)) {
        std::cerr << "Error : couldn't write " << outputFileName << std::endl;
        leave(-1);
    }
    if (timing)
        std::cerr << "{\"w2x_cli_timing_ms\": {\"imread\": " << t_read - t_start << ", \"convertWithModels\": " << t_conv
                  << ", \"cuda_context_wait\": " << t_ctx_wait << ", \"colour_resize_plumbing\": " << (t_write0 - t_read) - t_conv - t_ctx_wait
                  << ", \"imwrite\": " << now() - t_write0
                  << ", \"total\": " << now() - t_start << "}}" << std::endl;
    std::cout << "process successfully done!" << std::endl;
    if (gpu_warmup.joinable()) gpu_warmup.join();
    if (!std::getenv("W2X_CLI_FULL_TEARDOWN")) {   // the file is written and closed: skip the CUDA context / page-locked memory teardown (~0.1 s)
        std::cout.flush();
        std::cerr.flush();
        std::_Exit(0);
    }
    return 0;
}
