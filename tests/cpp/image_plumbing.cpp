// image_plumbing.cpp -- the device image plumbing's arithmetic (csrc/image_math.h, host flavour) against host/imgproc.hpp,
// and the host side of the device image tests (tests/test_image_plumbing.py, tests/test_gpu_image.py).
//   image_plumbing selftest                                  every stage, random images, bitwise; prints ALL OK
//   image_plumbing yuv <in.u8> <w> <h> <out.f32>             from_u8 + rgb2yuv of B,G,R bytes [h][w][3] -> planes [3][h][w]
//   image_plumbing resize <in.f32> <w> <h> <dw> <dh> <nearest|cubic|linear> <out.f32>   planes [3][h][w] -> [3][dh][dw]
//   image_plumbing rgb8 <in.f32> <w> <h> <out.u8>            yuv2rgb + to_u8 of planes [3][h][w] -> B,G,R bytes [h][w][3]
// "Bitwise" means equal bit patterns; two NaNs count as equal whatever their payloads (x86 and the GPU pick different ones).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <limits>
#include <random>
#include <string>
#include <vector>

#include "image_math.h"
#include "imgproc.hpp"

namespace img = w2x::img;
using Planes = std::vector<float>;   // [3][h][w]

static Planes planes_of(const w2ximg::Image3f &im) {
    Planes p((size_t)3 * im.width * im.height);
    for (int c = 0; c < 3; c++) w2ximg::get_channel(im, c, p.data() + (size_t)c * im.width * im.height, (size_t)im.width);
    return p;
}
static w2ximg::Image3f image_of(const Planes &p, int w, int h) {
    w2ximg::Image3f im(w, h);
    for (int c = 0; c < 3; c++) w2ximg::set_channel(im, c, p.data() + (size_t)c * w * h, (size_t)w);
    return im;
}

// ---- the device kernels' loops (image.cu), on the host ----
static Planes dev_yuv(const uint8_t *bgr, int w, int h) {
    Planes p((size_t)3 * w * h);
    const size_t n = (size_t)w * h;
    for (size_t i = 0; i < n; i++) img::bgr8_to_yuv(bgr + i * 3, &p[i], &p[n + i], &p[2 * n + i]);
    return p;
}
static std::vector<uint8_t> dev_rgb8(const Planes &p, int w, int h) {
    const size_t n = (size_t)w * h;
    std::vector<uint8_t> out(n * 3);
    for (size_t i = 0; i < n; i++) img::yuv_to_bgr8(p[i], p[n + i], p[2 * n + i], &out[i * 3]);
    return out;
}
static Planes dev_resize(const Planes &p, int w, int h, int dw, int dh, const std::string &interp) {
    Planes out((size_t)3 * dw * dh);
    const double sx = (double)w / dw, sy = (double)h / dh;
    for (int c = 0; c < 3; c++) {
        const float *src = p.data() + (size_t)c * w * h;
        float *dst = out.data() + (size_t)c * dw * dh;
        for (int y = 0; y < dh; y++)
            for (int x = 0; x < dw; x++) {
                float v;
                int xi[4], yi[4];
                float xw[4], yw[4];
                if (interp == "nearest") {
                    v = src[(size_t)img::nearest_index(y, sy, h) * w + img::nearest_index(x, sx, w)];
                } else if (interp == "cubic") {
                    img::cubic_coeffs(sx, x, w, xi, xw);
                    img::cubic_coeffs(sy, y, h, yi, yw);
                    v = img::sample<4>(src, w, xi, xw, yi, yw);
                } else {
                    img::linear_coeffs(sx, x, w, xi, xw);
                    img::linear_coeffs(sy, y, h, yi, yw);
                    v = img::sample<2>(src, w, xi, xw, yi, yw);
                }
                dst[(size_t)y * dw + x] = v;
            }
    }
    return out;
}

// ---- host/imgproc.hpp, as host/main.cpp calls it ----
static Planes host_yuv(const uint8_t *bgr, int w, int h) {
    w2ximg::Image3f im = w2ximg::from_u8(bgr, w, h);
    w2ximg::rgb2yuv(im);
    return planes_of(im);
}
static std::vector<uint8_t> host_rgb8(const Planes &p, int w, int h) {
    w2ximg::Image3f im = image_of(p, w, h);
    w2ximg::yuv2rgb(im);
    return w2ximg::to_u8(im);
}
static Planes host_resize(const Planes &p, int w, int h, int dw, int dh, const std::string &interp) {
    const w2ximg::Image3f im = image_of(p, w, h);
    if (interp == "nearest") {                                 // resize_nearest_channel, what main.cpp uses for the Y plane
        Planes out((size_t)3 * dw * dh);
        for (int c = 0; c < 3; c++) w2ximg::resize_nearest_channel(im, c, dw, dh, out.data() + (size_t)c * dw * dh, (size_t)dw);
        return out;
    }
    return planes_of(w2ximg::resize(im, dw, dh, interp == "cubic" ? w2ximg::CUBIC : w2ximg::LINEAR));
}

static bool same(float a, float b) {
    uint32_t x, y;
    std::memcpy(&x, &a, 4);
    std::memcpy(&y, &b, 4);
    return x == y || (std::isnan(a) && std::isnan(b));
}
static int failures = 0;
template <typename V>
static void compare(const V &got, const V &ref, const char *stage, int w, int h) {
    size_t bad = 0, first = 0;
    if (got.size() != ref.size()) bad = 1;
    for (size_t i = 0; i < got.size() && i < ref.size(); i++)
        if (!same((float)got[i], (float)ref[i])) {
            if (!bad++) first = i;
        }
    if (bad) {
        failures++;
        std::printf("MISMATCH %s %dx%d: %zu elements differ, first at %zu (%.9g vs %.9g)\n", stage, w, h, bad, first,
                    first < got.size() ? (double)got[first] : 0.0, first < ref.size() ? (double)ref[first] : 0.0);
    }
}

static Planes random_yuv(std::mt19937 &rng, int w, int h) {
    // mostly in range, some out of range, and NaN, +-0, +-inf sprinkled in
    std::uniform_real_distribution<float> u(-0.25f, 1.25f), big(-1e4f, 1e4f);
    std::uniform_int_distribution<int> pick(0, 99);
    Planes p((size_t)3 * w * h);
    for (auto &v : p) {
        const int k = pick(rng);
        v = k < 85 ? u(rng) : k < 90 ? big(rng) : k < 93 ? 0.f : k < 96 ? -0.f : k < 98 ? std::numeric_limits<float>::quiet_NaN()
          : (k == 98 ? 1.f : -1.f) * std::numeric_limits<float>::infinity();
    }
    return p;
}

static int selftest() {
    std::mt19937 rng(12345);
    std::uniform_int_distribution<int> byte(0, 255);
    const int sizes[][2] = {{1, 1}, {2, 3}, {37, 29}, {45, 33}, {640, 400}};
    for (auto &s : sizes) {
        const int w = s[0], h = s[1];
        std::vector<uint8_t> bgr((size_t)w * h * 3);
        for (auto &b : bgr) b = (uint8_t)byte(rng);
        compare(dev_yuv(bgr.data(), w, h), host_yuv(bgr.data(), w, h), "from_u8+rgb2yuv", w, h);
        const Planes yuv = random_yuv(rng, w, h);
        compare(dev_resize(yuv, w, h, 2 * w, 2 * h, "nearest"), host_resize(yuv, w, h, 2 * w, 2 * h, "nearest"), "nearest2x", w, h);
        compare(dev_resize(yuv, w, h, 2 * w, 2 * h, "cubic"), host_resize(yuv, w, h, 2 * w, 2 * h, "cubic"), "bicubic2x", w, h);
        compare(dev_rgb8(yuv, w, h), host_rgb8(yuv, w, h), "yuv2rgb+to_u8", w, h);
        // the shrink of main.cpp (src/main.cpp:104-108, 158-167) for ratios that are not powers of two
        for (double ratio : {3.0, 1.5, 2.5, 0.5}) {
            const int iter = static_cast<int>(std::ceil(std::log2(ratio)));
            double shrink = 0.0;
            if (static_cast<int>(ratio) != std::pow(2, iter)) shrink = ratio / std::pow(2.0, static_cast<double>(iter));
            int cw = w, ch = h;
            for (int i = 0; i < iter; i++) { cw *= 2; ch *= 2; }
            const int lw = static_cast<int>(static_cast<double>(cw * shrink)), lh = static_cast<int>(static_cast<double>(ch * shrink));
            if (shrink == 0.0 || lw < 1 || lh < 1) continue;
            const Planes big = random_yuv(rng, cw, ch);
            char stage[64];
            std::snprintf(stage, sizeof stage, "linear x%g -> %dx%d", ratio, lw, lh);
            compare(dev_resize(big, cw, ch, lw, lh, "linear"), host_resize(big, cw, ch, lw, lh, "linear"), stage, cw, ch);
        }
    }
    if (failures) return 1;
    std::printf("ALL OK\n");
    return 0;
}

template <typename T>
static std::vector<T> load(const char *path, size_t n) {
    std::vector<T> v(n);
    std::ifstream f(path, std::ios::binary);
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize)(n * sizeof(T)));
    if (!f) { std::fprintf(stderr, "short read: %s\n", path); std::exit(1); }
    return v;
}
template <typename V>
static void dump(const char *path, const V &v) {
    std::ofstream f(path, std::ios::binary);
    f.write(reinterpret_cast<const char *>(v.data()), (std::streamsize)(v.size() * sizeof(v[0])));
}

int main(int argc, char **argv) {
    if (argc < 2) return 2;
    const std::string op = argv[1];
    if (op == "selftest" && argc == 2) return selftest();
    if (op == "yuv" && argc == 6) {
        const int w = std::atoi(argv[3]), h = std::atoi(argv[4]);
        dump(argv[5], host_yuv(load<uint8_t>(argv[2], (size_t)w * h * 3).data(), w, h));
        return 0;
    }
    if (op == "resize" && argc == 9) {
        const int w = std::atoi(argv[3]), h = std::atoi(argv[4]);
        dump(argv[8], host_resize(load<float>(argv[2], (size_t)3 * w * h), w, h, std::atoi(argv[5]), std::atoi(argv[6]), argv[7]));
        return 0;
    }
    if (op == "rgb8" && argc == 6) {
        const int w = std::atoi(argv[3]), h = std::atoi(argv[4]);
        dump(argv[5], host_rgb8(load<float>(argv[2], (size_t)3 * w * h), w, h));
        return 0;
    }
    return 2;
}
