// main.cpp -- `raytracing_hw5 <scene.txt> <out.ppm>`: the reference's command line
// (src/main.cpp:6-19, run.sh) on top of the C-ABI.  Extra, optional environment knobs:
//   RTC_DEVICE=<n>   CUDA device (default 0)      RTC_SEED=<n>   RNG seed (default 0)
//   RTC_SAMPLES / RTC_WIDTH / RTC_HEIGHT / RTC_RAY_DEPTH   override the scene file
//   RTC_DEVICES=<list>   render on several devices of the machine, e.g. "0,1,2,3" or "0-7" (samples split over them,
//                        summed over NVLink peer access on the first): Scene::Render uses the whole machine too
//   RTC_ADAPTIVE=<tau>   adaptive sampling (rtc_render_adaptive, one device): every 8x8 tile takes samples until its
//                        noise is below tau display units (1/255 = one 8-bit level), at most the scene's SAMPLES (after
//                        RTC_SAMPLES); 0 renders every pixel at SAMPLES.  A value that is not a finite number >= 0 or a
//                        list of several RTC_DEVICES is an error.
//   RTC_DENOISE=<k>      filter the render with non-local means of strength k (rtc_render_denoised, one device; 0.45 is
//                        the recommended strength, 0 leaves the image as rendered): every pixel at SAMPLES, or with
//                        RTC_ADAPTIVE=<tau> adaptive sampling as above.  A value that is not a finite number >= 0 or a list
//                        of several RTC_DEVICES is an error.
//   RTC_TIMING=1     phase times on stderr (with RTC_ADAPTIVE or RTC_DENOISE also the passes and paths rendered)
// The same program serves the four earlier homework snapshots (hwN/run.sh -> build/raytracing_hwN): the dialect
// is the digit in the name it is called by (raytracing_hw1 .. raytracing_hw4 are links to this binary), or
// RTC_DIALECT=<1..5>.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include <string>
#include <vector>

#include "rtc_b200.h"

// "0,2,3" / "0-7" / "0-3,6" -> device indices
static std::vector<int> parse_devices(const char* text) {
    std::vector<int> out;
    const std::string t(text ? text : "");
    size_t i = 0;
    while (i < t.size()) {
        size_t j = t.find(',', i);
        if (j == std::string::npos) j = t.size();
        const std::string item = t.substr(i, j - i);
        const size_t dash = item.find('-');
        if (!item.empty()) {
            if (dash == std::string::npos) out.push_back(std::atoi(item.c_str()));
            else {
                const int a = std::atoi(item.substr(0, dash).c_str()), b = std::atoi(item.substr(dash + 1).c_str());
                for (int d = a; d <= b && (int)out.size() < 64; ++d) out.push_back(d);
            }
        }
        i = j + 1;
    }
    return out;
}

// "P6\nW H\n255\n" + bytes (src/scene.cpp:206-208, 243-251), as rtc_render_ppm writes it
static bool write_ppm(const char* path, uint32_t w, uint32_t h, const std::vector<uint8_t>& img) {
    FILE* f = std::fopen(path, "wb");
    if (!f) return false;
    std::fprintf(f, "P6\n%u %u\n255\n", w, h);
    const bool ok = std::fwrite(img.data(), 1, img.size(), f) == img.size();
    return std::fclose(f) == 0 && ok;
}

static int env_int(const char* name, int dflt) {
    const char* v = std::getenv(name);
    return v && *v ? std::atoi(v) : dflt;
}

int main(int argc, const char* argv[]) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: %s <scene.txt> <out.ppm>\n", argv[0]);
        return 2;
    }
    int dialect = RTC_DIALECT_HW5;
    const char* base = std::strrchr(argv[0], '/');
    base = base ? base + 1 : argv[0];
    if (std::strncmp(base, "raytracing_hw", 13) == 0 && base[13] >= '1' && base[13] <= '5' && base[14] == 0) dialect = base[13] - '0';
    dialect = env_int("RTC_DIALECT", dialect);
    const bool timing = std::getenv("RTC_TIMING") != nullptr;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count();
    };
    const auto t_start = now();
    const std::vector<int> devices = parse_devices(std::getenv("RTC_DEVICES"));
    const int device0 = devices.empty() ? env_int("RTC_DEVICE", 0) : devices[0];
    const char* adaptive = std::getenv("RTC_ADAPTIVE");
    if (adaptive && !*adaptive) adaptive = nullptr;
    float tau = 0.f;
    if (adaptive) {
        char* end = nullptr;
        tau = std::strtof(adaptive, &end);
        if (end == adaptive || *end || !std::isfinite(tau) || tau < 0.f) {
            std::fprintf(stderr, "raytracing_hw5: RTC_ADAPTIVE=%s is not a finite number >= 0\n", adaptive);
            return 1;
        }
        if (devices.size() > 1) {
            std::fprintf(stderr, "raytracing_hw5: RTC_ADAPTIVE renders on one device; RTC_DEVICES lists %zu\n", devices.size());
            return 1;
        }
    }
    const char* denoise = std::getenv("RTC_DENOISE");
    if (denoise && !*denoise) denoise = nullptr;
    float strength = 0.f;
    if (denoise) {
        char* end = nullptr;
        strength = std::strtof(denoise, &end);
        if (end == denoise || *end || !std::isfinite(strength) || strength < 0.f) {
            std::fprintf(stderr, "raytracing_hw5: RTC_DENOISE=%s is not a finite number >= 0\n", denoise);
            return 1;
        }
        if (devices.size() > 1) {
            std::fprintf(stderr, "raytracing_hw5: RTC_DENOISE renders on one device; RTC_DEVICES lists %zu\n", devices.size());
            return 1;
        }
    }
    rtc_scene* scene = rtc_scene_load_dialect(argv[1], device0, dialect);
    if (!scene) {
        std::fprintf(stderr, "raytracing_hw5: %s\n", rtc_last_error());
        return 1;
    }
    const auto t_loaded = now();
    int rc = rtc_scene_override(scene, env_int("RTC_WIDTH", -1), env_int("RTC_HEIGHT", -1), env_int("RTC_SAMPLES", -1),
                                env_int("RTC_RAY_DEPTH", -1));
    if (rc != RTC_OK) {
        std::fprintf(stderr, "raytracing_hw5: %s\n", rtc_last_error());
        rtc_scene_free(scene);
        return 1;
    }
    uint32_t info[8];
    rtc_scene_info(scene, info);
    uint64_t astats[4] = {0, 0, 0, 0};
    bool written_error = false;
    if (adaptive || denoise) {
        std::vector<uint8_t> img(3 * (size_t)info[0] * info[1]);
        const uint32_t seed = (uint32_t)env_int("RTC_SEED", 0);
        // without RTC_ADAPTIVE: min_samples = SAMPLES (at least 2) renders every pixel at SAMPLES
        const uint32_t min_samples = adaptive ? 16u : (info[3] > 2 ? info[3] : 2u);
        if (denoise) rc = rtc_render_denoised(scene, seed, tau, min_samples, 0, strength, img.data(), nullptr, astats);
        else rc = rtc_render_adaptive(scene, seed, tau, min_samples, 0, img.data(), nullptr, nullptr, astats);
        if (rc == RTC_OK && !write_ppm(argv[2], info[0], info[1], img)) {
            std::fprintf(stderr, "raytracing_hw5: cannot write %s\n", argv[2]);
            rc = RTC_ERR_IO;
            written_error = true;
        }
    } else if (devices.size() > 1) rc = rtc_render_ppm_multi(scene, devices.data(), (int)devices.size(), (uint32_t)env_int("RTC_SEED", 0), argv[2]);
    else rc = rtc_render_ppm(scene, (uint32_t)env_int("RTC_SEED", 0), argv[2]);
    if (rc != RTC_OK && !written_error) std::fprintf(stderr, "raytracing_hw5: %s\n", rtc_last_error());
    const auto t_rendered = now();
    if (timing)
        std::fprintf(stderr, "[rtc timing] %-28s %8.1f ms\n[rtc timing] %-28s %8.1f ms\n",
                     "load (file -> HBM, CUDA init)", ms(t_start, t_loaded), "render + PPM", ms(t_loaded, t_rendered));
    if (timing && (adaptive || denoise))
        std::fprintf(stderr, "[rtc timing] adaptive: %llu passes, %llu paths, %llu of %llu tiles stopped below SAMPLES\n",
                     (unsigned long long)astats[0], (unsigned long long)astats[1], (unsigned long long)astats[3],
                     (unsigned long long)astats[2]);
    // The image is on disk: leave without unmapping 2 GB of device memory buffer by buffer (0.15 - 1.1 s measured on the
    // B200 box); the driver reclaims everything when the process ends, as it does for the reference's own heap.
    std::fflush(nullptr);
    std::_Exit(rc == RTC_OK ? 0 : 1);
    return rc == RTC_OK ? 0 : 1;
}
