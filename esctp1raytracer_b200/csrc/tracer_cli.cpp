// tracer_cli.cpp — the reference's host flow (src/main.cpp:417-695) with the GPU renderer in the
// place of its accelerator call:  arg parse -> model::loadobj -> camera -> render -> PPM.
// Same flags as the reference where they exist (-m -o -v -l, main.cpp:467-529); `-w W,H` really sets
// the window here (in the reference it overwrites `look`, main.cpp:515-529); `--cuda` is accepted
// for symmetry with `--ispc`.  The CPU/ISPC modes (--thread, --ispc) do not exist in this build.  `--bvh` does what the
// reference's --bvh intends (main.cpp:566-567 flatten + sort, then a BVH render): the flatten+sort pass of --sorted, then
// the optional BVH mode (opts.accel = 1), so its output is the bytes of --sorted.
// `--gpus N` renders the frame on N GPUs of the box (interleaved 8-row bands, NCCL gather: tracer_cuda_init_multi), with the
// same generator and, for a given --seed, the same bytes as one GPU;
// `--spp S` = S stratified jittered samples per pixel (extension); `--sorted` runs the reference's optional
// flatten+sort pass (src/simplify/flatten.cpp:50-82) before rendering.
// `--eye x,y,z` (repeatable) renders one view per eye, all looking at -l, in one tracer_cuda_render_views call on a resident
// scene; with -o out.ppm they are written to out_0.ppm, out_1.ppm, ...  Each is the frame `-v x,y,z` gives with the same
// --seed.  Not with -v, --gpus > 1 or --cull.
// `--crop x,y,w,h` renders only that window of the -w frame (columns x .. x+w-1 of PPM rows y .. y+h-1, row 0 at the top) and
// writes a w x h PPM: the same pixels as the whole frame's, in every --rng mode, with --cull and --bvh.  Not with --eye or
// --gpus > 1.
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/tracer_host.h"

static void parse_triple(const char *s, float out[3]) {
    if (std::sscanf(s, "%f,%f,%f", &out[0], &out[1], &out[2]) != 3) throw std::runtime_error(std::string("expected x,y,z: ") + s);
}

int main(int argc, char *argv[]) {
    try {
        std::string model, output;
        float eye[3] = {0, 1, 3}, look[3] = {0, 1, 0}; // main.cpp:426
        int W = 1024, H = 768;                          // main.cpp:427
        int device = 0, p6 = 0, bundle_cull = 0, gpus = 1, spp = 0;
        bool sorted = false;
        int accel = 0;
        int crop[4] = {0, 0, 0, 0}; // x, y, w, h; all 0 = the whole frame
        bool have_seed = false, have_v = false, have_crop = false;
        std::vector<std::array<float, 3>> eyes;
        unsigned seed = 0;
        int rng = TRACER_RNG_MT19937; // the serial path's generator
        for (int a = 1; a < argc; ++a) {
            const std::string f = argv[a];
            auto need = [&](const char *what) -> const char * {
                if (a + 1 >= argc) throw std::runtime_error(std::string("missing value for ") + what);
                return argv[++a];
            };
            if (f == "--cuda" || f == "--debug" || f == "--trace" || f == "--test") continue;
            if (f == "--thread" || f == "--ispc")
                throw std::runtime_error(f + ": CPU/ISPC modes are not part of this build (GPU renderer only)");
            if (f == "-m") model = need("-m");
            else if (f == "-o") output = need("-o");
            else if (f == "-v") parse_triple(need("-v"), eye), have_v = true;
            else if (f == "--eye") {
                eyes.emplace_back();
                parse_triple(need("--eye"), eyes.back().data());
            }
            else if (f == "-l") parse_triple(need("-l"), look);
            else if (f == "-w") {
                if (std::sscanf(need("-w"), "%d,%d", &W, &H) != 2) throw std::runtime_error("expected -w W,H");
            } else if (f == "--seed") seed = (unsigned)std::strtoul(need("--seed"), nullptr, 10), have_seed = true;
            else if (f == "--rng") {
                const std::string r = need("--rng");
                rng = r == "hash" ? TRACER_RNG_HASH : TRACER_RNG_MT19937;
            } else if (f == "--device") device = std::atoi(need("--device"));
            else if (f == "--p6") p6 = 1;
            else if (f == "--cull") bundle_cull = 3; // optional bundle-cull mode: same bytes out, much faster on big scenes
            else if (f == "--gpus") gpus = std::atoi(need("--gpus"));
            else if (f == "--spp") spp = std::atoi(need("--spp"));
            else if (f == "--sorted") sorted = true;
            else if (f == "--bvh") sorted = true, accel = 1;
            else if (f == "--crop") {
                if (std::sscanf(need("--crop"), "%d,%d,%d,%d", &crop[0], &crop[1], &crop[2], &crop[3]) != 4)
                    throw std::runtime_error("expected --crop x,y,w,h");
                if (crop[2] < 1 || crop[3] < 1) throw std::runtime_error("--crop needs a width and height >= 1");
                have_crop = true;
            } else throw std::runtime_error("Unknown argument: " + f); // main.cpp:531-534
        }
        if (!eyes.empty() && have_v) throw std::runtime_error("--eye and -v do not combine: give every view as --eye");
        if (!eyes.empty() && gpus > 1) throw std::runtime_error("--eye renders on one GPU: --gpus must be 1");
        if (!eyes.empty() && bundle_cull) throw std::runtime_error("--eye does not combine with --cull");
        if (have_crop && !eyes.empty()) throw std::runtime_error("--crop does not combine with --eye");
        if (have_crop && gpus > 1) throw std::runtime_error("--crop renders on one GPU: --gpus must be 1");
        tracer_scene_host *scene = nullptr;
        tracer_scene_flat empty{};
        const int32_t zero_off[1] = {0};
        empty.geom_tri_offset = zero_off;
        const tracer_scene_flat *flat = &empty; // no -m: empty scene, black image (main.cpp:537-543)
        if (!model.empty()) {
            if (tracer_scene_load_obj(model.c_str(), &scene)) throw std::runtime_error(tracer_host_last_error());
            flat = tracer_scene_host_flat(scene);
        }
        tracer_scene_host *sorted_scene = nullptr;
        if (sorted && scene) { // main.cpp:566-567 runs flatten_scene before rendering
            if (tracer_scene_flatten_sorted(flat, &sorted_scene)) throw std::runtime_error(tracer_host_last_error());
            flat = tracer_scene_host_flat(sorted_scene);
        }
        tracer_camera cam;
        const float vup[3] = {0, 1, 0};
        tracer_camera_lookat(eye, look, vup, 60.f, float(W) / H, &cam); // main.cpp:548-551
        if (gpus > 1) {
            if (tracer_cuda_init_multi(gpus)) throw std::runtime_error(tracer_cuda_last_error());
        } else if (tracer_cuda_init(device)) throw std::runtime_error(tracer_cuda_last_error());
        tracer_render_opts o{};
        o.struct_size = sizeof o;
        o.rng_mode = rng;
        o.bundle_cull = bundle_cull;
        o.accel = accel;
        o.samples_per_pixel = spp;
        if (spp > 1 && rng == TRACER_RNG_MT19937) o.rng_mode = rng = TRACER_RNG_HASH; // the serial replay is 1 spp only
        o.seed = have_seed ? seed : std::random_device{}(); // main.cpp:587-588
        if (!eyes.empty()) { // one resident scene, one call for every view
            std::vector<tracer_camera> cams(eyes.size());
            for (size_t v = 0; v < eyes.size(); ++v) tracer_camera_lookat(eyes[v].data(), look, vup, 60.f, float(W) / H, &cams[v]);
            tracer_scene_dev *dev = nullptr;
            if (tracer_cuda_scene_create(flat, &dev)) throw std::runtime_error(tracer_cuda_last_error());
            std::vector<uint8_t> rgb(eyes.size() * (size_t)W * H * 3);
            const auto t0 = std::chrono::high_resolution_clock::now();
            const int rc = tracer_cuda_render_views(dev, cams.data(), (int32_t)cams.size(), W, H, &o, rgb.data());
            const auto t1 = std::chrono::high_resolution_clock::now();
            tracer_cuda_scene_destroy(dev);
            if (rc) throw std::runtime_error(tracer_cuda_last_error());
            std::cerr << "\n CUDA      : true" << std::endl;
            std::cerr << "\n Views     : " << eyes.size() << std::endl;
            std::cerr << "\n Duration  : " << std::chrono::duration_cast<std::chrono::milliseconds>(t1 - t0).count() << std::endl;
            if (!output.empty()) {
                const size_t dot = output.rfind('.'), slash = output.rfind('/');
                const bool has_ext = dot != std::string::npos && (slash == std::string::npos || dot > slash);
                const std::string stem = has_ext ? output.substr(0, dot) : output, ext = has_ext ? output.substr(dot) : "";
                for (size_t v = 0; v < eyes.size(); ++v) {
                    const std::string path = stem + "_" + std::to_string(v) + ext;
                    if (tracer_write_ppm(path.c_str(), rgb.data() + v * (size_t)W * H * 3, W, H, p6))
                        throw std::runtime_error(tracer_host_last_error());
                    std::cout << "Rendered image in: " << path << std::endl;
                }
            } else {
                std::cout << "Nothing saved: use -o to save rendered image" << std::endl;
            }
            tracer_scene_host_free(sorted_scene);
            tracer_scene_host_free(scene);
            tracer_cuda_shutdown();
            return 0;
        }
        o.crop_x = crop[0], o.crop_y = crop[1], o.crop_w = crop[2], o.crop_h = crop[3];
        const int out_w = have_crop ? crop[2] : W, out_h = have_crop ? crop[3] : H;
        std::vector<uint8_t> rgb((size_t)out_w * out_h * 3);
        const auto t0 = std::chrono::high_resolution_clock::now(); // main.cpp:583
        if (tracer_cuda_render(flat, &cam, W, H, &o, rgb.data())) throw std::runtime_error(tracer_cuda_last_error());
        const auto t1 = std::chrono::high_resolution_clock::now();
        std::cerr << "\n CUDA      : true" << std::endl;
        std::cerr << "\n GPUs      : " << gpus << std::endl;
        std::cerr << "\n Duration  : " << std::chrono::duration_cast<std::chrono::milliseconds>(t1 - t0).count() << std::endl;
        if (!output.empty()) {
            if (tracer_write_ppm(output.c_str(), rgb.data(), out_w, out_h, p6)) throw std::runtime_error(tracer_host_last_error());
            std::cout << "Rendered image in: " << output << std::endl; // main.cpp:688
        } else {
            std::cout << "Nothing saved: use -o to save rendered image" << std::endl;
        }
        tracer_scene_host_free(sorted_scene);
        tracer_scene_host_free(scene);
        tracer_cuda_shutdown();
        return 0;
    } catch (const std::exception &e) {
        std::cerr << "error: " << e.what() << std::endl;
        return 1;
    }
}
