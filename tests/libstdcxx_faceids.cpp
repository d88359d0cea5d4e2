// libstdcxx_faceids.cpp — test infrastructure: the faceIDs of a seeded frame drawn by libstdc++ itself (std::mt19937,
// std::uniform_int_distribution<int>, std::uniform_real_distribution<float>) in the order the reference's scan_row
// consumes them: the replay loop of oracle/ref_harness.cpp ref_render_frame (src/main.cpp:743-754).  Built and run by
// tests/test_abi.py; not part of the library.
//
//   libstdcxx_faceids W H seed F_0 ... F_{L-1}  < hit mask (W*H bytes, image index h*W+w)  > faceids (int32 [W*H, L])
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

int main(int argc, char **argv) {
    if (argc < 4) return 2;
    const int W = std::atoi(argv[1]), H = std::atoi(argv[2]);
    const unsigned seed = (unsigned)std::strtoul(argv[3], nullptr, 10);
    std::vector<int> faces;
    for (int k = 4; k < argc; ++k) faces.push_back(std::atoi(argv[k]));
    const int L = (int)faces.size();
    std::vector<uint8_t> hit((size_t)W * H);
    if (std::fread(hit.data(), 1, hit.size(), stdin) != hit.size()) return 3;
    std::vector<int32_t> faceid((size_t)W * H * L, -1);
    std::mt19937 replay(seed);
    std::uniform_real_distribution<float> distrib2(0, 1.f);
    for (int hh = H - 1; hh >= 0; --hh) {
        for (int w = 0; w < W; ++w) {
            const size_t i = (size_t)hh * W + w;
            if (!hit[i]) continue;
            for (int l = 0; l < L; ++l) {
                std::uniform_int_distribution<int> d1(0, faces[l] - 1);
                faceid[i * L + l] = d1(replay);
                (void)float(distrib2(replay));
                (void)float(distrib2(replay));
            }
        }
    }
    return std::fwrite(faceid.data(), sizeof(int32_t), faceid.size(), stdout) == faceid.size() ? 0 : 4;
}
