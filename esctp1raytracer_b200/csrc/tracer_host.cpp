// tracer_host.cpp — host-side pieces of the C ABI that need no device:
// the reference camera, the std::mt19937 replay of scan_row's draws, band maths.
#include <cmath>
#include <cstdint>
#include <cstring>

#include "../../include/tracer_cuda.h"

namespace {

struct V3 {
    float x, y, z;
};
inline V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 mul(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
inline V3 dvd(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
inline float dot(V3 a, V3 b) {
    float s = 0;
    s += a.x * b.x;
    s += a.y * b.y;
    s += a.z * b.z;
    return s;
}
inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline V3 normalize(V3 a) { return dvd(a, std::sqrt(dot(a, a))); }

// The 32-bit Mersenne Twister with the std::mt19937 parameters.
struct Mt19937 {
    uint32_t mt[624];
    int idx;
    explicit Mt19937(uint32_t seed) {
        mt[0] = seed;
        for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
        idx = 624;
    }
    void refill() {
        for (int i = 0; i < 624; ++i) {
            const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
            mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        idx = 0;
    }
    uint32_t next() {
        if (idx >= 624) refill();
        uint32_t y = mt[idx++];
        y ^= (y >> 11);
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= (y >> 18);
        return y;
    }
    // libstdc++'s uniform_int_distribution<int>(0, range-1) over a 32-bit engine
    // (Lemire's nearly-divisionless reduction, bits/uniform_int_dist.h)
    int below(uint32_t range) {
        uint64_t product = (uint64_t)next() * (uint64_t)range;
        uint32_t low = (uint32_t)product;
        if (low < range) {
            const uint32_t threshold = (0u - range) % range;
            while (low < threshold) {
                product = (uint64_t)next() * (uint64_t)range;
                low = (uint32_t)product;
            }
        }
        return (int)(product >> 32);
    }
};

}  // namespace

extern "C" {

int tracer_cuda_abi_version(void) { return TRACER_CUDA_ABI_VERSION; }

// src/scene/camera.h:16-29.  camera.h:20 calls tan() on a float whose value is fixed by the literal vfov = 60.f
// (main.cpp:549): the optimised reference build folds the call at compile time to the correctly rounded float
// (0x3f13cd3a), where glibc's run-time tanf — what an -O0 or instrumented build of the same source calls — returns
// the neighbouring float and moves most pixels by an ulp.  tan in double, narrowed once, gives the folded value;
// the oracle pin test holds it to the reference's -O3 camera bit for bit.
void tracer_camera_lookat(const float eye[3], const float look[3], const float vup[3], float vfov_deg, float aspect,
                          tracer_camera *out) {
    const float theta = (float)(vfov_deg * M_PI / 180);
    const float half_height = (float)std::tan((double)(theta / 2));
    const float half_width = aspect * half_height;
    const V3 origin{eye[0], eye[1], eye[2]};
    const V3 w = normalize(sub(origin, V3{look[0], look[1], look[2]}));
    const V3 u = normalize(cross(V3{vup[0], vup[1], vup[2]}, w));
    const V3 v = cross(w, u);
    const V3 llc = sub(sub(sub(origin, mul(u, half_width)), mul(v, half_height)), w);
    const V3 hor = mul(mul(u, 2.f), half_width);
    const V3 ver = mul(mul(v, 2.f), half_height);
    const V3 src[4] = {origin, llc, hor, ver};
    float *dst[4] = {out->origin, out->lower_left_corner, out->horizontal, out->vertical};
    for (int i = 0; i < 4; ++i) dst[i][0] = src[i].x, dst[i][1] = src[i].y, dst[i][2] = src[i].z;
}

int32_t tracer_band_row_count(int32_t height, int32_t band_rows, int32_t band_index, int32_t band_count) {
    if (band_count <= 1) return height;
    if (band_rows <= 0 || band_index < 0 || band_index >= band_count) return -1;
    const int n_bands = (height + band_rows - 1) / band_rows;
    int rows = 0;
    for (int b = band_index; b < n_bands; b += band_count) {
        const int r0 = b * band_rows;
        const int r1 = r0 + band_rows < height ? r0 + band_rows : height;
        rows += r1 - r0;
    }
    return rows;
}

// scan_row draws, per hit pixel and light, in scan order (main.cpp:628, 704, 740-754):
//   faceID = uniform_int_distribution<int>(0, F-1)(gen); two uniform_real<float> draws
//   (one engine output each for a 32-bit engine and a 24-bit mantissa).
// `hit` and `faceid` are in image index order h*W+w.
int tracer_mt19937_faceids(const tracer_scene_flat *scene, int32_t width, int32_t height, uint32_t seed,
                           const uint8_t *hit, int32_t *faceid) {
    if (!scene || !hit || !faceid || width <= 0 || height <= 0) return TRACER_ERR_INVALID;
    Mt19937 gen(seed);
    const int L = scene->n_lights;
    for (int h = height - 1; h >= 0; --h) {
        for (int w = 0; w < width; ++w) {
            const size_t i = (size_t)h * width + w;
            for (int l = 0; l < L; ++l) {
                int fid = -1;
                if (hit[i]) {
                    const int lg = scene->light_geom[l];
                    const uint32_t F = (uint32_t)(scene->geom_tri_offset[lg + 1] - scene->geom_tri_offset[lg]);
                    fid = gen.below(F);
                    (void)gen.next();
                    (void)gen.next();
                }
                faceid[i * L + l] = fid;
            }
        }
    }
    return TRACER_OK;
}

}  // extern "C"
