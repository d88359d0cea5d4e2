// strict_host_shim.cpp — test infrastructure: csrc/strict_math.cuh (the device's restatement of the reference's
// arithmetic) compiled for the HOST by plain g++, with the correctly-rounded CUDA intrinsics mapped to the IEEE
// operations they are defined as (-ffp-contract=off: no FMA contraction, SSE scalar: every operation rounds once).
// tests/test_strict_host.py compares it, pair by pair and bit by bit, with the pinned oracle (oracle/restated.c), so an
// edit of strict_math.cuh that changes an operation or its order is caught on the CPU, before any GPU run.
// tests/test_powf_glibc.py compares its strict::powf_glibc with libm's powf the same way, over every float of the
// ranges that matter; the comparison loops are here, in C and threaded, and Python only reads the counts.
#include <algorithm>
#include <array>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>
#include <cuda_runtime.h> // plain g++: __device__ / __forceinline__ expand to nothing special, float4 etc. are defined

static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __fsqrt_rn(float a) { return std::sqrt(a); }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline float __double2float_rn(double a) { return (float)a; }

#include "../esctp1raytracer_b200/csrc/strict_math.cuh"

extern "C" {
// n pairs: orig[3n], dir[3n], tri[9n], t_in[n] -> hit[n], t_out[n], v_out[n] (t, v unchanged on a miss; v enters as 0)
void strict_host_intersect_triangles(int n, const float *orig, const float *dir, const float *tri, const float *t_in,
                                     uint8_t *hit, float *t_out, float *v_out) {
    for (int i = 0; i < n; ++i) {
        float t = t_in[i], v = 0.f;
        const float *p = tri + 9 * (size_t)i;
        hit[i] = strict::intersect_triangle(strict::ld(orig + 3 * (size_t)i), strict::ld(dir + 3 * (size_t)i), strict::ld(p),
                                            strict::ld(p + 3), strict::ld(p + 6), t, v);
        t_out[i] = t, v_out[i] = v;
    }
}
// extension (no reference code): cr = centre, radius
void strict_host_intersect_spheres(int n, const float *orig, const float *dir, const float *cr, const float *t_in, uint8_t *hit,
                                   float *t_out) {
    for (int i = 0; i < n; ++i) {
        float t = t_in[i];
        const float *c = cr + 4 * (size_t)i;
        hit[i] = strict::intersect_sphere(strict::ld(orig + 3 * (size_t)i), strict::ld(dir + 3 * (size_t)i), make_float4(c[0], c[1], c[2], c[3]), t);
        t_out[i] = t;
    }
}
// vec.h helpers on n vectors: dot, cross, normalize, length
void strict_host_vec(int n, const float *a, const float *b, float *dot, float *cross, float *norm, float *len) {
    for (int i = 0; i < n; ++i) {
        const strict::f3 x = strict::ld(a + 3 * (size_t)i), y = strict::ld(b + 3 * (size_t)i);
        dot[i] = strict::dot(x, y);
        const strict::f3 c = strict::cross(x, y), nn = strict::normalize(x);
        cross[3 * i] = c.x, cross[3 * i + 1] = c.y, cross[3 * i + 2] = c.z;
        norm[3 * i] = nn.x, norm[3 * i + 1] = nn.y, norm[3 * i + 2] = nn.z;
        len[i] = strict::length(x);
    }
}

// ---- powf ----------------------------------------------------------------------------------------------------------
// The x of a range: every stride-th float bit pattern from lo_bits up to hi_bits (inclusive), i.e.
// n = (hi_bits - lo_bits) / stride + 1 values.
static int64_t range_count(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride) {
    return hi_bits < lo_bits || stride == 0 ? 0 : ((int64_t)hi_bits - lo_bits) / stride + 1;
}
static float bits_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static uint32_t float_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

void strict_host_powf_range(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride, float y, float *out) {
    const int64_t n = range_count(lo_bits, hi_bits, stride);
    for (int64_t i = 0; i < n; ++i) out[i] = strict::powf_glibc(bits_float(lo_bits + (uint32_t)(i * stride)), y);
}
void strict_host_powf_pairs(int64_t n, const float *x, const float *y, float *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = strict::powf_glibc(x[i], y[i]);
}
// the tables that powf_glibc's tables are checked against (tests/test_powf_glibc.py)
void strict_host_powf_tables(double *log2_tab32, uint64_t *exp2_tab32) {
    for (int i = 0; i < 16; ++i) log2_tab32[2 * i] = strict::POWF_LOG2_TAB[i][0], log2_tab32[2 * i + 1] = strict::POWF_LOG2_TAB[i][1];
    for (int i = 0; i < 32; ++i) exp2_tab32[i] = strict::POWF_EXP2_TAB[i];
}
int strict_host_has_fma_avx2(void) { return __builtin_cpu_supports("fma") && __builtin_cpu_supports("avx2"); }
}

namespace {
// the function under test: 0 = strict::powf_glibc, 1 = (float)pow((double)x, (double)y) (what the shading used to
// compute)
float impl_powf(int impl, float x, float y) {
    return impl == 0 ? strict::powf_glibc(x, y) : (float)std::pow((double)x, (double)y);
}
bool same(float a, float b) { return float_bits(a) == float_bits(b) || (std::isnan(a) && std::isnan(b)); }

// counts i in [0, n) with got(i) != want(i) (two NaNs are equal) on n_threads threads; the first max_rep mismatches in
// index order go to rep as (x, y, got, want)
template <class XY, class Got, class Want>
int64_t count_mismatches(int64_t n, int n_threads, XY xy, Got got, Want want, float *rep, int max_rep) {
    const int64_t block = 1 << 20;
    std::atomic<int64_t> next{0}, total{0};
    std::vector<std::vector<std::pair<int64_t, std::array<float, 4>>>> first(std::max(n_threads, 1));
    auto work = [&](int tid) {
        int64_t mine = 0;
        for (int64_t b; (b = next.fetch_add(block)) < n;) {
            const int64_t e = std::min(n, b + block);
            for (int64_t i = b; i < e; ++i) {
                float x, y;
                xy(i, x, y);
                const float g = got(i, x, y), w = want(x, y);
                if (same(g, w)) continue;
                ++mine;
                auto &f = first[tid];
                if ((int)f.size() < max_rep) f.push_back({i, {x, y, g, w}});
            }
        }
        total += mine;
    };
    std::vector<std::thread> th;
    for (int t = 1; t < n_threads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto &t : th) t.join();
    std::vector<std::pair<int64_t, std::array<float, 4>>> all;
    for (auto &f : first) all.insert(all.end(), f.begin(), f.end());
    std::sort(all.begin(), all.end(), [](const auto &a, const auto &b) { return a.first < b.first; });
    for (int k = 0; k < max_rep && k < (int)all.size(); ++k)
        for (int j = 0; j < 4; ++j) rep[4 * k + j] = all[k].second[j];
    return total;
}
float libm_powf(float x, float y) { return powf(x, y); }
} // namespace

extern "C" {
// impl (0: the port, 1: the old formula) against libm powf over a range of x (see strict_host_powf_range)
int64_t strict_host_powf_check_range(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride, float y, int impl, int n_threads,
                                     float *rep, int max_rep) {
    return count_mismatches(
        range_count(lo_bits, hi_bits, stride), n_threads, [&](int64_t i, float &x, float &yy) { x = bits_float(lo_bits + (uint32_t)(i * stride)), yy = y; },
        [&](int64_t, float x, float yy) { return impl_powf(impl, x, yy); }, libm_powf, rep, max_rep);
}
int64_t strict_host_powf_check_pairs(int64_t n, const float *x, const float *y, int impl, int n_threads, float *rep, int max_rep) {
    return count_mismatches(
        n, n_threads, [&](int64_t i, float &xx, float &yy) { xx = x[i], yy = y[i]; },
        [&](int64_t, float xx, float yy) { return impl_powf(impl, xx, yy); }, libm_powf, rep, max_rep);
}
// results computed elsewhere (the device build of the port) against the host build of the port
int64_t strict_host_powf_compare_range(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride, float y, const float *got,
                                       int n_threads, float *rep, int max_rep) {
    return count_mismatches(
        range_count(lo_bits, hi_bits, stride), n_threads, [&](int64_t i, float &x, float &yy) { x = bits_float(lo_bits + (uint32_t)(i * stride)), yy = y; },
        [&](int64_t i, float, float) { return got[i]; }, [](float x, float yy) { return strict::powf_glibc(x, yy); }, rep, max_rep);
}
int64_t strict_host_powf_compare_pairs(int64_t n, const float *x, const float *y, const float *got, int n_threads, float *rep,
                                       int max_rep) {
    return count_mismatches(
        n, n_threads, [&](int64_t i, float &xx, float &yy) { xx = x[i], yy = y[i]; }, [&](int64_t i, float, float) { return got[i]; },
        [](float xx, float yy) { return strict::powf_glibc(xx, yy); }, rep, max_rep);
}
}
