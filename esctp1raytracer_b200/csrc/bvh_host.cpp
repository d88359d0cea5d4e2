// bvh_host.cpp — internal hooks (tests only, no GPU needed): the BVH of the optional mode (bvh.cuh) built and traversed on
// the host, from the same source as the device build and kernels, in front of the host build of strict_math.cuh's
// strict::intersect_triangle.  Compiled by the host compiler with -ffp-contract=off: every float operation rounds once,
// as the device's _rn intrinsics do; the intrinsics the headers use are defined here as the IEEE operations they are.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include <cuda_runtime.h> // host compiler: __device__ / __host__ expand to nothing, float4 etc. are defined

static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __fsqrt_rn(float a) { return std::sqrt(a); }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline float __double2float_rn(double a) { return (float)a; }

#include "bvh.cuh"

namespace {
// post-order: fill in node i's children from theirs (the device's refit_kernel, sequentially)
void refit(std::vector<bvh::Node> &nodes, const std::vector<bvh::TriInfo> &ti, int i) {
    bvh::Node &nd = nodes[i];
    float4 lo[2], hi[2];
    int mn[2];
    for (int c = 0; c < 2; ++c) {
        const int ch = nd.child[c];
        if (ch < 0) {
            const bvh::TriInfo &t = ti[~ch];
            lo[c] = make_float4(t.lo[0], t.lo[1], t.lo[2], t.sigma), hi[c] = make_float4(t.hi[0], t.hi[1], t.hi[2], 0.f), mn[c] = ~ch;
        } else {
            refit(nodes, ti, ch);
            bvh::merge(nodes[ch], lo[c], hi[c], mn[c]);
        }
    }
    nd.lo0 = lo[0], nd.hi0 = hi[0], nd.lo1 = lo[1], nd.hi1 = hi[1], nd.mn[0] = mn[0], nd.mn[1] = mn[1];
}
}  // namespace

extern "C" {

// The construction of the device build for n triangles (verts [n*9]).  nodes_out: [max(n-1, 1) * 20] words (bvh::Node:
// lo0, hi0, lo1, hi1 as float4 with lo.w = sigma, then child[2], mn[2] as int32); always_out [n]: the always-test list,
// ascending.  Returns the number of triangles in the tree (n_in); the root is node 0 (n_in >= 2) or leaf
// *root_leaf (n_in == 1).
int tracer__bvh_build_host(int n, const float *verts, float *nodes_out, int *root_leaf, int *always_out, int *n_always) {
    std::vector<bvh::TriInfo> ti((size_t)std::max(n, 1));
    float clo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, chi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int i = 0; i < n; ++i) {
        ti[i] = bvh::tri_info(verts + 9 * (size_t)i);
        if (ti[i].in_tree)
            for (int c = 0; c < 3; ++c) clo[c] = std::min(clo[c], ti[i].c[c]), chi[c] = std::max(chi[c], ti[i].c[c]);
    }
    std::vector<unsigned long long> keys((size_t)n);
    for (int i = 0; i < n; ++i)
        keys[i] = ti[i].in_tree ? ((unsigned long long)bvh::morton(ti[i].c, clo, chi) << 32) | (uint32_t)i : bvh::KEY_ALWAYS | (uint32_t)i;
    std::sort(keys.begin(), keys.end());
    int n_in = 0;
    while (n_in < n && keys[n_in] < bvh::KEY_ALWAYS) ++n_in;
    *n_always = n - n_in;
    for (int j = n_in; j < n; ++j) always_out[j - n_in] = (int)(keys[j] & 0xffffffffull);
    *root_leaf = n_in == 1 ? (int)(keys[0] & 0xffffffffull) : -1;
    if (n_in >= 2) {
        std::vector<bvh::Node> nodes((size_t)n_in - 1);
        for (int i = 0; i < n_in - 1; ++i) {
            int l, r, split;
            bool ll, rl;
            bvh::karras_node(keys.data(), n_in, i, l, r, ll, rl, split);
            nodes[i].child[0] = l, nodes[i].child[1] = r;
        }
        refit(nodes, ti, 0);
        std::memcpy(nodes_out, nodes.data(), nodes.size() * sizeof(bvh::Node));
    }
    return n_in;
}

// n_rays queries (o, d: [n_rays*3], t: [n_rays]) against a tree from tracer__bvh_build_host.  mode 0: closest hit (the
// strict test with t = FLT_MAX per triangle, merged as (t, index); t is ignored) -> idx_out / t_out = index and t, or -1;
// mode 1: first occluder with the ray's own t -> the lowest accepted index and its t2, or -1.  brute != 0 answers by
// testing every triangle in index order instead of traversing.  m: the dilation (bvh::frame_margin), dscale: 1 = the
// derived margins, 0 = none.  *tests_out: strict tests done.
void tracer__bvh_query_host(int n, const float *verts, const float *nodes, int n_in, int root_leaf, const int *always, int n_always,
                            int n_rays, const float *o, const float *d, const float *t, int mode, int brute, float m, float dscale,
                            int *idx_out, float *t_out, long long *tests_out) {
    std::vector<unsigned long long> akeys((size_t)std::max(n_always, 1));
    for (int i = 0; i < n_always; ++i) akeys[i] = bvh::KEY_ALWAYS | (uint32_t)always[i];
    const bvh::Tree tr{reinterpret_cast<const bvh::Node *>(nodes), n_in, root_leaf, akeys.data(), n_always};
    long long tests = 0;
    for (int r = 0; r < n_rays; ++r) {
        const float *orr = o + 3 * (size_t)r, *dr = d + 3 * (size_t)r;
        const strict::f3 so = strict::ld(orr), sd = strict::ld(dr);
        auto strict_t = [&](int tri, float t0, float &t2) {
            ++tests;
            const float *q = verts + 9 * (size_t)tri;
            float tt = t0, v = 0.f;
            const bool hit = strict::intersect_triangle(so, sd, strict::ld(q), strict::ld(q + 3), strict::ld(q + 6), tt, v);
            t2 = tt;
            return hit;
        };
        const bvh::RayBox rb = bvh::make_ray(orr, dr, m, dscale);
        unsigned long long key = bvh::KEY_NONE;
        if (mode == 0) {
            auto test = [&](int tri) -> unsigned long long {
                float t2;
                return strict_t(tri, FLT_MAX, t2) ? ((unsigned long long)bvh::f2u(t2) << 32) | (uint32_t)tri : bvh::KEY_NONE;
            };
            if (brute)
                for (int i = 0; i < n; ++i) key = std::min(key, test(i));
            else
                bvh::closest(tr, rb, key, test);
            idx_out[r] = key == bvh::KEY_NONE ? -1 : (int)(key & 0xffffffffull);
            t_out[r] = key == bvh::KEY_NONE ? 0.f : bvh::u2f((uint32_t)(key >> 32));
        } else {
            auto test = [&](int tri) -> long long {
                float t2;
                return strict_t(tri, t[r], t2) ? (long long)bvh::f2u(t2) : -1;
            };
            if (brute) {
                for (int i = 0; i < n && key == bvh::KEY_NONE; ++i) {
                    const long long t2 = test(i);
                    if (t2 >= 0) key = ((unsigned long long)(uint32_t)i << 32) | (uint32_t)t2;
                }
            } else {
                key = bvh::occluder(tr, rb, t[r], test);
            }
            idx_out[r] = key == bvh::KEY_NONE ? -1 : (int)(key >> 32);
            t_out[r] = key == bvh::KEY_NONE ? 0.f : bvh::u2f((uint32_t)(key & 0xffffffffull));
        }
    }
    *tests_out = tests;
}

float tracer__bvh_margin(double ext, double lmax) { return bvh::frame_margin(ext, lmax); }

}  // extern "C"
