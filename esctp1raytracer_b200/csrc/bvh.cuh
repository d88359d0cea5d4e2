// bvh.cuh — OPTIONAL mode (opts.accel = 1): a linear BVH (Karras 2012) over the triangles, built on the device, and a
// conservative traversal in front of the reference's own test (strict::intersect_triangle).  The tree only ever decides
// which (ray, triangle) pairs reach the strict test; the results are merged as the sweeps merge them (closest hit: the
// minimum of t << 32 | index; first occluder: the minimum of index << 32 | t2), so a traversal that never skips a pair
// the strict test accepts gives the bytes of the brute-force sweeps.  Why it never does is argued at the constants below.
//
//   construction (device: build kernels below + cub::DeviceRadixSort in tracer_cuda.cu; host: tracer__bvh_build_host)
//     1. per triangle: box, centre, sigma = |e1| |e2| (tri_info).  Triangles whose vertices, box or sigma are not finite,
//        or whose sigma is >= SIGMA_MAX, stay out of the tree: every ray tests them after the tree ("always" list).
//     2. keys = 30-bit Morton code of the centre (10 bits per axis over the centres' box) << 32 | index, sorted; the
//        always-list triangles get the key 0xffffffff << 32 | index and sort last, in index order.
//     3. internal node i of the n_in - 1: Karras' longest-common-prefix split of the sorted keys (karras_node).
//     4. bottom-up refit with one arrival flag per node: each node stores its two children's boxes, the smallest
//        triangle index below each child (first-occluder pruning) and the largest sigma below each child.
//   traversal (closest / occluder): one thread per ray, a stack, the children's boxes dilated per node (child_test).
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "strict_math.cuh"

namespace bvh {

// one rounding per operation and no contraction: the device's _rn intrinsics, a host build's IEEE operations (the host
// translation unit is compiled with -ffp-contract=off), so the host hooks run the device's arithmetic
__host__ __device__ __forceinline__ float fadd(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ float fsub(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ float fmul(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ float fdiv(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}
__host__ __device__ __forceinline__ double dmad(double a, double b, double c) { // a*b + c, two roundings
#ifdef __CUDA_ARCH__
    return __dadd_rn(__dmul_rn(a, b), c);
#else
    return a * b + c;
#endif
}
__host__ __device__ __forceinline__ double dsqrt(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return std::sqrt(a);
#endif
}
__host__ __device__ __forceinline__ uint32_t f2u(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
__host__ __device__ __forceinline__ float u2f(uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
}
__host__ __device__ __forceinline__ uint32_t ord(float f) { // order-preserving float -> uint
    const uint32_t u = f2u(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float unord(uint32_t u) { return u2f((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }
__host__ __device__ __forceinline__ int clz64(unsigned long long x) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}

constexpr unsigned long long KEY_NONE = 0xffffffffffffffffull;
constexpr unsigned long long KEY_ALWAYS = 0xffffffffull << 32; // | index: triangles outside the tree sort last

// ---- the conservative test -------------------------------------------------------------------------------------
// Notation: u = 2^-24 (unit roundoff), eps = FLT_EPSILON = 2u; o, d the ray's float origin and direction (|d| <= 1.0001:
// every ray is a float-normalised vector); v0 and the float edges E1 = fl(v1 - v0), E2 = fl(v2 - v0) as the strict test
// forms them; sigma = |E1| |E2|; det* = d . (E2 x E1), (u*, v*, t*) the exact solution of o + t* d = v0 + u* E1 + v* E2.
//
// Suppose the strict test accepts the pair with (u, v, t2).  Float error analysis of its dot and cross products
// (gamma_3 per dot product, gamma_2 per cross component):
//   |det_f - det*|                    <= 6 u |d| sigma                                   (det_f = fl(E1 . fl(d x E2)))
//   |fl(T . Pv) - (o - v0).(d x E2)|  <= 7 u |d| |E2| |o - v0|      (likewise the v and t numerators with |E1|, sigma)
//   u = num / det_f * (1 + eta), |eta| <= 1.01 u                    (double division and product, rounding to float)
// The test rejects |det_f| < eps.  With sigma < SIGMA_MAX = 1/8, |det*| >= 2u - 6 * 1.0001 * u / 8 >= 1.25 u: the ray is
// not parallel to the plane and t* is finite.  (A larger triangle can be accepted by a ray that runs in its plane, where
// det_f is only rounding noise and u, v, t2 can be anything; such triangles go on the always list.)  Then
//   (u* - u) det* = -(numerator error) - eta num + u (det_f - det*)   =>   |u* - u| |E1| <= |d| sigma (6.5 |o - v0| + 4.8 |E1|)
// and the same for v with E2, so the point X = o + t* d of the exact line lies within
//   |X - (v0 + u E1 + v E2)| <= |d| sigma (13 |o - v0| + 4.8 (|E1| + |E2|))                                         (LAT)
// of a point of the triangle (u, v >= eps, u + v <= 1 up to one rounding), and its parameter satisfies
//   |t* - t2| <= 6.3 sigma |o - v0| + 4.8 |d| sigma t2                                                              (LON)
// Note that eps cancels: the strict test's absolute threshold on det bounds the error by geometry, not by eps times it.
// Per node and ray, with Lo = sum_c max |o_c - box_c| (>= |o - v0| for every v0 in the box, and >= half the box's L1
// extent, hence |E1| + |E2| <= 4 Lo (1 + u)):
//   LAT <= 1.0001 * 32.2 sigma Lo <= C_LAT sigma Lo,   LON <= C_ABS sigma Lo + C_REL sigma t2
// so the box dilated by m + C_LAT sigma_max Lo (m below) contains X, at a parameter t* in
// [-C_ABS sigma Lo, t_ref (1 + C_REL sigma) + C_ABS sigma Lo] whenever t2 <= t_ref (t2 >= eps > 0, C_REL sigma < 1).
// The traversal prunes a child only when the exact line misses that dilated box on that parameter range.
constexpr float SIGMA_MAX = 0.125f;
constexpr float C_LAT = 48.f; // 32.2 with every |d|, rounding and (1 + u) factor, rounded up generously
constexpr float C_ABS = 7.f;  // 6.3 -> 7
constexpr float C_REL = 5.f;  // 4.8 * 1.0001 -> 5
// Margin terms are themselves evaluated in float (a handful of roundings, relative error < 10 u): multiplied by SAFE.
constexpr float SAFE = 1.0001f;
// Slab entries and exits: fl((fl(box - D) - o) * fl(1/d)) is the exact (box' - o) / d times (1 + theta), |theta| <=
// gamma_3 ~ 3u (Ize 2013: robust BVH traversal); scaling by (1 -+ 8u) (the scaling's own rounding included) moves the
// entry down and the exit up past every exact value.  The rounding of fl(box -+ D) itself moves a plane by at most
// u |box -+ D|, covered by m (u |coordinate| part) and SAFE (u D part).
constexpr float WIDEN = 4.f * TRC_EPS; // 8u
// m: absolute dilation per frame, from the K analysis of the sweeps (kernels.cuh "Margin"): the float triangle
// (v0, v0 + E1, v0 + E2) lies within u max|edge| of the true one, and the dilated planes round by u |coordinate|.  Both
// are far below CK eps (ext + lmax), ext = the largest |coordinate| of the tree's box and the ray origins' box (eye,
// scene), lmax the reach bound of the rays (diag for primary rays, (k+1) diag for light k).  CK = 64 as for K.
constexpr double M_CK = 64.0;
__host__ __device__ __forceinline__ float frame_margin(double ext, double lmax) {
    return (float)(M_CK * (double)TRC_EPS * (ext + lmax) * 1.0001);
}

struct Node {            // 80 bytes; child c: box lo_c.xyz / hi_c.xyz, lo_c.w = largest sigma below it
    float4 lo0, hi0, lo1, hi1;
    int child[2];        // >= 0 internal node, < 0 leaf: triangle ~child
    int mn[2];           // smallest triangle index below each child
};

struct TriInfo {
    float lo[3], hi[3], c[3], sigma;
    bool in_tree;
};

__host__ __device__ __forceinline__ bool finite_f(float x) { return fabsf(x) <= FLT_MAX; } // false for inf and NaN

// box, centre, sigma of one triangle (v: its 9 vertex floats)
__host__ __device__ __forceinline__ TriInfo tri_info(const float *v) {
    TriInfo ti;
    bool ok = true;
    double n1 = 0.0, n2 = 0.0;
    for (int c = 0; c < 3; ++c) {
        ti.lo[c] = fminf(fminf(v[c], v[3 + c]), v[6 + c]);
        ti.hi[c] = fmaxf(fmaxf(v[c], v[3 + c]), v[6 + c]);
        ti.c[c] = fmul(0.5f, fadd(ti.lo[c], ti.hi[c]));
        ok = ok && finite_f(v[c]) && finite_f(v[3 + c]) && finite_f(v[6 + c]) && finite_f(ti.c[c]);
        const double e1 = (double)fsub(v[3 + c], v[c]), e2 = (double)fsub(v[6 + c], v[c]); // the strict test's float edges
        n1 = dmad(e1, e1, n1), n2 = dmad(e2, e2, n2);
    }
    // |E1| |E2| rounded up: the double evaluation is within 4 double ulps, the factor adds 2^-20, the cast to float loses
    // at most 2^-24 relative
    const double sg = dsqrt(n1) * dsqrt(n2) * (1.0 + 0x1p-20);
    ti.sigma = (float)sg;
    ti.in_tree = ok && finite_f(ti.sigma) && ti.sigma < SIGMA_MAX;
    if (!ti.in_tree) ti.sigma = 0.f;
    return ti;
}

__host__ __device__ __forceinline__ uint32_t expand10(uint32_t x) {
    x &= 0x3ffu;
    x = (x | (x << 16)) & 0x030000ffu;
    x = (x | (x << 8)) & 0x0300f00fu;
    x = (x | (x << 4)) & 0x030c30c3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}
// centres' box clo/chi -> 30-bit Morton code (quality only: any key order gives a correct tree)
__host__ __device__ __forceinline__ uint32_t morton(const float c[3], const float clo[3], const float chi[3]) {
    uint32_t m = 0;
    for (int a = 0; a < 3; ++a) {
        const float ext = fsub(chi[a], clo[a]);
        const float f = ext > 0.f ? fdiv(fsub(c[a], clo[a]), ext) : 0.f;
        const uint32_t q = (uint32_t)fminf(fmaxf(fmul(f, 1024.f), 0.f), 1023.f);
        m |= expand10(q) << a;
    }
    return m;
}

__host__ __device__ __forceinline__ int lcp(const unsigned long long *k, int n, int i, int j) {
    return (j < 0 || j >= n) ? -1 : clz64(k[i] ^ k[j]); // keys are unique (they carry the index)
}
// Karras 2012, internal node i of the n - 1 over the n sorted unique keys: its two children (leaf = ~triangle) and
// which slot of its children's parents it is
__host__ __device__ __forceinline__ void karras_node(const unsigned long long *k, int n, int i, int &left, int &right,
                                                     bool &left_leaf, bool &right_leaf, int &split) {
    const int d = lcp(k, n, i, i + 1) > lcp(k, n, i, i - 1) ? 1 : -1;
    const int dmin = lcp(k, n, i, i - d);
    int lmax = 2;
    while (lcp(k, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (lcp(k, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = lcp(k, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (lcp(k, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    split = i + s * d + (d < 0 ? -1 : 0);
    const int first = i < j ? i : j, last = i < j ? j : i;
    left_leaf = first == split, right_leaf = last == split + 1;
    left = left_leaf ? ~(int)(uint32_t)(k[split] & 0xffffffffull) : split;
    right = right_leaf ? ~(int)(uint32_t)(k[split + 1] & 0xffffffffull) : split + 1;
}

// the union of a node's two children: lo.w = largest sigma
__host__ __device__ __forceinline__ void merge(const Node &nd, float4 &lo, float4 &hi, int &mn) {
    lo = make_float4(fminf(nd.lo0.x, nd.lo1.x), fminf(nd.lo0.y, nd.lo1.y), fminf(nd.lo0.z, nd.lo1.z), fmaxf(nd.lo0.w, nd.lo1.w));
    hi = make_float4(fmaxf(nd.hi0.x, nd.hi1.x), fmaxf(nd.hi0.y, nd.hi1.y), fmaxf(nd.hi0.z, nd.hi1.z), 0.f);
    mn = nd.mn[0] < nd.mn[1] ? nd.mn[0] : nd.mn[1];
}

struct Tree {
    const Node *nodes;               // [n_in - 1]
    int n_in;                        // triangles in the tree (0: none; 1: the root is that leaf)
    int root_leaf;                   // the triangle when n_in == 1
    const unsigned long long *always; // [n_always] keys KEY_ALWAYS | index, ascending index
    int n_always;
};

__host__ __device__ __forceinline__ Node load_node(const Node *p) {
#ifdef __CUDA_ARCH__
    const float4 *q = reinterpret_cast<const float4 *>(p);
    Node n;
    n.lo0 = __ldg(q), n.hi0 = __ldg(q + 1), n.lo1 = __ldg(q + 2), n.hi1 = __ldg(q + 3);
    const int4 c = __ldg(reinterpret_cast<const int4 *>(q + 4));
    n.child[0] = c.x, n.child[1] = c.y, n.mn[0] = c.z, n.mn[1] = c.w;
    return n;
#else
    return *p;
#endif
}

struct RayBox {
    float o[3], inv[3];
    float m;      // absolute dilation of this frame (frame_margin)
    float dscale; // 1: the derived margins; 0: none (tests only: show that they are needed)
};
__host__ __device__ __forceinline__ RayBox make_ray(const float o[3], const float d[3], float m, float dscale) {
    RayBox r;
    for (int c = 0; c < 3; ++c) r.o[c] = o[c], r.inv[c] = fdiv(1.f, d[c]); // d_c = +-0: inv = +-inf
    r.m = m * dscale, r.dscale = dscale;
    return r;
}
// the parameter bound of a child: t_ref (1 + C_REL sigma) + C_ABS sigma Lo  (see above; FLT_MAX -> inf: no bound)
__host__ __device__ __forceinline__ float t_upper(float t_ref, float sig, float lo_term) {
    return fadd(fmul(t_ref, fadd(1.f, fmul(C_REL * SAFE, sig))), fmul(C_ABS * SAFE, lo_term));
}
// Does the exact line o + s d meet the child's box dilated by m + C_LAT sigma Lo for some s in
// [-C_ABS sigma Lo, t_upper(t_ref)]?  Returns the (widened) entry in `entry` and sigma * Lo in `sl` (to re-check on pop).
__host__ __device__ __forceinline__ bool child_test(const RayBox &r, const float4 &lo, const float4 &hi, float t_ref, float &entry,
                                                    float &sl) {
    float Lo = 0.f;
    for (int c = 0; c < 3; ++c) {
        const float bl = c == 0 ? lo.x : (c == 1 ? lo.y : lo.z), bh = c == 0 ? hi.x : (c == 1 ? hi.y : hi.z);
        Lo = fadd(Lo, fmaxf(fabsf(fsub(r.o[c], bl)), fabsf(fsub(r.o[c], bh))));
    }
    Lo = fminf(fmul(Lo, SAFE), FLT_MAX); // finite, so that sigma = 0 gives 0, never 0 * inf
    sl = fmul(fmul(lo.w, r.dscale), Lo);
    const float D = fadd(r.m, fmul(C_LAT * SAFE, sl));
    float n = fmul(-C_ABS * SAFE, sl), f = t_upper(t_ref, fmul(lo.w, r.dscale), sl);
    for (int c = 0; c < 3; ++c) {
        const float bl = c == 0 ? lo.x : (c == 1 ? lo.y : lo.z), bh = c == 0 ? hi.x : (c == 1 ? hi.y : hi.z);
        const float x0 = fmul(fsub(fsub(bl, D), r.o[c]), r.inv[c]);
        const float x1 = fmul(fsub(fadd(bh, D), r.o[c]), r.inv[c]);
        float cn = fminf(x0, x1), cf = fmaxf(x0, x1);
        // NaN only from 0 * inf: d_c = 0 with o_c exactly on a dilated plane, so the line lies in the closed slab for
        // every s.  (fminf / fmaxf would return the other operand, +-inf, and could reject the box.)
        if (x0 != x0 || x1 != x1) cn = -INFINITY, cf = INFINITY;
        cn = fmul(cn, cn > 0.f ? 1.f - WIDEN : 1.f + WIDEN);
        cf = fmul(cf, cf > 0.f ? 1.f + WIDEN : 1.f - WIDEN);
        n = fmaxf(n, cn), f = fminf(f, cf);
    }
    entry = n;
    return n <= f;
}

constexpr int STACK = 64; // the tree's depth is at most 64: every level below the root adds a bit to a 64-bit key prefix

// Closest hit.  key: in/out t bits << 32 | index (KEY_NONE: none yet).  test(tri) runs the strict test of one triangle
// with t = FLT_MAX and returns its key or KEY_NONE.  The nearer child goes first; a popped child is re-checked against
// the t found meanwhile.
template <class Test>
__host__ __device__ __forceinline__ void closest(const Tree &tr, const RayBox &r, unsigned long long &key, Test test) {
    auto tref = [&]() { return key == KEY_NONE ? FLT_MAX : u2f((uint32_t)(key >> 32)); };
    auto leaf = [&](int tri) {
        const unsigned long long k = test(tri);
        if (k < key) key = k;
    };
    if (tr.n_in == 1) leaf(tr.root_leaf);
    if (tr.n_in >= 2) {
        int st_node[STACK];
        float st_entry[STACK], st_sig[STACK], st_sl[STACK];
        int sp = 0;
        int node = 0;
        for (;;) {
            const Node nd = load_node(tr.nodes + node);
            const float t_ref = tref();
            float e0, e1, s0, s1;
            const bool h0 = child_test(r, nd.lo0, nd.hi0, t_ref, e0, s0);
            const bool h1 = child_test(r, nd.lo1, nd.hi1, t_ref, e1, s1);
            int next = -1;
            // leaves are tested at once; of two internal children the nearer is visited next, the other pushed
            const bool first1 = h1 && (!h0 || e1 < e0);
            for (int q = 0; q < 2; ++q) {
                const int c = (q == 0) == first1 ? 1 : 0;
                if (!(c ? h1 : h0)) continue;
                const int ch = nd.child[c];
                if (ch < 0) {
                    leaf(~ch);
                } else if (next < 0) {
                    next = ch;
                } else {
                    st_node[sp] = ch, st_entry[sp] = c ? e1 : e0, st_sig[sp] = c ? nd.lo1.w : nd.lo0.w, st_sl[sp] = c ? s1 : s0;
                    ++sp;
                }
            }
            if (next >= 0) {
                node = next;
                continue;
            }
            node = -1;
            while (sp > 0) {
                --sp;
                if (st_entry[sp] <= t_upper(tref(), fmul(st_sig[sp], r.dscale), st_sl[sp])) {
                    node = st_node[sp];
                    break;
                }
            }
            if (node < 0) break;
        }
    }
    for (int i = 0; i < tr.n_always; ++i) leaf((int)(uint32_t)(tr.always[i] & 0xffffffffull));
}

// First occluder in index order: the lowest index the strict test accepts with the ray's own t_ray.  test(tri) -> t2 bits
// or -1 (rejected).  Children whose smallest index is >= the best index found are pruned; the child with the lower
// smallest index goes first.  Returns index << 32 | t2 bits, or KEY_NONE.
template <class Test>
__host__ __device__ __forceinline__ unsigned long long occluder(const Tree &tr, const RayBox &r, float t_ray, Test test) {
    int best = 0x7fffffff;
    uint32_t best_t = 0;
    auto leaf = [&](int tri) {
        if (tri >= best) return;
        const long long t2 = test(tri);
        if (t2 >= 0) best = tri, best_t = (uint32_t)t2;
    };
    if (tr.n_in == 1) leaf(tr.root_leaf);
    if (tr.n_in >= 2) {
        int st_node[STACK], st_mn[STACK];
        int sp = 0;
        int node = 0;
        for (;;) {
            const Node nd = load_node(tr.nodes + node);
            float e, s;
            const bool h0 = nd.mn[0] < best && child_test(r, nd.lo0, nd.hi0, t_ray, e, s);
            const bool h1 = nd.mn[1] < best && child_test(r, nd.lo1, nd.hi1, t_ray, e, s);
            const bool first1 = h1 && (!h0 || nd.mn[1] < nd.mn[0]);
            int next = -1;
            for (int q = 0; q < 2; ++q) {
                const int c = (q == 0) == first1 ? 1 : 0;
                if (!(c ? h1 : h0) || nd.mn[c] >= best) continue;
                const int ch = nd.child[c];
                if (ch < 0) {
                    leaf(~ch);
                } else if (next < 0) {
                    next = ch;
                } else {
                    st_node[sp] = ch, st_mn[sp] = nd.mn[c];
                    ++sp;
                }
            }
            if (next >= 0) {
                node = next;
                continue;
            }
            node = -1;
            while (sp > 0) {
                --sp;
                if (st_mn[sp] < best) {
                    node = st_node[sp];
                    break;
                }
            }
            if (node < 0) break;
        }
    }
    for (int i = 0; i < tr.n_always; ++i) leaf((int)(uint32_t)(tr.always[i] & 0xffffffffull));
    return best == 0x7fffffff ? KEY_NONE : ((unsigned long long)(uint32_t)best << 32) | best_t;
}

}  // namespace bvh

#ifdef __CUDACC__
#include "kernels.cuh"

namespace bvh {

// ---- device build ------------------------------------------------------------------------------------------------
struct BuildHdr {
    uint32_t cb[6]; // centres' box of the tree's triangles, ord() bits: min x y z, max x y z
    uint32_t bb[6]; // boxes' union, same encoding
    int n_in;
};

__global__ void prep_kernel(const float *__restrict__ verts, int n, float4 *__restrict__ tlo, float4 *__restrict__ thi,
                            BuildHdr *hdr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t mn[6], mx[6];
    for (int c = 0; c < 6; ++c) mn[c] = 0xffffffffu, mx[c] = 0u;
    bool in = false;
    if (i < n) {
        const TriInfo ti = tri_info(verts + 9 * (size_t)i);
        in = ti.in_tree;
        tlo[i] = make_float4(ti.lo[0], ti.lo[1], ti.lo[2], ti.sigma);
        thi[i] = make_float4(ti.hi[0], ti.hi[1], ti.hi[2], in ? 1.f : 0.f);
        if (in)
            for (int c = 0; c < 3; ++c) {
                mn[c] = mx[c] = ord(ti.c[c]);
                mn[3 + c] = ord(ti.lo[c]), mx[3 + c] = ord(ti.hi[c]);
            }
    }
    for (int c = 0; c < 6; ++c)
        for (int o = 16; o; o >>= 1) {
            mn[c] = min(mn[c], __shfl_down_sync(0xffffffffu, mn[c], o));
            mx[c] = max(mx[c], __shfl_down_sync(0xffffffffu, mx[c], o));
        }
    const unsigned cnt = __popc(__ballot_sync(0xffffffffu, in));
    if ((threadIdx.x & 31) == 0 && cnt) {
        for (int c = 0; c < 3; ++c) {
            atomicMin(&hdr->cb[c], mn[c]), atomicMax(&hdr->cb[3 + c], mx[c]);
            atomicMin(&hdr->bb[c], mn[3 + c]), atomicMax(&hdr->bb[3 + c], mx[3 + c]);
        }
        atomicAdd(&hdr->n_in, (int)cnt);
    }
}

__global__ void key_kernel(const float4 *__restrict__ tlo, const float4 *__restrict__ thi, int n, const BuildHdr *hdr,
                           unsigned long long *__restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 l = tlo[i], h = thi[i];
    if (h.w == 0.f) {
        keys[i] = KEY_ALWAYS | (uint32_t)i;
        return;
    }
    float clo[3], chi[3], c[3] = {fmul(0.5f, fadd(l.x, h.x)), fmul(0.5f, fadd(l.y, h.y)), fmul(0.5f, fadd(l.z, h.z))};
    for (int a = 0; a < 3; ++a) clo[a] = unord(hdr->cb[a]), chi[a] = unord(hdr->cb[3 + a]);
    keys[i] = ((unsigned long long)morton(c, clo, chi) << 32) | (uint32_t)i;
}

__global__ void nodes_kernel(const unsigned long long *__restrict__ keys, int n_in, Node *__restrict__ nodes, int *__restrict__ parent,
                             int *__restrict__ leaf_parent, int *__restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_in - 1) return;
    int l, r, split;
    bool ll, rl;
    karras_node(keys, n_in, i, l, r, ll, rl, split);
    nodes[i].child[0] = l, nodes[i].child[1] = r;
    if (ll) leaf_parent[split] = i;
    else parent[split] = i;
    if (rl) leaf_parent[split + 1] = i;
    else parent[split + 1] = i;
    flags[i] = 0;
    if (i == 0) parent[0] = -1;
}

// bottom-up: one thread per leaf; at every node the second arrival fills in both children (the first has published its
// child before its atomic, behind a fence; the second reads past L1)
__global__ void refit_kernel(const unsigned long long *__restrict__ keys, int n_in, const float4 *__restrict__ tlo,
                             const float4 *__restrict__ thi, Node *nodes, const int *__restrict__ parent,
                             const int *__restrict__ leaf_parent, int *flags) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_in) return;
    int node = leaf_parent[p];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&flags[node], 1) == 0) return;
        __threadfence();
        Node &nd = nodes[node];
        const int ch[2] = {__ldcg(&nd.child[0]), __ldcg(&nd.child[1])};
        float4 lo[2], hi[2];
        int mn[2];
        for (int c = 0; c < 2; ++c) {
            if (ch[c] < 0) {
                const int t = ~ch[c];
                lo[c] = tlo[t], hi[c] = thi[t], mn[c] = t;
                hi[c].w = 0.f;
            } else {
                const float4 *q = reinterpret_cast<const float4 *>(nodes + ch[c]);
                Node cn;
                cn.lo0 = __ldcg(q), cn.hi0 = __ldcg(q + 1), cn.lo1 = __ldcg(q + 2), cn.hi1 = __ldcg(q + 3);
                cn.mn[0] = __ldcg(&nodes[ch[c]].mn[0]), cn.mn[1] = __ldcg(&nodes[ch[c]].mn[1]);
                merge(cn, lo[c], hi[c], mn[c]);
            }
        }
        nd.lo0 = lo[0], nd.hi0 = hi[0], nd.lo1 = lo[1], nd.hi1 = hi[1];
        nd.mn[0] = mn[0], nd.mn[1] = mn[1];
        node = parent[node];
    }
}

// ---- render kernels ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void count_tests(sweep::Counters *ctr, unsigned long long *slot, unsigned n) {
    for (int o = 16; o; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0 && n) {
        atomicAdd(slot, (unsigned long long)n);
        atomicAdd(&ctr->strict_evals, (unsigned long long)n);
    }
}

// closest hit, one thread per primary ray (direction exactly as the sweeps' candidate path builds it, bands and jitter
// included): the merged key the sweeps leave in best[], for resolve_primary_kernel
__global__ void __launch_bounds__(128) primary_kernel(const trk::Views views, const trk::Bands bands, const Tree tr, float m,
                                                      const float *__restrict__ tri_verts, unsigned long long *__restrict__ best,
                                                      sweep::Counters *ctr) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned tests = 0;
    if (k < bands.n_px) {
        int w, h, local;
        const trk::Cam &cam = views.cams[views.split(k, local)];
        bands.map(local, w, h);
        const strict::f3 d = trk::primary_dir(cam, bands, w, h), o = strict::ld(cam.o);
        const float df[3] = {d.x, d.y, d.z};
        const RayBox r = make_ray(cam.o, df, m, 1.f);
        unsigned long long key = KEY_NONE;
        closest(tr, r, key, [&](int tri) -> unsigned long long {
            ++tests;
            const float *q = tri_verts + 9 * (size_t)tri;
            float t = FLT_MAX, v = 0.f; // main.cpp:715-717
            if (strict::intersect_triangle(o, d, strict::mk(__ldg(q), __ldg(q + 1), __ldg(q + 2)), strict::mk(__ldg(q + 3), __ldg(q + 4), __ldg(q + 5)),
                                           strict::mk(__ldg(q + 6), __ldg(q + 7), __ldg(q + 8)), t, v))
                return ((unsigned long long)__float_as_uint(t) << 32) | (unsigned)tri;
            return KEY_NONE;
        });
        best[k] = key;
    }
    count_tests(ctr, &ctr->tests_primary, tests);
}

// first occluder, one thread per pixel with a shadow ray (px.rj >= 0; origin, direction and length as light_step_kernel
// left them); rays without a triangle occluder then run the spheres as shadow_spheres_kernel does.  Writes every
// pixel's best_occ (KEY_NONE: none, or no shadow ray).
__global__ void __launch_bounds__(128) shadow_kernel(const Tree tr, const trk::PixelState px, int n_px, float m,
                                                     const float *__restrict__ tri_verts, const float4 *__restrict__ spheres,
                                                     int n_spheres, int n_tris, sweep::Counters *ctr) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned tests = 0;
    if (k < n_px) {
        unsigned long long key = KEY_NONE;
        if (px.rj[k] >= 0) {
            const size_t n = (size_t)n_px;
            const float of[3] = {px.ro[k], px.ro[n + k], px.ro[2 * n + k]}, df[3] = {px.rd[k], px.rd[n + k], px.rd[2 * n + k]};
            const strict::f3 o = strict::ld(of), d = strict::ld(df);
            const float t_ray = px.rt[k];
            key = occluder(tr, make_ray(of, df, m, 1.f), t_ray, [&](int tri) -> long long {
                ++tests;
                const float *q = tri_verts + 9 * (size_t)tri;
                float t = t_ray, v = 0.f; // the ray has no occluder yet: t is its initial length (main.cpp:764)
                if (strict::intersect_triangle(o, d, strict::mk(__ldg(q), __ldg(q + 1), __ldg(q + 2)), strict::mk(__ldg(q + 3), __ldg(q + 4), __ldg(q + 5)),
                                               strict::mk(__ldg(q + 6), __ldg(q + 7), __ldg(q + 8)), t, v))
                    return (long long)__float_as_uint(t);
                return -1;
            });
            if (key == KEY_NONE && n_spheres > 0) key = trk::sphere_occluder(o, d, t_ray, spheres, n_spheres, n_tris);
        }
        px.best_occ[k] = key;
    }
    count_tests(ctr, &ctr->tests_shadow, tests);
}

}  // namespace bvh
#endif
