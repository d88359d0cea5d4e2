// kernels.cuh — device kernels of the render path (see sweep.cuh for the sweeps).
//
//   build_origin_table   per (point O, triangle): the 32-byte span row and the 48-byte three-row filter row
//   primary_kernel       raygen (camera.h:31-34) + closest hit (main.cpp:176-192)
//   light_step_kernel    per pixel, per light: finish light k-1 (main.cpp:772-788),
//                        set up the shadow ray of light k (main.cpp:740-770)
//   list_prefix / list_scatter   group shadow rays by light vertex
//   shadow_kernel        first in-order occluder (main.cpp:314-329)
//   quantise_kernel      clamp + int(x*255) -> packed u8 RGB (main.cpp:679-684)
//   assemble_bands_kernel  rank 0: band-packed rank buffers -> one frame
#pragma once
#include "cull.cuh"
#include "sweep.cuh"

namespace trk {

using strict::f3;

struct Cam {
    float o[3], llc[3], hor[3], ver[3];
};

// local pixel k (row-major over the PPM rows this rank renders) -> (w, h)
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

struct Bands {
    int W, H, band_rows, band_index, band_count, n_px;
    // extension (parity unpinned): spp_n x spp_n stratified jitter; sample = 0 .. spp_n^2-1
    int spp_n, sample;
    uint32_t seed;
    // image-plane parameters of pixel (w,h): the reference's s = w/(W-1), t = h/(H-1) (main.cpp:709-710);
    // with jitter, w and h are displaced inside the pixel's stratum first.  Strict arithmetic: the
    // restatement (oracle/restated.c:pixel_st) computes the same bits.
    __device__ __forceinline__ void pixel_st(int w, int h, float &s, float &t) const {
        float fw = (float)w, fh = (float)h;
        if (spp_n > 1) {
            const uint32_t h1 = mix32(mix32((seed ^ 0x51ed270bu) + (uint32_t)(h * W + w)) ^ ((uint32_t)sample * 0x9e3779b1u + 0x7f4a7c15u));
            const uint32_t h2 = mix32(h1 + 0x632be5abu);
            const float u1 = __fmul_rn((float)(h1 >> 8), 5.9604644775390625e-08f);
            const float u2 = __fmul_rn((float)(h2 >> 8), 5.9604644775390625e-08f);
            const float jx = __fdiv_rn(__fadd_rn((float)(sample % spp_n), u1), (float)spp_n);
            const float jy = __fdiv_rn(__fadd_rn((float)(sample / spp_n), u2), (float)spp_n);
            fw = __fadd_rn(fw, __fsub_rn(jx, 0.5f));
            fh = __fadd_rn(fh, __fsub_rn(jy, 0.5f));
        }
        s = __fdiv_rn(fw, (float)(W - 1));
        t = __fdiv_rn(fh, (float)(H - 1));
    }
    __host__ __device__ __forceinline__ void map(int k, int &w, int &h) const {
        const int lr = k / W;
        w = k - lr * W;
        int pr = lr;
        if (band_count > 1) {
            const int lb = lr / band_rows;
            pr = (band_index + lb * band_count) * band_rows + (lr - lb * band_rows);
        }
        h = H - 1 - pr; // PPM row 0 is h = H-1 (main.cpp:662)
    }
};

// main.cpp:709-710 + camera.h:31-34, strict
__device__ __forceinline__ f3 primary_dir(const Cam &c, const Bands &b, int w, int h) {
    float s, tt;
    b.pixel_st(w, h, s, tt);
    const f3 o = strict::ld(c.o), llc = strict::ld(c.llc), hor = strict::ld(c.hor), ver = strict::ld(c.ver);
    return strict::normalize(strict::sub(strict::add(strict::add(llc, strict::mul(hor, s)), strict::mul(ver, tt)), o));
}

// ---------------------------------------------------------------------------------
// Filter rows for lines through O (see sweep.cuh).  Computed in FP64 from the float
// vertices, rounded once.  lmax bounds the length of any ray segment that will be
// swept against this table (0 for the eye table: rays start AT O).
//
// Margin: the reference evaluates u' (etc.) as float dot/cross products of
// tvec = orig - v0, dir, edges: absolute error <= ~8 eps |tvec||dir||edge|, with
// |tvec| <= lmax + |a|.  Our own evaluation adds <= ~4 eps |a||edge|, and the
// shadow ray's float direction misses O by <= ~3 eps len.  All are bounded by
// K = CK eps * max|edge| * (lmax + |a| + |b| + |c|) with CK = 64.
// If O is within the same noise of the triangle's plane the side s is undefined
// (e.g. a light vertex against its own light's faces): the row is made
// "always candidate" and the pair is always decided by the strict path.
//
// Direction parametrisation of the ray group this table serves: d' = p*U + q*V + W with
// |d'| <= dmax.  A 3-D row (vec, K) valid for unit directions becomes the affine 2-D row
// (U.vec, V.vec, W.vec + K*dmax): d'.vec + K|d'| >= 0 is relaxed to d'.vec + K*dmax >= 0.
//
// SATURATING FORM.  The sweeps decide "all three rows >= 0" in the FMA pipe: each row value is
// clamped to [0,1] by the FFMA itself (fma.sat) and the three are multiplied, so a pair is a
// candidate iff the product is exactly 1.  For that every row carries a SECOND margin K2 (equal to the
// first one, K*dmax, for edge rows) and is scaled by a power of two S with S * 0.9 * K2 >= 1: a pair the
// reference could accept evaluates to >= 0 without K2, hence to >= K2 less a few ulps with it,
// hence to >= 1 after the (exact, power-of-two) scaling — it saturates to exactly 1 on all three
// rows.  Sign tests on the scaled rows (bundle-cull mode) remain valid: they are only looser.
struct TableParam {
    double o[3], U[3], V[3], W[3], dmax, lmax;
};

// K: the margin for unit directions; K2u: the second margin (same units); returns the scaled float row
// row3: the same row before the second margin and the scaling, in FP64: a pair the reference could accept satisfies
// p*row3[0] + q*row3[1] + row3[2] >= 0 in exact arithmetic (input of the span rows, span_rows below)
__host__ __device__ __forceinline__ float4 project_row(const TableParam &tp, double vx, double vy, double vz, double K, double K2u, double *row3) {
    const double A = tp.U[0] * vx + tp.U[1] * vy + tp.U[2] * vz;
    const double B = tp.V[0] * vx + tp.V[1] * vy + tp.V[2] * vz;
    const double K1 = K2u * tp.dmax;
    const double C0 = tp.W[0] * vx + tp.W[1] * vy + tp.W[2] * vz + K * tp.dmax * 1.0001; // first margin
    row3[0] = A, row3[1] = B, row3[2] = C0;
    const double C = C0 + K1; // + K2
    // S = 2^k >= 1 / (0.9 K2).  |row| / K2 is bounded by ~1/(8 eps) by construction, so the scaled row stays far inside
    // the float range; should that ever fail (or K2 be 0) the row becomes "always candidate": the strict path decides.
    const double mag = fmax(fabs(A), fmax(fabs(B), fabs(C)));
    if (!(K1 > 0.0) || !(mag < 1e30)) return make_float4(0.f, 0.f, 1.f, 0.f);
    const int k = (int)ceil(-log2(0.9 * K1));
    if (k > 100 || k < -100 || k + (int)ceil(log2(mag)) > 100) return make_float4(0.f, 0.f, 1.f, 0.f);
    // (float)x * 2^k is exact at these magnitudes, so the scaled row is the float row times S and its evaluation is
    // S times the unscaled evaluation, bit for bit
    const float Sf = (float)exp2((double)k);
    return make_float4((float)A * Sf, (float)B * Sf, (float)C * Sf, 0.f);
}

// SPAN rows (sweep.cuh, 4.): the three exact rows  p*A_i + q*B_i + C_i >= 0  as two lower and two upper bounds of p.
//   A_i > 0:  p >= q*beta + gamma     A_i < 0:  p <= q*beta + gamma      beta = -B_i/A_i, gamma = -C_i/A_i
// stored in row units with the +1 of the saturating test:  lower (-S*beta, 1 - S*gamma + M),  upper (S*beta, 1 + S*gamma + M).
// M covers the float evaluation of the bound (coefficients rounded to float, one or two FFMA roundings, |q| <= QMAX):
// M = 8 eps (QMAX S|beta| + S|gamma| + 1), so that a pair satisfying the exact row reaches >= 1 and saturates to exactly 1.
// A row whose A is tiny against its other terms (|A| < 1e-9 (PMAX|A| + QMAX|B| + |C|)) barely depends on p: it is replaced
// by (A', B, C + PMAX(|A'| + |A|)) with |A'| = that threshold, which is weaker for every |p| <= PMAX, and may take either
// sign, i.e. fill a lower or an upper slot.  Three bounds on the same side (a triangle whose cone reaches around the
// parametrisation plane: only for triangles that span tens of degrees as seen from O) keep the two that lose the least
// area of the (p,q) box; dropping a bound only loosens the filter.  Rows that are not finite make the triangle "always
// candidate" (the strict path decides).
constexpr double SPAN_PMAX = 1.0625, SPAN_QMAX = 1.0625; // |p|, |q| of every ray swept in span form (image plane: [0,1]; cube faces: [-1,1])

struct SpanBound {
    double beta, gamma;
};
__host__ __device__ __forceinline__ void span_rows(const double (&rows)[3][3], float4 &lo, float4 &hi) {
    const double S = (double)sweep::SPAN_S, eps = (double)TRC_EPS;
    const float OPEN = sweep::SPAN_OPEN;
    lo = make_float4(0.f, OPEN, 0.f, OPEN), hi = make_float4(0.f, OPEN, 0.f, OPEN); // no bound at all: always candidate
    SpanBound L[3], U[3];
    int nl = 0, nu = 0;
    double flexB[3], flexC[3], flexA[3]; // rows that barely depend on p: B, widened C, |A'|
    int nf = 0;
    for (int i = 0; i < 3; ++i) {
        const double A = rows[i][0], B = rows[i][1], C = rows[i][2];
        const double mag = SPAN_PMAX * fabs(A) + SPAN_QMAX * fabs(B) + fabs(C);
        if (!(mag < 1e30)) return;  // inf / NaN: always candidate
        if (mag == 0.0) continue;   // 0 >= 0: no bound
        const double amin = 1e-9 * mag;
        if (fabs(A) < amin) {
            flexA[nf] = amin, flexB[nf] = B, flexC[nf] = C + SPAN_PMAX * (amin + fabs(A)), ++nf;
        } else if (A > 0.0) {
            L[nl].beta = -B / A, L[nl].gamma = -C / A, ++nl;
        } else {
            U[nu].beta = -B / A, U[nu].gamma = -C / A, ++nu;
        }
    }
    for (int i = 0; i < nf; ++i) { // A' = +|A'| is a lower bound, A' = -|A'| an upper one: take the side with room
        if (nl <= nu) L[nl].beta = -flexB[i] / flexA[i], L[nl].gamma = -flexC[i] / flexA[i], ++nl;
        else U[nu].beta = flexB[i] / flexA[i], U[nu].gamma = flexC[i] / flexA[i], ++nu;
    }
    // three bounds on one side: drop the one whose removal adds the least area inside the box (sampled in q)
    auto drop_one = [&](SpanBound *b, int &n, bool lower) {
        if (n < 3) return;
        double loss[3] = {0, 0, 0};
        for (int sidx = 0; sidx < 17; ++sidx) {
            const double q = -SPAN_QMAX + 2.0 * SPAN_QMAX * sidx / 16.0;
            double c[3];
            for (int i = 0; i < 3; ++i) c[i] = fmin(SPAN_PMAX, fmax(-SPAN_PMAX, q * b[i].beta + b[i].gamma));
            for (int j = 0; j < 3; ++j) {
                const double o1 = c[(j + 1) % 3], o2 = c[(j + 2) % 3];
                if (lower) loss[j] += fmax(0.0, c[j] - fmax(o1, o2)); // lower bounds: the binding one is the maximum
                else loss[j] += fmax(0.0, fmin(o1, o2) - c[j]);
            }
        }
        int j = 0;
        if (loss[1] < loss[j]) j = 1;
        if (loss[2] < loss[j]) j = 2;
        b[j] = b[2];
        n = 2;
    };
    drop_one(L, nl, true), drop_one(U, nu, false);
    float *lof = &lo.x, *hif = &hi.x;
    for (int i = 0; i < nl; ++i) {
        const double M = 8.0 * eps * (SPAN_QMAX * S * fabs(L[i].beta) + S * fabs(L[i].gamma) + 1.0);
        const double b = -S * L[i].beta, c = 1.0 - S * L[i].gamma + M;
        if (!(fabs(b) < 1e30) || !(fabs(c) < 1e30)) continue; // cannot be represented: leave the bound open
        lof[2 * i] = (float)b, lof[2 * i + 1] = (float)c;
    }
    for (int i = 0; i < nu; ++i) {
        const double M = 8.0 * eps * (SPAN_QMAX * S * fabs(U[i].beta) + S * fabs(U[i].gamma) + 1.0);
        const double b = S * U[i].beta, c = 1.0 + S * U[i].gamma + M;
        if (!(fabs(b) < 1e30) || !(fabs(c) < 1e30)) continue;
        hif[2 * i] = (float)b, hif[2 * i + 1] = (float)c;
    }
}

// The filter rows of ONE triangle (p: its 9 vertex floats) for the origin / parametrisation tp: the 48-byte three-row form
// (rb, rc, rd) and, if want_span, the 32-byte span row (slo, shi).  Host-callable: tests/test_filter_rows.py checks the
// construction on the CPU against the reference's own intersection test (tracer__origin_rows in tracer_cuda.cu).
__host__ __device__ __forceinline__ void origin_rows(const float *__restrict__ p, const TableParam &tp, bool want_span, float4 &rb,
                                                     float4 &rc, float4 &rd, float4 &slo, float4 &shi) {
    const double ox = tp.o[0], oy = tp.o[1], oz = tp.o[2], lmax = tp.lmax;
    double rows[3][3] = {{0, 0, 1}, {0, 0, 1}, {0, 0, 1}}; // exact rows behind rb, rc, rd (always true unless set)
    const double v0x = p[0], v0y = p[1], v0z = p[2];
    const double e1x = (double)p[3] - v0x, e1y = (double)p[4] - v0y, e1z = (double)p[5] - v0z;
    const double e2x = (double)p[6] - v0x, e2y = (double)p[7] - v0y, e2z = (double)p[8] - v0z;
    const double ax = v0x - ox, ay = v0y - oy, az = v0z - oz;
    // B = a x e2, C = e1 x a, Nn = e2 x e1, D = Nn - B - C
    const double Bx = ay * e2z - az * e2y, By = az * e2x - ax * e2z, Bz = ax * e2y - ay * e2x;
    const double Cx = e1y * az - e1z * ay, Cy = e1z * ax - e1x * az, Cz = e1x * ay - e1y * ax;
    const double Nx = e2y * e1z - e2z * e1y, Ny = e2z * e1x - e2x * e1z, Nz = e2x * e1y - e2y * e1x;
    const double Dx = Nx - Bx - Cx, Dy = Ny - By - Cy, Dz = Nz - Bz - Cz;
    const double tprime = e2x * Cx + e2y * Cy + e2z * Cz; // e2 . (tvec x e1), tvec = -a
    const double la = sqrt(ax * ax + ay * ay + az * az);
    const double lb = sqrt((ax + e1x) * (ax + e1x) + (ay + e1y) * (ay + e1y) + (az + e1z) * (az + e1z));
    const double lc = sqrt((ax + e2x) * (ax + e2x) + (ay + e2y) * (ay + e2y) + (az + e2z) * (az + e2z));
    const double l1 = sqrt(e1x * e1x + e1y * e1y + e1z * e1z), l2 = sqrt(e2x * e2x + e2y * e2y + e2z * e2z);
    const double l3 = sqrt((e2x - e1x) * (e2x - e1x) + (e2y - e1y) * (e2y - e1y) + (e2z - e1z) * (e2z - e1z));
    const double emax = fmax(l1, fmax(l2, l3));
    const double reach = lmax + la + lb + lc;
    const double eps = (double)TRC_EPS;
    const double K = (double)sweep::CK * eps * emax * reach;
    const double tau = (double)sweep::CK * eps * l1 * l2 * reach;
    if (!(fabs(tprime) > tau)) {
        // O lies within the noise of the triangle's plane: the side s is undefined.  A line through
        // O can then only reach the (noise-dilated) triangle if it runs almost inside that plane:
        // |d.n| <= (h + delta) / (rho - delta), with h the distance of O from the plane, rho a lower
        // bound of the distance from O to the triangle and delta the positional noise scaled by the
        // triangle's aspect.  Two of the three rows encode that slab (+n and -n), the third is
        // always true.  When O is (nearly) ON the triangle — a light vertex against its own light's
        // faces — the slab degenerates and the row is "always candidate": the strict path decides.
        rb = rc = rd = make_float4(0.f, 0.f, 1.f, 0.f);
        const double area2 = sqrt(Nx * Nx + Ny * Ny + Nz * Nz);
        if (area2 > 0.0 && emax > 0.0) {
            const double shape = emax * emax / area2;
            const double delta = 4.0 * (double)sweep::CK * eps * reach * shape;
            const double rho = fmax(la, fmax(lb, lc)) - emax;
            const double h = fabs(tprime) / area2;
            if (rho > 4.0 * delta) {
                const double kappa = (h + delta) / (rho - delta) * 1.01 + 8.0 * eps;
                if (kappa < 1.0) {
                    // second margin: a fraction of the slab's own width, never below the evaluation noise of a unit row
                    const double k2 = fmax(kappa / 8.0, 16.0 * eps);
                    rb = project_row(tp, Nx / area2, Ny / area2, Nz / area2, kappa * 1.0000002 + 1e-37, k2, rows[0]);
                    rc = project_row(tp, -Nx / area2, -Ny / area2, -Nz / area2, kappa * 1.0000002 + 1e-37, k2, rows[1]);
                }
            }
        }
    } else {
        const double s = tprime > 0 ? 1.0 : -1.0;
        // round K up a little so the float row never under-states it
        const double Kd = K * 1.0000002 + 1e-37;
        rb = project_row(tp, s * Bx, s * By, s * Bz, Kd, Kd, rows[0]);
        rc = project_row(tp, s * Cx, s * Cy, s * Cz, Kd, Kd, rows[1]);
        rd = project_row(tp, s * Dx, s * Dy, s * Dz, Kd, Kd, rows[2]);
    }
    // rb.w (bundle-cull mode only): a lower bound of the distance from O to any point X of the triangle,
    // |X - O| >= |V - O| - |X - V| >= max(la, lb, lc) - emax, less a slack far above the float noise of the
    // reference's own t2.  A shadow ray that ends at O and is shorter than this cannot hit the triangle.
    if (lmax > 0.0) rb.w = (float)fmax(0.0, (fmax(la, fmax(lb, lc)) - emax - 1e-4 * reach) * 0.999999);
    if (want_span) span_rows(rows, slo, shi);
}

// table: the 48-byte three-row table (MODE_OWNQ sweeps, bundle-cull mode) or null; span: the 32-byte span table or null
__global__ void build_origin_table(const float *__restrict__ tri_verts, int n_tris, int n_pad, const TableParam tp,
                                   float4 *__restrict__ table, float4 *__restrict__ span) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    float4 rb, rc, rd, slo, shi;
    if (i >= n_tris) { // padding rows: never candidate
        rb = rc = rd = make_float4(0.f, 0.f, -1.f, 0.f);
        slo = make_float4(0.f, -sweep::SPAN_OPEN, 0.f, -sweep::SPAN_OPEN), shi = make_float4(0.f, sweep::SPAN_OPEN, 0.f, sweep::SPAN_OPEN);
    } else {
        origin_rows(tri_verts + 9 * (size_t)i, tp, span != nullptr, rb, rc, rd, slo, shi);
    }
    if (table) {
        table[3 * (size_t)i] = rb;
        table[3 * (size_t)i + 1] = rc;
        table[3 * (size_t)i + 2] = rd;
    }
    if (span) {
        span[2 * (size_t)i] = slo;
        span[2 * (size_t)i + 1] = shi;
    }
}

// every row a candidate: the group of rays whose assumptions failed (never observed in practice)
__global__ void build_allcand_table(int n_tris, int n_pad, float4 *__restrict__ table, float4 *__restrict__ span) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    const float4 r = make_float4(0.f, 0.f, i < n_tris ? 1.f : -1.f, 0.f);
    table[3 * (size_t)i] = table[3 * (size_t)i + 1] = table[3 * (size_t)i + 2] = r;
    const float lo = i < n_tris ? sweep::SPAN_OPEN : -sweep::SPAN_OPEN;
    span[2 * (size_t)i] = make_float4(0.f, lo, 0.f, lo);
    span[2 * (size_t)i + 1] = make_float4(0.f, sweep::SPAN_OPEN, 0.f, sweep::SPAN_OPEN);
}

// ---------------------------------------------------------------------------------
// Work decomposition of the sweeps: (ray block) x (triangle slice).  Closest hit is the
// lexicographic minimum of (t, index) over all valid hits (ray_triangle.h:46-50: t2 >= t rejects,
// so among equal t the lowest index stays) and the first occluder is the minimum index over all
// valid hits, so triangle slices can be swept independently and merged with a 64-bit atomicMin:
//   closest hit  key = t bits << 32 | index      (t > 0: float order == unsigned order)
//   occluder     key = index << 32  | t2 bits
// Slicing gives enough work items for every SM on small frames, late shadow chunks and when the
// frame is split over several GPUs.
constexpr unsigned long long KEY_NONE = 0xffffffffffffffffull;

struct PrimaryParams {
    Cam cam;
    Bands bands;
    const float4 *table; // eye table: span rows (MODE_SHAREDQ, MODE_QBAR) or the three-row table (MODE_OWNQ)
    int n_tiles, n_tris;
    const float *tri_verts;
    unsigned long long *best; // [n_px] merged closest-hit keys over triangles, KEY_NONE = miss
    sweep::Counters *counters;
    int *work;
    int n_blocks, n_slices;
    int tiles_x, n_rows; // ray blocks are screen tiles of (TX*R) x (512/TX) pixels, TX = 1 << tx_log2: n_blocks = tiles_x * tiles_y
    int tx_log2;         // threads across a tile (the host picks the shape that wastes the fewest pixels at the frame's edges)
};

// The reference's own test for the rays (bits of mask) of one thread against triangle tri, eye rays
// (cpp_intersect, main.cpp:176-192).  Every accepted pair is merged into the pixel's closest-hit key; the
// lexicographic minimum of (t, index) over all accepted pairs is what the serial loop ends with (t2 >= t
// rejects, ray_triangle.h:49, so among equal t the lowest index stays), whatever the order of evaluation.
// k0: local pixel index of the thread's ray 0 (ray r = pixel k0 + r).  filt: rays the filter passed (validation).
// Returns evaluations | filter misses << 16.
__device__ __noinline__ unsigned strict_primary(const PrimaryParams &p, int k0, unsigned mask, int tri, unsigned filt) {
    const float *q = p.tri_verts + 9 * (size_t)tri;
    const f3 v0 = strict::mk(__ldg(q), __ldg(q + 1), __ldg(q + 2));
    const f3 v1 = strict::mk(__ldg(q + 3), __ldg(q + 4), __ldg(q + 5));
    const f3 v2 = strict::mk(__ldg(q + 6), __ldg(q + 7), __ldg(q + 8));
    const f3 o = strict::ld(p.cam.o);
    unsigned ret = 0;
    while (mask) {
        const int r = __ffs(mask) - 1;
        mask &= mask - 1;
        int w, h;
        p.bands.map(k0 + r, w, h);
        const f3 d = primary_dir(p.cam, p.bands, w, h);
        float t = FLT_MAX, v = 0.f; // main.cpp:715-717
        ++ret;
        if (strict::intersect_triangle(o, d, v0, v1, v2, t, v)) {
            atomicMin(&p.best[k0 + r], ((unsigned long long)__float_as_uint(t) << 32) | (unsigned)tri);
            if (!((filt >> r) & 1u)) ret += 1u << 16;
        }
    }
    return ret;
}

// Ray block = screen tile, each thread holding R horizontally consecutive pixels of ONE image row.  Without
// jitter those R rays share the filter parameter q exactly (MODE_SHAREDQ): the four bounds of a triangle's span row are
// evaluated once per thread and triangle.  With jittered samples (extension) the rays of a thread are the same sample
// of R pixels of one image row: their q lie inside one stratum, 1/(spp_n (H-1)) wide, and the bounds are evaluated at
// the thread's mean q plus |B| x spread (MODE_QBAR, as the shadow sweeps do); the candidate path uses each ray's own q.
// MODE_OWNQ (three-row table, every ray its own q) remains for frames too small for the span rows' |p|,|q| range.
template <int R, bool EXHAUSTIVE, int MODE>
__global__ void __launch_bounds__(sweep::NT, sweep::MINB) primary_kernel(const __grid_constant__ PrimaryParams p) {
    constexpr bool SHAREDQ = MODE == sweep::MODE_SHAREDQ;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using Smem = sweep::SmemT<sweep::Rows<MODE>::N>;
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    const int tid = threadIdx.x;
    sweep::smem_init(sm);
    unsigned gtile = 0, n_strict = 0, n_swept = 0, n_miss = 0, n_pipe_err = 0;
    unsigned long long tests = 0;
    const int n_items = p.n_blocks * p.n_slices;
    for (;;) {
        if (tid == 0) sm.blk = atomicAdd(p.work, 1);
        __syncthreads();
        const int item = sm.blk;
        if (item >= n_items) break;
        // slice-major order: all CTAs stream the same table tiles at about the same time (L2 reuse)
        const int slice = item / p.n_blocks, blk = item - slice * p.n_blocks;
        const int tile_lo = (int)((long long)p.n_tiles * slice / p.n_slices);
        const int tile_hi = (int)((long long)p.n_tiles * (slice + 1) / p.n_slices);
        const int W = p.bands.W;
        const int tile_y = blk / p.tiles_x, tile_x = blk - tile_y * p.tiles_x;
        const int txn = 1 << p.tx_log2;
        const int x0 = (tile_x * txn + (tid & (txn - 1))) * R, ly = tile_y * (sweep::NT >> p.tx_log2) + (tid >> p.tx_log2);
        float rp[R], rq[R];
        unsigned valid = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (x0 + r < W && ly < p.n_rows) valid |= 1u << r;
            int w, h;
            p.bands.map(min(ly, p.n_rows - 1) * W + min(x0 + r, W - 1), w, h);
            // filter parameters: the ray's own (s,t) on the image plane (main.cpp:709-710)
            p.bands.pixel_st(w, h, rp[r], rq[r]);
        }
        if (SHAREDQ) { // same image row, no jitter: every rq[r] holds the same bits; say so to the compiler
            const float q0 = rq[0];
#pragma unroll
            for (int r = 1; r < R; ++r) rq[r] = q0;
        }
        const int k0 = ly * W + x0; // valid rays are pixels k0 + r
        unsigned done = 0;
        float qbar = 0.f, qdelta = 0.f;
        if (MODE == sweep::MODE_QBAR) { // (rays past the frame's edge are duplicates of edge pixels: all R values count)
            float qmin = rq[0], qmax = rq[0];
#pragma unroll
            for (int r = 1; r < R; ++r) qmin = fminf(qmin, rq[r]), qmax = fmaxf(qmax, rq[r]);
            qbar = 0.5f * (qmin + qmax);
            // >= max |q_r - qbar| with room for the roundings of this line and of the one extra FFMA per bound
            qdelta = fmaxf(qmax - qbar, qbar - qmin) * 1.0001f + 2.4e-7f * (fabsf(qbar) + 1.f);
        }
        sweep::sweep_table<R, MODE, false, EXHAUSTIVE>(
            sm, p.table, tile_lo, tile_hi, p.n_tris, rp, rq, qbar, qdelta, valid, done, gtile, n_swept,
            [&](unsigned mask, int tri, unsigned filt) {
                const unsigned c = strict_primary(p, k0, mask, tri, filt);
                n_strict += c & 0xffffu, n_miss += c >> 16;
                return 0u;
            },
            &n_pipe_err);
        const int t_lo = min(tile_lo * sweep::TILE, p.n_tris), t_hi = min(tile_hi * sweep::TILE, p.n_tris);
        tests += (unsigned long long)__popc(valid) * (unsigned)(t_hi - t_lo);
        __syncthreads(); // sm.blk is rewritten by the next item
    }
    atomicAdd(&p.counters->tests_primary, tests);
    atomicAdd(&p.counters->strict_evals, (unsigned long long)n_strict);
    if (EXHAUSTIVE) atomicAdd(&p.counters->filter_misses, (unsigned long long)n_miss);
    if (EXHAUSTIVE && n_pipe_err) atomicAdd(&p.counters->pipeline_errors, (unsigned long long)n_pipe_err);
}

// ---------------------------------------------------------------------------------
constexpr int NFACE = 7; // ray groups per light vertex: 6 cube faces + 1 "all candidates"

struct LightInfo {              // device arrays describing the lights
    const int *light_vbase;     // [L+1] prefix sum of F_l: index of light l's first vertex/table
    const float *light_verts;   // [V*3] light.vertex[faceID] positions (main.cpp:749)
};

struct PixelState {
    const unsigned long long *best;     // [n_px] merged closest-hit keys from primary_kernel
    unsigned long long *best_occ;       // [n_px] merged first-occluder keys of the current light
    int *hit_tri;
    float *hit_t, *hit_v;
    float *carry_t;       // the `t` variable of scan_row across lights (main.cpp:715, 764, occlusion's t2)
    float *nrm;           // [3][n_px]
    float *accum;         // [3][n_px]
    float *ro, *rd;       // [3][n_px] shadow ray origin, strict unit dir
    float *re;            // [2][n_px] filter parameters (p,q) on the ray's cube face
    float *rt;            // [n_px] tmax of the current shadow ray
    int *rj;              // [n_px] ray group within the current light: faceID*NFACE + cube face, -1 none
};

// After the sliced closest-hit sweep: unpack the merged (t, index) key, recover v by one strict
// re-evaluation of the winning triangle (same arithmetic, same bits as in the sweep), then the
// extension: analytic spheres, tested after all triangles in object order with the running t.
__global__ void __launch_bounds__(256) resolve_primary_kernel(Cam cam, Bands bands, const unsigned long long *__restrict__ best,
                                                              const float *__restrict__ tri_verts, int n_tris,
                                                              const float4 *__restrict__ spheres, int n_spheres,
                                                              int *__restrict__ hit_tri, float *__restrict__ hit_t,
                                                              float *__restrict__ hit_v) {
    const int kpx = blockIdx.x * blockDim.x + threadIdx.x;
    if (kpx >= bands.n_px) return;
    const unsigned long long key = best[kpx];
    int tri = key == KEY_NONE ? -1 : (int)(unsigned)(key & 0xffffffffu);
    float t = FLT_MAX, v = 0.f; // main.cpp:715-717
    if (tri >= 0 || n_spheres > 0) {
        int w, h;
        bands.map(kpx, w, h);
        const f3 o = strict::ld(cam.o);
        const f3 d = primary_dir(cam, bands, w, h);
        if (tri >= 0) {
            const float *q = tri_verts + 9 * (size_t)tri;
            strict::intersect_triangle(o, d, strict::ld(q), strict::ld(q + 3), strict::ld(q + 6), t, v);
        }
        for (int s = 0; s < n_spheres; ++s)
            if (strict::intersect_sphere(o, d, __ldg(&spheres[s]), t)) tri = n_tris + s;
    }
    hit_tri[kpx] = tri, hit_t[kpx] = t, hit_v[kpx] = v;
}

struct LightStepParams {
    Cam cam;
    Bands bands;
    PixelState px;
    LightInfo li;
    int k, L, n_tris;
    const float *tri_verts, *tri_normals;
    const int *tri_geom, *geom_has_normals;
    const float *geom_material, *sphere_material;
    const float4 *spheres;
    int rng_mode;
    uint32_t seed;
    const int *faceid; // [n_px*L] local pixel order (explicit / mt19937 modes)
    double lmax;
    int *seg_count;    // [F_k] histogram of rays per light vertex
    sweep::Counters *counters;
    int *dbg_occ;      // [n_px*L] or null
    int cull_cells;    // also write a 64-bit sort key: 1 = group << 32 | Morton code of (p,q) (bundle-cull mode),
                       // 2 = group << 32 | order-preserving bits of q (default mode with shared q-terms)
    unsigned long long *rkey; // [n_px] sort keys (bundle-cull mode), all-ones for pixels without a shadow ray
};

// counter-based faceID: uniform in [0,F), keyed by (seed, image index, light)
__host__ __device__ __forceinline__ int hash_faceid(uint32_t seed, uint32_t image_index, uint32_t light, uint32_t F) {
    uint32_t h = mix32((seed ^ 0x9e3779b9u) + image_index);
    h = mix32(h ^ (light * 0x85ebca6bu + 0xc2b2ae35u));
    return (int)(((unsigned long long)h * F) >> 32);
}

__global__ void __launch_bounds__(256) light_step_kernel(const LightStepParams p) {
    const int kpx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = kpx < p.bands.n_px;
    int my_j = -1;
    unsigned long long ref_tests = 0, rkey_mine = KEY_NONE;
    unsigned n_hit = 0;
    if (in_range) {
        const int n = p.bands.n_px;
        const int tri = p.px.hit_tri[kpx];
        n_hit = (p.k == 0) && tri >= 0;
        if (tri < 0) {
            if (p.k == 0) p.px.accum[kpx] = p.px.accum[n + kpx] = p.px.accum[2 * n + kpx] = 0.f; // vec3 ctor, vec.h:44
            if (p.k < p.L) {
                p.px.rj[kpx] = -1;
                if (p.dbg_occ) p.dbg_occ[(size_t)kpx * p.L + p.k] = -2;
            }
        } else {
            int w, h;
            p.bands.map(kpx, w, h);
            const f3 origin = strict::ld(p.cam.o);
            const f3 dir = primary_dir(p.cam, p.bands, w, h);
            const float *mat;
            f3 N;
            float t;
            f3 acc;
            if (p.k == 0) {
                t = p.px.hit_t[kpx];
                if (tri < p.n_tris) {
                    const float *q = p.tri_verts + 9 * (size_t)tri;
                    const f3 v0 = strict::ld(q), v1 = strict::ld(q + 3), v2 = strict::ld(q + 6);
                    N = strict::normalize(strict::cross(strict::sub(v1, v0), strict::sub(v2, v0))); // main.cpp:728-731
                    const int g = p.tri_geom[tri];
                    if (p.geom_has_normals && p.geom_has_normals[g]) { // main.cpp:733-738, u == 0
                        const float *nq = p.tri_normals + 9 * (size_t)tri;
                        const f3 N0 = strict::ld(nq), N1 = strict::ld(nq + 3), N2 = strict::ld(nq + 6);
                        const float u = 0.f, v = p.px.hit_v[kpx];
                        const float wgt = __fsub_rn(__fsub_rn(1.f, u), v);
                        N = strict::normalize(strict::add(strict::add(strict::mul(N1, u), strict::mul(N2, v)), strict::mul(N0, wgt)));
                    }
                } else { // extension: sphere normal
                    const float4 cr = p.spheres[tri - p.n_tris];
                    N = strict::normalize(strict::sub(strict::add(origin, strict::mul(dir, t)), strict::mk(cr.x, cr.y, cr.z)));
                }
                p.px.nrm[kpx] = N.x, p.px.nrm[n + kpx] = N.y, p.px.nrm[2 * n + kpx] = N.z;
                acc = strict::mk(0.f, 0.f, 0.f);
            } else {
                N = strict::mk(p.px.nrm[kpx], p.px.nrm[n + kpx], p.px.nrm[2 * n + kpx]);
                acc = strict::mk(p.px.accum[kpx], p.px.accum[n + kpx], p.px.accum[2 * n + kpx]);
                // what occlusion() left in t: t2 of the first occluder, else tmax (main.cpp:320-324, 764)
                const unsigned long long ok = p.px.best_occ[kpx];
                t = ok == KEY_NONE ? p.px.rt[kpx] : __uint_as_float((unsigned)(ok & 0xffffffffu));
            }
            mat = (tri < p.n_tris) ? p.geom_material + 13 * (size_t)p.tri_geom[tri]
                                   : p.sphere_material + 13 * (size_t)(tri - p.n_tris);
            const float fL = (float)p.L;
            if (p.k > 0) { // finish light k-1: main.cpp:768-788
                const unsigned long long ok = p.px.best_occ[kpx];
                const int occ = ok == KEY_NONE ? -1 : (int)(unsigned)(ok >> 32);
                if (p.dbg_occ) p.dbg_occ[(size_t)kpx * p.L + (p.k - 1)] = occ;
                ref_tests += (occ >= 0 && occ < p.n_tris) ? (unsigned)(occ + 1) : (unsigned)p.n_tris;
                if (occ < 0) {
                    const f3 Lv = strict::mk(p.px.rd[kpx], p.px.rd[n + kpx], p.px.rd[2 * n + kpx]);
                    const float d = strict::dot(N, Lv);
                    if (d > 0.f) {
                        const f3 ka = strict::ld(mat), kd = strict::ld(mat + 3), ks = strict::ld(mat + 6), ke = strict::ld(mat + 9);
                        const float Ns = mat[12];
                        f3 c = strict::div(strict::add(strict::mul(ka, 0.5f), ke), fL);
                        const f3 Hh = strict::normalize(strict::mul(strict::add(N, Lv), 2.f));
                        const float pw = strict::powf_glibc(strict::dot(N, Hh), Ns); // glibc powf, bit for bit
                        c = strict::add(c, strict::div(strict::add(strict::mul(kd, d), strict::mul(ks, pw)), fL));
                        acc = strict::add(acc, c);
                    }
                }
            }
            p.px.accum[kpx] = acc.x, p.px.accum[n + kpx] = acc.y, p.px.accum[2 * n + kpx] = acc.z;
            if (p.k < p.L) { // set up light k: main.cpp:740-766
                const int vb = p.li.light_vbase[p.k];
                const int F = p.li.light_vbase[p.k + 1] - vb;
                int fid;
                if (p.rng_mode == 0)
                    fid = hash_faceid(p.seed, (uint32_t)(h * p.bands.W + w), (uint32_t)p.k, (uint32_t)F);
                else
                    fid = p.faceid[(size_t)kpx * p.L + p.k];
                fid = min(max(fid, 0), F - 1);
                const f3 v0 = strict::ld(p.li.light_verts + 3 * (size_t)(vb + fid));
                // P = v0 + ((v1-v0)*r1 + (v2-v0)*r2) with v1 = v2 = v0 (main.cpp:749-754)
                const f3 zero = strict::sub(v0, v0);
                const f3 P = strict::add(v0, strict::add(strict::mul(zero, 0.5f), strict::mul(zero, 0.5f)));
                const f3 hit = strict::add(origin, strict::mul(dir, __fsub_rn(t, TRC_EPS)));
                f3 Lv = strict::sub(P, hit);
                const float len = strict::length(Lv);
                t = __fsub_rn(len, TRC_EPS);
                Lv = strict::normalize(Lv);
                p.px.ro[kpx] = hit.x, p.px.ro[n + kpx] = hit.y, p.px.ro[2 * n + kpx] = hit.z;
                p.px.rd[kpx] = Lv.x, p.px.rd[n + kpx] = Lv.y, p.px.rd[2 * n + kpx] = Lv.z;
                p.px.rt[kpx] = t;
                // filter parameters: the line through the light vertex towards the hit point, on the cube
                // face of its dominant axis: (p,q) = (d_a, d_b)/|d_c|.  A ray longer than the table's reach
                // bound (never expected) or a degenerate one goes to the "all candidates" group instead.
                const float fd[3] = {hit.x - v0.x, hit.y - v0.y, hit.z - v0.z};
                const float ax = fabsf(fd[0]), ay = fabsf(fd[1]), az = fabsf(fd[2]);
                const int c = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
                const float dc = fd[c];
                const float inv = 1.0f / fabsf(dc);
                const bool ok = (fabsf(dc) > 0.f) && ((double)len <= p.lmax) && isfinite(inv);
                const int face = ok ? 2 * c + (dc < 0.f ? 1 : 0) : NFACE - 1;
                const float da = c == 0 ? fd[1] : (c == 1 ? fd[2] : fd[0]); // axis (c+1)%3
                const float db = c == 0 ? fd[2] : (c == 1 ? fd[0] : fd[1]); // axis (c+2)%3
                p.px.re[kpx] = ok ? da * inv : 0.f;
                p.px.re[n + kpx] = ok ? db * inv : 0.f;
                const int key = fid * NFACE + face;
                if (p.cull_cells == 2) { // sort key: ray group, then q (default mode: the rays of a thread share a q-term)
                    const unsigned qb = __float_as_uint(ok ? db * inv : 0.f);
                    rkey_mine = ((unsigned long long)(unsigned)key << 32) | ((qb & 0x80000000u) ? ~qb : (qb | 0x80000000u));
                } else if (p.cull_cells) { // sort key: ray group, then the 16+16-bit Morton code of (p,q) on the face
                    unsigned mx = ok ? (unsigned)fminf(65535.f, fmaxf(0.f, (da * inv + 1.f) * 32767.5f)) : 0u;
                    unsigned my = ok ? (unsigned)fminf(65535.f, fmaxf(0.f, (db * inv + 1.f) * 32767.5f)) : 0u;
                    mx = (mx | (mx << 8)) & 0x00ff00ffu, mx = (mx | (mx << 4)) & 0x0f0f0f0fu, mx = (mx | (mx << 2)) & 0x33333333u, mx = (mx | (mx << 1)) & 0x55555555u;
                    my = (my | (my << 8)) & 0x00ff00ffu, my = (my | (my << 4)) & 0x0f0f0f0fu, my = (my | (my << 2)) & 0x33333333u, my = (my | (my << 1)) & 0x55555555u;
                    rkey_mine = ((unsigned long long)(unsigned)key << 32) | (mx | (my << 1));
                }
                p.px.rj[kpx] = key;
                my_j = key;
            }
        }
    }
    if (p.k < p.L && p.cull_cells && in_range) p.rkey[kpx] = rkey_mine;
    if (p.k < p.L) { // histogram of rays per light vertex, warp-aggregated
        const unsigned active = __ballot_sync(0xffffffffu, my_j >= 0);
        if (my_j >= 0) {
            const unsigned peers = __match_any_sync(active, my_j);
            if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&p.seg_count[my_j], __popc(peers));
        }
    }
    if (p.k > 0) {
        for (int o = 16; o; o >>= 1) ref_tests += __shfl_down_sync(0xffffffffu, ref_tests, o);
        if ((threadIdx.x & 31) == 0 && ref_tests) atomicAdd(&p.counters->tests_shadow_ref, ref_tests);
    } else {
        for (int o = 16; o; o >>= 1) n_hit += __shfl_down_sync(0xffffffffu, n_hit, o);
        if ((threadIdx.x & 31) == 0 && n_hit) atomicAdd(&p.counters->n_hits, (unsigned long long)n_hit);
    }
}

// seg_count[F] -> seg_off[F+1] (fixed for this light), cursors zeroed
__global__ void list_prefix_kernel(const int *seg_count, int F, int *seg_off, int *cursor) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int so = 0;
        for (int j = 0; j < F; ++j) {
            seg_off[j] = so;
            cursor[j] = 0;
            so += seg_count[j];
        }
        seg_off[F] = so;
    }
}

// before each triangle chunk: live-ray counts per ray group -> ray-block offsets; reset the
// survivors' counters and the work counter
// The triangle-slice count of the chunk is chosen here, on the device, from the live block count (so the
// host never has to wait for it): enough (block, slice) items to keep every SM busy, >= 4 tiles per slice.
__global__ void chunk_prefix_kernel(const int *cnt_in, int F, int rays_per_block, int n_tiles_chunk, int n_sms, int *blk_off,
                                    int *cnt_out, int *work, int *n_slices_out, int items_per_sm = 6, int min_tiles = 4) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int bo = 0;
        for (int j = 0; j < F; ++j) {
            blk_off[j] = bo;
            cnt_out[j] = 0;
            bo += (cnt_in[j] + rays_per_block - 1) / rays_per_block;
        }
        blk_off[F] = bo;
        *work = 0;
        const int possible = max(1, n_tiles_chunk / min_tiles);
        int sl = bo >= items_per_sm * n_sms ? 1 : (items_per_sm * n_sms + max(bo, 1) - 1) / max(bo, 1);
        *n_slices_out = max(1, min(sl, possible));
    }
}

__global__ void iota_kernel(int *a, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

// ---------------------------------------------------------------------------------
// First in-order occluder (occlusion(), main.cpp:314-329): ONE persistent cooperative kernel per light.
// Rays are grouped by (light vertex, cube face): segment j of the q-sorted list, table j.  The triangle table is cut
// into chunks; inside the kernel every chunk is
//     A. swept: (ray block, triangle slice) work items pulled from an atomic counter, merged by atomicMin on
//        index<<32|t2;                                                                         grid barrier
//     B. compacted, order preserving (the lists stay sorted by q): survivors counted per block of CBLK entries,
//                                                                                              grid barrier
//     C. ... and written in list order to the other list; new per-group counts;               grid barrier
// so the pairs actually swept track the reference's own early-exit count (main.cpp:324) and the host is not in
// the loop at all: block offsets, slice counts, the chunk scheme and the early stop ("every ray has its occluder")
// are decided on the device.  Round 1 ran A/B/C as 4 launches per chunk with host read-backs in between.
constexpr int SHADOW_R = 16;    // rays per thread of a full shadow-ray block (blocks of NT * SHADOW_R consecutive list entries).
                                // 32 measured slower (C4: 397 vs 330 ms): a thread's strict evaluations serialise over twice the
                                // rays and the CTAs that hold them are the stragglers of every chunk barrier (23 % waiting)
constexpr int SL_MAXF = 1022;   // ray groups per launch (the host batches bigger lights: 146 vertices x NFACE)
constexpr int SL_MAXCHUNK = 64;
constexpr int CBLK = 1024;      // list entries per compaction block

struct ShadowLightParams {
    const float4 *tables;  // face tables of this launch's first light vertex: group g=(j,f<6) at + (j*6+f)*table_stride
    const float4 *allcand; // table of group f == 6
    size_t table_stride;   // in float4
    int n_tris, n_tiles, F, n_px; // F = ray groups of this launch (light vertices * NFACE)
    int n_chunks[2];              // [0] geometric scheme (few rays), [1] equal chunks (>= many_rays live rays)
    int bounds[2][SL_MAXCHUNK + 1]; // chunk boundaries in tiles
    long long many_rays;
    int items_per_cta;            // (ray block, slice) items wanted per resident CTA
    int min_tiles;                // smallest slice, in tiles
    long long run_pairs;          // longest run of items handed to a CTA at once, in (ray, triangle) pairs
    const float *tri_verts;
    int *list[2];                 // ping-pong ray lists, [0] = the sorted input
    const int *seg_off;           // [F+1] segment starts of this launch's groups (absolute list positions)
    int *cnt[2];                  // [F] live rays per group, ping-pong; [0] = initial counts
    int *blk_cnt;                 // compaction scratch: survivors per compaction block (<= n_px/CBLK + F entries)
    PixelState px;
    const float4 *spheres;        // extension: tested after all triangles by the rays that found none
    int n_spheres;
    sweep::Counters *counters;
    int *work;                    // [SL_MAXCHUNK] work counters, zeroed by the host
    unsigned long long *timeline; // development (TRACER_SHADOW_DIAG=2): [SL_MAXCHUNK][gridDim.x][2] globaltimer ns at which a CTA
                                  // ran out of sweep items / left the barrier after the sweep, or null
};

// The reference's own test for the rays (bits of mask) of one thread against triangle tri, shadow rays
// (occlusion(), main.cpp:314-329): the first accepted face in order ends the ray and leaves t = t2 behind (the
// multi-light carry).  Origin, direction and length stay in the pixel state and are fetched on demand: only a
// few rays per work item ever get here.  Ray r of the thread is list entry min(e0 + r, e_last).
// Returns newly occluded rays (bits 0-31) | evaluations << 32 | filter misses << 48.
__device__ __noinline__ unsigned long long strict_shadow(const PixelState &px, const float *__restrict__ tri_verts, const int *__restrict__ list_in,
                                               int n_px, int e0, int e_last, unsigned mask, int tri, unsigned filt) {
    const float *q = tri_verts + 9 * (size_t)tri;
    const f3 v0 = strict::mk(__ldg(q), __ldg(q + 1), __ldg(q + 2));
    const f3 v1 = strict::mk(__ldg(q + 3), __ldg(q + 4), __ldg(q + 5));
    const f3 v2 = strict::mk(__ldg(q + 6), __ldg(q + 7), __ldg(q + 8));
    const size_t n = (size_t)n_px;
    unsigned long long ret = 0;
    while (mask) {
        const int r = __ffs(mask) - 1;
        mask &= mask - 1;
        const int k = list_in[min(e0 + r, e_last)];
        const f3 o = strict::mk(px.ro[k], px.ro[n + k], px.ro[2 * n + k]);
        const f3 d = strict::mk(px.rd[k], px.rd[n + k], px.rd[2 * n + k]);
        float t = px.rt[k], v = 0.f; // the ray has no occluder yet, so t is its initial length (main.cpp:764)
        ret += 1ull << 32;
        if (strict::intersect_triangle(o, d, v0, v1, v2, t, v)) {
            atomicMin(&px.best_occ[k], ((unsigned long long)(unsigned)tri << 32) | __float_as_uint(t));
            ret |= 1ull << r;
            if (!((filt >> r) & 1u)) ret += 1ull << 48;
        }
    }
    return ret;
}

// one (ray block, triangle slice) work item with RR rays per thread.  The list is ordered by q inside each group
// (and compaction keeps it so); a thread takes RR CONSECUTIVE rays, whose q differ by ~1e-6, and evaluates them
// with one q-term per edge row (sweep::MODE_QBAR).
template <int RR, bool EXHAUSTIVE>
__device__ __forceinline__ void shadow_item(sweep::SmemT<2> &sm, const ShadowLightParams &p, const int *__restrict__ list_in, int base,
                                            int seg_end, int lo, int hi, const float4 *__restrict__ tab, unsigned &gtile,
                                            unsigned &n_strict, unsigned &n_miss, unsigned long long &tests, unsigned &n_pipe_err) {
    const int tid = threadIdx.x, n = p.n_px;
    float rp[RR], rq[RR];
    unsigned valid = 0, done = 0;
    const int e0 = base + tid * RR;
#pragma unroll
    for (int r = 0; r < RR; ++r) {
        if (e0 + r < seg_end) valid |= 1u << r;
        const int k = list_in[min(e0 + r, seg_end - 1)];
        rp[r] = p.px.re[k], rq[r] = p.px.re[n + k];
        // an earlier slice may already have published an occluder below this slice: nothing to do
        const unsigned long long seen = p.px.best_occ[k];
        if (seen != KEY_NONE && (int)(unsigned)(seen >> 32) < lo * sweep::TILE) done |= 1u << r;
    }
    // rays past the end of the list are duplicates of the last one, so all RR values count
    float qmin = rq[0], qmax = rq[0];
#pragma unroll
    for (int r = 1; r < RR; ++r) qmin = fminf(qmin, rq[r]), qmax = fmaxf(qmax, rq[r]);
    const float qbar = 0.5f * (qmin + qmax);
    // >= max |q_r - qbar| with room for the roundings of this line and of the one extra FFMA per row
    const float qdelta = fmaxf(qmax - qbar, qbar - qmin) * 1.0001f + 2.4e-7f * (fabsf(qbar) + 1.f);
    unsigned swept = 0;
    sweep::sweep_table<RR, sweep::MODE_QBAR, true, EXHAUSTIVE>(
        sm, tab, lo, hi, p.n_tris, rp, rq, qbar, qdelta, valid, done, gtile, swept, [&](unsigned mask, int tri, unsigned filt) {
            const unsigned long long c = strict_shadow(p.px, p.tri_verts, list_in, n, e0, seg_end - 1, mask, tri, filt);
            n_strict += (unsigned)(c >> 32) & 0xffffu, n_miss += (unsigned)(c >> 48);
            return (unsigned)c;
        },
        &n_pipe_err);
    tests += (unsigned long long)swept * sweep::TILE * __popc(valid);
}

// exclusive prefix over the F groups of ceil(cnt[j] / unit), by the whole CTA into shared memory; returns the total
__device__ __forceinline__ int cta_group_prefix(const int *__restrict__ cnt, int F, int unit, int *out /*[F+1] shared*/, int *scratch) {
    constexpr int PER = (SL_MAXF + 1 + sweep::NT - 1) / sweep::NT;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    int v[PER], sum = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int j = tid * PER + i;
        v[i] = j < F ? (cnt[j] + unit - 1) / unit : 0;
        sum += v[i];
    }
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    __syncthreads(); // scratch / out may still be read from the previous use
    if (lane == 31) scratch[w] = incl;
    __syncthreads();
    int base = 0, total = 0;
    for (int i = 0; i < sweep::NT / 32; ++i) {
        if (i < w) base += scratch[i];
        total += scratch[i];
    }
    int run = base + incl - sum;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int j = tid * PER + i;
        if (j <= F) out[j] = run;
        run += v[i];
    }
    __syncthreads();
    return total;
}

// group of block b: largest j with off[j] <= b (off is non-decreasing, off[F] = total > b)
__device__ __forceinline__ int group_of_block(const int *off, int F, int b) {
    int lo = 0, hi = F; // invariant: off[lo] <= b < off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= b) lo = mid;
        else hi = mid;
    }
    return lo;
}

// All CTAs of the launch are co-resident (cooperative launch).  Monotonic counter: arrive, then wait for the epoch's
// total.  The counter is zeroed by the host before the launch.
__device__ __forceinline__ void grid_barrier(unsigned *bar, unsigned &epoch) {
    __syncthreads();
    if (threadIdx.x == 0) {
        ++epoch;
        __threadfence();
        atomicAdd(bar, 1u);
        const unsigned want = epoch * gridDim.x;
        while (*(volatile unsigned *)bar < want) __nanosleep(20);
        __threadfence();
    }
    __syncthreads();
}

template <bool EXHAUSTIVE>
__global__ void __launch_bounds__(sweep::NT, sweep::MINB) shadow_light_kernel(const __grid_constant__ ShadowLightParams p, unsigned *bar) {
    static_assert(CBLK % sweep::NT == 0, "compaction block must be a multiple of the CTA size");
    constexpr int R = SHADOW_R, CPT = CBLK / sweep::NT; // rays per thread of a full ray block; list entries per thread of a compaction block
    extern __shared__ __align__(128) unsigned char smem_raw[];
    sweep::SmemT<2> &sm = *reinterpret_cast<sweep::SmemT<2> *>(smem_raw); // the any-hit sweeps read span tables only
    __shared__ int s_blk_off[SL_MAXF + 1], s_cblk_off[SL_MAXF + 1], s_scratch[sweep::NT / 32], s_off;
    const int tid = threadIdx.x, F = p.F;
    sweep::smem_init(sm);
    unsigned gtile = 0, n_strict = 0, n_miss = 0, epoch = 0, n_pipe_err = 0;
    unsigned long long tests = 0;
    long long c_items = 0, c_bar = 0, c_comp = 0, n_it = 0, n_run = 0; // time split (thread 0)
    const long long c_begin = clock64();
    // chunk scheme: equal chunks keep the pairs swept past a ray's occluder lowest and win when the light has many
    // rays; with few rays the per-chunk tails weigh more and boundaries that start fine and coarsen geometrically win
    const long long live0 = cta_group_prefix(p.cnt[0], F, 1, s_blk_off, s_scratch);
    const int scheme = live0 >= p.many_rays ? 1 : 0;
    const int n_chunks = p.n_chunks[scheme];
    const int *bounds = p.bounds[scheme];
    int cur = 0;
    for (int c = 0; c < n_chunks; ++c) {
        const int *list_in = p.list[cur], *cnt_in = p.cnt[cur];
        int *list_out = p.list[cur ^ 1], *cnt_out = p.cnt[cur ^ 1];
        const int total_blocks = cta_group_prefix(cnt_in, F, sweep::NT * R, s_blk_off, s_scratch);
        if (total_blocks == 0) break; // every shadow ray of this light already has its occluder (same on every CTA)
        const int total_cblocks = cta_group_prefix(cnt_in, F, CBLK, s_cblk_off, s_scratch);
        const int tile_lo = bounds[c], tile_hi = bounds[c + 1], n_tiles = tile_hi - tile_lo;
        // (ray block, triangle slice) items, slices of >= min_tiles tiles.  Items are BLOCK-major (consecutive items = consecutive
        // slices of one ray block) and handed out in runs whose length shrinks as the chunk drains (guided self-scheduling):
        // long runs while there is plenty of work (one ray set-up per run), single smallest slices at the end, so the
        // chunk's tail — every CTA waits at the grid barrier for the last item — is one small slice long.  This is what
        // the 8-GPU band shares need: their chunks are only ~1 ms long.
        const int want = p.items_per_cta * (int)gridDim.x;
        const int n_slices = max(1, min(total_blocks >= want ? 1 : (want + total_blocks - 1) / total_blocks, max(1, n_tiles / p.min_tiles)));
        const int n_items = total_blocks * n_slices;
        // Runs are also capped in absolute size.  Guided self-scheduling assumes CTAs of equal speed, and the four CTAs of an
        // SM are not: the hardware's warp arbiter favours some of them, the starved one is still inside a long run when the
        // others find the queue empty (measured with TRACER_SHADOW_DIAG=2 at C4: 3/4 of the CTAs waited ~0.7 ms of every
        // 6 ms chunk for the 4th CTA of each SM).  Short runs bound that tail; each costs one ray set-up (a few us).
        const long long item_pairs = (long long)(sweep::NT * R) * sweep::TILE * max(1, n_tiles / n_slices);
        const int g_cap = (int)max(1ll, p.run_pairs / item_pairs);
        // ---- A: sweep --------------------------------------------------------------------------------------
        for (;;) {
            if (tid == 0) {
                const int seen = *(volatile int *)&p.work[c];
                const int g = max(1, min(min((n_items - seen) / (2 * (int)gridDim.x), n_slices), g_cap));
                const int it = atomicAdd(&p.work[c], g);
                sm.blk = it < n_items ? it : -1, sm.seg = min(it + g, n_items);
            }
            __syncthreads();
            int it = sm.blk;
            const int it_end = sm.seg;
            if (it < 0) break;
            const long long c_run = clock64();
            ++n_run;
            while (it < it_end) { // (uniform) one run per ray block touched
                ++n_it;
                const int blk = it / n_slices, sl0 = it - blk * n_slices, sl1 = min(n_slices, sl0 + (it_end - it));
                it += sl1 - sl0;
                const int j = group_of_block(s_blk_off, F, blk);
                const int lo = tile_lo + (int)((long long)n_tiles * sl0 / n_slices);
                const int hi = tile_lo + (int)((long long)n_tiles * sl1 / n_slices);
                const int seg_begin = p.seg_off[j], seg_end = seg_begin + cnt_in[j];
                const int base = seg_begin + (blk - s_blk_off[j]) * (sweep::NT * R);
                const int face = j % NFACE;
                const float4 *tab = face == NFACE - 1 ? p.allcand : p.tables + (size_t)((j / NFACE) * 6 + face) * p.table_stride;
                // The last block of a ray group is rarely full.  A block with at most NT*RR rays is swept with RR rays per
                // thread instead of dragging empty lanes through every triangle (late chunks have few rays in many groups).
                const int cnt = seg_end - base;
                if (cnt > 8 * sweep::NT)
                    shadow_item<SHADOW_R, EXHAUSTIVE>(sm, p, list_in, base, seg_end, lo, hi, tab, gtile, n_strict, n_miss, tests, n_pipe_err);
                else if (cnt > 4 * sweep::NT)
                    shadow_item<8, EXHAUSTIVE>(sm, p, list_in, base, seg_end, lo, hi, tab, gtile, n_strict, n_miss, tests, n_pipe_err);
                else if (cnt > 2 * sweep::NT)
                    shadow_item<4, EXHAUSTIVE>(sm, p, list_in, base, seg_end, lo, hi, tab, gtile, n_strict, n_miss, tests, n_pipe_err);
                else
                    shadow_item<2, EXHAUSTIVE>(sm, p, list_in, base, seg_end, lo, hi, tab, gtile, n_strict, n_miss, tests, n_pipe_err);
                __syncthreads(); // every warp is out of the tile pipeline before the next run re-arms it
            }
            c_items += clock64() - c_run;
        }
        if (p.timeline && tid == 0) {
            unsigned long long ns;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
            p.timeline[((size_t)c * gridDim.x + blockIdx.x) * 2] = ns;
        }
        if (c == n_chunks - 1) break; // nothing left to sweep: the lists are not needed compacted
        long long c0 = clock64();
        grid_barrier(bar, epoch);
        c_bar += clock64() - c0, c0 = clock64();
        if (p.timeline && tid == 0) {
            unsigned long long ns;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
            p.timeline[((size_t)c * gridDim.x + blockIdx.x) * 2 + 1] = ns;
        }
        // ---- B: survivors per compaction block ------------------------------------------------------------------
        for (int cb = blockIdx.x; cb < total_cblocks; cb += gridDim.x) {
            const int j = group_of_block(s_cblk_off, F, cb), bx = cb - s_cblk_off[j];
            const int begin = p.seg_off[j], count = cnt_in[j];
            int alive = 0;
#pragma unroll
            for (int q = 0; q < CPT; ++q) {
                const int i = bx * CBLK + tid * CPT + q;
                if (i < count && p.px.best_occ[list_in[begin + i]] == KEY_NONE) ++alive;
            }
            for (int o = 16; o; o >>= 1) alive += __shfl_down_sync(0xffffffffu, alive, o);
            __syncthreads();
            if ((tid & 31) == 0) s_scratch[tid >> 5] = alive;
            __syncthreads();
            if (tid == 0) {
                int t = 0;
                for (int w = 0; w < sweep::NT / 32; ++w) t += s_scratch[w];
                p.blk_cnt[cb] = t;
            }
        }
        c_comp += clock64() - c0, c0 = clock64();
        grid_barrier(bar, epoch);
        c_bar += clock64() - c0, c0 = clock64();
        // ---- C: write the survivors in list order ---------------------------------------------------------------
        for (int cb = blockIdx.x; cb < total_cblocks; cb += gridDim.x) {
            const int j = group_of_block(s_cblk_off, F, cb), bx = cb - s_cblk_off[j];
            const int begin = p.seg_off[j], count = cnt_in[j];
            int before = 0; // survivors in the group's blocks before this one
            for (int b = tid; b < bx; b += sweep::NT) before += p.blk_cnt[s_cblk_off[j] + b];
            for (int o = 16; o; o >>= 1) before += __shfl_down_sync(0xffffffffu, before, o);
            __syncthreads();
            if ((tid & 31) == 0) s_scratch[tid >> 5] = before;
            __syncthreads();
            if (tid == 0) {
                int t = 0;
                for (int w = 0; w < sweep::NT / 32; ++w) t += s_scratch[w];
                s_off = t;
            }
            __syncthreads();
            const int off = s_off;
            int ks[CPT], alive = 0;
#pragma unroll
            for (int q = 0; q < CPT; ++q) {
                const int i = bx * CBLK + tid * CPT + q;
                int k = -1;
                if (i < count) {
                    k = list_in[begin + i];
                    if (p.px.best_occ[k] != KEY_NONE) k = -1;
                }
                ks[q] = k;
                alive += k >= 0;
            }
            int incl = alive; // inclusive scan over the CTA
            const int lane = tid & 31, w = tid >> 5;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            __syncthreads(); // s_scratch is reused
            if (lane == 31) s_scratch[w] = incl;
            __syncthreads();
            int wbase = 0;
            for (int i = 0; i < w; ++i) wbase += s_scratch[i];
            int pos = off + wbase + incl - alive;
#pragma unroll
            for (int q = 0; q < CPT; ++q)
                if (ks[q] >= 0) list_out[begin + pos++] = ks[q];
            if ((bx + 1) * CBLK >= count && tid == sweep::NT - 1) cnt_out[j] = off + wbase + incl; // the group's last block
            __syncthreads();
        }
        // groups without entries keep a zero count
        for (int j = blockIdx.x * sweep::NT + tid; j < F; j += gridDim.x * sweep::NT)
            if (cnt_in[j] == 0) cnt_out[j] = 0;
        c_comp += clock64() - c0, c0 = clock64();
        grid_barrier(bar, epoch);
        c_bar += clock64() - c0;
        cur ^= 1;
    }
    // ---- extension: spheres come after all triangles in the object order --------------------------------------------
    if (p.n_spheres > 0) {
        grid_barrier(bar, epoch); // every sweep of the last chunk has published its occluders
        const int *list_in = p.list[cur], *cnt_in = p.cnt[cur];
        const size_t n = (size_t)p.n_px;
        for (int j = 0; j < F; ++j) {
            const int begin = p.seg_off[j], count = cnt_in[j];
            for (int i = blockIdx.x * sweep::NT + tid; i < count; i += gridDim.x * sweep::NT) {
                const int k = list_in[begin + i];
                if (p.px.best_occ[k] != KEY_NONE) continue;
                const f3 o = strict::mk(p.px.ro[k], p.px.ro[n + k], p.px.ro[2 * n + k]);
                const f3 d = strict::mk(p.px.rd[k], p.px.rd[n + k], p.px.rd[2 * n + k]);
                float t = p.px.rt[k];
                for (int s = 0; s < p.n_spheres; ++s)
                    if (strict::intersect_sphere(o, d, __ldg(&p.spheres[s]), t)) {
                        p.px.best_occ[k] = ((unsigned long long)(unsigned)(p.n_tris + s) << 32) | __float_as_uint(t);
                        break;
                    }
            }
        }
    }
    atomicAdd(&p.counters->tests_shadow, tests);
    atomicAdd(&p.counters->strict_evals, (unsigned long long)n_strict);
    if (EXHAUSTIVE) atomicAdd(&p.counters->filter_misses, (unsigned long long)n_miss);
    if (EXHAUSTIVE && n_pipe_err) atomicAdd(&p.counters->pipeline_errors, (unsigned long long)n_pipe_err);
    if (tid == 0) {
        atomicAdd(&p.counters->cyc_items, (unsigned long long)c_items), atomicAdd(&p.counters->cyc_barrier, (unsigned long long)c_bar);
        atomicAdd(&p.counters->cyc_compact, (unsigned long long)c_comp), atomicAdd(&p.counters->cyc_total, (unsigned long long)(clock64() - c_begin));
        atomicAdd(&p.counters->n_items, (unsigned long long)n_it), atomicAdd(&p.counters->n_runs, (unsigned long long)n_run);
    }
}

// extension: spheres are tested after all triangles, in order, by the rays that found no triangle
__global__ void shadow_spheres_kernel(const int *__restrict__ list, const int *__restrict__ seg_off, const int *__restrict__ cnt,
                                      int F, PixelState px, int n_px, const float4 *__restrict__ spheres, int n_spheres,
                                      int n_tris) {
    const int j = blockIdx.y;
    if (j >= F) return;
    const int begin = seg_off[j], count = cnt[j];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const int k = list[begin + i];
        if (px.best_occ[k] != KEY_NONE) continue;
        const f3 o = strict::mk(px.ro[k], px.ro[n_px + k], px.ro[2 * n_px + k]);
        const f3 d = strict::mk(px.rd[k], px.rd[n_px + k], px.rd[2 * n_px + k]);
        float t = px.rt[k];
        for (int s = 0; s < n_spheres; ++s)
            if (strict::intersect_sphere(o, d, __ldg(&spheres[s]), t)) {
                px.best_occ[k] = ((unsigned long long)(unsigned)(n_tris + s) << 32) | __float_as_uint(t);
                break;
            }
    }
}

// ---------------------------------------------------------------------------------
// OPTIONAL bundle-cull mode (cull.cuh): same results, hierarchical evaluation of the filter.
struct PrimaryCullParams {
    Cam cam;
    Bands bands;
    const float4 *table;
    int n_tiles, n_tris, n_rows, tiles_x, tiles_y, n_slices;
    cull::Emitter em;
    sweep::Counters *counters;
    int *work;
};

// rays of block blk of the primary tiling: 128 x 32 pixels per block, 32 x 8 per warp, R = 8 rows per thread
template <int R>
__device__ __forceinline__ void load_primary_bundle(const PrimaryCullParams &p, int blk, int warp, float (&rp)[R], float (&rq)[R],
                                                    float (&rl)[R], int (&kp)[R], unsigned &valid) {
    const int lane = threadIdx.x & 31, W = p.bands.W;
    const int ty = blk / p.tiles_x, tx = blk - ty * p.tiles_x;
    const int x = tx * 128 + (warp & 3) * 32 + lane, y0 = ty * 32 + (warp >> 2) * 8;
    valid = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int ly = y0 + r;
        if (x < W && ly < p.n_rows) valid |= 1u << r;
        const int k = min(ly, p.n_rows - 1) * W + min(x, W - 1); // clamp: duplicates of valid rays keep the boxes tight
        kp[r] = k;
        int w, h;
        p.bands.map(k, w, h);
        p.bands.pixel_st(w, h, rp[r], rq[r]);
        rl[r] = FLT_MAX; // primary rays are unbounded (main.cpp:715)
    }
}

// work item = screen tile of 128 x 32 pixels (warp: 32 x 8) x triangle slice; emits candidate pairs
__global__ void __launch_bounds__(sweep::THREADS, 2) primary_cull_kernel(const PrimaryCullParams p) {
    constexpr int R = 8;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    cull::EmitSmem &sm = *reinterpret_cast<cull::EmitSmem *>(smem_raw);
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < cull::CSTAGES; ++s) sweep::mbar_init(&sm.full_bar[s], 1);
        sweep::fence_barrier_init();
    }
    __syncthreads();
    unsigned gtile = 0;
    unsigned long long tests = 0;
    cull::WarpChunk wc{0, cull::CHUNK}; // no chunk yet
    const int n_blocks = p.tiles_x * p.tiles_y, n_items = n_blocks * p.n_slices;
    for (;;) {
        if (tid == 0) sm.blk = atomicAdd(p.work, 1);
        __syncthreads();
        const int item = sm.blk;
        if (item >= n_items) break;
        const int slice = item / n_blocks, blk = item - slice * n_blocks;
        const int tile_lo = (int)((long long)p.n_tiles * slice / p.n_slices);
        const int tile_hi = (int)((long long)p.n_tiles * (slice + 1) / p.n_slices);
        float rp[R], rq[R], rl[R];
        int kp[R];
        unsigned valid = 0;
        load_primary_bundle<R>(p, blk, threadIdx.x >> 5, rp, rq, rl, kp, valid);
        cull::Box wb, cb;
        cull::bundle_boxes<R>(rp, rq, rl, sm.scratch, wb, cb);
        cull::sweep_cull_emit<R>(sm, p.table, tile_lo, tile_hi, rp, rq, valid, kp, gtile, cb, wb, p.em, wc, nullptr);
        const int t_lo = min(tile_lo * cull::CTILE, p.n_tris), t_hi = min(tile_hi * cull::CTILE, p.n_tris);
        tests += (unsigned long long)__popc(valid) * (unsigned)(t_hi - t_lo);
        __syncthreads();
    }
    cull::chunk_close(p.em, wc);
    atomicAdd(&p.counters->tests_primary, tests);
}

// One thread per candidate pair, in whatever order the culled sweep emitted them.  Closest hit (cpp_intersect,
// main.cpp:176-192) is the lexicographic minimum of (t, index) over all valid hits and the first occluder
// (occlusion(), main.cpp:314-329) the minimum index over all valid hits, so — exactly like the triangle slices
// of the default mode — every pair is evaluated independently with the reference's arithmetic and merged with
// a 64-bit atomicMin; no sort of the candidates is needed.  *count may exceed cap (entries beyond cap were
// dropped by the emitter): that is reported through counters->cull_overflow and fails the frame.
__global__ void strict_primary_pairs(const unsigned long long *__restrict__ cand, const unsigned long long *__restrict__ count,
                                     unsigned long long cap, Cam cam, Bands bands, const float *__restrict__ tri_verts,
                                     unsigned long long *best, sweep::Counters *counters) {
    unsigned long long n = *count;
    if (n > cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&counters->cull_overflow, 1ull);
        n = cap;
    }
    unsigned n_strict = 0;
    const f3 o = strict::ld(cam.o);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long key = cand[i];
        const unsigned ray = (unsigned)(key >> 32);
        if (ray == 0xffffffffu) continue; // unused tail of a warp's chunk
        const int tr = (int)(unsigned)(key & 0xffffffffu);
        int w, h;
        bands.map((int)ray, w, h);
        const f3 d = primary_dir(cam, bands, w, h);
        const float *q = tri_verts + 9 * (size_t)tr;
        float t = FLT_MAX, v = 0.f; // main.cpp:715-717
        ++n_strict;
        if (strict::intersect_triangle(o, d, strict::ld(q), strict::ld(q + 3), strict::ld(q + 6), t, v))
            atomicMin(&best[ray], ((unsigned long long)__float_as_uint(t) << 32) | (unsigned)tr);
    }
    for (int o2 = 16; o2; o2 >>= 1) n_strict += __shfl_down_sync(0xffffffffu, n_strict, o2);
    if ((threadIdx.x & 31) == 0 && n_strict) atomicAdd(&counters->strict_evals, (unsigned long long)n_strict);
}

struct ShadowCullParams {
    const float4 *tables;
    const float4 *allcand;
    size_t table_stride;
    int n_tiles, n_tris, n_groups, n_px, cells_per_group;
    const int *n_slices;
    const int *list, *seg_off, *seg_cnt, *blk_off;
    PixelState px;
    cull::Emitter em;
    sweep::Counters *counters;
    int *work;
};

// rays of block blk of group j: 512*R consecutive rays of the (group, Morton)-sorted list, 32*R consecutive per warp
template <int R>
__device__ __forceinline__ void load_shadow_bundle(const ShadowCullParams &p, int blk, int warp, int j, float (&rp)[R], float (&rq)[R],
                                                   float (&rl)[R], int (&kp)[R], unsigned &valid) {
    const int lane = threadIdx.x & 31, n = p.n_px;
    const int seg_begin = p.seg_off[j], seg_end = seg_begin + p.seg_cnt[j];
    const int base = seg_begin + (blk - p.blk_off[j]) * (sweep::THREADS * R) + warp * (32 * R) + lane * R;
    valid = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        int e = base + r; // a warp holds 32*R consecutive rays of the sorted list, a lane R consecutive ones: compact cell ranges
        if (e < seg_end) valid |= 1u << r;
        e = min(e, seg_end - 1);
        const int k = p.list[e];
        kp[r] = k;
        rp[r] = p.px.re[k], rq[r] = p.px.re[n + k];
        // the ray ends at the light vertex O and starts len = t + eps away from it (main.cpp:762-764): an accepted
        // hit (eps <= t2 < t) lies within len of O
        rl[r] = (p.px.rt[k] + 2.f * TRC_EPS) * 1.0001f;
    }
}

// work item = 512*8 consecutive rays of the cell-sorted list of one (light vertex, face) group x triangle slice
__global__ void __launch_bounds__(sweep::THREADS, 2) shadow_cull_kernel(const ShadowCullParams p) {
    constexpr int R = 8;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    cull::EmitSmem &sm = *reinterpret_cast<cull::EmitSmem *>(smem_raw);
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < cull::CSTAGES; ++s) sweep::mbar_init(&sm.full_bar[s], 1);
        sweep::fence_barrier_init();
    }
    __syncthreads();
    const int total_blocks = p.blk_off[p.n_groups];
    const int n_slices = *p.n_slices;
    const int n_items = total_blocks * n_slices;
    unsigned gtile = 0;
    unsigned long long tests = 0;
    cull::WarpChunk wc{0, cull::CHUNK}; // no chunk yet
    for (;;) {
        if (tid == 0) {
            const int it = atomicAdd(p.work, 1);
            int j = 0, b = 0, sl = 0;
            if (it < n_items) {
                sl = it / total_blocks, b = it - sl * total_blocks;
                while (b >= p.blk_off[j + 1]) ++j;
            }
            sm.blk = it < n_items ? b : -1;
            sm.seg = j;
            sm.slice = sl;
        }
        __syncthreads();
        const int blk = sm.blk, j = sm.seg, slice = sm.slice;
        if (blk < 0) break;
        const int lo = (int)((long long)p.n_tiles * slice / n_slices), hi = (int)((long long)p.n_tiles * (slice + 1) / n_slices);
        float rp[R], rq[R], rl[R];
        int kp[R];
        unsigned valid = 0;
        load_shadow_bundle<R>(p, blk, threadIdx.x >> 5, j, rp, rq, rl, kp, valid);
        cull::Box wb, cb;
        cull::bundle_boxes<R>(rp, rq, rl, sm.scratch, wb, cb);
        const int face = j % NFACE;
        const float4 *tab = face == NFACE - 1 ? p.allcand : p.tables + (size_t)((j / NFACE) * 6 + face) * p.table_stride;
        cull::sweep_cull_emit<R>(sm, tab, lo, hi, rp, rq, valid, kp, gtile, cb, wb, p.em, wc, p.counters);
        tests += (unsigned long long)(hi - lo) * cull::CTILE * __popc(valid);
        __syncthreads();
    }
    cull::chunk_close(p.em, wc);
    atomicAdd(&p.counters->tests_shadow, tests);
}

// shadow rays: one thread per candidate pair; an accepted pair leaves t = t2 behind (the multi-light carry)
__global__ void strict_shadow_pairs(const unsigned long long *__restrict__ cand, const unsigned long long *__restrict__ count,
                                    unsigned long long cap, PixelState px, int n_px, const float *__restrict__ tri_verts,
                                    sweep::Counters *counters) {
    unsigned long long n = *count;
    if (n > cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&counters->cull_overflow, 1ull);
        n = cap;
    }
    unsigned n_strict = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long key = cand[i];
        const unsigned ray = (unsigned)(key >> 32);
        if (ray == 0xffffffffu) continue;
        const int tr = (int)(unsigned)(key & 0xffffffffu);
        // the answer is the LOWEST accepted index: once some lower-index occluder of this ray has been published,
        // this pair cannot change it (best_occ only ever decreases, so a stale read is merely conservative).  The
        // emitter walks each warp's triangles in ascending order, so this recovers most of occlusion()'s early exit.
        if ((unsigned)(px.best_occ[ray] >> 32) < (unsigned)tr) continue;
        const f3 o = strict::mk(px.ro[ray], px.ro[n_px + ray], px.ro[2 * (size_t)n_px + ray]);
        const f3 d = strict::mk(px.rd[ray], px.rd[n_px + ray], px.rd[2 * (size_t)n_px + ray]);
        float t = px.rt[ray], v;
        const float *q = tri_verts + 9 * (size_t)tr;
        ++n_strict;
        if (strict::intersect_triangle(o, d, strict::ld(q), strict::ld(q + 3), strict::ld(q + 6), t, v))
            atomicMin(&px.best_occ[ray], ((unsigned long long)(unsigned)tr << 32) | __float_as_uint(t));
    }
    for (int o2 = 16; o2; o2 >>= 1) n_strict += __shfl_down_sync(0xffffffffu, n_strict, o2);
    if ((threadIdx.x & 31) == 0 && n_strict) atomicAdd(&counters->strict_evals, (unsigned long long)n_strict);
}

// ---- two-phase bundle cull (cull.cuh: "block lists") -----------------------------------------------
// boxes of every ray block (CTA box for phase A, warp boxes for phase B), from exactly the rays the block holds
__global__ void __launch_bounds__(sweep::THREADS) primary_boxes_kernel(const PrimaryCullParams p, cull::BlockBoxes *__restrict__ out,
                                                                       int *__restrict__ blk_off) {
    constexpr int R = 8;
    __shared__ float scratch[5 * sweep::THREADS / 32];
    const int blk = blockIdx.x;
    float rp[R], rq[R], rl[R];
    int kp[R];
    unsigned valid;
    load_primary_bundle<R>(p, blk, threadIdx.x >> 5, rp, rq, rl, kp, valid);
    cull::Box wb, cb;
    cull::bundle_boxes<R>(rp, rq, rl, scratch, wb, cb);
    if ((threadIdx.x & 31) == 0) out[blk].warp[threadIdx.x >> 5] = wb;
    if (threadIdx.x == 0) out[blk].cta = cb;
    if (blk == 0 && threadIdx.x == 0) blk_off[0] = 0, blk_off[1] = p.tiles_x * p.tiles_y; // one group
}

__global__ void __launch_bounds__(sweep::THREADS) shadow_boxes_kernel(const ShadowCullParams p, cull::BlockBoxes *__restrict__ out) {
    constexpr int R = 8;
    __shared__ float scratch[5 * sweep::THREADS / 32];
    const int blk = blockIdx.x;
    if (blk >= p.blk_off[p.n_groups]) return;
    int j = 0;
    while (blk >= p.blk_off[j + 1]) ++j;
    float rp[R], rq[R], rl[R];
    int kp[R];
    unsigned valid;
    load_shadow_bundle<R>(p, blk, threadIdx.x >> 5, j, rp, rq, rl, kp, valid);
    cull::Box wb, cb;
    cull::bundle_boxes<R>(rp, rq, rl, scratch, wb, cb);
    if ((threadIdx.x & 31) == 0) out[blk].warp[threadIdx.x >> 5] = wb;
    if (threadIdx.x == 0) out[blk].cta = cb;
}

struct BlockLists {
    const cull::BlockBoxes *boxes;
    const unsigned long long *keys; // sorted (block*16+warp)<<tri_bits|triangle survivors of phase A
    unsigned long long n_keys;
    int tri_bits;
};

// phase B.  Work item = a fixed-size segment of the sorted key array, taken by ONE warp (so a warp with a very
// long survivor list — e.g. shadow rays that straddle a Morton-order jump and have a huge box — is spread over
// many warps of the grid, and short lists share one); a key's high part names the (ray block, warp) whose rays
// the executing warp loads when it changes.
constexpr unsigned long long CULL_SEG = 2048;

struct PrimaryBundles {
    PrimaryCullParams p;
    __device__ __forceinline__ const float4 *table_of(int) const { return p.table; }
    template <int R>
    __device__ __forceinline__ void load(int blk, int warp, float (&rp)[R], float (&rq)[R], float (&rl)[R], int (&kp)[R],
                                         unsigned &valid) const {
        load_primary_bundle<R>(p, blk, warp, rp, rq, rl, kp, valid);
    }
};
struct ShadowBundles {
    ShadowCullParams p;
    __device__ __forceinline__ int group_of(int blk) const {
        int j = 0;
        while (blk >= p.blk_off[j + 1]) ++j;
        return j;
    }
    __device__ __forceinline__ const float4 *table_of(int blk) const {
        return cull::group_table(p.tables, p.allcand, p.table_stride, NFACE, group_of(blk));
    }
    template <int R>
    __device__ __forceinline__ void load(int blk, int warp, float (&rp)[R], float (&rq)[R], float (&rl)[R], int (&kp)[R],
                                         unsigned &valid) const {
        load_shadow_bundle<R>(p, blk, warp, group_of(blk), rp, rq, rl, kp, valid);
    }
};

template <class Bundles>
__device__ __forceinline__ void cull2_body(const Bundles &bd, const BlockLists bl, int *work, const cull::Emitter em,
                                           sweep::Counters *counters) {
    constexpr int R = 8, NW = sweep::THREADS / 32;
    __shared__ cull::WarpListSmem lsm;
    const int lane = threadIdx.x & 31, ws = threadIdx.x >> 5;
    const unsigned long long n_items = (bl.n_keys + CULL_SEG - 1) / CULL_SEG;
    const unsigned tri_mask = (1u << bl.tri_bits) - 1u;
    unsigned d_l1 = 0;
    cull::WarpChunk wc{0, cull::CHUNK}; // no chunk yet
    int cur = -1;                       // (block, warp) whose rays this warp holds
    const float4 *tab = nullptr;
    float rp[R], rq[R], rl[R];
    int kp[R];
    unsigned valid = 0;
    cull::Box lane_box{};
    for (;;) {
        int it = 0;
        if (lane == 0) it = atomicAdd(work, 1);
        const unsigned long long item = (unsigned long long)__shfl_sync(0xffffffffu, it, 0);
        if (item >= n_items) break;
        const unsigned long long pos = item * CULL_SEG, end = min(bl.n_keys, pos + CULL_SEG);
        for (unsigned long long i0 = pos; i0 < end; i0 += 32) {
            const int n = (int)min((unsigned long long)32, end - i0);
            __syncwarp(); // the previous step's rows are consumed
            if (lane < n) { // gather: one key and its row per lane
                const unsigned long long key = bl.keys[i0 + lane];
                const int kb = (int)(key >> bl.tri_bits);
                const float4 *t = kb == cur ? tab : bd.table_of(kb / NW);
                const unsigned tri = (unsigned)key & tri_mask;
                lsm.key[ws][lane] = key;
                lsm.row[ws][3 * lane] = __ldg(&t[3 * (size_t)tri]);
                lsm.row[ws][3 * lane + 1] = __ldg(&t[3 * (size_t)tri + 1]);
                lsm.row[ws][3 * lane + 2] = __ldg(&t[3 * (size_t)tri + 2]);
            }
            __syncwarp();
#pragma unroll 1
            for (int e = 0; e < n; ++e) {
                const unsigned long long key = lsm.key[ws][e];
                const int kb = (int)(key >> bl.tri_bits);
                if (kb != cur) { // warp-uniform
                    cur = kb;
                    tab = bd.table_of(kb / NW);
                    bd.template load<R>(kb / NW, kb % NW, rp, rq, rl, kp, valid);
                    lane_box = cull::lane_box_of<R>(rp, rq, rl);
                }
                const float4 rb = lsm.row[ws][3 * e], rc = lsm.row[ws][3 * e + 1], rd = lsm.row[ws][3 * e + 2];
                unsigned mask = 0;
                ++d_l1;
                if (!(cull::box_sign(rb, rc, rd, lane_box) >> 31)) { // the box of this lane's own R rays
#pragma unroll
                    for (int r = 0; r < R; ++r)
                        mask |= ((unsigned)sweep::edge_pass(rb, rc, rd, rp[r], rq[r]) & (unsigned)(rb.w <= rl[r])) << r;
                    mask &= valid;
                }
                if (__ballot_sync(0xffffffffu, mask != 0) == 0) continue;
                cull::emit_pairs<R>(em, wc, mask, kp, (unsigned)key & tri_mask);
            }
        }
    }
    cull::chunk_close(em, wc);
    if (lane == 0) atomicAdd(&counters->cull_l1, (unsigned long long)d_l1);
}

__global__ void __launch_bounds__(sweep::THREADS, 2) primary_cull2_kernel(const PrimaryCullParams p, const BlockLists bl) {
    cull2_body(PrimaryBundles{p}, bl, p.work, p.em, p.counters);
}

__global__ void __launch_bounds__(sweep::THREADS, 2) shadow_cull2_kernel(const ShadowCullParams p, const BlockLists bl) {
    cull2_body(ShadowBundles{p}, bl, p.work, p.em, p.counters);
}

// ---------------------------------------------------------------------------------
// main.cpp:679-684: x>1 -> 1, int(x*255) truncation.  u8 cannot carry the
// reference's negative / INT_MIN (NaN) prints: those clamp to 0.
__device__ __forceinline__ unsigned quant(float x) {
    x = (x > 1.f) ? 1.f : x;
    const float y = __fmul_rn(x, 255.f);
    if (!(y >= 0.f)) return 0u;
    const int q = (int)y;
    return (unsigned)(q > 255 ? 255 : q);
}

// 16 pixels per thread: 48 contiguous bytes = three 128-bit stores, fully coalesced
__global__ void quantise_kernel(const float *__restrict__ accum, int n_px, uint8_t *__restrict__ rgb8) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int k0 = g * 16;
    if (k0 >= n_px) return;
    if (k0 + 16 <= n_px && ((uintptr_t)rgb8 & 15u) == 0) {
        unsigned bytes[48];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 *src = reinterpret_cast<const float4 *>(accum + (size_t)c * n_px + k0);
            const bool al = (((uintptr_t)src) & 15u) == 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float4 f;
                if (al)
                    f = src[q];
                else {
                    const float *s1 = accum + (size_t)c * n_px + k0 + 4 * q;
                    f = make_float4(s1[0], s1[1], s1[2], s1[3]);
                }
                bytes[(4 * q + 0) * 3 + c] = quant(f.x);
                bytes[(4 * q + 1) * 3 + c] = quant(f.y);
                bytes[(4 * q + 2) * 3 + c] = quant(f.z);
                bytes[(4 * q + 3) * 3 + c] = quant(f.w);
            }
        }
        uint4 *dst = reinterpret_cast<uint4 *>(rgb8 + (size_t)k0 * 3);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            uint4 o;
            unsigned *ow = &o.x;
#pragma unroll
            for (int wv = 0; wv < 4; ++wv) {
                const int b = (q * 4 + wv) * 4;
                ow[wv] = bytes[b] | (bytes[b + 1] << 8) | (bytes[b + 2] << 16) | (bytes[b + 3] << 24);
            }
            dst[q] = o;
        }
    } else {
        for (int k = k0; k < min(k0 + 16, n_px); ++k)
            for (int c = 0; c < 3; ++c) rgb8[(size_t)k * 3 + c] = (uint8_t)quant(accum[(size_t)c * n_px + k]);
    }
}

// extension: sum of the per-sample colours (sample order fixed => deterministic), final mean
__global__ void accumulate_kernel(const float *__restrict__ accum, float *__restrict__ total, size_t n3, int first, int last,
                                  float n_samples) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n3) return;
    float v = first ? accum[i] : __fadd_rn(total[i], accum[i]);
    if (last) v = __fdiv_rn(v, n_samples);
    total[i] = v;
}

// hit mask in local pixel order (= the reference's scan order) for the mt19937 replay
__global__ void hitmask_kernel(const int *__restrict__ hit_tri, int n_px, uint8_t *__restrict__ mask) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_px) mask[k] = hit_tri[k] >= 0;
}

// rank 0 after the gather: rank r's buffer holds its bands back to back
__global__ void assemble_bands_kernel(const uint8_t *__restrict__ gathered, uint8_t *__restrict__ frame, int W, int H,
                                      int band_rows, int band_count, int rows_pad) {
    const size_t row_bytes = (size_t)W * 3;
    const size_t total = row_bytes * H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int pr = (int)(i / row_bytes);
        const size_t x = i - (size_t)pr * row_bytes;
        const int gb = pr / band_rows;
        const int rank = gb % band_count;
        const int lb = gb / band_count;
        const int lr = lb * band_rows + (pr - gb * band_rows);
        frame[i] = gathered[((size_t)rank * rows_pad + lr) * row_bytes + x];
    }
}

}  // namespace trk
