// sweep.cuh — the O(rays x triangles) sweeps (closest hit and first-occluder),
// B200-native formulation.
//
// What the reference does per (ray, triangle) pair: full Moller-Trumbore with
// a double-precision divide (ray_triangle.h:7-57, ~52 flop).  What this kernel
// does per pair: half a packed add and half a three-input min (4., hot rows), plus
// 8 ops per thread and triangle (12 with a mean q); the closest-hit and shadow sweeps do nothing per pair, one packed add
// per thread and triangle on the thread's extreme rays (segment_pass).  The saving comes from these observations.
//
//  1. Every sweep is a bundle of rays through ONE common point.  Primary rays
//     all start at the eye (camera.h:31-34).  A shadow ray runs from the hit
//     point to the sampled light point, and the reference's light "sample" is
//     always exactly a light vertex (main.cpp:749-754: v0=v1=v2), so all
//     shadow rays toward the same light vertex lie on lines through that
//     vertex.  For a fixed point O and triangle (v0,v1,v2), with a=v0-O,
//     e1=v1-v0, e2=v2-v0, the three Moller-Trumbore numerators are LINEAR in
//     the line direction d:   u' = d.(a x e2)   v' = d.(e1 x a)
//     w' = det-u'-v' = d.(e2 x e1 - a x e2 - e1 x a),  and the side of the
//     plane O lies on, s = sign(e2.(e1 x a)), is a per-triangle constant.
//     A line through O can only hit the triangle if s*u', s*v', s*w' >= 0.
//
//  1b. Directions through one point have two degrees of freedom.  Each ray group
//     uses a parametrisation d' = p*U + q*V + W (the image plane for primary
//     rays: U,V,W = horizontal, vertical, llc-origin and (p,q) = the reference's
//     own (s,t); a cube face around a light vertex for shadow rays), so each
//     edge function becomes AFFINE in (p,q):  u'(p,q) = p*(U.B) + q*(V.B) + (W.B + K|d'|max).
//
//  2. The test above is used as a CONSERVATIVE FILTER only: K bounds every
//     rounding difference between this evaluation and the reference's own
//     float/double evaluation (see build_origin_table), so a pair the
//     reference would accept is never filtered out.  Pairs that pass (a few
//     per ray out of N) are re-evaluated in the reference's exact arithmetic
//     (strict_math.cuh), so closest-hit ties, the `first occluder in order`
//     rule and all the chaotic self-shadow decisions come out bit-identical
//     to the serial path.  The strict results are MERGED IN GLOBAL MEMORY with
//     one 64-bit atomicMin per accepted pair:
//        closest hit  key = t bits << 32 | index   (cpp_intersect keeps the lexicographic
//                                                   minimum of (t, index): t2 >= t rejects)
//        occluder     key = index << 32  | t2 bits (occlusion() returns the lowest index)
//     so the sweep keeps NO per-ray state in shared memory: a CTA's shared
//     memory is the table-tile pipeline only.
//
//  3. The R rays of a thread share q.  Closest-hit ray blocks are screen tiles in which a
//     thread holds R consecutive pixels of one image row: same q exactly (MODE_SHAREDQ).
//     Shadow-ray lists are sorted by q, then by p in short serpentine stripes; a thread takes R consecutive
//     rays and evaluates the q-dependent terms at qbar with |B|*qdelta added, qdelta >= max|q_r - qbar|, which is
//     >= every ray's own term, so the test stays a necessary condition (MODE_QBAR; also used
//     for jittered primary samples, whose q lie inside one stratum).
//
//  4. SPAN form.  For rays that share q, the three affine rows are half-lines in p: with
//     beta = -B/A, gamma = -C/A (divided once per (origin, triangle) in FP64) row i says
//     p >= q*beta_i + gamma_i where A_i > 0 and p <= q*beta_i + gamma_i where A_i < 0.  A
//     triangle has two lower bounds and one upper bound or the reverse, so the table row is
//     two lower + two upper bounds = 32 bytes, the thread evaluates the four at its q and keeps
//     the binding ones, and each PAIR is a two-sided span test (below).  The tables store the rows
//     in HOT form (hot_row): the test's +1s, the clamp and the margin folded into the constants, so
//     the thread's set-up is 4 FFMA + 2 FMNMX3 + 2 FADD per triangle.
//     MODE_OWNQ (every ray its own q) keeps the 48-byte three-row table: 3 x (A,B,C,-).
//
// Mapping to the SM (choices measured with tools/sweep_mb2-4.cu, see DESIGN.md):
//  * rows stream HBM/L2 -> shared memory in tiles of 256 triangles via TMA 1-D bulk copies
//    (cp.async.bulk + mbarrier complete_tx, UBLKCP in SASS), STAGES deep;
//  * every lane of every warp reads the SAME row at the same time, so the two LDS.128 per
//    triangle are pure broadcasts, amortised over R rays per thread held in registers
//    (R = 64 closest hit, 32 any-hit);
//  * closest hit (MODE_SHAREDQ) and any-hit (MODE_QBAR): one two-sided test on the thread's least and greatest 2*S*p per
//    triangle (segment_pass);
//  * jittered primary samples: each pair is ONE interval test |2*S*p + nc2| <= h2 (hot rows, below): per two pairs one packed
//    FADD2 and one FMNMX3 running minimum, no saturation, no integer op.  History on this part
//    (cycles per pair, closest hit): round 1 sign bits through LOP3 on the half-rate ALU pipe 7.9,
//    three saturating rows with a product accumulate 6.8, span form with two saturating adds 4.0;
//  * the inner loop has NO per-triangle branch: a batch of 16 triangles yields one verdict bit per
//    triangle; candidates (a few per ray per sweep) then go through a warp-wide pass: the flagged triangles'
//    (owner lane, ray, triangle) pairs are queued in shared memory and drained one pair per lane, so the
//    strict evaluations of a thread's R rays no longer serialise on that thread;
//  * NO block-wide barrier per tile in either sweep: every warp counts itself out of a
//    tile stage (shared-memory atomicAdd) and the last one issues the refill, so warps
//    run up to STAGES-1 tiles apart.  An any-hit warp whose rays all have their occluder
//    stops evaluating (it only keeps the stage counts going);
//  * SWEEP_NT threads per CTA, SWEEP_MINB CTAs per SM (launch bounds cap the registers; the 64-ray closest-hit
//    kernel has its own, SWEEP_MINB64 in kernels.cuh).
#pragma once
#include <cmath>
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "strict_math.cuh"

#ifndef SWEEP_NT
#define SWEEP_NT 128
#endif
#ifndef SWEEP_MINB
#define SWEEP_MINB 4
#endif
#ifndef SWEEP_STAGES
#define SWEEP_STAGES 4
#endif

namespace sweep {

constexpr int TILE = 256;          // triangles per shared-memory stage (48-byte rows: 12 KB)
constexpr int BATCH = 16;          // triangles between candidate checks of the three-row form
constexpr int STAGES = SWEEP_STAGES; // TMA pipeline depth
constexpr int THREADS = 512;       // threads per CTA of the bundle-cull kernels (cull.cuh)
constexpr int NT = SWEEP_NT;       // threads per CTA of the default sweeps
constexpr int MINB = SWEEP_MINB;   // CTAs per SM of the default sweeps
constexpr float CK = 64.f;         // safety factor of the filter margins (units of FLT_EPSILON)
constexpr uint32_t TILE_BYTES = TILE * 3 * sizeof(float4); // 48-byte rows (MODE_OWNQ, bundle-cull mode, tools/)
constexpr float SPAN_S = 65536.f;  // span rows: row units per unit of p (a power of two: p * SPAN_S is exact)
constexpr float SPAN_OPEN = 1e30f; // span rows: an unused bound

// MODE_OWNQ sweeps the 48-byte three-row table (every ray its own q: jittered primary rays); MODE_SHAREDQ and MODE_QBAR
// sweep the 32-byte SPAN table (4. below)
enum { MODE_OWNQ = 0, MODE_SHAREDQ = 1, MODE_QBAR = 2 };
template <int MODE>
struct Rows {
    static constexpr int N = MODE == MODE_OWNQ ? 3 : 2;                // float4 per triangle
    static constexpr uint32_t BYTES = TILE * N * sizeof(float4);      // per staged tile
};

// ---- mbarrier / TMA bulk-copy primitives (sm_90+; sm_100a here) -------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float4 lds128_opaque(const float4 *p) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
    return v;
}

// ---- shared memory of one sweep CTA: the table-tile pipeline and each warp's candidate queue -------------------
constexpr int QCAP = 32; // candidate pairs per warp queue: one per lane and drain
template <int ROWS> // float4 per triangle of the table the kernel sweeps: 2 (span rows) or 3 (three-row table)
struct __align__(128) SmemT {
    float4 tile[STAGES][TILE * ROWS];
    uint64_t full_bar[STAGES];
    int consumed[STAGES]; // warps that have finished the tile in this stage
    int blk, seg, slice;  // the work item the CTA is on
    unsigned queue[NT / 32][QCAP];             // candidate pairs: ray | owner lane << 6 | triangle in tile << 11 | filt << 19
    unsigned long long qdone[NT / 32][32];     // any-hit: rays of each owner lane accepted during a drain (zero between drains)
};
using Smem = SmemT<3>;

struct Counters {
    unsigned long long tests_primary, tests_shadow, strict_evals, tests_shadow_ref, n_hits, filter_misses;
    unsigned long long cull_l0, cull_l1, cull_tiles_any, cull_tiles_fallback; // bundle-cull diagnostics
    unsigned long long cull_overflow; // bundle-cull: a candidate buffer was too small (the frame is rejected)
    unsigned long long pipeline_errors; // validation mode: staged tiles that differed from their source (must be 0)
    // shadow_light_kernel time split, SM cycles summed over CTAs (thread 0's clock; TRACER_SHADOW_DIAG prints them):
    // inside work items, waiting at grid barriers, compaction passes, everything else (work-queue pops, prefix sums)
    unsigned long long cyc_items, cyc_barrier, cyc_compact, cyc_total, n_items, n_runs;
    // shadow_light_kernel: (thread, triangle) verdicts the hot loop flagged, and (ray, triangle) pairs queued for the drain
    unsigned long long n_flagged, n_queued;
    // shadow_light_kernel: SM cycles of the candidate path (from a batch's first flag to its last drain), lane 0 of every warp
    unsigned long long cyc_cand;
};

template <int ROWS>
__device__ __forceinline__ void smem_init(SmemT<ROWS> &sm) {
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&sm.full_bar[s], 1), sm.consumed[s] = 0;
        fence_barrier_init();
    }
    if (threadIdx.x < NT) sm.qdone[threadIdx.x >> 5][threadIdx.x & 31] = 0;
    __syncthreads();
}

// One 48-byte row triple per triangle: rb = (A,B,C,-) of s*u', rc of s*v', rd of s*w', in SATURATING FORM
// (kernels.cuh, build_origin_table): a pair the reference could accept evaluates to >= 1 on all three rows.
// Per-ray test used by the (rare) candidate path: bit clear = some row < 1.
__host__ __device__ __forceinline__ bool edge_pass(const float4 rb, const float4 rc, const float4 rd, float p, float q) {
    const float x = fmaf(p, rb.x, fmaf(q, rb.y, rb.z));
    const float y = fmaf(p, rc.x, fmaf(q, rc.y, rc.z));
    const float z = fmaf(p, rd.x, fmaf(q, rd.y, rd.z));
    return fminf(fminf(x, y), z) >= 1.f;
}
// Sign word of the three edge functions at the ray parameters (p,q): sign bit clear <=> all three >= 0 (bundle-cull
// mode and the LOP3 form of the hot loop; only looser than the saturating test on the same rows).
__device__ __forceinline__ unsigned edge_sign(const float4 rb, const float4 rc, const float4 rd, float p, float q) {
    const float x = fmaf(p, rb.x, fmaf(q, rb.y, rb.z));
    const float y = fmaf(p, rc.x, fmaf(q, rc.y, rc.z));
    const float z = fmaf(p, rd.x, fmaf(q, rd.y, rd.z));
    return __float_as_uint(x) | __float_as_uint(y) | __float_as_uint(z);
}

// QBAR form: the R rays of a thread are evaluated with ONE q-term per edge row.  With qbar the thread's mean q and
// qdelta >= max |q_r - qbar| the row value p*A + (qbar*B + |B|*qdelta + C) is >= the ray's own p*A + q_r*B + C, so
// the test stays a necessary condition while the inner term costs 2 FFMA per thread instead of 1 per ray
// (shadow rays sorted by q: qdelta ~ 1e-6, far inside the margin K already in C).
__device__ __forceinline__ float qterm_qbar(const float4 row, float qbar, float qdelta) {
    return fmaf(fabsf(row.y), qdelta, fmaf(qbar, row.y, row.z));
}

// ---- three-row form (MODE_OWNQ; also tools/sweep_mb2,3.cu): BATCH triangles of a staged tile against the R rays of this thread ---
// Everything runs in the FMA pipe (measured on B200, tools/sweep_mb3.cu: a scalar FMA-pipe instruction costs ~1.3
// issue cycles, a LOP3/SHF/FMNMX on the half-rate ALU pipe ~2, and the two do not overlap in this loop):
//   x' = sat(p*A_u + q_u)   y' = sat(p*A_v + q_v)   z' = sat(p*A_w + q_w)      3 FFMA.SAT per pair
//   acc += (x' * y') * z'                                                        1 FMUL + 1 FFMA per pair (packed: below)
// A candidate pair contributes exactly 1, any other pair something in [0,1), so after GROUP triangles
// "sum of the accumulators >= 1" is a necessary condition for the group to hold a candidate.  Straight-line FFMA /
// FMUL / LDS.128 stream, no branch per triangle.  Returns bit g set = triangles [g*GROUP, (g+1)*GROUP) may hold one.
// The conjunction runs on ray PAIRS in packed form (FMUL2 + FFMA2, fma.rn.f32x2): on this part a packed instruction
// costs ~2.2 issue cycles for two FMAs against ~2.6 for two scalar ones; the saturating row evaluations stay scalar
// (fma.sat has no f32x2 form).  Measured (tools/sweep_mb3.cu, shared q): scalar conjunction 5.05 Tpairs/s at R = 8,
// packed 5.41 at R = 8 and 5.71 at R = 12.
template <int R>
struct Batch {
    static_assert(R % 2 == 0, "rays are evaluated in pairs");
    static constexpr int GROUP = R >= 12 ? 4 : 8;                   // triangles per accumulator group
    static constexpr int NACC = R >= 16 ? 4 : R >= 12 ? 3 : (R >= 4 ? 2 : 1); // independent packed accumulators (FFMA2 chains) per group
    static_assert(R <= 32, "ray masks of the three-row form are 32 bits wide");
    static constexpr int NGROUPS = BATCH / GROUP;
};

template <int R, int MODE>
__device__ __forceinline__ unsigned eval_batch(const float4 *__restrict__ tp, const float (&rp)[R], const float (&rq)[R], float qbar,
                                               float qdelta) {
    constexpr int GROUP = Batch<R>::GROUP, NA = Batch<R>::NACC;
    unsigned cand = 0;
#pragma unroll
    for (int g = 0; g < BATCH / GROUP; ++g) {
        float2 acc[NA];
#pragma unroll
        for (int a = 0; a < NA; ++a) acc[a] = make_float2(0.f, 0.f);
#pragma unroll
        for (int kk = 0; kk < GROUP; ++kk) {
            const int k = g * GROUP + kk;
            const float4 rb = tp[3 * k], rc = tp[3 * k + 1], rd = tp[3 * k + 2];
            if (MODE == MODE_OWNQ) {
#pragma unroll
                for (int r = 0; r < R; r += 2) {
                    const float2 x = make_float2(__saturatef(fmaf(rp[r], rb.x, fmaf(rq[r], rb.y, rb.z))),
                                                 __saturatef(fmaf(rp[r + 1], rb.x, fmaf(rq[r + 1], rb.y, rb.z))));
                    const float2 y = make_float2(__saturatef(fmaf(rp[r], rc.x, fmaf(rq[r], rc.y, rc.z))),
                                                 __saturatef(fmaf(rp[r + 1], rc.x, fmaf(rq[r + 1], rc.y, rc.z))));
                    const float2 z = make_float2(__saturatef(fmaf(rp[r], rd.x, fmaf(rq[r], rd.y, rd.z))),
                                                 __saturatef(fmaf(rp[r + 1], rd.x, fmaf(rq[r + 1], rd.y, rd.z))));
                    acc[(r / 2) % NA] = __ffma2_rn(__fmul2_rn(x, y), z, acc[(r / 2) % NA]);
                }
            } else {
                const float qx = MODE == MODE_QBAR ? qterm_qbar(rb, qbar, qdelta) : fmaf(rq[0], rb.y, rb.z);
                const float qy = MODE == MODE_QBAR ? qterm_qbar(rc, qbar, qdelta) : fmaf(rq[0], rc.y, rc.z);
                const float qz = MODE == MODE_QBAR ? qterm_qbar(rd, qbar, qdelta) : fmaf(rq[0], rd.y, rd.z);
#pragma unroll
                for (int r = 0; r < R; r += 2) {
                    const float2 x = make_float2(__saturatef(fmaf(rp[r], rb.x, qx)), __saturatef(fmaf(rp[r + 1], rb.x, qx)));
                    const float2 y = make_float2(__saturatef(fmaf(rp[r], rc.x, qy)), __saturatef(fmaf(rp[r + 1], rc.x, qy)));
                    const float2 z = make_float2(__saturatef(fmaf(rp[r], rd.x, qz)), __saturatef(fmaf(rp[r + 1], rd.x, qz)));
                    acc[(r / 2) % NA] = __ffma2_rn(__fmul2_rn(x, y), z, acc[(r / 2) % NA]);
                }
            }
        }
        float sum = 0.f;
#pragma unroll
        for (int a = 0; a < NA; ++a) sum += acc[a].x + acc[a].y;
        if (sum >= 1.f) cand |= 1u << g;
    }
    return cand;
}

// ---- SPAN form -------------------------------------------------------------------------------------------------------
// For rays that share q the three affine rows p*A_i + (q*B_i + C_i) >= 0 are half-lines in p: p >= c_i(q) where A_i > 0,
// p <= c_i(q) where A_i < 0, with c_i(q) = q*beta_i + gamma_i, beta = -B/A, gamma = -C/A (divided once per (origin,
// triangle) in FP64, kernels.cuh: build_origin_table).  A triangle in front of the parametrisation plane has two lower
// bounds and one upper bound or the reverse, so the 32-byte span row holds two of each, already in row units and with the
// +1 of the saturating test folded in:
//     lo = (Bl1, Cl1, Bl2, Cl2):  a_i = q*Bl_i + Cl_i = 1 - S*(c_i(q) - margin)      ax = min(a_1, a_2)
//     hi = (Bu1, Cu1, Bu2, Cu2):  b_i = q*Bu_i + Cu_i = 1 + S*(c_i(q) + margin)      ay = min(b_1, b_2)
// and a pair is a candidate iff  x = sat(S*p + ax)  and  y = sat(ay - S*p)  are both exactly 1.  Per thread and triangle:
// 4 FFMA + 2 FMNMX (8 FFMA in MODE_QBAR, which adds |B|*qdelta to every bound); per PAIR: 2 FADD.SAT + half a packed
// FFMA2 (acc += x*y), against 3 FFMA.SAT + FMUL2/2 + FFMA2/2 of the three-row form.  Measured (tools/sweep_mb4.cu, B200):
// 8.9 Tpairs/s at 16 rays per thread, 9.3 at 24, 9.5 at 32, against 5.7 for the three-row loop at 12.
__host__ __device__ __forceinline__ void span_terms(const float4 lo, const float4 hi, float q, float &ax, float &ay) {
    ax = fminf(fmaf(q, lo.x, lo.y), fmaf(q, lo.z, lo.w));
    ay = fminf(fmaf(q, hi.x, hi.y), fmaf(q, hi.z, hi.w));
}
__host__ __device__ __forceinline__ void span_terms_qbar(const float4 lo, const float4 hi, float qbar, float qdelta, float &ax, float &ay) {
    ax = fminf(fmaf(fabsf(lo.x), qdelta, fmaf(qbar, lo.x, lo.y)), fmaf(fabsf(lo.z), qdelta, fmaf(qbar, lo.z, lo.w)));
    ay = fminf(fmaf(fabsf(hi.x), qdelta, fmaf(qbar, hi.x, hi.y)), fmaf(fabsf(hi.z), qdelta, fmaf(qbar, hi.z, hi.w)));
}
// per-ray test of the (rare) candidate path: ps = p * SPAN_S, the ray's own q
__host__ __device__ __forceinline__ bool span_pass(const float4 lo, const float4 hi, float ps, float q) {
    float ax, ay;
    span_terms(lo, hi, q, ax, ay);
    return fminf(ps + ax, ay - ps) >= 1.f;
}

// ---- INTERVAL form of the span test (the hot loop of MODE_SHAREDQ and MODE_QBAR) -----------------------------------------
// For one thread's shared q a triangle's span row is ONE interval of S*p:  x = y = 1  <=>  1 - ax <= S*p <= ay - 1, i.e.
// |S*p - c| <= h with c the interval's centre and h its half width.  Per thread and triangle (span_interval):
//     lo = max(1 - ax, -SPAN_BOX)   hi = min(ay - 1, SPAN_BOX)   nc = -(lo + hi)/2   h = (hi - lo)/2 + SPAN_DELTA
// and per ray PAIR one packed FADD2 {S*p_r, S*p_r+1} + nc and one three-input FMNMX3 m = min(m, |e_r|, |e_r+1|) (|.| is
// an operand modifier): 1 FMA-pipe instruction per two pairs, against 2 FFMA.SAT + half an FFMA2 per pair of the
// saturating form, whose .sat has no packed f32x2 form on sm_100a.  After the R rays, m <= h is the triangle's verdict.
//
// SPAN_DELTA makes the interval test pass every pair the saturating test passes (which the table's margins make pass every
// pair the reference accepts).  Let u = 2^-24 (float unit roundoff), P = SPAN_BOX, |S*p| <= S*SPAN_PMAX = P - 1 for every
// ray swept in span form (kernels.cuh).  A pair with fl(S*p + ax) >= 1 and fl(ay - S*p) >= 1 has, exactly,
// S*p >= (1 - ax) - u/2 and S*p <= (ay - 1) + u/2 (a sum rounds up to 1 from 1 - u/2 at the least).  Then:
//   lo: either -P (< S*p) or fl(1 - ax) > -P, and then 1 - ax lies in (-P, P): lo <= S*p + e, e = u/2 + u*P; same for hi.
//       So lo, hi lie in [-P, P] and S*p in [lo - e, hi + e]: |S*p - (lo+hi)/2| <= (hi-lo)/2 + e.
//   nc: one rounding of a sum of magnitude <= 2P (the halving is exact): |nc + (lo+hi)/2| <= u*P.
//   h:  fl(hi - lo) is off by <= 2u*P, the fma's one rounding by <= u*(P + SPAN_DELTA): h >= (hi-lo)/2 + SPAN_DELTA - 2.1u*P.
//   e = fl(S*p + nc): S*p + nc has magnitude <= 2P + 1, one rounding <= 2.1u*P.
// so |e| <= (hi-lo)/2 + u/2 + u*P + u*P + 2.1u*P <= h whenever SPAN_DELTA >= 6.3u*P; SPAN_DELTA = 8 FLT_EPSILON * P = 16u*P
// (0.066 row units, 1/250 of a 3840-wide frame's pixel).  The clamp is what bounds every term by P: without it an open
// bound (SPAN_OPEN = 1e30) would put c near 5e29 and round S*p away.  Padding rows (ax = -SPAN_OPEN) give lo = 1e30 > hi, so
// h ~ -5e29 and the triangle is never a candidate; always-candidate rows (ax = ay = SPAN_OPEN) give c = 0, h > P > |S*p|.
// NaN cannot reach h (fminf/fmaxf drop it) and a NaN |e| is ignored by the minimum, so neither can hide a candidate.
constexpr float SPAN_BOX = SPAN_S * 1.0625f + 1.f;                  // S * SPAN_PMAX + 1 (kernels.cuh checks the match)
constexpr float SPAN_DELTA = 8.f * 1.1920928955078125e-7f * SPAN_BOX; // 8 FLT_EPSILON * SPAN_BOX
#ifndef SWEEP_SPAN_BATCH
#define SWEEP_SPAN_BATCH 16
#endif
constexpr int SPAN_BATCH = SWEEP_SPAN_BATCH; // triangles between candidate checks of the interval form (<= 32: a bit each)
static_assert(SPAN_BATCH <= 32 && TILE % SPAN_BATCH == 0, "one verdict bit per triangle of a batch");

// (ax, ay) from span_terms / span_terms_qbar -> the negated centre and the widened half width of the interval of S*p
// (box, delta: SPAN_BOX, SPAN_DELTA; other values only in the test hook tracer__interval_pass)
// span_terms, span_pass and span_interval are the reference form of the span test: the tables store the HOT form of the
// same rows (hot_row below), which is proven against them.
__host__ __device__ __forceinline__ void span_interval(float ax, float ay, float &nc, float &h, float box = SPAN_BOX,
                                                      float delta = SPAN_DELTA) {
    const float lo = fmaxf(1.f - ax, -box), hi = fminf(ay - 1.f, box);
    nc = -0.5f * (lo + hi);
    h = fmaf(0.5f, hi - lo, delta);
}
// the interval test of one pair, as the hot loop evaluates it (ps = p * SPAN_S)
__host__ __device__ __forceinline__ bool interval_pass(float nc, float h, float ps) { return fabsf(ps + nc) <= h; }

// min(a, b, c): one FMNMX3 on sm_100 (NaN inputs are dropped, as fminf drops them)
__host__ __device__ __forceinline__ float fmin3(float a, float b, float c) {
#ifdef __CUDA_ARCH__
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
#else
    return fminf(fminf(a, b), c);
#endif
}
// min(m, |a|, |b|): one FMNMX3 with both absolute values as operand modifiers (sm_100)
__device__ __forceinline__ float fmin3_abs(float m, float a, float b) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(m), "f"(fabsf(a)), "f"(fabsf(b)));
    return d;
}

// ---- HOT rows: the span row as the tables store it (the hot loop of MODE_SHAREDQ and MODE_QBAR) ---------------------------
// The +1 of the saturating test, the clamp and the interval's margin are folded into the row.  build_origin_table stores
// span_rows' row with both constants of every bound shifted:  C' = C - (1 - HOT_DELTA), rounded toward +inf (hot_row), the
// q coefficients unchanged.  A thread with shared q then forms, per triangle,
//     A = min3(q*Bl1 + Cl1', q*Bl2 + Cl2', HOT_CLAMP) ~ -lo + delta     B = min3(q*Bu1 + Cu1', q*Bu2 + Cu2', HOT_CLAMP) ~ hi + delta
//     nc2 = A - B  (the negated centre of the interval of 2*S*p)          h2 = A + B  (its full width, 2*delta included)
// and per ray pair |2*S*p_r + nc2| <= h2: the two 1s cancel, delta is in the row and the clamp is the third input of the
// FMNMX3.  Rays hold 2*S*p (exact: a power of two).  Per thread and triangle 4 FFMA + 2 FMNMX3 + 2 FADD (MODE_QBAR: 8 FFMA,
// the |B|*qdelta widening kept, with qdelta scaled by HOT_QD_SCALE), against 4 FFMA + 2 FMNMX + 8 for span_interval.
//
// Why every pair the saturating test passes (fl(S*p + ax) >= 1 and fl(ay - S*p) >= 1, ax and ay from span_terms or
// span_terms_qbar on the unshifted row) passes the hot test.  u = 2^-24, C = HOT_CLAMP, s = 1 - delta, P0 = S*SPAN_PMAX =
// C - 1 >= |S*p|, Q = C + 2.  Take one lower bound, a = fl(G) its saturating value, G = |Bl|*qd + t0 exactly, t0 = fl(z),
// z = q*Bl + Cl (qd = 0 and t0 = z with a shared q), and its hot value A_i = fl(G'), G' = |Bl|*qd' + t, t = fl(q*Bl + Cl').
//   the pass: a >= ax and fl(S*p + ax) >= 1 give a >= 1 - u/2 - S*p (a sum rounds to 1 from 1 - u/2 at the least).
//   shift:    Cl' >= Cl - s exactly (rounded up), so t >= fl(z - s) >= z - s - u|z| - u, and t0 <= z + u|z|.
//   qdelta:   qd' = fl(qd * (1 + 2^-20)) >= qd (1 + 14u), and |z| <= (1 + 2u)(|G| + |Bl|*qd), so
//             G' - G >= 14u|Bl|qd - s - u - 2(1 + 2u)u(|G| + |Bl|qd) >= -s - u - 2.1u|G|.
//   a <= Q:   |G - a| <= uQ, G' >= a - s - 3.2uQ - u, and A_i = fl(G') >= min(C, a - s - 4.2uQ - 3u).
//   a > Q:    G > Q(1 - u), G' > C + 1 - 4.3uQ > C, A_i >= C.
// So A = min3(A_1, A_2, C) >= min(C, -S*p + delta - e) = -S*p + delta - e, e = 4.2uQ + 3.5u (C >= P0 + delta); the same
// for B >= S*p + delta - e, and |A|, |B| <= C.  Then, with one rounding each (u times a magnitude <= 2C):
//   h2 >= A + B - 2uC;   |2*S*p + A - B| <= A + B - 2*delta + 2e;   nc2 is off by <= 2uC and the FADD2 by <= 2uC(1 + u),
// so |fl(2*S*p + nc2)| <= h2 whenever delta >= e + 3uC + u^2 C ~ 7.2uC = 0.030 row units.  HOT_DELTA = 8 FLT_EPSILON * C
// (0.066, as SPAN_DELTA) and HOT_CLAMP = SPAN_BOX >= P0 + HOT_DELTA.  The FMNMX3 and the final compare are exact.
// Padding rows (Cl = -SPAN_OPEN, shifted: still -1e30) give A = -1e30, B = C, h2 = -1e30 < 0: never a candidate;
// always-candidate rows (every constant SPAN_OPEN) give A = B = C, nc2 = 0, h2 = 2C > |2*S*p|.  A NaN bound is dropped by
// the min3 (the clamp stays), a NaN |e| by the running minimum: neither can hide a candidate.
//
// SEGMENT verdict (closest-hit sweep, MODE_SHAREDQ: segment_pass).  The R rays of a thread share q bit for bit, so they
// share (nc2, h2), and the hot loop's verdict "some ray r has |fl(ps2_r + nc2)| <= h2" needs no per-ray work.  Let
// pmin2 <= ps2_r <= pmax2 for every r (a min and a max over all R values, whatever their order).  Round-to-nearest
// addition is monotone, a <= b => fl(a + c) <= fl(b + c), so a passing ray r gives
//     fl(pmin2 + nc2) <= fl(ps2_r + nc2) <= h2     and     fl(pmax2 + nc2) >= fl(ps2_r + nc2) >= -h2,
// and the two-sided test on the thread's extreme rays passes every (thread, triangle) the per-ray verdict passes: no new
// margin, no new rounding.  It costs one FADD2 and the compares per thread and triangle in place of R/2 FADD2 + R/2
// FMNMX3.  It is looser only where a triangle's interval falls between two neighbouring rays of the thread (narrower than
// a pixel); the candidate path rebuilds the per-ray mask with hot_pass, so the pairs handed to the strict test are the same.
// A NaN sum counts as a pass.
//
// MEAN-q SEGMENT verdict (shadow sweeps, MODE_QBAR with ANYHIT: the same segment_pass after hot_terms_qbar).  The R rays of
// a shadow thread do not share q, but the per-ray loop already gives them one (nc2, h2): hot_terms_qbar at the thread's qbar
// with the bounds widened by |B| * qdh, qdh = hot_qdelta(qdelta), qdelta >= max |q_r - qbar| over all R values (shadow_item's
// formula: the spread times 1.0001 plus 2.4e-7 (|qbar| + 1) covers the roundings of qbar and of the spread for any spread).
// The hot-row proof above already takes any qdelta: its qdelta step bounds G' - G with |z| <= (1 + 2u)(|G| + |Bl| qd) and the
// HOT_QD_SCALE term, neither of which assumes qd small, and a large qd only moves A_i, B_i towards the clamp C.  So every pair
// the exact row passes, at the ray's own q, passes |fl(ps2_r + nc2)| <= h2 with these shared (nc2, h2), and the monotonicity
// argument above then carries over word for word: pmin2 <= ps2_r <= pmax2 over the thread's R values gives
// fl(pmin2 + nc2) <= h2 and fl(pmax2 + nc2) >= -h2 for any passing ray.  No new margin, no new rounding.  The R values include
// the duplicated tail entries of a short list and rays already done: both only widen [pmin2, pmax2], so only loosen it.
// It pays once a thread's rays form a compact cell in (p, q): the default mode's shadow lists are sorted by q, then by p in
// serpentine stripes of about sqrt(128 n) entries (order_shadow_rays), so [pmin2, pmax2] spans a few triangle widths.  The
// widened bounds pass most of a flagged thread's rays, so the candidate path rebuilds with each ray's own q (sweep_table).
constexpr float HOT_CLAMP = SPAN_BOX;
constexpr float HOT_DELTA = 8.f * 1.1920928955078125e-7f * HOT_CLAMP;
constexpr float HOT_QD_SCALE = 1.f + 0x1p-20f;
static_assert((double)HOT_CLAMP >= (double)SPAN_S * 1.0625 + (double)HOT_DELTA, "the clamp lies outside every swept ray");

// C - (1 - delta) rounded toward +inf: an exact sum in FP64 (TwoSum), then the nearest float, moved up if below
__host__ __device__ __forceinline__ float hot_shift(float c, float delta) {
    const double a = (double)c, b = (double)delta - 1.0; // exact
    const double d = a + b, bb = d - a, err = (a - (d - bb)) + (b - bb); // a + b = d + err exactly
    float f = (float)d;
    if ((double)f < d || ((double)f == d && err > 0.0)) f = nextafterf(f, INFINITY);
    return f;
}
// span_rows' row (lo, hi) -> its hot form, in place (build_origin_table, build_allcand_table; delta: tests only)
__host__ __device__ __forceinline__ void hot_row(float4 &lo, float4 &hi, float delta = HOT_DELTA) {
    lo.y = hot_shift(lo.y, delta), lo.w = hot_shift(lo.w, delta);
    hi.y = hot_shift(hi.y, delta), hi.w = hot_shift(hi.w, delta);
}
__host__ __device__ __forceinline__ float hot_qdelta(float qdelta) { return qdelta * HOT_QD_SCALE; }
// (nc2, h2) of a hot row at q: a shared exact q, or q = qbar with the bounds widened by |B| * qdh, qdh = hot_qdelta(qdelta)
__host__ __device__ __forceinline__ void hot_terms(const float4 lo, const float4 hi, float q, float &nc2, float &h2) {
    const float A = fmin3(fmaf(q, lo.x, lo.y), fmaf(q, lo.z, lo.w), HOT_CLAMP);
    const float B = fmin3(fmaf(q, hi.x, hi.y), fmaf(q, hi.z, hi.w), HOT_CLAMP);
    nc2 = A - B, h2 = A + B;
}
__host__ __device__ __forceinline__ void hot_terms_qbar(const float4 lo, const float4 hi, float qbar, float qdh, float &nc2, float &h2) {
    const float A = fmin3(fmaf(fabsf(lo.x), qdh, fmaf(qbar, lo.x, lo.y)), fmaf(fabsf(lo.z), qdh, fmaf(qbar, lo.z, lo.w)), HOT_CLAMP);
    const float B = fmin3(fmaf(fabsf(hi.x), qdh, fmaf(qbar, hi.x, hi.y)), fmaf(fabsf(hi.z), qdh, fmaf(qbar, hi.z, hi.w)), HOT_CLAMP);
    nc2 = A - B, h2 = A + B;
}
// the hot test of one pair (ps2 = p * 2 * SPAN_S)
__host__ __device__ __forceinline__ bool hot_pass(float nc2, float h2, float ps2) { return fabsf(ps2 + nc2) <= h2; }
// the segment verdict of a thread's rays with a shared q (pmin2, pmax2: least and greatest ps2 over all of them; above HOT_CLAMP):
// true whenever hot_pass holds for one of them.  Device: one packed FADD2; host: the same two RN adds.
__host__ __device__ __forceinline__ bool segment_pass(float nc2, float h2, float pmin2, float pmax2) {
#ifdef __CUDA_ARCH__
    const float2 e = __fadd2_rn(make_float2(pmin2, pmax2), make_float2(nc2, nc2));
#else
    const float2 e = make_float2(pmin2 + nc2, pmax2 + nc2);
#endif
    return !(e.x > h2) && !(-e.y > h2);
}

// ray masks of the sweeps: a bit per ray of a thread
template <int R>
using RayMask = typename std::conditional<(R > 32), unsigned long long, unsigned>::type;
template <class M>
__device__ __forceinline__ int lowest_ray(M m) { return sizeof(M) == 8 ? __ffsll((long long)m) - 1 : __ffs((int)m) - 1; }

// SPAN_BATCH triangles of a staged hot-row tile against the R rays of this thread (ps2[r] = p_r * 2 * SPAN_S).  One minimum
// chain per triangle: the SPAN_BATCH chains are independent, which is the loop's instruction-level parallelism.
// qdh: hot_qdelta(qdelta) (MODE_QBAR).  Returns bit k set = triangle k may hold a candidate.
template <int R, int MODE>
__device__ __forceinline__ unsigned eval_interval(const float4 *__restrict__ tp, const float (&ps2)[R], float q, float qdh) {
    static_assert(R % 2 == 0, "rays are evaluated in pairs");
    unsigned cand = 0;
#pragma unroll
    for (int k = 0; k < SPAN_BATCH; ++k) {
        float nc2, h2;
        if (MODE == MODE_QBAR) hot_terms_qbar(tp[2 * k], tp[2 * k + 1], q, qdh, nc2, h2);
        else hot_terms(tp[2 * k], tp[2 * k + 1], q, nc2, h2);
        float m = __int_as_float(0x7f800000); // +inf
#pragma unroll
        for (int r = 0; r < R; r += 2) {
            const float2 e = __fadd2_rn(make_float2(ps2[r], ps2[r + 1]), make_float2(nc2, nc2));
            m = fmin3_abs(m, e.x, e.y);
        }
        cand |= (unsigned)(m <= h2) << k;
    }
    return cand;
}
// The same verdict bits from the thread's extreme rays (segment_pass; closest-hit sweep with MODE_SHAREDQ, shadow sweeps with
// MODE_QBAR): per triangle the set-up of hot_terms (hot_terms_qbar), one FADD2 and the compares, whatever R.  Bit k set =
// triangle k may hold a candidate.
template <int MODE>
__device__ __forceinline__ unsigned eval_segment(const float4 *__restrict__ tp, float pmin2, float pmax2, float q, float qdh) {
    unsigned cand = 0;
#pragma unroll
    for (int k = 0; k < SPAN_BATCH; ++k) {
        float nc2, h2;
        if (MODE == MODE_QBAR) hot_terms_qbar(tp[2 * k], tp[2 * k + 1], q, qdh, nc2, h2);
        else hot_terms(tp[2 * k], tp[2 * k + 1], q, nc2, h2);
        cand |= (unsigned)segment_pass(nc2, h2, pmin2, pmax2) << k;
    }
    return cand;
}

// The LOP3 form of the same loop (round 1; kept for tools/sweep_mb3.cu): sign bits OR-ed per ray, AND-ed over rays,
// shifted into a bit register.  Returns bit (BATCH-1-k) CLEAR = some ray of this thread may hit triangle k.
template <int R, int MODE, int UNROLL>
__device__ __forceinline__ unsigned eval_batch_lop3(const float4 *__restrict__ tp, const float (&rp)[R], const float (&rq)[R], float qbar,
                                                    float qdelta) {
    unsigned neg = 0xffffffffu;
#pragma unroll UNROLL
    for (int k = 0; k < BATCH; ++k) {
        const float4 rb = tp[3 * k], rc = tp[3 * k + 1], rd = tp[3 * k + 2];
        unsigned A = 0xffffffffu;
        if (MODE == MODE_OWNQ) {
#pragma unroll
            for (int r = 0; r < R; ++r) A &= edge_sign(rb, rc, rd, rp[r], rq[r]);
        } else {
            const float qx = MODE == MODE_QBAR ? qterm_qbar(rb, qbar, qdelta) : fmaf(rq[0], rb.y, rb.z);
            const float qy = MODE == MODE_QBAR ? qterm_qbar(rc, qbar, qdelta) : fmaf(rq[0], rc.y, rc.z);
            const float qz = MODE == MODE_QBAR ? qterm_qbar(rd, qbar, qdelta) : fmaf(rq[0], rd.y, rd.z);
#pragma unroll
            for (int r = 0; r < R; ++r)
                A &= __float_as_uint(fmaf(rp[r], rb.x, qx)) | __float_as_uint(fmaf(rp[r], rc.x, qy)) |
                     __float_as_uint(fmaf(rp[r], rd.x, qz));
        }
        neg = __funnelshift_l(A, neg, 1);
    }
    return neg;
}

// ---- the sweep over tiles [tile_lo, tile_hi) of one origin table, for the R rays of each thread ---
// rp/rq: the rays' parameters in the table's direction parametrisation (rq is read by MODE_OWNQ only; MODE_SHAREDQ takes
//        the common q from rq[0], MODE_QBAR from qbar/qdelta; span forms keep only 2*S*p in registers)
// valid: bit r set = ray r exists; done: bit r set = ray r needs no more tests (RayMask<R>: 64 bits for R > 32)
// gtile: running tile counter of this CTA (mbarrier phase bookkeeping across work items)
// strict(otid, r, tri, filt, row) -> accepted: the reference's own test of ray r of thread otid (a thread of the calling
//        lane's warp) against triangle tri (kernels.cuh), run by whichever lane drains the pair; filt = the filter passed
//        the pair (false only in EXHAUSTIVE validation mode), row = the triangle's staged row (still resident)
// n_flag, n_queue (may be null; not counted in EXHAUSTIVE mode): add this thread's flagged (thread, triangle) verdicts and the
//        pairs it queued
// n_cyc (may be null): lane 0 adds the SM cycles its warp spends in the candidate path
// own (any-hit MODE_QBAR only, required there): the rays of every thread of the CTA in shared memory, (2*S*p, q) of ray r of
//        thread t at own[t * R + ((r + t) & (R - 1))] (rotated by the lane, so that neither the stores nor the loads conflict)
template <int R, int MODE, bool ANYHIT, bool EXHAUSTIVE, class Strict>
__device__ __forceinline__ void sweep_table(SmemT<Rows<MODE>::N> &sm, const float4 *__restrict__ table, int tile_lo, int tile_hi, int n_tris,
                                            const float (&rp)[R], const float (&rq)[R], float qbar, float qdelta, RayMask<R> valid,
                                            RayMask<R> &done, unsigned &gtile, unsigned &n_tiles_swept, Strict &&strict,
                                            unsigned *n_pipe_err = nullptr, unsigned *n_flag = nullptr, unsigned *n_queue = nullptr,
                                            unsigned long long *n_cyc = nullptr, const float2 *own = nullptr) {
    using Mask = RayMask<R>;
    static_assert(R <= 32 || MODE != MODE_OWNQ, "the three-row form's rays fit one 32-bit mask");
    constexpr int ROWS = Rows<MODE>::N;
    constexpr uint32_t BYTES = Rows<MODE>::BYTES;
    constexpr bool SPAN = MODE != MODE_OWNQ;
    const int tid = threadIdx.x;
    const int n_tiles = tile_hi - tile_lo;
    const float4 *__restrict__ src = table + (size_t)tile_lo * TILE * ROWS;
    if (tid == 0) {
        const int first = n_tiles < STAGES ? n_tiles : STAGES;
        for (int i = 0; i < first; ++i) {
            const unsigned g = gtile + i;
            mbar_expect_tx(&sm.full_bar[g % STAGES], BYTES);
            tma_load_1d(sm.tile[g % STAGES], src + (size_t)i * TILE * ROWS, BYTES, &sm.full_bar[g % STAGES]);
        }
    }
    float ps2[R]; // span form: the rays' 2 p in row units (exact: SPAN_S is a power of two)
#pragma unroll
    for (int r = 0; r < R; ++r) ps2[r] = rp[r] * (2.f * SPAN_S);
    const float qhot = MODE == MODE_QBAR ? qbar : rq[0], qdh = hot_qdelta(qdelta);
    // closest hit with a shared q, and the shadow sweeps (mean q): the hot loop decides each triangle from the extreme rays
    // (segment_pass); jittered primary samples (MODE_QBAR, closest hit) keep the per-ray loop
    constexpr bool SEGMENT = (!ANYHIT && MODE == MODE_SHAREDQ) || (ANYHIT && MODE == MODE_QBAR);
    // the shadow sweeps rebuild a flagged triangle's candidates with each ray's own q, one ray per lane (below)
    constexpr bool OWNQ_REBUILD = ANYHIT && MODE == MODE_QBAR;
    static_assert(!OWNQ_REBUILD || 32 % R == 0, "a warp rebuilds whole threads' rays");
    float pmin2 = ps2[0], pmax2 = ps2[0];
    if (SEGMENT) {
#pragma unroll
        for (int r = 1; r < R; ++r) pmin2 = fminf(pmin2, ps2[r]), pmax2 = fmaxf(pmax2, ps2[r]);
    }
    const unsigned lane = tid & 31;
    unsigned *queue = sm.queue[tid >> 5];
#ifndef SWEEP_NO_STRICT
    // the first n queued pairs, one per lane: the reference's own test, then (any-hit) the accepted rays into done
    auto drain = [&](const float4 *__restrict__ tp, int it, int n) {
        __syncwarp();
        if ((int)lane < n) {
            const unsigned e = queue[lane];
            const int r = e & 63, owner = (e >> 6) & 31, k = (e >> 11) & 255;
            const int otid = (tid & ~31) | owner;
            if (strict(otid, r, (tile_lo + it) * TILE + k, (bool)(e >> 19), tp + ROWS * k) && ANYHIT)
                atomicOr(&sm.qdone[tid >> 5][owner], 1ull << r);
        }
        __syncwarp();
        if (ANYHIT) {
            done |= (Mask)sm.qdone[tid >> 5][lane];
            sm.qdone[tid >> 5][lane] = 0;
        }
        __syncwarp();
    };
#endif
    for (int it = 0; it < n_tiles; ++it) {
        const unsigned g = gtile + it;
        const int s = g % STAGES;
        mbar_wait(&sm.full_bar[s], (g / STAGES) & 1u);
        // Validation mode doubles as the pipeline's own race check (compute-sanitizer is not available on this pool):
        // every warp compares the staged tile with its source in global memory when the tile arrives AND after it has
        // used it — a copy that had not landed, or a refill issued while a warp was still reading, shows up here.
        auto tile_differs = [&]() {
            unsigned bad = 0;
            const uint4 *a = reinterpret_cast<const uint4 *>(sm.tile[s]);
            const uint4 *b = reinterpret_cast<const uint4 *>(src + (size_t)it * TILE * ROWS);
            for (int i = tid & 31; i < TILE * ROWS; i += 32) {
                const uint4 x = a[i], y = __ldcg(&b[i]);
                bad |= (x.x ^ y.x) | (x.y ^ y.y) | (x.z ^ y.z) | (x.w ^ y.w);
            }
            return __any_sync(0xffffffffu, bad != 0);
        };
        if (EXHAUSTIVE && n_pipe_err && tile_differs() && (tid & 31) == 0) ++*n_pipe_err;
        // any-hit: a warp whose rays all have their occluder has nothing left to evaluate
        const bool idle = ANYHIT && __all_sync(0xffffffffu, (Mask)(done | ~valid) == (Mask)~(Mask)0);
        if (!idle) {
            ++n_tiles_swept;
            const float4 *__restrict__ tp = sm.tile[s];
            // triangles per hot-loop call, and per bit of its verdict: the interval form (span rows) flags single
            // triangles, the three-row form groups of GROUP
            constexpr int NB = SPAN ? SPAN_BATCH : BATCH, UNIT = SPAN ? 1 : Batch<SPAN ? 2 : R>::GROUP;
            // pairs in this warp's queue.  The shadow sweeps keep them across the tile's batches and drain when the queue is
            // full and at the end of the tile: a drain is a chain of dependent loads and FP64 work, and fewer, fuller drains
            // hide more of it.  A ray that finds its occluder meanwhile only adds strict tests of later triangles, which the
            // minimum merge ignores.  The other sweeps drain after each batch.
            int fill = 0;
#pragma unroll 1
            for (int b0 = 0; b0 < TILE; b0 += NB) {
                unsigned cand;
                if constexpr (SEGMENT) cand = eval_segment<MODE>(tp + ROWS * b0, pmin2, pmax2, qhot, qdh);
                else if constexpr (SPAN) cand = eval_interval<R, MODE>(tp + ROWS * b0, ps2, qhot, qdh);
                else cand = eval_batch<R, MODE>(tp + ROWS * b0, rp, rq, qbar, qdelta);
#ifdef SWEEP_NO_STRICT // development microbenchmark only (tools/sweep_mb2.cu): timing without the strict path
                if (cand) ++done;
#else
                // validation mode: every triangle goes to the strict path; the hot loop's own verdict is kept so that an
                // accepted pair whose triangle (group) it would have skipped counts as a filter miss too
                const unsigned cand_hot = cand;
                if (!EXHAUSTIVE && n_flag) *n_flag += __popc(cand);
                if (EXHAUSTIVE) cand = NB / UNIT == 32 ? 0xffffffffu : (1u << (NB / UNIT)) - 1u;
                // rare: some lane flagged a triangle (group of UNIT triangles).  The warp rebuilds, lane by lane, the per-ray
                // candidate mask of each flagged triangle, queues the (owner lane, ray, triangle) pairs and drains the queue one
                // pair per lane, so a thread's candidates no longer serialise while the rest of the warp idles.
                unsigned wcand = __reduce_or_sync(0xffffffffu, cand);
                if (wcand) {
                    const long long c_cand = n_cyc ? clock64() : 0;
                    if constexpr (OWNQ_REBUILD) {
                        // Shadow sweeps: the thread's verdict used the mean-q bounds widened over all its rays, so most
                        // flagged rays fail their own test.  Each flagged (owner lane, triangle) is rebuilt one ray per lane:
                        // lane = slot * R + r tests ray r of the slot's owner, read from shared memory, with the exact test at
                        // its own q (hot_terms, hot_pass), and the pairs that pass and are live go straight to the queue.
                        // Every pair the reference accepts passes this test (hot_row), so the drain needs no second filter.
                        constexpr int OPW = 32 / R; // owner lanes per round
                        const int slot = lane / R, r = lane & (R - 1);
                        while (wcand) {
                            const int gq = __ffs(wcand) - 1, k = b0 + gq; // ascending triangle order
                            wcand &= wcand - 1;
                            if ((tile_lo + it) * TILE + k >= n_tris) break; // padding (warp-uniform), and so is the rest
                            const float4 lo = lds128_opaque(&tp[2 * k]), hi = lds128_opaque(&tp[2 * k + 1]);
                            const Mask live = valid & ~done;
                            unsigned owners = __ballot_sync(0xffffffffu, (cand >> gq) & 1u);
                            while (owners) {
                                unsigned m = owners;
                                for (int i = 0; i < slot; ++i) m &= m - 1;
                                const int o = m ? __ffs(m) - 1 : 0;
                                const Mask olive = __shfl_sync(0xffffffffu, live, o);
                                const unsigned ohot = __shfl_sync(0xffffffffu, cand_hot, o);
                                bool filt = false, in = false;
                                if (m) {
                                    const float2 pq = own[((tid & ~31) | o) * R + ((r + o) & (R - 1))];
                                    float nc2, h2;
                                    hot_terms(lo, hi, pq.y, nc2, h2);
                                    filt = hot_pass(nc2, h2, pq.x) && (!EXHAUSTIVE || ((ohot >> gq) & 1u));
                                    in = ((olive >> r) & 1u) && (EXHAUSTIVE || filt);
                                }
                                const unsigned ins = __ballot_sync(0xffffffffu, in);
                                const int n = __popc(ins), pos = fill + __popc(ins & ((1u << lane) - 1u));
                                const unsigned e = (unsigned)r | (unsigned)o << 6 | (unsigned)k << 11 | (unsigned)filt << 19;
                                if (in && pos < QCAP) queue[pos] = e;
                                if (fill + n >= QCAP) {
                                    drain(tp, it, QCAP);
                                    if (in && pos >= QCAP) queue[pos - QCAP] = e;
                                    fill += n - QCAP;
                                } else {
                                    fill += n;
                                }
                                if (!EXHAUSTIVE && n_queue) *n_queue += in;
#pragma unroll
                                for (int i = 0; i < OPW; ++i) owners &= owners - 1;
                            }
                        }
                    } else {
                        while (wcand) {
                            const int gq = __ffs(wcand) - 1; // ascending triangle order
                            wcand &= wcand - 1;
                            const bool mine = (cand >> gq) & 1u;
#pragma unroll 1
                            for (int kk = 0; kk < UNIT; ++kk) {
                                const int k = b0 + gq * UNIT + kk;
                                if ((tile_lo + it) * TILE + k >= n_tris) break; // padding (warp-uniform)
                                Mask filt = 0;
                                if (mine) {
                                    // The rows are re-read through opaque loads so that the compiler cannot merge this with the
                                    // hot evaluation.
                                    if (SPAN) {
                                        // the hot loop's own test, ray by ray: it passes every pair span_pass passes (hot_row); exact
                                        // with a common q
                                        const float4 lo = lds128_opaque(&tp[2 * k]), hi = lds128_opaque(&tp[2 * k + 1]);
                                        float nc2, h2;
                                        if (MODE == MODE_QBAR) hot_terms_qbar(lo, hi, qhot, qdh, nc2, h2);
                                        else hot_terms(lo, hi, qhot, nc2, h2);
#pragma unroll
                                        for (int r = 0; r < R; ++r) filt |= (Mask)hot_pass(nc2, h2, ps2[r]) << r;
                                    } else {
                                        const float4 rb = lds128_opaque(&tp[3 * k]), rc = lds128_opaque(&tp[3 * k + 1]), rd = lds128_opaque(&tp[3 * k + 2]);
#pragma unroll
                                        for (int r = 0; r < R; ++r) filt |= (Mask)edge_pass(rb, rc, rd, rp[r], rq[r]) << r;
                                    }
                                    if (EXHAUSTIVE && !((cand_hot >> gq) & 1u)) filt = 0;
                                }
                                const Mask live = valid & ~done;
                                Mask pend = mine ? (EXHAUSTIVE ? live : filt & live) : (Mask)0;
                                if (!EXHAUSTIVE && n_queue) *n_queue += __popcll((unsigned long long)pend);
                                while (__any_sync(0xffffffffu, pend != 0)) {
                                    // this lane's pairs go to queue slots [fill + before, ...): as many as fit, the rest after a drain
                                    const int n = __popcll((unsigned long long)pend);
                                    int incl = n;
#pragma unroll
                                    for (int o = 1; o < 32; o <<= 1) {
                                        const int y = __shfl_up_sync(0xffffffffu, incl, o);
                                        if (lane >= o) incl += y;
                                    }
                                    for (int slot = fill + incl - n; pend && slot < QCAP; ++slot) {
                                        const int r = lowest_ray(pend);
                                        pend &= pend - 1;
                                        queue[slot] = (unsigned)r | lane << 6 | (unsigned)k << 11 | (unsigned)((filt >> r) & 1u) << 19;
                                    }
                                    fill = min(QCAP, fill + __shfl_sync(0xffffffffu, incl, 31));
                                    if (fill == QCAP) drain(tp, it, fill), fill = 0;
                                }
                            }
                        }
                    }
                    if (!OWNQ_REBUILD && fill) drain(tp, it, fill), fill = 0;
                    if (n_cyc && lane == 0) *n_cyc += clock64() - c_cand;
                }
#endif
            }
#ifndef SWEEP_NO_STRICT
            if (OWNQ_REBUILD && __any_sync(0xffffffffu, fill != 0)) {
                const long long c_cand = n_cyc ? clock64() : 0;
                drain(tp, it, fill);
                if (n_cyc && lane == 0) *n_cyc += clock64() - c_cand;
            }
#endif
        }
        if (EXHAUSTIVE && n_pipe_err && tile_differs() && (tid & 31) == 0) ++*n_pipe_err;
        // No block-wide barrier per tile: every warp counts itself out of stage s, and the LAST one refills it.
        // Warps run up to STAGES-1 tiles apart, which absorbs the skew of the (rare, long) strict evaluations
        // instead of stalling every warp behind one.
        __syncwarp();
        if ((tid & 31) == 0) {
            __threadfence_block(); // this warp's reads of the stage are done before the count is visible
            if (atomicAdd(&sm.consumed[s], 1) == (int)(blockDim.x >> 5) - 1) {
                sm.consumed[s] = 0;
                __threadfence_block();
                if (it + STAGES < n_tiles) {
                    mbar_expect_tx(&sm.full_bar[s], BYTES);
                    tma_load_1d(sm.tile[s], src + (size_t)(it + STAGES) * TILE * ROWS, BYTES, &sm.full_bar[s]);
                }
            }
        }
    }
    gtile += n_tiles; // every issued tile has been waited for
}

}  // namespace sweep
