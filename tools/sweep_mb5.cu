// sweep_mb5.cu — round-3 microbenchmark of the INTERVAL form of the span test, against the span loop it replaces.
//
// For one thread's shared q a triangle's span row is one interval of S*p: the pair passes the span test
//     x = sat(S*p + ax) = 1  and  y = sat(ay - S*p) = 1      <=>     lo = 1 - ax  <=  S*p  <=  hi = ay - 1
// i.e. |S*p - c| <= h with c = (lo+hi)/2, h = (hi-lo)/2.  Per thread and triangle the bounds are clamped to the swept
// box and turned into (c, h); per ray PAIR the loop issues
//     e = S*{p_r, p_r+1} - c          one packed FFMA2 (or FADD2 on pre-scaled p)
//     m = min(m, |e.x|, |e.y|)        one three-input FMNMX3, |.| an operand modifier
// and after the R rays "m <= h" is the triangle's verdict: 1 FMA-pipe instruction per two pairs, against 2 FFMA.SAT +
// half an FFMA2 per pair (= 5 per two pairs) of the span loop (tools/sweep_mb4.cu, F_ADD: the library's form).
// saturation has no packed form on sm_100a (ptxas rejects .sat on f32x2), so the span loop cannot pack its two adds.
// The FMNMX3 chain kernel times the three-input min alone, to find its issue cost and pipe.
// F_HOT is the loop on the HOT rows the tables store now (csrc/sweep.cuh, hot_row): the +1s, the clamp and the margin
// folded into the row, per thread and triangle 4 FFMA + 2 FMNMX3 + 2 FADD (8 FFMA with a mean q), the rays holding 2*S*p.
// F_SEG is the segment verdict of the closest-hit sweep (csrc/sweep.cuh, segment_pass): the set-up of F_HOT, then one
// FADD2 {pmin, pmax} + nc2 and the two-sided compare per thread and triangle, nothing per pair (round 7).  Its
// "cyc/warp-tri" column is the loop's cost per (warp, triangle), whatever R.
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <vector>

constexpr int TILE = 256, BATCH = 16;
enum { MODE_SHAREDQ = 1, MODE_QBAR = 2 };
enum { F_SPAN = 0, F_IV_FMA2 = 1, F_IV_ADD2 = 2, F_HOT = 3, F_SEG = 4 };

__device__ __forceinline__ float min3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// the library's span loop (round 2): returns a bit per group of GROUP triangles
template <int R, int MODE, int GROUP, int NACC2>
__device__ __forceinline__ unsigned eval_span(const float4 *__restrict__ tp, const float (&ps)[R], float q, float qdelta) {
    unsigned cand = 0;
#pragma unroll
    for (int g = 0; g < BATCH / GROUP; ++g) {
        float2 acc[NACC2];
#pragma unroll
        for (int a = 0; a < NACC2; ++a) acc[a] = make_float2(0.f, 0.f);
#pragma unroll
        for (int kk = 0; kk < GROUP; ++kk) {
            const int k = g * GROUP + kk;
            const float4 lo = tp[2 * k], hi = tp[2 * k + 1];
            float a1 = fmaf(q, lo.x, lo.y), a2 = fmaf(q, lo.z, lo.w), b1 = fmaf(q, hi.x, hi.y), b2 = fmaf(q, hi.z, hi.w);
            if (MODE == MODE_QBAR) {
                a1 = fmaf(fabsf(lo.x), qdelta, a1), a2 = fmaf(fabsf(lo.z), qdelta, a2);
                b1 = fmaf(fabsf(hi.x), qdelta, b1), b2 = fmaf(fabsf(hi.z), qdelta, b2);
            }
            const float ax = fminf(a1, a2), ay = fminf(b1, b2);
#pragma unroll
            for (int r = 0; r < R; r += 2) {
                const float2 x = make_float2(__saturatef(ps[r] + ax), __saturatef(ps[r + 1] + ax));
                const float2 y = make_float2(__saturatef(ay - ps[r]), __saturatef(ay - ps[r + 1]));
                acc[(r / 2) % NACC2] = __ffma2_rn(x, y, acc[(r / 2) % NACC2]);
            }
        }
        float s = 0.f;
#pragma unroll
        for (int a = 0; a < NACC2; ++a) s += acc[a].x + acc[a].y;
        if (s >= 1.f) cand |= 1u << g;
    }
    return cand;
}

// the interval form: returns a bit per triangle; NCH independent min chains per triangle
template <int R, int MODE, int FORM, int NCH>
__device__ __forceinline__ unsigned eval_interval(const float4 *__restrict__ tp, const float (&rp)[R], const float (&ps)[R], float q, float qdelta,
                                                  float S, float pmin, float pmax) {
    constexpr float P = 65536.f * 1.0625f + 1.f, DELTA = 8.f * 1.1920929e-7f * P;
    unsigned cand = 0;
#pragma unroll
    for (int k = 0; k < BATCH; ++k) {
        const float4 lo = tp[2 * k], hi = tp[2 * k + 1];
        float a1 = fmaf(q, lo.x, lo.y), a2 = fmaf(q, lo.z, lo.w), b1 = fmaf(q, hi.x, hi.y), b2 = fmaf(q, hi.z, hi.w);
        if (MODE == MODE_QBAR) {
            a1 = fmaf(fabsf(lo.x), qdelta, a1), a2 = fmaf(fabsf(lo.z), qdelta, a2);
            b1 = fmaf(fabsf(hi.x), qdelta, b1), b2 = fmaf(fabsf(hi.z), qdelta, b2);
        }
        float nc, h;
        if (FORM == F_HOT || FORM == F_SEG) { // (ps holds 2*S*p here)
            const float A = min3(a1, a2, P), B = min3(b1, b2, P);
            nc = A - B, h = A + B;
        } else {
            const float l = fmaxf(1.f - fminf(a1, a2), -P), u = fminf(fminf(b1, b2) - 1.f, P);
            nc = -0.5f * (l + u), h = fmaf(0.5f, u - l, DELTA);
        }
        bool pass;
        if constexpr (FORM == F_SEG) { // the thread's extreme rays only
            const float2 e = __fadd2_rn(make_float2(pmin, pmax), make_float2(nc, nc));
            pass = !(e.x > h) && !(-e.y > h);
        } else {
            float m[NCH];
#pragma unroll
            for (int j = 0; j < NCH; ++j) m[j] = __int_as_float(0x7f800000);
#pragma unroll
            for (int r = 0; r < R; r += 2) {
                const float2 e = FORM == F_IV_FMA2 ? __ffma2_rn(make_float2(rp[r], rp[r + 1]), make_float2(S, S), make_float2(nc, nc))
                                                   : __fadd2_rn(make_float2(ps[r], ps[r + 1]), make_float2(nc, nc));
                float &mm = m[(r / 2) % NCH];
                mm = min3(mm, fabsf(e.x), fabsf(e.y));
            }
            float mn = m[0];
#pragma unroll
            for (int j = 1; j < NCH; ++j) mn = fminf(mn, m[j]);
            pass = mn <= h;
        }
        cand |= (unsigned)pass << k;
    }
    return cand;
}

template <int R, int MODE, int FORM, int NTH, int MINBLK, int GROUP, int NACC2>
__global__ void __launch_bounds__(NTH, MINBLK) k_loop(const float4 *tile_g, int reps, float *out, float seed, float S) {
    __shared__ __align__(16) float4 tile[TILE * 2];
    for (int i = threadIdx.x; i < TILE * 2; i += blockDim.x) tile[i] = tile_g[i];
    __syncthreads();
    float rp[R], ps[R];
#pragma unroll
    for (int r = 0; r < R; ++r) rp[r] = seed * (threadIdx.x + 1) * (r + 1), ps[r] = rp[r] * (FORM >= F_HOT ? 2.f * S : S);
    float pmin = ps[0], pmax = ps[0];
#pragma unroll
    for (int r = 1; r < R; ++r) pmin = fminf(pmin, ps[r]), pmax = fmaxf(pmax, ps[r]);
    const float q = seed * (threadIdx.x + 7) * 3, qdelta = 1e-6f * (1 + (threadIdx.x & 3));
    int hits = 0;
    for (int rep = 0; rep < reps; ++rep) {
#pragma unroll 1
        for (int b0 = 0; b0 < TILE; b0 += BATCH) {
            const unsigned c = FORM == F_SPAN ? eval_span<R, MODE, GROUP, NACC2>(tile + 2 * b0, ps, q, qdelta)
                                              : eval_interval<R, MODE, FORM, NACC2>(tile + 2 * b0, rp, ps, q, qdelta, S, pmin, pmax);
            if (c) {
                hits += 1;
                asm volatile("" ::: "memory");
            }
        }
    }
    if (hits == 123456789) out[0] = hits;
}

// FMNMX3 alone: NCH independent chains of `min3(m, |a|, |b|)` over register operands that change every iteration
template <int NCH, int NTH, int MINBLK>
__global__ void __launch_bounds__(NTH, MINBLK) k_fmnmx3(int reps, float *out, float seed) {
    float m[NCH], a[8];
#pragma unroll
    for (int j = 0; j < NCH; ++j) m[j] = seed * (j + threadIdx.x);
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = seed * (i + 3) - 0.5f;
    for (int rep = 0; rep < reps; ++rep) {
#pragma unroll
        for (int i = 0; i < 64; ++i) {
            float &mm = m[i % NCH];
            asm volatile("min.f32 %0, %1, %2, %3;" : "=f"(mm) : "f"(mm), "f"(fabsf(a[i % 8])), "f"(fabsf(a[(i + 3) % 8])));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = __int_as_float(__float_as_int(a[i]) ^ 1);
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NCH; ++j) s += m[j];
    if (s == 123456789.f) out[0] = s;
}

static int g_sms = 0;
static double g_clk = 1.965e9;
template <typename K, typename F>
void run(const char *tag, K kern, int nth, int minblk, F launch, double pairs_per_thread_rep, int R) {
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nth, 0);
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, kern);
    const int blocks = occ < minblk ? occ : minblk;
    const int reps = 300;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    for (int i = 0; i < 2; ++i) launch(g_sms * blocks, reps);
    cudaEventRecord(e0);
    const int iters = 4;
    for (int i = 0; i < iters; ++i) launch(g_sms * blocks, reps);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaError_t err = cudaGetLastError();
    const double units = (double)g_sms * blocks * nth * pairs_per_thread_rep * reps;
    const double tp = units * iters / (ms * 1e-3) / 1e12;
    // issue cycles per unit of one warp on one SM sub-partition (4 per SM)
    const double cyc = (double)g_sms * 4 * g_clk / (tp * 1e12) * 32;
    if (R > 0)
        printf("%-40s R=%-2d %4dthr x%d (%3d regs) %8.3f ms  %6.3f Tpairs/s  %5.1f cyc/warp-tri  %5.2f cyc/pair  %s\n", tag, R, nth,
               blocks, fa.numRegs, ms / iters, tp, cyc * R, cyc, err == cudaSuccess ? "" : cudaGetErrorString(err));
    else
        printf("%-40s       %4dthr x%d (%3d regs) %8.3f ms  %6.3f Tinstr/s  %5.2f issue cyc per warp instruction  %s\n", tag, nth, blocks,
               fa.numRegs, ms / iters, tp, cyc, err == cudaSuccess ? "" : cudaGetErrorString(err));
    fflush(stdout);
}

#define LOOP(R, MODE, FORM, NTH, MB, G, NA)                                                                                                 \
    run(#MODE " " #FORM " g" #G " x" #NA, k_loop<R, MODE, FORM, NTH, MB, G, NA>, NTH, MB,                                                   \
        [&](int grid, int reps) { k_loop<R, MODE, FORM, NTH, MB, G, NA><<<grid, NTH>>>(tile_g, reps, out, 1e-3f, 65536.f); },             \
        (double)R * TILE, R)
#define MINCHAIN(NCH, NTH, MB)                                                                                                              \
    run("FMNMX3 chain x" #NCH, k_fmnmx3<NCH, NTH, MB>, NTH, MB, [&](int grid, int reps) { k_fmnmx3<NCH, NTH, MB><<<grid, NTH>>>(reps, out, 1e-3f); }, \
        64.0, 0)

int main() {
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, 0);
    int clk_khz = 0;
    cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    if (clk_khz > 0) g_clk = clk_khz * 1e3;
    cudaDeviceProp prop{};
    cudaGetDeviceProperties(&prop, 0);
    printf("# %s, %d SMs, cycle columns at %.0f MHz (the reported max SM clock)\n", prop.name, g_sms, g_clk / 1e6);
    std::vector<float> h(TILE * 8);
    for (size_t i = 0; i < h.size(); ++i) h[i] = (i & 1) ? -1e4f - 3.f * (float)(i % 97) : 0.5f + 0.01f * (float)(i % 13); // never a candidate
    float4 *tile_g;
    float *out;
    cudaMalloc(&tile_g, h.size() * 4);
    cudaMemcpy(tile_g, h.data(), h.size() * 4, cudaMemcpyHostToDevice);
    cudaMalloc(&out, 64);
    printf("-- FMNMX3 alone (64 per iteration, independent chains)\n");
    MINCHAIN(1, 128, 4);
    MINCHAIN(4, 128, 4);
    MINCHAIN(8, 128, 4);
    MINCHAIN(8, 256, 4);
    printf("-- shared q: span loop (library round 2) vs interval form\n");
    LOOP(16, MODE_SHAREDQ, F_SPAN, 128, 4, 4, 4);
    LOOP(16, MODE_SHAREDQ, F_IV_FMA2, 128, 4, 1, 1);
    LOOP(16, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 1);
    LOOP(16, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 2);
    LOOP(24, MODE_SHAREDQ, F_SPAN, 128, 4, 4, 4);
    LOOP(24, MODE_SHAREDQ, F_IV_FMA2, 128, 4, 1, 1);
    LOOP(24, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 1);
    LOOP(24, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 2);
    LOOP(32, MODE_SHAREDQ, F_SPAN, 128, 4, 4, 4);
    LOOP(32, MODE_SHAREDQ, F_IV_FMA2, 128, 4, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_IV_ADD2, 128, 4, 1, 2);
    LOOP(32, MODE_SHAREDQ, F_IV_ADD2, 256, 2, 1, 1);
    printf("-- shared q: hot rows (R = 32, 64) against the interval form\n");
    LOOP(32, MODE_SHAREDQ, F_HOT, 128, 4, 1, 1);
    LOOP(64, MODE_SHAREDQ, F_IV_ADD2, 128, 2, 1, 1);
    LOOP(64, MODE_SHAREDQ, F_HOT, 128, 2, 1, 1);
    LOOP(64, MODE_SHAREDQ, F_HOT, 128, 3, 1, 1);
    printf("-- shared q: segment verdict (closest hit, round 7) against the hot loop, R = 32 and 64, 2 and 3 CTAs/SM\n");
    LOOP(32, MODE_SHAREDQ, F_HOT, 128, 2, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_SEG, 128, 2, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_HOT, 128, 3, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_SEG, 128, 3, 1, 1);
    LOOP(32, MODE_SHAREDQ, F_SEG, 128, 4, 1, 1);
    LOOP(64, MODE_SHAREDQ, F_SEG, 128, 2, 1, 1);
    LOOP(64, MODE_SHAREDQ, F_SEG, 128, 3, 1, 1);
    printf("-- any-hit (qbar + |B| qdelta): span loop vs interval form\n");
    LOOP(16, MODE_QBAR, F_SPAN, 128, 4, 4, 4);
    LOOP(16, MODE_QBAR, F_IV_FMA2, 128, 4, 1, 1);
    LOOP(16, MODE_QBAR, F_IV_ADD2, 128, 4, 1, 1);
    LOOP(16, MODE_QBAR, F_IV_ADD2, 128, 4, 1, 2);
    LOOP(32, MODE_QBAR, F_IV_ADD2, 128, 4, 1, 1);
    LOOP(16, MODE_QBAR, F_HOT, 128, 4, 1, 1);
    return 0;
}
