// sweep_mb2.cu — round-2 development microbenchmark of the sweep's hot loop (sweep::eval_batch, the code the
// production kernels run) at different occupancies: threads per CTA x CTAs per SM (launch bounds cap the
// registers), rays per thread, unroll.  The tile sits in shared memory and is swept repeatedly, so only the
// issue/pipe behaviour is measured; the PROD rows run the full TMA tile pipeline (sweep::sweep_table).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo tools/sweep_mb2.cu -o tools/sweep_mb2.bin
#define SWEEP_NO_STRICT
#include "../esctp1raytracer_b200/csrc/sweep.cuh"
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <vector>

using namespace sweep;

template <int R, int MODE, int NTH, int MINBLK, int UNROLL>
__global__ void __launch_bounds__(NTH, MINBLK) k_loop(const float4 *tile_g, int reps, float *out, float seed) {
    __shared__ __align__(16) float4 tile[TILE * 3];
    for (int i = threadIdx.x; i < TILE * 3; i += blockDim.x) tile[i] = tile_g[i];
    __syncthreads();
    float rp[R], rq[R];
#pragma unroll
    for (int r = 0; r < R; ++r) rp[r] = seed * (threadIdx.x + 1) * (r + 1), rq[r] = seed * (threadIdx.x + 7) * (MODE == MODE_OWNQ ? r + 3 : 3);
    const float qbar = rq[0], qdelta = 1e-6f * (1 + (threadIdx.x & 3));
    int hits = 0;
    for (int rep = 0; rep < reps; ++rep) {
#pragma unroll 1
        for (int b0 = 0; b0 < TILE; b0 += BATCH) {
            const unsigned neg = eval_batch_lop3<R, MODE, UNROLL>(tile + 3 * b0, rp, rq, qbar, qdelta);
            if (~neg & 0xffffu) {
                hits += 1;
                asm volatile("" ::: "memory");
            }
        }
    }
    if (hits == 123456789) out[0] = hits;
}

// the production data path (TMA tile stream + mbarrier + per-warp stage recycling) without the strict path
template <int R, int MODE, bool ANYHIT, int NTH, int MINBLK>
__global__ void __launch_bounds__(NTH, MINBLK) k_prod(const float4 *table, int n_tiles, int n_blocks, int *work, float *out, float seed) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using SmemM = SmemT<Rows<MODE>::N>; // (round 2, span form: MODE_SHAREDQ / MODE_QBAR sweep 32-byte rows)
    SmemM &sm = *reinterpret_cast<SmemM *>(smem_raw);
    const int tid = threadIdx.x;
    smem_init(sm);
    unsigned gtile = 0, n_swept = 0, acc = 0;
    for (;;) {
        if (tid == 0) sm.blk = atomicAdd(work, 1);
        __syncthreads();
        const int blk = sm.blk;
        if (blk >= n_blocks) break;
        float rp[R], rq[R];
#pragma unroll
        for (int r = 0; r < R; ++r) rp[r] = seed * (tid + 1) * (r + 1 + blk), rq[r] = seed * (tid + 7) * 3;
        unsigned done = 0;
        sweep_table<R, MODE, ANYHIT, false>(sm, table, 0, n_tiles, n_tiles * TILE, rp, rq, rq[0], 1e-6f, (1u << R) - 1u, done, gtile, n_swept,
                                            [&](int, int, int, bool, const float4 *) { return false; });
        acc += done;
        __syncthreads();
    }
    if (acc == 123456789u) out[0] = acc;
}

static int g_sms = 0;

template <typename F>
void run(const char *name, F launch, double pairs_per_launch, double flop_per_pair, int ctas_per_sm_expected) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    for (int i = 0; i < 2; ++i) launch();
    cudaEventRecord(e0);
    const int iters = 4;
    for (int i = 0; i < iters; ++i) launch();
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaError_t err = cudaGetLastError();
    const double tp = pairs_per_launch * iters / (ms * 1e-3) / 1e12;
    printf("%-44s %8.3f ms  %6.3f Tpairs/s  %6.2f TFLOP/s executed  %s\n", name, ms / iters, tp, tp * flop_per_pair,
           err == cudaSuccess ? "" : cudaGetErrorString(err));
    fflush(stdout);
}

template <int R, int MODE, int NTH, int MINBLK, int UNROLL>
void bench_loop(const float4 *tile_g, float *out, int reps) {
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_loop<R, MODE, NTH, MINBLK, UNROLL>, NTH, 0);
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, k_loop<R, MODE, NTH, MINBLK, UNROLL>);
    const int blocks = occ < MINBLK ? occ : MINBLK;
    char name[96];
    snprintf(name, sizeof name, "%s R=%-2d %4dthr x%d (occ %d, %3d regs) u%d", MODE == MODE_SHAREDQ ? "SQ  " : MODE == MODE_QBAR ? "QBAR" : "OWNQ", R, NTH,
             blocks, occ, fa.numRegs, UNROLL);
    const double flop = MODE == MODE_SHAREDQ ? 2.0 * (3 + 3 * R) / R : MODE == MODE_QBAR ? 2.0 * (6 + 3 * R) / R : 12.0;
    run(name, [&] { k_loop<R, MODE, NTH, MINBLK, UNROLL><<<g_sms * blocks, NTH>>>(tile_g, reps, out, 1e-3f); },
        (double)g_sms * blocks * NTH * R * TILE * reps, flop, blocks);
}

template <int R, int MODE, bool ANYHIT, int NTH, int MINBLK>
void bench_prod(const float4 *table, int n_tiles, int *work, float *out, int items_per_cta) {
    const size_t smem = sizeof(Smem);
    cudaFuncSetAttribute(k_prod<R, MODE, ANYHIT, NTH, MINBLK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_prod<R, MODE, ANYHIT, NTH, MINBLK>, NTH, smem);
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, k_prod<R, MODE, ANYHIT, NTH, MINBLK>);
    const int blocks = occ < MINBLK ? occ : MINBLK;
    const int n_blocks = g_sms * blocks * items_per_cta;
    char name[96];
    snprintf(name, sizeof name, "PROD %s%s R=%d %4dthr x%d (occ %d, %3d regs) %d items", MODE == MODE_SHAREDQ ? "SQ  " : MODE == MODE_QBAR ? "QBAR" : "OWNQ",
             ANYHIT ? " any" : "", R, NTH, blocks, occ, fa.numRegs, items_per_cta);
    const double flop = MODE == MODE_SHAREDQ ? 2.0 * (3 + 3 * R) / R : MODE == MODE_QBAR ? 2.0 * (6 + 3 * R) / R : 12.0;
    run(name, [&] { cudaMemset(work, 0, 4); k_prod<R, MODE, ANYHIT, NTH, MINBLK><<<g_sms * blocks, NTH, smem>>>(table, n_tiles, n_blocks, work, out, 1e-3f); },
        (double)n_blocks * NTH * R * TILE * n_tiles, flop, blocks);
}

int main() {
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, 0);
    std::vector<float> h(TILE * 12);
    for (size_t i = 0; i < h.size(); ++i) h[i] = -0.5f - 0.001f * (float)(i % 97); // never a candidate
    float4 *tile_g;
    float *out;
    cudaMalloc(&tile_g, h.size() * 4);
    cudaMemcpy(tile_g, h.data(), h.size() * 4, cudaMemcpyHostToDevice);
    cudaMalloc(&out, 64);
    const int reps = 300;
    printf("-- closest-hit loop (shared q): occupancy sweep\n");
    bench_loop<8, MODE_SHAREDQ, 512, 1, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 512, 2, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 512, 2, 2>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 512, 2, 1>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 512, 2, 8>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 1024, 1, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 256, 2, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 256, 3, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 256, 4, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 256, 5, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 256, 6, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 384, 2, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 384, 3, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 128, 8, 4>(tile_g, out, reps);
    bench_loop<8, MODE_SHAREDQ, 128, 6, 4>(tile_g, out, reps);
    printf("-- rays per thread\n");
    bench_loop<4, MODE_SHAREDQ, 512, 2, 4>(tile_g, out, reps);
    bench_loop<6, MODE_SHAREDQ, 512, 2, 4>(tile_g, out, reps);
    bench_loop<10, MODE_SHAREDQ, 512, 2, 4>(tile_g, out, reps);
    bench_loop<12, MODE_SHAREDQ, 512, 2, 2>(tile_g, out, reps);
    bench_loop<12, MODE_SHAREDQ, 256, 3, 2>(tile_g, out, reps);
    bench_loop<16, MODE_SHAREDQ, 256, 3, 2>(tile_g, out, reps);
    bench_loop<16, MODE_SHAREDQ, 256, 2, 2>(tile_g, out, reps);
    bench_loop<16, MODE_SHAREDQ, 512, 1, 2>(tile_g, out, reps);
    bench_loop<16, MODE_SHAREDQ, 384, 2, 2>(tile_g, out, reps);
    printf("-- any-hit loop (one q-term per thread: qbar + |B| qdelta)\n");
    bench_loop<8, MODE_QBAR, 512, 1, 4>(tile_g, out, reps);
    bench_loop<8, MODE_QBAR, 512, 2, 4>(tile_g, out, reps);
    bench_loop<8, MODE_QBAR, 512, 2, 2>(tile_g, out, reps);
    bench_loop<8, MODE_QBAR, 256, 3, 4>(tile_g, out, reps);
    bench_loop<8, MODE_QBAR, 256, 4, 4>(tile_g, out, reps);
    bench_loop<8, MODE_QBAR, 384, 2, 4>(tile_g, out, reps);
    bench_loop<12, MODE_QBAR, 256, 3, 2>(tile_g, out, reps);
    bench_loop<4, MODE_QBAR, 512, 2, 4>(tile_g, out, reps);
    bench_loop<2, MODE_QBAR, 512, 2, 4>(tile_g, out, reps);
    printf("-- one q per ray (jittered primary rays: 6 FFMA per pair)\n");
    bench_loop<8, MODE_OWNQ, 512, 1, 4>(tile_g, out, reps);
    bench_loop<8, MODE_OWNQ, 512, 2, 4>(tile_g, out, reps);
    bench_loop<8, MODE_OWNQ, 512, 2, 2>(tile_g, out, reps);
    bench_loop<8, MODE_OWNQ, 256, 3, 4>(tile_g, out, reps);
    bench_loop<6, MODE_OWNQ, 512, 2, 4>(tile_g, out, reps);
    {   // production data path
        const int n_tiles = 400;
        std::vector<float> ht((size_t)n_tiles * TILE * 12, 0.f);
        for (size_t i = 0; i < ht.size(); ++i) ht[i] = ((i % 4) == 2) ? -1.f : 0.0001f * (float)(i % 89); // C = -1: never candidate
        float4 *table;
        int *work;
        cudaMalloc(&table, ht.size() * 4);
        cudaMemcpy(table, ht.data(), ht.size() * 4, cudaMemcpyHostToDevice);
        cudaMalloc(&work, 4);
        printf("-- production data path (TMA tile pipeline, per-warp stage recycling), %d tiles per item\n", n_tiles);
        bench_prod<12, MODE_SHAREDQ, false, 256, 2>(table, n_tiles, work, out, 2);
        bench_prod<12, MODE_SHAREDQ, false, 256, 2>(table, n_tiles, work, out, 8);
        bench_prod<8, MODE_SHAREDQ, false, 256, 2>(table, n_tiles, work, out, 2);
        bench_prod<12, MODE_QBAR, true, 256, 2>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_QBAR, true, 256, 2>(table, n_tiles, work, out, 2);
        bench_prod<12, MODE_OWNQ, false, 256, 2>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_SHAREDQ, false, 512, 1>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_SHAREDQ, false, 512, 2>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_SHAREDQ, false, 256, 3>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_SHAREDQ, false, 256, 4>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_QBAR, true, 512, 1>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_QBAR, true, 512, 2>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_QBAR, true, 256, 3>(table, n_tiles, work, out, 2);
        bench_prod<4, MODE_QBAR, true, 512, 2>(table, n_tiles, work, out, 2);
        bench_prod<8, MODE_OWNQ, false, 512, 2>(table, n_tiles, work, out, 2);
    }
    return 0;
}
