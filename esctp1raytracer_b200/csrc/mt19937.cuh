// mt19937.cuh — the seeded serial path's std::mt19937 draws (main.cpp:743-754), replayed on the device.
//
// scan_row consumes one std::mt19937(seed) stream y0, y1, ... in scan order (PPM row 0 = h = H-1 first, w ascending).
// Per hit pixel and light l: faceID = libstdc++'s uniform_int_distribution (Lemire's mapping) over F_l faces, which
// redraws while low < 2^32 mod F_l (tested only when low < F_l), then two outputs for the two uniform_real<float> draws.
// Miss pixels consume nothing.  tracer_mt19937_faceids (tracer_host.cpp) is the sequential statement of this.
//
//   stream      one CTA keeps the 624-word state in shared memory and emits 227 words per step: x[k+624] =
//               x[k+397] ^ twist(x[k], x[k+1]) needs only the current window for k < n+227.
//   automaton   the consumption is a machine of 3L states (light l, phase faceID / real1 / real2); a rejected faceID draw
//               stays in its state, the last phase of the last light completes a hit pixel.  Pass 1 simulates every chunk
//               of the stream from every state (end state, hits completed); a walk over the chunks' maps gives each
//               chunk's true start state and first hit ordinal; pass 2 re-simulates each chunk from it and writes the
//               faceIDs by hit ordinal.  Exact for any F, however often draws reject.
//   ordinals    a hit pixel's place in the stream: hits in all earlier PPM rows of the frame + hits before it in its row.
//               Per-row counts are the only thing a banded render needs from the other bands.
//
// __host__ __device__ throughout: mt19937_host.cpp builds the same functions for the host (tests/test_mt19937_replay.py).
#pragma once
#include <cstdint>
#include <vector>
#ifdef __CUDACC__
#include <cub/block/block_scan.cuh>
#endif

namespace mt {

constexpr int N = 624, M = 397, STEP = N - M; // words per step of the stream generator
constexpr uint32_t MATRIX_A = 0x9908b0dfu;

__host__ __device__ __forceinline__ uint32_t seed_word(uint32_t prev, uint32_t i) { return 1812433253u * (prev ^ (prev >> 30)) + i; }

// x[k+624] from x[k], x[k+1] and x[k+397]
__host__ __device__ __forceinline__ uint32_t twist(uint32_t xk, uint32_t xk1, uint32_t xkm) {
    const uint32_t y = (xk & 0x80000000u) | (xk1 & 0x7fffffffu);
    return xkm ^ (y >> 1) ^ ((y & 1u) ? MATRIX_A : 0u);
}

__host__ __device__ __forceinline__ uint32_t temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    return y ^ (y >> 18);
}

// ring[k % 624] holds x[k] for the window x[n .. n+623]; word j < STEP of the step at n is x[n+624+j], which the caller
// stores into ring[(n+j) % 624] only after every word of the step has been read: word j reads x[n+j+1], the slot word j+1
// overwrites.  Stream output y_i = temper(x[624+i]), so the step at n = STEP*s emits y[STEP*s .. STEP*s+226].
__host__ __device__ __forceinline__ uint32_t step_word(const uint32_t *ring, int base, int j) {
    int a = base + j, b = a + 1, c = a + M;
    a -= a >= N ? N : 0, b -= b >= N ? N : 0, c -= c >= N ? N : 0;
    return twist(ring[a], ring[b], ring[c]);
}

__host__ __device__ __forceinline__ void seed_ring(uint32_t seed, uint32_t *ring) {
    ring[0] = seed;
    for (int i = 1; i < N; ++i) ring[i] = seed_word(ring[i - 1], (uint32_t)i);
}

// Lemire rejection threshold of libstdc++'s uniform_int_distribution over F values: 2^32 mod F (0 for F = 0, which then
// maps every draw to 0 as the host replay does)
__host__ __device__ __forceinline__ uint32_t threshold(uint32_t F) { return F ? (0u - F) % F : 0u; }

// The automaton over words y[0 .. n) from state 3*l + phase.  faceid(hit, l, fid) is called for every accepted faceID
// draw, hit counting the hit pixels completed since the start.  Returns the end state; hits += completed pixels.
// F and thr: [L] face counts and their thresholds.
template <class Emit>
__host__ __device__ __forceinline__ int run(const uint32_t *y, int64_t n, int state, int L, const uint32_t *F, const uint32_t *thr,
                                            int64_t &hits, Emit faceid) {
    int l = state / 3, ph = state - 3 * l;
    for (int64_t i = 0; i < n; ++i) {
        if (ph == 0) {
            const uint64_t p = (uint64_t)y[i] * F[l];
            const uint32_t low = (uint32_t)p;
            if (low < F[l] && low < thr[l]) continue; // rejected: the next word is a new faceID draw
            faceid(hits, l, (int)(p >> 32));
            ph = 1;
        } else if (ph == 1) {
            ph = 2;
        } else {
            ph = 0;
            if (++l == L) l = 0, ++hits;
        }
    }
    return 3 * l + ph;
}

// Pass 1, chunk c (words [c*C, min((c+1)*C, D))) from start state s of S = 3L: end[c*S+s], cnt[c*S+s] = hits completed
__host__ __device__ __forceinline__ void chunk_map(const uint32_t *y, int64_t D, int64_t C, int64_t c, int s, int L, const uint32_t *F,
                                                   const uint32_t *thr, int *end, int *cnt) {
    const int64_t w0 = c * C, n = (w0 + C < D ? w0 + C : D) - w0;
    int64_t hits = 0;
    end[c * 3 * L + s] = run(y + w0, n, s, L, F, thr, hits, [](int64_t, int, int) {});
    cnt[c * 3 * L + s] = (int)hits;
}

// The walk over the chunks' maps from state 0 at ordinal 0: every chunk's true start; returns the hits the stream completes
__host__ __device__ __forceinline__ int64_t chain(int64_t n_chunks, int L, const int *end, const int *cnt, int *start_state, int64_t *start_ord) {
    int st = 0;
    int64_t ord = 0;
    for (int64_t c = 0; c < n_chunks; ++c) {
        start_state[c] = st, start_ord[c] = ord;
        ord += cnt[c * 3 * L + st];
        st = end[c * 3 * L + st];
    }
    return ord;
}

// Pass 2, chunk c from its true start: fid_ord[ordinal*L + l] for every hit ordinal < T whose faceID it draws
__host__ __device__ __forceinline__ void chunk_faceids(const uint32_t *y, int64_t D, int64_t C, int64_t c, int state, int64_t ord0, int64_t T,
                                                       int L, const uint32_t *F, const uint32_t *thr, int *fid_ord) {
    const int64_t w0 = c * C, n = (w0 + C < D ? w0 + C : D) - w0;
    int64_t hits = 0;
    run(y + w0, n, state, L, F, thr, hits, [&](int64_t h, int l, int fid) {
        if (ord0 + h < T) fid_ord[(ord0 + h) * L + l] = fid;
    });
}

// ---- hit ordinals (host) -------------------------------------------------------------------------------------------------
// PPM row of local row lr of the band selection (band_count <= 1: the whole frame), as trk::Bands::map orders them
inline int ppm_row(int lr, int band_rows, int band_index, int band_count) {
    if (band_count <= 1) return lr;
    const int lb = lr / band_rows;
    return (band_index + lb * band_count) * band_rows + (lr - lb * band_rows);
}

// this call's per-local-row hit counts -> the frame's [H] row counts, other rows 0 (what the exchange hook receives)
inline void own_rows(const int *local, int n_rows, int band_rows, int band_index, int band_count, int *frame, int H) {
    for (int r = 0; r < H; ++r) frame[r] = 0;
    for (int lr = 0; lr < n_rows; ++lr) frame[ppm_row(lr, band_rows, band_index, band_count)] = local[lr];
}

// after the exchange: own rows unchanged, every count in [0, W]
inline bool rows_valid(const int *local, int n_rows, int band_rows, int band_index, int band_count, const int *frame, int H, int W) {
    for (int r = 0; r < H; ++r)
        if (frame[r] < 0 || frame[r] > W) return false;
    for (int lr = 0; lr < n_rows; ++lr)
        if (frame[ppm_row(lr, band_rows, band_index, band_count)] != local[lr]) return false;
    return true;
}

// first hit ordinal of every local row (an exclusive scan over the frame's rows), and the frame's hit count
inline int64_t row_bases(const int *frame, int H, int n_rows, int band_rows, int band_index, int band_count, int64_t *base) {
    std::vector<int64_t> ex((size_t)H + 1, 0);
    for (int r = 0; r < H; ++r) ex[r + 1] = ex[r] + frame[r];
    for (int lr = 0; lr < n_rows; ++lr) base[lr] = ex[ppm_row(lr, band_rows, band_index, band_count)];
    return ex[H];
}

#ifdef __CUDACC__
// ---- kernels ---------------------------------------------------------------------------------------------------------------
constexpr int GEN_THREADS = 256, SCAN_THREADS = 256, AUTO_THREADS = 128;

// y[0 .. n) of std::mt19937(seed): one CTA, STEP words per step
__global__ void __launch_bounds__(GEN_THREADS) stream_kernel(uint32_t seed, int64_t n, uint32_t *__restrict__ y) {
    __shared__ uint32_t ring[N];
    if (threadIdx.x == 0) seed_ring(seed, ring);
    __syncthreads();
    const int j = threadIdx.x;
    int base = 0;
    for (int64_t i0 = 0; i0 < n; i0 += STEP) {
        const uint32_t v = j < STEP ? step_word(ring, base, j) : 0u;
        __syncthreads(); // every word of the step read before any slot is overwritten
        if (j < STEP) {
            const int slot = base + j - (base + j >= N ? N : 0);
            ring[slot] = v;
            if (i0 + j < n) y[i0 + j] = temper(v);
        }
        __syncthreads();
        base += STEP - (base + STEP >= N ? N : 0);
    }
}

// one CTA per local row: rank[k] = hits before pixel k in its row, row_hits[lr] = the row's hits (hit: hit_tri >= 0)
__global__ void __launch_bounds__(SCAN_THREADS) row_rank_kernel(const int *__restrict__ hit_tri, int W, int *__restrict__ rank,
                                                                int *__restrict__ row_hits) {
    using Scan = cub::BlockScan<int, SCAN_THREADS>;
    __shared__ typename Scan::TempStorage tmp;
    const size_t row = (size_t)blockIdx.x * W;
    int carry = 0;
    for (int w0 = 0; w0 < W; w0 += SCAN_THREADS) {
        const int w = w0 + threadIdx.x;
        int ex, tot;
        Scan(tmp).ExclusiveSum(w < W && hit_tri[row + w] >= 0 ? 1 : 0, ex, tot);
        if (w < W) rank[row + w] = carry + ex;
        carry += tot;
        __syncthreads(); // tmp is reused
    }
    if (threadIdx.x == 0) row_hits[blockIdx.x] = carry;
}

// lights = F[L] then thr[L]
__global__ void chunk_map_kernel(const uint32_t *__restrict__ y, int64_t D, int64_t C, int64_t n_chunks, int L,
                                 const uint32_t *__restrict__ lights, int *__restrict__ end, int *__restrict__ cnt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_chunks * 3 * L) chunk_map(y, D, C, t / (3 * L), (int)(t % (3 * L)), L, lights, lights + L, end, cnt);
}

// ord[n_chunks] = the hits the whole stream completes
__global__ void chain_kernel(int64_t n_chunks, int L, const int *__restrict__ end, const int *__restrict__ cnt, int *__restrict__ start,
                             int64_t *__restrict__ ord) {
    ord[n_chunks] = chain(n_chunks, L, end, cnt, start, ord);
}

__global__ void chunk_faceids_kernel(const uint32_t *__restrict__ y, int64_t D, int64_t C, int64_t n_chunks, int64_t T, int L,
                                     const uint32_t *__restrict__ lights, const int *__restrict__ start, const int64_t *__restrict__ ord,
                                     int *__restrict__ fid_ord) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_chunks) chunk_faceids(y, D, C, c, start[c], ord[c], T, L, lights, lights + L, fid_ord);
}

// faceid[k*L + l] of every hit local pixel k: its hit ordinal = base[local row] + rank[k]
__global__ void gather_kernel(const int *__restrict__ hit_tri, int W, int n_px, int L, const int64_t *__restrict__ base,
                              const int *__restrict__ rank, const int *__restrict__ fid_ord, int *__restrict__ faceid) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_px || hit_tri[k] < 0) return;
    const int64_t o = base[k / W] + rank[k];
    for (int l = 0; l < L; ++l) faceid[(size_t)k * L + l] = fid_ord[o * L + l];
}
#endif

} // namespace mt
