// mt19937_host.cpp — internal hooks (tests only, no GPU needed): the device replay of the seeded draws (mt19937.cuh)
// run on the host from the same source — the stream in 227-word steps, the chunked automaton, the per-row hit ordinals.
#include <algorithm>
#include <cstdint>
#include <vector>
#include <cuda_runtime.h> // host compiler: __device__ / __host__ expand to nothing

#include "../../include/tracer_cuda.h"
#include "mt19937.cuh"

namespace {
// y[0 .. n) of std::mt19937(seed), generated step by step as the device's generator does
std::vector<uint32_t> stream(uint32_t seed, int64_t n) {
    std::vector<uint32_t> y((size_t)n);
    uint32_t ring[mt::N], next[mt::STEP];
    mt::seed_ring(seed, ring);
    for (int64_t i0 = 0, base = 0; i0 < n; i0 += mt::STEP, base = (base + mt::STEP) % mt::N) {
        for (int j = 0; j < mt::STEP; ++j) next[j] = mt::step_word(ring, (int)base, j);
        for (int j = 0; j < mt::STEP; ++j) {
            ring[(base + j) % mt::N] = next[j];
            if (i0 + j < n) y[(size_t)(i0 + j)] = mt::temper(next[j]);
        }
    }
    return y;
}
} // namespace

extern "C" {

// out[i] = y[start + i], i < n
void tracer__mt19937_words_host(uint32_t seed, int64_t start, int64_t n, uint32_t *out) {
    const std::vector<uint32_t> y = stream(seed, start + n);
    std::copy(y.begin() + start, y.end(), out);
}

// The device replay's algorithm on a scan-order hit mask: stream of 3*L*T words (T = hits), lengthened while rejections
// leave it short, automaton in chunks of `chunk` words (pass 1, chain, pass 2), gather by hit ordinal.  faceid_scan
// [n_px*L], -1 for misses — what tracer_mt19937_faceids gives in scan order.  Returns the stream words used.
int64_t tracer__mt19937_replay_host(uint32_t seed, int32_t L, const int32_t *faces, int64_t n_px, const uint8_t *hit_scan, int64_t chunk,
                                    int32_t *faceid_scan) {
    std::fill(faceid_scan, faceid_scan + n_px * L, -1);
    int64_t T = 0;
    for (int64_t k = 0; k < n_px; ++k) T += hit_scan[k] != 0;
    if (L == 0 || T == 0 || chunk < 1) return 0;
    std::vector<uint32_t> F((size_t)L), thr((size_t)L);
    for (int l = 0; l < L; ++l) F[l] = (uint32_t)faces[l], thr[l] = mt::threshold(F[l]);
    const int S = 3 * L;
    std::vector<int> fid_ord((size_t)(T * L), -1);
    for (int64_t D = 3 * L * T;;) {
        const std::vector<uint32_t> y = stream(seed, D);
        const int64_t n_chunks = (D + chunk - 1) / chunk;
        std::vector<int> end((size_t)(n_chunks * S)), cnt((size_t)(n_chunks * S)), st((size_t)n_chunks);
        std::vector<int64_t> ord((size_t)n_chunks);
        for (int64_t c = 0; c < n_chunks; ++c)
            for (int s = 0; s < S; ++s) mt::chunk_map(y.data(), D, chunk, c, s, L, F.data(), thr.data(), end.data(), cnt.data());
        const int64_t done = mt::chain(n_chunks, L, end.data(), cnt.data(), st.data(), ord.data());
        if (done < T) {
            D += 3 * L * (T - done) + (D >> 4);
            continue;
        }
        for (int64_t c = 0; c < n_chunks; ++c)
            mt::chunk_faceids(y.data(), D, chunk, c, st[c], ord[c], T, L, F.data(), thr.data(), fid_ord.data());
        int64_t o = 0;
        for (int64_t k = 0; k < n_px; ++k)
            if (hit_scan[k]) std::copy(&fid_ord[(size_t)(o * L)], &fid_ord[(size_t)(o * L)] + L, faceid_scan + k * L), ++o;
        return D;
    }
}

// Hit ordinals of the rows a band selection renders, as the library computes them: own per-row counts, the other rows'
// counts filled in as an exchange would (from the whole mask here), the check of the exchanged counts, the scan over the
// frame's rows, plus the in-row rank.  hit_img [H*W] in image order h*W+w; ord_out [n_rows*W] local order, -1 for misses.
// Returns the number of local rows, or -1 when the exchanged counts fail the library's check.
int tracer__mt19937_band_ordinals_host(int32_t W, int32_t H, int32_t band_rows, int32_t band_index, int32_t band_count,
                                       const uint8_t *hit_img, int64_t *ord_out) {
    const int bi = band_count > 1 ? band_index : 0, br = band_count > 1 ? band_rows : H;
    const int n_rows = tracer_band_row_count(H, band_rows, band_index, band_count);
    if (n_rows < 0) return -1;
    auto hits_in = [&](int pr) {
        int n = 0;
        for (int w = 0; w < W; ++w) n += hit_img[(size_t)(H - 1 - pr) * W + w] != 0;
        return n;
    };
    std::vector<int> local((size_t)n_rows), frame((size_t)H);
    for (int lr = 0; lr < n_rows; ++lr) local[lr] = hits_in(mt::ppm_row(lr, br, bi, band_count));
    mt::own_rows(local.data(), n_rows, br, bi, band_count, frame.data(), H);
    for (int pr = 0; pr < H; ++pr) // the all-reduce: every other row's owner adds its count
        if (band_count > 1 && (pr / br) % band_count != bi) frame[pr] += hits_in(pr);
    if (!mt::rows_valid(local.data(), n_rows, br, bi, band_count, frame.data(), H, W)) return -1;
    std::vector<int64_t> base((size_t)std::max(n_rows, 1));
    mt::row_bases(frame.data(), H, n_rows, br, bi, band_count, base.data());
    for (int lr = 0; lr < n_rows; ++lr) {
        const int h = H - 1 - mt::ppm_row(lr, br, bi, band_count);
        int64_t r = base[lr];
        for (int w = 0; w < W; ++w) ord_out[(size_t)lr * W + w] = hit_img[(size_t)h * W + w] ? r++ : -1;
    }
    return n_rows;
}

} // extern "C"
