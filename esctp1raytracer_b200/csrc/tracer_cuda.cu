// tracer_cuda.cu — C ABI (include/tracer_cuda.h) over the sm_100a kernels.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/tracer_cuda.h"
#include <cub/device/device_radix_sort.cuh>
#include <dlfcn.h>
#include <nccl.h>
#include <thread>

#include "kernels.cuh"

// Internal (tests only, no GPU needed): the row construction of build_origin_table and the sweeps' per-ray tests,
// compiled for the host from the same source.  rows9 = three exact rows (A, B, C); row8 = lo.xyzw, hi.xyzw.
extern "C" void tracer__span_rows(const double *rows9, float *row8) {
    double rows[3][3];
    for (int i = 0; i < 9; ++i) rows[i / 3][i % 3] = rows9[i];
    float4 lo, hi;
    trk::span_rows(rows, lo, hi);
    row8[0] = lo.x, row8[1] = lo.y, row8[2] = lo.z, row8[3] = lo.w, row8[4] = hi.x, row8[5] = hi.y, row8[6] = hi.z, row8[7] = hi.w;
}
// qdelta < 0: the ray's own q (candidate path); else the hot loop's shared-q form (q = qbar, bounds widened by |B| qdelta)
extern "C" int tracer__span_pass(const float *row8, float p, float q, float qdelta) {
    const float4 lo = make_float4(row8[0], row8[1], row8[2], row8[3]), hi = make_float4(row8[4], row8[5], row8[6], row8[7]);
    const float ps = p * sweep::SPAN_S;
    if (qdelta < 0.f) return sweep::span_pass(lo, hi, ps, q) ? 1 : 0;
    float ax, ay;
    sweep::span_terms_qbar(lo, hi, q, qdelta, ax, ay);
    return fminf(ps + ax, ay - ps) >= 1.f ? 1 : 0;
}

// The whole row construction of build_origin_table for ONE triangle (tri9: its 9 vertex floats).  tp18 = origin[3], U[3], V[3],
// W[3] of the direction parametrisation d' = p*U + q*V + W, then dmax >= |d'| and lmax (the reach bound of the table).
// out20 = rb, rc, rd (three-row form), lo, hi (span row).
extern "C" void tracer__origin_rows(const float *tri9, const double *tp14, float *out20) {
    trk::TableParam tp{};
    for (int i = 0; i < 3; ++i) tp.o[i] = tp14[i], tp.U[i] = tp14[3 + i], tp.V[i] = tp14[6 + i], tp.W[i] = tp14[9 + i];
    tp.dmax = tp14[12], tp.lmax = tp14[13];
    float4 r[5];
    trk::origin_rows(tri9, tp, true, r[0], r[1], r[2], r[3], r[4]);
    for (int i = 0; i < 5; ++i) out20[4 * i] = r[i].x, out20[4 * i + 1] = r[i].y, out20[4 * i + 2] = r[i].z, out20[4 * i + 3] = r[i].w;
}
// n rays (p, q) against the rows of one triangle: bit 0 = the three-row test (sweep::edge_pass), bit 1 = the span test with
// the ray's own q (sweep::span_pass), bit 2 = the span test in the hot loop's shared-q form (q = qbar, bounds widened by
// |B| * qdelta; only meaningful when |q - qbar| <= qdelta)
extern "C" void tracer__filter_pass(const float *rows20, int n, const float *p, const float *q, float qbar, float qdelta, unsigned char *out) {
    float4 rr[5];
    for (int i = 0; i < 5; ++i) rr[i] = make_float4(rows20[4 * i], rows20[4 * i + 1], rows20[4 * i + 2], rows20[4 * i + 3]);
    float ax, ay;
    sweep::span_terms_qbar(rr[3], rr[4], qbar, qdelta, ax, ay);
    for (int i = 0; i < n; ++i) {
        const float ps = p[i] * sweep::SPAN_S;
        out[i] = (unsigned char)((sweep::edge_pass(rr[0], rr[1], rr[2], p[i], q[i]) ? 1 : 0) | (sweep::span_pass(rr[3], rr[4], ps, q[i]) ? 2 : 0) |
                                 (fminf(ps + ax, ay - ps) >= 1.f ? 4 : 0));
    }
}

// Internal (tests only): strict::powf_glibc as the device computes it, for every stride-th float bit pattern x from
// lo_bits up to hi_bits (inclusive) -> host_out[(hi_bits - lo_bits) / stride + 1], or for n (x, y) pairs.  Runs on the
// current device (tracer_cuda_init first) in chunks; tests/test_gpu_specular.py compares with the host build.
__global__ void powf_range_kernel(uint32_t lo_bits, uint32_t stride, uint32_t n, float y, float *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = strict::powf_glibc(__uint_as_float(lo_bits + i * stride), y);
}
__global__ void powf_pairs_kernel(const float *x, const float *y, uint32_t n, float *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = strict::powf_glibc(x[i], y[i]);
}
extern "C" int tracer__device_powf(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride, float y, float *host_out);
extern "C" int tracer__device_powf_pairs(int64_t n, const float *x, const float *y, float *host_out);

extern "C" int tracer__mt19937_scan(uint32_t seed, int32_t n_lights, const int32_t *faces_per_light, int64_t n_px,
                                    const uint8_t *hit_scan, int32_t *faceid_scan);

namespace {


thread_local std::string g_err = "";

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CK_CUDA(call)                                                                                       \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess)                                                                              \
            return fail(TRACER_ERR_CUDA, std::string(#call) + " failed (tracer_cuda.cu:" + std::to_string(__LINE__) + "): " + cudaGetErrorString(e_)); \
    } while (0)

// A cudaMalloc'ed buffer of the test hooks, freed on every return path.
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
};

// Device-memory pool: the drop-in call (tracer_cuda_render) creates and destroys a resident scene per
// frame; cudaMalloc/cudaFree of a few GB of tables and workspace would cost more than the upload itself.
// Freed blocks are kept (up to a quarter of the device memory) and handed out again by size.
struct Pool {
    std::mutex mu;
    std::unordered_map<void *, size_t> live;     // pointer -> bytes of blocks handed out
    std::multimap<size_t, void *> free_blocks;   // bytes -> pointer
    size_t cached = 0, limit = 0;
    void *alloc(size_t bytes) {
        bytes = (bytes + 255) & ~(size_t)255;
        std::lock_guard<std::mutex> lk(mu);
        auto it = free_blocks.lower_bound(bytes);
        if (it != free_blocks.end() && it->first <= bytes + bytes / 2 + (1 << 20)) {
            void *p = it->second;
            cached -= it->first;
            live[p] = it->first;
            free_blocks.erase(it);
            return p;
        }
        void *p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) {
            cudaGetLastError();
            release_all_locked(); // make room and retry once
            if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
        }
        live[p] = bytes;
        return p;
    }
    void release(void *p) {
        if (!p) return;
        std::lock_guard<std::mutex> lk(mu);
        auto it = live.find(p);
        if (it == live.end()) {
            cudaFree(p);
            return;
        }
        const size_t bytes = it->second;
        live.erase(it);
        if (cached + bytes <= limit) {
            free_blocks.insert({bytes, p});
            cached += bytes;
        } else {
            cudaFree(p);
        }
    }
    void release_all_locked() {
        for (auto &kv : free_blocks) cudaFree(kv.second);
        free_blocks.clear();
        cached = 0;
    }
    void release_all() {
        std::lock_guard<std::mutex> lk(mu);
        release_all_locked();
    }
};

// One context per GPU.  tracer_cuda_init(d) sets up device d and makes it the process's CURRENT context (what
// scene_create uses); tracer_cuda_init_multi sets up several.  A resident scene remembers its context.
constexpr int MAX_GPUS = 16;
struct Ctx {
    bool inited = false;
    int device = -1;
    int n_sms = 0;
    cudaStream_t stream = nullptr;
    cudaDeviceProp prop{};
    Pool pool;
    int sl_ctas[2] = {0, 0}; // co-resident CTAs per SM of shadow_light_kernel<false/true> (cooperative launch limit)
} g_ctx[MAX_GPUS];
Ctx *g_cur = nullptr;
thread_local Pool *t_pool = nullptr; // pool of the context the calling thread is working on

template <typename T>
int dev_alloc(T **p, size_t n) {
    if (n == 0) n = 1;
    *p = (T *)t_pool->alloc(n * sizeof(T));
    if (!*p) return fail(TRACER_ERR_NOMEM, "device memory allocation of " + std::to_string((n * sizeof(T)) >> 20) + " MiB failed");
    return 0;
}
template <typename T>
void dev_free(T *&p) {
    t_pool->release((void *)p);
    p = nullptr;
}

}  // namespace

struct tracer_scene_multi {
    std::vector<tracer_scene_dev *> dev; // one replica per GPU
    tracer_frame_stats stats{};
};

struct tracer_scene_dev {
    Ctx *ctx = nullptr;
    int n_geoms = 0, n_tris = 0, n_pad = 0, n_lights = 0, n_spheres = 0, V = 0;
    float *tri_verts = nullptr, *tri_normals = nullptr, *geom_material = nullptr, *sphere_material = nullptr;
    int *tri_geom = nullptr, *geom_has_normals = nullptr;
    float4 *spheres = nullptr;
    int *light_vbase = nullptr;
    float *light_verts = nullptr;
    std::vector<int> h_light_vbase, h_light_F;
    std::vector<float> h_light_verts;
    double bb_lo[3], bb_hi[3];
    float4 *eye_table = nullptr, *light_tables = nullptr, *allcand_table = nullptr; // 48-byte three-row tables
    float4 *eye_span = nullptr, *light_spans = nullptr, *allcand_span = nullptr;    // 32-byte span tables (same slots)
    std::vector<double> table_lmax; // per (light vertex, cube face): reach bound it was built for, < 0 = not built
    int table_slots = 1;            // light vertices whose 6 face tables fit at once (and per persistent-kernel launch)
    bool tables_resident = true;    // every light vertex has its own slot: tables are kept across lights and frames
    bool allcand_built = false;
    size_t table_stride = 0, span_stride = 0; // float4 per table
    // per-frame workspace
    int ws_npx = 0, ws_L = 0;
    int *hit_tri = nullptr, *rj = nullptr, *list = nullptr, *list_b = nullptr, *faceid = nullptr, *dbg_occ = nullptr;
    unsigned long long *best = nullptr, *best_occ = nullptr;
    float *hit_t = nullptr, *hit_v = nullptr, *carry = nullptr, *nrm = nullptr, *accum = nullptr, *ro = nullptr,
          *rd = nullptr, *re = nullptr, *rt = nullptr;
    uint8_t *rgb8 = nullptr, *mask = nullptr;
    float *accum_total = nullptr;
    // bundle-cull mode: candidate (ray<<32|triangle) buffers, their count, radix-sort scratch
    unsigned long long *cand_a = nullptr, *cand_b = nullptr, *cand_count = nullptr, *rkey = nullptr, *rkey_sorted = nullptr;
    int *blk_cnt = nullptr;            // order-preserving compaction: survivors per (group, block of CBLK entries)
    size_t blk_cnt_cap = 0;
    cull::BlockBoxes *boxes = nullptr; // two-phase bundle cull: boxes of every ray block
    size_t boxes_cap = 0;
    int *iota = nullptr;
    size_t pair_bytes = 0;
    void *pair_tmp = nullptr;
    int rkey_npx = 0;
    size_t cand_cap = 0, sort_bytes = 0;
    int cull_grow = 1; // candidate buffers hold 24 * cull_grow pairs per ray (grown after an overflow)
    void *sort_tmp = nullptr;
    int *seg_count = nullptr, *seg_off = nullptr, *blk_off = nullptr, *cursor = nullptr, *cnt_b = nullptr, *work = nullptr,
        *n_slices = nullptr;
    int maxF = 0;
    sweep::Counters *counters = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> ev_shadow;
    tracer_frame_stats stats{};
};

namespace {

int ensure_workspace(tracer_scene_dev *s, int n_px, bool want_dbg_occ) {
    const int L = std::max(1, s->n_lights);
    if (n_px > s->ws_npx) {
        dev_free(s->hit_tri), dev_free(s->rj), dev_free(s->best), dev_free(s->best_occ), dev_free(s->list), dev_free(s->list_b);
        dev_free(s->faceid), dev_free(s->hit_t), dev_free(s->hit_v), dev_free(s->carry), dev_free(s->nrm), dev_free(s->accum);
        dev_free(s->ro), dev_free(s->rd), dev_free(s->re), dev_free(s->rt), dev_free(s->rgb8), dev_free(s->mask);
        dev_free(s->dbg_occ), dev_free(s->accum_total);
        s->ws_npx = 0;
        const size_t n = (size_t)n_px;
        int rc = 0;
        rc |= dev_alloc(&s->hit_tri, n) | dev_alloc(&s->rj, n) | dev_alloc(&s->best, n) | dev_alloc(&s->best_occ, n);
        rc |= dev_alloc(&s->list, n);
        rc |= dev_alloc(&s->list_b, n);
        rc |= dev_alloc(&s->faceid, n * L);
        rc |= dev_alloc(&s->hit_t, n) | dev_alloc(&s->hit_v, n) | dev_alloc(&s->carry, n);
        rc |= dev_alloc(&s->nrm, 3 * n) | dev_alloc(&s->accum, 3 * n + 16) | dev_alloc(&s->ro, 3 * n);
        rc |= dev_alloc(&s->rd, 3 * n) | dev_alloc(&s->re, 2 * n) | dev_alloc(&s->rt, n);
        rc |= dev_alloc(&s->rgb8, 3 * n + 64) | dev_alloc(&s->mask, n);
        if (rc) return TRACER_ERR_NOMEM;
        s->ws_npx = n_px;
    }
    if (want_dbg_occ && !s->dbg_occ) {
        if (dev_alloc(&s->dbg_occ, (size_t)s->ws_npx * L)) return TRACER_ERR_NOMEM;
    }
    return 0;
}

template <int R, bool EX, int MODE>
int launch_primary_q(const trk::PrimaryParams &p, int grid, cudaStream_t st) {
    const size_t smem = sizeof(sweep::SmemT<sweep::Rows<MODE>::N>);
    CK_CUDA(cudaFuncSetAttribute(trk::primary_kernel<R, EX, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    trk::primary_kernel<R, EX, MODE><<<grid, sweep::NT, smem, st>>>(p);
    CK_CUDA(cudaGetLastError());
    return 0;
}
int scene_create_on(Ctx &g, const tracer_scene_flat *sc, tracer_scene_dev **out);

// NCCL is needed by the multi-GPU entry points only: resolved at tracer_cuda_init_multi, so that a single-GPU user
// (and a box without NCCL) never touches it.  Types come from <nccl.h>; libnccl.so.2 is whichever copy the process
// already maps (torch bundles one) or the system's.
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string &err) {
        if (lib) return true;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) {
            err = std::string("multi-GPU needs NCCL: ") + dlerror();
            return false;
        }
        auto sym = [&](const char *n) { return dlsym(lib, n); };
        CommInitAll = (decltype(CommInitAll))sym("ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
        GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
        Send = (decltype(Send))sym("ncclSend");
        Recv = (decltype(Recv))sym("ncclRecv");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
        if (!CommInitAll || !CommDestroy || !GroupStart || !GroupEnd || !Send || !Recv || !GetErrorString) {
            err = "libnccl lacks a symbol this library needs";
            lib = nullptr;
            return false;
        }
        return true;
    }
} g_nccl;

struct Multi {
    int n = 0; // GPUs set up by tracer_cuda_init_multi (0: not called)
    bool have_comms = false;
    ncclComm_t comms[MAX_GPUS] = {};
    uint8_t *band_buf[MAX_GPUS] = {}; // GPU d's packed bands (send buffer), d > 0
    size_t band_cap[MAX_GPUS] = {};
    uint8_t *gathered = nullptr, *frame = nullptr; // GPU 0
    size_t gathered_cap = 0, frame_cap = 0;
} g_multi;

void multi_shutdown() {
    for (int d = 0; d < MAX_GPUS; ++d) {
        if (g_multi.have_comms && g_multi.comms[d] && g_nccl.CommDestroy) g_nccl.CommDestroy(g_multi.comms[d]);
        g_multi.comms[d] = nullptr;
        if (g_multi.band_buf[d] && g_ctx[d].inited) {
            cudaSetDevice(d);
            g_ctx[d].pool.release(g_multi.band_buf[d]);
        }
        g_multi.band_buf[d] = nullptr, g_multi.band_cap[d] = 0;
    }
    if (g_ctx[0].inited) {
        cudaSetDevice(0);
        g_ctx[0].pool.release(g_multi.gathered), g_ctx[0].pool.release(g_multi.frame);
    }
    g_multi.gathered = g_multi.frame = nullptr;
    g_multi.gathered_cap = g_multi.frame_cap = 0;
    g_multi.have_comms = false;
    g_multi.n = 0;
}
constexpr int WORK_INTS = trk::SL_MAXCHUNK + 8; // per-chunk work counters + the grid-barrier counter of the persistent kernel

template <bool EX>
int launch_shadow_light_t(Ctx &g, const trk::ShadowLightParams &p, unsigned *bar, cudaStream_t st) {
    const size_t smem = sizeof(sweep::SmemT<2>);
    int &ctas_per_sm = g.sl_ctas[EX ? 1 : 0]; // co-resident CTAs: a cooperative launch may not exceed them
    if (!ctas_per_sm) {
        CK_CUDA(cudaFuncSetAttribute(trk::shadow_light_kernel<EX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, trk::shadow_light_kernel<EX>, sweep::NT, smem));
        if (ctas_per_sm < 1) return fail(TRACER_ERR_CUDA, "shadow_light_kernel does not fit on an SM");
        ctas_per_sm = std::min(ctas_per_sm, sweep::MINB);
    }
    void *args[] = {(void *)&p, (void *)&bar};
    CK_CUDA(cudaLaunchCooperativeKernel((const void *)trk::shadow_light_kernel<EX>, dim3((unsigned)(ctas_per_sm * g.n_sms)), dim3(sweep::NT), args, smem, st));
    return 0;
}
int launch_shadow_light(Ctx &g, bool ex, const trk::ShadowLightParams &p, unsigned *bar, cudaStream_t st) {
    return ex ? launch_shadow_light_t<true>(g, p, bar, st) : launch_shadow_light_t<false>(g, p, bar, st);
}
// qmode: sweep::MODE_SHAREDQ (no jitter), MODE_QBAR (jittered samples, span table) or MODE_OWNQ (jittered, three-row table)
int launch_primary(int R, bool ex, int qmode, const trk::PrimaryParams &p, int grid, cudaStream_t st) {
    constexpr int OQ = sweep::MODE_OWNQ, SQ = sweep::MODE_SHAREDQ, QB = sweep::MODE_QBAR;
    if (qmode == OQ) { // every ray its own q, three-row table
        if (R == 12) return ex ? launch_primary_q<12, true, OQ>(p, grid, st) : launch_primary_q<12, false, OQ>(p, grid, st);
        if (R == 8) return ex ? launch_primary_q<8, true, OQ>(p, grid, st) : launch_primary_q<8, false, OQ>(p, grid, st);
        if (R == 4) return ex ? launch_primary_q<4, true, OQ>(p, grid, st) : launch_primary_q<4, false, OQ>(p, grid, st);
        return ex ? launch_primary_q<2, true, OQ>(p, grid, st) : launch_primary_q<2, false, OQ>(p, grid, st);
    }
    if (qmode == QB) {
        if (R == 32) return ex ? launch_primary_q<32, true, QB>(p, grid, st) : launch_primary_q<32, false, QB>(p, grid, st);
        if (R == 16) return ex ? launch_primary_q<16, true, QB>(p, grid, st) : launch_primary_q<16, false, QB>(p, grid, st);
        if (R == 8) return ex ? launch_primary_q<8, true, QB>(p, grid, st) : launch_primary_q<8, false, QB>(p, grid, st);
        if (R == 4) return ex ? launch_primary_q<4, true, QB>(p, grid, st) : launch_primary_q<4, false, QB>(p, grid, st);
        return ex ? launch_primary_q<2, true, QB>(p, grid, st) : launch_primary_q<2, false, QB>(p, grid, st);
    }
    if (R == 32) return ex ? launch_primary_q<32, true, SQ>(p, grid, st) : launch_primary_q<32, false, SQ>(p, grid, st);
    if (R == 24) return ex ? launch_primary_q<24, true, SQ>(p, grid, st) : launch_primary_q<24, false, SQ>(p, grid, st);
    if (R == 16) return ex ? launch_primary_q<16, true, SQ>(p, grid, st) : launch_primary_q<16, false, SQ>(p, grid, st);
    if (R == 8) return ex ? launch_primary_q<8, true, SQ>(p, grid, st) : launch_primary_q<8, false, SQ>(p, grid, st);
    if (R == 4) return ex ? launch_primary_q<4, true, SQ>(p, grid, st) : launch_primary_q<4, false, SQ>(p, grid, st);
    return ex ? launch_primary_q<2, true, SQ>(p, grid, st) : launch_primary_q<2, false, SQ>(p, grid, st);
}
// Work decomposition of a sweep: R rays per thread (8 preferred: best amortisation of the row loads) and
// n_slices triangle slices, chosen so that ray blocks x slices keeps every SM busy for several items.
struct Decomp {
    int R, n_blocks, n_slices;
};
// (ray block, triangle slice) work items wanted per resident CTA: the tail of a sweep is at most one item long, and
// an item's set-up (ray parameters; the shadow sweeps gather theirs through the sorted list) is a few microseconds.
// (TRACER_ITEMS_PER_CTA overrides: development knob.)
int items_per_cta() {
    static const int forced = [] {
        const char *e = std::getenv("TRACER_ITEMS_PER_CTA");
        return e ? std::atoi(e) : 0;
    }();
    return forced > 0 ? forced : 96;
}

Decomp pick_decomp(int64_t n_rays, int n_tiles, int n_sms, int forced_R, int extra_blocks, int qmode) {
    const int slices_possible = std::max(1, n_tiles / 4); // at least 4 tiles per slice
    auto blocks_for = [&](int R) {
        return (int)((n_rays + (int64_t)sweep::NT * R - 1) / ((int64_t)sweep::NT * R)) + extra_blocks;
    };
    Decomp d{2, blocks_for(2), 1};
    // rays per thread: span form with one exact q (no jitter) 32, 16, 8, 4 or 2 (24 on request); span form with a shared
    // mean q (jittered samples) 16, 8, 4 or 2; three-row form (own q) 12, 8, 4 or 2
    // (C4 closest-hit sweep on one B200: 997 ms at 16, 944 at 24, 905 at 32)
    const bool own_q = qmode == sweep::MODE_OWNQ;
    const int big = own_q ? 12 : 32, mid = own_q ? 8 : 16;
    if (forced_R == 2 || forced_R == 4 || forced_R == 8 || forced_R == mid || forced_R == big || (qmode == sweep::MODE_SHAREDQ && forced_R == 24)) {
        d.R = forced_R, d.n_blocks = blocks_for(forced_R);
    } else {
        for (int R : {big, mid, 8, 4, 2}) {
            d.R = R, d.n_blocks = blocks_for(R);
            if ((int64_t)d.n_blocks * slices_possible >= 4 * (int64_t)n_sms) break;
        }
    }
    const int64_t ips = (int64_t)items_per_cta() * sweep::MINB;
    const int64_t want = (ips * (int64_t)n_sms + d.n_blocks - 1) / std::max(1, d.n_blocks);
    d.n_slices = d.n_blocks >= ips * n_sms ? 1 : (int)std::max<int64_t>(1, std::min<int64_t>(want, slices_possible));
    return d;
}

// both forms of the filter table of one origin: the 48-byte rows (jittered primary rays, bundle-cull mode) and the
// 32-byte span rows (default sweeps)
int build_table(const tracer_scene_dev *s, const trk::TableParam &tp, float4 *table, float4 *span, cudaStream_t st) {
    const int th = 128;
    trk::build_origin_table<<<(s->n_pad + th - 1) / th, th, 0, st>>>(s->tri_verts, s->n_tris, s->n_pad, tp, table, span);
    CK_CUDA(cudaGetLastError());
    return 0;
}

// cube face f around point o: d' = p*e_a + q*e_b + sg*e_c, c = f/2, a = (c+1)%3, b = (c+2)%3, |d'| <= sqrt(3)
trk::TableParam face_param(const float *o, int f, double lmax) {
    trk::TableParam tp{};
    const int c = f / 2, a = (c + 1) % 3, b = (c + 2) % 3;
    for (int i = 0; i < 3; ++i) tp.o[i] = o[i];
    tp.U[a] = 1.0, tp.V[b] = 1.0, tp.W[c] = (f & 1) ? -1.0 : 1.0;
    tp.dmax = std::sqrt(3.0);
    tp.lmax = lmax;
    return tp;
}

}  // namespace

extern "C" {

const char *tracer_cuda_last_error(void) { return g_err.c_str(); }

}  // extern "C"

namespace {
int init_device(int device_ordinal) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(TRACER_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count=0"));
    if (device_ordinal < 0 || device_ordinal >= n || device_ordinal >= MAX_GPUS) return fail(TRACER_ERR_INVALID, "device ordinal out of range");
    Ctx &g = g_ctx[device_ordinal];
    CK_CUDA(cudaSetDevice(device_ordinal));
    CK_CUDA(cudaGetDeviceProperties(&g.prop, device_ordinal));
    if (g.prop.major < 10)
        return fail(TRACER_ERR_NO_DEVICE, std::string("kernels are built for sm_100a only; device is sm_") +
                                              std::to_string(g.prop.major) + std::to_string(g.prop.minor));
    if (!g.stream) CK_CUDA(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    g.device = device_ordinal;
    g.n_sms = g.prop.multiProcessorCount;
    g.pool.limit = g.prop.totalGlobalMem / 4;
    g.inited = true;
    g_cur = &g;
    t_pool = &g.pool;
    return TRACER_OK;
}
}  // namespace

extern "C" {

int tracer_cuda_init(int device_ordinal) {
    multi_shutdown(); // "use this GPU": ends a multi-GPU set-up, the drop-in call renders on this device again
    return init_device(device_ordinal);
}

void tracer_cuda_shutdown(void) {
    multi_shutdown();
    for (Ctx &g : g_ctx) {
        if (!g.inited) continue;
        cudaSetDevice(g.device);
        g.pool.release_all();
        if (g.stream) cudaStreamDestroy(g.stream);
        g.stream = nullptr;
        g.inited = false;
    }
    g_cur = nullptr;
}

int tracer_cuda_device_info(tracer_device_info *out) {
    if (!out) return fail(TRACER_ERR_INVALID, "null out");
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    const Ctx &g = *g_cur;
    std::memset(out, 0, sizeof *out);
    std::snprintf(out->name, sizeof out->name, "%.127s", g.prop.name);
    out->sm_count = g.prop.multiProcessorCount;
    out->cc_major = g.prop.major, out->cc_minor = g.prop.minor;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g.device);
    out->clock_khz = khz;
    out->total_mem = (int64_t)g.prop.totalGlobalMem;
    out->l2_bytes = g.prop.l2CacheSize;
    return TRACER_OK;
}

int tracer__device_powf(uint32_t lo_bits, uint32_t hi_bits, uint32_t stride, float y, float *host_out) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    if (!host_out || stride == 0 || hi_bits < lo_bits) return fail(TRACER_ERR_INVALID, "tracer__device_powf: bad range");
    const int64_t n = ((int64_t)hi_bits - lo_bits) / stride + 1;
    const int64_t chunk = std::min<int64_t>(n, 1 << 24);
    DevBuf out;
    CK_CUDA(cudaMalloc(&out.p, chunk * sizeof(float)));
    for (int64_t b = 0; b < n; b += chunk) {
        const uint32_t m = (uint32_t)std::min(chunk, n - b);
        powf_range_kernel<<<(m + 255) / 256, 256, 0, g_cur->stream>>>(lo_bits + (uint32_t)(b * stride), stride, m, y, (float *)out.p);
        CK_CUDA(cudaGetLastError());
        CK_CUDA(cudaMemcpyAsync(host_out + b, out.p, m * sizeof(float), cudaMemcpyDeviceToHost, g_cur->stream));
        CK_CUDA(cudaStreamSynchronize(g_cur->stream));
    }
    return TRACER_OK;
}

int tracer__device_powf_pairs(int64_t n, const float *x, const float *y, float *host_out) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    if (n < 0 || (n && (!x || !y || !host_out))) return fail(TRACER_ERR_INVALID, "tracer__device_powf_pairs: bad arguments");
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(n, 1 << 24));
    DevBuf dx, dy, dout;
    CK_CUDA(cudaMalloc(&dx.p, chunk * sizeof(float)));
    CK_CUDA(cudaMalloc(&dy.p, chunk * sizeof(float)));
    CK_CUDA(cudaMalloc(&dout.p, chunk * sizeof(float)));
    cudaStream_t st = g_cur->stream;
    for (int64_t b = 0; b < n; b += chunk) {
        const uint32_t m = (uint32_t)std::min(chunk, n - b);
        CK_CUDA(cudaMemcpyAsync(dx.p, x + b, m * sizeof(float), cudaMemcpyHostToDevice, st));
        CK_CUDA(cudaMemcpyAsync(dy.p, y + b, m * sizeof(float), cudaMemcpyHostToDevice, st));
        powf_pairs_kernel<<<(m + 255) / 256, 256, 0, st>>>((const float *)dx.p, (const float *)dy.p, m, (float *)dout.p);
        CK_CUDA(cudaGetLastError());
        CK_CUDA(cudaMemcpyAsync(host_out + b, dout.p, m * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK_CUDA(cudaStreamSynchronize(st));
    }
    return TRACER_OK;
}

void tracer_cuda_scene_destroy(tracer_scene_dev *s) {
    if (!s) return;
    if (s->ctx) {
        cudaSetDevice(s->ctx->device);
        cudaDeviceSynchronize(); // nothing of this scene is in flight (on any stream) when its blocks return to the pool
        t_pool = &s->ctx->pool;
    }
    dev_free(s->tri_verts), dev_free(s->tri_normals), dev_free(s->geom_material), dev_free(s->sphere_material);
    dev_free(s->tri_geom), dev_free(s->geom_has_normals), dev_free(s->spheres), dev_free(s->light_vbase);
    dev_free(s->light_verts), dev_free(s->eye_table), dev_free(s->light_tables), dev_free(s->allcand_table);
    dev_free(s->eye_span), dev_free(s->light_spans), dev_free(s->allcand_span);
    dev_free(s->hit_tri), dev_free(s->rj), dev_free(s->best), dev_free(s->best_occ), dev_free(s->list), dev_free(s->list_b);
    dev_free(s->faceid), dev_free(s->dbg_occ), dev_free(s->cnt_b), dev_free(s->accum_total);
    dev_free(s->hit_t), dev_free(s->hit_v), dev_free(s->carry), dev_free(s->nrm), dev_free(s->accum);
    dev_free(s->ro), dev_free(s->rd), dev_free(s->re), dev_free(s->rt), dev_free(s->rgb8), dev_free(s->mask);
    dev_free(s->seg_count), dev_free(s->seg_off), dev_free(s->blk_off), dev_free(s->cursor), dev_free(s->work);
    dev_free(s->n_slices);
    dev_free(s->cand_a), dev_free(s->cand_b), dev_free(s->cand_count), dev_free(s->rkey), dev_free(s->rkey_sorted), dev_free(s->iota);
    dev_free(s->boxes), dev_free(s->blk_cnt);
    t_pool->release(s->sort_tmp), t_pool->release(s->pair_tmp);
    dev_free(s->counters);
    for (auto &e : s->ev)
        if (e) cudaEventDestroy(e);
    for (auto &e : s->ev_shadow) cudaEventDestroy(e);
    delete s;
}

int tracer_cuda_scene_create(const tracer_scene_flat *sc, tracer_scene_dev **out) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    return scene_create_on(*g_cur, sc, out);
}

}  // extern "C"

namespace {
int scene_create_on(Ctx &g, const tracer_scene_flat *sc, tracer_scene_dev **out) {
    if (!out) return fail(TRACER_ERR_INVALID, "null out");
    *out = nullptr;
    if (!g.inited) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    t_pool = &g.pool;
    if (!sc || sc->n_geoms < 0 || sc->n_lights < 0 || sc->n_spheres < 0) return fail(TRACER_ERR_INVALID, "bad scene");
    if (sc->n_geoms > 0 && (!sc->geom_tri_offset || !sc->geom_material)) return fail(TRACER_ERR_INVALID, "null scene array");
    const int G = sc->n_geoms;
    const int N = G > 0 ? sc->geom_tri_offset[G] : 0;
    if (N < 0 || (N > 0 && !sc->tri_verts)) return fail(TRACER_ERR_INVALID, "bad triangle arrays");
    for (int g2 = 0; g2 < G; ++g2)
        if (sc->geom_tri_offset[g2] > sc->geom_tri_offset[g2 + 1] || sc->geom_tri_offset[g2] < 0)
            return fail(TRACER_ERR_INVALID, "geom_tri_offset must be non-decreasing");
    if (sc->n_lights > 0 && !sc->light_geom) return fail(TRACER_ERR_INVALID, "null light_geom");
    if (sc->n_spheres > 0 && (!sc->sphere_cr || !sc->sphere_material)) return fail(TRACER_ERR_INVALID, "null sphere arrays");
    bool any_normals = false;
    for (int g2 = 0; g2 < G && sc->geom_has_normals; ++g2) any_normals |= sc->geom_has_normals[g2] != 0;
    if (any_normals && !sc->tri_normals) return fail(TRACER_ERR_INVALID, "geom_has_normals set but tri_normals is null");

    CK_CUDA(cudaSetDevice(g.device));
    auto *s = new tracer_scene_dev();
    s->ctx = &g;
    s->n_geoms = G, s->n_tris = N, s->n_lights = sc->n_lights, s->n_spheres = sc->n_spheres;
    s->n_pad = std::max(1, (N + cull::CTILE - 1) / cull::CTILE) * cull::CTILE; // multiple of both tile sizes
    s->table_stride = (size_t)s->n_pad * 3, s->span_stride = (size_t)s->n_pad * 2;
#define TRY(x)                         \
    do {                               \
        int rc_ = (x);                 \
        if (rc_) {                     \
            tracer_cuda_scene_destroy(s); \
            return rc_;                \
        }                              \
    } while (0)
#define TRY_CUDA(call)                                                                                      \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) {                                                                            \
            tracer_cuda_scene_destroy(s);                                                                   \
            return fail(TRACER_ERR_CUDA, std::string(#call) + " failed (tracer_cuda.cu:" + std::to_string(__LINE__) + "): " + cudaGetErrorString(e_)); \
        }                                                                                                   \
    } while (0)
    TRY(dev_alloc(&s->tri_verts, (size_t)N * 9));
    TRY_CUDA(cudaMemcpyAsync(s->tri_verts, sc->tri_verts, (size_t)N * 9 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
    if (any_normals) {
        TRY(dev_alloc(&s->tri_normals, (size_t)N * 9));
        TRY_CUDA(cudaMemcpyAsync(s->tri_normals, sc->tri_normals, (size_t)N * 9 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
        TRY(dev_alloc(&s->geom_has_normals, (size_t)G));
        TRY_CUDA(cudaMemcpyAsync(s->geom_has_normals, sc->geom_has_normals, (size_t)G * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    }
    TRY(dev_alloc(&s->geom_material, (size_t)G * 13));
    TRY_CUDA(cudaMemcpyAsync(s->geom_material, sc->geom_material, (size_t)G * 13 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
    std::vector<int> tg((size_t)std::max(N, 1)); // lives until the upload has been waited for
    {
        for (int g2 = 0; g2 < G; ++g2)
            for (int t = sc->geom_tri_offset[g2]; t < sc->geom_tri_offset[g2 + 1]; ++t) tg[t] = g2;
        TRY(dev_alloc(&s->tri_geom, (size_t)N));
        TRY_CUDA(cudaMemcpyAsync(s->tri_geom, tg.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    }
    if (sc->n_spheres > 0) {
        TRY(dev_alloc(&s->spheres, (size_t)sc->n_spheres));
        TRY_CUDA(cudaMemcpyAsync(s->spheres, sc->sphere_cr, (size_t)sc->n_spheres * 4 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
        TRY(dev_alloc(&s->sphere_material, (size_t)sc->n_spheres * 13));
        TRY_CUDA(cudaMemcpy(s->sphere_material, sc->sphere_material, (size_t)sc->n_spheres * 13 * sizeof(float),
                            cudaMemcpyHostToDevice));
    }
    // bounding box of everything a ray can start from or end at
    for (int c = 0; c < 3; ++c) s->bb_lo[c] = 1e300, s->bb_hi[c] = -1e300;
    for (size_t i = 0; i < (size_t)N * 3; ++i)
        for (int c = 0; c < 3; ++c) {
            const double x = sc->tri_verts[3 * i + c];
            s->bb_lo[c] = std::min(s->bb_lo[c], x), s->bb_hi[c] = std::max(s->bb_hi[c], x);
        }
    for (int i = 0; i < sc->n_spheres; ++i)
        for (int c = 0; c < 3; ++c) {
            const double x = sc->sphere_cr[4 * i + c], r = std::fabs(sc->sphere_cr[4 * i + 3]);
            s->bb_lo[c] = std::min(s->bb_lo[c], x - r), s->bb_hi[c] = std::max(s->bb_hi[c], x + r);
        }
    // lights: light.vertex[faceID], faceID in [0, F) (main.cpp:743-751) = the first F de-indexed vertices
    s->h_light_vbase.assign(1, 0);
    for (int l = 0; l < sc->n_lights; ++l) {
        const int lg = sc->light_geom[l];
        if (lg < 0 || lg >= G) {
            tracer_cuda_scene_destroy(s);
            return fail(TRACER_ERR_INVALID, "light_geom index out of range");
        }
        const int t0 = sc->geom_tri_offset[lg], F = sc->geom_tri_offset[lg + 1] - t0;
        if (F <= 0) {
            tracer_cuda_scene_destroy(s);
            return fail(TRACER_ERR_INVALID, "light geometry has no faces");
        }
        s->h_light_F.push_back(F);
        for (int f = 0; f < F; ++f)
            for (int c = 0; c < 3; ++c) s->h_light_verts.push_back(sc->tri_verts[9 * (size_t)t0 + 3 * (size_t)f + c]);
        s->h_light_vbase.push_back(s->h_light_vbase.back() + F);
        s->maxF = std::max(s->maxF, F);
    }
    s->V = s->h_light_vbase.back();
    TRY(dev_alloc(&s->light_vbase, s->h_light_vbase.size()));
    TRY_CUDA(cudaMemcpyAsync(s->light_vbase, s->h_light_vbase.data(), s->h_light_vbase.size() * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    TRY(dev_alloc(&s->light_verts, s->h_light_verts.size()));
    TRY_CUDA(cudaMemcpyAsync(s->light_verts, s->h_light_verts.data(), s->h_light_verts.size() * sizeof(float), cudaMemcpyHostToDevice, g.stream));
    {   // Filter tables of the shadow sweeps: 6 cube-face tables of 48 B per triangle for every light vertex.  Two quad
        // lights need 0.6 GB at 1M triangles; an emissive MESH with hundreds of faces would need more than the GPU has.
        // Budget = half of the free HBM: when all vertices fit, every vertex owns a slot and its tables are built once
        // and kept; otherwise the slots are reused batch by batch within each light (rebuilt per frame: O(N) per table,
        // small next to the O(rays x N) sweep it serves).  The reference renders any light size, and so does this.
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t per_vertex = 6 * (s->table_stride + s->span_stride) * sizeof(float4);
        const size_t budget = free_b / 2;
        const char *cap_env = std::getenv("TRACER_TABLE_SLOTS"); // test knob: pretend only this many vertices fit
        size_t fit = std::max<size_t>(1, budget / per_vertex);
        if (cap_env) fit = std::max<size_t>(1, std::min<size_t>(fit, (size_t)std::atoll(cap_env)));
        s->tables_resident = (size_t)s->V <= fit;
        s->table_slots = (int)std::min<size_t>(fit, (size_t)trk::SL_MAXF / trk::NFACE);
    }
    TRY(dev_alloc(&s->eye_table, s->table_stride));
    TRY(dev_alloc(&s->light_tables, s->table_stride * 6 * (size_t)std::max(1, s->tables_resident ? s->V : s->table_slots)));
    TRY(dev_alloc(&s->allcand_table, s->table_stride));
    TRY(dev_alloc(&s->eye_span, s->span_stride));
    TRY(dev_alloc(&s->light_spans, s->span_stride * 6 * (size_t)std::max(1, s->tables_resident ? s->V : s->table_slots)));
    TRY(dev_alloc(&s->allcand_span, s->span_stride));
    s->table_lmax.assign((size_t)6 * s->V, -1.0);
    const size_t n_groups = (size_t)s->maxF * trk::NFACE;
    TRY(dev_alloc(&s->seg_count, n_groups + 1));
    TRY(dev_alloc(&s->seg_off, n_groups + 2));
    TRY(dev_alloc(&s->blk_off, n_groups + 2));
    TRY(dev_alloc(&s->cursor, n_groups + 1));
    TRY(dev_alloc(&s->cnt_b, n_groups + 1));
    TRY(dev_alloc(&s->work, (size_t)WORK_INTS));
    TRY(dev_alloc(&s->n_slices, 1));
    TRY(dev_alloc(&s->counters, 1));
    for (auto &e : s->ev) TRY_CUDA(cudaEventCreate(&e));
    s->ev_shadow.resize(2 * (size_t)std::max(1, s->n_lights));
    for (auto &e : s->ev_shadow) TRY_CUDA(cudaEventCreate(&e));
    // uploads were queued on the context's stream (truly asynchronous from pinned host memory): one wait for all
    if (cudaError_t e_ = cudaStreamSynchronize(g.stream); e_ != cudaSuccess) {
        tracer_cuda_scene_destroy(s);
        return fail(TRACER_ERR_CUDA, std::string("scene upload failed: ") + cudaGetErrorString(e_));
    }
#undef TRY
#undef TRY_CUDA
    *out = s;
    return TRACER_OK;
}
}  // namespace

extern "C" {

int tracer_cuda_render_scene(tracer_scene_dev *s, const tracer_camera *cam, int32_t W, int32_t H,
                             const tracer_render_opts *opts_in, uint8_t *rgb_out) {
    if (!s || !cam || !rgb_out) return fail(TRACER_ERR_INVALID, "null argument");
    if (!s->ctx || !s->ctx->inited) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    Ctx &g = *s->ctx;
    t_pool = &g.pool;
    if (W < 2 || H < 2) return fail(TRACER_ERR_INVALID, "width and height must be >= 2 (the reference divides by W-1, H-1)");
    // per-pixel planes are indexed with int (3 planes of n_px floats): keep 3 * n_px below 2^31
    if ((int64_t)W * H > (int64_t)700 * 1000 * 1000) return fail(TRACER_ERR_INVALID, "frame too large (limit 7e8 pixels per call; render bands)");
    tracer_render_opts o;
    std::memset(&o, 0, sizeof o);
    if (opts_in) std::memcpy(&o, opts_in, std::min<size_t>(sizeof o, opts_in->struct_size ? opts_in->struct_size : sizeof o));
    // extension (parity unpinned): samples_per_pixel = n*n stratified jittered samples per pixel
    int spp_n = 1;
    if (o.samples_per_pixel > 1) {
        spp_n = (int)std::lround(std::sqrt((double)o.samples_per_pixel));
        if (spp_n * spp_n != o.samples_per_pixel || spp_n > 16)
            return fail(TRACER_ERR_INVALID, "samples_per_pixel must be a square number <= 256");
        if (o.rng_mode == TRACER_RNG_MT19937)
            return fail(TRACER_ERR_INVALID, "TRACER_RNG_MT19937 reproduces the 1-sample serial path only");
    }
    const int S = spp_n * spp_n;
    const int band_count = o.band_count <= 1 ? 1 : o.band_count;
    const int band_rows = band_count > 1 ? o.band_rows : H;
    if (band_count > 1 && (band_rows <= 0 || o.band_index < 0 || o.band_index >= band_count))
        return fail(TRACER_ERR_INVALID, "bad band selection");
    if (o.rng_mode == TRACER_RNG_MT19937 && band_count > 1)
        return fail(TRACER_ERR_INVALID, "TRACER_RNG_MT19937 needs the whole frame in one call (band_count <= 1)");
    if (o.rng_mode == TRACER_RNG_EXPLICIT && !o.faceid && s->n_lights > 0)
        return fail(TRACER_ERR_INVALID, "TRACER_RNG_EXPLICIT needs opts->faceid");
    if (o.rng_mode < 0 || o.rng_mode > 2) return fail(TRACER_ERR_INVALID, "bad rng_mode");
    const int n_rows = tracer_band_row_count(H, band_rows, band_count > 1 ? o.band_index : 0, band_count);
    const int n_px = n_rows * W;
    const int L = s->n_lights;
    CK_CUDA(cudaSetDevice(g.device));
    cudaStream_t st = o.cuda_stream ? (cudaStream_t)o.cuda_stream : g.stream;
    std::memset(&s->stats, 0, sizeof s->stats);
    s->stats.n_sms = g.n_sms;
    s->stats.n_pixels = n_px;
    if (n_px == 0) return TRACER_OK;
    if (int rc = ensure_workspace(s, n_px, o.out_occ_tri != nullptr)) return rc;
    int launches = 0;

    trk::Cam dc;
    std::memcpy(dc.o, cam->origin, 12), std::memcpy(dc.llc, cam->lower_left_corner, 12);
    std::memcpy(dc.hor, cam->horizontal, 12), std::memcpy(dc.ver, cam->vertical, 12);
    trk::Bands bands{W, H, band_rows, band_count > 1 ? o.band_index : 0, band_count, n_px};
    bands.spp_n = spp_n, bands.sample = 0, bands.seed = o.seed;

    // reach bound for shadow segments: len_k <= (k+1) * diag(bbox U eye)  (t carries over lights, main.cpp:764)
    double lo[3], hi[3], diag2 = 0;
    for (int c = 0; c < 3; ++c) {
        lo[c] = std::min(s->bb_lo[c], (double)cam->origin[c]), hi[c] = std::max(s->bb_hi[c], (double)cam->origin[c]);
        if (hi[c] >= lo[c]) diag2 += (hi[c] - lo[c]) * (hi[c] - lo[c]);
    }
    // shadow segments of light k are bounded by len_k <= (k+1) * diag: t carries over lights (main.cpp:764)
    const double diag = std::sqrt(diag2) * 1.001 + 1e-30;
    CK_CUDA(cudaEventRecord(s->ev[0], st));
    {   // eye table on the image plane: d'(s,t) = (llc - origin) + s*horizontal + t*vertical (camera.h:31-34)
        trk::TableParam tp{};
        for (int c = 0; c < 3; ++c) {
            tp.o[c] = cam->origin[c], tp.U[c] = cam->horizontal[c], tp.V[c] = cam->vertical[c];
            tp.W[c] = (double)cam->lower_left_corner[c] - (double)cam->origin[c];
        }
        for (int corner = 0; corner < 4; ++corner) { // |d'| is convex in (s,t): its maximum is at a corner
            double n2 = 0;
            for (int c = 0; c < 3; ++c) {
                const double v = tp.W[c] + (corner & 1) * tp.U[c] + (corner >> 1) * tp.V[c];
                n2 += v * v;
            }
            tp.dmax = std::max(tp.dmax, std::sqrt(n2));
        }
        tp.lmax = 0.0;
        if (int rc = build_table(s, tp, s->eye_table, s->eye_span, st)) return rc;
        ++launches;
    }
    CK_CUDA(cudaMemsetAsync(s->counters, 0, sizeof(sweep::Counters), st));
    CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int), st));

    const int n_tiles = s->n_pad / sweep::TILE;
    // bundle_cull: 1 two-phase, 2 streaming, 3 auto = two-phase unless the default sweeps are estimated to be the
    // faster of the two (tiny scenes: the mode has a fixed cost of a few ms in sorts and count read-backs)
    const double est_default_ms = (double)n_px * (double)s->n_tris * (1.0 + 0.25 * L) / 4.0e9;
    // (the optional mode keeps every light vertex's tables resident; a light too big for that renders in the default mode)
    const bool cull = s->tables_resident && (o.bundle_cull == 3 ? est_default_ms > 6.0 : o.bundle_cull != 0);
    if (cull) { // candidate buffers: 24 per ray + slack (a few per ray are typical), sorted with a radix sort
        const size_t cap = (size_t)n_px * 24 * (size_t)s->cull_grow + ((size_t)1 << 22);
        if (cap > s->cand_cap) {
            dev_free(s->cand_a), dev_free(s->cand_b), dev_free(s->cand_count);
            t_pool->release(s->sort_tmp);
            s->sort_tmp = nullptr, s->cand_cap = 0;
            if (dev_alloc(&s->cand_a, cap) || dev_alloc(&s->cand_b, cap) || dev_alloc(&s->cand_count, 1)) return TRACER_ERR_NOMEM;
            CK_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, s->sort_bytes, s->cand_a, s->cand_b, cap, 0, 64, st));
            if (!(s->sort_tmp = t_pool->alloc(s->sort_bytes))) return fail(TRACER_ERR_NOMEM, "sort scratch");
            s->cand_cap = cap;
        }
    }
    // default mode: shadow rays ordered by (group, q) so that the rays of a thread can share a q-term (sweep::MODE_QBAR);
    // bundle-cull mode: ordered by (group, Morton code of (p,q)).  Either way a radix sort of (key, pixel) pairs.
    if (s->rkey_npx < n_px) {
        dev_free(s->rkey), dev_free(s->rkey_sorted), dev_free(s->iota);
        t_pool->release(s->pair_tmp);
        s->pair_tmp = nullptr;
        if (dev_alloc(&s->rkey, (size_t)n_px) || dev_alloc(&s->rkey_sorted, (size_t)n_px) || dev_alloc(&s->iota, (size_t)n_px)) return TRACER_ERR_NOMEM;
        CK_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, s->pair_bytes, s->rkey, s->rkey_sorted, s->iota, s->list, n_px, 0, 64, st));
        if (!(s->pair_tmp = t_pool->alloc(s->pair_bytes))) return fail(TRACER_ERR_NOMEM, "sort scratch");
        trk::iota_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(s->iota, n_px);
        CK_CUDA(cudaGetLastError());
        s->rkey_npx = n_px;
    }
    // two-phase bundle cull (cull.cuh "block lists"): phase A emits block<<32|triangle into cand_a; the sorted
    // keys land in cand_b, which phase B reads while it emits its ray<<32|triangle candidates into cand_a again.
    // Returns the number of keys, or -1 when the survivor lists would not fit (then the streaming kernels run).
    // test knob: pretend the bundle-cull candidate buffer holds only this many pairs (exercises the overflow fallback)
    const char *cand_env = std::getenv("TRACER_CAND_CAP");
    const unsigned long long em_cap = cand_env ? std::min<unsigned long long>((unsigned long long)std::atoll(cand_env), s->cand_cap) : (unsigned long long)s->cand_cap;
    double flop_primary = 0.0; // executed FP32 flops per swept pair of the closest-hit sweep (default mode)
    const bool two_phase = cull && o.bundle_cull != 2;
    int64_t host_tests_primary = 0, host_tests_shadow = 0; // pairs considered by two-phase sweeps (every block x every triangle)
    auto ensure_boxes = [&](size_t n_blocks) -> int {
        if (n_blocks <= s->boxes_cap) return 0;
        dev_free(s->boxes);
        s->boxes_cap = 0;
        if (dev_alloc(&s->boxes, n_blocks)) return TRACER_ERR_NOMEM;
        s->boxes_cap = n_blocks;
        return 0;
    };
    int tri_bits = 1;
    while (((int64_t)1 << tri_bits) < s->n_pad) ++tri_bits;
    auto block_lists = [&](cull::L0Params lp, int max_blocks, long long &n_keys) -> int {
        lp.boxes = s->boxes, lp.keys = s->cand_a, lp.count = s->cand_count, lp.cap = (unsigned long long)s->cand_cap; /* phase-A keys: their own limit (TRACER_L0_CAP) */
        lp.n_tris = s->n_tris, lp.tri_bits = tri_bits, lp.diag = s->counters;
        CK_CUDA(cudaMemsetAsync(s->cand_count, 0, sizeof(unsigned long long), st));
        const dim3 grid((unsigned)((s->n_tris + cull::L0_THREADS - 1) / cull::L0_THREADS), (unsigned)lp.n_groups);
        cull::cull_l0_kernel<<<grid, cull::L0_THREADS, 0, st>>>(lp);
        CK_CUDA(cudaGetLastError());
        unsigned long long n = 0;
        CK_CUDA(cudaMemcpyAsync(&n, s->cand_count, sizeof n, cudaMemcpyDeviceToHost, st));
        CK_CUDA(cudaStreamSynchronize(st));
        CK_CUDA(cudaMemsetAsync(s->cand_count, 0, sizeof(unsigned long long), st));
        launches += 2;
        if (getenv("TRACER_CULL_DIAG")) fprintf(stderr, "cull diag: phase A kept %llu (block, triangle) pairs over %d groups, <= %d blocks\n", n, lp.n_groups, max_blocks);
        const char *cap_env = getenv("TRACER_L0_CAP"); // development/test knob: pretend the key buffer is this small
        if (n > s->cand_cap || (cap_env && n > (unsigned long long)std::atoll(cap_env))) {
            n_keys = -1;
            return 0;
        }
        int blk_bits = 1;
        while ((1 << blk_bits) < max_blocks * (sweep::THREADS / 32)) ++blk_bits; // keys name a (block, warp)
        if (n) CK_CUDA(cub::DeviceRadixSort::SortKeys(s->sort_tmp, s->sort_bytes, s->cand_a, s->cand_b, n, 0, tri_bits + blk_bits, st));
        n_keys = (long long)n;
        return 0;
    };
    double ms_primary_acc = 0, ms_shadow_acc = 0;
    if (S > 1 && !s->accum_total && dev_alloc(&s->accum_total, 3 * (size_t)s->ws_npx)) return TRACER_ERR_NOMEM;
    for (int smp = 0; smp < S; ++smp) {
    bands.sample = smp;
    const uint32_t seed_s = o.seed + (uint32_t)smp * 0x9e3779b1u; // faceID stream of this sample
    // ---- primary: raygen + closest hit ----------------------------------------------
    CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int), st));
    CK_CUDA(cudaMemsetAsync(s->best, 0xff, sizeof(unsigned long long) * (size_t)n_px, st));
    CK_CUDA(cudaEventRecord(s->ev[1], st));
    if (cull) { // OPTIONAL bundle-cull mode: screen tiles of 128 x 32 pixels -> candidates -> sort -> strict
        trk::PrimaryCullParams p{};
        const int c_tiles = s->n_pad / cull::CTILE;
        p.cam = dc, p.bands = bands, p.table = s->eye_table, p.n_tiles = c_tiles, p.n_tris = s->n_tris, p.n_rows = n_rows;
        p.tiles_x = (W + 127) / 128, p.tiles_y = (n_rows + 31) / 32;
        const int blocks = p.tiles_x * p.tiles_y;
        p.n_slices = blocks >= 12 * g.n_sms ? 1 : std::max(1, std::min((12 * g.n_sms + blocks - 1) / blocks, std::max(1, c_tiles / 8)));
        p.em = cull::Emitter{s->cand_a, s->cand_count, em_cap};
        p.counters = s->counters, p.work = s->work;
        long long n_keys = -1;
        if (two_phase) {
            if (int rc = ensure_boxes((size_t)blocks)) return rc;
            trk::primary_boxes_kernel<<<blocks, sweep::THREADS, 0, st>>>(p, s->boxes, s->blk_off);
            CK_CUDA(cudaGetLastError());
            cull::L0Params lp{};
            lp.tables = s->eye_table, lp.n_groups = 1, lp.nface = 0, lp.blk_off = s->blk_off;
            if (int rc = block_lists(lp, blocks, n_keys)) return rc;
        }
        if (n_keys >= 0) {
            trk::primary_cull2_kernel<<<2 * g.n_sms, sweep::THREADS, 0, st>>>(p, trk::BlockLists{s->boxes, s->cand_b, (unsigned long long)n_keys, tri_bits});
            CK_CUDA(cudaGetLastError());
            host_tests_primary += (int64_t)n_px * s->n_tris;
        } else {
            CK_CUDA(cudaMemsetAsync(s->cand_count, 0, sizeof(unsigned long long), st));
            const size_t smem = sizeof(cull::EmitSmem);
            CK_CUDA(cudaFuncSetAttribute(trk::primary_cull_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            trk::primary_cull_kernel<<<std::min(blocks * p.n_slices, 2 * g.n_sms), sweep::THREADS, smem, st>>>(p);
            CK_CUDA(cudaGetLastError());
        }
        trk::strict_primary_pairs<<<8 * g.n_sms, 256, 0, st>>>(s->cand_a, s->cand_count, em_cap, dc, bands,
                                                               s->tri_verts, s->best, s->counters);
        CK_CUDA(cudaGetLastError());
        trk::resolve_primary_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(dc, bands, s->best, s->tri_verts, s->n_tris, s->spheres,
                                                                        s->n_spheres, s->hit_tri, s->hit_t, s->hit_v);
        CK_CUDA(cudaGetLastError());
        launches += 3;
    } else {
        // no jitter: the rays of a thread share q exactly; jittered samples (extension): they share a mean q (span table)
        // unless the frame is so small that a jittered (s,t) can leave the span rows' |p|,|q| <= 1.0625 range
        const int qmode = bands.spp_n <= 1 ? sweep::MODE_SHAREDQ : (W >= 16 && H >= 16 ? sweep::MODE_QBAR : sweep::MODE_OWNQ);
        const Decomp d = pick_decomp(n_px, n_tiles, g.n_sms, o.rays_per_thread, 0, qmode);
        trk::PrimaryParams p{};
        p.cam = dc, p.bands = bands, p.table = qmode == sweep::MODE_OWNQ ? s->eye_table : s->eye_span, p.n_tiles = n_tiles, p.n_tris = s->n_tris;
        p.tri_verts = s->tri_verts;
        p.best = s->best, p.counters = s->counters, p.work = s->work;
        p.n_rows = n_rows, p.n_blocks = 0; // ray blocks = screen tiles of (TX R) x (NT / TX) pixels: least edge waste wins
        for (int lg = 3; lg <= 6; ++lg) {
            const int tw = (1 << lg) * d.R, th = sweep::NT >> lg;
            const int tx = (W + tw - 1) / tw, nb = tx * ((n_rows + th - 1) / th);
            if (!p.n_blocks || nb < p.n_blocks) p.n_blocks = nb, p.tiles_x = tx, p.tx_log2 = lg;
        }
        p.n_slices = d.n_slices;
        const int want_items = items_per_cta() * sweep::MINB * g.n_sms;
        if (p.n_blocks < want_items) // same sizing rule as pick_decomp, on the real block count
            p.n_slices = std::max(1, std::min((want_items + p.n_blocks - 1) / p.n_blocks, std::max(1, n_tiles / 4)));
        const int grid = std::min(p.n_blocks * p.n_slices, sweep::MINB * g.n_sms);
        // executed FP32 flops per pair: span form 2 FADD + 1 FFMA per pair and 4 FFMA per thread and triangle; three-row
        // form with every ray its own q: 6 FFMA.SAT + FMUL + FFMA
        flop_primary = qmode == sweep::MODE_OWNQ ? 15.0 : 4.0 + (qmode == sweep::MODE_QBAR ? 16.0 : 8.0) / d.R;
        if (int rc = launch_primary(d.R, o.exhaustive_strict != 0, qmode, p, grid, st)) return rc;
        trk::resolve_primary_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(dc, bands, s->best, s->tri_verts, s->n_tris, s->spheres,
                                                                        s->n_spheres, s->hit_tri, s->hit_t, s->hit_v);
        CK_CUDA(cudaGetLastError());
        launches += 2;
    }
    CK_CUDA(cudaEventRecord(s->ev[2], st));

    // ---- faceIDs ------------------------------------------------------------------------
    if (smp == 0 && L > 0 && o.rng_mode == TRACER_RNG_EXPLICIT) {
        std::vector<int> loc((size_t)n_px * L);
        for (int k = 0; k < n_px; ++k) {
            int w, h;
            bands.map(k, w, h);
            std::memcpy(&loc[(size_t)k * L], o.faceid + ((size_t)h * W + w) * L, sizeof(int) * L);
        }
        CK_CUDA(cudaMemcpyAsync(s->faceid, loc.data(), loc.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        CK_CUDA(cudaStreamSynchronize(st));
    } else if (smp == 0 && L > 0 && o.rng_mode == TRACER_RNG_MT19937) {
        trk::hitmask_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(s->hit_tri, n_px, s->mask);
        CK_CUDA(cudaGetLastError());
        ++launches;
        std::vector<uint8_t> hm((size_t)n_px);
        CK_CUDA(cudaMemcpyAsync(hm.data(), s->mask, (size_t)n_px, cudaMemcpyDeviceToHost, st));
        CK_CUDA(cudaStreamSynchronize(st));
        std::vector<int> fid((size_t)n_px * L);
        tracer__mt19937_scan(o.seed, L, s->h_light_F.data(), n_px, hm.data(), fid.data()); // local order == scan order
        CK_CUDA(cudaMemcpyAsync(s->faceid, fid.data(), fid.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        CK_CUDA(cudaStreamSynchronize(st));
    }

    // ---- lights: (finish k-1, set up k) -> group by light vertex -> first-occluder sweep ----
    auto build_face_tables = [&](int k, const std::vector<int> &group_cnt) -> int { // lazily, for groups that have rays
        for (int gi = 0; gi < (int)group_cnt.size(); ++gi) {
            if (!group_cnt[gi]) continue;
            const int face = gi % trk::NFACE, vtx = s->h_light_vbase[k] + gi / trk::NFACE;
            if (face == trk::NFACE - 1) {
                if (!s->allcand_built) {
                    trk::build_allcand_table<<<(s->n_pad + 255) / 256, 256, 0, st>>>(s->n_tris, s->n_pad, s->allcand_table, s->allcand_span);
                    CK_CUDA(cudaGetLastError());
                    s->allcand_built = true, ++launches;
                }
                continue;
            }
            double &built = s->table_lmax[(size_t)vtx * 6 + face];
            const double need = (k + 1) * diag;
            if (built >= need) continue;
            built = need * 1.5; // head-room so that camera moves rarely trigger a rebuild
            const trk::TableParam tp = face_param(&s->h_light_verts[3 * (size_t)vtx], face, built);
            if (int rc = build_table(s, tp, s->light_tables + ((size_t)vtx * 6 + face) * s->table_stride,
                                     s->light_spans + ((size_t)vtx * 6 + face) * s->span_stride, st))
                return rc;
            ++launches;
        }
        return 0;
    };
    trk::PixelState px{s->best, s->best_occ, s->hit_tri, s->hit_t, s->hit_v, s->carry, s->nrm, s->accum,
                       s->ro,   s->rd,       s->re,      s->rt,    s->rj};
    for (int k = 0; k <= L; ++k) {
        trk::LightStepParams lp{};
        lp.cam = dc, lp.bands = bands, lp.px = px;
        lp.li = trk::LightInfo{s->light_vbase, s->light_verts};
        lp.k = k, lp.L = L, lp.n_tris = s->n_tris;
        lp.tri_verts = s->tri_verts, lp.tri_normals = s->tri_normals, lp.tri_geom = s->tri_geom;
        lp.geom_has_normals = s->geom_has_normals, lp.geom_material = s->geom_material;
        lp.sphere_material = s->sphere_material, lp.spheres = s->spheres;
        lp.rng_mode = o.rng_mode, lp.seed = seed_s, lp.faceid = s->faceid, lp.lmax = (k + 1) * diag;
        lp.seg_count = s->seg_count, lp.counters = s->counters;
        lp.dbg_occ = o.out_occ_tri ? s->dbg_occ : nullptr;
        lp.cull_cells = cull ? 1 : 2, lp.rkey = s->rkey;
        if (k < L) CK_CUDA(cudaMemsetAsync(s->seg_count, 0, sizeof(int) * ((size_t)s->maxF * trk::NFACE + 1), st));
        trk::light_step_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(lp);
        CK_CUDA(cudaGetLastError());
        ++launches;
        if (k == L) break;
        const int F = s->h_light_F[k] * trk::NFACE; // ray groups: (light vertex, cube face)
        if (cull) {
            // OPTIONAL bundle-cull mode: rays sorted by (group, Morton code of (p,q)), one culled sweep over all triangles per light
            const int rpb = sweep::THREADS * 8;
            int group_bits = 1;
            while ((1 << group_bits) < F) ++group_bits;
            trk::list_prefix_kernel<<<1, 32, 0, st>>>(s->seg_count, F, s->seg_off, s->cursor);
            CK_CUDA(cudaGetLastError());
            trk::chunk_prefix_kernel<<<1, 32, 0, st>>>(s->seg_count, F, rpb, s->n_pad / cull::CTILE, 2 * g.n_sms, s->blk_off, s->cnt_b, s->work,
                                                       s->n_slices, 24, 16);
            CK_CUDA(cudaGetLastError());
            CK_CUDA(cub::DeviceRadixSort::SortPairs(s->pair_tmp, s->pair_bytes, s->rkey, s->rkey_sorted, s->iota, s->list, n_px, 0,
                                                    32 + group_bits + 1, st));
            CK_CUDA(cudaMemcpyAsync(s->cursor, s->seg_count, sizeof(int) * F, cudaMemcpyDeviceToDevice, st));
            CK_CUDA(cudaMemsetAsync(s->best_occ, 0xff, sizeof(unsigned long long) * (size_t)n_px, st));
            std::vector<int> gcnt((size_t)F);
            CK_CUDA(cudaMemcpyAsync(gcnt.data(), s->cursor, sizeof(int) * F, cudaMemcpyDeviceToHost, st));
            CK_CUDA(cudaStreamSynchronize(st));
            CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k], st));
            if (int rc = build_face_tables(k, gcnt)) return rc;
            trk::ShadowCullParams sp{};
            sp.tables = s->light_tables + (size_t)s->h_light_vbase[k] * 6 * s->table_stride, sp.table_stride = s->table_stride;
            sp.allcand = s->allcand_table, sp.n_tiles = s->n_pad / cull::CTILE, sp.n_tris = s->n_tris, sp.n_groups = F, sp.n_px = n_px;
            sp.cells_per_group = 0, sp.n_slices = s->n_slices;
            sp.list = s->list, sp.seg_off = s->seg_off, sp.seg_cnt = s->cursor, sp.blk_off = s->blk_off, sp.px = px;
            sp.counters = s->counters, sp.work = s->work;
            sp.em = cull::Emitter{s->cand_a, s->cand_count, em_cap};
            long long n_keys = -1;
            if (two_phase) {
                const int max_blocks = n_px / rpb + F + 1;
                if (int rc = ensure_boxes((size_t)max_blocks)) return rc;
                trk::shadow_boxes_kernel<<<max_blocks, sweep::THREADS, 0, st>>>(sp, s->boxes);
                CK_CUDA(cudaGetLastError());
                cull::L0Params lp{};
                lp.tables = sp.tables, lp.allcand = sp.allcand, lp.table_stride = sp.table_stride;
                lp.n_groups = F, lp.nface = trk::NFACE, lp.blk_off = s->blk_off;
                if (int rc = block_lists(lp, max_blocks, n_keys)) return rc;
            }
            if (n_keys >= 0) {
                trk::shadow_cull2_kernel<<<2 * g.n_sms, sweep::THREADS, 0, st>>>(sp, trk::BlockLists{s->boxes, s->cand_b, (unsigned long long)n_keys, tri_bits});
                CK_CUDA(cudaGetLastError());
                for (int c : gcnt) host_tests_shadow += (int64_t)c * s->n_pad;
            } else {
                CK_CUDA(cudaMemsetAsync(s->cand_count, 0, sizeof(unsigned long long), st));
                const size_t smem = sizeof(cull::EmitSmem);
                CK_CUDA(cudaFuncSetAttribute(trk::shadow_cull_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                trk::shadow_cull_kernel<<<2 * g.n_sms, sweep::THREADS, smem, st>>>(sp);
                CK_CUDA(cudaGetLastError());
            }
            trk::strict_shadow_pairs<<<8 * g.n_sms, 256, 0, st>>>(s->cand_a, s->cand_count, em_cap, px, n_px,
                                                                  s->tri_verts, s->counters);
            CK_CUDA(cudaGetLastError());
            launches += 4;
            if (s->n_spheres > 0) {
                const dim3 sgrid((unsigned)std::min(1024, (n_px + 255) / 256), (unsigned)F);
                trk::shadow_spheres_kernel<<<sgrid, 256, 0, st>>>(s->list, s->seg_off, s->cursor, F, px, n_px, s->spheres, s->n_spheres,
                                                                   s->n_tris);
                CK_CUDA(cudaGetLastError());
                ++launches;
            }
            CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k + 1], st));
            continue;
        }
        // ---- default mode: q-sorted lists, then ONE persistent cooperative kernel per batch of light vertices ----
        trk::list_prefix_kernel<<<1, 32, 0, st>>>(s->seg_count, F, s->seg_off, s->cursor);
        CK_CUDA(cudaGetLastError());
        { // group-major, q-minor order (pixels without a shadow ray carry the all-ones key and sort last)
            int group_bits = 1;
            while ((1 << group_bits) < F) ++group_bits;
            CK_CUDA(cub::DeviceRadixSort::SortPairs(s->pair_tmp, s->pair_bytes, s->rkey, s->rkey_sorted, s->iota, s->list, n_px, 0,
                                                    32 + group_bits + 1, st));
            CK_CUDA(cudaMemcpyAsync(s->cursor, s->seg_count, sizeof(int) * F, cudaMemcpyDeviceToDevice, st));
            const size_t need = (size_t)n_px / trk::CBLK + (size_t)F + 2;
            if (need > s->blk_cnt_cap) {
                dev_free(s->blk_cnt);
                s->blk_cnt_cap = 0;
                if (dev_alloc(&s->blk_cnt, need)) return TRACER_ERR_NOMEM;
                s->blk_cnt_cap = need;
            }
        }
        launches += 2;
        CK_CUDA(cudaMemsetAsync(s->best_occ, 0xff, sizeof(unsigned long long) * (size_t)n_px, st));
        CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k], st));
        if (!s->allcand_built) {
            trk::build_allcand_table<<<(s->n_pad + 255) / 256, 256, 0, st>>>(s->n_tris, s->n_pad, s->allcand_table, s->allcand_span);
            CK_CUDA(cudaGetLastError());
            s->allcand_built = true, ++launches;
        }
        // Triangle chunks: after each one the still-unoccluded rays are compacted (early exit, main.cpp:324).  Equal chunks
        // keep the pairs swept past a ray's occluder lowest (x1.056 at 64 chunks; x1.11 at 32) and win when a light has many
        // shadow rays; with few rays (small frames, one band share of a multi-GPU frame) a chunk's fixed cost (three grid
        // barriers, the compaction passes, the sweep's tail: ~0.1 ms) weighs more, and 20 chunks that start fine (1/64 of the
        // triangles: most occluded rays find their occluder early) and coarsen win (x1.10).  The kernel picks the scheme from
        // the live-ray count it finds.  opts.shadow_chunks asks for that many equal chunks.
        trk::ShadowLightParams sp{};
        {
            const int nc = std::min({n_tiles, trk::SL_MAXCHUNK, o.shadow_chunks > 0 ? o.shadow_chunks : std::max(1, std::min(64, n_tiles / 8))});
            sp.n_chunks[1] = nc;
            for (int c = 0; c <= nc; ++c) sp.bounds[1][c] = (int)((int64_t)n_tiles * c / nc);
            if (o.shadow_chunks > 0 || n_tiles < 64) {
                sp.n_chunks[0] = nc;
                std::memcpy(sp.bounds[0], sp.bounds[1], sizeof sp.bounds[0]);
            } else {
                std::vector<int> fr{0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 32, 40, 48, 56, 64};
                int den = 64;
                if (const char *e = std::getenv("TRACER_GEO")) { // development knob: "den,f1,f2,...,den"
                    fr.assign(1, 0);
                    den = std::atoi(e);
                    for (const char *q = std::strchr(e, ','); q; q = std::strchr(q + 1, ',')) fr.push_back(std::atoi(q + 1));
                }
                sp.n_chunks[0] = (int)fr.size() - 1;
                for (size_t c = 0; c < fr.size(); ++c) sp.bounds[0][c] = (int)((int64_t)n_tiles * fr[c] / den);
            }
        }
        sp.many_rays = (long long)1 << 20;
        sp.items_per_cta = items_per_cta();
        sp.run_pairs = std::getenv("TRACER_RUN_PAIRS") ? std::max(1ll, std::atoll(std::getenv("TRACER_RUN_PAIRS"))) : 6000000ll;
        sp.min_tiles = std::getenv("TRACER_MIN_TILES") ? std::max(1, std::atoi(std::getenv("TRACER_MIN_TILES"))) : 1;
        sp.allcand = s->allcand_span, sp.table_stride = s->span_stride; // the default sweeps read the span tables
        sp.n_tris = s->n_tris, sp.n_tiles = n_tiles, sp.n_px = n_px, sp.tri_verts = s->tri_verts;
        sp.list[0] = s->list, sp.list[1] = s->list_b;
        sp.blk_cnt = s->blk_cnt, sp.px = px, sp.spheres = s->spheres, sp.n_spheres = s->n_spheres;
        sp.counters = s->counters;
        // light vertices in batches: as many as have table slots (all of them unless the light is a big mesh)
        const int Fk = s->h_light_F[k], vb = s->h_light_vbase[k];
        for (int b0 = 0; b0 < Fk; b0 += s->table_slots) {
            const int b1 = std::min(Fk, b0 + s->table_slots);
            for (int v = b0; v < b1; ++v)
                for (int face = 0; face < 6; ++face) {
                    // every vertex has its own slot when they all fit (tables are then kept across frames and lights);
                    // otherwise the slots are reused batch by batch and rebuilt every time
                    const size_t slot = s->tables_resident ? (size_t)(vb + v) : (size_t)(v - b0);
                    const double need = (k + 1) * diag;
                    if (s->tables_resident) {
                        double &built = s->table_lmax[slot * 6 + face];
                        if (built >= need) continue;
                        built = need * 1.5; // head-room so that camera moves rarely trigger a rebuild
                    }
                    const trk::TableParam tp = face_param(&s->h_light_verts[3 * (size_t)(vb + v)], face, need * 1.5);
                    if (int rc = build_table(s, tp, s->light_tables + (slot * 6 + face) * s->table_stride,
                                             s->light_spans + (slot * 6 + face) * s->span_stride, st))
                        return rc;
                    ++launches;
                }
            sp.tables = s->light_spans + (s->tables_resident ? (size_t)(vb + b0) : 0) * 6 * s->span_stride;
            sp.F = (b1 - b0) * trk::NFACE;
            sp.seg_off = s->seg_off + b0 * trk::NFACE;
            sp.cnt[0] = s->cursor + b0 * trk::NFACE, sp.cnt[1] = s->cnt_b + b0 * trk::NFACE;
            sp.work = s->work;
            CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int) * WORK_INTS, st));
            // development: TRACER_SHADOW_DIAG=2 dumps, for every light, when each CTA ran out of sweep items in each chunk
            static const bool want_timeline = std::getenv("TRACER_SHADOW_DIAG") && std::atoi(std::getenv("TRACER_SHADOW_DIAG")) >= 2;
            const size_t tl_n = (size_t)trk::SL_MAXCHUNK * 8 * (size_t)g.n_sms * 2;
            unsigned long long *tl = nullptr;
            if (want_timeline) {
                tl = (unsigned long long *)t_pool->alloc(tl_n * sizeof(unsigned long long));
                if (tl) CK_CUDA(cudaMemsetAsync(tl, 0, tl_n * sizeof(unsigned long long), st));
            }
            sp.timeline = tl;
            if (int rc = launch_shadow_light(g, o.exhaustive_strict != 0, sp, (unsigned *)(s->work + trk::SL_MAXCHUNK), st)) return rc;
            ++launches;
            if (tl) {
                std::vector<unsigned long long> h(tl_n);
                CK_CUDA(cudaMemcpyAsync(h.data(), tl, tl_n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
                CK_CUDA(cudaStreamSynchronize(st));
                t_pool->release(tl);
                char name[128];
                std::snprintf(name, sizeof name, "gpurun_out/shadow_timeline_light%d.bin", k);
                if (FILE *f = std::fopen(name, "wb")) {
                    const int hdr[2] = {trk::SL_MAXCHUNK, 8 * g.n_sms};
                    std::fwrite(hdr, sizeof hdr, 1, f), std::fwrite(h.data(), sizeof(unsigned long long), h.size(), f), std::fclose(f);
                }
            }
        }
        CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k + 1], st));
    }
    if (S > 1) { // sum the samples in a fixed order; the last pass divides by S
        const size_t n3 = 3 * (size_t)n_px;
        trk::accumulate_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(s->accum, s->accum_total, n3, smp == 0, smp == S - 1,
                                                                              (float)S);
        CK_CUDA(cudaGetLastError());
        ++launches;
        CK_CUDA(cudaStreamSynchronize(st));
        float msx = 0;
        cudaEventElapsedTime(&msx, s->ev[1], s->ev[2]);
        ms_primary_acc += msx;
        for (int k = 0; k < L; ++k) {
            cudaEventElapsedTime(&msx, s->ev_shadow[2 * k], s->ev_shadow[2 * k + 1]);
            ms_shadow_acc += msx;
        }
    }
    } // samples

    // ---- quantise + pack ------------------------------------------------------------------
    uint8_t *dst8 = o.rgb_out_is_device ? rgb_out : s->rgb8;
    const float *final_accum = S > 1 ? s->accum_total : s->accum;
    trk::quantise_kernel<<<((n_px + 15) / 16 + 127) / 128, 128, 0, st>>>(final_accum, n_px, dst8);
    CK_CUDA(cudaGetLastError());
    ++launches;
    CK_CUDA(cudaEventRecord(s->ev[3], st));
    if (!o.rgb_out_is_device) CK_CUDA(cudaMemcpyAsync(rgb_out, s->rgb8, (size_t)n_px * 3, cudaMemcpyDeviceToHost, st));

    // ---- optional debug read-backs -----------------------------------------------------------
    if (o.out_tri) CK_CUDA(cudaMemcpyAsync(o.out_tri, s->hit_tri, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_t) CK_CUDA(cudaMemcpyAsync(o.out_t, s->hit_t, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_v) CK_CUDA(cudaMemcpyAsync(o.out_v, s->hit_v, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_occ_tri && L > 0)
        CK_CUDA(cudaMemcpyAsync(o.out_occ_tri, s->dbg_occ, (size_t)n_px * L * 4, cudaMemcpyDeviceToHost, st));
    std::vector<float> acc;
    if (o.out_rgb) {
        acc.resize((size_t)n_px * 3);
        CK_CUDA(cudaMemcpyAsync(acc.data(), final_accum, acc.size() * 4, cudaMemcpyDeviceToHost, st));
    }
    sweep::Counters hc;
    CK_CUDA(cudaMemcpyAsync(&hc, s->counters, sizeof hc, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    if (o.out_rgb)
        for (int k = 0; k < n_px; ++k)
            for (int c = 0; c < 3; ++c) o.out_rgb[(size_t)k * 3 + c] = acc[(size_t)c * n_px + k];

    float ms = 0;
    cudaEventElapsedTime(&ms, s->ev[0], s->ev[3]);
    s->stats.ms_total = ms;
    cudaEventElapsedTime(&ms, s->ev[1], s->ev[2]);
    s->stats.ms_primary = S > 1 ? ms_primary_acc : ms;
    double sh = 0;
    for (int k = 0; k < L; ++k) {
        cudaEventElapsedTime(&ms, s->ev_shadow[2 * k], s->ev_shadow[2 * k + 1]);
        sh += ms;
    }
    if (S > 1) sh = ms_shadow_acc;
    s->stats.ms_shadow = sh;
    s->stats.ms_other = s->stats.ms_total - s->stats.ms_primary - sh;
    s->stats.n_primary_rays = (int64_t)n_px * S;
    s->stats.n_shadow_rays = (int64_t)hc.n_hits * L;
    s->stats.tests_primary = (int64_t)hc.tests_primary + host_tests_primary;
    s->stats.tests_shadow = (int64_t)hc.tests_shadow + host_tests_shadow;
    s->stats.tests_shadow_ref = (int64_t)hc.tests_shadow_ref;
    s->stats.strict_evals = (int64_t)hc.strict_evals;
    s->stats.filter_misses = (int64_t)hc.filter_misses;
    s->stats.pipeline_errors = (int64_t)hc.pipeline_errors;
    s->stats.kernel_launches = launches;
    // FP32 flops the sweeps' formulation needs per swept pair (all in the FMA pipe; FFMA = 2, FADD = 1).  Span form: two
    // saturating adds + one multiply-add per pair, plus the bound FFMAs per thread and triangle: 4 (one exact q) or 8 (mean q
    // + |B| * spread: shadow sweeps, jittered primary samples) over the R rays of the thread.
    s->stats.flop_primary = cull ? 0.0 : flop_primary, s->stats.flop_shadow = cull ? 0.0 : 4.0 + 16.0 / trk::SHADOW_R;
    // of which multiply-adds that evaluate bounds (the rest is the two saturating adds and the accumulate of each pair)
    s->stats.flop_primary_edges = cull ? 0.0 : (flop_primary >= 15.0 ? 12.0 : flop_primary - 4.0);
    s->stats.flop_shadow_edges = cull ? 0.0 : 16.0 / trk::SHADOW_R;
    if (hc.cull_overflow) {
        // the optional mode's candidate buffer (24 per ray + slack) was too small for this scene's depth complexity: render
        // the frame again with a 4x larger one while that fits comfortably, else by the default sweeps, which need no such
        // buffer — same bytes out either way
        tracer_render_opts o2 = o;
        o2.struct_size = sizeof o2;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t next_bytes = ((size_t)n_px * 24 * (size_t)s->cull_grow * 4 + ((size_t)1 << 22)) * sizeof(unsigned long long) * 3;
        if (!std::getenv("TRACER_CAND_CAP") && s->cull_grow < 64 && next_bytes < free_b / 2 + s->cand_cap * 24)
            s->cull_grow *= 4;
        else
            o2.bundle_cull = 0;
        return tracer_cuda_render_scene(s, cam, W, H, &o2, rgb_out);
    }
    if (getenv("TRACER_SHADOW_DIAG") && hc.cyc_total)
        fprintf(stderr, "shadow diag: CTA cycles %.3e total = items %.1f %% + grid barriers %.1f %% + compaction %.1f %% + other %.1f %%; %llu items in %llu runs\n",
                (double)hc.cyc_total, 100.0 * hc.cyc_items / hc.cyc_total, 100.0 * hc.cyc_barrier / hc.cyc_total, 100.0 * hc.cyc_compact / hc.cyc_total,
                100.0 * ((double)hc.cyc_total - hc.cyc_items - hc.cyc_barrier - hc.cyc_compact) / hc.cyc_total, hc.n_items, hc.n_runs);
    if (getenv("TRACER_CULL_DIAG"))
        fprintf(stderr, "cull diag (shadow): l0 survivors %llu, tiles with any %llu, fallback tiles %llu, l1 warp-passes %llu, item-tiles %llu\n", hc.cull_l0,
                hc.cull_tiles_any, hc.cull_tiles_fallback, hc.cull_l1, (unsigned long long)(hc.tests_shadow / 4096 / cull::CTILE));
    return TRACER_OK;
}

int tracer_cuda_last_stats(tracer_scene_dev *s, tracer_frame_stats *out) {
    if (!s || !out) return fail(TRACER_ERR_INVALID, "null argument");
    *out = s->stats;
    return TRACER_OK;
}

int tracer_cuda_render(const tracer_scene_flat *scene, const tracer_camera *cam, int32_t width, int32_t height,
                       const tracer_render_opts *opts, uint8_t *rgb_out) {
    if (g_multi.n > 1) return tracer_cuda_render_multi(scene, cam, width, height, opts, rgb_out);
    tracer_scene_dev *s = nullptr;
    if (int rc = tracer_cuda_scene_create(scene, &s)) return rc;
    const int rc = tracer_cuda_render_scene(s, cam, width, height, opts, rgb_out);
    tracer_cuda_scene_destroy(s);
    return rc;
}

int tracer_cuda_assemble_bands(const uint8_t *gathered_dev, uint8_t *frame_dev, int32_t width, int32_t height,
                               int32_t band_rows, int32_t band_count, int32_t rows_per_rank_padded, void *cuda_stream) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    Ctx &g = *g_cur;
    if (!gathered_dev || !frame_dev || width <= 0 || height <= 0 || band_rows <= 0 || band_count <= 0)
        return fail(TRACER_ERR_INVALID, "bad argument");
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : g.stream;
    trk::assemble_bands_kernel<<<g.n_sms * 8, 256, 0, st>>>(gathered_dev, frame_dev, width, height, band_rows, band_count,
                                                            rows_per_rank_padded);
    CK_CUDA(cudaGetLastError());
    CK_CUDA(cudaStreamSynchronize(st));
    return TRACER_OK;
}


/* ---- all GPUs of one box behind one call ---------------------------------------------------------------------
 * SURVEY 5 / 8e: one process, a context (stream, pool, scene replica) per GPU, one host thread per GPU while a frame
 * renders, ONE NCCL communicator set (ncclCommInitAll).  PPM rows are cut into 8-row bands, band b -> GPU b % n;
 * every GPU quantises its bands straight into its send buffer, the packed bands go to GPU 0 with grouped
 * ncclSend / ncclRecv over NVLink (this NCCL has no ncclGather), GPU 0 scatters them into PPM order. */
int tracer_cuda_init_multi(int n_gpus) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(TRACER_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count=0"));
    if (n_gpus < 1 || n_gpus > n || n_gpus > MAX_GPUS) return fail(TRACER_ERR_INVALID, "n_gpus out of range (" + std::to_string(n) + " devices visible)");
    multi_shutdown();
    for (int d = n_gpus - 1; d >= 0; --d) // device 0 last: it stays the current context
        if (int rc = init_device(d)) return rc;
    if (n_gpus > 1) {
        std::string err;
        if (!g_nccl.load(err)) return fail(TRACER_ERR_CUDA, err);
        int devs[MAX_GPUS];
        for (int d = 0; d < n_gpus; ++d) devs[d] = d;
        const ncclResult_t r = g_nccl.CommInitAll(g_multi.comms, n_gpus, devs);
        if (r != ncclSuccess) return fail(TRACER_ERR_CUDA, std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r));
        g_multi.have_comms = true;
    }
    g_multi.n = n_gpus;
    return TRACER_OK;
}

int tracer_cuda_multi_gpu_count(void) { return g_multi.n; }

void tracer_cuda_scene_destroy_multi(tracer_scene_multi *ms) {
    if (!ms) return;
    for (tracer_scene_dev *d : ms->dev) tracer_cuda_scene_destroy(d);
    delete ms;
}

int tracer_cuda_scene_create_multi(const tracer_scene_flat *sc, tracer_scene_multi **out) {
    if (!out) return fail(TRACER_ERR_INVALID, "null out");
    *out = nullptr;
    if (g_multi.n < 1) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init_multi not called");
    auto *ms = new tracer_scene_multi();
    ms->dev.assign((size_t)g_multi.n, nullptr);
    std::vector<int> rc((size_t)g_multi.n, 0);
    std::vector<std::string> err((size_t)g_multi.n);
    auto work = [&](int d) { // replicate: every GPU uploads over its own PCIe link
        rc[d] = scene_create_on(g_ctx[d], sc, &ms->dev[d]);
        if (rc[d]) err[d] = g_err;
    };
    std::vector<std::thread> th;
    for (int d = 1; d < g_multi.n; ++d) th.emplace_back(work, d);
    work(0);
    for (auto &t : th) t.join();
    for (int d = 0; d < g_multi.n; ++d)
        if (rc[d]) {
            const int r = rc[d];
            const std::string m = "GPU " + std::to_string(d) + ": " + err[d];
            tracer_cuda_scene_destroy_multi(ms);
            return fail(r, m);
        }
    *out = ms;
    return TRACER_OK;
}

int tracer_cuda_render_scene_multi(tracer_scene_multi *ms, const tracer_camera *cam, int32_t W, int32_t H,
                                   const tracer_render_opts *opts_in, uint8_t *rgb_out) {
    if (!ms || !cam || !rgb_out) return fail(TRACER_ERR_INVALID, "null argument");
    const int n = (int)ms->dev.size();
    if (n != g_multi.n || n < 1) return fail(TRACER_ERR_STATE, "scene was created for a different GPU set");
    if (n == 1) {
        const int rc = tracer_cuda_render_scene(ms->dev[0], cam, W, H, opts_in, rgb_out);
        ms->stats = ms->dev[0]->stats;
        return rc;
    }
    tracer_render_opts o;
    std::memset(&o, 0, sizeof o);
    if (opts_in) std::memcpy(&o, opts_in, std::min<size_t>(sizeof o, opts_in->struct_size ? opts_in->struct_size : sizeof o));
    if (o.band_count > 1) return fail(TRACER_ERR_INVALID, "the multi-GPU call partitions the frame itself: leave band_count at 0");
    if (o.out_tri || o.out_t || o.out_v || o.out_occ_tri || o.out_rgb) return fail(TRACER_ERR_INVALID, "debug outputs are per-GPU: use tracer_cuda_render_scene with bands");
    if (W < 2 || H < 2 || (int64_t)W * H > (int64_t)2000 * 1000 * 1000) return fail(TRACER_ERR_INVALID, "bad frame size");
    const int band_rows = o.band_rows > 0 ? o.band_rows : 8;
    int rows_pad = 0;
    for (int d = 0; d < n; ++d) rows_pad = std::max(rows_pad, tracer_band_row_count(H, band_rows, d, n));
    const size_t row_bytes = (size_t)W * 3, pad_bytes = (size_t)rows_pad * row_bytes, frame_bytes = row_bytes * H;
    // device 0: gather buffer (slot d = GPU d's packed bands; GPU 0 renders straight into slot 0) and the assembled frame
    Ctx &g0 = g_ctx[0];
    CK_CUDA(cudaSetDevice(0));
    t_pool = &g0.pool;
    if (g_multi.gathered_cap < pad_bytes * n + 64) {
        dev_free(g_multi.gathered);
        g_multi.gathered_cap = 0;
        if (dev_alloc(&g_multi.gathered, pad_bytes * n + 64)) return TRACER_ERR_NOMEM;
        g_multi.gathered_cap = pad_bytes * n + 64;
    }
    if (g_multi.frame_cap < frame_bytes + 64) {
        dev_free(g_multi.frame);
        g_multi.frame_cap = 0;
        if (dev_alloc(&g_multi.frame, frame_bytes + 64)) return TRACER_ERR_NOMEM;
        g_multi.frame_cap = frame_bytes + 64;
    }
    std::vector<int> rc((size_t)n, 0);
    std::vector<std::string> err((size_t)n);
    auto work = [&](int d) {
        Ctx &g = g_ctx[d];
        uint8_t *dst = g_multi.gathered; // GPU 0
        if (d > 0) {
            if (cudaSetDevice(d) != cudaSuccess) { rc[d] = TRACER_ERR_CUDA, err[d] = "cudaSetDevice"; return; }
            t_pool = &g.pool;
            if (g_multi.band_cap[d] < pad_bytes + 64) {
                dev_free(g_multi.band_buf[d]);
                g_multi.band_cap[d] = 0;
                if (dev_alloc(&g_multi.band_buf[d], pad_bytes + 64)) { rc[d] = TRACER_ERR_NOMEM, err[d] = g_err; return; }
                g_multi.band_cap[d] = pad_bytes + 64;
            }
            dst = g_multi.band_buf[d];
        }
        tracer_render_opts od = o;
        od.struct_size = sizeof od;
        od.band_rows = band_rows, od.band_index = d, od.band_count = n;
        od.rgb_out_is_device = 1, od.cuda_stream = nullptr; // the GPU's own stream: the send below is queued behind the frame
        rc[d] = tracer_cuda_render_scene(ms->dev[d], cam, W, H, &od, dst);
        if (rc[d]) err[d] = g_err;
    };
    std::vector<std::thread> th;
    for (int d = 1; d < n; ++d) th.emplace_back(work, d);
    work(0);
    for (auto &t : th) t.join();
    for (int d = 0; d < n; ++d)
        if (rc[d]) return fail(rc[d], "GPU " + std::to_string(d) + ": " + err[d]);
    // the one exchange step: packed bands -> GPU 0
    ncclResult_t r = g_nccl.GroupStart();
    for (int d = 1; d < n && r == ncclSuccess; ++d) {
        const size_t bytes = (size_t)tracer_band_row_count(H, band_rows, d, n) * row_bytes;
        if (!bytes) continue;
        r = g_nccl.Send(g_multi.band_buf[d], bytes, ncclUint8, 0, g_multi.comms[d], g_ctx[d].stream);
        if (r == ncclSuccess) r = g_nccl.Recv(g_multi.gathered + (size_t)d * pad_bytes, bytes, ncclUint8, d, g_multi.comms[0], g0.stream);
    }
    const ncclResult_t r2 = g_nccl.GroupEnd();
    if (r != ncclSuccess || r2 != ncclSuccess)
        return fail(TRACER_ERR_CUDA, std::string("NCCL band gather: ") + g_nccl.GetErrorString(r != ncclSuccess ? r : r2));
    CK_CUDA(cudaSetDevice(0));
    uint8_t *frame_dst = o.rgb_out_is_device ? rgb_out : g_multi.frame;
    trk::assemble_bands_kernel<<<g0.n_sms * 8, 256, 0, g0.stream>>>(g_multi.gathered, frame_dst, W, H, band_rows, n, rows_pad);
    CK_CUDA(cudaGetLastError());
    if (!o.rgb_out_is_device) CK_CUDA(cudaMemcpyAsync(rgb_out, g_multi.frame, frame_bytes, cudaMemcpyDeviceToHost, g0.stream));
    for (int d = n - 1; d >= 0; --d) { // the senders' streams too: their buffers are reused by the next frame
        CK_CUDA(cudaSetDevice(d));
        CK_CUDA(cudaStreamSynchronize(g_ctx[d].stream));
    }
    // whole-frame statistics: counts summed over the GPUs, times of the slowest
    tracer_frame_stats t{};
    for (int d = 0; d < n; ++d) {
        const tracer_frame_stats &x = ms->dev[d]->stats;
        t.ms_total = std::max(t.ms_total, x.ms_total), t.ms_primary = std::max(t.ms_primary, x.ms_primary);
        t.ms_shadow = std::max(t.ms_shadow, x.ms_shadow), t.ms_other = std::max(t.ms_other, x.ms_other);
        t.n_pixels += x.n_pixels, t.n_primary_rays += x.n_primary_rays, t.n_shadow_rays += x.n_shadow_rays;
        t.tests_primary += x.tests_primary, t.tests_shadow += x.tests_shadow, t.tests_shadow_ref += x.tests_shadow_ref;
        t.strict_evals += x.strict_evals, t.filter_misses += x.filter_misses, t.kernel_launches += x.kernel_launches;
        t.pipeline_errors += x.pipeline_errors;
        t.n_sms += x.n_sms;
        t.flop_primary = x.flop_primary, t.flop_shadow = x.flop_shadow;
        t.flop_primary_edges = x.flop_primary_edges, t.flop_shadow_edges = x.flop_shadow_edges;
    }
    t.kernel_launches += 1; // assemble
    ms->stats = t;
    return TRACER_OK;
}

int tracer_cuda_last_stats_multi(tracer_scene_multi *ms, tracer_frame_stats *out) {
    if (!ms || !out) return fail(TRACER_ERR_INVALID, "null argument");
    *out = ms->stats;
    return TRACER_OK;
}

int tracer_cuda_render_multi(const tracer_scene_flat *scene, const tracer_camera *cam, int32_t width, int32_t height,
                             const tracer_render_opts *opts, uint8_t *rgb_out) {
    tracer_scene_multi *ms = nullptr;
    if (int rc = tracer_cuda_scene_create_multi(scene, &ms)) return rc;
    const int rc = tracer_cuda_render_scene_multi(ms, cam, width, height, opts, rgb_out);
    tracer_cuda_scene_destroy_multi(ms);
    return rc;
}

}  // extern "C"
