// tracer_cuda.cu — C ABI (include/tracer_cuda.h) over the sm_100a kernels.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/tracer_cuda.h"
#include <cub/device/device_radix_sort.cuh>
#include <dlfcn.h>
#include <nccl.h>
#include <thread>

#include "bvh.cuh" // (includes kernels.cuh)
#include "mt19937.cuh"

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
// n rays (p) of one thread against one span row (row8 = lo.xyzw, hi.xyzw) in the hot loop's shared-q form: qdelta < 0 = one
// exact q (MODE_SHAREDQ), else q = qbar and the bounds widened by |B| * qdelta (MODE_QBAR).  bit 0 = the interval form with
// clamp box and margin delta (sweep::SPAN_BOX, sweep::SPAN_DELTA in the sweeps), bit 1 = the saturating form it replaces
// (x = sat(S p + ax) and y = sat(ay - S p) both 1), bit 2 = the candidate path's span_pass with q as the ray's own q.
extern "C" void tracer__interval_pass(const float *row8, int n, const float *p, float q, float qdelta, float box, float delta,
                                      unsigned char *out) {
    const float4 lo = make_float4(row8[0], row8[1], row8[2], row8[3]), hi = make_float4(row8[4], row8[5], row8[6], row8[7]);
    float ax, ay, nc, h;
    if (qdelta < 0.f) sweep::span_terms(lo, hi, q, ax, ay);
    else sweep::span_terms_qbar(lo, hi, q, qdelta, ax, ay);
    sweep::span_interval(ax, ay, nc, h, box, delta);
    for (int i = 0; i < n; ++i) {
        const float ps = p[i] * sweep::SPAN_S;
        out[i] = (unsigned char)((sweep::interval_pass(nc, h, ps) ? 1 : 0) | (fminf(ps + ax, ay - ps) >= 1.f ? 2 : 0) |
                                 (sweep::span_pass(lo, hi, ps, q) ? 4 : 0));
    }
}
extern "C" void tracer__interval_consts(float *out2) { out2[0] = sweep::SPAN_BOX, out2[1] = sweep::SPAN_DELTA; }
// n rays (p, own q) of one thread against one span row (row8 = lo.xyzw, hi.xyzw as span_rows makes it), stored in the hot form
// with margin delta (sweep::hot_row; sweep::HOT_DELTA in the tables).  Shared-q form: qdelta < 0 = one exact q = qbar
// (MODE_SHAREDQ), else q = qbar with the bounds widened by |B| * qdelta (MODE_QBAR).  bit 0 = the hot loop's test in the
// shared-q form, bit 1 = the candidate path's hot test with the ray's own q, bit 2 = the saturating form in the same shared-q
// form, bit 3 = span_pass with the ray's own q, bit 4 = the interval form (span_interval, SPAN_BOX, SPAN_DELTA) it replaces.
// hot8 (may be null) receives the stored hot row.
extern "C" void tracer__hot_row_pass(const float *row8, int n, const float *p, const float *q, float qbar, float qdelta, float delta,
                                     unsigned char *out, float *hot8) {
    const float4 lo = make_float4(row8[0], row8[1], row8[2], row8[3]), hi = make_float4(row8[4], row8[5], row8[6], row8[7]);
    float4 hlo = lo, hhi = hi;
    sweep::hot_row(hlo, hhi, delta);
    if (hot8) hot8[0] = hlo.x, hot8[1] = hlo.y, hot8[2] = hlo.z, hot8[3] = hlo.w, hot8[4] = hhi.x, hot8[5] = hhi.y, hot8[6] = hhi.z, hot8[7] = hhi.w;
    float nc2, h2, ax, ay, nc, h;
    if (qdelta < 0.f) sweep::hot_terms(hlo, hhi, qbar, nc2, h2), sweep::span_terms(lo, hi, qbar, ax, ay);
    else sweep::hot_terms_qbar(hlo, hhi, qbar, sweep::hot_qdelta(qdelta), nc2, h2), sweep::span_terms_qbar(lo, hi, qbar, qdelta, ax, ay);
    sweep::span_interval(ax, ay, nc, h);
    for (int i = 0; i < n; ++i) {
        const float ps = p[i] * sweep::SPAN_S, ps2 = p[i] * (2.f * sweep::SPAN_S);
        float rnc2, rh2;
        sweep::hot_terms(hlo, hhi, q[i], rnc2, rh2);
        out[i] = (unsigned char)((sweep::hot_pass(nc2, h2, ps2) ? 1 : 0) | (sweep::hot_pass(rnc2, rh2, ps2) ? 2 : 0) |
                                 (fminf(ps + ax, ay - ps) >= 1.f ? 4 : 0) | (sweep::span_pass(lo, hi, ps, q[i]) ? 8 : 0) |
                                 (sweep::interval_pass(nc, h, ps) ? 16 : 0));
    }
}
extern "C" void tracer__hot_consts(float *out3) { out3[0] = sweep::HOT_CLAMP, out3[1] = sweep::HOT_DELTA, out3[2] = sweep::HOT_QD_SCALE; }
// n rays (p, in any order, duplicates allowed) of one closest-hit thread with the shared q against one span row (row8 as
// span_rows makes it, stored in the hot form as the tables store it).  out2[0] = the segment verdict (sweep::segment_pass on
// the least and greatest 2 S p, as sweep_table forms them), out2[1] = the OR of the per-ray hot tests (the verdict of the
// per-ray loop it replaces).  terms2 (may be null) receives (nc2, h2).
extern "C" void tracer__segment_pass(const float *row8, int n, const float *p, float q, unsigned char *out2, float *terms2) {
    float4 lo = make_float4(row8[0], row8[1], row8[2], row8[3]), hi = make_float4(row8[4], row8[5], row8[6], row8[7]);
    sweep::hot_row(lo, hi);
    float nc2, h2;
    sweep::hot_terms(lo, hi, q, nc2, h2);
    bool any = false;
    float pmin2 = p[0] * (2.f * sweep::SPAN_S), pmax2 = pmin2;
    for (int i = 0; i < n; ++i) {
        const float ps2 = p[i] * (2.f * sweep::SPAN_S);
        pmin2 = fminf(pmin2, ps2), pmax2 = fmaxf(pmax2, ps2);
        any |= sweep::hot_pass(nc2, h2, ps2);
    }
    out2[0] = sweep::segment_pass(nc2, h2, pmin2, pmax2), out2[1] = any;
    if (terms2) terms2[0] = nc2, terms2[1] = h2;
}
// The same for n rays (p, q) of one shadow-sweep thread (mean-q form): (nc2, h2) from hot_terms_qbar at qbar with the bounds
// widened by hot_qdelta(qdelta), as shadow_item and sweep_table form them.  out3[0] = the segment verdict, out3[1] = the OR of
// the per-ray hot tests at qbar (the per-ray loop it replaces), out3[2] = the OR of the hot tests with each ray's own q (the
// drain's test).  terms2 (may be null) receives (nc2, h2).
extern "C" void tracer__segment_pass_qbar(const float *row8, int n, const float *p, const float *q, float qbar, float qdelta,
                                          unsigned char *out3, float *terms2) {
    float4 lo = make_float4(row8[0], row8[1], row8[2], row8[3]), hi = make_float4(row8[4], row8[5], row8[6], row8[7]);
    sweep::hot_row(lo, hi);
    float nc2, h2;
    sweep::hot_terms_qbar(lo, hi, qbar, sweep::hot_qdelta(qdelta), nc2, h2);
    bool any = false, own = false;
    float pmin2 = p[0] * (2.f * sweep::SPAN_S), pmax2 = pmin2;
    for (int i = 0; i < n; ++i) {
        const float ps2 = p[i] * (2.f * sweep::SPAN_S);
        pmin2 = fminf(pmin2, ps2), pmax2 = fmaxf(pmax2, ps2);
        any |= sweep::hot_pass(nc2, h2, ps2);
        float rnc2, rh2;
        sweep::hot_terms(lo, hi, q[i], rnc2, rh2);
        own |= sweep::hot_pass(rnc2, rh2, ps2);
    }
    out3[0] = sweep::segment_pass(nc2, h2, pmin2, pmax2), out3[1] = any, out3[2] = own;
    if (terms2) terms2[0] = nc2, terms2[1] = h2;
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
// Buffers of one capacity cap, grown to n elements each when n > cap (the old contents are lost); cap is 0 while any may be
// missing, so that a failed grow is tried again by the next call
template <typename... T>
int dev_grow(size_t &cap, size_t n, T *&...p) {
    if (n <= cap) return 0;
    (dev_free(p), ...);
    cap = 0;
    if ((dev_alloc(&p, n) || ...)) return TRACER_ERR_NOMEM;
    cap = n;
    return 0;
}

// Buffers of the device replay of the seeded draws (mt19937.cuh), grown as frames need them
struct MtWork {
    int *rank = nullptr, *row_hits = nullptr, *maps = nullptr, *start = nullptr, *fid_ord = nullptr;
    uint32_t *words = nullptr, *lights = nullptr;
    int64_t *base = nullptr, *ord = nullptr;
    size_t rank_cap = 0, rows_cap = 0, maps_cap = 0, start_cap = 0, fid_cap = 0, words_cap = 0, lights_cap = 0, base_cap = 0, ord_cap = 0;
    // a crop window's covering rows: the closest-hit pass's merged keys and hits, and the faceIDs replayed for them
    unsigned long long *cov_best = nullptr;
    int *cov_tri = nullptr, *cov_fid = nullptr;
    float *cov_t = nullptr, *cov_v = nullptr;
    size_t cov_cap = 0, cov_fid_cap = 0;
    void release() {
        dev_free(rank), dev_free(row_hits), dev_free(maps), dev_free(start), dev_free(fid_ord), dev_free(words), dev_free(lights);
        dev_free(base), dev_free(ord);
        dev_free(cov_best), dev_free(cov_tri), dev_free(cov_fid), dev_free(cov_t), dev_free(cov_v);
        rank_cap = rows_cap = maps_cap = start_cap = fid_cap = words_cap = lights_cap = base_cap = ord_cap = cov_cap = cov_fid_cap = 0;
    }
};

// The per-frame buffers of a scene, per pixel of the largest call so far (npx); dbg_occ and accum_total once a call needs them
struct Workspace {
    int npx = 0;
    int *hit_tri = nullptr, *rj = nullptr, *list = nullptr, *list_b = nullptr, *faceid = nullptr, *dbg_occ = nullptr;
    unsigned long long *best = nullptr, *best_occ = nullptr;
    float *hit_t = nullptr, *hit_v = nullptr, *carry = nullptr, *nrm = nullptr, *accum = nullptr, *ro = nullptr, *rd = nullptr,
          *re = nullptr, *rt = nullptr, *accum_total = nullptr;
    uint8_t *rgb8 = nullptr;
    void release() {
        dev_free(hit_tri), dev_free(rj), dev_free(best), dev_free(best_occ), dev_free(list), dev_free(list_b), dev_free(faceid);
        dev_free(hit_t), dev_free(hit_v), dev_free(carry), dev_free(nrm), dev_free(accum), dev_free(ro), dev_free(rd), dev_free(re);
        dev_free(rt), dev_free(rgb8), dev_free(dbg_occ), dev_free(accum_total);
        npx = 0;
    }
    trk::PixelState px() const { return {best, best_occ, hit_tri, hit_t, hit_v, carry, nrm, accum, ro, rd, re, rt, rj}; }
};

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
    std::vector<int> h_light_vbase, h_light_F, h_light_t0; // per light: first light vertex, faces, first triangle
    std::vector<float> h_light_verts;
    double bb_lo[3], bb_hi[3];
    void *box_work = nullptr; // bbox_partial_kernel's per-block bounds, then the 6 doubles of the box
    float4 *eye_table = nullptr, *light_tables = nullptr, *allcand_table = nullptr; // 48-byte three-row tables
    float4 *eye_span = nullptr, *light_spans = nullptr, *allcand_span = nullptr;    // 32-byte span tables (same slots)
    size_t eye_table_cap = 0, eye_span_cap = 0; // float4 of eye_table / eye_span: the eye tables of one view or more
    trk::Cam *cams = nullptr;       // the call's cameras, one per view
    size_t cams_cap = 0;
    std::vector<double> table_lmax; // per (light vertex, cube face): reach bound it was built for, < 0 = not built
    int table_slots = 1;            // light vertices whose 6 face tables fit at once (and per persistent-kernel launch)
    bool tables_resident = true;    // every light vertex has its own slot: tables are kept across lights and frames
    bool allcand_built = false;
    size_t table_stride = 0, span_stride = 0; // float4 per table
    Workspace ws;
    MtWork mt;
    // bundle-cull mode: candidate (ray<<32|triangle) buffers, their count, radix-sort scratch
    unsigned long long *cand_a = nullptr, *cand_b = nullptr, *cand_count = nullptr, *rkey = nullptr, *rkey_sorted = nullptr;
    int *blk_cnt = nullptr;            // order-preserving compaction: survivors per (group, block of CBLK entries)
    size_t blk_cnt_cap = 0;
    cull::BlockBoxes *boxes = nullptr; // two-phase bundle cull: boxes of every ray block
    size_t boxes_cap = 0;
    int *iota = nullptr;
    size_t pair_bytes = 0, pair_cap = 0;
    unsigned char *pair_tmp = nullptr;
    size_t rkey_cap = 0;
    size_t cand_cap = 0, sort_bytes = 0, sort_cap = 0, count_cap = 0;
    int cull_grow = 1; // candidate buffers hold 24 * cull_grow pairs per ray (grown after an overflow)
    unsigned char *sort_tmp = nullptr;
    int *seg_count = nullptr, *seg_off = nullptr, *blk_off = nullptr, *cursor = nullptr, *cnt_b = nullptr, *work = nullptr,
        *n_slices = nullptr;
    int maxF = 0;
    sweep::Counters *counters = nullptr;
    // optional BVH mode: built on the first BVH render, kept until the scene is destroyed
    bool bvh_built = false;
    bvh::Node *bvh_nodes = nullptr;
    unsigned long long *bvh_keys = nullptr; // sorted keys; the always-test list is the tail from bvh_tree.n_in on
    bvh::Tree bvh_tree{};
    double bvh_ext = 0.0; // largest |coordinate| of the tree's triangles
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> ev_shadow;
    tracer_frame_stats stats{};
};

namespace {

// L: faceIDs (and first occluders) per pixel
int ensure_workspace(Workspace &w, int n_px, int L, bool want_dbg_occ) {
    if (n_px > w.npx) {
        w.release();
        const size_t n = (size_t)n_px;
        int rc = 0;
        rc |= dev_alloc(&w.hit_tri, n) | dev_alloc(&w.rj, n) | dev_alloc(&w.best, n) | dev_alloc(&w.best_occ, n);
        rc |= dev_alloc(&w.list, n);
        rc |= dev_alloc(&w.list_b, n);
        rc |= dev_alloc(&w.faceid, n * L);
        rc |= dev_alloc(&w.hit_t, n) | dev_alloc(&w.hit_v, n) | dev_alloc(&w.carry, n);
        rc |= dev_alloc(&w.nrm, 3 * n) | dev_alloc(&w.accum, 3 * n + 16) | dev_alloc(&w.ro, 3 * n);
        rc |= dev_alloc(&w.rd, 3 * n) | dev_alloc(&w.re, 2 * n) | dev_alloc(&w.rt, n);
        rc |= dev_alloc(&w.rgb8, 3 * n + 64);
        if (rc) return TRACER_ERR_NOMEM;
        w.npx = n_px;
    }
    if (want_dbg_occ && !w.dbg_occ) {
        if (dev_alloc(&w.dbg_occ, (size_t)w.npx * L)) return TRACER_ERR_NOMEM;
    }
    return 0;
}

template <int R, bool EX, int MODE, bool VIEWS>
int launch_primary_v(const trk::PrimaryParams &p, int grid, cudaStream_t st) {
    const size_t smem = sizeof(sweep::SmemT<sweep::Rows<MODE>::N>);
    CK_CUDA(cudaFuncSetAttribute(trk::primary_kernel<R, EX, MODE, VIEWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    trk::primary_kernel<R, EX, MODE, VIEWS><<<grid, sweep::NT, smem, st>>>(p);
    CK_CUDA(cudaGetLastError());
    return 0;
}
// views: the launch covers several views (primary_kernel's per-item view decode); one view reads camera and table as parameters
template <int R, bool EX, int MODE>
int launch_primary_q(const trk::PrimaryParams &p, bool views, int grid, cudaStream_t st) {
    return views ? launch_primary_v<R, EX, MODE, true>(p, grid, st) : launch_primary_v<R, EX, MODE, false>(p, grid, st);
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
    const size_t smem = trk::SHADOW_SMEM;
    int &ctas_per_sm = g.sl_ctas[EX ? 1 : 0]; // co-resident CTAs: a cooperative launch may not exceed them
    if (!ctas_per_sm) {
        CK_CUDA(cudaFuncSetAttribute(trk::shadow_light_kernel<EX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, trk::shadow_light_kernel<EX>, sweep::NT, smem));
        if (ctas_per_sm < 1) return fail(TRACER_ERR_CUDA, "shadow_light_kernel does not fit on an SM");
        ctas_per_sm = std::min(ctas_per_sm, SHADOW_MINB);
    }
    void *args[] = {(void *)&p, (void *)&bar};
    CK_CUDA(cudaLaunchCooperativeKernel((const void *)trk::shadow_light_kernel<EX>, dim3((unsigned)(ctas_per_sm * g.n_sms)), dim3(sweep::NT), args, smem, st));
    return 0;
}
int launch_shadow_light(Ctx &g, bool ex, const trk::ShadowLightParams &p, unsigned *bar, cudaStream_t st) {
    return ex ? launch_shadow_light_t<true>(g, p, bar, st) : launch_shadow_light_t<false>(g, p, bar, st);
}
// Rays per thread R of each form of the closest-hit sweep, largest first: the primary_kernel instantiations there are.
// qmode sweep::MODE_SHAREDQ: no jitter, the rays of a thread share one exact q (span table); MODE_QBAR: jittered samples
// sharing a mean q (span table); MODE_OWNQ: jittered, every ray its own q (three-row table)
template <int QMODE, int... Rs>
struct RaysPerThread {
    static constexpr int n = sizeof...(Rs);
    static constexpr int r[] = {Rs...};
};
template <typename Fn>
auto with_rays_per_thread(int qmode, Fn &&fn) {
    if (qmode == sweep::MODE_OWNQ) return fn(RaysPerThread<sweep::MODE_OWNQ, 12, 8, 4, 2>{});
    if (qmode == sweep::MODE_QBAR) return fn(RaysPerThread<sweep::MODE_QBAR, 32, 16, 8, 4, 2>{});
    return fn(RaysPerThread<sweep::MODE_SHAREDQ, 64, 32, 24, 16, 8, 4, 2>{});
}
// the form's instantiation for r rays per thread (its last, 2, for an r it lacks)
template <int QMODE, int R, int... Rs>
int launch_primary_r(int r, bool ex, const trk::PrimaryParams &p, bool views, int grid, cudaStream_t st) {
    if constexpr (sizeof...(Rs) > 0)
        if (r != R) return launch_primary_r<QMODE, Rs...>(r, ex, p, views, grid, st);
    return ex ? launch_primary_q<R, true, QMODE>(p, views, grid, st) : launch_primary_q<R, false, QMODE>(p, views, grid, st);
}
template <int QMODE, int... Rs>
int launch_primary_of(RaysPerThread<QMODE, Rs...>, int r, bool ex, const trk::PrimaryParams &p, bool views, int grid, cudaStream_t st) {
    return launch_primary_r<QMODE, Rs...>(r, ex, p, views, grid, st);
}
int launch_primary(int R, bool ex, int qmode, const trk::PrimaryParams &p, bool views, int grid, cudaStream_t st) {
    return with_rays_per_thread(qmode, [&](auto rays) { return launch_primary_of(rays, R, ex, p, views, grid, st); });
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

Decomp pick_decomp(int64_t n_rays, int n_tiles, int n_sms, int forced_R, int qmode) {
    const int slices_possible = std::max(1, n_tiles / 4); // at least 4 tiles per slice
    auto blocks_for = [&](int R) { return (int)((n_rays + (int64_t)sweep::NT * R - 1) / ((int64_t)sweep::NT * R)); };
    Decomp d{2, blocks_for(2), 1};
    // rays per thread: forced_R when the form has it, else the largest that gives enough work items (24 only on request)
    // (C4 closest-hit sweep on one B200: 997 ms at 16, 944 at 24, 905 at 32 with the saturating span loop)
    const auto [rs, n_rs] = with_rays_per_thread(qmode, [](auto rays) { return std::make_pair(rays.r, rays.n); });
    if (std::find(rs, rs + n_rs, forced_R) != rs + n_rs) {
        d.R = forced_R, d.n_blocks = blocks_for(forced_R);
    } else {
        for (const int *R = rs; R != rs + n_rs; ++R) {
            if (*R == 24) continue;
            d.R = *R, d.n_blocks = blocks_for(*R);
            if ((int64_t)d.n_blocks * slices_possible >= 4 * (int64_t)n_sms) break;
        }
    }
    const int64_t ips = (int64_t)items_per_cta() * trk::primary_minb(d.R);
    const int64_t want = (ips * (int64_t)n_sms + d.n_blocks - 1) / std::max(1, d.n_blocks);
    d.n_slices = d.n_blocks >= ips * n_sms ? 1 : (int)std::max<int64_t>(1, std::min<int64_t>(want, slices_possible));
    return d;
}

// both forms of the filter table of one origin: the 48-byte rows (jittered primary rays, bundle-cull mode) and the
// 32-byte span rows (default sweeps).  count >= 0: only the rows of triangles [first, first + count) (a scene update; a
// row depends on tp and its own triangle only, so they equal those of a full build); the padding rows are left alone.
int build_table(const tracer_scene_dev *s, const trk::TableParam &tp, float4 *table, float4 *span, cudaStream_t st, int first = 0,
                int count = -1) {
    const int th = 128;
    const int n_tris = count < 0 ? s->n_tris : count, n_pad = count < 0 ? s->n_pad : count;
    if (n_pad == 0) return 0;
    trk::build_origin_table<<<(n_pad + th - 1) / th, th, 0, st>>>(s->tri_verts + 9 * (size_t)first, n_tris, n_pad, tp,
                                                                  table + 3 * (size_t)first, span + 2 * (size_t)first);
    CK_CUDA(cudaGetLastError());
    return 0;
}

// ---- the scene's bounding box, on the device --------------------------------------------------------------------------------
// What the host loop over the flat arrays gave: in order, every triangle vertex (double)x, then every sphere's x -/+ |r| in
// double, folded with lo = std::min(lo, x), hi = std::max(hi, x) from (1e300, -1e300).  A NaN never replaces a bound (it
// fails every comparison) and infinities count.  A parallel fold gives the same bits when each bound carries the ordinal of
// the item that set it and, between equal values (only -0.0 and +0.0 differ in their bits), the lower ordinal wins: the
// sequential loop keeps the first of equal values.
struct BoxArg {
    double v;
    long long i; // ordinal: vertex k -> k, sphere j -> 3 n_tris + j
};
constexpr int BOX_THREADS = 256, BOX_MAX_BLOCKS = 1024;
__device__ __forceinline__ void box_take(BoxArg &a, double v, long long i, bool upper) {
    if ((upper ? v > a.v : v < a.v) || (v == a.v && i < a.i)) a.v = v, a.i = i;
}
// b = 0..2: lo x y z, 3..5: hi x y z; folds the block's threads into a[*] of thread 0
__device__ void box_block_fold(BoxArg (&a)[6]) {
    __shared__ BoxArg sh[6][BOX_THREADS];
    for (int b = 0; b < 6; ++b) sh[b][threadIdx.x] = a[b];
    __syncthreads();
    for (int w = BOX_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w)
            for (int b = 0; b < 6; ++b) {
                const BoxArg o = sh[b][threadIdx.x + w];
                box_take(sh[b][threadIdx.x], o.v, o.i, b >= 3);
            }
        __syncthreads();
    }
    for (int b = 0; b < 6; ++b) a[b] = sh[b][0];
}
__global__ void __launch_bounds__(BOX_THREADS) bbox_partial_kernel(const float *__restrict__ verts, long long n_verts,
                                                                   const float4 *__restrict__ spheres, int n_spheres, BoxArg *partial) {
    BoxArg a[6];
    for (int b = 0; b < 6; ++b) a[b] = BoxArg{b < 3 ? 1e300 : -1e300, LLONG_MAX};
    const long long n = n_verts + n_spheres, stride = (long long)gridDim.x * BOX_THREADS;
    for (long long k = blockIdx.x * (long long)BOX_THREADS + threadIdx.x; k < n; k += stride) {
        if (k < n_verts) {
            for (int c = 0; c < 3; ++c) {
                const double x = verts[3 * k + c];
                box_take(a[c], x, k, false), box_take(a[3 + c], x, k, true);
            }
        } else {
            const float4 sp = spheres[k - n_verts];
            const double r = fabs((double)sp.w), xs[3] = {sp.x, sp.y, sp.z};
            for (int c = 0; c < 3; ++c) box_take(a[c], xs[c] - r, k, false), box_take(a[3 + c], xs[c] + r, k, true);
        }
    }
    box_block_fold(a);
    if (threadIdx.x == 0)
        for (int b = 0; b < 6; ++b) partial[6 * (size_t)blockIdx.x + b] = a[b];
}
__global__ void __launch_bounds__(BOX_THREADS) bbox_final_kernel(const BoxArg *__restrict__ partial, int n_blocks, double *out6) {
    BoxArg a[6];
    for (int b = 0; b < 6; ++b) a[b] = BoxArg{b < 3 ? 1e300 : -1e300, LLONG_MAX};
    for (int k = threadIdx.x; k < n_blocks; k += BOX_THREADS)
        for (int b = 0; b < 6; ++b) box_take(a[b], partial[6 * (size_t)k + b].v, partial[6 * (size_t)k + b].i, b >= 3);
    box_block_fold(a);
    if (threadIdx.x == 0)
        for (int b = 0; b < 6; ++b) out6[b] = a[b].v;
}

// The BVH of the optional mode (bvh.cuh), on stream st: prep (boxes, sigma, bounds) -> Morton keys -> radix sort ->
// Karras nodes -> bottom-up refit.  One read-back when it is built (tree size and bounds, for the per-frame margin).
int ensure_bvh(tracer_scene_dev *s, cudaStream_t st) {
    if (s->bvh_built) return 0;
    const int n = s->n_tris;
    float4 *tlo = nullptr, *thi = nullptr;
    unsigned long long *keys = nullptr;
    int *parent = nullptr, *leaf_parent = nullptr, *flags = nullptr;
    bvh::BuildHdr *hdr = nullptr;
    void *tmp = nullptr;
    struct Scratch { // build-only buffers, back to the pool on every return path
        float4 *&a, *&b;
        unsigned long long *&k;
        int *&p, *&lp, *&f;
        bvh::BuildHdr *&h;
        void *&t;
        ~Scratch() { dev_free(a), dev_free(b), dev_free(k), dev_free(p), dev_free(lp), dev_free(f), dev_free(h), t_pool->release(t); }
    } scratch{tlo, thi, keys, parent, leaf_parent, flags, hdr, tmp};
    const size_t N = (size_t)std::max(n, 1);
    dev_free(s->bvh_nodes), dev_free(s->bvh_keys);
    if (dev_alloc(&tlo, N) || dev_alloc(&thi, N) || dev_alloc(&keys, N) || dev_alloc(&s->bvh_keys, N) || dev_alloc(&parent, N) ||
        dev_alloc(&leaf_parent, N) || dev_alloc(&flags, N) || dev_alloc(&s->bvh_nodes, N) || dev_alloc(&hdr, 1))
        return TRACER_ERR_NOMEM;
    bvh::BuildHdr h0{};
    for (int c = 0; c < 6; ++c) h0.cb[c] = h0.bb[c] = c < 3 ? 0xffffffffu : 0u;
    CK_CUDA(cudaMemcpyAsync(hdr, &h0, sizeof h0, cudaMemcpyHostToDevice, st));
    const int th = 256, blocks = (int)((N + th - 1) / th);
    if (n > 0) {
        bvh::prep_kernel<<<blocks, th, 0, st>>>(s->tri_verts, n, tlo, thi, hdr);
        CK_CUDA(cudaGetLastError());
        bvh::key_kernel<<<blocks, th, 0, st>>>(tlo, thi, n, hdr, keys);
        CK_CUDA(cudaGetLastError());
        size_t tmp_bytes = 0;
        CK_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, keys, s->bvh_keys, n, 0, 64, st));
        if (!(tmp = t_pool->alloc(tmp_bytes))) return fail(TRACER_ERR_NOMEM, "BVH sort scratch");
        CK_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, keys, s->bvh_keys, n, 0, 64, st));
    }
    bvh::BuildHdr hh{};
    CK_CUDA(cudaMemcpyAsync(&hh, hdr, sizeof hh, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    const int n_in = hh.n_in;
    if (n_in >= 2) {
        bvh::nodes_kernel<<<(n_in - 1 + th - 1) / th, th, 0, st>>>(s->bvh_keys, n_in, s->bvh_nodes, parent, leaf_parent, flags);
        CK_CUDA(cudaGetLastError());
        bvh::refit_kernel<<<(n_in + th - 1) / th, th, 0, st>>>(s->bvh_keys, n_in, tlo, thi, s->bvh_nodes, parent, leaf_parent, flags);
        CK_CUDA(cudaGetLastError());
    }
    int root_leaf = -1;
    if (n_in == 1) {
        unsigned long long k0 = 0;
        CK_CUDA(cudaMemcpyAsync(&k0, s->bvh_keys, sizeof k0, cudaMemcpyDeviceToHost, st));
        CK_CUDA(cudaStreamSynchronize(st));
        root_leaf = (int)(k0 & 0xffffffffull);
    }
    CK_CUDA(cudaStreamSynchronize(st)); // the scratch buffers go back to the pool when this returns
    s->bvh_tree = bvh::Tree{s->bvh_nodes, n_in, root_leaf, s->bvh_keys + n_in, n - n_in};
    s->bvh_ext = 0.0;
    if (n_in > 0)
        for (int c = 0; c < 6; ++c) s->bvh_ext = std::max(s->bvh_ext, (double)std::fabs(bvh::unord(hh.bb[c])));
    s->bvh_built = true;
    if (std::getenv("TRACER_BVH_DIAG"))
        std::fprintf(stderr, "bvh: %d triangles in the tree, %d on the always-test list (non-finite or sigma >= %g)\n", n_in, n - n_in,
                     (double)bvh::SIGMA_MAX);
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

// The shadow filter tables (both forms) of cube face `face` of light vertex vtx, in table slot `slot`: vtx itself when every
// vertex has its own slot (tables_resident: kept across lights and frames), else its place in the batch of vertices whose
// tables the slots hold (rebuilt every time).  A full build serves shadow segments up to `need`, with 1.5x head-room so
// that camera moves rarely trigger a rebuild; a resident table already built for `need` or more is kept.  count >= 0 (a
// scene update): only rows [first, first + count) of a built resident table, for the bound it was built with.
int build_face_table(tracer_scene_dev *s, int vtx, int face, size_t slot, double need, cudaStream_t st, int &launches, int first = 0,
                     int count = -1) {
    double lmax = need * 1.5;
    if (s->tables_resident) {
        double &built = s->table_lmax[(size_t)vtx * 6 + face];
        if (count >= 0) lmax = built;
        else if (built >= need) return 0;
        else built = lmax;
    }
    const trk::TableParam tp = face_param(&s->h_light_verts[3 * (size_t)vtx], face, lmax);
    if (int rc = build_table(s, tp, s->light_tables + (slot * 6 + face) * s->table_stride, s->light_spans + (slot * 6 + face) * s->span_stride,
                             st, first, count))
        return rc;
    ++launches;
    return 0;
}

// The table of every light vertex's last ray group (trk::NFACE - 1), every row a candidate: built once per scene
int ensure_allcand_table(tracer_scene_dev *s, cudaStream_t st, int &launches) {
    if (s->allcand_built) return 0;
    trk::build_allcand_table<<<(s->n_pad + 255) / 256, 256, 0, st>>>(s->n_tris, s->n_pad, s->allcand_table, s->allcand_span);
    CK_CUDA(cudaGetLastError());
    s->allcand_built = true, ++launches;
    return 0;
}

// s->bb_lo, s->bb_hi from the scene's device arrays (bbox_partial_kernel): two launches on st, one read-back, a synchronise
int scene_bbox(tracer_scene_dev *s, cudaStream_t st) {
    if (!s->box_work && !(s->box_work = t_pool->alloc(sizeof(BoxArg) * 6 * BOX_MAX_BLOCKS + sizeof(double) * 6)))
        return fail(TRACER_ERR_NOMEM, "bounding-box scratch");
    BoxArg *partial = (BoxArg *)s->box_work;
    double *out6 = (double *)(partial + 6 * BOX_MAX_BLOCKS);
    const long long n_verts = 3 * (long long)s->n_tris, n = n_verts + s->n_spheres;
    const int blocks = (int)std::max(1LL, std::min<long long>(BOX_MAX_BLOCKS, (n + BOX_THREADS - 1) / BOX_THREADS));
    bbox_partial_kernel<<<blocks, BOX_THREADS, 0, st>>>(s->tri_verts, n_verts, s->spheres, s->n_spheres, partial);
    CK_CUDA(cudaGetLastError());
    bbox_final_kernel<<<1, BOX_THREADS, 0, st>>>(partial, blocks, out6);
    CK_CUDA(cudaGetLastError());
    double box[6];
    CK_CUDA(cudaMemcpyAsync(box, out6, sizeof box, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    for (int c = 0; c < 3; ++c) s->bb_lo[c] = box[c], s->bb_hi[c] = box[3 + c];
    return 0;
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
    dev_free(s->eye_span), dev_free(s->light_spans), dev_free(s->allcand_span), dev_free(s->cams);
    s->ws.release();
    dev_free(s->seg_count), dev_free(s->seg_off), dev_free(s->blk_off), dev_free(s->cursor), dev_free(s->cnt_b), dev_free(s->work);
    dev_free(s->n_slices);
    dev_free(s->cand_a), dev_free(s->cand_b), dev_free(s->cand_count), dev_free(s->rkey), dev_free(s->rkey_sorted), dev_free(s->iota);
    dev_free(s->boxes), dev_free(s->blk_cnt);
    dev_free(s->sort_tmp), dev_free(s->pair_tmp);
    dev_free(s->counters);
    dev_free(s->bvh_nodes), dev_free(s->bvh_keys);
    t_pool->release(s->box_work);
    s->mt.release();
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

    // lives until the upload has been waited for: declared before the scene, whose destroy waits for the device
    std::vector<int> tg((size_t)std::max(N, 1));
    CK_CUDA(cudaSetDevice(g.device));
    // destroyed on every failure return, handed out on success
    std::unique_ptr<tracer_scene_dev, void (*)(tracer_scene_dev *)> s(new tracer_scene_dev(), tracer_cuda_scene_destroy);
    s->ctx = &g;
    s->n_geoms = G, s->n_tris = N, s->n_lights = sc->n_lights, s->n_spheres = sc->n_spheres;
    s->n_pad = std::max(1, (N + cull::CTILE - 1) / cull::CTILE) * cull::CTILE; // multiple of both tile sizes
    s->table_stride = (size_t)s->n_pad * 3, s->span_stride = (size_t)s->n_pad * 2;
    if (int rc = dev_alloc(&s->tri_verts, (size_t)N * 9)) return rc;
    CK_CUDA(cudaMemcpyAsync(s->tri_verts, sc->tri_verts, (size_t)N * 9 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
    if (any_normals) {
        if (int rc = dev_alloc(&s->tri_normals, (size_t)N * 9)) return rc;
        CK_CUDA(cudaMemcpyAsync(s->tri_normals, sc->tri_normals, (size_t)N * 9 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
        if (int rc = dev_alloc(&s->geom_has_normals, (size_t)G)) return rc;
        CK_CUDA(cudaMemcpyAsync(s->geom_has_normals, sc->geom_has_normals, (size_t)G * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    }
    if (int rc = dev_alloc(&s->geom_material, (size_t)G * 13)) return rc;
    CK_CUDA(cudaMemcpyAsync(s->geom_material, sc->geom_material, (size_t)G * 13 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
    for (int g2 = 0; g2 < G; ++g2)
        for (int t = sc->geom_tri_offset[g2]; t < sc->geom_tri_offset[g2 + 1]; ++t) tg[t] = g2;
    if (int rc = dev_alloc(&s->tri_geom, (size_t)N)) return rc;
    CK_CUDA(cudaMemcpyAsync(s->tri_geom, tg.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    if (sc->n_spheres > 0) {
        if (int rc = dev_alloc(&s->spheres, (size_t)sc->n_spheres)) return rc;
        CK_CUDA(cudaMemcpyAsync(s->spheres, sc->sphere_cr, (size_t)sc->n_spheres * 4 * sizeof(float), cudaMemcpyHostToDevice, g.stream));
        if (int rc = dev_alloc(&s->sphere_material, (size_t)sc->n_spheres * 13)) return rc;
        CK_CUDA(cudaMemcpy(s->sphere_material, sc->sphere_material, (size_t)sc->n_spheres * 13 * sizeof(float),
                            cudaMemcpyHostToDevice));
    }
    // bounding box of everything a ray can start from or end at, from the uploaded arrays (the kernel an update uses too)
    if (int rc = scene_bbox(s.get(), g.stream)) return rc;
    // lights: light.vertex[faceID], faceID in [0, F) (main.cpp:743-751) = the first F de-indexed vertices
    s->h_light_vbase.assign(1, 0);
    for (int l = 0; l < sc->n_lights; ++l) {
        const int lg = sc->light_geom[l];
        if (lg < 0 || lg >= G) return fail(TRACER_ERR_INVALID, "light_geom index out of range");
        const int t0 = sc->geom_tri_offset[lg], F = sc->geom_tri_offset[lg + 1] - t0;
        if (F <= 0) return fail(TRACER_ERR_INVALID, "light geometry has no faces");
        s->h_light_F.push_back(F);
        s->h_light_t0.push_back(t0);
        for (int f = 0; f < F; ++f)
            for (int c = 0; c < 3; ++c) s->h_light_verts.push_back(sc->tri_verts[9 * (size_t)t0 + 3 * (size_t)f + c]);
        s->h_light_vbase.push_back(s->h_light_vbase.back() + F);
        s->maxF = std::max(s->maxF, F);
    }
    s->V = s->h_light_vbase.back();
    if (int rc = dev_alloc(&s->light_vbase, s->h_light_vbase.size())) return rc;
    CK_CUDA(cudaMemcpyAsync(s->light_vbase, s->h_light_vbase.data(), s->h_light_vbase.size() * sizeof(int), cudaMemcpyHostToDevice, g.stream));
    if (int rc = dev_alloc(&s->light_verts, s->h_light_verts.size())) return rc;
    CK_CUDA(cudaMemcpyAsync(s->light_verts, s->h_light_verts.data(), s->h_light_verts.size() * sizeof(float), cudaMemcpyHostToDevice, g.stream));
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
    if (int rc = dev_grow(s->eye_table_cap, s->table_stride, s->eye_table)) return rc;
    if (int rc = dev_alloc(&s->light_tables, s->table_stride * 6 * (size_t)std::max(1, s->tables_resident ? s->V : s->table_slots))) return rc;
    if (int rc = dev_alloc(&s->allcand_table, s->table_stride)) return rc;
    if (int rc = dev_grow(s->eye_span_cap, s->span_stride, s->eye_span)) return rc;
    if (int rc = dev_alloc(&s->light_spans, s->span_stride * 6 * (size_t)std::max(1, s->tables_resident ? s->V : s->table_slots))) return rc;
    if (int rc = dev_alloc(&s->allcand_span, s->span_stride)) return rc;
    s->table_lmax.assign((size_t)6 * s->V, -1.0);
    const size_t n_groups = (size_t)s->maxF * trk::NFACE;
    if (int rc = dev_alloc(&s->seg_count, n_groups + 1)) return rc;
    if (int rc = dev_alloc(&s->seg_off, n_groups + 2)) return rc;
    if (int rc = dev_alloc(&s->blk_off, n_groups + 2)) return rc;
    if (int rc = dev_alloc(&s->cursor, n_groups + 1)) return rc;
    if (int rc = dev_alloc(&s->cnt_b, n_groups + 1)) return rc;
    if (int rc = dev_alloc(&s->work, (size_t)WORK_INTS)) return rc;
    if (int rc = dev_alloc(&s->n_slices, 1)) return rc;
    if (int rc = dev_alloc(&s->counters, 1)) return rc;
    for (auto &e : s->ev) CK_CUDA(cudaEventCreate(&e));
    s->ev_shadow.resize(2 * (size_t)std::max(1, s->n_lights));
    for (auto &e : s->ev_shadow) CK_CUDA(cudaEventCreate(&e));
    // uploads were queued on the context's stream (truly asynchronous from pinned host memory): one wait for all
    if (cudaError_t e_ = cudaStreamSynchronize(g.stream); e_ != cudaSuccess)
        return fail(TRACER_ERR_CUDA, std::string("scene upload failed: ") + cudaGetErrorString(e_));
    *out = s.release();
    return TRACER_OK;
}
}  // namespace

namespace {
// ---- the seeded draws (TRACER_RNG_MT19937), replayed on the device: mt19937.cuh -------------------------------------------
// In-row hit ranks of the n_rows local rows (on the device) and their hit counts (read back into `local`)
int mt_count_rows(MtWork &m, const int *hit_tri, int W, int n_rows, cudaStream_t st, std::vector<int> &local) {
    local.assign((size_t)n_rows, 0);
    if (n_rows == 0) return 0;
    if (dev_grow(m.rank_cap, (size_t)n_rows * W, m.rank) || dev_grow(m.rows_cap, (size_t)n_rows, m.row_hits)) return TRACER_ERR_NOMEM;
    mt::row_rank_kernel<<<n_rows, mt::SCAN_THREADS, 0, st>>>(hit_tri, W, m.rank, m.row_hits);
    CK_CUDA(cudaGetLastError());
    CK_CUDA(cudaMemcpyAsync(local.data(), m.row_hits, sizeof(int) * (size_t)n_rows, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// The frame's [H] row hit counts from this call's own: the whole frame, or a band selection completed by the caller's hook
int mt_frame_rows(const tracer_render_opts &o, int W, int H, int band_rows, int band_count, const std::vector<int> &local,
                  std::vector<int> &frame) {
    const int bi = band_count > 1 ? o.band_index : 0, n_rows = (int)local.size();
    frame.assign((size_t)H, 0);
    mt::own_rows(local.data(), n_rows, band_rows, bi, band_count, frame.data(), H);
    if (band_count <= 1) return 0;
    const int32_t r = o.row_hits_exchange(o.row_hits_user, H, frame.data());
    if (r != 0) return fail(TRACER_ERR_STATE, "row_hits_exchange returned " + std::to_string(r));
    if (!mt::rows_valid(local.data(), n_rows, band_rows, bi, band_count, frame.data(), H, W))
        return fail(TRACER_ERR_INVALID, "row_hits_exchange changed this call's rows or gave a count outside [0, width]");
    return 0;
}

// faceid[k*L + l] of every hit local pixel k, from the frame's row counts: the stream, the automaton, the gather
// (rank_off: where these rows' in-row ranks start in m.rank, when mt_count_rows counted more rows than these)
int mt_replay(MtWork &m, uint32_t seed, const std::vector<int> &faces, const std::vector<int> &frame, int W, int band_rows,
              int band_index, int band_count, int n_rows, const int *hit_tri, int *faceid, cudaStream_t st, int &launches,
              size_t rank_off = 0) {
    const int L = (int)faces.size(), S = 3 * L, n_px = n_rows * W;
    if (L == 0 || n_rows == 0) return 0;
    std::vector<int64_t> base((size_t)n_rows);
    const int64_t T = mt::row_bases(frame.data(), (int)frame.size(), n_rows, band_rows, band_index, band_count, base.data());
    if (T == 0) return 0;
    std::vector<uint32_t> lights((size_t)2 * L);
    for (int l = 0; l < L; ++l) lights[l] = (uint32_t)faces[l], lights[L + l] = mt::threshold((uint32_t)faces[l]);
    if (dev_grow(m.lights_cap, lights.size(), m.lights) || dev_grow(m.base_cap, base.size(), m.base) ||
        dev_grow(m.fid_cap, (size_t)T * L, m.fid_ord))
        return TRACER_ERR_NOMEM;
    CK_CUDA(cudaMemcpyAsync(m.lights, lights.data(), sizeof(uint32_t) * lights.size(), cudaMemcpyHostToDevice, st));
    CK_CUDA(cudaMemcpyAsync(m.base, base.data(), sizeof(int64_t) * base.size(), cudaMemcpyHostToDevice, st));
    // 3L words per hit pixel without rejections; when rejections leave the stream short, a longer one is generated
    int64_t D = 3 * (int64_t)L * T, C = 0, n_chunks = 0;
    for (;;) {
        C = std::max<int64_t>(256, (D + 2047) / 2048), n_chunks = (D + C - 1) / C;
        if (dev_grow(m.words_cap, (size_t)D, m.words) || dev_grow(m.maps_cap, (size_t)(2 * n_chunks * S), m.maps) ||
            dev_grow(m.start_cap, (size_t)n_chunks, m.start) || dev_grow(m.ord_cap, (size_t)n_chunks + 1, m.ord))
            return TRACER_ERR_NOMEM;
        mt::stream_kernel<<<1, mt::GEN_THREADS, 0, st>>>(seed, D, m.words);
        CK_CUDA(cudaGetLastError());
        const int64_t n_maps = n_chunks * S;
        mt::chunk_map_kernel<<<(unsigned)((n_maps + mt::AUTO_THREADS - 1) / mt::AUTO_THREADS), mt::AUTO_THREADS, 0, st>>>(
            m.words, D, C, n_chunks, L, m.lights, m.maps, m.maps + n_maps);
        CK_CUDA(cudaGetLastError());
        mt::chain_kernel<<<1, 1, 0, st>>>(n_chunks, L, m.maps, m.maps + n_maps, m.start, m.ord);
        CK_CUDA(cudaGetLastError());
        launches += 3;
        int64_t done = 0;
        CK_CUDA(cudaMemcpyAsync(&done, m.ord + n_chunks, sizeof done, cudaMemcpyDeviceToHost, st));
        CK_CUDA(cudaStreamSynchronize(st));
        if (done >= T) break;
        D += 3 * (int64_t)L * (T - done) + D / 16;
    }
    mt::chunk_faceids_kernel<<<(unsigned)((n_chunks + mt::AUTO_THREADS - 1) / mt::AUTO_THREADS), mt::AUTO_THREADS, 0, st>>>(
        m.words, D, C, n_chunks, T, L, m.lights, m.start, m.ord, m.fid_ord);
    CK_CUDA(cudaGetLastError());
    mt::gather_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(hit_tri, W, n_px, L, m.base, m.rank + rank_off, m.fid_ord, faceid);
    CK_CUDA(cudaGetLastError());
    launches += 2;
    return 0;
}

// Eye tables kept per call: views in groups whose tables (both forms, n_pad x 80 B per view) fit a quarter of the free
// device memory, one closest-hit launch per group.  (TRACER_VIEW_GROUP caps the group size: development/test knob.)
int view_group_size(tracer_scene_dev *s, int n_views) {
    const char *e = std::getenv("TRACER_VIEW_GROUP");
    const int cap = e ? std::max(1, std::atoi(e)) : INT_MAX;
    const size_t held = s->eye_table_cap / s->table_stride; // views whose tables the scene already holds
    if ((size_t)n_views <= held) return std::min(n_views, cap);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const size_t per_view = (s->table_stride + s->span_stride) * sizeof(float4);
    const size_t fit = std::max<size_t>(held, free_b / 4 / per_view);
    return (int)std::max<size_t>(1, std::min<size_t>({fit, (size_t)cap, (size_t)n_views}));
}

// The caller's options; fields past a caller's struct_size are 0
tracer_render_opts read_opts(const tracer_render_opts *in) {
    tracer_render_opts o;
    std::memset(&o, 0, sizeof o);
    if (in) std::memcpy(&o, in, std::min<size_t>(sizeof o, in->struct_size ? in->struct_size : sizeof o));
    return o;
}
// any crop field set: the call renders a window of the frame (render_views checks it)
bool has_crop(const tracer_render_opts &o) { return o.crop_x || o.crop_y || o.crop_w || o.crop_h; }

// ---- one render call: n_views frames of one scene, one per camera (V = 1: tracer_cuda_render_scene) -------------------------
// The call's pixels run view-major (k = view * W * n_rows + local); every per-pixel buffer, sort and list spans all of them,
// and the shadow sweeps take the rays of every view at once.  Only the closest-hit sweep is per view: one eye table each, in
// groups (DESIGN §4e).  Per sample: closest hit, faceIDs (first sample), then per light a light step and a shadow sweep.

// The render modes.  The values are light_step_kernel's cull_cells: which shadow-ray sort key it writes.
enum Mode { BVH = 0, CULL = 1, SWEEPS = 2 };
// Frame::render's outcome when the bundle-cull candidate buffer overflowed (not a status code: render_views renders again)
constexpr int CAND_OVERFLOW = 1;

// A closest-hit pass: its pixels (bands.n_px, in local rows of bands.crop_w), the local rows they span, and the planes it
// leaves its merged keys and hits in
struct HitPass {
    trk::Bands bands;
    trk::Views views;
    int n_rows;
    unsigned long long *best;
    int *hit_tri;
    float *hit_t, *hit_v;
};

// One attempt at the frames of one call: the scene, the checked options, what follows from them, and the counts it adds up
struct Frame {
    tracer_scene_dev *s;
    Ctx &g;
    const tracer_render_opts &o;
    const tracer_camera *cams;
    cudaStream_t st;
    int W, H, n_rows, view_px, n_px, n_views, L, S; // S: samples per pixel; n_rows, view_px: local rows of bands.crop_w pixels
    trk::Bands bands;
    // a crop window with TRACER_RNG_MT19937: the closest-hit pass covers PPM rows [0, cover_rows) at full width, whose hits
    // fix the crop's faceIDs (DESIGN §4f); 0 = the pass covers the call's own pixels
    int cover_rows;
    trk::Views views{};
    std::vector<trk::Cam> h_cams;
    double diag = 0;    // reach bound of a primary ray's hit point; light k's shadow segments are bounded by (k+1) * diag
    double bvh_ext = 0; // BVH mode: largest |coordinate| of the tree and every eye
    Mode mode = SWEEPS;
    bool two_phase = false;        // bundle-cull mode: block lists first (cull.cuh), not only the streaming kernels
    int group = 1, n_groups = 1;   // eye tables: n_groups groups of up to `group` views
    unsigned long long em_cap = 0; // candidate pairs the bundle-cull kernels may emit
    int tri_bits = 1;              // bits of a triangle index in a block-list key
    trk::PixelState px{};
    int launches = 0;
    int64_t host_tests_primary = 0, host_tests_shadow = 0; // pairs considered by two-phase sweeps (every block x every triangle)
    double flop_primary = 0.0;       // executed FP32 flops per swept pair of the closest-hit sweep (default mode)
    double flop_primary_edges = 0.0; // of which bound-evaluating multiply-adds
    double ms_primary = 0, ms_shadow = 0; // event times, summed over the samples

    int render(uint8_t *rgb_out, std::vector<int> &frame_rows, bool &rows_known);
    int setup();
    int build_eye_tables(int v0, int v1);
    size_t hit_px() const { return cover_rows ? (size_t)W * cover_rows : (size_t)n_px; }
    HitPass hit_pass() const;
    int closest_hit();
    int primary_sweeps(const HitPass &hp);
    int primary_cull(const HitPass &hp);
    int primary_bvh(const HitPass &hp);
    int block_lists(cull::L0Params lp, int max_blocks, long long &n_keys);
    int faceids(std::vector<int> &frame_rows, bool &rows_known);
    int light(int k, uint32_t seed);
    int order_shadow_rays(int F);
    int shadow_sweeps(int k);
    int shadow_cull(int k);
    int shadow_bvh(int k);
    int accumulate(int smp);
    void add_sample_times();
    int finish_frame(uint8_t *rgb_out);
};

// frame_rows, rows_known: the frame's row hit counts (TRACER_RNG_MT19937), known once the exchange hook has run; a render
// again after an overflow checks its own against them (the hook runs once per frame)
int Frame::render(uint8_t *rgb_out, std::vector<int> &frame_rows, bool &rows_known) {
    CK_CUDA(cudaSetDevice(g.device));
    std::memset(&s->stats, 0, sizeof s->stats);
    s->stats.n_sms = g.n_sms;
    s->stats.n_pixels = n_px;
    if (n_px == 0)
        return o.rng_mode == TRACER_RNG_MT19937 && bands.band_count > 1 ? mt_frame_rows(o, W, H, bands.band_rows, bands.band_count, {}, frame_rows)
                                                                         : TRACER_OK;
    if (int rc = setup()) return rc;
    for (int smp = 0; smp < S; ++smp) {
        bands.sample = smp;
        if (int rc = closest_hit()) return rc;
        if (smp == 0)
            if (int rc = faceids(frame_rows, rows_known)) return rc;
        const uint32_t seed = o.seed + (uint32_t)smp * 0x9e3779b1u; // faceID stream of this sample
        for (int k = 0; k <= L; ++k)
            if (int rc = light(k, seed)) return rc;
        if (S > 1)
            if (int rc = accumulate(smp)) return rc;
    }
    return finish_frame(rgb_out);
}

// Workspace, cameras, reach bound, mode, and the buffers and tables the mode needs before the first sample
int Frame::setup() {
    if (int rc = ensure_workspace(s->ws, n_px, std::max(1, L), o.out_occ_tri != nullptr)) return rc;
    h_cams.resize((size_t)n_views);
    for (int v = 0; v < n_views; ++v) {
        trk::Cam &c = h_cams[v];
        std::memcpy(c.o, cams[v].origin, 12), std::memcpy(c.llc, cams[v].lower_left_corner, 12);
        std::memcpy(c.hor, cams[v].horizontal, 12), std::memcpy(c.ver, cams[v].vertical, 12);
    }
    if (dev_grow(s->cams_cap, (size_t)n_views, s->cams)) return TRACER_ERR_NOMEM;
    CK_CUDA(cudaMemcpyAsync(s->cams, h_cams.data(), sizeof(trk::Cam) * (size_t)n_views, cudaMemcpyHostToDevice, st));
    views = trk::Views{s->cams, view_px};

    // reach bound for shadow segments: len_k <= (k+1) * diag(bbox U every eye)  (t carries over lights, main.cpp:764).  One
    // bound for all views: a view's own would be smaller, and a table built for a larger bound is only looser (DESIGN §4e)
    double lo[3], hi[3], diag2 = 0;
    for (int c = 0; c < 3; ++c) {
        lo[c] = s->bb_lo[c], hi[c] = s->bb_hi[c];
        for (int v = 0; v < n_views; ++v) lo[c] = std::min(lo[c], (double)cams[v].origin[c]), hi[c] = std::max(hi[c], (double)cams[v].origin[c]);
        if (hi[c] >= lo[c]) diag2 += (hi[c] - lo[c]) * (hi[c] - lo[c]);
    }
    diag = std::sqrt(diag2) * 1.001 + 1e-30;

    // bundle_cull: 1 two-phase, 2 streaming, 3 auto = two-phase unless the default sweeps are estimated to be the
    // faster of the two (tiny scenes: the mode has a fixed cost of a few ms in sorts and count read-backs)
    const double est_default_ms = (double)n_px * (double)s->n_tris * (1.0 + 0.25 * L) / 4.0e9;
    // (the optional mode keeps every light vertex's tables resident; a light too big for that renders in the default mode)
    if (o.accel == 1) mode = BVH;
    else if (s->tables_resident && (o.bundle_cull == 3 ? est_default_ms > 6.0 : o.bundle_cull != 0)) mode = CULL;
    two_phase = mode == CULL && o.bundle_cull != 2;

    group = mode == BVH ? n_views : view_group_size(s, n_views), n_groups = (n_views + group - 1) / group;
    if (mode != BVH && (dev_grow(s->eye_table_cap, s->table_stride * group, s->eye_table) ||
                        dev_grow(s->eye_span_cap, s->span_stride * group, s->eye_span)))
        return TRACER_ERR_NOMEM;
    CK_CUDA(cudaEventRecord(s->ev[0], st));
    if (mode == BVH) {
        if (int rc = ensure_bvh(s, st)) return rc;
    } else if (n_groups == 1) { // one group: its tables serve every sample; otherwise each group builds its own in turn
        if (int rc = build_eye_tables(0, n_views)) return rc;
    }
    CK_CUDA(cudaMemsetAsync(s->counters, 0, sizeof(sweep::Counters), st));
    CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int), st));

    if (cover_rows) { // the covering pass's planes
        const size_t n = hit_px();
        if (dev_grow(s->mt.cov_cap, n, s->mt.cov_best, s->mt.cov_tri, s->mt.cov_t, s->mt.cov_v) ||
            dev_grow(s->mt.cov_fid_cap, n * std::max(1, L), s->mt.cov_fid))
            return TRACER_ERR_NOMEM;
    }
    if (mode == CULL) { // candidate buffers: 24 per ray + slack (a few per ray are typical), sorted with a radix sort
        const size_t cap = hit_px() * 24 * (size_t)s->cull_grow + ((size_t)1 << 22);
        if (cap > s->cand_cap) {
            if (dev_grow(s->cand_cap, cap, s->cand_a, s->cand_b)) return TRACER_ERR_NOMEM;
            CK_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, s->sort_bytes, s->cand_a, s->cand_b, cap, 0, 64, st));
        }
        if (dev_grow(s->count_cap, 1, s->cand_count) || dev_grow(s->sort_cap, s->sort_bytes, s->sort_tmp)) return TRACER_ERR_NOMEM;
    }
    // shadow rays ordered by a radix sort of (key, pixel) pairs (order_shadow_rays)
    if (mode != BVH) {
        if ((size_t)n_px > s->rkey_cap) {
            if (dev_grow(s->rkey_cap, (size_t)n_px, s->rkey, s->rkey_sorted, s->iota)) return TRACER_ERR_NOMEM;
            CK_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, s->pair_bytes, s->rkey, s->rkey_sorted, s->iota, s->ws.list, n_px, 0, 64, st));
            trk::iota_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(s->iota, n_px);
            CK_CUDA(cudaGetLastError());
        }
        if (dev_grow(s->pair_cap, s->pair_bytes, s->pair_tmp)) return TRACER_ERR_NOMEM;
    }
    // test knob: pretend the bundle-cull candidate buffer holds only this many pairs (exercises the overflow fallback)
    const char *cand_env = std::getenv("TRACER_CAND_CAP");
    em_cap = cand_env ? std::min<unsigned long long>((unsigned long long)std::atoll(cand_env), s->cand_cap) : (unsigned long long)s->cand_cap;
    while (((int64_t)1 << tri_bits) < s->n_pad) ++tri_bits;
    if (S > 1 && !s->ws.accum_total && dev_alloc(&s->ws.accum_total, 3 * (size_t)s->ws.npx)) return TRACER_ERR_NOMEM;
    px = s->ws.px();
    // BVH mode: the tree's dilation m (bvh.cuh frame_margin) from the largest |coordinate| of the tree and the eye, with
    // the reach bound diag of the primary rays' hit points, (k+1) diag for light k
    bvh_ext = s->bvh_ext; // (every view's eye: the tree serves them all)
    for (int v = 0; v < n_views; ++v)
        for (int c = 0; c < 3; ++c) bvh_ext = std::max(bvh_ext, (double)std::fabs(cams[v].origin[c]));
    return 0;
}

// eye tables: views [v0, v1) into slots 0 .. v1 - v0, on the image plane: d'(s,t) = (llc - origin) + s*horizontal +
// t*vertical (camera.h:31-34)
int Frame::build_eye_tables(int v0, int v1) {
    for (int v = v0; v < v1; ++v) {
        const tracer_camera *cv = &cams[v];
        trk::TableParam tp{};
        for (int c = 0; c < 3; ++c) {
            tp.o[c] = cv->origin[c], tp.U[c] = cv->horizontal[c], tp.V[c] = cv->vertical[c];
            tp.W[c] = (double)cv->lower_left_corner[c] - (double)cv->origin[c];
        }
        for (int corner = 0; corner < 4; ++corner) { // |d'| is convex in (s,t): its maximum is at a corner
            double n2 = 0;
            for (int c = 0; c < 3; ++c) {
                const double x = tp.W[c] + (corner & 1) * tp.U[c] + (corner >> 1) * tp.V[c];
                n2 += x * x;
            }
            tp.dmax = std::max(tp.dmax, std::sqrt(n2));
        }
        tp.lmax = 0.0;
        if (int rc = build_table(s, tp, s->eye_table + (size_t)(v - v0) * s->table_stride, s->eye_span + (size_t)(v - v0) * s->span_stride, st))
            return rc;
        ++launches;
    }
    return 0;
}

// ---- primary: raygen + closest hit -> hit_tri, hit_t, hit_v -------------------------------------------------------------
// The call's own pixels into the workspace, or a seeded crop's covering rows (the whole frame's first cover_rows PPM rows,
// full width) into their own planes
HitPass Frame::hit_pass() const {
    if (!cover_rows) return {bands, views, n_rows, s->ws.best, s->ws.hit_tri, s->ws.hit_t, s->ws.hit_v};
    trk::Bands b = bands;
    b.crop_x = 0, b.crop_w = W, b.crop_y = 0, b.n_px = (int)hit_px();
    return {b, trk::Views{s->cams, b.n_px}, cover_rows, s->mt.cov_best, s->mt.cov_tri, s->mt.cov_t, s->mt.cov_v};
}

int Frame::closest_hit() {
    const HitPass hp = hit_pass();
    const int n = hp.bands.n_px;
    CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int), st));
    CK_CUDA(cudaMemsetAsync(hp.best, 0xff, sizeof(unsigned long long) * (size_t)n, st));
    CK_CUDA(cudaEventRecord(s->ev[1], st));
    if (int rc = mode == BVH ? primary_bvh(hp) : mode == CULL ? primary_cull(hp) : primary_sweeps(hp)) return rc;
    trk::resolve_primary_kernel<<<(n + 255) / 256, 256, 0, st>>>(hp.views, hp.bands, hp.best, s->tri_verts, s->n_tris, s->spheres,
                                                                 s->n_spheres, hp.hit_tri, hp.hit_t, hp.hit_v);
    CK_CUDA(cudaGetLastError());
    ++launches;
    CK_CUDA(cudaEventRecord(s->ev[2], st));
    return 0;
}

int Frame::primary_bvh(const HitPass &hp) {
    bvh::primary_kernel<<<(hp.bands.n_px + 127) / 128, 128, 0, st>>>(hp.views, hp.bands, s->bvh_tree, bvh::frame_margin(bvh_ext, diag),
                                                                      s->tri_verts, hp.best, s->counters);
    CK_CUDA(cudaGetLastError());
    ++launches;
    return 0;
}

// OPTIONAL bundle-cull mode: screen tiles of 128 x 32 pixels -> candidates -> sort -> strict
int Frame::primary_cull(const HitPass &hp) {
    trk::PrimaryCullParams p{};
    const int c_tiles = s->n_pad / cull::CTILE;
    p.cam = h_cams[0], p.bands = hp.bands, p.table = s->eye_table, p.n_tiles = c_tiles, p.n_tris = s->n_tris, p.n_rows = hp.n_rows;
    p.tiles_x = (hp.bands.crop_w + 127) / 128, p.tiles_y = (hp.n_rows + 31) / 32;
    const int blocks = p.tiles_x * p.tiles_y;
    p.n_slices = blocks >= 12 * g.n_sms ? 1 : std::max(1, std::min((12 * g.n_sms + blocks - 1) / blocks, std::max(1, c_tiles / 8)));
    p.em = cull::Emitter{s->cand_a, s->cand_count, em_cap};
    p.counters = s->counters, p.work = s->work;
    long long n_keys = -1;
    if (two_phase) {
        if (dev_grow(s->boxes_cap, (size_t)blocks, s->boxes)) return TRACER_ERR_NOMEM;
        trk::primary_boxes_kernel<<<blocks, sweep::THREADS, 0, st>>>(p, s->boxes, s->blk_off);
        CK_CUDA(cudaGetLastError());
        cull::L0Params lp{};
        lp.tables = s->eye_table, lp.n_groups = 1, lp.nface = 0, lp.blk_off = s->blk_off;
        if (int rc = block_lists(lp, blocks, n_keys)) return rc;
    }
    if (n_keys >= 0) {
        trk::primary_cull2_kernel<<<2 * g.n_sms, sweep::THREADS, 0, st>>>(p, trk::BlockLists{s->boxes, s->cand_b, (unsigned long long)n_keys, tri_bits});
        CK_CUDA(cudaGetLastError());
        host_tests_primary += (int64_t)hp.bands.n_px * s->n_tris;
    } else {
        CK_CUDA(cudaMemsetAsync(s->cand_count, 0, sizeof(unsigned long long), st));
        const size_t smem = sizeof(cull::EmitSmem);
        CK_CUDA(cudaFuncSetAttribute(trk::primary_cull_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        trk::primary_cull_kernel<<<std::min(blocks * p.n_slices, 2 * g.n_sms), sweep::THREADS, smem, st>>>(p);
        CK_CUDA(cudaGetLastError());
    }
    trk::strict_primary_pairs<<<8 * g.n_sms, 256, 0, st>>>(s->cand_a, s->cand_count, em_cap, h_cams[0], hp.bands, s->tri_verts, hp.best,
                                                           s->counters);
    CK_CUDA(cudaGetLastError());
    launches += 2;
    return 0;
}

// Default mode: one primary_kernel launch per group of views (all of them unless their eye tables did not fit at once)
int Frame::primary_sweeps(const HitPass &hp) {
    const int n_tiles = s->n_pad / sweep::TILE, row_w = hp.bands.crop_w;
    // no jitter: the rays of a thread share q exactly; jittered samples (extension): they share a mean q (span table)
    // unless the frame is so small that a jittered (s,t) can leave the span rows' |p|,|q| <= 1.0625 range
    const int qmode = bands.spp_n <= 1 ? sweep::MODE_SHAREDQ : (W >= 16 && H >= 16 ? sweep::MODE_QBAR : sweep::MODE_OWNQ);
    for (int v0 = 0; v0 < n_views; v0 += group) {
        const int nv = std::min(group, n_views - v0);
        if (n_groups > 1) {
            if (int rc = build_eye_tables(v0, v0 + nv)) return rc;
            if (v0 > 0) CK_CUDA(cudaMemsetAsync(s->work, 0, sizeof(int), st));
        }
        const Decomp d = pick_decomp((int64_t)nv * hp.views.view_px, n_tiles, g.n_sms, o.rays_per_thread, qmode);
        trk::PrimaryParams p{};
        p.views = hp.views, p.cam = h_cams[v0], p.bands = hp.bands, p.n_tiles = n_tiles, p.n_tris = s->n_tris;
        p.table = qmode == sweep::MODE_OWNQ ? s->eye_table : s->eye_span;
        p.table_stride = (long long)(qmode == sweep::MODE_OWNQ ? s->table_stride : s->span_stride), p.view0 = v0;
        p.tri_verts = s->tri_verts;
        p.best = hp.best, p.counters = s->counters, p.work = s->work;
        p.n_rows = hp.n_rows, p.view_blocks = 0; // ray blocks = screen tiles of (TX R) x (NT / TX) pixels: least edge waste wins
        for (int lg = d.R > 32 ? 2 : 3; lg <= 6; ++lg) { // (64 rays per thread: from 4 x 64 = 256 pixels wide)
            const int tw = (1 << lg) * d.R, th = sweep::NT >> lg;
            const int tx = (row_w + tw - 1) / tw, nb = tx * ((hp.n_rows + th - 1) / th);
            if (!p.view_blocks || nb < p.view_blocks) p.view_blocks = nb, p.tiles_x = tx, p.tx_log2 = lg;
        }
        p.n_blocks = nv * p.view_blocks;
        p.n_slices = d.n_slices;
        const int minb = trk::primary_minb(d.R);
        const int want_items = items_per_cta() * minb * g.n_sms;
        if (p.n_blocks < want_items) // same sizing rule as pick_decomp, on the real block count
            p.n_slices = std::max(1, std::min((want_items + p.n_blocks - 1) / p.n_blocks, std::max(1, n_tiles / 4)));
        const int grid = std::min(p.n_blocks * p.n_slices, minb * g.n_sms);
        // executed FP32 flops per pair: hot form half a packed FADD2 per pair (the three-input mins are no flops), and
        // per thread and triangle 4 FFMA for the bounds + the 2 FADD of nc2 and h2 (10 flops; 8 more FFMA-flops with a
        // mean q); three-row form with every ray its own q: 6 FFMA.SAT + FMUL + FFMA
        // shared q: per thread and triangle the set-up's 10 flops and one FADD2 (segment_pass), nothing per pair
        flop_primary = qmode == sweep::MODE_OWNQ ? 15.0 : qmode == sweep::MODE_QBAR ? 1.0 + 18.0 / d.R : 12.0 / d.R;
        flop_primary_edges = qmode == sweep::MODE_OWNQ ? 12.0 : (qmode == sweep::MODE_QBAR ? 16.0 : 8.0) / d.R;
        if (int rc = launch_primary(d.R, o.exhaustive_strict != 0, qmode, p, nv > 1, grid, st)) return rc;
        ++launches;
    }
    return 0;
}

// two-phase bundle cull (cull.cuh "block lists"): phase A emits block<<32|triangle into cand_a; the sorted
// keys land in cand_b, which phase B reads while it emits its ray<<32|triangle candidates into cand_a again.
// n_keys = the number of keys, or -1 when the survivor lists would not fit (then the streaming kernels run).
int Frame::block_lists(cull::L0Params lp, int max_blocks, long long &n_keys) {
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
}

// ---- faceIDs (first sample): the caller's (TRACER_RNG_EXPLICIT) or the seeded draws' (TRACER_RNG_MT19937) --------------
int Frame::faceids(std::vector<int> &frame_rows, bool &rows_known) {
    if (L > 0 && o.rng_mode == TRACER_RNG_EXPLICIT) {
        std::vector<int> loc((size_t)n_px * L);
        for (int k = 0; k < n_px; ++k) { // view v's faceids: opts->faceid[v][W*H*L], image index order
            int w, h;
            const int v = k / view_px;
            bands.map(k - v * view_px, w, h);
            std::memcpy(&loc[(size_t)k * L], o.faceid + ((size_t)v * H * W + (size_t)h * W + w) * L, sizeof(int) * L);
        }
        CK_CUDA(cudaMemcpyAsync(s->ws.faceid, loc.data(), loc.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        CK_CUDA(cudaStreamSynchronize(st));
    } else if (o.rng_mode == TRACER_RNG_MT19937) {
        // a bundle-cull closest-hit pass whose candidates overflowed has lost hits: its row counts must not be used or sent,
        // so the frame is rendered again before the exchange (read back with the row counts, at the same synchronise)
        unsigned long long primary_overflow = 0;
        if (mode == CULL) CK_CUDA(cudaMemcpyAsync(&primary_overflow, &s->counters->cull_overflow, sizeof primary_overflow, cudaMemcpyDeviceToHost, st));
        // the row hits of every view in one pass (view-major rows), then each view replays its own std::mt19937(seed) draws,
        // as a separate render of that view would.  A crop window: those of its covering rows (full-width rows from PPM row 0,
        // the prefix of a whole frame), then its own pixels' hits and faceIDs are gathered from them.
        const HitPass hp = hit_pass();
        const int rows = hp.n_rows, vpx = hp.views.view_px;
        int *const fid = cover_rows ? s->mt.cov_fid : s->ws.faceid;
        std::vector<int> all_rows;
        if (int rc = mt_count_rows(s->mt, hp.hit_tri, W, n_views * rows, st, all_rows)) return rc;
        ++launches;
        if (primary_overflow) return CAND_OVERFLOW;
        for (int v = 0; v < n_views; ++v) {
            const std::vector<int> local(all_rows.begin() + (size_t)v * rows, all_rows.begin() + (size_t)(v + 1) * rows);
            if (rows_known) {
                if (!mt::rows_valid(local.data(), rows, bands.band_rows, bands.band_index, bands.band_count, frame_rows.data(), H, W))
                    return fail(TRACER_ERR_STATE, "bundle-cull re-render: the closest-hit pass found other hits than the first pass");
            } else if (int rc = mt_frame_rows(o, W, H, bands.band_rows, bands.band_count, local, frame_rows)) {
                return rc;
            }
            const size_t off = (size_t)v * vpx;
            if (int rc = mt_replay(s->mt, o.seed, s->h_light_F, frame_rows, W, bands.band_rows, bands.band_index, bands.band_count, rows,
                                   hp.hit_tri + off, fid + off * L, st, launches, off))
                return rc;
        }
        rows_known = true;
        if (cover_rows) {
            trk::crop_gather_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(bands, hp.hit_tri, hp.hit_t, hp.hit_v, fid, L, s->ws.hit_tri,
                                                                        s->ws.hit_t, s->ws.hit_v, s->ws.faceid);
            CK_CUDA(cudaGetLastError());
            ++launches;
        }
    }
    return 0;
}

// ---- light k: (finish k-1, set up k) -> group by light vertex -> first-occluder sweep; k = L only finishes L-1 --------------
int Frame::light(int k, uint32_t seed) {
    trk::LightStepParams lp{};
    lp.views = views, lp.bands = bands, lp.px = px;
    lp.li = trk::LightInfo{s->light_vbase, s->light_verts};
    lp.k = k, lp.L = L, lp.n_tris = s->n_tris;
    lp.tri_verts = s->tri_verts, lp.tri_normals = s->tri_normals, lp.tri_geom = s->tri_geom;
    lp.geom_has_normals = s->geom_has_normals, lp.geom_material = s->geom_material;
    lp.sphere_material = s->sphere_material, lp.spheres = s->spheres;
    lp.rng_mode = o.rng_mode, lp.seed = seed, lp.faceid = s->ws.faceid, lp.lmax = (k + 1) * diag;
    lp.seg_count = s->seg_count, lp.counters = s->counters;
    lp.dbg_occ = o.out_occ_tri ? s->ws.dbg_occ : nullptr;
    lp.cull_cells = mode, lp.rkey = s->rkey;
    if (k < L) CK_CUDA(cudaMemsetAsync(s->seg_count, 0, sizeof(int) * ((size_t)s->maxF * trk::NFACE + 1), st));
    trk::light_step_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(lp);
    CK_CUDA(cudaGetLastError());
    ++launches;
    if (k == L) return 0;
    if (int rc = mode == BVH ? shadow_bvh(k) : mode == CULL ? shadow_cull(k) : shadow_sweeps(k)) return rc;
    CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k + 1], st));
    return 0;
}

// The shadow rays of one light in list order, grouped by ray group (light vertex, cube face): seg_off = where each group
// starts, cursor = its count, best_occ = no occluder yet.  Keys (light_step_kernel): default mode (group, q), so that the rays
// of a thread can share a q-term (sweep::MODE_QBAR); bundle-cull mode (group, Morton code of (p,q)).  Pixels without a
// shadow ray carry the all-ones key and sort last.  Default mode then cuts each group's q-sorted run into stripes of about
// sqrt(128 n) entries (n: the group's rays; SHADOW_CELL_C) and sorts every stripe by p, serpentine (stripe_key_kernel): a
// thread's SHADOW_R consecutive entries form a compact cell in (p, q).
// TRACER_SHADOW_STRIPE (development) sets one stripe length for every group; 1 gives the plain (group, q) order.
int Frame::order_shadow_rays(int F) {
    trk::list_prefix_kernel<<<1, 32, 0, st>>>(s->seg_count, F, s->seg_off, s->cursor);
    CK_CUDA(cudaGetLastError());
    int group_bits = 1;
    while ((1 << group_bits) < F) ++group_bits;
    int *first = mode == SWEEPS ? s->ws.list_b : s->ws.list;
    CK_CUDA(cub::DeviceRadixSort::SortPairs(s->pair_tmp, s->pair_bytes, s->rkey, s->rkey_sorted, s->iota, first, n_px, 0,
                                            32 + group_bits + 1, st));
    if (mode == SWEEPS) {
        const char *e = std::getenv("TRACER_SHADOW_STRIPE");
        const int len = e ? std::max(1, std::atoi(e)) : 0; // 0: each group's own stripe length
        trk::stripe_key_kernel<<<(n_px + 255) / 256, 256, 0, st>>>(s->rkey_sorted, first, s->ws.re, s->seg_off, n_px, len, s->rkey);
        CK_CUDA(cudaGetLastError());
        int pos_bits = 1;
        while (((int64_t)1 << pos_bits) < n_px) ++pos_bits;
        CK_CUDA(cub::DeviceRadixSort::SortPairs(s->pair_tmp, s->pair_bytes, s->rkey, s->rkey_sorted, first, s->ws.list, n_px, 0,
                                                32 + pos_bits, st));
        launches += 2;
    }
    CK_CUDA(cudaMemcpyAsync(s->cursor, s->seg_count, sizeof(int) * F, cudaMemcpyDeviceToDevice, st));
    CK_CUDA(cudaMemsetAsync(s->ws.best_occ, 0xff, sizeof(unsigned long long) * (size_t)n_px, st));
    return 0;
}

// one thread per pixel: first occluder through the tree, then the spheres
int Frame::shadow_bvh(int k) {
    CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k], st));
    bvh::shadow_kernel<<<(n_px + 127) / 128, 128, 0, st>>>(s->bvh_tree, px, n_px, bvh::frame_margin(bvh_ext, (k + 1) * diag), s->tri_verts,
                                                            s->spheres, s->n_spheres, s->n_tris, s->counters);
    CK_CUDA(cudaGetLastError());
    ++launches;
    return 0;
}

// OPTIONAL bundle-cull mode: rays sorted by (group, Morton code of (p,q)), one culled sweep over all triangles per light
int Frame::shadow_cull(int k) {
    const int F = s->h_light_F[k] * trk::NFACE; // ray groups: (light vertex, cube face)
    const int rpb = sweep::THREADS * 8;
    if (int rc = order_shadow_rays(F)) return rc;
    trk::chunk_prefix_kernel<<<1, 32, 0, st>>>(s->seg_count, F, rpb, s->n_pad / cull::CTILE, 2 * g.n_sms, s->blk_off, s->cnt_b, s->work,
                                               s->n_slices, 24, 16);
    CK_CUDA(cudaGetLastError());
    std::vector<int> gcnt((size_t)F);
    CK_CUDA(cudaMemcpyAsync(gcnt.data(), s->cursor, sizeof(int) * F, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k], st));
    for (int gi = 0; gi < F; ++gi) { // the tables of the groups that have rays
        if (!gcnt[gi]) continue;
        const int face = gi % trk::NFACE, vtx = s->h_light_vbase[k] + gi / trk::NFACE;
        if (int rc = face == trk::NFACE - 1 ? ensure_allcand_table(s, st, launches) : build_face_table(s, vtx, face, vtx, (k + 1) * diag, st, launches))
            return rc;
    }
    trk::ShadowCullParams sp{};
    sp.tables = s->light_tables + (size_t)s->h_light_vbase[k] * 6 * s->table_stride, sp.table_stride = s->table_stride;
    sp.allcand = s->allcand_table, sp.n_tiles = s->n_pad / cull::CTILE, sp.n_tris = s->n_tris, sp.n_groups = F, sp.n_px = n_px;
    sp.cells_per_group = 0, sp.n_slices = s->n_slices;
    sp.list = s->ws.list, sp.seg_off = s->seg_off, sp.seg_cnt = s->cursor, sp.blk_off = s->blk_off, sp.px = px;
    sp.counters = s->counters, sp.work = s->work;
    sp.em = cull::Emitter{s->cand_a, s->cand_count, em_cap};
    long long n_keys = -1;
    if (two_phase) {
        const int max_blocks = n_px / rpb + F + 1;
        if (dev_grow(s->boxes_cap, (size_t)max_blocks, s->boxes)) return TRACER_ERR_NOMEM;
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
    trk::strict_shadow_pairs<<<8 * g.n_sms, 256, 0, st>>>(s->cand_a, s->cand_count, em_cap, px, n_px, s->tri_verts, s->counters);
    CK_CUDA(cudaGetLastError());
    launches += 4;
    if (s->n_spheres > 0) {
        const dim3 sgrid((unsigned)std::min(1024, (n_px + 255) / 256), (unsigned)F);
        trk::shadow_spheres_kernel<<<sgrid, 256, 0, st>>>(s->ws.list, s->seg_off, s->cursor, F, px, n_px, s->spheres, s->n_spheres, s->n_tris);
        CK_CUDA(cudaGetLastError());
        ++launches;
    }
    return 0;
}

// Triangle chunks of the default shadow sweep: after each one the still-unoccluded rays are compacted (early exit,
// main.cpp:324).  Equal chunks keep the pairs swept past a ray's occluder lowest (x1.056 at 64 chunks; x1.11 at 32) and win
// when a light has many shadow rays.  8 of them: since flagged triangles are rebuilt with each ray's own q, a chunk's grid
// barriers and tail cost more than the pairs swept past occluders that more chunks would save (C4: 142 ms of shadow sweep
// at 8 chunks, 146 at 10 and 12, 153 at 6, 170 with 32 chunks and the earlier run cap; profiles/r12_e).  With few rays (small frames, one band
// share of a multi-GPU frame) a chunk's fixed cost (three grid barriers, the compaction passes, the sweep's tail: ~0.1 ms)
// weighs more, and 20 chunks that start fine (1/64 of the triangles: most occluded rays find their occluder early) and
// coarsen win (x1.10).  The kernel picks the scheme from the live-ray count it finds.  opts.shadow_chunks asks for that many
// equal chunks.
void chunk_schemes(trk::ShadowLightParams &sp, int n_tiles, int shadow_chunks) {
    const int nc = std::min({n_tiles, trk::SL_MAXCHUNK, shadow_chunks > 0 ? shadow_chunks : std::max(1, std::min(8, n_tiles / 8))});
    sp.n_chunks[1] = nc;
    for (int c = 0; c <= nc; ++c) sp.bounds[1][c] = (int)((int64_t)n_tiles * c / nc);
    if (shadow_chunks > 0 || n_tiles < 64) {
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

// ---- default mode: q-sorted lists, then ONE persistent cooperative kernel per batch of light vertices ----
int Frame::shadow_sweeps(int k) {
    const int F = s->h_light_F[k] * trk::NFACE, n_tiles = s->n_pad / sweep::TILE; // ray groups: (light vertex, cube face)
    if (int rc = order_shadow_rays(F)) return rc;
    launches += 2;
    if (dev_grow(s->blk_cnt_cap, (size_t)n_px / trk::CBLK + (size_t)F + 2, s->blk_cnt)) return TRACER_ERR_NOMEM;
    CK_CUDA(cudaEventRecord(s->ev_shadow[2 * k], st));
    if (int rc = ensure_allcand_table(s, st, launches)) return rc;
    trk::ShadowLightParams sp{};
    chunk_schemes(sp, n_tiles, o.shadow_chunks);
    sp.many_rays = (long long)1 << 20;
    sp.items_per_cta = items_per_cta();
    // run cap and smallest slice measured together with the chunk count at C4 (profiles/r12_e): 24 M pairs and 4 tiles at
    // 8 chunks; 6 M and 1 tile (the values for 32 chunks) cost 16 ms more
    sp.run_pairs = std::getenv("TRACER_RUN_PAIRS") ? std::max(1ll, std::atoll(std::getenv("TRACER_RUN_PAIRS"))) : 24000000ll;
    sp.min_tiles = std::getenv("TRACER_MIN_TILES") ? std::max(1, std::atoi(std::getenv("TRACER_MIN_TILES"))) : 4;
    sp.allcand = s->allcand_span, sp.table_stride = s->span_stride; // the default sweeps read the span tables
    sp.n_tris = s->n_tris, sp.n_tiles = n_tiles, sp.n_px = n_px, sp.tri_verts = s->tri_verts;
    sp.list[0] = s->ws.list, sp.list[1] = s->ws.list_b;
    sp.blk_cnt = s->blk_cnt, sp.px = px, sp.spheres = s->spheres, sp.n_spheres = s->n_spheres;
    sp.counters = s->counters;
    // light vertices in batches: as many as have table slots (all of them unless the light is a big mesh)
    const int Fk = s->h_light_F[k], vb = s->h_light_vbase[k];
    for (int b0 = 0; b0 < Fk; b0 += s->table_slots) {
        const int b1 = std::min(Fk, b0 + s->table_slots);
        for (int v = b0; v < b1; ++v)
            for (int face = 0; face < 6; ++face)
                if (int rc = build_face_table(s, vb + v, face, s->tables_resident ? vb + v : v - b0, (k + 1) * diag, st, launches)) return rc;
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
    return 0;
}

// S > 1: sum the samples in a fixed order; the last pass divides by S
int Frame::accumulate(int smp) {
    const size_t n3 = 3 * (size_t)n_px;
    trk::accumulate_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(s->ws.accum, s->ws.accum_total, n3, smp == 0, smp == S - 1, (float)S);
    CK_CUDA(cudaGetLastError());
    ++launches;
    CK_CUDA(cudaStreamSynchronize(st));
    add_sample_times();
    return 0;
}

// The event times of the sample just rendered (after a synchronise): its closest-hit pass and its shadow sweeps
void Frame::add_sample_times() {
    float ms = 0;
    cudaEventElapsedTime(&ms, s->ev[1], s->ev[2]);
    ms_primary += ms;
    for (int k = 0; k < L; ++k) {
        cudaEventElapsedTime(&ms, s->ev_shadow[2 * k], s->ev_shadow[2 * k + 1]);
        ms_shadow += ms;
    }
}

// ---- quantise + pack, read-backs, stats --------------------------------------------------------------------------------
int Frame::finish_frame(uint8_t *rgb_out) {
    uint8_t *dst8 = o.rgb_out_is_device ? rgb_out : s->ws.rgb8;
    const float *final_accum = S > 1 ? s->ws.accum_total : s->ws.accum;
    trk::quantise_kernel<<<((n_px + 15) / 16 + 127) / 128, 128, 0, st>>>(final_accum, n_px, dst8);
    CK_CUDA(cudaGetLastError());
    ++launches;
    CK_CUDA(cudaEventRecord(s->ev[3], st));
    if (!o.rgb_out_is_device) CK_CUDA(cudaMemcpyAsync(rgb_out, s->ws.rgb8, (size_t)n_px * 3, cudaMemcpyDeviceToHost, st));
    // optional debug read-backs
    if (o.out_tri) CK_CUDA(cudaMemcpyAsync(o.out_tri, s->ws.hit_tri, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_t) CK_CUDA(cudaMemcpyAsync(o.out_t, s->ws.hit_t, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_v) CK_CUDA(cudaMemcpyAsync(o.out_v, s->ws.hit_v, (size_t)n_px * 4, cudaMemcpyDeviceToHost, st));
    if (o.out_occ_tri && L > 0)
        CK_CUDA(cudaMemcpyAsync(o.out_occ_tri, s->ws.dbg_occ, (size_t)n_px * L * 4, cudaMemcpyDeviceToHost, st));
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
    if (S == 1) add_sample_times();
    s->stats.ms_primary = ms_primary;
    s->stats.ms_shadow = ms_shadow;
    s->stats.ms_other = s->stats.ms_total - s->stats.ms_primary - ms_shadow;
    s->stats.n_primary_rays = (int64_t)hit_px() * S;
    s->stats.n_shadow_rays = (int64_t)hc.n_hits * L;
    s->stats.tests_primary = (int64_t)hc.tests_primary + host_tests_primary;
    s->stats.tests_shadow = (int64_t)hc.tests_shadow + host_tests_shadow;
    s->stats.tests_shadow_ref = (int64_t)hc.tests_shadow_ref;
    s->stats.strict_evals = (int64_t)hc.strict_evals;
    s->stats.filter_misses = (int64_t)hc.filter_misses;
    s->stats.pipeline_errors = (int64_t)hc.pipeline_errors;
    s->stats.kernel_launches = launches;
    // FP32 flops the sweeps' formulation needs per swept pair (FFMA = 2, FADD = FMUL = 1, a minimum 0).  Shadow sweeps: the
    // segment verdict, per thread and triangle 8 bound FFMAs (mean q + |B| * spread), 2 FADD for the interval and one packed
    // FADD2 on the thread's extreme rays, over the R rays; nothing per pair.
    const bool no_flops = mode != SWEEPS; // the optional modes: no fixed per-pair cost
    s->stats.flop_primary = no_flops ? 0.0 : flop_primary, s->stats.flop_shadow = no_flops ? 0.0 : 20.0 / trk::SHADOW_R;
    // of which multiply-adds that evaluate bounds (the rest is each pair's interval test and the per-triangle interval)
    s->stats.flop_primary_edges = no_flops ? 0.0 : flop_primary_edges;
    s->stats.flop_shadow_edges = no_flops ? 0.0 : 16.0 / trk::SHADOW_R;
    if (hc.cull_overflow) return CAND_OVERFLOW; // (with TRACER_RNG_MT19937 only the shadow sweeps' candidates can have overflowed by now)
    if (getenv("TRACER_SHADOW_DIAG") && hc.cyc_total)
        fprintf(stderr, "shadow diag: CTA cycles %.3e total = items %.1f %% + grid barriers %.1f %% + compaction %.1f %% + other %.1f %%; %llu items in %llu runs; "
                        "flagged (thread, triangle) %llu, queued pairs %llu, strict evals %llu; candidate path %.1f %% of item cycles; %d CTAs per SM\n",
                (double)hc.cyc_total, 100.0 * hc.cyc_items / hc.cyc_total, 100.0 * hc.cyc_barrier / hc.cyc_total, 100.0 * hc.cyc_compact / hc.cyc_total,
                100.0 * ((double)hc.cyc_total - hc.cyc_items - hc.cyc_barrier - hc.cyc_compact) / hc.cyc_total, hc.n_items, hc.n_runs,
                hc.n_flagged, hc.n_queued, hc.strict_evals, 100.0 * hc.cyc_cand / (sweep::NT / 32) / std::max(1.0, (double)hc.cyc_items), g.sl_ctas[0]);
    if (getenv("TRACER_CULL_DIAG"))
        fprintf(stderr, "cull diag (shadow): l0 survivors %llu, tiles with any %llu, fallback tiles %llu, l1 warp-passes %llu, item-tiles %llu\n", hc.cull_l0,
                hc.cull_tiles_any, hc.cull_tiles_fallback, hc.cull_l1, (unsigned long long)(hc.tests_shadow / 4096 / cull::CTILE));
    return TRACER_OK;
}

// Checks the call, then renders it: again after a bundle-cull candidate overflow, with a 4x larger candidate buffer while
// that fits comfortably, else by the default sweeps, which need no such buffer (same bytes out either way).  The stats are
// those of the last attempt.
int render_views(tracer_scene_dev *s, const tracer_camera *cams, int n_views, int32_t W, int32_t H, const tracer_render_opts *opts_in,
                 uint8_t *rgb_out) {
    if (!s || !cams || !rgb_out) return fail(TRACER_ERR_INVALID, "null argument");
    if (!s->ctx || !s->ctx->inited) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    Ctx &g = *s->ctx;
    t_pool = &g.pool;
    if (W < 2 || H < 2) return fail(TRACER_ERR_INVALID, "width and height must be >= 2 (the reference divides by W-1, H-1)");
    tracer_render_opts o = read_opts(opts_in);
    const bool crop = has_crop(o);
    if (crop && (o.crop_w < 1 || o.crop_h < 1 || o.crop_x < 0 || o.crop_y < 0 || (int64_t)o.crop_x + o.crop_w > W ||
                 (int64_t)o.crop_y + o.crop_h > H))
        return fail(TRACER_ERR_INVALID, "crop window (" + std::to_string(o.crop_x) + ", " + std::to_string(o.crop_y) + ") " +
                                            std::to_string(o.crop_w) + " x " + std::to_string(o.crop_h) + " is not inside the " +
                                            std::to_string(W) + " x " + std::to_string(H) + " frame");
    // per-pixel planes are indexed with int (3 planes of n_px floats): keep 3 * n_px below 2^31
    constexpr int64_t PX_LIMIT = (int64_t)700 * 1000 * 1000;
    if ((crop ? (int64_t)o.crop_w * o.crop_h : (int64_t)n_views * W * H) > PX_LIMIT)
        return fail(TRACER_ERR_INVALID, "frame too large (limit 7e8 pixels per call, over all views; render bands or fewer views)");
    if (crop && (int64_t)W * H >= ((int64_t)1 << 31)) // a crop pixel's image index h*W + w is an int
        return fail(TRACER_ERR_INVALID, "a crop window needs a frame of fewer than 2^31 pixels");
    if (crop && o.rng_mode == TRACER_RNG_MT19937 && (int64_t)W * (o.crop_y + o.crop_h) > PX_LIMIT)
        return fail(TRACER_ERR_INVALID, "seeded crop window too low in the frame: its covering rows (every PPM row down to its last, "
                                        "full width) exceed the limit of 7e8 pixels per call");
    // extension (parity unpinned): samples_per_pixel = n*n stratified jittered samples per pixel
    int spp_n = 1;
    if (o.samples_per_pixel > 1) {
        spp_n = (int)std::lround(std::sqrt((double)o.samples_per_pixel));
        if (spp_n * spp_n != o.samples_per_pixel || spp_n > 16)
            return fail(TRACER_ERR_INVALID, "samples_per_pixel must be a square number <= 256");
        if (o.rng_mode == TRACER_RNG_MT19937)
            return fail(TRACER_ERR_INVALID, "TRACER_RNG_MT19937 reproduces the 1-sample serial path only");
    }
    const int band_count = o.band_count <= 1 ? 1 : o.band_count;
    const int band_rows = band_count > 1 ? o.band_rows : H;
    if (band_count > 1 && (band_rows <= 0 || o.band_index < 0 || o.band_index >= band_count))
        return fail(TRACER_ERR_INVALID, "bad band selection");
    if (crop && band_count > 1) return fail(TRACER_ERR_INVALID, "a crop window does not combine with bands (band_count > 1)");
    if (o.rng_mode == TRACER_RNG_MT19937 && band_count > 1 && !o.row_hits_exchange)
        return fail(TRACER_ERR_INVALID, "TRACER_RNG_MT19937 with band_count > 1 needs opts->row_hits_exchange (the other bands' row hit counts)");
    if (o.rng_mode == TRACER_RNG_EXPLICIT && !o.faceid && s->n_lights > 0)
        return fail(TRACER_ERR_INVALID, "TRACER_RNG_EXPLICIT needs opts->faceid");
    if (o.rng_mode < 0 || o.rng_mode > 2) return fail(TRACER_ERR_INVALID, "bad rng_mode");
    if (o.accel < 0 || o.accel > 1) return fail(TRACER_ERR_INVALID, "bad accel (0 = sweeps, 1 = BVH)");
    if (o.accel == 1 && (o.bundle_cull != 0 || o.exhaustive_strict != 0))
        return fail(TRACER_ERR_INVALID, "accel = 1 (BVH) does not combine with bundle_cull or exhaustive_strict (a debug mode of the sweeps' filter)");
    const int band_index = band_count > 1 ? o.band_index : 0;
    const int n_rows = crop ? o.crop_h : tracer_band_row_count(H, band_rows, band_index, band_count);
    const int row_w = crop ? o.crop_w : W;
    const int view_px = n_rows * row_w, n_px = n_views * view_px;
    trk::Bands bands{W, H, band_rows, band_index, band_count, n_px};
    bands.spp_n = spp_n, bands.sample = 0, bands.seed = o.seed;
    bands.crop_x = crop ? o.crop_x : 0, bands.crop_w = row_w, bands.crop_y = crop ? o.crop_y : 0;
    const int cover_rows = crop && o.rng_mode == TRACER_RNG_MT19937 ? o.crop_y + o.crop_h : 0;
    const cudaStream_t st = o.cuda_stream ? (cudaStream_t)o.cuda_stream : g.stream;
    std::vector<int> frame_rows;
    bool rows_known = false;
    for (;;) {
        Frame f{s, g, o, cams, st, W, H, n_rows, view_px, n_px, n_views, s->n_lights, spp_n * spp_n, bands, cover_rows};
        const int rc = f.render(rgb_out, frame_rows, rows_known);
        if (rc != CAND_OVERFLOW) return rc;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t next_bytes = (f.hit_px() * 24 * (size_t)s->cull_grow * 4 + ((size_t)1 << 22)) * sizeof(unsigned long long) * 3;
        if (!std::getenv("TRACER_CAND_CAP") && s->cull_grow < 64 && next_bytes < free_b / 2 + s->cand_cap * 24)
            s->cull_grow *= 4;
        else
            o.bundle_cull = 0;
    }
}
}  // namespace

extern "C" {

int tracer_cuda_render_scene(tracer_scene_dev *s, const tracer_camera *cam, int32_t W, int32_t H,
                             const tracer_render_opts *opts_in, uint8_t *rgb_out) {
    return render_views(s, cam, 1, W, H, opts_in, rgb_out);
}

int tracer_cuda_render_views(tracer_scene_dev *s, const tracer_camera *cams, int32_t n_views, int32_t W, int32_t H,
                             const tracer_render_opts *opts_in, uint8_t *rgb_out) {
    if (n_views < 1) return fail(TRACER_ERR_INVALID, "n_views must be >= 1");
    if (!cams) return fail(TRACER_ERR_INVALID, "null cameras");
    const tracer_render_opts o = read_opts(opts_in);
    if (o.band_count > 1) return fail(TRACER_ERR_INVALID, "tracer_cuda_render_views renders whole views: band_count must be <= 1");
    if (o.bundle_cull != 0) return fail(TRACER_ERR_INVALID, "tracer_cuda_render_views does not combine with bundle_cull");
    if (has_crop(o)) return fail(TRACER_ERR_INVALID, "tracer_cuda_render_views renders whole views: no crop window");
    return render_views(s, cams, n_views, W, H, opts_in, rgb_out);
}
}  // extern "C"

namespace {
// ---- scene updates (tracer_cuda_scene_update) -----------------------------------------------------------------------------
// The checks of one replica that need no device: the struct, the triangle range, data for a count, normals
int update_check(const tracer_scene_dev *s, const tracer_scene_update *u) {
    if (!s || !u) return fail(TRACER_ERR_INVALID, "null argument");
    if (u->struct_size < sizeof(tracer_scene_update)) return fail(TRACER_ERR_INVALID, "tracer_scene_update.struct_size too small");
    if (!s->ctx || !s->ctx->inited) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    if (u->tri_first < 0 || u->tri_count < 0 || (int64_t)u->tri_first + u->tri_count > s->n_tris)
        return fail(TRACER_ERR_INVALID, "triangle range [" + std::to_string(u->tri_first) + ", +" + std::to_string(u->tri_count) +
                                            ") outside the scene's " + std::to_string(s->n_tris) + " triangles");
    if (u->tri_count > 0 && !u->tri_verts && !u->tri_normals) return fail(TRACER_ERR_INVALID, "tri_count > 0 needs tri_verts or tri_normals");
    if (u->tri_normals && !s->tri_normals) return fail(TRACER_ERR_INVALID, "tri_normals given for a scene created without normals");
    return 0;
}
// data_is_device: every pointer the update reads is device or managed memory of GPU `device`
int update_check_pointers(const tracer_scene_dev *s, const tracer_scene_update *u, int device) {
    if (!u->data_is_device) return 0;
    const struct {
        const void *p;
        bool read;
        const char *name;
    } args[] = {{u->tri_verts, u->tri_count > 0, "tri_verts"},          {u->tri_normals, u->tri_count > 0, "tri_normals"},
                {u->geom_material, s->n_geoms > 0, "geom_material"},    {u->sphere_cr, s->n_spheres > 0, "sphere_cr"},
                {u->sphere_material, s->n_spheres > 0, "sphere_material"}};
    for (const auto &a : args) {
        if (!a.p || !a.read) continue;
        cudaPointerAttributes at{};
        const cudaError_t e = cudaPointerGetAttributes(&at, a.p);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(TRACER_ERR_INVALID, std::string(a.name) + ": not a CUDA pointer (" + cudaGetErrorString(e) + ")");
        }
        if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != device)
            return fail(TRACER_ERR_INVALID, std::string(a.name) + ": data_is_device, but not device memory of GPU " + std::to_string(device));
    }
    return 0;
}
bool update_is_noop(const tracer_scene_update *u) {
    return u->tri_count == 0 && !u->tri_verts && !u->tri_normals && !u->geom_material && !u->sphere_cr && !u->sphere_material;
}

// The device work of a checked update on one replica, on stream st.  src_device: the GPU the data lives on, -1 = host.
// 1. copies; 2. the box (vertices or spheres changed); 3. the light vertices, compared bit for bit with the old ones;
// 4. resident shadow tables: a moved light vertex's six are dropped (table_lmax = -1, rebuilt lazily by the next render as
// on a fresh scene), every other built table gets rows [tri_first, +tri_count) again, from the TableParam it was built
// with; 5. the BVH is marked stale.  Ends with a synchronise of st.
int update_apply(tracer_scene_dev *s, const tracer_scene_update &u, int src_device, cudaStream_t st) {
    Ctx &g = *s->ctx;
    t_pool = &g.pool;
    CK_CUDA(cudaSetDevice(g.device));
    auto copy = [&](void *dst, const void *src, size_t bytes) -> int {
        if (!src || !bytes) return 0;
        if (src_device >= 0 && src_device != g.device) CK_CUDA(cudaMemcpyPeerAsync(dst, g.device, src, src_device, bytes, st));
        else CK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, st));
        return 0;
    };
    const size_t tri_bytes = (size_t)u.tri_count * 9 * sizeof(float), tri0 = 9 * (size_t)u.tri_first;
    const bool verts = u.tri_verts && u.tri_count > 0, spheres = u.sphere_cr && s->n_spheres > 0;
    int rc = copy(s->tri_verts + tri0, u.tri_verts, tri_bytes);
    if (!rc && u.tri_normals) rc = copy(s->tri_normals + tri0, u.tri_normals, tri_bytes);
    if (!rc) rc = copy(s->geom_material, u.geom_material, (size_t)s->n_geoms * 13 * sizeof(float));
    if (!rc) rc = copy(s->spheres, u.sphere_cr, (size_t)s->n_spheres * sizeof(float4));
    if (!rc) rc = copy(s->sphere_material, u.sphere_material, (size_t)s->n_spheres * 13 * sizeof(float));
    if (rc) return rc;
    if (verts || spheres) {
        if (int r = scene_bbox(s, st)) return r;
    }
    if (verts) {
        if (s->V > 0) { // light l's vertices are the first 3 F floats of its geometry's triangles
            for (int l = 0; l < s->n_lights; ++l)
                CK_CUDA(cudaMemcpyAsync(s->light_verts + 3 * (size_t)s->h_light_vbase[l], s->tri_verts + 9 * (size_t)s->h_light_t0[l],
                                        3 * (size_t)s->h_light_F[l] * sizeof(float), cudaMemcpyDeviceToDevice, st));
            const std::vector<float> old = s->h_light_verts;
            CK_CUDA(cudaMemcpyAsync(s->h_light_verts.data(), s->light_verts, old.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
            CK_CUDA(cudaStreamSynchronize(st));
            int launches = 0; // (an update keeps no launch count)
            for (int v = 0; s->tables_resident && v < s->V; ++v) {
                const bool moved = std::memcmp(&old[3 * (size_t)v], &s->h_light_verts[3 * (size_t)v], 3 * sizeof(float)) != 0;
                for (int face = 0; face < 6; ++face) {
                    double &built = s->table_lmax[(size_t)v * 6 + face];
                    if (built < 0) continue;
                    if (moved) {
                        built = -1.0;
                        continue;
                    }
                    if (int r = build_face_table(s, v, face, v, built, st, launches, u.tri_first, u.tri_count)) return r;
                }
            }
        }
        s->bvh_built = false; // rebuilt by the next BVH render (ensure_bvh)
    }
    CK_CUDA(cudaStreamSynchronize(st));
    return 0;
}
}  // namespace

extern "C" {

int tracer_cuda_last_stats(tracer_scene_dev *s, tracer_frame_stats *out) {
    if (!s || !out) return fail(TRACER_ERR_INVALID, "null argument");
    *out = s->stats;
    return TRACER_OK;
}

int tracer_cuda_scene_update(tracer_scene_dev *s, const tracer_scene_update *u) {
    if (int rc = update_check(s, u)) return rc;
    CK_CUDA(cudaSetDevice(s->ctx->device));
    if (int rc = update_check_pointers(s, u, s->ctx->device)) return rc;
    if (update_is_noop(u)) return TRACER_OK;
    return update_apply(s, *u, u->data_is_device ? s->ctx->device : -1, u->cuda_stream ? (cudaStream_t)u->cuda_stream : s->ctx->stream);
}

// Internal (tests only): the scene's bounding box as the render uses it, lo xyz then hi xyz
int tracer__scene_bbox(tracer_scene_dev *s, double *out6) {
    if (!s || !out6) return fail(TRACER_ERR_INVALID, "null argument");
    for (int c = 0; c < 3; ++c) out6[c] = s->bb_lo[c], out6[3 + c] = s->bb_hi[c];
    return TRACER_OK;
}

// Internal (measurement): (re)build the scene's BVH on its context's stream, timed with CUDA events around the build and
// a synchronise; *ms_out = the build's device time.  The next BVH render uses this tree.
int tracer__bvh_prepare(tracer_scene_dev *s, double *ms_out) {
    if (!s || !s->ctx || !s->ctx->inited) return fail(TRACER_ERR_INVALID, "null scene");
    t_pool = &s->ctx->pool;
    CK_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    s->bvh_built = false;
    CK_CUDA(cudaEventRecord(s->ev[0], st));
    if (int rc = ensure_bvh(s, st)) return rc;
    CK_CUDA(cudaEventRecord(s->ev[3], st));
    CK_CUDA(cudaEventSynchronize(s->ev[3]));
    float ms = 0.f;
    CK_CUDA(cudaEventElapsedTime(&ms, s->ev[0], s->ev[3]));
    if (ms_out) *ms_out = ms;
    return TRACER_OK;
}

// Internal (tests, measurement): the device replay of the seeded draws, on the current device, for one whole frame's hit
// mask in scan order (n_rows rows of W pixels).  faceid_scan [W*n_rows*L]: what tracer_mt19937_faceids gives, in scan
// order, -1 for misses.  *ms_out (may be NULL): CUDA events around the replay, from the per-row hit count to the gather.
int tracer__mt19937_faceids_device(uint32_t seed, int32_t L, const int32_t *faces, int32_t W, int32_t n_rows, const uint8_t *hit_scan,
                                   int32_t *faceid_scan, double *ms_out) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    if (L < 0 || W < 1 || n_rows < 1 || (int64_t)W * n_rows * std::max(L, 1) >= ((int64_t)1 << 31) || !hit_scan || !faceid_scan || (L && !faces))
        return fail(TRACER_ERR_INVALID, "bad argument");
    Ctx &g = *g_cur;
    t_pool = &g.pool;
    CK_CUDA(cudaSetDevice(g.device));
    cudaStream_t st = g.stream;
    const int n_px = W * n_rows;
    struct Bufs {
        MtWork m;
        int *tri = nullptr, *fid = nullptr;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        ~Bufs() {
            m.release(), dev_free(tri), dev_free(fid);
            for (cudaEvent_t e : ev)
                if (e) cudaEventDestroy(e);
        }
    } b;
    std::vector<int> tri((size_t)n_px);
    for (int k = 0; k < n_px; ++k) tri[k] = hit_scan[k] ? 0 : -1;
    if (dev_alloc(&b.tri, (size_t)n_px) || dev_alloc(&b.fid, (size_t)n_px * std::max(L, 1))) return TRACER_ERR_NOMEM;
    CK_CUDA(cudaEventCreate(&b.ev[0]));
    CK_CUDA(cudaEventCreate(&b.ev[1]));
    CK_CUDA(cudaMemcpyAsync(b.tri, tri.data(), sizeof(int) * (size_t)n_px, cudaMemcpyHostToDevice, st));
    CK_CUDA(cudaMemsetAsync(b.fid, 0xff, sizeof(int) * (size_t)n_px * std::max(L, 1), st));
    CK_CUDA(cudaEventRecord(b.ev[0], st));
    std::vector<int> local, frame;
    tracer_render_opts whole{};
    int launches = 0;
    if (int rc = mt_count_rows(b.m, b.tri, W, n_rows, st, local)) return rc;
    if (int rc = mt_frame_rows(whole, W, n_rows, n_rows, 1, local, frame)) return rc;
    if (int rc = mt_replay(b.m, seed, std::vector<int>(faces, faces + L), frame, W, n_rows, 0, 1, n_rows, b.tri, b.fid, st, launches))
        return rc;
    CK_CUDA(cudaEventRecord(b.ev[1], st));
    CK_CUDA(cudaMemcpyAsync(faceid_scan, b.fid, sizeof(int) * (size_t)n_px * L, cudaMemcpyDeviceToHost, st));
    CK_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    CK_CUDA(cudaEventElapsedTime(&ms, b.ev[0], b.ev[1]));
    if (ms_out) *ms_out = ms;
    return TRACER_OK;
}

// Internal (measurement): the replay's stream generator on its own, n words of std::mt19937(seed) on the current device;
// *ms_out = CUDA events around the one launch.
int tracer__mt19937_stream_device(uint32_t seed, int64_t n, double *ms_out) {
    if (!g_cur) return fail(TRACER_ERR_NO_DEVICE, "tracer_cuda_init not called");
    if (n < 1 || !ms_out) return fail(TRACER_ERR_INVALID, "bad argument");
    Ctx &g = *g_cur;
    t_pool = &g.pool;
    CK_CUDA(cudaSetDevice(g.device));
    cudaStream_t st = g.stream;
    struct Bufs {
        uint32_t *words = nullptr;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        ~Bufs() {
            dev_free(words);
            for (cudaEvent_t e : ev)
                if (e) cudaEventDestroy(e);
        }
    } b;
    if (dev_alloc(&b.words, (size_t)n)) return TRACER_ERR_NOMEM;
    CK_CUDA(cudaEventCreate(&b.ev[0]));
    CK_CUDA(cudaEventCreate(&b.ev[1]));
    CK_CUDA(cudaEventRecord(b.ev[0], st));
    mt::stream_kernel<<<1, mt::GEN_THREADS, 0, st>>>(seed, n, b.words);
    CK_CUDA(cudaGetLastError());
    CK_CUDA(cudaEventRecord(b.ev[1], st));
    CK_CUDA(cudaEventSynchronize(b.ev[1]));
    float ms = 0.f;
    CK_CUDA(cudaEventElapsedTime(&ms, b.ev[0], b.ev[1]));
    *ms_out = ms;
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

}  // extern "C"

namespace {
// TRACER_RNG_MT19937 on several GPUs: their row hit counts summed between their threads, a barrier and a shared [H]
// array.  A GPU whose render fails before the exchange arrives after it, with an error flag, so that no thread waits
// forever; every GPU's exchange then fails.
struct RowExchange {
    std::mutex mu;
    std::condition_variable cv;
    int n = 0, arrived = 0;
    bool error = false;
    std::vector<int> sum;
    bool arrive(int32_t *rows, int32_t H, bool failed) {
        std::unique_lock<std::mutex> lk(mu);
        if (failed) error = true;
        else {
            if ((int)sum.size() < H) sum.resize((size_t)H, 0);
            for (int r = 0; r < H; ++r) sum[r] += rows[r];
        }
        if (++arrived == n) cv.notify_all();
        else cv.wait(lk, [&] { return arrived == n; });
        if (error) return false;
        if (rows) std::copy(sum.begin(), sum.begin() + H, rows);
        return true;
    }
};
struct RowExchangeSeat {
    RowExchange *x = nullptr;
    bool arrived = false, peer_failed = false;
};
int32_t row_exchange_hook(void *user, int32_t H, int32_t *rows) {
    auto *seat = (RowExchangeSeat *)user;
    seat->arrived = true;
    if (seat->x->arrive(rows, H, false)) return 0;
    seat->peer_failed = true;
    return 1;
}
}  // namespace

extern "C" {

// Internal (tests only, no GPU needed): the multi-GPU call's row-count exchange between n threads.  Thread d offers
// rows_in[d*H ..] through the hook, or — fails[d] != 0 — arrives as a GPU whose render failed before the exchange does.
// rows_out[d*H ..] = what thread d's hook left in its array, rc_out[d] = the hook's return (-1 for a failed thread).
void tracer__row_exchange_host(int32_t n, int32_t H, const int32_t *rows_in, const uint8_t *fails, int32_t *rows_out, int32_t *rc_out) {
    RowExchange xchg;
    xchg.n = n;
    std::vector<RowExchangeSeat> seats((size_t)n);
    auto work = [&](int d) {
        int32_t *rows = rows_out + (size_t)d * H;
        std::copy(rows_in + (size_t)d * H, rows_in + (size_t)(d + 1) * H, rows);
        seats[d].x = &xchg;
        rc_out[d] = fails[d] ? -1 : row_exchange_hook(&seats[d], H, rows);
        if (!seats[d].arrived) xchg.arrive(nullptr, 0, true);
    };
    std::vector<std::thread> th;
    for (int d = 1; d < n; ++d) th.emplace_back(work, d);
    work(0);
    for (auto &t : th) t.join();
}

int tracer_cuda_render_scene_multi(tracer_scene_multi *ms, const tracer_camera *cam, int32_t W, int32_t H,
                                   const tracer_render_opts *opts_in, uint8_t *rgb_out) {
    if (!ms || !cam || !rgb_out) return fail(TRACER_ERR_INVALID, "null argument");
    const int n = (int)ms->dev.size();
    if (n != g_multi.n || n < 1) return fail(TRACER_ERR_STATE, "scene was created for a different GPU set");
    const tracer_render_opts o = read_opts(opts_in);
    if (has_crop(o)) return fail(TRACER_ERR_INVALID, "the multi-GPU call renders whole frames: use tracer_cuda_render_scene for a crop window");
    if (n == 1) {
        const int rc = tracer_cuda_render_scene(ms->dev[0], cam, W, H, opts_in, rgb_out);
        ms->stats = ms->dev[0]->stats;
        return rc;
    }
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
    if (dev_grow(g_multi.gathered_cap, pad_bytes * n + 64, g_multi.gathered) || dev_grow(g_multi.frame_cap, frame_bytes + 64, g_multi.frame))
        return TRACER_ERR_NOMEM;
    std::vector<int> rc((size_t)n, 0);
    std::vector<std::string> err((size_t)n);
    const bool mt = o.rng_mode == TRACER_RNG_MT19937;
    RowExchange xchg;
    xchg.n = n;
    std::vector<RowExchangeSeat> seats((size_t)n);
    auto render_on = [&](int d) {
        Ctx &g = g_ctx[d];
        uint8_t *dst = g_multi.gathered; // GPU 0
        if (d > 0) {
            if (cudaSetDevice(d) != cudaSuccess) { rc[d] = TRACER_ERR_CUDA, err[d] = "cudaSetDevice"; return; }
            t_pool = &g.pool;
            if (dev_grow(g_multi.band_cap[d], pad_bytes + 64, g_multi.band_buf[d])) { rc[d] = TRACER_ERR_NOMEM, err[d] = g_err; return; }
            dst = g_multi.band_buf[d];
        }
        tracer_render_opts od = o;
        od.struct_size = sizeof od;
        od.band_rows = band_rows, od.band_index = d, od.band_count = n;
        od.rgb_out_is_device = 1, od.cuda_stream = nullptr; // the GPU's own stream: the send below is queued behind the frame
        if (mt) seats[d].x = &xchg, od.row_hits_exchange = row_exchange_hook, od.row_hits_user = &seats[d];
        rc[d] = tracer_cuda_render_scene(ms->dev[d], cam, W, H, &od, dst);
        if (rc[d]) err[d] = g_err;
    };
    auto work = [&](int d) {
        render_on(d);
        if (mt && !seats[d].arrived) xchg.arrive(nullptr, 0, true); // failed before the exchange: release the others
    };
    std::vector<std::thread> th;
    for (int d = 1; d < n; ++d) th.emplace_back(work, d);
    work(0);
    for (auto &t : th) t.join();
    for (int pass = 0; pass < 2; ++pass) // the error of a GPU that failed on its own before the others' exchange failures
        for (int d = 0; d < n; ++d)
            if (rc[d] && (pass == 1 || !seats[d].peer_failed)) return fail(rc[d], "GPU " + std::to_string(d) + ": " + err[d]);
    // the band gather: packed bands -> GPU 0
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

// Every replica is checked before any changes; then they are updated one after the other.  Replica 0 goes first, on
// cuda_stream, and its update ends with a synchronise of that stream: device data produced on it is complete before the
// other replicas' peer copies from device 0 start on their own streams.
int tracer_cuda_scene_update_multi(tracer_scene_multi *ms, const tracer_scene_update *u) {
    if (!ms || !u) return fail(TRACER_ERR_INVALID, "null argument");
    const int n = (int)ms->dev.size();
    if (n != g_multi.n || n < 1) return fail(TRACER_ERR_STATE, "scene was created for a different GPU set");
    for (int d = 0; d < n; ++d)
        if (int rc = update_check(ms->dev[d], u)) return rc;
    CK_CUDA(cudaSetDevice(0));
    if (int rc = update_check_pointers(ms->dev[0], u, 0)) return rc;
    if (update_is_noop(u)) return TRACER_OK;
    for (int d = 0; d < n; ++d) {
        const cudaStream_t st = d == 0 && u->cuda_stream ? (cudaStream_t)u->cuda_stream : g_ctx[d].stream;
        if (int rc = update_apply(ms->dev[d], *u, u->data_is_device ? 0 : -1, st)) return fail(rc, "GPU " + std::to_string(d) + ": " + g_err);
    }
    return TRACER_OK;
}

int tracer_cuda_render_multi(const tracer_scene_flat *scene, const tracer_camera *cam, int32_t width, int32_t height,
                             const tracer_render_opts *opts, uint8_t *rgb_out) {
    if (has_crop(read_opts(opts)))
        return fail(TRACER_ERR_INVALID, "the multi-GPU call renders whole frames: use tracer_cuda_render_scene for a crop window");
    tracer_scene_multi *ms = nullptr;
    if (int rc = tracer_cuda_scene_create_multi(scene, &ms)) return rc;
    const int rc = tracer_cuda_render_scene_multi(ms, cam, width, height, opts, rgb_out);
    tracer_cuda_scene_destroy_multi(ms);
    return rc;
}

}  // extern "C"
