/* tracer_cuda.h — C ABI of the B200 (sm_100a) renderer for the per-pixel hot
 * path of pg42819/EscTp1RayTracer.
 *
 * Position in the reference: this library is called exactly where the
 * reference calls its ISPC accelerator,
 *     ispc::trace(W, H, ispc_cam, nTri, tris, nLights, lights, nLightFaces,
 *                 lightFaces, flat_image, debug, test)        src/main.cpp:619-624
 * (export declared at src/ispc/trace.ispc:86-92), after the scene has been
 * flattened to plain arrays (src/simplify/flatten_iscp.cpp:35-111) and the
 * camera marshalled (flatten_iscp.cpp:117-128).  It computes what the serial
 * path computes in scan_row (src/main.cpp:698-791) followed by the quantiser
 * of the PPM writer (src/main.cpp:679-684).
 *
 * Plain pointers and sizes only; no C++ or torch types.  All functions return
 * 0 on success or a negative tracer_status; the message is available from
 * tracer_cuda_last_error().  There is NO CPU fallback: without a CUDA device
 * (or without the sm_100a kernels) every compute entry point fails with
 * TRACER_ERR_NO_DEVICE / TRACER_ERR_CUDA.
 */
#ifndef TRACER_CUDA_H
#define TRACER_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRACER_CUDA_ABI_VERSION 1

typedef enum tracer_status {
    TRACER_OK = 0,
    TRACER_ERR_INVALID = -1,   /* bad argument (NULL, negative size, bad index) */
    TRACER_ERR_NO_DEVICE = -2, /* no CUDA device / tracer_cuda_init not called  */
    TRACER_ERR_CUDA = -3,      /* a CUDA runtime call or kernel failed          */
    TRACER_ERR_NOMEM = -4,
    TRACER_ERR_STATE = -5      /* handle destroyed / wrong call order           */
} tracer_status;

/* Flat scene, structure of arrays, HOST pointers, caller owned.
 * Replaces ispc_triangle[] / ispc_light[] (src/ispc/ispc_helpers.h:16-29,
 * 52-56) and tracer::scene (src/scene/scene.h:9-44).
 * Triangle order MUST be the reference's iteration order — geometry major,
 * face minor (src/main.cpp:179-180) — because ties keep the lower index
 * (ray_triangle.h:49) and occlusion() returns the first face in order
 * (src/main.cpp:317-325).  The reference's ISPC flatten sorts by centroid x
 * (flatten_iscp.cpp:110); do NOT sort for serial-path parity. */
typedef struct tracer_scene_flat {
    int32_t n_geoms;
    const int32_t *geom_tri_offset;  /* [n_geoms+1] first triangle of geometry g; last = n_tris */
    const float *tri_verts;          /* [n_tris*9]  v0 v1 v2 (de-indexed, sceneloader.cpp:78-82) */
    const float *tri_normals;        /* [n_tris*9]  per-corner normals, or NULL                  */
    const int32_t *geom_has_normals; /* [n_geoms]   (!normals.empty(), main.cpp:733) or NULL     */
    const float *geom_material;      /* [n_geoms*13] ka[3] kd[3] ks[3] ke[3] Ns (scene.h:11-18)  */
    int32_t n_lights;
    const int32_t *light_geom;       /* [n_lights]  geometry index, in light_sources order       */
    /* Extension with no reference behaviour (src/intersect.h is empty):
     * analytic spheres, tested after all triangles, object index n_tris+s. */
    int32_t n_spheres;
    const float *sphere_cr;          /* [n_spheres*4]  centre xyz, radius */
    const float *sphere_material;    /* [n_spheres*13] */
} tracer_scene_flat;

/* The four vectors tracer::camera precomputes (src/scene/camera.h:16-29);
 * replaces ispc_cam (ispc_helpers.h:59-65). */
typedef struct tracer_camera {
    float origin[3];
    float lower_left_corner[3];
    float horizontal[3];
    float vertical[3];
} tracer_camera;

/* Host helper: the reference camera constructor, same arithmetic
 * (camera.h:16-29; main.cpp:548-551 uses vfov=60, vup=(0,1,0), aspect=W/H). */
void tracer_camera_lookat(const float eye[3], const float look[3], const float vup[3], float vfov_deg,
                          float aspect, tracer_camera *out);

typedef enum tracer_rng_mode {
    /* counter-based hash of (seed, pixel, light): independent of GPU count and
     * of scan order.  Production default. */
    TRACER_RNG_HASH = 0,
    /* std::mt19937(seed) consumed exactly as scan_row does (main.cpp:743-754,
     * three draws per hit pixel per light, scan order h=H-1..0, w=0..W-1,
     * libstdc++ uniform_int_distribution): reproduces the seeded serial path.
     * The draws are replayed on the device.  A pixel's draws depend on the hits
     * of every earlier row of the frame, so a call that renders bands
     * (band_count > 1) needs opts->row_hits_exchange to learn the other rows'
     * hit counts; 1 sample per pixel only. */
    TRACER_RNG_MT19937 = 1,
    /* faceID per (pixel, light) supplied by the caller in opts->faceid. */
    TRACER_RNG_EXPLICIT = 2
} tracer_rng_mode;

typedef struct tracer_render_opts {
    uint32_t struct_size;  /* = sizeof(tracer_render_opts) */
    int32_t rng_mode;      /* tracer_rng_mode */
    uint32_t seed;
    const int32_t *faceid; /* HOST [W*H*n_lights], image index h*W+w; TRACER_RNG_EXPLICIT only */

    /* Row-band partition for multi-GPU (1 process per GPU).  The frame's PPM
     * rows (row 0 = h=H-1, main.cpp:662) are cut into bands of band_rows
     * rows; this call renders the bands b with b % band_count == band_index,
     * packed back to back in the output.  band_count<=1 renders everything (or, with crop_x .. crop_h at the end
     * of this struct, one rectangular window of the frame). */
    int32_t band_rows;
    int32_t band_index;
    int32_t band_count;

    int32_t rgb_out_is_device; /* rgb_out is a device pointer (stays in HBM, e.g. for an NCCL gather) */
    void *cuda_stream;         /* cudaStream_t to launch on; NULL = the library's own (non-blocking) stream.  To order the
                                  render with work on the legacy default stream pass cudaStreamLegacy (0x1), not 0 */

    int32_t exhaustive_strict; /* debug: bypass the conservative filter, strict-test every pair */
    int32_t samples_per_pixel; /* extension (parity unpinned): 0/1 = reference; n*n stratified jitter */
    int32_t rays_per_thread;   /* tuning: 0 = auto, else 2, 4, 8, 16, 24, 32 or 64 rays per thread in the closest-hit sweep
                                  (2, 4, 8 or 12 with jittered samples) */
    int32_t shadow_chunks;     /* tuning: 0 = auto; triangle chunks between shadow-ray compactions */
    int32_t bundle_cull;       /* OPTIONAL mode: hierarchical (bundle box -> warp box -> ray) evaluation of the same
                                  conservative filter; identical results.  1 = two-phase (dense block-box pass, then
                                  per-block survivor lists), 2 = single streaming sweep (also the fall-back of 1),
                                  3 = auto: two-phase unless the scene is so small that the default sweeps are faster */

    /* optional debug outputs, HOST pointers, indexed like the output rows
     * (local pixel k = local_row*W + w), any may be NULL */
    int32_t *out_tri;     /* closest-hit flat triangle index (n_tris+s for spheres), -1 miss */
    float *out_t;         /* closest-hit t */
    float *out_v;         /* closest-hit v */
    int32_t *out_occ_tri; /* [n_px*n_lights] first in-order occluder, -1 none, -2 no shadow ray */
    float *out_rgb;       /* [n_px*3] float accumulator before quantisation */

    int32_t accel;        /* OPTIONAL mode: 0 = the modes above; 1 = BVH: a linear BVH over the triangles (built on the
                             device on the first BVH render of a scene, kept until the scene is destroyed or an
                             update moves vertices, tracer_cuda_scene_update) with a
                             conservative traversal in front of the reference's own test; identical results.  Not
                             combinable with bundle_cull or exhaustive_strict (TRACER_ERR_INVALID); rays_per_thread and
                             shadow_chunks are ignored.  In this mode tests_primary / tests_shadow = strict_evals = the
                             triangle tests done at leaves, flop_* = 0, and the tree's build time is part of ms_other.
                             Appended last: callers with an older struct_size get 0. */

    /* TRACER_RNG_MT19937 with band_count > 1 only (required there, ignored otherwise): the frame's per-row hit counts.
     * The call invokes it exactly once, after its closest-hit pass, also when its band selection covers no row.  On
     * entry row_hits[r] (r = PPM row, 0 .. height-1) holds this call's hit count for every row it renders and 0
     * elsewhere; on return it must hold the counts of every row of the frame (each row has one owner, so an all-reduce
     * sum over the calls that render the frame does it) and return 0.  A non-zero return fails the render with
     * TRACER_ERR_STATE; this call's rows changed or a count outside [0, width] fails it with TRACER_ERR_INVALID.  The
     * scene stays usable either way.  A call that fails before its closest-hit pass ends does not invoke it.
     * Appended last: callers with an older struct_size get NULL. */
    int32_t (*row_hits_exchange)(void *user, int32_t height, int32_t *row_hits);
    void *row_hits_user;

    /* Crop window: render only columns [crop_x, crop_x + crop_w) of PPM rows [crop_y, crop_y + crop_h) (PPM row 0 =
     * h = H-1, as for bands).  The frame is still width x height: the camera, the image-plane (s, t), the faceID hash,
     * the jitter and the explicit faceid array (still [W*H*n_lights]) are those of the whole frame.  rgb_out holds
     * crop_h rows of crop_w pixels in PPM order, and the debug outputs are indexed k = local_row * crop_w + column.
     * Contract: every byte and debug value equals the same pixel of the whole frame rendered with the same options, in
     * every mode, rng_mode and sample count and with exhaustive_strict.  With TRACER_RNG_MT19937 a pixel's draws depend
     * on the hits of every pixel before it in scan order, so the call first runs the closest-hit pass over the covering
     * rows [0, crop_y + crop_h) at full width; tests_primary, strict_evals and n_primary_rays count that pass, n_pixels
     * counts the crop.  All four 0 = the whole frame.  Refused with TRACER_ERR_INVALID: a window not inside the frame,
     * crop_w < 1 or crop_h < 1 while any field is set, band_count > 1, tracer_cuda_render_views and the multi-GPU calls.
     * Appended last: callers with an older struct_size get 0. */
    int32_t crop_x, crop_y, crop_w, crop_h;
} tracer_render_opts;

typedef struct tracer_frame_stats {
    double ms_total;        /* CUDA events around all launches of the frame            */
    double ms_primary;      /* closest-hit sweep                                       */
    double ms_shadow;       /* any-hit sweeps, all lights                              */
    double ms_other;        /* table build, ray set-up, shading, quantise              */
    int64_t n_pixels;       /* pixels rendered by this call (a crop's)                 */
    int64_t n_primary_rays; /* (a seeded crop: those of its covering rows)             */
    int64_t n_shadow_rays;
    int64_t tests_primary;  /* ray-triangle pairs swept (filter evaluations), primary  */
    int64_t tests_shadow;   /* same, shadow sweeps                                     */
    int64_t tests_shadow_ref; /* sum over shadow rays of (first occluder index+1, else N): the reference's count */
    int64_t strict_evals;   /* pairs re-evaluated in reference arithmetic              */
    int64_t filter_misses;  /* exhaustive_strict only: strict accepts the filter would have lost (must be 0) */
    int32_t kernel_launches;
    int32_t n_sms;
    double flop_primary;    /* FP32 flops the closest-hit sweep executes per swept pair (FFMA = 2, FADD = FMUL = 1, a
                               minimum 0).  Hot rows (no jitter: the R rays of a thread share q): per thread and
                               triangle 4 FFMA for the bounds, 2 FADD for the interval and one packed FADD2 for the
                               thread's extreme rays (segment verdict), nothing per pair: 12/R.  Jittered samples with
                               a shared mean q (8 FFMA, and per pair half a packed FADD2): 1 + 18/R.  Three-row form (every ray its own q): 6 FFMA + FMUL + FFMA = 15.
                               0 in bundle-cull mode                                                              */
    double flop_shadow;     /* same for the any-hit sweeps (hot rows, R = 32 rays of one (p, q) cell share a mean q:
                               8 FFMA + 2 FADD per thread and triangle and one packed FADD2 for the thread's extreme
                               rays (segment verdict), nothing per pair): 20/R                                    */
    /* of which the multiply-adds that evaluate the bounds / edge rows (the rest is each pair's conjunction) */
    double flop_primary_edges;
    double flop_shadow_edges;
    int64_t pipeline_errors; /* exhaustive_strict only: the sweeps' own race check — staged table tiles (TMA pipeline,
                                per-warp stage recycling) that differed from their source when a warp started or
                                finished using them (must be 0) */
} tracer_frame_stats;

typedef struct tracer_device_info {
    char name[128];
    int32_t sm_count;
    int32_t cc_major, cc_minor;
    int32_t clock_khz; /* cudaDevAttrClockRate */
    int64_t total_mem;
    int64_t l2_bytes;
} tracer_device_info;

typedef struct tracer_scene_dev tracer_scene_dev; /* opaque: scene resident in HBM */

/* ---- lifetime ------------------------------------------------------------ */
int tracer_cuda_abi_version(void);
int tracer_cuda_init(int device_ordinal); /* cudaSetDevice + stream; makes that GPU the current context */
void tracer_cuda_shutdown(void);
const char *tracer_cuda_last_error(void);
int tracer_cuda_device_info(tracer_device_info *out);

/* ---- the drop-in call: host buffers in, packed 8-bit RGB out --------------
 * rgb_out: caller-owned, n_rows_of_this_call * W * 3 bytes (a crop: crop_h * crop_w * 3), PPM row order,
 * fully overwritten (unlike ispc::trace, which += into an un-zeroed malloc,
 * trace.ispc:262-265 / main.cpp:593).  Uploads the scene, renders, downloads. */
int tracer_cuda_render(const tracer_scene_flat *scene, const tracer_camera *cam, int32_t width, int32_t height,
                       const tracer_render_opts *opts, uint8_t *rgb_out);

/* ---- resident-scene variant (scene stays in HBM across frames) ------------ */
int tracer_cuda_scene_create(const tracer_scene_flat *scene, tracer_scene_dev **out);
void tracer_cuda_scene_destroy(tracer_scene_dev *scene);
int tracer_cuda_render_scene(tracer_scene_dev *scene, const tracer_camera *cam, int32_t width, int32_t height,
                             const tracer_render_opts *opts, uint8_t *rgb_out);
int tracer_cuda_last_stats(tracer_scene_dev *scene, tracer_frame_stats *out);

/* n_views frames of one resident scene, one per camera, in one call.  rgb_out: n_views * height * width * 3 bytes,
 * view-major, each view in PPM row order (host, or device with opts->rgb_out_is_device).  Debug outputs are view-major
 * too ([n_views * height * width] ...), and with TRACER_RNG_EXPLICIT opts->faceid is [n_views][W*H*n_lights].
 * View v is the frame tracer_cuda_render_scene gives for cams[v] with the same opts: packed bytes, hit ids, t, v,
 * first occluders and the float accumulator, in every rng_mode (TRACER_RNG_MT19937: each view draws from its own
 * std::mt19937(seed), as a separate run of the serial path would), with jittered samples, in the default and the BVH
 * mode, with exhaustive_strict.  Refused with TRACER_ERR_INVALID: n_views < 1, cams NULL, band_count > 1, bundle_cull != 0,
 * a crop window, n_views * width * height above the per-call pixel limit.  Stats (tracer_cuda_last_stats) are totals over the call.
 * The views share the camera-independent work of a frame: the shadow rays of every view go through one sweep per light
 * vertex batch; only the closest-hit sweep runs per view (one eye table each). */
int tracer_cuda_render_views(tracer_scene_dev *scene, const tracer_camera *cams, int32_t n_views, int32_t width,
                             int32_t height, const tracer_render_opts *opts, uint8_t *rgb_out);

/* ---- updating a resident scene between frames --------------------------------
 * Replaces vertices, normals, materials and spheres of a resident scene in place, without re-creating it.
 * Topology is fixed: the triangle, geometry, light and sphere counts, geom_tri_offset, light_geom and
 * geom_has_normals stay those of the create call (changing any of them means creating a new scene), and
 * triangle order stays the reference's iteration order.  A frame rendered after an update is the frame a
 * freshly created scene of the updated arrays gives, in every mode, rng_mode and band selection, packed bytes
 * and every debug output alike.
 * The library refreshes what depends on the geometry: the scene's bounding box (on the device), the light
 * vertices, the rows [tri_first, tri_first + tri_count) of every resident shadow filter table (tables of a
 * light vertex that moved are dropped and rebuilt by the next render that needs them) and, when vertices
 * changed, the BVH of the optional mode (rebuilt by the next BVH render).
 * Every check runs before anything is copied: a NULL pointer where tri_count needs data, a range outside
 * [0, n_tris], struct_size < sizeof(tracer_scene_update), tri_normals for a scene created without normals, and
 * with data_is_device a pointer that is not device or managed memory of the scene's GPU (multi: device 0).
 * A refused update returns TRACER_ERR_INVALID and leaves the scene as it was; the multi form checks every
 * replica before it changes any.  After TRACER_ERR_CUDA the scene's contents are undefined: destroy it.
 * The call is synchronous: it returns once the update is complete on the device, so the caller may reuse or
 * free its buffers.  Its copies and kernels run on cuda_stream, so data produced on that stream is ordered
 * before them (multi: cuda_stream is a stream of device 0; the other replicas wait for it, then copy from
 * device 0 with peer copies on their own streams).  tri_count = 0 and every pointer NULL is a no-op. */
typedef struct tracer_scene_update {
    uint32_t struct_size;          /* = sizeof(tracer_scene_update) */
    int32_t data_is_device;        /* 1: every pointer below is device memory on the scene's GPU (multi: device 0) */
    void *cuda_stream;             /* stream the copies and kernels run on; NULL = the library's own */
    int32_t tri_first, tri_count;  /* triangles [tri_first, tri_first + tri_count) */
    const float *tri_verts;        /* [tri_count*9] new vertices, or NULL */
    const float *tri_normals;      /* [tri_count*9] or NULL; only for scenes created with normals */
    const float *geom_material;    /* [n_geoms*13] or NULL */
    const float *sphere_cr;        /* [n_spheres*4] or NULL */
    const float *sphere_material;  /* [n_spheres*13] or NULL */
} tracer_scene_update;
int tracer_cuda_scene_update(tracer_scene_dev *scene, const tracer_scene_update *u);

/* ---- all GPUs of one box behind one call ------------------------------------
 * The reference has no multi-device path (its closest analogue is thread-per-row,
 * src/main.cpp:629-643).  One process; a context, stream and scene replica per GPU; one
 * host thread per GPU while a frame renders; one NCCL communicator set (ncclCommInitAll).
 * The frame's PPM rows are cut into bands of opts->band_rows (default 8) rows, band b is
 * rendered by GPU b % n_gpus, every GPU quantises its bands straight into its send
 * buffer and the packed bands are gathered on GPU 0 with grouped ncclSend/ncclRecv over
 * NVLink.  Results are byte-identical to a single-GPU frame, in every rng_mode: with
 * TRACER_RNG_MT19937 the GPUs exchange their per-row hit counts between their threads
 * (opts->row_hits_exchange is the call's own), and every GPU replays the draws itself.
 * After tracer_cuda_init_multi(n > 1) the drop-in tracer_cuda_render() uses all n GPUs. */
typedef struct tracer_scene_multi tracer_scene_multi; /* opaque: one scene replica per GPU */
int tracer_cuda_init_multi(int n_gpus);               /* devices 0 .. n_gpus-1 */
int tracer_cuda_multi_gpu_count(void);                /* 0 before tracer_cuda_init_multi */
int tracer_cuda_render_multi(const tracer_scene_flat *scene, const tracer_camera *cam, int32_t width, int32_t height,
                             const tracer_render_opts *opts, uint8_t *rgb_out);
int tracer_cuda_scene_create_multi(const tracer_scene_flat *scene, tracer_scene_multi **out);
void tracer_cuda_scene_destroy_multi(tracer_scene_multi *scene);
int tracer_cuda_render_scene_multi(tracer_scene_multi *scene, const tracer_camera *cam, int32_t width, int32_t height,
                                   const tracer_render_opts *opts, uint8_t *rgb_out); /* rgb_out: host, or GPU 0 if rgb_out_is_device */
int tracer_cuda_last_stats_multi(tracer_scene_multi *scene, tracer_frame_stats *out); /* counts summed, times of the slowest GPU */
int tracer_cuda_scene_update_multi(tracer_scene_multi *scene, const tracer_scene_update *u); /* every replica; see tracer_cuda_scene_update */

/* number of PPM rows the band selection (band_rows, band_index, band_count) covers */
int32_t tracer_band_row_count(int32_t height, int32_t band_rows, int32_t band_index, int32_t band_count);

/* Rank 0 after the gather: scatter band-packed rank buffers (each padded to
 * rows_per_rank_padded rows) into one PPM-ordered frame.  Device pointers. */
int tracer_cuda_assemble_bands(const uint8_t *gathered_dev, uint8_t *frame_dev, int32_t width, int32_t height,
                               int32_t band_rows, int32_t band_count, int32_t rows_per_rank_padded, void *cuda_stream);

/* ---- host utilities -------------------------------------------------------- */
/* std::mt19937 replay of the reference's draws (main.cpp:743-754): hit is the
 * full-frame mask in image index order; faceid [W*H*n_lights]. */
int tracer_mt19937_faceids(const tracer_scene_flat *scene, int32_t width, int32_t height, uint32_t seed,
                           const uint8_t *hit, int32_t *faceid);

/* ---- measurement: FP32 peak microbenchmark ---------------------------------
 * variant 0: scalar FFMA chains; 1: packed FFMA2 (fma.rn.f32x2) chains;
 * returns achieved TFLOP/s (2 flop per FMA) over `iters` launches timed with
 * CUDA events. */
int tracer_cuda_fp32_peak(int32_t variant, int32_t iters, double *tflops_out, double *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* TRACER_CUDA_H */
