/*
 * rt_b200.h -- C ABI of the B200-native sphere ray tracer (librt_b200.so).
 *
 * This is the drop-in boundary for the reference's one data-parallel hot path
 * (camera rays -> brute-force ray/sphere closest hit -> Phong + shadow rays -> reflection
 * bounces -> 8-bit RGB).  Plain pointers and sizes only: no C++ types, no torch types, no
 * exceptions and no exit() cross this line.  Every function returns 0 on success or a
 * negative rt_status; rt_last_error() returns the text of the calling thread's last failure.
 *
 * What each entry point replaces in the reference (paths relative to the reference root):
 *
 *   rt_scene_load / rt_scene_*     include/scene_loader.h:27-135   load_scene(filename)
 *   rt_upload_scene                src/main_hybrid.cpp:196-279     GPUResources::upload_scene
 *                                  src/kernel.cu:202-207           upload_lights_and_ambience
 *                                  include/camera.h:10-15          Camera::Camera (basis vectors)
 *   rt_render / rt_render_bands    src/main.cpp:146-157,185-199    the pixel loop + trace_ray
 *                                  src/kernel.cu:185-200           launch_gpu_kernel (tile launch)
 *                                  src/main.cpp:84-86              the 8-bit quantiser of write_ppm
 *   rt_render_tile                 src/kernel.cu:185-200           launch_gpu_kernel (tile + stream + float3 fb)
 *   rt_create_multi / rt_multi_*   src/main.cpp:185-199            the OpenMP pixel loop, sharded by row bands over GPUs
 *   rt_set_option("antialias")     src/main_gpu.cu:249-258,327-333 ray_cuda -a (2x2 supersampling)
 *   rt_write_ppm                   src/main.cpp:69-91              write_ppm (P3 text)
 *
 * Semantics are those of the reference's SERIAL renderer (FP64; src/main.cpp + include/ *.h),
 * not of its CUDA kernels: hit / sphere-index selection is bit-exact with ties to the lowest
 * sphere index, 8-bit RGB within 1 LSB.
 *
 * Threading: one host thread per rt_ctx at a time.  A ctx owns one CUDA device, one stream
 * and all device memory it allocates.  Renders of ONE ctx are serialised on the device, whatever
 * streams the caller passes (they share the ctx's ray queues and counters): a render enqueued on
 * stream B waits -- on the device, not on the host -- for the ctx's previous render on stream A, so
 * the reference's "tiles round-robin over three streams" loop (src/main_hybrid.cpp:611-622) is safe,
 * it just does not overlap tiles of the same ctx.  Camera, lights and ambient live in one
 * __constant__ bank per DEVICE (as in the reference, src/kernel.cu:7-9): contexts that share a
 * device may interleave renders freely; the bank is rewritten when it changes hands, stream-ordered
 * behind the previous owner's last render.  rt_upload_scene waits (on the host) for every render of
 * the ctx that is still in flight, also those enqueued on caller streams; rt_set_camera takes its place in the same
 * device-side render order instead (see there).  There is no CPU
 * fallback: every render entry point fails with RT_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 1
#define RT_MAX_LEVELS 32          /* reflection levels tracked in rt_stats.alive[]            */
#define RT_SPHERE_STRIDE 10       /* cx cy cz r R G B metallic roughness shininess (file order)*/
#define RT_LIGHT_STRIDE 7         /* x y z R G B intensity                         (file order)*/

typedef enum rt_status {
  RT_OK = 0,
  RT_ERR_ARG = -1,      /* bad argument (NULL pointer, non-positive size, ...)                 */
  RT_ERR_CUDA = -2,     /* CUDA runtime / driver error, or no usable sm_100 device             */
  RT_ERR_STATE = -3,    /* call order violated (e.g. render before upload)                     */
  RT_ERR_IO = -4,       /* file could not be opened / written                                  */
  RT_ERR_NOMEM = -5,
  RT_ERR_UNSUPPORTED = -6
} rt_status;

typedef struct rt_ctx rt_ctx;       /* opaque: device, stream, device-resident scene + buffers */
typedef struct rt_scene rt_scene;   /* opaque: a parsed scene file (host memory only)          */

/* Counters of one render.  Ray counts follow the oracle's definition (SURVEY 8d):
 * closest_queries = find_intersection calls issued by trace_ray (R_c), shadow_queries =
 * in_shadow calls (R_s = lights x hits).  They are properties of (scene, W, H, depth).  */
typedef struct rt_stats {
  double ms_device;             /* CUDA-event time of the kernels of this call on the stream   */
  double ms_host;               /* host wall-clock of the whole call, copies included          */
  double ms_level0;             /* device time of reflection level 0 (camera rays + their shadows + shading) */
  double ms_closest0;           /* ... of which: the camera-ray closest-hit kernel             */
  double ms_shadow0;            /* ... of which: the level-0 shadow kernel (the dominant one)  */
  uint64_t closest_queries;
  uint64_t hits;
  uint64_t shadow_queries;
  uint64_t occluded;
  uint64_t alive[RT_MAX_LEVELS];/* closest queries per reflection level                        */
  uint64_t fp64_intersections;  /* exact FP64 sphere evaluations the kernels needed            */
  uint64_t sphere_tests;        /* ray/sphere tests of the brute-force algorithm: N x (R_c + R_s)*/
  uint64_t filter_violations;   /* self-check of the FP32 filter; must be 0 (see DESIGN.md)    */
  int32_t kernel_launches;      /* kernels launched by this call                               */
  int32_t rows_rendered;        /* image rows this call produced (all of H unless banded)      */
  uint64_t bundle_walks;        /* warp-level table walks that used bundle culling (DESIGN.md)  */
  uint64_t bundle_candidates;   /* spheres left after culling, summed over those walks          */
  uint64_t bundle_fallbacks;    /* LBVH bundles that fell back to one traversal per ray          */
} rt_stats;

/* ---- library ------------------------------------------------------------------------- */
int rt_abi_version(void);
const char *rt_last_error(void);
/* Number of CUDA devices usable by this library (0 when none; never fails). */
int rt_device_count(void);

/* ---- scene files (host only; usable without a GPU) -------------------------------------
 * Same grammar and skip/warn behaviour as include/scene_loader.h:27-135: '#' comments,
 * "sphere x y z r R G B metallic roughness shininess", "light x y z R G B intensity",
 * "ambient R G B", "camera px py pz lx ly lz fov"; malformed or unknown lines are reported
 * on stderr and skipped; a file that cannot be opened is RT_ERR_IO.  Defaults when a line
 * type is absent: ambient (0,0,0), camera (0,0,0)->(0,0,-1) fov 60 (include/scene.h:22,31).
 * If verbose != 0 prints "Loaded scene: N spheres, M lights" like scene_loader.h:131-132.  */
int rt_scene_load(const char *path, int verbose, rt_scene **out);
int rt_scene_counts(const rt_scene *s, int *nspheres, int *nlights, int *has_camera);
/* Pointers stay valid until rt_scene_free.  spheres: N x RT_SPHERE_STRIDE, lights:
 * L x RT_LIGHT_STRIDE, ambient[3], camera[7] = pos xyz, look_at xyz, fov (degrees).       */
int rt_scene_data(const rt_scene *s, const double **spheres, const double **lights,
                  const double **ambient, const double **camera);
void rt_scene_free(rt_scene *s);

/* ---- context ---------------------------------------------------------------------------- */
int rt_create(int device, rt_ctx **out);
void rt_destroy(rt_ctx *ctx);
/* Integer options: "mode" 0 = fast FP32-filter kernels (default), 1 = exact FP64 brute force
 * (diagnostic; same results, slower); "counters" 0/1 = collect ray counters (default 1);
 * "accel" 0 = automatic (LBVH from 1024 spheres), 1 = table walks only, 2 = LBVH always (read at the
 * next rt_upload_scene); "wave_levels" 1..32 = reflection levels run as wavefront kernels before
 * the fused tail; "antialias" 0/1 = 2x2 supersampling as the reference's `ray_cuda -a`
 * (src/main_gpu.cu:249-258,327-333: samples at pixel offsets (0,0) (.5,0) (0,.5) (.5,.5),
 * averaged before the 8-bit quantiser); with it on, the debug buffers of rt_render_debug are
 * per sample: [2H][2W][max_depth], sample (a,b) of pixel (i,j) at (2j+b, 2i+a);
 * "level_timing" 0/1 = record CUDA events between the level-0 kernels so that rt_stats carries
 * ms_closest0 / ms_shadow0 / ms_level0 (default 0: the events break the back-to-back programmatic
 * dependent launches of the production path, so timing renders run a slightly different launch
 * sequence; without it those three fields equal ms_device / 0 / ms_device).                   */
int rt_set_option(rt_ctx *ctx, const char *key, long long value);

/* Copies the scene to the device (host -> device inside the call) and precomputes the
 * per-origin sphere tables.  Arrays are in scene-file column order (see rt_scene_data).
 * roughness and light intensity are accepted and ignored, as in the reference.            */
int rt_upload_scene(rt_ctx *ctx, const double *spheres, int nspheres, const double *lights,
                    int nlights, const double ambient[3], const double cam_pos[3],
                    const double cam_look[3], double fov_deg);

/* Moves the camera of the uploaded scene without uploading it again (turntables, fly-throughs, several views of one
 * scene).  Afterwards every render entry point produces exactly what rt_upload_scene of the same spheres, lights and
 * ambient with this camera would produce: pixels, debug buffers and every rt_stats counter (kernel_launches and the
 * times aside).  fov and look-at are taken as rt_upload_scene takes them.  The table layout chosen at the last upload is
 * kept (a new "accel" option still waits for the next upload).
 * Asynchronous on `stream` (NULL = the ctx stream), in the render order of the ctx: it waits on the device for the ctx's
 * previous render, and renders on other streams wait for it.  A new position rebuilds the camera's sphere table on the
 * device; a new look-at or fov alone launches nothing.  Exception: a camera that moves beyond the extent of the lights
 * and spheres (or back inside it) changes the FP32 filter slack of every table; then the call rebuilds the scene from a
 * host copy of the last upload and SYNCHRONISES like rt_upload_scene.  RT_ERR_STATE before any upload.               */
int rt_set_camera(rt_ctx *ctx, const double cam_pos[3], const double cam_look[3], double fov_deg, void *stream);

/* Renders the full frame and copies it to host_rgb: W*H*3 bytes, row j = 0 is the BOTTOM of
 * the image (src/main.cpp:153-154), channel value int(255.99*min(1,c)).  stats may be NULL. */
int rt_render(rt_ctx *ctx, int width, int height, int max_depth, uint8_t *host_rgb,
              rt_stats *stats);

/* As rt_render, additionally returning (each may be NULL), for every pixel p = j*W+i and
 * reflection level k < max_depth: hit_idx[p*max_depth+k] = sphere index, -1 = miss,
 * -2 = level not reached; shadow_mask[...] bit l = light l occluded at that hit.            */
int rt_render_debug(rt_ctx *ctx, int width, int height, int max_depth, uint8_t *host_rgb,
                    int32_t *hit_idx, uint32_t *shadow_mask, rt_stats *stats);

/* Row-band sharded render into DEVICE memory (no host copy, asynchronous on `stream`).
 * Bands are band_h rows tall; rank r of nranks owns bands b with b % nranks == r and writes
 * its rows, in ascending j, compactly into dev_rgb (rt_band_rows()*W*3 bytes, 16-byte
 * aligned).  nranks = 1 renders the whole frame.  stream is a cudaStream_t passed as void*
 * (NULL = the ctx stream); dev_rgb must belong to the ctx's device.  stats (may be NULL) is
 * filled after a stream synchronise only when counters are enabled.                        */
int rt_render_bands(rt_ctx *ctx, int width, int height, int max_depth, int band_h, int rank,
                    int nranks, void *dev_rgb, void *stream, rt_stats *stats);
/* As rt_render_bands, but the rows this rank owns are stored at their IMAGE positions of an assembled
 * H*W*3-byte frame (row j at dev_frame + j*W*3).  dev_frame may be memory of this GPU or peer-mapped
 * memory of another GPU of the box (rt_ipc_open): the ranks' kernels then write rank 0's frame directly
 * over NVLink while they compute, and the "gather" of SURVEY 8e shrinks to a completion signal
 * (rt_peer_signal / rt_peer_wait).  Not available with supersampling.                         */
int rt_render_bands_frame(rt_ctx *ctx, int width, int height, int max_depth, int band_h, int rank,
                          int nranks, void *dev_frame, void *stream, rt_stats *stats);
/* Device memory that processes of one box can share (one process per GPU, as under torchrun):
 * rt_dev_alloc = zeroed cudaMalloc on the ctx's device; rt_ipc_export writes the 64-byte CUDA IPC
 * handle of such an allocation; rt_ipc_open maps an exported allocation of another process (peer
 * access is enabled on demand) and returns a device pointer valid in the calling process.     */
int rt_dev_alloc(rt_ctx *ctx, size_t bytes, void **dev_ptr);
int rt_dev_free(rt_ctx *ctx, void *dev_ptr);
int rt_ipc_export(rt_ctx *ctx, void *dev_ptr, unsigned char handle[64]);
int rt_ipc_open(rt_ctx *ctx, const unsigned char handle[64], void **dev_ptr);
int rt_ipc_close(rt_ctx *ctx, void *dev_ptr);
/* Completion signalling on `stream` (NULL = ctx stream).  rt_peer_signal: after everything already
 * enqueued on the stream, store `value` to *flag (typically flag = rank 0's flags + rank, peer
 * mapped) with system-scope release ordering.  rt_peer_wait: enqueue a wait until flags[0..n) have
 * all reached `value` (n <= 64); on a ~2 s timeout it writes 1 + the missing index to *dev_err
 * (a device uint32 the caller zeroed) and returns to the stream.                               */
int rt_peer_signal(rt_ctx *ctx, uint32_t *flag, uint32_t value, void *stream);
int rt_peer_wait(rt_ctx *ctx, uint32_t *flags, int n, uint32_t value, uint32_t *dev_err, void *stream);

/* Tile render with the calling convention of the reference's launch_gpu_kernel
 * (src/kernel.cu:185-200; caller src/main_hybrid.cpp:461-466): renders pixels
 * [tile_x, tile_x+tile_w) x [tile_y, tile_y+tile_h) of a width x height image into the CALLER's
 * device framebuffer as FP32 RGB, dev_fb[(j*width + i)*3 + c] (= the reference's float3
 * d_framebuffer[pixel_idx]), row j = 0 = bottom, asynchronously on `stream` (NULL = ctx
 * stream).  The scene is the ctx's (rt_upload_scene replaces GPUResources::upload_scene +
 * upload_lights_and_ambience).  Pixels outside the tile are not touched.                   */
int rt_render_tile(rt_ctx *ctx, int width, int height, int max_depth, int tile_x, int tile_y,
                   int tile_w, int tile_h, float *dev_fb, void *stream);
/* Rows owned by `rank` under the band rule above. */
int rt_band_rows(int height, int band_h, int rank, int nranks);
/* Writes the owned row indices (ascending) into rows[rt_band_rows()]. */
int rt_band_row_list(int height, int band_h, int rank, int nranks, int32_t *rows);

/* ---- one frame on several GPUs of the box, in ONE process ---------------------------------
 * rt_create_multi(ngpus): ranks 0..ngpus-1, rank r on device r (r modulo the device count when the
 * box has fewer GPUs: same frame, no speed-up), each with its own rt_ctx (device, stream, scene
 * replica, buffers).  rt_multi_render: rank r renders the interleaved bands b with b % ngpus == r
 * (band = band_h rows; the rule of rt_render_bands) and copies them over ITS OWN host link to their
 * image positions in host_rgb (W*H*3, row 0 = bottom); the call returns when the frame is complete.
 * host_rgb is page-locked for the duration if it is not already (rt_host_alloc avoids that).
 * stats (may be NULL): counters summed over the ranks, times = the slowest rank.  rt_multi_ctx gives
 * the per-rank context for the calls that have no multi form (valid until rt_multi_destroy).     */
typedef struct rt_multi rt_multi;
int rt_create_multi(int ngpus, rt_multi **out);
void rt_multi_destroy(rt_multi *m);
int rt_multi_ranks(const rt_multi *m);
rt_ctx *rt_multi_ctx(rt_multi *m, int rank);
int rt_multi_set_option(rt_multi *m, const char *key, long long value);
int rt_multi_upload_scene(rt_multi *m, const double *spheres, int nspheres, const double *lights,
                          int nlights, const double ambient[3], const double cam_pos[3],
                          const double cam_look[3], double fov_deg);
/* rt_set_camera on every rank (each on its ctx stream). */
int rt_multi_set_camera(rt_multi *m, const double cam_pos[3], const double cam_look[3], double fov_deg);
int rt_multi_render(rt_multi *m, int width, int height, int max_depth, int band_h, uint8_t *host_rgb,
                    rt_stats *stats);
/* A camera path frame-parallel over the ranks: whole frames go to different GPUs instead of every frame being split into
 * bands, so each GPU renders full frames at its single-GPU efficiency.  cameras: K rows of 7 host doubles, px py pz lx ly
 * lz fov (the scene file's order).  dev_frames: K*H*W*3 bytes of device memory on RANK 0's device; frame k starts at
 * k*H*W*3 (any alignment), row 0 = bottom.  Rank k % ngpus renders frame k exactly as rt_set_camera with cameras[k]
 * followed by a full-frame render on that rank would, so every frame is byte-identical to the same path rendered on one
 * context with the same options (mode, accel, antialias, wave_levels).  A rank renders into a frame buffer on its own
 * device and copies it into place (a peer copy from another device; peer access is enabled on demand, and a device pair
 * without it is RT_ERR_UNSUPPORTED -- nothing is staged through host memory).
 * Asynchronous: every rank works on its ctx stream, in that ctx's render order, and the host enqueues the ranks' frames
 * on parallel threads (one per device; ranks that share a device share one), joined before the call returns.  No
 * frame is written before the work already on `stream` at the call has finished, and `stream` waits, on the device, for
 * every frame: the caller consumes them on `stream` without a host synchronisation.  `stream` is a cudaStream_t of rank
 * 0's device passed as void* (NULL = rank 0's ctx stream).  The one host synchronisation is rt_set_camera's: a camera
 * that leaves the extent of the lights and spheres (or comes back inside it) makes that rank rebuild its scene and wait.
 * Afterwards every rank's camera is cameras[K-1].  There is no rt_stats argument: per-frame counters would need a host
 * synchronisation per frame.  RT_ERR_ARG for a NULL pointer, K < 1, a size below 1, max_depth < 0 or dev_frames not on
 * rank 0's device; RT_ERR_STATE before rt_multi_upload_scene; when ranks fail, the error of the lowest failing rank,
 * after every thread has joined.  With more ranks than devices the frames are the same, without a speed-up.        */
int rt_multi_render_path(rt_multi *m, const double *cameras, int K, int width, int height, int max_depth,
                         void *dev_frames, void *stream);

/* One process per GPU (torchrun): as rt_multi_render's per-rank half.  Every rank calls it with the SAME host frame
 * (shared memory, W*H*3 bytes, row 0 = bottom) and its own (rank, nranks); the rank's bands are rendered and copied to
 * their image positions over this GPU's host link.  Returns when this rank's rows have landed; the frame is complete
 * when every rank has returned (the caller synchronises the ranks).  Page-lock the frame in every process first
 * (rt_host_register) or the copies are staged through pageable memory.                          */
int rt_render_bands_host(rt_ctx *ctx, int width, int height, int max_depth, int band_h, int rank,
                         int nranks, uint8_t *host_rgb, rt_stats *stats);

/* ---- pinned host memory -----------------------------------------------------------------
 * Page-locked buffers so that the frame copy of rt_render runs at full host-link rate.
 * (The reference does the same for its bulk copy: src/main_hybrid.cpp:524.)                 */
int rt_host_alloc(size_t bytes, void **out);
void rt_host_free(void *p);
/* Page-locks / releases memory the caller allocated itself (e.g. a POSIX shared-memory frame).   */
int rt_host_register(void *p, size_t bytes);
int rt_host_unregister(void *p);

/* ---- measurement -------------------------------------------------------------------------
 * FP32 FFMA issue peak of `device` in FLOP/s (8 independent chains/thread, all SMs busy) and
 * the SM clock seen while it ran.  bench.py divides the algorithmic FLOP/s by this.          */
int rt_measure_fp32_peak(int device, double *flops_per_s, double *sm_clock_mhz);

/* ---- PPM (host only) -------------------------------------------------------------------- */
/* P3 text, byte-identical to src/main.cpp:69-91: "P3\nW H\n255\n", rows j = H-1 .. 0, one
 * "r g b\n" per pixel.  rgb is bottom-row-first as produced by rt_render.                   */
int rt_write_ppm(const char *path, const uint8_t *rgb, int width, int height);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
