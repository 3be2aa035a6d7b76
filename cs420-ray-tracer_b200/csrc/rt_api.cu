// rt_api.cu -- host side of the C ABI declared in include/rt_b200.h.
//
// Owns the context (device, stream, device-resident scene), converts the reference's
// AoS/FP64 data model (include/sphere.h:8-20, include/scene.h:10-38) into the device layout
// described in rt_device.h, and sequences the kernels.  No rendering arithmetic happens on
// the host; there is no CPU fallback.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "rt_device.h"
#include "rt_internal.h"
#include "rt_kernels.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

// ------------------------------------------------------------------------------------------
// errors
static thread_local std::string g_last_error;
int rt_fail(int code, const std::string &msg) { g_last_error = msg; return code; }
extern "C" const char *rt_last_error(void) { return g_last_error.c_str(); }
extern "C" int rt_abi_version(void) { return RT_ABI_VERSION; }

#define RT_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return rt_fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));             \
  } while (0)

extern "C" int rt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// ------------------------------------------------------------------------------------------
// context
struct rt_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evm[3] = {nullptr, nullptr, nullptr};
  // Every render of a ctx shares one set of work buffers (queues, counters, hit blocks) and the device's __constant__
  // bank, so renders of one ctx are SERIALISED on the device whatever streams the caller hands in: ev_last is recorded
  // behind the last kernel of each render and the next render's stream waits for it when it is a different stream.
  cudaEvent_t ev_last = nullptr;
  cudaStream_t last_stream = nullptr;
  bool last_valid = false;
  int pend_launches = 0, pend_rows = 0; bool pend_counters = false, pend_marks = false; cudaStream_t pend_stream = nullptr;   // collect_stats
  int level_timing = 0;  // 1: event records between the level-0 kernels (rt_stats.ms_closest0 / ms_shadow0); turns PDL off
  int mode = 0;          // 0 fast, 1 exact
  int counters_on = 1;
  int accel = 0;         // 0 auto, 1 table walks, 2 LBVH (takes effect at the next rt_upload_scene)
  int antialias = 0;     // 2x2 supersampling (the reference's ray_cuda -a)
  // scene
  bool have_scene = false;
  int N = 0, L = 0;
  double fov = 60.0;
  RtFrameConst frame;
  unsigned long long scene_version = 0;
  // host copy of the last upload, for rt_set_camera's full rebuild when the camera changes delta64; up_accel = the accel
  // option that upload was built with (the table layout rt_set_camera keeps)
  std::vector<double> h_sph, h_lig;
  double h_amb[3] = {0, 0, 0};
  int up_accel = 0;
  double4 *d_sph64 = nullptr;
  float4 *d_mat = nullptr;
  float2 *d_matx = nullptr;
  RtFastScene fast;      // FP32 filter tables (rt_kernels.h)
  // per-resolution tables
  int tabW = 0, tabH = 0, tab_aa = 0;
  double tab_fov = 0;
  double *d_su = nullptr, *d_sv = nullptr;
  bool tab_valid = false;   // d_su / d_sv hold the coordinates of (tabW, tabH, tab_aa, tab_fov)
  float *d_fb = nullptr; size_t fb_cap = 0;   // float sample frame of a supersampled render
  // buffers
  uint8_t *d_rgb = nullptr; size_t rgb_cap = 0;
  uint8_t *d_part = nullptr; size_t part_cap = 0;   // compact band buffer of rt_render_bands_host / rt_multi_render
  int32_t *d_hit = nullptr; size_t hit_cap = 0;
  uint32_t *d_mask = nullptr; size_t mask_cap = 0;
  unsigned long long *d_counters = nullptr;
  RtFastWork work;       // queues / accumulators of the fast path
};

// which (ctx, scene_version) last wrote each device's __constant__ bank
static std::mutex g_const_mutex;
static const rt_ctx *g_const_owner[64] = {nullptr};
static unsigned long long g_const_version[64] = {0};

extern "C" void rt_destroy(rt_ctx *c);
extern "C" int rt_create(int device, rt_ctx **out) {
  if (!out) return rt_fail(RT_ERR_ARG, "rt_create: NULL out");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return rt_fail(RT_ERR_CUDA, "rt_create: no CUDA device (this library has no CPU fallback)");
  }
  if (device < 0 || device >= n || device >= 64) return rt_fail(RT_ERR_ARG, "rt_create: bad device index");
  cudaDeviceProp prop;
  RT_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return rt_fail(RT_ERR_CUDA, std::string("rt_create: device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                    ", this library is built for sm_100a only");
  RT_CUDA(cudaSetDevice(device));
  rt_ctx *c = new (std::nothrow) rt_ctx();
  if (!c) return rt_fail(RT_ERR_NOMEM, "rt_create: out of memory");
  c->device = device;
  memset(&c->frame, 0, sizeof(c->frame));
  memset(&c->fast, 0, sizeof(c->fast));
  memset(&c->work, 0, sizeof(c->work));
  c->work.num_sms = prop.multiProcessorCount;
  // (a failure below must not leak the half-built context: rt_destroy copes with null members)
  cudaError_t ce = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaEventCreate(&c->ev0);
  if (ce == cudaSuccess) ce = cudaEventCreate(&c->ev1);
  for (int k = 0; k < 3 && ce == cudaSuccess; k++) ce = cudaEventCreate(&c->evm[k]);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&c->ev_last, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaMalloc(&c->d_counters, RT_CNT_TOTAL * sizeof(unsigned long long));
  if (ce != cudaSuccess) {
    rt_destroy(c);
    return rt_fail(RT_ERR_CUDA, std::string("rt_create: ") + cudaGetErrorString(ce));
  }
  int r = rtk_fast_init(c->device);
  if (r != 0) {
    rt_destroy(c);
    return rt_fail(RT_ERR_CUDA, std::string("rt_create: kernel attribute setup failed: ") + cudaGetErrorString((cudaError_t)-r));
  }
  *out = c;
  return RT_OK;
}

static void free_scene(rt_ctx *c) {
  c->d_sph64 = nullptr; c->d_mat = nullptr; c->d_matx = nullptr;   // (they point into the table arena)
  rtk_fast_free_scene(&c->fast, 1);
  c->have_scene = false;
}

extern "C" void rt_destroy(rt_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->last_valid) cudaEventSynchronize(c->ev_last);       // renders enqueued on caller streams
  {
    std::lock_guard<std::mutex> lk(g_const_mutex);
    if (g_const_owner[c->device] == c) g_const_owner[c->device] = nullptr;
  }
  free_scene(c);
  rtk_fast_free_work(&c->work);
  cudaFree(c->d_su); cudaFree(c->d_sv);
  cudaFree(c->d_part);
  cudaFree(c->d_rgb); cudaFree(c->d_hit); cudaFree(c->d_mask); cudaFree(c->d_counters); cudaFree(c->d_fb);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  for (int k = 0; k < 3; k++) if (c->evm[k]) cudaEventDestroy(c->evm[k]);
  if (c->ev_last) cudaEventDestroy(c->ev_last);
  if (c->stream) cudaStreamDestroy(c->stream);
  cudaGetLastError();
  delete c;
}

extern "C" int rt_set_option(rt_ctx *c, const char *key, long long value) {
  if (!c || !key) return rt_fail(RT_ERR_ARG, "rt_set_option: NULL argument");
  if (!strcmp(key, "mode")) {
    if (value != 0 && value != 1) return rt_fail(RT_ERR_ARG, "rt_set_option: mode must be 0 or 1");
    c->mode = (int)value;
    return RT_OK;
  }
  if (!strcmp(key, "counters")) { c->counters_on = value != 0; return RT_OK; }
  if (!strcmp(key, "antialias")) { c->antialias = value != 0; return RT_OK; }
  if (!strcmp(key, "level_timing")) { c->level_timing = value != 0; return RT_OK; }
  if (!strcmp(key, "accel")) {
    if (value < 0 || value > 2) return rt_fail(RT_ERR_ARG, "rt_set_option: accel must be 0 (auto), 1 (tables) or 2 (LBVH)");
    c->accel = (int)value;
    return RT_OK;
  }
  if (!strcmp(key, "wave_levels")) {
    if (value < 1 || value > RT_MAX_LEVELS) return rt_fail(RT_ERR_ARG, "rt_set_option: wave_levels must be 1..32");
    c->work.wave_levels = (int)value;
    return RT_OK;
  }
  return rt_fail(RT_ERR_ARG, std::string("rt_set_option: unknown key ") + key);
}

// ------------------------------------------------------------------------------------------
// scene upload
namespace {
struct V3 { double x, y, z; };
inline V3 vsub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline double vlen(V3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
inline V3 vnorm(V3 a) { double l = vlen(a); return {a.x / l, a.y / l, a.z / l}; }
inline V3 vcross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

// include/camera.h:10-15, in double on the host
void set_camera_basis(RtFrameConst &f, const double cam_pos[3], const double cam_look[3]) {
  V3 pos{cam_pos[0], cam_pos[1], cam_pos[2]}, look{cam_look[0], cam_look[1], cam_look[2]};
  V3 fwd = vnorm(vsub(look, pos));
  V3 right = vnorm(vcross(fwd, V3{0, 1, 0}));
  V3 up = vnorm(vcross(right, fwd));
  f.cam_pos[0] = pos.x; f.cam_pos[1] = pos.y; f.cam_pos[2] = pos.z;
  f.fwd[0] = fwd.x; f.fwd[1] = fwd.y; f.fwd[2] = fwd.z;
  f.right[0] = right.x; f.right[1] = right.y; f.right[2] = right.z;
  f.up[0] = up.x; f.up[1] = up.y; f.up[2] = up.z;
}
}  // namespace

// The upload proper; the rows may be the ctx's own host copy (rt_set_camera's full rebuild).
static int upload_scene(rt_ctx *c, const double *spheres, int N, const double *lights, int L, const double ambient[3],
                        const double cam_pos[3], const double cam_look[3], double fov_deg, int accel) {
  RT_CUDA(cudaSetDevice(c->device));
  RT_CUDA(cudaStreamSynchronize(c->stream));
  // the tables are rebuilt in place: renders of this ctx still running on a CALLER's stream must finish first
  if (c->last_valid) RT_CUDA(cudaEventSynchronize(c->ev_last));
  c->have_scene = false;
  rtk_fast_free_scene(&c->fast, 0);              // keeps the table allocation for reuse
  c->N = N; c->L = L; c->fov = fov_deg;

  RtFrameConst &f = c->frame;
  memset(&f, 0, sizeof(f));
  set_camera_basis(f, cam_pos, cam_look);
  for (int l = 0; l < L; l++) {
    const double *r = lights + (size_t)l * RT_LIGHT_STRIDE;
    for (int k = 0; k < 3; k++) { f.light_pos[l][k] = r[k]; f.light_col[l][k] = (float)r[3 + k]; }
  }
  for (int k = 0; k < 3; k++) f.ambient[k] = (float)ambient[k];
  f.nlights = L; f.nspheres = N;

  // exact geometry, materials and the FP32 filter tables: one staged arena, one host->device copy (rt_kernels.cu)
  int r = rtk_fast_build_scene(&c->fast, spheres, N, &f, accel, c->stream);
  if (r != 0) return rt_fail(RT_ERR_CUDA, std::string("rt_upload_scene: filter table build failed: ") + cudaGetErrorString((cudaError_t)-r));
  c->d_sph64 = (double4 *)c->fast.sph64; c->d_mat = (float4 *)c->fast.mat; c->d_matx = (float2 *)c->fast.matx;
  c->up_accel = accel;
  c->scene_version++;
  c->have_scene = true;
  return RT_OK;
}

extern "C" int rt_upload_scene(rt_ctx *c, const double *spheres, int N, const double *lights, int L,
                               const double ambient[3], const double cam_pos[3], const double cam_look[3],
                               double fov_deg) {
  if (!c || N < 0 || L < 0 || (N > 0 && !spheres) || (L > 0 && !lights) || !ambient || !cam_pos || !cam_look)
    return rt_fail(RT_ERR_ARG, "rt_upload_scene: bad argument");
  if (L > RT_MAX_LIGHTS)
    return rt_fail(RT_ERR_UNSUPPORTED, "rt_upload_scene: more than " + std::to_string(RT_MAX_LIGHTS) + " lights");
  c->h_sph.assign(spheres, spheres + (size_t)N * RT_SPHERE_STRIDE);
  c->h_lig.assign(lights, lights + (size_t)L * RT_LIGHT_STRIDE);
  for (int k = 0; k < 3; k++) c->h_amb[k] = ambient[k];
  return upload_scene(c, c->h_sph.data(), N, c->h_lig.data(), L, c->h_amb, cam_pos, cam_look, fov_deg, c->accel);
}

// Moves the camera of the uploaded scene (DESIGN.md "Camera moves").  Only table 0, the camera basis / position of the
// constant bank and the camera-plane tables depend on the camera; everything else the upload built stays.
extern "C" int rt_set_camera(rt_ctx *c, const double cam_pos[3], const double cam_look[3], double fov_deg, void *stream) {
  if (!c || !cam_pos || !cam_look) return rt_fail(RT_ERR_ARG, "rt_set_camera: NULL argument");
  if (!c->have_scene) return rt_fail(RT_ERR_STATE, "rt_set_camera: no scene uploaded (call rt_upload_scene first)");
  RT_CUDA(cudaSetDevice(c->device));
  if (rtk_delta64(c->fast.sabs_scene, cam_pos) != c->fast.delta64) {
    // the camera changes the slack of every table (it is now the farthest point of the scene, or no longer): full
    // rebuild with the layout of the last upload; synchronises like rt_upload_scene
    std::vector<double> sph, lig;   // (upload_scene may be handed the ctx's own copies: keep them apart from the call)
    sph.swap(c->h_sph); lig.swap(c->h_lig);
    const double amb[3] = {c->h_amb[0], c->h_amb[1], c->h_amb[2]};
    const int rc = upload_scene(c, sph.data(), c->N, lig.data(), c->L, amb, cam_pos, cam_look, fov_deg, c->up_accel);
    sph.swap(c->h_sph); lig.swap(c->h_lig);
    return rc;
  }
  const cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
  // table 0 is rewritten in place: after the ctx's last render, whatever stream that was on
  if (c->last_valid && c->last_stream != s) RT_CUDA(cudaStreamWaitEvent(s, c->ev_last, 0));
  if (memcmp(cam_pos, c->frame.cam_pos, sizeof(c->frame.cam_pos)) != 0) {
    const int r = rtk_fast_camera_table(&c->fast, cam_pos, s);
    if (r != 0) return rt_fail(RT_ERR_CUDA, std::string("rt_set_camera: camera table rebuild failed: ") + cudaGetErrorString((cudaError_t)-r));
  }
  set_camera_basis(c->frame, cam_pos, cam_look);
  c->fov = fov_deg;
  c->scene_version++;                                 // the next render rewrites the constant bank
  {
    std::lock_guard<std::mutex> lk(g_const_mutex);
    RT_CUDA(cudaEventRecord(c->ev_last, s));          // a render on another stream waits for the rebuild
    c->last_stream = s; c->last_valid = true;
  }
  return RT_OK;
}

// ------------------------------------------------------------------------------------------
// render
// Per-column / per-row camera-plane coordinates.  aa = 1: the 2W x 2H SAMPLE grid of the 2x2 supersampling
// (sample (a, b) of pixel (i, j) sits at index (2i + a, 2j + b); u = (i + a/2)/(W-1), src/main_gpu.cu:253-256).
// The coordinates are computed on the device (k_cam_plane: the operations of include/camera.h:18-22 and
// src/main.cpp:151-152 in the same order, correctly rounded, tan evaluated here), stream ordered behind the ctx's previous
// render: a new fov (rt_set_camera) regenerates them in place without a host sync.  A new size reallocates them.
static int ensure_tables(rt_ctx *c, int W, int H, int aa, cudaStream_t stream) {
  if (c->tab_valid && c->tabW == W && c->tabH == H && c->tab_fov == c->fov && c->tab_aa == aa) return RT_OK;
  const int m = aa ? 2 : 1;
  if (!c->d_su || c->tabW != W || c->tabH != H || c->tab_aa != aa) {
    c->tab_valid = false;
    cudaFree(c->d_su); cudaFree(c->d_sv); c->d_su = c->d_sv = nullptr;
    RT_CUDA(cudaMalloc(&c->d_su, (size_t)W * m * sizeof(double)));
    RT_CUDA(cudaMalloc(&c->d_sv, (size_t)H * m * sizeof(double)));
    c->tabW = W; c->tabH = H; c->tab_aa = aa;
  }
  const double scale = std::tan(c->fov * 0.5 * M_PI / 180.0);
  const int r = rtk_camera_plane(c->d_su, W * m, c->d_sv, H * m, m, W, H, scale, stream);
  if (r != 0) return rt_fail(RT_ERR_CUDA, std::string("render: camera-plane tables: ") + cudaGetErrorString((cudaError_t)-r));
  c->tab_fov = c->fov; c->tab_valid = true;
  return RT_OK;
}

template <typename T>
static int ensure_cap(T *&ptr, size_t &cap, size_t need) {
  if (cap >= need && ptr) return RT_OK;
  cudaFree(ptr); ptr = nullptr; cap = 0;
  RT_CUDA(cudaMalloc(&ptr, need * sizeof(T)));
  cap = need;
  return RT_OK;
}

extern "C" int rt_band_rows(int H, int band_h, int rank, int nranks) {
  if (H < 0 || band_h < 1 || nranks < 1 || rank < 0 || rank >= nranks) return rt_fail(RT_ERR_ARG, "rt_band_rows: bad argument");
  int rows = 0;
  for (int b = rank; b * band_h < H; b += nranks) {
    int j0 = b * band_h, j1 = j0 + band_h < H ? j0 + band_h : H;
    rows += j1 - j0;
  }
  return rows;
}

extern "C" int rt_band_row_list(int H, int band_h, int rank, int nranks, int32_t *rows) {
  int n = rt_band_rows(H, band_h, rank, nranks);
  if (n < 0) return n;
  if (!rows) return rt_fail(RT_ERR_ARG, "rt_band_row_list: NULL rows");
  int k = 0;
  for (int b = rank; b * band_h < H; b += nranks)
    for (int j = b * band_h; j < (b + 1) * band_h && j < H; j++) rows[k++] = j;
  return n;
}

static void fill_stats(rt_stats *st, const unsigned long long *cnt) {
  st->closest_queries = cnt[RT_CNT_CLOSEST];
  st->hits = cnt[RT_CNT_HITS];
  st->shadow_queries = cnt[RT_CNT_SHADOW];
  st->occluded = cnt[RT_CNT_OCCLUDED];
  st->fp64_intersections = cnt[RT_CNT_FP64];
  st->sphere_tests = cnt[RT_CNT_TESTS];
  st->filter_violations = cnt[RT_CNT_VIOLATIONS];
  st->bundle_walks = cnt[RT_CNT_WALKS];
  st->bundle_candidates = cnt[RT_CNT_CAND];
  st->bundle_fallbacks = cnt[RT_CNT_FALLBACKS];
  for (int k = 0; k < RT_MAX_LEVELS; k++) st->alive[k] = cnt[RT_CNT_ALIVE0 + k];
}

// Launches the kernels of one (possibly banded) render on `stream`.  When `stats` is given the
// call synchronises the stream and fills it.  With supersampling on, the kernels render the 2W x 2H sample
// grid into a float frame and k_resolve_aa averages it into dev_rgb; debug buffers are per SAMPLE then.
// Second half of a render that asked for stats: waits for the stream and fills *stats.  Split from the launch half so
// that a multi-GPU frame (rt_multi_render) can enqueue every rank's share before it waits for any of them.
static int collect_stats(rt_ctx *c, rt_stats *stats) {
  RT_CUDA(cudaSetDevice(c->device));
  RT_CUDA(cudaStreamSynchronize(c->pend_stream));
  float ms = 0;
  RT_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  memset(stats, 0, sizeof(*stats));
  stats->ms_device = ms;
  stats->ms_level0 = ms;
  stats->ms_closest0 = ms; stats->ms_shadow0 = 0;
  if (c->pend_marks) {
    float m0 = 0, m1 = 0, m2 = 0;
    RT_CUDA(cudaEventElapsedTime(&m0, c->ev0, c->evm[0]));
    RT_CUDA(cudaEventElapsedTime(&m1, c->evm[0], c->evm[1]));
    RT_CUDA(cudaEventElapsedTime(&m2, c->ev0, c->evm[2]));
    stats->ms_closest0 = m0; stats->ms_shadow0 = m1; stats->ms_level0 = m2;
  }
  stats->kernel_launches = c->pend_launches;
  stats->rows_rendered = c->pend_rows;
  if (c->mode == 0 && c->pend_rows > 0) {
    // compute-sanitizer cannot run on this pool: the kernels guard their own queue bounds and report here
    unsigned int word = 0;
    const int er = rtk_fast_last_error(&c->work, &word);
    if (er != 0) return rt_fail(RT_ERR_CUDA, std::string("render: reading the error word failed: ") + cudaGetErrorString((cudaError_t)-er));
    if (word != 0)
      return rt_fail(RT_ERR_STATE, "render: device-side guard tripped (bit 0: hit-block buffer, bit 1: ray queue): word " +
                                       std::to_string(word));
  }
  if (c->pend_counters) {
    unsigned long long cnt[RT_CNT_TOTAL];
    RT_CUDA(cudaMemcpy(cnt, c->d_counters, sizeof(cnt), cudaMemcpyDeviceToHost));
    fill_stats(stats, cnt);
  }
  return RT_OK;
}

struct TileSpec { int x, y, w, h; float *fb; int frame; };   // rt_render_tile: float output into the caller's full-frame buffer;
                                                            // frame = 1 (rt_render_bands_frame): 8-bit rows at their image positions
static int render_common(rt_ctx *c, int W, int H, int depth, int band_h, int rank, int nranks, uint8_t *dev_rgb,
                         int32_t *dev_hit, uint32_t *dev_mask, cudaStream_t stream, rt_stats *stats, const TileSpec *tile = nullptr,
                         bool defer_collect = false) {
  if (!c->have_scene) return rt_fail(RT_ERR_STATE, "render: no scene uploaded (call rt_upload_scene first)");
  if (W < 1 || H < 1 || depth < 0) return rt_fail(RT_ERR_ARG, "render: bad image size or depth");
  if (depth > RT_MAX_LEVELS) return rt_fail(RT_ERR_UNSUPPORTED, "render: max_depth above RT_MAX_LEVELS");
  const bool frame_mode = tile && tile->frame;
  if (frame_mode) tile = nullptr;
  if (frame_mode && c->antialias) return rt_fail(RT_ERR_UNSUPPORTED, "rt_render_bands_frame: not with supersampling");
  const int aa = (c->antialias && !tile) ? 1 : 0, m = aa ? 2 : 1;
  if ((aa || tile || frame_mode) && c->mode == 1) return rt_fail(RT_ERR_UNSUPPORTED, "render: supersampling / tile renders need mode 0");
  int rows = rt_band_rows(H, band_h, rank, nranks);
  if (rows < 0) return rows;
  RT_CUDA(cudaSetDevice(c->device));
  // renders of one ctx are serialised on the device (shared work buffers): a render on another stream than the
  // previous one first waits for that one's last kernel
  if (c->last_valid && c->last_stream != stream) RT_CUDA(cudaStreamWaitEvent(stream, c->ev_last, 0));
  int rc = ensure_tables(c, W, H, aa, stream);   // (after the wait: the tables may be rewritten in place)
  if (rc) return rc;
  {
    // The camera / lights / ambient bank is one __constant__ symbol per device.  It is rewritten only when its
    // content changes hands, and only after the previous owner's last render has finished (its ev_last); the copy is
    // stream ordered before this render's kernels, and later renders of this ctx are ordered behind it by ev_last.
    std::lock_guard<std::mutex> lk(g_const_mutex);
    if (g_const_owner[c->device] != c || g_const_version[c->device] != c->scene_version) {
      const rt_ctx *prev = g_const_owner[c->device];
      if (prev && prev != c && prev->last_valid) RT_CUDA(cudaStreamWaitEvent(stream, prev->ev_last, 0));
      RT_CUDA(rtk_set_frame_const(&c->frame, stream));
      g_const_owner[c->device] = c;
      g_const_version[c->device] = c->scene_version;
    }
  }
  const bool want_counters = c->counters_on && stats != nullptr;
  RtRenderArgs a;
  memset(&a, 0, sizeof(a));
  a.W = W * m; a.H = H * m; a.max_depth = depth;
  a.bands.band_h = band_h * m; a.bands.rank = rank; a.bands.nranks = nranks; a.bands.local_rows = rows * m;
  a.su = c->d_su; a.sv = c->d_sv;
  a.sph64 = c->d_sph64; a.mat = c->d_mat; a.matx = c->d_matx;
  a.rgb = dev_rgb; a.hit_idx = dev_hit; a.shadow_mask = dev_mask;
  if (aa) {
    if ((rc = ensure_cap(c->d_fb, c->fb_cap, (size_t)a.W * a.bands.local_rows * 3 + 4))) return rc;
    a.fb = c->d_fb;
    if (depth <= 0) RT_CUDA(cudaMemsetAsync(c->d_fb, 0, (size_t)a.W * a.bands.local_rows * 3 * sizeof(float), stream));
  }
  if (tile) {
    // the tile is a W' x H' frame whose camera-plane coordinates start at (tile.x, tile.y) of the full image's tables
    a.W = tile->w; a.H = tile->h;
    a.bands.band_h = tile->h; a.bands.rank = 0; a.bands.nranks = 1; a.bands.local_rows = tile->h;
    a.su = c->d_su + tile->x; a.sv = c->d_sv + tile->y;
    a.fb = tile->fb; a.rgb = nullptr;
    a.out_remap = 1; a.out_pitch = W; a.out_x0 = tile->x; a.out_y0 = tile->y;
    rows = tile->h;
    if (depth <= 0) RT_CUDA(cudaMemset2DAsync(tile->fb + ((size_t)tile->y * W + tile->x) * 3, (size_t)W * 12, 0, (size_t)tile->w * 12, tile->h, stream));
  }
  if (frame_mode) {
    a.out_remap = 2;
    if (depth <= 0)                                  // src/main.cpp:17-18: black; this rank's bands only
      for (int b = rank; b * band_h < H; b += nranks) {
        const int j0 = b * band_h, j1 = j0 + band_h < H ? j0 + band_h : H;
        RT_CUDA(cudaMemsetAsync(dev_rgb + (size_t)j0 * W * 3, 0, (size_t)(j1 - j0) * W * 3, stream));
      }
  }
  a.counters = want_counters ? c->d_counters : nullptr;
  if (want_counters) RT_CUDA(cudaMemsetAsync(c->d_counters, 0, RT_CNT_TOTAL * sizeof(unsigned long long), stream));
  if (stats) RT_CUDA(cudaEventRecord(c->ev0, stream));
  int launches = 0;
  if (rows > 0) {
    if (c->mode == 1) launches = rtk_launch_exact(a, stream);
    else launches = rtk_launch_fast(a, &c->fast, &c->work, stream, (stats && depth > 0 && c->level_timing) ? c->evm : nullptr);
    if (launches < 0) return rt_fail(RT_ERR_CUDA, std::string("render: launch failed: ") + cudaGetErrorString((cudaError_t)-launches));
    if (aa) {
      const int r2 = rtk_resolve_aa(c->d_fb, W, rows, dev_rgb, stream);
      if (r2 < 0) return rt_fail(RT_ERR_CUDA, std::string("render: resolve launch failed: ") + cudaGetErrorString((cudaError_t)-r2));
      launches += r2;
    }
  }
  {
    std::lock_guard<std::mutex> lk(g_const_mutex);   // (another ctx's render may look at ev_last when the constant bank changes hands)
    RT_CUDA(cudaEventRecord(c->ev_last, stream));
    c->last_stream = stream; c->last_valid = true;
  }
  if (stats) {
    RT_CUDA(cudaEventRecord(c->ev1, stream));
    c->pend_launches = launches; c->pend_rows = rows; c->pend_counters = want_counters;
    c->pend_marks = rows > 0 && c->mode == 0 && depth > 0 && c->level_timing;
    c->pend_stream = stream;
    if (!defer_collect) return collect_stats(c, stats);
  }
  return RT_OK;
}

// Renders the tile [tile_x, tile_x + tile_w) x [tile_y, tile_y + tile_h) of a width x height image into the
// caller's device framebuffer as FP32 RGB: dev_fb[(j * width + i) * 3 + c], row j = 0 = bottom, asynchronously on
// `stream` -- the calling convention of the reference's tile launcher (src/kernel.cu:185-200).
extern "C" int rt_render_tile(rt_ctx *c, int W, int H, int depth, int tile_x, int tile_y, int tile_w, int tile_h,
                              float *dev_fb, void *stream) {
  if (!c || !dev_fb) return rt_fail(RT_ERR_ARG, "rt_render_tile: NULL argument");
  if (tile_x < 0 || tile_y < 0 || tile_w < 1 || tile_h < 1 || tile_x + tile_w > W || tile_y + tile_h > H)
    return rt_fail(RT_ERR_ARG, "rt_render_tile: tile outside the image");
  const TileSpec t = {tile_x, tile_y, tile_w, tile_h, dev_fb, 0};
  return render_common(c, W, H, depth, H, 0, 1, nullptr, nullptr, nullptr, stream ? (cudaStream_t)stream : c->stream, nullptr, &t);
}

extern "C" int rt_render_bands(rt_ctx *c, int W, int H, int depth, int band_h, int rank, int nranks, void *dev_rgb,
                               void *stream, rt_stats *stats) {
  if (!c || !dev_rgb) return rt_fail(RT_ERR_ARG, "rt_render_bands: NULL argument");
  cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
  auto t0 = std::chrono::steady_clock::now();
  int rc = render_common(c, W, H, depth, band_h, rank, nranks, (uint8_t *)dev_rgb, nullptr, nullptr, s, stats);
  if (rc == RT_OK && stats)
    stats->ms_host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

// As rt_render_bands, but the rows this rank owns are stored at their IMAGE positions of an assembled H x W x 3 frame:
// dev_frame may be memory of this GPU or peer-mapped memory of another GPU of the box (rt_ipc_open), so that the ranks'
// kernels write rank 0's frame directly over NVLink and no gather / de-interleave step is left.
extern "C" int rt_render_bands_frame(rt_ctx *c, int W, int H, int depth, int band_h, int rank, int nranks, void *dev_frame,
                                     void *stream, rt_stats *stats) {
  if (!c || !dev_frame) return rt_fail(RT_ERR_ARG, "rt_render_bands_frame: NULL argument");
  const TileSpec t = {0, 0, 0, 0, nullptr, 1};
  return render_common(c, W, H, depth, band_h, rank, nranks, (uint8_t *)dev_frame, nullptr, nullptr,
                       stream ? (cudaStream_t)stream : c->stream, stats, &t);
}

// ---- device memory that can be shared between the processes of one box (one process per GPU) ----------------------
extern "C" int rt_dev_alloc(rt_ctx *c, size_t bytes, void **out) {
  if (!c || !out || bytes == 0) return rt_fail(RT_ERR_ARG, "rt_dev_alloc: bad argument");
  RT_CUDA(cudaSetDevice(c->device));
  RT_CUDA(cudaMalloc(out, bytes));
  RT_CUDA(cudaMemset(*out, 0, bytes));
  return RT_OK;
}
extern "C" int rt_dev_free(rt_ctx *c, void *p) {
  if (!c) return rt_fail(RT_ERR_ARG, "rt_dev_free: NULL ctx");
  RT_CUDA(cudaSetDevice(c->device));
  RT_CUDA(cudaFree(p));
  return RT_OK;
}
extern "C" int rt_ipc_export(rt_ctx *c, void *dev_ptr, unsigned char handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  if (!c || !dev_ptr || !handle) return rt_fail(RT_ERR_ARG, "rt_ipc_export: NULL argument");
  RT_CUDA(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  RT_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
  memcpy(handle, &h, 64);
  return RT_OK;
}
extern "C" int rt_ipc_open(rt_ctx *c, const unsigned char handle[64], void **out) {
  if (!c || !handle || !out) return rt_fail(RT_ERR_ARG, "rt_ipc_open: NULL argument");
  RT_CUDA(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  RT_CUDA(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
  return RT_OK;
}
extern "C" int rt_ipc_close(rt_ctx *c, void *p) {
  if (!c) return rt_fail(RT_ERR_ARG, "rt_ipc_close: NULL ctx");
  RT_CUDA(cudaSetDevice(c->device));
  RT_CUDA(cudaIpcCloseMemHandle(p));
  return RT_OK;
}
extern "C" int rt_peer_signal(rt_ctx *c, uint32_t *flag, uint32_t value, void *stream) {
  if (!c || !flag) return rt_fail(RT_ERR_ARG, "rt_peer_signal: NULL argument");
  RT_CUDA(cudaSetDevice(c->device));
  const int r = rtk_peer_signal(flag, value, stream ? (cudaStream_t)stream : c->stream);
  return r < 0 ? rt_fail(RT_ERR_CUDA, std::string("rt_peer_signal: ") + cudaGetErrorString((cudaError_t)-r)) : RT_OK;
}
extern "C" int rt_peer_wait(rt_ctx *c, uint32_t *flags, int n, uint32_t value, uint32_t *dev_err, void *stream) {
  if (!c || !flags || !dev_err || n < 1 || n > 64) return rt_fail(RT_ERR_ARG, "rt_peer_wait: bad argument");
  RT_CUDA(cudaSetDevice(c->device));
  const int r = rtk_peer_wait(flags, n, value, dev_err, stream ? (cudaStream_t)stream : c->stream);
  return r < 0 ? rt_fail(RT_ERR_CUDA, std::string("rt_peer_wait: ") + cudaGetErrorString((cudaError_t)-r)) : RT_OK;
}

extern "C" int rt_render_debug(rt_ctx *c, int W, int H, int depth, uint8_t *host_rgb, int32_t *hit_idx,
                               uint32_t *shadow_mask, rt_stats *stats) {
  if (!c || !host_rgb) return rt_fail(RT_ERR_ARG, "rt_render: NULL argument");
  if (W < 1 || H < 1 || depth < 0) return rt_fail(RT_ERR_ARG, "rt_render: bad image size or depth");
  auto t0 = std::chrono::steady_clock::now();
  RT_CUDA(cudaSetDevice(c->device));
  const size_t npx = (size_t)W * H;
  int rc = ensure_cap(c->d_rgb, c->rgb_cap, npx * 3 + 16);
  if (rc) return rc;
  // debug buffers are per SAMPLE when supersampling is on: [2H][2W][depth]
  const size_t nlev = npx * (size_t)(c->antialias ? 4 : 1) * (size_t)(depth > 0 ? depth : 1);
  if (hit_idx && (rc = ensure_cap(c->d_hit, c->hit_cap, nlev))) return rc;
  if (shadow_mask && (rc = ensure_cap(c->d_mask, c->mask_cap, nlev))) return rc;
  rc = render_common(c, W, H, depth, H, 0, 1, c->d_rgb, hit_idx ? c->d_hit : nullptr,
                     shadow_mask ? c->d_mask : nullptr, c->stream, stats);
  if (rc) return rc;
  RT_CUDA(cudaMemcpyAsync(host_rgb, c->d_rgb, npx * 3, cudaMemcpyDeviceToHost, c->stream));
  if (hit_idx && depth > 0) RT_CUDA(cudaMemcpyAsync(hit_idx, c->d_hit, nlev * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  if (shadow_mask && depth > 0) RT_CUDA(cudaMemcpyAsync(shadow_mask, c->d_mask, nlev * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  RT_CUDA(cudaStreamSynchronize(c->stream));
  if (stats) stats->ms_host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return RT_OK;
}

extern "C" int rt_render(rt_ctx *c, int W, int H, int depth, uint8_t *host_rgb, rt_stats *stats) {
  return rt_render_debug(c, W, H, depth, host_rgb, nullptr, nullptr, stats);
}

// Pinned host memory for callers that want the frame copy to run at full PCIe rate.
extern "C" int rt_host_alloc(size_t bytes, void **out) {
  if (!out || bytes == 0) return rt_fail(RT_ERR_ARG, "rt_host_alloc: bad argument");
  RT_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return RT_OK;
}
extern "C" void rt_host_free(void *p) { if (p) cudaFreeHost(p); }

// FP32 FFMA issue peak of the device, measured live: the roofline denominator of bench.py.
extern "C" int rt_measure_fp32_peak(int device, double *flops_per_s, double *sm_clock_mhz) {
  if (!flops_per_s) return rt_fail(RT_ERR_ARG, "rt_measure_fp32_peak: NULL argument");
  if (rt_device_count() <= device || device < 0) return rt_fail(RT_ERR_CUDA, "rt_measure_fp32_peak: no such CUDA device");
  double v = rtk_measure_fp32_peak(device, sm_clock_mhz);
  if (v < 0) return rt_fail(RT_ERR_CUDA, "rt_measure_fp32_peak: probe kernel failed");
  *flops_per_s = v;
  return RT_OK;
}

// ------------------------------------------------------------------------------------------
// Multi-GPU frame in ONE process (SURVEY 8b: "rt_create(int ngpus, ...): the ctx owns devices, streams and comms").
// rank r of n renders the interleaved row bands b with b % n == r (SURVEY 8e) on its own device and stream, compactly,
// and copies them -- every rank over ITS OWN host link, all ranks concurrently -- to their image positions of the
// caller's host frame: a band is band_h consecutive rows = one contiguous run both in the rank's compact buffer and in
// the frame, so the whole share of a rank is ONE strided copy (cudaMemcpy2DAsync; + one for a ragged last band).
// Nothing crosses between the GPUs: for a frame that ends in host memory the gather of 8e is the host frame itself.
// One rank's share of a frame that ends in HOST memory: renders the bands b with b % nranks == rank compactly into the
// ctx's own device buffer and enqueues their copies to their image positions in host_rgb on the ctx stream.  A band is
// band_h consecutive rows = one contiguous run both in the compact buffer and in the frame, so the full bands of a rank
// are ONE strided copy (cudaMemcpy2DAsync), a ragged last band (H % band_h rows) one more.  Does not wait.
static int enqueue_bands_to_host(rt_ctx *c, int W, int H, int depth, int band_h, int rank, int nranks, uint8_t *host_rgb, rt_stats *stats) {
  const size_t row_bytes = (size_t)W * 3, band_bytes = row_bytes * (size_t)band_h;
  const int rows = rt_band_rows(H, band_h, rank, nranks);
  if (rows < 0) return rows;
  RT_CUDA(cudaSetDevice(c->device));
  int rc = ensure_cap(c->d_part, c->part_cap, (size_t)(rows > 0 ? rows : 1) * row_bytes + 16);
  if (rc) return rc;
  rc = render_common(c, W, H, depth, band_h, rank, nranks, c->d_part, nullptr, nullptr, c->stream, stats, nullptr, true);
  if (rc) return rc;
  if (rows == 0) return RT_OK;
  const int nb_all = (H + band_h - 1) / band_h;
  int nb = 0, nfull = 0;
  for (int b = rank; b < nb_all; b += nranks) { nb++; if ((b + 1) * band_h <= H) nfull++; }
  if (nfull > 0)
    RT_CUDA(cudaMemcpy2DAsync(host_rgb + (size_t)rank * band_bytes, (size_t)nranks * band_bytes, c->d_part, band_bytes, band_bytes, (size_t)nfull,
                              cudaMemcpyDeviceToHost, c->stream));
  if (nb > nfull) {
    const int b = rank + nfull * nranks, tail_rows = H - b * band_h;
    RT_CUDA(cudaMemcpyAsync(host_rgb + (size_t)b * band_bytes, c->d_part + (size_t)nfull * band_bytes, (size_t)tail_rows * row_bytes,
                            cudaMemcpyDeviceToHost, c->stream));
  }
  return RT_OK;
}

// One process per GPU (torchrun): every rank calls this with the SAME host frame -- shared memory that each process has
// page-locked (rt_host_register) -- and its own (rank, nranks).  Every rank's bands travel over its own host link, all
// ranks concurrently; nothing crosses between the GPUs.  Returns when this rank's rows have landed.
extern "C" int rt_render_bands_host(rt_ctx *c, int W, int H, int depth, int band_h, int rank, int nranks, uint8_t *host_rgb, rt_stats *stats) {
  if (!c || !host_rgb) return rt_fail(RT_ERR_ARG, "rt_render_bands_host: NULL argument");
  if (W < 1 || H < 1 || depth < 0 || band_h < 1) return rt_fail(RT_ERR_ARG, "rt_render_bands_host: bad image size, depth or band height");
  auto t0 = std::chrono::steady_clock::now();
  int rc = enqueue_bands_to_host(c, W, H, depth, band_h, rank, nranks, host_rgb, stats);
  if (rc) return rc;
  if (stats && (rc = collect_stats(c, stats))) return rc;
  RT_CUDA(cudaStreamSynchronize(c->stream));
  if (stats) stats->ms_host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return RT_OK;
}

// Page-locks memory the caller allocated (e.g. a POSIX shared-memory frame) so that device -> host copies into it are
// asynchronous and run at full link rate; portable across the contexts of the process.
extern "C" int rt_host_register(void *p, size_t bytes) {
  if (!p || bytes == 0) return rt_fail(RT_ERR_ARG, "rt_host_register: bad argument");
  RT_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  return RT_OK;
}
extern "C" int rt_host_unregister(void *p) {
  if (!p) return rt_fail(RT_ERR_ARG, "rt_host_unregister: NULL argument");
  RT_CUDA(cudaHostUnregister(p));
  return RT_OK;
}

struct rt_multi {
  int n = 0;
  std::vector<rt_ctx *> ctx;
  void *registered = nullptr; size_t registered_bytes = 0;   // host frame pinned by us (cudaHostRegister) for async copies
  // rt_multi_render_path: ev_in on rank 0's device (the caller's stream at the call), ev_done[r] on rank r's device (its
  // last frame copy)
  cudaEvent_t ev_in = nullptr;
  std::vector<cudaEvent_t> ev_done;
};

extern "C" void rt_multi_destroy(rt_multi *m) {
  if (!m) return;
  for (int r = 0; r < (int)m->ctx.size(); r++) {
    if (!m->ctx[r]) continue;
    cudaSetDevice(m->ctx[r]->device);
    cudaStreamSynchronize(m->ctx[r]->stream);
    if (r < (int)m->ev_done.size() && m->ev_done[r]) cudaEventDestroy(m->ev_done[r]);
    if (r == 0 && m->ev_in) cudaEventDestroy(m->ev_in);
    rt_destroy(m->ctx[r]);
  }
  if (m->registered) cudaHostUnregister(m->registered);
  cudaGetLastError();
  delete m;
}

extern "C" int rt_create_multi(int ngpus, rt_multi **out) {
  if (!out || ngpus < 1 || ngpus > 64) return rt_fail(RT_ERR_ARG, "rt_create_multi: bad argument (1 <= ngpus <= 64)");
  const int ndev = rt_device_count();
  if (ndev == 0) return rt_fail(RT_ERR_CUDA, "rt_create_multi: no CUDA device (this library has no CPU fallback)");
  rt_multi *m = new (std::nothrow) rt_multi();
  if (!m) return rt_fail(RT_ERR_NOMEM, "rt_create_multi: out of memory");
  m->n = ngpus;
  m->ctx.assign((size_t)ngpus, nullptr);
  m->ev_done.assign((size_t)ngpus, nullptr);
  for (int r = 0; r < ngpus; r++) {
    // more ranks than devices: ranks share devices round robin (same frame, no speed-up) -- lets a 1-GPU box run the
    // N-rank code path
    const int rc = rt_create(r % ndev, &m->ctx[r]);
    if (rc != RT_OK) { const std::string msg = g_last_error; rt_multi_destroy(m); return rt_fail(rc, msg); }
    // (rt_create left the rank's device current)
    cudaError_t e = cudaEventCreateWithFlags(&m->ev_done[r], cudaEventDisableTiming);
    if (e == cudaSuccess && r == 0) e = cudaEventCreateWithFlags(&m->ev_in, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      rt_multi_destroy(m);
      return rt_fail(RT_ERR_CUDA, std::string("rt_create_multi: ") + cudaGetErrorString(e));
    }
  }
  *out = m;
  return RT_OK;
}

extern "C" int rt_multi_ranks(const rt_multi *m) { return m ? m->n : 0; }
extern "C" rt_ctx *rt_multi_ctx(rt_multi *m, int rank) { return (m && rank >= 0 && rank < m->n) ? m->ctx[rank] : nullptr; }

extern "C" int rt_multi_set_option(rt_multi *m, const char *key, long long value) {
  if (!m) return rt_fail(RT_ERR_ARG, "rt_multi_set_option: NULL argument");
  for (int r = 0; r < m->n; r++) { const int rc = rt_set_option(m->ctx[r], key, value); if (rc != RT_OK) return rc; }
  return RT_OK;
}

extern "C" int rt_multi_upload_scene(rt_multi *m, const double *spheres, int N, const double *lights, int L,
                                     const double ambient[3], const double cam_pos[3], const double cam_look[3], double fov_deg) {
  if (!m) return rt_fail(RT_ERR_ARG, "rt_multi_upload_scene: NULL argument");
  // every rank holds a full scene replica (SURVEY 8e); the per-rank table builds are independent: one host thread each
  std::vector<int> rc((size_t)m->n, RT_OK);
  std::vector<std::string> msg((size_t)m->n);
  auto one = [&](int r) {
    rc[r] = rt_upload_scene(m->ctx[r], spheres, N, lights, L, ambient, cam_pos, cam_look, fov_deg);
    if (rc[r] != RT_OK) msg[r] = g_last_error;          // (thread local: copy it out of the worker thread)
  };
  if (m->n == 1) one(0);
  else {
    std::vector<std::thread> th;
    for (int r = 0; r < m->n; r++) th.emplace_back(one, r);
    for (auto &t : th) t.join();
  }
  for (int r = 0; r < m->n; r++) if (rc[r] != RT_OK) return rt_fail(rc[r], msg[r]);
  return RT_OK;
}

extern "C" int rt_multi_set_camera(rt_multi *m, const double cam_pos[3], const double cam_look[3], double fov_deg) {
  if (!m || !cam_pos || !cam_look) return rt_fail(RT_ERR_ARG, "rt_multi_set_camera: NULL argument");
  for (int r = 0; r < m->n; r++) { const int rc = rt_set_camera(m->ctx[r], cam_pos, cam_look, fov_deg, nullptr); if (rc != RT_OK) return rc; }
  return RT_OK;
}

extern "C" int rt_multi_render(rt_multi *m, int W, int H, int depth, int band_h, uint8_t *host_rgb, rt_stats *stats) {
  if (!m || !host_rgb) return rt_fail(RT_ERR_ARG, "rt_multi_render: NULL argument");
  if (W < 1 || H < 1 || depth < 0 || band_h < 1) return rt_fail(RT_ERR_ARG, "rt_multi_render: bad image size, depth or band height");
  auto t0 = std::chrono::steady_clock::now();
  const int n = m->n;
  const size_t row_bytes = (size_t)W * 3;
  // asynchronous device -> host copies need page-locked memory: pin the caller's frame once (kept while it stays the same
  // buffer); a frame that is already pinned (rt_host_alloc) reports cudaErrorHostMemoryAlreadyRegistered -- fine
  if (n > 1 && (m->registered != host_rgb || m->registered_bytes != row_bytes * H)) {
    if (m->registered) { cudaHostUnregister(m->registered); m->registered = nullptr; }
    const cudaError_t e = cudaHostRegister(host_rgb, row_bytes * H, cudaHostRegisterPortable);
    if (e == cudaSuccess) { m->registered = host_rgb; m->registered_bytes = row_bytes * H; }
    else cudaGetLastError();                           // already pinned, or not pinnable: the copies still work (staged)
  }
  for (int r = 0; r < n; r++) {
    const int rc = enqueue_bands_to_host(m->ctx[r], W, H, depth, band_h, r, n, host_rgb, stats);
    if (rc) return rc;
  }
  rt_stats acc;
  memset(&acc, 0, sizeof(acc));
  for (int r = 0; r < n; r++) {
    rt_ctx *c = m->ctx[r];
    RT_CUDA(cudaSetDevice(c->device));
    if (stats) {
      rt_stats s;
      const int rc = collect_stats(c, &s);
      if (rc) return rc;
      // time-like fields: the slowest rank; counters: summed (every ray of the frame is traced by exactly one rank)
      acc.ms_device = std::fmax(acc.ms_device, s.ms_device); acc.ms_level0 = std::fmax(acc.ms_level0, s.ms_level0);
      acc.ms_closest0 = std::fmax(acc.ms_closest0, s.ms_closest0); acc.ms_shadow0 = std::fmax(acc.ms_shadow0, s.ms_shadow0);
      acc.closest_queries += s.closest_queries; acc.hits += s.hits; acc.shadow_queries += s.shadow_queries; acc.occluded += s.occluded;
      for (int k = 0; k < RT_MAX_LEVELS; k++) acc.alive[k] += s.alive[k];
      acc.fp64_intersections += s.fp64_intersections; acc.sphere_tests += s.sphere_tests; acc.filter_violations += s.filter_violations;
      acc.kernel_launches += s.kernel_launches; acc.rows_rendered += s.rows_rendered;
      acc.bundle_walks += s.bundle_walks; acc.bundle_candidates += s.bundle_candidates; acc.bundle_fallbacks += s.bundle_fallbacks;
    }
    RT_CUDA(cudaStreamSynchronize(c->stream));         // also: this rank's device -> host copies have landed
  }
  if (stats) {
    *stats = acc;
    stats->ms_host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  return RT_OK;
}

// ---- a camera path frame-parallel over the ranks ---------------------------------------------------------------------
// One frame of rt_multi_render_path on rank c: rt_set_camera + a full-frame render into the ctx's own frame buffer (the
// kernels store 16-byte row segments, so they never write the caller's frames directly), then one copy to `dst` on
// rank 0's device (peer memory unless c lives there).  wait_first: the first frame of the rank waits for the caller's
// stream before its copy, so the rendering itself overlaps the caller's earlier work.
static int path_frame(rt_ctx *c, const double *cam, int W, int H, int depth, uint8_t *dst, cudaEvent_t wait_first) {
  int rc = rt_set_camera(c, cam, cam + 3, cam[6], nullptr);
  if (rc) return rc;
  const size_t bytes = (size_t)W * H * 3;
  RT_CUDA(cudaSetDevice(c->device));
  if ((rc = ensure_cap(c->d_rgb, c->rgb_cap, bytes + 16))) return rc;
  if ((rc = render_common(c, W, H, depth, H, 0, 1, c->d_rgb, nullptr, nullptr, c->stream, nullptr))) return rc;
  if (wait_first) RT_CUDA(cudaStreamWaitEvent(c->stream, wait_first, 0));
  RT_CUDA(cudaMemcpyAsync(dst, c->d_rgb, bytes, cudaMemcpyDeviceToDevice, c->stream));
  return RT_OK;
}

extern "C" int rt_multi_render_path(rt_multi *m, const double *cameras, int K, int W, int H, int depth, void *dev_frames,
                                    void *stream) {
  if (!m || !cameras || !dev_frames) return rt_fail(RT_ERR_ARG, "rt_multi_render_path: NULL argument");
  if (K < 1 || W < 1 || H < 1 || depth < 0) return rt_fail(RT_ERR_ARG, "rt_multi_render_path: bad frame count, image size or depth");
  const int n = m->n, dev0 = m->ctx[0]->device;
  for (int r = 0; r < n; r++)
    if (!m->ctx[r]->have_scene) return rt_fail(RT_ERR_STATE, "rt_multi_render_path: no scene uploaded (call rt_multi_upload_scene first)");
  cudaPointerAttributes pa;
  RT_CUDA(cudaPointerGetAttributes(&pa, dev_frames));
  if (pa.type != cudaMemoryTypeDevice || pa.device != dev0)
    return rt_fail(RT_ERR_ARG, "rt_multi_render_path: dev_frames must be device memory of rank 0's device " + std::to_string(dev0));
  // the devices in rank order; ranks that share a device are enqueued by one thread, because the device's __constant__
  // bank changes hands between its contexts in the order their renders are enqueued (render_common), which needs one order
  std::vector<int> devs;
  for (int r = 0; r < n; r++) {
    const int d = m->ctx[r]->device;
    bool seen = false;
    for (int x : devs) seen |= x == d;
    if (seen) continue;
    devs.push_back(d);
    if (d == dev0) continue;
    // the ranks copy their frames into rank 0's memory: peer access, enabled on demand; no staging through the host
    int can = 0;
    RT_CUDA(cudaDeviceCanAccessPeer(&can, d, dev0));
    if (!can)
      return rt_fail(RT_ERR_UNSUPPORTED, "rt_multi_render_path: device " + std::to_string(d) + " has no peer access to device " +
                                             std::to_string(dev0));
    RT_CUDA(cudaSetDevice(d));
    const cudaError_t e = cudaDeviceEnablePeerAccess(dev0, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
    else if (e != cudaSuccess) return rt_fail(RT_ERR_CUDA, std::string("rt_multi_render_path: cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
  }
  const cudaStream_t s0 = stream ? (cudaStream_t)stream : m->ctx[0]->stream;
  RT_CUDA(cudaSetDevice(dev0));
  RT_CUDA(cudaEventRecord(m->ev_in, s0));

  const size_t bytes = (size_t)W * H * 3;
  const double *last = cameras + (size_t)(K - 1) * 7;
  std::vector<int> rc((size_t)n, RT_OK);
  std::vector<std::string> msg((size_t)n);
  std::vector<char> wrote((size_t)n, 0);              // the rank's stream waited for ev_in: `stream` must wait for it
  auto one_device = [&](int dev) {
    int bad = -1, e = RT_OK;
    for (int k = 0; k < K && e == RT_OK; k++) {       // rank k % n renders frame k
      const int r = k % n;
      if (m->ctx[r]->device != dev) continue;
      const bool first = !wrote[r];
      wrote[r] = 1;
      e = path_frame(m->ctx[r], cameras + (size_t)k * 7, W, H, depth, (uint8_t *)dev_frames + (size_t)k * bytes,
                     first ? m->ev_in : nullptr);
      if (e != RT_OK) bad = r;
    }
    for (int r = 0; r < n; r++) {
      if (m->ctx[r]->device != dev) continue;
      if (wrote[r]) {                                 // (also after a failure: `stream` waits for whatever was enqueued)
        const cudaError_t ce = cudaEventRecord(m->ev_done[r], m->ctx[r]->stream);
        if (ce != cudaSuccess && e == RT_OK) { e = rt_fail(RT_ERR_CUDA, std::string("rt_multi_render_path: cudaEventRecord: ") + cudaGetErrorString(ce)); bad = r; }
      }
      // every rank ends on the last camera, as Renderer.render_path does
      if (e == RT_OK && r != (K - 1) % n && (e = rt_set_camera(m->ctx[r], last, last + 3, last[6], nullptr)) != RT_OK) bad = r;
    }
    if (bad >= 0) { rc[bad] = e; msg[bad] = g_last_error; }   // (thread local: copy it out of the worker thread)
  };
  if (devs.size() == 1) one_device(devs[0]);
  else {
    std::vector<std::thread> th;
    for (int d : devs) th.emplace_back(one_device, d);
    for (auto &t : th) t.join();
  }
  // `stream` waits on the device for every frame copy; also after a failure, so that no copy outlives the caller's buffer
  RT_CUDA(cudaSetDevice(dev0));
  for (int r = 0; r < n; r++)
    if (wrote[r]) RT_CUDA(cudaStreamWaitEvent(s0, m->ev_done[r], 0));
  for (int r = 0; r < n; r++) if (rc[r] != RT_OK) return rt_fail(rc[r], msg[r]);
  return RT_OK;
}
