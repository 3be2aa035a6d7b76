// rt_kernels.h -- host-callable launchers implemented in rt_kernels.cu.
#ifndef RT_KERNELS_H
#define RT_KERNELS_H

#include <cuda_runtime.h>

#include "rt_device.h"

// Copies the frame constants into this device's __constant__ bank (async on `stream`).
cudaError_t rtk_set_frame_const(const RtFrameConst *host_const, cudaStream_t stream);

// mode 1: exact FP64 brute force.  Returns the number of kernels launched (or <0: -cudaError).
int rtk_launch_exact(const RtRenderArgs &args, cudaStream_t stream);

// mode 0: FP32-filter fast path (kernels_fast.cuh).
struct RtFastScene {
  int N, L, npairs, ngroups;
  void *tabs;             // device: (1+L) shared-origin tables (pairs | gmin | perm), then the general table
  size_t tabs_cap;        // bytes allocated behind tabs (reused by the next upload when large enough)
  // the exact geometry / materials live in the same device arena, behind the tables: ONE pinned staging buffer and ONE
  // host->device copy per upload
  void *sph64, *mat, *matx;   // device: N x double4, N x float4, N x float2
  void *h_stage; size_t h_stage_cap;   // pinned host staging of the whole arena
  void *raw_dev; size_t raw_cap;       // large LBVH scenes: the raw sphere rows on the device (tables are built there)
  unsigned tstride;       // bytes per shared-origin table
  unsigned gmin_off, perm_off, inv_off, cullA_off, cullB_off;
  size_t bytes_primary;   // staged by k_primary: (1+L) * tstride
  size_t bytes_bounce;    // staged by k_bounce : L * tstride + npairs * 32
  float d64;              // absolute FP64/geometry slack (delta64)
  float gS2;              // squared radius bound of the recentred scene
  float g_dtmax;          // additive bound of the general filter's centre projection
  unsigned long long generation;   // bumped by every rtk_fast_build_scene
  double c0[3];           // recentring offset of the general table
  // device-built LBVH over the recentred spheres (bvh.cuh); built when the scene has >= bvh_min spheres
  void *bvh_nodes, *bvh_leaves;   // bvh_nodes = bvh_nodes_buf when the current scene has a hierarchy, else NULL
  void *bvh_nodes_buf, *bvh_scratch;   // grow-only allocations kept across uploads
  size_t bvh_nodes_cap, bvh_scratch_cap;
  int bvh_nleaf;
  int nbig, big[8];       // spheres kept out of the LBVH because their boxes would cover most of it
  double bvh_build_ms;    // device time of the build
  // camera moves without a re-upload (rtk_fast_camera_table): what the upload decided and kept for it
  double sabs_scene;      // magnitude bound of the lights and spheres, without the camera
  double delta64;         // the slack the tables were built with (fs->d64 is its float rounding)
  int lookup_only, device_build;   // table layout: index-order lookup tables (LBVH scenes); written by k_build_lookup
  void *geo;              // device, inside the arena: N x double4 (cx, cy, cz, r); NULL when device_build (raw_dev)
  void *cam_scratch; size_t cam_scratch_cap;   // sort scratch of the camera table (sorted layouts), grow-only
};
struct RtFastWork {
  int num_sms;
  int wave_levels;       // reflection levels run as wavefront kernels before the fused tail (0 = automatic)
  // automatic choice: the per-level ray counts of the previous frame of the same (scene, size, depth) are read back
  // asynchronously (136 bytes) and decide where the next frame switches from wavefront levels to the tail
  unsigned int *h_fb;    // pinned: rays entering level k of the frame the read-back was taken from
  cudaEvent_t fb_event;
  int fb_pending, fb_levels;
  unsigned long long fb_key, fb_pending_key;
  void *queue[2];        // reflected-ray records, ping-pong between levels
  size_t queue_cap;      // records per queue
  unsigned int *ctl;     // device control words (zeroed before every frame): tile counter, per-level chunk counters, queue counts
  unsigned int *last_err; // device: error word of the last frame launched (bounds guards)
  void *hits;            // HitRec queue of the current level (kernels_wave.cuh), 64-slot blocks
  unsigned int *hit_n;   // hits per block
  void *cand;            // LBVH scenes: closest-hit candidate per queued ray (k_closest1_dyn -> k_closest1)
  size_t cand_cap;
  unsigned char *occ;    // [L][hit_cap] occlusion bytes of the current level
  size_t hit_cap, occ_bytes;
  unsigned int *tile_ray; // per level-0 tile: its reflected rays, then their first position in the level-1 queue
  size_t tile_cap;
};
int rtk_fast_init(int device);
// accel: 0 = automatic (LBVH from kBvhAutoSpheres spheres), 1 = table walks only, 2 = LBVH whenever N > 0
int rtk_fast_build_scene(RtFastScene *fs, const double *spheres, int N, const RtFrameConst *frame, int accel, cudaStream_t stream);
void rtk_fast_free_scene(RtFastScene *fs, int release_tables);   // release_tables = 0: keep the table allocation
// delta64 of a scene whose lights and spheres have the magnitude bound sabs_scene, seen from cam_pos
double rtk_delta64(double sabs_scene, const double cam_pos[3]);
// Rewrites table 0 (the camera's shared-origin table) in place for a new camera position, on the device, asynchronously
// on `stream`; the bytes equal those rtk_fast_build_scene writes for that camera as long as rtk_delta64 is unchanged.
// Plain launches (no programmatic dependent launch): the next render's k_closest0 starts after the last of them.
int rtk_fast_camera_table(RtFastScene *fs, const double cam_pos[3], cudaStream_t stream);
// su[0..nu) / sv[0..nv): the camera-plane coordinates of ensure_tables (rt_api.cu), computed on the device.
int rtk_camera_plane(double *su, int nu, double *sv, int nv, int m, int W, int H, double scale, cudaStream_t stream);
void rtk_fast_free_work(RtFastWork *w);
int rtk_fast_last_error(const RtFastWork *w, unsigned int *word);
// marks (may be null): 3 events recorded after the level-0 closest-hit, shadow and shade kernels.
int rtk_launch_fast(const RtRenderArgs &args, const RtFastScene *fs, RtFastWork *w, cudaStream_t stream,
                    const cudaEvent_t *marks);

// Completion signalling of the peer-memory frame assembly (flags live in rank 0's memory, n <= 64).
int rtk_peer_signal(unsigned int *flag, unsigned int value, cudaStream_t stream);
int rtk_peer_wait(unsigned int *flags, int n, unsigned int value, unsigned int *err, cudaStream_t stream);

// 2x2 supersampling resolve: float sample frame (2W x 2rows) -> 8-bit rows x W.
int rtk_resolve_aa(const float *fb, int W, int rows, uint8_t *rgb, cudaStream_t stream);

// FP32 FFMA issue peak of `device`, measured live (FLOP/s); used by bench.py as the roofline
// denominator because MEASURED_PEAKS.json carries no FP32 entry.  Returns <0: -cudaError.
double rtk_measure_fp32_peak(int device, double *sm_clock_mhz);

#endif
