// kernels_wave.cuh -- the phase-separated wavefront used for reflection levels 0 and 1 (every level in LBVH scenes).
//
// Profiling a fused per-warp pipeline (one kernel per level) showed that the packed FP32 sphere
// loops were only ~30 % of its time: the rest was FP64 geometry, shading and slow-path code that
// is latency bound at 16 warps/SM and too large for the instruction cache.  Here every phase is its
// own kernel and every warp is full because each phase consumes a COMPACTED queue:
//
//   k_closest0   pixels      -> camera-table walk -> exact t -> hit point / normal -> HitRec block
//                               (sky pixels are final: staged per warp, 128-bit stores)
//   k_closest1   RayRec queue-> general-origin loop -> same, for reflected rays (misses are final)
//   k_shadow     HitRec blocks (two hits per lane) x lights -> light-table walk -> one occlusion bit per (light, hit)
//                               in the hit's record (a byte array when the scene has more than 32 lights)
//   k_shade      HitRec      -> Phong (include/scene.h:89-121) -> final pixel, or the reflected
//                               ray appended to the RayRec queue (warp-ballot compaction)
// Where the candidate spheres of a query come from is the template mode of k_closest0 / k_shadow (kTab*): a bundle-culled
// table staged in shared memory, a table streamed through a ring of TMA tiles, or the LBVH (bundle traversal at level 0;
// k_closest1_dyn / k_shadow_dyn -- per-ray traversal with dynamic ray fetch -- from level 1 on).
// Levels >= 2 of small scenes hold a few percent of the rays; they run in the fused tail kernel of
// kernels_fast.cuh (k_bounce), one launch for all remaining levels.  Every kernel but the first of a frame is launched with
// programmatic dependent launch (RT_PDL_SYNC).
#ifndef RT_KERNELS_WAVE_CUH
#define RT_KERNELS_WAVE_CUH

#include <type_traits>

#include "kernels_fast.cuh"

namespace rtf {

// A camera-ray hit (level 0) has no queue record, carries weight 1 and no colour yet: there the words of (vy, vz), (src, wt)
// and (ar, ag) hold the EXACT unit direction of the camera ray as three doubles (finish_hit / hit_d0x..z: k_closest0 has it;
// the shading pass would otherwise redo its two FP64 normalisations for every hit that reflects); view direction = -(float)d0.
// The word of vx holds, for a camera-ray hit whose path continues, its rank among the reflected rays of its 16x4 tile in
// slot order (k_closest0): k_shade stores the reflected ray at the tile's offset + rank (tile-ordered level-1 queue).
// (Plain fields and register-level bit casts, not a union: the record keeps moving as five 128-bit words.)
struct __align__(16) HitRec {      // 80 bytes
  double px, py, pz;               // exact FP64 hit point (src/main.cpp:32)
  float nx, ny, nz;                // unit normal, FP32 (colour + lit-side test only)
  float vx, vy, vz;                // view direction = -ray direction, FP32 (colour only; level >= 1)
  int idx;                         // sphere index
  unsigned pix;                    // local pixel index lr*W + x
  unsigned src;                    // level >= 1: index of the ray in the level's RayRec queue
  float wt, ar, ag, ab;            // carried weight / colour (front to back)
  unsigned pad;                    // occlusion bits of the hit's shadow queries (bit l = light l occluded; scenes with <= 32 lights)
};
__device__ __forceinline__ double hit_d0x(const HitRec &h) { return __hiloint2double(__float_as_int(h.vz), __float_as_int(h.vy)); }
__device__ __forceinline__ double hit_d0y(const HitRec &h) { return __hiloint2double(__float_as_int(h.wt), (int)h.src); }
__device__ __forceinline__ double hit_d0z(const HitRec &h) { return __hiloint2double(__float_as_int(h.ag), __float_as_int(h.ar)); }
__device__ __forceinline__ unsigned hit_ray_rank(const HitRec &h) { return __float_as_uint(h.vx); }
static_assert(sizeof(HitRec) == 80, "hit record layout");

struct WaveArgs {
  FastArgs f;
  // Blocked hit queue: the hits of one warp work item (a 16x4 tile / 64 queued rays) occupy ONE 64-slot block,
  // compacted to its front, so that the bundle of shadow rays a warp handles later stays spatially coherent.
  HitRec *hits; unsigned int *hit_count;   // *hit_count = 64 x blocks in use
  unsigned int *hit_n;             // hits per block
  unsigned hit_cap;                // slots
  unsigned char *occ;              // [L][hit_cap] occlusion bytes (scenes with more than 32 lights)
  int occ_bits;                    // <= 32 lights: the occlusion bits travel in the hit record itself (HitRec::pad): one word
                                   // written by the shadow pass, read with the record by the shading pass
  unsigned int *work_counter;      // per-launch chunk counter
  Best *cand;                      // LBVH scenes, level >= 1: per queued ray, the closest-hit candidate k_closest1_dyn found
  unsigned int *work_counter2;     // ... and that kernel's item counter
  // per level-0 tile (tile order): the number of its reflected rays (written by k_closest0 for every tile, so never
  // cleared), turned in place into the position of its first ray in the level-1 queue by CTA 0 of the level-0 k_shadow
  unsigned int *tile_ray;
};

// Control words (u32) of one frame: [0] tile counter, [5] error word; per level k <= 33: tail chunk counter, shadow /
// shade / closest work counters, hits of level k (x64: blocks in use), rays entering level k
enum { CTL_TILE = 0, CTL_ERR = 5, CTL_TAIL = 8, CTL_SHADOW = 48, CTL_SHADE = 88, CTL_CLOSEST = 128, CTL_HITS = 168, CTL_RAYS = 208,
       CTL_WORDS = 256 };

// Allocates the block of a work item with (m0, m1) = ballots of its candidate hits; slot[r] = where this
// lane's hit r goes.  One atomic per work item.
__device__ __forceinline__ void hit_block(const WaveArgs &w, unsigned m0, unsigned m1, unsigned (&slot)[2]) {
  const int lane = threadIdx.x & 31;
  const unsigned n = (unsigned)(__popc(m0) + __popc(m1));
  unsigned base = 0;
  if (n != 0u) {
    if (lane == 0) {
      base = atomicAdd(w.hit_count, 64u);
      if (base + 64u > w.hit_cap) { atomicOr(w.f.err, (unsigned)RT_GUARD_HIT_BLOCKS); base = 0u; }   // guard: never past the buffer (flagged; block 0 is sacrificed)
      w.hit_n[base >> 6] = n;
    }
    base = __shfl_sync(kFull, base, 0);
  }
  const unsigned lt = (1u << lane) - 1u;
  slot[0] = base + (unsigned)__popc(m0 & lt);
  slot[1] = base + (unsigned)__popc(m0) + (unsigned)__popc(m1 & lt);
}

// 32-bit per-thread counters, reduced once per warp at kernel end (cold path, out of line)
__device__ __noinline__ void flush_counts(unsigned long long *counters, int level, unsigned closest, unsigned hits, unsigned shadow,
                                          unsigned occluded, unsigned fp64, unsigned violations, unsigned long long n_spheres,
                                          unsigned cand = 0, unsigned walks = 0, unsigned fallbacks = 0) {
  unsigned v[6] = {closest, hits, shadow, occluded, fp64, violations};
#pragma unroll
  for (int k = 0; k < 6; k++) v[k] = __reduce_add_sync(kFull, v[k]);
  if ((threadIdx.x & 31) == 0) {
    if (v[0]) { atomicAdd(&counters[RT_CNT_CLOSEST], (unsigned long long)v[0]); if (level < 32) atomicAdd(&counters[RT_CNT_ALIVE0 + level], (unsigned long long)v[0]); }
    if (v[1]) atomicAdd(&counters[RT_CNT_HITS], (unsigned long long)v[1]);
    if (v[2]) atomicAdd(&counters[RT_CNT_SHADOW], (unsigned long long)v[2]);
    if (v[3]) atomicAdd(&counters[RT_CNT_OCCLUDED], (unsigned long long)v[3]);
    if (v[4]) atomicAdd(&counters[RT_CNT_FP64], (unsigned long long)v[4]);
    if (v[5]) atomicAdd(&counters[RT_CNT_VIOLATIONS], (unsigned long long)v[5]);
    if (v[0] + v[2]) atomicAdd(&counters[RT_CNT_TESTS], (unsigned long long)(v[0] + v[2]) * n_spheres);
    if (walks) { atomicAdd(&counters[RT_CNT_CAND], (unsigned long long)cand); atomicAdd(&counters[RT_CNT_WALKS], (unsigned long long)walks); }   // warp-uniform
    if (fallbacks) atomicAdd(&counters[RT_CNT_FALLBACKS], (unsigned long long)fallbacks);
  }
}

// Exact t of the winner + hit record (out of line: FP64 heavy, once per hit ray); returns the sphere hit, -1 = none
__device__ __noinline__ int finish_hit(const FastArgs &a, Best b, RaySrc src, unsigned pix, unsigned srcidx, float wt, float ar, float ag,
                                        float ab, HitRec *out, unsigned *viol, unsigned *nfp64) {
  const ExactRay e = exact_ray(src);
  double t = b.t;
  bool ok = b.exact;
  if (!ok) { (*nfp64)++; ok = exact_sphere(a.r.sph64, b.idx, e.o, e.d, e.a, t) && t < 1e20; }
  int bi = b.idx;
  if (!ok) { (*viol)++; bi = exact_bruteforce(a.r.sph64, a.N, e.o, e.d, e.a, t); }
  if (bi < 0) return -1;
  const HitGeom g = hit_geometry(a.r.sph64, bi, e.o, e.d, t);
  // (the words of the record are formed first and stored unconditionally, in order: five 128-bit stores)
  float vx = -(float)e.d.x, vy = -(float)e.d.y, vz = -(float)e.d.z;   // view_dir = -d up to rounding (src/main.cpp:38)
  if (src.rec == nullptr) {                      // camera ray: the exact direction travels with the hit (see HitRec)
    vx = 0.f; ab = 0.f;
    vy = __int_as_float(__double2loint(e.d.x)); vz = __int_as_float(__double2hiint(e.d.x));
    srcidx = (unsigned)__double2loint(e.d.y); wt = __int_as_float(__double2hiint(e.d.y));
    ar = __int_as_float(__double2loint(e.d.z)); ag = __int_as_float(__double2hiint(e.d.z));
  }
  out->px = g.p.x; out->py = g.p.y; out->pz = g.p.z;
  out->nx = g.nx; out->ny = g.ny; out->nz = g.nz;
  out->vx = vx; out->vy = vy; out->vz = vz;
  out->idx = bi; out->pix = pix; out->src = srcidx; out->wt = wt; out->ar = ar; out->ag = ag; out->ab = ab; out->pad = 0;
  return bi;
}

// ---------------------------------------------------------------------------------------------
// Table modes of the two table-walking kernels of level 0:
//   kTabSmem    the kernel's tables staged once per CTA with one TMA bulk copy (they fit)
//   kTabStream  tables larger than shared memory: every CTA streams the (sorted) table through a
//               two-stage ring of 32 KB tiles -- cp.async.bulk into stage k+1 while the eight warps
//               test their rays against stage k (full barriers = mbarriers with expect_tx, the
//               "stage is free again" edge = the CTA barrier that also votes on early termination).
enum { kTabSmem = 1, kTabStream = 2, kTabBvh = 3 };   // kTabBvh: candidates from the LBVH, tables in global memory
constexpr int kTilePairs = 1024;                                   // sphere pairs per streamed tile
constexpr unsigned kTileBytes = kTilePairs * 32u;                  // 32 KB per stage

__device__ __forceinline__ void ring_init(unsigned char *smem) {
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem);
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); }
  __syncthreads();
}
__device__ __forceinline__ float4 *ring_stage(unsigned char *smem, int st) {
  return reinterpret_cast<float4 *>(smem + kSmemHeader + (unsigned)st * kTileBytes);
}
// thread 0 only: arm the stage's barrier and start the bulk copy of `npairs_tile` pairs
__device__ __forceinline__ void ring_issue(unsigned char *smem, int st, const float4 *gsrc, int npairs_tile) {
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem) + st;
  const unsigned bytes = (unsigned)npairs_tile * 32u;
  mbar_expect_tx(bar, bytes);
  tma_bulk_g2s(ring_stage(smem, st), gsrc, bytes, bar);
}
// all threads: wait until the stage's copy has landed; phase bit per stage flips per use
__device__ __forceinline__ void ring_wait(unsigned char *smem, int st, unsigned &phase) {
  mbar_wait(reinterpret_cast<unsigned long long *>(smem) + st, (phase >> st) & 1u);
  phase ^= 1u << st;
}
// CTA-uniform work fetch (streamed kernels walk a table together, so the CTA takes 8 items at once)
__device__ __forceinline__ int cta_fetch(unsigned int *counter, unsigned char *smem) {
  int *slot = reinterpret_cast<int *>(smem + 32);
  if (threadIdx.x == 0) *slot = (int)atomicAdd(counter, 1u);
  __syncthreads();
  const int v = *slot;
  __syncthreads();
  return v;
}

// ---------------------------------------------------------------------------------------------
// LEVEL 0 closest hit: each warp pulls 16x4-pixel tiles, two vertically adjacent pixels per lane.
// Level-0 tiles that contain hits are written ONCE, as whole 16-byte row segments, by the shading pass (shade_body): it
// knows the finished hit pixels and recomputes the sky colour of the others exactly as k_closest0 would have (same FP64
// camera direction, same FP32 normalisation).  tile_path() = the output modes where that applies; k_closest0 then stores
// only tiles WITHOUT hits itself.
__device__ __forceinline__ bool tile_path(const FastArgs &a) {
  return a.r.fb == nullptr && (a.r.out_remap == 0 || a.r.out_remap == 2) && (a.r.W & 15) == 0 &&
         (reinterpret_cast<unsigned long long>(a.r.rgb) & 15ull) == 0ull && a.r.hit_idx == nullptr;
}
__device__ __forceinline__ float camera_dir_y(const FastArgs &a, int x, int j, float &fx_, float &fz_) {
  // include/camera.h:21-22 in FP64 (un-normalised), then an FP32 unit vector
  const d3 v = rtx::add(rtx::add(ldc3(g_frame.fwd), rtx::scale(ldc3(g_frame.right), a.r.su[x])), rtx::scale(ldc3(g_frame.up), a.r.sv[j]));
  const float fx = (float)v.x, fy = (float)v.y, fz = (float)v.z;
  const float inv = rsqrtf(fmaf(fz, fz, fmaf(fy, fy, fx * fx)));
  fx_ = fx * inv; fz_ = fz * inv;
  return fy * inv;
}
// sky (src/main.cpp:26-30) quantised: r | g << 8 | b << 16
__device__ __forceinline__ unsigned sky_rgb8(float dy) {
  const Rgb c = sky_colour(dy);
  return quant8(c.r) | (quant8(c.g) << 8) | (quant8(c.b) << 16);
}

// tabs: where table 0 (the camera table) is read from (shared memory when staged); wbase: the per-warp compacted tables
template <int kMode>
__device__ __forceinline__ void closest0_body(const WaveArgs &w, unsigned char *smem, const unsigned char *tabs, unsigned char *wbase) {
  const FastArgs &a = w.f;
  const bool defer_mixed = tile_path(a);             // tiles with hits are stored by the shading pass
  const Tab camg = tab_at(a.tabs, a, 0);             // global view (gmin / perm of the streamed mode)
  const Tab cam = tab_at(tabs, a, 0);
  const WarpBuf wb = warp_buf(wbase);                                                                                // kTabSmem / kTabBvh
  const BundleBuf bb = bundle_buf(smem + kSmemHeader + kWarps * kWarpBufBytes);                                      // kTabBvh only
  unsigned ring_phase = 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char *s_rgb = smem + 64 + warp * (kWTileH * kWTileW * 3);
  const int W = a.r.W, rows = a.r.bands.local_rows, depth = a.r.max_depth;
  const bool kBytes = a.r.fb == nullptr && a.r.out_remap != 1;   // 8-bit frame (compact or assembled): staged tile rows, 128-bit stores
  const bool kFrame = a.r.out_remap == 2;                        // rows go to their image positions (maybe in a peer GPU's memory)
  unsigned c_closest = 0, c_hits = 0, c_fp64 = 0, c_viol = 0, c_cand = 0, c_walks = 0, c_fall = 0;
  for (;;) {
    int tile;
    if (kMode == kTabStream) {
      const int ct = cta_fetch(a.tile_counter, smem);
      if (ct * kWarps >= a.nwtiles) break;
      tile = ct * kWarps + warp;
    } else {
      tile = warp_fetch(a.tile_counter);
      if (tile >= a.nwtiles) break;
    }
    const bool tile_ok = tile < a.nwtiles;
    const int tx0 = (tile % a.wtiles_x) * kWTileW, ty0 = (tile / a.wtiles_x) * kWTileH;
    const int x = tx0 + (lane & 15);
    int lr[2], j[2];
    unsigned pix[2];
    bool live[2];
    float dx[2], dy[2], dz[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      lr[r] = ty0 + (lane >> 4) * 2 + r;
      live[r] = tile_ok && x < W && lr[r] < rows && depth > 0;
      j[r] = 0; pix[r] = 0; dx[r] = dy[r] = dz[r] = 0.f;
      if (tile_ok && x < W && lr[r] < rows) {
        j[r] = rt_local_to_global_row(a.r.bands, lr[r]);
        pix[r] = (unsigned)lr[r] * (unsigned)W + (unsigned)x;
      }
      if (live[r]) {
        // include/camera.h:21-22 in FP64 (un-normalised), then an FP32 unit vector for the filter
        const d3 v = rtx::add(rtx::add(ldc3(g_frame.fwd), rtx::scale(ldc3(g_frame.right), a.r.su[x])),
                              rtx::scale(ldc3(g_frame.up), a.r.sv[j[r]]));
        const float fx = (float)v.x, fy = (float)v.y, fz = (float)v.z;
        const float inv = rsqrtf(fmaf(fz, fz, fmaf(fy, fy, fx * fx)));
        dx[r] = fx * inv; dy[r] = fy * inv; dz[r] = fz * inv;
        if (a.r.hit_idx) for (int k = 0; k < depth; k++) a.r.hit_idx[(size_t)pix[r] * depth + k] = -2;
        if (a.r.shadow_mask) for (int k = 0; k < depth; k++) a.r.shadow_mask[(size_t)pix[r] * depth + k] = 0u;
      }
    }
    Best best[2];
    best_init(best[0]); best_init(best[1]);
    const RaySrc src[2] = {{a.r.su, a.r.sv, x, j[0], nullptr}, {a.r.su, a.r.sv, x, j[1], nullptr}};
    if (kMode == kTabSmem) {
      closest_shared_culled<2>(cam, a.npairs, wb, dx, dy, dz, live, a.d64, a.r.sph64, src, best, c_cand, c_walks);
    } else if (kMode == kTabBvh) {
      const float3 o = recentred(a, g_frame.cam_pos);
      // the tile's rays descend the hierarchy as ONE bundle; a per-ray traversal only if the bundle is too wide
      const Cone cone = warp_cone<2>(dx, dy, dz, live);
      bool done = false;
      // (camera tiles: the bundle walk costs about the same per tile whatever the scene size, a per-ray traversal grows
      // with it -- measured crossover between 10 k and 100 k spheres; the shadow bundles win at both sizes)
      if (cone.ok && a.N >= 32768) {
        ClosestQ<2> q;
        closest_begin(q);
        c_walks++;
        const BundleBox bx = bundle_box<2>(o, dx, dy, dz, live);
        done = bundle_traverse(a, bx, -1e-3f, 3.0e38f, bb, [&](int n) {
          c_cand += (unsigned)n;
          const int np = bundle_fill(cam, bb.cand, n, wb);
          closest_shared_range<2>(q, wb.pairs, wb.gmin, wb.perm, 0, np, dx, dy, dz, live, a.d64, a.r.sph64, src);
          __syncwarp();
          return q.wcut;
        });
        if (done) { best[0] = q.best[0]; best[1] = q.best[1]; }
      }
      if (!done) {
        c_fall++;
#pragma unroll 1
        for (int r = 0; r < 2; r++)
          if (live[r]) best[r] = bvh_closest_shared(a, cam, o, dx[r], dy[r], dz[r], src[r]);
      }
    } else {
      // the eight warps of the CTA walk the sorted camera table together, tile by tile
      ClosestQ<2> q;
      closest_begin(q);
      bool need = true;
      const int ntiles = (a.npairs + kTilePairs - 1) / kTilePairs;
      if (threadIdx.x == 0) ring_issue(smem, 0, camg.pairs, min(kTilePairs, a.npairs));
      for (int k = 0; k < ntiles; k++) {
        const int st = k & 1, p0 = k * kTilePairs, np = min(kTilePairs, a.npairs - p0);
        if (threadIdx.x == 0 && k + 1 < ntiles)
          ring_issue(smem, st ^ 1, camg.pairs + (size_t)(p0 + kTilePairs) * 2, min(kTilePairs, a.npairs - p0 - kTilePairs));
        ring_wait(smem, st, ring_phase);
        if (need) need = closest_shared_range<2>(q, ring_stage(smem, st) - (size_t)p0 * 2, camg.gmin, camg.perm, p0, p0 + np, dx, dy, dz,
                                              live, a.d64, a.r.sph64, src);
        const int more = __syncthreads_or(need ? 1 : 0);        // also: stage st is free again
        if (!more || k + 1 == ntiles) { if (k + 1 < ntiles) ring_wait(smem, st ^ 1, ring_phase); break; }
      }
      best[0] = q.best[0]; best[1] = q.best[1];
    }
    unsigned hslot[2];
    const unsigned hm0 = __ballot_sync(kFull, live[0] && best[0].idx >= 0), hm1 = __ballot_sync(kFull, live[1] && best[1].idx >= 0);
    hit_block(w, hm0, hm1, hslot);
    // a whole tile with a hit block: the shading pass stores it (tile_path)
    const bool deferred = defer_mixed && (hm0 | hm1) != 0u && tx0 + kWTileW <= W && ty0 + kWTileH <= rows;
    bool cont[2];                                    // the hit's path continues (shade_one's test): a level-1 ray
#pragma unroll
    for (int r = 0; r < 2; r++) {
      bool hit = false;
      cont[r] = false;
      if (live[r]) {
        c_closest++; c_fp64 += best[r].nfp64;
        if (best[r].idx >= 0) {
          HitRec *rec = w.hits + hslot[r];
          const int hi = finish_hit(a, best[r], src[r], pix[r], 0u, 1.0f, 0.f, 0.f, 0.f, rec, &c_viol, &c_fp64);
          hit = hi >= 0;
          if (!hit) { rec->idx = -1; rec->pix = pix[r]; }   // (filter violation resolved to a miss: dead slot)
          else cont[r] = depth > 1 && __ldg(&a.r.matx[hi]).y > 0.5f;
          if (a.r.hit_idx) a.r.hit_idx[(size_t)pix[r] * depth] = hit ? rec->idx : -1;
        } else if (a.r.hit_idx) a.r.hit_idx[(size_t)pix[r] * depth] = -1;
      }
      c_hits += hit;
      // sky (src/main.cpp:26-30) is final now; hit pixels are written by k_shade / later levels
      const Rgb skyc = sky_colour(dy[r]);
      const bool sky = live[r] && !hit;
      if (kBytes) {
        unsigned char *q = s_rgb + (((lane >> 4) * 2 + r) * kWTileW + (lane & 15)) * 3;
        q[0] = (unsigned char)quant8(sky ? skyc.r : 0.f);
        q[1] = (unsigned char)quant8(sky ? skyc.g : 0.f);
        q[2] = (unsigned char)quant8(sky ? skyc.b : 0.f);
      } else if (sky) {
        write_final(a.r, pix[r], skyc.r, skyc.g, skyc.b);
      }
    }
    {
      // the tile's reflected rays: their count, and each one's rank in slot order (hit_block: the r = 0 hits, then r = 1)
      const unsigned k0 = __ballot_sync(kFull, cont[0]), k1 = __ballot_sync(kFull, cont[1]), lt = (1u << lane) - 1u;
      if (cont[0]) w.hits[hslot[0]].vx = __uint_as_float((unsigned)__popc(k0 & lt));
      if (cont[1]) w.hits[hslot[1]].vx = __uint_as_float((unsigned)(__popc(k0) + __popc(k1 & lt)));
      if (lane == 0 && tile_ok) w.tile_ray[tile] = (unsigned)(__popc(k0) + __popc(k1));
    }
    if (!kBytes) continue;                           // float / remapped output: only finished pixels are written
    __syncwarp();
    if (!tile_ok || deferred) { __syncwarp(); continue; }
    if (tx0 + kWTileW <= W && (W & 15) == 0) {
      // 3 x 16-byte stores per 48-byte row segment (src/main.cpp:84-86 quantiser applied above)
      if (lane < kWTileH * 3) {
        const int ty = lane / 3, seg = lane % 3;
        if (ty0 + ty < rows) {
          const size_t orow = kFrame ? (size_t)rt_local_to_global_row(a.r.bands, ty0 + ty) : (size_t)(ty0 + ty);
          *reinterpret_cast<uint4 *>(a.r.rgb + (orow * W + tx0) * 3 + seg * 16) =
              *reinterpret_cast<const uint4 *>(s_rgb + ty * kWTileW * 3 + seg * 16);
        }
      }
    } else {
#pragma unroll
      for (int r = 0; r < 2; r++) {
        if (x < W && lr[r] < rows) {
          const unsigned char *q = s_rgb + (((lane >> 4) * 2 + r) * kWTileW + (lane & 15)) * 3;
          unsigned char *o = a.r.rgb + (kFrame ? ((size_t)j[r] * W + x) : (size_t)pix[r]) * 3;
          o[0] = q[0]; o[1] = q[1]; o[2] = q[2];
        }
      }
    }
    __syncwarp();
  }
  if (a.r.counters) flush_counts(a.r.counters, 0, c_closest, c_hits, 0, 0, c_fp64, c_viol, (unsigned long long)a.N, c_cand, c_walks, c_fall);
}
// 2 CTAs/SM (128 registers) for the table kernels k_closest0 / k_closest1 / k_shadow: more CTAs at fewer registers spill
// and were slower (DESIGN §5d)
constexpr int kTableCtas = 2;
template <int kMode>
__global__ void __launch_bounds__(kThreads, kTableCtas) k_closest0(const WaveArgs w) {
  extern __shared__ __align__(128) unsigned char smem[];
  const FastArgs &a = w.f;
  const unsigned char *tabs = a.tabs;
  if (kMode == kTabSmem) { stage_tables(smem, a.tabs, a.stage_bytes); tabs = smem + kSmemHeader; }
  if (kMode == kTabStream) ring_init(smem);
  RT_PDL_SYNC();
  closest0_body<kMode>(w, smem, tabs, smem + kSmemHeader + (kMode == kTabBvh ? 0u : ((a.stage_bytes + 127u) & ~127u)));
}

// ---------------------------------------------------------------------------------------------
// LEVEL >= 1 closest hit: reflected rays from the RayRec queue, 64 per warp fetch, two per lane.
// gen: the general table (shared memory when staged); kCull (gen staged): bundle-culled walk, survivors listed in the
// header's per-warp staging area (unused in this kernel: kGenIds 16-bit slots of its 192 bytes)
template <bool kBvh, bool kCull = false>
__device__ __forceinline__ void closest1_body(const WaveArgs &w, const float4 *gen, unsigned char *smem) {
  const FastArgs &a = w.f;
  const unsigned nq = __ldcg(a.q_in_count);
  if (nq == 0u) return;
  const int lane = threadIdx.x & 31, depth = a.r.max_depth, level = a.level;
  unsigned c_closest = 0, c_hits = 0, c_fp64 = 0, c_viol = 0, c_cand = 0, c_walks = 0;
  const RayRec *qin = a.q_in;
  static_assert(kGenIds * 2 <= kWTileH * kWTileW * 3, "survivor list in the header's per-warp staging area");
  unsigned short *ids = kCull ? reinterpret_cast<unsigned short *>(smem + 64 + (threadIdx.x >> 5) * (kWTileH * kWTileW * 3)) : nullptr;
  // few rays (deep levels): one ray per lane, so that twice as many warps share the work
  const bool two = nq >= gridDim.x * (unsigned)kWarps * 64u * a.two_mult;
  const unsigned per = two ? 64u : 32u;
  for (;;) {
    const int chunk = warp_fetch(w.work_counter);
    if ((unsigned)chunk * per >= nq) break;
    bool live[2];
    unsigned qi[2], pix[2];
    float ox[2], oy[2], oz[2], dx[2], dy[2], dz[2], wt[2], cr[2], cg[2], cb[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      qi[r] = two ? (unsigned)chunk * 64u + 2u * lane + r : (unsigned)chunk * 32u + lane;
      live[r] = qi[r] < nq && (two || r == 0);
      ox[r] = oy[r] = oz[r] = dx[r] = dy[r] = dz[r] = 0.f; wt[r] = cr[r] = cg[r] = cb[r] = 0.f; pix[r] = 0;
      if (live[r]) {
        const RayRec &q = qin[qi[r]];
        ox[r] = (float)(q.ox - a.c0[0]); oy[r] = (float)(q.oy - a.c0[1]); oz[r] = (float)(q.oz - a.c0[2]);
        dx[r] = (float)q.dx; dy[r] = (float)q.dy; dz[r] = (float)q.dz;
        pix[r] = q.pix; wt[r] = q.wt; cr[r] = q.ar; cg[r] = q.ag; cb[r] = q.ab;
      }
    }
    Best best[2];
    best_init(best[0]); best_init(best[1]);
    const RaySrc src[2] = {{nullptr, nullptr, 0, 0, qin + qi[0]}, {nullptr, nullptr, 0, 0, qin + qi[1]}};
    if (kBvh) {                                      // the traversal already ran (k_closest1_dyn): pick up its result
#pragma unroll
      for (int r = 0; r < 2; r++)
        if (live[r]) best[r] = w.cand[qi[r]];
    } else if (kCull) {
      closest_general_culled<2>(gen, a.npairs, a.N, ox, oy, oz, dx, dy, dz, live, a.d64, a.gS2, a.g_dtmax, a.r.sph64, src, best, ids,
                                c_cand, c_walks);
    } else {
      closest_general<2>(gen, a.npairs, a.N, ox, oy, oz, dx, dy, dz, live, a.d64, a.gS2, a.g_dtmax, a.r.sph64, src, best);
    }
    unsigned hslot[2];
    hit_block(w, __ballot_sync(kFull, live[0] && best[0].idx >= 0), __ballot_sync(kFull, live[1] && best[1].idx >= 0), hslot);
#pragma unroll
    for (int r = 0; r < 2; r++) {
      bool hit = false;
      if (live[r]) {
        c_closest++; c_fp64 += best[r].nfp64;
        if (best[r].idx >= 0) {
          HitRec *rec = w.hits + hslot[r];
          hit = finish_hit(a, best[r], src[r], pix[r], qi[r], wt[r], cr[r], cg[r], cb[r], rec, &c_viol, &c_fp64) >= 0;
          if (!hit) rec->idx = -1;
        }
        if (a.r.hit_idx) a.r.hit_idx[(size_t)pix[r] * depth + level] = hit ? w.hits[hslot[r]].idx : -1;
        if (!hit) {                                // sky through the mirror(s): the pixel is final
          const Rgb skyc = sky_colour(dy[r]);
          float fr = cr[r], fg = cg[r], fb = cb[r];
          add_scaled(fr, fg, fb, wt[r], skyc.r, skyc.g, skyc.b);
          write_final(a.r, pix[r], fr, fg, fb);
        }
      }
      c_hits += hit;
    }
  }
  if (a.r.counters) flush_counts(a.r.counters, level, c_closest, c_hits, 0, 0, c_fp64, c_viol, (unsigned long long)a.N, c_cand, c_walks);
}
template <bool kSmem, bool kBvh>
__global__ void __launch_bounds__(kThreads, kTableCtas) k_closest1(const WaveArgs w) {
  extern __shared__ __align__(128) unsigned char smem[];
  const FastArgs &a = w.f;
  // staged: the general table only (it follows the (1+L) shared-origin tables)
  const unsigned char *tabs = a.tabs + (size_t)(a.L + 1) * a.tstride;
  if (kSmem) { stage_tables(smem, tabs, a.stage_bytes); tabs = smem + kSmemHeader; }
  RT_PDL_SYNC();
  closest1_body<kBvh, kSmem && !kBvh>(w, reinterpret_cast<const float4 *>(tabs), smem);
}

// ---------------------------------------------------------------------------------------------
// SHADE of ONE hit (lane local, no warp-level operations): include/scene.h:89-121 in FP32 with the occlusion bits of
// the shadow queries (bit l of occm = light l occluded), then src/main.cpp:43-55 -- the pixel is final (written here),
// or the path continues: returns true and *rec is the exact FP64 reflected ray for the next level's queue.
// stage != nullptr: a final pixel is not written to the frame but quantised into stage[0..2] (the caller emits whole
// 16-byte row segments of its tile), *is_final tells which it was.
__device__ __forceinline__ bool shade_one(const WaveArgs &w, const int level, const HitRec &hr, unsigned long long occm, RayRec &rec,
                                          unsigned char *stage = nullptr) {
  const FastArgs &a = w.f;
  const int L = a.L;
  const float4 m = __ldg(&a.r.mat[hr.idx]);
  const float2 mx = __ldg(&a.r.matx[hr.idx]);
  float sr = g_frame.ambient[0] * m.x, sg = g_frame.ambient[1] * m.y, sb = g_frame.ambient[2] * m.z;
  const bool cam = level == 0;                  // camera-ray hit: exact direction in the record, weight 1, no colour yet
  const float vx = cam ? -(float)hit_d0x(hr) : hr.vx, vy = cam ? -(float)hit_d0y(hr) : hr.vy, vz = cam ? -(float)hit_d0z(hr) : hr.vz;
  for (int l = 0; l < L; l++)
    if (!((occm >> l) & 1ull)) phong_light(l, hr.px, hr.py, hr.pz, hr.nx, hr.ny, hr.nz, vx, vy, vz, m, mx.x, sr, sg, sb);
  if (a.r.shadow_mask) a.r.shadow_mask[(size_t)hr.pix * a.r.max_depth + level] = (unsigned)(occm & 0xffffffffull);
  float cr = cam ? 0.f : hr.ar, cg = cam ? 0.f : hr.ag, cb = cam ? 0.f : hr.ab, wt = cam ? 1.0f : hr.wt;
  bool cont = false;
  if (mx.y > 0.5f) {                          // reflectivity > 0, decided in double on the host
    const float refl = m.w, k = __fmul_rn(wt, __fsub_rn(1.0f, refl));
    add_scaled(cr, cg, cb, k, sr, sg, sb);
    wt = __fmul_rn(wt, refl);
    if (level + 1 < a.r.max_depth) {
      // exact reflected ray: the incoming direction comes with the record (camera ray) or from the ray's queue record,
      // the normal from the exact hit point (src/main.cpp:35,45-48)
      d3 din;
      if (cam) din = rtx::mk(hit_d0x(hr), hit_d0y(hr), hit_d0z(hr));
      else { const RayRec &q = a.q_in[hr.src]; din = rtx::mk(q.dx, q.dy, q.dz); }
      const double4 s = ld_sph64(&a.r.sph64[hr.idx]);
      const d3 p = rtx::mk(hr.px, hr.py, hr.pz);
      reflected_ray_from_center(din, p, rtx::mk(s.x, s.y, s.z), &rec);
      rec.pix = hr.pix; rec.wt = wt; rec.ar = cr; rec.ag = cg; rec.ab = cb; rec.pad = 0;
      cont = true;
    }
  } else {
    add_scaled(cr, cg, cb, wt, sr, sg, sb);
  }
  if (!cont) {
    if (stage) { stage[0] = (unsigned char)quant8(cr); stage[1] = (unsigned char)quant8(cg); stage[2] = (unsigned char)quant8(cb); }
    else write_final(a.r, hr.pix, cr, cg, cb);
  }
  return cont;
}

// ---------------------------------------------------------------------------------------------
// SHADOW: a warp fetch is 64 consecutive hits; a lane owns hits 2*lane and 2*lane+1 of the chunk and
// runs their shadow queries against every light in turn (the hit records are read once).
// Output: one occlusion byte per (light, hit).
//
// Self-shadow shortcut: if the point faces away from the light (n.l < -4 EPS / r) the shadow-ray
// origin p + l*EPS lies strictly inside the sphere the point is on, so the reference's query returns
// that sphere's exit distance, which is shorter than the distance to any light outside that sphere
// (flag bit 30 of Tab::inv, set on the host): occluded, no table walk needed.
// tabs: where the L light tables are read from (shared memory when staged); wbase: the per-warp compacted tables.
template <int kMode>
__device__ __forceinline__ void shadow_body(const WaveArgs &w, unsigned char *smem, const unsigned char *tabs, unsigned char *wbase) {
  const FastArgs &a = w.f;
  const unsigned char *gtabs = a.tabs + a.tstride;
  const unsigned nh = __ldcg(w.hit_count);
  if (nh == 0u || a.L == 0) return;
  const WarpBuf wb = warp_buf(wbase);                                                                                // kTabSmem / kTabBvh
  const BundleBuf bb = bundle_buf(smem + kSmemHeader + kWarps * kWarpBufBytes);                                      // kTabBvh only
  unsigned ring_phase = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // few hits (deep levels): one hit per lane, so that twice as many warps share the work
  const bool two = kMode == kTabStream || nh >= gridDim.x * (unsigned)kWarps * 64u * a.two_mult;
  const unsigned nchunks = two ? nh / 64u : nh / 32u;            // nh = 64 x blocks
  // few chunks (reflection levels >= 1): one (chunk, light) item per fetch instead of (chunk, all lights) -- L times
  // as many, L times shorter items, so the warps of the machine share them evenly
  const bool lightpar = kMode != kTabStream && a.L > 1 && nchunks < a.lp_mult * gridDim.x * (unsigned)kWarps;
  const unsigned nitems = lightpar ? nchunks * (unsigned)a.L : nchunks;
  unsigned c_fp64 = 0, c_cand = 0, c_walks = 0, c_fall = 0;
  for (;;) {
    unsigned chunk;
    if (kMode == kTabStream) {
      const unsigned cc = (unsigned)cta_fetch(w.work_counter, smem);
      if (cc * kWarps >= nchunks) break;
      chunk = cc * kWarps + warp;
    } else {
      chunk = (unsigned)warp_fetch(w.work_counter);
      if (chunk >= nitems) break;
    }
    int l_beg = 0, l_end = a.L;
    if (lightpar) { l_beg = (int)(chunk % (unsigned)a.L); l_end = l_beg + 1; chunk /= (unsigned)a.L; }
    const unsigned h0 = two ? chunk * 64u + 2u * lane : chunk * 32u + lane;
    const unsigned hend = (h0 & ~63u) + (h0 < nh ? w.hit_n[h0 >> 6] : 0u);   // end of the block's live slots
    bool have[2];
    int self[2];
    float nx[2], ny[2], nz[2], backthr[2];
    d3 p[2];
    const double *pp[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {
      have[r] = h0 + r < hend && (two || r == 0) && w.hits[h0 + r].idx >= 0;
      self[r] = -1; nx[r] = ny[r] = nz[r] = 0.f; backthr[r] = 0.f; p[r] = rtx::mk(0, 0, 0); pp[r] = &w.hits[0].px;
      if (have[r]) {
        const HitRec &hr = w.hits[h0 + r];
        pp[r] = &hr.px;
        p[r] = rtx::mk(hr.px, hr.py, hr.pz);
        self[r] = hr.idx;
        nx[r] = hr.nx; ny[r] = hr.ny; nz[r] = hr.nz;
        backthr[r] = -fmaxf(4.0f * kEps * rsqrtf((float)a.r.sph64[hr.idx].w), 1e-4f);     // -4 EPS / r
      }
    }
    const double *const ppc[2] = {pp[0], pp[1]};
    for (int l = l_beg; l < l_end; l++) {
      const Tab T = tab_at(kMode == kTabStream ? gtabs : tabs, a, l);
      const d3 lp = ldc3(g_frame.light_pos[l]);
      bool want[2], occ[2], shortcut[2];
      float dx[2], dy[2], dz[2], so[2], cosl[2];
#pragma unroll
      for (int r = 0; r < 2; r++) {
        dx[r] = dy[r] = dz[r] = 0.f; so[r] = 0.f; cosl[r] = 0.f; shortcut[r] = false;
        if (have[r]) {
          // direction light -> point: FP64 difference, FP32 normalisation (error <= 12u, see filter_math.cuh)
          const d3 wv = rtx::sub(p[r], lp);
          const float wx = (float)wv.x, wy = (float)wv.y, wz = (float)wv.z;
          const float l2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx));
          const float inv = rsqrtf(l2);
          dx[r] = wx * inv; dy[r] = wy * inv; dz[r] = wz * inv;
          so[r] = l2 * inv - kEps;
          cosl[r] = -(nx[r] * dx[r] + ny[r] * dy[r] + nz[r] * dz[r]);       // n . light_dir
          shortcut[r] = cosl[r] < backthr[r] && (T.inv[self[r]] & 0x40000000) != 0;
        }
        want[r] = have[r] && !shortcut[r];
      }
      int n64 = 0;
      if (kMode == kTabBvh) {
        const float3 o = recentred(a, g_frame.light_pos[l]);
        occ[0] = occ[1] = false;
        if (__any_sync(kFull, want[0] || want[1])) {
          // the block's shadow rays towards this light descend the hierarchy as one bundle (from the light)
          const Cone cone = warp_cone<2>(dx, dy, dz, want);
          ShadowQ<2> q;
          shadow_begin<2>(q, T.inv, so, want, self, cosl);
          q.sslot[0] = q.sslot[1] = -1;              // (no pre-clearing of the lit self sphere here: slow_shadow skips it)
          bool done = false;
          if (cone.ok) c_walks++;
          if (cone.ok)
            done = bundle_traverse(a, bundle_box<2>(o, dx, dy, dz, want), -(kEps + fmaxf(q.m[0], q.m[1])), q.wcut, bb, [&](int n) {
              c_cand += (unsigned)n;
              const int np = bundle_fill(T, bb.cand, n, wb);
              shadow_range<2>(q, wb.pairs, wb.gmin, wb.perm, 0, np, l, dx, dy, dz, so, self, cosl, ppc, a.d64, a.r.sph64, n64);
              __syncwarp();
              return q.wcut < -1.0e38f ? -1.0f : q.wcut;
            });
          if (!done) c_fall++;
#pragma unroll 1
          for (int r = 0; r < 2; r++) {
            occ[r] = q.occ[r];
            if (!done && q.open[r]) occ[r] = bvh_shadow(a, T, o, l, dx[r], dy[r], dz[r], so[r], self[r], cosl[r], ppc[r], n64);
          }
        }
      } else if (kMode == kTabSmem) {
        occ[0] = occ[1] = false;
        if (__any_sync(kFull, want[0] || want[1]))
          shadow_light_culled<2>(T, a.npairs, wb, l, dx, dy, dz, so, want, self, cosl, ppc, a.d64, a.r.sph64, occ, n64, c_cand, c_walks);
      } else {
        // the eight warps of the CTA walk this light's sorted table together, tile by tile
        const Tab TG = tab_at(gtabs, a, l);
        ShadowQ<2> q;
        shadow_begin<2>(q, TG.inv, so, want, self, cosl);
        bool need = q.wcut > -1.0e38f;
        if (__syncthreads_or(need ? 1 : 0)) {
          const int ntiles = (a.npairs + kTilePairs - 1) / kTilePairs;
          if (threadIdx.x == 0) ring_issue(smem, 0, TG.pairs, min(kTilePairs, a.npairs));
          for (int k = 0; k < ntiles; k++) {
            const int st = k & 1, p0 = k * kTilePairs, np = min(kTilePairs, a.npairs - p0);
            if (threadIdx.x == 0 && k + 1 < ntiles)
              ring_issue(smem, st ^ 1, TG.pairs + (size_t)(p0 + kTilePairs) * 2, min(kTilePairs, a.npairs - p0 - kTilePairs));
            ring_wait(smem, st, ring_phase);
            if (need) need = shadow_range<2>(q, ring_stage(smem, st) - (size_t)p0 * 2, TG.gmin, TG.perm, p0, p0 + np, l, dx, dy, dz, so, self,
                                          cosl, ppc, a.d64, a.r.sph64, n64);
            const int more = __syncthreads_or(need ? 1 : 0);      // also: stage st is free again
            if (!more || k + 1 == ntiles) { if (k + 1 < ntiles) ring_wait(smem, st ^ 1, ring_phase); break; }
          }
        }
        occ[0] = q.occ[0]; occ[1] = q.occ[1];
      }
      c_fp64 += (unsigned)n64;
      if (w.occ_bits) {                                // one fire-and-forget RED.OR per OCCLUDED (hit, light) into the hit record
        if (have[0] && (occ[0] || shortcut[0])) atomicOr(&w.hits[h0].pad, 1u << l);
        if (have[1] && (occ[1] || shortcut[1])) atomicOr(&w.hits[h0 + 1].pad, 1u << l);
        continue;
      }
      // two adjacent bytes per lane -> one 16-bit store when both exist
      const unsigned o0 = (occ[0] || shortcut[0]) ? 1u : 0u, o1 = (occ[1] || shortcut[1]) ? 256u : 0u;
      unsigned char *o = w.occ + (size_t)l * w.hit_cap + h0;
      if (have[1]) *reinterpret_cast<unsigned short *>(o) = (unsigned short)(o0 | o1);
      else if (have[0]) o[0] = (unsigned char)o0;
    }
  }
  if (a.r.counters) flush_counts(a.r.counters, 99, 0, 0, 0, 0, c_fp64, 0, (unsigned long long)a.N, c_cand, c_walks, c_fall);
}
// Level 0, one CTA: the per-tile ray counts become exclusive offsets in tile order, in place, and their sum the number of
// rays entering level 1.  The queue position of a reflected ray is thus a function of its tile, not of when a warp got
// to it: a warp of k_closest1 takes 64 rays of a short horizontal strip of consecutive tiles (complex.txt at 1080p: about
// 10 reflected rays per tile), and the order is the same in every run.  Each thread scans a contiguous run of tiles (whole uint4: tile_ray is allocated to that size); s =
// 8 words of scratch shared memory.
__device__ __noinline__ void tile_offsets(unsigned int *tile_ray, int n, unsigned int *rays, unsigned *s) {
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int seg = (n + 4 * kThreads - 1) / (4 * kThreads);        // uint4 per thread
  uint4 *v = reinterpret_cast<uint4 *>(tile_ray) + (size_t)t * seg;
  const int i0 = t * seg * 4;
  unsigned sum = 0;
#pragma unroll 8
  for (int k = 0; k < seg; k++) {
    const uint4 c = v[k];
    const int i = i0 + 4 * k;
    sum += (i < n ? c.x : 0u) + (i + 1 < n ? c.y : 0u) + (i + 2 < n ? c.z : 0u) + (i + 3 < n ? c.w : 0u);
  }
  unsigned incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned y = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) s[warp] = incl;
  __syncthreads();
  unsigned run = incl - sum, total = 0;
  for (int k = 0; k < kWarps; k++) { const unsigned x = s[k]; if (k < warp) run += x; total += x; }
#pragma unroll 8
  for (int k = 0; k < seg; k++) {
    const uint4 c = v[k];
    const int i = i0 + 4 * k;
    uint4 o;
    o.x = run; run += i < n ? c.x : 0u;
    o.y = run; run += i + 1 < n ? c.y : 0u;
    o.z = run; run += i + 2 < n ? c.z : 0u;
    o.w = run; run += i + 3 < n ? c.w : 0u;
    v[k] = o;
  }
  if (t == 0) *rays = total;
  __syncthreads();
}

template <int kMode>
__global__ void __launch_bounds__(kThreads, kTableCtas) k_shadow(const WaveArgs w) {
  extern __shared__ __align__(128) unsigned char smem[];
  const FastArgs &a = w.f;
  // staged: the L light tables
  const unsigned char *tabs = a.tabs + a.tstride;
  // (the pointer is switched UNCONDITIONALLY in this mode -- a scene without lights never dereferences it -- so that the
  // compiler knows the tables are in shared memory: LDS instead of generic loads in every walk)
  if (kMode == kTabSmem) { if (a.L > 0) stage_tables(smem, tabs, a.stage_bytes); tabs = smem + kSmemHeader; }
  if (kMode == kTabStream) ring_init(smem);
  RT_PDL_SYNC();
  if (a.level == 0 && blockIdx.x == 0) tile_offsets(w.tile_ray, a.nwtiles, a.q_out_count, reinterpret_cast<unsigned *>(smem + 64));   // (the header's staging area)
  shadow_body<kMode>(w, smem, tabs, smem + kSmemHeader + (kMode == kTabBvh ? 0u : ((a.stage_bytes + 127u) & ~127u)));
}

// ---------------------------------------------------------------------------------------------
// CLOSEST HIT through the LBVH with DYNAMIC RAY FETCH (large scenes, reflection levels >= 1; see k_shadow_dyn for the
// scheme).  Only the traversal runs here: a lane's result is the candidate bracket (Best) of its ray, stored per queued
// ray; k_closest1 then does the exact finish for 64 neighbouring rays at a time, as before.
constexpr int kDynCtas = 4;     // the traversal kernels are memory-latency bound: 64 registers / 32 warps per SM beat 97 / 16 (measured)
__global__ void __launch_bounds__(kThreads, kDynCtas) k_closest1_dyn(const WaveArgs w) {
  const FastArgs &a = w.f;
  RT_PDL_SYNC();
  const unsigned nq = *a.q_in_count;
  if (nq == 0u) return;
  const float4 *gen = reinterpret_cast<const float4 *>(a.tabs + (size_t)(a.L + 1) * a.tstride);
  const RayRec *qin = a.q_in;
  const int lane = threadIdx.x & 31;
  rtb::BvhIter it;
  Best b;
  best_init(b);
  bool active = false, more = true;
  unsigned qi = 0;
  int big_k = 0;
  float ox = 0.f, oy = 0.f, oz = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
  for (;;) {
    const unsigned idle = __ballot_sync(kFull, !active);
    if (more && (__popc(idle) >= 8 || idle == kFull)) {
      unsigned base = 0;
      if (lane == __ffs(idle) - 1) base = atomicAdd(w.work_counter2, (unsigned)__popc(idle));
      base = __shfl_sync(kFull, base, __ffs(idle) - 1);
      if (base + (unsigned)__popc(idle) >= nq) more = false;
      if (!active) {
        qi = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (qi < nq) {
          const RayRec &q = qin[qi];
          ox = (float)(q.ox - a.c0[0]); oy = (float)(q.oy - a.c0[1]); oz = (float)(q.oz - a.c0[2]);
          dx = (float)q.dx; dy = (float)q.dy; dz = (float)q.dz;
          best_init(b);
          rtb::bvh_begin(it, rtb::bvh_ray(ox, oy, oz, dx, dy, dz), -1e-3f, 3.0e38f);
          big_k = 0;
          active = true;
        }
      }
    }
    if (!__any_sync(kFull, active)) { if (!more) break; else continue; }
#pragma unroll 1
    for (int step = 0; step < 6; step++) {
      if (active) {
        int cnd;
        if (big_k < a.nbig) cnd = a.big[big_k++];
        else cnd = rtb::bvh_next(a.bvh, it, 6);
        if (cnd >= 0) {
          const RaySrc src = {nullptr, nullptr, 0, 0, qin + qi};
          b = slow_closest_general(b, gen, cnd >> 1, a.N, ox, oy, oz, dx, dy, dz, a.d64, a.gS2, a.r.sph64, src);
          if (b.idx >= 0) it.t1 = fminf(it.t1, __fmaf_ru(b.hi, 1e-6f, b.hi) + 1e-6f);     // prune by the best bracket so far
        } else if (cnd == -1) {
          w.cand[qi] = b;
          active = false;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// SHADOW through the LBVH with DYNAMIC RAY FETCH (large scenes).  Work item = one (light, hit slot) shadow ray.  The
// traversal lengths of neighbouring rays differ by an order of magnitude once rays are incoherent (k_shadow<kTabBvh> ran
// at 5-6 active lanes of 32 from reflection level 1 on), so here a lane does not wait for its warp: whenever enough
// lanes are idle they fetch the next items together (one atomic per refill) and everybody goes on traversing
// (persistent threads, Aila & Laine 2009).  Same queries, same slow paths, same occlusion bytes as k_shadow.
__global__ void __launch_bounds__(kThreads, kDynCtas) k_shadow_dyn(const WaveArgs w) {
  const FastArgs &a = w.f;
  RT_PDL_SYNC();
  const unsigned nh = *w.hit_count;
  if (nh == 0u || a.L == 0) return;
  const unsigned total = nh * (unsigned)a.L;         // item = light * nh + slot: neighbouring lanes start on neighbouring hits
  const unsigned char *gtabs = a.tabs + a.tstride;
  const int lane = threadIdx.x & 31;
  rtb::BvhIter it;
  bool active = false, more = true;                  // more: the item counter has not run out yet
  unsigned slot = 0;
  int light = 0, self = -1, big_k = 0;
  float dx = 0.f, dy = 0.f, dz = 0.f, so = 0.f, m = 0.f, cosl = 0.f;
  unsigned c_fp64 = 0;
  for (;;) {
    // ---- refill: idle lanes take the next items (skipped while few lanes are idle, to amortise the atomic)
    const unsigned idle = __ballot_sync(kFull, !active);
    if (more && (__popc(idle) >= 8 || idle == kFull)) {
      unsigned base = 0;
      if (lane == __ffs(idle) - 1) base = atomicAdd(w.work_counter, (unsigned)__popc(idle));
      base = __shfl_sync(kFull, base, __ffs(idle) - 1);
      if (base + (unsigned)__popc(idle) >= total) more = false;
      if (!active) {
        const unsigned item = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (item < total) {
          light = (int)(item / nh); slot = item - (unsigned)light * nh;
          const HitRec &hr = w.hits[slot];
          if ((slot & 63u) < w.hit_n[slot >> 6] && hr.idx >= 0) {
            self = hr.idx;
            // direction light -> point: FP64 difference, FP32 normalisation (error <= 12u, see filter_math.cuh)
            const d3 wv = rtx::sub(rtx::mk(hr.px, hr.py, hr.pz), ldc3(g_frame.light_pos[light]));
            const float wx = (float)wv.x, wy = (float)wv.y, wz = (float)wv.z;
            const float l2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx));
            const float inv = rsqrtf(l2);
            dx = wx * inv; dy = wy * inv; dz = wz * inv;
            so = l2 * inv - kEps;
            cosl = -(hr.nx * dx + hr.ny * dy + hr.nz * dz);                       // n . light_dir
            const Tab T = tab_at(gtabs, a, light);
            const float backthr = -fmaxf(4.0f * kEps * rsqrtf((float)a.r.sph64[self].w), 1e-4f);   // -4 EPS / r
            if (cosl < backthr && (T.inv[self] & 0x40000000) != 0) {
              if (w.occ_bits) atomicOr(&w.hits[slot].pad, 1u << light); else w.occ[(size_t)light * w.hit_cap + slot] = 1;   // self-shadow shortcut (see k_shadow)
            } else {
              m = __fmaf_ru(1.9073486e-6f, so + kEps, 1e-7f);                     // as in shadow_begin
              const float3 o = recentred(a, g_frame.light_pos[light]);
              rtb::bvh_begin(it, rtb::bvh_ray(o.x, o.y, o.z, dx, dy, dz), -(kEps + m), so + m);
              big_k = 0;
              active = true;
            }
          }
        }
      }
    }
    if (!__any_sync(kFull, active)) { if (!more) break; else continue; }
    // ---- a few traversal steps for every active lane, then look at the warp again
#pragma unroll 1
    for (int step = 0; step < 6; step++) {
      if (active) {
        int cand;
        if (big_k < a.nbig) cand = a.big[big_k++];                                // the spheres kept out of the tree first
        else cand = rtb::bvh_next(a.bvh, it, 6);
        if (cand >= 0) {
          const Tab T = tab_at(gtabs, a, light);
          const int sl = __ldg(&T.inv[cand]) & 0x3fffffff;
          const int rc = slow_shadow(T.pairs, T.perm, sl >> 1, dx, dy, dz, so, m, self, cosl, &w.hits[slot].px, light, a.d64, a.r.sph64);
          c_fp64 += (unsigned)(rc >> 1);
          if (rc & 1) { if (w.occ_bits) atomicOr(&w.hits[slot].pad, 1u << light); else w.occ[(size_t)light * w.hit_cap + slot] = 1; active = false; }
        } else if (cand == -1) {
          if (!w.occ_bits) w.occ[(size_t)light * w.hit_cap + slot] = 0;
          active = false;
        }
      }
    }
  }
  if (a.r.counters) flush_counts(a.r.counters, 99, 0, 0, 0, 0, c_fp64, 0, 0);
}

// ---------------------------------------------------------------------------------------------
// SHADE: one hit per lane.  include/scene.h:89-121 in FP32 with the occlusion bytes of k_shadow, then
// src/main.cpp:43-55: final pixel, or the reflected ray (exact FP64) appended to the RayRec queue.
__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
// a reflected ray of level 0 at its place in the tile-ordered queue (tile offset + rank); the capacity guard of queue_push
__device__ __forceinline__ void queue_put(const WaveArgs &w, unsigned pos, const RayRec &rec) {
  if (pos < w.f.queue_cap) w.f.q_out[pos] = rec;
  else atomicOr(w.f.err, (unsigned)RT_GUARD_RAY_QUEUE);
}

// The items of this phase cost the same (one hit per lane), so the chunks are dealt out STATICALLY -- warp g of G takes
// chunks g, g + G, ... -- instead of through an atomic counter: the counter's round trip was a third of this
// memory-latency-bound kernel's stall samples.  The record of the lane's NEXT hit is prefetched into L1 meanwhile.
// Level 0: the reflected rays go to their tile-ordered places (tile_offsets); levels >= 1 append them in arrival order
// (queue_push).
__device__ __forceinline__ void shade_body(const WaveArgs &w) {
  const FastArgs &a = w.f;
  const int level = a.level;
  const bool ordered = level == 0;
  const unsigned nh = __ldcg(w.hit_count);
  if (nh == 0u) return;
  const int lane = threadIdx.x & 31, L = a.L;
  unsigned c_shadow = 0, c_occ = 0;
  const unsigned G = gridDim.x * (unsigned)kWarps;
  // Level 0, 8-bit frame: the 64 slots of a hit block are the hits of ONE 16x4-pixel tile.  The warp takes the whole
  // block and stores the whole tile as twelve 16-byte row segments: every pixel starts as the sky colour of its camera
  // ray (what k_closest0 would have written), the finished hits overwrite theirs in shared memory, the hits whose path
  // continues are overwritten later by the level that finishes them.  k_closest0 leaves such tiles alone (tile_path).
  if (ordered && tile_path(a)) {
    __shared__ __align__(16) unsigned char s_tiles[kWarps][kWTileH * kWTileW * 3];
    unsigned char *s_tile = s_tiles[threadIdx.x >> 5];
    const unsigned W = (unsigned)a.r.W, rows = (unsigned)a.r.bands.local_rows;
    const bool frame = a.r.out_remap == 2;
    for (unsigned blk = blockIdx.x * (unsigned)kWarps + (threadIdx.x >> 5); blk * 64u < nh; blk += G) {
      {
        const unsigned bn = blk + G;
        if (bn * 64u < nh) {
          // the whole next block: 64 records of 80 bytes = 40 lines of 128 bytes, one or two per lane; its occlusion bytes
          const unsigned char *q = reinterpret_cast<const unsigned char *>(w.hits + bn * 64u) + lane * 128;
          prefetch_l1(q);
          if (lane < 8) prefetch_l1(q + 32 * 128);
          if (lane == 0) prefetch_l1(w.hit_n + bn);
          if (!w.occ_bits && lane < L) prefetch_l1(w.occ + (size_t)lane * w.hit_cap + bn * 64u);
        }
      }
      const unsigned nslots = w.hit_n[blk];
      const unsigned pix0 = w.hits[blk * 64u].pix;                  // slot 0 of a block in use always carries its pixel
      const unsigned ty0 = (pix0 / W) & ~(unsigned)(kWTileH - 1), tx0 = (pix0 % W) & ~(unsigned)(kWTileW - 1);
      const bool whole = ty0 + kWTileH <= rows;                      // (W % 16 == 0: every tile is whole in x)
      const unsigned qbase = w.tile_ray[(ty0 / kWTileH) * (unsigned)a.wtiles_x + tx0 / kWTileW];
      if (whole) {
#pragma unroll
        for (int r = 0; r < 2; r++) {                                // the lane's two pixels of the tile, as in k_closest0
          const unsigned ly = (unsigned)(lane >> 4) * 2u + (unsigned)r, lx = (unsigned)lane & 15u;
          float fx, fz;
          const unsigned c = sky_rgb8(camera_dir_y(a, (int)(tx0 + lx), rt_local_to_global_row(a.r.bands, (int)(ty0 + ly)), fx, fz));
          unsigned char *q = s_tile + (ly * kWTileW + lx) * 3;
          q[0] = (unsigned char)c; q[1] = (unsigned char)(c >> 8); q[2] = (unsigned char)(c >> 16);
        }
      }
      __syncwarp();
#pragma unroll 1
      for (int half = 0; half < 2; half++) {
        const unsigned h = blk * 64u + (unsigned)half * 32u + lane;
        const bool live = (h & 63u) < nslots && w.hits[h].idx >= 0;
        bool cont = false;
        RayRec rec;
        unsigned rank = 0;
        if (live) {
          const HitRec hr = w.hits[h];
          unsigned long long occm = hr.pad;
          if (!w.occ_bits) {
            occm = 0ull;
            for (int l = 0; l < L; l++)
              if (w.occ[(size_t)l * w.hit_cap + h]) occm |= 1ull << l;
          }
          c_shadow += (unsigned)L; c_occ += (unsigned)__popcll(occm);
          const unsigned y = hr.pix / W, x = hr.pix - y * W;
          cont = shade_one(w, level, hr, occm, rec, whole ? s_tile + ((y - ty0) * kWTileW + (x - tx0)) * 3 : nullptr);
          rank = hit_ray_rank(hr);
        }
        if (cont) queue_put(w, qbase + rank, rec);
      }
      __syncwarp();
      if (whole && lane < kWTileH * 3) {
        const unsigned ty = (unsigned)lane / 3u, sg = (unsigned)lane % 3u;
        const size_t orow = frame ? (size_t)rt_local_to_global_row(a.r.bands, (int)(ty0 + ty)) : (size_t)(ty0 + ty);
        *reinterpret_cast<uint4 *>(a.r.rgb + (orow * W + tx0) * 3 + sg * 16) = *reinterpret_cast<const uint4 *>(s_tile + lane * 16);
      }
      __syncwarp();
    }
    if (a.r.counters) flush_counts(a.r.counters, 99, 0, 0, c_shadow, c_occ, 0, 0, (unsigned long long)a.N);
    return;
  }
  for (unsigned chunk = blockIdx.x * (unsigned)kWarps + (threadIdx.x >> 5); chunk * 32u < nh; chunk += G) {
    const unsigned h = chunk * 32u + lane;
    {
      const unsigned hn = h + G * 32u;
      if (hn < nh) {
        const unsigned char *q = reinterpret_cast<const unsigned char *>(w.hits + hn);
        prefetch_l1(q); prefetch_l1(q + 64);
        if (lane == 0) prefetch_l1(w.hit_n + (hn >> 6));
        if (!w.occ_bits && lane < L) prefetch_l1(w.occ + (size_t)lane * w.hit_cap + hn);
      }
    }
    const bool live = (h & 63u) < w.hit_n[h >> 6] && w.hits[h].idx >= 0;
    bool cont = false;
    RayRec rec;
    unsigned qpos = 0;
    if (live) {
      const HitRec hr = w.hits[h];
      unsigned long long occm = hr.pad;
      if (!w.occ_bits) {
        occm = 0ull;
        for (int l = 0; l < L; l++)
          if (w.occ[(size_t)l * w.hit_cap + h]) occm |= 1ull << l;
      }
      c_shadow += (unsigned)L; c_occ += (unsigned)__popcll(occm);
      cont = shade_one(w, level, hr, occm, rec);
      if (ordered && cont) {
        const unsigned y = hr.pix / (unsigned)a.r.W, x = hr.pix - y * (unsigned)a.r.W;
        qpos = w.tile_ray[(y / kWTileH) * (unsigned)a.wtiles_x + x / kWTileW] + hit_ray_rank(hr);
      }
    }
    if (ordered) { if (cont) queue_put(w, qpos, rec); }
    else queue_push(cont, rec, a.q_out, a.q_out_count, a.queue_cap, a.err);
  }
  if (a.r.counters) flush_counts(a.r.counters, 99, 0, 0, c_shadow, c_occ, 0, 0, (unsigned long long)a.N);
}
constexpr int kShadeCtas = 4;   // memory-latency bound: 64 registers / 32 warps per SM
__global__ void __launch_bounds__(kThreads, kShadeCtas) k_shade(const WaveArgs w) {
  RT_PDL_SYNC();
  shade_body(w);
}

}  // namespace rtf
#endif
