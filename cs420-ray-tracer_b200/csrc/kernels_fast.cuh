// kernels_fast.cuh -- "mode 0": the production path.  sm_100a only.
//
// Work decomposition (wavefront with compacted queues, warps schedule themselves):
//   levels 0 and 1 run as phase-separated wavefront kernels (kernels_wave.cuh); this file holds the
//   query primitives they share and
//   k_bounce    the tail (levels >= 2, one launch): consumes the ray queue, <= 32 rays per warp fetch,
//               general-origin closest hit per lane, the (hit, light) shadow queries of the warp packed
//               onto its lanes (shadow_mixed), Phong; each lane follows its ray to termination, the
//               queue record is updated in place.
// Sphere tables are staged once per CTA into shared memory with ONE TMA bulk copy
// (cp.async.bulk + mbarrier) when they fit; larger ones are streamed tile by tile (kernels_wave.cuh) or, from
// 1024 spheres on, replaced as the source of candidates by the device-built LBVH (bvh.cuh).
//
// Shared-origin tables (camera, each light) are SORTED by the distance of the sphere's nearest
// point from that origin; a query stops at the first 8-sphere group that lies entirely beyond
// its cutoff (current best hit / distance to the shaded point), so "any hit" really is early out.
//
// Bundle culling (tables staged in shared memory): the rays a warp works on at one time share their
// origin (camera / one light) and form a narrow bundle.  The warp bounds them by a cone, tests every
// sphere of the table against that cone ONCE (one sphere per lane, warp ballot), compacts the
// survivors into a per-warp shared-memory table and runs the per-ray tests over that table only:
// a handful of spheres instead of all N.  The cone test is conservative (see cull_round).
//
// What is FP32 and what is FP64:  every ray/sphere TEST is 4 packed-FP32 FMAs per sphere pair
// (FFMA2; shared origin) or 10 (general origin).  The tests are conservative (filter_math.cuh);
// the few spheres they flag are bracketed in FP32 interval arithmetic and, only where brackets
// touch, decided by the reference's own FP64 formula (exact_fp64.cuh).  Hit points, normals and
// reflected rays -- everything that feeds the NEXT query -- are FP64 in the reference's
// operation order, so hit indices and shadow booleans are bit-exact.  Colour is FP32.
#ifndef RT_KERNELS_FAST_CUH
#define RT_KERNELS_FAST_CUH

#include "bvh.cuh"
#include "exact_fp64.cuh"
#include "filter_math.cuh"
#include "rt_device.h"

namespace rtf {

using rtx::d3;

#ifndef RT_THREADS
#define RT_THREADS 256
#endif
constexpr int kThreads = RT_THREADS;
constexpr int kWarps = kThreads / 32;
constexpr int kWTileW = 16, kWTileH = 4;  // pixels per warp tile (32 lanes x 2 pixels)
constexpr int kGroupPairs = 4;            // sphere pairs per fast-path group (8 spheres)
constexpr int kSmemHeader = 2048;         // [0,8) mbarrier, [64, 64+8*192) per-warp RGB staging
constexpr float kEps = 0.001f;            // EPSILON, include/ray_math_constants.h:22
constexpr unsigned kSign = 0x80000000u;
constexpr unsigned kFull = 0xffffffffu;

struct __align__(16) RayRec {             // one queued reflected ray (80 bytes)
  double ox, oy, oz, dx, dy, dz;          // exact FP64 origin / unit direction (src/main.cpp:45-48)
  unsigned pix;                           // local pixel index lr*W + x
  float wt;                               // product of reflectivities so far
  float ar, ag, ab;                       // colour accumulated so far (front to back)
  unsigned pad;
};

struct FastArgs {
  RtRenderArgs r;
  const unsigned char *tabs;  // (1+L) shared-origin tables (tstride bytes each: pairs | gmin | perm), then the general table
  int npairs, ngroups;        // npairs is a multiple of kGroupPairs; ngroups = npairs / kGroupPairs
  int N, L;
  unsigned tstride, gmin_off, perm_off, inv_off, cullA_off, cullB_off;
  unsigned stage_bytes;       // bytes this kernel stages into shared memory
  float d64;                  // absolute slack covering FP64 rounding / geometry (delta64)
  float gS2;                  // squared radius bound S^2 of the recentred scene (general filter)
  float g_dtmax;              // 16u*S: bound of |fl32 dot - true| for the general filter
  double c0[3];               // recentring offset of the general table
  int wtiles_x, nwtiles;
  unsigned int *tile_counter;
  RayRec *q_out; unsigned int *q_out_count;
  RayRec *q_in; const unsigned int *q_in_count;
  unsigned int *chunk_counter;
  int level;
  int tables_in_smem;
  rtb::BvhView bvh;           // large scenes: candidates come from the LBVH instead of a table walk (bvh.cuh)
  int nbig, big[8];           // spheres too large for the LBVH (a ground sphere ...): tested for every ray instead
  unsigned two_mult, lp_mult; // work-granularity thresholds in units of (warps of the grid): two rays / hits per lane from
                              // two_mult x 64 per warp on; one (chunk, light) item per fetch below lp_mult chunks per warp
  unsigned queue_cap;         // records per ray queue
  unsigned int *err;          // the frame's error word (bounds guards; 0 = clean)
};

// One shared-origin table: sphere pairs in sorted order, per-group minimum distance, original indices
struct Tab {
  const float4 *pairs;   // 2 float4 per pair: (x0,x1,y0,y1) (z0,z1,w0,w1)
  const float *gmin;     // per group of 8 spheres: lower bound of |oc| - r over the group (ascending)
  const int *perm;       // original sphere index per sorted slot, -1 = padding
  const int *inv;        // sorted slot of each original sphere index; bit 30: the origin is strictly outside it
  const float4 *cullA;   // per slot: unit vector origin -> centre, cos(alpha); alpha = angular radius seen from the origin
  const float *cullB;    // per slot: sin(alpha)
};

// ---------------------------------------------------------------------------------------------
// small helpers
__device__ __forceinline__ unsigned fbits(float x) { return __float_as_uint(x); }
__device__ __forceinline__ float f_rd(double x) { return __double2float_rd(x); }
__device__ __forceinline__ float f_ru(double x) { return __double2float_ru(x); }
__device__ __forceinline__ d3 ldc3(const double *p) { return rtx::mk(p[0], p[1], p[2]); }
__device__ __forceinline__ double4 ld_sph64(const double4 *p) {
  const double2 *q = reinterpret_cast<const double2 *>(p);
  double2 a = __ldg(q), b = __ldg(q + 1);
  return make_double4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ unsigned long long wsum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float wmaxf(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}
__device__ __forceinline__ unsigned quant8(float c) { return (unsigned)(int)(255.99f * fminf(1.0f, c)); }

// ---- colour arithmetic with a FIXED operation order.  Several kernels (and several inlined copies inside one kernel: the tile
// and the pixel path of k_shade, the wavefront and the tail) compute the colour of the same pixel, and their results must
// agree bit for bit (assembled N-GPU frames are compared with single-GPU ones).  Written as ordinary expressions the compiler
// contracts a*b + c*d into an FMA one way in one copy and the other way in the next; explicit intrinsics are never contracted.
struct Rgb { float r, g, b; };
__device__ __forceinline__ Rgb sky_colour(float dy) {              // src/main.cpp:26-30: (1-t) white + t (0.5, 0.7, 1)
  const float ts = __fmul_rn(0.5f, __fadd_rn(dy, 1.0f)), w = __fsub_rn(1.0f, ts);
  Rgb c;
  c.r = __fmaf_rn(0.5f, ts, w); c.g = __fmaf_rn(0.7f, ts, w); c.b = __fadd_rn(w, ts);
  return c;
}
__device__ __forceinline__ void add_scaled(float &cr, float &cg, float &cb, float k, float sr, float sg, float sb) {
  cr = __fmaf_rn(k, sr, cr); cg = __fmaf_rn(k, sg, cg); cb = __fmaf_rn(k, sb, cb);
}
// Phong terms of ONE un-occluded light at a hit (include/scene.h:104-117): point p (exact), unit normal n, view direction v,
// material m = (R, G, B, reflectivity), shininess; adds to (sr, sg, sb)
__device__ __forceinline__ void phong_light(int l, double px, double py, double pz, float nx, float ny, float nz, float vx, float vy, float vz,
                                            float4 m, float shin, float &sr, float &sg, float &sb) {
  // light_dir = normalized(light - point): FP64 difference, FP32 normalisation (colour only)
  const float wx = (float)__dsub_rn(g_frame.light_pos[l][0], px), wy = (float)__dsub_rn(g_frame.light_pos[l][1], py),
              wz = (float)__dsub_rn(g_frame.light_pos[l][2], pz);
  const float inv = rsqrtf(__fmaf_rn(wz, wz, __fmaf_rn(wy, wy, __fmul_rn(wx, wx))));
  const float lx = __fmul_rn(wx, inv), ly = __fmul_rn(wy, inv), lz = __fmul_rn(wz, inv);
  const float nl = __fmaf_rn(nz, lz, __fmaf_rn(ny, ly, __fmul_rn(nx, lx)));
  const float kd = __fmul_rn(__fsub_rn(1.0f, m.w), fmaxf(0.0f, nl));
  // reflect(-light_dir, n) = -l + 2 (l.n) n   (include/vec3.h:31-33)
  const float t2 = __fmul_rn(2.0f, nl);
  const float rx = __fmaf_rn(t2, nx, -lx), ry = __fmaf_rn(t2, ny, -ly), rz = __fmaf_rn(t2, nz, -lz);
  const float rdv = fmaxf(0.0f, __fmaf_rn(rz, vz, __fmaf_rn(ry, vy, __fmul_rn(rx, vx))));
  const float spec = __fmul_rn(0.5f, shin == 0.0f ? 1.0f : __powf(rdv, shin));
  sr = __fadd_rn(sr, __fmaf_rn(g_frame.light_col[l][0], spec, __fmul_rn(m.x, kd)));
  sg = __fadd_rn(sg, __fmaf_rn(g_frame.light_col[l][1], spec, __fmul_rn(m.y, kd)));
  sb = __fadd_rn(sb, __fmaf_rn(g_frame.light_col[l][2], spec, __fmul_rn(m.z, kd)));
}
// A finished pixel: 8-bit quantised (src/main.cpp:84-86) or, for tile renders / supersampling, FP32 colour.
__device__ __forceinline__ void write_final(const RtRenderArgs &r, unsigned pix, float cr, float cg, float cb) {
  size_t o = pix;
  if (r.out_remap) {
    const unsigned lr = pix / (unsigned)r.W, x = pix - lr * (unsigned)r.W;
    if (r.out_remap == 2) o = (size_t)rt_local_to_global_row(r.bands, (int)lr) * (size_t)r.W + x;
    else o = (size_t)(lr + (unsigned)r.out_y0) * (size_t)r.out_pitch + x + (unsigned)r.out_x0;
  }
  if (r.fb) { float *f = r.fb + o * 3; f[0] = cr; f[1] = cg; f[2] = cb; }
  else { unsigned char *q = r.rgb + o * 3; q[0] = (unsigned char)quant8(cr); q[1] = (unsigned char)quant8(cg); q[2] = (unsigned char)quant8(cb); }
}
__device__ __forceinline__ int warp_fetch(unsigned int *counter) {
  int v = 0;
  if ((threadIdx.x & 31) == 0) v = (int)atomicAdd(counter, 1u);
  return __shfl_sync(kFull, v, 0);
}

// Programmatic dependent launch: everything a kernel does BEFORE this point (table staging) may overlap the tail of the
// previous kernel of the stream; after it, that kernel has completed and its writes are visible.  The early
// launch_dependents lets the NEXT kernel's CTAs take SM slots as soon as ours exit (they wait at their own RT_PDL_SYNC).
// Both are no-ops for a launch without the PDL attribute.
#define RT_PDL_SYNC() do { asm volatile("griddepcontrol.wait;" ::: "memory"); asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); } while (0)

// mbarrier + TMA bulk copy (global -> shared), one phase, used once per CTA
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
  unsigned d = (unsigned)__cvta_generic_to_shared(dst), b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(src),
               "r"(bytes), "r"(b)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(a), "r"(parity)
      : "memory");
}

// Stages `bytes` from gsrc into shared memory behind the header with ONE TMA bulk copy.
__device__ __forceinline__ void stage_tables(unsigned char *smem, const unsigned char *gsrc, unsigned bytes) {
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, bytes);
    tma_bulk_g2s(smem + kSmemHeader, gsrc, bytes, bar);
  }
  __syncthreads();
  mbar_wait(bar, 0);
}

__device__ __forceinline__ Tab tab_at(const unsigned char *base, const FastArgs &a, int t) {
  const unsigned char *p = base + (size_t)t * a.tstride;
  Tab T;
  T.pairs = reinterpret_cast<const float4 *>(p);
  T.gmin = reinterpret_cast<const float *>(p + a.gmin_off);
  T.perm = reinterpret_cast<const int *>(p + a.perm_off);
  T.inv = reinterpret_cast<const int *>(p + a.inv_off);
  T.cullA = reinterpret_cast<const float4 *>(p + a.cullA_off);
  T.cullB = reinterpret_cast<const float *>(p + a.cullB_off);
  return T;
}

// ---------------------------------------------------------------------------------------------
// exact (FP64) deciders.  Everything here is OUT OF LINE on purpose: it is rare, register hungry
// and large (IEEE double sqrt / div expand to dozens of instructions); one copy per kernel keeps
// the instruction footprint of the kernels inside the instruction cache.
struct ExactRay { d3 o, d; double a; };

// Where a query's exact FP64 ray comes from: the camera (pixel x, row j) or a queue record.
struct RaySrc { const double *su, *sv; int x, j; const RayRec *rec; };

__device__ __noinline__ ExactRay exact_ray(RaySrc s) {
  ExactRay e;
  if (s.rec) {
    e.o = rtx::mk(s.rec->ox, s.rec->oy, s.rec->oz);
    e.d = rtx::mk(s.rec->dx, s.rec->dy, s.rec->dz);
  } else {
    e.o = ldc3(g_frame.cam_pos);
    e.d = rtx::camera_dir(ldc3(g_frame.fwd), ldc3(g_frame.right), ldc3(g_frame.up), s.su[s.x], s.sv[s.j]);
  }
  e.a = rtx::dot(e.d, e.d);
  return e;
}
__device__ __noinline__ bool exact_sphere(const double4 *sph64, int idx, d3 o, d3 d, double a, double &t) {
  double4 s = ld_sph64(&sph64[idx]);
  return rtx::intersect(o, d, a, rtx::mk(s.x, s.y, s.z), s.w, t);
}
// include/scene.h:70-85 for ONE sphere: the reference's own formula on the reference's own shadow ray
__device__ __noinline__ bool exact_shadow_sphere(const double4 *sph64, int idx, d3 p, int light) {
  d3 o, d; double ldist, tt;
  rtx::shadow_ray(p, ldc3(g_frame.light_pos[light]), 0.001, o, d, ldist);
  return exact_sphere(sph64, idx, o, d, rtx::dot(d, d), tt) && tt < 1e20 && tt < ldist;
}
// safety net only: full FP64 brute force for one ray (a filter violation was detected)
__device__ __noinline__ int exact_bruteforce(const double4 *sph64, int n, d3 o, d3 d, double a, double &tbest) {
  double t = 1e20; int idx = -1;
  for (int i = 0; i < n; i++) {
    double tt;
    if (exact_sphere(sph64, i, o, d, a, tt) && tt < t) { t = tt; idx = i; }
  }
  tbest = t;
  return idx;
}
// src/main.cpp:32,35 : the exact hit point, and the unit normal as an FP32 vector.  The normal of the hit record feeds the
// colour and two sign tests with wide margins (lit side: n.l > 1e-3, self-shadow shortcut: n.l < -1e-4) -- FP32 accuracy
// is all they need, so it is the exact FP64 difference p - c normalised in FP32 (2-3 ulp) instead of the reference's FP64
// normalisation (one FP64 square root and three divisions per hit: a quarter of the exact finish).  The EXACT normal the
// reflected ray is built from is formed where a ray continues (reflected_ray_from_center).  One copy of this code serves
// every kernel, so a hit gets the same FP32 normal whichever kernel finishes it.
struct HitGeom { d3 p; float nx, ny, nz; };
__device__ __noinline__ HitGeom hit_geometry(const double4 *sph64, int idx, d3 o, d3 d, double t) {
  const double4 s = ld_sph64(&sph64[idx]);
  HitGeom h;
  h.p = rtx::hit_point(o, d, t);
  const float fx = (float)rtx::dsub(h.p.x, s.x), fy = (float)rtx::dsub(h.p.y, s.y), fz = (float)rtx::dsub(h.p.z, s.z);
  const float inv = rsqrtf(__fmaf_rn(fz, fz, __fmaf_rn(fy, fy, __fmul_rn(fx, fx))));
  h.nx = __fmul_rn(fx, inv); h.ny = __fmul_rn(fy, inv); h.nz = __fmul_rn(fz, inv);
  return h;
}
// src/main.cpp:35,45-48 from the exact hit point and the sphere centre: exact normal, reflected ray as the Ray ctor stores it
__device__ __noinline__ void reflected_ray_from_center(d3 d, d3 p, d3 c, RayRec *rec) {
  const d3 n = rtx::normal_at(p, c);
  d3 o2, d2;
  rtx::reflect_ray(d, p, n, 0.001, o2, d2);
  rec->ox = o2.x; rec->oy = o2.y; rec->oz = o2.z; rec->dx = d2.x; rec->dy = d2.y; rec->dz = d2.z;
}

// ---------------------------------------------------------------------------------------------
// closest-hit bookkeeping: best candidate as an FP32 bracket, exact FP64 t only when needed.
// All comparisons are order independent: (t, index) lexicographic, i.e. the reference's strict '<'
// scan in ascending index order (include/scene.h:47-56), whatever order spheres are visited in.
struct Best {
  float lo, hi;
  int idx;
  int nfp64;      // FP64 sphere evaluations spent on this query
  double t;       // valid iff exact
  bool exact;
};
__device__ __forceinline__ void best_init(Best &b) { b.lo = 3.0e38f; b.hi = 3.0e38f; b.idx = -1; b.t = 1e20; b.exact = false; b.nfp64 = 0; }
__device__ __forceinline__ void best_set_exact(Best &b, int idx, double t) {
  b.idx = idx; b.t = t; b.exact = true; b.lo = f_rd(t); b.hi = f_ru(t);
}

// brackets touch, or the sphere itself is ambiguous: decide in FP64, lowest index wins ties (rare, out of line)
__device__ __noinline__ Best closest_consider_exact(Best b, int i, const double4 *sph64, RaySrc src) {
  const ExactRay e = exact_ray(src);
  double tn;
  b.nfp64++;
  const bool hn = exact_sphere(sph64, i, e.o, e.d, e.a, tn);
  if (!hn || !(tn < 1e20)) return b;              // INFINITY_DOUBLE init of include/scene.h:42
  if (b.idx >= 0 && !b.exact) {
    const float tl = f_rd(tn), th = f_ru(tn);
    if (tl > b.hi) return b;
    if (th < b.lo) { best_set_exact(b, i, tn); return b; }
    double tb;
    b.nfp64++;
    const bool hb = exact_sphere(sph64, b.idx, e.o, e.d, e.a, tb);
    if (hb) best_set_exact(b, b.idx, tb); else { const int k = b.nfp64; best_init(b); b.nfp64 = k; }   // (else: filter violation, caught later)
  }
  if (b.idx < 0 || tn < b.t || (tn == b.t && i < b.idx)) best_set_exact(b, i, tn);
  return b;
}
// the common outcomes are decided inline on the FP32 brackets
__device__ __forceinline__ void closest_consider(Best &b, int i, int status, float lo, float hi, const double4 *sph64, RaySrc src) {
  if (status == RT_MISS || i == b.idx) return;     // (BVH candidates can name a sphere twice)
  if (status == RT_HIT) {
    if (b.idx < 0) { b.lo = lo; b.hi = hi; b.idx = i; b.exact = false; return; }
    if (lo > b.hi) return;                        // strictly farther
    if (hi < b.lo) { b.lo = lo; b.hi = hi; b.idx = i; b.exact = false; return; }
  }
  b = closest_consider_exact(b, i, sph64, src);
}

// scalar re-evaluation of one sphere of a shared-origin table (same operations as the fast path)
__device__ __forceinline__ void shared_origin_eval(float ocx, float ocy, float ocz, float ncc, float dx, float dy, float dz,
                                                   float &tca, float &Dp) {
  tca = __fmul_rn(ocx, dx);
  tca = __fmaf_rn(ocy, dy, tca);
  tca = __fmaf_rn(ocz, dz, tca);
  Dp = __fmaf_rn(tca, tca, ncc);
}

// Brackets the roots of sphere (oc, ncc) of a shared-origin table.  False = discriminant sign uncertain.
__device__ __forceinline__ bool shared_origin_roots(float ocx, float ocy, float ocz, float ncc, float tca, float Dp, float d64,
                                                    Roots &r) {
  float oc2 = __fmaf_ru(ocz, ocz, __fmaf_ru(ocy, ocy, __fmul_ru(ocx, ocx)));
  float E = disc_margin(oc2, d64);
  // D* <= Dp (+ rounding), D* >= Dp - 2E - ulp(ncc) (- rounding): see DESIGN.md "filter margins"
  float slop = __fmul_ru(4.8e-7f, fabsf(Dp) + fabsf(ncc));
  float Dhi = __fadd_ru(Dp, slop);
  float E2 = __fadd_ru(__fadd_ru(__fmul_ru(2.0f, E), slop), slop);
  float dt = __fmul_ru(RT_ETA * 1.001f, __fsqrt_ru(oc2));
  return bracket_roots(tca, Dhi, E2, dt, r);
}

// ---- slow paths: one flagged sphere PAIR for ONE ray.  The FP32 bracketing is inline (a call would
// spill the caller's registers to local memory around it); only the FP64 deciders are out of line.
#ifndef RT_SLOW
#define RT_SLOW __forceinline__
#endif
__device__ RT_SLOW Best slow_closest_shared(Best b, const float4 *pairs, const int *perm, int pi, float dx, float dy, float dz,
                                                 float d64, const double4 *sph64, RaySrc src) {
  const float4 A = pairs[2 * pi], B = pairs[2 * pi + 1];
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    const int i = perm[2 * pi + h];
    if (i < 0) continue;
    const float ocx = h ? A.y : A.x, ocy = h ? A.w : A.z, ocz = h ? B.y : B.x, ncc = h ? B.w : B.z;
    float tca, Dp;
    shared_origin_eval(ocx, ocy, ocz, ncc, dx, dy, dz, tca, Dp);
    if (!(Dp >= 0.0f)) continue;
    Roots rt;
    int status = RT_AMBIG;
    float lo = 0, hi = 0;
    if (shared_origin_roots(ocx, ocy, ocz, ncc, tca, Dp, d64, rt)) status = select_root(rt, lo, hi);
    closest_consider(b, i, status, lo, hi, sph64, src);
  }
  return b;
}

// returns bit 0 = an occluder was found in this pair, bits 1.. = FP64 evaluations spent
__device__ RT_SLOW int slow_shadow(const float4 *pairs, const int *perm, int pi, float dx, float dy, float dz, float so, float m,
                                        int self, float cosl, const double *p3, int light, float d64, const double4 *sph64) {
  const float so_lo = so - m, so_hi = so + m, e_lo = -kEps - m, e_hi = -kEps + m;
  const float4 A = pairs[2 * pi], B = pairs[2 * pi + 1];
  int n64 = 0, found = 0;
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    const int i = perm[2 * pi + h];
    if (i < 0) continue;
    if (i == self && cosl > 1e-3f) continue;
    const float ocx = h ? A.y : A.x, ocy = h ? A.w : A.z, ocz = h ? B.y : B.x, ncc = h ? B.w : B.z;
    float tca, Dp;
    shared_origin_eval(ocx, ocy, ocz, ncc, dx, dy, dz, tca, Dp);
    if (!(Dp >= 0.0f)) continue;
    Roots rt;
    if (shared_origin_roots(ocx, ocy, ocz, ncc, tca, Dp, d64, rt)) {
      const bool no = (rt.n_lo > so_hi) || (rt.f_hi < e_lo) || (rt.n_hi < e_lo && rt.f_lo > so_hi);
      const bool yes = (rt.f_lo > e_hi && rt.f_hi < so_lo) || (rt.f_lo > so_hi && rt.n_lo > e_hi && rt.n_hi < so_lo);
      if (no) continue;
      if (yes) { found = 1; break; }
    }
    n64++;
    if (exact_shadow_sphere(sph64, i, rtx::mk(p3[0], p3[1], p3[2]), light)) { found = 1; break; }
  }
  return found | (n64 << 1);
}

__device__ RT_SLOW Best slow_closest_general(Best b, const float4 *pairs, int pi, int N, float ox, float oy, float oz, float dx,
                                                  float dy, float dz, float d64, float gS2, const double4 *sph64, RaySrc src) {
  const float sS = __fsqrt_ru(gS2);
  const float4 A = pairs[2 * pi], B = pairs[2 * pi + 1];
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    const int i = 2 * pi + h;
    if (i >= N) break;
    const float cx = h ? A.y : A.x, cy = h ? A.w : A.z, cz = h ? B.y : B.x, rho = h ? B.w : B.z;
    // explicit-margin evaluation (independent of the inflation tricks of the fast path)
    const float x = __fsub_rn(cx, ox), y = __fsub_rn(cy, oy), z = __fsub_rn(cz, oz);
    float tca = __fmul_rn(x, dx); tca = __fmaf_rn(y, dy, tca); tca = __fmaf_rn(z, dz, tca);
    const float oc2 = __fmaf_ru(z, z, __fmaf_ru(y, y, __fmul_ru(x, x)));
    // |X - oc*| <= u(2S + |oc|)  =>  D error <= u (8.1 S |oc| + 16 |oc|^2 + 4 rho) + d64   (DESIGN.md)
    const float ocn = __fsqrt_ru(oc2);
    const float Eg = __fadd_ru(__fmul_ru(5.9604645e-8f, __fmaf_ru(8.2f * sS, ocn, __fmaf_ru(16.5f, oc2, 4.5f * fabsf(rho)))), d64);
    const float Dc = __fmaf_rn(tca, tca, __fsub_rn(rho, oc2));      // rho = r^2 + margins
    const float Dhi = __fadd_ru(Dc, Eg);
    if (!(Dhi >= 0.0f)) continue;
    Roots rt;
    int status = RT_AMBIG;
    float lo = 0, hi = 0;
    const float dt = __fmul_ru(RT_ETA * 1.001f, __fadd_ru(ocn, sS));
    // rho' - r^2 = 40u r^2 + 12u S r + 64u^2 S^2 + d64 (host), bounded here from rho' itself
    const float rm = __fadd_ru(__fmul_ru(5.9604645e-8f, __fmaf_ru(12.5f * sS, __fsqrt_ru(fabsf(rho)), __fmaf_ru(41.0f, fabsf(rho), 1e-4f * gS2))), d64);
    if (bracket_roots(tca, Dhi, __fadd_ru(__fmul_ru(2.0f, Eg), rm), dt, rt)) status = select_root(rt, lo, hi);
    closest_consider(b, i, status, lo, hi, sph64, src);
  }
  return b;
}

// The packed FP32 test of up to 32 sphere PAIRS (one "chunk") of a shared-origin table against the
// NR rays of a lane.  For every pair and ray one bit is shifted into a history word: 1 = neither
// sphere of the pair can be hit (D' = (oc.d)^2 + ncc < 0 for both), 0 = flagged.  No branch, no vote:
// flagged pairs are resolved afterwards, all lanes together (see the drain loops below).
constexpr int kChunkPairs = 32;
__device__ __forceinline__ unsigned push_sign(unsigned hist, unsigned v) { return __funnelshift_l(v, hist, 1); }

template <int NR>
__device__ __forceinline__ void chunk_test_shared(const float4 *__restrict__ pairs, int p0, int np, const float2 (&dx)[NR],
                                                  const float2 (&dy)[NR], const float2 (&dz)[NR], unsigned (&h)[NR]) {
#pragma unroll
  for (int r = 0; r < NR; r++) h[r] = kFull;
#pragma unroll 1
  for (int p = p0; p < p0 + np; p += kGroupPairs) {
#pragma unroll
    for (int k = 0; k < kGroupPairs; k++) {
      const float4 A = pairs[2 * (p + k)], B = pairs[2 * (p + k) + 1];
      const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w), Z = make_float2(B.x, B.y), Wv = make_float2(B.z, B.w);
#pragma unroll
      for (int r = 0; r < NR; r++) {
        float2 t = __fmul2_rn(X, dx[r]); t = __ffma2_rn(Y, dy[r], t); t = __ffma2_rn(Z, dz[r], t);
        const float2 D = __ffma2_rn(t, t, Wv);
        h[r] = push_sign(h[r], fbits(D.x) & fbits(D.y));
      }
    }
  }
}
// history word -> flagged-pair bits (bit i <-> pair p0 + np - 1 - i)
__device__ __forceinline__ unsigned flagged_bits(unsigned hist, int np, bool live) {
  const unsigned pm = np >= 32 ? kFull : ((1u << np) - 1u);
  return live ? (~hist & pm) : 0u;
}

// ---------------------------------------------------------------------------------------------
// LANE-COOPERATIVE chunk tests (the tail kernel at its deep levels: a warp that holds only a few live rays).  The chunk
// tests above give every lane ITS ray and walk the pairs serially; with a handful of live lanes that is one warp's
// dependency chain over the whole table for a few rays' worth of work.  Here the roles are swapped: for each live ray
// in turn (its direction broadcast by shuffle) all 32 lanes test 32 DIFFERENT pairs of the chunk at once, and the ballot
// of the flags, reordered to the history-word convention of flagged_bits (bit i <-> pair p0 + np - 1 - i), goes to the
// lane that owns the ray.  Per (ray, pair) the arithmetic is exactly that of chunk_test_shared / closest_general, so
// the flags -- and everything that follows from them -- are identical.
__device__ __forceinline__ unsigned coop_chunk_shared(const float4 *__restrict__ pairs, int p0, int np, float dx, float dy, float dz, bool live) {
  const int lane = threadIdx.x & 31;
  unsigned mine = 0u, lm = __ballot_sync(kFull, live);
  float4 A = make_float4(0.f, 0.f, 0.f, 0.f), B = A;
  if (lane < np) { A = pairs[2 * (p0 + lane)]; B = pairs[2 * (p0 + lane) + 1]; }
  const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w), Z = make_float2(B.x, B.y), Wv = make_float2(B.z, B.w);
  while (lm != 0u) {
    const int k = __ffs(lm) - 1;
    lm &= lm - 1u;
    const float bx = __shfl_sync(kFull, dx, k), by = __shfl_sync(kFull, dy, k), bz = __shfl_sync(kFull, dz, k);
    float2 t = __fmul2_rn(X, make_float2(bx, bx)); t = __ffma2_rn(Y, make_float2(by, by), t); t = __ffma2_rn(Z, make_float2(bz, bz), t);
    const float2 D = __ffma2_rn(t, t, Wv);
    const bool flagged = lane < np && ((fbits(D.x) & fbits(D.y)) & kSign) == 0u;      // not (both spheres certainly missed)
    const unsigned m = __ballot_sync(kFull, flagged);
    if (lane == k) mine = __brev(m) >> (32 - np);
  }
  return mine;
}
__device__ __forceinline__ unsigned coop_chunk_general(const float4 *__restrict__ pairs, int p0, int np, float nox, float noy, float noz,
                                                       float idx, float idy, float idz, float dtmax, bool live) {
  const int lane = threadIdx.x & 31;
  unsigned mine = 0u, lm = __ballot_sync(kFull, live);
  float4 A = make_float4(0.f, 0.f, 0.f, 0.f), B = A;
  if (lane < np) { A = pairs[2 * (p0 + lane)]; B = pairs[2 * (p0 + lane) + 1]; }
  const float2 CX = make_float2(A.x, A.y), CY = make_float2(A.z, A.w), CZ = make_float2(B.x, B.y), NR_ = make_float2(-B.z, -B.w);
  const float2 dtm = make_float2(dtmax, dtmax);
  while (lm != 0u) {
    const int k = __ffs(lm) - 1;
    lm &= lm - 1u;
    const float ox = __shfl_sync(kFull, nox, k), oy = __shfl_sync(kFull, noy, k), oz = __shfl_sync(kFull, noz, k);
    const float ix = __shfl_sync(kFull, idx, k), iy = __shfl_sync(kFull, idy, k), iz = __shfl_sync(kFull, idz, k);
    const float2 x = __fadd2_rn(CX, make_float2(ox, ox)), y = __fadd2_rn(CY, make_float2(oy, oy)), z = __fadd2_rn(CZ, make_float2(oz, oz));
    float2 t = __ffma2_rn(x, make_float2(ix, ix), dtm); t = __ffma2_rn(y, make_float2(iy, iy), t); t = __ffma2_rn(z, make_float2(iz, iz), t);
    float2 q = __ffma2_rn(x, x, NR_); q = __ffma2_rn(y, y, q); q = __ffma2_rn(z, z, q);
    const float2 D = __ffma2_rn(t, t, make_float2(-q.x, -q.y));
    const unsigned rej = (fbits(D.x) | (fbits(t.x) & ~fbits(q.x))) & (fbits(D.y) | (fbits(t.y) & ~fbits(q.y)));
    const unsigned m = __ballot_sync(kFull, lane < np && (rej & kSign) == 0u);
    if (lane == k) mine = __brev(m) >> (32 - np);
  }
  return mine;
}
// ... and for queries that each walk their OWN shared-origin table (shadow_mixed below: lane k's query goes to light
// light[k], whose table starts at tabs + light[k] * tstride): the table of the query in turn is read by all lanes
__device__ __forceinline__ unsigned coop_chunk_mixed(const unsigned char *tabs, unsigned tstride, int light, int p0, int np, float dx, float dy,
                                                     float dz, bool live) {
  const int lane = threadIdx.x & 31;
  unsigned mine = 0u, lm = __ballot_sync(kFull, live);
  while (lm != 0u) {
    const int k = __ffs(lm) - 1;
    lm &= lm - 1u;
    const float4 *pk = reinterpret_cast<const float4 *>(tabs + (size_t)__shfl_sync(kFull, light, k) * tstride);
    float4 A = make_float4(0.f, 0.f, 0.f, 0.f), B = A;
    if (lane < np) { A = pk[2 * (p0 + lane)]; B = pk[2 * (p0 + lane) + 1]; }
    const float2 X = make_float2(A.x, A.y), Y = make_float2(A.z, A.w), Z = make_float2(B.x, B.y), Wv = make_float2(B.z, B.w);
    const float bx = __shfl_sync(kFull, dx, k), by = __shfl_sync(kFull, dy, k), bz = __shfl_sync(kFull, dz, k);
    float2 t = __fmul2_rn(X, make_float2(bx, bx)); t = __ffma2_rn(Y, make_float2(by, by), t); t = __ffma2_rn(Z, make_float2(bz, bz), t);
    const float2 D = __ffma2_rn(t, t, Wv);
    const bool flagged = lane < np && ((fbits(D.x) & fbits(D.y)) & kSign) == 0u;
    const unsigned m = __ballot_sync(kFull, flagged);
    if (lane == k) mine = __brev(m) >> (32 - np);
  }
  return mine;
}
constexpr int kCoopMaxLive = 12;     // a warp with at most this many live rays tests them lane-cooperatively

// ---------------------------------------------------------------------------------------------
// Bundle culling.
//
// Cone of a warp's rays: axis a = normalised sum of the (FP32, unit) directions, cos(theta) = the
// smallest d.a over the active rays, lowered by 2e-6 (FP32 rounding of the dot products and of |a|).
// A ray of the bundle -- extended to a LINE, because include/sphere.h:37 also reports tangent hits
// behind the origin -- can meet a sphere whose centre direction is u and whose angular radius is
// alpha only if |u.a| >= cos(theta + alpha).  Spheres failing that by more than 2e-5 are culled:
// that margin is >= 10x every FP32 error involved (direction 12u, dot 4u, table entries 1u; the
// host rounds cos(alpha) down and sin(alpha) up and inflates r by 1e-6) and ~1e9 x the FP64 rounding
// of the reference's own discriminant, so a culled sphere is a certain miss for the reference.
// Spheres containing the origin carry cos(alpha) = -4 (never culled), padding slots +4 (always).
// Bundles wider than 60 degrees are not culled at all (the caller walks the whole table).
struct Cone { float ax, ay, az, cth, sth; bool ok; };

template <int NR>
__device__ __forceinline__ Cone warp_cone(const float (&dx)[NR], const float (&dy)[NR], const float (&dz)[NR], const bool (&act)[NR]) {
  float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
  for (int r = 0; r < NR; r++)
    if (act[r]) { sx += dx[r]; sy += dy[r]; sz += dz[r]; }
  // any axis is valid (cos(theta) is measured against it), so a fixed-point integer reduction will do
  const float ax = (float)__reduce_add_sync(kFull, __float2int_rn(sx * 65536.f));
  const float ay = (float)__reduce_add_sync(kFull, __float2int_rn(sy * 65536.f));
  const float az = (float)__reduce_add_sync(kFull, __float2int_rn(sz * 65536.f));
  const float l2 = fmaf(az, az, fmaf(ay, ay, ax * ax));
  const float inv = rsqrtf(fmaxf(l2, 1.0f));
  Cone c;
  c.ax = ax * inv; c.ay = ay * inv; c.az = az * inv;
  float mn = 1.0f;
#pragma unroll
  for (int r = 0; r < NR; r++)
    if (act[r]) mn = fminf(mn, fmaf(dz[r], c.az, fmaf(dy[r], c.ay, dx[r] * c.ax)));
  mn = fmaxf(mn, 0.0f);                              // non-negative floats order like their bit patterns
  c.cth = __uint_as_float(__reduce_min_sync(kFull, __float_as_uint(mn))) - 2e-6f;
  c.ok = l2 >= 1.0f && c.cth >= 0.5f;
#ifdef RT_NO_CULL
  c.ok = false;                                      // diagnostics build: every walk covers the whole table
#endif
  c.sth = fmaf(sqrtf(fmaxf(0.0f, fmaf(-c.cth, c.cth, 1.0f))), 1.0001f, 1e-4f);
  return c;
}

// Per-warp compacted table in shared memory: same layout as a shared-origin table, so the chunk test
// and the slow paths run on it unchanged.  kCandMax candidates = one 32-pair chunk per fill.
constexpr int kCandMax = 96;             // room for one more DOUBLE culling round (64 slots) on top of 32 collected candidates
constexpr unsigned kWarpBufBytes = kCandMax * 16 + kCandMax * 4 + 48 + 80;   // pairs | perm | gmin | pad -> 2048 (multiple of 128)
static_assert(kWarpBufBytes % 128 == 0 && kCandMax % 8 == 0, "warp table layout");
struct WarpBuf { float4 *pairs; int *perm; float *gmin; };
__device__ __forceinline__ WarpBuf warp_buf(unsigned char *base) {
  unsigned char *p = base + (threadIdx.x >> 5) * kWarpBufBytes;
  WarpBuf b;
  b.pairs = reinterpret_cast<float4 *>(p);
  b.perm = reinterpret_cast<int *>(p + kCandMax * 16);
  b.gmin = reinterpret_cast<float *>(p + kCandMax * 16 + kCandMax * 4);
  return b;
}

// One culling round: lane l looks at slot base + l of table T.  Survivors (ballot order = table order,
// so the compacted table stays sorted) are copied to positions ncand.. of the warp's table.  `wcut`:
// spheres whose group lies beyond it are dropped as well.  Returns the survivors' ballot mask.
__device__ __forceinline__ unsigned cull_round(const Tab &T, int base, int nslots, const Cone &c, float wcut, const WarpBuf &wb,
                                               int ncand) {
  const int lane = threadIdx.x & 31, slot = base + lane;
  bool keep = false;
  if (slot < nslots) {
    const float4 u = T.cullA[slot];
    const float sA = T.cullB[slot];
    const float dotv = fabsf(fmaf(u.z, c.az, fmaf(u.y, c.ay, u.x * c.ax)));
    keep = !(dotv < fmaf(c.cth, u.w, -fmaf(c.sth, sA, 2e-5f))) && !(T.gmin[slot >> 3] > wcut);
  }
  const unsigned mk = __ballot_sync(kFull, keep);
  if (keep) {
    const int rank = ncand + __popc(mk & ((1u << lane) - 1u));
    const float *src = reinterpret_cast<const float *>(T.pairs) + (slot >> 1) * 8 + (slot & 1);
    float *dst = reinterpret_cast<float *>(wb.pairs) + (rank >> 1) * 8 + (rank & 1);
    dst[0] = src[0]; dst[2] = src[2]; dst[4] = src[4]; dst[6] = src[6];
    wb.perm[rank] = T.perm[slot];
    if ((rank & 7) == 0) wb.gmin[rank >> 3] = T.gmin[slot >> 3];    // lower bound of this and every later key
  }
  return mk;
}
// Two culling rounds at once: lane l looks at slots base + l AND base + 32 + l.  The two cone tests are independent
// dependency chains in one basic block (the single round is bound by its own chain: shared-memory load -> 5 dependent FMAs
// -> compare -> ballot -> compaction), and half the loop iterations, ballots and cut-off checks remain.  Same test, same
// survivor order (table order), so the compacted table is the one two single rounds would have produced.
__device__ __forceinline__ void cull_round2(const Tab &T, int base, int nslots, const Cone &c, float wcut, const WarpBuf &wb, int ncand,
                                            unsigned &mk0, unsigned &mk1) {
  const int lane = threadIdx.x & 31, s0 = base + lane, s1 = s0 + 32;
  const int i0 = min(s0, nslots - 1), i1 = min(s1, nslots - 1);
  const float4 u0 = T.cullA[i0], u1 = T.cullA[i1];
  const float a0 = T.cullB[i0], a1 = T.cullB[i1];
  const float g0 = T.gmin[i0 >> 3], g1 = T.gmin[i1 >> 3];
  const float d0 = fabsf(fmaf(u0.z, c.az, fmaf(u0.y, c.ay, u0.x * c.ax))), d1 = fabsf(fmaf(u1.z, c.az, fmaf(u1.y, c.ay, u1.x * c.ax)));
  const bool keep0 = s0 < nslots && !(d0 < fmaf(c.cth, u0.w, -fmaf(c.sth, a0, 2e-5f))) && !(g0 > wcut);
  const bool keep1 = s1 < nslots && !(d1 < fmaf(c.cth, u1.w, -fmaf(c.sth, a1, 2e-5f))) && !(g1 > wcut);
  mk0 = __ballot_sync(kFull, keep0);
  mk1 = __ballot_sync(kFull, keep1);
  const unsigned lt = (1u << lane) - 1u;
  if (keep0) {
    const int rank = ncand + __popc(mk0 & lt);
    const float *src = reinterpret_cast<const float *>(T.pairs) + (s0 >> 1) * 8 + (s0 & 1);
    float *dst = reinterpret_cast<float *>(wb.pairs) + (rank >> 1) * 8 + (rank & 1);
    dst[0] = src[0]; dst[2] = src[2]; dst[4] = src[4]; dst[6] = src[6];
    wb.perm[rank] = T.perm[s0];
    if ((rank & 7) == 0) wb.gmin[rank >> 3] = g0;
  }
  if (keep1) {
    const int rank = ncand + __popc(mk0) + __popc(mk1 & lt);
    const float *src = reinterpret_cast<const float *>(T.pairs) + (s1 >> 1) * 8 + (s1 & 1);
    float *dst = reinterpret_cast<float *>(wb.pairs) + (rank >> 1) * 8 + (rank & 1);
    dst[0] = src[0]; dst[2] = src[2]; dst[4] = src[4]; dst[6] = src[6];
    wb.perm[rank] = T.perm[s1];
    if ((rank & 7) == 0) wb.gmin[rank >> 3] = g1;
  }
}
// Pads the warp's table to a whole group of 8 spheres with never-hit entries; returns its pair count.
__device__ __forceinline__ int cull_finish(const WarpBuf &wb, int ncand) {
  const int lane = threadIdx.x & 31, padded = (ncand + 7) & ~7, rank = ncand + lane;
  if (rank < padded) {
    float *dst = reinterpret_cast<float *>(wb.pairs) + (rank >> 1) * 8 + (rank & 1);
    dst[0] = 0.f; dst[2] = 0.f; dst[4] = 0.f; dst[6] = -1.0f;
    wb.perm[rank] = -1;
  }
  __syncwarp();
  return padded >> 1;
}

// ---------------------------------------------------------------------------------------------
// CLOSEST HIT, shared origin (camera table, sorted by nearest-point distance).  NR rays per lane.
// The query is resumable over pair ranges so that a table larger than shared memory can be streamed
// through it tile by tile: `pairs` is indexed with ABSOLUTE pair numbers (a tile buffer is passed as
// buffer - 2*first_pair), gmin / perm may live in global memory.
template <int NR>
struct ClosestQ {
  Best best[NR];
  float wcut;                                        // warp-uniform: farthest cutoff of any live ray
};
template <int NR>
__device__ __forceinline__ void closest_begin(ClosestQ<NR> &q) {
#pragma unroll
  for (int r = 0; r < NR; r++) best_init(q.best[r]);
  q.wcut = 3.0e38f;
}

// returns false once every remaining sphere of the (sorted) table is beyond every ray's best hit
template <int NR>
__device__ __forceinline__ bool closest_shared_range(ClosestQ<NR> &q, const float4 *__restrict__ pairs, const float *gmin, const int *perm,
                                                     int pbeg, int pend, const float (&dx)[NR], const float (&dy)[NR],
                                                     const float (&dz)[NR], const bool (&live)[NR], float d64, const double4 *sph64,
                                                     const RaySrc (&src)[NR]) {
  float2 dx2[NR], dy2[NR], dz2[NR];
#pragma unroll
  for (int r = 0; r < NR; r++) { dx2[r] = make_float2(dx[r], dx[r]); dy2[r] = make_float2(dy[r], dy[r]); dz2[r] = make_float2(dz[r], dz[r]); }
#pragma unroll 1
  for (int p0 = pbeg; p0 < pend; p0 += kChunkPairs) {
    if (gmin[p0 / kGroupPairs] > q.wcut) return false;
    const int np = min(kChunkPairs, pend - p0);
    unsigned h[NR], f[NR], any = 0u;
    chunk_test_shared<NR>(pairs, p0, np, dx2, dy2, dz2, h);
#pragma unroll
    for (int r = 0; r < NR; r++) { f[r] = flagged_bits(h[r], np, live[r]); any |= f[r]; }
    if (__any_sync(kFull, any != 0u)) {
      // drain: every lane resolves its own flagged pairs, nearest first, one per iteration
#pragma unroll
      for (int r = 0; r < NR; r++) {
        unsigned fr = f[r];
        while (__any_sync(kFull, fr != 0u)) {
          if (fr != 0u) {
            const int bit = 31 - __clz(fr);
            const int pi = p0 + np - 1 - bit;
            fr &= ~(1u << bit);
            if (gmin[pi / kGroupPairs] > q.best[r].hi) fr = 0u;       // sorted: the rest is farther still
            else q.best[r] = slow_closest_shared(q.best[r], pairs, perm, pi, dx[r], dy[r], dz[r], d64, sph64, src[r]);
          }
        }
      }
      float c = -3.0e38f;
#pragma unroll
      for (int r = 0; r < NR; r++) c = fmaxf(c, live[r] ? q.best[r].hi : -3.0e38f);
      q.wcut = wmaxf(c);
    }
  }
  return true;
}

template <int NR>
__device__ __forceinline__ void closest_shared(const Tab T, int npairs, const float (&dx)[NR], const float (&dy)[NR],
                                               const float (&dz)[NR], const bool (&live)[NR], float d64, const double4 *sph64,
                                               const RaySrc (&src)[NR], Best (&best)[NR]) {
  ClosestQ<NR> q;
  closest_begin(q);
  closest_shared_range<NR>(q, T.pairs, T.gmin, T.perm, 0, npairs, dx, dy, dz, live, d64, sph64, src);
#pragma unroll
  for (int r = 0; r < NR; r++) best[r] = q.best[r];
}

// The same query with bundle culling (T staged in shared memory, wb = this warp's compacted table).
template <int NR>
__device__ __forceinline__ void closest_shared_culled(const Tab T, int npairs, const WarpBuf &wb, const float (&dx)[NR],
                                                      const float (&dy)[NR], const float (&dz)[NR], const bool (&live)[NR], float d64,
                                                      const double4 *sph64, const RaySrc (&src)[NR], Best (&best)[NR],
                                                      unsigned &c_cand, unsigned &c_walks) {
  const Cone cone = warp_cone<NR>(dx, dy, dz, live);
  if (!cone.ok) { closest_shared<NR>(T, npairs, dx, dy, dz, live, d64, sph64, src, best); return; }
  c_walks++;
  ClosestQ<NR> q;
  closest_begin(q);
  const int nslots = 2 * npairs;
  int ncand = 0;
  bool more = true;
  // (the candidates collected so far are walked BEFORE the loop is left at the cut-off: the rounds since the last fill may
  // hold a sphere nearer than the best hit the cut-off was computed from -- found by scripts/fuzz_parity.py on a
  // 1705-sphere scene: a fill, then a round with <= 32 survivors, then the cut-off; tests/test_gpu_parity.py keeps the scene)
  int base = 0;
#pragma unroll 1
  for (;;) {
    const bool last = base >= nslots || T.gmin[base >> 3] > q.wcut;   // nothing further to collect: the table ends, or its
    if (!last) {                                                      // rest is beyond every ray's best hit
      unsigned mk0, mk1;
      cull_round2(T, base, nslots, cone, q.wcut, wb, ncand, mk0, mk1);
      ncand += __popc(mk0) + __popc(mk1);
      base += 64;
      if (ncand <= kCandMax - 64 && base < nslots) continue;
    }
    if (ncand > 0) {
      c_cand += (unsigned)ncand;
      const int np = cull_finish(wb, ncand);
      more = closest_shared_range<NR>(q, wb.pairs, wb.gmin, wb.perm, 0, np, dx, dy, dz, live, d64, sph64, src);
      __syncwarp();
      ncand = 0;
    }
    if (last || !more || base >= nslots) break;
  }
#pragma unroll
  for (int r = 0; r < NR; r++) best[r] = q.best[r];
}

// ---------------------------------------------------------------------------------------------
// CLOSEST HIT, general origin (bounce rays).  Table pair = (cx0,cx1,cy0,cy1) (cz0,cz1,rho0,rho1)
// with recentred centres, index order.  Per sphere: X = c - o, tu = X.d(1+24u) + dtmax (an UPPER
// bound of the true centre projection), q = |X|^2 - rho' (>= 0 => origin strictly outside),
// D' = tu^2 - q.  A sphere is skipped when D' < 0, or when it lies behind an origin that is outside
// it (tu < 0 and q >= 0): that removes the sphere the ray just left without any extra arithmetic.
// kIds: the walk covers the pairs ids[0..npairs) (ascending, npairs even) instead of 0..npairs (closest_general_culled).
template <int NR, bool kIds = false>
__device__ __forceinline__ void closest_general(const float4 *__restrict__ pairs, int npairs, int N, const float (&ox)[NR],
                                                const float (&oy)[NR], const float (&oz)[NR], const float (&dx)[NR],
                                                const float (&dy)[NR], const float (&dz)[NR], const bool (&live)[NR], float d64,
                                                float gS2, float dtmax, const double4 *sph64, const RaySrc (&src)[NR],
                                                Best (&best)[NR], const bool coop = false, const unsigned short *ids = nullptr) {
  const float kInfl = 1.0f + 24.0f * 5.9604645e-8f;
  float2 nox[NR], noy[NR], noz[NR], idx2[NR], idy2[NR], idz2[NR];
  const float2 dtm = make_float2(dtmax, dtmax);
#pragma unroll
  for (int r = 0; r < NR; r++) {
    nox[r] = make_float2(-ox[r], -ox[r]); noy[r] = make_float2(-oy[r], -oy[r]); noz[r] = make_float2(-oz[r], -oz[r]);
    float ix = __fmul_rn(dx[r], kInfl), iy = __fmul_rn(dy[r], kInfl), iz = __fmul_rn(dz[r], kInfl);
    idx2[r] = make_float2(ix, ix); idy2[r] = make_float2(iy, iy); idz2[r] = make_float2(iz, iz);
  }
#pragma unroll 1
  for (int p0 = 0; p0 < npairs; p0 += kChunkPairs) {
    const int np = min(kChunkPairs, npairs - p0);
    unsigned h[NR];
#pragma unroll
    for (int r = 0; r < NR; r++) h[r] = kFull;
    if (NR == 1 && coop) {
      // (flagged bits -> history word: flagged_bits() below inverts it again)
      h[0] = ~coop_chunk_general(pairs, p0, np, nox[0].x, noy[0].x, noz[0].x, idx2[0].x, idy2[0].x, idz2[0].x, dtmax, live[0]);
    } else
#pragma unroll 1
    for (int p = p0; p < p0 + np; p += 2) {
#pragma unroll
      for (int k = 0; k < 2; k++) {
        const int pk = kIds ? (int)ids[p + k] : p + k;
        const float4 A = pairs[2 * pk], B = pairs[2 * pk + 1];
        const float2 CX = make_float2(A.x, A.y), CY = make_float2(A.z, A.w), CZ = make_float2(B.x, B.y);
        const float2 NR_ = make_float2(-B.z, -B.w);
#pragma unroll
        for (int r = 0; r < NR; r++) {
          const float2 x = __fadd2_rn(CX, nox[r]), y = __fadd2_rn(CY, noy[r]), z = __fadd2_rn(CZ, noz[r]);
          float2 t = __ffma2_rn(x, idx2[r], dtm); t = __ffma2_rn(y, idy2[r], t); t = __ffma2_rn(z, idz2[r], t);
          float2 q = __ffma2_rn(x, x, NR_); q = __ffma2_rn(y, y, q); q = __ffma2_rn(z, z, q);
          const float2 D = __ffma2_rn(t, t, make_float2(-q.x, -q.y));
          // rejected  <=>  D' < 0  or  (tu < 0 and q >= 0)
          h[r] = push_sign(h[r], (fbits(D.x) | (fbits(t.x) & ~fbits(q.x))) & (fbits(D.y) | (fbits(t.y) & ~fbits(q.y))));
        }
      }
    }
#pragma unroll
    for (int r = 0; r < NR; r++) {
      unsigned fr = flagged_bits(h[r], np, live[r]);
      while (__any_sync(kFull, fr != 0u)) {
        if (fr != 0u) {
          const int bit = 31 - __clz(fr);
          const int pi = kIds ? (int)ids[p0 + np - 1 - bit] : p0 + np - 1 - bit;
          fr &= ~(1u << bit);
          best[r] = slow_closest_general(best[r], pairs, pi, N, ox[r], oy[r], oz[r], dx[r], dy[r], dz[r], d64, gS2, sph64, src[r]);
        }
      }
    }
  }
}

// The same walk with bundle culling (general table in shared memory; k_closest1 takes 64 consecutive rays of the
// tile-ordered level-1 queue, a strip of neighbouring level-0 tiles, so its rays leave a small region in similar directions).  Bound of the bundle: its directions by the cone
// of warp_cone (axis a, cos/sin theta), its FP32 origins by a ball (centre m = one live ray's origin, radius rb = the
// largest |o - m|, rounded up).  Per pair, each sphere is tested once for the whole warp; a pair is dropped when neither
// sphere can be flagged by the filter above for ANY ray of the bundle, so the surviving pairs -- ascending, in the warp's
// ids[] -- are flagged and decided exactly as in the full walk, in the same order (same hits, same FP64 evaluations).
//
// Margin argument (u = 2^-24; X = c - o with the FP32 table centre c and FP32 origin o taken as exact reals, T = X.d,
// L = |m - c| + rb >= |X|):
//   * tu - T <= Dl = dtmax + 64u L: the filter's tu = fl(X).d(1 + 24u) + dtmax is an upper bound of T by construction;
//     fl(X) (u|X|), the inflated direction (25u |X|) and three FMA roundings add at most 32u |X| more.
//   * q >= |X|^2 (1 - 8u) - rho' (1 + 8u)   (fl(X) and three FMA roundings).
//   * |d| = 1 +- 3u (FP32 of an exact unit vector): the distance of c from the line is h^2 = |X|^2 - T^2 / |d|^2
//     <= |X|^2 - T^2 + 7u L^2.
//   Flagged with T >= 0 (tu >= 0, tu^2 >= q): h^2 <= rho' (1 + 8u) + 2 L Dl + Dl^2 + 15u L^2 <= Re^2 with
//     Re^2 = rho' (1 + 16u) + 2 L Dl + Dl^2 + 64u L^2: the FORWARD ray from o passes within Re of c.
//   Flagged with T < 0: then 0 <= tu < Dl, so |X|^2 <= Re^2: o lies within Re of c.  (Flagged because q < 0: the same.)
//   Shift by o - m (|o - m| <= rb): the forward ray from m with the same direction meets the ball B(c, R2), R2 = Re + rb.
//   m outside that ball (|c - m| = dist > R2): the directions from m that meet it form a cone of half-angle alpha around
//   (c - m) / dist, sin alpha = R2 / dist; it meets the bundle's cone iff angle(a, c - m) <= theta + alpha (theta <= 60,
//   alpha < 90 degrees: cos is monotonic there), i.e. (c - m).a >= cos(theta) sqrt(dist^2 - R2^2) - sin(theta) R2.
//   A sphere is culled when that fails by more than 2e-5 (dist + R2): >= 100x the FP32 errors of this test itself (the
//   rounding of c - m, the dot product, dist; cos theta is already lowered and sin theta raised by warp_cone, R2 is rounded
//   up, the square root rounded down).  So a culled sphere is rejected by the filter for every ray of the bundle.
// Only the forward ray matters: the filter rejects a sphere behind an origin outside it (the tangent-behind case of
// include/sphere.h:37 is not reproduced by the general filter in the first place, DESIGN.md section 4).
// ids: this warp's kGenIds 16-bit slots; survivors are walked in batches of at most kGenIds - 1 (+1: a culled pair pads
// an odd count to the even length the packed loop needs -- it is rejected for every ray, so its bit never drains).
constexpr int kGenIds = 96;
template <int NR>
__device__ __forceinline__ void closest_general_culled(const float4 *__restrict__ pairs, int npairs, int N, const float (&ox)[NR],
                                                       const float (&oy)[NR], const float (&oz)[NR], const float (&dx)[NR],
                                                       const float (&dy)[NR], const float (&dz)[NR], const bool (&live)[NR], float d64,
                                                       float gS2, float dtmax, const double4 *sph64, const RaySrc (&src)[NR],
                                                       Best (&best)[NR], unsigned short *ids, unsigned &c_cand, unsigned &c_walks) {
  const Cone cone = warp_cone<NR>(dx, dy, dz, live);
  if (!cone.ok) { closest_general<NR>(pairs, npairs, N, ox, oy, oz, dx, dy, dz, live, d64, gS2, dtmax, sph64, src, best); return; }
  c_walks++;
  const int lane = threadIdx.x & 31;
  // the ball: centre = the origin of one live ray (cone.ok: the warp has one), radius rounded up
  bool any = false;
  float mx = 0.f, my = 0.f, mz = 0.f;
#pragma unroll
  for (int r = NR - 1; r >= 0; r--)
    if (live[r]) { any = true; mx = ox[r]; my = oy[r]; mz = oz[r]; }
  const int ml = __ffs(__ballot_sync(kFull, any)) - 1;
  mx = __shfl_sync(kFull, mx, ml); my = __shfl_sync(kFull, my, ml); mz = __shfl_sync(kFull, mz, ml);
  float rb = 0.f;
#pragma unroll
  for (int r = 0; r < NR; r++)
    if (live[r]) {
      const float ex = __fsub_rn(ox[r], mx), ey = __fsub_rn(oy[r], my), ez = __fsub_rn(oz[r], mz);
      rb = fmaxf(rb, __fsqrt_ru(__fmaf_ru(ez, ez, __fmaf_ru(ey, ey, __fmul_ru(ex, ex)))));
    }
  rb = __fmul_ru(__uint_as_float(__reduce_max_sync(kFull, __float_as_uint(rb))), 1.00001f);   // (non-negative: bit order)
  const float u = 5.9604645e-8f;
  auto keep = [&](float cx, float cy, float cz, float rho) -> bool {
    const float wx = __fsub_rn(cx, mx), wy = __fsub_rn(cy, my), wz = __fsub_rn(cz, mz);
    const float d2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx)), dist = sqrtf(d2);
    const float Lx = __fadd_ru(__fmul_ru(dist, 1.0001f), rb);
    const float Dl = __fmaf_ru(64.0f * u, Lx, dtmax);
    const float re2 = __fmaf_ru(Dl, Dl, __fmaf_ru(__fmul_ru(2.0f, Lx), Dl, __fmaf_ru(__fmul_ru(64.0f * u, Lx), Lx, __fmul_ru(rho, 1.0f + 16.0f * u))));
    const float R2 = __fadd_ru(__fmul_ru(__fsqrt_ru(re2), 1.00001f), rb);
    const float R22 = __fmul_ru(R2, R2), d2lo = __fmul_rd(d2, 0.99998f);
    if (!(d2lo > R22)) return true;                                // (written so that a NaN keeps the sphere)
    const float wa = fmaf(wz, cone.az, fmaf(wy, cone.ay, wx * cone.ax));
    return wa >= cone.cth * __fsqrt_rd(__fsub_rd(d2lo, R22)) - cone.sth * R2 - 2e-5f * (dist + R2);
  };
  const unsigned lt = (1u << lane) - 1u;
  int n = 0, spare = 0;
#pragma unroll 1
  for (int base = 0; base < npairs; base += 32) {
    const int p = base + lane;
    bool k = false;
    if (p < npairs) {
      const float4 A = pairs[2 * p], B = pairs[2 * p + 1];
      k = (2 * p < N && keep(A.x, A.z, B.x, B.z)) || (2 * p + 1 < N && keep(A.y, A.w, B.y, B.w));
    }
    const unsigned km = __ballot_sync(kFull, k), cm = __ballot_sync(kFull, p < npairs && !k);
    if (k) ids[n + __popc(km & lt)] = (unsigned short)p;
    n += __popc(km);
    if (cm) spare = base + 31 - __clz(cm);
    if (n + 33 <= kGenIds && base + 32 < npairs) continue;
    // (the batch saw whole 32-pair rounds or ended at npairs, a multiple of kGroupPairs: an even number of pairs, so an odd
    // n means that one of them was culled, and `spare` names a culled pair)
    c_cand += 2u * (unsigned)n;                                     // (spheres, as the level-0 counts)
    if (n & 1) { if (lane == 0) ids[n] = (unsigned short)spare; n++; }
    __syncwarp();
    if (n > 0) {
      closest_general<NR, true>(pairs, n, N, ox, oy, oz, dx, dy, dz, live, d64, gS2, dtmax, sph64, src, best, false, ids);
      __syncwarp();
    }
    n = 0;
  }
}

// ---------------------------------------------------------------------------------------------
// SHADOW (any hit, early out), light table sorted by distance from the light.  dl = unit vector FROM
// THE LIGHT TOWARDS the shaded point, so = distance light -> shadow-ray origin (= |L-p| - EPS), both
// FP32 with known error.  Roots s are measured from the light; the reference's t = so - s
// (include/scene.h:70-85):   occluded  <=>  (-EPS < s2 <= so)  or  (s2 > so and -EPS < s1 <= so).
// self[r] / cosl[r]: the sphere the point lies on and n.light_dir there.  Its surface passes through
// the point, so the filter flags it for every query; on its lit side it cannot occlude (the shadow
// origin is outside it and moving away), so its flag is cleared up front unless its pair partner
// is a candidate too.  p64[r] points at the exact hit point (only read if FP64 is needed).
template <int NR>
struct ShadowQ {
  bool open[NR], occ[NR];                            // still undecided / found an occluder
  float m[NR], cut[NR], wcut;
  int tslot[NR];                                     // slot of the lit self sphere in this light's table, or -1
  int sslot[NR];                                     // ... its position in the table shadow_range is walking, or -1
};
template <int NR>
__device__ __forceinline__ void shadow_begin(ShadowQ<NR> &q, const int *inv, const float (&so)[NR], const bool (&want)[NR],
                                             const int (&self)[NR], const float (&cosl)[NR]) {
  float c = -3.0e38f;
#pragma unroll
  for (int r = 0; r < NR; r++) {
    q.open[r] = want[r]; q.occ[r] = false;
    q.m[r] = __fmaf_ru(1.9073486e-6f, so[r] + kEps, 1e-7f);   // 2^-19 |L-p|: covers the FP32 length error
    q.cut[r] = want[r] ? so[r] + q.m[r] : -3.0e38f;           // nothing farther from the light can matter
    q.tslot[r] = (want[r] && cosl[r] > 1e-3f) ? (inv[self[r]] & 0x3fffffff) : -1;
    q.sslot[r] = q.tslot[r];
    c = fmaxf(c, q.cut[r]);
  }
  q.wcut = wmaxf(c);
}

// returns false once the warp needs nothing further from this (sorted) table
// kMixed: every lane walks the table of ITS OWN light (pairs / gmin / perm / light differ per lane; all tables have the same
// shape), so "nothing further" is a vote over the lanes' own cut-offs instead of one comparison with the warp's;
// mixed_tabs / tstride: where table t starts (for the lane-cooperative chunk test of that mode)
template <int NR, bool kMixed = false>
__device__ __forceinline__ bool shadow_range(ShadowQ<NR> &q, const float4 *__restrict__ pairs, const float *gmin, const int *perm, int pbeg,
                                             int pend, int light, const float (&dx)[NR], const float (&dy)[NR], const float (&dz)[NR],
                                             const float (&so)[NR], const int (&self)[NR], const float (&cosl)[NR],
                                             const double *const (&p64)[NR], float d64, const double4 *sph64, int &n_fp64,
                                             const bool coop = false, const unsigned char *mixed_tabs = nullptr, unsigned tstride = 0u,
                                             unsigned long long *prof = nullptr) {
  float2 dx2[NR], dy2[NR], dz2[NR];
#pragma unroll
  for (int r = 0; r < NR; r++) { dx2[r] = make_float2(dx[r], dx[r]); dy2[r] = make_float2(dy[r], dy[r]); dz2[r] = make_float2(dz[r], dz[r]); }
#pragma unroll 1
  for (int p0 = pbeg; p0 < pend; p0 += kChunkPairs) {
    if (kMixed) { if (!__any_sync(kFull, q.open[0] && !(gmin[p0 / kGroupPairs] > q.cut[0]))) return false; }
    else if (gmin[p0 / kGroupPairs] > q.wcut) return false;
    const int np = min(kChunkPairs, pend - p0);
    unsigned h[NR], f[NR], any = 0u;
    long long pt0 = 0;
    if (prof) pt0 = clock64();
    if (NR == 1 && kMixed && coop) h[0] = ~coop_chunk_mixed(mixed_tabs, tstride, light, p0, np, dx[0], dy[0], dz[0], q.open[0]);
    else if (NR == 1 && coop) h[0] = ~coop_chunk_shared(pairs, p0, np, dx[0], dy[0], dz[0], q.open[0]);
    else chunk_test_shared<NR>(pairs, p0, np, dx2, dy2, dz2, h);
#pragma unroll
    for (int r = 0; r < NR; r++) {
      f[r] = flagged_bits(h[r], np, q.open[r]);
      const int sp = q.sslot[r] >> 1;                // pair of the lit self sphere (or -1)
      if (sp >= p0 && sp < p0 + np) {
        const int ph = (q.sslot[r] & 1) ^ 1;         // partner = the other half of the pair
        const float4 A = pairs[2 * sp], B = pairs[2 * sp + 1];
        float tca, Dp;
        shared_origin_eval(ph ? A.y : A.x, ph ? A.w : A.z, ph ? B.y : B.x, ph ? B.w : B.z, dx[r], dy[r], dz[r], tca, Dp);
        if (!(Dp >= 0.0f)) f[r] &= ~(1u << (p0 + np - 1 - sp));
      }
      any |= f[r];
    }
    if (prof) { const long long t = clock64(); prof[0] += (unsigned long long)(t - pt0); prof[3]++; pt0 = t; }
    if (__any_sync(kFull, any != 0u)) {
#pragma unroll
      for (int r = 0; r < NR; r++) {
        unsigned fr = f[r];
        while (__any_sync(kFull, fr != 0u)) {
          if (prof) prof[2]++;
          if (fr != 0u) {
            const int bit = 31 - __clz(fr);
            const int pi = p0 + np - 1 - bit;
            fr &= ~(1u << bit);
            if (gmin[pi / kGroupPairs] > q.cut[r]) {
              fr = 0u;                                // sorted: everything after this pair is farther still
            } else {
              const int rc = slow_shadow(pairs, perm, pi, dx[r], dy[r], dz[r], so[r], q.m[r], self[r], cosl[r], p64[r], light, d64, sph64);
              n_fp64 += rc >> 1;
              if (rc & 1) { q.occ[r] = true; q.open[r] = false; fr = 0u; }
            }
          }
        }
      }
      float c = -3.0e38f;
#pragma unroll
      for (int r = 0; r < NR; r++) c = fmaxf(c, q.open[r] ? q.cut[r] : -3.0e38f);   // decided rays stop holding the warp
      q.wcut = wmaxf(c);
      if (prof) prof[1] += (unsigned long long)(clock64() - pt0);
      if (q.wcut < -1.0e38f) return false;
    }
  }
  return true;
}

template <int NR>
__device__ __forceinline__ void shadow_light(const Tab T, int npairs, int light, const float (&dx)[NR], const float (&dy)[NR],
                                             const float (&dz)[NR], const float (&so)[NR], const bool (&want)[NR],
                                             const int (&self)[NR], const float (&cosl)[NR], const double *const (&p64)[NR], float d64,
                                             const double4 *sph64, bool (&occ)[NR], int &n_fp64, const bool coop = false) {
  ShadowQ<NR> q;
  shadow_begin<NR>(q, T.inv, so, want, self, cosl);
  shadow_range<NR>(q, T.pairs, T.gmin, T.perm, 0, npairs, light, dx, dy, dz, so, self, cosl, p64, d64, sph64, n_fp64, coop);
#pragma unroll
  for (int r = 0; r < NR; r++) occ[r] = q.occ[r];
}

// One any-hit query PER LANE, each towards its own light (the tail kernel packs the (hit, light) queries of a warp onto
// its lanes: ceil(hits x L / 32) walks instead of L walks with the lanes of the missed rays idle).  Same chunk tests, same
// slow paths and deciders per (ray, sphere) as shadow_light, so the same booleans.
__device__ __forceinline__ bool shadow_mixed(const unsigned char *tabs, const FastArgs &a, int light, float dx, float dy, float dz, float so,
                                             bool want, int self, float cosl, const double *p64, int &n_fp64, const bool coop,
                                             unsigned long long *prof = nullptr) {
  const Tab T = tab_at(tabs, a, light);
  const float dxa[1] = {dx}, dya[1] = {dy}, dza[1] = {dz}, soa[1] = {so}, cosla[1] = {cosl};
  const bool wanta[1] = {want};
  const int selfa[1] = {self};
  const double *const pa[1] = {p64};
  ShadowQ<1> q;
  shadow_begin<1>(q, T.inv, soa, wanta, selfa, cosla);
  shadow_range<1, true>(q, T.pairs, T.gmin, T.perm, 0, a.npairs, light, dxa, dya, dza, soa, selfa, cosla, pa, a.d64, a.r.sph64, n_fp64, coop, tabs,
                        a.tstride, prof);
  return q.occ[0];
}

// The same query with bundle culling (T staged in shared memory, wb = this warp's compacted table).
template <int NR>
__device__ __forceinline__ void shadow_light_culled(const Tab T, int npairs, const WarpBuf &wb, int light, const float (&dx)[NR],
                                                    const float (&dy)[NR], const float (&dz)[NR], const float (&so)[NR],
                                                    const bool (&want)[NR], const int (&self)[NR], const float (&cosl)[NR],
                                                    const double *const (&p64)[NR], float d64, const double4 *sph64, bool (&occ)[NR],
                                                    int &n_fp64, unsigned &c_cand, unsigned &c_walks) {
  const Cone cone = warp_cone<NR>(dx, dy, dz, want);
  if (!cone.ok) { shadow_light<NR>(T, npairs, light, dx, dy, dz, so, want, self, cosl, p64, d64, sph64, occ, n_fp64); return; }
  c_walks++;
  ShadowQ<NR> q;
  shadow_begin<NR>(q, T.inv, so, want, self, cosl);
#pragma unroll
  for (int r = 0; r < NR; r++) q.sslot[r] = -1;
  const int nslots = 2 * npairs;
  int ncand = 0;
  bool more = true;
#pragma unroll 1
  for (int base = 0; base < nslots && more; base += 64) {
    bool beyond = T.gmin[base >> 3] > q.wcut;        // the rest of the table is farther from the light than every open point
    if (!beyond) {
      unsigned mk0, mk1;
      cull_round2(T, base, nslots, cone, q.wcut, wb, ncand, mk0, mk1);
#pragma unroll
      for (int r = 0; r < NR; r++) {                 // where did this ray's lit self sphere go?
        const unsigned b = (unsigned)(q.tslot[r] - base);
        if (b < 32u) { if ((mk0 >> b) & 1u) q.sslot[r] = ncand + __popc(mk0 & ((1u << b) - 1u)); }
        else if (b < 64u) { if ((mk1 >> (b - 32u)) & 1u) q.sslot[r] = ncand + __popc(mk0) + __popc(mk1 & ((1u << (b - 32u)) - 1u)); }
      }
      ncand += __popc(mk0) + __popc(mk1);
      beyond = base + 32 < nslots && T.gmin[(base + 32) >> 3] > q.wcut;   // (the second half already ran into the cut-off)
    }
    if (beyond || ncand > kCandMax - 64 || base + 64 >= nslots) {
      if (ncand > 0) {
        c_cand += (unsigned)ncand;
        const int np = cull_finish(wb, ncand);
        more = shadow_range<NR>(q, wb.pairs, wb.gmin, wb.perm, 0, np, light, dx, dy, dz, so, self, cosl, p64, d64, sph64, n_fp64);
        __syncwarp();
        ncand = 0;
#pragma unroll
        for (int r = 0; r < NR; r++) q.sslot[r] = -1;
      }
      if (beyond) break;
    }
  }
#pragma unroll
  for (int r = 0; r < NR; r++) occ[r] = q.occ[r];
}

// ---------------------------------------------------------------------------------------------
// LBVH queries (large scenes).  Per lane: the traversal (bvh.cuh) names candidate spheres, each candidate
// goes through the SAME slow paths as a flagged sphere of a table walk (the pair it sits in is evaluated
// as a whole: its partner is a real sphere too, so considering it can only confirm the right answer).
// Forward traversal only: the include/sphere.h:37 oddity (a ray whose LINE is exactly tangent to a sphere
// BEHIND its origin counts as a hit with t < 0) is not reproduced in this mode, as in closest_general.
__device__ __forceinline__ float3 recentred(const FastArgs &a, const double *p) {
  return make_float3((float)(p[0] - a.c0[0]), (float)(p[1] - a.c0[1]), (float)(p[2] - a.c0[2]));
}
// closest hit of a ray from the shared origin O of table T (camera)
__device__ __forceinline__ Best bvh_closest_shared(const FastArgs &a, const Tab T, float3 o, float dx, float dy, float dz, RaySrc src) {
  Best b;
  best_init(b);
  const rtb::BvhRay r = rtb::bvh_ray(o.x, o.y, o.z, dx, dy, dz);
  auto leaf = [&](int i) {
    const int slot = __ldg(&T.inv[i]) & 0x3fffffff;
    b = slow_closest_shared(b, T.pairs, T.perm, slot >> 1, dx, dy, dz, a.d64, a.r.sph64, src);
    return b.idx >= 0 ? __fmaf_ru(b.hi, 1e-6f, b.hi) + 1e-6f : 3.0e38f;
  };
  float t1 = 3.0e38f;
#pragma unroll 1
  for (int k = 0; k < a.nbig; k++) t1 = leaf(a.big[k]);      // first: their hit distance prunes the traversal
  rtb::bvh_traverse(a.bvh, r, -1e-3f, t1, leaf);
  return b;
}
// closest hit of a general-origin ray (recentred FP32 origin o)
__device__ __forceinline__ Best bvh_closest_general(const FastArgs &a, const float4 *gen, float ox, float oy, float oz, float dx, float dy,
                                                    float dz, RaySrc src) {
  Best b;
  best_init(b);
  const rtb::BvhRay r = rtb::bvh_ray(ox, oy, oz, dx, dy, dz);
  auto leaf = [&](int i) {
    b = slow_closest_general(b, gen, i >> 1, a.N, ox, oy, oz, dx, dy, dz, a.d64, a.gS2, a.r.sph64, src);
    return b.idx >= 0 ? __fmaf_ru(b.hi, 1e-6f, b.hi) + 1e-6f : 3.0e38f;
  };
  float t1 = 3.0e38f;
#pragma unroll 1
  for (int k = 0; k < a.nbig; k++) t1 = leaf(a.big[k]);
  rtb::bvh_traverse(a.bvh, r, -1e-3f, t1, leaf);
  return b;
}
// any-hit shadow query, traversed FROM THE LIGHT (origin o = light, recentred) along dl up to the shaded point
__device__ __forceinline__ bool bvh_shadow(const FastArgs &a, const Tab T, float3 o, int light, float dx, float dy, float dz, float so, int self,
                                           float cosl, const double *p64, int &n_fp64) {
  const float m = __fmaf_ru(1.9073486e-6f, so + kEps, 1e-7f);           // as in shadow_begin
  bool occ = false;
  const rtb::BvhRay r = rtb::bvh_ray(o.x, o.y, o.z, dx, dy, dz);
  const float t1 = so + m;
  auto leaf = [&](int i) {
    const int slot = __ldg(&T.inv[i]) & 0x3fffffff;
    const int rc = slow_shadow(T.pairs, T.perm, slot >> 1, dx, dy, dz, so, m, self, cosl, p64, light, a.d64, a.r.sph64);
    n_fp64 += rc >> 1;
    if (rc & 1) occ = true;
    return occ ? -3.0e38f : t1;
  };
#pragma unroll 1
  for (int k = 0; k < a.nbig && !occ; k++) leaf(a.big[k]);
  if (!occ) rtb::bvh_traverse(a.bvh, r, -(kEps + m), t1, leaf);
  return occ;
}

// ---------------------------------------------------------------------------------------------
// BUNDLE TRAVERSAL of the LBVH: bundle culling (see cull_round) for scenes too large for a table scan.  The warp's
// ray bundle descends the hierarchy BREADTH FIRST with the lanes working on 32 frontier nodes at a time: a child
// survives when the interval-arithmetic slab test (bundle_slab) cannot exclude that some ray of the bundle touches its
// (inflated) box within the distance cutoff.  Surviving leaves name candidate spheres; these are gathered into the warp's compacted table
// (any order: its group minima are -inf, so nothing relies on sortedness) and the unchanged chunk test + slow paths
// run over it.  O(candidates x depth / 32) warp steps instead of one traversal per ray.  Coherent bundles only
// (camera tiles, the shadow rays of one hit block): incoherent ones use the per-lane traversals above.
constexpr int kFront = 192;                          // frontier capacity (nodes per BVH level that touch the cone)
constexpr int kCandList = 128;                       // candidate list capacity; processed (and emptied) in fills of kCandMax
constexpr int kBundleMaxCand = 1 << 20;              // candidate budget of one bundle (measured: giving up early at 96 did not pay; the frontier bound decides)
constexpr unsigned kBundleBufBytes = (2 * kFront + kCandList) * 4;
struct BundleBuf { int *cur, *nxt, *cand; };
__device__ __forceinline__ BundleBuf bundle_buf(unsigned char *base) {
  int *p = reinterpret_cast<int *>(base + (threadIdx.x >> 5) * kBundleBufBytes);
  BundleBuf b;
  b.cur = p; b.nxt = p + kFront; b.cand = p + 2 * kFront;
  return b;
}
// The bundle as a "direction box": per axis the interval [1/d] of the reciprocal direction components of its rays
// (+-inf when the components change sign: no constraint from that axis).  bundle_slab is the slab test in interval
// arithmetic: a lower bound of every ray's entry distance and an upper bound of every exit distance; the box can be
// touched by SOME ray of the bundle only if these overlap -- conservative, and tight for coherent rays even for the
// elongated boxes of the upper levels (a bounding-sphere test lets most of them through).
struct BundleBox { float ox, oy, oz, ilo[3], ihi[3]; };
__device__ __forceinline__ float wredf(float v, bool want_max) {
  int i = __float_as_int(v);
  i = i >= 0 ? i : i ^ 0x7fffffff;                   // order-preserving map float -> int
  i = want_max ? __reduce_max_sync(kFull, i) : __reduce_min_sync(kFull, i);
  return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff);
}
template <int NR>
__device__ __forceinline__ BundleBox bundle_box(float3 o, const float (&dx)[NR], const float (&dy)[NR], const float (&dz)[NR], const bool (&act)[NR]) {
  float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f};
#pragma unroll
  for (int r = 0; r < NR; r++)
    if (act[r]) {
      lo[0] = fminf(lo[0], dx[r]); hi[0] = fmaxf(hi[0], dx[r]);
      lo[1] = fminf(lo[1], dy[r]); hi[1] = fmaxf(hi[1], dy[r]);
      lo[2] = fminf(lo[2], dz[r]); hi[2] = fmaxf(hi[2], dz[r]);
    }
  BundleBox b;
  b.ox = o.x; b.oy = o.y; b.oz = o.z;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float dl = wredf(lo[k], false) - 2e-6f, dh = wredf(hi[k], true) + 2e-6f;   // 12u direction error and more
    if (dl <= 0.f && dh >= 0.f) { b.ilo[k] = -INFINITY; b.ihi[k] = INFINITY; }
    else {
      const float i0 = __frcp_rn(dl), i1 = __frcp_rn(dh);
      const float mn = fminf(i0, i1), mx = fmaxf(i0, i1);
      b.ilo[k] = mn - fabsf(mn) * 1e-6f; b.ihi[k] = mx + fabsf(mx) * 1e-6f;
    }
  }
  return b;
}
// lower bound of the entry distance of any ray of the bundle into the box, or 3e38 when no ray with t in [t0, t1] can touch it
__device__ __forceinline__ float bundle_slab(const BundleBox &b, float lx, float ly, float lz, float hx, float hy, float hz, float t0, float t1) {
  float tn = -3.0e38f, tf = 3.0e38f;
  const float lo[3] = {lx - b.ox, ly - b.oy, lz - b.oz}, hi[3] = {hx - b.ox, hy - b.oy, hz - b.oz};
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float a0 = lo[k] * b.ilo[k], a1 = lo[k] * b.ihi[k], a2 = hi[k] * b.ilo[k], a3 = hi[k] * b.ihi[k];
    tn = fmaxf(tn, fminf(fminf(a0, a1), fminf(a2, a3)));      // (fminf / fmaxf drop the NaN of 0 * inf)
    tf = fminf(tf, fmaxf(fmaxf(a0, a1), fmaxf(a2, a3)));
  }
  tn = tn - fabsf(tn) * 1e-6f;
  tf = tf + fabsf(tf) * 1e-6f;
  return (tn <= tf && tn <= t1 && tf >= t0) ? tn : 3.0e38f;
}

// Gathers candidates [0, n) (n <= kCandMax) from table T (global memory) into the warp's compacted table; returns its pair count.
__device__ __forceinline__ int bundle_fill(const Tab &T, const int *cand, int n, const WarpBuf &wb) {
  const int lane = threadIdx.x & 31;
  for (int k = lane; k < n; k += 32) {
    const int id = cand[k], slot = __ldg(&T.inv[id]) & 0x3fffffff;
    const float *src = reinterpret_cast<const float *>(T.pairs) + (slot >> 1) * 8 + (slot & 1);
    float *dst = reinterpret_cast<float *>(wb.pairs) + (k >> 1) * 8 + (k & 1);
    dst[0] = __ldg(src); dst[2] = __ldg(src + 2); dst[4] = __ldg(src + 4); dst[6] = __ldg(src + 6);
    wb.perm[k] = id;
  }
  if (lane < kCandMax / 8) wb.gmin[lane] = -3.0e38f;
  return cull_finish(wb, n);
}

// Walks the hierarchy; calls process(n) -- warp-uniform, consumes bb.cand[0, n), returns the new distance cutoff (a
// negative value: the query is finished) -- whenever kCandMax candidates are collected and at the end.  Returns false
// when a frontier overflowed (the caller falls back to per-ray traversal; nothing has been processed then... the
// candidates processed so far are harmless: the queries are resumable and idempotent per sphere).
template <typename F>
__device__ __forceinline__ bool bundle_traverse(const FastArgs &a, const BundleBox &bx, float t0, float wcut, const BundleBuf &bb, F &&process) {
  const int lane = threadIdx.x & 31;
  int ncur = 1, ncand = 0, ntotal = 0;
  if (lane == 0) bb.cur[0] = 0;
  // the spheres kept out of the tree are candidates of every bundle; tested first: a hit on them (the ground) bounds
  // the depth the bundle has to search
  if (a.nbig > 0) {
    if (lane < a.nbig) bb.cand[lane] = a.big[lane];
    __syncwarp();
    wcut = process(a.nbig);
    if (wcut < 0.f) return true;
  }
  __syncwarp();
  int *cur = bb.cur, *nxt = bb.nxt;
  while (ncur > 0) {
    int nnxt = 0;
    for (int base = 0; base < ncur; base += 32) {
      bool p0 = false, p1 = false;
      int c0 = 0, c1 = 0;
      if (base + lane < ncur) {
        const rtb::BvhNode *nd = a.bvh.nodes + cur[base + lane];
        const float4 A = __ldg(&nd->a), B = __ldg(&nd->b), C = __ldg(&nd->c);
        const int4 D = __ldg(&nd->d);
        c0 = D.x; c1 = D.y;
        p0 = bundle_slab(bx, A.x, A.y, A.z, A.w, B.x, B.y, t0, wcut) < 3.0e38f;
        p1 = bundle_slab(bx, B.z, B.w, C.x, C.y, C.z, C.w, t0, wcut) < 3.0e38f;
      }
      // leaves -> candidate list, internal nodes -> next frontier (ballot compaction, child 0 then child 1)
#pragma unroll
      for (int k = 0; k < 2; k++) {
        const bool p = k ? p1 : p0;
        const int ch = k ? c1 : c0;
        const unsigned ml = __ballot_sync(kFull, p && ch < 0), mi = __ballot_sync(kFull, p && ch >= 0);
        const unsigned lt = (1u << lane) - 1u;
        if (nnxt + __popc(mi) > kFront) return false;
        if (p && ch >= 0) nxt[nnxt + __popc(mi & lt)] = ch;
        nnxt += __popc(mi);
        if (p && ch < 0) bb.cand[ncand + __popc(ml & lt)] = ~ch;
        ncand += __popc(ml);
        ntotal += __popc(ml);
        if (ntotal > kBundleMaxCand) return false;     // a wide bundle: per-ray traversals are cheaper from here on
        __syncwarp();
        if (ncand > kCandList - 32) {                  // room for one more ballot's worth is gone: consume one fill now
          wcut = process(kCandMax);
          if (wcut < 0.f) return true;
          const int rem = ncand - kCandMax;            // <= kCandList - kCandMax = 64: two values per lane
          const int v0 = lane < rem ? bb.cand[kCandMax + lane] : 0, v1 = lane + 32 < rem ? bb.cand[kCandMax + lane + 32] : 0;
          __syncwarp();
          if (lane < rem) bb.cand[lane] = v0;
          if (lane + 32 < rem) bb.cand[lane + 32] = v1;
          ncand = rem;
          __syncwarp();
        }
      }
    }
    int *t = cur; cur = nxt; nxt = t;
    ncur = nnxt;
    __syncwarp();
  }
  while (ncand > 0) {
    const int n = min(ncand, kCandMax);
    wcut = process(n);
    if (wcut < 0.f) return true;
    const int rem = ncand - n;
    const int v0 = lane < rem ? bb.cand[n + lane] : 0, v1 = lane + 32 < rem ? bb.cand[n + lane + 32] : 0;
    __syncwarp();
    if (lane < rem) bb.cand[lane] = v0;
    if (lane + 32 < rem) bb.cand[lane + 32] = v1;
    ncand = rem;
    __syncwarp();
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
// warp-ballot compaction: rays still alive are appended densely to the next level's queue
// Guard (compute-sanitizer is not available on this pool, so the kernels check their own queue bounds): a push that
// would run past the queue's capacity is dropped and flagged in the frame's error word instead of written.
enum { RT_GUARD_HIT_BLOCKS = 1u, RT_GUARD_RAY_QUEUE = 2u };
__device__ __forceinline__ void queue_push(bool want, const RayRec &rec, RayRec *q, unsigned int *count, unsigned cap, unsigned int *err) {
  const unsigned mk = __ballot_sync(kFull, want);
  if (mk == 0) return;
  const int lane = threadIdx.x & 31, leader = __ffs(mk) - 1;
  unsigned base = 0;
  if (lane == leader) base = atomicAdd(count, (unsigned)__popc(mk));
  base = __shfl_sync(kFull, base, leader);
  if (base + (unsigned)__popc(mk) > cap) { if (lane == leader) atomicOr(err, (unsigned)RT_GUARD_RAY_QUEUE); return; }
  if (want) q[base + __popc(mk & ((1u << lane) - 1u))] = rec;
}

struct Counters {
  unsigned long long closest, hits, shadow, occluded, fp64, violations;
};

__device__ __forceinline__ void flush_counters(const FastArgs &a, Counters &c, int &n_fp64, int level) {
  if (!a.r.counters) return;
  c.fp64 += (unsigned long long)n_fp64;
  unsigned long long v[6] = {c.closest, c.hits, c.shadow, c.occluded, c.fp64, c.violations};
#pragma unroll
  for (int k = 0; k < 6; k++) v[k] = wsum(v[k]);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&a.r.counters[RT_CNT_CLOSEST], v[0]);
    atomicAdd(&a.r.counters[RT_CNT_HITS], v[1]);
    atomicAdd(&a.r.counters[RT_CNT_SHADOW], v[2]);
    atomicAdd(&a.r.counters[RT_CNT_OCCLUDED], v[3]);
    atomicAdd(&a.r.counters[RT_CNT_FP64], v[4]);
    atomicAdd(&a.r.counters[RT_CNT_VIOLATIONS], v[5]);
    atomicAdd(&a.r.counters[RT_CNT_TESTS], (v[0] + v[2]) * (unsigned long long)a.N);
    if (level < 32) atomicAdd(&a.r.counters[RT_CNT_ALIVE0 + level], v[0]);
  }
  c.closest = c.hits = c.shadow = c.occluded = c.fp64 = c.violations = 0;
  n_fp64 = 0;
}

// ---------------------------------------------------------------------------------------------
// THE TAIL (levels >= wave_levels): reflected rays from the queue, one per lane, <= 32 per warp fetch;
// every lane follows its ray to termination, the queue record is updated in place.  Few rays are
// left at these levels (a few percent of the frame), so the kernel is bound by the latency of one
// warp's chain: closest hit -> exact t / geometry -> shadow queries -> Phong -> reflect.  The shadow
// queries were two thirds of that chain when every light was walked in turn with the lanes of the missed
// rays idle; now the self-shadow shortcut settles the back-facing half and the rest is packed 32 per walk
// (profiles/r02_tail_phase_trace.txt; -DRT_TAIL_TRACE builds the phase stamps in).
#ifndef RT_TAIL_THREADS
#define RT_TAIL_THREADS 128
#endif
#ifndef RT_TAIL_CTAS
#define RT_TAIL_CTAS 3
#endif
constexpr int kTailThreads = RT_TAIL_THREADS;
#ifdef RT_TAIL_TRACE
// diagnostics build only (scripts/probe_tail_trace.py): per warp (first chunk), per level, SM-clock stamps of the phases
constexpr int kTraceWarps = 4096, kTraceLevels = 6, kTraceStamps = 12;
__device__ unsigned long long g_tail_trace[kTraceWarps * kTraceLevels * kTraceStamps];
#define RT_TT(k, extra) do { const unsigned long long x_ = (unsigned long long)(extra);   /* (warp-wide: ballots inside) */ \
    if (tt_on && lane == 0 && level - a.level < kTraceLevels) g_tail_trace[(tt_warp * kTraceLevels + (level - a.level)) * kTraceStamps + (k)] = (unsigned long long)clock64() | (x_ << 48); } while (0)
#define RT_TG(k) do { if (tt_on && lane == 0 && level - a.level < kTraceLevels) { unsigned long long t_; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_)); g_tail_trace[(tt_warp * kTraceLevels + (level - a.level)) * kTraceStamps + (k)] = t_; } } while (0)
#else
#define RT_TT(k, extra) do { } while (0)
#define RT_TG(k) do { } while (0)
#endif
template <bool kSmem, bool kBvh>
__global__ void __launch_bounds__(kTailThreads, RT_TAIL_CTAS) k_bounce(const FastArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  // staged: [L light tables][general table], contiguous in global memory in that order
  const unsigned char *tabs = a.tabs + a.tstride;
  if (kSmem) { stage_tables(smem, tabs, a.stage_bytes); tabs = smem + kSmemHeader; }
  RT_PDL_SYNC();
  const unsigned nq = *a.q_in_count;
  if (nq == 0u) return;                             // nothing survived to this level
  const WarpBuf wb = warp_buf(smem + kSmemHeader + ((a.stage_bytes + 127u) & ~127u));
  const float4 *gen = reinterpret_cast<const float4 *>(tabs + (size_t)a.L * a.tstride);
  const int lane = threadIdx.x & 31;
  const int depth = a.r.max_depth, L = a.L;
  Counters cnt = {0, 0, 0, 0, 0, 0};
  int n_fp64 = 0;
  unsigned c_cand = 0, c_walks = 0;
  RayRec *qin = a.q_in;
  // rays per warp fetch: the queue is spread over ALL resident warps (a warp's chain gets shorter with fewer rays: its
  // drain loops run for the slowest lane, and from kCoopMaxLive live rays down the tests turn lane-cooperative), 32 at most
  const unsigned nwarps = gridDim.x * (unsigned)(kTailThreads / 32);
  const unsigned per = min(32u, max(4u, (nq + nwarps - 1u) / nwarps));
#ifdef RT_TAIL_TRACE
  const unsigned tt_warp = blockIdx.x * (unsigned)(kTailThreads / 32) + (threadIdx.x >> 5);
  bool tt_on = tt_warp < (unsigned)kTraceWarps;
#endif
  for (;;) {
    const int chunk = warp_fetch(a.chunk_counter);
    if ((unsigned)chunk * per >= nq) break;
    const unsigned qi = (unsigned)chunk * per + lane;
    bool live[1] = {(unsigned)lane < per && qi < nq};
    unsigned pix = 0;
    float ox[1] = {0.f}, oy[1] = {0.f}, oz[1] = {0.f}, dx[1] = {0.f}, dy[1] = {0.f}, dz[1] = {0.f};
    float wt = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
    if (live[0]) {
      const RayRec &q = qin[qi];
      // recentred FP32 origin and FP32 direction for the filter (exact values stay in the record)
      ox[0] = (float)(q.ox - a.c0[0]); oy[0] = (float)(q.oy - a.c0[1]); oz[0] = (float)(q.oz - a.c0[2]);
      dx[0] = (float)q.dx; dy[0] = (float)q.dy; dz[0] = (float)q.dz;
      pix = q.pix; wt = q.wt; cr = q.ar; cg = q.ag; cb = q.ab;
    }
    const RaySrc src[1] = {{nullptr, nullptr, 0, 0, qin + qi}};
    for (int level = a.level;; level++) {
      Best best[1];
      best_init(best[0]);
      // few live rays in this warp (the deep levels): the sphere tests run lane-cooperatively (coop_chunk_*)
      const bool coop = kSmem && !kBvh && __popc(__ballot_sync(kFull, live[0])) <= kCoopMaxLive;
      RT_TT(0, __popc(__ballot_sync(kFull, live[0]))); RT_TG(6);
      if (kBvh) { if (live[0]) best[0] = bvh_closest_general(a, gen, ox[0], oy[0], oz[0], dx[0], dy[0], dz[0], src[0]); }
      else closest_general<1>(gen, a.npairs, a.N, ox, oy, oz, dx, dy, dz, live, a.d64, a.gS2, a.g_dtmax, a.r.sph64, src, best, coop);
      RT_TT(1, 0);
      bool hit = false, final_ = false, cont = false;
      int idx[1] = {-1};
      double t64 = 0;
      d3 o64 = rtx::mk(0, 0, 0), d64v = o64;
      if (live[0]) {
        cnt.closest++;
        n_fp64 += best[0].nfp64;
        if (best[0].idx >= 0) {
          const ExactRay e = exact_ray(src[0]);
          // exact FP64 t of the winner (or the brute-force safety net if the filter contradicted itself)
          double t = best[0].t;
          bool ok = best[0].exact;
          if (!ok) { n_fp64++; ok = exact_sphere(a.r.sph64, best[0].idx, e.o, e.d, e.a, t) && t < 1e20; }
          int bi = best[0].idx;
          if (!ok) { cnt.violations++; bi = exact_bruteforce(a.r.sph64, a.N, e.o, e.d, e.a, t); }
          if (bi >= 0) { hit = true; idx[0] = bi; t64 = t; cnt.hits++; }
          o64 = e.o; d64v = e.d;
        }
        if (a.r.hit_idx) a.r.hit_idx[(size_t)pix * depth + level] = idx[0];
        if (!hit) {                                  // sky, src/main.cpp:26-30
          const Rgb sky = sky_colour(dy[0]);
          add_scaled(cr, cg, cb, wt, sky.r, sky.g, sky.b);
          final_ = true;
        }
      }
      RT_TT(2, __popc(__ballot_sync(kFull, hit)));
      // ---- shading of the hit (include/scene.h:89-121 in FP32, shadow booleans exact)
      d3 p = rtx::mk(0, 0, 0);
      float nx = 0.f, ny = 0.f, nz = 0.f, vx = 0.f, vy = 0.f, vz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, backthr = 0.f;
      float4 m = make_float4(0, 0, 0, 0); float2 mx = make_float2(0, 0);
      unsigned smask = 0u;
      if (hit) {
        const HitGeom hg = hit_geometry(a.r.sph64, idx[0], o64, d64v, t64);   // src/main.cpp:32,35
        p = hg.p;
        m = __ldg(&a.r.mat[idx[0]]); mx = __ldg(&a.r.matx[idx[0]]);
        nx = hg.nx; ny = hg.ny; nz = hg.nz;
        // view_dir = normalized(origin - hit) = -d up to rounding (src/main.cpp:38); colour only
        vx = -(float)d64v.x; vy = -(float)d64v.y; vz = -(float)d64v.z;
        sr = g_frame.ambient[0] * m.x; sg = g_frame.ambient[1] * m.y; sb = g_frame.ambient[2] * m.z;
        backthr = -fmaxf(4.0f * kEps * rsqrtf((float)a.r.sph64[idx[0]].w), 1e-4f);          // -4 EPS / r (self-shadow shortcut, see k_shadow)
      }
      RT_TT(3, 0);
#ifdef RT_TAIL_TRACE
      unsigned long long tt_prof[4] = {0ull, 0ull, 0ull, 0ull};
#endif
      // ---- the shadow queries of the warp's hits: occm = occlusion bits of this lane's hit (bit l = light l)
      unsigned long long occm = 0ull;
      const unsigned hm = __ballot_sync(kFull, hit);
      // per hit and light: the self-shadow shortcut (the point faces away from the light and the light is outside its sphere:
      // occluded by that sphere, no walk; see k_shadow) settles about half of the queries; `need` = the lights left to walk
      unsigned long long need = 0ull;
      if (kSmem && !kBvh && hit) {
        for (int l = 0; l < L; l++) {
          const d3 w = rtx::sub(p, ldc3(g_frame.light_pos[l]));
          const float wx = (float)w.x, wy = (float)w.y, wz = (float)w.z;
          const float inv = rsqrtf(fmaf(wz, wz, fmaf(wy, wy, wx * wx)));
          const float cosl = -(nx * (wx * inv) + ny * (wy * inv) + nz * (wz * inv));
          if (cosl < backthr && (tab_at(tabs, a, l).inv[idx[0]] & 0x40000000) != 0) occm |= 1ull << l; else need |= 1ull << l;
        }
      }
      const int Qn = kSmem && !kBvh ? (int)__reduce_add_sync(kFull, (unsigned)__popcll(need)) : 0;
      if (kSmem && !kBvh && L > 1 && (Qn + 31) / 32 < L) {
        // few queries: they are PACKED onto the lanes, 32 per round -- each lane walks the table of its own query's light
        // (shadow_mixed) -- ceil(Qn / 32) walks instead of L walks with the lanes of missed rays and settled queries idle.
        // A round's queries are listed in the warp's scratch table (owner lane << 8 | light); the hit's data comes from
        // its owner lane by shuffle, the answers go back as a ballot.
        int *list = wb.perm;
        unsigned long long rem = need;
        while (__any_sync(kFull, rem != 0ull)) {
          const int c = __popcll(rem);
          int incl = c;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += v; }
          const int excl = incl - c, take = max(0, min(c, 32 - excl));
          unsigned long long taken = 0ull;
          for (int k = 0; k < take; k++) {
            const int l = __ffsll((long long)rem) - 1;
            rem &= rem - 1ull; taken |= 1ull << l;
            list[excl + k] = (lane << 8) | l;
          }
          __syncwarp();
          const int total = min(32, __shfl_sync(kFull, incl, 31));
          const bool act = lane < total;
          const int e = act ? list[lane] : 0;
          __syncwarp();
          const int owner = e >> 8, l = e & 255;
          d3 pq;
          pq.x = __shfl_sync(kFull, p.x, owner); pq.y = __shfl_sync(kFull, p.y, owner); pq.z = __shfl_sync(kFull, p.z, owner);
          const float qnx = __shfl_sync(kFull, nx, owner), qny = __shfl_sync(kFull, ny, owner), qnz = __shfl_sync(kFull, nz, owner);
          const int qself = __shfl_sync(kFull, idx[0], owner);
          float sdx = 0.f, sdy = 0.f, sdz = 0.f, so = 0.f, cosl = 0.f;
          if (act) {
            // direction light -> point: FP64 difference, FP32 normalisation (error <= 12u, see filter_math.cuh)
            const d3 w = rtx::sub(pq, ldc3(g_frame.light_pos[l]));
            const float wx = (float)w.x, wy = (float)w.y, wz = (float)w.z;
            const float l2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx));
            const float inv = rsqrtf(l2);
            sdx = wx * inv; sdy = wy * inv; sdz = wz * inv;
            so = l2 * inv - kEps;
            cosl = -(qnx * sdx + qny * sdy + qnz * sdz);                        // n . light_dir
          }
#ifdef RT_TAIL_TRACE
          const bool o = shadow_mixed(tabs, a, l, sdx, sdy, sdz, so, act, qself, cosl, &pq.x, n_fp64, total <= kCoopMaxLive, tt_prof);
#else
          const bool o = shadow_mixed(tabs, a, l, sdx, sdy, sdz, so, act, qself, cosl, &pq.x, n_fp64, total <= kCoopMaxLive);
#endif
          const unsigned wm = __ballot_sync(kFull, act && o);
          for (int k = 0; taken != 0ull; k++) {          // this lane's queries of the round: list positions excl, excl + 1, ...
            const int l2 = __ffsll((long long)taken) - 1;
            taken &= taken - 1ull;
            if ((wm >> (excl + k)) & 1u) occm |= 1ull << l2;
          }
        }
      } else if (kBvh || hm != 0u) {
        for (int l = 0; l < L; l++) {
          float sdx[1] = {0.f}, sdy[1] = {0.f}, sdz[1] = {0.f}, so[1] = {0.f}, cosl[1] = {0.f};
          bool occ[1] = {false};
          bool shortcut = false;
          if (hit) {
            // direction light -> point: FP64 difference, FP32 normalisation (error <= 12u, see filter_math.cuh)
            const d3 w = rtx::sub(p, ldc3(g_frame.light_pos[l]));
            const float wx = (float)w.x, wy = (float)w.y, wz = (float)w.z;
            const float l2 = fmaf(wz, wz, fmaf(wy, wy, wx * wx));
            const float inv = rsqrtf(l2);
            sdx[0] = wx * inv; sdy[0] = wy * inv; sdz[0] = wz * inv;
            so[0] = l2 * inv - kEps;
            cosl[0] = -(nx * sdx[0] + ny * sdy[0] + nz * sdz[0]);             // n . light_dir
            shortcut = cosl[0] < backthr && (tab_at(tabs, a, l).inv[idx[0]] & 0x40000000) != 0;   // (self-shadow shortcut, see k_shadow)
          }
          const bool want[1] = {hit && !shortcut};
          const double *const pp[1] = {&p.x};
          if (!kBvh && !__any_sync(kFull, want[0])) { if (shortcut) occm |= 1ull << l; continue; }
          if (kBvh) { if (want[0]) occ[0] = bvh_shadow(a, tab_at(tabs, a, l), recentred(a, g_frame.light_pos[l]), l, sdx[0], sdy[0], sdz[0], so[0], idx[0], cosl[0], &p.x, n_fp64); }
          else if (kSmem && coop) shadow_light<1>(tab_at(tabs, a, l), a.npairs, l, sdx, sdy, sdz, so, want, idx, cosl, pp, a.d64, a.r.sph64, occ, n_fp64, true);
          else if (kSmem) shadow_light_culled<1>(tab_at(tabs, a, l), a.npairs, wb, l, sdx, sdy, sdz, so, want, idx, cosl, pp, a.d64, a.r.sph64, occ, n_fp64, c_cand, c_walks);
          else shadow_light<1>(tab_at(tabs, a, l), a.npairs, l, sdx, sdy, sdz, so, want, idx, cosl, pp, a.d64, a.r.sph64, occ, n_fp64);
          if (occ[0] || shortcut) occm |= 1ull << l;
        }
      }
      // ---- Phong of the un-occluded lights (include/scene.h:104-117 in FP32)
      if (hit) {
        cnt.shadow += L; cnt.occluded += __popcll(occm);
        smask = (unsigned)(occm & 0xffffffffull);
        for (int l = 0; l < L; l++)
          if (!((occm >> l) & 1ull)) phong_light(l, p.x, p.y, p.z, nx, ny, nz, vx, vy, vz, m, mx.x, sr, sg, sb);
      }
      RT_TT(4, 0);
#ifdef RT_TAIL_TRACE
      if (tt_on && lane == 0 && level - a.level < kTraceLevels)
        for (int k = 0; k < 4; k++) g_tail_trace[(tt_warp * kTraceLevels + (level - a.level)) * kTraceStamps + 8 + k] = tt_prof[k];
#endif
      // continuation: src/main.cpp:43-55 unrolled front to back
      if (hit) {
        if (a.r.shadow_mask) a.r.shadow_mask[(size_t)pix * a.r.max_depth + level] = smask;
        if (mx.y > 0.5f) {                          // reflectivity > 0, decided in double on the host
          const float refl = m.w, k = __fmul_rn(wt, __fsub_rn(1.0f, refl));
          add_scaled(cr, cg, cb, k, sr, sg, sb);
          wt = __fmul_rn(wt, refl);
          if (level + 1 < a.r.max_depth) {
            RayRec *rec = qin + qi;                 // in place: the exact ray of the next level is re-read from here
            const double4 sc = ld_sph64(&a.r.sph64[idx[0]]);
            reflected_ray_from_center(d64v, p, rtx::mk(sc.x, sc.y, sc.z), rec);
            ox[0] = (float)(rec->ox - a.c0[0]); oy[0] = (float)(rec->oy - a.c0[1]); oz[0] = (float)(rec->oz - a.c0[2]);
            dx[0] = (float)rec->dx; dy[0] = (float)rec->dy; dz[0] = (float)rec->dz;
            cont = true;
          } else {
            final_ = true;                          // depth exhausted: the child contributes black
          }
        } else {
          add_scaled(cr, cg, cb, wt, sr, sg, sb);
          final_ = true;
        }
      }
      if (live[0] && final_) write_final(a.r, pix, cr, cg, cb);
      if (a.r.counters) {
        flush_counters(a, cnt, n_fp64, level);
        if (lane == 0 && c_walks) { atomicAdd(&a.r.counters[RT_CNT_CAND], (unsigned long long)c_cand); atomicAdd(&a.r.counters[RT_CNT_WALKS], (unsigned long long)c_walks); }
        c_cand = c_walks = 0;
      }
      RT_TT(5, __popc(__ballot_sync(kFull, cont))); RT_TG(7);
      live[0] = cont;
      if (!__any_sync(kFull, cont)) break;
    }
#ifdef RT_TAIL_TRACE
    tt_on = false;                                   // (first chunk of the warp only)
#endif
  }
}

}  // namespace rtf
#endif
