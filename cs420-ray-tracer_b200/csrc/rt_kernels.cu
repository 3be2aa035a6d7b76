// rt_kernels.cu -- the single device translation unit of librt_b200.so (sm_100a only).
#include "rt_kernels.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <thread>
#include <tuple>
#include <vector>

// Camera basis, lights and ambient: one copy per device, refreshed by rt_upload_scene.
__constant__ RtFrameConst g_frame;

#include "kernels_exact.cuh"
#include "kernels_fast.cuh"
#include "kernels_wave.cuh"

cudaError_t rtk_set_frame_const(const RtFrameConst *host_const, cudaStream_t stream) {
  return cudaMemcpyToSymbolAsync(g_frame, host_const, sizeof(RtFrameConst), 0, cudaMemcpyHostToDevice, stream);
}

int rtk_launch_exact(const RtRenderArgs &args, cudaStream_t stream) {
  dim3 block(128);
  dim3 grid((args.W + 31) / 32, (args.bands.local_rows + 3) / 4);
  rtk::k_exact<<<grid, block, 0, stream>>>(args);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 1 : -(int)e;
}

// ---------------------------------------------------------------------------------------------
// fast path, host side
namespace {

constexpr size_t kMaxSmemTables = 90 * 1024;    // stage a kernel's tables in shared memory up to this size (2 CTAs/SM stay resident)
constexpr int kCtlWords = rtf::CTL_WORDS;        // device control words per frame, layout: enum CTL_* (kernels_wave.cuh)

#define RTK_TRY(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return -(int)e_; } while (0)

}  // namespace

int rtk_fast_init(int) {
  const int big = 224 * 1024;        // (some kernels carry a little static shared memory on top)
  RTK_TRY(cudaFuncSetAttribute(rtf::k_bounce<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_closest0<rtf::kTabSmem>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_closest0<rtf::kTabStream>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_closest1<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_shadow<rtf::kTabSmem>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_shadow<rtf::kTabStream>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_shadow<rtf::kTabBvh>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtf::k_closest0<rtf::kTabBvh>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
  RTK_TRY(cudaFuncSetAttribute(rtb::k_bvh_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((16 * rtb::kSortThreads + 32) * sizeof(unsigned))));
  return 0;
}

constexpr int RT_MAX_LEVELS_INTERNAL = 32;
constexpr int kBvhAutoSpheres = 1024;   // automatic mode: scenes from this size on are traversed through the LBVH

// Device build of the LBVH (bvh.cuh) over cen[i] = (c_i - C0, r_i) in FP32; eps inflates every box.
// Inputs of the device LBVH build, written ON THE DEVICE from the raw sphere rows (no host loop, no host -> device copy
// of a second sphere array): cen[k] = (c - C0 in FP32, radius rounded up), orig[k] = sphere index, for the spheres that
// are not in `big` (at most 8, ascending k keeps index order).
struct BuildBig { int n; int idx[8]; };
__global__ void k_bvh_inputs(const double *__restrict__ raw, int N, double c0x, double c0y, double c0z, BuildBig big,
                             float4 *__restrict__ cen, int *__restrict__ orig) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int before = 0;
  for (int k = 0; k < big.n; k++) { if (big.idx[k] == i) return; before += big.idx[k] < i; }
  const double *s = raw + (size_t)i * 10;
  cen[i - before] = make_float4((float)(s[0] - c0x), (float)(s[1] - c0y), (float)(s[2] - c0z), __double2float_ru(fabs(s[3])));
  orig[i - before] = i;
}

// the inputs are produced on the device by k_bvh_inputs from the raw rows (raw_dev)
static int bvh_build(RtFastScene *fs, int n, const double *raw_dev, int N_all, const double *c0, const BuildBig &big, float eps,
                     cudaStream_t stream) {
  const int nleaf = (n + rtb::kLeafSize - 1) / rtb::kLeafSize, nint = nleaf > 1 ? nleaf - 1 : 1;
  // one scratch arena and the node array, both kept (grow-only) across uploads: cudaMalloc / cudaFree cost milliseconds
  // each once gigabytes of frame buffers are allocated, and a build needs seventeen arrays
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  int rc = 0;
#define BV(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = -(int)e_; goto done; } } while (0)
  size_t off = 0;
  auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t o_cen = carve((size_t)n * 16), o_orig = carve((size_t)n * 4), o_k0 = carve((size_t)n * 4), o_k1 = carve((size_t)n * 4),
               o_v0 = carve((size_t)n * 4), o_v1 = carve((size_t)n * 4), o_bounds = carve(6 * 4), o_llo = carve((size_t)nleaf * 16),
               o_lhi = carve((size_t)nleaf * 16), o_lkey = carve((size_t)nleaf * 4), o_nlo = carve((size_t)nint * 16),
               o_nhi = carve((size_t)nint * 16), o_left = carve((size_t)nint * 4), o_right = carve((size_t)nint * 4),
               o_pi = carve((size_t)nint * 4), o_pl = carve((size_t)nleaf * 4), o_flags = carve((size_t)nint * 4);
  if (fs->bvh_scratch_cap < off) {
    cudaFree(fs->bvh_scratch); fs->bvh_scratch = nullptr; fs->bvh_scratch_cap = 0;
    if (cudaMalloc(&fs->bvh_scratch, off) != cudaSuccess) return -(int)cudaErrorMemoryAllocation;
    fs->bvh_scratch_cap = off;
  }
  if (fs->bvh_nodes_cap < (size_t)nint * sizeof(rtb::BvhNode)) {
    cudaFree(fs->bvh_nodes_buf); fs->bvh_nodes_buf = nullptr; fs->bvh_nodes_cap = 0;
    if (cudaMalloc(&fs->bvh_nodes_buf, (size_t)nint * sizeof(rtb::BvhNode)) != cudaSuccess) return -(int)cudaErrorMemoryAllocation;
    fs->bvh_nodes_cap = (size_t)nint * sizeof(rtb::BvhNode);
  }
  unsigned char *sc = (unsigned char *)fs->bvh_scratch;
  float4 *d_cen = (float4 *)(sc + o_cen), *leaf_lo = (float4 *)(sc + o_llo), *leaf_hi = (float4 *)(sc + o_lhi),
         *node_lo = (float4 *)(sc + o_nlo), *node_hi = (float4 *)(sc + o_nhi);
  unsigned *keys[2] = {(unsigned *)(sc + o_k0), (unsigned *)(sc + o_k1)}, *leaf_key = (unsigned *)(sc + o_lkey);
  int *vals[2] = {(int *)(sc + o_v0), (int *)(sc + o_v1)}, *d_orig = (int *)(sc + o_orig), *bounds = (int *)(sc + o_bounds),
      *left = (int *)(sc + o_left), *right = (int *)(sc + o_right), *par_i = (int *)(sc + o_pi), *par_l = (int *)(sc + o_pl),
      *flags = (int *)(sc + o_flags);
  fs->bvh_nodes = fs->bvh_nodes_buf;
  BV(cudaEventCreate(&e0)); BV(cudaEventCreate(&e1));
  k_bvh_inputs<<<(N_all + 255) / 256, 256, 0, stream>>>(raw_dev, N_all, c0[0], c0[1], c0[2], big, d_cen, d_orig);
  {
    const int init[6] = {0x7f7fffff, 0x7f7fffff, 0x7f7fffff, (int)0x80800000, (int)0x80800000, (int)0x80800000};   // ord(+max) / ord(-max)
    BV(cudaMemcpyAsync(bounds, init, sizeof(init), cudaMemcpyHostToDevice, stream));
  }
  BV(cudaMemsetAsync(flags, 0, (size_t)nint * 4, stream));
  BV(cudaMemsetAsync(par_l, 0xff, (size_t)nleaf * 4, stream));
  BV(cudaMemsetAsync(par_i, 0xff, (size_t)nint * 4, stream));
  BV(cudaEventRecord(e0, stream));
  {
    const int tb = 256, gb = (n + tb - 1) / tb, gl = (nleaf + tb - 1) / tb;
    rtb::k_bvh_bounds<<<gb < 592 ? gb : 592, tb, 0, stream>>>(d_cen, n, bounds);
    rtb::k_bvh_morton<<<gb, tb, 0, stream>>>(d_cen, n, bounds, keys[0], vals[0]);
    const size_t sort_smem = (16 * rtb::kSortThreads + 32) * sizeof(unsigned);   // (attribute set by rtk_fast_init)
    rtb::k_bvh_sort<<<1, rtb::kSortThreads, sort_smem, stream>>>(keys[0], vals[0], keys[1], vals[1], n, 8);   // 8 x 4 bits, result in [0]
    rtb::k_bvh_leaves<<<gl, tb, 0, stream>>>(d_cen, keys[0], vals[0], n, nleaf, eps, leaf_lo, leaf_hi, leaf_key);
    if (nleaf > 1) {
      rtb::k_bvh_hier<<<(nleaf - 1 + tb - 1) / tb, tb, 0, stream>>>(leaf_key, nleaf, left, right, par_i, par_l);
      rtb::k_bvh_refit<<<gl, tb, 0, stream>>>(nleaf, left, right, par_i, par_l, leaf_lo, leaf_hi, node_lo, node_hi, flags);
    }
    rtb::k_bvh_pack<<<(nint + tb - 1) / tb, tb, 0, stream>>>(nleaf, left, right, vals[0], d_orig, leaf_lo, leaf_hi, node_lo, node_hi, (rtb::BvhNode *)fs->bvh_nodes);
  }
  BV(cudaGetLastError());
  BV(cudaEventRecord(e1, stream));
  BV(cudaStreamSynchronize(stream));
  { float ms = 0; BV(cudaEventElapsedTime(&ms, e0, e1)); fs->bvh_build_ms = ms; }
  fs->bvh_nleaf = nleaf;
done:
#undef BV
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (rc != 0) fs->bvh_nodes = nullptr;
  return rc;
}

// ---------------------------------------------------------------------------------------------
// The bytes of a table slot, defined once for the host build (sorted tables, at upload), k_cam_fill (the sorted camera
// table, rt_set_camera) and k_build_lookup (lookup tables, at upload and rt_set_camera).  The FP32 filter tables are
// computed in double and rounded conservatively (DESIGN.md "filter margins"; error model in filter_math.cuh):
//   shared-origin table for origin O (camera, each light), spheres SORTED by key = |oc| - r (lookup layouts: index order):
//       oc = c_i - O (double -> nearest float), w = round_up(E_i - (|oc|^2 - r_i^2)),
//       E_i = 2.01 * 2^-20 * |oc|^2 + delta64;  gmin[g] = round_down(key of the group's first sphere)
//       perm[slot] = original sphere index (-1 = padding)
//   general table (index order): c' = c_i - C0 (nearest float),
//       rho' = round_up(r^2 (1+40u) + 12u S r + 64u^2 S^2 + delta64)
// Every double operation is one correctly rounded IEEE operation, in the same order on both sides, so host and device
// write the same bytes.  On the device each is an explicit _rn intrinsic, which nvcc never contracts into an FMA; on the
// host it is the plain operator, which stays one rounding only because NVFLAGS (Makefile) compile the host side with
// -ffp-contract=off.  The conversions to float round to nearest, up or down, correctly on both sides.
#ifdef __CUDA_ARCH__
#define RT_RN(device, host) (device)
#else
#define RT_RN(device, host) (host)
#endif
namespace rn {
inline float host_up(double x) {                // smallest float >= x
  float f = (float)x;
  if ((double)f < x) f = std::nextafterf(f, INFINITY);
  return f;
}
inline float host_down(double x) {              // largest float <= x
  float f = (float)x;
  if ((double)f > x) f = std::nextafterf(f, -INFINITY);
  return f;
}
__host__ __device__ __forceinline__ double mul(double a, double b) { return RT_RN(__dmul_rn(a, b), a * b); }
__host__ __device__ __forceinline__ double add(double a, double b) { return RT_RN(__dadd_rn(a, b), a + b); }
__host__ __device__ __forceinline__ double sub(double a, double b) { return RT_RN(__dsub_rn(a, b), a - b); }
__host__ __device__ __forceinline__ double div(double a, double b) { return RT_RN(__ddiv_rn(a, b), a / b); }
__host__ __device__ __forceinline__ double sqrt(double a) { return RT_RN(__dsqrt_rn(a), std::sqrt(a)); }
__host__ __device__ __forceinline__ float to_float(double a) { return RT_RN(__double2float_rn(a), (float)a); }
__host__ __device__ __forceinline__ float up(double a) { return RT_RN(__double2float_ru(a), host_up(a)); }
__host__ __device__ __forceinline__ float down(double a) { return RT_RN(__double2float_rd(a), host_down(a)); }
}  // namespace rn
#undef RT_RN

// Sphere PAIRS are interleaved for the packed FP32x2 test: (x0,x1,y0,y1) (z0,z1,w0,w1).
__host__ __device__ __forceinline__ void put_pair(float4 *pairs, int slot, float x, float y, float z, float w) {
  float4 *A = pairs + (size_t)(slot >> 1) * 2, *B = A + 1;
  if (slot & 1) { A->y = x; A->w = y; B->y = z; B->w = w; } else { A->x = x; A->z = y; B->x = z; B->z = w; }
}

// oc = c - O of a row (cx, cy, cz, r, ...), |oc|^2, and the sort key |oc| - |r|
struct Oc { double x, y, z, oc2; };
__host__ __device__ __forceinline__ Oc offset(const double *row, const double O[3]) {
  Oc v;
  v.x = rn::sub(row[0], O[0]); v.y = rn::sub(row[1], O[1]); v.z = rn::sub(row[2], O[2]);
  v.oc2 = rn::add(rn::add(rn::mul(v.x, v.x), rn::mul(v.y, v.y)), rn::mul(v.z, v.z));
  return v;
}
__host__ __device__ __forceinline__ double sort_key(const Oc &v, const double *row) { return rn::sub(rn::sqrt(v.oc2), fabs(row[3])); }

// Byte layout of a shared-origin table (RtFastScene)
struct TabLayout { unsigned tstride, gmin_off, perm_off, inv_off, cullA_off, cullB_off; };

// Slot `slot` of the shared-origin table at `base` seen from O: sphere i with row[0..3] = (cx, cy, cz, r), or padding
// when i < 0.  The slot heading a group also writes the group's gmin.  kSorted: a table sorted by key, with cull data
// (table scenes); else a lookup table of an LBVH scene in index order without cull data (nothing walks it in order,
// the hierarchy names the candidates).
template <bool kSorted>
__host__ __device__ __forceinline__ void shared_origin_slot(unsigned char *base, const TabLayout &t, int slot, int i, const double *row,
                                                            const double O[3], double delta64) {
  float4 *pairs = reinterpret_cast<float4 *>(base);
  float *gmin = reinterpret_cast<float *>(base + t.gmin_off);
  int *perm = reinterpret_cast<int *>(base + t.perm_off), *inv = reinterpret_cast<int *>(base + t.inv_off);
  float4 *cullA = reinterpret_cast<float4 *>(base + t.cullA_off);
  float *cullB = reinterpret_cast<float *>(base + t.cullB_off);
  constexpr int kGroupSlots = 2 * rtf::kGroupPairs;
  if (i < 0) {                                         // padding: never a candidate, always culled
    put_pair(pairs, slot, 0.f, 0.f, 0.f, -1.0f); perm[slot] = -1;
    if (kSorted) { cullA[slot] = make_float4(0.f, 0.f, 0.f, 4.0f); cullB[slot] = 0.f; }
    if (slot % kGroupSlots == 0) gmin[slot / kGroupSlots] = 3.0e38f;
    return;
  }
  const Oc v = offset(row, O);
  const double r2 = rn::mul(row[3], row[3]);
  const double E = rn::add(rn::mul(rn::mul(2.01 * 9.5367431640625e-07, v.oc2), 1 + 1e-9), delta64);
  put_pair(pairs, slot, rn::to_float(v.x), rn::to_float(v.y), rn::to_float(v.z), rn::up(rn::sub(E, rn::sub(v.oc2, r2))));
  perm[slot] = i;
  // bit 30: the table origin (camera / light) is strictly outside sphere i, with a generous margin
  inv[i] = slot | (rn::sub(v.oc2, r2) > rn::add(rn::mul(1e-6, rn::add(v.oc2, r2)), rn::mul(4.0, delta64)) ? 0x40000000 : 0);
  if (kSorted) {
    // bundle culling (kernels_fast.cuh, margins: see Cone): unit vector to the centre, cos / sin of the angular radius
    const double n = rn::sqrt(v.oc2), r = rn::add(rn::mul(fabs(row[3]), 1.0 + 1e-6), 1e-12);
    if (n > rn::mul(r, 1.0 + 1e-6)) {
      const double sa = rn::div(r, n), ca = rn::sqrt(rn::mul(rn::sub(1.0, sa), rn::add(1.0, sa)));
      cullA[slot] = make_float4(rn::to_float(rn::div(v.x, n)), rn::to_float(rn::div(v.y, n)), rn::to_float(rn::div(v.z, n)), rn::down(ca));
      cullB[slot] = rn::up(sa);
    } else {                                           // the origin is inside (or on) the sphere: never culled
      cullA[slot] = make_float4(0.f, 0.f, 0.f, -4.0f); cullB[slot] = 0.f;
    }
  }
  if (slot % kGroupSlots == 0) {                       // (index order: never a reason to stop)
    const double k = sort_key(v, row);
    gmin[slot / kGroupSlots] = kSorted ? rn::down(rn::sub(rn::sub(rn::sub(k, rn::mul(fabs(k), 1e-6)), 1e-6), delta64)) : -3.0e38f;
  }
}

// Slot i of the general table (index order, recentred by c0) and the exact geometry / material rows of sphere i, from
// its row of 10 columns in file order; row == nullptr: a padding slot.
__host__ __device__ __forceinline__ void general_slot(float4 *pairs, double4 *s64, float4 *mat, float2 *matx, int i, const double *row,
                                                      const double c0[3], double S, double delta64) {
  if (!row) { put_pair(pairs, i, 0.f, 0.f, 0.f, -1.0e30f); return; }
  constexpr double u = 0x1p-24;
  const double r = fabs(row[3]);
  const double rho = rn::add(rn::add(rn::add(rn::mul(rn::mul(r, r), 1 + 40 * u), rn::mul(rn::mul(12 * u, S), r)),
                                     rn::mul(rn::mul(rn::mul(64 * u, u), S), S)), delta64);
  put_pair(pairs, i, rn::to_float(rn::sub(row[0], c0[0])), rn::to_float(rn::sub(row[1], c0[1])), rn::to_float(rn::sub(row[2], c0[2])),
           rn::up(rho));
  s64[i] = make_double4(row[0], row[1], row[2], rn::mul(row[3], row[3]));
  mat[i] = make_float4(rn::to_float(row[4]), rn::to_float(row[5]), rn::to_float(row[6]), rn::to_float(row[7]));
  matx[i] = make_float2(rn::to_float(row[9]), row[7] > 0 ? 1.0f : 0.0f);   // recurse flag decided in double
}

// The tables of LBVH scenes, written on the device from the raw rows: one thread per (table, slot).  blockIdx.y <= L:
// the lookup table of origin y (camera, lights); L + 1: the general table, exact geometry and materials.
struct BuildArgs {
  const double *raw;          // N x 10 sphere rows (file column order), device
  unsigned char *arena;       // tables | general table | ... (layout of RtFastScene)
  double4 *s64;
  float4 *mat;
  float2 *matx;
  TabLayout tab;
  double origin[RT_MAX_LIGHTS + 1][3];
  int N, L, nslots;
  double delta64, c0[3], S;
};
__global__ void k_build_lookup(const BuildArgs b) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (slot >= b.nslots) return;
  const double *row = slot < b.N ? b.raw + (size_t)slot * 10 : nullptr;
  if (t <= b.L)
    shared_origin_slot<false>(b.arena + (size_t)t * b.tab.tstride, b.tab, slot, row ? slot : -1, row, b.origin[t], b.delta64);
  else
    general_slot(reinterpret_cast<float4 *>(b.arena + (size_t)(b.L + 1) * b.tab.tstride), b.s64, b.mat, b.matx, slot, row, b.c0, b.S,
                 b.delta64);
}

// ---------------------------------------------------------------------------------------------
// Sorted camera table (table 0) rebuilt on the device for a new camera position (rt_set_camera), byte-identical to the
// host build.  Input: geo[i] = (cx, cy, cz, r) as in the file (r signed).
//   k_cam_keys    key_i = sqrt(|c_i - O|^2) - |r_i| as an order-preserving 64-bit integer, split in two 32-bit words
//   k_bvh_sort    (bvh.cuh) stable LSD radix sort on the low words, then on the high words gathered through the first
//                 permutation (k_cam_gather): together the order of std::stable_sort on the doubles, ties by index
//   k_cam_fill    shared_origin_slot of every slot in the sorted order
struct CamFillArgs {
  const double4 *geo;
  const int *order;
  unsigned char *base;        // table 0 = the start of the arena
  TabLayout tab;
  int N, nslots;
  double O[3], delta64;
};
__global__ void k_cam_keys(const double4 *__restrict__ geo, int N, double ox, double oy, double oz, unsigned *__restrict__ klo,
                           unsigned *__restrict__ khi, int *__restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double4 g = geo[i];
  const double row[4] = {g.x, g.y, g.z, g.w}, O[3] = {ox, oy, oz};
  const double key = __dadd_rn(sort_key(offset(row, O), row), 0.0);   // (-0 -> +0: the two compare equal)
  unsigned long long u = (unsigned long long)__double_as_longlong(key);
  u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
  klo[i] = (unsigned)u; khi[i] = (unsigned)(u >> 32); vals[i] = i;
}
__global__ void k_cam_gather(const unsigned *__restrict__ src, const int *__restrict__ perm, unsigned *__restrict__ dst, int N) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < N) dst[k] = src[perm[k]];
}
__global__ void k_cam_fill(const CamFillArgs b) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= b.nslots) return;
  if (slot >= b.N) { shared_origin_slot<true>(b.base, b.tab, slot, -1, nullptr, b.O, b.delta64); return; }
  const int i = b.order[slot];
  const double4 g = b.geo[i];
  const double row[4] = {g.x, g.y, g.z, g.w};
  shared_origin_slot<true>(b.base, b.tab, slot, i, row, b.O, b.delta64);
}

// Per-column / per-row camera-plane coordinates (include/camera.h:18-22, src/main.cpp:151-152) in the operation order of
// the reference; aspect = 1, scale = tan(fov / 2) evaluated once on the host.  m = 2: the 2W x 2H supersampling grid.
__global__ void k_cam_plane(double *__restrict__ su, int nu, double *__restrict__ sv, int nv, int m, int W, int H, double scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nu) {
    const double u = __ddiv_rn(__dadd_rn((double)(i / m), __dmul_rn(0.5, (double)(i % m))), (double)(W - 1));
    su[i] = __dmul_rn(__dsub_rn(u, 0.5), scale);
  }
  if (i < nv) {
    const double v = __ddiv_rn(__dadd_rn((double)(i / m), __dmul_rn(0.5, (double)(i % m))), (double)(H - 1));
    sv[i] = __dmul_rn(__dsub_rn(v, 0.5), scale);
  }
}

int rtk_camera_plane(double *su, int nu, double *sv, int nv, int m, int W, int H, double scale, cudaStream_t stream) {
  const int n = nu > nv ? nu : nv;
  k_cam_plane<<<(n + 255) / 256, 256, 0, stream>>>(su, nu, sv, nv, m, W, H, scale);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : -(int)e;
}

static TabLayout tab_layout(const RtFastScene *fs) {
  return {fs->tstride, fs->gmin_off, fs->perm_off, fs->inv_off, fs->cullA_off, fs->cullB_off};
}

// k_build_lookup's arguments for the lookup tables of fs: table 0 seen from cam_pos, tables 1..L from light_pos, the
// general table recentred with the extent bound S.  rt_set_camera rebuilds table 0 only and passes no lights and no S.
static BuildArgs lookup_args(const RtFastScene *fs, const double cam_pos[3], const double (*light_pos)[3], double S) {
  BuildArgs b;
  memset(&b, 0, sizeof(b));
  b.raw = (const double *)fs->raw_dev; b.arena = (unsigned char *)fs->tabs;
  b.s64 = (double4 *)fs->sph64; b.mat = (float4 *)fs->mat; b.matx = (float2 *)fs->matx;
  b.tab = tab_layout(fs);
  for (int k = 0; k < 3; k++) { b.origin[0][k] = cam_pos[k]; b.c0[k] = fs->c0[k]; }
  if (light_pos)
    for (int l = 0; l < fs->L; l++) for (int k = 0; k < 3; k++) b.origin[l + 1][k] = light_pos[l][k];
  b.N = fs->N; b.L = fs->L; b.nslots = 2 * fs->npairs;
  b.delta64 = fs->delta64; b.S = S;
  return b;
}

int rtk_fast_build_scene(RtFastScene *fs, const double *sph, int N, const RtFrameConst *f, int accel, cudaStream_t stream) {
  const int L = f->nlights;
  int npairs = (N + 1) / 2;
  npairs = ((npairs + rtf::kGroupPairs - 1) / rtf::kGroupPairs) * rtf::kGroupPairs;
  if (npairs == 0) npairs = rtf::kGroupPairs;
  const int ngroups = npairs / rtf::kGroupPairs, nslots = 2 * npairs;
  fs->N = N; fs->L = L; fs->npairs = npairs; fs->ngroups = ngroups;
  // identity of the scene for the wave-level feedback: re-uploading the SAME scene (an end-to-end loop does, every frame)
  // keeps the ray statistics valid.  a 64-bit multiplicative hash over the input doubles; large scenes (LBVH: no feedback) just get a new id.
  if (N < 4096) {
    unsigned long long hsh = 1469598103934665603ull;
    auto mix = [&](const void *p, size_t n) {       // 8 bytes per step (n is a multiple of 8 for both inputs)
      const unsigned char *b = (const unsigned char *)p;
      for (size_t i = 0; i + 8 <= n; i += 8) { unsigned long long w; memcpy(&w, b + i, 8); hsh = (hsh ^ w) * 0x9E3779B97F4A7C15ull; hsh ^= hsh >> 29; }
    };
    mix(sph, (size_t)N * 10 * sizeof(double)); mix(f, sizeof(*f));
    fs->generation = hsh;
  } else {
    fs->generation++;
  }
  const double u = std::ldexp(1.0, -24);

  // absolute magnitude bound of every coordinate the reference touches -> delta64.  The part without the camera is kept:
  // rt_set_camera recomputes sabs = fmax(sabs_scene, |cam_pos|), the same value (fmax of non-negative terms in any order).
  double sabs = 0;
  auto upd = [&](double x, double y, double z, double r) { sabs = std::fmax(sabs, std::sqrt(x * x + y * y + z * z) + r); };
  for (int l = 0; l < L; l++) upd(f->light_pos[l][0], f->light_pos[l][1], f->light_pos[l][2], 0);
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (int i = 0; i < N; i++) {
    const double *s = sph + (size_t)i * 10;
    upd(s[0], s[1], s[2], std::fabs(s[3]));
    for (int k = 0; k < 3; k++) { lo[k] = std::fmin(lo[k], s[k]); hi[k] = std::fmax(hi[k], s[k]); }
  }
  fs->sabs_scene = sabs;
  const double delta64 = rtk_delta64(sabs, f->cam_pos);
  fs->delta64 = delta64;
  fs->d64 = rn::up(delta64);
  for (int k = 0; k < 3; k++) fs->c0[k] = N > 0 ? 0.5 * (lo[k] + hi[k]) : 0.0;
  double S = 0;
  for (int i = 0; i < N; i++) {
    const double *s = sph + (size_t)i * 10;
    const double x = s[0] - fs->c0[0], y = s[1] - fs->c0[1], z = s[2] - fs->c0[2];
    S = std::fmax(S, std::sqrt(x * x + y * y + z * z) + std::fabs(s[3]));
  }
  S += 0.01;
  fs->gS2 = rn::up(S * S * 1.0001);
  fs->g_dtmax = rn::up(80.0 * u * S);

  // LBVH scenes: the candidates of every query come from the hierarchy, the tables are only LOOKED UP by sphere (inv ->
  // slot -> pair); nothing walks them in order, prunes by gmin or culls by cone.  So they keep index order -- no sort
  // (five stable sorts of 100 k keys were most of a config-5 upload) -- and carry no cull data, and a kernel writes them
  // from the raw rows (k_build_lookup) instead of staging them on the host.
  const bool lookup_only = N > 0 && (accel == 2 || (accel == 0 && N >= kBvhAutoSpheres));
  fs->lookup_only = lookup_only;
  // byte layout of one shared-origin table
  const unsigned pairs_bytes = (unsigned)npairs * 32u;
  const unsigned gmin_bytes = ((unsigned)ngroups * 4u + 15u) & ~15u;
  const unsigned perm_bytes = (unsigned)nslots * 4u;
  const unsigned inv_bytes = (((unsigned)(N > 0 ? N : 1)) * 4u + 15u) & ~15u;
  const unsigned cullA_bytes = lookup_only ? 0u : (unsigned)nslots * 16u, cullB_bytes = lookup_only ? 0u : (unsigned)nslots * 4u;
  fs->gmin_off = pairs_bytes; fs->perm_off = pairs_bytes + gmin_bytes; fs->inv_off = fs->perm_off + perm_bytes;
  fs->cullA_off = fs->inv_off + inv_bytes; fs->cullB_off = fs->cullA_off + cullA_bytes;
  fs->tstride = fs->cullB_off + cullB_bytes;
  // stride = 32 (mod 128) bytes: when the lanes of a warp walk DIFFERENT lights' tables in step (shadow_mixed), the same
  // pair of four consecutive tables lies in four different bank groups of shared memory
  fs->tstride += (32u + 128u - fs->tstride % 128u) % 128u;
  fs->bytes_bounce = (size_t)L * fs->tstride + pairs_bytes;
  const size_t total = (size_t)(L + 1) * fs->tstride + pairs_bytes;
  // arena = tables | sph64 | mat | matx | geo in one device allocation (grow-only).  geo = (cx, cy, cz, r) per sphere, sorted
  // layouts only: the input of the device rebuild of the camera table (rtk_fast_camera_table); lookup layouts read raw_dev
  const size_t n1 = (size_t)(N > 0 ? N : 1);
  const size_t o_s64 = (total + 255) & ~(size_t)255, o_mat = o_s64 + n1 * sizeof(double4), o_matx = o_mat + n1 * sizeof(float4);
  const size_t o_geo = ((o_matx + n1 * sizeof(float2)) + 255) & ~(size_t)255;
  const size_t arena = lookup_only ? o_geo : ((o_geo + n1 * sizeof(double4)) + 255) & ~(size_t)255;
  if (fs->tabs_cap < arena) {
    cudaFree(fs->tabs); fs->tabs = nullptr; fs->tabs_cap = 0;
    RTK_TRY(cudaMalloc(&fs->tabs, arena));
    fs->tabs_cap = arena;
  }
  fs->sph64 = (unsigned char *)fs->tabs + o_s64; fs->mat = (unsigned char *)fs->tabs + o_mat; fs->matx = (unsigned char *)fs->tabs + o_matx;
  fs->geo = lookup_only ? nullptr : (unsigned char *)fs->tabs + o_geo;
  if (lookup_only) {
    const size_t raw_bytes = (size_t)N * 10 * sizeof(double);
    if (fs->raw_cap < raw_bytes) {
      cudaFree(fs->raw_dev); fs->raw_dev = nullptr; fs->raw_cap = 0;
      RTK_TRY(cudaMalloc(&fs->raw_dev, raw_bytes));
      fs->raw_cap = raw_bytes;
    }
    RTK_TRY(cudaMemcpyAsync(fs->raw_dev, sph, raw_bytes, cudaMemcpyHostToDevice, stream));
    RTK_TRY(cudaMemsetAsync(fs->tabs, 0, total, stream));   // the gaps of the layout, as the host build clears them
    const BuildArgs b = lookup_args(fs, f->cam_pos, f->light_pos, S);
    k_build_lookup<<<dim3((unsigned)(nslots + 255) / 256, (unsigned)(L + 2)), 256, 0, stream>>>(b);
    RTK_TRY(cudaGetLastError());
  } else {
    // scratch of the camera-table sort (keys: 3 x N words, values: 2 x N), grow-only: rt_set_camera allocates nothing
    const size_t need = 5 * (((size_t)N * 4 + 255) & ~(size_t)255);
    if (fs->cam_scratch_cap < need) {
      cudaFree(fs->cam_scratch); fs->cam_scratch = nullptr; fs->cam_scratch_cap = 0;
      RTK_TRY(cudaMalloc(&fs->cam_scratch, need));
      fs->cam_scratch_cap = need;
    }
    if (fs->h_stage_cap < arena) {
      if (fs->h_stage) cudaFreeHost(fs->h_stage);
      fs->h_stage = nullptr; fs->h_stage_cap = 0;
      RTK_TRY(cudaHostAlloc(&fs->h_stage, arena, cudaHostAllocDefault));
      fs->h_stage_cap = arena;
    }
    unsigned char *h = (unsigned char *)fs->h_stage;
    memset(h, 0, total);
    const TabLayout tab = tab_layout(fs);
    std::vector<int> order((size_t)(N > 0 ? N : 1));
    std::vector<double> key((size_t)(N > 0 ? N : 1));
    auto build_table = [&](int t, std::vector<int> &order, std::vector<double> &key) {
      const double *O = t == 0 ? f->cam_pos : f->light_pos[t - 1];
      for (int i = 0; i < N; i++) {
        const double *s = sph + (size_t)i * 10;
        key[i] = sort_key(offset(s, O), s);
        order[i] = i;
      }
      std::stable_sort(order.begin(), order.begin() + N, [&](int p, int q) { return key[p] < key[q]; });
      for (int slot = 0; slot < nslots; slot++) {
        const int i = slot < N ? order[slot] : -1;
        shared_origin_slot<true>(h + (size_t)t * fs->tstride, tab, slot, i, i < 0 ? nullptr : sph + (size_t)i * 10, O, delta64);
      }
    };
    // the (1+L) tables are independent: large scenes build them on separate host threads
    if (N >= 4096 && L >= 1) {
      std::vector<std::thread> th;
      for (int t = 0; t <= L; t++)
        th.emplace_back([&, t]() { std::vector<int> o2((size_t)N); std::vector<double> k2((size_t)N); build_table(t, o2, k2); });
      for (auto &x : th) x.join();
    } else {
      for (int t = 0; t <= L; t++) build_table(t, order, key);
    }
    float4 *gen = reinterpret_cast<float4 *>(h + (size_t)(L + 1) * fs->tstride);
    double4 *s64 = reinterpret_cast<double4 *>(h + o_s64), *geo = reinterpret_cast<double4 *>(h + o_geo);
    float4 *mat = reinterpret_cast<float4 *>(h + o_mat);
    float2 *matx = reinterpret_cast<float2 *>(h + o_matx);
    for (int i = 0; i < nslots; i++) {
      const double *s = i < N ? sph + (size_t)i * 10 : nullptr;
      general_slot(gen, s64, mat, matx, i, s, fs->c0, S, delta64);
      if (s) geo[i] = make_double4(s[0], s[1], s[2], s[3]);
    }
    if (N == 0) { s64[0] = make_double4(0, 0, 0, 0); mat[0] = make_float4(0, 0, 0, 0); matx[0] = make_float2(0, 0); }
    RTK_TRY(cudaMemcpyAsync(fs->tabs, h, arena, cudaMemcpyHostToDevice, stream));
  }
  RTK_TRY(cudaStreamSynchronize(stream));   // the staging buffer / the caller's sphere rows may be reused from here on
  fs->bvh_nodes = nullptr; fs->bvh_nleaf = 0; fs->bvh_build_ms = 0; fs->nbig = 0;
  if (lookup_only) {
    // Spheres far larger than the typical one (a ground sphere ...) stay out of the hierarchy: their boxes would make
    // every ancestor cover the scene, so every ray would walk that whole root-to-leaf path.  They are tested per ray.
    std::vector<double> rad((size_t)N);
    for (int i = 0; i < N; i++) rad[i] = std::fabs(sph[(size_t)i * 10 + 3]);
    std::vector<double> srt(rad);
    std::nth_element(srt.begin(), srt.begin() + N / 2, srt.end());
    const double big_r = 16.0 * srt[N / 2];
    std::vector<int> bigs;
    for (int i = 0; i < N; i++) if (rad[i] > big_r) bigs.push_back(i);
    std::sort(bigs.begin(), bigs.end(), [&](int p, int q) { return rad[p] > rad[q]; });
    if (bigs.size() > 8 || (int)bigs.size() == N) bigs.resize(bigs.size() > 8 ? 8 : 0);
    fs->nbig = (int)bigs.size();
    for (int k = 0; k < fs->nbig; k++) fs->big[k] = bigs[k];
    // box inflation: FP32 rounding of recentred centres / ray origins (<= u S each) and the 12u direction error over
    // any distance <= 2S inside the scene ball, with a 2x reserve: 64u * 3S
    const float eps = rn::up(64.0 * u * 3.0 * S);
    BuildBig big;
    memset(&big, 0, sizeof(big));
    big.n = fs->nbig;
    for (int k = 0; k < fs->nbig; k++) big.idx[k] = fs->big[k];
    const int r = bvh_build(fs, N - fs->nbig, (const double *)fs->raw_dev, N, fs->c0, big, eps, stream);
    if (r != 0) return r;
  }
  return 0;
}

double rtk_delta64(double sabs_scene, const double cam_pos[3]) {
  const double sabs = std::fmax(sabs_scene, std::sqrt(cam_pos[0] * cam_pos[0] + cam_pos[1] * cam_pos[1] + cam_pos[2] * cam_pos[2]) + 0);
  return std::ldexp(4.0 * sabs * sabs, -40) + 1e-30;
}

int rtk_fast_camera_table(RtFastScene *fs, const double cam_pos[3], cudaStream_t stream) {
  const int N = fs->N, nslots = 2 * fs->npairs, tb = 256;
  if (N == 0) return 0;                                // (padding only: nothing depends on the camera)
  if (fs->lookup_only) {
    // table 0 of the kernel that built the tables at upload
    k_build_lookup<<<dim3((unsigned)(nslots + tb - 1) / tb, 1u), tb, 0, stream>>>(lookup_args(fs, cam_pos, nullptr, 0.0));
    RTK_TRY(cudaGetLastError());
    return 0;
  }
  CamFillArgs a;
  memset(&a, 0, sizeof(a));
  a.geo = (const double4 *)fs->geo; a.base = (unsigned char *)fs->tabs; a.tab = tab_layout(fs);
  a.N = N; a.nslots = nslots;
  for (int k = 0; k < 3; k++) a.O[k] = cam_pos[k];
  a.delta64 = fs->delta64;
  const size_t w = ((size_t)N * 4 + 255) & ~(size_t)255;
  unsigned char *sc = (unsigned char *)fs->cam_scratch;
  unsigned *k0 = (unsigned *)sc, *k1 = (unsigned *)(sc + w), *k2 = (unsigned *)(sc + 2 * w);
  int *v0 = (int *)(sc + 3 * w), *v1 = (int *)(sc + 4 * w);
  const size_t sort_smem = (16 * rtb::kSortThreads + 32) * sizeof(unsigned);
  k_cam_keys<<<(N + tb - 1) / tb, tb, 0, stream>>>(a.geo, N, cam_pos[0], cam_pos[1], cam_pos[2], k0, k2, v0);
  rtb::k_bvh_sort<<<1, rtb::kSortThreads, sort_smem, stream>>>(k0, v0, k1, v1, N, 8);   // low words; result in (k0, v0)
  k_cam_gather<<<(N + tb - 1) / tb, tb, 0, stream>>>(k2, v0, k1, N);
  rtb::k_bvh_sort<<<1, rtb::kSortThreads, sort_smem, stream>>>(k1, v0, k0, v1, N, 8);   // high words; order in v0
  a.order = v0;
  k_cam_fill<<<(nslots + tb - 1) / tb, tb, 0, stream>>>(a);
  RTK_TRY(cudaGetLastError());
  return 0;
}

void rtk_fast_free_scene(RtFastScene *fs, int release_tables) {
  if (release_tables) {
    cudaFree(fs->cam_scratch); fs->cam_scratch = nullptr; fs->cam_scratch_cap = 0;
    cudaFree(fs->tabs); fs->tabs = nullptr; fs->tabs_cap = 0;
    if (fs->h_stage) cudaFreeHost(fs->h_stage);
    fs->h_stage = nullptr; fs->h_stage_cap = 0;
    fs->sph64 = fs->mat = fs->matx = nullptr;
    cudaFree(fs->bvh_nodes_buf); cudaFree(fs->bvh_scratch); cudaFree(fs->raw_dev);
    fs->bvh_nodes_buf = fs->bvh_scratch = nullptr; fs->bvh_nodes_cap = fs->bvh_scratch_cap = 0;
    fs->raw_dev = nullptr; fs->raw_cap = 0;
  }
  fs->bvh_nodes = nullptr; fs->bvh_nleaf = 0;
}

// The error word of the last frame launched (call after the stream has been synchronised): bounds guards of the hit /
// ray queues.  0 = clean.
int rtk_fast_last_error(const RtFastWork *w, unsigned int *word) {
  *word = 0;
  if (!w->last_err) return 0;
  RTK_TRY(cudaMemcpy(word, w->last_err, sizeof(unsigned int), cudaMemcpyDeviceToHost));
  return 0;
}

void rtk_fast_free_work(RtFastWork *w) {
  cudaFree(w->queue[0]); cudaFree(w->queue[1]); cudaFree(w->ctl); cudaFree(w->hits); cudaFree(w->occ); cudaFree(w->hit_n); cudaFree(w->cand);
  w->last_err = nullptr;
  w->cand = nullptr; w->cand_cap = 0;
  cudaFree(w->tile_ray); w->tile_ray = nullptr; w->tile_cap = 0;
  if (w->h_fb) { cudaFreeHost(w->h_fb); cudaEventDestroy(w->fb_event); }
  w->h_fb = nullptr; w->fb_pending = 0; w->fb_levels = 0;
  w->queue[0] = w->queue[1] = nullptr; w->ctl = nullptr; w->hits = nullptr; w->occ = nullptr; w->hit_n = nullptr;
  w->queue_cap = w->hit_cap = w->occ_bytes = 0;
}

namespace {
// persistent grid: as many CTAs as can be resident
template <typename K>
int resident_grid(K kernel, size_t smem, int num_sms, int threads = rtf::kThreads) {
  // cached: the occupancy query costs microseconds of host time per launch
  static std::mutex mu;
  static std::map<std::tuple<const void *, size_t, int>, int> cache;
  const auto key = std::make_tuple((const void *)kernel, smem, threads);
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(key);
  if (it == cache.end()) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) nb = 1;
    it = cache.emplace(key, nb).first;
  }
  return std::max(1, it->second * num_sms);
}
// Launch with programmatic dependent launch (PDL): the grid may start while the previous kernel of the stream is
// still draining, run its prologue (table staging) and then block in griddepcontrol.wait (RT_PDL_SYNC in the kernels)
// until that kernel has completed and flushed.  Hides launch latency + prologue behind the predecessor's tail.
// The first failing launch of a frame is remembered (g_launch_err, thread local) and reported by rtk_launch_fast.
thread_local cudaError_t g_launch_err = cudaSuccess;
template <typename K, typename A>
void launch(K kernel, int grid, int block, size_t smem, cudaStream_t stream, bool pdl, const A &arg) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1u : 0u;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, arg);
  if (e != cudaSuccess && g_launch_err == cudaSuccess) g_launch_err = e;
}
// dynamic shared memory of a kernel that stages `bytes` of tables: header | tables | per-warp compacted tables
// ... of the LBVH level-0 kernels: header | per-warp compacted tables | per-warp bundle-traversal frontiers
inline size_t bvh_smem() { return rtf::kSmemHeader + rtf::kWarps * (size_t)(rtf::kWarpBufBytes + rtf::kBundleBufBytes); }
inline size_t staged_smem(size_t bytes) { return rtf::kSmemHeader + ((bytes + 127) & ~(size_t)127) + rtf::kWarps * (size_t)rtf::kWarpBufBytes; }
// control words (u32): [0] tile counter; per level k <= 33: tail chunk counter, shadow / shade / closest work
// counters, hits of level k, rays entering level k
using rtf::CTL_TILE; using rtf::CTL_TAIL; using rtf::CTL_SHADOW; using rtf::CTL_SHADE; using rtf::CTL_CLOSEST; using rtf::CTL_HITS; using rtf::CTL_RAYS;
}  // namespace

int rtk_launch_fast(const RtRenderArgs &args, const RtFastScene *fs, RtFastWork *w, cudaStream_t stream,
                    const cudaEvent_t *marks) {
  const size_t npix = (size_t)args.W * args.bands.local_rows;
  if (!w->ctl) RTK_TRY(cudaMalloc(&w->ctl, kCtlWords * sizeof(unsigned int)));
  // blocked hit queue: one 64-slot block per 16x4 tile (level 0: tiles x 64 >= pixels) or per 64 queued rays (level >= 1:
  // at most pixels / 64 + 1 blocks).  With few rays (fewer than one per lane of the resident grid) k_closest1 takes 32 rays
  // per block instead: fewer than grid x 8 warps x 2 blocks; the slack term covers the largest resident grid (4 CTAs/SM).
  const size_t hit_cap = ((size_t)((args.W + rtf::kWTileW - 1) / rtf::kWTileW) * ((args.bands.local_rows + rtf::kWTileH - 1) / rtf::kWTileH) + 2) * 64 +
                         (size_t)w->num_sms * 4 * rtf::kWarps * 128 * (size_t)rtf::kTwoMult;
  if (w->hit_cap < hit_cap || w->occ_bytes < hit_cap * (size_t)(fs->L > 0 ? fs->L : 1) || (args.max_depth > 1 && w->queue_cap < npix)) {
    RTK_TRY(cudaStreamSynchronize(stream));
    cudaFree(w->queue[0]); cudaFree(w->queue[1]); cudaFree(w->hits); cudaFree(w->occ); cudaFree(w->hit_n);
    w->queue[0] = w->queue[1] = nullptr; w->hits = nullptr; w->occ = nullptr; w->hit_n = nullptr; w->queue_cap = w->hit_cap = w->occ_bytes = 0;
    RTK_TRY(cudaMalloc(&w->hits, hit_cap * sizeof(rtf::HitRec)));
    RTK_TRY(cudaMalloc(&w->hit_n, (hit_cap / 64) * sizeof(unsigned int)));
    w->occ_bytes = hit_cap * (size_t)(fs->L > 0 ? fs->L : 1);
    RTK_TRY(cudaMalloc(&w->occ, w->occ_bytes));
    w->hit_cap = hit_cap;
    if (args.max_depth > 1) {
      RTK_TRY(cudaMalloc(&w->queue[0], npix * sizeof(rtf::RayRec)));
      RTK_TRY(cudaMalloc(&w->queue[1], npix * sizeof(rtf::RayRec)));
      w->queue_cap = npix;
    }

  }
  if (fs->bvh_nodes && args.max_depth > 1 && w->cand_cap < npix) {
    RTK_TRY(cudaStreamSynchronize(stream));
    cudaFree(w->cand); w->cand = nullptr; w->cand_cap = 0;
    RTK_TRY(cudaMalloc(&w->cand, npix * sizeof(rtf::Best)));
    w->cand_cap = npix;
  }
  // per level-0 tile: reflected-ray count, then queue offset (rounded up to whole uint4 segments of the scan, k_shadow)
  const size_t ntiles = (size_t)((args.W + rtf::kWTileW - 1) / rtf::kWTileW) * ((args.bands.local_rows + rtf::kWTileH - 1) / rtf::kWTileH);
  const size_t tile_cap = (ntiles + 4 * rtf::kThreads - 1) / (4 * rtf::kThreads) * (4 * rtf::kThreads);
  if (w->tile_cap < tile_cap) {
    RTK_TRY(cudaStreamSynchronize(stream));
    cudaFree(w->tile_ray); w->tile_ray = nullptr; w->tile_cap = 0;
    RTK_TRY(cudaMalloc(&w->tile_ray, tile_cap * sizeof(unsigned int)));
    w->tile_cap = tile_cap;
  }
  RTK_TRY(cudaMemsetAsync(w->ctl, 0, kCtlWords * sizeof(unsigned int), stream));
  if (args.max_depth <= 0 && !args.fb && !args.out_remap) RTK_TRY(cudaMemsetAsync(args.rgb, 0, npix * 3, stream));   // src/main.cpp:17-18: black (other output modes: the caller clears)

  g_launch_err = cudaSuccess;
  rtf::WaveArgs wa;
  memset(&wa, 0, sizeof(wa));
  rtf::FastArgs &a = wa.f;
  a.r = args;
  a.tabs = (const unsigned char *)fs->tabs;
  a.npairs = fs->npairs; a.ngroups = fs->ngroups; a.N = fs->N; a.L = fs->L;
  a.tstride = fs->tstride; a.gmin_off = fs->gmin_off; a.perm_off = fs->perm_off; a.inv_off = fs->inv_off;
  a.cullA_off = fs->cullA_off; a.cullB_off = fs->cullB_off;
  a.d64 = fs->d64; a.gS2 = fs->gS2; a.g_dtmax = fs->g_dtmax;
  for (int k = 0; k < 3; k++) a.c0[k] = fs->c0[k];
  a.wtiles_x = (args.W + rtf::kWTileW - 1) / rtf::kWTileW;
  a.nwtiles = a.wtiles_x * ((args.bands.local_rows + rtf::kWTileH - 1) / rtf::kWTileH);
  a.tile_counter = w->ctl + CTL_TILE;
  a.two_mult = rtf::kTwoMult; a.lp_mult = rtf::kLpMult;
  a.queue_cap = (unsigned)w->queue_cap; a.err = w->ctl + rtf::CTL_ERR;
  w->last_err = a.err;
  wa.hits = (rtf::HitRec *)w->hits; wa.hit_cap = (unsigned)hit_cap;   // THIS frame's slot count = the stride of the per-light occlusion rows (the allocation may be
                                                          // larger; with its size as stride a scene with more lights than the one the buffers were sized
                                                          // for would index past occ_bytes)
  wa.occ = w->occ; wa.hit_n = w->hit_n; wa.tile_ray = w->tile_ray;
  wa.occ_bits = fs->L <= 32;
  const size_t pairs_bytes = (size_t)fs->npairs * 32;
  const size_t light_bytes = (size_t)fs->L * fs->tstride;
  // per kernel: its tables are staged whole when they fit, else streamed (shared-origin tables) or read through L1/L2 (general table)
  const bool cam_smem = fs->tstride <= kMaxSmemTables, light_smem = light_bytes <= kMaxSmemTables;
  const bool gen_smem = pairs_bytes <= kMaxSmemTables, in_smem = fs->bytes_bounce <= kMaxSmemTables;
  a.tables_in_smem = in_smem;
  const bool bvh = fs->bvh_nodes != nullptr;
  a.bvh.nodes = (const rtb::BvhNode *)fs->bvh_nodes;
  a.nbig = fs->nbig;
  for (int k = 0; k < 8; k++) a.big[k] = fs->big[k];
  // larger tables are streamed through a two-stage ring of TMA tiles (kernels_wave.cuh, kTabStream)
  const size_t stream_smem = rtf::kSmemHeader + 2 * (size_t)rtf::kTileBytes;
  int launches = 0;
  // event records between the kernels (stats) break the launch adjacency PDL needs
  const bool pdl = marks == nullptr;

  // levels below wave_levels run as phase-separated wavefront kernels; the (few) rays left after that are
  // followed to termination by one fused launch
  // (large scenes: every level has enough rays to fill the machine, and the tail's one-warp chains would dominate)
  // small shares of a frame (one rank's bands of many): level 1 has too few rays to pay for three more launches
  int wave_levels = w->wave_levels > 0 ? w->wave_levels : (fs->bvh_nodes ? RT_MAX_LEVELS_INTERNAL : (npix >= 750000 ? 2 : 1));
  // ... better: the ray counts of the previous frame of this very (scene, size, depth).  A level runs as a wavefront when
  // at least kWaveMinRays rays enter it (measured break-even: 67 k rays still win as a wavefront, 55 k do not), the rest goes to the tail.
  const unsigned long long fb_key = fs->generation * 1000003ull + (unsigned long long)npix * 131ull + (unsigned long long)args.max_depth;
  const bool fb_auto = w->wave_levels <= 0 && !fs->bvh_nodes && args.max_depth > 1;
  if (fb_auto) {
    if (!w->h_fb) {
      RTK_TRY(cudaHostAlloc(&w->h_fb, 34 * sizeof(unsigned int), cudaHostAllocDefault));
      RTK_TRY(cudaEventCreateWithFlags(&w->fb_event, cudaEventDisableTiming));
    }
    const cudaError_t fbq = w->fb_pending ? cudaEventQuery(w->fb_event) : cudaErrorNotReady;
    if (fbq != cudaSuccess) cudaGetLastError();      // (cudaErrorNotReady must not surface as this call's launch error)
    if (w->fb_pending && fbq == cudaSuccess) {
      constexpr unsigned kWaveMinRays = 60000u;
      int lv = 1;
      while (lv < 33 && w->h_fb[lv] >= kWaveMinRays) lv++;
      w->fb_levels = lv; w->fb_key = w->fb_pending_key; w->fb_pending = 0;
    }
    if (w->fb_levels > 0 && w->fb_key == fb_key) wave_levels = w->fb_levels;
  }
  for (int level = 0; level < args.max_depth && level < wave_levels; level++) {
    a.level = level;
    wa.hit_count = w->ctl + CTL_HITS + level;
    // ---- closest hit
    if (level == 0) {
      a.stage_bytes = fs->tstride;
      const size_t smem = cam_smem ? staged_smem(a.stage_bytes) : stream_smem;
      const int cta_tiles = (a.nwtiles + rtf::kWarps - 1) / rtf::kWarps;
      if (bvh) { int g = resident_grid(rtf::k_closest0<rtf::kTabBvh>, bvh_smem(), w->num_sms); launch(rtf::k_closest0<rtf::kTabBvh>, g < cta_tiles ? g : cta_tiles, rtf::kThreads, bvh_smem(), stream, false, wa); }
      else if (cam_smem) { int g = resident_grid(rtf::k_closest0<rtf::kTabSmem>, smem, w->num_sms); launch(rtf::k_closest0<rtf::kTabSmem>, g < cta_tiles ? g : cta_tiles, rtf::kThreads, smem, stream, false, wa); }
      else { int g = resident_grid(rtf::k_closest0<rtf::kTabStream>, smem, w->num_sms); launch(rtf::k_closest0<rtf::kTabStream>, g < cta_tiles ? g : cta_tiles, rtf::kThreads, smem, stream, false, wa); }
    } else {
      a.q_in = (rtf::RayRec *)w->queue[(level - 1) & 1];
      a.q_in_count = w->ctl + CTL_RAYS + level;
      wa.work_counter = w->ctl + CTL_CLOSEST + level;
      a.stage_bytes = (unsigned)pairs_bytes;
      const size_t smem = rtf::kSmemHeader + (gen_smem ? a.stage_bytes : 0);
      if (bvh) {
        // incoherent rays: traversal with dynamic ray fetch, then the coherent finish
        wa.cand = (rtf::Best *)w->cand;
        wa.work_counter2 = w->ctl + CTL_TAIL + level;       // (the tail's counters are unused in LBVH scenes)
        launch(rtf::k_closest1_dyn, resident_grid(rtf::k_closest1_dyn, 0, w->num_sms), rtf::kThreads, 0, stream, pdl, wa);
        launches++;
        launch(rtf::k_closest1<false, true>, resident_grid(rtf::k_closest1<false, true>, rtf::kSmemHeader, w->num_sms), rtf::kThreads, rtf::kSmemHeader, stream, pdl, wa);
      }
      else if (gen_smem) launch(rtf::k_closest1<true, false>, resident_grid(rtf::k_closest1<true, false>, smem, w->num_sms), rtf::kThreads, smem, stream, pdl, wa);
      else launch(rtf::k_closest1<false, false>, resident_grid(rtf::k_closest1<false, false>, smem, w->num_sms), rtf::kThreads, smem, stream, pdl, wa);
    }
    launches++;
    if (level == 0 && marks) RTK_TRY(cudaEventRecord(marks[0], stream));
    a.q_out = (rtf::RayRec *)w->queue[level & 1];
    a.q_out_count = w->ctl + CTL_RAYS + level + 1;
    // ---- shadow queries: (light, hit) items.  At level 0 also without lights: its CTA 0 turns the per-tile ray counts
    // into the level-1 queue offsets that k_shade writes to
    if (fs->L > 0 || level == 0) {
      wa.work_counter = w->ctl + CTL_SHADOW + level;
      a.stage_bytes = (unsigned)light_bytes;
      const size_t smem = light_smem ? staged_smem(a.stage_bytes) : stream_smem;
      // camera-ray hits are coherent: the warp-synchronous kernel wins at level 0 (4.3 vs 5.9 ms on config 4); from level 1 on
      // the rays are not, and the dynamic-fetch kernel does (levels >= 1 of config 5: 57.6 -> 38 ms)
      if (bvh && level > 0) launch(rtf::k_shadow_dyn, resident_grid(rtf::k_shadow_dyn, 0, w->num_sms), rtf::kThreads, 0, stream, pdl, wa);
      else if (bvh) launch(rtf::k_shadow<rtf::kTabBvh>, resident_grid(rtf::k_shadow<rtf::kTabBvh>, bvh_smem(), w->num_sms), rtf::kThreads, bvh_smem(), stream, pdl, wa);
      else if (light_smem) launch(rtf::k_shadow<rtf::kTabSmem>, resident_grid(rtf::k_shadow<rtf::kTabSmem>, smem, w->num_sms), rtf::kThreads, smem, stream, pdl, wa);
      else launch(rtf::k_shadow<rtf::kTabStream>, resident_grid(rtf::k_shadow<rtf::kTabStream>, smem, w->num_sms), rtf::kThreads, smem, stream, pdl, wa);
      launches++;
    }
    if (level == 0 && marks) RTK_TRY(cudaEventRecord(marks[1], stream));
    // ---- shade + continuation
    wa.work_counter = w->ctl + CTL_SHADE + level;
    launch(rtf::k_shade, resident_grid(rtf::k_shade, 0, w->num_sms), rtf::kThreads, 0, stream, pdl, wa);
    launches++;
    if (level == 0 && marks) RTK_TRY(cudaEventRecord(marks[2], stream));
  }
  // ---- levels >= 2: one fused launch that follows every remaining ray to termination
  if (args.max_depth > wave_levels) {
    const int level = wave_levels;
    a.level = level;
    a.q_in = (rtf::RayRec *)w->queue[(level - 1) & 1];
    a.q_in_count = w->ctl + CTL_RAYS + level;
    a.q_out = (rtf::RayRec *)w->queue[level & 1];
    a.q_out_count = w->ctl + CTL_RAYS + level + 1;
    a.chunk_counter = w->ctl + CTL_TAIL + level;
    a.stage_bytes = (unsigned)fs->bytes_bounce;
    const size_t smem = in_smem ? staged_smem(fs->bytes_bounce) : rtf::kSmemHeader;
    if (bvh) launch(rtf::k_bounce<false, true>, resident_grid(rtf::k_bounce<false, true>, rtf::kSmemHeader, w->num_sms, rtf::kTailThreads), rtf::kTailThreads, rtf::kSmemHeader, stream, pdl, a);
    else if (in_smem) launch(rtf::k_bounce<true, false>, resident_grid(rtf::k_bounce<true, false>, smem, w->num_sms, rtf::kTailThreads), rtf::kTailThreads, smem, stream, pdl, a);
    else launch(rtf::k_bounce<false, false>, resident_grid(rtf::k_bounce<false, false>, smem, w->num_sms, rtf::kTailThreads), rtf::kTailThreads, smem, stream, pdl, a);
    launches++;
  }
  if (fb_auto && !w->fb_pending) {
    RTK_TRY(cudaMemcpyAsync(w->h_fb, w->ctl + CTL_RAYS, 34 * sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
    RTK_TRY(cudaEventRecord(w->fb_event, stream));
    w->fb_pending = 1; w->fb_pending_key = fb_key;
  }
  cudaError_t e = cudaGetLastError();
  if (g_launch_err != cudaSuccess) e = g_launch_err;
  return e == cudaSuccess ? launches : -(int)e;
}

// ---------------------------------------------------------------------------------------------
// Frame assembly over peer memory (rt_render_bands_frame): every rank's kernels store their finished rows straight
// into rank 0's frame over NVLink; what is left of the "gather" is this completion signal.
//   k_peer_signal  (every rank, after its render, same stream): system-scope fence, then flag[rank] = value in rank 0's
//                  memory -- ordered after all pixel stores of the rank.
//   k_peer_wait    (rank 0): spins until every flag has reached `value`; gives up after ~2 s and reports through err.
__global__ void k_peer_signal(volatile unsigned int *flag, unsigned int value) {
  __threadfence_system();
  *flag = value;
  __threadfence_system();
}
__global__ void k_peer_wait(volatile unsigned int *flags, int n, unsigned int value, unsigned int *err) {
  const int k = threadIdx.x;
  if (k >= n) return;
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
  while ((int)(flags[k] - value) < 0) {
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
    if (t1 - t0 > 2000000000ULL) { atomicExch(err, 1u + (unsigned)k); break; }    // 2 s of wall clock (ns timer), whatever the SM clock
    __nanosleep(200);
  }
  __threadfence_system();
}
int rtk_peer_signal(unsigned int *flag, unsigned int value, cudaStream_t stream) {
  k_peer_signal<<<1, 1, 0, stream>>>(flag, value);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 1 : -(int)e;
}
int rtk_peer_wait(unsigned int *flags, int n, unsigned int value, unsigned int *err, cudaStream_t stream) {
  k_peer_wait<<<1, 64, 0, stream>>>(flags, n, value, err);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 1 : -(int)e;
}

// ---------------------------------------------------------------------------------------------
// 2x2 supersampling resolve (the reference's ray_cuda -a, src/main_gpu.cu:249-258,327-333): the four samples of
// output pixel (i, j) are the pixels (2i + a, 2j + b) of the float sample frame; summed in the reference's order
// s = 0..3 = (0,0) (1,0) (0,1) (1,1), scaled by 1/4, then quantised (src/main_gpu.cu:347-349).
__global__ void k_resolve_aa(const float *__restrict__ fb, int W, int rows, uint8_t *__restrict__ rgb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= W || j >= rows) return;
  const size_t W2 = 2 * (size_t)W;
  const float *s0 = fb + ((size_t)(2 * j) * W2 + 2 * i) * 3, *s2 = s0 + W2 * 3;
  uint8_t *o = rgb + ((size_t)j * W + i) * 3;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    const float v = (((s0[c] + s0[3 + c]) + s2[c]) + s2[3 + c]) * 0.25f;
    o[c] = (uint8_t)(int)(255.99f * fminf(1.0f, v));
  }
}
int rtk_resolve_aa(const float *fb, int W, int rows, uint8_t *rgb, cudaStream_t stream) {
  if (rows <= 0) return 0;
  k_resolve_aa<<<dim3((W + 127) / 128, rows), 128, 0, stream>>>(fb, W, rows, rgb);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 1 : -(int)e;
}

// ---------------------------------------------------------------------------------------------
// FP32 peak probe: 8 independent FFMA chains per thread, 8 CTAs x 256 threads per SM
__global__ void k_fp32_peak(float *out, int iters, float a, float b, unsigned long long *clk) {
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; i++) x[i] = threadIdx.x * 0.001f + i;
  unsigned long long c0 = clock64(), g0;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g0));
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int k = 0; k < 16; k++)
#pragma unroll
      for (int i = 0; i < 8; i++) x[i] = fmaf(x[i], a, b);
  }
  unsigned long long c1 = clock64(), g1;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g1));
  float s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += x[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  if (threadIdx.x == 0 && blockIdx.x == 0) { clk[0] = c1 - c0; clk[1] = g1 - g0; }
}

double rtk_measure_fp32_peak(int device, double *sm_clock_mhz) {
  cudaDeviceProp p;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&p, device) != cudaSuccess) return -1;
  const int grid = p.multiProcessorCount * 8, block = 256, iters = 2048;
  float *buf = nullptr; unsigned long long *clk = nullptr;
  if (cudaMalloc(&buf, (size_t)grid * block * sizeof(float)) != cudaSuccess) return -2;
  if (cudaMalloc(&clk, 16) != cudaSuccess) { cudaFree(buf); return -2; }
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e30f;
  for (int rep = 0; rep < 6; rep++) {
    cudaEventRecord(e0);
    k_fp32_peak<<<grid, block>>>(buf, iters, 1.0001f, 0.5f, clk);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    if (rep >= 2 && ms < best) best = ms;
  }
  unsigned long long h[2] = {0, 1};
  cudaMemcpy(h, clk, 16, cudaMemcpyDeviceToHost);
  if (sm_clock_mhz) *sm_clock_mhz = (double)h[0] / (double)h[1] * 1e3;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(buf); cudaFree(clk);
  if (cudaGetLastError() != cudaSuccess) return -3;
  return 2.0 * grid * block * (double)iters * 16 * 8 / (best * 1e-3);
}
