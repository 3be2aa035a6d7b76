// kernel_shim.cu -> libkernel_shim.so : the reference's tile-launch C ABI, symbol for symbol, on top of librt_b200.
//
// The reference's hybrid renderer links `kernel.o` for exactly two extern "C" functions
//     launch_gpu_kernel            src/kernel.cu:185-200   (declared src/main_hybrid.cpp:104-109, called :461-466, :615-621)
//     upload_lights_and_ambience   src/kernel.cu:202-207   (declared src/main_hybrid.cpp:170-171, called :238)
// This library exports both with the same names, argument lists and conventions (caller-owned device buffers, float3
// framebuffer indexed [row * image_width + column] with row 0 = bottom, asynchronous on the caller's stream, void
// return, process-global light state), so `ray_hybrid` links against it unchanged in place of kernel.o:
//     g++ -fopenmp -I include -I $CUDA/include -c src/main_hybrid.cpp
//     g++ main_hybrid.o -o ray_hybrid -L<pkg> -lkernel_shim -lrt_b200 -L$CUDA/lib64 -lcudart -lgomp
// Only the BINARY LAYOUT of the argument structs is mirrored here (include/gpu_shared.h:85-100 GPUMaterial/GPUSphere
// 36 bytes, :145-149 GPULight 28 bytes, :155-166 GPUCamera 88 bytes); none of the reference's code is used.
//
// What differs, by necessity: the reference's caller hands the scene over as FP32 device structs, so the scene this
// shim renders is the FP32-rounded one (exactly what the reference's own kernel sees); it is rendered with the serial
// renderer's semantics by librt_b200 (rt_render_tile).  The sphere array and the camera are read back from the device
// once per (sphere pointer, camera pointer, sphere count, light count) and cached; call kernel_shim_invalidate() after
// changing them in place.  Errors cannot be
// returned through a void function: like the reference's CUDA_CHECK (include/gpu_shared.h:14-22) they are printed and
// the process exits.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "rt_b200.h"

// (namespace scope, not anonymous: a function whose parameter types have internal linkage would not be exported)
struct ShimMaterial { float3 albedo; float metallic; float shininess; };
struct ShimSphere { float3 center; float radius; ShimMaterial material; };
struct ShimLight { float3 position; float3 color; float intensity; };
struct ShimCamera { float3 origin, lower_left, horizontal, vertical, forward, right, up; float fov; };
static_assert(sizeof(ShimSphere) == 36 && sizeof(ShimLight) == 28 && sizeof(ShimCamera) == 88, "layout of include/gpu_shared.h");

namespace {

std::mutex g_mu;
rt_ctx *g_ctx = nullptr;
std::vector<double> g_lights;            // L x 7, file column order
double g_ambient[3] = {0, 0, 0};
const void *g_spheres_ptr = nullptr, *g_camera_ptr = nullptr;
int g_nspheres = -1, g_nlights = -1;
bool g_dirty = true;

[[noreturn]] void die(const char *what) {
  std::fprintf(stderr, "kernel_shim: %s: %s\n", what, rt_last_error());
  std::exit(1);
}
void die_cuda(const char *what, cudaError_t e) {
  if (e == cudaSuccess) return;
  std::fprintf(stderr, "kernel_shim: %s: %s\n", what, cudaGetErrorString(e));
  std::exit(1);
}

}  // namespace

extern "C" void kernel_shim_invalidate(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_dirty = true;
}

extern "C" void upload_lights_and_ambience(ShimLight *lights, int count, float3 ambience) {
  std::lock_guard<std::mutex> lk(g_mu);
  g_lights.assign((size_t)(count > 0 ? count : 0) * RT_LIGHT_STRIDE, 0.0);
  for (int l = 0; l < count; l++) {
    double *r = &g_lights[(size_t)l * RT_LIGHT_STRIDE];
    r[0] = lights[l].position.x; r[1] = lights[l].position.y; r[2] = lights[l].position.z;
    r[3] = lights[l].color.x; r[4] = lights[l].color.y; r[5] = lights[l].color.z;
    r[6] = lights[l].intensity;
  }
  g_ambient[0] = ambience.x; g_ambient[1] = ambience.y; g_ambient[2] = ambience.z;
  g_dirty = true;
}

extern "C" void launch_gpu_kernel(float3 *d_framebuffer, ShimSphere *d_spheres, int num_spheres, int num_lights, ShimCamera *camera,
                                  int tile_x, int tile_y, int tile_width, int tile_height, int image_width, int image_height,
                                  int max_depth, cudaStream_t stream) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_ctx) {
    int dev = 0;
    die_cuda("cudaGetDevice", cudaGetDevice(&dev));
    if (rt_create(dev, &g_ctx) != RT_OK) die("rt_create");
  }
  if (g_dirty || d_spheres != g_spheres_ptr || camera != g_camera_ptr || num_spheres != g_nspheres ||
      num_lights != g_nlights) {
    // (blocking copies: once per scene; they also order this read behind the caller's own uploads)
    std::vector<ShimSphere> hs((size_t)(num_spheres > 0 ? num_spheres : 0));
    if (num_spheres > 0) die_cuda("read spheres", cudaMemcpy(hs.data(), d_spheres, hs.size() * sizeof(ShimSphere), cudaMemcpyDeviceToHost));
    ShimCamera cam;
    die_cuda("read camera", cudaMemcpy(&cam, camera, sizeof(cam), cudaMemcpyDeviceToHost));
    std::vector<double> sph((size_t)hs.size() * RT_SPHERE_STRIDE);
    for (size_t i = 0; i < hs.size(); i++) {
      double *r = &sph[i * RT_SPHERE_STRIDE];
      r[0] = hs[i].center.x; r[1] = hs[i].center.y; r[2] = hs[i].center.z; r[3] = hs[i].radius;
      r[4] = hs[i].material.albedo.x; r[5] = hs[i].material.albedo.y; r[6] = hs[i].material.albedo.z;
      r[7] = hs[i].material.metallic; r[8] = 1.0 - hs[i].material.metallic; r[9] = hs[i].material.shininess;
    }
    int L = (int)(g_lights.size() / RT_LIGHT_STRIDE);
    if (num_lights < L) L = num_lights;                // the caller's count rules, as in the reference's kernel
    const double pos[3] = {cam.origin.x, cam.origin.y, cam.origin.z};
    const double look[3] = {pos[0] + (double)cam.forward.x, pos[1] + (double)cam.forward.y, pos[2] + (double)cam.forward.z};
    if (rt_upload_scene(g_ctx, sph.data(), (int)hs.size(), g_lights.data(), L, g_ambient, pos, look, (double)cam.fov) != RT_OK)
      die("rt_upload_scene");
    g_spheres_ptr = d_spheres; g_camera_ptr = camera; g_nspheres = num_spheres; g_nlights = num_lights; g_dirty = false;
  }
  if (rt_render_tile(g_ctx, image_width, image_height, max_depth, tile_x, tile_y, tile_width, tile_height,
                     reinterpret_cast<float *>(d_framebuffer), (void *)stream) != RT_OK)
    die("rt_render_tile");
}
