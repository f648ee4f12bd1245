// TEST INFRASTRUCTURE ONLY -- never linked into, loaded by, or shipped with the product.
//
// oracle/_ref/libptref_gpu.so: the reference's OWN render entry and kernels -- src/raytraceKernel.cu, included from
// where it lies under the reference checkout (nothing is copied) -- compiled for sm_100a.  Its kernels are the TODO stubs the
// reference ships: raytraceRay writes per-pixel noise (src/raytraceKernel.cu:93-104, generateRandomNumberFromThread
// :29-36), sendImageToPBO converts the image to 8 bits (:58-89).  Running it on the GPU box gives the outputs of the
// reference ITSELF for the pieces it does implement:
//   * tests/test_gpu_reference_stub.py compares pt_reference_stub_image / pt_resolve_rgba8 with them, bit for bit;
//   * ref_noise_host is the same generator evaluated by the reference's host build (argument evaluation order of g++).
#include "raytraceKernel.cu"

#include <cstring>
#include <vector>

extern "C" {

// One call of the reference's cudaRaytraceCore on a W x H frame: image_inout (W*H*3 floats, host) is what
// renderCam->image holds before and after; pbo_out (W*H*4 bytes, host) receives the device PBO.  Returns 0, or a CUDA
// error code from the allocations here (the reference itself exits on its own errors).
int ref_cudaRaytraceCore(int W, int H, int iterations, float* image_inout, unsigned char* pbo_out) {
  camera cam;
  glm::vec3 pos(0, 4.5f, 12), view(0, 0, -1), up(0, 1, 0);
  cam.resolution = glm::vec2(W, H);
  cam.positions = &pos; cam.views = &view; cam.ups = &up;
  cam.frames = 1;
  cam.fov = glm::vec2(25, 25);
  cam.iterations = 5000;
  cam.image = reinterpret_cast<glm::vec3*>(image_inout);
  cam.rayList = NULL;
  geom g;
  glm::vec3 t(0, 0, 0), r(0, 0, 0), s(1, 1, 1);
  cudaMat4 I;
  I.x = glm::vec4(1, 0, 0, 0); I.y = glm::vec4(0, 1, 0, 0); I.z = glm::vec4(0, 0, 1, 0); I.w = glm::vec4(0, 0, 0, 1);
  g.type = SPHERE; g.materialid = 0; g.frames = 1;
  g.translations = &t; g.rotations = &r; g.scales = &s; g.transforms = &I; g.inverseTransforms = &I;
  material m;
  std::memset(&m, 0, sizeof(m));
  uchar4* pbo = NULL;
  cudaError_t e = cudaMalloc(&pbo, (size_t)W * H * sizeof(uchar4));
  if (e != cudaSuccess) return (int)e;
  cudaMemset(pbo, 0xAB, (size_t)W * H * sizeof(uchar4));
  cudaRaytraceCore(pbo, &cam, 0, iterations, &m, 1, &g, 1);
  e = cudaMemcpy(pbo_out, pbo, (size_t)W * H * sizeof(uchar4), cudaMemcpyDeviceToHost);
  cudaFree(pbo);
  return (int)e;
}

// generateRandomNumberFromThread on the host (the reference's host build of the same function)
void ref_noise_host(int W, int H, float time, float* out) {
  for (int y = 0; y < H; y++)
    for (int x = 0; x < W; x++) {
      glm::vec3 c = generateRandomNumberFromThread(glm::vec2(W, H), time, x, y);
      float* o = out + 3 * ((size_t)y * W + x);
      o[0] = c.x; o[1] = c.y; o[2] = c.z;
    }
}

}  // extern "C"
