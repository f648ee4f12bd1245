// pt_sampling.cuh -- surface-point / direction sampling and Beer-Lambert transmission (sm_100a).
//
// Reference functions re-implemented here (paths relative to the reference repo root):
//   hash                                  src/intersections.h:26-34
//   getRadiuses                           src/intersections.h:120-129
//   getRandomPointOnCube                  src/intersections.h:133-175   (implemented there: bit-exact, see below)
//   getRandomPointOnSphere (stub)         src/intersections.h:179-182
//   getRandomDirectionInSphere (stub)     src/interactions.h:93-95
//   calculateTransmission (stub)          src/interactions.h:31-33
//   thrust::minstd_rand / uniform_real_distribution<float>   (the generator the reference seeds at :135-137)
//   generateRandomNumberFromThread        src/raytraceKernel.cu:29-36   (the noise its raytraceRay stub writes, :93-104)
//
// getRandomPointOnCube is evaluation-order dependent in the reference (`glm::vec3(u02(rng), u02(rng), .5)`): its host
// build draws the SECOND random coordinate first (g++ evaluates arguments right to left).  The oracle is pinned to
// that build, so this file draws in the same order explicitly.  Same arithmetic contract as pt_device.cuh.
#pragma once
#include "pt_device.cuh"

namespace ptd {

__device__ __forceinline__ uint32_t ref_hash(uint32_t a) {
  a = (a + 0x7ed55d16u) + (a << 12);
  a = (a ^ 0xc761c23cu) ^ (a >> 19);
  a = (a + 0x165667b1u) + (a << 5);
  a = (a + 0xd3a2646cu) ^ (a << 9);
  a = (a + 0xfd7046c5u) + (a << 3);
  a = (a ^ 0xb55a4f09u) ^ (a >> 16);
  return a;
}

// LCG(48271, 0, 2^31 - 1); seed s -> s mod m, 0 -> 1; uniform = (float)(x - 1) / 2^31 * (b - a) + a
struct Minstd { uint32_t x; };
__device__ __forceinline__ void minstd_seed(Minstd& r, uint32_t s) {
  const uint32_t v = s % 2147483647u;
  r.x = v == 0 ? 1u : v;
}
__device__ __forceinline__ float minstd_uniform(Minstd& r, float a, float b) {
  r.x = (uint32_t)(((uint64_t)r.x * 48271u) % 2147483647u);
  float res = (float)(r.x - 1u);
  res = res / 2147483648.0f;  // 1.0f + (float)(max - min) rounds to 2^31
  return (res * (b - a)) + a;
}

__device__ __forceinline__ f3 radiuses(float4 f0, float4 f1, float4 f2) {
  const f3 origin = mulMV(f0, f1, f2, 0.0f, 0.0f, 0.0f, 1.0f);
  const f3 xmax = mulMV(f0, f1, f2, 0.5f, 0.0f, 0.0f, 1.0f);
  const f3 ymax = mulMV(f0, f1, f2, 0.0f, 0.5f, 0.0f, 1.0f);
  const f3 zmax = mulMV(f0, f1, f2, 0.0f, 0.0f, 0.5f, 1.0f);
  return mk(length(xmax - origin), length(ymax - origin), length(zmax - origin));
}

// body of src/intersections.h:140-172 given the three draws (roulette in [0,1), a and b in [-.5,.5))
__device__ __forceinline__ f3 cube_point(float4 f0, float4 f1, float4 f2, float roulette, float a, float b) {
  const f3 radii = radiuses(f0, f1, f2);
  const float side1 = radii.x * radii.y * 4.0f;
  const float side2 = radii.z * radii.y * 4.0f;
  const float side3 = radii.x * radii.z * 4.0f;
  const float totalarea = 2.0f * (side1 + side2 + side3);
  f3 p;
  if (roulette < (side1 / totalarea)) p = mk(a, b, 0.5f);
  else if (roulette < ((side1 * 2) / totalarea)) p = mk(a, b, -0.5f);
  else if (roulette < (((side1 * 2) + (side2)) / totalarea)) p = mk(0.5f, a, b);
  else if (roulette < (((side1 * 2) + (side2 * 2)) / totalarea)) p = mk(-0.5f, a, b);
  else if (roulette < (((side1 * 2) + (side2 * 2) + (side3)) / totalarea)) p = mk(a, 0.5f, b);
  else p = mk(a, -0.5f, b);
  return mulMV(f0, f1, f2, p.x, p.y, p.z, 1.0f);
}

// the same with the five face thresholds precomputed per geom (pt_api.cu: build_lights evaluates the expressions above
// in the same binary32 order on the host); th = (th0..th3), th4
__device__ __forceinline__ f3 cube_point_th(float4 f0, float4 f1, float4 f2, float4 th, float th4, float roulette, float a, float b) {
  f3 p;
  if (roulette < th.x) p = mk(a, b, 0.5f);
  else if (roulette < th.y) p = mk(a, b, -0.5f);
  else if (roulette < th.z) p = mk(0.5f, a, b);
  else if (roulette < th.w) p = mk(-0.5f, a, b);
  else if (roulette < th4) p = mk(a, 0.5f, b);
  else p = mk(a, -0.5f, b);
  return mulMV(f0, f1, f2, p.x, p.y, p.z, 1.0f);
}

__device__ __forceinline__ f3 sphere_point(float4 f0, float4 f1, float4 f2, float u0, float u1) {
  const f3 d = sphere_dir(u0, u1);
  return mulMV(f0, f1, f2, 0.5f * d.x, 0.5f * d.y, 0.5f * d.z, 1.0f);
}

// getRandomPointOnCube / getRandomPointOnSphere with the reference's generator construction
__device__ __forceinline__ f3 random_point_on_geom(int type, float4 f0, float4 f1, float4 f2, float randomSeed) {
  Minstd rng;
  minstd_seed(rng, ref_hash((uint32_t)randomSeed));
  if (type == 0) {
    const float u0 = minstd_uniform(rng, 0.0f, 1.0f);
    const float u1 = minstd_uniform(rng, 0.0f, 1.0f);
    return sphere_point(f0, f1, f2, u0, u1);
  }
  const float roulette = minstd_uniform(rng, 0.0f, 1.0f);
  const float b = minstd_uniform(rng, -0.5f, 0.5f);  // the host build's order: second coordinate first
  const float a = minstd_uniform(rng, -0.5f, 0.5f);
  return cube_point(f0, f1, f2, roulette, a, b);
}

// generateRandomNumberFromThread (src/raytraceKernel.cu:29-36), what the reference's raytraceRay stub writes into every
// pixel (:93-104): index = x + y * resolution.x in binary32, seed = hash((unsigned)(index * time)), three draws of
// uniform(0,1).  The three draws are arguments of one glm::vec3(...) call, so their order is the compiler's: reversed =
// false draws x, y, z (what the reference's kernel does on the device), true draws z, y, x (its host build under g++).
__device__ __forceinline__ f3 reference_noise(float res_x, float time, int x, int y, bool reversed) {
  const int index = (int)((float)x + ((float)y * res_x));
  Minstd rng;
  minstd_seed(rng, ref_hash((uint32_t)((float)index * time)));
  const float a = minstd_uniform(rng, 0.0f, 1.0f), b = minstd_uniform(rng, 0.0f, 1.0f), c = minstd_uniform(rng, 0.0f, 1.0f);
  return reversed ? mk(c, b, a) : mk(a, b, c);
}
__global__ void k_reference_stub(int W, int H, float time, int reversed, float* rgb) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= W || y >= H) return;
  const f3 c = reference_noise((float)W, time, x, y, reversed != 0);
  float* o = rgb + 3 * ((size_t)y * W + x);
  o[0] = c.x; o[1] = c.y; o[2] = c.z;
}

// ---- parity entry points (lists) ----
// mode 0: one float seed per point (the reference's generator); mode 1: three given uniforms per point
__global__ void k_points_on_geom(int type, float4 f0, float4 f1, float4 f2, int mode, int n, const float* in, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  f3 p;
  if (mode == 0) p = random_point_on_geom(type, f0, f1, f2, in[i]);
  else if (type == 0) p = sphere_point(f0, f1, f2, in[3 * i], in[3 * i + 1]);
  else p = cube_point(f0, f1, f2, in[3 * i], in[3 * i + 1] - 0.5f, in[3 * i + 2] - 0.5f);
  out[3 * i] = p.x; out[3 * i + 1] = p.y; out[3 * i + 2] = p.z;
}
__global__ void k_sphere_dirs(int n, const float* xi1, const float* xi2, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const f3 d = sphere_dir(xi1[i], xi2[i]);
  out[3 * i] = d.x; out[3 * i + 1] = d.y; out[3 * i + 2] = d.z;
}
__global__ void k_transmission(int n, const float* absorption, const float* distance, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const f3 t = transmission(mk(absorption[3 * i], absorption[3 * i + 1], absorption[3 * i + 2]), distance[i]);
  out[3 * i] = t.x; out[3 * i + 1] = t.y; out[3 * i + 2] = t.z;
}
// u = (xi1, xi2, xf) per entry: the three uniforms the renderer takes from the segment's Philox block (u[0], u[1], u[3])
__global__ void k_sample_medium(int n, const float* absorption, const float* scatter, const float* distance, const float* u,
                                int32_t* scattered, float* s, float* dir, float* weight) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const MediumSample e = sample_medium(mk(absorption[3 * i], absorption[3 * i + 1], absorption[3 * i + 2]), scatter[i], distance[i],
                                       u[3 * i], u[3 * i + 1], u[3 * i + 2]);
  scattered[i] = e.scattered ? 1 : 0;
  s[i] = e.s;
  dir[3 * i] = e.dir.x; dir[3 * i + 1] = e.dir.y; dir[3 * i + 2] = e.dir.z;
  weight[3 * i] = e.weight.x; weight[3 * i + 1] = e.weight.y; weight[3 * i + 2] = e.weight.z;
}
// u = (u0, u1) per entry: the two uniforms the renderer takes from the segment's Philox block (u[0], u[1]); the shading
// normal faces the incident direction as in shade()
__global__ void k_sample_glossy(int n, const float* normal, const float* incident, const float* exponent, const float* u,
                                float* dir) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const f3 nn = mk(normal[3 * i], normal[3 * i + 1], normal[3 * i + 2]);
  const f3 d = mk(incident[3 * i], incident[3 * i + 1], incident[3 * i + 2]);
  const f3 ns = dot(d, nn) < 0 ? nn : neg(nn);
  const f3 g = sample_glossy(ns, d, exponent[i], u[2 * i], u[2 * i + 1]);
  dir[3 * i] = g.x; dir[3 * i + 1] = g.y; dir[3 * i + 2] = g.z;
}

}  // namespace ptd
