// pt_compat.h -- source-compatible C++ entry point of the reference's hot path.
//
// libpt_b200.so exports the reference's own symbol
//
//     void cudaRaytraceCore(uchar4*, camera*, int, int, material*, int, geom*, int);      (C++ linkage)
//
// declared at reference src/raytraceKernel.h:17 and called from src/main.cpp:110.  A reference build keeps its own
// src/sceneStructs.h + src/raytraceKernel.h, drops src/raytraceKernel.cu from the link and links -lpt_b200 instead
// (INTEGRATION.md).  This header is for callers that do NOT have the reference's headers (and GLM): it declares
// layout-identical types under the same names, which is all the mangled symbol depends on.
//
// Do not include this header together with the reference's sceneStructs.h (same type names).
#ifndef PT_COMPAT_H
#define PT_COMPAT_H

#include <vector_types.h>  // uchar4 (CUDA toolkit)

#include <string>

namespace ptc {
struct vec2 { float x, y; };
struct vec3 { float x, y, z; };
struct vec4 { float x, y, z, w; };
}  // namespace ptc

struct cudaMat4 { ptc::vec4 x, y, z, w; };  // src/cudaMat4.h:18-23: four ROWS

enum GEOMTYPE { SPHERE, CUBE, MESH };  // src/sceneStructs.h:14

struct ray {  // src/sceneStructs.h:16-19
  ptc::vec3 origin;
  ptc::vec3 direction;
};

struct geom {  // src/sceneStructs.h:21-30 (56 bytes)
  enum GEOMTYPE type;
  int materialid;
  int frames;  // never initialised by the reference loader (SURVEY.md D5); not read
  ptc::vec3* translations;
  ptc::vec3* rotations;
  ptc::vec3* scales;
  cudaMat4* transforms;
  cudaMat4* inverseTransforms;
};

struct camera {  // src/sceneStructs.h:50-61 (96 bytes)
  ptc::vec2 resolution;
  ptc::vec3* positions;
  ptc::vec3* views;
  ptc::vec3* ups;
  int frames;
  ptc::vec2 fov;
  unsigned int iterations;
  ptc::vec3* image;  // running mean, W*H, index = x + y*W
  ray* rayList;
  std::string imageName;
};

struct material {  // src/sceneStructs.h:63-74 (64 bytes)
  ptc::vec3 color;
  float specularExponent;
  ptc::vec3 specularColor;
  float hasReflective;
  float hasRefractive;
  float indexOfRefraction;
  float hasScatter;
  ptc::vec3 absorptionCoefficient;
  float reducedScatterCoefficient;
  float emittance;
};

// One iteration (one sample per pixel), exactly the reference's contract (src/raytraceKernel.cu:108-165):
//   * `iterations` is the 1-based sample number (src/main.cpp:95); sample `iterations` is folded into
//     renderCam->image as a running mean (image = (image*(k-1) + L_k) / k), which is what the reference's save path
//     expects (divisor 1, src/main.cpp:127-131);
//   * `frame` selects [frame] of every per-frame array;
//   * PBOpos is a DEVICE pointer to W*H uchar4 (mapped PBO) or NULL (headless); it receives sendImageToPBO's bytes;
//   * synchronous: the image is complete on return (cudaThreadSynchronize at :162);
//   * on a CUDA error it prints "Cuda error: ..." to stderr and exits (checkCUDAError, :19-25) unless
//     pt_compat_set_exit_on_error(0) was called, in which case pt_compat_last_status() reports it.
void cudaRaytraceCore(uchar4* PBOpos, camera* renderCam, int frame, int iterations, material* materials,
                      int numberOfMaterials, geom* geoms, int numberOfGeoms);

extern "C" {
// the reference hard-codes traceDepth = 1 as a placeholder (src/raytraceKernel.cu:110); default here is 8
int pt_compat_set_trace_depth(int depth);
int pt_compat_set_seed(unsigned long long seed);
int pt_compat_set_device(int device);
int pt_compat_set_lens(float aperture, float focal_distance);
int pt_compat_set_exit_on_error(int on);
/* samples traced ahead of the calls per group (default 8, 1..64; two groups are in flight): a sequence of calls
 * iterations = k, k+1, ... then only adds one traced sample per call; results do not depend on it */
int pt_compat_set_ahead(int samples);
int pt_compat_set_direct_lighting(int on); /* pt_set_direct_lighting for the calls that follow (default off) */
int pt_compat_set_subsurface(int on);      /* pt_set_subsurface for the calls that follow (default off) */
int pt_compat_set_glossy(int on);          /* pt_set_glossy for the calls that follow (default off) */
/* 1: cudaRaytraceCore behaves exactly like the UNMODIFIED reference does today -- its raytraceRay is a stub that fills
 * renderCam->image with per-pixel noise and converts that to the PBO (src/raytraceKernel.cu:93-104,149-154) -- so a
 * build can be checked against the reference before the renderer is switched on (default 0) */
int pt_compat_set_reference_stub(int on);
int pt_compat_last_status(void);
// drop the cached context (the reference's cudaDeviceReset() between frames, src/main.cpp:155)
void pt_compat_reset(void);
}

#endif  // PT_COMPAT_H
