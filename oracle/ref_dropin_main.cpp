// TEST INFRASTRUCTURE ONLY -- proves the drop-in claim of INTEGRATION.md section 1 by building it.
//
// A headless host program compiled against the REFERENCE'S OWN headers (src/scene.h, src/sceneStructs.h,
// src/raytraceKernel.h, src/image.h, src/utilities.h, included from where they lie under the reference checkout) and linked
// with the reference's own scene.cpp / utilities.cpp / image.cpp / stb_image_write.c -- but NOT with its
// raytraceKernel.cu: the symbol cudaRaytraceCore(uchar4*, camera*, int, int, material*, int, geom*, int) declared at
// src/raytraceKernel.h:17 is resolved by libpt_b200.so.  What the program does is what the reference's application does
// per frame without a window (src/main.cpp:16-55 scene load, :93-113 one cudaRaytraceCore call per iteration with freshly
// packed geom / material arrays, :118-139 mirrored copy into an `image` and saveImageRGB); a plain cudaMalloc'ed uchar4
// buffer stands in for the mapped GL pixel buffer.  Built by `make -C oracle dropin` into oracle/_ref/ref_dropin.
//
// usage: ref_dropin scene=<file> [iterations=N] [frame=F] [depth=D] [seed=S] [out=<name.png|name.bmp>] [pbo=<raw rgba8 dump>]
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>
#include <string>

#include "image.h"
#include "raytraceKernel.h"
#include "scene.h"
#include "sceneStructs.h"
#include "utilities.h"

// knobs of the replacement library (include/pt_compat.h; that header re-declares the reference's struct names, so it
// cannot be included next to sceneStructs.h)
extern "C" int pt_compat_set_trace_depth(int depth);
extern "C" int pt_compat_set_seed(unsigned long long seed);
extern "C" void pt_compat_reset(void);

int main(int argc, char** argv) {
  std::string scene_file, out_name, pbo_name;
  int n_iter = 4, frame = 0, depth = 8;
  unsigned long long seed = 0;
  for (int i = 1; i < argc; i++) {
    std::string key, val;
    std::istringstream arg(argv[i]);
    getline(arg, key, '=');
    getline(arg, val, '=');
    if (key == "scene") scene_file = val;
    else if (key == "iterations") n_iter = atoi(val.c_str());
    else if (key == "frame") frame = atoi(val.c_str());
    else if (key == "depth") depth = atoi(val.c_str());
    else if (key == "seed") seed = strtoull(val.c_str(), nullptr, 10);
    else if (key == "out") out_name = val;
    else if (key == "pbo") pbo_name = val;
  }
  if (scene_file.empty()) {
    std::cerr << "usage: ref_dropin scene=<file> [iterations=N] [frame=F] [depth=D] [seed=S] [out=<file>]" << std::endl;
    return 2;
  }
  scene* world = new scene(scene_file);  // never deleted: scene::~scene() is declared but not defined (src/scene.h:27)
  camera* cam = &world->renderCam;
  if (frame < 0 || frame >= cam->frames) frame = 0;
  const int W = (int)cam->resolution.x, H = (int)cam->resolution.y;

  pt_compat_set_trace_depth(depth);
  pt_compat_set_seed(seed);
  uchar4* pbo = nullptr;  // stands in for cudaGLMapBufferObject's device pointer
  if (cudaMalloc(&pbo, sizeof(uchar4) * (size_t)W * H) != cudaSuccess) {
    std::cerr << "cudaMalloc failed" << std::endl;
    return 1;
  }
  for (int it = 1; it <= n_iter; it++) {
    const int ng = (int)world->objects.size(), nm = (int)world->materials.size();
    geom* geoms = new geom[ng];
    material* mats = new material[nm];
    for (int i = 0; i < ng; i++) geoms[i] = world->objects[i];
    for (int i = 0; i < nm; i++) mats[i] = world->materials[i];
    cudaRaytraceCore(pbo, cam, frame, it, mats, nm, geoms, ng);
    delete[] geoms;
    delete[] mats;
  }
  if (!pbo_name.empty()) {
    std::string bytes((size_t)W * H * 4, '\0');
    cudaMemcpy(&bytes[0], pbo, bytes.size(), cudaMemcpyDeviceToHost);
    FILE* f = fopen(pbo_name.c_str(), "wb");
    if (f) { fwrite(bytes.data(), 1, bytes.size(), f); fclose(f); }
  }
  cudaFree(pbo);

  image out(W, H);
  for (int x = 0; x < W; x++)
    for (int y = 0; y < H; y++) out.writePixelRGB(W - 1 - x, y, cam->image[x + y * W]);
  gammaSettings gs;
  gs.applyGamma = true;
  gs.gamma = 1.0;
  gs.divisor = 1.0;
  out.setGammaSettings(gs);
  std::string name = out_name.empty() ? cam->imageName : out_name;
  std::ostringstream fr;
  fr << frame;
  utilityCore::replaceString(name, ".bmp", "." + fr.str() + ".bmp");
  utilityCore::replaceString(name, ".png", "." + fr.str() + ".png");
  out.saveImageRGB(name);
  std::cout << "Saved frame " << frame << " to " << name << " after " << n_iter << " iterations" << std::endl;
  pt_compat_reset();
  return 0;
}
