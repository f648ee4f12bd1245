// TEST INFRASTRUCTURE ONLY -- never linked into, loaded by, or shipped with the product.
//
// extern "C" wrappers around the reference's own scene loader and image writer, compiled
// from the reference checkout's src/{scene,utilities,image}.cpp and external stb_image_write.c where
// they lie (see oracle/Makefile).  Used by oracle/gen_golden.py and by the in-container
// pinning tests.  Reference entry points wrapped:
//   scene::scene(string)            src/scene.cpp:11-35
//   runCuda() save path             src/main.cpp:118-139 (re-stated here verbatim in behaviour,
//                                   because main.cpp needs GL and cannot be compiled)
//   image::saveImageRGB             src/image.cpp:46-88
#include "scene.h"
#include "image.h"
#include <cstring>
#include <sstream>

extern "C" {

void* refscene_load(const char* path) {
  // scene::~scene is declared but never defined (SURVEY.md D6) -> never deleted.
  return new scene(std::string(path));
}

void refscene_counts(void* h, int* n_geoms, int* n_mats, int* cam_frames, int* iterations, int* w, int* hgt) {
  scene* s = (scene*)h;
  *n_geoms = (int)s->objects.size();
  *n_mats = (int)s->materials.size();
  *cam_frames = s->renderCam.frames;
  *iterations = (int)s->renderCam.iterations;
  *w = (int)s->renderCam.resolution.x;
  *hgt = (int)s->renderCam.resolution.y;
}

// Flatten frame `frame` exactly like cudaRaytraceCore does (src/raytraceKernel.cu:123-134).
void refscene_static_geoms(void* h, int frame, void* out172) {
  scene* s = (scene*)h;
  staticGeom* out = (staticGeom*)out172;
  for (size_t i = 0; i < s->objects.size(); i++) {
    staticGeom g;
    std::memset(&g, 0, sizeof(g));
    g.type = s->objects[i].type;
    g.materialid = s->objects[i].materialid;
    g.translation = s->objects[i].translations[frame];
    g.rotation = s->objects[i].rotations[frame];
    g.scale = s->objects[i].scales[frame];
    g.transform = s->objects[i].transforms[frame];
    g.inverseTransform = s->objects[i].inverseTransforms[frame];
    out[i] = g;
  }
}

void refscene_materials(void* h, void* out64) {
  scene* s = (scene*)h;
  std::memcpy(out64, s->materials.data(), s->materials.size() * sizeof(material));
}

// cameraData packed like src/raytraceKernel.cu:141-146
void refscene_camera(void* h, int frame, void* out52, char* name, int name_cap) {
  scene* s = (scene*)h;
  cameraData c;
  c.resolution = s->renderCam.resolution;
  c.position = s->renderCam.positions[frame];
  c.view = s->renderCam.views[frame];
  c.up = s->renderCam.ups[frame];
  c.fov = s->renderCam.fov;
  std::memcpy(out52, &c, sizeof(c));
  std::strncpy(name, s->renderCam.imageName.c_str(), name_cap - 1);
  name[name_cap - 1] = 0;
}

// The save path of runCuda(), src/main.cpp:118-139: mirror x, gamma{true,1.0,1}, frame number
// spliced into the name, image::saveImageRGB.  rgb is renderCam->image (W*H*3 floats).
void ref_save_image(const float* rgb, int W, int H, const char* image_name, int frame, char* out_name, int cap) {
  image outputImage(W, H);
  for (int x = 0; x < W; x++) {
    for (int y = 0; y < H; y++) {
      int index = x + (y * W);
      outputImage.writePixelRGB(W - 1 - x, y, glm::vec3(rgb[3 * index], rgb[3 * index + 1], rgb[3 * index + 2]));
    }
  }
  gammaSettings gamma;
  gamma.applyGamma = true;
  gamma.gamma = 1.0;
  gamma.divisor = 1.0;
  outputImage.setGammaSettings(gamma);
  std::string filename = image_name;
  std::stringstream out;
  out << frame;
  std::string s = out.str();
  utilityCore::replaceString(filename, ".bmp", "." + s + ".bmp");
  utilityCore::replaceString(filename, ".png", "." + s + ".png");
  outputImage.saveImageRGB(filename);
  std::strncpy(out_name, filename.c_str(), cap - 1);
  out_name[cap - 1] = 0;
}

}  // extern "C"
