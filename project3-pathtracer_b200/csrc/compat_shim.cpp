// compat_shim.cpp -- cudaRaytraceCore with the reference's exact C++ signature, on top of the C ABI.
//
// Replaces reference src/raytraceKernel.cu:108-165 (declared at src/raytraceKernel.h:17, called at src/main.cpp:110).
// Differences inside the call: the scene is re-uploaded only when its bytes change, device buffers live in a cached
// context instead of being malloc'ed and freed per call (:118-119,136-137,157-159), and while calls arrive in
// sequence (k, k+1, ...) the exact running SUM stays in HBM, so the per-call H2D of the image (:120) disappears;
// the D2H of the running mean into renderCam->image (:154) is kept because the caller owns and reads that buffer.
// The samples themselves are traced AHEAD of the calls, a group at a time (pt_stream_*: the reference's loop calls again
// with k + 1, src/main.cpp:93-95), so a call in sequence only adds its sample to the sum and copies the mean.  A call
// that does not continue the sequence (other scene, frame, camera, iteration number, depth, seed) drops what was traced
// ahead: it restarts from renderCam->image or from zero exactly as before.
#include "../../include/pt_b200.h"
#include "../../include/pt_compat.h"

#include <cuda_runtime_api.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

static_assert(sizeof(geom) == 56 && sizeof(material) == 64 && sizeof(cudaMat4) == 64 && sizeof(ray) == 24,
              "reference struct layouts (SURVEY.md appendix B)");
static_assert(sizeof(pt_material) == sizeof(material), "material image");

namespace {
struct Cache {
  pt_context* ctx = nullptr;
  int W = 0, H = 0, device = 0;
  std::vector<pt_static_geom> geoms;
  std::vector<pt_material> mats;
  pt_camera_data cam{};
  pt_lens lens{0.0f, 0.0f};
  const camera* last_cam = nullptr;
  int last_frame = -1, last_iter = 0;
  bool streaming = false;  // a sample stream is open on ctx: samples last_iter, last_iter + 1, ... are traced ahead
  int stream_depth = 0, stream_direct = 0, stream_sss = 0, stream_glossy = 0;
  unsigned long long stream_seed = 0;
  int direct_applied = -1; // pt_set_direct_lighting drops the stream: only called when the value changes
  int sss_applied = -1;    // ... and so does pt_set_subsurface
  int glossy_applied = -1; // ... and pt_set_glossy
  std::vector<float> scaled;
  void* pinned = nullptr;  // renderCam->image, page-locked in place while a sequence of calls keeps arriving for it
  size_t pinned_bytes = 0;
  void* pin_failed = nullptr;  // ... or the buffer that could not be locked (not retried on every call)
} g;
int g_depth = 8;
unsigned long long g_seed = 0;
int g_device = 0;
pt_lens g_lens{0.0f, 0.0f};
int g_exit_on_error = 1;
int g_ahead = 8;   // samples per group traced ahead of the calls (pt_compat_set_ahead)
int g_direct = 0;  // pt_compat_set_direct_lighting
int g_sss = 0;     // pt_compat_set_subsurface
int g_glossy = 0;  // pt_compat_set_glossy
int g_stub = 0;    // pt_compat_set_reference_stub
int g_status = PT_OK;

void fail(int rc) {
  g_status = rc;
  if (g_exit_on_error) {
    // checkCUDAError, src/raytraceKernel.cu:19-25
    fprintf(stderr, "Cuda error: %s: %s.\n", "Kernel failed!", pt_last_error());
    exit(EXIT_FAILURE);
  }
}
}  // namespace

extern "C" int pt_compat_set_trace_depth(int depth) {
  if (depth < 1 || depth > 64) return PT_ERR_INVALID;
  g_depth = depth;
  return PT_OK;
}
extern "C" int pt_compat_set_seed(unsigned long long seed) { g_seed = seed; return PT_OK; }
extern "C" int pt_compat_set_device(int device) { g_device = device; return PT_OK; }
extern "C" int pt_compat_set_lens(float aperture, float focal_distance) {
  g_lens.aperture = aperture;
  g_lens.focal_distance = focal_distance;
  return PT_OK;
}
extern "C" int pt_compat_set_exit_on_error(int on) { g_exit_on_error = on; return PT_OK; }
extern "C" int pt_compat_set_ahead(int samples) {
  if (samples < 1 || samples > 64) return PT_ERR_INVALID;
  if (samples != g_ahead) pt_compat_reset();  // the cached context sized its wavefront for the old group
  g_ahead = samples;
  return PT_OK;
}
extern "C" int pt_compat_set_direct_lighting(int on) { g_direct = on != 0; return PT_OK; }
extern "C" int pt_compat_set_subsurface(int on) { g_sss = on != 0; return PT_OK; }
extern "C" int pt_compat_set_glossy(int on) { g_glossy = on != 0; return PT_OK; }
extern "C" int pt_compat_set_reference_stub(int on) { g_stub = on != 0; return PT_OK; }
extern "C" int pt_compat_last_status(void) { return g_status; }
// The caller reads renderCam->image after every call (src/main.cpp:118-131), so its D2H copy cannot go away; but a
// pageable destination makes it a staged ~10 GB/s copy.  Page-locking the caller's buffer in place (it lives as long as
// the scene, src/scene.cpp:207-214) turns it into one DMA.  Failure to lock is harmless: the copy stays pageable.
// The registration is renewed at the start of every sequence (iterations == 1) and whenever pointer or size change: a
// host that frees and re-creates its image between renders (the reference rebuilds scenes) never leaves a stale
// registration behind for longer than the sequence that owned it.
static void unpin() {
  if (g.pinned) { cudaHostUnregister(g.pinned); cudaGetLastError(); g.pinned = nullptr; g.pinned_bytes = 0; }
}
static void pin(void* image, size_t bytes, bool new_sequence) {
  if (!new_sequence && ((g.pinned == image && g.pinned_bytes == bytes) || g.pin_failed == image)) return;
  unpin();
  const cudaError_t e = cudaHostRegister(image, bytes, cudaHostRegisterDefault);
  if (e == cudaSuccess) { g.pinned = image; g.pinned_bytes = bytes; g.pin_failed = nullptr; }
  else { cudaGetLastError(); g.pin_failed = image; }
  if (getenv("PT_COMPAT_DEBUG")) fprintf(stderr, "pt_compat: cudaHostRegister(%p, %zu) -> %s\n", image, bytes, cudaGetErrorString(e));
}
extern "C" void pt_compat_reset(void) {
  unpin();
  if (g.ctx) pt_context_destroy(g.ctx);
  g = Cache();
}

void cudaRaytraceCore(uchar4* PBOpos, camera* renderCam, int frame, int iterations, material* materials,
                      int numberOfMaterials, geom* geoms, int numberOfGeoms) {
  g_status = PT_OK;
  if (!renderCam || !materials || !geoms || numberOfGeoms <= 0 || numberOfMaterials <= 0 || iterations < 1 ||
      !renderCam->image) {
    fprintf(stderr, "cudaRaytraceCore: bad arguments\n");
    g_status = PT_ERR_INVALID;
    if (g_exit_on_error) exit(EXIT_FAILURE);
    return;
  }
  // package geometry and camera for `frame`, like src/raytraceKernel.cu:123-146
  std::vector<pt_static_geom> sg((size_t)numberOfGeoms);
  for (int i = 0; i < numberOfGeoms; i++) {
    pt_static_geom& s = sg[i];
    memset(&s, 0, sizeof(s));
    s.type = (int)geoms[i].type;
    s.materialid = geoms[i].materialid;
    memcpy(s.translation, &geoms[i].translations[frame], 12);
    memcpy(s.rotation, &geoms[i].rotations[frame], 12);
    memcpy(s.scale, &geoms[i].scales[frame], 12);
    memcpy(s.transform, &geoms[i].transforms[frame], 64);
    memcpy(s.inverseTransform, &geoms[i].inverseTransforms[frame], 64);
  }
  pt_camera_data cam;
  cam.resolution[0] = renderCam->resolution.x; cam.resolution[1] = renderCam->resolution.y;
  memcpy(cam.position, &renderCam->positions[frame], 12);
  memcpy(cam.view, &renderCam->views[frame], 12);
  memcpy(cam.up, &renderCam->ups[frame], 12);
  cam.fov[0] = renderCam->fov.x; cam.fov[1] = renderCam->fov.y;
  const int W = (int)cam.resolution[0], H = (int)cam.resolution[1];
  const size_t npix = (size_t)W * H;
  const pt_material* pm = reinterpret_cast<const pt_material*>(materials);

  int rc;
  bool scene_changed = false;
  if (g.ctx && (g.W != W || g.H != H || g.device != g_device)) pt_compat_reset();
  if (!g.ctx) {
    if ((rc = pt_context_create(sg.data(), numberOfGeoms, pm, numberOfMaterials, &cam, &g_lens, g_device, &g.ctx))) return fail(rc);
    // samples are traced ahead a group at a time: one wavefront per group
    if ((rc = pt_set_wavefront_paths(g.ctx, npix * (size_t)g_ahead))) return fail(rc);
    g.W = W; g.H = H; g.device = g_device;
    scene_changed = true;
  } else if (g.geoms.size() != sg.size() || memcmp(g.geoms.data(), sg.data(), sg.size() * sizeof(pt_static_geom)) ||
             g.mats.size() != (size_t)numberOfMaterials || memcmp(g.mats.data(), pm, g.mats.size() * sizeof(pt_material)) ||
             memcmp(&g.cam, &cam, sizeof(cam)) || memcmp(&g.lens, &g_lens, sizeof(g_lens))) {
    if ((rc = pt_update_scene(g.ctx, sg.data(), numberOfGeoms, pm, numberOfMaterials, &cam, &g_lens))) return fail(rc);
    scene_changed = true;
  }
  if (scene_changed) {
    g.geoms = sg;
    g.mats.assign(pm, pm + numberOfMaterials);
    g.cam = cam;
    g.lens = g_lens;
  }

  if (g_stub) {
    // what the unmodified reference does today (src/raytraceKernel.cu:93-104,149-154): every pixel overwritten with
    // generateRandomNumberFromThread(resolution, (float)iterations, x, y), the PBO converted from that image
    float* im = reinterpret_cast<float*>(renderCam->image);
    if ((rc = pt_reference_stub_image(g_device, W, H, iterations, PT_STUB_ORDER_DEVICE, im))) return fail(rc);
    if (PBOpos) {
      if ((rc = pt_upload_sum(g.ctx, im))) return fail(rc);
      if ((rc = pt_resolve_rgba8(g.ctx, 1, nullptr, PBOpos))) return fail(rc);
    }
    g.last_cam = nullptr;  // the next real call resumes from the caller's image
    g.streaming = false;   // (pt_upload_sum above dropped any samples traced ahead)
    return;
  }
  const bool in_sequence = !scene_changed && g.last_cam == renderCam && g.last_frame == frame && iterations == g.last_iter + 1;
  // the stream of samples traced ahead goes on if this call is the next iteration with the same settings
  const bool stream_ok = g.streaming && in_sequence && g.stream_depth == g_depth && g.stream_seed == g_seed &&
                         g.stream_direct == g_direct && g.stream_sss == g_sss && g.stream_glossy == g_glossy;
  if (!stream_ok) {
    if (g.streaming) { g.streaming = false; if ((rc = pt_stream_end(g.ctx))) return fail(rc); }
    if (iterations == 1) {
      if ((rc = pt_clear(g.ctx))) return fail(rc);
    } else if (!in_sequence) {
      // resume from the caller's running mean: sum = image * (k-1)
      g.scaled.resize(npix * 3);
      const float k1 = (float)(iterations - 1);
      const float* im = reinterpret_cast<const float*>(renderCam->image);
      for (size_t i = 0; i < npix * 3; i++) g.scaled[i] = im[i] * k1;
      if ((rc = pt_upload_sum(g.ctx, g.scaled.data()))) return fail(rc);
    }  // (in sequence with other settings: the exact sum of the samples so far is in HBM and stays)
    if (g.direct_applied != g_direct) {
      if ((rc = pt_set_direct_lighting(g.ctx, g_direct))) return fail(rc);
      g.direct_applied = g_direct;
    }
    if (g.sss_applied != g_sss) {
      if ((rc = pt_set_subsurface(g.ctx, g_sss))) return fail(rc);
      g.sss_applied = g_sss;
    }
    if (g.glossy_applied != g_glossy) {
      if ((rc = pt_set_glossy(g.ctx, g_glossy))) return fail(rc);
      g.glossy_applied = g_glossy;
    }
    if ((rc = pt_stream_begin(g.ctx, (uint32_t)(iterations - 1), (uint32_t)(iterations - 1), g_depth, g_seed, (uint32_t)g_ahead))) return fail(rc);
    g.streaming = true; g.stream_depth = g_depth; g.stream_seed = g_seed; g.stream_direct = g_direct; g.stream_sss = g_sss;
    g.stream_glossy = g_glossy;
  }
  if (in_sequence || iterations == 1) pin(renderCam->image, npix * 3 * sizeof(float), iterations == 1);  // a render loop, not a one-off call
  if ((rc = pt_stream_next(g.ctx, reinterpret_cast<float*>(renderCam->image), PBOpos, nullptr))) return fail(rc);
  g.last_cam = renderCam;
  g.last_frame = frame;
  g.last_iter = iterations;
}
