// pt_main.cpp -- headless driver: the reference's main()/runCuda() loop without GL.
//
// Follows reference src/main.cpp:16-61 (argv tokens `scene=<file>` and `frame=<n>` split on '='), :88-159 (iterate
// until renderCam->iterations, save with the frame number spliced into the name, advance to the next frame unless
// frame= was given) -- but renders all samples of a frame in one pt_render call per GPU instead of one
// cudaRaytraceCore call per sample, keeps the image in HBM, and writes PNG (out= / bmp=1 to override).
//
//   pt_render scene=<file> [frame=<n>] [spp=<n>] [depth=<n>] [seed=<n>] [gpus=<n>] [out=<name>] [bmp=1]
//             [rotat=degrees] [wavefront=<paths>] [json=1] [direct=1] [sss=1] [glossy=1]
//
// direct=1 turns on direct light sampling at diffuse bounces (pt_set_direct_lighting); sss=1 turns on subsurface
// scattering inside refractive geoms whose material has SCATTER and RSCTCOEFF (pt_set_subsurface); glossy=1 turns on
// glossy reflection for reflective materials with SPECEX > 0 (pt_set_glossy).
//
// gpus=N shards the samples of each frame over N GPUs by contiguous sample-index blocks (one host thread and one
// context per GPU) and combines the accumulation buffers with one NCCL reduce.
#include "pt_b200.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

static int die(const char* what) {
  fprintf(stderr, "pt_render: %s: %s\n", what, pt_last_error());
  return 1;
}

int main(int argc, char** argv) {
  std::string scene_path, out_name;
  int frame = -1, spp = -1, depth = 8, gpus = 1, bmp = 0, rot_deg = 0, json = 0, direct = 0, sss = 0, glossy = 0;
  unsigned long long seed = 0, wavefront = 0;
  for (int i = 1; i < argc; i++) {
    std::string tok = argv[i];
    size_t eq = tok.find('=');
    if (eq == std::string::npos) continue;
    std::string k = tok.substr(0, eq), v = tok.substr(eq + 1);
    if (k == "scene") scene_path = v;
    else if (k == "frame") frame = atoi(v.c_str());
    else if (k == "spp") spp = atoi(v.c_str());
    else if (k == "depth") depth = atoi(v.c_str());
    else if (k == "seed") seed = strtoull(v.c_str(), nullptr, 10);
    else if (k == "gpus") gpus = atoi(v.c_str());
    else if (k == "out") out_name = v;
    else if (k == "bmp") bmp = atoi(v.c_str());
    else if (k == "rotat") rot_deg = (v == "degrees");
    else if (k == "wavefront") wavefront = strtoull(v.c_str(), nullptr, 10);
    else if (k == "json") json = atoi(v.c_str());
    else if (k == "direct") direct = atoi(v.c_str());
    else if (k == "sss") sss = atoi(v.c_str());
    else if (k == "glossy") glossy = atoi(v.c_str());
  }
  if (scene_path.empty()) {
    // main.cpp:38-41
    fprintf(stderr, "Error: scene file needed!\nusage: pt_render scene=<file> [frame=<n>] [spp=<n>] [depth=<n>] [seed=<n>] "
                    "[gpus=<n>] [out=<name>] [bmp=1] [rotat=degrees] [wavefront=<paths>] [json=1] [direct=1] [sss=1] [glossy=1]\n");
    return 1;
  }
  pt_scene* sc = nullptr;
  if (pt_scene_load(scene_path.c_str(), rot_deg, &sc)) return die("scene");
  int n_geoms, n_mats, n_frames, W, H, iterations;
  char name[512];
  pt_scene_info(sc, &n_geoms, &n_mats, &n_frames, &W, &H, &iterations, name, sizeof(name));
  if (spp <= 0) spp = iterations;
  if (out_name.empty()) out_name = name[0] ? name : "render.png";
  int ndev = 0;
  if (pt_device_count(&ndev) || ndev < 1) return die("no CUDA device (there is no CPU fallback)");
  if (gpus < 1 || gpus > ndev) { fprintf(stderr, "pt_render: gpus=%d but %d device(s) present\n", gpus, ndev); return 1; }

  const int f0 = frame >= 0 ? frame : 0, f1 = frame >= 0 ? frame : n_frames - 1;  // singleFrameMode, main.cpp:32-35
  std::vector<pt_static_geom> geoms(n_geoms);
  std::vector<pt_material> mats(n_mats);
  pt_camera_data cam;
  pt_lens lens;
  std::vector<pt_context*> ctx(gpus, nullptr);
  std::vector<float> img((size_t)W * H * 3);
  for (int f = f0; f <= f1; f++) {
    if (pt_scene_frame(sc, f, geoms.data(), mats.data(), &cam, &lens)) return die("frame");
    for (int g = 0; g < gpus; g++) {
      int rc = ctx[g] ? pt_update_scene(ctx[g], geoms.data(), n_geoms, mats.data(), n_mats, &cam, &lens)
                      : pt_context_create(geoms.data(), n_geoms, mats.data(), n_mats, &cam, &lens, g, &ctx[g]);
      if (rc) return die("context");
      if (wavefront && pt_set_wavefront_paths(ctx[g], wavefront)) return die("wavefront");
      if (pt_set_direct_lighting(ctx[g], direct)) return die("direct");
      if (pt_set_subsurface(ctx[g], sss)) return die("sss");
      if (pt_set_glossy(ctx[g], glossy)) return die("glossy");
      if (pt_clear(ctx[g])) return die("clear");
    }
    auto t0 = std::chrono::steady_clock::now();
    std::vector<int> rcs(gpus, 0);
    std::vector<std::string> errs(gpus);  // pt_last_error() is per thread: the worker keeps its own message
    std::vector<std::thread> th;
    for (int g = 0; g < gpus; g++) {
      // contiguous blocks of sample indices; the union over GPUs is exactly [0, spp)
      const unsigned s_begin = (unsigned)((long long)spp * g / gpus), s_end = (unsigned)((long long)spp * (g + 1) / gpus);
      th.emplace_back([&, g, s_begin, s_end] {
        rcs[g] = s_end > s_begin ? pt_render(ctx[g], s_begin, s_end - s_begin, depth, seed) : 0;
        if (!rcs[g]) rcs[g] = pt_sync(ctx[g]);
        if (rcs[g]) errs[g] = pt_last_error();
      });
    }
    for (auto& t : th) t.join();
    for (int g = 0; g < gpus; g++)
      if (rcs[g]) { fprintf(stderr, "pt_render: render on GPU %d failed (%d): %s\n", g, rcs[g], errs[g].c_str()); return 1; }
    if (gpus > 1 && pt_reduce_to_first(ctx.data(), gpus)) return die("reduce");
    if (pt_download_mean(ctx[0], img.data(), (unsigned)spp)) return die("download");
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    unsigned long long paths = 0, segs = 0;
    for (int g = 0; g < gpus; g++) {
      unsigned long long p = 0, s = 0;
      uint64_t live[64];
      if (pt_counters(ctx[g], (uint64_t*)&p, (uint64_t*)&s, live)) return die("counters");
      paths += p; segs += s;
    }
    char saved[1024];
    if (pt_save_image(img.data(), W, H, out_name.c_str(), f, bmp ? 0 : 1, saved, sizeof(saved))) return die("save");
    if (json)
      printf("{\"frame\": %d, \"file\": \"%s\", \"width\": %d, \"height\": %d, \"spp\": %d, \"depth\": %d, \"gpus\": %d, "
             "\"paths\": %llu, \"segments\": %llu, \"seconds\": %.6f, \"mseg_per_s\": %.3f, \"spp_per_s\": %.3f}\n",
             f, saved, W, H, spp, depth, gpus, paths, segs, secs, segs / secs / 1e6, spp / secs);
    else
      printf("Saved frame %d to %s  (%d spp, %llu segments, %.3f s, %.1f Mseg/s)\n", f, saved, spp, segs, secs, segs / secs / 1e6);
  }
  for (pt_context* c : ctx) pt_context_destroy(c);
  pt_scene_free(sc);
  return 0;
}
