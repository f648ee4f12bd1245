/* pt_b200.h -- C ABI of the B200-native wavefront path tracer (libpt_b200.so).
 *
 * Drop-in boundary for the hot path of CIS565-Fall-2014/Project3-Pathtracer.  Every entry point names the
 * reference interface it replaces (paths relative to the reference repo root).  Plain pointers and sizes only;
 * all pointers are HOST pointers unless a name says `device`.  Every function returns 0 on success and a
 * negative pt_status otherwise; pt_last_error() gives the message.  The library never calls exit() (the
 * reference does: src/raytraceKernel.cu:19-25) and never throws across the boundary.
 *
 * There is no CPU fallback: without a CUDA device every compute entry point fails with PT_ERR_CUDA.
 *
 * A context is not thread-safe (the reference is single-threaded: src/main.cpp:63-82); use one per GPU.
 */
#ifndef PT_B200_H
#define PT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PT_ABI_VERSION 1

typedef enum {
  PT_OK = 0,
  PT_ERR_INVALID = -1, /* bad argument */
  PT_ERR_CUDA = -2,    /* CUDA runtime error or no device */
  PT_ERR_IO = -3,      /* file could not be read / written */
  PT_ERR_PARSE = -4,   /* malformed scene file */
  PT_ERR_STATE = -5    /* call order (e.g. render on a destroyed context) */
} pt_status;

/* ---- POD images of the reference's structs (byte-for-byte the same layout) ---- */

/* staticGeom, src/sceneStructs.h:32-40 (172 bytes); cudaMat4 = 4 ROWS x,y,z,w, src/cudaMat4.h:18-23 */
typedef struct {
  int32_t type;       /* GEOMTYPE src/sceneStructs.h:14: 0 SPHERE, 1 CUBE, 2 MESH (never hit) */
  int32_t materialid;
  float translation[3];
  float rotation[3];
  float scale[3];
  float transform[16];
  float inverseTransform[16];
} pt_static_geom;

/* material, src/sceneStructs.h:63-74 (64 bytes) */
typedef struct {
  float color[3];
  float specularExponent;
  float specularColor[3];
  float hasReflective;
  float hasRefractive;
  float indexOfRefraction;
  float hasScatter;
  float absorptionCoefficient[3];
  float reducedScatterCoefficient;
  float emittance;
} pt_material;

/* cameraData, src/sceneStructs.h:42-48 (52 bytes); fov = half-angles in degrees (src/scene.cpp:203-207) */
typedef struct {
  float resolution[2];
  float position[3];
  float view[3];
  float up[3];
  float fov[2];
} pt_camera_data;

/* Thin lens for depth of field.  The reference camera has no such field (src/sceneStructs.h:50-61); the scene
 * loader reads it from a new top-level LENS block, which the reference's dispatcher ignores (src/scene.cpp:22-31). */
typedef struct {
  float aperture;       /* lens radius, 0 = pinhole */
  float focal_distance; /* plane of focus, measured along the view axis */
} pt_lens;

typedef struct pt_context pt_context;

/* ---- library ---- */
int pt_abi_version(void);
const char* pt_last_error(void);
int pt_device_count(int* count);

/* ---- context: replaces the per-call cudaMalloc/upload/free of cudaRaytraceCore (src/raytraceKernel.cu:118-138,
 * 157-159).  Geometry (one frame, already flattened as in :123-134), materials (never uploaded by the reference,
 * SURVEY.md D11) and the camera (:141-146) are uploaded once and stay resident in HBM. ---- */
int pt_context_create(const pt_static_geom* geoms, int n_geoms, const pt_material* materials, int n_materials,
                      const pt_camera_data* cam, const pt_lens* lens /* may be NULL */, int device,
                      pt_context** out);
int pt_context_destroy(pt_context* ctx);
/* replace the scene of an existing context (next animation frame: src/main.cpp:147-157); keeps the image size */
int pt_update_scene(pt_context* ctx, const pt_static_geom* geoms, int n_geoms, const pt_material* materials,
                    int n_materials, const pt_camera_data* cam, const pt_lens* lens);
/* upper bound on paths in flight per wavefront (rounded down to whole samples of the frame, at least one).
 * Default: 16 Mi paths. Path state costs 224 bytes of HBM per path of capacity: two wavefronts are in flight at a time
 * (on two internal streams, so that the tail of one overlaps the head of the other), each with two ping-pong buffers
 * of 3 float4. */
int pt_set_wavefront_paths(pt_context* ctx, uint64_t max_paths);
/* run on a caller-owned cudaStream_t instead of the context's own stream (NULL restores it) */
int pt_set_stream(pt_context* ctx, void* cuda_stream);
/* Which kernels trace a wavefront of a scene with few geoms -- a tuning / test knob; results never depend on it.
 *   bounce_kernel   depths >= 1: 0 = automatic (per depth, by the share of paths the scene keeps alive), 1 = always the
 *                   kernel that re-batches exact test + shading by winner type (k_bounce_q), 2 = always the fused one */
int pt_set_kernel_policy(pt_context* ctx, int bounce_kernel);
/* Pixels per wavefront band.  0 (default) = automatic: the whole frame, or bands of 1 Mi pixels when the float4
 * accumulation image exceeds 48 MB (e.g. 3840x2160: +9 %), so that the radiance atomics of the wavefronts in flight stay in
 * L2.  A wavefront then covers [band] x [more samples].  Results do not depend on it. */
int pt_set_band_pixels(pt_context* ctx, uint32_t pixels);

/* ---- render: replaces the raytraceRay launch (src/raytraceKernel.cu:149) and its per-iteration host round trip.
 * Traces samples [first_sample, first_sample + n_samples) of every pixel to at most max_depth segments and ADDS
 * their radiance to the accumulation buffer in HBM.  Asynchronous; pt_sync / pt_download_* wait for it.
 * The reference's `iterations` argument (1-based sample number, src/main.cpp:95) is first_sample + 1. ---- */
int pt_render(pt_context* ctx, uint32_t first_sample, uint32_t n_samples, int max_depth, uint64_t seed);
int pt_sync(pt_context* ctx);
/* zero the accumulation buffer and the counters: clearImage (src/raytraceKernel.cu:48-55) */
int pt_clear(pt_context* ctx);
/* GPU time of the most recent pt_render call, CUDA events on the launching stream; waits for it */
int pt_last_render_ms(pt_context* ctx, float* ms);

/* ---- image out: replaces the D2H of renderCam->image (src/raytraceKernel.cu:154).  rgb = W*H*3 floats in the
 * renderCam->image layout (index = x + y*W, src/main.cpp:122). ---- */
int pt_download_sum(pt_context* ctx, float* rgb);
int pt_download_mean(pt_context* ctx, float* rgb, uint32_t spp); /* sum / spp */
/* ---- sample streaming: the reference's loop reads the running mean after EVERY sample (src/main.cpp:93-113: one
 * cudaRaytraceCore per iteration, image copied back at src/raytraceKernel.cu:154).  Tracing one sample per call costs
 * eight small, latency-bound launches per sample; a stream traces samples AHEAD in groups at the throughput of a large
 * wavefront, forms their running means ahead as well, and lets a call only copy its mean to the host.
 *   pt_stream_begin  starts tracing samples first_sample, first_sample + 1, ... on top of the current sum, which holds
 *                    spp_before samples (two groups of `group` samples are in flight, each sample in an image of its own:
 *                    about 2 * group * W * H * 28 bytes of HBM)
 *   pt_stream_next   hands out the running mean after the next sample: rgb (host, W*H*3 floats) = (sum + that sample and all
 *                    streamed before it) / (spp_before + their number), the same binary32 adds in the same order as one
 *                    pt_render per sample when at most one path per pixel and sample carries radiance (no direct light
 *                    sampling); if device_rgba8 is not NULL that DEVICE buffer gets sendImageToPBO's bytes of the mean;
 *                    *spp (may be NULL) = the divisor used.  Returns when rgb is complete.
 *   pt_stream_end    folds the samples handed out so far into the accumulation buffer and drops the rest (every call that
 *                    reads or changes the buffer, the scene or the settings does the same implicitly) */
int pt_stream_begin(pt_context* ctx, uint32_t first_sample, uint32_t spp_before, int max_depth, uint64_t seed, uint32_t group);
int pt_stream_next(pt_context* ctx, float* rgb, void* device_rgba8, uint32_t* spp);
int pt_stream_end(pt_context* ctx);
/* overwrite the accumulation buffer (resume, or the running mean of the compat shim) */
int pt_upload_sum(pt_context* ctx, const float* rgb);
/* sendImageToPBO (src/raytraceKernel.cu:58-89): uchar4{r,g,b,0} = min(mean*255, 255), truncated.
 * Either destination may be NULL.  device_rgba8 is a DEVICE pointer (the reference's mapped PBO, src/main.cpp:96). */
int pt_resolve_rgba8(pt_context* ctx, uint32_t spp, uint8_t* host_rgba8, void* device_rgba8);
/* the float4[W*H] accumulation buffer itself (DEVICE pointer), for the multi-GPU reduce done by the host plumbing */
int pt_accum_device_ptr(pt_context* ctx, void** device_ptr, size_t* bytes);

/* Multi-GPU in ONE process (the headless driver): n contexts, one per GPU, each rendered a different range of
 * sample indices of the same frame; sums their accumulation buffers into ctxs[0] with one ncclReduce over NVLink.
 * (The reference is single-GPU: src/main.cpp:222.)  NCCL is loaded at run time; missing NCCL is an error. */
int pt_reduce_to_first(pt_context* const* ctxs, int n);

/* ---- counters (SURVEY.md 8d): paths started, segments traced (= sum of live), live[d] = paths for which
 * closest-hit ran at depth d; live must have room for 64 entries.  Waits for outstanding renders. ---- */
int pt_counters(pt_context* ctx, uint64_t* paths, uint64_t* segments, uint64_t* live);
/* number of this library's kernels launched for this context so far (render + resolve kernels) */
int pt_launch_count(pt_context* ctx, uint64_t* launches);

/* ---- stage entry points (same kernels' device functions; used by the parity tests and by callers that want one
 * stage).  All buffers are host buffers of n elements (x3 floats for vectors). ---- */
/* raycastFromCameraKernel (src/raytraceKernel.cu:40-45) + depth of field */
int pt_raygen(pt_context* ctx, uint64_t seed, int n, const uint32_t* pixel, const uint32_t* sample, float* origin,
              float* direction);
/* closest hit over all geoms: sphereIntersectionTest / boxIntersectionTest (src/intersections.h:74-117);
 * geom_id = -1 and t = -1 on a miss */
int pt_intersect(pt_context* ctx, int n, const float* origin, const float* direction, int32_t* geom_id, float* t,
                 float* point, float* normal);
/* the stream-compaction primitive (README.md:63-70) on its own: keeps values[i] where flags[i] != 0, order
 * preserved; out must have room for n entries */
int pt_compact_u32(int device, const uint32_t* values, const uint8_t* flags, uint64_t n, uint32_t* out,
                   uint64_t* n_out);
/* how pt_compact_u32 runs: 0 (default) = three launches -- per-tile counts (warp ballot / popc, block reduce), exclusive
 * scan of the tile aggregates (block scan + decoupled look-back across CTAs), scatter -- so that no streaming CTA ever
 * waits for another; 1 = the single-pass kernel with the look-back inside (half the throughput on B200) */
int pt_set_compact_mode(int mode);
/* the same, and the kernel(s) alone timed on the device (CUDA events, mean of `iters` launches after one warm-up) */
int pt_compact_u32_timed(int device, const uint32_t* values, const uint8_t* flags, uint64_t n, uint32_t* out,
                         uint64_t* n_out, int iters, float* kernel_ms);

/* Closest hit runs as a conservative filter over all geoms followed by the reference-exact test of the best
 * candidate, falling back to the exact scan of every geom when the filter cannot separate two surfaces
 * (csrc/pt_filter.cuh).  The answers are identical by construction; these entry points let callers check that.
 * pt_intersect_ex: mode PT_HIT_FILTERED is pt_intersect; PT_HIT_EXACT_SCAN runs the exact test on every geom in index
 * order (the specification).  fallbacks (may be NULL) = rays of this call that took the fallback. */
#define PT_HIT_FILTERED 0
#define PT_HIT_EXACT_SCAN 1
int pt_intersect_ex(pt_context* ctx, int mode, int n, const float* origin, const float* direction, int32_t* geom_id,
                    float* t, float* point, float* normal, uint64_t* fallbacks);
/* multiply every rounding-error term of the filter's bounds by `scale` (1 = shipped).  Test hook: parity must hold
 * at 1 with margin, i.e. also at scales well below 1; 0 disables the margins. */
int pt_set_filter_scale(pt_context* ctx, float scale);
/* Primary rays of a pinhole camera (no lens) in a scene of the pair scan first try a per-pixel candidate, worked out
 * once per pixel for the whole pixel footprint (DESIGN.md 3a "primary rays"); the filter scan runs only for rays that
 * candidate does not settle.  The table is rebuilt by pt_context_create, pt_update_scene and pt_set_filter_scale (its
 * margin scales with the filter's).
 * pt_primary_hit: the primary ray of each (pixel, sample) pair (as pt_raygen makes it with `seed`) through that depth-0
 * closest hit, with the results of pt_intersect_ex; decided[i] = 1 if the table's candidate settled ray i.  Scenes of the
 * pair scan only (PT_ERR_STATE otherwise).
 * pt_primary_table_info: *active = 1 if the current scene and camera have the table; build_ms (may be NULL) = the time
 * of one rebuild, measured by rebuilding it. */
int pt_primary_hit(pt_context* ctx, uint64_t seed, int n, const uint32_t* pixel, const uint32_t* sample, int32_t* geom_id,
                   float* t, float* point, float* normal, uint8_t* decided, uint64_t* fallbacks);
int pt_primary_table_info(pt_context* ctx, int* active, float* build_ms);
/* segments of pt_render calls since the last pt_clear whose closest hit took the exact-scan fallback */
int pt_filter_stats(pt_context* ctx, uint64_t* fallbacks);
/* scenes with a hierarchy: segments (and shadow rays) since pt_clear whose nearest candidate was not confirmed by its exact
 * test but whose closest hit the exact test of the SECOND candidate settled (the traversal keeps two) -- they are not
 * counted by pt_filter_stats, which counts the exact traversals */
int pt_filter_retries(pt_context* ctx, uint64_t* retries);

/* exhaustive check (all 2^32 inputs) of the kernels' single-guard IEEE sqrt, reciprocal and 1/sqrt against the generic
 * operators; bad[0..2] = number of differing results of each (must be 0) */
int pt_selftest_math(int device, uint64_t bad[3]);

/* ---- direct light sampling (SURVEY.md 8f rank 3; README.md "Sphere surface point sampling") ----
 * Off by default (every result above is then unchanged).  On: at each diffuse bounce that is not the path's last
 * allowed segment, one emissive sphere / cube is picked uniformly, one point on it is drawn with
 * getRandomPointOnCube's area-weighted face rule (src/intersections.h:140-172) or the sphere sampler (:179-182),
 * a shadow ray is traced through the same closest hit, and a visible point adds
 * thr * Le * cos cos' / (pi t^2) * area * lights * w, w = 1 / (1 + G K) (balance heuristic against the direction the bounce
 * samples itself; G = cos cos' / t^2, K = area * lights / pi); the continuing path weights the emission it meets at its
 * next hit by the complementary x / (1 + x) (DESIGN.md 4).  Same expected image, less noise; shadow rays are counted
 * apart from the path segments.  The shadow rays of a depth are queued (64 bytes each, one queue entry per path of
 * wavefront capacity, allocated by the first render that needs them) and traced by a launch of their own. */
int pt_set_direct_lighting(pt_context* ctx, int on);
/* ---- subsurface scattering (calculateScatterAndAbsorption, stub at src/interactions.h:36-39; README.md "subsurface
 * scattering") ----
 * Off by default: SCATTER and RSCTCOEFF are then carried but ignored, and every result is unchanged.  On: a sphere / cube
 * whose material has REFR > 0, SCATTER > 0 and RSCTCOEFF > 0 holds a homogeneous medium -- scattering coefficient
 * RSCTCOEFF (isotropic phase function), absorption ABSCOEFF per channel, the refractive surface as its boundary.  A
 * segment that ran inside it ends at a free-flight distance s = -log(1 - u) / RSCTCOEFF if that comes first: the path
 * goes on from there in a uniform direction, weighted by calculateTransmission over s, and the next emission it meets
 * counts in full (no light sample at such an event).  Each scattering event is one segment of max_depth.  Media block
 * shadow rays like any refractive geom; nested or overlapping media are not modelled.  Drops an open sample stream. */
int pt_set_subsurface(pt_context* ctx, int on);
/* ---- glossy reflection (material.specularExponent, SPECEX in the scene format) ----
 * Off by default: SPECEX is then carried but ignored, and every reflective material is a perfect mirror.  On: a sphere /
 * cube whose material has REFL > 0, REFR <= 0, SPECEX > 0 and EMITTANCE <= 0 reflects into a Phong lobe of exponent SPECEX
 * around the mirror direction (cos of the lobe angle distributed as c^(SPECEX+1)); a direction below the surface is
 * folded back above it, so the lobe's albedo is exactly SPECRGB.  A glossy event is specular for direct light sampling:
 * no light sample there, and the next emission its path meets counts in full.  Refractive materials keep ignoring
 * SPECEX.  As SPECEX grows the lobe becomes the mirror.  Drops an open sample stream. */
int pt_set_glossy(pt_context* ctx, int on);
/* shadow rays traced by pt_render calls since the last pt_clear; n_lights (may be NULL) = emissive geoms of the scene */
int pt_shadow_rays(pt_context* ctx, uint64_t* shadow_rays, int* n_lights);

/* ---- surface-point / direction sampling and absorption (host buffers; one launch each) ---- */
/* getRandomPointOnCube (src/intersections.h:133-175, implemented there: results are bit-identical to the reference's
 * host build, including its right-to-left argument evaluation order) and getRandomPointOnSphere (stub at :179-182;
 * uniform on the object-space sphere of radius .5), chosen by geom->type.  One world-space point per float seed:
 * generator = thrust minstd seeded with hash((unsigned)seed) like the reference; seeds must lie in [0, 2^32). */
int pt_random_points_on_geom(int device, const pt_static_geom* geom, int n, const float* seeds, float* points);
/* the same samplers driven by caller-supplied uniforms in [0,1): u = n x 3 (face roulette, two in-face coordinates
 * for a cube; z and azimuth for a sphere, third ignored) */
int pt_points_on_geom_u(int device, const pt_static_geom* geom, int n, const float* u, float* points);
/* getRandomDirectionInSphere (stub at src/interactions.h:93-95): uniform unit vectors from (xi1, xi2) */
int pt_random_directions_in_sphere(int device, int n, const float* xi1, const float* xi2, float* dirs);
/* calculateTransmission (stub at src/interactions.h:31-33): Beer-Lambert exp(-absorption * distance) per channel;
 * absorption = n x 3, distance = n.  pt_render applies it to every segment that runs inside a refractive geom whose
 * material has ABSCOEFF > 0. */
int pt_calculate_transmission(int device, int n, const float* absorption, const float* distance, float* out);
/* calculateScatterAndAbsorption (stub at src/interactions.h:36-39): the free flight pt_set_subsurface traces, for n
 * segments of length distance[i] inside a medium with absorption[i] (x3) and scattering coefficient scatter[i] > 0,
 * driven by u[i] = (xi1, xi2, xf) in [0,1): s[i] = -log(1 - xf) / scatter[i]; if s[i] < distance[i] then scattered[i] = 1,
 * direction[i] = getRandomDirectionInSphere(xi1, xi2), weight[i] = calculateTransmission over s[i]; otherwise
 * scattered[i] = 0, direction[i] = 0 and weight[i] = calculateTransmission over distance[i]. */
int pt_sample_medium(int device, int n, const float* absorption, const float* scatter, const float* distance, const float* u,
                     int32_t* scattered, float* s, float* direction, float* weight);
/* the glossy lobe pt_set_glossy samples, for n reflections: outward normal[i] (x3) of the surface, incident[i] (x3) the
 * unit direction of the arriving ray, exponent[i] = SPECEX > 0, u[i] = (u0, u1) in [0,1).  ns = normal[i] turned to face
 * incident[i], r = reflect(ns, incident[i]); direction[i] = the sample of the lobe around r (unit length, dot with ns
 * >= 0). */
int pt_sample_glossy(int device, int n, const float* normal, const float* incident, const float* exponent, const float* u,
                     float* direction);

/* What the reference's own cudaRaytraceCore leaves in renderCam->image TODAY: its raytraceRay is a stub that overwrites
 * every pixel with generateRandomNumberFromThread(resolution, (float)iterations, x, y) (src/raytraceKernel.cu:29-36,
 * 93-104).  Reproduced bit for bit so that a maintainer can check the drop-in against the unmodified reference: order
 * PT_STUB_ORDER_DEVICE = the draw order of the reference's kernel on the GPU, PT_STUB_ORDER_HOST = of its host build
 * (the three draws are arguments of one constructor call, so their order is the compiler's). */
#define PT_STUB_ORDER_DEVICE 0
#define PT_STUB_ORDER_HOST 1
int pt_reference_stub_image(int device, int width, int height, int iterations, int order, float* rgb);

/* ---- scene file and image file (host side; same formats as the reference) ---- */
typedef struct pt_scene pt_scene;
/* scene::scene(string), src/scene.cpp:11-35.  rotat_degrees = 0 reproduces the reference exactly (ROTAT is
 * consumed as radians, SURVEY.md D1); 1 converts ROTAT from degrees. */
int pt_scene_load(const char* path, int rotat_degrees, pt_scene** out);
int pt_scene_free(pt_scene* s);
int pt_scene_info(const pt_scene* s, int* n_geoms, int* n_materials, int* n_frames, int* width, int* height,
                  int* iterations, char* image_name, int image_name_cap);
/* flatten one frame the way cudaRaytraceCore does (src/raytraceKernel.cu:123-146); arrays sized by pt_scene_info */
int pt_scene_frame(const pt_scene* s, int frame, pt_static_geom* geoms, pt_material* materials,
                   pt_camera_data* cam, pt_lens* lens);
/* the save path of runCuda (src/main.cpp:118-139) + image::saveImageRGB (src/image.cpp:46-88): mirror x, identity
 * gamma, clamp(f*255,0,255) truncated, ".<frame>" spliced before .png/.bmp, BMP iff the name ends in "bmp".
 * force_png = 1 rewrites a trailing .bmp to .png first (headless default).  out_name may be NULL. */
int pt_save_image(const float* rgb, int width, int height, const char* image_name, int frame, int force_png,
                  char* out_name, int out_name_cap);
/* the 8-bit conversion alone: rgb8 = W*H*3 bytes, rows top-down, x mirrored (what the file holds) */
int pt_image_to_rgb8(const float* rgb, int width, int height, uint8_t* rgb8);

#ifdef __cplusplus
}
#endif
#endif /* PT_B200_H */
