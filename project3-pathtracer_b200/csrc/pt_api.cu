// pt_api.cu -- the C ABI (include/pt_b200.h) over the wavefront kernels.
//
// Replaces the body of cudaRaytraceCore (reference src/raytraceKernel.cu:108-165): instead of malloc / upload /
// launch / download / free once per sample, a context keeps the scene, the path-state ping-pong buffers and the
// accumulation image resident in HBM, and pt_render() traces any number of samples with no host round trip.
//
// Compiled with -fmad=false (see pt_device.cuh: the arithmetic contract).
#include "../../include/pt_b200.h"
#include "pt_kernels.cuh"

#include <nvtx3/nvToolsExt.h>  // header-only; ranges cost nothing unless a profiler is attached

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <thread>
#include <utility>
#include <functional>
#include <vector>

using namespace ptd;

// NVTX range around a stage of the render (profiler timelines: "pt_render", "band", "wavefront", "reduce")
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------- errors
static thread_local std::string g_err;
extern "C" void pt_set_error_(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}
extern "C" const char* pt_last_error(void) { return g_err.c_str(); }
extern "C" int pt_abi_version(void) { return PT_ABI_VERSION; }

#define CU(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) {                                                                 \
      pt_set_error_("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return PT_ERR_CUDA;                                                                    \
    }                                                                                        \
  } while (0)

extern "C" int pt_device_count(int* count) {
  if (!count) { pt_set_error_("count is NULL"); return PT_ERR_INVALID; }
  *count = 0;
  CU(cudaGetDeviceCount(count));
  return PT_OK;
}

// ---------------------------------------------------------------- context
// the filter constants build_filter gave one geom of the pair scan (the primary-ray table is built from them)
struct FiltGeom {
  int key, cls, geom;  // key = 2 * pair + half, as the scan reports its candidate
  float c[3], k[6], wk[6], ew_c, ew_w;
};
struct pt_context {
  int device = 0;
  int sm_count = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  // scene
  int n_geoms = 0, n_mats = 0;
  float4* d_rows = nullptr;  // 6 arrays of n_geoms float4
  int2* d_meta = nullptr;
  float4* d_normals = nullptr;  // kNormalRows float4 per geom: face normals + sphere centre (k_normal_table)
  float4* d_mats = nullptr;
  float4* d_lights = nullptr;  // direct light sampling: 3 float4 per emissive sphere / cube (build_lights)
  float* d_light_k = nullptr;  // per geom: K = area * n_lights / pi of a light, 0 otherwise
  int n_lights = 0;
  bool nee = false;            // pt_set_direct_lighting
  bool sss = false;            // pt_set_subsurface
  int n_media = 0;             // spheres / cubes whose material makes them a scattering medium (DESIGN.md 4)
  bool glossy = false;         // pt_set_glossy
  int n_glossy = 0;            // spheres / cubes whose material makes them glossy reflectors (DESIGN.md 4)
  int rr_first = 0;            // pt_set_russian_roulette: first roulette depth, 0 = off
  float4* d_filt = nullptr;   // kFiltRows arrays of n_pairs float4: filter geometry (pt_filter.cuh)
  int2* d_filt_ids = nullptr;
  FiltSoA filt{};
  int filt_cap = 0;
  float4* d_bvh_nodes = nullptr;   // hierarchy over the filter tests (pt_bvh.cuh), scenes with >= kBvhMinGeoms geoms
  float4* d_bvh_leaves = nullptr;
  int2* d_bvh_meta = nullptr;
  BvhSoA bvh{};
  float filter_scale = 1.0f;  // multiplies every error-model term of the filter (test hook; 1 = the shipped bounds)
  std::vector<pt_static_geom> h_geoms;  // host copy, to rebuild the filter when the scale changes
  std::vector<FiltGeom> filt_geoms;  // the filter constants of every geom (build_filter), for the primary-ray table
  uint32_t* d_ptab = nullptr;  // per pixel: candidate of the primary rays (k_primary_table), npix words
  PrimRec* d_prim = nullptr;   // the table's per-geom records (kMaxPrimRecs)
  bool ptab_on = false;        // d_ptab holds the table of the current scene, camera and filter scale
  GeomSoA g{};
  RaygenConsts cam{};
  uint32_t W = 0, H = 0, npix = 0;
  // wavefront
  uint64_t wf_capacity = 0;  // paths
  uint32_t band_pixels = 0;  // pixels per wavefront band; 0 = automatic (pt_set_band_pixels)
  // Two wavefronts are in flight at a time, each on its own internal stream with its own path-state buffers and control
  // block: the tail of one wavefront's launch (its last units) overlaps the head of the other's instead of idling SMs.
#ifndef PT_WF_SLOTS
#define PT_WF_SLOTS 2
#endif
  static const int kSlots = PT_WF_SLOTS;
  float4* d_shadow = nullptr;   // direct light sampling: per slot 4 arrays of shadow_cap float4 (the depth's queue of shadow rays)
  uint64_t shadow_cap = 0;      // ... allocated when the first render with direct lighting needs it (ensure_shadow)
  int shadow_slots = 0;
  int grid_blocks_shadow = 0;   // resident CTAs of k_shadow_lin / k_shadow_bvh ...
  int shadow_cfg_mode = -1;     // ... worked out for this scene mode and this much filter geometry
  size_t shadow_cfg_smem = 0;
  float4* d_state = nullptr; // per slot (state_bytes): 6 arrays of wf_capacity float4: o0 d0 t0 o1 d1 t1, then wf_capacity float4 (hierarchy results)
  WfCtrl* d_ctrl = nullptr;  // per slot
  int n_slots = kSlots;      // slots in use (1 for frames whose accumulation image alone fills the L2)
  cudaStream_t wf_stream[kSlots] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kSlots] = {};
  unsigned long long* d_live = nullptr;  // kMaxDepth totals, then fallbacks, then shadow rays
  uint64_t paths_total = 0;
  uint64_t launches = 0;     // kernels of this library launched on behalf of this context
  // image
  float4* d_accum = nullptr;
  float* d_rgb = nullptr;      // staging for packed RGB
  uchar4* d_rgba8 = nullptr;   // staging for the 8-bit resolve
  // persistent grid of each entry of the kernel tables (kBounceKernels), 0 = no such kernel
  int grid_blocks[2][2][kFxSets] = {};  // [FIRST][LAST][FX]: k_bounce, or k_bounce_bvh in the hierarchy mode
  int grid_blocks_q[2][kFxSets] = {};   // [LAST][FX]: k_bounce_q (depths >= 1 of the linear mode)
  size_t q_smem_total = 0;            // k_bounce_q: filter geometry + the warps' candidate queues
  int q_mode = 0;                     // depths >= 1, few geoms: 0 = per depth by the scene's measured survival (h_policy),
                                      // 1 = always k_bounce_q, 2 = always the fused k_bounce (PT_B200_FUSED=1 / =0 force 2 / 1)
  void* d_scratch = nullptr;          // grow-only device arena of the list entry points (pt_raygen, pt_intersect_ex): no
  size_t scratch_bytes = 0;           // cudaMalloc / cudaFree per call
  int* h_policy = nullptr;            // mapped host memory, kMaxDepth + 1 ints written by k_accum_counts: 0 unknown, 1 q, 2 fused
  int* d_policy = nullptr;            // ... its device address
  // sample streaming (pt_stream_*): samples are traced ahead in groups into per-sample images ("slabs") on ahead_stream,
  // folded into d_accum one per call on the caller's stream, and the running mean leaves through copy_stream
  cudaStream_t copy_stream = nullptr, ahead_stream = nullptr;
  cudaEvent_t ev_res = nullptr, ev_copy = nullptr, ev_ready[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  float4* d_slab = nullptr;           // 2 groups x stream_group images of npix float4
  float* d_means = nullptr;           // 2 groups x stream_group running means (npix * 3 floats each), computed ahead
  float4* d_base[2] = {nullptr, nullptr};  // d_base[s]: the sum before the group that lives in slot s
  uint32_t slab_group = 0;            // images per group the buffers above were allocated for
  bool stream_open = false;
  uint32_t stream_base = 0, stream_next = 0, stream_group = 0;  // first sample of the stream, next sample to hand out, samples per group
  uint32_t stream_spp0 = 0;           // samples in the sum before the stream's first sample
  int stream_depth = 0;
  uint64_t stream_seed = 0;
  int mode = -1;                      // 0: linear scan over pairs staged in shared memory, 1: hierarchy (pt_bvh.cuh)
  size_t smem_bytes = 0;   // k_bounce: filter geometry
  size_t geom_smem = 0;    // filter geometry only (k_intersect_list)
};

static const uint64_t kDefaultWavefrontPaths = 16ull << 20;
static const int kMaxSmemPairs = 64;    // the linear scan serves scenes below kBvhMinGeoms geoms: at most 16 + 3 pairs, 3 KB of shared memory

// ---------------------------------------------------------------- filter constants (pt_filter.cuh, DESIGN.md "filter")
// largest eigenvalue of the symmetric 3x3 matrix S (cyclic Jacobi, binary64)
static void sym3_eigen_range(double S[3][3], double* emin, double* emax) {
  for (int sweep = 0; sweep < 32; sweep++) {
    double off = fabs(S[0][1]) + fabs(S[0][2]) + fabs(S[1][2]);
    if (off < 1e-300) break;
    for (int p = 0; p < 2; p++)
      for (int q = p + 1; q < 3; q++) {
        if (S[p][q] == 0.0) continue;
        const double th = (S[q][q] - S[p][p]) / (2.0 * S[p][q]);
        const double t = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < 3; k++) {  // S <- S * J
          const double skp = S[k][p], skq = S[k][q];
          S[k][p] = c * skp - sn * skq; S[k][q] = sn * skp + c * skq;
        }
        for (int k = 0; k < 3; k++) {  // S <- J^T * S
          const double spk = S[p][k], sqk = S[q][k];
          S[p][k] = c * spk - sn * sqk; S[q][k] = sn * spk + c * sqk;
        }
      }
  }
  *emin = fmin(S[0][0], fmin(S[1][1], S[2][2]));
  *emax = fmax(S[0][0], fmax(S[1][1], S[2][2]));
}
static float round_down(double x) {  // a float <= x
  float f = (float)x;
  if ((double)f > x) f = nextafterf(f, -INFINITY);
  return nextafterf(f, -INFINITY);
}
static float round_up(double x) {  // smallest-ish float >= x (x >= 0)
  float f = (float)x;
  if ((double)f < x) f = nextafterf(f, INFINITY);
  return nextafterf(f, INFINITY);
}

struct HostFilter {
  std::vector<float4> rows;  // [n_pairs][kFiltRows]
  std::vector<int2> ids;     // per pair: geom index of half A, half B
  int end[kFiltClasses] = {0, 0, 0, 0};
  float r_scene = 0.0f;
  // hierarchy (pt_bvh.cuh); empty when the scene is small enough for the pair scan
  std::vector<float4> nodes, leaves;
  std::vector<int2> leaf_meta;
  int root = 0;  // reference of the hierarchy's root: node 0, or the only leaf
  float ew_c_max = 0.0f, ew_w_max = 0.0f;
  std::vector<FiltGeom> geoms;  // every real geom of the pair scan
};
static const int kBvhMinGeoms = 33;  // scenes with fewer geoms use the linear pair scan (shared memory, packed)
static bool inv3(const double a[3][3], double r[3][3]) {
  const double c00 = a[1][1] * a[2][2] - a[1][2] * a[2][1], c01 = a[1][2] * a[2][0] - a[1][0] * a[2][2],
               c02 = a[1][0] * a[2][1] - a[1][1] * a[2][0];
  const double det = a[0][0] * c00 + a[0][1] * c01 + a[0][2] * c02;
  if (!(fabs(det) > 0) || !std::isfinite(det)) return false;
  const double id = 1.0 / det;
  r[0][0] = c00 * id; r[0][1] = (a[0][2] * a[2][1] - a[0][1] * a[2][2]) * id; r[0][2] = (a[0][1] * a[1][2] - a[0][2] * a[1][1]) * id;
  r[1][0] = c01 * id; r[1][1] = (a[0][0] * a[2][2] - a[0][2] * a[2][0]) * id; r[1][2] = (a[0][2] * a[1][0] - a[0][0] * a[1][2]) * id;
  r[2][0] = c02 * id; r[2][1] = (a[0][1] * a[2][0] - a[0][0] * a[2][1]) * id; r[2][2] = (a[0][0] * a[1][1] - a[0][1] * a[1][0]) * id;
  return true;
}
// Per-geom coefficients of the error model (DESIGN.md "filter").  u = 2^-24 (unit roundoff).  `scale` multiplies
// every rounding-error term (test hook; geometry terms such as the 1e-4 pull-back are not scaled).
static HostFilter build_filter(const pt_static_geom* geoms, int n_geoms, double scale) {
  HostFilter F;
  const double u = ldexp(1.0, -24);
  const double s3 = 1.7320508075688772;
  struct Per {
    int geom, cls;
    double KA[3], T[3];
    float k[8];      // object-space constants (classes 1, 3)
    float c[3];      // world point that inverseTransform maps to the object origin (classes 0, 2)
    float wk[6];     // class 0: Wc, Ww, Wr;  class 2: Hc.xyz, Hw.xyz
    float wd[3];     // the DEFLATED shape's constants at w = 0 (sure-hit bound, pt_bvh.cuh): class 0: Wc'; class 2: Hd.xyz
    float ew_c, ew_w;
    double bc[3], bh[3], p1, p2;  // world AABB (centre, half extents) of the inflated shape at w = 0; pad coefficients
  };
  std::vector<Per> per;
  // pass 1: scene bound
  double r_scene = 0.0;
  std::vector<double> sigM(n_geoms, 0.0);
  for (int i = 0; i < n_geoms; i++) {
    if (geoms[i].type > 1) continue;
    const float* M = geoms[i].transform;
    double MtM[3][3], tm2 = 0.0, lo, hi;
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        MtM[a][b] = 0.0;
        for (int r = 0; r < 3; r++) MtM[a][b] += (double)M[4 * r + a] * M[4 * r + b];
      }
    sym3_eigen_range(MtM, &lo, &hi);
    sigM[i] = sqrt(fmax(hi, 0.0)) * 1.001;
    for (int r = 0; r < 3; r++) tm2 += (double)M[4 * r + 3] * M[4 * r + 3];
    // bound on |p| over the geom's surface: |translation| + sigma_max(M) * (half diagonal of the unit cube)
    r_scene = fmax(r_scene, sqrt(tm2) + sigM[i] * 0.8661);
  }
  F.r_scene = round_up(r_scene * 1.001);
  const double Rs = (double)F.r_scene;
  // pass 2: per-geom constants and class
  for (int i = 0; i < n_geoms; i++) {
    const pt_static_geom& g = geoms[i];
    if (g.type > 1) continue;
    const float* A = g.inverseTransform;
    const float* M = g.transform;
    Per q;
    q.geom = i;
    double A3[3][3], AtA[3][3], Ai[3][3];
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        A3[a][b] = (double)A[4 * a + b];
        AtA[a][b] = 0.0;
        for (int r = 0; r < 3; r++) AtA[a][b] += (double)A[4 * r + a] * A[4 * r + b];
      }
    double lmin, lmax;
    sym3_eigen_range(AtA, &lmin, &lmax);
    const double isigA = lmin > 0 ? 1.001 / sqrt(lmin) : INFINITY;  // 1 / sigma_min(A): bound on |d| / |A d|
    double KM = 0, TM = 0, EMw = 0, EMc = 0, rlin = 0, rt = 0;
    for (int r = 0; r < 3; r++) {
      q.KA[r] = fabs((double)A[4 * r]) + fabs((double)A[4 * r + 1]) + fabs((double)A[4 * r + 2]);
      q.T[r] = fabs((double)A[4 * r + 3]);
    }
    for (int r = 0; r < 3; r++) {
      const double m0 = fabs((double)M[4 * r]), m1 = fabs((double)M[4 * r + 1]), m2 = fabs((double)M[4 * r + 2]);
      KM = fmax(KM, m0 + m1 + m2);
      TM = fmax(TM, fabs((double)M[4 * r + 3]));
      EMw = fmax(EMw, m0 * q.KA[0] + m1 * q.KA[1] + m2 * q.KA[2]);
      EMc = fmax(EMc, m0 * q.T[0] + m1 * q.T[1] + m2 * q.T[2]);
      // residual of transform * inverseTransform - I (both are rounded binary32 matrices)
      double lin = 0.0;
      for (int c = 0; c < 4; c++) {
        double acc = c == 3 ? (double)M[4 * r + 3] : 0.0;
        for (int j = 0; j < 3; j++) acc += (double)M[4 * r + j] * A[4 * j + c];
        if (c < 3) lin += fabs(acc - (c == r ? 1.0 : 0.0)); else rt = fmax(rt, fabs(acc));
      }
      rlin = fmax(rlin, lin);
    }
    const double KAn = sqrt(q.KA[0] * q.KA[0] + q.KA[1] * q.KA[1] + q.KA[2] * q.KA[2]);
    const double Tn = sqrt(q.T[0] * q.T[0] + q.T[1] * q.T[1] + q.T[2] * q.T[2]);
    // world slack: pull-back of 1e-4 object units (NOT scaled: it is geometry, not rounding) + rounding of both
    // paths mapped through the forward transform + residual of M*A - I
    double ew_w = scale * s3 * 2.0 * 2.25 * u * EMw;
    double ew_c = scale * s3 * 2.0 * (9.0 * u * (EMc + 0.5 * KM) + 4.0 * u * (0.51 * KM + TM) + rlin * Rs + rt) + 1.0001e-4 * isigA;
    double objk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (g.type == 0) {
      const double alpha = 6.0 * u * KAn * isigA;
      ew_w += scale * 16.0 * u * isigA * KAn * 0.25;
      ew_c += scale * 16.0 * u * isigA * Tn;
      // R2c, R2w, R2r
      objk[0] = 0.25 + scale * (28.0 * u * Tn + alpha); objk[1] = scale * 7.0 * u * KAn; objk[2] = scale * (64.0 * u + 4.0 * alpha);
      q.k[0] = round_up(objk[0]); q.k[1] = round_up(objk[1]); q.k[2] = round_up(objk[2]);
    } else {
      // hc.xyz, hw.xyz
      for (int r = 0; r < 3; r++) {
        objk[r] = 0.5 + scale * u * (32.0 * q.T[r] + 16.0);
        objk[3 + r] = scale * 13.2 * u * q.KA[r];
        q.k[r] = round_up(objk[r]); q.k[3 + r] = round_up(objk[3 + r]);
      }
    }
    q.ew_c = round_up(ew_c); q.ew_w = round_up(ew_w);
    // ---- world-space classes: c = the world point that A maps to the object origin ----
    q.cls = g.type == 0 ? 1 : 3;
    q.wd[0] = q.wd[1] = q.wd[2] = -INFINITY;  // (never a sure hit)
    if (inv3(A3, Ai)) {
      double cw[3], dc = 0.0;
      for (int r = 0; r < 3; r++) {
        cw[r] = -(Ai[r][0] * A[3] + Ai[r][1] * A[7] + Ai[r][2] * A[11]);
        q.c[r] = (float)cw[r];
        dc = fmax(dc, fabs(cw[r] - (double)q.c[r]) + u * fabs(cw[r]));  // rounding of c to binary32 (+ its use)
      }
      const bool finite = std::isfinite(cw[0]) && std::isfinite(cw[1]) && std::isfinite(cw[2]);
      // world AABB of the inflated shape { x : A (x - c) in inflated unit shape }, split into its value at w = 0 and
      // the pad coefficients of P1*w + P2*D^2 (pt_bvh.cuh)
      q.p1 = q.p2 = 0.0;
      for (int r = 0; r < 3; r++) {
        q.bc[r] = cw[r];
        if (g.type == 1) {
          q.bh[r] = fabs(Ai[r][0]) * objk[0] + fabs(Ai[r][1]) * objk[1] + fabs(Ai[r][2]) * objk[2] + 2.0 * dc;
          q.p1 = fmax(q.p1, fabs(Ai[r][0]) * objk[3] + fabs(Ai[r][1]) * objk[4] + fabs(Ai[r][2]) * objk[5]);
        } else {
          // |x - c|_r <= |row r of A^-1| * sqrt(R2),  sqrt(R2) <= sqrt(R2c) + R2w w + R2r |ro|^2,  |ro|^2 <= lmax D^2
          const double rown = sqrt(Ai[r][0] * Ai[r][0] + Ai[r][1] * Ai[r][1] + Ai[r][2] * Ai[r][2]);
          q.bh[r] = sqrt(objk[0]) * rown * 1.000001 + 2.0 * dc;
          q.p1 = fmax(q.p1, objk[1] * rown);
          q.p2 = fmax(q.p2, objk[2] * lmax * rown * 1.001);
        }
      }
      q.p1 += scale * 16.0 * u;  // rounding of the node slab test itself, in units of w
      if (!finite) { q.bh[0] = q.bh[1] = q.bh[2] = INFINITY; q.bc[0] = q.bc[1] = q.bc[2] = 0.0; }
      if (g.type == 0 && finite && lmin > 0 && (lmax - lmin) <= 1e-5 * lmax) {
        // |A x|^2 >= lmin |x|^2: a line within R_obj of the object origin is within R_obj / sqrt(lmin) of c;
        // |ro|^2 <= lmax |o - c|^2
        const double rad = 0.5 / sqrt(lmin);
        q.wk[0] = round_up(objk[0] / lmin + 4.0 * rad * dc);
        q.wk[1] = round_up(objk[1] / lmin);
        q.wk[2] = round_up(objk[2] * (lmax / lmin) + scale * 32.0 * u);
        // deflated: a world point within r' of c maps to within sqrt(lmax) r' of the object origin
        q.wd[0] = round_down((0.5 - objk[0]) / lmax * (1.0 - 1e-6) - 4.0 * rad * dc);
        q.cls = 0;
      } else if (g.type == 1 && finite) {
        // world AABB of the inflated cube { x : |A (x - c)|_j <= h_j }: half extents sum_j |Ai_ij| h_j
        bool tight = true;
        for (int r = 0; r < 3; r++) {
          double dom = 0.0, sum = 0.0;
          for (int j = 0; j < 3; j++) { dom = fmax(dom, fabs(Ai[r][j])); sum += fabs(Ai[r][j]); }
          if (!((sum - dom) <= 1e-4 * dom)) tight = false;  // the AABB must hug the cube, else near misses fall back
          q.wk[r] = round_up(fabs(Ai[r][0]) * objk[0] + fabs(Ai[r][1]) * objk[1] + fabs(Ai[r][2]) * objk[2] + 2.0 * dc);
          q.wk[3 + r] = round_up(fabs(Ai[r][0]) * objk[3] + fabs(Ai[r][1]) * objk[4] + fabs(Ai[r][2]) * objk[5] + scale * 16.0 * u);
        }
        if (tight) {
          q.cls = 2;
          // deflated: a world AABB {|x_r| <= H'_r} INSIDE the cube deflated to half extents 1 - objk[j]:
          // sum_r |A_jr| H'_r <= 1 - objk[j] for every object axis j (checked, with a growing shrink factor)
          for (double eps = 1e-3; eps < 0.6; eps *= 4.0) {
            double Hd[3];
            bool ok = true;
            for (int r = 0; r < 3; r++) {
              int jd = 0;  // the object axis this world axis runs along
              for (int j = 1; j < 3; j++) if (fabs(Ai[r][j]) > fabs(Ai[r][jd])) jd = j;
              Hd[r] = fabs(Ai[r][jd]) * (1.0 - objk[jd]) * (1.0 - eps) - 2.0 * dc;
              if (!(Hd[r] > 0)) ok = false;
            }
            for (int j = 0; j < 3 && ok; j++)
              if (!(fabs(A3[j][0]) * Hd[0] + fabs(A3[j][1]) * Hd[1] + fabs(A3[j][2]) * Hd[2] <= (1.0 - objk[j]) * (1.0 - 1e-6))) ok = false;
            if (ok) { for (int r = 0; r < 3; r++) q.wd[r] = round_down(Hd[r]); break; }
          }
        }
      }
    }
    else {  // singular inverseTransform: cannot be bounded, always visited
      q.bc[0] = q.bc[1] = q.bc[2] = 0.0; q.bh[0] = q.bh[1] = q.bh[2] = INFINITY; q.p1 = q.p2 = 0.0;
    }
    per.push_back(q);
  }
  // pairs of one class; an odd geom out is paired with a copy of itself that can never be a candidate (-inf bounds)
  const float ninf = -INFINITY;
  for (int cls = 0; cls < kFiltClasses; cls++) {
    std::vector<int> m;
    for (int k = 0; k < (int)per.size(); k++) if (per[k].cls == cls) m.push_back(k);
    for (size_t j = 0; j < m.size(); j += 2) {
      const Per& x = per[m[j]];
      const bool dummy = j + 1 >= m.size();
      Per y = per[dummy ? m[j] : m[j + 1]];
      if (dummy) {  // radius^2 / half extents -inf: discriminant -inf, tnear = +inf > tfar = -inf: proven miss
        if (cls == 0) y.wk[0] = ninf;
        if (cls == 1) y.k[0] = ninf;
        if (cls == 2) y.wk[0] = y.wk[1] = y.wk[2] = ninf;
        if (cls == 3) y.k[0] = y.k[1] = y.k[2] = ninf;
      }
      float4 r[kFiltRows];
      for (int t = 0; t < kFiltRows; t++) r[t] = make_float4(0, 0, 0, 0);
      if (cls == 0) {
        r[0] = make_float4(x.c[0], y.c[0], x.c[1], y.c[1]);
        r[1] = make_float4(x.c[2], y.c[2], x.wk[0], y.wk[0]);
        r[2] = make_float4(x.wk[1], y.wk[1], x.wk[2], y.wk[2]);
        r[3] = make_float4(x.ew_c, y.ew_c, x.ew_w, y.ew_w);
      } else if (cls == 2) {
        r[0] = make_float4(x.c[0], y.c[0], x.c[1], y.c[1]);
        r[1] = make_float4(x.c[2], y.c[2], x.wk[0], y.wk[0]);
        r[2] = make_float4(x.wk[1], y.wk[1], x.wk[2], y.wk[2]);
        r[3] = make_float4(x.wk[3], y.wk[3], x.wk[4], y.wk[4]);
        r[4] = make_float4(x.wk[5], y.wk[5], x.ew_c, y.ew_c);
        r[5] = make_float4(x.ew_w, y.ew_w, 0, 0);
      } else {
        const float* A = geoms[x.geom].inverseTransform;
        const float* B = geoms[y.geom].inverseTransform;
        for (int t = 0; t < 3; t++) {
          r[2 * t] = make_float4(A[4 * t], B[4 * t], A[4 * t + 1], B[4 * t + 1]);
          r[2 * t + 1] = make_float4(A[4 * t + 2], B[4 * t + 2], A[4 * t + 3], B[4 * t + 3]);
        }
        if (cls == 1) {
          r[6] = make_float4(x.k[0], y.k[0], x.k[1], y.k[1]);
          r[7] = make_float4(x.k[2], y.k[2], x.ew_c, y.ew_c);
          r[8] = make_float4(x.ew_w, y.ew_w, 0, 0);
        } else {
          r[6] = make_float4(x.k[0], y.k[0], x.k[1], y.k[1]);
          r[7] = make_float4(x.k[2], y.k[2], x.k[3], y.k[3]);
          r[8] = make_float4(x.k[4], y.k[4], x.k[5], y.k[5]);
          r[9] = make_float4(x.ew_c, y.ew_c, x.ew_w, y.ew_w);
        }
      }
      F.rows.insert(F.rows.end(), r, r + kFiltRows);
      for (int half = 0; half < (dummy ? 1 : 2); half++) {
        const Per& z = half ? y : x;
        FiltGeom e;
        e.key = 2 * (int)F.ids.size() + half; e.cls = cls; e.geom = z.geom;
        memcpy(e.c, z.c, sizeof(e.c)); memcpy(e.k, z.k, sizeof(e.k)); memcpy(e.wk, z.wk, sizeof(e.wk));
        e.ew_c = z.ew_c; e.ew_w = z.ew_w;
        F.geoms.push_back(e);
      }
      F.ids.push_back(make_int2(x.geom, y.geom));
    }
    F.end[cls] = (int)F.ids.size();
  }
  if (F.ids.empty()) { F.rows.assign(kFiltRows, make_float4(0, 0, 0, 0)); F.ids.push_back(make_int2(0, 0)); }

  // ---- hierarchy for scenes with many geoms: surface-area heuristic, one geom per leaf ----
  const int n = (int)per.size();
  if (n >= kBvhMinGeoms) {
    F.leaves.assign((size_t)n * kBvhLeafRows, make_float4(0, 0, 0, 0));
    F.leaf_meta.resize(n);
    for (int k = 0; k < n; k++) {
      const Per& x = per[k];
      float4* L = &F.leaves[(size_t)k * kBvhLeafRows];
      const float* A = geoms[x.geom].inverseTransform;
      if (x.cls == 0) {
        L[0] = make_float4(x.c[0], x.c[1], x.c[2], x.wk[0]);
        L[1] = make_float4(x.wk[1], x.wk[2], x.ew_c, x.ew_w);
        L[2] = make_float4(x.wd[0], 0, 0, 0);
      } else if (x.cls == 2) {
        L[0] = make_float4(x.c[0], x.c[1], x.c[2], x.ew_c);
        L[1] = make_float4(x.wk[0], x.wk[1], x.wk[2], x.ew_w);
        L[2] = make_float4(x.wk[3], x.wk[4], x.wk[5], 0);
        L[3] = make_float4(x.wd[0], x.wd[1], x.wd[2], 0);
      } else {
        for (int t = 0; t < 3; t++) L[t] = make_float4(A[4 * t], A[4 * t + 1], A[4 * t + 2], A[4 * t + 3]);
        if (x.cls == 1) { L[3] = make_float4(x.k[0], x.k[1], x.k[2], x.ew_c); L[4] = make_float4(x.ew_w, 0, 0, 0); }
        else { L[3] = make_float4(x.k[0], x.k[1], x.k[2], x.ew_c); L[4] = make_float4(x.k[3], x.k[4], x.k[5], x.ew_w); }
      }
      F.leaf_meta[k] = make_int2(x.cls, x.geom);
      F.ew_c_max = fmaxf(F.ew_c_max, x.ew_c);
      F.ew_w_max = fmaxf(F.ew_w_max, x.ew_w);
    }
    struct Box { double lo[3], hi[3], p1, p2; };
    auto leaf_box = [&](int k) {
      Box b;
      for (int r = 0; r < 3; r++) { b.lo[r] = per[k].bc[r] - per[k].bh[r]; b.hi[r] = per[k].bc[r] + per[k].bh[r]; }
      b.p1 = per[k].p1; b.p2 = per[k].p2;
      return b;
    };
    auto merge = [](const Box& a, const Box& b) {
      Box m;
      for (int r = 0; r < 3; r++) { m.lo[r] = fmin(a.lo[r], b.lo[r]); m.hi[r] = fmax(a.hi[r], b.hi[r]); }
      m.p1 = fmax(a.p1, b.p1); m.p2 = fmax(a.p2, b.p2);
      return m;
    };
    auto down = [](double x) { float f = (float)x; if ((double)f > x) f = nextafterf(f, -INFINITY); return nextafterf(f, -INFINITY); };
    auto up = [](double x) { float f = (float)x; if ((double)f < x) f = nextafterf(f, INFINITY); return nextafterf(f, INFINITY); };
    auto area = [](const Box& b) {  // half the surface area; +inf for an unbounded box
      const double x = b.hi[0] - b.lo[0], y = b.hi[1] - b.lo[1], z = b.hi[2] - b.lo[2];
      const double a = x * y + y * z + z * x;
      return std::isfinite(a) ? a : INFINITY;
    };
    std::vector<int> idx(n);
    for (int k = 0; k < n; k++) idx[k] = k;
    std::vector<Box> lbox(n);
    for (int k = 0; k < n; k++) lbox[k] = leaf_box(k);
    std::vector<double> suffix(n);
    struct BNode { Box b[2]; int c[2]; };  // the binary tree; collapsed into 4-wide nodes below
    std::vector<BNode> bnodes((size_t)(n > 1 ? n - 1 : 1));
    std::atomic<int> next_node{0};  // (subtrees are built by several host threads: node numbers are handed out atomically)
    // Returns the child reference (node index, or ~leaf) and the box of idx[first, last).  Split rule: the cheapest, by
    // the surface-area heuristic (area x count of each side), of
    //   * the largest geom on its own (a ground slab among pebbles: whatever group it stayed in would inherit its
    //     extent, level after level; a sweep over centroids cannot single it out),
    //   * every split position of the centroids sorted along x, y and z;
    // the median along the widest axis when the levels left are only just enough to finish by halving (the traversal
    // stack need of the collapsed tree is checked below: kBvhStack) or when nothing has a finite cost.
    bool median_only = getenv("PT_B200_BVH_MEDIAN") != nullptr;  // measurement knob: the plain median-split tree
    std::function<int(int, int, int, Box&)> build = [&](int first, int last, int depth, Box& box) -> int {
      const int cnt = last - first;
      if (cnt == 1) { box = lbox[idx[first]]; return ~idx[first]; }
      int levels = 0;
      while ((1 << levels) < cnt) levels++;
      const bool must_halve = depth + levels + 2 >= kBvhBinaryDepth || median_only;
      int mid = -1;
      if (!must_halve && cnt > 2) {
        int big = first;
        for (int i = first + 1; i < last; i++)
          if (area(lbox[idx[i]]) > area(lbox[idx[big]])) big = i;
        std::swap(idx[first], idx[big]);
        Box rest = lbox[idx[first + 1]];
        for (int i = first + 2; i < last; i++) rest = merge(rest, lbox[idx[i]]);
        double best_cost = area(lbox[idx[first]]) + area(rest) * (cnt - 1);  // the largest geom on its own
        int best_axis = -1, best_mid = first + 1;
        if (std::isfinite(area(lbox[idx[first]]))) {
          for (int axis = 0; axis < 3; axis++) {
            std::sort(idx.begin() + first, idx.begin() + last, [&](int a, int b) { return per[a].bc[axis] < per[b].bc[axis]; });
            Box acc = lbox[idx[last - 1]];
            suffix[last - 1] = area(acc);
            for (int i = last - 2; i > first; i--) { acc = merge(acc, lbox[idx[i]]); suffix[i] = area(acc); }
            acc = lbox[idx[first]];
            for (int i = first + 1; i < last; i++) {  // left = [first, i), right = [i, last)
              const double cost = area(acc) * (i - first) + suffix[i] * (last - i);
              if (cost < best_cost) { best_cost = cost; best_axis = axis; best_mid = i; }
              acc = merge(acc, lbox[idx[i]]);
            }
          }
        }
        if (best_axis >= 0) {
          if (best_axis != 2)
            std::sort(idx.begin() + first, idx.begin() + last, [&](int a, int b) { return per[a].bc[best_axis] < per[b].bc[best_axis]; });
          mid = best_mid;
        } else if (std::isfinite(best_cost) || !std::isfinite(area(lbox[idx[big]]))) {
          // (the sorts moved the largest geom: bring it back to the front)
          big = first;
          for (int i = first + 1; i < last; i++)
            if (area(lbox[idx[i]]) > area(lbox[idx[big]])) big = i;
          std::swap(idx[first], idx[big]);
          mid = first + 1;
        }
      }
      if (mid < 0) {
        double clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (int i = first; i < last; i++)
          for (int r = 0; r < 3; r++) { clo[r] = fmin(clo[r], per[idx[i]].bc[r]); chi[r] = fmax(chi[r], per[idx[i]].bc[r]); }
        int axis = 0;
        if (chi[1] - clo[1] > chi[axis] - clo[axis]) axis = 1;
        if (chi[2] - clo[2] > chi[axis] - clo[axis]) axis = 2;
        mid = first + cnt / 2;
        std::nth_element(idx.begin() + first, idx.begin() + mid, idx.begin() + last,
                         [&](int a, int b) { return per[a].bc[axis] < per[b].bc[axis]; });
      }
      const int me = next_node++;
      Box b0, b1;
      int c0, c1;
      if (depth < 3 && cnt >= 2048) {  // the two halves are independent (disjoint ranges of idx / suffix): up to 8 threads
        std::thread left([&] { c0 = build(first, mid, depth + 1, b0); });
        c1 = build(mid, last, depth + 1, b1);
        left.join();
      } else {
        c0 = build(first, mid, depth + 1, b0);
        c1 = build(mid, last, depth + 1, b1);
      }
      bnodes[me].b[0] = b0; bnodes[me].b[1] = b1; bnodes[me].c[0] = c0; bnodes[me].c[1] = c1;
      box = merge(b0, b1);
      return me;
    };
    Box root;
    for (int attempt = 0; attempt < 2; attempt++) {
      next_node = 0;
      for (int k = 0; k < n; k++) idx[k] = k;
      const int root_ref = build(0, n, 0, root);
      // ---- collapse into 4-wide nodes: a node's slots start as its two children; while there is room, the inner slot
      // with the largest box is replaced by its own two children.  One fetch then serves up to four boxes, and the chain
      // of dependent fetches of a traversal is about half as long. ----
      F.nodes.clear();
      int stack_need = 0;
      std::function<int(int, int&)> collapse = [&](int b, int& need) -> int {
        int ref[4], cnt = 2;
        Box bx[4];
        bx[0] = bnodes[b].b[0]; bx[1] = bnodes[b].b[1]; ref[0] = bnodes[b].c[0]; ref[1] = bnodes[b].c[1];
        while (cnt < 4) {
          int pick = -1;
          for (int i = 0; i < cnt; i++)
            if (ref[i] >= 0 && (pick < 0 || area(bx[i]) > area(bx[pick]))) pick = i;
          if (pick < 0) break;
          const BNode& q = bnodes[ref[pick]];
          bx[pick] = q.b[0]; ref[pick] = q.c[0];
          bx[cnt] = q.b[1]; ref[cnt] = q.c[1];
          cnt++;
        }
        const int me = (int)(F.nodes.size() / kBvhNodeRows);
        F.nodes.resize(F.nodes.size() + kBvhNodeRows, make_float4(0, 0, 0, 0));
        int child[4], deepest = 0;
        for (int i = 0; i < 4; i++) {
          child[i] = kBvhNoChild;
          if (i < cnt) {
            int sub = 0;
            // (a leaf's reference carries its filter class, so that a traversal fetches the leaf's record without
            // waiting for its meta word: one dependent fetch less per leaf)
            child[i] = ref[i] >= 0 ? collapse(ref[i], sub) : bvh_leaf_ref(~ref[i], per[~ref[i]].cls);
            deepest = std::max(deepest, sub);
          }
        }
        need = (cnt - 1) + deepest;  // the children not taken wait on the stack while the deepest one is walked
        float4* N = &F.nodes[(size_t)me * kBvhNodeRows];
        const float pinf = INFINITY, ninf = -INFINITY;
        float cf[4];
        memcpy(cf, child, sizeof(cf));
        float p1n = 0.0f, p2n = 0.0f;  // (128-byte nodes: the pads of the node = the largest of its children's)
        for (int i = 0; i < cnt; i++) { p1n = fmaxf(p1n, up(bx[i].p1)); p2n = fmaxf(p2n, up(bx[i].p2 * 1.000002)); }
        for (int h = 0; h < 2; h++) {  // two blocks in the layout child_entries reads: children (0, 1) and (2, 3)
          const int i0 = 2 * h, i1 = 2 * h + 1;
          auto lo = [&](int i, int r) { return i < cnt ? down(bx[i].lo[r]) : pinf; };  // an empty slot: a box nothing enters
          auto hi = [&](int i, int r) { return i < cnt ? up(bx[i].hi[r]) : ninf; };
          auto p1 = [&](int i) { return i < cnt ? up(bx[i].p1) : 0.0f; };
          auto p2 = [&](int i) { return i < cnt ? up(bx[i].p2 * 1.000002) : 0.0f; };  // x 1.000002: rounding of D^2 in child_entries
          float4* Nh = N + (PT_BVH_NODE128 ? 3 : 4) * h;
          Nh[0] = make_float4(lo(i0, 0), lo(i1, 0), lo(i0, 1), lo(i1, 1));
          Nh[1] = make_float4(lo(i0, 2), lo(i1, 2), hi(i0, 0), hi(i1, 0));
          Nh[2] = make_float4(hi(i0, 1), hi(i1, 1), hi(i0, 2), hi(i1, 2));
          if (!PT_BVH_NODE128) Nh[3] = make_float4(p1(i0), p1(i1), p2(i0), p2(i1));
        }
        if (PT_BVH_NODE128) {
          N[6] = make_float4(cf[0], cf[1], cf[2], cf[3]);
          N[7] = make_float4(p1n, p2n, 0.0f, 0.0f);
        } else {
          N[8] = make_float4(cf[0], cf[1], cf[2], cf[3]);
        }
        return me;
      };
      F.root = root_ref >= 0 ? 0 : bvh_leaf_ref(~root_ref, per[~root_ref].cls);
      if (root_ref >= 0) collapse(root_ref, stack_need);
      if (getenv("PT_B200_BVH_DEBUG"))
        fprintf(stderr, "pt_b200 bvh: %d leaves, %d binary nodes, %zu wide nodes, stack need %d of %d%s\n", n, next_node.load(),
                F.nodes.size() / kBvhNodeRows, stack_need, kBvhStack, median_only ? " (median splits)" : "");
      if (stack_need + 2 <= kBvhStack || median_only) break;
      median_only = true;  // a degenerate tree: the balanced one needs 3 entries per two binary levels at most
    }
  }
  return F;
}

// host-side camera constants (DESIGN.md "raygen"): binary32, unfused, in this exact order -- the parity tests compare bits
static f3 h_mk(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
static f3 h_normalize(f3 v) {
  float sqr = (v.x * v.x + v.y * v.y) + v.z * v.z;
  float inv = 1.0f / sqrtf(sqr);
  return h_mk(v.x * inv, v.y * inv, v.z * inv);
}
static f3 h_cross(f3 x, f3 y) { return h_mk(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y); }
static RaygenConsts make_raygen(const pt_camera_data& c, const pt_lens* lens) {
  RaygenConsts R;
  R.eye = h_mk(c.position[0], c.position[1], c.position[2]);
  R.w = h_normalize(h_mk(c.view[0], c.view[1], c.view[2]));
  R.right = h_normalize(h_cross(R.w, h_mk(c.up[0], c.up[1], c.up[2])));
  R.vup = h_cross(R.right, R.w);
  float tx = tanf(c.fov[0] * 0.017453292f);
  float ty = tanf(c.fov[1] * 0.017453292f);
  R.Hh = h_mk(R.right.x * tx, R.right.y * tx, R.right.z * tx);
  R.Vv = h_mk(R.vup.x * ty, R.vup.y * ty, R.vup.z * ty);
  R.fw = c.resolution[0];
  R.fh = c.resolution[1];
  R.W = (uint32_t)(int)c.resolution[0];
  R.npix = R.W * (uint32_t)(int)c.resolution[1];
  R.divW = make_fastdiv(R.W);
  R.aperture = lens ? lens->aperture : 0.0f;
  R.focal = lens ? lens->focal_distance : 0.0f;
  return R;
}

// The features the bounce kernels of segment kind (first, last) are instantiated with; a launch runs a subset of them.
//   direct light sampling: unless first and last -- the last segment never samples a light, but it honours the
//     no-emission flag, and a first-and-last segment cannot carry that flag either
//   subsurface scattering: unless last -- a scattering event there ends the path exactly as the refraction it replaces
//     does (neither adds radiance, and no later depth counts the path), so image and live counts are those of the plain
//     kernel
//   glossy reflection: unless last, for the same reason -- the last segment stores no direction, so the direction a
//     glossy event samples there is never used
//   Russian roulette: unless first, whose throughput is 1, or last, which continues nowhere (DESIGN.md 4)
constexpr uint32_t variants_of(bool first, bool last) {
  return (first && last ? 0u : kFxNee) | (last ? 0u : kFxMedium | kFxGlossy) | (first || last ? 0u : kFxRoulette);
}

// The kernel tables: kBounceKernels[first][last][FX] holds the bounce kernels of that segment kind and feature set, null
// where FX is not a subset of variants_of(first, last) -- no such kernel is instantiated.  (k_bounce_q and k_bounce_bvh
// take no FIRST: the kinds (true, L) and (false, L) share their instantiations.)
using BounceKernel = void (*)(BounceParams);
struct BounceKernels {
  BounceKernel fused, queued, bvh;  // k_bounce, k_bounce_q, k_bounce_bvh
};
template <bool F, bool L, uint32_t FX>
constexpr BounceKernels bounce_kernels() {
  if constexpr ((FX & ~variants_of(F, L)) != 0) return {nullptr, nullptr, nullptr};
  else return {k_bounce<F, L, FX>, k_bounce_q<L, FX>, k_bounce_bvh<L, FX>};
}
template <bool F, bool L, uint32_t... FX>
constexpr std::array<BounceKernels, kFxSets> kernel_table(std::integer_sequence<uint32_t, FX...>) {
  return {{bounce_kernels<F, L, FX>()...}};
}
using EveryFx = std::make_integer_sequence<uint32_t, kFxSets>;
static const std::array<BounceKernels, kFxSets> kBounceKernels[2][2] = {
    {kernel_table<false, false>(EveryFx{}), kernel_table<false, true>(EveryFx{})},
    {kernel_table<true, false>(EveryFx{}), kernel_table<true, true>(EveryFx{})}};

// the persistent grid of one bounce kernel with `smem` bytes of dynamic shared memory: resident CTAs on the whole
// device, 0 for a null table entry
static int fit_grid(pt_context* c, BounceKernel kernel, int threads, size_t smem, bool carveout, const char* name, int* grid) {
  *grid = 0;
  if (!kernel) return PT_OK;
  int per_sm = 0;
  CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (carveout) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  if (per_sm < 1) { pt_set_error_("%s does not fit on an SM", name); return PT_ERR_CUDA; }
  *grid = per_sm * c->sm_count;
  return PT_OK;
}

// ---- direct light sampling: the light table (DESIGN.md "direct light sampling"; same binary32 expressions, in the same
// order, as getRadiuses / getRandomPointOnCube, src/intersections.h:120-129,140-147) ----
static float h_length3(float x, float y, float z) { return sqrtf((x * x + y * y) + z * z); }
static void h_mulMV(const float* m, float vx, float vy, float vz, float vw, float out[3]) {
  for (int r = 0; r < 3; r++) out[r] = (m[4 * r] * vx) + (m[4 * r + 1] * vy) + (m[4 * r + 2] * vz) + (m[4 * r + 3] * vw);
}
static void h_radiuses(const pt_static_geom& g, float r[3]) {
  float o[3], x[3], y[3], z[3];
  h_mulMV(g.transform, 0, 0, 0, 1, o);
  h_mulMV(g.transform, .5f, 0, 0, 1, x);
  h_mulMV(g.transform, 0, .5f, 0, 1, y);
  h_mulMV(g.transform, 0, 0, .5f, 1, z);
  r[0] = h_length3(x[0] - o[0], x[1] - o[1], x[2] - o[2]);
  r[1] = h_length3(y[0] - o[0], y[1] - o[1], y[2] - o[2]);
  r[2] = h_length3(z[0] - o[0], z[1] - o[1], z[2] - o[2]);
}
static std::vector<float4> build_lights(const pt_static_geom* geoms, int n_geoms, const pt_material* mats, std::vector<float>* geom_k) {
  std::vector<float4> T;
  geom_k->assign((size_t)n_geoms, 0.0f);
  std::vector<float> area;
  std::vector<int> ids;
  for (int i = 0; i < n_geoms; i++) {
    const pt_static_geom& g = geoms[i];
    if (g.type != 0 && g.type != 1) continue;
    if (!(mats[g.materialid].emittance > 0)) continue;
    float r[3], th[5] = {0, 0, 0, 0, 0}, a;
    h_radiuses(g, r);
    if (g.type == 1) {
      const float side1 = r[0] * r[1] * 4.0f;
      const float side2 = r[2] * r[1] * 4.0f;
      const float side3 = r[0] * r[2] * 4.0f;
      const float totalarea = 2.0f * (side1 + side2 + side3);
      th[0] = (side1 / totalarea);
      th[1] = ((side1 * 2) / totalarea);
      th[2] = (((side1 * 2) + (side2)) / totalarea);
      th[3] = (((side1 * 2) + (side2 * 2)) / totalarea);
      th[4] = (((side1 * 2) + (side2 * 2) + (side3)) / totalarea);
      a = totalarea;
    } else {
      a = 4.1887903f * ((r[0] * r[1] + r[1] * r[2]) + r[0] * r[2]);  // 4 pi / 3 * (...): 4 pi r^2 for a uniform scale
    }
    int gi = i, ty = g.type;
    float gf, tf;
    memcpy(&gf, &gi, 4); memcpy(&tf, &ty, 4);
    T.push_back(make_float4(0, 0, 0, gf));
    T.push_back(make_float4(th[0], th[1], th[2], th[3]));
    T.push_back(make_float4(th[4], tf, 0, 0));
    area.push_back(a);
    ids.push_back(i);
  }
  const int n = (int)ids.size();
  for (int k = 0; k < n; k++) {
    const pt_material& m = mats[geoms[ids[k]].materialid];
    const float kk = (area[k] * (float)n) * 0.31830987f;  // area * lights / pi = K of the balance heuristic
    T[3 * k + 2].z = kk;
    (*geom_k)[ids[k]] = kk;
    T[3 * k].x = (m.color[0] * m.emittance) * kk;
    T[3 * k].y = (m.color[1] * m.emittance) * kk;
    T[3 * k].z = (m.color[2] * m.emittance) * kk;
  }
  return T;
}

static int upload_filter(pt_context* c) {
  const HostFilter F = build_filter(c->h_geoms.data(), (int)c->h_geoms.size(), (double)c->filter_scale);
  if (F.end[3] != c->filt.end[3] || !c->d_filt) {
    if (c->d_filt) CU(cudaFree(c->d_filt));
    if (c->d_filt_ids) CU(cudaFree(c->d_filt_ids));
    c->d_filt = nullptr; c->d_filt_ids = nullptr;
    CU(cudaMalloc(&c->d_filt, F.rows.size() * sizeof(float4)));
    CU(cudaMalloc(&c->d_filt_ids, F.ids.size() * sizeof(int2)));
  }
  CU(cudaMemcpyAsync(c->d_filt, F.rows.data(), F.rows.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_filt_ids, F.ids.data(), F.ids.size() * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));  // F dies at return
  c->filt.rows = c->d_filt;
  c->filt.ids = c->d_filt_ids;
  for (int k = 0; k < kFiltClasses; k++) c->filt.end[k] = F.end[k];
  c->filt.r_scene = F.r_scene;
  c->filt_geoms = F.geoms;
  // hierarchy
  if (c->d_bvh_nodes) CU(cudaFree(c->d_bvh_nodes));
  if (c->d_bvh_leaves) CU(cudaFree(c->d_bvh_leaves));
  if (c->d_bvh_meta) CU(cudaFree(c->d_bvh_meta));
  c->d_bvh_nodes = nullptr; c->d_bvh_leaves = nullptr; c->d_bvh_meta = nullptr;
  c->bvh = BvhSoA{};
  if (!F.leaf_meta.empty()) {
    CU(cudaMalloc(&c->d_bvh_nodes, F.nodes.size() * sizeof(float4)));
    CU(cudaMalloc(&c->d_bvh_leaves, F.leaves.size() * sizeof(float4)));
    CU(cudaMalloc(&c->d_bvh_meta, F.leaf_meta.size() * sizeof(int2)));
    CU(cudaMemcpy(c->d_bvh_nodes, F.nodes.data(), F.nodes.size() * sizeof(float4), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_bvh_leaves, F.leaves.data(), F.leaves.size() * sizeof(float4), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_bvh_meta, F.leaf_meta.data(), F.leaf_meta.size() * sizeof(int2), cudaMemcpyHostToDevice));
    c->bvh.nodes = c->d_bvh_nodes; c->bvh.leaves = c->d_bvh_leaves; c->bvh.leaf_meta = c->d_bvh_meta;
    c->bvh.n_leaves = (int)F.leaf_meta.size(); c->bvh.ew_c_max = F.ew_c_max; c->bvh.ew_w_max = F.ew_w_max;
    c->bvh.root = F.root;
  }
  return PT_OK;
}

// The primary-ray table (pt_kernels.cuh: k_primary_table, DESIGN.md 3a "primary rays"), for pinhole cameras of
// pair-scan scenes: one record per filter shape at the eye, in binary64, from the binary32 constants the filter itself
// uses (each term rounded up), then one device thread per pixel.  Anything that cannot be bounded leaves the table off:
// depth 0 then runs the filter scan for every ray, exactly as without a table.
static int build_primary_table(pt_context* c) {
  c->ptab_on = false;
  if (c->mode != 0 || c->cam.aperture > 0.0f || c->filt_geoms.empty() || c->filt_geoms.size() > (size_t)kMaxPrimRecs) return PT_OK;
  const double up = 1.0 + 1e-6;
  const double o[3] = {c->cam.eye.x, c->cam.eye.y, c->cam.eye.z};
  const double omax = fmax(fmax(fabs(o[0]), fabs(o[1])), fabs(o[2]));
  const double w = (4.0 * omax + (double)c->filt.r_scene) * up;  // (make_scan_ray's w, rounding included)
  std::vector<PrimRec> recs;
  for (const FiltGeom& e : c->filt_geoms) {
    if (e.key >= (int)kKeyMask) return PT_OK;
    PrimRec r;
    memset(&r, 0, sizeof(r));
    r.ball = e.cls <= 1;
    r.key = e.key;
    double ctr[3], half[3];  // world box around the shape: centre, half extents
    if (e.cls == 0 || e.cls == 2) {  // world space: the frame is the world translated to the centre
      double oc2 = 0.0;
      for (int i = 0; i < 3; i++) {
        r.A[4 * i] = 1.0;
        ctr[i] = e.c[i];
        r.ro[i] = o[i] - ctr[i];
        r.g[i] = 1.0;
        oc2 += r.ro[i] * r.ro[i];
      }
      if (e.cls == 0) {
        r.h[0] = sqrt(((double)e.wk[0] + (double)e.wk[1] * w + (double)e.wk[2] * oc2) * up);
        for (int i = 0; i < 3; i++) half[i] = r.h[0];
      } else {
        for (int i = 0; i < 3; i++) half[i] = r.h[i] = ((double)e.wk[i] + (double)e.wk[3 + i] * w) * up;
      }
    } else {  // object space
      const float* A = c->h_geoms[e.geom].inverseTransform;
      double A3[3][3], Ai[3][3], AtA[3][3], ro2 = 0.0;
      for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) { A3[i][j] = A[4 * i + j]; r.A[3 * i + j] = A3[i][j]; }
        r.ro[i] = (double)A[4 * i] * o[0] + (double)A[4 * i + 1] * o[1] + (double)A[4 * i + 2] * o[2] + (double)A[4 * i + 3];
        ro2 += r.ro[i] * r.ro[i];
      }
      if (!inv3(A3, Ai)) return PT_OK;
      for (int i = 0; i < 3; i++) ctr[i] = -(Ai[i][0] * A[3] + Ai[i][1] * A[7] + Ai[i][2] * A[11]);
      if (e.cls == 1) {
        for (int a = 0; a < 3; a++)
          for (int b = 0; b < 3; b++) { AtA[a][b] = 0.0; for (int k = 0; k < 3; k++) AtA[a][b] += A3[k][a] * A3[k][b]; }
        double lmin, lmax;
        sym3_eigen_range(AtA, &lmin, &lmax);
        r.h[0] = sqrt(((double)e.k[0] + (double)e.k[1] * w + (double)e.k[2] * ro2) * up);
        r.g[0] = sqrt(fmax(lmax, 0.0)) * 1.001;  // sigma_max(A): a world ball of radius rho fits in an object ball of g rho
        for (int i = 0; i < 3; i++) half[i] = r.h[0] * sqrt(Ai[i][0] * Ai[i][0] + Ai[i][1] * Ai[i][1] + Ai[i][2] * Ai[i][2]) * 1.001;
      } else {
        for (int i = 0; i < 3; i++) {
          r.h[i] = ((double)e.k[i] + (double)e.k[3 + i] * w) * up;
          r.g[i] = sqrt(A3[i][0] * A3[i][0] + A3[i][1] * A3[i][1] + A3[i][2] * A3[i][2]) * 1.001;  // |row i of A|
        }
        for (int i = 0; i < 3; i++) half[i] = (fabs(Ai[i][0]) * r.h[0] + fabs(Ai[i][1]) * r.h[1] + fabs(Ai[i][2]) * r.h[2]) * 1.001;
      }
    }
    double D2 = 0.0;
    for (int i = 0; i < 3; i++) { const double q = fabs(o[i] - ctr[i]) + half[i]; D2 += q * q; }
    r.D = sqrt(D2) * 1.001;
    r.ew = ((double)e.ew_c + (double)e.ew_w * w) * up;
    bool finite = std::isfinite(r.D) && std::isfinite(r.ew);
    for (int i = 0; i < 3; i++) finite = finite && std::isfinite(r.ro[i]) && std::isfinite(r.h[i]) && std::isfinite(r.g[i]);
    if (!finite) return PT_OK;
    recs.push_back(r);
  }
  if (!c->d_ptab) CU(cudaMalloc(&c->d_ptab, (size_t)c->npix * sizeof(uint32_t)));
  if (!c->d_prim) CU(cudaMalloc(&c->d_prim, (size_t)kMaxPrimRecs * sizeof(PrimRec)));
  CU(cudaMemcpyAsync(c->d_prim, recs.data(), recs.size() * sizeof(PrimRec), cudaMemcpyHostToDevice, c->stream));
  k_primary_table<<<(c->npix + 127) / 128, 128, 0, c->stream>>>(c->cam, c->d_prim, (int)recs.size(), (double)c->filter_scale, c->d_ptab);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(c->stream));  // recs dies at return
  c->ptab_on = true;
  return PT_OK;
}

static int upload_scene(pt_context* c, const pt_static_geom* geoms, int n_geoms, const pt_material* mats, int n_mats,
                        const pt_camera_data* cam, const pt_lens* lens, bool first) {
  if (!geoms || n_geoms <= 0 || !mats || n_mats <= 0 || !cam) {
    pt_set_error_("geoms, materials and camera are required and must be non-empty");
    return PT_ERR_INVALID;
  }
  const int Wi = (int)cam->resolution[0], Hi = (int)cam->resolution[1];
  if (Wi <= 0 || Hi <= 0 || (uint64_t)Wi * (uint64_t)Hi > (1ull << 31)) {
    pt_set_error_("bad resolution %d x %d", Wi, Hi);
    return PT_ERR_INVALID;
  }
  if (!first && ((uint32_t)Wi != c->W || (uint32_t)Hi != c->H)) {
    pt_set_error_("pt_update_scene cannot change the resolution (%ux%u -> %dx%d)", c->W, c->H, Wi, Hi);
    return PT_ERR_INVALID;
  }
  for (int i = 0; i < n_geoms; i++) {
    if (geoms[i].type <= 1 && (geoms[i].materialid < 0 || geoms[i].materialid >= n_mats)) {
      pt_set_error_("object %d references material %d, but there are %d materials", i, geoms[i].materialid, n_mats);
      return PT_ERR_INVALID;
    }
  }
  // array of structures (172-byte staticGeom) -> structure of arrays of float4 rows
  std::vector<float4> rows((size_t)6 * n_geoms);
  std::vector<int2> meta(n_geoms);
  for (int i = 0; i < n_geoms; i++) {
    const float* inv = geoms[i].inverseTransform;
    const float* fwd = geoms[i].transform;
    for (int r = 0; r < 3; r++) {
      rows[(size_t)r * n_geoms + i] = make_float4(inv[4 * r], inv[4 * r + 1], inv[4 * r + 2], inv[4 * r + 3]);
      rows[(size_t)(3 + r) * n_geoms + i] = make_float4(fwd[4 * r], fwd[4 * r + 1], fwd[4 * r + 2], fwd[4 * r + 3]);
    }
    meta[i] = make_int2(geoms[i].type, geoms[i].type <= 1 ? geoms[i].materialid : 0);
  }
  c->h_geoms.assign(geoms, geoms + n_geoms);
  if (c->h_policy) {  // a new scene: its survival is unknown (wavefronts of the old one have finished: callers synchronise)
    for (int i = 0; i <= kMaxDepth; i++) ((volatile int*)c->h_policy)[i] = 0;
  }
  int rcf;
  if ((rcf = upload_filter(c))) return rcf;
  if (n_geoms != c->n_geoms) {
    if (c->d_rows) CU(cudaFree(c->d_rows));
    if (c->d_meta) CU(cudaFree(c->d_meta));
    if (c->d_normals) CU(cudaFree(c->d_normals));
    c->d_rows = nullptr; c->d_meta = nullptr; c->d_normals = nullptr;
    CU(cudaMalloc(&c->d_rows, rows.size() * sizeof(float4)));
    CU(cudaMalloc(&c->d_meta, meta.size() * sizeof(int2)));
    CU(cudaMalloc(&c->d_normals, (size_t)n_geoms * kNormalRows * sizeof(float4)));
  }
  if (n_mats != c->n_mats) {
    if (c->d_mats) CU(cudaFree(c->d_mats));
    c->d_mats = nullptr;
    CU(cudaMalloc(&c->d_mats, (size_t)n_mats * sizeof(pt_material)));
  }
  CU(cudaMemcpyAsync(c->d_rows, rows.data(), rows.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_meta, meta.data(), meta.size() * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_mats, mats, (size_t)n_mats * sizeof(pt_material), cudaMemcpyHostToDevice, c->stream));
  c->n_media = 0;
  c->n_glossy = 0;
  for (int i = 0; i < n_geoms; i++) {
    if (geoms[i].type > 1) continue;
    const pt_material& mm = mats[geoms[i].materialid];
    if (mm.hasRefractive > 0 && mm.hasScatter > 0 && mm.reducedScatterCoefficient > 0) c->n_media++;
    if (!(mm.emittance > 0) && !(mm.hasRefractive > 0) && mm.hasReflective > 0 && mm.specularExponent > 0) c->n_glossy++;
  }
  std::vector<float> geom_k;
  const std::vector<float4> lights = build_lights(geoms, n_geoms, mats, &geom_k);
  if (c->d_light_k) CU(cudaFree(c->d_light_k));
  c->d_light_k = nullptr;
  CU(cudaMalloc(&c->d_light_k, (size_t)n_geoms * sizeof(float)));
  CU(cudaMemcpyAsync(c->d_light_k, geom_k.data(), (size_t)n_geoms * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  if (c->d_lights) CU(cudaFree(c->d_lights));
  c->d_lights = nullptr;
  c->n_lights = (int)(lights.size() / 3);
  if (c->n_lights > 0) {
    CU(cudaMalloc(&c->d_lights, lights.size() * sizeof(float4)));
    CU(cudaMemcpyAsync(c->d_lights, lights.data(), lights.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));  // the host vectors die at return
  c->n_geoms = n_geoms;
  c->n_mats = n_mats;
  c->g.inv0 = c->d_rows; c->g.inv1 = c->d_rows + n_geoms; c->g.inv2 = c->d_rows + 2 * (size_t)n_geoms;
  c->g.fwd0 = c->d_rows + 3 * (size_t)n_geoms; c->g.fwd1 = c->d_rows + 4 * (size_t)n_geoms;
  c->g.fwd2 = c->d_rows + 5 * (size_t)n_geoms;
  c->g.meta = c->d_meta;
  k_normal_table<<<(n_geoms + 127) / 128, 128, 0, c->stream>>>(c->g, n_geoms, reinterpret_cast<const float4*>(c->d_mats), c->d_normals);
  CU(cudaGetLastError());
  c->cam = make_raygen(*cam, lens);
  c->W = (uint32_t)Wi; c->H = (uint32_t)Hi; c->npix = c->W * c->H;
  const int cap = c->filt.end[3] < 1 ? 1 : (c->filt.end[3] < kMaxSmemPairs ? c->filt.end[3] : kMaxSmemPairs);
  const int mode = c->bvh.n_leaves > 0 ? 1 : 0;  // fewer than kBvhMinGeoms geoms always fit: at most 16 pairs per class
  if (cap != c->filt_cap || mode != c->mode) {
    c->filt_cap = cap;
    c->geom_smem = filt_smem_bytes(cap);
    c->mode = mode;
    c->smem_bytes = mode == 0 ? c->geom_smem : kBvhSmemBytes;  // k_bounce: filter geometry; k_bounce_bvh: pool results, retry list, stacks
    if (mode == 0) c->q_smem_total = c->geom_smem + q_smem_bytes();
    for (int f = 0; f < 2; f++)
      for (int l = 0; l < 2; l++)
        for (uint32_t fx = 0; fx < kFxSets; fx++) {
          const BounceKernels& k = kBounceKernels[f][l][fx];
          // (many geoms: one kernel for every depth, primary rays come from k_raygen_wf)
          int rc = mode ? fit_grid(c, k.bvh, kBvhThreads, kBvhSmemBytes, false, "k_bounce", &c->grid_blocks[f][l][fx])
                        : fit_grid(c, k.fused, kBounceThreads, c->smem_bytes, false, "k_bounce", &c->grid_blocks[f][l][fx]);
          if (!rc && mode == 0 && !f) rc = fit_grid(c, k.queued, kQThreads, c->q_smem_total, true, "k_bounce_q", &c->grid_blocks_q[l][fx]);
          if (rc) return rc;
        }
    CU(cudaFuncSetAttribute(k_intersect_list, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->geom_smem));
    CU(cudaFuncSetAttribute(k_primary_list, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->geom_smem));
  }
  return build_primary_table(c);
}

// bytes of one wavefront slot: two ping-pong buffers of three float4 arrays, and the hierarchy kernel's per-path results
// (two candidate leaves and two bounds: k_bounce_bvh keeps them in HBM so that a warp's pool of rays can be as long as it likes)
static size_t state_bytes(uint64_t cap) { return (((size_t)cap * (7 * sizeof(float4))) + 255) & ~(size_t)255; }
static int alloc_wavefront(pt_context* c, uint64_t max_paths) {
  uint64_t spp = max_paths / c->npix;
  if (spp < 1) spp = 1;
  const uint64_t cap = spp * c->npix;
  if (cap > 0xFFFFFF00ull) { pt_set_error_("wavefront of %llu paths exceeds 2^32", (unsigned long long)cap); return PT_ERR_INVALID; }
  if (cap == c->wf_capacity) return PT_OK;
  // ... as long as the accumulation image leaves room in the 126 MB L2 for two wavefronts' streams: at 3840x2160 (133 MB
  // of float4 sums) a second concurrent sweep over the image costs more in missed RED atomics than the overlap gains
  int n_slots = pt_context::kSlots;  // (frames larger than that are rendered band by band, pt_render, so the rule below holds again)
  if (const char* env = getenv("PT_B200_SLOTS")) n_slots = atoi(env) >= 2 ? pt_context::kSlots : 1;  // developer knob
  // the internal streams exist only when they are used
  if (n_slots > 1 && !c->wf_stream[0]) {
    CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < pt_context::kSlots; i++) {
      CU(cudaStreamCreateWithFlags(&c->wf_stream[i], cudaStreamNonBlocking));
      CU(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
    }
  }
  // the old buffers go first (the two together may not fit), but a failed allocation must not leave the context
  // without any: fall back to the previous capacity, and report the error
  const uint64_t old_cap = c->wf_capacity;
  const int old_slots = c->n_slots;
  if (c->d_state) CU(cudaFree(c->d_state));
  c->d_state = nullptr; c->wf_capacity = 0;
  if (cudaMalloc(&c->d_state, (size_t)n_slots * state_bytes(cap)) != cudaSuccess) {
    const cudaError_t e = cudaGetLastError();
    c->d_state = nullptr;
    if (old_cap && cudaMalloc(&c->d_state, (size_t)old_slots * state_bytes(old_cap)) == cudaSuccess) {
      c->wf_capacity = old_cap; c->n_slots = old_slots;
    } else {
      cudaGetLastError();
      c->d_state = nullptr;  // pt_render refuses to run until pt_set_wavefront_paths succeeds
    }
    pt_set_error_("cudaMalloc of %llu wavefront paths failed: %s", (unsigned long long)cap, cudaGetErrorString(e));
    return PT_ERR_CUDA;
  }
  c->n_slots = n_slots;
  c->wf_capacity = cap;
  return PT_OK;
}

extern "C" int pt_context_destroy(pt_context* c) {
  if (!c) return PT_OK;
  cudaSetDevice(c->device);
  // every stream that may still carry work of this context (samples traced ahead, the running mean on its way out)
  cudaStream_t streams[] = {c->stream, c->ahead_stream, c->copy_stream, c->wf_stream[0], c->wf_stream[1], c->own_stream};
  for (cudaStream_t st : streams)
    if (st) cudaStreamSynchronize(st);
  const bool dbg = getenv("PT_B200_DEBUG_DESTROY") != nullptr;
  auto chk = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && dbg) fprintf(stderr, "pt_context_destroy: %s -> %s\n", what, cudaGetErrorString(e));
  };
#define PT_FREE(p) chk(cudaFree(p), #p)
  PT_FREE(c->d_rows); PT_FREE(c->d_meta); PT_FREE(c->d_normals); PT_FREE(c->d_mats); PT_FREE(c->d_lights); PT_FREE(c->d_state);
  PT_FREE(c->d_filt); PT_FREE(c->d_filt_ids); PT_FREE(c->d_bvh_nodes); PT_FREE(c->d_bvh_leaves); PT_FREE(c->d_bvh_meta);
  PT_FREE(c->d_ctrl); PT_FREE(c->d_live); PT_FREE(c->d_accum); PT_FREE(c->d_rgb); PT_FREE(c->d_rgba8);
  PT_FREE(c->d_scratch); PT_FREE(c->d_light_k); PT_FREE(c->d_shadow); PT_FREE(c->d_ptab); PT_FREE(c->d_prim);
  PT_FREE(c->d_slab); PT_FREE(c->d_means); PT_FREE(c->d_base[0]); PT_FREE(c->d_base[1]);
#undef PT_FREE
  for (int i = 0; i < pt_context::kSlots; i++) {
    if (c->wf_stream[i]) chk(cudaStreamDestroy(c->wf_stream[i]), "wf_stream");
    if (c->ev_join[i]) chk(cudaEventDestroy(c->ev_join[i]), "ev_join");
  }
  if (c->ev_fork) chk(cudaEventDestroy(c->ev_fork), "ev_fork");
  if (c->ahead_stream) chk(cudaStreamDestroy(c->ahead_stream), "ahead_stream");
  if (c->copy_stream) chk(cudaStreamDestroy(c->copy_stream), "copy_stream");
  if (c->ev_res) chk(cudaEventDestroy(c->ev_res), "ev_res");
  if (c->ev_copy) chk(cudaEventDestroy(c->ev_copy), "ev_copy");
  for (int i = 0; i < 2; i++) {
    if (c->ev_ready[i]) chk(cudaEventDestroy(c->ev_ready[i]), "ev_ready");
    if (c->ev_consumed[i]) chk(cudaEventDestroy(c->ev_consumed[i]), "ev_consumed");
  }
  if (c->h_policy) chk(cudaFreeHost(c->h_policy), "h_policy");
  if (c->ev0) chk(cudaEventDestroy(c->ev0), "ev0");
  if (c->ev1) chk(cudaEventDestroy(c->ev1), "ev1");
  if (c->own_stream) chk(cudaStreamDestroy(c->own_stream), "own_stream");
  cudaGetLastError();  // nothing of this context's teardown may surface in a later call's error check
  delete c;
  return PT_OK;
}

extern "C" int pt_context_create(const pt_static_geom* geoms, int n_geoms, const pt_material* materials,
                                 int n_materials, const pt_camera_data* cam, const pt_lens* lens, int device,
                                 pt_context** out) {
  if (!out) { pt_set_error_("out is NULL"); return PT_ERR_INVALID; }
  *out = nullptr;
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { pt_set_error_("device %d out of range (%d devices)", device, ndev); return PT_ERR_INVALID; }
  CU(cudaSetDevice(device));
  pt_context* c = new pt_context();
  c->device = device;
  int rc = PT_OK;
  auto fail = [&](int code) { std::string keep = g_err; pt_context_destroy(c); g_err = keep; return code; };
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { pt_set_error_("cudaGetDeviceProperties failed"); return fail(PT_ERR_CUDA); }
  c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    pt_set_error_("stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
    return fail(PT_ERR_CUDA);
  }
  c->stream = c->own_stream;
  if (const char* env = getenv("PT_B200_FUSED")) c->q_mode = atoi(env) == 0 ? 1 : 2;  // developer knob: A/B runs
  if (cudaHostAlloc(&c->h_policy, (kMaxDepth + 1) * sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(&c->d_policy, c->h_policy, 0) != cudaSuccess) {
    pt_set_error_("cudaHostAlloc (policy words) failed: %s", cudaGetErrorString(cudaGetLastError()));
    return fail(PT_ERR_CUDA);
  }
  memset(c->h_policy, 0, (kMaxDepth + 1) * sizeof(int));
  if ((rc = upload_scene(c, geoms, n_geoms, materials, n_materials, cam, lens, true))) return fail(rc);
  if (cudaMalloc(&c->d_accum, (size_t)c->npix * sizeof(float4)) != cudaSuccess ||
      cudaMalloc(&c->d_rgb, (size_t)c->npix * 3 * sizeof(float)) != cudaSuccess ||
      cudaMalloc(&c->d_rgba8, (size_t)c->npix * sizeof(uchar4)) != cudaSuccess ||
      cudaMalloc(&c->d_ctrl, pt_context::kSlots * sizeof(WfCtrl)) != cudaSuccess ||
      cudaMalloc(&c->d_live, (kMaxDepth + 3) * sizeof(unsigned long long)) != cudaSuccess) {
    pt_set_error_("cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    return fail(PT_ERR_CUDA);
  }
  if ((rc = alloc_wavefront(c, kDefaultWavefrontPaths))) return fail(rc);
  if ((rc = pt_clear(c))) return fail(rc);
  *out = c;
  return PT_OK;
}

static int stream_discard(pt_context* c);  // pt_stream_*: drop the samples traced ahead

#define CTX(c)                                                       \
  do {                                                               \
    if (!(c)) { pt_set_error_("context is NULL"); return PT_ERR_STATE; } \
    CU(cudaSetDevice((c)->device));                                  \
  } while (0)

extern "C" int pt_update_scene(pt_context* c, const pt_static_geom* geoms, int n_geoms, const pt_material* materials,
                               int n_materials, const pt_camera_data* cam, const pt_lens* lens) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return upload_scene(c, geoms, n_geoms, materials, n_materials, cam, lens, false);
}

extern "C" int pt_set_wavefront_paths(pt_context* c, uint64_t max_paths) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  return alloc_wavefront(c, max_paths);
}

extern "C" int pt_set_kernel_policy(pt_context* c, int bounce_kernel) {
  CTX(c);
  if (bounce_kernel < 0 || bounce_kernel > 2) { pt_set_error_("bounce_kernel %d (0 = automatic, 1 = re-batched, 2 = fused)", bounce_kernel); return PT_ERR_INVALID; }
  CU(cudaStreamSynchronize(c->stream));
  c->q_mode = bounce_kernel;
  return PT_OK;
}

extern "C" int pt_set_band_pixels(pt_context* c, uint32_t pixels) {
  CTX(c);
  CU(cudaStreamSynchronize(c->stream));
  c->band_pixels = pixels;
  return PT_OK;
}

extern "C" int pt_set_stream(pt_context* c, void* cuda_stream) {
  CTX(c);
  CU(cudaStreamSynchronize(c->stream));
  c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
  return PT_OK;
}

extern "C" int pt_clear(pt_context* c) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaMemsetAsync(c->d_accum, 0, (size_t)c->npix * sizeof(float4), c->stream));
  CU(cudaMemsetAsync(c->d_live, 0, (kMaxDepth + 3) * sizeof(unsigned long long), c->stream));
  c->paths_total = 0;
  return PT_OK;
}

// the features a launch at `depth` runs: those switched on that the scene has a use for, roulette from its first depth
// on, and only those its segment kind has variants for
static uint32_t launch_features(const pt_context* c, bool first, bool last, uint32_t depth) {
  uint32_t fx = 0;
  if (c->nee && c->n_lights > 0) fx |= kFxNee;
  if (c->sss && c->n_media > 0) fx |= kFxMedium;  // (no medium in the scene: the plain kernels, same results)
  if (c->glossy && c->n_glossy > 0) fx |= kFxGlossy;  // (likewise without a glossy geom)
  if (c->rr_first > 0 && depth >= (uint32_t)c->rr_first) fx |= kFxRoulette;  // (a roulette depth)
  return fx & variants_of(first, last);
}

static cudaError_t launch_bounce(pt_context* c, bool first, bool last, const BounceParams& P, uint32_t n_upper, cudaStream_t st) {
  const uint32_t fx = launch_features(c, first, last, P.depth);
  const BounceKernels& k = kBounceKernels[first][last][fx];
  uint32_t grid = (uint32_t)c->grid_blocks[first][last][fx];
  // depths >= 1, few geoms: second half re-batched by winner type -- unless the scene keeps nearly all its paths alive
  // at this depth (closed rooms), where the fused kernel is faster; unknown yet (first wavefronts of a scene): re-batched
  const bool use_q = c->q_mode == 1 || (c->q_mode == 0 && ((volatile int*)c->h_policy)[P.depth] != 2);
  if (!first && !c->mode && use_q) {
    uint32_t gq = (uint32_t)c->grid_blocks_q[last][fx];
    const uint32_t ctas = (n_upper + kQThreads - 1) / kQThreads;  // one unit per warp at least
    if (ctas < gq) gq = ctas ? ctas : 1;
    k.queued<<<gq, kQThreads, c->q_smem_total, st>>>(P);
  } else if (c->mode) {
    if (first) {  // primary rays into the wavefront's input buffers
      const uint32_t blocks = (n_upper + 255u) / 256u, most = (uint32_t)c->sm_count * 8u;
      k_raygen_wf<<<blocks < most ? (blocks ? blocks : 1u) : most, 256, 0, st>>>(P);
      c->launches++;
    }
    const uint32_t ctas = (n_upper + kPoolMin * (kBvhThreads / 32) - 1) / (kPoolMin * (kBvhThreads / 32));  // a (smallest) pool per warp at least
    if (ctas < grid) grid = ctas ? ctas : 1;
    k.bvh<<<grid, kBvhThreads, kBvhSmemBytes, st>>>(P);
  } else {
    const uint32_t ctas = (n_upper + kBounceThreads - 1) / kBounceThreads;  // one unit per warp at least
    if (ctas < grid) grid = ctas ? ctas : 1;
    k.fused<<<grid, kBounceThreads, c->smem_bytes, st>>>(P);
  }
  c->launches++;
  return cudaGetLastError();
}

// the shadow-ray queues of direct light sampling: one per wavefront slot, as long as a wavefront (a path queues at most
// one shadow ray per depth, and a depth's queue is traced before the next depth fills it again)
static int ensure_shadow(pt_context* c) {
  if (!(c->d_shadow && c->shadow_cap == c->wf_capacity && c->shadow_slots == c->n_slots)) {
    if (c->d_shadow) CU(cudaFree(c->d_shadow));
    c->d_shadow = nullptr; c->shadow_cap = 0;
    if (cudaMalloc(&c->d_shadow, (size_t)c->n_slots * 4 * c->wf_capacity * sizeof(float4)) != cudaSuccess) {
      const cudaError_t e = cudaGetLastError();
      c->d_shadow = nullptr;
      pt_set_error_("cudaMalloc of the shadow-ray queues (%llu paths) failed: %s", (unsigned long long)c->wf_capacity, cudaGetErrorString(e));
      return PT_ERR_CUDA;
    }
    c->shadow_cap = c->wf_capacity; c->shadow_slots = c->n_slots;
  }
  if (c->shadow_cfg_mode == c->mode && c->shadow_cfg_smem == c->geom_smem) return PT_OK;
  int per_sm = 0;
  if (c->mode) {
    CU(cudaFuncSetAttribute(k_shadow_bvh, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBvhSmemBytes));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_shadow_bvh, kBvhThreads, kBvhSmemBytes));
  } else {
    CU(cudaFuncSetAttribute(k_shadow_lin, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shadow_lin_smem(c->geom_smem)));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_shadow_lin, kBounceThreads, shadow_lin_smem(c->geom_smem)));
  }
  if (per_sm < 1) { pt_set_error_("k_shadow does not fit on an SM"); return PT_ERR_CUDA; }
  c->grid_blocks_shadow = per_sm * c->sm_count;
  c->shadow_cfg_mode = c->mode; c->shadow_cfg_smem = c->geom_smem;
  return PT_OK;
}
// trace the shadow rays the depth-P.depth launch queued (n_upper: how many there can be at most)
static cudaError_t launch_shadow(pt_context* c, BounceParams P, uint32_t n_upper, cudaStream_t st) {
  P.in_o = P.sq_o; P.in_d = P.sq_d;  // the traversal reads its rays from the queue
  uint32_t grid = (uint32_t)c->grid_blocks_shadow;
  if (c->mode) {
    const uint32_t ctas = (n_upper + kPoolMin * (kBvhThreads / 32) - 1) / (kPoolMin * (kBvhThreads / 32));
    if (ctas < grid) grid = ctas ? ctas : 1;
    k_shadow_bvh<<<grid, kBvhThreads, kBvhSmemBytes, st>>>(P);
  } else {
    const uint32_t ctas = (n_upper + kBounceThreads - 1) / kBounceThreads;
    if (ctas < grid) grid = ctas ? ctas : 1;
    k_shadow_lin<<<grid, kBounceThreads, shadow_lin_smem(c->geom_smem), st>>>(P);
  }
  c->launches++;
  return cudaGetLastError();
}

// Trace samples [first_sample, first_sample + n_samples) of every pixel, enqueued behind `stream0`.  Radiance goes to
// accum[(s - acc_s0) * acc_stride + pixel] (stride 0: one image).
static int render_into(pt_context* c, uint32_t first_sample, uint32_t n_samples, int max_depth, uint64_t seed, cudaStream_t stream0,
                       float4* accum, uint32_t acc_s0, uint32_t acc_stride, bool timed) {
  if (max_depth < 1 || max_depth > kMaxDepth) { pt_set_error_("max_depth %d outside [1,%d]", max_depth, kMaxDepth); return PT_ERR_INVALID; }
  if ((uint64_t)first_sample + n_samples > 0xFFFFFFFFull) { pt_set_error_("sample index overflow"); return PT_ERR_INVALID; }
  if (!c->d_state || c->wf_capacity == 0) {
    pt_set_error_("no wavefront buffers (a previous pt_set_wavefront_paths failed): call it again with a size that fits");
    return PT_ERR_STATE;
  }
  const bool nee_on = c->nee && c->n_lights > 0 && max_depth > 1;
  if (nee_on) { if (int rc = ensure_shadow(c)) return rc; }
  NvtxRange nvtx_render("pt_render");
  if (timed) CU(cudaEventRecord(c->ev0, stream0));
  const uint64_t cap = c->wf_capacity;
  // Bands: a frame whose float4 accumulation image does not leave room in the 126 MB L2 (> 48 MB, e.g. 3840x2160) is
  // rendered in bands of 1 Mi pixels (16 MB of sums) with proportionally more samples per wavefront, so that the radiance
  // atomics of the wavefronts in flight keep hitting L2 instead of DRAM.  Results do not depend on it (RNG streams are
  // keyed by pixel and sample).  3840x2160, Gseg/s by band size: 0.5 Mi 27.3, 1 Mi 27.2, 2 Mi 26.9, 4 Mi 22.1, unbanded 24.9.
  uint32_t band_cap = c->band_pixels ? c->band_pixels
                                     : ((size_t)c->npix * sizeof(float4) <= ((size_t)48 << 20) ? c->npix : (1u << 20));
  if (band_cap > c->npix) band_cap = c->npix;
  if ((uint64_t)band_cap > cap) band_cap = (uint32_t)cap;
  const uint32_t spp_band = (uint32_t)(cap / band_cap);  // samples per wavefront of a full band (>= 1)
  // fork: wavefront i runs on internal stream i % kSlots, after everything queued on the caller's stream so far
  const uint64_t n_bands = ((uint64_t)c->npix + band_cap - 1) / band_cap;
  const uint64_t n_wf = n_bands * (((uint64_t)n_samples + spp_band - 1) / spp_band);
  const int slots_used = n_wf < (uint64_t)c->n_slots ? (int)n_wf : c->n_slots;
  const bool forked = slots_used > 1;  // a single wavefront in flight simply runs on the caller's stream
  if (forked) {
    CU(cudaEventRecord(c->ev_fork, stream0));
    for (int i = 0; i < slots_used; i++) CU(cudaStreamWaitEvent(c->wf_stream[i], c->ev_fork, 0));
  }
  uint64_t wf = 0;
  for (uint32_t pix0 = 0; pix0 < c->npix; pix0 += band_cap) {
  NvtxRange nvtx_band("band");
  const uint32_t band = c->npix - pix0 < band_cap ? c->npix - pix0 : band_cap;
  const uint32_t spp_wf = (uint32_t)(cap / band);
  for (uint32_t s0 = 0; s0 < n_samples; s0 += spp_wf, wf++) {
    NvtxRange nvtx_wf("wavefront");
    const int sl = (int)(wf % (uint64_t)slots_used);
    cudaStream_t st = forked ? c->wf_stream[sl] : stream0;
    float4* S = reinterpret_cast<float4*>(reinterpret_cast<char*>(c->d_state) + (size_t)sl * state_bytes(cap));
    WfCtrl* ctrl = c->d_ctrl + sl;
    const uint32_t ns = (n_samples - s0 < spp_wf) ? (n_samples - s0) : spp_wf;
    const uint32_t n_first = ns * band;
    CU(cudaMemsetAsync(ctrl, 0, sizeof(WfCtrl), st));
    for (int depth = 0; depth < max_depth; depth++) {
      BounceParams P;
      const int in = depth & 1, outb = in ^ 1;
      P.in_o = S + (3 * in + 0) * cap; P.in_d = S + (3 * in + 1) * cap; P.in_t = S + (3 * in + 2) * cap;
      P.out_o = S + (3 * outb + 0) * cap; P.out_d = S + (3 * outb + 1) * cap; P.out_t = S + (3 * outb + 2) * cap;
      P.accum = accum; P.acc_s0 = acc_s0; P.acc_stride = acc_stride;
      P.g = c->g; P.n_geoms = c->n_geoms;
      P.normals = c->d_normals;
      P.filt = c->filt; P.filt_cap = c->filt_cap;
      P.bvh = c->bvh;
      P.bvh_res = S + 6 * cap;
      float4* const SQ = nee_on ? c->d_shadow + (size_t)sl * 4 * cap : nullptr;
      P.sq_o = SQ; P.sq_d = SQ ? SQ + cap : nullptr; P.sq_t = SQ ? SQ + 2 * cap : nullptr; P.sq_x = SQ ? SQ + 3 * cap : nullptr;
      P.mats = c->d_mats;
      P.lights = c->d_lights; P.n_lights = c->n_lights; P.light_k = c->d_light_k;
      P.cam = c->cam;
      P.ctrl = ctrl;
      P.depth = (uint32_t)depth;
      P.keys = philox_keys(seed);
      P.first_sample = first_sample + s0;
      P.n_first = n_first;
      P.pix0 = pix0; P.band = band;
      P.div_band = make_fastdiv(band);
      P.q_offset = (uint32_t)c->geom_smem;
      P.cap = (uint32_t)cap;
      P.ptab = c->ptab_on ? c->d_ptab : nullptr;
      const bool first = depth == 0, last = depth == max_depth - 1;
      cudaError_t e = launch_bounce(c, first, last, P, n_first, st);
      if (e != cudaSuccess) { pt_set_error_("k_bounce launch failed: %s", cudaGetErrorString(e)); return PT_ERR_CUDA; }
      // direct light sampling: the shadow rays this depth queued, before the next depth queues its own
      if (nee_on && !last && (e = launch_shadow(c, P, n_first, st)) != cudaSuccess) {
        pt_set_error_("k_shadow launch failed: %s", cudaGetErrorString(e));
        return PT_ERR_CUDA;
      }
    }
    k_accum_counts<<<1, kMaxDepth, 0, st>>>(ctrl, c->d_live, max_depth, c->q_mode == 0 && !c->mode ? c->d_policy : nullptr);
    c->launches++;
    CU(cudaGetLastError());
    c->paths_total += n_first;
  }
  }
  // join: the caller's stream continues when both internal streams are done
  for (int i = 0; forked && i < slots_used; i++) {
    CU(cudaEventRecord(c->ev_join[i], c->wf_stream[i]));
    CU(cudaStreamWaitEvent(stream0, c->ev_join[i], 0));
  }
  if (timed) {
    CU(cudaEventRecord(c->ev1, stream0));
    c->timed = true;
  }
  return PT_OK;
}

extern "C" int pt_render(pt_context* c, uint32_t first_sample, uint32_t n_samples, int max_depth, uint64_t seed) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;  // samples traced ahead share the path-state buffers
  return render_into(c, first_sample, n_samples, max_depth, seed, c->stream, c->d_accum, 0u, 0u, true);
}

extern "C" int pt_sync(pt_context* c) {
  CTX(c);
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}

extern "C" int pt_last_render_ms(pt_context* c, float* ms) {
  CTX(c);
  if (!ms) { pt_set_error_("ms is NULL"); return PT_ERR_INVALID; }
  if (!c->timed) { pt_set_error_("no render has been recorded"); return PT_ERR_STATE; }
  CU(cudaEventSynchronize(c->ev1));
  CU(cudaEventElapsedTime(ms, c->ev0, c->ev1));
  return PT_OK;
}

static int download_rgb(pt_context* c, float* rgb, float spp, int divide) {
  if (!rgb) { pt_set_error_("rgb is NULL"); return PT_ERR_INVALID; }
  if (int rc = stream_discard(c)) return rc;  // a sample stream keeps the sum up to date lazily
  const uint32_t blocks = (c->npix + 255) / 256;
  k_resolve_rgb<<<blocks, 256, 0, c->stream>>>(c->d_accum, c->npix, spp, divide, c->d_rgb);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(rgb, c->d_rgb, (size_t)c->npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}
extern "C" int pt_download_sum(pt_context* c, float* rgb) { CTX(c); return download_rgb(c, rgb, 1.0f, 0); }
extern "C" int pt_download_mean(pt_context* c, float* rgb, uint32_t spp) {
  CTX(c);
  if (spp == 0) { pt_set_error_("spp is 0"); return PT_ERR_INVALID; }
  return download_rgb(c, rgb, (float)spp, 1);
}

// ---- sample streaming: the reference's loop asks for the running mean after EVERY sample (src/main.cpp:93-113) ----
// A one-sample render of an 800x800 frame is 8 launches of 20-55 us, each bound by its own latency chains
// (profiles/r02_shim_notes.txt).  Here samples are traced AHEAD, a group at a time, each into an image of its own
// ("slab"), at the throughput of a large wavefront; k_stream_prefix then forms the group's running means (the same
// binary32 adds, in the same order, as one atomic add per sample into the sum).  A call only copies its mean to the
// host.  Two groups alternate: while one is handed out the other is traced.  d_accum holds the sum before the oldest
// group that is not used up; stream_close() folds in the samples already handed out of that group.
static int stream_close(pt_context* c, bool keep_consumed) {
  if (!c->stream_open) return PT_OK;
  c->stream_open = false;
  CU(cudaStreamSynchronize(c->ahead_stream));
  CU(cudaStreamSynchronize(c->copy_stream));
  const uint32_t G = c->stream_group, rel = c->stream_next - c->stream_base;
  const uint32_t j = rel % G;
  const int slot = (int)((rel / G) & 1u);
  if (keep_consumed && j > 0) {
    k_stream_apply<<<(c->npix + 255) / 256, 256, 0, c->stream>>>(c->d_accum, c->d_slab + (size_t)slot * G * c->npix, c->npix, j);
    c->launches++;
    CU(cudaGetLastError());
  }
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}
static int stream_discard(pt_context* c) { return stream_close(c, true); }
extern "C" int pt_stream_end(pt_context* c) {
  CTX(c);
  return stream_close(c, true);
}
// trace the group that starts at sample `first` into slab group `slot` (all zeros here) and form its running means;
// everything on ahead_stream
static int stream_trace_group(pt_context* c, int slot, uint32_t first) {
  const uint32_t G = c->stream_group;
  if ((uint64_t)first + G > 0xFFFFFFFFull) return PT_OK;  // the sample index space ends: nothing more to trace ahead
  float4* slabs = c->d_slab + (size_t)slot * G * c->npix;
  int rc = render_into(c, first, G, c->stream_depth, c->stream_seed, c->ahead_stream, slabs, first, c->npix, false);
  if (rc) return rc;
  const float spp0 = (float)(c->stream_spp0 + (first - c->stream_base) + 1u);  // samples in the sum once the group's first one is in
  k_stream_prefix<<<(c->npix + 255) / 256, 256, 0, c->ahead_stream>>>(c->d_base[slot], slabs, c->npix, G, spp0,
                                                                       c->d_means + (size_t)slot * G * c->npix * 3, c->d_base[slot ^ 1]);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ev_ready[slot], c->ahead_stream));
  return PT_OK;
}
extern "C" int pt_stream_begin(pt_context* c, uint32_t first_sample, uint32_t spp_before, int max_depth, uint64_t seed, uint32_t group) {
  CTX(c);
  if (max_depth < 1 || max_depth > kMaxDepth) { pt_set_error_("max_depth %d outside [1,%d]", max_depth, kMaxDepth); return PT_ERR_INVALID; }
  if (group < 1 || group > 64) { pt_set_error_("group %u outside [1,64]", group); return PT_ERR_INVALID; }
  if (int rc = stream_close(c, true)) return rc;
  if (!c->ahead_stream) {
    CU(cudaStreamCreateWithFlags(&c->ahead_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&c->ev_res, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
      CU(cudaEventCreateWithFlags(&c->ev_ready[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming));
    }
  }
  if (c->slab_group != group) {
    cudaFree(c->d_slab); cudaFree(c->d_means); cudaFree(c->d_base[0]); cudaFree(c->d_base[1]);
    c->d_slab = nullptr; c->d_means = nullptr; c->d_base[0] = c->d_base[1] = nullptr; c->slab_group = 0;
    CU(cudaMalloc(&c->d_slab, (size_t)2 * group * c->npix * sizeof(float4)));
    CU(cudaMalloc(&c->d_means, (size_t)2 * group * c->npix * 3 * sizeof(float)));
    CU(cudaMalloc(&c->d_base[0], (size_t)c->npix * sizeof(float4)));
    CU(cudaMalloc(&c->d_base[1], (size_t)c->npix * sizeof(float4)));
    c->slab_group = group;
  }
  CU(cudaStreamSynchronize(c->stream));  // whatever the caller queued (clear, upload, scene) is done before samples are traced
  CU(cudaMemsetAsync(c->d_slab, 0, (size_t)2 * group * c->npix * sizeof(float4), c->ahead_stream));
  CU(cudaMemcpyAsync(c->d_base[0], c->d_accum, (size_t)c->npix * sizeof(float4), cudaMemcpyDeviceToDevice, c->ahead_stream));
  c->stream_base = c->stream_next = first_sample;
  c->stream_spp0 = spp_before;
  c->stream_group = group; c->stream_depth = max_depth; c->stream_seed = seed;
  c->stream_open = true;
  for (int slot = 0; slot < 2; slot++)
    if (int rc = stream_trace_group(c, slot, first_sample + (uint32_t)slot * group)) { c->stream_open = false; return rc; }
  return PT_OK;
}
extern "C" int pt_stream_next(pt_context* c, float* rgb, void* device_rgba8, uint32_t* spp) {
  CTX(c);
  if (!c->stream_open) { pt_set_error_("no sample stream is open (pt_stream_begin)"); return PT_ERR_STATE; }
  if (!rgb) { pt_set_error_("rgb is NULL"); return PT_ERR_INVALID; }
  const uint32_t G = c->stream_group, rel = c->stream_next - c->stream_base;
  const uint32_t q = rel / G, j = rel % G;
  const int slot = (int)(q & 1u);
  if ((uint64_t)c->stream_base + (uint64_t)(q + 1) * G > 0xFFFFFFFFull) { pt_set_error_("sample index overflow"); return PT_ERR_INVALID; }
  const float* mean = c->d_means + ((size_t)slot * G + j) * c->npix * 3;
  CU(cudaStreamWaitEvent(c->copy_stream, c->ev_ready[slot], 0));
  CU(cudaMemcpyAsync(rgb, mean, (size_t)c->npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->copy_stream));
  CU(cudaEventRecord(c->ev_copy, c->copy_stream));
  if (device_rgba8) {
    CU(cudaStreamWaitEvent(c->stream, c->ev_ready[slot], 0));
    k_rgb_to_rgba8<<<(c->npix + 255) / 256, 256, 0, c->stream>>>(mean, c->npix, (uchar4*)device_rgba8);
    c->launches++;
    CU(cudaGetLastError());
  }
  c->stream_next++;
  if (spp) *spp = c->stream_spp0 + rel + 1u;
  int rc = PT_OK;
  if (j == G - 1) {
    // this group is used up: the sum moves past it (= the base of the other group), its slabs are cleared, and it takes
    // the samples after the other group's -- all behind this call's copy and conversion
    if (device_rgba8) { CU(cudaEventRecord(c->ev_res, c->stream)); CU(cudaStreamWaitEvent(c->ahead_stream, c->ev_res, 0)); }
    CU(cudaStreamWaitEvent(c->ahead_stream, c->ev_copy, 0));
    CU(cudaMemcpyAsync(c->d_accum, c->d_base[slot ^ 1], (size_t)c->npix * sizeof(float4), cudaMemcpyDeviceToDevice, c->ahead_stream));
    CU(cudaMemsetAsync(c->d_slab + (size_t)slot * G * c->npix, 0, (size_t)G * c->npix * sizeof(float4), c->ahead_stream));
    rc = stream_trace_group(c, slot, c->stream_base + (q + 2) * G);
  }
  CU(cudaEventSynchronize(c->ev_copy));
  if (device_rgba8) CU(cudaStreamSynchronize(c->stream));
  return rc;
}

extern "C" int pt_upload_sum(pt_context* c, const float* rgb) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  if (!rgb) { pt_set_error_("rgb is NULL"); return PT_ERR_INVALID; }
  CU(cudaMemcpyAsync(c->d_rgb, rgb, (size_t)c->npix * 3 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  k_upload_rgb<<<(c->npix + 255) / 256, 256, 0, c->stream>>>(c->d_rgb, c->npix, c->d_accum);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}

extern "C" int pt_resolve_rgba8(pt_context* c, uint32_t spp, uint8_t* host_rgba8, void* device_rgba8) {
  CTX(c);
  if (spp == 0) { pt_set_error_("spp is 0"); return PT_ERR_INVALID; }
  if (int rc = stream_discard(c)) return rc;
  uchar4* dst = device_rgba8 ? (uchar4*)device_rgba8 : c->d_rgba8;
  k_resolve_rgba8<<<(c->npix + 255) / 256, 256, 0, c->stream>>>(c->d_accum, c->npix, (float)spp, dst);
  CU(cudaGetLastError());
  if (host_rgba8) CU(cudaMemcpyAsync(host_rgba8, dst, (size_t)c->npix * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}

extern "C" int pt_accum_device_ptr(pt_context* c, void** device_ptr, size_t* bytes) {
  CTX(c);
  if (device_ptr) *device_ptr = c->d_accum;
  if (bytes) *bytes = (size_t)c->npix * sizeof(float4);
  return PT_OK;
}

extern "C" int pt_launch_count(pt_context* c, uint64_t* launches) {
  CTX(c);
  if (!launches) { pt_set_error_("launches is NULL"); return PT_ERR_INVALID; }
  *launches = c->launches;
  return PT_OK;
}

extern "C" int pt_counters(pt_context* c, uint64_t* paths, uint64_t* segments, uint64_t* live) {
  CTX(c);
  unsigned long long h[kMaxDepth];
  CU(cudaMemcpyAsync(h, c->d_live, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  uint64_t seg = 0;
  for (int i = 0; i < kMaxDepth; i++) { seg += h[i]; if (live) live[i] = h[i]; }
  if (segments) *segments = seg;
  if (paths) *paths = c->paths_total;
  return PT_OK;
}

// ---------------------------------------------------------------- stage entry points
template <typename T>
struct DevBuf {
  T* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t n) { return cudaMalloc(&p, (n ? n : 1) * sizeof(T)); }
};

// Carves the list entry points' device buffers out of one grow-only arena owned by the context (256-byte aligned pieces).
struct Arena {
  pt_context* c;
  size_t used = 0;
  explicit Arena(pt_context* ctx) : c(ctx) {}
  static size_t up(size_t b) { return (b + 255) & ~(size_t)255; }
  int reserve(size_t total) {
    if (total <= c->scratch_bytes) return PT_OK;
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_scratch) CU(cudaFree(c->d_scratch));
    c->d_scratch = nullptr; c->scratch_bytes = 0;
    CU(cudaMalloc(&c->d_scratch, total));
    c->scratch_bytes = total;
    return PT_OK;
  }
  template <typename T>
  T* take(size_t count) {
    T* p = reinterpret_cast<T*>(static_cast<char*>(c->d_scratch) + used);
    used += up((count ? count : 1) * sizeof(T));
    return p;
  }
};

extern "C" int pt_raygen(pt_context* c, uint64_t seed, int n, const uint32_t* pixel, const uint32_t* sample,
                         float* origin, float* direction) {
  CTX(c);
  if (n < 0 || (n > 0 && (!pixel || !sample || !origin || !direction))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (n == 0) return PT_OK;
  for (int i = 0; i < n; i++)
    if (pixel[i] >= c->npix) { pt_set_error_("pixel[%d] = %u outside the %u-pixel frame", i, pixel[i], c->npix); return PT_ERR_INVALID; }
  Arena A(c);
  if (int rc = A.reserve(2 * Arena::up(n * sizeof(uint32_t)) + 2 * Arena::up(3 * (size_t)n * sizeof(float)))) return rc;
  uint32_t *dp = A.take<uint32_t>(n), *ds = A.take<uint32_t>(n);
  float *dor = A.take<float>(3 * (size_t)n), *ddr = A.take<float>(3 * (size_t)n);
  CU(cudaMemcpyAsync(dp, pixel, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(ds, sample, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  k_raygen_list<<<(n + 255) / 256, 256, 0, c->stream>>>(c->cam, seed, n, dp, ds, dor, ddr);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(origin, dor, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(direction, ddr, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return PT_OK;
}

extern "C" int pt_intersect_ex(pt_context* c, int mode, int n, const float* origin, const float* direction,
                               int32_t* geom_id, float* t, float* point, float* normal, uint64_t* fallbacks) {
  CTX(c);
  if (n < 0 || (n > 0 && (!origin || !direction || !geom_id || !t || !point || !normal))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (mode != PT_HIT_FILTERED && mode != PT_HIT_EXACT_SCAN) { pt_set_error_("mode %d is neither PT_HIT_FILTERED nor PT_HIT_EXACT_SCAN", mode); return PT_ERR_INVALID; }
  if (fallbacks) *fallbacks = 0;
  if (n == 0) return PT_OK;
  const size_t v = 3 * (size_t)n;
  Arena A(c);
  if (int rc = A.reserve(4 * Arena::up(v * sizeof(float)) + Arena::up(n * sizeof(float)) + Arena::up(n * sizeof(int)) + 256)) return rc;
  float *dor = A.take<float>(v), *ddr = A.take<float>(v), *dt = A.take<float>(n), *dpnt = A.take<float>(v), *dn = A.take<float>(v);
  int* did = A.take<int>(n);
  unsigned long long* dfb = A.take<unsigned long long>(1);
  CU(cudaMemcpyAsync(dor, origin, v * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(ddr, direction, v * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(dfb, 0, sizeof(unsigned long long), c->stream));
  k_intersect_list<<<(n + kTile - 1) / kTile, kTile, c->geom_smem, c->stream>>>(
      c->g, c->n_geoms, c->filt, c->filt_cap, c->bvh, mode == PT_HIT_FILTERED ? c->d_normals : nullptr, mode, n, dor, ddr,
      did, dt, dpnt, dn, dfb);
  c->launches++;
  CU(cudaGetLastError());
  unsigned long long fb = 0;
  CU(cudaMemcpyAsync(geom_id, did, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(t, dt, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(point, dpnt, v * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(normal, dn, v * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(&fb, dfb, sizeof(fb), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (fallbacks) *fallbacks = fb;
  return PT_OK;
}
extern "C" int pt_intersect(pt_context* c, int n, const float* origin, const float* direction, int32_t* geom_id,
                            float* t, float* point, float* normal) {
  return pt_intersect_ex(c, PT_HIT_FILTERED, n, origin, direction, geom_id, t, point, normal, nullptr);
}

extern "C" int pt_primary_hit(pt_context* c, uint64_t seed, int n, const uint32_t* pixel, const uint32_t* sample, int32_t* geom_id,
                              float* t, float* point, float* normal, uint8_t* decided, uint64_t* fallbacks) {
  CTX(c);
  if (n < 0 || (n > 0 && (!pixel || !sample || !geom_id || !t || !point || !normal || !decided))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (c->mode != 0) { pt_set_error_("pt_primary_hit: the scene has %d geoms and uses the hierarchy, not the pair scan", c->n_geoms); return PT_ERR_STATE; }
  if (fallbacks) *fallbacks = 0;
  if (n == 0) return PT_OK;
  for (int i = 0; i < n; i++)
    if (pixel[i] >= c->npix) { pt_set_error_("pixel[%d] = %u outside the %u-pixel frame", i, pixel[i], c->npix); return PT_ERR_INVALID; }
  const size_t v = 3 * (size_t)n;
  Arena A(c);
  if (int rc = A.reserve(2 * Arena::up(n * sizeof(uint32_t)) + 2 * Arena::up(v * sizeof(float)) + Arena::up(n * sizeof(float)) +
                         Arena::up(n * sizeof(int)) + Arena::up(n) + 256)) return rc;
  uint32_t *dp = A.take<uint32_t>(n), *ds = A.take<uint32_t>(n);
  float *dt = A.take<float>(n), *dpnt = A.take<float>(v), *dn = A.take<float>(v);
  int* did = A.take<int>(n);
  uint8_t* ddec = A.take<uint8_t>(n);
  unsigned long long* dfb = A.take<unsigned long long>(1);
  CU(cudaMemcpyAsync(dp, pixel, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(ds, sample, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemsetAsync(dfb, 0, sizeof(unsigned long long), c->stream));
  k_primary_list<<<(n + kTile - 1) / kTile, kTile, c->geom_smem, c->stream>>>(c->cam, seed, c->g, c->n_geoms, c->filt, c->d_normals,
                                                                               c->ptab_on ? c->d_ptab : nullptr, n, dp, ds, did, dt, dpnt, dn, ddec, dfb);
  c->launches++;
  CU(cudaGetLastError());
  unsigned long long fb = 0;
  CU(cudaMemcpyAsync(geom_id, did, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(t, dt, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(point, dpnt, v * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(normal, dn, v * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(decided, ddec, n, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(&fb, dfb, sizeof(fb), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (fallbacks) *fallbacks = fb;
  return PT_OK;
}

extern "C" int pt_primary_table_info(pt_context* c, int* active, float* build_ms) {
  CTX(c);
  if (!active) { pt_set_error_("active is NULL"); return PT_ERR_INVALID; }
  *active = c->ptab_on ? 1 : 0;
  if (build_ms) {
    // time one rebuild, host records to finished kernel: what a scene update or a filter-scale change pays for it
    CU(cudaStreamSynchronize(c->stream));
    const auto t0 = std::chrono::steady_clock::now();
    if (int rc = build_primary_table(c)) return rc;
    *build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  return PT_OK;
}

extern "C" int pt_set_filter_scale(pt_context* c, float scale) {
  CTX(c);
  if (!(scale >= 0.0f) || !(scale <= 1e6f)) { pt_set_error_("filter scale %g outside [0, 1e6]", (double)scale); return PT_ERR_INVALID; }
  CU(cudaStreamSynchronize(c->stream));
  c->filter_scale = scale;
  if (int rc = upload_filter(c)) return rc;
  return build_primary_table(c);  // (its margin scales with the filter's)
}

extern "C" int pt_filter_stats(pt_context* c, uint64_t* fallbacks) {
  CTX(c);
  if (!fallbacks) { pt_set_error_("fallbacks is NULL"); return PT_ERR_INVALID; }
  unsigned long long h = 0;
  CU(cudaMemcpyAsync(&h, c->d_live + kMaxDepth, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *fallbacks = h;
  return PT_OK;
}

extern "C" int pt_filter_retries(pt_context* c, uint64_t* retries) {
  CTX(c);
  if (!retries) { pt_set_error_("retries is NULL"); return PT_ERR_INVALID; }
  unsigned long long h = 0;
  CU(cudaMemcpyAsync(&h, c->d_live + kMaxDepth + 2, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *retries = h;
  return PT_OK;
}

extern "C" int pt_set_direct_lighting(pt_context* c, int on) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  c->nee = on != 0;
  return PT_OK;
}
extern "C" int pt_set_subsurface(pt_context* c, int on) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  c->sss = on != 0;
  return PT_OK;
}
extern "C" int pt_set_glossy(pt_context* c, int on) {
  CTX(c);
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  c->glossy = on != 0;
  return PT_OK;
}
extern "C" int pt_set_russian_roulette(pt_context* c, int first_depth) {
  CTX(c);
  if (first_depth < 0 || first_depth > kMaxDepth - 1) {
    pt_set_error_("first_depth %d: Russian roulette takes 0 (off) or a first depth in [1, %d]", first_depth, kMaxDepth - 1);
    return PT_ERR_INVALID;
  }
  if (int rc = stream_discard(c)) return rc;
  CU(cudaStreamSynchronize(c->stream));
  c->rr_first = first_depth;
  return PT_OK;
}
extern "C" int pt_shadow_rays(pt_context* c, uint64_t* shadow_rays, int* n_lights) {
  CTX(c);
  if (!shadow_rays) { pt_set_error_("shadow_rays is NULL"); return PT_ERR_INVALID; }
  unsigned long long h = 0;
  CU(cudaMemcpyAsync(&h, c->d_live + kMaxDepth + 1, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *shadow_rays = h;
  if (n_lights) *n_lights = c->n_lights;
  return PT_OK;
}

static int g_compact_mode = 0;  // 0: count / scan / scatter (three launches), 1: k_compact_u32 (single pass)
extern "C" int pt_set_compact_mode(int mode) {
  if (mode != 0 && mode != 1) { pt_set_error_("compact mode %d (0 = three kernels, 1 = single pass)", mode); return PT_ERR_INVALID; }
  g_compact_mode = mode;
  return PT_OK;
}
static int compact_impl(int device, const uint32_t* values, const uint8_t* flags, uint64_t n, uint32_t* out,
                        uint64_t* n_out, int timed_iters, float* kernel_ms) {
  if (!n_out || (n > 0 && (!values || !flags || !out))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  *n_out = 0;
  if (kernel_ms) *kernel_ms = 0.0f;
  if (n == 0) return PT_OK;
  if (n > 0xFFFFFF00ull) { pt_set_error_("n too large"); return PT_ERR_INVALID; }
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { pt_set_error_("device %d out of range", device); return PT_ERR_INVALID; }
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  DevBuf<uint32_t> dv, dout, dctl, dcount, dprefix;
  DevBuf<uint8_t> df;
  DevBuf<uint64_t> dst, dst2;
  const uint64_t tiles = (n + kCompactTile - 1) / kCompactTile;
  const uint64_t chunks = (tiles + kScanChunk - 1) / kScanChunk;  // CTAs of k_compact_scan: <= 1024, all resident
  CU(dv.alloc(n)); CU(dout.alloc(n)); CU(dctl.alloc(3)); /* ticket of k_compact_u32, n_out, ticket of k_compact_scan */ CU(df.alloc(n)); CU(dst.alloc(tiles));
  CU(dcount.alloc(tiles)); CU(dprefix.alloc(tiles)); CU(dst2.alloc(chunks));
  CU(cudaMemset(dst2.p, 0, chunks * sizeof(uint64_t)));
  CU(cudaMemcpy(dv.p, values, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(df.p, flags, n, cudaMemcpyHostToDevice));
  CU(cudaMemset(dst.p, 0, tiles * sizeof(uint64_t)));
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_compact_u32, kCompactThreads, 0));
  uint64_t grid = (uint64_t)per_sm * prop.multiProcessorCount;
  if (tiles < grid) grid = tiles;
  int per_sm_c = 0, per_sm_s = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_c, k_compact_count, kCompactThreads, 0));
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_s, k_compact_scatter, kCompactThreads, 0));
  uint64_t grid_c = (uint64_t)per_sm_c * prop.multiProcessorCount, grid_s = (uint64_t)per_sm_s * prop.multiProcessorCount;
  if (tiles < grid_c) grid_c = tiles;
  if (tiles < grid_s) grid_s = tiles;
  // the status words carry the launch epoch, so repeated launches need no clearing in between
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (timed_iters > 0) { CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1)); }
  const int launches = timed_iters > 0 ? timed_iters + 1 : 1;  // one warm-up launch before the timed ones
  for (int it = 0; it < launches; it++) {
    CU(cudaMemsetAsync(dctl.p, 0, 3 * sizeof(uint32_t), 0));
    if (timed_iters > 0 && it == 1) CU(cudaEventRecord(e0, 0));
    if (g_compact_mode == 1) {
      k_compact_u32<<<(unsigned)grid, kCompactThreads>>>(dv.p, df.p, (uint32_t)n, dout.p, dctl.p + 1, dctl.p, dst.p, (uint32_t)(it + 1));
    } else {
      k_compact_count<<<(unsigned)grid_c, kCompactThreads>>>(df.p, (uint32_t)n, (uint32_t)tiles, dcount.p);
      k_compact_scan<<<(unsigned)chunks, kScanThreads>>>(dcount.p, (uint32_t)tiles, dprefix.p, dctl.p + 1, dctl.p + 2, dst2.p, (uint32_t)(it + 1));
      k_compact_scatter<<<(unsigned)grid_s, kCompactThreads>>>(dv.p, df.p, (uint32_t)n, (uint32_t)tiles, dprefix.p, dout.p);
    }
    CU(cudaGetLastError());
  }
  if (timed_iters > 0) {
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    float ms = 0.0f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (kernel_ms) *kernel_ms = ms / timed_iters;  // includes one 8-byte memset per launch
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  uint32_t cnt = 0;
  CU(cudaMemcpy(&cnt, dctl.p + 1, sizeof(cnt), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(out, dout.p, (size_t)cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  *n_out = cnt;
  return PT_OK;
}
extern "C" int pt_compact_u32(int device, const uint32_t* values, const uint8_t* flags, uint64_t n, uint32_t* out,
                              uint64_t* n_out) {
  return compact_impl(device, values, flags, n, out, n_out, 0, nullptr);
}
extern "C" int pt_compact_u32_timed(int device, const uint32_t* values, const uint8_t* flags, uint64_t n, uint32_t* out,
                                    uint64_t* n_out, int iters, float* kernel_ms) {
  if (iters < 1 || !kernel_ms) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  return compact_impl(device, values, flags, n, out, n_out, iters, kernel_ms);
}

extern "C" int pt_selftest_math(int device, uint64_t bad[3]) {
  if (!bad) { pt_set_error_("bad is NULL"); return PT_ERR_INVALID; }
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { pt_set_error_("device %d out of range (%d devices)", device, ndev); return PT_ERR_INVALID; }
  CU(cudaSetDevice(device));
  DevBuf<unsigned long long> d;
  CU(d.alloc(3));
  CU(cudaMemset(d.p, 0, 3 * sizeof(unsigned long long)));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  k_selftest_math<<<prop.multiProcessorCount * 8, 256>>>(d.p);
  CU(cudaGetLastError());
  unsigned long long h[3];
  CU(cudaMemcpy(h, d.p, sizeof(h), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 3; i++) bad[i] = h[i];
  return PT_OK;
}

// ---------------------------------------------------------------- sampling / transmission parity entry points
static int select_device_(int device) {
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { pt_set_error_("device %d out of range (%d devices)", device, ndev); return PT_ERR_INVALID; }
  CU(cudaSetDevice(device));
  return PT_OK;
}
static int points_impl(int device, const pt_static_geom* g, int mode, int n, const float* in, float* points) {
  if (!g || n < 0 || (n > 0 && (!in || !points))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (g->type != 0 && g->type != 1) { pt_set_error_("geom type %d has no surface sampler (sphere = 0, cube = 1)", g->type); return PT_ERR_INVALID; }
  if (n == 0) return PT_OK;
  if (mode == 0)  // the reference converts the seed float -> unsigned (src/intersections.h:135): defined for [0, 2^32) only
    for (int i = 0; i < n; i++)
      if (!(in[i] >= 0.0f && in[i] < 4294967296.0f)) { pt_set_error_("seeds[%d] = %g outside [0, 2^32)", i, (double)in[i]); return PT_ERR_INVALID; }
  if (int rc = select_device_(device)) return rc;
  const size_t per = mode == 0 ? 1 : 3;
  DevBuf<float> din, dout;
  CU(din.alloc(per * n)); CU(dout.alloc(3 * (size_t)n));
  CU(cudaMemcpy(din.p, in, per * n * sizeof(float), cudaMemcpyHostToDevice));
  const float* T = g->transform;
  k_points_on_geom<<<(n + 255) / 256, 256>>>(g->type, make_float4(T[0], T[1], T[2], T[3]), make_float4(T[4], T[5], T[6], T[7]),
                                             make_float4(T[8], T[9], T[10], T[11]), mode, n, din.p, dout.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(points, dout.p, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}
extern "C" int pt_random_points_on_geom(int device, const pt_static_geom* geom, int n, const float* seeds, float* points) {
  return points_impl(device, geom, 0, n, seeds, points);
}
extern "C" int pt_points_on_geom_u(int device, const pt_static_geom* geom, int n, const float* u, float* points) {
  return points_impl(device, geom, 1, n, u, points);
}
extern "C" int pt_random_directions_in_sphere(int device, int n, const float* xi1, const float* xi2, float* dirs) {
  if (n < 0 || (n > 0 && (!xi1 || !xi2 || !dirs))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (n == 0) return PT_OK;
  if (int rc = select_device_(device)) return rc;
  DevBuf<float> d1, d2, dout;
  CU(d1.alloc(n)); CU(d2.alloc(n)); CU(dout.alloc(3 * (size_t)n));
  CU(cudaMemcpy(d1.p, xi1, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d2.p, xi2, n * sizeof(float), cudaMemcpyHostToDevice));
  k_sphere_dirs<<<(n + 255) / 256, 256>>>(n, d1.p, d2.p, dout.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(dirs, dout.p, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}
extern "C" int pt_calculate_transmission(int device, int n, const float* absorption, const float* distance, float* out) {
  if (n < 0 || (n > 0 && (!absorption || !distance || !out))) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  if (n == 0) return PT_OK;
  if (int rc = select_device_(device)) return rc;
  DevBuf<float> da, dd, dout;
  CU(da.alloc(3 * (size_t)n)); CU(dd.alloc(n)); CU(dout.alloc(3 * (size_t)n));
  CU(cudaMemcpy(da.p, absorption, 3 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(dd.p, distance, n * sizeof(float), cudaMemcpyHostToDevice));
  k_transmission<<<(n + 255) / 256, 256>>>(n, da.p, dd.p, dout.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, dout.p, 3 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}

extern "C" int pt_sample_medium(int device, int n, const float* absorption, const float* scatter, const float* distance,
                                const float* u, int32_t* scattered, float* s, float* direction, float* weight) {
  if (n < 0 || (n > 0 && (!absorption || !scatter || !distance || !u || !scattered || !s || !direction || !weight))) {
    pt_set_error_("bad arguments");
    return PT_ERR_INVALID;
  }
  if (n == 0) return PT_OK;
  if (int rc = select_device_(device)) return rc;
  const size_t n3 = 3 * (size_t)n;
  // one arena: absorption, scatter, distance, u in; s, direction, weight out (floats), then the flags
  DevBuf<float> buf;
  CU(buf.alloc(n3 + n + n + n3 + n + n3 + n3 + n));
  float *da = buf.p, *dsc = da + n3, *dd = dsc + n, *du = dd + n, *ds = du + n3, *ddir = ds + n, *dw = ddir + n3;
  int32_t* dflag = reinterpret_cast<int32_t*>(dw + n3);
  CU(cudaMemcpy(da, absorption, n3 * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(dsc, scatter, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(dd, distance, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(du, u, n3 * sizeof(float), cudaMemcpyHostToDevice));
  k_sample_medium<<<(n + 255) / 256, 256>>>(n, da, dsc, dd, du, dflag, ds, ddir, dw);
  CU(cudaGetLastError());
  CU(cudaMemcpy(scattered, dflag, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(s, ds, n * sizeof(float), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(direction, ddir, n3 * sizeof(float), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(weight, dw, n3 * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}

extern "C" int pt_sample_glossy(int device, int n, const float* normal, const float* incident, const float* exponent,
                                const float* u, float* direction) {
  if (n < 0 || (n > 0 && (!normal || !incident || !exponent || !u || !direction))) {
    pt_set_error_("bad arguments");
    return PT_ERR_INVALID;
  }
  if (n == 0) return PT_OK;
  if (int rc = select_device_(device)) return rc;
  const size_t n3 = 3 * (size_t)n;
  // one arena: normal, incident, exponent, u in; direction out
  DevBuf<float> buf;
  CU(buf.alloc(n3 + n3 + n + 2 * (size_t)n + n3));
  float *dn = buf.p, *di = dn + n3, *de = di + n3, *du = de + n, *ddir = du + 2 * (size_t)n;
  CU(cudaMemcpy(dn, normal, n3 * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(di, incident, n3 * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(de, exponent, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(du, u, 2 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
  k_sample_glossy<<<(n + 255) / 256, 256>>>(n, dn, di, de, du, ddir);
  CU(cudaGetLastError());
  CU(cudaMemcpy(direction, ddir, n3 * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}

extern "C" int pt_reference_stub_image(int device, int width, int height, int iterations, int order, float* rgb) {
  if (width <= 0 || height <= 0 || !rgb || (order != 0 && order != 1) || (uint64_t)width * height > (1ull << 28)) {
    pt_set_error_("bad arguments");
    return PT_ERR_INVALID;
  }
  if (int rc = select_device_(device)) return rc;
  DevBuf<float> d;
  const size_t n = (size_t)width * height * 3;
  CU(d.alloc(n));
  const dim3 block(8, 8), grid((width + 7) / 8, (height + 7) / 8);  // the reference's launch shape, src/raytraceKernel.cu:113-115
  k_reference_stub<<<grid, block>>>(width, height, (float)iterations, order, d.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(rgb, d.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return PT_OK;
}

// ---------------------------------------------------------------- multi-GPU combine (single process, one context per GPU)
// One ncclReduce(sum) of the float4 accumulation images to ctxs[0] over NVLink / NVSwitch.  NCCL is resolved at run
// time (dlopen) so that a process that already carries its own libnccl (PyTorch) keeps a single copy; processes
// launched one-per-GPU (bench.py under torchrun) do the same reduce through torch.distributed instead.
#include <dlfcn.h>
namespace {
typedef struct ncclComm* nccl_comm_t;
struct NcclApi {
  void* h = nullptr;
  int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*Reduce)(const void*, void*, size_t, int, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::vector<int> devs;
  std::vector<nccl_comm_t> comms;
} g_nccl;
bool load_nccl() {
  if (g_nccl.h) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.h) break;
  }
  if (!g_nccl.h) { pt_set_error_("NCCL not found (dlopen libnccl.so.2): %s", dlerror()); return false; }
  *(void**)&g_nccl.CommInitAll = dlsym(g_nccl.h, "ncclCommInitAll");
  *(void**)&g_nccl.CommDestroy = dlsym(g_nccl.h, "ncclCommDestroy");
  *(void**)&g_nccl.GroupStart = dlsym(g_nccl.h, "ncclGroupStart");
  *(void**)&g_nccl.GroupEnd = dlsym(g_nccl.h, "ncclGroupEnd");
  *(void**)&g_nccl.Reduce = dlsym(g_nccl.h, "ncclReduce");
  *(void**)&g_nccl.GetErrorString = dlsym(g_nccl.h, "ncclGetErrorString");
  if (!g_nccl.CommInitAll || !g_nccl.GroupStart || !g_nccl.GroupEnd || !g_nccl.Reduce) {
    pt_set_error_("libnccl lacks ncclCommInitAll/ncclReduce");
    g_nccl.h = nullptr;
    return false;
  }
  return true;
}
}  // namespace

#define NC(call)                                                                                  \
  do {                                                                                            \
    int r_ = (call);                                                                              \
    if (r_ != 0) {                                                                                \
      pt_set_error_("%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
      return PT_ERR_CUDA;                                                                         \
    }                                                                                             \
  } while (0)

extern "C" int pt_reduce_to_first(pt_context* const* ctxs, int n) {
  if (!ctxs || n < 1) { pt_set_error_("bad arguments"); return PT_ERR_INVALID; }
  for (int i = 0; i < n; i++) {
    if (!ctxs[i]) { pt_set_error_("context %d is NULL", i); return PT_ERR_STATE; }
    if (ctxs[i]->npix != ctxs[0]->npix) { pt_set_error_("context %d has a different frame size", i); return PT_ERR_INVALID; }
    for (int j = 0; j < i; j++)
      if (ctxs[j]->device == ctxs[i]->device) { pt_set_error_("contexts %d and %d share device %d", j, i, ctxs[i]->device); return PT_ERR_INVALID; }
  }
  if (n == 1) return PT_OK;
  NvtxRange nvtx_reduce("reduce");
  if (!load_nccl()) return PT_ERR_CUDA;
  std::vector<int> devs(n);
  for (int i = 0; i < n; i++) devs[i] = ctxs[i]->device;
  if (devs != g_nccl.devs) {
    for (nccl_comm_t c : g_nccl.comms) if (g_nccl.CommDestroy) g_nccl.CommDestroy(c);
    g_nccl.comms.assign(n, nullptr);
    g_nccl.devs.clear();
    NC(g_nccl.CommInitAll(g_nccl.comms.data(), n, devs.data()));
    g_nccl.devs = devs;
  }
  NC(g_nccl.GroupStart());
  for (int i = 0; i < n; i++) {
    CU(cudaSetDevice(ctxs[i]->device));
    // ncclFloat32 = 7, ncclSum = 0, root = rank 0
    NC(g_nccl.Reduce(ctxs[i]->d_accum, ctxs[i]->d_accum, (size_t)ctxs[i]->npix * 4, 7, 0, 0, g_nccl.comms[i], ctxs[i]->stream));
  }
  NC(g_nccl.GroupEnd());
  // (path / segment counters stay per context: callers add them up, pt_main.cpp)
  for (int i = 0; i < n; i++) {
    CU(cudaSetDevice(ctxs[i]->device));
    CU(cudaStreamSynchronize(ctxs[i]->stream));
  }
  return PT_OK;
}

#ifdef PT_BVH_STACK_HIST
extern "C" int pt_debug_sp_hist(unsigned long long* out64) {
  return cudaMemcpyFromSymbol(out64, ptd::g_sp_hist, 64 * sizeof(unsigned long long)) == cudaSuccess ? 0 : 1;
}
#endif
