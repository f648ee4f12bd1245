// pt_kernels.cuh -- the wavefront kernels (sm_100a).
//
//   k_bounce<FIRST,LAST,NEE,MEDIUM,GLOSSY>  one path segment for every live path of the wavefront, fused (few geoms: depth 0, and every depth
//                           of scenes that keep nearly all their paths alive):
//                           [FIRST: raygen + depth of field]  (raycastFromCameraKernel, src/raytraceKernel.cu:40-45)
//                           closest hit over SoA geometry staged in shared memory (src/intersections.h:74-117)
//                           BSDF sampling with Philox (calculateBSDF, src/interactions.h:99-104), absorption inside glass
//                           (calculateTransmission, :31-33), [NEE: direct light sampling, src/intersections.h:133-182]
//                           [MEDIUM: subsurface scattering inside media, calculateScatterAndAbsorption, :36-39]
//                           [GLOSSY: glossy reflection, a Phong lobe around the mirror direction (SPECEX)]
//                           radiance accumulation in HBM (the running image of src/raytraceKernel.cu:118-120,154)
//                           stream compaction of the survivors (README.md:63-70): warp ballot -> ranks inside a 32-path
//                           unit, one slot-reserving atomic per unit, survivors written once to the other ping-pong
//                           buffer.
//                         Persistent CTAs; warps take units from a ticket counter and never wait for each other; the
//                         live count never visits the host.
//   k_bounce_q<LAST,NEE,MEDIUM,GLOSSY>  depths >= 1 of few-geom scenes: the same segment with its second half (exact test of the filter's
//                         candidate, shading, compaction) re-batched by winner type in per-warp shared-memory queues
//   k_raygen_wf + k_bounce_bvh<LAST,NEE,MEDIUM,GLOSSY>   scenes with many geoms: primary rays into the wavefront's buffers, then one kernel
//                         for every depth -- pooled traversal of the hierarchy (pt_bvh.cuh) with lane refill, exact
//                         tests and shading unit by unit
//   k_shadow_lin / k_shadow_bvh   direct light sampling: the shadow rays a depth queued, traced by a launch of their own
//   k_raygen_list / k_intersect_list   the same device functions on caller-supplied lists (parity entry points)
//   k_compact_u32                      the stable compaction primitive on its own: ballot -> block scan -> decoupled look-back
//   k_points_on_geom / k_sphere_dirs / k_transmission (pt_sampling.cuh)   sampling and absorption parity entry points
//   k_resolve_*                        accumulation buffer -> float RGB / uchar4 (sendImageToPBO, :58-89)
#pragma once
#include "pt_device.cuh"
#include "pt_filter.cuh"
#include "pt_bvh.cuh"
#include "pt_sampling.cuh"

namespace ptd {

constexpr int kMaxDepth = 64;
constexpr int kTile = 256;  // paths per tile = threads per CTA (list kernels, k_compact_u32)
#ifndef PT_BOUNCE_THREADS
#define PT_BOUNCE_THREADS 256  // threads per CTA of k_bounce (tuning knob together with PT_MIN_BLOCKS, see profiles/)
#endif
constexpr int kBounceThreads = PT_BOUNCE_THREADS;
#ifndef PT_MIN_BLOCKS
#define PT_MIN_BLOCKS 4  // resident CTAs per SM the register allocation aims for (tuning knob, see profiles/)
#endif

// per-wavefront control block in HBM, zeroed before each wavefront
struct WfCtrl {
  uint32_t count[kMaxDepth + 1];     // count[d] = live paths entering depth d
  uint32_t tile_ctr[kMaxDepth + 1];  // ticket counter of the depth-d launch
  uint32_t fallbacks;                // rays whose filtered closest hit fell back to the exact scan (statistics)
  uint32_t retries;                  // hierarchy: rays whose nearest candidate was not confirmed and whose second candidate settled them (statistics)
  unsigned long long shadow;         // shadow rays traced by direct light sampling
  uint32_t shadow_ctr[kMaxDepth + 1];  // ticket counter of the depth-d shadow launch (k_shadow_*)
};

// ---- decoupled look-back (Merrill & Garland 2016) on 64-bit status words ----
// word = epoch[63:34] | state[33:32] | value[31:0]; a word is valid only if its epoch equals the launch's, so the
// array never needs clearing between launches (or CUDA-graph replays).
constexpr uint32_t kStAggregate = 1u, kStPrefix = 2u;
__device__ __forceinline__ uint64_t st_pack(uint32_t epoch, uint32_t state, uint32_t value) {
  return ((uint64_t)epoch << 34) | ((uint64_t)state << 32) | (uint64_t)value;
}
__device__ __forceinline__ void st_store(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t st_load(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Called by ONE full warp of the CTA that owns `tile`.  aggregate = number of survivors in this tile.
// Returns the number of survivors in all earlier tiles (exclusive prefix) to every lane.
// (Inspecting 128 instead of 32 predecessors per look-back step -- four independent loads per lane -- was tried for
// k_compact_u32 and did not help: tiles do not wait for the prefix wave but for the slowest load among ALL their
// predecessors, see profiles/r01_compact_u32.txt.)
__device__ __forceinline__ uint32_t lookback_exclusive(uint64_t* status, uint32_t tile, uint32_t epoch,
                                                       uint32_t aggregate) {
  const uint32_t lane = threadIdx.x & 31u;
  if (lane == 0) st_store(status + tile, st_pack(epoch, tile == 0 ? kStPrefix : kStAggregate, aggregate));
  if (tile == 0) return 0;
  uint32_t exclusive = 0;
  int look = (int)tile - 1;
  for (;;) {
    const int t = look - (int)lane;
    uint32_t state = kStPrefix, value = 0;  // tiles before the first one: empty prefix
    if (t >= 0) {
      uint64_t w;
      do { w = st_load(status + t); } while ((uint32_t)(w >> 34) != epoch);
      state = (uint32_t)(w >> 32) & 3u;
      value = (uint32_t)w;
    }
    const uint32_t pmask = __ballot_sync(0xffffffffu, state == kStPrefix);
    const int firstp = pmask ? (__ffs(pmask) - 1) : 31;
    uint32_t contrib = ((int)lane <= firstp) ? value : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
    exclusive += contrib;
    if (pmask) break;
    look -= 32;
  }
  if (lane == 0) st_store(status + tile, st_pack(epoch, kStPrefix, exclusive + aggregate));
  return exclusive;
}

struct BounceParams {
  const float4 *in_o, *in_d, *in_t;  // path state in:  (origin.xyz, pixel) (direction.xyz, sample) (throughput.xyz, -)
  float4 *out_o, *out_d, *out_t;     // survivors out, compacted
  float4* accum;                     // per-pixel radiance sums
  GeomSoA g;                         // per-geom rows in HBM (the winner's exact test / material lookup)
  const float4* normals;             // per-geom table of face normals and sphere centres (k_normal_table)
  int n_geoms;
  FiltSoA filt;                      // filter geometry (pt_filter.cuh): pairs of geoms, four classes
  int filt_cap;                      // pairs that fit in shared memory
  BvhSoA bvh;                        // hierarchy over the same filter tests for scenes with many geoms (pt_bvh.cuh)
  float4* bvh_res;                   // k_bounce_bvh: per path of the wavefront (lo2, lo3, bits of the candidate leaves k1, k2), between its two phases
  const float4* mats;                // 4 float4 per material
  const float4* lights;              // direct light sampling: 3 float4 per light (E.xyz | geom) (th0..th3) (th4, type, K, -)
  const float* light_k;              // per geom: K = area * n_lights / pi of a light, 0 otherwise (balance heuristic at emissive hits)
  int n_lights;
  RaygenConsts cam;
  WfCtrl* ctrl;
  uint32_t depth;
  PhiloxKeys keys;                   // round keys of the render's seed
  uint32_t first_sample, n_first;    // FIRST only: paths to generate = band * samples in this wavefront
  uint32_t pix0, band;               // FIRST only: the wavefront covers pixels [pix0, pix0 + band) (the whole frame unless banded)
  FastDiv div_band;                  // FIRST only: path index -> (sample, pixel of the band)
  float4 *sq_o, *sq_d, *sq_t, *sq_x; // direct light sampling: the wavefront's queue of shadow rays (origin | pixel) (direction | sample)
                                     // (throughput * emittance | cosine at the surface) (distance to the light point, K, light geom, -)
  uint32_t q_offset;                 // k_bounce_q: byte offset of the warps' candidate queues in dynamic shared memory
  uint32_t cap;                      // paths the in / out buffers hold (debug checks)
  uint32_t acc_s0, acc_stride;       // radiance of sample s goes to accum[(s - acc_s0) * acc_stride + pixel]: stride 0 = one image for
                                     // all samples (the rule), stride = pixels per frame = one image per sample (pt_stream_*)
  const uint32_t* ptab;              // FIRST only: per-pixel candidate of the primary rays (k_primary_table), null = none
                                     // (last member: the other kernels read the members before it at unchanged offsets)
};

// ---- the primary-ray table (DESIGN.md 3a "primary rays"): pinhole cameras, pair-scan scenes ----
// Every primary ray of a pixel starts at the eye and points into the pixel's footprint, so the filter's answer is nearly
// always the same for all of them.  k_primary_table works it out once per pixel, in binary64, for the footprint's
// central ray against every filter shape grown by rho = D * (largest angle between a ray of the footprint and the
// central ray): a grown shape the central ray enters at world distance s is entered by no ray of the footprint before
// s.  Entry per pixel: (bits(lo2) & ~kKeyMask) | key of the candidate, kKeyMask = "no table decision".
struct PrimRec {      // one filter shape at the eye, in the frame where it is a unit-free ball or box
  double A[9];        // ray direction -> shape frame (identity for the world-space classes 0 and 2)
  double ro[3];       // the eye in the shape frame
  double h[3];        // ball: radius in h[0]; box: half extents
  double g[3];        // growth of h per unit of world distance rho (ball: sigma_max(A) in g[0]; box: |row i of A|)
  double D;           // no point of the shape is farther than D from the eye
  double ew;          // world slack E_w of the filter at the eye
  int ball, key;      // shape kind; 2 * pair + half of the filter scan
};
constexpr int kMaxPrimRecs = 128;
// the pixel's footprint: d_c = unit central direction; returns the largest angle between d_c and the direction of any
// primary ray raygen() makes for the pixel, rounding included, or a negative value when no bound is possible
__device__ __forceinline__ double footprint_angle(const RaygenConsts& C, uint32_t pixel, double dc[3]) {
  const double u = 5.9604644775390625e-8;  // 2^-24
  const uint32_t yi = pixel / C.W;
  const double x = (double)(pixel - yi * C.W), y = (double)yi, fw = C.fw, fh = C.fh;
  // sx = 1 - 2 ((x + u0) / fw), u0 in [0, 1): the real interval, widened by the binary32 evaluation's error
  const double ex = 16.0 * u * (1.0 + 2.0 * (x + 1.0) / fw), ey = 16.0 * u * (1.0 + 2.0 * (y + 1.0) / fh);
  const double sx0 = 1.0 - 2.0 * (x + 1.0) / fw - ex, sx1 = 1.0 - 2.0 * x / fw + ex;
  const double sy0 = 1.0 - 2.0 * (y + 1.0) / fh - ey, sy1 = 1.0 - 2.0 * y / fh + ey;
  const double w[3] = {C.w.x, C.w.y, C.w.z}, H[3] = {C.Hh.x, C.Hh.y, C.Hh.z}, V[3] = {C.Vv.x, C.Vv.y, C.Vv.z};
  // every v = w + H sx + V sy lies in one plane: |v| >= the plane's distance from the origin
  double n[3] = {H[1] * V[2] - H[2] * V[1], H[2] * V[0] - H[0] * V[2], H[0] * V[1] - H[1] * V[0]};
  const double nn = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
  const double vmin = fabs(w[0] * n[0] + w[1] * n[1] + w[2] * n[2]) / nn;
  const double nw = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]), nH = sqrt(H[0] * H[0] + H[1] * H[1] + H[2] * H[2]),
               nV = sqrt(V[0] * V[0] + V[1] * V[1] + V[2] * V[2]);
  // binary32 error of (w + H sx) + V sy, and of the normalisation, as an angle
  const double ev = 8.0 * u * (nw + nH * fmax(fabs(sx0), fabs(sx1)) + nV * fmax(fabs(sy0), fabs(sy1)));
  if (!(nn > 0) || !(vmin > 16.0 * ev)) return -1.0;
  const double th_r = 2.0 * ev / vmin + 8.0 * u;
  const double sxc = 0.5 * (sx0 + sx1), syc = 0.5 * (sy0 + sy1);
  double l = 0.0;
  for (int i = 0; i < 3; i++) { dc[i] = w[i] + H[i] * sxc + V[i] * syc; l += dc[i] * dc[i]; }
  l = sqrt(l);
  for (int i = 0; i < 3; i++) dc[i] /= l;
  // the angle to d_c is quasi-convex over the rectangle (its sublevel sets are a plane cut through a convex cone), so
  // its maximum is at a corner
  double th = 0.0;
  for (int k = 0; k < 4; k++) {
    const double sx = (k & 1) ? sx1 : sx0, sy = (k & 2) ? sy1 : sy0;
    double v[3];
    for (int i = 0; i < 3; i++) v[i] = w[i] + H[i] * sx + V[i] * sy;
    const double cx = v[1] * dc[2] - v[2] * dc[1], cy = v[2] * dc[0] - v[0] * dc[2], cz = v[0] * dc[1] - v[1] * dc[0];
    th = fmax(th, atan2(sqrt(cx * cx + cy * cy + cz * cz), v[0] * dc[0] + v[1] * dc[1] + v[2] * dc[2]));
  }
  th = (th + th_r) * (1.0 + 1e-6) + 1e-12;
  return th < 1.0 ? th : -1.0;  // (a cone of half-angle >= 1 rad: no table decision)
}
// smallest s >= 0 at which ro + s rw lies in the grown shape (rounded so that it is no later than the exact value),
// +inf when it never does.  Both shapes are inflated by 1e-9 of their scale first, far above binary64 rounding.
__device__ __forceinline__ double prim_entry(const PrimRec& R, const double rw[3], double rho) {
  if (R.ball) {
    const double r = R.h[0] + rho * R.g[0];
    const double ro2 = R.ro[0] * R.ro[0] + R.ro[1] * R.ro[1] + R.ro[2] * R.ro[2];
    const double a = rw[0] * rw[0] + rw[1] * rw[1] + rw[2] * rw[2];
    const double b = R.ro[0] * rw[0] + R.ro[1] * rw[1] + R.ro[2] * rw[2];
    const double c = ro2 - (r * r + 1e-9 * (ro2 + r * r));
    const double disc = b * b - a * c;
    if (disc < 0.0) return INFINITY;
    const double sq = sqrt(disc);
    if (-b + sq < 0.0) return INFINITY;  // behind the eye
    return fmax((-b - sq) / a, 0.0);
  }
  double tn = 0.0, tf = INFINITY;
  for (int i = 0; i < 3; i++) {
    const double h = (R.h[i] + rho * R.g[i]) * (1.0 + 1e-9) + 1e-9 * fabs(R.ro[i]);
    if (rw[i] == 0.0) {
      if (fabs(R.ro[i]) > h) return INFINITY;
      continue;
    }
    const double t1 = (-h - R.ro[i]) / rw[i], t2 = (h - R.ro[i]) / rw[i];
    tn = fmax(tn, fmin(t1, t2));
    tf = fmin(tf, fmax(t1, t2));
  }
  return tn <= tf ? tn : INFINITY;
}
__global__ void __launch_bounds__(128) k_primary_table(RaygenConsts C, const PrimRec* recs, int n_recs, double scale, uint32_t* tab) {
  const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= C.npix) return;
  double dc[3];
  const double th = footprint_angle(C, pixel, dc);
  uint32_t entry = kKeyMask;
  if (th >= 0.0) {
    double lo1 = INFINITY, lo2 = INFINITY;
    int k1 = -1;
    for (int j = 0; j < n_recs; j++) {
      const PrimRec& R = recs[j];
      double rw[3];
      for (int i = 0; i < 3; i++) rw[i] = R.A[3 * i] * dc[0] + R.A[3 * i + 1] * dc[1] + R.A[3 * i + 2] * dc[2];
      const double rho = scale * R.D * th * (1.0 + 1e-6);
      const double s = prim_entry(R, rw, rho);
      if (!(s < INFINITY)) continue;  // a proven miss for the whole footprint
      const double lo = fmax(s - R.ew, 0.0);
      if (lo < lo1) { lo2 = lo1; lo1 = lo; k1 = R.key; }
      else lo2 = fmin(lo2, lo);
    }
    if (k1 >= 0 && lo2 > lo1) {
      // lo2 rounded down to binary32 (a finite value: an entry's bits must not read as NaN), then its key bits cleared
      float f = (float)fmin(lo2, 3.0e38);
      if ((double)f > lo2) f = nextafterf(f, 0.0f);
      entry = (__float_as_uint(f) & ~kKeyMask) | (uint32_t)k1;
    }
  }
  tab[pixel] = entry;
}

// Closest hit of a primary ray, by a whole warp: the exact test of the table's candidate (`tab`, may be null) and, for
// the lanes it does not settle, the filter scan and the exact test of its candidate -- ONE copy of the exact test for
// both -- and, where that does not settle the ray either, the exact scan (return value: it ran).  The acceptance rule
// is resolve_scan's, so the answer is the exact scan's, bit for bit.  `decided`: the table's candidate was confirmed.
__device__ __forceinline__ bool primary_hit(const uint32_t* tab, const float4* fs, const FiltSoA& filt, const GeomSoA& g, int n_geoms,
                                            bool valid, uint32_t pixel, f3 o, f3 d, Hit& h, bool& decided) {
  ScanBest best;
  best.k1 = -1; best.lo2 = 0.0f;
  bool scan = valid, open = valid, from_tab = false, fell_back = false;
  decided = false;
  if (tab != nullptr && valid) {
    const uint32_t e = __ldg(tab + pixel);
    if ((e & kKeyMask) != kKeyMask) {
      best.k1 = (int)(e & kKeyMask); best.lo2 = __uint_as_float(e & ~kKeyMask);
      scan = false; from_tab = true;
    }
  }
#pragma unroll 1
  for (;;) {
    if (__any_sync(0xffffffffu, scan)) {
      if (scan) {
        scan_init(best);
        const ScanRay ray = make_scan_ray(o, d, filt.r_scene, filt.end[2] > filt.end[1]);
        filter_scan(fs, 0, filt.end[3], filt.end, ray, best);
      }
    }
    bool retry = false;
    if (open && best.k1 >= 0) {
      const int gi = __ldg(reinterpret_cast<const int*>(filt.ids) + best.k1);
      const int type = best.k1 < 2 * filt.end[1] ? 0 : 1;
      float dist;
      f3 P;
      int ncode;
      DeferredGuard m;
      const bool hit = exact_hit(type, __ldg(g.inv0 + gi), __ldg(g.inv1 + gi), __ldg(g.inv2 + gi), __ldg(g.fwd0 + gi),
                                 __ldg(g.fwd1 + gi), __ldg(g.fwd2 + gi), o, d, dist, P, ncode, m);
      if (!m.bad && hit && dist > 0 && dist < best.lo2) {
        h.t = dist; h.id = gi; h.p = P; h.ncode = ncode;
        decided = from_tab;
      } else if (from_tab) {
        retry = true;  // the footprint's candidate is not this ray's: the filter decides
      } else {
        closest_hit_exact(g, n_geoms, o, d, h);
        fell_back = true;
      }
    }
    if (!__any_sync(0xffffffffu, retry)) break;
    scan = retry; open = retry; from_tab = false;
  }
  return fell_back;
}

// what changes from one depth of a wavefront to the next: the ping-pong buffers and the depth itself (a launch per depth
// takes it from its parameters).  A single cooperative launch stepping through all depths of a small wavefront was
// measured and dropped: a 640 k-path wavefront is bound by per-unit latency chains, not by launches -- 377 us in one
// launch with grid-wide barriers against 295 us as 8 launches (profiles/r02_shim_notes.txt).
struct DepthIO {
  const float4 *in_o, *in_d, *in_t;
  float4 *out_o, *out_d, *out_t;
  uint32_t depth;
};
__device__ __forceinline__ DepthIO depth_io(const BounceParams& P) {
  DepthIO io;
  io.in_o = P.in_o; io.in_d = P.in_d; io.in_t = P.in_t;
  io.out_o = P.out_o; io.out_d = P.out_d; io.out_t = P.out_t;
  io.depth = P.depth;
  return io;
}

// Work decomposition of k_bounce: the unit of work is ONE WARP x 32 consecutive paths.  Warps take units from a
// global ticket counter and never synchronise with the other warps of their CTA (an earlier version with
// barrier-delimited 1024-path CTA tiles left a third of the resident warps parked at __syncthreads() and the
// look-back warp spinning: profiles/r01_k_bounce_v1_*, r01_k_bounce_v5_*).
// Stream compaction of the survivors (README.md:63-70): warp ballot -> rank of each survivor inside its unit
// (order preserved inside a unit); the unit's base slot is reserved with ONE atomic on the next depth's live count,
// issued by lane 0 as soon as the ballot is known; the survivors go straight from registers to base + rank,
// coalesced.  Units finish in roughly ticket order, so the output stays roughly ordered, but it is not the stable
// compaction a scan would give: at 32-path granularity (4 700 units in flight, 470 finishing per microsecond) a
// decoupled look-back has to walk ~15 windows of 32 predecessors per unit and cost 40 % more instructions than the
// tracing itself (profiles/r01_k_bounce_v6_lookback32_*); the ordered, look-back based primitive remains available
// as k_compact_u32 / pt_compact_u32.  Results do not depend on the slot order (RNG streams are keyed by pixel and
// sample, radiance goes through atomics).
constexpr int kUnit = 32;  // paths per unit = one warp

// radiance into the accumulation image: one 16-byte vector reduction (REDG.E.ADD.F32x4) instead of three scalar ones; each
// component is the same binary32 add (w += 0), a third of the atomic transactions in L2
__device__ __forceinline__ void accum_add(float4* px, f3 L) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(px), "f"(L.x), "f"(L.y), "f"(L.z), "f"(0.0f) : "memory");
}

__device__ __forceinline__ float4* accum_at(const BounceParams& P, uint32_t pixel, uint32_t sample) {
  return P.accum + pixel + (size_t)(sample - P.acc_s0) * P.acc_stride;
}

__device__ __forceinline__ uint32_t atom_add_u32(uint32_t* p, uint32_t v) {  // plain ATOMG, no warp-aggregation code
  uint32_t old;
  asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}

// A ticket is kTicketUnits consecutive units: the ticket counter sees one atomic per 128 paths (atomics on one address
// serialise in L2 at about one per clock; a ticket per unit put the counter at a third of that limit).
#ifndef PT_TICKET_UNITS
#define PT_TICKET_UNITS 4
#endif
constexpr uint32_t kTicketUnits = PT_TICKET_UNITS;

// closest hit of one ray on its own (direct light sampling's shadow rays).  LINEAR: pair scan over `fs`, else hierarchy.
template <bool LINEAR>
__device__ __forceinline__ void closest_hit_one(const BounceParams& P, const float4* fs, f3 o, f3 d, Hit& h) {
  ScanBest best;
  scan_init(best);
  bool fell_back;
  if (LINEAR) {
    const ScanRay ray = make_scan_ray(o, d, P.filt.r_scene, P.filt.end[2] > P.filt.end[1]);
    filter_scan(fs, 0, P.filt.end[3], P.filt.end, ray, best);
    fell_back = resolve_scan(best, P.filt, P.g, P.n_geoms, o, d, h);
  } else {
    const ScanRay ray = make_scan_ray(o, d, P.filt.r_scene, true);
    bvh_traverse<false>(P.bvh, P.g, ray, best, h);
    fell_back = resolve_bvh(best, P.bvh, P.g, P.filt.r_scene, o, d, h);
  }
  if (fell_back) atomicAdd(&P.ctrl->fallbacks, 1u);
}

// Direct light sampling (DESIGN.md "direct light sampling"; oracle: or_render_ex), by a whole warp; `active` lanes
// have just sampled a diffuse bounce: o = new path origin, ns = shading normal, thr = throughput after the bounce.
#ifndef PT_NEE_QUEUE
#define PT_NEE_QUEUE 1
#endif
// The light sample's contribution once the closest hit `h` of its shadow ray (direction wd, unit length) is known.
// TE = throughput * emittance, cs = cosine at the surface, dy = distance to the sampled point y, gl = the light's geom.
template <bool TABLE>
__device__ __forceinline__ void shadow_resolve(const BounceParams& P, const Hit& h, f3 wd, f3 TE, float cs, float dy, float K, int gl,
                                               uint32_t pixel, uint32_t sample) {
  // y is visible iff the ray arrives ON the light AT y (its far side is hidden by the light itself)
  if (h.id != gl || !((dy - h.t) < 1e-3f * dy + 1e-3f)) return;
  const f3 n2 = TABLE ? hit_normal_table(P.normals, h)
                      : hit_normal(__ldg(P.g.fwd0 + gl), __ldg(P.g.fwd1 + gl), __ldg(P.g.fwd2 + gl), h);
  const float cl = -dot(n2, wd);
  if (!(cl > 0)) return;
  const float G = (cs * cl) / (h.t * h.t);
  const float wl = 1.0f / (1.0f + G * K);  // balance heuristic: p_bsdf / p_light = G * K, K = area * n_lights / pi
  const f3 Ld = (TE * G) * wl;
  PT_CHECK(pixel < P.cam.npix);
  accum_add(accum_at(P, pixel, sample), Ld);
}

// One light, one point on it (getRandomPointOnCube's area-weighted faces / the sphere sampler, Philox block 65 + depth),
// one shadow ray through the ordinary closest hit.
#ifndef PT_NEE_INLINE
#define PT_NEE_INLINE __forceinline__  // measured: 19.75 G rays/s inlined, 19.25 out of line (sample scene, direct light on)
#endif
// `alive` lanes continue as path `slot` of the next depth's wavefront; `active` ones among them bounced diffusely.
template <bool TABLE, bool LINEAR>
__device__ PT_NEE_INLINE void direct_light(const BounceParams& P, const DepthIO& io, const float4* fs, uint32_t lane, bool active, bool alive,
                                          uint32_t slot, f3 ns, f3 o, f3 thr, uint32_t pixel, uint32_t sample) {
  bool traced = false;
  f3 wd = mk(0, 0, 1), E = mk(0, 0, 0);
  float cs = 0.0f, dy = 0.0f, K = 0.0f;
  int gl = -1;
  if (active) {
    float v[4];
    rng4(P.keys, pixel, sample, 65u + io.depth, v);
    int li = (int)(v[0] * (float)P.n_lights);
    if (li > P.n_lights - 1) li = P.n_lights - 1;
    const float4 L0 = __ldg(P.lights + 3 * li), L1 = __ldg(P.lights + 3 * li + 1), L2 = __ldg(P.lights + 3 * li + 2);
    gl = __float_as_int(L0.w);
    E = mk(L0.x, L0.y, L0.z);
    K = L2.z;
    const float4 f0 = __ldg(P.g.fwd0 + gl), f1 = __ldg(P.g.fwd1 + gl), f2 = __ldg(P.g.fwd2 + gl);
    const f3 y = __float_as_int(L2.y) == 0 ? sphere_point(f0, f1, f2, v[1], v[2])
                                           : cube_point_th(f0, f1, f2, L1, L2.x, v[1], v[2] - 0.5f, v[3] - 0.5f);
    const f3 wv = y - o;
    wd = normalize(wv);
    dy = length(wv);
    cs = dot(ns, wd);
    traced = cs > 0;
  }
  const uint32_t tmask = __ballot_sync(0xffffffffu, traced);
#if PT_NEE_QUEUE
  // The shadow rays are not traced here -- a few lanes of a warp in the middle of the shading code -- but QUEUED: a launch
  // of its own traces the depth's shadow rays as dense units (k_shadow_lin) or through the pooled traversal (k_shadow_bvh).
  // Everything the contribution needs travels with the ray; the operations are the ones below, in the same order.
  // The queue is indexed like the next depth's wavefront -- the shadow ray of the path that continues in slot i is entry
  // i -- so it needs no slot reservation of its own (a second atomic per unit next to the compaction's, on the same L2
  // slice, halved the bounce kernels' speed); a path that continues without a shadow ray marks its entry empty.
  if (lane == 0 && tmask) atomicAdd(&P.ctrl->shadow, (unsigned long long)__popc(tmask));
  if (alive) {
    PT_CHECK(slot < P.cap);
    if (traced) {
      const f3 TE = thr * E;
      __stcs(P.sq_o + slot, make_float4(o.x, o.y, o.z, __uint_as_float(pixel)));
      __stcs(P.sq_d + slot, make_float4(wd.x, wd.y, wd.z, __uint_as_float(sample)));
      __stcs(P.sq_t + slot, make_float4(TE.x, TE.y, TE.z, cs));
      __stcs(P.sq_x + slot, make_float4(dy, K, __int_as_float(gl), 0.0f));
    } else {
      __stcs(P.sq_x + slot, make_float4(0.0f, 0.0f, __int_as_float(-1), 0.0f));  // no shadow ray
    }
  }
#else
  if (lane == 0 && tmask) atomicAdd(&P.ctrl->shadow, (unsigned long long)__popc(tmask));
  if (!traced) return;
  Hit h;
  h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
  closest_hit_one<LINEAR>(P, fs, o, wd, h);
  shadow_resolve<TABLE>(P, h, wd, thr * E, cs, dy, K, gl, pixel, sample);
#endif
}

// The second half of a segment, by a whole warp: material lookup, reservation of the unit's output slots, BSDF
// sampling, radiance of finished paths, survivors written to base + rank.  `hit` lanes carry a closest hit in h.
// TABLE: normals from the per-geom table or from the winner's own rows.  LINEAR: shadow rays scan the filter pairs in
// shared memory (`fs`; few geoms) or walk the hierarchy (many geoms).  NEE: direct light sampling at diffuse bounces; `cos_b` > 0 = the path's
// previous event was one (the cosine of the direction it sampled travels in throughput.w): a light it reaches by itself is
// weighted by the balance heuristic against that event's light sample.  MEDIUM: subsurface scattering (shade() may return 4,
// a scattering event inside a medium geom: the path goes on, without a light sample).  GLOSSY: glossy reflection (a glossy
// event is kind 1, like a mirror: no light sample, and its path carries cos_b = 0).
// Deferred output (k_bounce_q): a batch's survivors wait in shared memory while the atomic that reserves their slots is
// in flight, and are written one batch later -- the warp never waits for the atomic (it was 7 % of the stall samples:
// one address per depth takes 0.6 atomics per nanosecond, and their latency under that load exceeds a whole shading pass).
#ifndef PT_MD_FROM_TABLE
#define PT_MD_FROM_TABLE 1
#endif
struct DeferredOut {
  float4* stage;      // [3][kUnit] in the warp's shared memory: the survivors' (origin | direction | throughput) rows, ranked
  uint32_t pend_raw;  // lane 0: slot base of the staged survivors (result of the atomic; read one batch later)
  uint32_t pend_n;    // warp-uniform: survivors staged, 0 = nothing pending
};
__device__ __forceinline__ void deferred_flush(DeferredOut& W, const BounceParams& P, const DepthIO& io, uint32_t lane) {
  if (W.pend_n == 0) return;
  const uint32_t base = __shfl_sync(0xffffffffu, W.pend_raw, 0);
  if (lane < W.pend_n) {
    PT_CHECK(base + lane < P.cap);
    __stcs(io.out_o + base + lane, W.stage[lane]);
    __stcs(io.out_d + base + lane, W.stage[kUnit + lane]);
    __stcs(io.out_t + base + lane, W.stage[2 * kUnit + lane]);
  }
  W.pend_n = 0;
  __syncwarp();  // the staging rows may be overwritten now
}

template <bool LAST, bool TABLE, bool NEE, bool DEFER = false, bool LINEAR = TABLE, bool MEDIUM = false, bool GLOSSY = false>
__device__ __forceinline__ void shade_and_compact(const BounceParams& P, const DepthIO& io, const float4* fs, uint32_t lane, bool hit, const Hit& h, f3 o, f3 d, f3 thr,
                                                  uint32_t pixel, uint32_t sample, float cos_b, DeferredOut* W = nullptr) {
  // a path survives this segment unless it left the scene or reached a light; the slot of the unit's survivors
  // is reserved before shading so that the atomic's latency hides behind it
  int mat = 0;
  float4 md = make_float4(0, 0, 0, 0);  // (absorption.yz, reducedScatter, emittance)
  if (hit) {
    mat = __ldg(P.g.meta + h.id).y;
    // (the per-geom table holds a copy of its material's fourth row: one load instead of two dependent ones ahead of the ballot)
    md = (TABLE && PT_MD_FROM_TABLE) ? __ldg(P.normals + (size_t)h.id * kNormalRows + kMatRow) : __ldg(P.mats + 4 * mat + 3);
  }
  const bool alive = hit && !(md.w > 0);
  uint32_t base_raw = 0, ballot = 0;
  if (!LAST) {
    ballot = __ballot_sync(0xffffffffu, alive);
    if (DEFER) {
      deferred_flush(*W, P, io, lane);  // the batch before this one: its atomic returned long ago
      W->pend_n = (uint32_t)__popc(ballot);
      if (lane == 0 && ballot) W->pend_raw = atom_add_u32(&P.ctrl->count[io.depth + 1], (uint32_t)__popc(ballot));
    } else if (lane == 0 && ballot) {
      base_raw = atom_add_u32(&P.ctrl->count[io.depth + 1], (uint32_t)__popc(ballot));
    }
  }
  bool sampled = false;  // NEE: this lane's bounce was diffuse and gets a light sample
  float cos_s = 0.0f;    // ... and the cosine its continuing path carries to the next hit
  f3 ns = mk(0, 0, 1);
  if (hit) {
    const int gi = h.id;
    const f3 n = TABLE ? hit_normal_table(P.normals, h)
                       : hit_normal(__ldg(P.g.fwd0 + gi), __ldg(P.g.fwd1 + gi), __ldg(P.g.fwd2 + gi), h);
    MatRows m;
    m.a = __ldg(P.mats + 4 * mat); m.b = __ldg(P.mats + 4 * mat + 1); m.c = __ldg(P.mats + 4 * mat + 2); m.d = md;
    f3 L;
    if (NEE && !LAST) ns = dot(d, n) < 0 ? n : neg(n);  // the shading normal shade() uses
    const float4* frame = nullptr;
    if (TABLE && h.ncode != 8) frame = P.normals + (size_t)gi * kNormalRows + kFrameRow0 + 4 * ((h.ncode & 3) + ((h.ncode & 4) ? 3 : 0));
    const int kind = shade<MEDIUM, GLOSSY>(m, P.g, gi, h.p, n, frame, P.keys, pixel, sample, io.depth, o, d, thr, L);
    if (kind == 3) {
      // a light reached by a direction the diffuse bounce before sampled itself: balance heuristic against that bounce's
      // light sample (cos_b = cosine of this direction at the bounce, 0 = camera ray / specular event: full weight)
      if (NEE && cos_b > 0) {
        const float clp = -dot(n, d);
        if (clp > 0) {
          const float x = ((cos_b * clp) / (h.t * h.t)) * __ldg(P.light_k + gi);
          const float wb = x / (1.0f + x);
          L = L * wb;
        }
      }
      PT_CHECK(pixel < P.cam.npix);
      accum_add(accum_at(P, pixel, sample), L);
    }
    sampled = NEE && !LAST && kind == 0 && P.n_lights > 0;
    if (sampled) cos_s = dot(ns, d);  // of the direction the bounce just sampled
  }
  if (!LAST) {
    const uint32_t rank = __popc(ballot & ((1u << lane) - 1u));
    uint32_t slot = 0;  // where an alive lane's path continues in the next depth's wavefront
    if (DEFER) {
      if (alive) {
        W->stage[rank] = make_float4(o.x, o.y, o.z, __uint_as_float(pixel));
        W->stage[kUnit + rank] = make_float4(d.x, d.y, d.z, __uint_as_float(sample));
        W->stage[2 * kUnit + rank] = make_float4(thr.x, thr.y, thr.z, sampled ? cos_s : 0.0f);
      }
      __syncwarp();
      if (NEE && PT_NEE_QUEUE) slot = __shfl_sync(0xffffffffu, W->pend_raw, 0) + rank;  // (the atomic was issued before the shading)
    } else {
      slot = __shfl_sync(0xffffffffu, base_raw, 0) + rank;
      if (alive) {
        PT_CHECK(slot < P.cap);
        __stcs(io.out_o + slot, make_float4(o.x, o.y, o.z, __uint_as_float(pixel)));
        __stcs(io.out_d + slot, make_float4(d.x, d.y, d.z, __uint_as_float(sample)));
        __stcs(io.out_t + slot, make_float4(thr.x, thr.y, thr.z, sampled ? cos_s : 0.0f));
      }
    }
    if (NEE && (PT_NEE_QUEUE ? ballot != 0u : __any_sync(0xffffffffu, sampled)))
      direct_light<TABLE, LINEAR>(P, io, fs, lane, sampled, alive, slot, ns, o, thr, pixel, sample);
  }
}

// Few geoms (every BASELINE config but the 10k one): linear scan over the filter pairs staged in shared memory.
// The body of one depth, by every warp of a persistent grid (`fs` = the staged filter pairs):
template <bool FIRST, bool LAST, bool NEE, bool MEDIUM, bool GLOSSY>
__device__ __forceinline__ void bounce_fused(const BounceParams& P, const DepthIO& io, const float4* fs, uint32_t lane) {
  const uint32_t n_in = FIRST ? P.n_first : P.ctrl->count[io.depth];
  if (FIRST && blockIdx.x == 0 && threadIdx.x == 0) P.ctrl->count[0] = n_in;
  const uint32_t n_units = (n_in + kUnit - 1) / kUnit;
  uint32_t* const ticket = &P.ctrl->tile_ctr[io.depth];

  uint32_t next_raw = 0;  // lane 0: the ticket taken ahead of time
  if (lane == 0) next_raw = atom_add_u32(ticket, 1u);

  for (;;) {
    const uint32_t unit0 = __shfl_sync(0xffffffffu, next_raw, 0) * kTicketUnits;
    if (unit0 >= n_units) break;
    if (lane == 0) next_raw = atom_add_u32(ticket, 1u);  // consumed after this ticket's units: its latency is hidden
#pragma unroll 1
    for (uint32_t unit = unit0; unit < min(unit0 + kTicketUnits, n_units); unit++) {
    const uint32_t idx = unit * kUnit + lane;
    const bool valid = idx < n_in;

    f3 o = mk(0, 0, 0), d = mk(0, 0, 1), thr = mk(1, 1, 1);
    uint32_t pixel = 0, sample = 0;
    float cos_b = 0.0f;
    if (valid) {
      if (FIRST) {
        const uint32_t si = fastdiv(idx, P.div_band);
        pixel = P.pix0 + (idx - si * P.band);
        sample = P.first_sample + si;
        raygen(P.cam, P.keys, pixel, sample, o, d);
      } else {
        const float4 a = __ldcs(io.in_o + idx), b = __ldcs(io.in_d + idx), c = __ldcs(io.in_t + idx);
        o = mk(a.x, a.y, a.z); pixel = __float_as_uint(a.w);
        d = mk(b.x, b.y, b.z); sample = __float_as_uint(b.w);
        thr = mk(c.x, c.y, c.z);
        if (NEE) cos_b = c.w;
      }
    }

    Hit h;
    h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
    if constexpr (FIRST) {  // primary rays: the per-pixel table first (pinhole cameras)
      PT_CHECK(!valid || pixel < P.cam.npix);
      bool decided;
      if (primary_hit(P.ptab, fs, P.filt, P.g, P.n_geoms, valid, pixel, o, d, h, decided)) atomicAdd(&P.ctrl->fallbacks, 1u);
    } else if (valid) {
      ScanBest best;
      scan_init(best);
      const ScanRay ray = make_scan_ray(o, d, P.filt.r_scene, P.filt.end[2] > P.filt.end[1]);
      filter_scan(fs, 0, P.filt.end[3], P.filt.end, ray, best);
      if (resolve_scan(best, P.filt, P.g, P.n_geoms, o, d, h)) atomicAdd(&P.ctrl->fallbacks, 1u);
    }

    shade_and_compact<LAST, true, NEE, false, true, MEDIUM, GLOSSY>(P, io, fs, lane, valid && h.id >= 0, h, o, d, thr, pixel, sample, cos_b);
    }
  }
}

template <bool FIRST, bool LAST, bool NEE = false, bool MEDIUM = false, bool GLOSSY = false>
__global__ void __launch_bounds__(kBounceThreads, PT_MIN_BLOCKS) k_bounce(const __grid_constant__ BounceParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // ---- filter geometry: staged once per CTA ----
  stage_filt(P.filt, 0, P.filt.end[3], reinterpret_cast<float4*>(smem_raw));
  __syncthreads();  // the only CTA-wide barrier
  bounce_fused<FIRST, LAST, NEE, MEDIUM, GLOSSY>(P, depth_io(P), reinterpret_cast<const float4*>(smem_raw), threadIdx.x & 31u);
}

// ---- k_bounce_q: the same segment with the second half RE-BATCHED BY WINNER TYPE (depths >= 1, few geoms) ----
// In k_bounce a warp carries its 32 paths through the exact test and the shading together: after the first bounce a
// third of them have left the scene in the filter scan and the rest are a mix of sphere and cube winners, so the
// second half of the segment -- two thirds of the kernel's instructions -- ran with 19-22 of 32 lanes
// (profiles/r01_k_bounce_v14_*).  Here each warp owns two queues in shared memory, one per winner type.  Per unit:
//   phase A  load 32 rays (origin, direction; the throughput is not touched), filter scan; every path that has a
//            candidate is pushed (ray + candidate + lo2 + path index, 48 bytes) onto the queue of its candidate's type
//            -- ranks by ballot, no atomics, the queues are private to the warp; paths without a candidate end here
//            (black background) and their throughput is never read from HBM;
//   phase B  whenever a queue holds >= 32 entries, 32 of them are popped (their throughputs are fetched now: the load's
//            latency hides behind the exact test) and run through exact test, shading and compaction with ALL 32
//            lanes busy and with ONE shape's code (the type is warp-uniform: the sphere and the
//            cube branch of exact_hit / hit_normal / the tangent frame are never both executed).
// When the ticket counter runs dry the queues are flushed as partial batches.  The two queues grow towards each other
// in one array of kQCap = 96 entries: before a push each holds <= 31, a push adds <= 32 in total.
// Results do not depend on the order in which paths are processed (RNG streams are keyed by pixel and sample,
// radiance goes through atomics), so images and live counts are the ones k_bounce produces, bit for bit.
constexpr int kQCap = 96;
#ifndef PT_Q_PREFETCH
#define PT_Q_PREFETCH 1  // the next unit's path state travels HBM -> shared memory (cp.async) while this unit is traced
#endif
#ifndef PT_Q_PREFETCH_EARLY
#define PT_Q_PREFETCH_EARLY 1
#endif
#ifndef PT_Q_DEFER_OUT
#define PT_Q_DEFER_OUT 1
#endif
// (A queue that carries only the path index, phase B fetching the throughput from HBM itself, was measured too: a first
// touch of HBM at the head of every batch, 58 % issue-slot utilisation, slower.)
struct QWarp {
  float4 o[kQCap];  // (origin.xyz, pixel)
  float4 d[kQCap];  // (direction.xyz, sample)
  float4 t[kQCap];  // (throughput.xyz, cos_b of direct light sampling)
  float4 c[kQCap];  // (lo2 = second-smallest lower bound, bits of the candidate's geom index, path index, -)
#if PT_Q_PREFETCH
  float4 st[3][kUnit];  // staging: the next unit's (origin | direction | throughput) rows, one slot per lane
#endif
#if PT_Q_DEFER_OUT
  float4 wst[3 * kUnit];  // the last batch's survivors, written to HBM one batch later (DeferredOut)
#endif
};
#ifndef PT_Q_THREADS
#define PT_Q_THREADS 256
#endif
#ifndef PT_Q_MIN_BLOCKS
#define PT_Q_MIN_BLOCKS 3  // 80 registers: the second half of a segment does not fit 64 without spilling its loop state
#endif
constexpr int kQThreads = PT_Q_THREADS;
__host__ __device__ inline size_t q_smem_bytes() { return sizeof(QWarp) * (size_t)(kQThreads / 32); }

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <bool LAST, bool NEE = false, bool MEDIUM = false, bool GLOSSY = false>
__global__ void __launch_bounds__(kQThreads, PT_Q_MIN_BLOCKS) k_bounce_q(const __grid_constant__ BounceParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t lt = (1u << lane) - 1u;
  const float4* const fs = reinterpret_cast<const float4*>(smem_raw);
  stage_filt(P.filt, 0, P.filt.end[3], reinterpret_cast<float4*>(smem_raw));
  __syncthreads();  // the only CTA-wide barrier
  QWarp& Q = reinterpret_cast<QWarp*>(smem_raw + P.q_offset)[threadIdx.x >> 5];
  const DepthIO io = depth_io(P);

  const uint32_t n_in = P.ctrl->count[P.depth];
  const uint32_t n_units = (n_in + kUnit - 1) / kUnit;
  uint32_t* const ticket = &P.ctrl->tile_ctr[P.depth];
  uint32_t next_raw = 0;  // lane 0: the ticket taken ahead of time
  if (lane == 0) next_raw = atom_add_u32(ticket, 1u);

#if PT_Q_DEFER_OUT
  DeferredOut W;
  W.stage = Q.wst; W.pend_raw = 0; W.pend_n = 0;
#endif
  uint32_t ns = 0, nc = 0;           // queue lengths (warp-uniform): spheres at [0, ns), cubes at [kQCap - nc, kQCap)
  uint32_t unit = 0, unit_end = 0;   // units left of the current ticket
  bool more = true;                  // the ticket counter has not run dry yet
  // the unit phase A works on next: taken from the ticket at hand or from the next ticket; with PT_Q_PREFETCH its path
  // state is requested at once, so that it arrives while the unit before it is traced
  auto advance = [&]() {
    if (unit == unit_end) {
      const uint32_t unit0 = __shfl_sync(0xffffffffu, next_raw, 0) * kTicketUnits;
      if (unit0 >= n_units) { more = false; return; }
      if (lane == 0) next_raw = atom_add_u32(ticket, 1u);  // consumed a ticket's worth of work later: its latency is hidden
      unit = unit0;
      unit_end = min(unit0 + kTicketUnits, n_units);
    }
#if PT_Q_PREFETCH
    const uint32_t idc = min(unit * kUnit + lane, n_in - 1u);  // lanes past the end fetch a copy of the last path
    cp_async16(&Q.st[0][lane], P.in_o + idc);
    cp_async16(&Q.st[1][lane], P.in_d + idc);
    cp_async16(&Q.st[2][lane], P.in_t + idc);
    cp_async_commit();
#endif
  };
  advance();
  for (;;) {
    // ---- phase B: full batches (every entry once the input is exhausted) ----
    for (;;) {
      const uint32_t need = more ? (uint32_t)kUnit : 1u;
      uint32_t n, slot0;
      int type;
      if (ns >= need) { type = 0; n = min(ns, (uint32_t)kUnit); ns -= n; slot0 = ns; }
      else if (nc >= need) { type = 1; n = min(nc, (uint32_t)kUnit); nc -= n; slot0 = kQCap - n - nc; }
      else break;
      // lanes beyond a partial batch (the final flush only) work on a copy of its first entry and are masked out below:
      // no defaults to set up, no divergence
      const bool valid = lane < n;
      const uint32_t slot = slot0 + (valid ? lane : 0u);
      PT_CHECK(slot < (uint32_t)kQCap && n >= 1u && n <= (uint32_t)kUnit);
      const float4 a = Q.o[slot], b = Q.d[slot];
      f3 o = mk(a.x, a.y, a.z), d = mk(b.x, b.y, b.z);
      const uint32_t pixel = __float_as_uint(a.w), sample = __float_as_uint(b.w);
      const float4 e = Q.c[slot];
      const int gi = __float_as_int(e.y);
      const float lo2 = e.x;
      Hit h;
      DeferredGuard m;  // (an argument outside the fast paths' range sends the lane to the exact scan, which guards every call)
      const bool hit = exact_hit(type, __ldg(P.g.inv0 + gi), __ldg(P.g.inv1 + gi), __ldg(P.g.inv2 + gi), __ldg(P.g.fwd0 + gi),
                                 __ldg(P.g.fwd1 + gi), __ldg(P.g.fwd2 + gi), o, d, h.t, h.p, h.ncode, m);
      h.id = gi;
      if (m.bad || !(hit && h.t > 0 && h.t < lo2)) {
        // the candidate is not confirmed: the exact scan decides (0.008 % of the segments on the sample scene)
        h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
        if (valid) {
          closest_hit_exact(P.g, P.n_geoms, o, d, h);
          atomicAdd(&P.ctrl->fallbacks, 1u);
        }
      }
      // the throughput is fetched only now: it is not needed before shading, and the exact test is where registers are scarce
      const float4 c = Q.t[slot];
      f3 thr = mk(c.x, c.y, c.z);
      const float cos_b = NEE ? c.w : 0.0f;
      __syncwarp();  // the popped entries are in registers: the next push may overwrite them
#if PT_Q_DEFER_OUT
      shade_and_compact<LAST, true, NEE, true, true, MEDIUM, GLOSSY>(P, io, fs, lane, valid && h.id >= 0, h, o, d, thr, pixel, sample, cos_b, &W);
#else
      shade_and_compact<LAST, true, NEE, false, true, MEDIUM, GLOSSY>(P, io, fs, lane, valid && h.id >= 0, h, o, d, thr, pixel, sample, cos_b);
#endif
    }
    if (!more) break;
    // ---- phase A: load, filter scan, push the candidates ----
    {
      const uint32_t idx = unit * kUnit + lane;
      unit++;
      const bool valid = idx < n_in;
#if PT_Q_PREFETCH
      cp_async_wait_all();  // every lane reads only the slots it requested itself
      const float4 a = Q.st[0][lane], b = Q.st[1][lane];
      float4 c = Q.st[2][lane];
#if PT_Q_PREFETCH_EARLY
      advance();  // this lane's staging slots are free again: the next unit's rows travel during this unit's scan as well
#endif
#else
      const uint32_t idc = valid ? idx : n_in - 1u;  // (n_in >= 1 here) lanes past the end scan a copy of the last path
      const float4 a = __ldcs(P.in_o + idc), b = __ldcs(P.in_d + idc);
      float4 c = __ldcs(P.in_t + idc);
#endif
      ScanBest best;
      scan_init(best);
      const ScanRay ray = make_scan_ray(mk(a.x, a.y, a.z), mk(b.x, b.y, b.z), P.filt.r_scene, P.filt.end[2] > P.filt.end[1]);
      filter_scan(fs, 0, P.filt.end[3], P.filt.end, ray, best);
      const bool cand = valid && best.k1 >= 0;
      const bool sphere = best.k1 < 2 * P.filt.end[1];
      const uint32_t bs = __ballot_sync(0xffffffffu, cand && sphere), bc = __ballot_sync(0xffffffffu, cand && !sphere);
      if (cand) {
        const int gi = __ldg(reinterpret_cast<const int*>(P.filt.ids) + best.k1);
        const uint32_t slot = sphere ? ns + __popc(bs & lt) : kQCap - 1 - (nc + __popc(bc & lt));
        PT_CHECK(slot < (uint32_t)kQCap && ns + nc + __popc(bs) + __popc(bc) <= (uint32_t)kQCap);
        PT_CHECK(idx < P.cap && gi >= 0 && gi < P.n_geoms);
        Q.o[slot] = a; Q.d[slot] = b;
        Q.t[slot] = c;
        Q.c[slot] = make_float4(best.lo2, __int_as_float(gi), __uint_as_float(idx), 0.0f);
      }
      ns += __popc(bs);
      nc += __popc(bc);
#if !(PT_Q_PREFETCH && PT_Q_PREFETCH_EARLY)
      advance();  // (the staged rows of this unit are in registers / in the queue by now)
#endif
      __syncwarp();
    }
  }
#if PT_Q_DEFER_OUT
  if (!LAST) deferred_flush(W, P, io, lane);  // the last batch's survivors
#endif
}

// Many geoms (BASELINE config "10k spheres/cubes"): the hierarchy of pt_bvh.cuh, read through L1/L2.  A ray's
// traversal takes anything from a handful to hundreds of steps, and neighbouring paths stop being neighbours in space
// after the first bounce, so a warp that walked 32 rays in lock step kept 9 of its 32 lanes busy on average
// (profiles/r01_bvh_v1_metrics.txt).  Work decomposition here, per warp:
//   a POOL of up to kPool consecutive paths is taken from the wavefront's counter (fewer towards the end of the
//   wavefront, so that the warps finish together);
//   phase 1  filter traversal of the pool: every lane walks one ray at a time and, when it is done, takes the next ray
//            of the pool, read from the wavefront's buffers right there (depth 0: k_raygen_wf wrote them); lanes are
//            refilled once kRefillMin of them are idle, so the refill code runs rarely.  The result of a ray -- two
//            candidate leaves and two bounds, 16 bytes -- goes to HBM: a pool costs no shared memory, so it can be long.
//            A pool ends with a tail in which the last long traversals run alone, and that tail is paid once per pool
//            (pools of 128 rays held in shared memory: 43 % of a warp's steps fell into tails; profiles/r02_bvh_notes.txt);
//   phase 2  unit by unit, all 32 lanes together: the rays once more (coalesced this time), exact test of each path's
//            candidate k1 and, where that does not settle the path, of k2 (bvh_resolve2), shading, compaction -- as in
//            k_bounce.  A path that two candidates do not settle (~0.1 %) is NOT traversed exactly on the spot -- that
//            would occupy the warp with one or two live lanes for a whole traversal -- but DEFERRED: its index goes to a
//            per-warp list, and whenever 32 have gathered they are run as a unit of their own (run_deferred).
#ifndef PT_BVH_POOL_UNITS
#define PT_BVH_POOL_UNITS 32
#endif
#ifndef PT_BVH_POOL_MIN_UNITS
#define PT_BVH_POOL_MIN_UNITS 4
#endif
#ifndef PT_BVH_REFILL_MIN
#define PT_BVH_REFILL_MIN 8
#endif
#ifndef PT_BVH_SMEM_STACK
#define PT_BVH_SMEM_STACK 0  // levels of a lane's traversal stack held in shared memory (pt_bvh.cuh: TravStack)
#endif
constexpr int kPoolUnits = PT_BVH_POOL_UNITS, kPool = kPoolUnits * kUnit, kPoolMin = PT_BVH_POOL_MIN_UNITS * kUnit;
constexpr int kRefillMin = PT_BVH_REFILL_MIN, kDeferCap = 2 * kUnit, kSmemStack = PT_BVH_SMEM_STACK;
#ifndef PT_BVH_THREADS
#define PT_BVH_THREADS 256
#endif
#ifndef PT_BVH_MIN_BLOCKS
#define PT_BVH_MIN_BLOCKS 4  // 64 registers, 32 resident warps per SM: +3 % over 3 x 80 registers (the kernel waits on node fetches)
#endif
constexpr int kBvhThreads = PT_BVH_THREADS;
struct BvhWarpSmem {
  uint32_t defer[kDeferCap];     // paths (index into the wavefront's input) waiting for the exact traversal
  StackEnt stk[kSmemStack > 0 ? kSmemStack * kUnit : 1];  // the lanes' traversal stacks, lowest levels
};
constexpr size_t kBvhSmemBytes = sizeof(BvhWarpSmem) * (kBvhThreads / 32);

// Depth 0 of a many-geom scene: the primary rays are GENERATED by a kernel of their own into the wavefront's input
// buffers (free at depth 0) and k_bounce_bvh then traces every depth alike.  96 bytes of HBM traffic per path -- 1.5 % of
// what the wavefront takes -- buy a traversal loop without the ray generator in its instruction footprint (generated in
// the loop's refill branch: 40 % of the stall samples were instruction fetches) and long pools at depth 0 as well.
__global__ void __launch_bounds__(256) k_raygen_wf(const __grid_constant__ BounceParams P) {
  if (blockIdx.x == 0 && threadIdx.x == 0) P.ctrl->count[0] = P.n_first;
  float4* const wo = const_cast<float4*>(P.in_o);
  float4* const wd = const_cast<float4*>(P.in_d);
  float4* const wt = const_cast<float4*>(P.in_t);
  for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < P.n_first; idx += gridDim.x * blockDim.x) {
    PT_CHECK(idx < P.cap);
    const uint32_t si = fastdiv(idx, P.div_band);
    const uint32_t pixel = P.pix0 + (idx - si * P.band), sample = P.first_sample + si;
    f3 o, d;
    raygen(P.cam, P.keys, pixel, sample, o, d);
    wo[idx] = make_float4(o.x, o.y, o.z, __uint_as_float(pixel));
    wd[idx] = make_float4(d.x, d.y, d.z, __uint_as_float(sample));
    wt[idx] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);  // throughput 1, no diffuse bounce behind the path
  }
}

// a path of the wavefront's input: ray, pixel, sample
__device__ __forceinline__ void load_path(const BounceParams& P, uint32_t idx, f3& o, f3& d, uint32_t& pixel, uint32_t& sample) {
  const float4 a = __ldg(P.in_o + idx), b = __ldg(P.in_d + idx);
  o = mk(a.x, a.y, a.z); pixel = __float_as_uint(a.w);
  d = mk(b.x, b.y, b.z); sample = __float_as_uint(b.w);
}

// shading + compaction of one unit of k_bounce_bvh: ONE copy of the code for the pool's units and the deferred units
// (the kernel's instruction footprint is what its warps wait for at depth 0: profiles/r02_bvh_notes.txt)
#ifndef PT_BVH_TABLE
#define PT_BVH_TABLE 0  // normals, tangent frames and the material row from the per-geom table, as in the few-geom kernels
#endif
template <bool LAST, bool NEE, bool MEDIUM, bool GLOSSY>
__device__ __noinline__ void shade_unit_bvh(const BounceParams& P, const DepthIO& io, uint32_t lane, bool hit, const Hit& h, f3 o, f3 d,
                                            f3 thr, uint32_t pixel, uint32_t sample, float cos_b) {
  shade_and_compact<LAST, PT_BVH_TABLE != 0, NEE, false, false, MEDIUM, GLOSSY>(P, io, nullptr, lane, hit, h, o, d, thr, pixel, sample, cos_b);
}

// `n` (<= 32, warp-uniform) deferred paths, taken from the top of the warp's list: paths whose two nearest candidates
// did not settle the closest hit (a third geom is in the way: ~0.1 % of the segments) go through the EXACT traversal --
// every candidate leaf along the ray that can still matter is tested exactly -- all lanes together, then shading and
// compaction as a unit of their own.
template <bool LAST, bool NEE, bool MEDIUM, bool GLOSSY>
__device__ __noinline__ void run_deferred(const BounceParams& P, const uint32_t* list, uint32_t n) {
  const uint32_t lane = threadIdx.x & 31u;
  const DepthIO io = depth_io(P);
  const bool valid = lane < n;
  f3 o = mk(0, 0, 0), d = mk(0, 0, 1), thr = mk(1, 1, 1);
  uint32_t pixel = 0, sample = 0;
  float cos_b = 0.0f;
  Hit h;
  h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
  if (valid) {
    const uint32_t idx = list[lane];
    load_path(P, idx, o, d, pixel, sample);
    { const float4 c = __ldg(P.in_t + idx); thr = mk(c.x, c.y, c.z); cos_b = NEE ? c.w : 0.0f; }
    bvh_exact(P.bvh, P.g, o, d, P.filt.r_scene, h);
  }
  if (lane == 0) atomicAdd(&P.ctrl->fallbacks, n);  // statistics: segments that needed the exact traversal
  shade_unit_bvh<LAST, NEE, MEDIUM, GLOSSY>(P, io, lane, valid && h.id >= 0, h, o, d, thr, pixel, sample, cos_b);
}

// the next pool of a warp: kPool paths while plenty are left, fewer (down to kPoolMin) when the wavefront runs out, so
// that the warps finish together.  Returns false when the wavefront is exhausted.  (`ticket` counts PATHS.)
__device__ __forceinline__ bool bvh_take_pool(uint32_t* ticket, uint32_t n_in, uint32_t n_warps, uint32_t lane, uint32_t& base, uint32_t& n_pool) {
  uint32_t chunk = 0;
  base = 0;
  if (lane == 0) {
    const uint32_t seen = *reinterpret_cast<volatile uint32_t*>(ticket);  // (a little stale: only sizes the chunk)
    chunk = kPool;
    if (seen < n_in) {
      const uint32_t fair = ((n_in - seen) / (2u * n_warps)) & ~(kUnit - 1u);
      chunk = min((uint32_t)kPool, max((uint32_t)kPoolMin, fair));
    }
    base = atom_add_u32(ticket, chunk);
  }
  base = __shfl_sync(0xffffffffu, base, 0);
  chunk = __shfl_sync(0xffffffffu, chunk, 0);
  if (base >= n_in) return false;
  n_pool = min(chunk, n_in - base);
  return true;
}

// phase 1 of a pool: filter traversal of paths [base, base + n_pool); the result of every path to P.bvh_res
// (SHADOW: the rays are the entries of the shadow queue, some of which are empty)
template <bool SHADOW = false>
__device__ __forceinline__ void bvh_phase1(const BounceParams& P, BvhWarpSmem& S, uint32_t lane, uint32_t n_in, uint32_t base, uint32_t n_pool) {
  {
    uint32_t next = 0;  // warp-uniform: first ray of the pool nobody has taken yet
    int ray = -1;       // this lane's ray, -1 = idle
    ScanRay r;
    TravRay tr;
    ScanBest best;
    StackEnt ov[kBvhStack - kSmemStack];
    TravStack<kSmemStack> st;
    st.sm = S.stk + lane; st.ov = ov;
    int cur = 0;
    r = make_scan_ray(mk(0, 0, 0), mk(0, 0, 1), 0.0f, true);
    tr = make_trav_ray(P.bvh, r);
    scan_init(best);
    for (;;) {
      const uint32_t idle = __ballot_sync(0xffffffffu, ray < 0);
      if (idle) {
        if (next < n_pool && (__popc(idle) >= kRefillMin || idle == 0xffffffffu)) {
          const uint32_t j = next + __popc(idle & ((1u << lane) - 1u));
          if (ray < 0 && j < n_pool) {
            ray = (int)j;
            f3 o, d;
            uint32_t pixel, sample;
            float reach = INFINITY;  // SHADOW: nothing beyond the sampled point of the light can change what the ray decides
            if (SHADOW) {
              const float4 x = __ldg(P.sq_x + base + j);
              if (__float_as_int(x.z) < 0) ray = -1;  // an empty entry: nothing to trace
              reach = __fmaf_rn(x.x, 1.002f, 2e-3f);
            }
            if (ray >= 0) {
            load_path(P, base + j, o, d, pixel, sample);
            r = make_scan_ray(o, d, P.filt.r_scene, true);
            tr = make_trav_ray(P.bvh, r);
            scan_init(best);
            // A shadow ray asks one thing: is its closest hit the light, at the sampled point's distance dy (within
            // 1e-3 dy + 1e-3)?  A light that is hit is hit no farther than the point sampled on its surface, so geoms whose
            // bound exceeds dy (1 + 2e-3) + 2e-3 cannot be that hit nor hide it: the traversal treats them like geoms
            // behind a sure hit.
            if (SHADOW) best.hi = reach;
            st.sp = 0;
            cur = bvh_root(P.bvh);
            }
          }
          next += __popc(idle);
          // the rays the next refill will take: on their way into L1 meanwhile (4 lines each of origins and directions)
          if (lane < 8u) {
            const uint32_t q = base + next + (lane & 3u) * 8u;
            if (q < n_in) asm volatile("prefetch.global.L1 [%0];" ::"l"((lane < 4u ? P.in_o : P.in_d) + q));
          }
        } else if (idle == 0xffffffffu) {
          break;
        }
      }
#ifdef PT_BVH_STACK_HIST
      {
        const uint32_t act = __ballot_sync(0xffffffffu, ray >= 0), atn = __ballot_sync(0xffffffffu, ray >= 0 && cur >= 0);
        if (lane == 0) {
          atomicAdd(&g_sp_hist[45], (unsigned long long)__popc(act));
          atomicAdd(&g_sp_hist[46], 1ull);
          if (next >= n_pool) { atomicAdd(&g_sp_hist[47], 1ull); atomicAdd(&g_sp_hist[48], (unsigned long long)__popc(act)); }
          atomicAdd(&g_sp_hist[49], (unsigned long long)__popc(atn));
        }
      }
#endif
      if (ray >= 0 && !filter_step(P.bvh, r, tr, best, cur, st)) {
        PT_CHECK(base + (uint32_t)ray < P.cap && best.k1 < P.bvh.n_leaves && best.k2 < P.bvh.n_leaves);
        P.bvh_res[base + (uint32_t)ray] = make_float4(best.lo2, best.lo3, __int_as_float(best.k1), __int_as_float(best.k2));
        ray = -1;
      }
    }
  }
}

// The closest hit of a path from the filter traversal's result res = (lo2, lo3, k1, k2), all lanes of a warp together:
// the nearest candidate k1 is tested exactly (k1 < 0: every geom is a proven miss) and decides if it reports a hit closer
// than lo2; where it does not, the second candidate joins in and the closer exact result wins if it is closer than lo3
// (every other geom is a proven miss or no closer than its bound >= lo3).  Returns true if that does not settle it
// either (a third geom is in the way): the caller runs the exact traversal.  `h` is filled in when a hit is settled.
__device__ __forceinline__ bool bvh_resolve2(const BounceParams& P, uint32_t lane, float4 res, f3 o, f3 d, Hit& h) {
  const float lo2 = res.x, lo3 = res.y;
  const int k1 = __float_as_int(res.z), k2 = __float_as_int(res.w);
  Hit e1;
  e1.t = INFINITY; e1.id = -1; e1.p = mk(0, 0, 0); e1.ncode = 0;
  bool hit1 = false, defer = false;
  if (k1 >= 0) hit1 = exact_leaf_call(k1, P.bvh, P.g, o, d, e1);
  const bool settled1 = k1 < 0 || (hit1 && e1.t < lo2) || (!hit1 && k2 < 0);
  if (hit1 && e1.t < lo2) h = e1;
  if (__any_sync(0xffffffffu, !settled1)) {
    if (!settled1) {
      Hit e2;
      const bool hit2 = exact_leaf_call(k2, P.bvh, P.g, o, d, e2);
      const bool second = hit2 && (!hit1 || e2.t < e1.t || (e2.t == e1.t && e2.id < e1.id));
      if (hit1 || hit2) {
        if (second) e1 = e2;
        if (e1.t < lo3) h = e1; else defer = true;
      } else {
        defer = lo3 < INFINITY;  // two misses: settled unless a third geom is a candidate
      }
    }
    const uint32_t n2 = __popc(__ballot_sync(0xffffffffu, !settled1 && !defer));
    if (lane == 0 && n2) atomicAdd(&P.ctrl->retries, n2);  // statistics: segments the second candidate settled
  }
  return defer;
}

// phase 2 of a pool: exact test of the candidates, shading, compaction, unit by unit; paths that two candidates do not
// settle go to the warp's list for the exact traversal, which is run whenever the list holds a unit's worth
template <bool LAST, bool NEE, bool MEDIUM, bool GLOSSY>
__device__ __forceinline__ void bvh_phase2(const BounceParams& P, const DepthIO& io, BvhWarpSmem& S, uint32_t lane, uint32_t base, uint32_t n_pool,
                                           uint32_t& n_defer) {
#pragma unroll 1
  for (uint32_t j0 = 0; j0 < n_pool; j0 += kUnit) {
    const uint32_t j = j0 + lane;
    const bool valid = j < n_pool;
    f3 o = mk(0, 0, 0), d = mk(0, 0, 1), thr = mk(1, 1, 1);
    uint32_t pixel = 0, sample = 0;
    float cos_b = 0.0f;
    Hit h;
    h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
    float4 res = make_float4(INFINITY, INFINITY, __int_as_float(-1), __int_as_float(-1));
    if (valid) {
      load_path(P, base + j, o, d, pixel, sample);
      res = P.bvh_res[base + j];  // (written by this warp: ordered by the __syncwarp after phase 1)
      { const float4 c = __ldcs(P.in_t + base + j); thr = mk(c.x, c.y, c.z); cos_b = NEE ? c.w : 0.0f; }
    }
    const bool defer = bvh_resolve2(P, lane, res, o, d, h);  // neither candidate settles it: the exact traversal decides (run_deferred)
    const uint32_t dmask = __ballot_sync(0xffffffffu, defer);
    PT_CHECK(n_defer + __popc(dmask) <= (uint32_t)kDeferCap);
    if (defer) S.defer[n_defer + __popc(dmask & ((1u << lane) - 1u))] = base + j;
    n_defer += __popc(dmask);
    shade_unit_bvh<LAST, NEE, MEDIUM, GLOSSY>(P, io, lane, valid && !defer && h.id >= 0, h, o, d, thr, pixel, sample, cos_b);
    if (n_defer >= kUnit) {
      __syncwarp();
      n_defer -= kUnit;
      run_deferred<LAST, NEE, MEDIUM, GLOSSY>(P, S.defer + n_defer, kUnit);
      __syncwarp();
    }
  }
}

// (Traversal and exact test + shading as two kernels were measured: the traversal loop alone fits 48 registers only with
// spills, and at 64 it takes as long as this kernel takes for both phases -- in one kernel the arithmetic of the warps in
// phase 2 fills the issue slots that the warps in phase 1 leave while they wait for nodes: 2.51 vs 3.00 Gseg/s.)
template <bool LAST, bool NEE = false, bool MEDIUM = false, bool GLOSSY = false>
__global__ void __launch_bounds__(kBvhThreads, PT_BVH_MIN_BLOCKS) k_bounce_bvh(const __grid_constant__ BounceParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const uint32_t lane = threadIdx.x & 31u;
  BvhWarpSmem& S = reinterpret_cast<BvhWarpSmem*>(smem_raw)[threadIdx.x >> 5];
  const DepthIO io = depth_io(P);
  const uint32_t n_in = P.ctrl->count[P.depth];  // (depth 0: set by k_raygen_wf)
  const uint32_t n_warps = gridDim.x * (kBvhThreads / 32);
  uint32_t n_defer = 0;  // warp-uniform
  uint32_t base, n_pool;
  while (bvh_take_pool(&P.ctrl->tile_ctr[P.depth], n_in, n_warps, lane, base, n_pool)) {
    bvh_phase1(P, S, lane, n_in, base, n_pool);
    __syncwarp();  // (the pool's results were written by this warp: ordered for its other lanes)
    bvh_phase2<LAST, NEE, MEDIUM, GLOSSY>(P, io, S, lane, base, n_pool, n_defer);
  }
  if (n_defer) {
    __syncwarp();
    run_deferred<LAST, NEE, MEDIUM, GLOSSY>(P, S.defer, n_defer);
  }
}

// ---- the shadow rays of direct light sampling, one launch per depth behind the depth's bounce launch ----
// P.in_o / P.in_d point at the queue's (origin | pixel) / (direction | sample) rows, P.depth names the queue.
// Few geoms: a unit of 32 queued rays per warp -- filter scan, exact test of the winner, visibility, contribution: the
// closest hit of direct_light's former inline trace, bit for bit, with all lanes busy.
constexpr int kShadowQ = 2 * kUnit;  // per warp: indices of queued shadow rays waiting for a full unit
__host__ __device__ inline size_t shadow_lin_smem(size_t geom_smem) { return geom_smem + (size_t)(kBounceThreads / 32) * kShadowQ * sizeof(uint32_t); }
__device__ __forceinline__ void shadow_trace_lin(const BounceParams& P, const float4* fs, uint32_t idx) {
  const float4 a = __ldcs(P.in_o + idx), b = __ldcs(P.in_d + idx), c = __ldcs(P.sq_t + idx), x = __ldcs(P.sq_x + idx);
  const f3 o = mk(a.x, a.y, a.z), wd = mk(b.x, b.y, b.z);
  Hit h;
  h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
  closest_hit_one<true>(P, fs, o, wd, h);
  shadow_resolve<true>(P, h, wd, mk(c.x, c.y, c.z), c.w, x.x, x.y, __float_as_int(x.z), __float_as_uint(a.w), __float_as_uint(b.w));
}
__global__ void __launch_bounds__(kBounceThreads, PT_MIN_BLOCKS) k_shadow_lin(const __grid_constant__ BounceParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const float4* const fs = reinterpret_cast<const float4*>(smem_raw);
  stage_filt(P.filt, 0, P.filt.end[3], reinterpret_cast<float4*>(smem_raw));
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t* const q = reinterpret_cast<uint32_t*>(smem_raw + P.q_offset) + (threadIdx.x >> 5) * kShadowQ;
  const uint32_t n = P.ctrl->count[P.depth + 1];  // entry i of the queue belongs to path i of the next depth's wavefront
  const uint32_t n_units = (n + kUnit - 1) / kUnit;
  uint32_t* const ticket = &P.ctrl->shadow_ctr[P.depth];
  uint32_t nq = 0;  // warp-uniform: indices waiting in q (< 32 between units)
  for (;;) {
    uint32_t t = 0;
    if (lane == 0) t = atom_add_u32(ticket, 1u);
    const uint32_t unit0 = __shfl_sync(0xffffffffu, t, 0) * kTicketUnits;
    if (unit0 >= n_units) break;
    const uint32_t unit_end = min(unit0 + kTicketUnits, n_units);
    // (the ticket's flags are requested together: one wait for HBM per ticket instead of one per unit)
    uint32_t has_bits = 0;
#pragma unroll
    for (uint32_t k = 0; k < kTicketUnits; k++) {
      const uint32_t idx = (unit0 + k) * kUnit + lane;
      const int gl = idx < n ? __float_as_int(__ldcs(&P.sq_x[idx].z)) : -1;
      has_bits |= (gl >= 0 ? 1u : 0u) << k;
    }
#pragma unroll 1
    for (uint32_t u = unit0; u < unit_end; u++) {
      // the entries of the queue that hold a ray (a path that continued without one left its entry empty) are gathered
      // until 32 are there: the trace below always runs with a full warp
      const uint32_t idx = u * kUnit + lane;
      const bool has = (has_bits >> (u - unit0)) & 1u;
      const uint32_t m = __ballot_sync(0xffffffffu, has);
      PT_CHECK(nq + __popc(m) <= (uint32_t)kShadowQ);
      if (has) q[nq + __popc(m & ((1u << lane) - 1u))] = idx;
      nq += __popc(m);
      __syncwarp();
      if (nq >= kUnit) {
        nq -= kUnit;
        const uint32_t i2 = q[nq + lane];
        __syncwarp();
        shadow_trace_lin(P, fs, i2);
      }
    }
  }
  if (lane < nq) shadow_trace_lin(P, fs, q[lane]);
}
// Many geoms: the queue goes through the pooled filter traversal like a wavefront of paths (bvh_phase1), then unit by
// unit through the two-candidate resolution; the few rays that leaves open take the exact traversal on the spot.
__global__ void __launch_bounds__(kBvhThreads, PT_BVH_MIN_BLOCKS) k_shadow_bvh(const __grid_constant__ BounceParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const uint32_t lane = threadIdx.x & 31u;
  BvhWarpSmem& S = reinterpret_cast<BvhWarpSmem*>(smem_raw)[threadIdx.x >> 5];
  const uint32_t n = P.ctrl->count[P.depth + 1];  // entry i of the queue belongs to path i of the next depth's wavefront
  const uint32_t n_warps = gridDim.x * (kBvhThreads / 32);
  uint32_t base, n_pool;
  while (bvh_take_pool(&P.ctrl->shadow_ctr[P.depth], n, n_warps, lane, base, n_pool)) {
    bvh_phase1<true>(P, S, lane, n, base, n_pool);
    __syncwarp();
#pragma unroll 1
    for (uint32_t j0 = 0; j0 < n_pool; j0 += kUnit) {
      const uint32_t j = j0 + lane;
      const bool valid = j < n_pool;
      f3 o = mk(0, 0, 0), wd = mk(0, 0, 1);
      uint32_t pixel = 0, sample = 0;
      float4 res = make_float4(INFINITY, INFINITY, __int_as_float(-1), __int_as_float(-1));
      Hit h;
      h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
      float4 x = make_float4(0.0f, 0.0f, __int_as_float(-1), 0.0f);
      if (valid) x = __ldcs(P.sq_x + base + j);
      const bool queued = __float_as_int(x.z) >= 0;  // (an empty entry has no ray and no traversal result)
      if (queued) {
        load_path(P, base + j, o, wd, pixel, sample);
        res = P.bvh_res[base + j];
      }
      if (bvh_resolve2(P, lane, res, o, wd, h)) {
        h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
        bvh_exact(P.bvh, P.g, o, wd, P.filt.r_scene, h);
        atomicAdd(&P.ctrl->fallbacks, 1u);
      }
      if (queued) {
        const float4 c = __ldcs(P.sq_t + base + j);
        shadow_resolve<false>(P, h, wd, mk(c.x, c.y, c.z), c.w, x.x, x.y, __float_as_int(x.z), pixel, sample);
      }
    }
    __syncwarp();
  }
}

// live_total[d] += count[d]; one tiny launch per wavefront.  `policy` (mapped host memory, may be null): policy[d] = which
// kernel suits depth d of THIS scene -- 1: k_bounce_q (a good part of the paths ends in the filter scan or on a light, so
// re-batching the rest pays), 2: the fused k_bounce (nearly every path goes on: closed rooms) -- judged by the share
// of depth d-1's paths that reach depth d.  The host reads it when it launches later wavefronts; results do not depend
// on the choice.
constexpr float kQSurvivalMax = 0.93f;
__global__ void k_accum_counts(const WfCtrl* ctrl, unsigned long long* live_total, int max_depth, volatile int* policy) {
  int d = threadIdx.x;
  // atomics: the two wavefront slots run on different streams and may fold their counts at the same time
  if (d < max_depth) atomicAdd(live_total + d, (unsigned long long)ctrl->count[d]);
  if (d == 0) atomicAdd(live_total + kMaxDepth, (unsigned long long)ctrl->fallbacks);
  if (d == 1) atomicAdd(live_total + kMaxDepth + 1, ctrl->shadow);
  if (d == 2) atomicAdd(live_total + kMaxDepth + 2, (unsigned long long)ctrl->retries);
  if (policy && d >= 1 && d < max_depth && ctrl->count[d - 1] >= 4096u)
    policy[d] = (float)ctrl->count[d] < kQSurvivalMax * (float)ctrl->count[d - 1] ? 1 : 2;
}

// the ray-independent part of hit_normal, once per scene: identical instructions, so identical bits
__global__ void k_normal_table(GeomSoA g, int n_geoms, const float4* mats, float4* tab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_geoms) return;
  const float4 f0 = g.fwd0[i], f1 = g.fwd1[i], f2 = g.fwd2[i];
  Hit h;
  h.t = 0.0f; h.id = i; h.p = mk(0, 0, 0);
  for (int face = 0; face < 6; face++) {
    h.ncode = (face % 3) | (face >= 3 ? 4 : 0);
    const f3 n = hit_normal(f0, f1, f2, h);
    tab[(size_t)i * kNormalRows + face] = make_float4(n.x, n.y, n.z, 0.0f);
    // the diffuse sampler's tangent frame for both shading normals of this face (shade(): ns = n or -n)
    f3 p1, p2;
    float4* fr = tab + (size_t)i * kNormalRows + kFrameRow0 + 4 * face;
    hemisphere_frame(n, p1, p2);
    fr[0] = make_float4(p1.x, p1.y, p1.z, 0.0f); fr[1] = make_float4(p2.x, p2.y, p2.z, 0.0f);
    hemisphere_frame(neg(n), p1, p2);
    fr[2] = make_float4(p1.x, p1.y, p1.z, 0.0f); fr[3] = make_float4(p2.x, p2.y, p2.z, 0.0f);
  }
  const f3 c = mulMV(f0, f1, f2, 0.0f, 0.0f, 0.0f, 1.0f);  // intersections.h:111: transform * (0,0,0,1)
  tab[(size_t)i * kNormalRows + 6] = make_float4(c.x, c.y, c.z, 0.0f);
  // the row of the geom's material that decides whether a path ends here (emittance) and how it scatters
  const int2 me = g.meta[i];
  tab[(size_t)i * kNormalRows + kMatRow] = me.x <= 1 ? mats[4 * me.y + 3] : make_float4(0, 0, 0, 0);
}

// ---- parity entry points ----
__global__ void k_raygen_list(RaygenConsts C, uint64_t seed, int n, const uint32_t* pixel, const uint32_t* sample,
                              float* o, float* d) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  f3 oo, dd;
  raygen(C, seed, pixel[i], sample[i], oo, dd);
  o[3 * i] = oo.x; o[3 * i + 1] = oo.y; o[3 * i + 2] = oo.z;
  d[3 * i] = dd.x; d[3 * i + 1] = dd.y; d[3 * i + 2] = dd.z;
}

__global__ void __launch_bounds__(kTile) k_intersect_list(GeomSoA g, int n_geoms, FiltSoA filt, int filt_cap, BvhSoA bvh, const float4* normals, int mode, int n,
                                                          const float* o, const float* d, int* id, float* t, float* p,
                                                          float* nrm, unsigned long long* fallbacks) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < n;
  f3 oo = mk(0, 0, 0), dd = mk(0, 0, 1);
  if (valid) { oo = mk(o[3 * i], o[3 * i + 1], o[3 * i + 2]); dd = mk(d[3 * i], d[3 * i + 1], d[3 * i + 2]); }
  Hit h;
  h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
  if (mode == 1) {  // the exact scan on its own (the specification; what the filtered path must reproduce)
    if (valid) closest_hit_exact(g, n_geoms, oo, dd, h);
  } else if (bvh.n_leaves > 0) {  // many geoms: the hierarchy
    if (valid) {
      const ScanRay ray = make_scan_ray(oo, dd, filt.r_scene, true);
      ScanBest best;
      scan_init(best);
      bvh_traverse<false>(bvh, g, ray, best, h);
      if (resolve_bvh(best, bvh, g, filt.r_scene, oo, dd, h)) atomicAdd(fallbacks, 1ull);
    }
  } else {
    const float4* fs = reinterpret_cast<const float4*>(smem_raw);
    const ScanRay ray = make_scan_ray(oo, dd, filt.r_scene, filt.end[2] > filt.end[1]);
    ScanBest best;
    scan_init(best);
    stage_filt(filt, 0, filt.end[3], reinterpret_cast<float4*>(smem_raw));
    __syncthreads();
    if (valid) filter_scan(fs, 0, filt.end[3], filt.end, ray, best);
    if (valid && resolve_scan(best, filt, g, n_geoms, oo, dd, h)) atomicAdd(fallbacks, 1ull);
  }
  if (!valid) return;
  f3 nn = mk(0, 0, 0);
  if (h.id >= 0) nn = normals ? hit_normal_table(normals, h) : hit_normal(__ldg(g.fwd0 + h.id), __ldg(g.fwd1 + h.id), __ldg(g.fwd2 + h.id), h);
  id[i] = h.id;
  t[i] = h.id >= 0 ? h.t : -1.0f;
  p[3 * i] = h.p.x; p[3 * i + 1] = h.p.y; p[3 * i + 2] = h.p.z;
  nrm[3 * i] = nn.x; nrm[3 * i + 1] = nn.y; nrm[3 * i + 2] = nn.z;
}

// primary rays of (pixel, sample) pairs through depth 0's closest hit (primary_hit): table first, then the filter
__global__ void __launch_bounds__(kTile) k_primary_list(RaygenConsts C, uint64_t seed, GeomSoA g, int n_geoms, FiltSoA filt,
                                                        const float4* normals, const uint32_t* tab, int n, const uint32_t* pixel,
                                                        const uint32_t* sample, int* id, float* t, float* p, float* nrm,
                                                        uint8_t* decided, unsigned long long* fallbacks) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < n;
  stage_filt(filt, 0, filt.end[3], reinterpret_cast<float4*>(smem_raw));
  __syncthreads();
  f3 oo = mk(0, 0, 0), dd = mk(0, 0, 1);
  uint32_t px = 0;
  if (valid) {
    px = pixel[i];
    PT_CHECK(px < C.npix);
    raygen(C, seed, px, sample[i], oo, dd);
  }
  Hit h;
  h.t = INFINITY; h.id = -1; h.p = mk(0, 0, 0); h.ncode = 0;
  bool dec;
  if (primary_hit(tab, reinterpret_cast<const float4*>(smem_raw), filt, g, n_geoms, valid, px, oo, dd, h, dec)) atomicAdd(fallbacks, 1ull);
  if (!valid) return;
  const f3 nn = h.id >= 0 ? hit_normal_table(normals, h) : mk(0, 0, 0);
  id[i] = h.id;
  t[i] = h.id >= 0 ? h.t : -1.0f;
  p[3 * i] = h.p.x; p[3 * i + 1] = h.p.y; p[3 * i + 2] = h.p.z;
  nrm[3 * i] = nn.x; nrm[3 * i + 1] = nn.y; nrm[3 * i + 2] = nn.z;
  decided[i] = dec ? 1 : 0;
}

// ---- stream compaction on its own (README.md:63-70): stable, single pass, decoupled look-back ----
// A tile is 256 threads x 16 elements = 4096 consecutive elements.  Each WARP owns 512 consecutive elements and loads
// them warp-striped -- lane l, step j reads the uint4 (and the 4 flag bytes) at element (j*32 + l)*4 of the warp's chunk
// -- so every load instruction covers 512 contiguous bytes.  Ranks in index order:
//   inside a lane's uint4      prefix of its 4 flags
//   across the lanes of a step  counts 0..4 per lane -> three ballots (one per bit of the count) + popc of the lanes below
//   across the 4 steps / 8 warps running sums; the warps' totals go through shared memory (block scan)
//   across tiles               64-bit status word per tile (epoch | state | value): the tile's aggregate is published as
//                               soon as it is known, warp 0 looks back over 32 predecessors per step until it meets an
//                               inclusive prefix, then publishes its own.  Tiles come from a ticket counter, so every
//                               predecessor is resident and the look-back cannot deadlock; the epoch tag makes clearing
//                               the status words between launches unnecessary.
// Kept elements are written straight to out[prefix + rank]: a lane's (up to 4) elements are adjacent and the lanes'
// ranges abut, so the sectors are filled within the warp.  HBM-bound: 5 B read per element + 4 B written per kept one.
#ifndef PT_COMPACT_THREADS
#define PT_COMPACT_THREADS 256
#endif
constexpr int kCompactThreads = PT_COMPACT_THREADS;
constexpr int kCompactItems = 16;                                // elements per thread
constexpr int kCompactTile = kCompactThreads * kCompactItems;    // 4096 elements per tile
#ifndef PT_COMPACT_BLOCKS
#define PT_COMPACT_BLOCKS (2048 / PT_COMPACT_THREADS)  // resident CTAs per SM: the kernel is latency-bound (one HBM and one L2 round trip per tile)
#endif
__global__ void __launch_bounds__(kCompactThreads, PT_COMPACT_BLOCKS) k_compact_u32(const uint32_t* __restrict__ values, const uint8_t* __restrict__ flags,
                                                       uint32_t n, uint32_t* __restrict__ out, uint32_t* n_out,
                                                       uint32_t* ticket, uint64_t* status, uint32_t epoch) {
  __shared__ uint32_t s_tile;
  __shared__ uint32_t s_warp[kCompactThreads / 32];  // per-warp totals, then exclusive offsets inside the tile
  __shared__ uint32_t s_base;              // exclusive prefix of the tile
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  const uint32_t n_tiles = (n + kCompactTile - 1) / kCompactTile;
  const bool aligned = (reinterpret_cast<uintptr_t>(values) & 15u) == 0 && (reinterpret_cast<uintptr_t>(flags) & 3u) == 0;
  for (;;) {
    __syncthreads();  // s_tile / s_warp / s_base of the previous tile are no longer read
    // (a ticket taken ahead of time would delay that tile's aggregate by a whole tile and stall every successor: measured -30 %)
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    if (tile >= n_tiles) break;
    const uint32_t chunk = tile * kCompactTile + warp * (32 * kCompactItems);  // first element of this warp's 512
    uint4 v[4];
    uint32_t f[4];       // 4 flag bytes per step, normalised to 0 / 1 per byte
    uint32_t cnt[4];     // kept elements of this lane in step j
    uint32_t before[4];  // kept elements of the warp before this lane's uint4 of step j
    uint32_t run = 0;    // running total of the warp over the steps
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t e = chunk + (j * 32 + lane) * 4;  // first of this lane's 4 elements
      uint32_t fb = 0;
      if (e + 4 <= n && aligned) {
        v[j] = __ldcs(reinterpret_cast<const uint4*>(values + e));
        fb = __ldcs(reinterpret_cast<const uint32_t*>(flags + e));
      } else {  // the ragged end of the input (or unaligned pointers): element by element
        uint32_t t[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < 4; k++)
          if (e + k < n) { t[k] = values[e + k]; fb |= (uint32_t)flags[e + k] << (8 * k); }
        v[j] = make_uint4(t[0], t[1], t[2], t[3]);
      }
      // byte != 0 -> 1, per byte (no carries across bytes: 0x7f + 0x7f < 0x100)
      f[j] = ((((fb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | fb) & 0x80808080u) >> 7;
      cnt[j] = (f[j] * 0x01010101u) >> 24;  // sum of the four bytes
      const uint32_t b0 = __ballot_sync(0xffffffffu, cnt[j] & 1u), b1 = __ballot_sync(0xffffffffu, cnt[j] & 2u),
                     b2 = __ballot_sync(0xffffffffu, cnt[j] & 4u);
      before[j] = run + __popc(b0 & lt) + 2u * __popc(b1 & lt) + 4u * __popc(b2 & lt);
      run += __popc(b0) + 2u * __popc(b1) + 4u * __popc(b2);
    }
    if (lane == 0) s_warp[warp] = run;
    __syncthreads();
    if (warp == 0) {
      const uint32_t c = lane < kCompactThreads / 32 ? s_warp[lane] : 0u;
      uint32_t incl = c;  // inclusive scan over the warps' totals
#pragma unroll
      for (int o = 1; o < kCompactThreads / 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)lane >= o) incl += t;
      }
      const uint32_t total = __shfl_sync(0xffffffffu, incl, kCompactThreads / 32 - 1);
      const uint32_t excl = lookback_exclusive(status, tile, epoch, total);
      if (lane < kCompactThreads / 32) s_warp[lane] = incl - c;
      if (lane == 0) {
        s_base = excl;
        if (tile == n_tiles - 1) *n_out = excl + total;
      }
    }
    __syncthreads();
    const uint32_t base = s_base + s_warp[warp];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      uint32_t pos = base + before[j];
      PT_CHECK(pos + ((f[j] * 0x01010101u) >> 24) <= n);
      if (f[j] & 0x00000001u) out[pos++] = v[j].x;
      if (f[j] & 0x00000100u) out[pos++] = v[j].y;
      if (f[j] & 0x00010000u) out[pos++] = v[j].z;
      if (f[j] & 0x01000000u) out[pos++] = v[j].w;
    }
  }
}

// ---- the same compaction with the ordered prefix taken out of the streaming kernels (three launches) ----
// k_compact_u32 keeps every resident CTA waiting in its look-back until the prefix wave reaches it, with no loads in
// flight meanwhile: it streams at 31-41 % of the HBM copy peak (profiles/r01_compact_u32.txt).  Here the dependency
// between tiles is confined to a tiny kernel over the tiles' aggregates:
//   k_compact_count    flags only (1 B per element): kept elements per 4096-element tile
//   k_compact_scan     exclusive prefix over the tile aggregates: 1024 aggregates per CTA, block scan, decoupled look-back
//                      across the CTAs (at most 1024 CTAs for 2^32 elements: all resident)
//   k_compact_scatter  values + flags again, ranks inside the tile exactly as k_compact_u32 computes them, base from the
//                      prefix array: no CTA ever waits for another
// Traffic 6 B read per element + 4 B written per kept one (the flags are read twice) against 5 + 4 algorithmic.
__device__ __forceinline__ uint32_t flag_bytes_to_bits(uint32_t fb) {  // byte != 0 -> 1, per byte
  return ((((fb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | fb) & 0x80808080u) >> 7;
}
__global__ void __launch_bounds__(kCompactThreads) k_compact_count(const uint8_t* __restrict__ flags, uint32_t n, uint32_t n_tiles,
                                                                   uint32_t* __restrict__ tile_count) {
  __shared__ uint32_t s_warp[kCompactThreads / 32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const bool aligned = (reinterpret_cast<uintptr_t>(flags) & 3u) == 0;
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const uint32_t chunk = tile * kCompactTile + warp * (32 * kCompactItems);
    uint32_t cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t e = chunk + (j * 32 + lane) * 4;
      uint32_t fb = 0;
      if (e + 4 <= n && aligned) fb = __ldg(reinterpret_cast<const uint32_t*>(flags + e));  // read again by the scatter: keep it cached
      else
        for (int k = 0; k < 4; k++)
          if (e + k < n) fb |= (uint32_t)flags[e + k] << (8 * k);
      cnt += (flag_bytes_to_bits(fb) * 0x01010101u) >> 24;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) s_warp[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t t = 0;
      for (int w = 0; w < kCompactThreads / 32; w++) t += s_warp[w];
      tile_count[tile] = t;
    }
    __syncthreads();
  }
}
constexpr int kScanThreads = 256, kScanItems = 4, kScanChunk = kScanThreads * kScanItems;
// Chunks are taken from a TICKET counter, not from blockIdx.x: a CTA that looks back at chunk t - 1 then knows that
// chunk's CTA has started (it took its ticket earlier), so the look-back makes progress however few CTAs are resident.
__global__ void __launch_bounds__(kScanThreads) k_compact_scan(const uint32_t* __restrict__ tile_count, uint32_t n_tiles,
                                                               uint32_t* __restrict__ tile_prefix, uint32_t* n_out,
                                                               uint32_t* ticket, uint64_t* status, uint32_t epoch) {
  __shared__ uint32_t s_warp[kScanThreads / 32];
  __shared__ uint32_t s_base, s_chunk;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_chunk = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t chunk = s_chunk;
  const uint32_t first = chunk * kScanChunk + threadIdx.x * kScanItems;
  uint32_t c[kScanItems], mine = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) { c[k] = first + k < n_tiles ? tile_count[first + k] : 0u; mine += c[k]; }
  uint32_t incl = mine;  // inclusive scan over the threads of the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if ((int)lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const uint32_t w = lane < kScanThreads / 32 ? s_warp[lane] : 0u;
    uint32_t wi = w;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if ((int)lane >= o) wi += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, wi, kScanThreads / 32 - 1);
    const uint32_t excl = lookback_exclusive(status, chunk, epoch, total);
    __syncwarp();
    if (lane < kScanThreads / 32) s_warp[lane] = wi - w;
    if (lane == 0) {
      s_base = excl;
      if (chunk == gridDim.x - 1) *n_out = excl + total;
    }
  }
  __syncthreads();
  uint32_t run = s_base + s_warp[warp] + (incl - mine);
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    if (first + k < n_tiles) tile_prefix[first + k] = run;
    run += c[k];
  }
}
__global__ void __launch_bounds__(kCompactThreads, PT_COMPACT_BLOCKS) k_compact_scatter(const uint32_t* __restrict__ values,
                                                                                        const uint8_t* __restrict__ flags, uint32_t n,
                                                                                        uint32_t n_tiles,
                                                                                        const uint32_t* __restrict__ tile_prefix,
                                                                                        uint32_t* __restrict__ out) {
  __shared__ uint32_t s_warp[kCompactThreads / 32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  const bool aligned = (reinterpret_cast<uintptr_t>(values) & 15u) == 0 && (reinterpret_cast<uintptr_t>(flags) & 3u) == 0;
  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const uint32_t chunk = tile * kCompactTile + warp * (32 * kCompactItems);
    uint4 v[4];
    uint32_t f[4], before[4], run = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t e = chunk + (j * 32 + lane) * 4;
      uint32_t fb = 0;
      if (e + 4 <= n && aligned) {
        v[j] = __ldcs(reinterpret_cast<const uint4*>(values + e));
        fb = __ldcs(reinterpret_cast<const uint32_t*>(flags + e));
      } else {
        uint32_t t[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < 4; k++)
          if (e + k < n) { t[k] = values[e + k]; fb |= (uint32_t)flags[e + k] << (8 * k); }
        v[j] = make_uint4(t[0], t[1], t[2], t[3]);
      }
      f[j] = flag_bytes_to_bits(fb);
      const uint32_t cnt = (f[j] * 0x01010101u) >> 24;
      const uint32_t b0 = __ballot_sync(0xffffffffu, cnt & 1u), b1 = __ballot_sync(0xffffffffu, cnt & 2u),
                     b2 = __ballot_sync(0xffffffffu, cnt & 4u);
      before[j] = run + __popc(b0 & lt) + 2u * __popc(b1 & lt) + 4u * __popc(b2 & lt);
      run += __popc(b0) + 2u * __popc(b1) + 4u * __popc(b2);
    }
    __syncthreads();  // s_warp of the previous tile is no longer read
    if (lane == 0) s_warp[warp] = run;
    __syncthreads();
    uint32_t base = __ldg(tile_prefix + tile);
    for (uint32_t w = 0; w < warp; w++) base += s_warp[w];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      uint32_t pos = base + before[j];
      PT_CHECK(pos + ((f[j] * 0x01010101u) >> 24) <= n);
      if (f[j] & 0x00000001u) out[pos++] = v[j].x;
      if (f[j] & 0x00000100u) out[pos++] = v[j].y;
      if (f[j] & 0x00010000u) out[pos++] = v[j].z;
      if (f[j] & 0x01000000u) out[pos++] = v[j].w;
    }
  }
}

// ---- exhaustive self-test of sqrt_ieee / rcp_ieee / inv_sqrt_ieee (pt_device.cuh) against the generic operators ----
// every one of the 2^32 bit patterns; NaN results compare equal to NaN results
__global__ void k_selftest_math(unsigned long long* bad) {
  const uint32_t stride = gridDim.x * blockDim.x;
  unsigned long long b0 = 0, b1 = 0, b2 = 0;
  auto same = [](float u, float v) { return __float_as_uint(u) == __float_as_uint(v) || (u != u && v != v); };
  for (uint64_t k = blockIdx.x * blockDim.x + threadIdx.x; k < (1ull << 32); k += stride) {
    const float x = __uint_as_float((uint32_t)k);
    b0 += !same(sqrt_ieee(x), sqrtf(x));
    b1 += !same(rcp_ieee(x), 1.0f / x);
    b2 += !same(inv_sqrt_ieee(x), 1.0f / sqrtf(x));
  }
  if (b0) atomicAdd(bad + 0, b0);
  if (b1) atomicAdd(bad + 1, b1);
  if (b2) atomicAdd(bad + 2, b2);
}

// ---- sample streaming (pt_stream_*): a group of samples, each traced into an image of its own ("slab") ----
// running means of the group, ahead of the calls that will ask for them: s = base; for each sample j: s += slab_j (one
// binary32 add per component: what the sample's atomic add into the sum would have done), mean_j = s / (spp0 + j) in the
// renderCam->image layout; the sum after the whole group goes to `final` (the base of the next group)
__global__ void k_stream_prefix(const float4* __restrict__ base, const float4* __restrict__ slabs, uint32_t npix, uint32_t group,
                                float spp0, float* __restrict__ means, float4* __restrict__ final) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  float4 a = base[i];
  for (uint32_t j = 0; j < group; j++) {
    const float4 b = __ldcs(slabs + (size_t)j * npix + i);
    a.x = a.x + b.x; a.y = a.y + b.y; a.z = a.z + b.z;
    const float spp = spp0 + (float)j;
    float* m = means + ((size_t)j * npix + i) * 3;
    __stcs(m, a.x / spp); __stcs(m + 1, a.y / spp); __stcs(m + 2, a.z / spp);
  }
  final[i] = a;
}
// the first `count` samples of a group folded into the sum (a stream that ends inside a group)
__global__ void k_stream_apply(float4* sum, const float4* __restrict__ slabs, uint32_t npix, uint32_t count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  float4 a = sum[i];
  for (uint32_t j = 0; j < count; j++) {
    const float4 b = slabs[(size_t)j * npix + i];
    a.x = a.x + b.x; a.y = a.y + b.y; a.z = a.z + b.z;
  }
  sum[i] = a;
}
// sendImageToPBO's bytes (src/raytraceKernel.cu:58-89) of a mean image in the renderCam->image layout
__global__ void k_rgb_to_rgba8(const float* __restrict__ rgb, uint32_t npix, uchar4* out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  float r = rgb[3 * i] * 255.0f, g = rgb[3 * i + 1] * 255.0f, b = rgb[3 * i + 2] * 255.0f;
  if (r > 255) r = 255;
  if (g > 255) g = 255;
  if (b > 255) b = 255;
  uchar4 px;
  px.x = (unsigned char)r; px.y = (unsigned char)g; px.z = (unsigned char)b; px.w = 0;
  out[i] = px;
}

// ---- image out ----
// packed float RGB (renderCam->image layout) = sum * 1 or sum / spp
__global__ void k_resolve_rgb(const float4* accum, uint32_t npix, float spp, int divide, float* rgb) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  float4 a = accum[i];
  if (divide) { a.x = a.x / spp; a.y = a.y / spp; a.z = a.z / spp; }
  rgb[3 * i] = a.x; rgb[3 * i + 1] = a.y; rgb[3 * i + 2] = a.z;
}
__global__ void k_upload_rgb(const float* rgb, uint32_t npix, float4* accum) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  accum[i] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], 0.0f);
}
// sendImageToPBO, src/raytraceKernel.cu:58-89: c = image*255.0; c > 255 -> 255; stored to uchar (truncation), w = 0.
// image*255.0 is a binary64 product of two binary32-representable values rounded to float, which equals the
// binary32 product (double rounding is innocuous for a single multiply).
__global__ void k_resolve_rgba8(const float4* accum, uint32_t npix, float spp, uchar4* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  float4 a = accum[i];
  float r = (a.x / spp) * 255.0f, g = (a.y / spp) * 255.0f, b = (a.z / spp) * 255.0f;
  if (r > 255) r = 255;
  if (g > 255) g = 255;
  if (b > 255) b = 255;
  uchar4 px;
  px.x = (unsigned char)r; px.y = (unsigned char)g; px.z = (unsigned char)b; px.w = 0;
  out[i] = px;
}

}  // namespace ptd
