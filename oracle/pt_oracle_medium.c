/* TEST INFRASTRUCTURE ONLY -- see pt_oracle_medium.h.
 *
 * Subsurface scattering (DESIGN.md 4), the (S) specification of the reference's calculateScatterAndAbsorption stub
 * (src/interactions.h:16-39), as an extension of the C restatement: this file compiles pt_oracle.c together with the
 * pieces below into libpt_oracle_medium.so, so that the restatement's own helpers (Philox addressing, the sphere-direction
 * sampler, Beer-Lambert transmission, the light table) are reused as they are and pt_oracle.c stays the frozen
 * specification of everything else.
 *
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fno-fast-math -fopenmp (oracle/oracle_medium.py), like pt_oracle.c.
 */
#include "pt_oracle.c"
#include "pt_oracle_medium.h"

/* (S) log(x) in binary32 with +,-,* only (Cephes logf): x = m * 2^e through the exponent field, m in [sqrt(1/2),
 * sqrt(2)), f = m - 1 exact, degree-9 polynomial in f, e * ln2 added in two parts (0.693359375 - 2.12194440e-4).  The same
 * operation sequence in the CUDA kernels (log_repro), so free-flight distances are bit-reproducible.  Defined for positive
 * normal x; anything below FLT_MIN (zero, subnormals, negatives, NaN) gives -inf. */
float or_log(float x) {
  if (!(x >= 1.17549435e-38f)) return -INFINITY;
  union { uint32_t u; float f; } b;
  b.f = x;
  int e = (int)(b.u >> 23) - 127;
  b.u = (b.u & 0x007fffffu) | 0x3f800000u; /* m in [1, 2) */
  float m = b.f;
  if (m > 1.41421356f) { m = m * 0.5f; e = e + 1; }
  const float f = m - 1.0f;
  const float z = f * f;
  float p = 7.0376836292e-2f;
  p = p * f - 1.1514610310e-1f;
  p = p * f + 1.1676998740e-1f;
  p = p * f - 1.2420140846e-1f;
  p = p * f + 1.4249322787e-1f;
  p = p * f - 1.6668057665e-1f;
  p = p * f + 2.0000714765e-1f;
  p = p * f - 2.4999993993e-1f;
  p = p * f + 3.3333331174e-1f;
  const float fe = (float)e;
  float y = (p * f) * z;
  y = y + fe * -2.12194440e-4f;
  y = y - 0.5f * z;
  return (f + y) + fe * 0.693359375f;
}

/* (S) calculateScatterAndAbsorption (stub at src/interactions.h:36-39, AbsorptionAndScatteringProperties :16-19) for a
 * homogeneous medium with an isotropic phase function: free-flight distance s = -log(1 - xf) / sigma_s (1 - xf is exact
 * for xf = k * 2^-24); if s < distance the path scatters at s into sphere_dir(xi1, xi2) and is weighted by
 * transmission(sigma_a, s), otherwise it leaves the medium after `distance` with weight transmission(sigma_a, distance) and
 * direction (0, 0, 0).  Returns 1 if it scattered. */
static inline int sample_medium(const float ab[3], float sigma_s, float distance, float xi1, float xi2, float xf, float* s,
                                v3* dir, float w[3]) {
  *s = -or_log(1.0f - xf) / sigma_s;
  if (*s < distance) {
    *dir = sphere_dir(xi1, xi2);
    or_calculateTransmission(ab, *s, w);
    return 1;
  }
  *dir = V(0, 0, 0);
  or_calculateTransmission(ab, distance, w);
  return 0;
}
int or_sample_medium(const float absorption[3], float scatter, float distance, const float u[3], float* s, float dir[3],
                     float weight[3]) {
  v3 d;
  int sc = sample_medium(absorption, scatter, distance, u[0], u[1], u[2], s, &d, weight);
  st3(dir, d);
  return sc;
}
void or_sample_medium_batch(int n, const float* absorption, const float* scatter, const float* distance, const float* u,
                            int32_t* scattered, float* s, float* dir, float* weight) {
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++)
    scattered[i] = or_sample_medium(absorption + 3 * i, scatter[i], distance[i], u + 3 * i, s + i, dir + 3 * i, weight + 3 * i);
}

/* (S) one shading event with subsurface scattering.  A medium geom (REFR > 0, SCATTER > 0, RSCTCOEFF > 0; not emissive)
 * reached from inside: the segment that ends here ran through the medium over t, and may have ended earlier, at a
 * scattering event drawn with u[3] of the depth's Philox block (the dimension or_shade leaves unused); the path then goes on
 * from o + d*s in the direction sphere_dir(u[0], u[1]) with throughput thr * transmission(ABSCOEFF, s) (kind 4).  Every
 * other case -- and every case while subsurface == 0 -- is or_shade, unchanged (absorption over t, then Fresnel with u[2]). */
int or_shade_sss(const or_scene* sc, int subsurface, int geom_id, float t, const float p[3], const float n[3], uint64_t seed,
                 uint32_t pixel, uint32_t sample, uint32_t depth, float o[3], float d[3], float thr[3], float L[3]) {
  const or_material* m = &sc->materials[sc->geoms[geom_id].materialid];
  if (subsurface && !(m->emittance > 0) && m->hasRefractive > 0 && m->hasScatter > 0 && m->reducedScatterCoefficient > 0 &&
      !(vdot(ld3(d), ld3(n)) < 0)) {
    float u[4], s, w[3];
    v3 dir;
    rng4(seed, pixel, sample, 1u + depth, u);
    if (sample_medium(m->absorptionCoefficient, m->reducedScatterCoefficient, t, u[0], u[1], u[3], &s, &dir, w)) {
      st3(o, vadd(ld3(o), vscale(ld3(d), s)));
      st3(d, dir);
      st3(thr, vmul(ld3(thr), ld3(w)));
      return 4;
    }
  }
  return or_shade(sc, geom_id, t, p, n, seed, pixel, sample, depth, o, d, thr, L);
}

/* (S) the path loop of or_render_ex (pt_oracle.c) with or_shade_sss in place of or_shade: a scattering event (kind 4) keeps
 * the path alive, uses one segment of max_depth and carries cos_b = 0 (no light sample there).  subsurface == 0 gives
 * or_render_ex's results bit for bit (tests/test_oracle_medium.py). */
double or_render_sss(const or_scene* sc, int subsurface, uint32_t first_sample, uint32_t n_samples, int max_depth,
                     uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb, uint64_t* live, int threads,
                     uint64_t* shadow_rays) {
  if (max_depth > 64) max_depth = 64;
#ifdef _OPENMP
  int nt = threads > 0 ? threads : omp_get_max_threads();
#else
  int nt = 1;
  (void)threads;
#endif
  or_light lights_buf[1024];  /* 36 KB on the stack; more lights than that are ignored (build_lights caps) */
  or_light* lights = lights_buf;
  int n_lights = 0;
  if (sc->direct_lighting) n_lights = build_lights(sc, lights, 1024);
  double t0 = now_s();
#pragma omp parallel num_threads(nt)
  {
    uint64_t mylive[64], myshadow = 0;
    memset(mylive, 0, sizeof(mylive));
#pragma omp for schedule(dynamic, 256)
    for (int64_t pix = (int64_t)pix_begin; pix < (int64_t)pix_end; pix++) {
      for (uint32_t s = first_sample; s < first_sample + n_samples; s++) {
        float o[3], d[3], thr[3] = {1.0f, 1.0f, 1.0f};
        float cos_b = 0.0f;  /* > 0: the previous event was a diffuse bounce with a light sample (MIS weight at the next light) */
        or_raygen(&sc->cam, &sc->lens, seed, (uint32_t)pix, s, o, d);
        for (int depth = 0; depth < max_depth; depth++) {
          mylive[depth]++;
          float t, p[3], n[3];
          int id = or_closest_hit(sc->geoms, sc->n_geoms, o, d, &t, p, n);
          if (id < 0) break;
          float L[3];
          v3 din = ld3(d);
          int kind = or_shade_sss(sc, subsurface, id, t, p, n, seed, (uint32_t)pix, s, (uint32_t)depth, o, d, thr, L);
          if (kind == 3) {
            if (cos_b > 0) {
              float clp = -vdot(ld3(n), din);
              if (clp > 0) {
                float Kh = 0.0f;
                for (int k = 0; k < n_lights; k++) if (lights[k].geom == id) Kh = lights[k].K;
                float x = ((cos_b * clp) / (t * t)) * Kh;
                float wb = x / (1.0f + x);
                L[0] = L[0] * wb; L[1] = L[1] * wb; L[2] = L[2] * wb;
              }
            }
            sum_rgb[3 * pix + 0] += L[0];
            sum_rgb[3 * pix + 1] += L[1];
            sum_rgb[3 * pix + 2] += L[2];
            break;
          }
          cos_b = 0.0f;
          if (kind == 0 && n_lights > 0 && depth + 1 < max_depth) {
            v3 N = ld3(n);
            v3 ns = vdot(din, N) < 0 ? N : vneg(N);
            cos_b = vdot(ns, ld3(d));  /* d = the direction the bounce sampled */
            float v[4];
            rng4(seed, (uint32_t)pix, s, 65u + (uint32_t)depth, v);
            int li = (int)(v[0] * (float)n_lights);
            if (li > n_lights - 1) li = n_lights - 1;
            const or_light* Lt = &lights[li];
            const or_static_geom* gl = &sc->geoms[Lt->geom];
            v3 y;
            if (gl->type == 0) {
              float yy[3];
              or_sphere_point_u(gl, v[1], v[2], yy);
              y = ld3(yy);
            } else {
              y = cube_point_th(gl, Lt->th, v[1], v[2] - 0.5f, v[3] - 0.5f);
            }
            v3 wv = vsub(y, ld3(o));
            v3 wd = vnormalize(wv);
            float dy = vlength(wv);
            float cs = vdot(ns, wd);
            if (cs > 0) {
              myshadow++;
              float wdv[3], t2, p2[3], n2[3];
              st3(wdv, wd);
              int id2 = or_closest_hit(sc->geoms, sc->n_geoms, o, wdv, &t2, p2, n2);
              /* y is visible iff the ray arrives ON the light AT y (a point on the light's far side is hidden by the
               * light itself: same geom, shorter distance) */
              if (id2 == Lt->geom && (dy - t2) < 1e-3f * dy + 1e-3f) {
                float cl = -vdot(ld3(n2), wd);
                if (cl > 0) {
                  float G = (cs * cl) / (t2 * t2);
                  float wl = 1.0f / (1.0f + G * Lt->K);
                  v3 Ld = vscale(vscale(vmul(ld3(thr), ld3(Lt->E)), G), wl);
                  sum_rgb[3 * pix + 0] += Ld.x;
                  sum_rgb[3 * pix + 1] += Ld.y;
                  sum_rgb[3 * pix + 2] += Ld.z;
                }
              }
            }
          }
        }
      }
    }
#pragma omp critical
    {
      for (int i = 0; i < max_depth; i++) live[i] += mylive[i];
      if (shadow_rays) *shadow_rays += myshadow;
    }
  }
  return now_s() - t0;
}
