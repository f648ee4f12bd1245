/* TEST INFRASTRUCTURE ONLY -- see pt_oracle_roulette.h.
 *
 * Russian roulette (DESIGN.md 4): from a depth the user chooses, a path whose throughput has fallen below 1 ends at random
 * with probability 1 - q and the survivors are divided by q, so that the estimator stays unbiased.  This file compiles
 * pt_oracle_glossy.c (and with it pt_oracle_medium.c and pt_oracle.c) unchanged, together with the pieces below, into
 * libpt_oracle_roulette.so.
 *
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fno-fast-math -fopenmp (oracle/oracle_roulette.py), like pt_oracle.c.
 */
#include "pt_oracle_glossy.c"
#include "pt_oracle_roulette.h"

/* (S) the roulette step.  m = max(thr) is exact.  q = m rounded up to a multiple of 2^-24 (every operation exact: the
 * scaling by 2^24 and 2^-24, and ceil), 1 for m >= 1.  u01 draws u = j * 2^-24, so P(u < q) is exactly q and u < q is
 * equivalent to u < m: weighting the survivors by 1/q is unbiased for the discrete draw.  A path with q == 1 goes on with
 * its throughput's bits and without a draw. */
int or_roulette(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, float thr[3]) {
  const float m = fmaxf(fmaxf(thr[0], thr[1]), thr[2]);
  const float q = m >= 1.0f ? 1.0f : ceilf(m * 16777216.0f) * 5.9604644775390625e-8f;
  if (q == 1.0f) return 1;
  float u[4];
  rng4(seed, pixel, sample, 129u + depth, u);
  if (!(u[0] < q)) return 0;
  thr[0] = thr[0] / q;
  thr[1] = thr[1] / q;
  thr[2] = thr[2] / q;
  return 1;
}

/* (S) the path loop of or_render_ext (pt_oracle_glossy.c) with the roulette step between the closest hit and
 * or_shade_ext.  It runs at depth d when first_depth >= 1, first_depth <= d < max_depth - 1 (none at depth 0, where the
 * throughput is 1, none on the last segment, which continues nowhere) and the hit geom is not emissive.  A path it ends
 * has traced segment d (it counts in live[d]) and gets no shading, no light sample and no further segment.  A survivor's
 * light sample uses the reweighted throughput.  first_depth == 0 gives or_render_ext's results bit for bit
 * (tests/test_oracle_roulette.py). */
double or_render_rr(const or_scene* sc, int subsurface, int glossy, int first_depth, uint32_t first_sample,
                    uint32_t n_samples, int max_depth, uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb,
                    uint64_t* live, int threads, uint64_t* shadow_rays) {
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
          if (first_depth > 0 && depth >= first_depth && depth < max_depth - 1 &&
              !(sc->materials[sc->geoms[id].materialid].emittance > 0) &&
              !or_roulette(seed, (uint32_t)pix, s, (uint32_t)depth, thr))
            break;
          float L[3];
          v3 din = ld3(d);
          int kind = or_shade_ext(sc, subsurface, glossy, id, t, p, n, seed, (uint32_t)pix, s, (uint32_t)depth, o, d, thr, L);
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
