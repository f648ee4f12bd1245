/* TEST INFRASTRUCTURE ONLY -- see pt_oracle_glossy.h.
 *
 * Glossy reflection (DESIGN.md 4): reflective materials with SPECEX > 0 sample a Phong lobe around the mirror direction
 * instead of the mirror direction itself.  This file compiles pt_oracle_medium.c (and with it pt_oracle.c) together with
 * the pieces below into libpt_oracle_glossy.so, so that the restatement's own helpers (Philox addressing, reflect,
 * sincos_2pi, the reproducible exp and log, the light table) are reused as they are and both files stay the frozen
 * specification of everything else.
 *
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fno-fast-math -fopenmp (oracle/oracle_glossy.py), like pt_oracle.c.
 */
#include "pt_oracle_medium.c"
#include "pt_oracle_glossy.h"

/* (S) the diffuse sampler's tangent frame (src/interactions.h:72-85, hemisphere_body) of an arbitrary unit vector */
static inline void frame3(v3 normal, v3* p1, v3* p2) {
  v3 dnn;
  if ((double)fabsf(normal.x) < OR_SQRT_OF_ONE_THIRD) {
    dnn = V(1, 0, 0);
  } else if ((double)fabsf(normal.y) < OR_SQRT_OF_ONE_THIRD) {
    dnn = V(0, 1, 0);
  } else {
    dnn = V(0, 0, 1);
  }
  *p1 = vnormalize(vcross(normal, dnn));
  *p2 = vnormalize(vcross(normal, *p1));
}

/* (S) the glossy lobe: a Phong lobe of exponent specex around r = reflect(ns, d).  The cosine c of the angle to r has
 * the CDF c^(specex + 1) on [0, 1]: c = exp(log(1 - u0) / (specex + 1)) with the reproducible exp and log (1 - u0 is
 * exact for u0 = k * 2^-24 and lies in (0, 1]); the azimuth 2*pi*u1 turns in the diffuse sampler's frame of r, with
 * hemisphere_in_frame's operand order.  A sample below the surface (dot(g, ns) <= 0) is folded back above it by the
 * mirror through the surface plane, so the path always continues and the lobe's albedo is exactly specularColor.  As
 * specex grows, c reaches 1 and g is r bit for bit: the mirror. */
static inline v3 sample_glossy(v3 ns, v3 d, float specex, float u0, float u1) {
  const v3 r = reflect3(ns, d);
  v3 p1, p2;
  frame3(r, &p1, &p2);
  const float c = or_exp(or_log(1.0f - u0) / (specex + 1.0f));
  const float s = sqrtf(fmaxf(0.0f, 1.0f - c * c));
  float sn, cs;
  or_sincos_2pi(u1, &sn, &cs);
  v3 g = vadd(vadd(vscale(r, c), vscale(p1, cs * s)), vscale(p2, sn * s));
  if (!(vdot(g, ns) > 0)) g = reflect3(ns, g);
  return g;
}
void or_sample_glossy(const float n[3], const float d[3], float specex, const float u[2], float out[3]) {
  const v3 N = ld3(n), D = ld3(d);
  const v3 ns = vdot(D, N) < 0 ? N : vneg(N);
  st3(out, sample_glossy(ns, D, specex, u[0], u[1]));
}
void or_sample_glossy_batch(int n, const float* normal, const float* incident, const float* exponent, const float* u,
                            float* direction) {
#pragma omp parallel for schedule(static)
  for (int i = 0; i < n; i++) or_sample_glossy(normal + 3 * i, incident + 3 * i, exponent[i], u + 2 * i, direction + 3 * i);
}

/* (S) one shading event with glossy reflection.  A glossy geom (REFL > 0, REFR <= 0, SPECEX > 0; not emissive) takes
 * the mirror branch of or_shade with the lobe's direction in place of the mirror direction, driven by u[0], u[1] of the
 * depth's Philox block (the dimensions the diffuse sampler uses): origin p + ns * RAY_BIAS_AMOUNT, throughput times
 * specularColor, kind 1 (a specular event: no light sample, the next emission counts in full).  Every other case -- and
 * every case while glossy == 0 -- is or_shade_sss, unchanged. */
int or_shade_ext(const or_scene* sc, int subsurface, int glossy, int geom_id, float t, const float p[3], const float n[3],
                 uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, float o[3], float d[3], float thr[3],
                 float L[3]) {
  const or_material* m = &sc->materials[sc->geoms[geom_id].materialid];
  if (glossy && !(m->emittance > 0) && !(m->hasRefractive > 0) && m->hasReflective > 0 && m->specularExponent > 0) {
    const v3 D = ld3(d), N = ld3(n);
    const v3 ns = vdot(D, N) < 0 ? N : vneg(N);
    float u[4];
    rng4(seed, pixel, sample, 1u + depth, u);
    const v3 g = sample_glossy(ns, D, m->specularExponent, u[0], u[1]);
    st3(o, vadd(ld3(p), vscale(ns, OR_RAY_BIAS_AMOUNT)));
    st3(d, g);
    st3(thr, vmul(ld3(thr), ld3(m->specularColor)));
    return 1;
  }
  return or_shade_sss(sc, subsurface, geom_id, t, p, n, seed, pixel, sample, depth, o, d, thr, L);
}

/* (S) the path loop of or_render_sss (pt_oracle_medium.c) with or_shade_ext in place of or_shade_sss.  A glossy event is
 * kind 1 like a mirror: it carries cos_b = 0.  glossy == 0 gives or_render_sss's results bit for bit
 * (tests/test_oracle_glossy.py). */
double or_render_ext(const or_scene* sc, int subsurface, int glossy, uint32_t first_sample, uint32_t n_samples,
                     int max_depth, uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb, uint64_t* live,
                     int threads, uint64_t* shadow_rays) {
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
