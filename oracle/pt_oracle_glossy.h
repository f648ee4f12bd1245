/* TEST INFRASTRUCTURE ONLY.
 *
 * Glossy reflection for the CPU oracle (pt_oracle.h, pt_oracle_medium.h): the (S) specification of the Phong lobe that
 * reflective materials with SPECEX > 0 sample around the mirror direction, and the path loop that uses it (DESIGN.md 4).
 * Same arithmetic contract as pt_oracle.h: binary32, round-to-nearest-even, unfused, in the order written; the CUDA
 * kernels (pt_set_glossy, pt_sample_glossy) follow it bit for bit.
 */
#ifndef PT_ORACLE_GLOSSY_H
#define PT_ORACLE_GLOSSY_H

#include "pt_oracle_medium.h"

#ifdef __cplusplus
extern "C" {
#endif

/* one glossy direction: ns = the outward normal n turned to face the incoming direction d, r = reflect(ns, d), a Phong
 * lobe of exponent specex around r driven by u = (u0, u1), folded above the surface */
void or_sample_glossy(const float n[3], const float d[3], float specex, const float u[2], float out[3]);
/* n entries: normal (x3), incident (x3), exponent, u (x2) -> direction (x3) */
void or_sample_glossy_batch(int n, const float* normal, const float* incident, const float* exponent, const float* u,
                            float* direction);
/* or_shade_sss with glossy reflection: while glossy != 0 a glossy geom (REFL > 0, REFR <= 0, SPECEX > 0, not emissive)
 * samples the lobe instead of the mirror direction (kind 1) */
int or_shade_ext(const or_scene* sc, int subsurface, int glossy, int geom_id, float t, const float p[3], const float n[3],
                 uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, float o[3], float d[3], float thr[3],
                 float L[3]);
/* or_render_sss with glossy reflection (glossy == 0: or_render_sss bit for bit) */
double or_render_ext(const or_scene* sc, int subsurface, int glossy, uint32_t first_sample, uint32_t n_samples,
                     int max_depth, uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb, uint64_t* live,
                     int threads, uint64_t* shadow_rays);

#ifdef __cplusplus
}
#endif
#endif
