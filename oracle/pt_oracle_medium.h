/* TEST INFRASTRUCTURE ONLY.
 *
 * Subsurface scattering for the CPU oracle (pt_oracle.h): the (S) specification of the reference's
 * calculateScatterAndAbsorption stub (src/interactions.h:16-39) and the path loop that uses it (DESIGN.md 4).  Same
 * arithmetic contract as pt_oracle.h: binary32, round-to-nearest-even, unfused, in the order written; the CUDA kernels
 * (pt_set_subsurface, pt_sample_medium) follow it bit for bit.
 */
#ifndef PT_ORACLE_MEDIUM_H
#define PT_ORACLE_MEDIUM_H

#include "pt_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* log with +,-,* only; positive normal x, else -inf */
float or_log(float x);
/* the free flight of calculateScatterAndAbsorption: u = (xi1, xi2, xf), s = -log(1 - xf) / scatter; returns 1 and
 * dir = uniform direction, weight = transmission over s if s < distance, else 0, dir = 0, weight = transmission over
 * distance */
int or_sample_medium(const float absorption[3], float scatter, float distance, const float u[3], float* s, float dir[3],
                     float weight[3]);
void or_sample_medium_batch(int n, const float* absorption, const float* scatter, const float* distance, const float* u,
                            int32_t* scattered, float* s, float* dir, float* weight);
/* or_shade with subsurface scattering: returns 4 for a scattering event inside a medium geom (subsurface != 0) */
int or_shade_sss(const or_scene* sc, int subsurface, int geom_id, float t, const float p[3], const float n[3], uint64_t seed,
                 uint32_t pixel, uint32_t sample, uint32_t depth, float o[3], float d[3], float thr[3], float L[3]);
/* or_render_ex with subsurface scattering (subsurface == 0: or_render_ex bit for bit) */
double or_render_sss(const or_scene* sc, int subsurface, uint32_t first_sample, uint32_t n_samples, int max_depth,
                     uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb, uint64_t* live, int threads,
                     uint64_t* shadow_rays);

#ifdef __cplusplus
}
#endif
#endif
