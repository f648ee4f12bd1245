/* TEST INFRASTRUCTURE ONLY.
 *
 * Russian roulette for the CPU oracle (pt_oracle.h, pt_oracle_medium.h, pt_oracle_glossy.h): the (S) specification of the
 * step that ends low-throughput paths at random from a chosen depth and reweights the survivors, and the path loop that
 * uses it (DESIGN.md 4).  Same arithmetic contract as pt_oracle.h: binary32, round-to-nearest-even, unfused, in the order
 * written; the CUDA kernels (pt_set_russian_roulette) follow it bit for bit.
 */
#ifndef PT_ORACLE_ROULETTE_H
#define PT_ORACLE_ROULETTE_H

#include "pt_oracle_glossy.h"

#ifdef __cplusplus
extern "C" {
#endif

/* one roulette step at depth `depth` on the path's incoming throughput: m = max channel, q = 1 for m >= 1, else m rounded
 * up to a multiple of 2^-24; q == 1 -> 1 (no draw, thr unchanged); else u = u[0] of Philox block 129 + depth: u < q -> 1
 * with thr = thr / q, otherwise 0 (the path ends) */
int or_roulette(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t depth, float thr[3]);
/* or_render_ext with Russian roulette from depth first_depth (0 = off: or_render_ext bit for bit): at every depth d with
 * first_depth <= d < max_depth - 1 whose closest hit is a non-emissive geom, or_roulette runs before the shading */
double or_render_rr(const or_scene* sc, int subsurface, int glossy, int first_depth, uint32_t first_sample,
                    uint32_t n_samples, int max_depth, uint64_t seed, uint32_t pix_begin, uint32_t pix_end, float* sum_rgb,
                    uint64_t* live, int threads, uint64_t* shadow_rays);

#ifdef __cplusplus
}
#endif
#endif
