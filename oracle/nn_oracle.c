/*
 * nn_oracle.c -- CPU restatement of the reference's nearest-neighbour index kernels.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in pvnet_b200/ may include, link, load or call this file; only tests/,
 * __graft_entry__.smoke() and benchmarks use it, through oracle/metrics_oracle.py, as the checker.
 *
 * What is restated (paths relative to the zju3dv/pvnet tree):
 *   pvo_find_nearest_point_idx   lib/utils/extend_utils/src/nearest_neighborhood.cu:48-117
 *                                (findNearestPoint{2D,3D}IdxKernel)
 *
 * Floating point.  The distance is the sequence nvcc 12.9 emits for the reference kernel on sm_100a (DESIGN.md
 * §2): d = ref - que per axis; 2-D fmaf(dx,dx,dy*dy), 3-D fmaf(dz,dz,fmaf(dx,dx,dy*dy)).  Selection: (FLT_MAX, 0)
 * start, strict `<`, increasing index.  Built with -ffp-contract=off (oracle/metrics.mk), so the compiler adds
 * or removes no FMA.  Offsets are 64-bit.
 *
 * Parity pin: tests/golden/ref_nn.npz holds the indices the reference kernel itself returned
 * (tests/golden/make_golden_nn.py); tests/test_metrics_cpu.py checks this file against them bit for bit.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define PVO_API __attribute__((visibility("default")))

/* ref [b,pn1,dim], que [b,pn2,dim] f32, idxs [b,pn2] */
PVO_API void pvo_find_nearest_point_idx(const float *ref, const float *que, int32_t *idxs, int b, int pn1, int pn2,
                                        int dim, int exclude_self)
{
    #pragma omp parallel for collapse(2) schedule(static)
    for (int bi = 0; bi < b; ++bi) {
        for (int qi = 0; qi < pn2; ++qi) {
            const float *q = que + ((size_t)bi * pn2 + qi) * dim;
            const float *r = ref + (size_t)bi * pn1 * dim;
            float min_dist = 3.40282346638528859812e+38F; /* FLT_MAX */
            int min_idx = 0;
            for (int i = 0; i < pn1; ++i) {
                if (exclude_self && i == qi) continue;
                const float dx = r[(size_t)i * dim] - q[0], dy = r[(size_t)i * dim + 1] - q[1];
                float dist = fmaf(dx, dx, dy * dy);
                if (dim == 3) {
                    const float dz = r[(size_t)i * dim + 2] - q[2];
                    dist = fmaf(dz, dz, dist);
                }
                if (dist < min_dist) {
                    min_dist = dist;
                    min_idx = i;
                }
            }
            idxs[(size_t)bi * pn2 + qi] = min_idx;
        }
    }
}
