// Test-only: the overlap sihl_od_quad_map_match_crowd gives a detection with a crowd ("don't care") quad — od_math.h's
// quad_ioa_hulls, the clamped hull intersection over the detection's hull area (sihl_b200/csrc/od_math.h) — compiled for
// the HOST with -ffp-contract=off, as the library is built with -fmad=false, so that the crowd oracle
// (tests/crowd_map_reference.py) sees the same fp32 bits as k_quad_map_iou_crowd.  Never part of the product library.
#include <vector>

#include "../sihl_b200/csrc/od_math.h"

// out[i * nb + j] = quad_ioa_hulls(a_i, b_j), each hull built once
extern "C" void shim_quad_ioa_grid(const float *a, long na, const float *b, long nb, float *out)
{
    std::vector<sihl::QuadHull> hb(nb);
    for (long j = 0; j < nb; ++j) hb[j] = sihl::quad_hull(b + 8 * j);
    for (long i = 0; i < na; ++i) {
        const sihl::QuadHull ha = sihl::quad_hull(a + 8 * i);
        for (long j = 0; j < nb; ++j) out[i * nb + j] = sihl::quad_ioa_hulls(ha, hb[j]);
    }
}
