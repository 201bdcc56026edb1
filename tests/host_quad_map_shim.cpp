// Test-only: the per-quad values sihl_od_quad_map_match matches with — the hull area and the hull IoU of od_math.h
// (sihl_b200/csrc/od_math.h) — compiled for the HOST with -ffp-contract=off, as the library is built with -fmad=false, so
// that the quad COCO oracle (tests/quad_map_reference.py) sees the same fp32 bits as the kernels.  Never part of the
// product library.
#include <vector>

#include "../sihl_b200/csrc/od_math.h"

// out[i] = the hull area of quad i (the area sihl_od_quad_map_match puts in the COCO area ranges)
extern "C" void shim_quad_hull_areas(const float *q, long n, float *out)
{
    for (long i = 0; i < n; ++i) out[i] = sihl::quad_hull(q + 8 * i).area;
}

// out[i * nb + j] = quad_iou(a_i, b_j), each hull built once (the matrix sihl_od_quad_map_match fills per image)
extern "C" void shim_quad_iou_grid(const float *a, long na, const float *b, long nb, float *out)
{
    std::vector<sihl::QuadHull> hb(nb);
    for (long j = 0; j < nb; ++j) hb[j] = sihl::quad_hull(b + 8 * j);
    for (long i = 0; i < na; ++i) {
        const sihl::QuadHull ha = sihl::quad_hull(a + 8 * i);
        for (long j = 0; j < nb; ++j) out[i * nb + j] = sihl::quad_iou_hulls(ha, hb[j]);
    }
}
