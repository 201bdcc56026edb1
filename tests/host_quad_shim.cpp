// Test-only: compiles the quad overlap of sihl_b200/csrc/od_math.h (the suppression test of sihl_od_batched_quad_nms and
// the value of sihl_od_quad_iou) for the HOST, and runs the plain greedy quad NMS on it: the oracle the GPU results must
// equal.  Built with -ffp-contract=off, as the library is with -fmad=false.  Never part of the product library.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "../sihl_b200/csrc/od_math.h"

// out[i] = quad_iou(a_i, b_i) for n pairs of quads (8 floats each)
extern "C" void shim_quad_iou_pairs(const float *a, const float *b, long n, float *out)
{
    for (long i = 0; i < n; ++i) out[i] = sihl::quad_iou(a + 8 * i, b + 8 * i);
}

// Greedy class-aware NMS of one list: visit by (score desc, index asc); a kept quad suppresses every later quad of its
// class with quad_iou > thr.  Pairs whose AABBs do not overlap have IoU 0: they are only tested when thr < 0.
// Returns the number of kept indices written to keep (in visit order).
extern "C" long shim_batched_quad_nms(const float *quads, const float *scores, const int64_t *classes, long n, float thr,
                                      int64_t *keep)
{
    std::vector<sihl::QuadHull> h(n);
    for (long i = 0; i < n; ++i) h[i] = sihl::quad_hull(quads + 8 * i);
    std::vector<long> order(n);
    for (long i = 0; i < n; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](long i, long j) {
        if (classes[i] != classes[j]) return classes[i] < classes[j];
        if (scores[i] != scores[j]) return scores[i] > scores[j];
        return i < j;
    });
    std::vector<char> dead(n, 0);
    std::vector<long> kept_idx;
    for (long s = 0; s < n;) {                       // one class at a time
        long e = s;
        while (e < n && classes[order[e]] == classes[order[s]]) ++e;
        std::vector<long> kept;                      // kept items of this class, to test later items against
        for (long p = s; p < e; ++p) {
            const long j = order[p];
            bool sup = false;
            for (long i : kept) {
                const sihl::QuadHull &a = h[i], &b = h[j];
                const bool apart = !(std::min(a.x2, b.x2) > std::max(a.x1, b.x1)) || !(std::min(a.y2, b.y2) > std::max(a.y1, b.y1));
                if (apart ? 0.f > thr : sihl::quad_iou_hulls(a, b) > thr) { sup = true; break; }
            }
            if (!sup) { kept.push_back(j); kept_idx.push_back(j); }
        }
        s = e;
    }
    // output order: score desc, index asc over the whole list
    std::sort(kept_idx.begin(), kept_idx.end(), [&](long i, long j) {
        if (scores[i] != scores[j]) return scores[i] > scores[j];
        return i < j;
    });
    for (size_t k = 0; k < kept_idx.size(); ++k) keep[k] = kept_idx[k];
    return (long)kept_idx.size();
}
