// od_quad.cu — the un-clamped, four-output variant of the top-k assignment (SURVEY.md §8f N1).
//
// Replaces QuadrilateralDetection.bbox_matching
// (ref: src/sihl/heads/quadrilateral_detection.py:266-294) and the per-image Python loop around it
// (:165-172).  Differences from ObjectDetection.bbox_matching (od_assign.cu):
//   * no clamp(0): every gt selects exactly k anchors by raw CIoU, negative values included (:277-278);
//   * per anchor the reference takes max over gts of (iou * is_topk_match): a selected gt contributes its
//     (possibly negative) value, every gt that did NOT select the anchor contributes a zero (:283);
//   * four outputs: o2m_assignments, o2o_mask (anchor is some gt's best match, :279-280,:286), o2m_iou
//     (absolute) and o2m_rel_iou = (max / best_iou[gt]).nan_to_num(0) (:289-293).
// Anchors are arbitrary here (the quadrilateral head's anchors are level-sized squares around every location,
// :159-163), so all A x G pairs are evaluated: one warp per gt sweeps the anchors 32 at a time and keeps a top-k
// buffer of 64-bit keys (order-preserving CIoU bits << 32 | ~anchor: value desc, anchor asc — ties: lowest index).
// Stage 2 is one CTA per (image, 512 anchors): shared-memory atomicMax on the order-preserving bits, then atomicMin
// of the gt among the maxima (torch.max: lowest gt), a per-anchor count of selecting gts (to know whether an
// unselected gt's zero takes part in the max) and the best-match flags.
//
// Canonical output (as for the clamped variant, SURVEY.md §3.4): assignment = -1 wherever rel_iou is not > 0 —
// there the reference's index is that of an arbitrary zero entry and nothing downstream reads it (:188,:201 index
// assignment[b, rel_iou > 0] only); iou / rel_iou of such anchors are 0 exactly as in the reference.
#include "od_common.cuh"

namespace sihl {

constexpr int kQuadSelWarps = 4;
constexpr int kQuadBuf = 64;
constexpr int kQuadResThreads = 128;

// float -> uint32 whose unsigned order is the float order (-0 folded into +0 first: torch.topk / max compare them equal)
__device__ __forceinline__ unsigned ord_bits(float v) { return f2ord(v + 0.f); }

__device__ __forceinline__ int quad_compress(unsigned long long *bk, int cnt, int topk, int lane)
{
    __syncwarp();
    const bool h0 = lane < cnt, h1 = lane + 32 < cnt;
    const unsigned long long k0 = h0 ? bk[lane] : 0ull, k1 = h1 ? bk[lane + 32] : 0ull;
    int r0 = 0, r1 = 0;
#pragma unroll 4
    for (int i = 0; i < cnt; ++i) {
        const unsigned long long ki = bk[i];
        r0 += ki > k0;
        r1 += ki > k1;
    }
    __syncwarp();
    if (h0 && r0 < topk) bk[r0] = k0;
    if (h1 && r1 < topk) bk[r1] = k1;
    __syncwarp();
    return cnt < topk ? cnt : topk;
}

// ref :277-278: topk(ious, k, dim=0) per gt — values descending, ties -> lowest anchor index.
__global__ void __launch_bounds__(kQuadSelWarps * 32)
k_quad_select(const float4 *__restrict__ anchors, const float4 *__restrict__ anchor_terms, int num_anchors,
              const float4 *__restrict__ gt_boxes, int total_gt, int topk, int32_t *__restrict__ sel_anchor,
              float *__restrict__ sel_val)
{
    __shared__ unsigned long long s_key[kQuadSelWarps][kQuadBuf];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * kQuadSelWarps + warp;
    if (g >= total_gt) return;
    unsigned long long *bk = s_key[warp];
    const BoxTerms gt = box_terms(to_box(__ldg(gt_boxes + g)));
    int cnt = 0;
    unsigned long long floor_key = 0ull;                 // k-th best so far once the buffer holds k entries
    for (int a0 = 0; a0 < num_anchors; a0 += 32) {
        const int a = a0 + lane;
        bool hit = false;
        unsigned long long key = 0ull;
        if (a < num_anchors) {
            const float4 bx = __ldg(anchors + a), t = __ldg(anchor_terms + a);   // (area, cx, cy, atan(w/h)): k_anchor_terms
            BoxTerms an;
            an.x1 = bx.x; an.y1 = bx.y; an.x2 = bx.z; an.y2 = bx.w; an.area = t.x; an.cx = t.y; an.cy = t.z; an.at = t.w;
            const float v = ciou_pair(an, gt);
            if (v == v) {                                // NaN never ranks (precondition: finite, non-degenerate boxes)
                key = ((unsigned long long)ord_bits(v) << 32) | (unsigned long long)(0xffffffffu - (unsigned)a);
                hit = key > floor_key;
            }
        }
        const unsigned m = __ballot_sync(kFullMask, hit);
        if (m) {
            if (hit) bk[cnt + __popc(m & ((1u << lane) - 1u))] = key;
            cnt += __popc(m);
            if (cnt > kQuadBuf - 32) {
                cnt = quad_compress(bk, cnt, topk, lane);
                if (cnt == topk) floor_key = bk[topk - 1];
            }
        }
    }
    cnt = quad_compress(bk, cnt, topk, lane);
    if (lane < topk) {
        const unsigned long long k = lane < cnt ? bk[lane] : 0ull;
        sel_anchor[(int64_t)g * topk + lane] = lane < cnt ? (int)(0xffffffffu - (unsigned)k) : -1;
        sel_val[(int64_t)g * topk + lane] = lane < cnt ? ord2f((unsigned)(k >> 32)) : 0.f;
    }
}

struct QuadResolveParams {
    const int32_t *sel_anchor; const float *sel_val; const int32_t *gt_offsets;
    int num_anchors, topk;
    float inv_topk;
    int64_t *assignment; uint8_t *o2o; float *iou; float *rel;
};

// torch.nan_to_num(x, nan=0): NaN -> 0, +-inf -> +-FLT_MAX (ref :293).
__device__ __forceinline__ float nan_to_num0(float x)
{
    if (x != x) return 0.f;
    if (x == CUDART_INF_F) return 3.402823466e+38f;
    if (x == -CUDART_INF_F) return -3.402823466e+38f;
    return x;
}

__global__ void __launch_bounds__(kQuadResThreads) k_quad_resolve(QuadResolveParams p)
{
    __shared__ unsigned s_v[kTile], s_g[kTile];
    __shared__ unsigned s_cnt[kTile];
    __shared__ unsigned char s_best[kTile];
    const int tid = threadIdx.x;
    const int b = blockIdx.y, a0 = blockIdx.x * kTile;
    const int A = p.num_anchors, na = min(kTile, A - a0);
    const int g0 = __ldg(p.gt_offsets + b), g1 = __ldg(p.gt_offsets + b + 1);
    const int n_gt = g1 - g0, n_entries = n_gt * p.topk;
    for (int i = tid; i < kTile; i += kQuadResThreads) { s_v[i] = 0u; s_g[i] = 0xffffffffu; s_cnt[i] = 0; s_best[i] = 0; }
    __syncthreads();
    const int32_t *sa = p.sel_anchor + (int64_t)g0 * p.topk;
    const float *sv = p.sel_val + (int64_t)g0 * p.topk;
    const bool recip = n_entries < (1 << 21);
    for (int e = tid; e < n_entries; e += kQuadResThreads) {
        const int a = __ldg(sa + e) - a0;
        if (a < 0 || a >= na) continue;
        const int g = recip ? (int)(((float)e + 0.5f) * p.inv_topk) : e / p.topk;
        atomicMax(&s_v[a], ord_bits(__ldg(sv + e)));     // ord_bits > 0 for every non-NaN value: 0 means "not selected"
        atomicAdd(&s_cnt[a], 1u);                        // how many gts selected this anchor
        if (e - g * p.topk == 0) s_best[a] = 1;          // ref :279-280 topk_idxs[0:1]
    }
    __syncthreads();
    for (int e = tid; e < n_entries; e += kQuadResThreads) {
        const int a = __ldg(sa + e) - a0;
        if (a < 0 || a >= na) continue;
        if (s_v[a] == ord_bits(__ldg(sv + e))) {
            const int g = recip ? (int)(((float)e + 0.5f) * p.inv_topk) : e / p.topk;
            atomicMin(&s_g[a], (unsigned)g);
        }
    }
    __syncthreads();
    for (int la = tid; la < na; la += kQuadResThreads) {
        const int64_t flat = (int64_t)b * A + a0 + la;
        const int cnt = (int)s_cnt[la];
        int64_t asg = -1;
        float iou = 0.f, rel = 0.f;
        if (cnt > 0) {
            const float v = ord2f(s_v[la]);
            const int g = (int)s_g[la];
            // the max of ref :283 runs over the selected values and one zero per gt that did not select this anchor
            if (v > 0.f || cnt == n_gt) {
                iou = v;
                rel = nan_to_num0(v / __ldg(sv + (int64_t)g * p.topk));     // best_ious_per_gt = topk_ious[0], ref :289-293
                if (rel > 0.f) asg = g;                                      // canonical form
            }
        }
        p.assignment[flat] = asg;
        p.o2o[flat] = cnt > 0 ? s_best[la] : 0;
        p.iou[flat] = iou;
        p.rel[flat] = rel;
    }
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_quad_matching(const float *anchors, int64_t num_anchors, const float *gt_boxes,
                                     const int32_t *gt_offsets, int batch, int total_gt, int topk,
                                     int64_t *assignment, uint8_t *o2o_mask, float *o2m_iou, float *rel_iou,
                                     int32_t *sel_anchor, float *sel_val, float *anchor_terms, void *stream)
{
    SIHL_CHECK_ARG(topk >= 1 && topk <= SIHL_OD_MAX_TOPK, "topk=%d outside 1..%d", topk, SIHL_OD_MAX_TOPK);
    SIHL_CHECK_ARG(batch >= 0 && batch <= 65535 && total_gt >= 0 && num_anchors >= 0 && num_anchors < (1ll << 30), "bad sizes");
    SIHL_CHECK_ARG(total_gt == 0 || num_anchors >= topk,
                   "selected index k out of range: %lld anchors < topk=%d (torch.topk raises in the reference)",
                   (long long)num_anchors, topk);
    SIHL_CHECK_ARG(assignment && o2o_mask && o2m_iou && rel_iou && gt_offsets, "NULL output / gt_offsets");
    SIHL_CHECK_ARG(total_gt == 0 || (anchors && gt_boxes && sel_anchor && sel_val && anchor_terms), "NULL input / workspace");
    if (batch == 0 || num_anchors == 0) return SIHL_OD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (total_gt > 0) {
        int rc = sihl_od_anchor_terms(anchors, num_anchors, anchor_terms, stream);   // per-anchor half of the CIoU, once
        if (rc) return rc;
        k_quad_select<<<(total_gt + kQuadSelWarps - 1) / kQuadSelWarps, kQuadSelWarps * 32, 0, st>>>(
            reinterpret_cast<const float4 *>(anchors), reinterpret_cast<const float4 *>(anchor_terms), (int)num_anchors,
            reinterpret_cast<const float4 *>(gt_boxes), total_gt, topk, sel_anchor, sel_val);
        SIHL_CHECK_LAUNCH("k_quad_select");
    }
    QuadResolveParams p;
    p.sel_anchor = sel_anchor; p.sel_val = sel_val; p.gt_offsets = gt_offsets; p.num_anchors = (int)num_anchors; p.topk = topk;
    p.inv_topk = 1.f / (float)topk;
    p.assignment = assignment; p.o2o = o2o_mask; p.iou = o2m_iou; p.rel = rel_iou;
    const dim3 grid((unsigned)((num_anchors + kTile - 1) / kTile), (unsigned)batch);
    k_quad_resolve<<<grid, kQuadResThreads, 0, st>>>(p);
    SIHL_CHECK_LAUNCH("k_quad_resolve");
    return SIHL_OD_OK;
}
