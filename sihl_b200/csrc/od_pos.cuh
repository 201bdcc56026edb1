// od_pos.cuh — device pieces of the losses (SURVEY.md §8 a5-a10) shared by the positive-row loss over
// dense maps (od_loss.cu) and the compact-row forward / backward of the training step (od_train.cu).
#pragma once

#include "od_common.cuh"

namespace sihl {

// ref object_detection.py:189 and :195 — decoded (normalised) prediction and target of one positive.
__device__ __forceinline__ void pos_boxes(float4 raw, float4 off, float4 sc, float4 gt, float img_w, float img_h,
                                          Box4 *pred, Box4 *tgt)
{
    *pred = Box4{decode_norm(off.x, sc.x, raw.x), decode_norm(off.y, sc.y, raw.y),
                 decode_norm(off.z, sc.z, raw.z), decode_norm(off.w, sc.w, raw.w)};
    *tgt = Box4{gt.x / img_w, gt.y / img_h, gt.z / img_w, gt.w / img_h};
}

// CIoU loss of one positive (thread per row).  ref :189-197.
__device__ __forceinline__ float pos_box_loss(float4 raw, float4 off, float4 sc, float4 gt, float img_w, float img_h)
{
    Box4 pred, tgt;
    pos_boxes(raw, off, sc, gt, img_w, img_h, &pred, &tgt);
    return ciou_loss_row(pred, tgt, nullptr);
}

// exp(x), x <= 0, inside a softmax denominator.  FAST: ex2.approx(x * log2 e), 2 instructions instead of the 8 of
// expf; relative error <= 2^-21 per term, i.e. <= 5e-7 absolute on a cross-entropy of O(1) — the class loss is held
// to 1e-5 relative (BASELINE.json north_star), not to bit equality, and only the forward tile kernel on the step's
// critical path uses it.  The backward kernels and the compact-row forward keep expf.
template <bool FAST>
__device__ __forceinline__ float softmax_exp(float x)
{
    return FAST ? __expf(x) : expf(x);
}

// Row statistics of a class-logit row by a group of 8 lanes (4 rows per warp): max and
// sum exp(z - max).  Every lane of the warp must call; lanes of a group share z and C.
template <bool FAST = false>
__device__ __forceinline__ void row_softmax_stats8(const float *__restrict__ z, int C, int gl, float *m_out,
                                                   float *s_out)
{
    float m = -CUDART_INF_F;
    for (int c = gl; c < C; c += 8) m = fmaxf(m, __ldg(z + c));
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
    float s = 0.f;
    for (int c = gl; c < C; c += 8) s += softmax_exp<FAST>(__ldg(z + c) - m);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    *m_out = m;
    *s_out = s;
}

// Same with 4 lanes per row and 16-byte loads (C % 4 == 0, 16-byte aligned rows): 8 rows per warp.
template <bool FAST = false>
__device__ __forceinline__ void row_softmax_stats4v(const float *__restrict__ z, int C, int gl, float *m_out, float *s_out)
{
    const float4 *z4 = reinterpret_cast<const float4 *>(z);
    const int C4 = C >> 2;
    float m = -CUDART_INF_F;
    for (int v = gl; v < C4; v += 4) {
        const float4 q = __ldg(z4 + v);
        m = fmaxf(m, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
    }
#pragma unroll
    for (int o = 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
    float s = 0.f;
    for (int v = gl; v < C4; v += 4) {
        const float4 q = __ldg(z4 + v);
        s += (softmax_exp<FAST>(q.x - m) + softmax_exp<FAST>(q.y - m)) + (softmax_exp<FAST>(q.z - m) + softmax_exp<FAST>(q.w - m));
    }
#pragma unroll
    for (int o = 2; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    *m_out = m;
    *s_out = s;
}

// The five losses [location, box, class, iou, total] from the 8 sums (layout in sihl_od.h).
__device__ __forceinline__ void finalize_losses(const double *sums, float *losses)
{
    const double loc = sums[0] / sums[1];                         // ref :163 (0/0 and x/0 as in the reference)
    if (sums[6] == 0.0) {                                         // ref :165-172, rel_iou.max() == 0
        losses[0] = (float)loc; losses[1] = 0.f; losses[2] = 0.f; losses[3] = 0.f; losses[4] = (float)loc;
        return;
    }
    const double iou = sums[2] / sums[3], box = sums[4] / sums[3], cls = sums[5] / sums[3];
    losses[0] = (float)loc; losses[1] = (float)box; losses[2] = (float)cls; losses[3] = (float)iou;
    losses[4] = (float)(loc + 10.0 * box + cls + iou);           // ref :210
}

}  // namespace sihl
