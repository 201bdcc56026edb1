// od_math.h — scalar arithmetic of the detection-head path, shared by every kernel.
//
// Plain C++ with no CUDA types so that tests/ can also compile these functions
// for the host (g++ -ffp-contract=off) and check the analytic gradients against
// torch autograd where no GPU exists.  The product only ever calls them from
// device code (compiled with -fmad=false, IEEE division, no fast-math).
//
// Operator order follows the torch / torchvision eager code line by line; see
// SURVEY.md §7.1 for why (bit equality of assignment indices with torch-CUDA).
#pragma once

#include <math.h>

#if defined(__CUDACC__)
#define SIHL_HD __host__ __device__ __forceinline__
#else
#define SIHL_HD static inline
#endif

namespace sihl {

struct Box4 {
    float x1, y1, x2, y2;
};

// Per-box terms of torchvision.ops.complete_box_iou hoisted out of the pair loop:
// tv:ops/boxes.py:273-303 (area), :470-473 (centres), :428-431 (atan(w/h)).
struct BoxTerms {
    float x1, y1, x2, y2, area, cx, cy, at;
};

SIHL_HD BoxTerms box_terms(Box4 b)
{
    BoxTerms t;
    t.x1 = b.x1; t.y1 = b.y1; t.x2 = b.x2; t.y2 = b.y2;
    const float w = b.x2 - b.x1, h = b.y2 - b.y1;
    t.area = w * h;
    t.cx = (b.x1 + b.x2) / 2.f;
    t.cy = (b.y1 + b.y2) / 2.f;
    t.at = atanf(w / h);
    return t;
}

#define SIHL_FOUR_OVER_PI2 ((float)(4.0 / (3.14159265358979323846 * 3.14159265358979323846)))

// complete_box_iou for one (anchor, gt) pair — tv:ops/boxes.py:404-434, :462-480, :308-341.
// Not clamped: the caller applies clamp(0) (ref object_detection.py:263).
SIHL_HD float ciou_pair(const BoxTerms &a, const BoxTerms &g)
{
    const float eps = 1e-7f;
    float w = fminf(a.x2, g.x2) - fmaxf(a.x1, g.x1);
    float h = fminf(a.y2, g.y2) - fmaxf(a.y1, g.y1);
    w = w < 0.f ? 0.f : w;
    h = h < 0.f ? 0.f : h;
    const float inter = w * h;
    const float uni = (a.area + g.area) - inter;
    const float iou = inter / uni;
    float wi = fmaxf(a.x2, g.x2) - fminf(a.x1, g.x1);
    float hi = fmaxf(a.y2, g.y2) - fminf(a.y1, g.y1);
    wi = wi < 0.f ? 0.f : wi;
    hi = hi < 0.f ? 0.f : hi;
    const float diag = ((wi * wi) + (hi * hi)) + eps;
    const float dx = a.cx - g.cx, dy = a.cy - g.cy;
    const float cd = (dx * dx) + (dy * dy);
    const float diou = iou - (cd / diag);
    const float da = a.at - g.at;
    const float v = SIHL_FOUR_OVER_PI2 * (da * da);
    const float alpha = v / (((1.f - iou) + v) + eps);
    return diou - (alpha * v);
}

// torchvision.ops.distance_box_iou for one pair (tv:ops/boxes.py _box_diou_iou, eps = 1e-7): the IoU in the operator
// order of the hard NMS, minus the squared distance of the centres over the squared diagonal of the enclosing box.
// area_a / area_b are (x2 - x1) * (y2 - y1).  Bitwise symmetric in (a, b); NaN only when both boxes have zero area.
// The DIoU-NMS suppression test (Zheng et al., AAAI 2020) is diou_pair(kept, later) > thr.
SIHL_HD float diou_pair(Box4 a, float area_a, Box4 b, float area_b)
{
    const float eps = 1e-7f;
    const float w = fmaxf(0.f, fminf(a.x2, b.x2) - fmaxf(a.x1, b.x1));
    const float h = fmaxf(0.f, fminf(a.y2, b.y2) - fmaxf(a.y1, b.y1));
    const float inter = w * h;
    const float iou = inter / ((area_a + area_b) - inter);
    const float wi = fmaxf(0.f, fmaxf(a.x2, b.x2) - fminf(a.x1, b.x1));
    const float hi = fmaxf(0.f, fmaxf(a.y2, b.y2) - fminf(a.y1, b.y1));
    const float diag = ((wi * wi) + (hi * hi)) + eps;
    const float dx = (a.x1 + a.x2) / 2.f - (b.x1 + b.x2) / 2.f;
    const float dy = (a.y1 + a.y2) / 2.f - (b.y1 + b.y2) / 2.f;
    const float cd = (dx * dx) + (dy * dy);
    return iou - (cd / diag);
}

// torchvision.ops.complete_box_iou_loss for one row — tv:ops/ciou_loss.py:47-64,
// tv:ops/diou_loss.py:64-91, tv:ops/_utils.py:87-106.  If grad != nullptr it receives
// dLoss/d(pred x1,y1,x2,y2) with alpha held constant (ciou_loss.py:61-62) and the
// intersection differentiable only where it is non-empty (_utils.py:101-103).
// max/min ties split the gradient evenly, as torch.max/min backward do.
SIHL_HD float ciou_loss_row(Box4 p, Box4 t, float *grad)
{
    const float eps = 1e-7f;
    const float xk1 = fmaxf(p.x1, t.x1), yk1 = fmaxf(p.y1, t.y1);
    const float xk2 = fminf(p.x2, t.x2), yk2 = fminf(p.y2, t.y2);
    const bool overlap = (yk2 > yk1) && (xk2 > xk1);
    const float iw = xk2 - xk1, ih = yk2 - yk1;
    const float inter = overlap ? iw * ih : 0.f;
    const float wp = p.x2 - p.x1, hp = p.y2 - p.y1;
    const float wg = t.x2 - t.x1, hg = t.y2 - t.y1;
    const float uni = ((wp * hp) + (wg * hg)) - inter;
    const float ue = uni + eps;
    const float iou = inter / ue;
    const float xc1 = fminf(p.x1, t.x1), yc1 = fminf(p.y1, t.y1);
    const float xc2 = fmaxf(p.x2, t.x2), yc2 = fmaxf(p.y2, t.y2);
    const float cw = xc2 - xc1, ch = yc2 - yc1;
    const float diag = ((cw * cw) + (ch * ch)) + eps;
    const float xp = (p.x2 + p.x1) / 2.f, yp = (p.y2 + p.y1) / 2.f;
    const float xg = (t.x1 + t.x2) / 2.f, yg = (t.y1 + t.y2) / 2.f;
    const float dx = xp - xg, dy = yp - yg;
    const float cd = (dx * dx) + (dy * dy);
    const float dterm = cd / diag;
    const float theta_g = atanf(wg / hg), theta_p = atanf(wp / hp);
    const float da = theta_g - theta_p;
    const float v = SIHL_FOUR_OVER_PI2 * (da * da);
    const float alpha = v / (((1.f - iou) + v) + eps);
    const float loss = ((1.f - iou) + dterm) + alpha * v;
    if (grad) {
        // d(inter)/d(pred): through max/min selectors, only where the boxes overlap
        auto sel_gt = [](float a, float b) { return a > b ? 1.f : (a == b ? 0.5f : 0.f); };   // d max(a,b)/da
        auto sel_lt = [](float a, float b) { return a < b ? 1.f : (a == b ? 0.5f : 0.f); };   // d min(a,b)/da
        const float ov = overlap ? 1.f : 0.f;
        const float di[4] = {-ov * ih * sel_gt(p.x1, t.x1), -ov * iw * sel_gt(p.y1, t.y1),
                             ov * ih * sel_lt(p.x2, t.x2), ov * iw * sel_lt(p.y2, t.y2)};
        const float dap[4] = {-hp, -wp, hp, wp};                                      // d(area_pred)
        const float dcw[4] = {-sel_lt(p.x1, t.x1), 0.f, sel_gt(p.x2, t.x2), 0.f};      // d(cw)
        const float dch[4] = {0.f, -sel_lt(p.y1, t.y1), 0.f, sel_gt(p.y2, t.y2)};      // d(ch)
        const float ddx[4] = {0.5f, 0.f, 0.5f, 0.f}, ddy[4] = {0.f, 0.5f, 0.f, 0.5f};
        const float r2 = (wp * wp) + (hp * hp);
        const float dth_dw = hp / r2, dth_dh = -wp / r2;                               // d atan(wp/hp)
        const float dth[4] = {-dth_dw, -dth_dh, dth_dw, dth_dh};
        for (int c = 0; c < 4; ++c) {
            const float duni = dap[c] - di[c];
            const float diou = (di[c] * ue - inter * duni) / (ue * ue);
            const float dcd = 2.f * dx * ddx[c] + 2.f * dy * ddy[c];
            const float ddiag = 2.f * cw * dcw[c] + 2.f * ch * dch[c];
            const float ddterm = (dcd * diag - cd * ddiag) / (diag * diag);
            const float dv = SIHL_FOUR_OVER_PI2 * 2.f * da * (-dth[c]);
            grad[c] = -diou + ddterm + alpha * dv;
        }
    }
    return loss;
}

// binary_cross_entropy_with_logits for one element, target t in {0,1}:
// (1-t)*x - log_sigmoid(x)  (aten/src/ATen/native/Loss.cpp).
SIHL_HD float bce_logits(float x, float t)
{
    return (1.f - t) * x + (fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x))));
}

// sigmoid as ATen: 1 / (1 + exp(-x)).
SIHL_HD float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// ref object_detection.py:121 / :189 — one normalised coordinate of the decoded box.
SIHL_HD float decode_norm(float off, float sc, float raw) { return off + sc * expf(raw); }

}  // namespace sihl
