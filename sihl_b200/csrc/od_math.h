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

// ---- quadrilateral overlap (sihl_od_batched_quad_nms, sihl_od_quad_iou) -------------------------------------------------
// A quad is 4 finite points (x, y) in pixels (finite is a precondition).  The overlap of two quads is the IoU of the
// CONVEX HULLS of their vertex sets: for a convex quad that is the polygon IoU whatever its start vertex and orientation,
// and a non-convex or self-intersecting ("bow-tie") vertex order still gets a defined value.
//   - The hull is a function of the point SET (the points are sorted first), so the result is bit-identical under any
//     permutation of a quad's vertices.
//   - A hull of zero area (collinear or repeated points) has IoU 0 with everything.  Disjoint AABBs give exactly 0, and
//     an AABB overlap of zero width counts as disjoint.
//   - inter is clamped to [0, min(area_a, area_b)];  iou = inter / ((area_a + area_b) - inter), 0 unless the union > 0.
//   - quad_iou(a, b) and quad_iou(b, a) are the same bits: the pair is put in a canonical order first.
//   - fp32 throughout, with +,-,*,/, explicit fmaf and comparisons only: -fmad=false on the device and -ffp-contract=off
//     on the host give the same bits.  Hull areas are taken about the hull's first vertex and the intersection about the lower corner of
//     the AABB intersection, never about the image origin, where shoelace terms of a small quad at x ~ 4096 cancel.
//   - The intersection clips hull A by the edges of hull B (Sutherland-Hodgman): every intermediate result is one closed
//     polygon, so a shared or touching edge whose side tests come out as rounding noise changes the area by noise only.

// Per-quad form, computed once per item: hull vertices CCW (3 of them repeat the third in slot 3; a zero-area hull has
// area 0), the hull area and the AABB of the points.
struct QuadHull {
    float x[4], y[4];
    float area;
    float x1, y1, x2, y2;
};

// ax * by - ay * bx with Kahan's difference of products (two fmaf, within 1.5 ulp): the plain form loses all digits of a
// thin slanted quad's area to cancellation.  fmaf is correctly rounded on the device and in the host's libm alike.
SIHL_HD float cross2(float ax, float ay, float bx, float by)
{
    const float w = ay * bx;
    const float e = fmaf(-ay, bx, w);
    const float f = fmaf(ax, by, -w);
    return f + e;
}

// compare-exchange on (x, y) lexicographic order
SIHL_HD void pt_sort2(float &ax, float &ay, float &bx, float &by)
{
    if (bx < ax || (bx == ax && by < ay)) {
        const float tx = ax, ty = ay;
        ax = bx; ay = by; bx = tx; by = ty;
    }
}

// p: x0, y0, x1, y1, x2, y2, x3, y3.  Andrew's monotone chain unrolled for four points.
SIHL_HD QuadHull quad_hull(const float *p)
{
    float x0 = p[0] + 0.f, y0 = p[1] + 0.f, x1 = p[2] + 0.f, y1 = p[3] + 0.f;   // + 0: -0 becomes +0, one order of zeros
    float x2 = p[4] + 0.f, y2 = p[5] + 0.f, x3 = p[6] + 0.f, y3 = p[7] + 0.f;
    QuadHull h;
    h.x1 = fminf(fminf(x0, x1), fminf(x2, x3)); h.x2 = fmaxf(fmaxf(x0, x1), fmaxf(x2, x3));
    h.y1 = fminf(fminf(y0, y1), fminf(y2, y3)); h.y2 = fmaxf(fmaxf(y0, y1), fmaxf(y2, y3));
    pt_sort2(x0, y0, x1, y1); pt_sort2(x2, y2, x3, y3);
    pt_sort2(x0, y0, x2, y2); pt_sort2(x1, y1, x3, y3);
    pt_sort2(x1, y1, x2, y2);
    // p0 and p3 are hull vertices; p1 / p2 lie below (c < 0), above (c > 0) or on the chord p0 -> p3
    const float dx = x3 - x0, dy = y3 - y0;
    const float c1 = cross2(dx, dy, x1 - x0, y1 - y0), c2 = cross2(dx, dy, x2 - x0, y2 - y0);
    bool k1 = c1 != 0.f, k2 = c2 != 0.f;
    if (c1 < 0.f && c2 < 0.f) {                             // both on the lower chain p0, p1, p2, p3
        k1 = cross2(x1 - x0, y1 - y0, x2 - x0, y2 - y0) > 0.f;
        k2 = !k1 || cross2(x2 - x1, y2 - y1, x3 - x1, y3 - y1) > 0.f;
    } else if (c1 > 0.f && c2 > 0.f) {                      // both on the upper chain p3, p2, p1, p0
        k2 = cross2(x2 - x3, y2 - y3, x1 - x3, y1 - y3) > 0.f;
        k1 = !k2 || cross2(x1 - x2, y1 - y2, x0 - x2, y0 - y2) > 0.f;
    }
    // CCW: p0, the kept lower points by x, p3, the kept upper points by decreasing x
    float hx[4] = {x0, x0, x0, x0}, hy[4] = {y0, y0, y0, y0};
    int m = 1;
    if (k1 && c1 < 0.f) { hx[m] = x1; hy[m] = y1; ++m; }
    if (k2 && c2 < 0.f) { hx[m] = x2; hy[m] = y2; ++m; }
    hx[m] = x3; hy[m] = y3; ++m;
    if (k2 && c2 > 0.f) { hx[m] = x2; hy[m] = y2; ++m; }
    if (k1 && c1 > 0.f) { hx[m] = x1; hy[m] = y1; ++m; }
    for (int i = m; i < 4; ++i) { hx[i] = hx[m - 1]; hy[i] = hy[m - 1]; }
    for (int i = 0; i < 4; ++i) { h.x[i] = hx[i]; h.y[i] = hy[i]; }
    const float t1 = cross2(hx[1] - hx[0], hy[1] - hy[0], hx[2] - hx[0], hy[2] - hy[0]);
    const float t2 = cross2(hx[2] - hx[0], hy[2] - hy[0], hx[3] - hx[0], hy[3] - hy[0]);
    h.area = m < 3 ? 0.f : (t1 + t2) * 0.5f;
    return h;
}

// true when hull b comes before hull a in the canonical order of a pair (lexicographic on the vertex slots, which
// determine the hull; no NaN and no -0 can occur there)
SIHL_HD bool quad_hull_before(const QuadHull &b, const QuadHull &a)
{
    for (int i = 0; i < 4; ++i) {
        if (b.x[i] != a.x[i]) return b.x[i] < a.x[i];
        if (b.y[i] != a.y[i]) return b.y[i] < a.y[i];
    }
    return false;
}

constexpr int kQuadClipMax = 8;     // a convex 4-gon clipped by 4 half-planes has at most 8 vertices

// Overlap of two hulls: the intersection, clamped to [0, min(area_a, area_b)], over the union (kIoA = false, the IoU) or
// over qa's area alone (kIoA = true, the IoA: COCOeval's overlap of a detection qa with a crowd region qb).  Both are 0
// for disjoint AABBs or a zero-area hull.  Sutherland-Hodgman of the first hull of the canonical pair against the
// second's edges, about the lower corner of the AABB intersection.  A vertex on an edge's line counts as inside; a
// crossing point is emitted only for a strict sign change.  Rounding on nearly collinear chains could in principle emit
// more than kQuadClipMax points: those past the cap are dropped, which keeps the result defined and changes the area by
// rounding noise only.  One body for both forms, so that the intersection they divide is the same bits.
template <bool kIoA>
SIHL_HD float quad_overlap_hulls(const QuadHull &qa, const QuadHull &qb)
{
    const bool swap = quad_hull_before(qb, qa);
    const QuadHull &a = swap ? qb : qa;
    const QuadHull &b = swap ? qa : qb;
    const float ox = fmaxf(a.x1, b.x1), oy = fmaxf(a.y1, b.y1);
    if (!(fminf(a.x2, b.x2) > ox) || !(fminf(a.y2, b.y2) > oy)) return 0.f;
    if (!(a.area > 0.f) || !(b.area > 0.f)) return 0.f;
    float px[kQuadClipMax], py[kQuadClipMax], qx[kQuadClipMax], qy[kQuadClipMax];
    int n = 4;
    for (int i = 0; i < 4; ++i) { px[i] = a.x[i] - ox; py[i] = a.y[i] - oy; }
    for (int e = 0; e < 4 && n > 0; ++e) {
        const float ex = b.x[e] - ox, ey = b.y[e] - oy;
        const float fx = b.x[(e + 1) & 3] - ox, fy = b.y[(e + 1) & 3] - oy;
        const float dx = fx - ex, dy = fy - ey;
        int m = 0;
        float sc = cross2(dx, dy, px[0] - ex, py[0] - ey);
        for (int i = 0; i < n; ++i) {
            const int j = i + 1 < n ? i + 1 : 0;
            const float sn = cross2(dx, dy, px[j] - ex, py[j] - ey);
            if (sc >= 0.f) {
                if (m < kQuadClipMax) { qx[m] = px[i]; qy[m] = py[i]; }
                ++m;
            }
            if ((sc > 0.f && sn < 0.f) || (sc < 0.f && sn > 0.f)) {
                const float t = sc / (sc - sn);
                if (m < kQuadClipMax) { qx[m] = px[i] + t * (px[j] - px[i]); qy[m] = py[i] + t * (py[j] - py[i]); }
                ++m;
            }
            sc = sn;
        }
        n = m < kQuadClipMax ? m : kQuadClipMax;
        for (int i = 0; i < n; ++i) { px[i] = qx[i]; py[i] = qy[i]; }
    }
    float s = 0.f;                                          // fan about the first vertex: no cancelling terms
    for (int i = 1; i + 1 < n; ++i) s = s + cross2(px[i] - px[0], py[i] - py[0], px[i + 1] - px[0], py[i + 1] - py[0]);
    const float lim = fminf(a.area, b.area);
    float inter = s * 0.5f;
    inter = inter > 0.f ? (inter < lim ? inter : lim) : 0.f;
    if (kIoA) return inter / qa.area;                       // qa.area > 0 here, and inter <= qa.area
    const float uni = (a.area + b.area) - inter;
    return uni > 0.f ? inter / uni : 0.f;
}

// IoU of two hulls
SIHL_HD float quad_iou_hulls(const QuadHull &qa, const QuadHull &qb) { return quad_overlap_hulls<false>(qa, qb); }

// intersection of two hulls over the area of the first
SIHL_HD float quad_ioa_hulls(const QuadHull &qa, const QuadHull &qb) { return quad_overlap_hulls<true>(qa, qb); }

// quad_iou of two quads given as 8 floats each
SIHL_HD float quad_iou(const float *a, const float *b) { return quad_iou_hulls(quad_hull(a), quad_hull(b)); }

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
