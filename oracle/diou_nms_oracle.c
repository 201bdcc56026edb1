/*
 * diou_nms_oracle.c — CPU restatement of class-aware DIoU-NMS (Zheng et al., "Distance-IoU Loss: Faster and Better
 * Learning for Bounding Box Regression", AAAI 2020), as include/sihl_od.h defines it for sihl_od_diou_nms_topk,
 * sihl_od_diou_nms_topk_split and sihl_od_batched_diou_nms.
 *
 * TEST INFRASTRUCTURE ONLY, beside od_oracle.c (whose greedy NMS and dense postprocess it mirrors with the DIoU test).
 * Arithmetic rules as there: fp32, one IEEE operation per source operator, built with -ffp-contract=off, never
 * -ffast-math.  The DIoU is torchvision's _box_diou_iou (tv:ops/boxes.py, eps = 1e-7) in its operator order.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define ORC_API __attribute__((visibility("default")))

/* distance_box_iou of boxes a and b (xyxy) */
ORC_API float orc_diou_pair(const float *a, const float *b)
{
    const float eps = 1e-7f;
    float area_a = (a[2] - a[0]) * (a[3] - a[1]);
    float area_b = (b[2] - b[0]) * (b[3] - b[1]);
    float w = fmaxf(0.f, fminf(a[2], b[2]) - fmaxf(a[0], b[0]));
    float h = fmaxf(0.f, fminf(a[3], b[3]) - fmaxf(a[1], b[1]));
    float inter = w * h;
    float iou = inter / ((area_a + area_b) - inter);
    float wi = fmaxf(0.f, fmaxf(a[2], b[2]) - fminf(a[0], b[0]));
    float hi = fmaxf(0.f, fmaxf(a[3], b[3]) - fminf(a[1], b[1]));
    float diag = ((wi * wi) + (hi * hi)) + eps;
    float dx = (a[0] + a[2]) / 2.f - (b[0] + b[2]) / 2.f;
    float dy = (a[1] + a[3]) / 2.f - (b[1] + b[3]) / 2.f;
    float cd = (dx * dx) + (dy * dy);
    return iou - (cd / diag);
}

typedef struct { float v; int64_t i; } orc_vi;
static int orc_cmp_desc(const void *x, const void *y)
{
    const orc_vi *a = (const orc_vi *)x, *b = (const orc_vi *)y;
    if (a->v > b->v) return -1;
    if (a->v < b->v) return 1;
    return (a->i < b->i) ? -1 : (a->i > b->i);
}

/* Visit boxes by (score desc, index asc); a kept box i suppresses every later box j of the same class with
 * diou(i, j) > thr (a NaN diou never suppresses).  keep: indices in visit order.  Returns M. */
ORC_API int64_t orc_batched_diou_nms(const float *boxes, const float *scores, const int64_t *classes,
                                     int64_t N, float thr, int64_t *keep)
{
    if (N == 0) return 0;
    orc_vi *ord = (orc_vi *)malloc(sizeof(orc_vi) * (size_t)N);
    for (int64_t i = 0; i < N; ++i) { ord[i].v = scores[i]; ord[i].i = i; }
    qsort(ord, (size_t)N, sizeof(orc_vi), orc_cmp_desc);
    unsigned char *dead = (unsigned char *)calloc((size_t)N, 1);
    int64_t m = 0;
    for (int64_t oi = 0; oi < N; ++oi) {
        int64_t i = ord[oi].i;
        if (dead[i]) continue;
        keep[m++] = i;
        for (int64_t oj = oi + 1; oj < N; ++oj) {
            int64_t j = ord[oj].i;
            if (dead[j] || classes[j] != classes[i]) continue;
            if (orc_diou_pair(boxes + 4 * i, boxes + 4 * j) > thr) dead[j] = 1;
        }
    }
    free(ord); free(dead);
    return m;
}

/* od_oracle.c's orc_dense_postprocess with DIoU-NMS: dense decode of every location (class = first argmax, score =
 * sigmoid(loc logit), candidates = score > score_thr, box decoded as ref :121), class-aware DIoU-NMS per image, the
 * first K kept detections in (score desc, location asc) order, zero padded. */
static inline float orc_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

ORC_API int orc_dense_postprocess_diou(const float *loc, const float *cls, const float *box_raw,
                                       int B, int64_t A, int C,
                                       const float *offsets, const float *scales, int img_w, int img_h,
                                       float score_thr, float diou_thr, int K,
                                       int64_t *num_instances, float *scores, int64_t *classes, float *boxes)
{
    const float size[4] = {(float)img_w, (float)img_h, (float)img_w, (float)img_h};
    float *cb = (float *)malloc(sizeof(float) * 4 * (size_t)A);
    float *cs = (float *)malloc(sizeof(float) * (size_t)A);
    int64_t *cc = (int64_t *)malloc(sizeof(int64_t) * (size_t)A);
    int64_t *keep = (int64_t *)malloc(sizeof(int64_t) * (size_t)A);
    for (int b = 0; b < B; ++b) {
        int64_t n = 0;
        for (int64_t a = 0; a < A; ++a) {
            int64_t flat = (int64_t)b * A + a;
            float s = orc_sigmoid(loc[flat]);
            if (!(s > score_thr)) continue;
            const float *z = cls + (int64_t)C * flat;
            int best = 0;
            for (int c = 1; c < C; ++c) if (z[c] > z[best]) best = c;
            for (int c = 0; c < 4; ++c)
                cb[4 * n + c] = (offsets[4 * a + c] + scales[4 * a + c] * expf(box_raw[4 * flat + c])) * size[c];
            cs[n] = s; cc[n] = best; ++n;
        }
        int64_t m = orc_batched_diou_nms(cb, cs, cc, n, diou_thr, keep);
        if (m > K) m = K;
        num_instances[b] = m;
        for (int k = 0; k < K; ++k) {
            int64_t r = (int64_t)b * K + k;
            if (k < m) {
                int64_t j = keep[k];
                scores[r] = cs[j]; classes[r] = cc[j];
                for (int c = 0; c < 4; ++c) boxes[4 * r + c] = cb[4 * j + c];
            } else {
                scores[r] = 0.f; classes[r] = 0;
                for (int c = 0; c < 4; ++c) boxes[4 * r + c] = 0.f;
            }
        }
    }
    free(cb); free(cs); free(cc); free(keep);
    return 0;
}
