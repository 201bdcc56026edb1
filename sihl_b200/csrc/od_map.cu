// od_map.cu — N3 (SURVEY.md §8f): the detection <-> ground-truth matching behind the validation mAP.
//
// The reference hands every validation batch to torchmetrics' MeanAveragePrecision (ref object_detection.py:219-237,
// :245; backend faster_coco_eval), whose compute() runs COCOeval on the CPU at epoch end: per image and category,
// detections in score order are greedily matched to the ground truth at the 10 IoU thresholds .50:.05:.95 and for
// the 4 area ranges (COCOeval.evaluateImg), then precision / recall curves are accumulated.  The matching is the
// part that scales with batch x detections x ground truth; it runs here, on the GPU, right after forward() —
// one CTA per image, one thread per (area range, IoU threshold) greedy chain, box IoU in fp64 as maskUtils.iou
// computes it on the xywh boxes torchmetrics builds (w = fl32(x2 - x1), h = fl32(y2 - y1)).
//
// Matching rule restated from pycocotools / faster_coco_eval COCOeval.evaluateImg (iscrowd == 0 for the plain entries;
// the _crowd entries add COCO's iscrowd and area annotations, see MapAnnotations and sihl_od.h):
//   gts of the category in input order, "ignored" ones (area outside the range) after the others;
//   for each detection d by (score desc, input order):  best = min(t, 1 - 1e-10), m = none
//       for each gt g in that order: skip g if already matched at this threshold;
//           stop if m is a regular gt and g is an ignored one; skip if iou(d, g) < best; best = iou(d, g), m = g
//       if m: d is matched to m (and inherits its ignore flag), m is taken
//       else: d is unmatched, and ignored iff its own area is outside the range.
// torchmetrics / faster_coco_eval are not installed in this environment: parity of this row is UNPINNED (the oracle,
// oracle/map_oracle.py, restates the same published algorithm).
#include "od_common.cuh"

namespace sihl {

constexpr int kMapMaxT = 16, kMapMaxA = 8, kMapMaxK = 1024;

struct MapParams {
    const float4 *det_boxes; const float *det_scores; const int64_t *det_classes; int K;
    const float4 *gt_boxes; const int64_t *gt_classes; const int32_t *gt_offsets;
    int n_thr, n_area;
    double thr[kMapMaxT];
    double area_lo[kMapMaxA], area_hi[kMapMaxA];
    int32_t *det_order;        // [B, K] rank -> detection
    int32_t *dt_match;         // [B, n_area, n_thr, K] by rank: global gt index or -1
    uint8_t *dt_ignore;        // [B, n_area, n_thr, K] by rank
    uint8_t *gt_ignore;        // [n_area, total_gt]
    int32_t *gt_taken;         // workspace [n_area, n_thr, total_gt]: 0 or 1 + rank of the detection that took the gt
    int total_gt;
};

__device__ __forceinline__ double box_area_d(float4 b)
{
    return (double)(b.z - b.x) * (double)(b.w - b.y);            // w, h rounded to fp32 first (torchmetrics box_convert)
}

// maskUtils.iou on xywh boxes (bbIou), in double: u = da + ga - i, or u = da against a crowd gt (kIoA, iscrowd = 1).
template <bool kIoA = false>
__device__ __forceinline__ double box_iou_d(float4 d, float4 g)
{
    const double dx = d.x, dy = d.y, dw = (double)(d.z - d.x), dh = (double)(d.w - d.y);
    const double gx = g.x, gy = g.y, gw = (double)(g.z - g.x), gh = (double)(g.w - g.y);
    const double w = fmin(dx + dw, gx + gw) - fmax(dx, gx);
    if (w <= 0.0) return 0.0;
    const double h = fmin(dy + dh, gy + gh) - fmax(dy, gy);
    if (h <= 0.0) return 0.0;
    const double i = w * h;
    const double u = kIoA ? dw * dh : dw * dh + gw * gh - i;
    return i / u;
}

// Where the chains of one image read their geometry: the box kernel computes IoU and area from the xyxy boxes, the quad
// kernel reads IoU from its precomputed matrix and areas from the hulls.  D is what a chain keeps of its detection.
// crowd_iou is the overlap with a crowd gt: the box IoA, or the matrix entry, which holds the IoA in crowd columns.
struct MapBoxGeometry {
    const float4 *db, *gb;
    __device__ __forceinline__ float4 det(int d) const { return __ldg(db + d); }
    __device__ __forceinline__ double det_area(float4 box) const { return box_area_d(box); }
    __device__ __forceinline__ double gt_area(int g) const { return box_area_d(__ldg(gb + g)); }
    __device__ __forceinline__ double iou(float4 box, int g) const { return box_iou_d(box, __ldg(gb + g)); }
    __device__ __forceinline__ double crowd_iou(float4 box, int g) const { return box_iou_d<true>(box, __ldg(gb + g)); }
};

// The optional COCO annotations of the ground truth (sihl_od_*map_match_crowd), [total_gt] each; NULL means none.
struct MapAnnotations {
    const uint8_t *crowd;             // nonzero: a crowd region
    const double *area;               // > 0: the area that places the gt in an area range
    __device__ __forceinline__ bool is_crowd(int g) const { return crowd != nullptr && __ldg(crowd + g) != 0; }
    __device__ __forceinline__ double range_area(int g, double computed) const
    {
        const double given = area != nullptr ? __ldg(area + g) : 0.0;
        return given > 0.0 ? given : computed;                  // NaN and <= 0 keep the computed area
    }
};

// No annotations: the plain entries.  Folds away, so their kernels are the code they were before annotations existed.
struct MapNoAnnotations {
    __device__ __forceinline__ bool is_crowd(int) const { return false; }
    __device__ __forceinline__ double range_area(int, double computed) const { return computed; }
};

// COCOeval.evaluateImg for image b (the rule above): rank the detections, flag the gts per area range, then one greedy
// chain per (area range, threshold) on a thread.  Shared by k_map_match and k_quad_map_match; inlined into each.
// Ann adds COCOeval's two gt annotations (MapAnnotations, the _crowd kernels): the annotated area replaces the computed
// one when it is > 0, and a crowd gt is ignored in every area range, overlaps a detection by crowd_iou and is never
// taken, so any number of detections may match it.
template <class Geo, class Ann>
__device__ __forceinline__ void map_match_image(const MapParams &p, const Geo &geo, const Ann &ann, int *s_order)
{
    const int b = blockIdx.x, tid = threadIdx.x, K = p.K;
    const float *sc = p.det_scores + (int64_t)b * K;
    const int64_t *dc = p.det_classes + (int64_t)b * K;
    const int g0 = __ldg(p.gt_offsets + b), g1 = __ldg(p.gt_offsets + b + 1);

    // detections by (score desc, input order): rank by counting (K <= 1024)
    for (int d = tid; d < K; d += blockDim.x) {
        const float s = __ldg(sc + d);
        int r = 0;
        for (int j = 0; j < K; ++j) {
            const float sj = __ldg(sc + j);
            r += (sj > s) || (sj == s && j < d);
        }
        s_order[r] = d;
        p.det_order[(int64_t)b * K + r] = d;
    }
    // ignore flags of this image's gts per area range; clear the "taken" markers
    for (int i = tid; i < (g1 - g0) * p.n_area; i += blockDim.x) {
        const int a = i / (g1 - g0), g = g0 + i % (g1 - g0);
        const double ar = ann.range_area(g, geo.gt_area(g));
        p.gt_ignore[(int64_t)a * p.total_gt + g] = (ann.is_crowd(g) || ar < p.area_lo[a] || ar > p.area_hi[a]) ? 1 : 0;
    }
    for (int i = tid; i < (g1 - g0) * p.n_area * p.n_thr; i += blockDim.x)
        p.gt_taken[(int64_t)(i / (g1 - g0)) * p.total_gt + g0 + i % (g1 - g0)] = 0;
    __syncthreads();

    // one greedy chain per (area range, threshold)
    for (int chain = tid; chain < p.n_area * p.n_thr; chain += blockDim.x) {
        const int a = chain / p.n_thr, t = chain % p.n_thr;
        const uint8_t *gig = p.gt_ignore + (int64_t)a * p.total_gt;
        int32_t *taken = p.gt_taken + (int64_t)chain * p.total_gt;
        int32_t *dtm = p.dt_match + (((int64_t)b * p.n_area + a) * p.n_thr + t) * K;
        uint8_t *dti = p.dt_ignore + (((int64_t)b * p.n_area + a) * p.n_thr + t) * K;
        const double thr = fmin(p.thr[t], 1.0 - 1e-10);
        for (int r = 0; r < K; ++r) {
            const int d = s_order[r];
            const int64_t cls = __ldg(dc + d);
            const auto det = geo.det(d);
            double best = thr;
            int m = -1;
            for (int pass = 0; pass < 2 && m < 0; ++pass) {        // regular gts first; ignored ones only while unmatched
                for (int g = g0; g < g1; ++g) {
                    if (__ldg(p.gt_classes + g) != cls || gig[g] != pass || taken[g] != 0) continue;
                    const double iou = ann.is_crowd(g) ? geo.crowd_iou(det, g) : geo.iou(det, g);
                    if (iou < best) continue;
                    best = iou;
                    m = g;
                }
            }
            if (m >= 0) {
                dtm[r] = m;
                dti[r] = gig[m];
                if (!ann.is_crowd(m)) taken[m] = r + 1;
            } else {
                const double ar = geo.det_area(det);
                dtm[r] = -1;
                dti[r] = (ar < p.area_lo[a] || ar > p.area_hi[a]) ? 1 : 0;
            }
        }
    }
}

__global__ void __launch_bounds__(128) k_map_match(const __grid_constant__ MapParams p)
{
    __shared__ int s_order[kMapMaxK];
    const MapBoxGeometry geo{p.det_boxes + (int64_t)blockIdx.x * p.K, p.gt_boxes};
    map_match_image(p, geo, MapNoAnnotations{}, s_order);
}

__global__ void __launch_bounds__(128) k_map_match_crowd(const __grid_constant__ MapParams p, MapAnnotations ann)
{
    __shared__ int s_order[kMapMaxK];
    const MapBoxGeometry geo{p.det_boxes + (int64_t)blockIdx.x * p.K, p.gt_boxes};
    map_match_image(p, geo, ann, s_order);
}

// ---- polygon IoU (sihl_od_quad_map_match): the same chains over quads ----------------------------------------------
// The overlap is od_math.h's hull IoU, the one sihl_od_batched_quad_nms suppresses with, and the area of a quad is its
// hull's polygon area.  A clip costs ~40x a box IoU, so it is not recomputed inside the chains (each chain would redo
// every pair of its image, 40 times per image, on one SM): k_quad_map_hulls builds every hull once, k_quad_map_iou fills
// the [K, G_b] fp32 IoU block of each image with the pairs spread over the whole GPU, and k_quad_map_match runs the
// chains above on that matrix.  Image b's block starts at K * gt_offsets[b]: the matrix is K * total_gt floats.
struct MapQuadGeometry {
    const float *m;                   // image b's [K, G_b] IoU block
    const QuadHull *dh, *gh;          // image b's detection hulls; every gt hull
    int g0, gn;
    __device__ __forceinline__ int det(int d) const { return d; }
    __device__ __forceinline__ double det_area(int d) const { return (double)__ldg(&dh[d].area); }
    __device__ __forceinline__ double gt_area(int g) const { return (double)__ldg(&gh[g].area); }
    __device__ __forceinline__ double iou(int d, int g) const { return (double)__ldg(m + (int64_t)d * gn + (g - g0)); }
    __device__ __forceinline__ double crowd_iou(int d, int g) const { return iou(d, g); }
};

// hulls[i] = quad_hull of detection i (i < n_det = B * K), then of gt i - n_det
__global__ void __launch_bounds__(256)
k_quad_map_hulls(const float *__restrict__ det_quads, int64_t n_det, const float *__restrict__ gt_quads, int64_t n_gt,
                 QuadHull *__restrict__ hulls)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_det + n_gt) return;
    const float *q = i < n_det ? det_quads + 8 * i : gt_quads + 8 * (i - n_det);
    float p[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) p[c] = __ldg(q + c);
    hulls[i] = quad_hull(p);
}

// One thread per (detection, gt) pair of the same image, grid-stride over the K * total_gt matrix.  Pair k lies in image
// b with K * g0 <= k < K * g1, i.e. gt_offsets[b] <= k / K < gt_offsets[b + 1].  Pairs of different classes are skipped
// (the chains test the class first and never read them); every same-class pair is written, an exact 0 included.  With
// kAnnotated, the columns of crowd gts hold the IoA of the detection instead (quad_ioa_hulls).
template <bool kAnnotated>
__device__ __forceinline__ void quad_map_iou_pairs(const QuadHull *__restrict__ hulls, const int64_t *__restrict__ det_classes,
                                                   const int64_t *__restrict__ gt_classes,
                                                   const int32_t *__restrict__ gt_offsets, int batch, int K, int total_gt,
                                                   const uint8_t *__restrict__ gt_crowd, float *__restrict__ iou)
{
    const int64_t n = (int64_t)K * total_gt, n_det = (int64_t)batch * K;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(k / K);                       // in [g0, g1) of the pair's image
        int lo = 0, hi = batch - 1;                         // last b with gt_offsets[b] <= row
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(gt_offsets + mid) <= row) lo = mid; else hi = mid - 1;
        }
        const int g0 = __ldg(gt_offsets + lo), gn = __ldg(gt_offsets + lo + 1) - g0;
        const int64_t local = k - (int64_t)K * g0;
        const int d = (int)(local / gn), g = g0 + (int)(local - (int64_t)d * gn);
        const int64_t di = (int64_t)lo * K + d;
        if (__ldg(det_classes + di) != __ldg(gt_classes + g)) continue;
        if (kAnnotated && gt_crowd != nullptr && __ldg(gt_crowd + g) != 0)
            iou[k] = quad_ioa_hulls(hulls[di], hulls[n_det + g]);
        else
            iou[k] = quad_iou_hulls(hulls[di], hulls[n_det + g]);
    }
}

__global__ void __launch_bounds__(256)
k_quad_map_iou(const QuadHull *__restrict__ hulls, const int64_t *__restrict__ det_classes,
               const int64_t *__restrict__ gt_classes, const int32_t *__restrict__ gt_offsets, int batch, int K,
               int total_gt, float *__restrict__ iou)
{
    quad_map_iou_pairs<false>(hulls, det_classes, gt_classes, gt_offsets, batch, K, total_gt, nullptr, iou);
}

__global__ void __launch_bounds__(256)
k_quad_map_iou_crowd(const QuadHull *__restrict__ hulls, const int64_t *__restrict__ det_classes,
                     const int64_t *__restrict__ gt_classes, const int32_t *__restrict__ gt_offsets, int batch, int K,
                     int total_gt, const uint8_t *__restrict__ gt_crowd, float *__restrict__ iou)
{
    quad_map_iou_pairs<true>(hulls, det_classes, gt_classes, gt_offsets, batch, K, total_gt, gt_crowd, iou);
}

// image b's geometry: its [K, G_b] block of the matrix, its detection hulls and every gt hull
__device__ __forceinline__ MapQuadGeometry quad_map_geometry(const MapParams &p, const float *iou, const QuadHull *hulls)
{
    const int b = blockIdx.x, g0 = __ldg(p.gt_offsets + b), g1 = __ldg(p.gt_offsets + b + 1);
    return MapQuadGeometry{iou + (int64_t)p.K * g0, hulls + (int64_t)b * p.K, hulls + (int64_t)gridDim.x * p.K, g0,
                           g1 - g0};
}

__global__ void __launch_bounds__(128)
k_quad_map_match(const __grid_constant__ MapParams p, const float *__restrict__ iou, const QuadHull *__restrict__ hulls)
{
    __shared__ int s_order[kMapMaxK];
    map_match_image(p, quad_map_geometry(p, iou, hulls), MapNoAnnotations{}, s_order);
}

__global__ void __launch_bounds__(128)
k_quad_map_match_crowd(const __grid_constant__ MapParams p, const float *__restrict__ iou,
                       const QuadHull *__restrict__ hulls, MapAnnotations ann)
{
    __shared__ int s_order[kMapMaxK];
    map_match_image(p, quad_map_geometry(p, iou, hulls), ann, s_order);
}

// workspace: the hulls of every detection and gt, the IoU matrix, the taken markers of the chains
struct QuadMapWorkspace {
    size_t hulls, iou, taken, bytes;
};

static QuadMapWorkspace quad_map_workspace(int batch, int k, int total_gt, int n_thresholds, int n_areas)
{
    QuadMapWorkspace w;
    w.hulls = 0;
    w.iou = round_up_256(((size_t)batch * k + total_gt) * sizeof(QuadHull));
    w.taken = w.iou + round_up_256((size_t)k * total_gt * sizeof(float));
    w.bytes = w.taken + (size_t)(total_gt > 0 ? total_gt : 1) * n_thresholds * n_areas * sizeof(int32_t);
    return w;
}

}  // namespace sihl

using namespace sihl;

extern "C" size_t sihl_od_map_workspace_bytes(int total_gt, int n_thresholds, int n_areas)
{
    if (total_gt < 0 || n_thresholds < 1 || n_areas < 1) return 0;
    return (size_t)(total_gt > 0 ? total_gt : 1) * (size_t)n_thresholds * (size_t)n_areas * sizeof(int32_t);
}

// sihl_od_map_match and sihl_od_map_match_crowd: ann with two NULL pointers launches the plain kernel.  empty_ok (the
// _crowd entry, as the quad entries): batch = 0 returns after the size checks, before the pointers are checked.
static int map_match_boxes(const float *det_boxes, const float *det_scores, const int64_t *det_classes, int batch, int k,
                           const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets, int total_gt,
                           MapAnnotations ann, const double *iou_thresholds_host, int n_thresholds,
                           const double *area_ranges_host, int n_areas, int32_t *det_order, int32_t *dt_match,
                           uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace, void *stream, bool empty_ok)
{
    if (empty_ok && batch == 0) {
        SIHL_CHECK_ARG(iou_thresholds_host && area_ranges_host, "NULL thresholds / area ranges");
        SIHL_CHECK_ARG(k >= 1 && k <= kMapMaxK && total_gt >= 0, "bad sizes (k=%d, at most %d detections per image)", k,
                       kMapMaxK);
        SIHL_CHECK_ARG(n_thresholds >= 1 && n_thresholds <= kMapMaxT && n_areas >= 1 && n_areas <= kMapMaxA,
                       "at most %d IoU thresholds and %d area ranges", kMapMaxT, kMapMaxA);
        return SIHL_OD_OK;                              // nothing is read or written: empty tensors may be NULL
    }
    SIHL_CHECK_ARG(det_boxes && det_scores && det_classes && gt_offsets && iou_thresholds_host && area_ranges_host, "NULL input");
    SIHL_CHECK_ARG(det_order && dt_match && dt_ignore && workspace, "NULL output / workspace");
    SIHL_CHECK_ARG(batch >= 0 && k >= 1 && k <= kMapMaxK && total_gt >= 0, "bad sizes (k=%d, at most %d detections per image)", k,
                   kMapMaxK);
    SIHL_CHECK_ARG(n_thresholds >= 1 && n_thresholds <= kMapMaxT && n_areas >= 1 && n_areas <= kMapMaxA,
                   "at most %d IoU thresholds and %d area ranges", kMapMaxT, kMapMaxA);
    SIHL_CHECK_ARG(total_gt == 0 || (gt_boxes && gt_classes && gt_ignore), "NULL ground truth");
    if (batch == 0) return SIHL_OD_OK;
    MapParams p;
    p.det_boxes = reinterpret_cast<const float4 *>(det_boxes); p.det_scores = det_scores; p.det_classes = det_classes; p.K = k;
    p.gt_boxes = reinterpret_cast<const float4 *>(gt_boxes); p.gt_classes = gt_classes; p.gt_offsets = gt_offsets;
    p.n_thr = n_thresholds; p.n_area = n_areas;
    for (int i = 0; i < n_thresholds; ++i) p.thr[i] = iou_thresholds_host[i];
    for (int i = 0; i < n_areas; ++i) { p.area_lo[i] = area_ranges_host[2 * i]; p.area_hi[i] = area_ranges_host[2 * i + 1]; }
    p.det_order = det_order; p.dt_match = dt_match; p.dt_ignore = dt_ignore; p.gt_ignore = gt_ignore;
    p.gt_taken = reinterpret_cast<int32_t *>(workspace); p.total_gt = total_gt;
    if (ann.crowd == nullptr && ann.area == nullptr) {
        k_map_match<<<batch, 128, 0, (cudaStream_t)stream>>>(p);
        SIHL_CHECK_LAUNCH("k_map_match");
    } else {
        k_map_match_crowd<<<batch, 128, 0, (cudaStream_t)stream>>>(p, ann);
        SIHL_CHECK_LAUNCH("k_map_match_crowd");
    }
    return SIHL_OD_OK;
}

extern "C" int sihl_od_map_match(const float *det_boxes, const float *det_scores, const int64_t *det_classes, int batch, int k,
                                 const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets, int total_gt,
                                 const double *iou_thresholds_host, int n_thresholds, const double *area_ranges_host,
                                 int n_areas, int32_t *det_order, int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore,
                                 void *workspace, void *stream)
{
    return map_match_boxes(det_boxes, det_scores, det_classes, batch, k, gt_boxes, gt_classes, gt_offsets, total_gt,
                           MapAnnotations{nullptr, nullptr}, iou_thresholds_host, n_thresholds, area_ranges_host, n_areas,
                           det_order, dt_match, dt_ignore, gt_ignore, workspace, stream, false);
}

extern "C" int sihl_od_map_match_crowd(const float *det_boxes, const float *det_scores, const int64_t *det_classes, int batch,
                                       int k, const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                                       int total_gt, const uint8_t *gt_crowd, const double *gt_area,
                                       const double *iou_thresholds_host, int n_thresholds, const double *area_ranges_host,
                                       int n_areas, int32_t *det_order, int32_t *dt_match, uint8_t *dt_ignore,
                                       uint8_t *gt_ignore, void *workspace, void *stream)
{
    return map_match_boxes(det_boxes, det_scores, det_classes, batch, k, gt_boxes, gt_classes, gt_offsets, total_gt,
                           MapAnnotations{gt_crowd, gt_area}, iou_thresholds_host, n_thresholds, area_ranges_host, n_areas,
                           det_order, dt_match, dt_ignore, gt_ignore, workspace, stream, true);
}

extern "C" size_t sihl_od_quad_map_workspace_bytes(int batch, int k, int total_gt, int n_thresholds, int n_areas)
{
    if (batch < 0 || k < 1 || k > kMapMaxK || total_gt < 0 || n_thresholds < 1 || n_thresholds > kMapMaxT ||
        n_areas < 1 || n_areas > kMapMaxA)
        return 0;
    return quad_map_workspace(batch, k, total_gt, n_thresholds, n_areas).bytes;
}

// sihl_od_quad_map_match and sihl_od_quad_map_match_crowd: ann with two NULL pointers launches the plain kernels
static int map_match_quads(const float *det_quads, const float *det_scores, const int64_t *det_classes, int batch, int k,
                           const float *gt_quads, const int64_t *gt_classes, const int32_t *gt_offsets, int total_gt,
                           MapAnnotations ann, const double *iou_thresholds_host, int n_thresholds,
                           const double *area_ranges_host, int n_areas, int32_t *det_order, int32_t *dt_match,
                           uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace, size_t workspace_bytes, void *stream)
{
    SIHL_CHECK_ARG(iou_thresholds_host && area_ranges_host, "NULL thresholds / area ranges");
    SIHL_CHECK_ARG(batch >= 0 && k >= 1 && k <= kMapMaxK && total_gt >= 0, "bad sizes (k=%d, at most %d detections per image)", k,
                   kMapMaxK);
    SIHL_CHECK_ARG(n_thresholds >= 1 && n_thresholds <= kMapMaxT && n_areas >= 1 && n_areas <= kMapMaxA,
                   "at most %d IoU thresholds and %d area ranges", kMapMaxT, kMapMaxA);
    if (batch == 0) return SIHL_OD_OK;                  // nothing is read or written: empty tensors may be NULL
    SIHL_CHECK_ARG(det_quads && det_scores && det_classes && gt_offsets, "NULL input");
    SIHL_CHECK_ARG(det_order && dt_match && dt_ignore && workspace, "NULL output / workspace");
    SIHL_CHECK_ARG(total_gt == 0 || (gt_quads && gt_classes && gt_ignore), "NULL ground truth");
    const QuadMapWorkspace w = quad_map_workspace(batch, k, total_gt, n_thresholds, n_areas);
    SIHL_CHECK_ARG(workspace_bytes >= w.bytes, "workspace of %zu bytes, %zu needed (sihl_od_quad_map_workspace_bytes)",
                   workspace_bytes, w.bytes);
    const bool annotated = ann.crowd != nullptr || ann.area != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    QuadHull *hulls = reinterpret_cast<QuadHull *>(ws + w.hulls);
    float *iou = reinterpret_cast<float *>(ws + w.iou);
    const int64_t n_det = (int64_t)batch * k;
    k_quad_map_hulls<<<(unsigned)((n_det + total_gt + 255) / 256), 256, 0, st>>>(det_quads, n_det, gt_quads, total_gt, hulls);
    SIHL_CHECK_LAUNCH("k_quad_map_hulls");
    if (total_gt > 0) {
        const int64_t pairs = (int64_t)k * total_gt;
        const int64_t blocks = (pairs + 255) / 256;
        const unsigned grid = (unsigned)(blocks < kNumSMs * 64 ? blocks : kNumSMs * 64);
        if (ann.crowd != nullptr) {                     // the area annotation does not change the matrix
            k_quad_map_iou_crowd<<<grid, 256, 0, st>>>(hulls, det_classes, gt_classes, gt_offsets, batch, k, total_gt,
                                                       ann.crowd, iou);
            SIHL_CHECK_LAUNCH("k_quad_map_iou_crowd");
        } else {
            k_quad_map_iou<<<grid, 256, 0, st>>>(hulls, det_classes, gt_classes, gt_offsets, batch, k, total_gt, iou);
            SIHL_CHECK_LAUNCH("k_quad_map_iou");
        }
    }
    MapParams p;
    p.det_boxes = nullptr; p.det_scores = det_scores; p.det_classes = det_classes; p.K = k;
    p.gt_boxes = nullptr; p.gt_classes = gt_classes; p.gt_offsets = gt_offsets;
    p.n_thr = n_thresholds; p.n_area = n_areas;
    for (int i = 0; i < n_thresholds; ++i) p.thr[i] = iou_thresholds_host[i];
    for (int i = 0; i < n_areas; ++i) { p.area_lo[i] = area_ranges_host[2 * i]; p.area_hi[i] = area_ranges_host[2 * i + 1]; }
    p.det_order = det_order; p.dt_match = dt_match; p.dt_ignore = dt_ignore; p.gt_ignore = gt_ignore;
    p.gt_taken = reinterpret_cast<int32_t *>(ws + w.taken); p.total_gt = total_gt;
    if (annotated) {
        k_quad_map_match_crowd<<<batch, 128, 0, st>>>(p, iou, hulls, ann);
        SIHL_CHECK_LAUNCH("k_quad_map_match_crowd");
    } else {
        k_quad_map_match<<<batch, 128, 0, st>>>(p, iou, hulls);
        SIHL_CHECK_LAUNCH("k_quad_map_match");
    }
    return SIHL_OD_OK;
}

extern "C" int sihl_od_quad_map_match(const float *det_quads, const float *det_scores, const int64_t *det_classes, int batch,
                                      int k, const float *gt_quads, const int64_t *gt_classes, const int32_t *gt_offsets,
                                      int total_gt, const double *iou_thresholds_host, int n_thresholds,
                                      const double *area_ranges_host, int n_areas, int32_t *det_order, int32_t *dt_match,
                                      uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace, size_t workspace_bytes,
                                      void *stream)
{
    return map_match_quads(det_quads, det_scores, det_classes, batch, k, gt_quads, gt_classes, gt_offsets, total_gt,
                           MapAnnotations{nullptr, nullptr}, iou_thresholds_host, n_thresholds, area_ranges_host, n_areas,
                           det_order, dt_match, dt_ignore, gt_ignore, workspace, workspace_bytes, stream);
}

extern "C" int sihl_od_quad_map_match_crowd(const float *det_quads, const float *det_scores, const int64_t *det_classes,
                                            int batch, int k, const float *gt_quads, const int64_t *gt_classes,
                                            const int32_t *gt_offsets, int total_gt, const uint8_t *gt_crowd,
                                            const double *gt_area, const double *iou_thresholds_host, int n_thresholds,
                                            const double *area_ranges_host, int n_areas, int32_t *det_order,
                                            int32_t *dt_match, uint8_t *dt_ignore, uint8_t *gt_ignore, void *workspace,
                                            size_t workspace_bytes, void *stream)
{
    return map_match_quads(det_quads, det_scores, det_classes, batch, k, gt_quads, gt_classes, gt_offsets, total_gt,
                           MapAnnotations{gt_crowd, gt_area}, iou_thresholds_host, n_thresholds, area_ranges_host, n_areas,
                           det_order, dt_match, dt_ignore, gt_ignore, workspace, workspace_bytes, stream);
}
