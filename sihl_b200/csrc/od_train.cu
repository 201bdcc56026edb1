// od_train.cu — the loss half of the drop-in head's training step (SURVEY.md §8 a5-a10, §7.4, §8f N2):
// one launch forward (four loss sums + finalize), one launch backward (four gradients), on head outputs
// of any of the three map types, with the number of positives read on the device.
//
//   k_train_loss      ref object_detection.py:157-217 (+ torchvision ciou_loss.py)
//   k_train_loss_bwd  d/d loc_logits, iou_preds, box rows, class rows
//
// Both kernels split their grid by role: the first `dense_blocks` CTAs stream the dense maps
// (loc_logits / iou_preds / rel_iou: HBM-bound, 12 B per anchor forward, 20 B backward), the others take
// the compact positive rows (gather-bound, (16+4C) B per positive).  The roles share nothing but the 8
// fp64 sums, so one launch does the dense losses, the positive-row losses and the finalize (and, backward,
// both gradient halves).
// Compact rows: row r of box_rows / cls_rows belongs to location pos_index[r]; only the first
// P = min(*pos_total, pos_capacity) rows are real (see sihl_od.h).
#include "od_common.cuh"
#include "od_pos.cuh"

namespace sihl {

constexpr int kTrainThreads = 256;

struct TrainLossParams {
    const void *loc; const void *iou_pred; const void *box_rows; const void *cls_rows;
    int64_t n_dense; int num_anchors; int num_classes;
    const float *rel; const int64_t *assignment;
    const int32_t *pos_index; int64_t pos_capacity; const int32_t *pos_total;
    const float4 *offsets; const float4 *scales; float img_w, img_h;
    const float4 *gt_boxes; const int64_t *gt_classes; const int32_t *gt_offsets;
    double *sums; float *losses;
    int dense_blocks, pos_blocks;
    int cls_vec;               // class rows are read / written 16 bytes at a time (C * sizeof(T) % 16 == 0, aligned bases)
    // backward
    const float *grad_losses; float grad_scale;
    void *dloc; void *diou; void *dbox; void *dcls;
};

__device__ __forceinline__ int64_t train_pos_count(const TrainLossParams &p)
{
    const int64_t m = __ldg(p.pos_total);
    return m < p.pos_capacity ? m : p.pos_capacity;
}

// binary_cross_entropy_with_logits term as the reference evaluates it on a map of type T (ref :160-161):
// ATen computes (1 - t) * x - log_sigmoid(x) with log_sigmoid run in the INPUT dtype — for half logits its result
// (min(0,x) - log1p(exp(-|x|)), evaluated in fp32) is rounded to half before it enters the fp32 expression.
template <typename T> __device__ __forceinline__ float bce_term(float x, float t)
{
    const float ls = fminf(0.f, x) - log1pf(expf(-fabsf(x)));
    return (1.f - t) * x - round_to<T>(ls);
}
template <> __device__ __forceinline__ float bce_term<float>(float x, float t) { return bce_logits(x, t); }

// Class target of positive row r (ref :201-203), or -1 if the label is outside [0, C).
__device__ __forceinline__ int pos_target(const TrainLossParams &p, int64_t flat, int b)
{
    const int g = __ldg(p.gt_offsets + b) + (int)__ldg(p.assignment + flat);
    const int64_t t = __ldg(p.gt_classes + g);
    return (t >= 0 && t < p.num_classes) ? (int)t : -1;
}

template <typename T>
__global__ void __launch_bounds__(kTrainThreads) k_train_loss(TrainLossParams p)
{
    __shared__ double s_red[5 * 32];
    __shared__ bool s_last;
    const int tid = threadIdx.x;
    if ((int)blockIdx.x < p.dense_blocks) {
        // ---- dense role: ref :157-163, :175-180
        const T *loc = reinterpret_cast<const T *>(p.loc), *iou_pred = reinterpret_cast<const T *>(p.iou_pred);
        double v[5] = {0, 0, 0, 0, 0};
        const int64_t n = p.n_dense, stride = (int64_t)p.dense_blocks * blockDim.x;
        for (int64_t base = (int64_t)blockIdx.x * blockDim.x + tid; base < n; base += 4 * stride) {
            float bce = 0.f, one = 0.f, mse = 0.f, rs = 0.f, np = 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t i = base + u * stride;
                if (i < n) {
                    const float r = __ldg(p.rel + i);
                    const float t = (r == 1.0f) ? 1.f : 0.f;
                    bce += bce_term<T>(ldf(loc + i), t);
                    one += t;
                    if (iou_pred != nullptr) { const float d = ldf(iou_pred + i) - r; mse += d * d; }
                    rs += r;
                    np += (r > 0.f) ? 1.f : 0.f;
                }
            }
            v[0] += bce; v[1] += one; v[2] += mse; v[3] += rs; v[4] += np;
        }
        const int slot[5] = {0, 1, 2, 3, 6};
        block_accumulate<5>(v, s_red, p.sums, slot);
    } else {
        // ---- positive-row role: ref :187-208
        const T *box_rows = reinterpret_cast<const T *>(p.box_rows), *cls_rows = reinterpret_cast<const T *>(p.cls_rows);
        const int64_t n = train_pos_count(p);
        const int A = p.num_anchors, C = p.num_classes;
        const int64_t first = (int64_t)((int)blockIdx.x - p.dense_blocks) * blockDim.x + tid;
        const int64_t nthreads = (int64_t)p.pos_blocks * blockDim.x;
        float acc_box = 0.f, acc_cls = 0.f;
        if (box_rows != nullptr) {                                    // thread per positive row
            for (int64_t r = first; r < n; r += nthreads) {
                const int64_t flat = __ldg(p.pos_index + r);
                const int b = (int)(flat / A), a = (int)(flat - (int64_t)b * A);
                const int g = __ldg(p.gt_offsets + b) + (int)__ldg(p.assignment + flat);
                const float l = pos_box_loss(ldf4(box_rows + 4 * r), __ldg(p.offsets + a), __ldg(p.scales + a),
                                             __ldg(p.gt_boxes + g), p.img_w, p.img_h);
                acc_box += __ldg(p.rel + flat) * l;                   // ref :197
            }
        }
        if (cls_rows != nullptr) {                                    // 4 lanes (16-byte loads) or 8 lanes per positive row
            const int lsh = p.cls_vec ? 2 : 3, lpr = 1 << lsh;
            const int gl = tid & (lpr - 1);
            const int64_t ngrp = nthreads >> lsh, grp = first >> lsh;
            const int64_t rounds = (n + ngrp - 1) / ngrp;
            for (int64_t it = 0; it < rounds; ++it) {
                const int64_t r = it * ngrp + grp;
                const bool ok = r < n;
                const int64_t rr = ok ? r : 0;
                const int64_t flat = __ldg(p.pos_index + rr);
                const int b = (int)(flat / A);
                const int tgt = pos_target(p, flat, b);
                const T *z = cls_rows + rr * C;
                float m = -CUDART_INF_F, s = 0.f;
                if (p.cls_vec) {                                      // 16-byte loads: 4 lanes x 64 contiguous bytes per step
                    constexpr int N = Vec16<T>::N;
                    const int CV = C / N;
                    for (int v = gl; v < CV; v += 4) {
                        float x[N];
                        ld_vec16(z + v * N, x);
#pragma unroll
                        for (int e = 0; e < N; ++e) m = fmaxf(m, x[e]);
                    }
                    m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 2));
                    m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 1));
                    for (int v = gl; v < CV; v += 4) {                // second pass: L1 hits
                        float x[N];
                        ld_vec16(z + v * N, x);
#pragma unroll
                        for (int e = 0; e < N; ++e) s += expf(x[e] - m);
                    }
                    s += __shfl_xor_sync(kFullMask, s, 2);
                    s += __shfl_xor_sync(kFullMask, s, 1);
                } else {
                    for (int c = gl; c < C; c += 8) m = fmaxf(m, ldf(z + c));
#pragma unroll
                    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
                    for (int c = gl; c < C; c += 8) s += expf(ldf(z + c) - m);
#pragma unroll
                    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
                }
                if (ok && gl == 0) {
                    const float ce = tgt >= 0 ? (logf(s) + m) - ldf(z + tgt) : CUDART_NAN_F;   // ref :205-207
                    acc_cls += __ldg(p.rel + flat) * ce;              // ref :208
                }
            }
        }
        double v[2] = {acc_box, acc_cls};
        const int slot[2] = {4, 5};
        block_accumulate<2>(v, s_red, p.sums, slot);
    }
    if (p.losses != nullptr) {                                        // last CTA out computes the five losses
        if (tid == 0) {
            __threadfence();
            s_last = atomicAdd(p.sums + 7, 1.0) == (double)(gridDim.x - 1);
        }
        __syncthreads();
        if (s_last && tid == 0) {
            __threadfence();
            finalize_losses(const_cast<const double *>(reinterpret_cast<volatile double *>(p.sums)), p.losses);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kTrainThreads) k_train_loss_bwd(TrainLossParams p)
{
    const int tid = threadIdx.x;
    const float gt_ = p.grad_losses ? __ldg(p.grad_losses + 4) : 1.f;        // d / d total, ref :210
    const bool early = p.sums[6] == 0.0;                                      // ref :165-172: only the location loss
    if ((int)blockIdx.x < p.dense_blocks) {
        const T *loc = reinterpret_cast<const T *>(p.loc), *iou_pred = reinterpret_cast<const T *>(p.iou_pred);
        T *dloc = reinterpret_cast<T *>(p.dloc), *diou = reinterpret_cast<T *>(p.diou);
        const float g_loc = ((p.grad_losses ? __ldg(p.grad_losses + 0) : 0.f) + gt_ * 1.f) * p.grad_scale;
        const float g_iou = ((p.grad_losses ? __ldg(p.grad_losses + 3) : 0.f) + gt_ * 1.f) * p.grad_scale;
        const float inv_one = (float)((double)g_loc / p.sums[1]);
        const float inv_rel2 = early ? 0.f : (float)(2.0 * (double)g_iou / p.sums[3]);
        const int64_t n = p.n_dense;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < n; i += (int64_t)p.dense_blocks * blockDim.x) {
            const float r = __ldg(p.rel + i);
            if (dloc != nullptr) dloc[i] = from_f<T>((sigmoid_f(ldf(loc + i)) - ((r == 1.0f) ? 1.f : 0.f)) * inv_one);
            if (diou != nullptr) diou[i] = from_f<T>(early ? 0.f : (ldf(iou_pred + i) - r) * inv_rel2);
        }
        return;
    }
    const T *box_rows = reinterpret_cast<const T *>(p.box_rows), *cls_rows = reinterpret_cast<const T *>(p.cls_rows);
    T *dbox = reinterpret_cast<T *>(p.dbox), *dcls = reinterpret_cast<T *>(p.dcls);
    const int64_t n = early ? 0 : train_pos_count(p);
    const int A = p.num_anchors, C = p.num_classes;
    const float g_box = ((p.grad_losses ? __ldg(p.grad_losses + 1) : 0.f) + gt_ * 10.f) * p.grad_scale;
    const float g_cls = ((p.grad_losses ? __ldg(p.grad_losses + 2) : 0.f) + gt_ * 1.f) * p.grad_scale;
    const float inv_w = early ? 0.f : (float)(1.0 / p.sums[3]);
    const int64_t first = (int64_t)((int)blockIdx.x - p.dense_blocks) * blockDim.x + tid;
    const int64_t nthreads = (int64_t)p.pos_blocks * blockDim.x;
    if (dbox != nullptr) {
        for (int64_t r = first; r < p.pos_capacity; r += nthreads) {
            float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < n) {
                const int64_t flat = __ldg(p.pos_index + r);
                const int b = (int)(flat / A), a = (int)(flat - (int64_t)b * A);
                const int g = __ldg(p.gt_offsets + b) + (int)__ldg(p.assignment + flat);
                const float4 raw = ldf4(box_rows + 4 * r), off = __ldg(p.offsets + a), sc = __ldg(p.scales + a);
                Box4 pred, tgt;
                pos_boxes(raw, off, sc, __ldg(p.gt_boxes + g), p.img_w, p.img_h, &pred, &tgt);
                float gr[4];
                ciou_loss_row(pred, tgt, gr);
                const float k = g_box * __ldg(p.rel + flat) * inv_w;      // ref :197, :210
                // d pred_j / d raw_j = scales_j * exp(raw_j) = pred_j - offsets_j
                out = make_float4(k * gr[0] * (pred.x1 - off.x), k * gr[1] * (pred.y1 - off.y),
                                  k * gr[2] * (pred.x2 - off.z), k * gr[3] * (pred.y2 - off.w));
            }
            stf4(dbox + 4 * r, out);
        }
    }
    if (dcls != nullptr) {
        const int lsh = p.cls_vec ? 2 : 3, lpr = 1 << lsh;             // 4 lanes (16-byte accesses) or 8 lanes per row
        const int gl = tid & (lpr - 1);
        const int64_t ngrp = nthreads >> lsh, grp = first >> lsh;
        const int64_t rounds = (p.pos_capacity + ngrp - 1) / ngrp;
        for (int64_t it = 0; it < rounds; ++it) {
            const int64_t r = it * ngrp + grp;
            if (r >= p.pos_capacity) continue;                        // group-uniform (the lanes of a group share r)
            T *out = dcls + r * C;
            constexpr int N = Vec16<T>::N;
            const int CV = C / N;
            if (r >= n) {                                             // padding row: zero gradient
                if (p.cls_vec) {
                    float zero[N];
#pragma unroll
                    for (int e = 0; e < N; ++e) zero[e] = 0.f;
                    for (int v = gl; v < CV; v += 4) st_vec16(out + v * N, zero);
                } else {
                    for (int c = gl; c < C; c += 8) out[c] = from_f<T>(0.f);
                }
                continue;
            }
            const int64_t flat = __ldg(p.pos_index + r);
            const int b = (int)(flat / A);
            const int tgt = pos_target(p, flat, b);
            const T *z = cls_rows + r * C;
            // the lanes of a group may diverge from the other groups of the warp: group-local shuffles
            const unsigned gmask = (lpr == 4 ? 0xfu : 0xffu) << ((tid & 31) & ~(lpr - 1));
            float m = -CUDART_INF_F, s = 0.f;
            if (p.cls_vec) {
                for (int v = gl; v < CV; v += 4) {
                    float x[N];
                    ld_vec16(z + v * N, x);
#pragma unroll
                    for (int e = 0; e < N; ++e) m = fmaxf(m, x[e]);
                }
                m = fmaxf(m, __shfl_xor_sync(gmask, m, 2));
                m = fmaxf(m, __shfl_xor_sync(gmask, m, 1));
                for (int v = gl; v < CV; v += 4) {
                    float x[N];
                    ld_vec16(z + v * N, x);
#pragma unroll
                    for (int e = 0; e < N; ++e) s += expf(x[e] - m);
                }
                s += __shfl_xor_sync(gmask, s, 2);
                s += __shfl_xor_sync(gmask, s, 1);
            } else {
                for (int c = gl; c < C; c += 8) m = fmaxf(m, ldf(z + c));
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(gmask, m, o));
                for (int c = gl; c < C; c += 8) s += expf(ldf(z + c) - m);
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(gmask, s, o);
            }
            const float k = tgt >= 0 ? g_cls * __ldg(p.rel + flat) * inv_w : CUDART_NAN_F;   // ref :208
            const float inv_s = 1.f / s;
            if (p.cls_vec) {
                for (int v = gl; v < CV; v += 4) {
                    float x[N];
                    ld_vec16(z + v * N, x);
#pragma unroll
                    for (int e = 0; e < N; ++e) x[e] = k * (expf(x[e] - m) * inv_s - ((v * N + e) == tgt ? 1.f : 0.f));
                    st_vec16(out + v * N, x);
                }
            } else {
                for (int c = gl; c < C; c += 8)
                    out[c] = from_f<T>(k * (expf(ldf(z + c) - m) * inv_s - (c == tgt ? 1.f : 0.f)));
            }
        }
    }
}

static int fill_train(TrainLossParams *out, const void *loc_logits, const void *iou_preds, const void *box_rows,
                      const void *cls_rows, int batch, int64_t num_anchors, int num_classes, const float *rel_iou,
                      const int64_t *assignment, const int32_t *pos_index, int64_t pos_capacity, const int32_t *pos_total,
                      const float *offsets, const float *scales, int img_w, int img_h, const float *gt_boxes,
                      const int64_t *gt_classes, const int32_t *gt_offsets)
{
    TrainLossParams &p = *out;
    SIHL_CHECK_ARG(rel_iou && assignment && gt_offsets, "NULL argument");
    SIHL_CHECK_ARG(batch >= 0 && num_anchors >= 0 && num_anchors < (1ll << 30) && (int64_t)batch * num_anchors < (1ll << 31),
                   "bad sizes: batch=%d anchors=%lld", batch, (long long)num_anchors);
    const bool rows = box_rows != nullptr || cls_rows != nullptr;
    SIHL_CHECK_ARG(!rows || (pos_index && pos_total && pos_capacity >= 0), "positive rows need pos_index / pos_total");
    SIHL_CHECK_ARG(box_rows == nullptr || (offsets && scales && img_w > 0 && img_h > 0),
                   "box loss needs offsets, scales and the image size");
    // gt_boxes / gt_classes may be NULL when the batch holds no ground truth at all (then P == 0 and no row is read)
    SIHL_CHECK_ARG(cls_rows == nullptr || num_classes > 0, "class loss needs num_classes");
    SIHL_CHECK_ARG(box_rows == nullptr || (reinterpret_cast<uintptr_t>(box_rows) & 15u) == 0, "box_rows must be 16-byte aligned");
    p.loc = loc_logits; p.iou_pred = iou_preds; p.box_rows = box_rows; p.cls_rows = cls_rows;
    p.n_dense = (int64_t)batch * num_anchors; p.num_anchors = (int)num_anchors; p.num_classes = num_classes;
    p.rel = rel_iou; p.assignment = assignment;
    p.pos_index = pos_index; p.pos_capacity = rows ? pos_capacity : 0; p.pos_total = pos_total;
    p.offsets = reinterpret_cast<const float4 *>(offsets); p.scales = reinterpret_cast<const float4 *>(scales);
    p.img_w = (float)img_w; p.img_h = (float)img_h;
    p.gt_boxes = reinterpret_cast<const float4 *>(gt_boxes); p.gt_classes = gt_classes; p.gt_offsets = gt_offsets;
    p.sums = nullptr; p.losses = nullptr; p.grad_losses = nullptr; p.grad_scale = 1.f;
    p.dloc = p.diou = p.dbox = p.dcls = nullptr;
    // Few, fat CTAs: every CTA ends with up to 5 fp64 atomics on ONE 64-byte line plus the completion ticket, and
    // same-line atomics serialise in one L2 slice (measured: 1776 CTAs spent 9 of 23 us there).  Dense role: 2 CTAs
    // per SM (4 elements per thread and pass); positive role: one row per thread for the box term, 4 or 8 lanes per
    // row for the class term, at most 6 CTAs per SM (one round over 9 x 6400 rows at cfg1).
    int64_t db = (p.n_dense + (int64_t)kTrainThreads * 4 - 1) / ((int64_t)kTrainThreads * 4);
    if (db > (int64_t)kNumSMs * 2) db = (int64_t)kNumSMs * 2;
    int64_t pb = (p.pos_capacity * 4 + kTrainThreads - 1) / kTrainThreads;
    if (pb > (int64_t)kNumSMs * 6) pb = (int64_t)kNumSMs * 6;
    p.dense_blocks = (int)db; p.pos_blocks = rows ? (int)(pb < 1 ? 1 : pb) : 0;
    p.cls_vec = 0;                                  // set per dtype by the callers (needs sizeof(T))
    return SIHL_OD_OK;
}

static int class_rows_vectorisable(int map_dtype, int num_classes, const void *a, const void *b)
{
    const int esz = map_dtype == SIHL_OD_F32 ? 4 : 2;
    if (num_classes <= 0 || ((size_t)num_classes * esz) % 16 != 0) return 0;
    if (a != nullptr && (reinterpret_cast<uintptr_t>(a) & 15u) != 0) return 0;
    if (b != nullptr && (reinterpret_cast<uintptr_t>(b) & 15u) != 0) return 0;
    return 1;
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_train_loss(const void *loc_logits, const void *iou_preds, const void *box_rows, const void *cls_rows,
                                  int map_dtype, int batch, int64_t num_anchors, int num_classes, const float *rel_iou,
                                  const int64_t *assignment, const int32_t *pos_index, int64_t pos_capacity,
                                  const int32_t *pos_total, const float *offsets, const float *scales, int img_w, int img_h,
                                  const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets, double *sums,
                                  float *losses, void *stream)
{
    TrainLossParams p;
    int rc = fill_train(&p, loc_logits, iou_preds, box_rows, cls_rows, batch, num_anchors, num_classes, rel_iou, assignment,
                        pos_index, pos_capacity, pos_total, offsets, scales, img_w, img_h, gt_boxes, gt_classes, gt_offsets);
    if (rc) return rc;
    SIHL_CHECK_ARG(loc_logits != nullptr && sums != nullptr, "loc_logits / sums is NULL");
    p.sums = sums; p.losses = losses;
    p.cls_vec = class_rows_vectorisable(map_dtype, num_classes, cls_rows, nullptr);
    const int blocks = p.dense_blocks + p.pos_blocks;
    if (blocks == 0) return SIHL_OD_OK;
    SIHL_DISPATCH_DTYPE(map_dtype, (k_train_loss<T><<<blocks, kTrainThreads, 0, (cudaStream_t)stream>>>(p)));
    SIHL_CHECK_LAUNCH("k_train_loss");
    return SIHL_OD_OK;
}

extern "C" int sihl_od_train_loss_bwd(const void *loc_logits, const void *iou_preds, const void *box_rows, const void *cls_rows,
                                      int map_dtype, int batch, int64_t num_anchors, int num_classes, const float *rel_iou,
                                      const int64_t *assignment, const int32_t *pos_index, int64_t pos_capacity,
                                      const int32_t *pos_total, const float *offsets, const float *scales, int img_w,
                                      int img_h, const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                                      const double *sums, const float *grad_losses, float grad_scale, void *dloc, void *diou,
                                      void *dbox_rows, void *dcls_rows, void *stream)
{
    TrainLossParams p;
    int rc = fill_train(&p, loc_logits, iou_preds, box_rows, cls_rows, batch, num_anchors, num_classes, rel_iou, assignment,
                        pos_index, pos_capacity, pos_total, offsets, scales, img_w, img_h, gt_boxes, gt_classes, gt_offsets);
    if (rc) return rc;
    SIHL_CHECK_ARG(sums != nullptr, "sums is NULL");
    SIHL_CHECK_ARG(dloc == nullptr || loc_logits != nullptr, "dloc needs loc_logits");
    SIHL_CHECK_ARG(diou == nullptr || iou_preds != nullptr, "diou needs iou_preds");
    SIHL_CHECK_ARG(dbox_rows == nullptr || box_rows != nullptr, "dbox_rows needs box_rows");
    SIHL_CHECK_ARG(dcls_rows == nullptr || cls_rows != nullptr, "dcls_rows needs cls_rows");
    SIHL_CHECK_ARG(dbox_rows == nullptr || (reinterpret_cast<uintptr_t>(dbox_rows) & 15u) == 0, "dbox_rows must be 16-byte aligned");
    p.sums = const_cast<double *>(sums); p.grad_losses = grad_losses; p.grad_scale = grad_scale;
    p.dloc = dloc; p.diou = diou; p.dbox = dbox_rows; p.dcls = dcls_rows;
    p.cls_vec = class_rows_vectorisable(map_dtype, num_classes, cls_rows, dcls_rows);
    if (dloc == nullptr && diou == nullptr) p.dense_blocks = 0;
    if (dbox_rows == nullptr && dcls_rows == nullptr) p.pos_blocks = 0;
    const int blocks = p.dense_blocks + p.pos_blocks;
    if (blocks == 0) return SIHL_OD_OK;
    SIHL_DISPATCH_DTYPE(map_dtype, (k_train_loss_bwd<T><<<blocks, kTrainThreads, 0, (cudaStream_t)stream>>>(p)));
    SIHL_CHECK_LAUNCH("k_train_loss_bwd");
    return SIHL_OD_OK;
}
