// od_assign.cu — CIoU top-k label assignment (SURVEY.md §8 a3/a4) and the streaming
// resolve pass with the dense losses (a5/a6) and the positive lists (a7) fused in.
//
// Replaces, per training step, the Python loop of B calls to ObjectDetection.bbox_matching
// (ref: src/sihl/heads/object_detection.py:143-148, :252-284), ~100 ATen launches, ~35
// [A,G] fp32 temporaries and ~7 host syncs per image, by two launches for the batch.
//
// Stage 1 (k_assign_select): one warp per ground-truth box.  CIoU > 0 implies IoU > 0
// (every subtracted term is >= 0), so only anchors whose cell overlaps the gt can be
// positive, and CIoU <= IoU - rho^2/c^2 bounds the distance between the centres: per
// pyramid level the candidates are the cells of a small window around the gt (overlap
// window intersected with the centre-distance window, both with slack; the decision is
// always the exact CIoU arithmetic on the real anchor table).  The windows of all
// levels form one flat candidate range that the warp sweeps 32 at a time.
// Lanes append positives to a per-warp shared-memory buffer with ballot/popc; a rank-by-
// counting pass (lexicographic (value desc, anchor asc)) keeps the top k and yields them
// sorted.  Bound: FP32 ALU / latency (≈45 flops + 4 IEEE divisions + atanf per pair);
// compulsory HBM traffic is 16 B per gt in, 8k+4 B per gt out.
//
// Stage 2 (k_assign_resolve): one CTA per (image, tile of 1024 anchors).  The image's
// <= G*k selections are max-reduced into 64-bit keys (value bits << 32 | ~gt) in shared
// memory — the torch.max rule "largest value, lowest gt index" in one atomicMax — then
// the CTA streams loc_logits / iou_preds (coalesced 4-byte loads), writes assignment
// (int64) and rel_iou, and reduces BCE / MSE / counts in registers -> shuffles -> one
// fp64 atomicAdd per CTA and term.  Bound: HBM, 20 B per anchor.
#include "od_common.cuh"
#include "od_pos.cuh"

namespace sihl {

int fill_level_table(const int32_t *level_hw_host, int n_levels, LevelTable *lv);   // od_anchors.cu

// ---------------------------------------------------------------------------
// Stage 1: select
// ---------------------------------------------------------------------------
constexpr int kSelWarps = 4;
constexpr int kSelMinBlocks = 12;     // <= 40 registers: the 1600 CTAs of cfg1 (6400 gts) fit in one wave of 148 x 12
constexpr int kBufCap = 64;

struct SelectParams {
    LevelTable lv;
    float inv_sx[SIHL_OD_MAX_LEVELS], inv_sy[SIHL_OD_MAX_LEVELS];   // cells per pixel (host-computed, only sizes the
    float cell_w[SIHL_OD_MAX_LEVELS], cell_h[SIHL_OD_MAX_LEVELS];   // conservative candidate windows)
    int use_levels;
    int num_anchors;
    int topk;
};

// Buffer entries are 64-bit keys: CIoU bits << 32 | ~anchor.  Values are > 0, so the unsigned order of the keys is
// (value desc, anchor asc) — the lexicographic rule of torch.topk ties in one integer comparison.
__device__ __forceinline__ unsigned long long sel_key(float v, int a)
{
    return ((unsigned long long)__float_as_uint(v) << 32) | (unsigned long long)(0xffffffffu - (unsigned)a);
}
__device__ __forceinline__ float sel_key_val(unsigned long long k) { return __uint_as_float((unsigned)(k >> 32)); }
__device__ __forceinline__ int sel_key_anchor(unsigned long long k) { return (int)(0xffffffffu - (unsigned)k); }

// Keep the top-k of the warp's buffer, sorted descending (rank by counting; keys are distinct); returns the new count.
__device__ __forceinline__ int select_compress(unsigned long long *bk, int cnt, int topk, int lane)
{
    __syncwarp();
    const bool h0 = lane < cnt, h1 = lane + 32 < cnt;
    const unsigned long long k0 = h0 ? bk[lane] : 0ull, k1 = h1 ? bk[lane + 32] : 0ull;
    int r0 = 0, r1 = 0;
    if (cnt <= 32) {
#pragma unroll 4
        for (int i = 0; i < cnt; ++i) r0 += bk[i] > k0;
    } else {
#pragma unroll 4
        for (int i = 0; i < cnt; ++i) {
            const unsigned long long ki = bk[i];
            r0 += ki > k0;
            r1 += ki > k1;
        }
    }
    __syncwarp();
    if (h0 && r0 < topk) bk[r0] = k0;
    if (h1 && r1 < topk) bk[r1] = k1;
    __syncwarp();
    return cnt < topk ? cnt : topk;
}

// How the kernel learns the ground-truth layout (sihl_od_train_assign):
//   kGtHost    total_gt is exact (legacy entry point), nothing else to do;
//   kGtByValue the per-image prefix sums arrive BY VALUE in the kernel parameters and block 0 writes them to
//              gt_offsets for the kernels that follow — ragged python lists reach the device without a copy or a sync;
//   kGtDevice  gt_offsets is already on the device: the true total is gt_offsets[batch], total_gt sizes the launch
//              (a captured graph can be replayed on new ground truth).
enum { kGtHost = 0, kGtByValue = 1, kGtDevice = 2 };
template <int MODE> struct GtLayoutArg { };                          // empty for kGtHost
template <> struct GtLayoutArg<kGtByValue> { int32_t *gt_offsets; int batch; int prefix[SIHL_OD_MAX_BATCH_BY_VALUE + 1]; };
template <> struct GtLayoutArg<kGtDevice> { const int32_t *gt_total; };

// anchor_terms (optional): per anchor (area, cx, cy, atan(w/h)) as sihl_od_anchor_terms writes them —
// the same fp32 operations box_terms() performs, hoisted out of the pair loop and cached with the tables.
template <int MODE>
__global__ void __launch_bounds__(kSelWarps * 32, kSelMinBlocks)
k_assign_select(SelectParams p, const float4 *__restrict__ anchors, const float4 *__restrict__ anchor_terms,
                const float4 *__restrict__ gt_boxes, int total_gt, int32_t *__restrict__ sel_anchor,
                float *__restrict__ sel_val, float *__restrict__ best_iou, double *__restrict__ sums,
                const __grid_constant__ GtLayoutArg<MODE> layout)
{
    __shared__ unsigned long long s_key[kSelWarps][kBufCap];
    __shared__ int4 s_tab[kSelWarps][SIHL_OD_MAX_LEVELS];

    if (sums != nullptr && blockIdx.x == 0 && threadIdx.x < SIHL_OD_NUM_SUMS) sums[threadIdx.x] = 0.0;
    if constexpr (MODE == kGtByValue) {
        if (blockIdx.x == 0)
            for (int i = threadIdx.x; i <= layout.batch; i += blockDim.x) layout.gt_offsets[i] = layout.prefix[i];
    }
    if constexpr (MODE == kGtDevice) {
        const int t = __ldg(layout.gt_total);
        total_gt = t < total_gt ? t : total_gt;
    }

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * kSelWarps + warp;
    if (g >= total_gt) return;                       // warp-uniform; no block barriers below

    unsigned long long *bk = s_key[warp];
    const int topk = p.topk;
    const BoxTerms gt = box_terms(to_box(__ldg(gt_boxes + g)));
    int cnt = 0;
    float thr = 0.f;                                 // k-th best so far once cnt == topk, else 0

    // Evaluate up to 32 candidates (one per lane) and append the ones that can still make the top k.
    // The arithmetic is ciou_pair() (od_math.h) cut in three so that a chunk leaves early when no lane
    // can still rank: no overlap => CIoU <= 0; IoU < thr => CIoU < thr (CIoU <= IoU).
    auto consider = [&](bool valid, int a) {
        BoxTerms an;
        an.x1 = an.y1 = an.x2 = an.y2 = an.area = an.cx = an.cy = an.at = 0.f;
        if (valid) {
            const float4 b = __ldg(anchors + a);
            if (anchor_terms != nullptr) {
                const float4 t = __ldg(anchor_terms + a);
                an.x1 = b.x; an.y1 = b.y; an.x2 = b.z; an.y2 = b.w;
                an.area = t.x; an.cx = t.y; an.cy = t.z; an.at = t.w;
            } else {
                an = box_terms(to_box(b));
            }
        }
        const float eps = 1e-7f;
        float w = fminf(an.x2, gt.x2) - fmaxf(an.x1, gt.x1);
        float h = fminf(an.y2, gt.y2) - fmaxf(an.y1, gt.y1);
        w = w < 0.f ? 0.f : w;
        h = h < 0.f ? 0.f : h;
        const float inter = w * h;
        bool live = valid && inter > 0.f;
        if (!__any_sync(kFullMask, live)) return;
        const float uni = (an.area + gt.area) - inter;
        const float iou = inter / uni;
        live = live && (thr > 0.f ? iou >= thr : true);
        if (!__any_sync(kFullMask, live)) return;
        float wi = fmaxf(an.x2, gt.x2) - fminf(an.x1, gt.x1);
        float hi = fmaxf(an.y2, gt.y2) - fminf(an.y1, gt.y1);
        wi = wi < 0.f ? 0.f : wi;
        hi = hi < 0.f ? 0.f : hi;
        const float diag = ((wi * wi) + (hi * hi)) + eps;
        const float dx = an.cx - gt.cx, dy = an.cy - gt.cy;
        const float cd = (dx * dx) + (dy * dy);
        const float diou = iou - (cd / diag);
        const float da = an.at - gt.at;
        const float vv = SIHL_FOUR_OVER_PI2 * (da * da);
        const float alpha = vv / (((1.f - iou) + vv) + eps);
        const float v = diou - (alpha * vv);
        const bool hit = live && (thr > 0.f ? v >= thr : v > 0.f);      // clamp(0): non-positives never rank
        const unsigned m = __ballot_sync(kFullMask, hit);
        if (m) {
            if (hit) bk[cnt + __popc(m & ((1u << lane) - 1u))] = sel_key(v, a);
            cnt += __popc(m);
            if (cnt > kBufCap - 32) {
                cnt = select_compress(bk, cnt, topk, lane);
                if (cnt == topk) thr = sel_key_val(bk[topk - 1]);
            }
        }
    };

    if (!p.use_levels) {
        for (int t0 = 0; t0 < p.num_anchors; t0 += 32) consider(t0 + lane < p.num_anchors, t0 + lane);
    } else {
        // Candidate windows, one pyramid level per lane.  A positive CIoU needs BOTH
        //  (i)  overlap (CIoU <= IoU): cells from floor((x1 - slack)/sx) to floor((x2 + slack)/sx), and
        //  (ii) rho^2 / c^2 < IoU (CIoU <= IoU - rho^2/c^2) with IoU <= min(area)/max(area) and, for
        //       overlapping boxes, c^2 <= (Wg+sx)^2 + (Hg+sy)^2: the cell centre lies within
        //       R = sqrt(IoU_max * c_max^2) of the gt centre in x and in y.
        // Both are supersets evaluated with slack (2 % + 0.01 px on R, 0.02 px on the overlap window); the
        // decision itself is always the exact CIoU arithmetic on the real anchor table above.
        int4 *tab = s_tab[warp];
        int n_l = 0;
        if (lane < p.lv.n) {
            const int l = lane;
            const int lw = p.lv.w[l], lh = p.lv.h[l];
            const float isx = p.inv_sx[l], isy = p.inv_sy[l], sx = p.cell_w[l], sy = p.cell_h[l];
            const float fw = (float)(lw - 1), fh = (float)(lh - 1);
            // (i) overlap window: cell j spans [j sx, (j+1) sx) up to the ~1e-4 px by which the real anchor table is off
            // the ideal lattice (linspace rounding, SURVEY.md §7.1); a cell whose span ends more than `slack` before
            // the gt starts (or starts more than `slack` after it ends) cannot intersect it.  slack = 0.02 px + 1e-5
            // of the coordinate is ~100x the lattice error and ~1000x the rounding of the products below — and costs
            // a fraction of a cell, where a whole extra cell per side (the first version) tripled the candidates of
            // a small gt on its best level (6 x 6 instead of 3 x 3 cells for a gt of two cells).
            const float ex = 0.02f + 1e-5f * fmaxf(fabsf(gt.x1), fabsf(gt.x2)), ey = 0.02f + 1e-5f * fmaxf(fabsf(gt.y1), fabsf(gt.y2));
            float jlo = floorf((gt.x1 - ex) * isx), jhi = floorf((gt.x2 + ex) * isx);
            float ilo = floorf((gt.y1 - ey) * isy), ihi = floorf((gt.y2 + ey) * isy);
            if (gt.area > 0.f) {
                const float cell = sx * sy;
                const float iou_max = __fdividef(fminf(cell, gt.area), fmaxf(cell, gt.area));
                const float wg = fabsf(gt.x2 - gt.x1) + sx, hg = fabsf(gt.y2 - gt.y1) + sy;
                const float R = sqrtf(iou_max * ((wg * wg) + (hg * hg) + 1.f)) * 1.02f + 0.01f;
                jlo = fmaxf(jlo, floorf((gt.cx - R) * isx - 0.5f));
                jhi = fminf(jhi, floorf((gt.cx + R) * isx - 0.5f) + 1.f);
                ilo = fmaxf(ilo, floorf((gt.cy - R) * isy - 0.5f));
                ihi = fminf(ihi, floorf((gt.cy + R) * isy - 0.5f) + 1.f);
            }
            const int j0 = (int)fminf(fmaxf(jlo, 0.f), fw), j1 = (int)fminf(fmaxf(jhi, 0.f), fw);
            const int i0 = (int)fminf(fmaxf(ilo, 0.f), fh), i1 = (int)fminf(fmaxf(ihi, 0.f), fh);
            const bool empty = !(jhi >= 0.f) || !(jlo <= fw) || !(ihi >= 0.f) || !(ilo <= fh) || j1 < j0 || i1 < i0;
            const int nj = empty ? 0 : j1 - j0 + 1, ni = empty ? 0 : i1 - i0 + 1;
            n_l = ni * nj;
            tab[l] = make_int4(p.lv.base[l] + i0 * lw + j0, nj, lw, __float_as_int(__fdividef(1.f, (float)(nj > 0 ? nj : 1))));
        }
        int incl = n_l;                              // inclusive prefix of the window sizes over the level lanes
#pragma unroll
        for (int o = 1; o < SIHL_OD_MAX_LEVELS; o <<= 1) {
            const int y = __shfl_up_sync(kFullMask, incl, o);
            if (lane >= o) incl += y;
        }
        int pre[SIHL_OD_MAX_LEVELS];                 // pre[k] = first flat candidate index of level k+1
#pragma unroll
        for (int k = 0; k < SIHL_OD_MAX_LEVELS; ++k) pre[k] = __shfl_sync(kFullMask, incl, k);
        const int total = pre[SIHL_OD_MAX_LEVELS - 1];
        __syncwarp();
        for (int t0 = 0; t0 < total; t0 += 32) {
            const int t = t0 + lane;
            const bool valid = t < total;
            int l = 0, first = 0;
#pragma unroll
            for (int k = 0; k < SIHL_OD_MAX_LEVELS - 1; ++k)
                if (t >= pre[k]) { l = k + 1; first = pre[k]; }
            const int4 e = tab[valid ? l : 0];
            const int tl = t - first;
            const int ri = (int)(((float)tl + 0.5f) * __int_as_float(e.w));     // tl / nj (margin 0.5/nj >> rounding)
            const int rj = tl - ri * e.y;
            consider(valid, e.x + ri * e.z + rj);
        }
    }

    cnt = select_compress(bk, cnt, topk, lane);
    const unsigned long long mine = lane < cnt ? bk[lane] : 0ull;
    const int my_anchor = lane < cnt ? sel_key_anchor(mine) : -1;
    if (lane < topk) {
        sel_anchor[(int64_t)g * topk + lane] = my_anchor;
        sel_val[(int64_t)g * topk + lane] = lane < cnt ? sel_key_val(mine) : 0.f;
    }
    if (lane == 0) best_iou[g] = cnt ? sel_key_val(mine) : 0.f;      // ref :277 topk_ious[0]
}

// Per-anchor terms of the CIoU (box_terms() of od_math.h), cached next to the anchor table.
__global__ void __launch_bounds__(256) k_anchor_terms(const float4 *__restrict__ anchors, int n, float4 *__restrict__ terms)
{
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < n; a += gridDim.x * blockDim.x) {
        const BoxTerms t = box_terms(to_box(__ldg(anchors + a)));
        terms[a] = make_float4(t.area, t.cx, t.cy, t.at);
    }
}

// ---------------------------------------------------------------------------
// Stage 2: resolve (+ dense losses, + compaction, + fused positive losses)
// ---------------------------------------------------------------------------
constexpr int kResThreads = 128;
constexpr int kChunks = kTile / kResThreads;
constexpr int kResWarps = kResThreads / 32;

struct ResolveParams {
    const int32_t *sel_anchor; const float *sel_val; const float *best_iou; const int32_t *gt_offsets;
    int num_anchors, topk, relative;
    const void *loc; const void *iou_pred;     // element type T of the kernel template (SIHL_OD_F32 / _F16 / _BF16)
    int64_t *assignment; float *out_iou; double *sums;
    int32_t *tile_pos_count; int32_t *tile_pos_rows;
    const void *prefetch_box; const void *prefetch_cls; int num_classes;     // L2 hints for k_pos_loss_tiles (same T)
    float inv_topk;            // 1 / topk: e / topk == (int)((e + 0.5f) * inv_topk) for e < 2^21 (checked for topk <= 64)
    int32_t *pos_chunks;       // work list for k_pos_loss_tiles: (slot << 10 | first_row / 32 << 6 | rows - 1)
    int2 *tile_pos_aux;        // per listed positive: (global gt index, rel bits) — saves that kernel two dependent hops
};

// BCE term of the fused pass for a map of type T.  fp32: the fast form above.  Half types: what the reference computes
// on half logits (ref :160-161 has no .to(float32)): (1 - t) x - log_sigmoid(x) with log_sigmoid rounded to the map type.
template <typename T> __device__ __forceinline__ float bce_fused(float x, float t)
{
    const float ax = fabsf(x);
    const float ls = fminf(0.f, x) - log1pf(expf(-ax));
    return (1.f - t) * x - round_to<T>(ls);
}
template <> __device__ __forceinline__ float bce_fused<float>(float x, float t) { return bce_logits_fast(x, t); }

template <typename T>
__global__ void __launch_bounds__(kResThreads) k_assign_resolve(ResolveParams p)
{
    const T *t_loc = reinterpret_cast<const T *>(p.loc), *t_iou = reinterpret_cast<const T *>(p.iou_pred);
    __shared__ unsigned s_v[kTile], s_g[kTile];
    __shared__ float s_rel[kTile];
    __shared__ unsigned short s_pos[kTile];
    __shared__ int s_seg[kChunks * kResWarps + 1];
    __shared__ double s_red[5 * 32];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y, tile = blockIdx.x, n_tiles = gridDim.x;
    const int A = p.num_anchors, a0 = tile * kTile;
    const int na = min(kTile, A - a0);
    const int g0 = __ldg(p.gt_offsets + b), g1 = __ldg(p.gt_offsets + b + 1);

    // issue the streaming loads first: they are independent of the key reduction below
    float x_loc[kChunks], x_iou[kChunks];
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
        const int la = c * kResThreads + tid;
        const int64_t flat = (int64_t)b * A + a0 + (la < na ? la : 0);
        x_loc[c] = t_loc != nullptr ? ldf(t_loc + flat) : 0.f;
        x_iou[c] = t_iou != nullptr ? ldf(t_iou + flat) : 0.f;
    }

    for (int i = tid; i < kTile; i += kResThreads) { s_v[i] = 0u; s_g[i] = 0xffffffffu; }
    __syncthreads();
    // per anchor: max value over the gts that selected it, ties -> lowest gt (ref :270), as two passes
    // of native 32-bit shared-memory atomics (max of the value bits, then min of the gt among the maxima)
    const int n_entries = (g1 - g0) * p.topk;
    const int32_t *sa = p.sel_anchor + (int64_t)g0 * p.topk;
    const float *sv = p.sel_val + (int64_t)g0 * p.topk;
    constexpr int kEntryBatch = 8;                                   // loads in flight per thread
    auto load_batch = [&](int e0, int (&ea)[kEntryBatch], unsigned (&ev)[kEntryBatch]) {
#pragma unroll
        for (int u = 0; u < kEntryBatch; ++u) {                         // all loads first: one L2 round trip per batch
            const int e = e0 + u * kResThreads + tid;
            const bool in = e < n_entries;
            ea[u] = in ? __ldg(sa + e) - a0 : -1;
            ev[u] = in ? __float_as_uint(__ldg(sv + e)) : 0u;           // values are > 0: bit order == value order
        }
    };
    auto pass_max = [&](const int (&ea)[kEntryBatch], const unsigned (&ev)[kEntryBatch]) {
#pragma unroll
        for (int u = 0; u < kEntryBatch; ++u)
            if (ea[u] >= 0 && ea[u] < na) atomicMax(&s_v[ea[u]], ev[u]);
    };
    auto pass_min = [&](int e0, const int (&ea)[kEntryBatch], const unsigned (&ev)[kEntryBatch]) {
#pragma unroll
        for (int u = 0; u < kEntryBatch; ++u)
            if (ea[u] >= 0 && ea[u] < na && s_v[ea[u]] == ev[u]) {
                const int e = e0 + u * kResThreads + tid;
                // e / topk without the ~20-instruction integer division: exact for e < 2^21 and topk <= 64
                const int g = e < (1 << 21) ? (int)(((float)e + 0.5f) * p.inv_topk) : e / p.topk;
                atomicMin(&s_g[ea[u]], (unsigned)g);
            }
    };
    if (n_entries <= kEntryBatch * kResThreads) {                    // one batch (<= 1024 selections per image: cfg1 has
        int ea[kEntryBatch];                                         // 900): the entries stay in registers for pass two
        unsigned ev[kEntryBatch];
        load_batch(0, ea, ev);
        pass_max(ea, ev);
        __syncthreads();
        pass_min(0, ea, ev);
    } else {
        for (int e0 = 0; e0 < n_entries; e0 += kEntryBatch * kResThreads) {
            int ea[kEntryBatch];
            unsigned ev[kEntryBatch];
            load_batch(e0, ea, ev);
            pass_max(ea, ev);
        }
        __syncthreads();
        for (int e0 = 0; e0 < n_entries; e0 += kEntryBatch * kResThreads) {
            int ea[kEntryBatch];
            unsigned ev[kEntryBatch];
            load_batch(e0, ea, ev);
            pass_min(e0, ea, ev);
        }
    }
    __syncthreads();

    float acc_bce = 0.f, acc_one = 0.f, acc_mse = 0.f, acc_rel = 0.f, acc_pos = 0.f;
    unsigned ballots[kChunks];
    bool flags[kChunks];
    const bool want_list = p.tile_pos_count != nullptr;
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
        const int la = c * kResThreads + tid;
        bool pos = false;
        if (la < na) {
            const unsigned vb = s_v[la];
            const int64_t flat = (int64_t)b * A + a0 + la;
            float rel = 0.f;
            int64_t asg = -1;
            if (vb != 0u) {
                const float v = __uint_as_float(vb);
                const int g = (int)s_g[la];
                rel = p.relative ? v / __ldg(p.best_iou + g0 + g) : v;          // ref :279-281
                pos = rel > 0.f;
                asg = pos ? g : -1;                                              // canonical form (sihl_od.h)
            }
            p.assignment[flat] = asg;
            p.out_iou[flat] = rel;
            s_rel[la] = rel;
            if (pos) {                                    // the positive-row kernel gathers these next: warm L2 now
                if (p.prefetch_box != nullptr)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const T *>(p.prefetch_box) + 4 * flat));
                if (p.prefetch_cls != nullptr) {
                    const char *row = reinterpret_cast<const char *>(reinterpret_cast<const T *>(p.prefetch_cls) + flat * p.num_classes);
                    const int bytes = p.num_classes * (int)sizeof(T);
                    for (int o = 0; o < bytes; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + o));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(row + bytes - 4));
                }
            }
            if (p.loc != nullptr) {
                const float t = (rel == 1.0f) ? 1.f : 0.f;                       // ref :159
                acc_bce += bce_fused<T>(x_loc[c], t);
                acc_one += t;
                if (p.iou_pred != nullptr) {
                    const float d = x_iou[c] - rel;                              // ref :177-179
                    acc_mse += d * d;
                }
                acc_rel += rel;
                acc_pos += pos ? 1.f : 0.f;
            }
        }
        flags[c] = pos;
        ballots[c] = __ballot_sync(kFullMask, pos);
        if (want_list && lane == 0) s_seg[c * kResWarps + warp] = __popc(ballots[c]);
    }

    int n_pos = 0;
    if (want_list) {
        // ordered compaction: segment (chunk, warp) order == ascending anchor order (ref :182-184)
        __syncthreads();
        if (warp == 0) {
            const int nseg = kChunks * kResWarps;
            int x = lane < nseg ? s_seg[lane] : 0;
            int incl = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += y;
            }
            if (lane < nseg) s_seg[lane] = incl - x;
            if (lane == 31) s_seg[nseg] = incl;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < kChunks; ++c)
            if (flags[c]) {
                const int r = s_seg[c * kResWarps + warp] + __popc(ballots[c] & ((1u << lane) - 1u));
                s_pos[r] = (unsigned short)(c * kResThreads + tid);
            }
        __syncthreads();
        n_pos = s_seg[kChunks * kResWarps];
        if (p.tile_pos_count != nullptr) {
            const int slot = b * n_tiles + tile;
            if (tid == 0) p.tile_pos_count[slot] = n_pos;
            // reserve ceil(n_pos/32) entries of the chunk list; the counter lives in sums[7] (zeroed by
            // k_assign_select together with the loss sums; integers are exact in fp64).  The atomic's
            // round trip overlaps the list writes below.
            const int nchunk = (n_pos + 31) >> 5;
            double base_d = 0.0;
            const bool publish = p.pos_chunks != nullptr && n_pos > 0 && warp == 0;
            if (publish && lane == 0) base_d = atomicAdd(p.sums + 7, (double)nchunk);
            for (int r = tid; r < n_pos; r += kResThreads) {
                const int la = s_pos[r];
                p.tile_pos_rows[(int64_t)slot * kTile + r] = (int32_t)((int64_t)b * A + a0 + la);
                if (p.tile_pos_aux != nullptr) {
                    p.tile_pos_aux[(int64_t)slot * kTile + r] = make_int2(g0 + (int)s_g[la], __float_as_int(s_rel[la]));
                }
            }
            if (publish) {
                const int base = __shfl_sync(kFullMask, (int)base_d, 0);
                if (lane < nchunk) {
                    const int rows = min(32, n_pos - 32 * lane);
                    p.pos_chunks[base + lane] = (slot << 10) | (lane << 6) | (rows - 1);
                }
            }
        }
    }

    if (p.sums != nullptr && p.loc != nullptr) {
        float v[5] = {acc_bce, acc_one, acc_mse, acc_rel, acc_pos};
        const int slot[5] = {0, 1, 2, 3, 6};
        block_accumulate_f<5>(v, s_red, p.sums, slot);
    }
}

// ---------------------------------------------------------------------------
// Tile lists -> one ascending pos_index (ref :182-184 row order)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_pos_compact(const int32_t *__restrict__ tile_pos_count, const int32_t *__restrict__ tile_pos_rows, int n_slots,
              int32_t *__restrict__ pos_index, int64_t capacity, int32_t *__restrict__ pos_total)
{
    __shared__ int s_red[32];
    const int slot = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int before = 0, total = 0;
    for (int i = tid; i < n_slots; i += blockDim.x) {
        const int c = __ldg(tile_pos_count + i);
        total += c;
        if (i < slot) before += c;
    }
    before = warp_sum(before);
    total = warp_sum(total);
    if (lane == 0) { s_red[warp] = before; s_red[16 + warp] = total; }
    __syncthreads();
    before = 0; total = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { before += s_red[w]; total += s_red[16 + w]; }
    if (tid == 0 && slot == 0) *pos_total = total;
    const int n = __ldg(tile_pos_count + slot);
    for (int r = tid; r < n; r += blockDim.x)
        if ((int64_t)before + r < capacity) pos_index[before + r] = __ldg(tile_pos_rows + (int64_t)slot * kTile + r);
    // rows [total, capacity) are gathered by the static-size MLP batch: any valid row will do
    for (int64_t r = (int64_t)total + (int64_t)slot * blockDim.x + tid; r < capacity; r += (int64_t)n_slots * blockDim.x)
        pos_index[r] = 0;
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_anchor_terms(const float *anchors, int64_t num_anchors, float *terms, void *stream)
{
    SIHL_CHECK_ARG(anchors && terms && num_anchors >= 0 && num_anchors < (1ll << 30), "bad arguments");
    if (num_anchors == 0) return SIHL_OD_OK;
    k_anchor_terms<<<(unsigned)((num_anchors + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4 *>(anchors), (int)num_anchors, reinterpret_cast<float4 *>(terms));
    SIHL_CHECK_LAUNCH("k_anchor_terms");
    return SIHL_OD_OK;
}

static int fill_select_params(SelectParams *out, int64_t num_anchors, const int32_t *level_hw_host, int n_levels,
                              int img_w, int img_h, int total_gt, int topk)
{
    SelectParams &p = *out;
    SIHL_CHECK_ARG(topk >= 1 && topk <= SIHL_OD_MAX_TOPK, "topk=%d outside 1..%d", topk, SIHL_OD_MAX_TOPK);
    SIHL_CHECK_ARG(total_gt >= 0 && num_anchors >= 0 && num_anchors < (1ll << 30), "bad sizes");
    SIHL_CHECK_ARG(total_gt == 0 || num_anchors >= topk,
                   "selected index k out of range: %lld anchors < topk=%d (torch.topk raises in the reference)",
                   (long long)num_anchors, topk);
    p.use_levels = level_hw_host != nullptr;
    for (int l = 0; l < SIHL_OD_MAX_LEVELS; ++l) { p.inv_sx[l] = p.inv_sy[l] = 0.f; p.cell_w[l] = p.cell_h[l] = 1.f; }
    if (p.use_levels) {
        int rc = fill_level_table(level_hw_host, n_levels, &p.lv);
        if (rc) return rc;
        SIHL_CHECK_ARG(p.lv.base[n_levels] == num_anchors, "levels hold %d anchors, table has %lld", p.lv.base[n_levels],
                       (long long)num_anchors);
        SIHL_CHECK_ARG(img_w > 0 && img_h > 0, "image size %dx%d", img_w, img_h);
        for (int l = 0; l < n_levels; ++l) {
            p.inv_sx[l] = (float)p.lv.w[l] / (float)img_w;
            p.inv_sy[l] = (float)p.lv.h[l] / (float)img_h;
            p.cell_w[l] = (float)img_w / (float)p.lv.w[l];
            p.cell_h[l] = (float)img_h / (float)p.lv.h[l];
        }
    } else {
        p.lv.n = 0;
        for (int l = 0; l < SIHL_OD_MAX_LEVELS; ++l) { p.lv.h[l] = p.lv.w[l] = 1; p.lv.base[l] = 0; }
        p.lv.base[SIHL_OD_MAX_LEVELS] = 0;
    }
    p.num_anchors = (int)num_anchors; p.topk = topk;
    return SIHL_OD_OK;
}

extern "C" int sihl_od_assign_select(const float *anchors, const float *anchor_terms, int64_t num_anchors,
                                     const int32_t *level_hw_host, int n_levels, int img_w, int img_h,
                                     const float *gt_boxes, const int32_t *gt_offsets, int batch, int total_gt,
                                     int topk, int32_t *sel_anchor, float *sel_val, float *best_iou, double *sums,
                                     void *stream)
{
    (void)gt_offsets; (void)batch;
    SelectParams p;
    int rc = fill_select_params(&p, num_anchors, level_hw_host, n_levels, img_w, img_h, total_gt, topk);
    if (rc) return rc;
    if (total_gt == 0 && sums == nullptr) return SIHL_OD_OK;
    const int blocks = total_gt > 0 ? (total_gt + kSelWarps - 1) / kSelWarps : 1;
    k_assign_select<kGtHost><<<blocks, kSelWarps * 32, 0, (cudaStream_t)stream>>>(
        p, reinterpret_cast<const float4 *>(anchors), reinterpret_cast<const float4 *>(anchor_terms),
        reinterpret_cast<const float4 *>(gt_boxes), total_gt, sel_anchor, sel_val, best_iou, sums, GtLayoutArg<kGtHost>{});
    SIHL_CHECK_LAUNCH("k_assign_select");
    return SIHL_OD_OK;
}

// ---------------------------------------------------------------------------
// The drop-in head's "before the MLPs" call: select -> resolve -> compaction, all scratch from one workspace.
// ---------------------------------------------------------------------------
namespace {
struct TrainWorkspace {
    int32_t *sel_anchor; float *sel_val; float *best_iou; int32_t *tile_pos_count; int32_t *tile_pos_rows;
    size_t bytes;
};
TrainWorkspace carve_train_workspace(void *base, int batch, int64_t num_anchors, int gt_capacity, int topk)
{
    const size_t n_tiles = (size_t)((num_anchors + kTile - 1) / kTile);
    const size_t gk = (size_t)(gt_capacity > 0 ? gt_capacity : 0) * (size_t)topk;
    unsigned char *b = reinterpret_cast<unsigned char *>(base);
    size_t o = 0;
    TrainWorkspace w;
    w.sel_anchor = reinterpret_cast<int32_t *>(b + o); o += round_up_256(gk * 4);
    w.sel_val = reinterpret_cast<float *>(b + o); o += round_up_256(gk * 4);
    w.best_iou = reinterpret_cast<float *>(b + o); o += round_up_256((size_t)(gt_capacity > 0 ? gt_capacity : 0) * 4);
    w.tile_pos_count = reinterpret_cast<int32_t *>(b + o); o += round_up_256((size_t)batch * n_tiles * 4);
    w.tile_pos_rows = reinterpret_cast<int32_t *>(b + o); o += round_up_256((size_t)batch * n_tiles * kTile * 4);
    w.bytes = o;
    return w;
}
}  // namespace

extern "C" size_t sihl_od_train_workspace_bytes(int batch, int64_t num_anchors, int gt_capacity, int topk)
{
    if (batch < 0 || num_anchors < 0 || topk < 1) return 0;
    return carve_train_workspace(nullptr, batch, num_anchors, gt_capacity, topk).bytes;
}

extern "C" int sihl_od_train_assign(const float *anchors, const float *anchor_terms, int64_t num_anchors,
                                    const int32_t *level_hw_host, int n_levels, int img_w, int img_h,
                                    const float *gt_boxes, const int32_t *gt_counts_host, int32_t *gt_offsets,
                                    int batch, int gt_capacity, int topk, int64_t *assignment, float *rel_iou,
                                    int32_t *pos_index, int64_t pos_capacity, int32_t *pos_total, double *sums,
                                    void *workspace, size_t workspace_bytes, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    SIHL_CHECK_ARG(anchors && gt_offsets && assignment && rel_iou && pos_index && pos_total && sums, "NULL argument");
    SIHL_CHECK_ARG(batch >= 1 && batch <= 65535 && gt_capacity >= 0 && pos_capacity >= 1, "bad sizes");
    SIHL_CHECK_ARG(gt_capacity == 0 || gt_boxes != nullptr, "gt_boxes is NULL");
    SIHL_CHECK_ARG(workspace != nullptr && workspace_bytes >= sihl_od_train_workspace_bytes(batch, num_anchors, gt_capacity, topk),
                   "workspace too small: %zu < %zu bytes", workspace_bytes,
                   sihl_od_train_workspace_bytes(batch, num_anchors, gt_capacity, topk));
    SIHL_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15u) == 0, "workspace must be 16-byte aligned");
    int total_gt = gt_capacity;
    GtLayoutArg<kGtByValue> table;
    if (gt_counts_host != nullptr) {
        SIHL_CHECK_ARG(batch <= SIHL_OD_MAX_BATCH_BY_VALUE, "batch=%d > %d: pass gt_offsets on the device instead of host counts",
                       batch, SIHL_OD_MAX_BATCH_BY_VALUE);
        table.gt_offsets = gt_offsets; table.batch = batch; table.prefix[0] = 0;
        for (int b = 0; b < batch; ++b) {
            SIHL_CHECK_ARG(gt_counts_host[b] >= 0, "negative gt count for image %d", b);
            table.prefix[b + 1] = table.prefix[b] + gt_counts_host[b];
        }
        total_gt = table.prefix[batch];
        SIHL_CHECK_ARG(total_gt <= gt_capacity, "gt counts add up to %d > gt_capacity=%d", total_gt, gt_capacity);
    }
    SelectParams sp;
    int rc = fill_select_params(&sp, num_anchors, level_hw_host, n_levels, img_w, img_h, total_gt, topk);
    if (rc) return rc;
    const TrainWorkspace w = carve_train_workspace(workspace, batch, num_anchors, gt_capacity, topk);
    const int blocks = total_gt > 0 ? (total_gt + kSelWarps - 1) / kSelWarps : 1;
    const float4 *an = reinterpret_cast<const float4 *>(anchors), *at = reinterpret_cast<const float4 *>(anchor_terms);
    const float4 *gb = reinterpret_cast<const float4 *>(gt_boxes);
    if (gt_counts_host != nullptr) {
        k_assign_select<kGtByValue><<<blocks, kSelWarps * 32, 0, st>>>(sp, an, at, gb, total_gt, w.sel_anchor, w.sel_val,
                                                                        w.best_iou, sums, table);
    } else {
        GtLayoutArg<kGtDevice> dv;
        dv.gt_total = gt_offsets + batch;
        k_assign_select<kGtDevice><<<blocks, kSelWarps * 32, 0, st>>>(sp, an, at, gb, total_gt, w.sel_anchor, w.sel_val,
                                                                       w.best_iou, sums, dv);
    }
    SIHL_CHECK_LAUNCH("k_assign_select");
    rc = sihl_od_assign_resolve(w.sel_anchor, w.sel_val, w.best_iou, gt_offsets, batch, num_anchors, topk, 1, nullptr, nullptr,
                                assignment, rel_iou, nullptr, w.tile_pos_count, w.tile_pos_rows, nullptr, nullptr, 0, nullptr,
                                nullptr, stream);
    if (rc) return rc;
    const int n_tiles = (int)((num_anchors + kTile - 1) / kTile);
    const int n_slots = batch * n_tiles;
    k_pos_compact<<<n_slots, 256, 0, st>>>(w.tile_pos_count, w.tile_pos_rows, n_slots, pos_index, pos_capacity, pos_total);
    SIHL_CHECK_LAUNCH("k_pos_compact");
    return SIHL_OD_OK;
}

extern "C" int sihl_od_resolve_tiles(int64_t num_anchors, int *n_tiles, int *tile)
{
    if (n_tiles) *n_tiles = (int)((num_anchors + kTile - 1) / kTile);
    if (tile) *tile = kTile;
    return SIHL_OD_OK;
}

extern "C" int sihl_od_assign_resolve(const int32_t *sel_anchor, const float *sel_val, const float *best_iou,
                                      const int32_t *gt_offsets, int batch, int64_t num_anchors, int topk, int relative,
                                      const float *loc_logits, const float *iou_preds, int64_t *assignment,
                                      float *out_iou, double *sums, int32_t *tile_pos_count, int32_t *tile_pos_rows,
                                      const float *prefetch_box_raw, const float *prefetch_cls_logits, int num_classes,
                                      int32_t *pos_chunks, int32_t *tile_pos_aux, void *stream)
{
    return sihl_od_assign_resolve_t(sel_anchor, sel_val, best_iou, gt_offsets, batch, num_anchors, topk, relative, loc_logits,
                                    iou_preds, SIHL_OD_F32, assignment, out_iou, sums, tile_pos_count, tile_pos_rows,
                                    prefetch_box_raw, prefetch_cls_logits, num_classes, pos_chunks, tile_pos_aux, stream);
}

extern "C" int sihl_od_assign_resolve_t(const int32_t *sel_anchor, const float *sel_val, const float *best_iou,
                                        const int32_t *gt_offsets, int batch, int64_t num_anchors, int topk, int relative,
                                        const void *loc_logits, const void *iou_preds, int map_dtype, int64_t *assignment,
                                        float *out_iou, double *sums, int32_t *tile_pos_count, int32_t *tile_pos_rows,
                                        const void *prefetch_box_raw, const void *prefetch_cls_logits, int num_classes,
                                        int32_t *pos_chunks, int32_t *tile_pos_aux, void *stream)
{
    SIHL_CHECK_ARG(topk >= 1 && topk <= SIHL_OD_MAX_TOPK, "topk=%d outside 1..%d", topk, SIHL_OD_MAX_TOPK);
    SIHL_CHECK_ARG(batch >= 0 && num_anchors >= 0 && num_anchors < (1ll << 30), "bad sizes");
    SIHL_CHECK_ARG(assignment && out_iou && gt_offsets, "assignment / out_iou / gt_offsets must not be NULL");
    SIHL_CHECK_ARG((tile_pos_count == nullptr) == (tile_pos_rows == nullptr), "tile_pos_count and tile_pos_rows go together");
    SIHL_CHECK_ARG(iou_preds == nullptr || loc_logits != nullptr, "iou_preds needs loc_logits");
    SIHL_CHECK_ARG(loc_logits == nullptr || sums != nullptr, "dense losses need sums");
    if (batch == 0 || num_anchors == 0) return SIHL_OD_OK;
    ResolveParams p;
    p.sel_anchor = sel_anchor; p.sel_val = sel_val; p.best_iou = best_iou; p.gt_offsets = gt_offsets;
    p.inv_topk = 1.f / (float)topk;
    p.num_anchors = (int)num_anchors; p.topk = topk; p.relative = relative;
    p.loc = loc_logits; p.iou_pred = iou_preds; p.assignment = assignment; p.out_iou = out_iou; p.sums = sums;
    p.tile_pos_count = tile_pos_count; p.tile_pos_rows = tile_pos_rows;
    p.prefetch_box = prefetch_box_raw; p.prefetch_cls = num_classes > 0 ? prefetch_cls_logits : nullptr; p.num_classes = num_classes;
    SIHL_CHECK_ARG(pos_chunks == nullptr || (tile_pos_count != nullptr && sums != nullptr), "pos_chunks needs the tile lists and sums");
    SIHL_CHECK_ARG(pos_chunks == nullptr || (int64_t)batch * ((num_anchors + kTile - 1) / kTile) < (1 << 21), "too many tiles for the chunk list");
    p.pos_chunks = pos_chunks;
    SIHL_CHECK_ARG(tile_pos_aux == nullptr || tile_pos_count != nullptr, "tile_pos_aux needs the tile lists");
    p.tile_pos_aux = reinterpret_cast<int2 *>(tile_pos_aux);
    const dim3 grid((unsigned)((num_anchors + kTile - 1) / kTile), (unsigned)batch);
    SIHL_CHECK_ARG(batch <= 65535, "batch=%d > 65535", batch);
    SIHL_DISPATCH_DTYPE(map_dtype, (k_assign_resolve<T><<<grid, kResThreads, 0, (cudaStream_t)stream>>>(p)));
    SIHL_CHECK_LAUNCH("k_assign_resolve");
    return SIHL_OD_OK;
}
