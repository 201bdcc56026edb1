// od_soft_nms.cu — class-aware Soft-NMS (Bodla et al., ICCV 2017, Algorithm 1; the semantics of mmcv's soft_nms), a
// second consumer of the candidate lists of the dense decode (sihl_od_soft_nms_topk) and the segment form of the
// stand-alone entry (sihl_od_batched_soft_nms).  Per image:
//
//   s = candidate scores (fp32); alive = candidates with s >= score_thr
//   until K detections are emitted or nothing is alive:
//     m = alive candidate with the largest (s, ~index) key     (index: location, or input index for the stand-alone entry)
//     emit m with its current s; alive -= {m}
//     every alive j of m's class: iou = box_iou(m, j) (NaN -> 0); s[j] *= w(iou); dead once !(s[j] >= score_thr)
//       linear:   w = iou > iou_thr ? 1 - iou : 1                        (fp32)
//       gaussian: w = (float)exp(-(double)iou * (double)iou / sigma)     (fp64 exp, rounded once to fp32)
//
// The Gaussian weight goes through fp64 because CUDA's expf and a host libm's disagree in the last ulp, and one ulp in a
// decayed score can flip a later argmax.  Rounded once from fp64, device and host agree (both fp64 exps are within an ulp
// of the exact value, so their fp32 roundings differ only when the exact value lies within ~2^-29 relative of an fp32
// rounding boundary), which lets the tests demand equality with oracle/soft_nms_oracle.py.
//
// Work split: one thread-block cluster per image (1..8 CTAs, sized on the host from the list capacity).  A list that
// fits one CTA's shared memory (steady-state step: a few hundred candidates) is handled by the cluster's first CTA alone,
// the others exit at once: one launch, two block barriers per selected detection.  Longer lists (crowds: one class with
// tens of thousands of candidates) are partitioned across the CTAs' shared memory, 28 B per candidate; every iteration
// each CTA decays its part with the previous winner and finds its best key, the CTAs publish their best (key, box,
// class, score) in a double-buffered shared-memory slot, and after one cluster barrier every CTA reads the others' slots
// through distributed shared memory and agrees on the winner.  Lists too long for the cluster's shared memory keep the
// same partition in a global workspace.
#include <cooperative_groups.h>

#include "od_common.cuh"

namespace cg = cooperative_groups;

namespace sihl {

constexpr int kSoftThreads = 512;
constexpr int kSoftItems = 4096;          // candidates per CTA held in shared memory
constexpr int kSoftMaxCluster = 8;        // portable cluster size
constexpr size_t kSoftItemBytes = 28;     // box 16 + score 4 + tie-break word 4 + class 4

struct __align__(16) SoftSlot {
    float4 box;
    unsigned long long key;    // (score order << 32) | ~index; 0: nothing alive in this CTA
    unsigned cls;
    float score;
};

struct SoftArrays {
    float4 *box;
    float *score;              // current (decayed) score; NaN once dead
    unsigned *lo;              // tie-break word of the key: ~location / ~input index
    unsigned *cls;
};

__device__ __forceinline__ SoftArrays carve_soft(unsigned char *base, int64_t items)
{
    SoftArrays a;
    a.box = reinterpret_cast<float4 *>(base);
    a.score = reinterpret_cast<float *>(base + (size_t)items * 16);
    a.lo = reinterpret_cast<unsigned *>(base + (size_t)items * 20);
    a.cls = reinterpret_cast<unsigned *>(base + (size_t)items * 24);
    return a;
}

__device__ __forceinline__ SoftArrays offset_soft(SoftArrays a, int64_t o)
{
    a.box += o; a.score += o; a.lo += o; a.cls += o;
    return a;
}

struct SoftParams {
    // mode 0: candidate lists written by the dense decode
    const int32_t *cand_count; int64_t cap;
    const unsigned long long *cand_key; const float4 *cand_box; const int32_t *cand_cls;
    int64_t *num_instances; float *out_scores; int64_t *out_classes; float4 *out_boxes;
    int reset_counts;
    // mode 1: stand-alone boxes / scores / classes + segment offsets
    const float4 *boxes; const float *scores; const int64_t *classes; const int32_t *seg_offsets;
    int64_t *keep; float *keep_scores; int32_t *keep_count;
    int mode, method;
    float iou_thr, score_thr;
    double sigma;
    int K;
    unsigned char *workspace; int64_t ws_items;   // workspace layout: carve_soft over ws_items (B * cap, or n)
    int smem_items;                               // candidates one CTA holds in its dynamic shared memory
};

__device__ __forceinline__ void warp_argmax(unsigned long long &key, int &idx)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long k = __shfl_xor_sync(kFullMask, key, o);
        const int i = __shfl_xor_sync(kFullMask, idx, o);
        if (k > key) { key = k; idx = i; }
    }
}

// One CTA's part of an image: items [start, start + cnt) of the list, stored at a[0 .. cnt).  solo: the CTA handles the
// whole list alone (block barriers only); otherwise the cluster's CTAs agree on every winner through their slots.
template <bool SMEM>
__device__ __forceinline__ void soft_body(const SoftParams &p, SoftArrays a, int img, int64_t g0, int start, int cnt, bool solo,
                                          SoftSlot *s_slot, unsigned long long *s_wkey, int *s_widx, int *s_best)
{
    if (SMEM) { __builtin_assume(__isShared(a.box)); __builtin_assume(__isShared(a.score)); __builtin_assume(__isShared(a.lo)); __builtin_assume(__isShared(a.cls)); }
    else { __builtin_assume(__isGlobal(a.box)); __builtin_assume(__isGlobal(a.score)); __builtin_assume(__isGlobal(a.lo)); __builtin_assume(__isGlobal(a.cls)); }
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5, T = blockDim.x;
    const int csize = solo ? 1 : (int)cluster.num_blocks(), rank = solo ? 0 : (int)cluster.block_rank();
    const float nan = __int_as_float(0x7fffffff);

    // every thread owns items tid, tid + T, ...: it alone reads and writes their scores inside the loop
    for (int l = tid; l < cnt; l += T) {
        const int i = start + l;
        float s;
        unsigned lo, c;
        float4 bx;
        if (p.mode == 0) {
            const unsigned long long key = __ldg(p.cand_key + g0 + i);
            s = __uint_as_float((unsigned)(key >> 32));
            lo = (unsigned)key;
            bx = __ldg(p.cand_box + g0 + i);
            c = (unsigned)__ldg(p.cand_cls + g0 + i);
        } else {
            s = __ldg(p.scores + g0 + i) + 0.f;                       // -0 -> +0: the key orders them like the values
            lo = ~(unsigned)i;
            bx = __ldg(p.boxes + g0 + i);
            c = (unsigned)__ldg(p.classes + g0 + i);
        }
        a.box[l] = bx;
        a.score[l] = s >= p.score_thr ? s : nan;
        a.lo[l] = lo;
        a.cls[l] = c;
    }

    float4 mbox = make_float4(0.f, 0.f, 0.f, 0.f);
    float marea = 0.f;
    unsigned mcls = 0u;
    bool have = false;
    int emitted = 0, par = 0;
    while (emitted < p.K) {
        // 1. decay the own items of the previous winner's class, then the thread's best key
        unsigned long long best = 0ull;
        int bidx = -1;
        for (int l = tid; l < cnt; l += T) {
            float s = a.score[l];
            if (isnan(s)) continue;
            if (have && a.cls[l] == mcls) {
                const float4 b = a.box[l];
                float iou = box_iou(mbox, marea, b, (b.z - b.x) * (b.w - b.y));
                if (isnan(iou)) iou = 0.f;                             // two zero-area boxes: weight 1
                float w;
                if (p.method == SIHL_OD_SOFT_NMS_LINEAR) w = iou > p.iou_thr ? 1.f - iou : 1.f;
                else w = (float)exp(-(double)iou * (double)iou / p.sigma);
                s = s * w + 0.f;                                       // (+0.f: a negative score decayed to -0 becomes +0)
                if (!(s >= p.score_thr)) { a.score[l] = nan; continue; }
                a.score[l] = s;
            }
            const unsigned long long key = ((unsigned long long)f2ord(s) << 32) | a.lo[l];
            if (key > best) { best = key; bidx = l; }
        }
        // 2. the CTA's best -> its slot
        warp_argmax(best, bidx);
        if (lane == 0) { s_wkey[warp] = best; s_widx[warp] = bidx; }
        __syncthreads();
        if (warp == 0) {
            unsigned long long k = lane < nwarps ? s_wkey[lane] : 0ull;
            int i = lane < nwarps ? s_widx[lane] : -1;
            warp_argmax(k, i);
            if (lane == 0) {
                SoftSlot &sl = s_slot[par];
                sl.key = k;
                if (k != 0ull) { sl.box = a.box[i]; sl.cls = a.cls[i]; sl.score = a.score[i]; }
                *s_best = i;
            }
        }
        if (solo) __syncthreads();
        else cluster.sync();
        // 3. the winner: the largest key over the cluster's slots (every CTA computes the same)
        unsigned long long gk = s_slot[par].key;
        int wr = rank;
        for (int r = 0; r < csize; ++r) {
            if (r == rank) continue;
            const unsigned long long k = cluster.map_shared_rank(&s_slot[par], (unsigned)r)->key;
            if (k > gk) { gk = k; wr = r; }
        }
        if (gk == 0ull) break;                                         // nothing alive anywhere (cluster-uniform)
        const SoftSlot *ws = wr == rank ? &s_slot[par] : cluster.map_shared_rank(&s_slot[par], (unsigned)wr);
        mbox = ws->box;
        mcls = ws->cls;
        const float msc = ws->score;
        marea = (mbox.z - mbox.x) * (mbox.w - mbox.y);
        have = true;
        if (wr == rank) {
            const int b = *s_best;
            if (b % T == tid) a.score[b] = nan;                        // its owner retires the winner
        }
        if (rank == 0 && tid == 0) {
            if (p.mode == 0) {
                const int64_t o = (int64_t)img * p.K + emitted;
                p.out_scores[o] = msc;
                p.out_classes[o] = (int64_t)mcls;
                p.out_boxes[o] = mbox;
            } else {
                p.keep[g0 + emitted] = g0 + (int64_t)(~(unsigned)gk);
                p.keep_scores[g0 + emitted] = msc;
            }
        }
        ++emitted;
        par ^= 1;
    }
    if (!solo) cluster.sync();                                         // no CTA leaves while another may read its slots
    if (rank != 0) return;
    if (p.mode == 0) {
        if (tid == 0) {
            p.num_instances[img] = emitted;
            if (p.reset_counts) const_cast<int32_t *>(p.cand_count)[img] = 0;
        }
        for (int k = emitted + tid; k < p.K; k += T) {
            const int64_t o = (int64_t)img * p.K + k;
            p.out_scores[o] = 0.f;
            p.out_classes[o] = 0;
            p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    } else if (tid == 0) {
        p.keep_count[img] = emitted;
    }
}

__global__ void __launch_bounds__(kSoftThreads) k_soft_nms(SoftParams p)
{
    extern __shared__ __align__(16) unsigned char s_soft[];
    __shared__ SoftSlot s_slot[2];
    __shared__ unsigned long long s_wkey[kSoftThreads / 32];
    __shared__ int s_widx[kSoftThreads / 32];
    __shared__ int s_best;
    cg::cluster_group cluster = cg::this_cluster();
    const int csize = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int img = (int)(blockIdx.x / (unsigned)csize);
    int n;
    int64_t g0;                                                        // the image's first item in the inputs / workspace
    if (p.mode == 0) {
        const int c = __ldg(p.cand_count + img);
        n = (int)(c < p.cap ? c : p.cap);
        g0 = (int64_t)img * p.cap;
    } else {
        g0 = __ldg(p.seg_offsets + img);
        n = __ldg(p.seg_offsets + img + 1) - (int)g0;
    }
    if (csize > 1) cluster.sync();                                     // all have read n before the first CTA may reset it
    const bool solo = csize == 1 || n <= p.smem_items;
    if (solo && rank != 0) return;
    const int parts = solo ? 1 : csize, part = solo ? 0 : rank;
    const int per = (n + parts - 1) / parts;
    const int start = min(n, part * per), cnt = min(n, start + per) - start;
    if (per <= p.smem_items) {
        soft_body<true>(p, carve_soft(s_soft, p.smem_items), img, g0, start, cnt, solo, s_slot, s_wkey, s_widx, &s_best);
    } else {
        const SoftArrays a = offset_soft(carve_soft(p.workspace, p.ws_items), g0 + start);
        soft_body<false>(p, a, img, g0, start, cnt, solo, s_slot, s_wkey, s_widx, &s_best);
    }
}

// CTAs per image for lists of up to `bound` candidates, and the candidates each one holds on chip
static void soft_shape(int64_t bound, int *csize, int *smem_items)
{
    int64_t c = (bound + kSoftItems - 1) / kSoftItems;
    if (c < 1) c = 1;
    if (c > kSoftMaxCluster) c = kSoftMaxCluster;
    const int64_t per = (bound + c - 1) / c;
    *csize = (int)c;
    *smem_items = (int)(per < kSoftItems ? (per < 1 ? 1 : per) : kSoftItems);
}

static bool soft_needs_workspace(int64_t bound) { return bound > (int64_t)kSoftMaxCluster * kSoftItems; }

static int launch_soft(SoftParams p, int n_images, int64_t bound, cudaStream_t st)
{
    int csize, smem_items;
    soft_shape(bound, &csize, &smem_items);
    p.smem_items = smem_items;
    static thread_local bool attr_set = false;
    if (!attr_set) {
        int rc = cuda_status(cudaFuncSetAttribute(k_soft_nms, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                  (int)(kSoftItems * kSoftItemBytes)),
                             "cudaFuncSetAttribute(k_soft_nms)");
        if (rc) return rc;
        attr_set = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((int64_t)n_images * csize));
    cfg.blockDim = dim3((unsigned)kSoftThreads);
    cfg.dynamicSmemBytes = (size_t)smem_items * kSoftItemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cuda_status(cudaLaunchKernelEx(&cfg, k_soft_nms, p), "cudaLaunchKernelEx(k_soft_nms)");
}

static int check_method(int method, float sigma)
{
    SIHL_CHECK_ARG(method == SIHL_OD_SOFT_NMS_LINEAR || method == SIHL_OD_SOFT_NMS_GAUSSIAN,
                   "soft-NMS method %d is not SIHL_OD_SOFT_NMS_LINEAR (1) or SIHL_OD_SOFT_NMS_GAUSSIAN (2)", method);
    SIHL_CHECK_ARG(method != SIHL_OD_SOFT_NMS_GAUSSIAN || sigma > 0.f, "gaussian soft-NMS needs sigma > 0 (got %g)", (double)sigma);
    return SIHL_OD_OK;
}

}  // namespace sihl

using namespace sihl;

extern "C" size_t sihl_od_soft_nms_workspace_bytes(int batch, int64_t cand_capacity)
{
    if (batch <= 0 || cand_capacity <= 0 || !soft_needs_workspace(cand_capacity)) return 0;
    return (size_t)batch * (size_t)cand_capacity * kSoftItemBytes;
}

extern "C" int sihl_od_soft_nms_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                                     const float *cand_box, const int32_t *cand_cls, int batch, int method, float iou_thr,
                                     float sigma, float score_thr, int k, int64_t *num_instances, float *scores,
                                     int64_t *classes, float *boxes, void *workspace, int reset_counts, void *stream)
{
    int rc = check_method(method, sigma);
    if (rc) return rc;
    SIHL_CHECK_ARG(cand_count && cand_key && cand_box && cand_cls, "NULL input");
    SIHL_CHECK_ARG(num_instances && scores && classes && boxes, "NULL output");
    SIHL_CHECK_ARG(cand_capacity >= 1 && cand_capacity < (1ll << 30) && batch >= 0 && k >= 1, "bad sizes");
    SIHL_CHECK_ARG(workspace != nullptr || sihl_od_soft_nms_workspace_bytes(batch, cand_capacity) == 0,
                   "workspace needed for capacity %lld", (long long)cand_capacity);
    if (batch == 0) return SIHL_OD_OK;
    SoftParams p = {};
    p.cand_count = cand_count; p.cap = cand_capacity;
    p.cand_key = reinterpret_cast<const unsigned long long *>(cand_key);
    p.cand_box = reinterpret_cast<const float4 *>(cand_box); p.cand_cls = cand_cls;
    p.num_instances = num_instances; p.out_scores = scores; p.out_classes = classes;
    p.out_boxes = reinterpret_cast<float4 *>(boxes); p.reset_counts = reset_counts;
    p.mode = 0; p.method = method; p.iou_thr = iou_thr; p.score_thr = score_thr; p.sigma = (double)sigma; p.K = k;
    p.workspace = static_cast<unsigned char *>(workspace); p.ws_items = (int64_t)batch * cand_capacity;
    return launch_soft(p, batch, cand_capacity, (cudaStream_t)stream);
}

extern "C" size_t sihl_od_batched_soft_nms_workspace_bytes(int64_t n)
{
    if (n <= 0 || !soft_needs_workspace(n)) return 0;
    return (size_t)n * kSoftItemBytes;
}

extern "C" int sihl_od_batched_soft_nms(const float *boxes, const float *scores, const int64_t *classes,
                                        const int32_t *seg_offsets, int n_images, int64_t n, int method, float iou_thr,
                                        float sigma, float score_thr, int max_out, int64_t *keep, float *keep_scores,
                                        int32_t *keep_count, void *workspace, void *stream)
{
    int rc = check_method(method, sigma);
    if (rc) return rc;
    SIHL_CHECK_ARG(seg_offsets && keep_count, "NULL argument");
    SIHL_CHECK_ARG(n >= 0 && n < (1ll << 30) && n_images >= 0 && max_out >= 1, "bad sizes");
    SIHL_CHECK_ARG(n == 0 || (boxes && scores && classes && keep && keep_scores), "NULL argument");
    SIHL_CHECK_ARG(workspace != nullptr || sihl_od_batched_soft_nms_workspace_bytes(n) == 0, "workspace needed for n=%lld",
                   (long long)n);
    if (n_images == 0) return SIHL_OD_OK;
    SoftParams p = {};
    p.boxes = reinterpret_cast<const float4 *>(boxes); p.scores = scores; p.classes = classes; p.seg_offsets = seg_offsets;
    p.keep = keep; p.keep_scores = keep_scores; p.keep_count = keep_count;
    p.mode = 1; p.method = method; p.iou_thr = iou_thr; p.score_thr = score_thr; p.sigma = (double)sigma; p.K = max_out;
    p.workspace = static_cast<unsigned char *>(workspace); p.ws_items = n;
    return launch_soft(p, n_images, n, (cudaStream_t)stream);
}
