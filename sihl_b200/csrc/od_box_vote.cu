// od_box_vote.cu — class-aware box voting (merge-NMS) after the greedy NMS entries of od_nms.cu.
//
// Gidaris & Komodakis (ICCV 2015); YOLOv5's non_max_suppression(..., merge=True).  Every emitted detection k of class c
// is replaced by the score-weighted mean of the boxes of its list that its own suppression test would claim:
//   V_k = { j in the image's list or the segment : cls_j == c  and  overlap(b_k, b_j) > thr }   (k itself included)
//   b'_k = sum_{j in V_k} s_j * b_j / sum_{j in V_k} s_j        per coordinate
// with the selection's overlap (overlap_gt<kIoU | kDIoU>, od_common.cuh) and threshold.  The products s_j * x_j of two
// fp32 values are exact in fp64; the sums are fp64 and the quotient is rounded once to fp32.  An empty cluster or a zero
// weight sum leaves b_k as it is.  The keep set, its order, the scores and the classes are not touched.
//
// Why the full list: the selection of the top-K entry may have run on the lazy ~200-candidate prefix only (od_nms.cu),
// but the members of a cluster can rank anywhere below it, so every lane strides the whole list of its image / segment.
//
// One warp per emitted detection (a slot of [B, K] or a position of keep [N]); slots past num_instances[b] /
// keep_count[s] exit.  The grid depends on the arguments only, and the pass uses no workspace: it can be captured in a
// CUDA graph after the NMS it follows.  The warp reads the kept box once before it writes, so the top-K entry can
// rewrite the NMS's boxes in place.  Each lane tests the class first, then the overlap; its fp64 partial sums are
// combined by a fixed xor-shuffle tree, so the result does not depend on scheduling.
#include "od_common.cuh"

namespace sihl {

constexpr int kVoteThreads = 256;         // 8 detections per CTA
constexpr int kVoteLists = 0;             // candidate lists of the top-K entries
constexpr int kVoteSegments = 1;          // flat segments of the batched entries

struct VoteParams {
    // kVoteLists: the candidate lists and the top-K outputs of the NMS (boxes rewritten in place)
    const int32_t *cand_count; int64_t cap;
    const unsigned long long *cand_key; const float4 *cand_box; const int32_t *cand_cls;
    int K; const int64_t *num_instances; const int64_t *out_classes; float4 *out_boxes;
    // kVoteSegments: batched NMS inputs, its keep / keep_count, and the voted boxes aligned with keep
    const float4 *boxes; const float *scores; const int64_t *classes; const int32_t *seg_offsets; int n_images;
    const int64_t *keep; const int32_t *keep_count; float4 *voted;
    int64_t n_slots;
    float thr;
};

template <int KIND, int LAYOUT>
__global__ void __launch_bounds__(kVoteThreads) k_box_vote(VoteParams p)
{
    const int64_t slot = ((int64_t)blockIdx.x * kVoteThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (slot >= p.n_slots) return;                       // warp-uniform, like every exit below

    int64_t lb, n;                                       // the list: [lb, lb + n)
    int64_t c;                                           // class of the detection
    float4 bk;
    float4 *dst;
    if (LAYOUT == kVoteLists) {
        const int img = (int)(slot / p.K), k = (int)(slot % p.K);
        if (k >= __ldg(p.num_instances + img)) return;
        const int cnt = __ldg(p.cand_count + img);
        lb = (int64_t)img * p.cap;
        n = cnt < p.cap ? cnt : p.cap;
        dst = p.out_boxes + slot;
        bk = *dst;
        c = (int64_t)(int32_t)p.out_classes[slot];       // the NMS emits the candidate's int32 class
    } else {
        // the segment holding this position: the last s with seg_offsets[s] <= slot
        int lo = 0, hi = p.n_images;                     // seg_offsets[lo] <= slot < seg_offsets[hi] once checked
        if (slot < __ldg(p.seg_offsets) || slot >= __ldg(p.seg_offsets + p.n_images)) return;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(p.seg_offsets + mid) <= slot) lo = mid; else hi = mid;
        }
        lb = __ldg(p.seg_offsets + lo);
        if (slot - lb >= __ldg(p.keep_count + lo)) return;
        n = __ldg(p.seg_offsets + lo + 1) - lb;
        const int64_t i = __ldg(p.keep + slot);
        bk = __ldg(p.boxes + i);
        c = __ldg(p.classes + i);
        dst = p.voted + slot;
    }
    const float ak = (bk.z - bk.x) * (bk.w - bk.y);

    double s = 0.0, sx1 = 0.0, sy1 = 0.0, sx2 = 0.0, sy2 = 0.0;
    for (int64_t j = lane; j < n; j += 32) {
        const int64_t cj = LAYOUT == kVoteLists ? (int64_t)__ldg(p.cand_cls + lb + j) : __ldg(p.classes + lb + j);
        if (cj != c) continue;
        const float4 bj = LAYOUT == kVoteLists ? __ldg(p.cand_box + lb + j) : __ldg(p.boxes + lb + j);
        if (!overlap_gt<KIND>(bk, ak, bj, (bj.z - bj.x) * (bj.w - bj.y), p.thr)) continue;
        const float sj = LAYOUT == kVoteLists ? __uint_as_float((unsigned)(__ldg(p.cand_key + lb + j) >> 32))
                                              : __ldg(p.scores + lb + j);
        const double w = (double)sj;
        s += w;
        sx1 += w * (double)bj.x; sy1 += w * (double)bj.y;
        sx2 += w * (double)bj.z; sy2 += w * (double)bj.w;
    }
    s = warp_sum(s);
    sx1 = warp_sum(sx1); sy1 = warp_sum(sy1); sx2 = warp_sum(sx2); sy2 = warp_sum(sy2);
    if (lane == 0) {
        float4 out = bk;
        if (s != 0.0) out = make_float4((float)(sx1 / s), (float)(sy1 / s), (float)(sx2 / s), (float)(sy2 / s));
        *dst = out;
    }
}

template <int LAYOUT>
static int launch_box_vote(const VoteParams &p, int kind, cudaStream_t st)
{
    if (p.n_slots == 0) return SIHL_OD_OK;
    const int64_t grid = (p.n_slots * 32 + kVoteThreads - 1) / kVoteThreads;
    if (kind == kDIoU) k_box_vote<kDIoU, LAYOUT><<<(unsigned)grid, kVoteThreads, 0, st>>>(p);
    else k_box_vote<kIoU, LAYOUT><<<(unsigned)grid, kVoteThreads, 0, st>>>(p);
    SIHL_CHECK_LAUNCH("k_box_vote");
    return SIHL_OD_OK;
}

// The argument checks mirror sihl_od_nms_topk's (the lists) and sihl_od_batched_nms's (the segments).
static int box_vote_topk_entry(int kind, const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                               const float *cand_box, const int32_t *cand_cls, int batch, float thr, int k,
                               const int64_t *num_instances, const int64_t *classes, float *boxes, void *stream)
{
    SIHL_CHECK_ARG(cand_count && cand_key && cand_box && cand_cls, "NULL input");
    SIHL_CHECK_ARG(num_instances && classes && boxes, "NULL output");
    SIHL_CHECK_ARG(cand_capacity >= 1 && cand_capacity < (1ll << 30) && k >= 1, "bad sizes");
    if (batch <= 0) return SIHL_OD_OK;
    VoteParams p = {};
    p.cand_count = cand_count; p.cap = cand_capacity;
    p.cand_key = reinterpret_cast<const unsigned long long *>(cand_key);
    p.cand_box = reinterpret_cast<const float4 *>(cand_box); p.cand_cls = cand_cls;
    p.K = k; p.num_instances = num_instances; p.out_classes = classes; p.out_boxes = reinterpret_cast<float4 *>(boxes);
    p.n_slots = (int64_t)batch * k; p.thr = thr;
    return launch_box_vote<kVoteLists>(p, kind, (cudaStream_t)stream);
}

static int batched_box_vote_entry(int kind, const float *boxes, const float *scores, const int64_t *classes,
                                  const int32_t *seg_offsets, int n_images, int64_t n, float thr, const int64_t *keep,
                                  const int32_t *keep_count, float *voted_boxes, void *stream)
{
    SIHL_CHECK_ARG(seg_offsets && keep_count, "NULL argument");
    SIHL_CHECK_ARG(n >= 0 && n < (1ll << 30) && n_images >= 0, "bad sizes");
    SIHL_CHECK_ARG(n == 0 || (boxes && scores && classes && keep && voted_boxes), "NULL argument");
    if (n_images == 0) return SIHL_OD_OK;
    VoteParams p = {};
    p.boxes = reinterpret_cast<const float4 *>(boxes); p.scores = scores; p.classes = classes;
    p.seg_offsets = seg_offsets; p.n_images = n_images;
    p.keep = keep; p.keep_count = keep_count; p.voted = reinterpret_cast<float4 *>(voted_boxes);
    p.n_slots = n; p.thr = thr;
    return launch_box_vote<kVoteSegments>(p, kind, (cudaStream_t)stream);
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_box_vote_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                                     const float *cand_box, const int32_t *cand_cls, int batch, float iou_thr, int k,
                                     const int64_t *num_instances, const int64_t *classes, float *boxes, void *stream)
{
    return box_vote_topk_entry(kIoU, cand_count, cand_capacity, cand_key, cand_box, cand_cls, batch, iou_thr, k,
                               num_instances, classes, boxes, stream);
}

extern "C" int sihl_od_diou_box_vote_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                                          const float *cand_box, const int32_t *cand_cls, int batch, float diou_thr, int k,
                                          const int64_t *num_instances, const int64_t *classes, float *boxes, void *stream)
{
    return box_vote_topk_entry(kDIoU, cand_count, cand_capacity, cand_key, cand_box, cand_cls, batch, diou_thr, k,
                               num_instances, classes, boxes, stream);
}

extern "C" int sihl_od_batched_box_vote(const float *boxes, const float *scores, const int64_t *classes,
                                        const int32_t *seg_offsets, int n_images, int64_t n, float iou_thr,
                                        const int64_t *keep, const int32_t *keep_count, float *voted_boxes, void *stream)
{
    return batched_box_vote_entry(kIoU, boxes, scores, classes, seg_offsets, n_images, n, iou_thr, keep, keep_count,
                                  voted_boxes, stream);
}

extern "C" int sihl_od_batched_diou_box_vote(const float *boxes, const float *scores, const int64_t *classes,
                                             const int32_t *seg_offsets, int n_images, int64_t n, float diou_thr,
                                             const int64_t *keep, const int32_t *keep_count, float *voted_boxes,
                                             void *stream)
{
    return batched_box_vote_entry(kDIoU, boxes, scores, classes, seg_offsets, n_images, n, diou_thr, keep, keep_count,
                                  voted_boxes, stream);
}
