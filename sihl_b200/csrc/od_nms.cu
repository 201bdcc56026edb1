// od_nms.cu — class-aware greedy NMS (SURVEY.md §8 a15; north-star extension, the
// reference has no NMS).  Semantics: torchvision's exact per-class path
// (_batched_nms_vanilla, tv:ops/boxes.py:102-120, over the CPU nms kernel): visit boxes by
// (score desc, index asc); a kept box suppresses every later box of the same class with
// inter / (area_i + area_j - inter) > thr.
//
// k_nms: one CTA per image (segment), sort-free, the list length (known only on the device) picks the body:
//   * n <= 256 (nms_small_body): 2 (top-K entry) or 4 lanes per candidate; ONE counting pass over the list gives every candidate its
//     rank (score desc, index asc), its class-major position and its class segment; suppression bitmasks per
//     candidate against the earlier boxes of its class (all pairs in parallel), greedy chain on bits.
//   * top-K entry with n > 256 and K <= 128 (lazy prefix): greedy NMS is prefix-closed — whether a box is kept
//     depends only on higher-ranked boxes — so the K best survivors are found among the ~200 highest-ranked
//     candidates whenever at least K of them survive: a 4-pass radix select picks that prefix (all ties with it),
//     the short-list body runs on it, and only if fewer than K survive does the full list get processed.
//   * longer lists (nms_medium_body): class buckets through a shared-memory hash table (count -> scan -> scatter),
//     rank by counting inside the class, 64-bit suppression masks for classes <= 64 boxes, 32-box chunks (all
//     pairs of a chunk in parallel by shuffles, then the chunk's kept boxes against the rest) by one warp per
//     class up to 2048 boxes and by the whole CTA beyond, top-K by radix select of the K-th score; arrays in
//     shared memory up to 4096 candidates, in the global workspace beyond (the top-K entry: always the workspace).
//   * more than 512 distinct classes (nms_big_body): the two-bitonic-sort fallback — sort by rank, sort by
//     (class, rank), per-segment suppression, ordered compaction.
// Footprint: the top-K entry runs next to the dense scan of the other steps in flight (two 256-thread scan CTAs per SM,
// 16 384 registers and ~46 KB of shared memory each).  Its CTA (k_nms<kNmsThreadsTopk>) therefore stays within half the
// register file (512 threads x <= 64 registers) and reserves no dynamic shared memory: its long-list arrays live in the
// per-image workspace (small and L2-resident), and the short-list body needs only the ~27 KB of static shared memory.
// The stand-alone entries (segment-mode batched NMS, the class-split sub-lists) run with 1024 threads and keep their
// long-list arrays on chip: with 512 threads and the workspace, batched NMS of 1 000-5 000 boxes took 8-63 % longer.
// tests/test_kernel_footprint.py checks the top-K budget on the built library.
// sihl_od_nms_topk_split deals an image's candidates to several CTAs by class; stand-alone batched NMS of
// 8192..90000 boxes takes the multi-CTA bitmask path of od_nms_wide.cu (whole GPU) instead of one CTA.
#include "od_common.cuh"

namespace sihl {

constexpr int kNmsThreadsTopk = 512;     // the top-K entry (beside the dense scan)
constexpr int kNmsThreadsAlone = 1024;   // the stand-alone entries
constexpr int kSmemItems = 4096;          // per-image candidates held on chip
constexpr int kBigSegment = 512;
constexpr int kSmallItems = 256;          // lists up to this size take the single-pass rank-sort kernel
constexpr size_t kSmemItemBytes = 47;     // dynamic shared memory per on-chip candidate: max over the two long-list layouts (41, 47)
constexpr size_t kWsItemBytes = 48;       // workspace stride per item (keeps every image 16-B aligned)

__device__ __forceinline__ unsigned f2ord_nms(float f)
{
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

struct NmsArrays {
    unsigned long long *key;   // [np] sort keys; after step 2: (class << 32 | r) by q
    float4 *box;               // [np] by q
    unsigned *val;             // [np] rank -> slot, later rank -> q
    float *area;               // [np] by q
    unsigned *slot;            // [np] by q
    int *seg;                  // [np] segment starts (+ sentinel)
    unsigned char *dead;       // [np] by q
};

__device__ __forceinline__ NmsArrays carve(unsigned char *base, int np)
{
    NmsArrays a;
    a.key = reinterpret_cast<unsigned long long *>(base);
    a.box = reinterpret_cast<float4 *>(base + (size_t)np * 8);
    a.val = reinterpret_cast<unsigned *>(base + (size_t)np * 24);
    a.area = reinterpret_cast<float *>(base + (size_t)np * 28);
    a.slot = reinterpret_cast<unsigned *>(base + (size_t)np * 32);
    a.seg = reinterpret_cast<int *>(base + (size_t)np * 36);
    a.dead = base + (size_t)np * 40;
    return a;
}

template <bool DESC>
__device__ __forceinline__ void bitonic_kv(unsigned long long *key, unsigned *val, int np)
{
    for (int k = 2; k <= np; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < np; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = key[i], b = key[ixj];
                    const bool first = (i & k) == 0;
                    const bool swap = DESC ? (first ? (a < b) : (a > b)) : (first ? (a > b) : (a < b));
                    if (swap) {
                        key[i] = b; key[ixj] = a;
                        if (val) { const unsigned t = val[i]; val[i] = val[ixj]; val[ixj] = t; }
                    }
                }
            }
            __syncthreads();
        }
}

// Ordered block compaction: emit(i, rank) for every i in [0,n) with flag(i); rank ascends with i.
template <class Flag, class Emit>
__device__ __forceinline__ int block_ordered_compact(int n, int *s_warp /* [33] */, Flag flag, Emit emit)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int running = 0;
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool f = i < n && flag(i);
        const unsigned m = __ballot_sync(kFullMask, f);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        if (warp == 0) {
            const int x = lane < nwarps ? s_warp[lane] : 0;
            int incl = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += y;
            }
            if (lane < nwarps) s_warp[lane] = incl - x;
            if (lane == 31) s_warp[32] = incl;
        }
        __syncthreads();
        if (f) emit(i, running + s_warp[warp] + __popc(m & ((1u << lane) - 1u)));
        running += s_warp[32];
        __syncthreads();
    }
    return running;
}

// torchvision/csrc/ops/cpu/nms_kernel.cpp: ovr = inter / (iarea + areas[j] - inter); ovr > thr
__device__ __forceinline__ bool iou_gt(float4 a, float area_a, float4 b, float area_b, float thr)
{
    const float w = fmaxf(0.f, fminf(a.z, b.z) - fmaxf(a.x, b.x));
    const float h = fmaxf(0.f, fminf(a.w, b.w) - fmaxf(a.y, b.y));
    const float inter = w * h;
    return inter / ((area_a + area_b) - inter) > thr;
}

__device__ __forceinline__ float4 shfl4(float4 v, int src)
{
    return make_float4(__shfl_sync(kFullMask, v.x, src), __shfl_sync(kFullMask, v.y, src), __shfl_sync(kFullMask, v.z, src),
                       __shfl_sync(kFullMask, v.w, src));
}

// Greedy suppression inside one 32-box chunk of a score-ordered class segment, by one warp (lane = box).
// `dead` = already suppressed by an earlier chunk.  Returns the kept bits of the chunk (same value in every lane):
// all 32 x 31 / 2 pairs are tested in parallel (boxes broadcast by shuffles), then the greedy chain runs on bits.
__device__ __forceinline__ unsigned chunk_greedy(float4 bi, float ai, bool dead, float thr, int lane)
{
    unsigned over = 0u;                                   // earlier boxes of the chunk that overlap this one
#pragma unroll 4
    for (int l = 0; l < 31; ++l) {
        const float4 bl = shfl4(bi, l);
        const float al = __shfl_sync(kFullMask, ai, l);
        if (l < lane && iou_gt(bl, al, bi, ai, thr)) over |= 1u << l;
    }
    const unsigned alive = __ballot_sync(kFullMask, !dead);
    unsigned kept = 0u;
#pragma unroll 4
    for (int l = 0; l < 32; ++l) {
        const unsigned ol = __shfl_sync(kFullMask, over, l);
        if (((alive >> l) & 1u) && (ol & kept) == 0u) kept |= 1u << l;
    }
    return kept;
}

// One warp, one class segment [q0, q0 + m) in score order: chunks of 32 boxes; the kept boxes of a chunk then
// suppress the later boxes of the segment (32 at a time).  m^2/2 pair tests like the serial formulation, but
// m/32 dependent steps instead of m.
template <bool SMEM>   // SMEM: the arrays live in shared memory (lets the compiler emit LDS/STS instead of generic accesses)
__device__ __forceinline__ void warp_segment_nms(const float4 *box, const float *area, unsigned char *dead_flag, int q0, int m,
                                                 float thr, int lane)
{
    if (SMEM) { __builtin_assume(__isShared(box)); __builtin_assume(__isShared(area)); __builtin_assume(__isShared(dead_flag)); }
    else { __builtin_assume(__isGlobal(box)); __builtin_assume(__isGlobal(area)); __builtin_assume(__isGlobal(dead_flag)); }
    for (int c0 = 0; c0 < m; c0 += 32) {
        __syncwarp();
        const int i = c0 + lane;
        const bool valid = i < m;
        const float4 bi = valid ? box[q0 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
        const float ai = valid ? area[q0 + i] : 0.f;
        const bool dead = valid ? dead_flag[q0 + i] != 0 : true;
        const unsigned kept = chunk_greedy(bi, ai, dead, thr, lane);
        if (valid && !dead && !((kept >> lane) & 1u)) dead_flag[q0 + i] = 1;
        for (int j0 = c0 + 32; j0 < m; j0 += 32) {
            const int j = j0 + lane;
            const bool live = j < m && dead_flag[q0 + j] == 0;
            const float4 bj = live ? box[q0 + j] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float aj = live ? area[q0 + j] : 0.f;
            bool kill = false;
            for (unsigned k = kept; k != 0u; k &= k - 1u) {              // warp-uniform
                const int l = __ffs(k) - 1;
                const float4 bl = shfl4(bi, l);
                const float al = __shfl_sync(kFullMask, ai, l);
                if (live && !kill && iou_gt(bl, al, bj, aj, thr)) kill = true;
            }
            if (kill) dead_flag[q0 + j] = 1;
        }
    }
}

// The whole CTA, one very long class segment: warp 0 resolves a chunk of 32 boxes and publishes its kept boxes in
// shared memory; every thread then tests its share of the later boxes against them.  2 barriers per 32 boxes.
struct ChunkScratch { float4 box[32]; float area[32]; unsigned kept; int n_big; int big[32]; };

template <bool SMEM>
__device__ __forceinline__ void cta_segment_nms(const float4 *box, const float *area, unsigned char *dead_flag, int q0, int m,
                                                float thr, ChunkScratch *sc)
{
    if (SMEM) { __builtin_assume(__isShared(box)); __builtin_assume(__isShared(area)); __builtin_assume(__isShared(dead_flag)); }
    else { __builtin_assume(__isGlobal(box)); __builtin_assume(__isGlobal(area)); __builtin_assume(__isGlobal(dead_flag)); }
    __builtin_assume(__isShared(sc));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int c0 = 0; c0 < m; c0 += 32) {
        __syncthreads();                                                  // flags of the previous pass are visible
        if (warp == 0) {
            const int i = c0 + lane;
            const bool valid = i < m;
            const float4 bi = valid ? box[q0 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float ai = valid ? area[q0 + i] : 0.f;
            const bool dead = valid ? dead_flag[q0 + i] != 0 : true;
            const unsigned kept = chunk_greedy(bi, ai, dead, thr, lane);
            if (valid && !dead && !((kept >> lane) & 1u)) dead_flag[q0 + i] = 1;
            sc->box[lane] = bi;
            sc->area[lane] = ai;
            if (lane == 0) sc->kept = kept;
        }
        __syncthreads();
        const unsigned kept = sc->kept;
        if (kept == 0u) continue;                                         // block-uniform
        for (int j = c0 + 32 + tid; j < m; j += blockDim.x) {
            if (dead_flag[q0 + j]) continue;
            const float4 bj = box[q0 + j];
            const float aj = area[q0 + j];
            for (unsigned k = kept; k != 0u; k &= k - 1u) {
                const int l = __ffs(k) - 1;
                if (iou_gt(sc->box[l], sc->area[l], bj, aj, thr)) { dead_flag[q0 + j] = 1; break; }
            }
        }
    }
    __syncthreads();
}

struct NmsParams {
    // mode 0: candidate lists written by k_dense_decode
    const int32_t *cand_count; int64_t cap;
    const unsigned long long *cand_key; const float4 *cand_box; const int32_t *cand_cls;
    // mode 1: torchvision.ops.batched_nms inputs + segment offsets
    const float4 *boxes; const float *scores; const int64_t *classes; const int32_t *seg_offsets;
    int mode;
    float iou_thr;
    int K; int64_t *num_instances; float *out_scores; int64_t *out_classes; float4 *out_boxes;   // mode 0
    int64_t *keep; int32_t *keep_count;                                                           // mode 1
    unsigned char *workspace; size_t ws_stride;   // mode 0: bytes per image; mode 1: unused (offset = 2*seg start)
    int reset_counts;          // mode 0: zero cand_count[img] once consumed (saves the next step's memset launch)
    // mode 0, class-split launch (sihl_od_nms_topk_split): list i starts at list_offsets[i] inside the candidate
    // arrays instead of i * cap, and the sort key of every emitted detection is written next to it
    const int32_t *list_offsets;
    unsigned long long *out_keys;
    int smem_items;            // candidates per list that the launch's dynamic shared memory holds (<= kSmemItems)
};

__device__ __forceinline__ int64_t list_base(const NmsParams &p, int img)
{
    return p.list_offsets != nullptr ? (int64_t)__ldg(p.list_offsets + img) : (int64_t)img * p.cap;
}
__device__ __forceinline__ unsigned char *list_workspace(const NmsParams &p, int img, int src0)
{
    if (p.mode != 0) return p.workspace + (size_t)2 * src0 * kWsItemBytes;
    if (p.list_offsets != nullptr) return p.workspace + (size_t)2 * __ldg(p.list_offsets + img) * kWsItemBytes;
    return p.workspace + (size_t)img * p.ws_stride;
}

__device__ __forceinline__ void nms_big_body(const NmsParams &p)
{
    extern __shared__ __align__(16) unsigned char s_dyn[];
    __shared__ int s_warp[33];

    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int64_t lb = p.mode == 0 ? list_base(p, img) : 0;
    int n, src0;
    if (p.mode == 0) {
        const int c = __ldg(p.cand_count + img);
        n = (int)(c < p.cap ? c : p.cap);
        src0 = 0;
    } else {
        src0 = __ldg(p.seg_offsets + img);
        n = __ldg(p.seg_offsets + img + 1) - src0;
    }
    int np = 2;
    while (np < n) np <<= 1;
    int n_kept = 0;

    if (n > 0) {
        unsigned char *base = s_dyn;
        if (np > p.smem_items)
            base = list_workspace(p, img, src0);
        const NmsArrays ar = carve(base, np);

        // 1. rank by (score desc, index asc)
        for (int i = tid; i < np; i += blockDim.x) {
            unsigned long long key = 0ull;
            if (i < n) {
                if (p.mode == 0) key = __ldg(p.cand_key + lb + i);
                else key = ((unsigned long long)f2ord_nms(__ldg(p.scores + src0 + i)) << 32) |
                           (unsigned long long)(0xffffffffu - (unsigned)i);
            }
            ar.key[i] = key;
            ar.val[i] = (unsigned)i;
        }
        __syncthreads();
        bitonic_kv<true>(ar.key, ar.val, np);

        // 2. class-major order; the rank in the low word keeps score order inside a class
        for (int r = tid; r < np; r += blockDim.x) {
            unsigned long long key = ~0ull;
            if (r < n) {
                const unsigned slot = ar.val[r];
                const unsigned c = p.mode == 0 ? (unsigned)__ldg(p.cand_cls + lb + slot)
                                               : (unsigned)__ldg(p.classes + src0 + slot);
                key = ((unsigned long long)c << 32) | (unsigned long long)r;
            }
            ar.key[r] = key;
        }
        __syncthreads();
        bitonic_kv<false>(ar.key, nullptr, np);
        for (int q = tid; q < n; q += blockDim.x) {
            const unsigned r = (unsigned)(ar.key[q] & 0xffffffffu), slot = ar.val[r];
            const float4 bx = p.mode == 0 ? __ldg(p.cand_box + lb + slot) : __ldg(p.boxes + src0 + slot);
            ar.box[q] = bx;
            ar.area[q] = (bx.z - bx.x) * (bx.w - bx.y);
            ar.slot[q] = slot;
            ar.dead[q] = 0;
        }
        __syncthreads();
        for (int q = tid; q < n; q += blockDim.x) ar.val[(unsigned)(ar.key[q] & 0xffffffffu)] = (unsigned)q;   // rank -> q

        // 3. class segments
        const int n_seg = block_ordered_compact(
            n, s_warp, [&](int q) { return q == 0 || (ar.key[q] >> 32) != (ar.key[q - 1] >> 32); },
            [&](int q, int s) { ar.seg[s] = q; });
        if (tid == 0) ar.seg[n_seg] = n;
        __syncthreads();
        bool any_big = false;
        for (int s = warp; s < n_seg; s += nwarps) {
            const int q0 = ar.seg[s], m = ar.seg[s + 1] - q0;
            if (m > kBigSegment) continue;
            for (int i = 0; i + 1 < m; ++i) {
                __syncwarp();
                if (ar.dead[q0 + i]) continue;
                const float4 bi = ar.box[q0 + i];
                const float ai = ar.area[q0 + i];
                for (int j = i + 1 + lane; j < m; j += 32)
                    if (!ar.dead[q0 + j] && iou_gt(bi, ai, ar.box[q0 + j], ar.area[q0 + j], p.iou_thr)) ar.dead[q0 + j] = 1;
            }
        }
        for (int s = 0; s < n_seg; ++s) any_big |= (ar.seg[s + 1] - ar.seg[s]) > kBigSegment;
        __syncthreads();
        if (any_big) {
            for (int s = 0; s < n_seg; ++s) {
                const int q0 = ar.seg[s], m = ar.seg[s + 1] - q0;
                if (m <= kBigSegment) continue;
                for (int i = 0; i + 1 < m; ++i) {
                    __syncthreads();
                    if (ar.dead[q0 + i]) continue;
                    const float4 bi = ar.box[q0 + i];
                    const float ai = ar.area[q0 + i];
                    for (int j = i + 1 + tid; j < m; j += blockDim.x)
                        if (!ar.dead[q0 + j] && iou_gt(bi, ai, ar.box[q0 + j], ar.area[q0 + j], p.iou_thr))
                            ar.dead[q0 + j] = 1;
                }
                __syncthreads();
            }
        }

        // 4. survivors in rank order
        n_kept = block_ordered_compact(
            n, s_warp, [&](int r) { return ar.dead[ar.val[r]] == 0; },
            [&](int r, int k) {
                const unsigned q = ar.val[r], slot = ar.slot[q];
                if (p.mode == 0) {
                    if (k < p.K) {
                        const int64_t o = (int64_t)img * p.K + k;
                        const unsigned long long ck = __ldg(p.cand_key + lb + slot);
                        p.out_scores[o] = __uint_as_float((unsigned)(ck >> 32));
                        p.out_classes[o] = (int64_t)(ar.key[q] >> 32);
                        p.out_boxes[o] = ar.box[q];
                        if (p.out_keys != nullptr) p.out_keys[o] = ck;
                    }
                } else {
                    p.keep[src0 + k] = (int64_t)src0 + slot;
                }
            });
    }

    if (p.mode == 0) {
        const int m = n_kept < p.K ? n_kept : p.K;
        if (tid == 0) {
            p.num_instances[img] = m;
            if (p.reset_counts) const_cast<int32_t *>(p.cand_count)[img] = 0;
        }
        for (int k = m + tid; k < p.K; k += blockDim.x) {
            const int64_t o = (int64_t)img * p.K + k;
            p.out_scores[o] = 0.f;
            p.out_classes[o] = 0;
            p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    } else if (tid == 0) {
        p.keep_count[img] = n_kept;
    }
}

// Short lists (n <= kSmallItems, the common case after a 0.05 score threshold).  THREADS / 256 lanes per
// candidate; ONE counting pass over shared memory yields, per candidate, its rank r in
// (score desc, index asc) order, its class-major position q, and the start / length of its
// class segment.  Suppression is then a per-candidate bitmask of earlier same-class boxes with
// IoU > thr (all pairs in parallel, no serial dependence), resolved by one lane per segment with
// pure bit operations — the greedy chain costs a few cycles per box instead of a shared-memory
// round trip per kept box.  Segments longer than 32 fall back to the broadcast loop of k_nms.
// `sel` (optional, shared memory): the body runs on the n_sel candidates lb + sel[0..n_sel) instead of the whole list
// (lazy top-K prefix).  Returns the number of survivors; with finalize == false the per-image epilogue
// (num_instances, zero padding, counter reset) is left to the caller.
template <int THREADS>
__device__ __forceinline__ int nms_small_body(const NmsParams &p, const int *sel = nullptr, int n_sel = 0, bool finalize = true)
{
    constexpr int kLanes = THREADS / kSmallItems;
    static_assert(kLanes * kSmallItems == THREADS && (kLanes == 2 || kLanes == 4), "short-list path: 2 or 4 lanes per candidate");
    __shared__ unsigned long long s_key[kSmallItems];
    __shared__ unsigned s_cls[kSmallItems];        // by slot
    __shared__ float4 s_box[kSmallItems];          // by q
    __shared__ float s_area[kSmallItems];          // by q
    __shared__ unsigned s_mask[kSmallItems];       // by q: earlier boxes of the segment that suppress q (if kept)
    __shared__ unsigned s_keep[kSmallItems];       // by segment start: kept bits of the segment
    __shared__ unsigned char s_dead[kSmallItems];  // by q (only for segments longer than 32)
    __shared__ unsigned short s_q_of_r[kSmallItems], s_slot_of_r[kSmallItems], s_seg0_of_q[kSmallItems], s_len_of_q[kSmallItems];
    __shared__ int s_warp[33];
    __shared__ int s_big;

    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int64_t lb = p.mode == 0 ? list_base(p, img) : 0;
    const int item = tid / kLanes, sub = tid % kLanes;
    int n, src0;
    if (p.mode == 0) {
        const int c = __ldg(p.cand_count + img);
        n = (int)(c < p.cap ? c : p.cap);
        src0 = 0;
    } else {
        src0 = __ldg(p.seg_offsets + img);
        n = __ldg(p.seg_offsets + img + 1) - src0;
    }
    if (sel != nullptr) n = n_sel;
    int n_kept = 0;
    if (n > 0) {
        const bool have = item < n;
        unsigned long long key = 0ull;
        unsigned cls = 0;
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        if (have) {
            if (p.mode == 0) {
                const int src = sel != nullptr ? sel[item] : item;
                key = __ldg(p.cand_key + lb + src);
                cls = (unsigned)__ldg(p.cand_cls + lb + src);
                bx = __ldg(p.cand_box + lb + src);
            } else {
                key = ((unsigned long long)f2ord_nms(__ldg(p.scores + src0 + item)) << 32) |
                      (unsigned long long)(0xffffffffu - (unsigned)item);
                cls = (unsigned)__ldg(p.classes + src0 + item);
                bx = __ldg(p.boxes + src0 + item);
            }
            if (sub == 0) { s_key[item] = key; s_cls[item] = cls; }
        }
        if (tid == 0) s_big = 0;
        // Keys are distinct in every valid list, which makes the ranks below a permutation of 0..n-1.  Should a caller
        // hand in a list with repeated entries (decode run twice without zeroing the counters), ranks collide and some
        // slots of the rank-indexed tables are never written: give them in-bounds defaults, so that such a list yields
        // a meaningless but memory-safe result instead of stale shared-memory indices (measured: a tie-break inside
        // the counting loop would do the same for 2 % of the candidate-first step; these five stores are free).
        if (sub == 0 && item < kSmallItems) {
            s_q_of_r[item] = 0; s_slot_of_r[item] = 0; s_seg0_of_q[item] = 0; s_len_of_q[item] = 1; s_mask[item] = 0u;
            s_keep[item] = 0u; s_dead[item] = 0; s_box[item] = make_float4(0.f, 0.f, 0.f, 0.f); s_area[item] = 0.f;
        }
        __syncthreads();
        // one pass: r = #better keys; seg0 = #smaller classes; k = #better keys of the same class; len = #same class
        int r = 0, seg0 = 0, k = 0, len = 0;
        if (have) {
#pragma unroll 4
            for (int j = sub; j < n; j += kLanes) {
                const unsigned long long kj = s_key[j];
                const unsigned cj = s_cls[j];
                const bool better = kj > key, same = cj == cls;
                r += better;
                seg0 += cj < cls;
                k += same && better;
                len += same;
            }
        }
#pragma unroll
        for (int o = kLanes / 2; o > 0; o >>= 1) {
            r += __shfl_xor_sync(kFullMask, r, o);
            seg0 += __shfl_xor_sync(kFullMask, seg0, o);
            k += __shfl_xor_sync(kFullMask, k, o);
            len += __shfl_xor_sync(kFullMask, len, o);
        }
        const int q = seg0 + k;
        if (have && sub == 0) {
            s_box[q] = bx;
            s_area[q] = (bx.z - bx.x) * (bx.w - bx.y);
            s_q_of_r[r] = (unsigned short)q;
            s_slot_of_r[r] = (unsigned short)item;
            s_seg0_of_q[q] = (unsigned short)seg0;
            s_len_of_q[q] = (unsigned short)len;
            s_dead[q] = 0;
            if (len > 32) s_big = 1;
        }
        __syncthreads();
        // suppressor masks: the lanes of a candidate split its earlier same-class boxes
        unsigned mask = 0;
        if (have && len <= 32) {
            const float area = (bx.z - bx.x) * (bx.w - bx.y);
            for (int j = sub; j < k; j += kLanes)
                if (iou_gt(s_box[seg0 + j], s_area[seg0 + j], bx, area, p.iou_thr)) mask |= 1u << j;
        }
#pragma unroll
        for (int o = kLanes / 2; o > 0; o >>= 1) mask |= __shfl_xor_sync(kFullMask, mask, o);
        if (have && sub == 0) s_mask[q] = mask;
        __syncthreads();
        if (have && sub == 0 && k == 0 && len <= 32) {          // segment leader: greedy pass on bits only
            unsigned kept = 1u;
            for (int i = 1; i < len; ++i)
                if ((s_mask[seg0 + i] & kept) == 0u) kept |= 1u << i;
            s_keep[seg0] = kept;
        }
        __syncthreads();
        if (s_big) {                                             // rare: a class with more than 32 candidates
            const int warp = tid >> 5, nwarps = blockDim.x >> 5;
            for (int qq = warp; qq < n; qq += nwarps) {          // a warp per long segment, found by its leader
                const int q0 = s_seg0_of_q[qq], m = s_len_of_q[qq];
                if (qq != q0 || m <= 32) continue;
                for (int i = 0; i + 1 < m; ++i) {
                    __syncwarp();
                    if (s_dead[q0 + i]) continue;
                    const float4 bi = s_box[q0 + i];
                    const float ai = s_area[q0 + i];
                    for (int j = i + 1 + lane; j < m; j += 32)
                        if (!s_dead[q0 + j] && iou_gt(bi, ai, s_box[q0 + j], s_area[q0 + j], p.iou_thr)) s_dead[q0 + j] = 1;
                }
            }
            __syncthreads();
        }
        // survivors in rank order
        n_kept = block_ordered_compact(
            n, s_warp,
            [&](int rr) {
                const int qq = s_q_of_r[rr], q0 = s_seg0_of_q[qq];
                return s_len_of_q[qq] <= 32 ? ((s_keep[q0] >> (qq - q0)) & 1u) != 0u : s_dead[qq] == 0;
            },
            [&](int rr, int kk) {
                const int qq = s_q_of_r[rr], slot = s_slot_of_r[rr];
                if (p.mode == 0) {
                    if (kk < p.K) {
                        const int64_t o = (int64_t)img * p.K + kk;
                        p.out_scores[o] = __uint_as_float((unsigned)(s_key[slot] >> 32));
                        p.out_classes[o] = (int64_t)s_cls[slot];
                        p.out_boxes[o] = s_box[qq];
                        if (p.out_keys != nullptr) p.out_keys[o] = s_key[slot];
                    }
                } else {
                    p.keep[src0 + kk] = (int64_t)src0 + slot;
                }
            });
    }
    if (!finalize) return n_kept;
    if (p.mode == 0) {
        const int m = n_kept < p.K ? n_kept : p.K;
        if (tid == 0) {
            p.num_instances[img] = m;
            if (p.reset_counts) const_cast<int32_t *>(p.cand_count)[img] = 0;
        }
        for (int kk = m + tid; kk < p.K; kk += blockDim.x) {
            const int64_t o = (int64_t)img * p.K + kk;
            p.out_scores[o] = 0.f;
            p.out_classes[o] = 0;
            p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    } else if (tid == 0) {
        p.keep_count[img] = n_kept;
    }
    return n_kept;
}

// Lazy prefix for the top-K entry (mode 0): pick the ~kLazyTarget highest-ranked candidates of a long list — every
// candidate whose score is >= the kLazyTarget-th largest score, i.e. a prefix of the visit order closed under
// ties — into s_sel.  4-pass MSB radix select on the score word of the key (scores are sigmoid outputs > 0: their
// bit patterns order like the values).  Returns the prefix length, or 0 if it would not fit (a tie wider than the
// short-list body) and the caller should process the full list.
constexpr int kLazyTarget = 200;
constexpr int kLazyMaxK = 128;
__device__ __forceinline__ int lazy_prefix_select(const NmsParams &p, int64_t lb, int n, int *s_sel, unsigned *s_hist,
                                                  unsigned *s_pick, int *s_count)
{
    const int tid = threadIdx.x, lane = tid & 31;
    unsigned prefix = 0u, mask = 0u, remaining = (unsigned)kLazyTarget;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
        for (int i0 = 0; i0 < n; i0 += blockDim.x) {
            const int i = i0 + tid;
            const bool ok = i < n;
            const unsigned u = ok ? (unsigned)(__ldg(p.cand_key + lb + i) >> 32) : 0u;
            const bool in = ok && ((u & mask) == prefix);
            const unsigned digit = (u >> shift) & 255u;
            const unsigned act = __ballot_sync(kFullMask, in);
            if (in) {                                       // warp-aggregated histogram update (scores cluster)
                const unsigned peers = __match_any_sync(act, digit);
                if (lane == __ffs(peers) - 1) atomicAdd(&s_hist[digit], (unsigned)__popc(peers));
            }
        }
        __syncthreads();
        if (tid < 32) {                                     // lane handles 8 digits, descending
            unsigned c[8], tot = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = s_hist[255 - (lane * 8 + j)]; tot += c[j]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned y = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += y;
            }
            unsigned before = incl - tot;
            if (before < remaining && remaining <= incl) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (before < remaining && remaining <= before + c[j]) {
                        s_pick[0] = 255u - (unsigned)(lane * 8 + j);
                        s_pick[1] = remaining - before;
                    }
                    before += c[j];
                }
            }
        }
        __syncthreads();
        prefix |= s_pick[0] << shift;
        mask |= 255u << shift;
        remaining = s_pick[1];
        __syncthreads();
    }
    // everything with score word >= prefix: kLazyTarget - remaining strictly above + the whole tie group
    if (tid == 0) *s_count = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + tid;
        if (i < n && (unsigned)(__ldg(p.cand_key + lb + i) >> 32) >= prefix) {
            const int pos = atomicAdd(s_count, 1);
            if (pos < kSmallItems) s_sel[pos] = i;
        }
    }
    __syncthreads();
    const int c = *s_count;
    return c <= kSmallItems ? c : 0;
}

// Medium and long lists (n > kSmallItems).  No global sort: candidates are bucketed by class through a small
// shared-memory hash table (count -> exclusive scan -> scatter), ranked INSIDE their class by counting
// (sum_c n_c^2 comparisons instead of n log^2 n sort stages with a barrier each), suppressed per class by one
// warp, and only the survivors are sorted by score (bitonic) for the output order.  Arrays live in shared
// memory up to kSmemItems candidates, in the global workspace beyond.  Returns false when the list defeats the
// table (more than kHashSlots/2 distinct classes): the caller then takes the two-sort path (nms_big_body).
constexpr int kWarpSegment = 2048;        // class segments up to this length are suppressed by one warp, longer ones by the CTA
constexpr int kHashSlots = 1024;
constexpr unsigned kHashEmpty = 0xffffffffu;
constexpr size_t kMedItemBytes = 47;      // U_key 8 + F_key 8 + F_box 16 + U_slot 4 + F_slot 4 + F_area 4 + B_id 2 + F_dead 1
static_assert(kMedItemBytes <= kSmemItemBytes && kMedItemBytes <= kWsItemBytes, "long-list layouts must fit the shared/workspace strides");

struct MedArrays {
    unsigned long long *u_key;   // bucketed by class, unordered inside a bucket; later: survivors to sort
    unsigned long long *f_key;   // by q (class-major, score-descending inside a class)
    float4 *f_box;
    unsigned *u_slot, *f_slot;
    float *f_area;
    unsigned short *b_id;        // hash slot of candidate i
    unsigned char *f_dead;
};

__device__ __forceinline__ MedArrays carve_med(unsigned char *base, int n_al)
{
    MedArrays a;
    a.u_key = reinterpret_cast<unsigned long long *>(base);
    a.f_key = reinterpret_cast<unsigned long long *>(base + (size_t)n_al * 8);
    a.f_box = reinterpret_cast<float4 *>(base + (size_t)n_al * 16);
    a.u_slot = reinterpret_cast<unsigned *>(base + (size_t)n_al * 32);
    a.f_slot = reinterpret_cast<unsigned *>(base + (size_t)n_al * 36);
    a.f_area = reinterpret_cast<float *>(base + (size_t)n_al * 40);
    a.b_id = reinterpret_cast<unsigned short *>(base + (size_t)n_al * 44);
    a.f_dead = base + (size_t)n_al * 46;
    return a;
}

// SMEM: the arrays are in shared memory (tells the compiler the address space: generic loads from shared are
// several times slower than LDS and do not pipeline in the counting loops).
template <bool SMEM, int THREADS>
__device__ __forceinline__ bool nms_medium_body(const NmsParams &p, int n, int src0, unsigned char *base, int n_al,
                                                int *s_warp, unsigned *h_cls, int *h_cnt, int *h_start, ChunkScratch *chunk_scratch,
                                                int *n_kept_out)
{
    if (SMEM) __builtin_assume(__isShared(base));
    else __builtin_assume(__isGlobal(base));
    __builtin_assume(__isShared(h_cls));
    __builtin_assume(__isShared(h_cnt));
    __builtin_assume(__isShared(h_start));
    int &s_distinct = h_start[0];                    // scratch until the scan overwrites h_start
    const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int64_t lb = p.mode == 0 ? list_base(p, img) : 0;
    const MedArrays ar = carve_med(base, n_al);

    auto key_of = [&](int i) -> unsigned long long {
        if (p.mode == 0) return __ldg(p.cand_key + lb + i);
        return ((unsigned long long)f2ord_nms(__ldg(p.scores + src0 + i)) << 32) | (unsigned long long)(0xffffffffu - (unsigned)i);
    };
    auto cls_of = [&](int i) -> unsigned {
        return p.mode == 0 ? (unsigned)__ldg(p.cand_cls + lb + i) : (unsigned)__ldg(p.classes + src0 + i);
    };

    for (int h = tid; h < kHashSlots; h += blockDim.x) { h_cls[h] = kHashEmpty; h_cnt[h] = 0; }
    if (tid == 0) s_distinct = 0;
    __syncthreads();
    // 1. class -> hash slot, per-slot counts
    for (int i = tid; i < n; i += blockDim.x) {
        const unsigned c = cls_of(i);
        unsigned h = (c * 2654435761u) >> 22;                      // 10 bits
        for (int probe = 0; probe < kHashSlots; ++probe) {
            const unsigned prev = atomicCAS(&h_cls[h], kHashEmpty, c);
            if (prev == kHashEmpty) { atomicAdd(&s_distinct, 1); break; }
            if (prev == c) break;
            h = (h + 1) & (kHashSlots - 1);
        }
        ar.b_id[i] = (unsigned short)h;
        atomicAdd(&h_cnt[h], 1);
    }
    __syncthreads();
    if (s_distinct > kHashSlots / 2) return false;                // block-uniform
    // 2. exclusive scan of the slot counts (kSlotsPerThread consecutive slots per thread)
    {
        constexpr int kSlotsPerThread = kHashSlots / THREADS;
        static_assert(kSlotsPerThread * THREADS == kHashSlots, "hash slots split evenly over the threads");
        int cs[kSlotsPerThread], c = 0;
#pragma unroll
        for (int j = 0; j < kSlotsPerThread; ++j) { cs[j] = h_cnt[kSlotsPerThread * tid + j]; c += cs[j]; }
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(kFullMask, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int x = lane < nwarps ? s_warp[lane] : 0;
            int wi = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(kFullMask, wi, o);
                if (lane >= o) wi += y;
            }
            s_warp[lane] = wi - x;
        }
        __syncthreads();
        int run = s_warp[warp] + incl - c;
#pragma unroll
        for (int j = 0; j < kSlotsPerThread; ++j) {                 // h_cnt becomes the fill cursor
            h_start[kSlotsPerThread * tid + j] = run;
            h_cnt[kSlotsPerThread * tid + j] = 0;
            run += cs[j];
        }
    }
    __syncthreads();
    // 3. scatter (key, slot) into the class buckets
    for (int i = tid; i < n; i += blockDim.x) {
        const int h = ar.b_id[i];
        const int pos = h_start[h] + atomicAdd(&h_cnt[h], 1);
        ar.u_key[pos] = key_of(i);
        ar.u_slot[pos] = (unsigned)i;
    }
    __syncthreads();
    // 4. rank inside the bucket by counting -> class-major position q; gather the box
    for (int pp = tid; pp < n; pp += blockDim.x) {
        const unsigned long long key = ar.u_key[pp];
        const unsigned slot = ar.u_slot[pp];
        const int h = ar.b_id[slot];
        const int s0 = h_start[h], e0 = s0 + h_cnt[h];
        int rank = 0;
        if (p.mode == 0) {                                   // candidate lists: (==, earlier position), see nms_small_body
            for (int j = s0; j < e0; ++j) {
                const unsigned long long kj = ar.u_key[j];
                rank += kj > key || (kj == key && j < pp);
            }
        } else {                                             // batched_nms: the keys carry the box index, always distinct
            for (int j = s0; j < e0; ++j) rank += ar.u_key[j] > key;
        }
        const int q = s0 + rank;
        const float4 bx = p.mode == 0 ? __ldg(p.cand_box + lb + slot) : __ldg(p.boxes + src0 + slot);
        ar.f_key[q] = key;
        ar.f_slot[q] = slot;
        ar.f_box[q] = bx;
        ar.f_area[q] = (bx.z - bx.x) * (bx.w - bx.y);
        ar.f_dead[q] = 0;
    }
    __syncthreads();
    // 5. suppression inside each class.  Segments of up to 64 boxes: every box gets the bitmask of the earlier
    //    boxes of its class that overlap it (all pairs in parallel, u_key is free to hold the masks), then one
    //    lane per class runs the greedy chain on bits.  Longer segments: one warp per class, the kept box is
    //    broadcast and 32 later boxes are tested per step.
    unsigned long long *mask = ar.u_key;
    if (tid == 0) chunk_scratch->n_big = 0;                       // visible after the barrier below
    for (int q = tid; q < n; q += blockDim.x) {
        const int h = ar.b_id[ar.f_slot[q]];
        const int s0 = h_start[h], m = h_cnt[h];
        unsigned long long bits = 0ull;
        if (m <= 64) {
            const float4 bq = ar.f_box[q];
            const float aq = ar.f_area[q];
            for (int j = s0; j < q; ++j)
                if (iou_gt(ar.f_box[j], ar.f_area[j], bq, aq, p.iou_thr)) bits |= 1ull << (j - s0);
        }
        mask[q] = bits;
    }
    __syncthreads();
    for (int h = tid; h < kHashSlots; h += blockDim.x) {          // one lane per class: greedy on bits
        const int m = h_cnt[h];
        if (m > kWarpSegment) {                                    // rare: remember it for the CTA-wide pass below
            const int k = atomicAdd(&chunk_scratch->n_big, 1);
            if (k < 32) chunk_scratch->big[k] = h;
        }
        if (m < 2 || m > 64) continue;
        const int s0 = h_start[h];
        unsigned long long kept = 1ull;
        for (int i = 1; i < m; ++i) {
            if ((mask[s0 + i] & kept) == 0ull) kept |= 1ull << i;
            else ar.f_dead[s0 + i] = 1;
        }
    }
    for (int h = warp; h < kHashSlots; h += nwarps) {             // long segments: one warp each, 32-box chunks
        const int m = h_cnt[h];
        if (m <= 64 || m > kWarpSegment) continue;
        warp_segment_nms<SMEM>(ar.f_box, ar.f_area, ar.f_dead, h_start[h], m, p.iou_thr, lane);
    }
    __syncthreads();
    const int n_big = chunk_scratch->n_big;                       // very long segments: the whole CTA, one after another
    if (n_big > 0) {                                              // (block-uniform)
        if (n_big <= 32) {
            for (int k = 0; k < n_big; ++k) {
                const int h = chunk_scratch->big[k];               // (cta_segment_nms only touches box / area / kept)
                cta_segment_nms<SMEM>(ar.f_box, ar.f_area, ar.f_dead, h_start[h], h_cnt[h], p.iou_thr, chunk_scratch);
            }
        } else {
            for (int h = 0; h < kHashSlots; ++h)
                if (h_cnt[h] > kWarpSegment)
                    cta_segment_nms<SMEM>(ar.f_box, ar.f_area, ar.f_dead, h_start[h], h_cnt[h], p.iou_thr, chunk_scratch);
        }
    }
    // 6. survivors -> u_key/u_slot (ballot compaction), then ordered by (score desc, index asc) WITHOUT a sort:
    //    mode 0 needs the K best only -> radix select of the K-th score + rank-by-counting of the few above it;
    //    mode 1 needs all of them     -> rank-by-counting over the survivors (bitonic only beyond 4096 of them).
    //    (Barrier-heavy sorts are slow here: every __syncthreads drains the shared-memory stores of 32 warps.)
    const int n_kept = block_ordered_compact(
        n, s_warp, [&](int q) { return ar.f_dead[q] == 0; },
        [&](int q, int k) { ar.u_key[k] = ar.f_key[q]; ar.u_slot[k] = (unsigned)q; });
    __syncthreads();
    auto emit = [&](int k_src, int rank) {                       // survivor k_src goes to output position rank
        const unsigned q = ar.u_slot[k_src], slot = ar.f_slot[q];
        if (p.mode == 0) {
            const int64_t o = (int64_t)img * p.K + rank;
            p.out_scores[o] = __uint_as_float((unsigned)(ar.u_key[k_src] >> 32));
            p.out_classes[o] = (int64_t)h_cls[ar.b_id[slot]];
            p.out_boxes[o] = ar.f_box[q];
            if (p.out_keys != nullptr) p.out_keys[o] = ar.u_key[k_src];
        } else {
            p.keep[src0 + rank] = (int64_t)src0 + slot;
        }
    };
    const int want = p.mode == 0 ? (n_kept < p.K ? n_kept : p.K) : n_kept;
    if (p.mode == 1 && n_kept > 4096) {
        int np = 2;
        while (np < n_kept) np <<= 1;
        for (int k = n_kept + tid; k < np; k += blockDim.x) { ar.u_key[k] = 0ull; ar.u_slot[k] = 0u; }
        __syncthreads();
        bitonic_kv<true>(ar.u_key, ar.u_slot, np);
        for (int k = tid; k < n_kept; k += blockDim.x) emit(k, k);
    } else {
        // threshold: with more survivors than outputs, only keys >= the want-th largest score can be emitted
        unsigned thr_hi = 0u;                                    // compare on the score word
        if (n_kept > want) {
            unsigned *hist = reinterpret_cast<unsigned *>(h_cnt);    // 1024 ints of scratch, free by now
            unsigned prefix = 0, mask = 0, remaining = (unsigned)want;
            for (int pass = 0; pass < 4; ++pass) {
                const int shift = 24 - 8 * pass;
                for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
                __syncthreads();
                for (int k0 = 0; k0 < n_kept; k0 += blockDim.x) {
                    const int k = k0 + tid;
                    const bool ok = k < n_kept;
                    const unsigned u = ok ? (unsigned)(ar.u_key[k] >> 32) : 0u;
                    const bool in = ok && ((u & mask) == prefix);
                    const unsigned digit = (u >> shift) & 255u;
                    const unsigned act = __ballot_sync(kFullMask, in);
                    if (in) {
                        const unsigned peers = __match_any_sync(act, digit);
                        if (lane == __ffs(peers) - 1) atomicAdd(&hist[digit], (unsigned)__popc(peers));
                    }
                }
                __syncthreads();
                if (warp == 0) {
                    unsigned c[8], tot = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) { c[j] = hist[255 - (lane * 8 + j)]; tot += c[j]; }
                    unsigned incl = tot;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const unsigned y = __shfl_up_sync(kFullMask, incl, o);
                        if (lane >= o) incl += y;
                    }
                    unsigned before = incl - tot;
                    if (before < remaining && remaining <= incl) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            if (before < remaining && remaining <= before + c[j]) {
                                hist[256] = 255u - (unsigned)(lane * 8 + j);
                                hist[257] = remaining - before;
                            }
                            before += c[j];
                        }
                    }
                }
                __syncthreads();
                prefix |= hist[256] << shift;
                mask |= 255u << shift;
                remaining = hist[257];
                __syncthreads();
            }
            thr_hi = prefix;
        }
        // rank-by-counting among the survivors that can make it (all of them when n_kept == want).  They are
        // compacted first (f_key is free by now) so that a few full warps do the counting instead of one lane
        // in every warp, and they only need to be ranked among themselves: everything else is smaller.
        unsigned long long *pass_key = ar.f_key;
        unsigned *pass_src = reinterpret_cast<unsigned *>(ar.f_area);
        __syncthreads();
        const int n_pass = block_ordered_compact(
            n_kept, s_warp, [&](int k) { return (unsigned)(ar.u_key[k] >> 32) >= thr_hi; },
            [&](int k, int r) { pass_key[r] = ar.u_key[k]; pass_src[r] = (unsigned)k; });
        __syncthreads();
        for (int r = tid; r < n_pass; r += blockDim.x) {
            const unsigned long long key = pass_key[r];
            int rank = 0;
            if (p.mode == 0) {
                for (int j = 0; j < n_pass; ++j) rank += pass_key[j] > key || (pass_key[j] == key && j < r);
            } else {
                for (int j = 0; j < n_pass; ++j) rank += pass_key[j] > key;
            }
            if (rank < want) emit((int)pass_src[r], rank);
        }
    }
    *n_kept_out = n_kept;
    return true;
}

// One launch for every path: the list length (known only on the device) picks the body.
template <int THREADS>   // <= 64 registers per thread either way: 512 threads take half the register file
__global__ void __launch_bounds__(THREADS, 1024 / THREADS) k_nms(NmsParams p)
{
    extern __shared__ __align__(16) unsigned char s_dyn_top[];
    __shared__ int s_warp_top[33];
    __shared__ unsigned s_hcls[kHashSlots];
    __shared__ int s_hcnt[kHashSlots], s_hstart[kHashSlots];
    __shared__ ChunkScratch s_chunk;
    int n, src0;
    if (p.mode == 0) {
        const int c = __ldg(p.cand_count + blockIdx.x);
        n = (int)(c < p.cap ? c : p.cap);
        src0 = 0;
    } else {
        src0 = __ldg(p.seg_offsets + blockIdx.x);
        n = __ldg(p.seg_offsets + blockIdx.x + 1) - src0;
    }
    if (n <= kSmallItems) { nms_small_body<THREADS>(p); return; }
    if (p.mode == 0 && p.K <= kLazyMaxK) {
        // top-K of a long list: try the highest-ranked ~200 candidates first (exact: see the file header)
        __shared__ int s_sel[kSmallItems];
        __shared__ unsigned s_pick[2];
        __shared__ int s_count;
        const int64_t lb = list_base(p, (int)blockIdx.x);
        const int m = lazy_prefix_select(p, lb, n, s_sel, reinterpret_cast<unsigned *>(s_hcnt), s_pick, &s_count);
        if (m > 0) {
            const int kept = nms_small_body<THREADS>(p, s_sel, m, false);
            if (kept >= p.K) {                             // the K best survivors are all inside the prefix: done
                if (threadIdx.x == 0) {
                    p.num_instances[blockIdx.x] = p.K;
                    if (p.reset_counts) const_cast<int32_t *>(p.cand_count)[blockIdx.x] = 0;
                }
                return;
            }
            __syncthreads();                               // fewer than K survived: the full list decides
        }
    }
    int n_al = 2;
    while (n_al < n) n_al <<= 1;
    int n_kept = 0;
    bool done;
    if (n_al <= p.smem_items) {
        done = nms_medium_body<true, THREADS>(p, n, src0, s_dyn_top, n_al, s_warp_top, s_hcls, s_hcnt, s_hstart, &s_chunk, &n_kept);
    } else {
        unsigned char *ws = list_workspace(p, (int)blockIdx.x, src0);
        done = nms_medium_body<false, THREADS>(p, n, src0, ws, n_al, s_warp_top, s_hcls, s_hcnt, s_hstart, &s_chunk, &n_kept);
    }
    if (done) {
        const int img = blockIdx.x, tid = threadIdx.x;
        if (p.mode == 0) {
            const int m = n_kept < p.K ? n_kept : p.K;
            if (tid == 0) {
                p.num_instances[img] = m;
                if (p.reset_counts) const_cast<int32_t *>(p.cand_count)[img] = 0;
            }
            for (int k = m + tid; k < p.K; k += blockDim.x) {
                const int64_t o = (int64_t)img * p.K + k;
                p.out_scores[o] = 0.f;
                p.out_classes[o] = 0;
                p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        } else if (tid == 0) {
            p.keep_count[img] = n_kept;
        }
        return;
    }
    __syncthreads();
    nms_big_body(p);
}

// ---------------------------------------------------------------------------
// Class-split NMS for long lists (mode 0).  Suppression never crosses classes, so an image's candidates can be
// dealt to S independent sub-lists by class (hash % S) and every sub-list handled by its own CTA — S SMs per image
// instead of one, and sub-lists short enough to stay in shared memory.  k_nms runs unchanged on the B*S sub-lists
// (each yields its K best survivors, sorted, with their keys); k_nms_merge then picks the image's K best of the
// S*K by rank = position in the own list + number of larger keys in every other list (binary search).
// ---------------------------------------------------------------------------
constexpr int kMaxSplit = 64;

__device__ __forceinline__ int sub_list_of(unsigned cls, int S) { return (int)(((cls * 2654435761u) >> 16) % (unsigned)S); }

struct SplitParams {
    int32_t *cand_count; int64_t cap;
    const unsigned long long *key; const float4 *box; const int32_t *cls;
    int S; int32_t *sub_count; int32_t *sub_offset;          // [B*S]
    unsigned long long *key2; float4 *box2; int32_t *cls2;     // [B*cap] re-bucketed copies
    int reset_counts;
};

__global__ void __launch_bounds__(1024) k_nms_split_lists(SplitParams p)
{
    __shared__ int s_cnt[kMaxSplit], s_start[kMaxSplit], s_cur[kMaxSplit];
    const int img = blockIdx.x, tid = threadIdx.x, S = p.S;
    const int c = __ldg(p.cand_count + img);
    const int n = (int)(c < p.cap ? c : p.cap);
    const int64_t lb = (int64_t)img * p.cap;
    if (tid < kMaxSplit) { s_cnt[tid] = 0; s_cur[tid] = 0; }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) atomicAdd(&s_cnt[sub_list_of((unsigned)__ldg(p.cls + lb + i), S)], 1);
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int s = 0; s < S; ++s) { s_start[s] = run; run += s_cnt[s]; }
    }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        const int cl = __ldg(p.cls + lb + i);
        const int s = sub_list_of((unsigned)cl, S);
        const int64_t dst = lb + s_start[s] + atomicAdd(&s_cur[s], 1);     // order inside a sub-list is irrelevant: keys carry it
        p.key2[dst] = __ldg(p.key + lb + i);
        p.box2[dst] = __ldg(p.box + lb + i);
        p.cls2[dst] = cl;
    }
    if (tid < S) {
        p.sub_count[img * S + tid] = s_cnt[tid];
        p.sub_offset[img * S + tid] = (int32_t)(lb + s_start[tid]);
    }
    if (tid == 0 && p.reset_counts) p.cand_count[img] = 0;
}

struct MergeParams {
    int S, K;
    const int64_t *sub_num; const unsigned long long *sub_keys; const float *sub_scores; const int64_t *sub_classes;
    const float4 *sub_boxes;                                   // [B*S] / [B*S, K]
    int64_t *num_instances; float *out_scores; int64_t *out_classes; float4 *out_boxes;
};

// STAGED: the S*K keys of the image are copied to shared memory first (the binary searches are chains of dependent
// loads: ~20 cycles each from shared memory, ~700 from L2).
template <bool STAGED>
__global__ void __launch_bounds__(512) k_nms_merge(MergeParams p)
{
    extern __shared__ __align__(16) unsigned char s_merge[];
    __shared__ int s_num[kMaxSplit];
    const int img = blockIdx.x, tid = threadIdx.x, S = p.S, K = p.K;
    if (tid < S) s_num[tid] = (int)__ldg(p.sub_num + img * S + tid);
    __syncthreads();
    const unsigned long long *keys = p.sub_keys + (int64_t)img * S * K;
    if (STAGED) {
        unsigned long long *sk = reinterpret_cast<unsigned long long *>(s_merge);
        for (int e = tid; e < S * K; e += blockDim.x) {
            const int s = e / K, k = e - s * K;
            if (k < s_num[s]) sk[e] = __ldg(keys + e);
        }
        __syncthreads();
        keys = sk;
    }
    int total = 0;
    for (int s = 0; s < S; ++s) total += s_num[s];
    const int m = total < K ? total : K;
    for (int e = tid; e < S * K; e += blockDim.x) {
        const int s = e / K, k = e - s * K;
        if (k >= s_num[s]) continue;
        const unsigned long long key = keys[e];
        int rank = k;                                          // the own list is sorted descending
        for (int t = 0; t < S && rank < K; ++t) {
            if (t == s) continue;
            const unsigned long long *other = keys + t * K;
            int lo = 0, hi = s_num[t];                         // number of keys of list t that are larger than key
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (other[mid] > key) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < K) {
            const int64_t src = ((int64_t)img * S + s) * K + k;
            const int64_t o = (int64_t)img * K + rank;
            p.out_scores[o] = __ldg(p.sub_scores + src);
            p.out_classes[o] = __ldg(p.sub_classes + src);
            p.out_boxes[o] = __ldg(p.sub_boxes + src);
        }
    }
    if (tid == 0) p.num_instances[img] = m;
    for (int k = m + tid; k < K; k += blockDim.x) {
        const int64_t o = (int64_t)img * K + k;
        p.out_scores[o] = 0.f;
        p.out_classes[o] = 0;
        p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

static int pow2ceil(int64_t n)
{
    int p = 2;
    while (p < n) p <<= 1;
    return p;
}

// smem_items: candidates per list whose long-list arrays the launch keeps in dynamic shared memory (0: none, every long
// list uses the workspace).  Dynamic shared memory is reserved only when a list can exceed the short-list path.
template <int THREADS>
static int launch_nms(NmsParams p, int n_images, int64_t max_items, cudaStream_t st, int smem_items)
{
    p.smem_items = smem_items;
    const size_t smem = max_items > kSmallItems ? (size_t)smem_items * kSmemItemBytes : 0;
    static thread_local bool attr_set = false;
    if (smem && !attr_set) {
        int rc = cuda_status(cudaFuncSetAttribute(k_nms<THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                  (int)((size_t)kSmemItems * kSmemItemBytes)),
                             "cudaFuncSetAttribute(k_nms)");
        if (rc) return rc;
        attr_set = true;
    }
    k_nms<THREADS><<<n_images, THREADS, smem, st>>>(p);
    SIHL_CHECK_LAUNCH("k_nms");
    return SIHL_OD_OK;
}

}  // namespace sihl

using namespace sihl;

extern "C" size_t sihl_od_nms_workspace_bytes(int batch, int64_t cand_capacity)
{
    if (batch <= 0 || cand_capacity <= 0) return 0;
    const int np = pow2ceil(cand_capacity);
    if (np <= kSmallItems) return 0;                           // every list fits the short-list body
    return (size_t)batch * (size_t)np * kWsItemBytes;
}

extern "C" int sihl_od_nms_topk(const int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                                const float *cand_box, const int32_t *cand_cls, int batch, float iou_thr, int k,
                                int64_t *num_instances, float *scores, int64_t *classes, float *boxes, void *workspace,
                                int reset_counts, void *stream)
{
    SIHL_CHECK_ARG(cand_count && cand_key && cand_box && cand_cls, "NULL input");
    SIHL_CHECK_ARG(num_instances && scores && classes && boxes, "NULL output");
    SIHL_CHECK_ARG(cand_capacity >= 1 && cand_capacity < (1ll << 30) && k >= 1, "bad sizes");
    SIHL_CHECK_ARG(workspace != nullptr || sihl_od_nms_workspace_bytes(batch, cand_capacity) == 0,
                   "workspace needed for capacity %lld", (long long)cand_capacity);
    if (batch <= 0) return SIHL_OD_OK;
    NmsParams p = {};
    p.cand_count = cand_count; p.cap = cand_capacity;
    p.cand_key = reinterpret_cast<const unsigned long long *>(cand_key);
    p.cand_box = reinterpret_cast<const float4 *>(cand_box); p.cand_cls = cand_cls;
    p.mode = 0; p.iou_thr = iou_thr; p.K = k; p.reset_counts = reset_counts;
    p.num_instances = num_instances; p.out_scores = scores; p.out_classes = classes;
    p.out_boxes = reinterpret_cast<float4 *>(boxes);
    p.workspace = static_cast<unsigned char *>(workspace);
    p.ws_stride = (size_t)pow2ceil(cand_capacity) * kWsItemBytes;
    // runs next to the dense scan of the neighbouring steps: no dynamic shared memory (see the file header)
    return launch_nms<kNmsThreadsTopk>(p, batch, cand_capacity, (cudaStream_t)stream, 0);
}

namespace sihl {                 // od_nms_wide.cu: the multi-CTA bitmask path for one long list
size_t wide_nms_workspace_bytes(int64_t n);
bool wide_nms_applies(int64_t n);
int launch_wide_batched_nms(const float *boxes, const float *scores, const int64_t *classes, const int32_t *seg_offsets,
                            int n_images, int64_t n, float iou_thr, int64_t *keep, int32_t *keep_count, void *workspace,
                            cudaStream_t st);
}

extern "C" size_t sihl_od_batched_nms_workspace_bytes(int64_t n)
{
    if (wide_nms_applies(n)) return wide_nms_workspace_bytes(n);
    if (n <= kSmemItems) return 0;
    return (size_t)(2 * n + 2) * kWsItemBytes;
}

extern "C" int sihl_od_batched_nms(const float *boxes, const float *scores, const int64_t *classes,
                                   const int32_t *seg_offsets, int n_images, int64_t n, float iou_thr, int64_t *keep,
                                   int32_t *keep_count, void *workspace, void *stream)
{
    SIHL_CHECK_ARG(seg_offsets && keep_count, "NULL argument");
    SIHL_CHECK_ARG(n >= 0 && n < (1ll << 30) && n_images >= 0, "bad sizes");
    SIHL_CHECK_ARG(n == 0 || (boxes && scores && classes && keep), "NULL argument");
    SIHL_CHECK_ARG(workspace != nullptr || sihl_od_batched_nms_workspace_bytes(n) == 0, "workspace needed for n=%lld",
                   (long long)n);
    if (n_images == 0) return SIHL_OD_OK;
    if (wide_nms_applies(n))        // 8192..90000 boxes: bitmask-parallel suppression over all SMs (od_nms_wide.cu)
        return launch_wide_batched_nms(boxes, scores, classes, seg_offsets, n_images, n, iou_thr, keep, keep_count, workspace,
                                       (cudaStream_t)stream);
    NmsParams p = {};
    p.boxes = reinterpret_cast<const float4 *>(boxes); p.scores = scores; p.classes = classes; p.seg_offsets = seg_offsets;
    p.mode = 1; p.iou_thr = iou_thr; p.keep = keep; p.keep_count = keep_count;
    p.workspace = static_cast<unsigned char *>(workspace); p.ws_stride = 0;
    return launch_nms<kNmsThreadsAlone>(p, n_images, n, (cudaStream_t)stream, kSmemItems);
}

// ---- class-split variant (long lists) ------------------------------------------------------------------
static int split_factor(int64_t cand_capacity)
{
    int64_t s = (cand_capacity + 2047) / 2048;                 // sub-lists of ~2k candidates at a full list
    if (s < 2) s = 2;
    if (s > 32) s = 32;
    return (int)s;
}

static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

extern "C" size_t sihl_od_nms_split_workspace_bytes(int batch, int64_t cand_capacity, int k)
{
    if (batch <= 0 || cand_capacity <= 0 || k <= 0) return 0;
    const size_t S = (size_t)split_factor(cand_capacity), B = (size_t)batch, cap = (size_t)cand_capacity, K = (size_t)k;
    size_t bytes = 0;
    bytes += align256(B * cap * 8) + align256(B * cap * 16) + align256(B * cap * 4);          // key2, box2, cls2
    bytes += 2 * align256(B * S * 4);                                                         // sub_count, sub_offset
    bytes += align256(B * S * 8) + align256(B * S * K * 8) + align256(B * S * K * 4) + align256(B * S * K * 8) +
             align256(B * S * K * 16);                                                        // per-sub-list outputs
    bytes += align256((size_t)(2 * B * cap + 2) * kWsItemBytes);                              // k_nms workspace for long sub-lists
    return bytes;
}

extern "C" int sihl_od_nms_topk_split(int32_t *cand_count, int64_t cand_capacity, const uint64_t *cand_key,
                                      const float *cand_box, const int32_t *cand_cls, int batch, float iou_thr, int k,
                                      int64_t *num_instances, float *scores, int64_t *classes, float *boxes, void *workspace,
                                      int reset_counts, void *stream)
{
    SIHL_CHECK_ARG(cand_count && cand_key && cand_box && cand_cls, "NULL input");
    SIHL_CHECK_ARG(num_instances && scores && classes && boxes && workspace, "NULL output / workspace");
    SIHL_CHECK_ARG(cand_capacity >= 1 && (int64_t)batch * cand_capacity < (1ll << 30) && k >= 1 && k <= 4096, "bad sizes");
    if (batch <= 0) return SIHL_OD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int S = split_factor(cand_capacity);
    const size_t B = (size_t)batch, cap = (size_t)cand_capacity, K = (size_t)k;
    unsigned char *w = static_cast<unsigned char *>(workspace);
    auto take = [&](size_t bytes) { unsigned char *ptr = w; w += align256(bytes); return ptr; };
    SplitParams sp;
    sp.cand_count = cand_count; sp.cap = cand_capacity;
    sp.key = reinterpret_cast<const unsigned long long *>(cand_key); sp.box = reinterpret_cast<const float4 *>(cand_box);
    sp.cls = cand_cls; sp.S = S; sp.reset_counts = reset_counts;
    sp.key2 = reinterpret_cast<unsigned long long *>(take(B * cap * 8));
    sp.box2 = reinterpret_cast<float4 *>(take(B * cap * 16));
    sp.cls2 = reinterpret_cast<int32_t *>(take(B * cap * 4));
    sp.sub_count = reinterpret_cast<int32_t *>(take(B * S * 4));
    sp.sub_offset = reinterpret_cast<int32_t *>(take(B * S * 4));
    int64_t *sub_num = reinterpret_cast<int64_t *>(take(B * S * 8));
    unsigned long long *sub_keys = reinterpret_cast<unsigned long long *>(take(B * S * K * 8));
    float *sub_scores = reinterpret_cast<float *>(take(B * S * K * 4));
    int64_t *sub_classes = reinterpret_cast<int64_t *>(take(B * S * K * 8));
    float4 *sub_boxes = reinterpret_cast<float4 *>(take(B * S * K * 16));
    unsigned char *nms_ws = take((size_t)(2 * B * cap + 2) * kWsItemBytes);
    k_nms_split_lists<<<batch, 1024, 0, st>>>(sp);
    SIHL_CHECK_LAUNCH("k_nms_split_lists");
    NmsParams p = {};
    p.cand_count = sp.sub_count; p.cap = cand_capacity; p.list_offsets = sp.sub_offset;
    p.cand_key = sp.key2; p.cand_box = sp.box2; p.cand_cls = sp.cls2;
    p.mode = 0; p.iou_thr = iou_thr; p.K = k; p.reset_counts = 0;
    p.num_instances = sub_num; p.out_scores = sub_scores; p.out_classes = sub_classes; p.out_boxes = sub_boxes;
    p.out_keys = sub_keys; p.workspace = nms_ws; p.ws_stride = 0;
    // sub-lists rarely exceed 2048 candidates: half the shared memory per CTA lets two of them share an SM
    int rc = launch_nms<kNmsThreadsAlone>(p, batch * S, cand_capacity, st, kSmemItems / 2);
    if (rc) return rc;
    MergeParams mp;
    mp.S = S; mp.K = k; mp.sub_num = sub_num; mp.sub_keys = sub_keys; mp.sub_scores = sub_scores; mp.sub_classes = sub_classes;
    mp.sub_boxes = sub_boxes; mp.num_instances = num_instances; mp.out_scores = scores; mp.out_classes = classes;
    mp.out_boxes = reinterpret_cast<float4 *>(boxes);
    const size_t stage = (size_t)S * K * 8;
    if (stage <= 96 * 1024) {
        static thread_local bool merge_attr = false;
        if (!merge_attr) {
            rc = cuda_status(cudaFuncSetAttribute(k_nms_merge<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024),
                             "cudaFuncSetAttribute(k_nms_merge)");
            if (rc) return rc;
            merge_attr = true;
        }
        k_nms_merge<true><<<batch, 512, stage, st>>>(mp);
    } else {
        k_nms_merge<false><<<batch, 512, 0, st>>>(mp);
    }
    SIHL_CHECK_LAUNCH("k_nms_merge");
    return SIHL_OD_OK;
}
