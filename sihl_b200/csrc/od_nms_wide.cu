// od_nms_wide.cu — class-aware greedy NMS for LONG lists on the whole GPU (SURVEY.md §8 a15; extension).
//
// od_nms.cu handles a segment (image) with one CTA: right for the few hundred candidates of the steady-state
// step, wrong for a single list of tens of thousands of boxes (30 000 boxes of one class took 92 ms on one SM
// while torchvision's CUDA op needs 16 ms on the whole GPU).  This path spreads the same exact semantics —
// torchvision's per-class greedy rule, visit order (score desc, index asc), keep test
// inter / (area_i + area_j - inter) > thr with IEEE division — over all SMs in five steps:
//
//   k_wide_count    all pairs of a segment, tiled 256 x 4096 over the grid: per item its position q in the order
//                   (class asc, score desc, index asc), its score rank r, the start / length of its class segment
//                   (rank by counting: no sort, no barrier chain; 4 integer comparisons per pair)
//   k_wide_scatter  items -> class-major order; k_wide_rowoff: exclusive scan of the mask-row lengths
//   k_wide_mask     bitmask-parallel IoU (k_wide_mask_diou: the DIoU test of DIoU-NMS): 64 x 64 tiles (row tile, column tile >= row tile) WITHIN class segments
//                   only; word w of row q holds the later same-class boxes of tile (first tile of the class + w)
//                   that q would suppress
//   k_wide_reduce   the serial greedy pass on mask words: one CTA per class segment, 64 rows per step — the
//                   in-tile chain runs on one 64-bit word in registers, the kept rows are OR-ed into the
//                   "removed" bitmap of the later tiles by the whole CTA (coalesced word loads)
//   k_wide_emit     survivors in (score desc, index asc) order per segment (ordered compaction by score rank)
//
// Memory: the mask needs sum_c n_c * (n_c / 64 + 2) words, bounded by N^2/64 + 3N for N items; the entry point
// takes this path for 8192 <= N <= 90 000 (1 GiB of mask at most) and the one-CTA-per-segment kernel otherwise.
//
// The quadrilateral NMS (sihl_od_batched_quad_nms, end of this file) runs the same pipeline for every N up to 90 000,
// with its own scatter (hulls) and mask (convex-hull IoU) kernels.
#include "od_common.cuh"

namespace sihl {

constexpr int kWideITile = 256;            // items per CTA of k_wide_count
constexpr int kWideJSlab = 4096;           // partner items per CTA of k_wide_count
constexpr int kWideColsPerCta = 8;         // column tiles per CTA of k_wide_mask
constexpr int kWideMaxWords = 1536;        // mask words per row the reduce kernel can hold (>= 90000 / 64 + 2)

struct WideBuffers {
    int *cnt_q, *cnt_r, *cnt_cs, *cnt_len;                 // [N] pair counters (zeroed)
    unsigned long long *akey;                              // [N] (class << 32 | ~ord(score)) by item
    int *seg_of;                                           // [N] segment of the item
    float4 *sbox; float *sarea; int *scs, *sce, *sidx, *sr;   // [N] by q: box, area, class-segment [start, end), item, score rank
    long long *rowoff;                                     // [N+1] first mask word of row q
    unsigned char *kept, *flag_by_r; int *idx_by_r;        // [N]
    unsigned long long *mask;                              // mask words
    size_t mask_words;
    size_t bytes;
};

static WideBuffers carve_wide(void *base, int64_t n)
{
    WideBuffers w;
    unsigned char *b = reinterpret_cast<unsigned char *>(base);
    size_t o = 0;
    const size_t N = (size_t)n;
    auto take = [&](size_t bytes) { unsigned char *ptr = b + o; o += round_up_256(bytes); return ptr; };
    w.cnt_q = reinterpret_cast<int *>(take(4 * N * 4));   // the four counter arrays are contiguous: one memset
    w.cnt_r = w.cnt_q + N; w.cnt_cs = w.cnt_r + N; w.cnt_len = w.cnt_cs + N;
    w.akey = reinterpret_cast<unsigned long long *>(take(N * 8));
    w.seg_of = reinterpret_cast<int *>(take(N * 4));
    w.sbox = reinterpret_cast<float4 *>(take(N * 16));
    w.sarea = reinterpret_cast<float *>(take(N * 4));
    w.scs = reinterpret_cast<int *>(take(N * 4));
    w.sce = reinterpret_cast<int *>(take(N * 4));
    w.sidx = reinterpret_cast<int *>(take(N * 4));
    w.sr = reinterpret_cast<int *>(take(N * 4));
    w.rowoff = reinterpret_cast<long long *>(take((N + 1) * 8));
    w.kept = take(N);
    w.flag_by_r = take(N);
    w.idx_by_r = reinterpret_cast<int *>(take(N * 4));
    w.mask_words = N * (N / 64 + 3);
    w.mask = reinterpret_cast<unsigned long long *>(take(w.mask_words * 8));
    w.bytes = o;
    return w;
}

size_t wide_nms_workspace_bytes(int64_t n) { return carve_wide(nullptr, n).bytes; }

bool wide_nms_applies(int64_t n) { return n >= 8192 && n <= 90000; }

// per item: sort key and segment
__global__ void __launch_bounds__(256)
k_wide_keys(const float *__restrict__ scores, const int64_t *__restrict__ classes, const int32_t *__restrict__ seg_offsets,
            int n_segments, int n, unsigned long long *__restrict__ akey, int *__restrict__ seg_of)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int lo = 0, hi = n_segments;                           // largest s with seg_offsets[s] <= i
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(seg_offsets + mid) <= i) lo = mid; else hi = mid;
    }
    seg_of[i] = lo;
    akey[i] = ((unsigned long long)(unsigned)__ldg(classes + i) << 32) | (unsigned long long)(~f2ord(__ldg(scores + i)));
}

// Rank by counting over all pairs of a segment.  CTA (x, y): items [256x, 256x+256) against the y-th slab of 4096
// partners of the union of their segments.  "j before i" in class-major order <=> (akey_j, j) < (akey_i, i).
__global__ void __launch_bounds__(kWideITile)
k_wide_count(const unsigned long long *__restrict__ akey, const int *__restrict__ seg_of,
             const int32_t *__restrict__ seg_offsets, int n, int *__restrict__ cnt_q, int *__restrict__ cnt_r,
             int *__restrict__ cnt_cs, int *__restrict__ cnt_len)
{
    __shared__ unsigned long long s_key[kWideITile];
    __shared__ int s_lo, s_hi;
    const int i = blockIdx.x * kWideITile + threadIdx.x;
    const bool have = i < n;
    int my_lo = 0, my_hi = 0;
    unsigned long long ki = 0ull;
    if (have) {
        const int s = __ldg(seg_of + i);
        my_lo = __ldg(seg_offsets + s); my_hi = __ldg(seg_offsets + s + 1);
        ki = __ldg(akey + i);
    }
    if (threadIdx.x == 0) {                                // items are ordered by segment: first / last item bound the union
        const int first = blockIdx.x * kWideITile, last = min(n, first + kWideITile) - 1;
        s_lo = __ldg(seg_offsets + __ldg(seg_of + first));
        s_hi = __ldg(seg_offsets + __ldg(seg_of + last) + 1);
    }
    __syncthreads();
    const int j0 = s_lo + (int)blockIdx.y * kWideJSlab;
    const int j1 = min(s_hi, j0 + kWideJSlab);
    if (j0 >= j1) return;                                  // block-uniform
    const unsigned ci = (unsigned)(ki >> 32), si = (unsigned)ki;
    int q = 0, r = 0, cs = 0, len = 0;
    for (int jb = j0; jb < j1; jb += kWideITile) {
        const int j = jb + threadIdx.x;
        __syncthreads();
        s_key[threadIdx.x] = j < j1 ? __ldg(akey + j) : 0ull;
        __syncthreads();
        const int cnt = min(kWideITile, j1 - jb);
        if (have) {
            // partners outside the item's own segment do not count (the tile may straddle segments)
            const int a = max(jb, my_lo) - jb, b = min(jb + cnt, my_hi) - jb;
#pragma unroll 4
            for (int t = a; t < b; ++t) {
                const unsigned long long kj = s_key[t];
                const int jj = jb + t;
                const unsigned cj = (unsigned)(kj >> 32), sj = (unsigned)kj;
                const bool first = jj < i;
                q += (kj < ki) || (kj == ki && first);
                r += (sj < si) || (sj == si && first);
                cs += cj < ci;
                len += cj == ci;
            }
        }
    }
    if (have) {
        if (q) atomicAdd(cnt_q + i, q);
        if (r) atomicAdd(cnt_r + i, r);
        if (cs) atomicAdd(cnt_cs + i, cs);
        if (len) atomicAdd(cnt_len + i, len);
    }
}

__global__ void __launch_bounds__(256)
k_wide_scatter(const float4 *__restrict__ boxes, const int *__restrict__ seg_of, const int32_t *__restrict__ seg_offsets, int n,
               WideBuffers w)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s0 = __ldg(seg_offsets + __ldg(seg_of + i));
    const int q = s0 + w.cnt_q[i];
    const float4 b = __ldg(boxes + i);
    const int cs = s0 + w.cnt_cs[i];
    w.sbox[q] = b;
    w.sarea[q] = (b.z - b.x) * (b.w - b.y);
    w.scs[q] = cs;
    w.sce[q] = cs + w.cnt_len[i];
    w.sidx[q] = i;
    w.sr[q] = s0 + w.cnt_r[i];
    w.kept[q] = 0;
}

// words per mask row of a class segment [cs, ce): one per 64-aligned tile it touches
__device__ __forceinline__ int class_words(int cs, int ce) { return ((ce - 1) >> 6) - (cs >> 6) + 1; }

// rowoff[q] = sum_{q' < q} words(q'): single CTA, 1024 threads, sequential chunks with a carried prefix.
__global__ void __launch_bounds__(1024) k_wide_rowoff(const int *__restrict__ scs, const int *__restrict__ sce, int n,
                                                      long long *__restrict__ rowoff)
{
    __shared__ long long s_warp[33];
    __shared__ long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int q = base + tid;
        const long long x = q < n ? (long long)class_words(__ldg(scs + q), __ldg(sce + q)) : 0;
        long long incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(kFullMask, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            long long v = s_warp[lane], inc2 = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(kFullMask, inc2, o);
                if (lane >= o) inc2 += y;
            }
            s_warp[lane] = inc2 - v;
            if (lane == 31) s_warp[32] = inc2;
        }
        __syncthreads();
        const long long carry = s_carry;
        if (q < n) rowoff[q] = carry + s_warp[warp] + incl - x;
        __syncthreads();
        if (tid == 0) s_carry = carry + s_warp[32];
        __syncthreads();
    }
    if (tid == 0) rowoff[n] = s_carry;
}

// CTA (R, y): row tile R (rows q = 64R + t, one per thread) against the column tiles Cg = R + 8y .. R + 8y + 7.
// Row q writes word (Cg - cs(q)/64) for every Cg from its own tile to the last tile of its class segment — every
// word of the mask is written exactly once (zero where nothing overlaps), so the mask needs no memset.
// t = threadIdx.x, read by the kernel, where the launch bound tells the compiler that t < 64.
template <int KIND>
__device__ __forceinline__ void wide_mask(WideBuffers w, int n, float thr, int t)
{
    __shared__ float4 s_box[64];
    __shared__ float s_area[64];
    __shared__ int s_cs[64];
    __shared__ int s_last;
    const int R = blockIdx.x;
    const int q = R * 64 + t;
    const bool have = q < n;
    int cs = 0, ce = 0;
    float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
    float aq = 0.f;
    long long off = 0;
    if (have) { cs = w.scs[q]; ce = w.sce[q]; bq = w.sbox[q]; aq = w.sarea[q]; off = w.rowoff[q]; }
    if (t == 0) s_last = 0;
    __syncthreads();
    if (have) atomicMax(&s_last, (ce - 1) >> 6);           // last column tile any row of this tile needs
    __syncthreads();
    const int c_first = R + (int)blockIdx.y * kWideColsPerCta;
    const int c_end = min(s_last, c_first + kWideColsPerCta - 1);
    for (int Cg = c_first; Cg <= c_end; ++Cg) {            // block-uniform bounds
        const int qc = Cg * 64 + t;
        __syncthreads();
        if (qc < n) { s_box[t] = w.sbox[qc]; s_area[t] = w.sarea[qc]; s_cs[t] = w.scs[qc]; }
        else s_cs[t] = -1;
        __syncthreads();
        if (!have || Cg > ((ce - 1) >> 6)) continue;       // past this row's class segment
        unsigned long long word = 0ull;
        const int b0 = Cg == R ? t + 1 : 0;                // only later boxes (q' > q)
        for (int b = b0; b < 64; ++b)
            if (s_cs[b] == cs && overlap_gt<KIND>(bq, aq, s_box[b], s_area[b], thr)) word |= 1ull << b;
        w.mask[off + (Cg - (cs >> 6))] = word;
    }
}

// the mask of greedy NMS (torchvision's IoU test) and of DIoU-NMS; every other step serves both
__global__ void __launch_bounds__(64) k_wide_mask(WideBuffers w, int n, float thr) { wide_mask<kIoU>(w, n, thr, threadIdx.x); }
__global__ void __launch_bounds__(64) k_wide_mask_diou(WideBuffers w, int n, float thr) { wide_mask<kDIoU>(w, n, thr, threadIdx.x); }

// One CTA per 64-tile of the class-major order; it serves every class segment that STARTS in its tile.
constexpr int kReduceThreads = 512;
__global__ void __launch_bounds__(kReduceThreads) k_wide_reduce(WideBuffers w, int n)
{
    __shared__ unsigned long long s_rem[kWideMaxWords];
    __shared__ unsigned long long s_diag[64];
    __shared__ long long s_off[64], s_kept_off[64];
    __shared__ unsigned long long s_kept;
    __shared__ int s_nkept;
    const int tid = threadIdx.x, tile = blockIdx.x;
    for (int lead = tile * 64; lead < min(n, tile * 64 + 64);) {
        const int cs = w.scs[lead];
        const int ce = w.sce[lead];
        if (cs != lead) { lead = ce; continue; }           // a class that started in an earlier tile: skip to its end
        const int W = class_words(cs, ce);
        const int g0 = cs >> 6;
        if (ce - cs == 1) {                                // a class of one box: kept
            if (tid == 0) w.kept[cs] = 1;
            lead = ce;
            continue;
        }
        for (int x = tid; x < W; x += kReduceThreads) s_rem[x] = 0ull;
        __syncthreads();
        for (int x = 0; x < W; ++x) {
            const int qa = max(cs, (g0 + x) * 64), qb = min(ce, (g0 + x) * 64 + 64);   // this class's rows in tile g0+x
            if (tid < 64) {
                const int qq = (g0 + x) * 64 + tid;
                const bool mine = qq >= qa && qq < qb;
                const long long off = mine ? w.rowoff[qq] : 0;
                s_off[tid] = off;
                s_diag[tid] = mine ? w.mask[off + x] : 0ull;
            }
            __syncthreads();
            if (tid == 0) {                                // the greedy chain of the tile, on bits
                unsigned long long cur = s_rem[x], kept = 0ull;
                int nk = 0;
                for (int b = qa - (g0 + x) * 64; b < qb - (g0 + x) * 64; ++b) {
                    if (!((cur >> b) & 1ull)) {
                        kept |= 1ull << b;
                        cur |= s_diag[b];
                        s_kept_off[nk++] = s_off[b];
                    }
                }
                s_kept = kept;
                s_nkept = nk;
            }
            __syncthreads();
            const unsigned long long kept = s_kept;
            const int nk = s_nkept;
            if (tid < 64 && ((kept >> tid) & 1ull)) w.kept[(g0 + x) * 64 + tid] = 1;
            // the kept rows suppress in the later tiles: thread per later word, loop over the kept rows
            for (int x2 = x + 1 + tid; x2 < W; x2 += kReduceThreads) {
                unsigned long long acc = 0ull;
                for (int k = 0; k < nk; ++k) acc |= w.mask[s_kept_off[k] + x2];
                s_rem[x2] |= acc;
            }
            __syncthreads();
        }
        lead = ce;
    }
}

__global__ void __launch_bounds__(256) k_wide_by_rank(WideBuffers w, int n)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const int r = w.sr[q];
    w.flag_by_r[r] = w.kept[q];
    w.idx_by_r[r] = w.sidx[q];
}

// One CTA per segment: ordered compaction of the survivors by score rank.
__global__ void __launch_bounds__(1024)
k_wide_emit(WideBuffers w, const int32_t *__restrict__ seg_offsets, int64_t *__restrict__ keep, int32_t *__restrict__ keep_count)
{
    __shared__ int s_warp[33];
    const int seg = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s0 = __ldg(seg_offsets + seg), s1 = __ldg(seg_offsets + seg + 1);
    int running = 0;
    for (int base = s0; base < s1; base += 1024) {
        const int r = base + tid;
        const bool f = r < s1 && w.flag_by_r[r] != 0;
        const unsigned m = __ballot_sync(kFullMask, f);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        if (warp == 0) {
            const int x = s_warp[lane];
            int incl = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += y;
            }
            s_warp[lane] = incl - x;
            if (lane == 31) s_warp[32] = incl;
        }
        __syncthreads();
        if (f) keep[s0 + running + s_warp[warp] + __popc(m & ((1u << lane) - 1u))] = (int64_t)w.idx_by_r[r];
        running += s_warp[32];
        __syncthreads();
    }
    if (tid == 0) keep_count[seg] = running;
}

// ---- quadrilateral NMS (sihl_od_batched_quad_nms): the same pipeline, with the hull overlap of od_math.h ---------------
// k_wide_scatter_quad writes the AABB into sbox, the hull area into sarea and the hull vertices into squad (two float4
// per item, class-major); k_wide_mask_quad tests the AABBs first and clips the hulls only for pairs whose AABBs overlap.
// Every other step is the box path's kernel.  The quad array is a separate argument: WideBuffers keeps its layout.
constexpr int kWideQuad = 2;                  // launch_wide_batched_nms's kind for quads (kIoU / kDIoU are the boxes')
constexpr int64_t kQuadNmsMax = 90000;        // the mask takes up to N^2/64 words: 1 GiB at this size

static size_t quad_nms_workspace_bytes(int64_t n)
{
    return n == 0 ? 0 : carve_wide(nullptr, n).bytes + round_up_256((size_t)n * 2 * sizeof(float4));
}

__global__ void __launch_bounds__(256)
k_wide_scatter_quad(const float *__restrict__ quads, const int *__restrict__ seg_of, const int32_t *__restrict__ seg_offsets,
                    int n, WideBuffers w, float4 *__restrict__ squad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s0 = __ldg(seg_offsets + __ldg(seg_of + i));
    const int q = s0 + w.cnt_q[i];
    float p[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) p[k] = __ldg(quads + (size_t)8 * i + k);
    const QuadHull h = quad_hull(p);
    const int cs = s0 + w.cnt_cs[i];
    w.sbox[q] = make_float4(h.x1, h.y1, h.x2, h.y2);
    w.sarea[q] = h.area;
    squad[2 * q] = make_float4(h.x[0], h.y[0], h.x[1], h.y[1]);
    squad[2 * q + 1] = make_float4(h.x[2], h.y[2], h.x[3], h.y[3]);
    w.scs[q] = cs;
    w.sce[q] = cs + w.cnt_len[i];
    w.sidx[q] = i;
    w.sr[q] = s0 + w.cnt_r[i];
    w.kept[q] = 0;
}

__device__ __forceinline__ QuadHull load_hull(float4 box, float area, float4 v0, float4 v1)
{
    QuadHull h;
    h.x[0] = v0.x; h.y[0] = v0.y; h.x[1] = v0.z; h.y[1] = v0.w;
    h.x[2] = v1.x; h.y[2] = v1.y; h.x[3] = v1.z; h.y[3] = v1.w;
    h.area = area;
    h.x1 = box.x; h.y1 = box.y; h.x2 = box.z; h.y2 = box.w;
    return h;
}

// wide_mask's tiling and word layout; the test of a pair is quad_iou_hulls(q, later) > thr, where AABBs that do not
// overlap (zero width included) give IoU 0 without a clip
__global__ void __launch_bounds__(64) k_wide_mask_quad(WideBuffers w, const float4 *__restrict__ squad, int n, float thr)
{
    __shared__ float4 s_box[64], s_v0[64], s_v1[64];
    __shared__ float s_area[64];
    __shared__ int s_cs[64];
    __shared__ int s_last;
    const int t = threadIdx.x;
    const int R = blockIdx.x;
    const int q = R * 64 + t;
    const bool have = q < n;
    const bool apart_hits = 0.f > thr;
    int cs = 0, ce = 0;
    long long off = 0;
    QuadHull hq = load_hull(make_float4(0.f, 0.f, 0.f, 0.f), 0.f, make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f));
    if (have) {
        cs = w.scs[q]; ce = w.sce[q]; off = w.rowoff[q];
        hq = load_hull(w.sbox[q], w.sarea[q], squad[2 * q], squad[2 * q + 1]);
    }
    if (t == 0) s_last = 0;
    __syncthreads();
    if (have) atomicMax(&s_last, (ce - 1) >> 6);
    __syncthreads();
    const int c_first = R + (int)blockIdx.y * kWideColsPerCta;
    const int c_end = min(s_last, c_first + kWideColsPerCta - 1);
    for (int Cg = c_first; Cg <= c_end; ++Cg) {            // block-uniform bounds
        const int qc = Cg * 64 + t;
        __syncthreads();
        if (qc < n) {
            s_box[t] = w.sbox[qc]; s_area[t] = w.sarea[qc]; s_cs[t] = w.scs[qc];
            s_v0[t] = squad[2 * qc]; s_v1[t] = squad[2 * qc + 1];
        } else {
            s_cs[t] = -1;
        }
        __syncthreads();
        if (!have || Cg > ((ce - 1) >> 6)) continue;       // past this row's class segment
        unsigned long long word = 0ull;
        const int b0 = Cg == R ? t + 1 : 0;                // only later quads (q' > q)
        for (int b = b0; b < 64; ++b) {
            if (s_cs[b] != cs) continue;
            const float4 bb = s_box[b];
            const bool apart = !(fminf(hq.x2, bb.z) > fmaxf(hq.x1, bb.x)) || !(fminf(hq.y2, bb.w) > fmaxf(hq.y1, bb.y));
            const bool hit = apart ? apart_hits : quad_iou_hulls(hq, load_hull(bb, s_area[b], s_v0[b], s_v1[b])) > thr;
            if (hit) word |= 1ull << b;
        }
        w.mask[off + (Cg - (cs >> 6))] = word;
    }
}

// sihl_od_quad_iou: one thread per pair
__global__ void __launch_bounds__(256)
k_quad_iou(const float *__restrict__ a, int64_t na, const float *__restrict__ b, int64_t nb, float *__restrict__ out)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= na * nb) return;
    const int64_t i = k / nb, j = k - i * nb;
    float pa[8], pb[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { pa[c] = __ldg(a + 8 * i + c); pb[c] = __ldg(b + 8 * j + c); }
    out[k] = quad_iou(pa, pb);
}

// kind: kIoU / kDIoU (boxes [N, 4]) or kWideQuad (quads [N, 8]: needs quad_nms_workspace_bytes(n), of which the first
// carve_wide(n).bytes are the box path's buffers)
int launch_wide_batched_nms(const float *boxes, const float *scores, const int64_t *classes, const int32_t *seg_offsets,
                            int n_images, int64_t n64, int kind, float iou_thr, int64_t *keep, int32_t *keep_count,
                            void *workspace, cudaStream_t st)
{
    const int n = (int)n64;
    WideBuffers w = carve_wide(workspace, n64);
    float4 *squad = reinterpret_cast<float4 *>(static_cast<unsigned char *>(workspace) + w.bytes);
    int rc = cuda_status(cudaMemsetAsync(w.cnt_q, 0, (size_t)4 * n * sizeof(int), st), "cudaMemsetAsync(wide counters)");
    if (rc) return rc;
    const int nb = (n + 255) / 256;
    k_wide_keys<<<nb, 256, 0, st>>>(scores, classes, seg_offsets, n_images, n, w.akey, w.seg_of);
    SIHL_CHECK_LAUNCH("k_wide_keys");
    const dim3 cgrid((unsigned)((n + kWideITile - 1) / kWideITile), (unsigned)((n + kWideJSlab - 1) / kWideJSlab));
    k_wide_count<<<cgrid, kWideITile, 0, st>>>(w.akey, w.seg_of, seg_offsets, n, w.cnt_q, w.cnt_r, w.cnt_cs, w.cnt_len);
    SIHL_CHECK_LAUNCH("k_wide_count");
    if (kind == kWideQuad) k_wide_scatter_quad<<<nb, 256, 0, st>>>(boxes, w.seg_of, seg_offsets, n, w, squad);
    else k_wide_scatter<<<nb, 256, 0, st>>>(reinterpret_cast<const float4 *>(boxes), w.seg_of, seg_offsets, n, w);
    SIHL_CHECK_LAUNCH("k_wide_scatter");
    k_wide_rowoff<<<1, 1024, 0, st>>>(w.scs, w.sce, n, w.rowoff);
    SIHL_CHECK_LAUNCH("k_wide_rowoff");
    const int tiles = (n + 63) / 64;
    const dim3 mgrid((unsigned)tiles, (unsigned)((tiles + kWideColsPerCta - 1) / kWideColsPerCta));
    if (kind == kWideQuad) k_wide_mask_quad<<<mgrid, 64, 0, st>>>(w, squad, n, iou_thr);
    else if (kind == kDIoU) k_wide_mask_diou<<<mgrid, 64, 0, st>>>(w, n, iou_thr);
    else k_wide_mask<<<mgrid, 64, 0, st>>>(w, n, iou_thr);
    SIHL_CHECK_LAUNCH("k_wide_mask");
    k_wide_reduce<<<tiles, kReduceThreads, 0, st>>>(w, n);
    SIHL_CHECK_LAUNCH("k_wide_reduce");
    k_wide_by_rank<<<nb, 256, 0, st>>>(w, n);
    SIHL_CHECK_LAUNCH("k_wide_by_rank");
    k_wide_emit<<<n_images, 1024, 0, st>>>(w, seg_offsets, keep, keep_count);
    SIHL_CHECK_LAUNCH("k_wide_emit");
    return SIHL_OD_OK;
}

}  // namespace sihl

using namespace sihl;

extern "C" size_t sihl_od_batched_quad_nms_workspace_bytes(int64_t n)
{
    return n >= 0 && n <= kQuadNmsMax ? quad_nms_workspace_bytes(n) : 0;
}

extern "C" int sihl_od_batched_quad_nms(const float *quads, const float *scores, const int64_t *classes,
                                        const int32_t *seg_offsets, int n_images, int64_t n, float iou_thr, int64_t *keep,
                                        int32_t *keep_count, void *workspace, void *stream)
{
    SIHL_CHECK_ARG(seg_offsets && keep_count, "NULL argument");
    SIHL_CHECK_ARG(n >= 0 && n_images >= 0, "bad sizes");
    SIHL_CHECK_ARG(n <= kQuadNmsMax, "n=%lld quads: sihl_od_batched_quad_nms takes at most %lld", (long long)n,
                   (long long)kQuadNmsMax);
    SIHL_CHECK_ARG(n == 0 || (quads && scores && classes && keep), "NULL argument");
    SIHL_CHECK_ARG(workspace != nullptr || n == 0, "workspace needed for n=%lld", (long long)n);
    if (n_images == 0) return SIHL_OD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0)
        return cuda_status(cudaMemsetAsync(keep_count, 0, (size_t)n_images * sizeof(int32_t), st), "cudaMemsetAsync(keep_count)");
    return launch_wide_batched_nms(quads, scores, classes, seg_offsets, n_images, n, kWideQuad, iou_thr, keep, keep_count,
                                   workspace, st);
}

extern "C" int sihl_od_quad_iou(const float *a, int64_t na, const float *b, int64_t nb, float *out, void *stream)
{
    SIHL_CHECK_ARG(na >= 0 && nb >= 0 && na < (1ll << 31) && nb < (1ll << 31), "bad sizes");
    SIHL_CHECK_ARG(na * nb <= (1ll << 38), "na * nb = %lld pairs: at most 2^38", (long long)(na * nb));
    if (na == 0 || nb == 0) return SIHL_OD_OK;
    SIHL_CHECK_ARG(a && b && out, "NULL argument");
    const int64_t blocks = (na * nb + 255) / 256;
    k_quad_iou<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, na, b, nb, out);
    SIHL_CHECK_LAUNCH("k_quad_iou");
    return SIHL_OD_OK;
}
