// od_infer.cu — inference tail of the detection head (SURVEY.md §8 a11 + the dense
// decode half of the a15 extension).
//
//   k_topk          ref object_detection.py:108-109  torch.topk(loc_logits, K, dim=1)
//   k_decode_rows   ref :113-121                     sigmoid / count / argmax / box decode on K rows
//   k_dense_decode* extension: the same per-location decode over ALL locations of the
//                   dense maps + score threshold, feeding class-aware NMS (od_nms.cu).
//                   This is the HBM-bound kernel of the path: 4*A*(C+5) B per image are read
//                   exactly once.  Three variants, picked by sihl_od_dense_decode():
//                     _tma  C % 4 == 0, C <= 128: TMA bulk copies into a shared-memory ring
//                     _v4   C % 4 == 0, larger C: 16-byte loads, 4 or 32 lanes per row
//                     plain any C: 4-byte loads, 8 lanes per row
#include <type_traits>

#include "od_common.cuh"

namespace sihl {

// Order-preserving map fp32 -> uint32 (ascending).
__device__ __forceinline__ unsigned f2ord(float f)
{
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// ---------------------------------------------------------------------------
// top-K of one row per CTA: 4-pass MSB radix select for the K-th largest value, one
// ordered pass that takes everything above it plus the lowest-index elements equal to
// it, then a bitonic sort of the K winners by (value desc, index asc).
// ---------------------------------------------------------------------------
constexpr int kTopkThreads = 1024;
constexpr int kTopkMaxK = 1024;

template <typename T>     // element type of the location map (upcast on load; half values are exact in fp32)
__global__ void __launch_bounds__(kTopkThreads)
k_topk(const T *__restrict__ loc, int A, int K, int KP /* pow2 >= K */, int64_t *__restrict__ idx_out,
       float *__restrict__ val_out)
{
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_pick[2];               // [0] = digit, [1] = remaining
    __shared__ int s_warp[33];
    __shared__ unsigned long long s_sel[kTopkMaxK];
    __shared__ int s_ngt;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const T *row = loc + (int64_t)blockIdx.x * A;

    unsigned prefix = 0, mask = 0, remaining = (unsigned)K;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0;
        __syncthreads();
        for (int i0 = 0; i0 < A; i0 += blockDim.x) {
            const int i = i0 + tid;
            const bool ok = i < A;
            const unsigned u = ok ? f2ord(ldf(row + i)) : 0u;
            const bool in = ok && ((u & mask) == prefix);
            const unsigned digit = (u >> shift) & 255u;
            // warp-aggregated histogram update (logits cluster in a few exponent buckets)
            const unsigned act = __ballot_sync(kFullMask, in);
            if (in) {
                const unsigned peers = __match_any_sync(act, digit);
                if (lane == __ffs(peers) - 1) atomicAdd(&s_hist[digit], (unsigned)__popc(peers));
            }
        }
        __syncthreads();
        if (warp == 0) {
            // lane handles 8 digits, descending: digit = 255 - (lane*8 + j)
            unsigned c[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = s_hist[255 - (lane * 8 + j)]; tot += c[j]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned y = __shfl_up_sync(kFullMask, incl, o);
                if (lane >= o) incl += y;
            }
            unsigned before = incl - tot;          // elements in strictly larger digits handled by lower lanes
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
    const unsigned kth = prefix;                 // ord-key of the K-th largest value
    const int need_eq = (int)remaining;          // how many elements equal to it are taken (lowest index first)
    if (tid == 0) s_ngt = 0;
    for (int i = tid; i < KP; i += blockDim.x) s_sel[i] = 0ull;
    __syncthreads();

    int eq_seen = 0;                             // block-uniform running count of equal elements
    for (int i0 = 0; i0 < A; i0 += blockDim.x) {
        const int i = i0 + tid;
        const unsigned u = (i < A) ? f2ord(ldf(row + i)) : 0u;
        const bool gt = (i < A) && u > kth, eq = (i < A) && u == kth;
        const unsigned long long key = ((unsigned long long)u << 32) | (unsigned long long)(0xffffffffu - (unsigned)i);
        if (gt) s_sel[atomicAdd(&s_ngt, 1)] = key;           // fewer than K of these by construction
        // ordered rank among the equal elements
        const unsigned beq = __ballot_sync(kFullMask, eq);
        if (lane == 0) s_warp[warp] = __popc(beq);
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
        if (eq) {
            const int r = eq_seen + s_warp[warp] + __popc(beq & ((1u << lane) - 1u));
            if (r < need_eq) s_sel[K - need_eq + r] = key;   // slots [K-need_eq, K) are reserved for the ties
        }
        eq_seen += s_warp[32];
        __syncthreads();
    }

    // bitonic sort, descending, of KP (>= K) composite keys; the zero padding sinks to the end
    for (int k = 2; k <= KP; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < KP; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = s_sel[i], b = s_sel[ixj];
                    const bool desc = (i & k) == 0;
                    if (desc ? (a < b) : (a > b)) { s_sel[i] = b; s_sel[ixj] = a; }
                }
            }
            __syncthreads();
        }
    for (int i = tid; i < K; i += blockDim.x) {
        const unsigned long long key = s_sel[i];
        idx_out[(int64_t)blockIdx.x * K + i] = (int64_t)(0xffffffffu - (unsigned)(key & 0xffffffffu));
        val_out[(int64_t)blockIdx.x * K + i] = ord2f((unsigned)(key >> 32));
    }
}

// ---------------------------------------------------------------------------
// First arg-max over a row of C logits by a group of 8 lanes (4 rows per warp).
// Lane gl visits c = gl, gl+8, ...; strict '>' keeps the lowest index inside a lane and
// the cross-lane reduction prefers the lower index on equal values (torch.max, ref :117).
// ---------------------------------------------------------------------------
template <int CPL>   // logits per lane when C == 8*CPL (fully unrolled, all loads in flight); 0 = runtime C
__device__ __forceinline__ int row_argmax8(const float *__restrict__ z, int C, int gl)
{
    float best = -CUDART_INF_F;
    int arg = 0x7fffffff;
    if (CPL > 0) {
        float v[CPL > 0 ? CPL : 1];
#pragma unroll
        for (int i = 0; i < CPL; ++i) v[i] = __ldcs(z + gl + 8 * i);      // streamed once: evict-first
#pragma unroll
        for (int i = 0; i < CPL; ++i)
            if (v[i] > best || arg == 0x7fffffff) { best = v[i]; arg = gl + 8 * i; }
    } else {
        for (int c = gl; c < C; c += 8) {
            const float x = __ldcs(z + c);
            if (x > best || arg == 0x7fffffff) { best = x; arg = c; }
        }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(kFullMask, best, o);
        const int oa = __shfl_xor_sync(kFullMask, arg, o);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    return arg;
}

// The same first arg-max on a row of element type T (half maps: 2-byte loads, upcast in registers).
template <typename T>
__device__ __forceinline__ int row_argmax8_t(const T *__restrict__ z, int C, int gl)
{
    float best = -CUDART_INF_F;
    int arg = 0x7fffffff;
    for (int c = gl; c < C; c += 8) {
        const float x = ldf(z + c);
        if (x > best || arg == 0x7fffffff) { best = x; arg = c; }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(kFullMask, best, o);
        const int oa = __shfl_xor_sync(kFullMask, arg, o);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    return arg;
}

// ref :113-121 on the K gathered rows of one image per CTA.  For half maps the reference's `.sigmoid()` and `.exp()`
// run in the map dtype (evaluated in fp32, rounded to half): round_to<T> reproduces that, so scores, the
// `scores > 0.5` count and the decoded boxes follow the reference under autocast too.
template <typename T>
__global__ void __launch_bounds__(256)
k_decode_rows(const float *__restrict__ top_logits, const int64_t *__restrict__ idx, int K,
              const T *__restrict__ cls_rows, int C, const T *__restrict__ box_rows,
              const float4 *__restrict__ offsets, const float4 *__restrict__ scales, float img_w, float img_h,
              int64_t *__restrict__ num_instances, float *__restrict__ scores, int64_t *__restrict__ classes,
              float *__restrict__ boxes)
{
    __shared__ int s_count;
    const int b = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_count = 0;
    __syncthreads();
    int local = 0;
    for (int k = tid; k < K; k += blockDim.x) {
        const int64_t r = (int64_t)b * K + k;
        const float s = round_to<T>(sigmoid_f(__ldg(top_logits + r)));     // ref :113
        scores[r] = s;
        local += (s > 0.5f) ? 1 : 0;                                       // ref :114
        const int a = (int)__ldg(idx + r);
        const float4 raw = ldf4(box_rows + 4 * r), off = __ldg(offsets + a), sc = __ldg(scales + a);
        *reinterpret_cast<float4 *>(boxes + 4 * r) =                       // ref :121
            make_float4((off.x + sc.x * round_to<T>(expf(raw.x))) * img_w, (off.y + sc.y * round_to<T>(expf(raw.y))) * img_h,
                        (off.z + sc.z * round_to<T>(expf(raw.z))) * img_w, (off.w + sc.w * round_to<T>(expf(raw.w))) * img_h);
    }
    local = warp_sum(local);
    if ((tid & 31) == 0 && local) atomicAdd(&s_count, local);
    const int gl = tid & 7, grp = tid >> 3, ngrp = blockDim.x >> 3;
    for (int k0 = 0; k0 < K; k0 += ngrp) {
        const int k = k0 + grp;
        const int64_t r = (int64_t)b * K + (k < K ? k : K - 1);
        const int arg = row_argmax8_t<T>(cls_rows + r * C, C, gl);         // ref :117
        if (k < K && gl == 0) classes[r] = arg;
    }
    __syncthreads();
    if (tid == 0) num_instances[b] = s_count;
}

// ---------------------------------------------------------------------------
// Dense decode (extension).  Grid-stride over rows (= locations of the whole batch),
// 8 lanes per row.  Candidates (sigmoid(loc) > thr) are appended to the image's list.
// ---------------------------------------------------------------------------
struct DenseDecodeParams {
    const float *loc; const float *cls; const float *box_raw;
    int batch, A, C;
    const float4 *offsets; const float4 *scales; float img_w, img_h, score_thr;
    float logit_thr;        // a logit below this cannot pass (conservative pre-filter; the sigmoid test decides)
    int32_t *cand_count; int64_t cap;
    unsigned long long *cand_key; float4 *cand_box; int32_t *cand_cls;
};

// Candidate test and append for one decoded location (one lane per row).
__device__ __forceinline__ void emit_candidate(const DenseDecodeParams &p, int64_t row, float x, int arg)
{
    const float s = sigmoid_f(x);
    if (!(s > p.score_thr)) return;
    const int b = (int)(row / p.A), a = (int)(row - (int64_t)b * p.A);
    const int slot = atomicAdd(p.cand_count + b, 1);
    if (slot >= p.cap) return;
    const float4 raw = __ldcs(reinterpret_cast<const float4 *>(p.box_raw) + row);
    const float4 off = __ldg(p.offsets + a), sc = __ldg(p.scales + a);
    const int64_t o = (int64_t)b * p.cap + slot;
    p.cand_key[o] = ((unsigned long long)__float_as_uint(s) << 32) | (unsigned long long)(0xffffffffu - (unsigned)a);
    p.cand_box[o] = make_float4(decode_norm(off.x, sc.x, raw.x) * p.img_w, decode_norm(off.y, sc.y, raw.y) * p.img_h,
                                decode_norm(off.z, sc.z, raw.z) * p.img_w, decode_norm(off.w, sc.w, raw.w) * p.img_h);
    p.cand_cls[o] = arg;
}

// Scalar variant (any C): 8 lanes per row, 4-byte loads.
template <int CPL>
__global__ void __launch_bounds__(256) k_dense_decode(DenseDecodeParams p)
{
    const int gl = threadIdx.x & 7;
    const int64_t rows = (int64_t)p.batch * p.A;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) >> 3;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const int64_t rounds = (rows + ngrp - 1) / ngrp;
    for (int64_t it = 0; it < rounds; ++it) {
        const int64_t row = it * ngrp + grp;
        const bool ok = row < rows;
        const int64_t rr = ok ? row : rows - 1;
        const float x = __ldcs(p.loc + rr);
        const int arg = row_argmax8<CPL>(p.cls + rr * p.C, p.C, gl);
        if (ok && gl == 0) emit_candidate(p, row, x, arg);
    }
}

// Vector variant (C % 4 == 0): LPR lanes per row, VPL 16-byte loads per lane and row, two rows
// per group and iteration, i.e. 2*VPL independent LDG.128 in flight per lane before the first
// use — enough bytes in flight (~160 B/lane) to cover HBM latency at 4 CTAs/SM.
// Lane gl owns float4 indices gl, gl+LPR, ...: ascending class index inside the lane, so a
// strict '>' keeps the first maximum; the cross-lane step prefers the lower index on ties.
template <int LPR, int VPL, bool EXACT>
__global__ void __launch_bounds__(256) k_dense_decode_v4(DenseDecodeParams p)
{
    const int gl = threadIdx.x & (LPR - 1);
    const int C4 = p.C >> 2;
    const int64_t rows = (int64_t)p.batch * p.A;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const float4 *cls4 = reinterpret_cast<const float4 *>(p.cls);
    for (int64_t row0 = grp; row0 < rows; row0 += 2 * ngrp) {       // rows is warp-uniform-safe: see clamp below
        const int64_t rowA = row0, rowB = row0 + ngrp;
        const bool okB = rowB < rows;
        const int64_t rb = okB ? rowB : rowA;
        float4 va[VPL], vb[VPL];
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            const int v = gl + LPR * i;
            const bool in = EXACT || v < C4;
            va[i] = in ? __ldcs(cls4 + rowA * C4 + v) : make_float4(0.f, 0.f, 0.f, 0.f);
            vb[i] = in ? __ldcs(cls4 + rb * C4 + v) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        const float xa = __ldcs(p.loc + rowA), xb = __ldcs(p.loc + rb);
        float bestA = -CUDART_INF_F, bestB = -CUDART_INF_F;
        int argA = 0x7fffffff, argB = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            const int v = gl + LPR * i;
            if (EXACT || v < C4) {
                const int c = 4 * v;
                const float ea[4] = {va[i].x, va[i].y, va[i].z, va[i].w};
                const float eb[4] = {vb[i].x, vb[i].y, vb[i].z, vb[i].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (ea[e] > bestA || argA == 0x7fffffff) { bestA = ea[e]; argA = c + e; }
                    if (eb[e] > bestB || argB == 0x7fffffff) { bestB = eb[e]; argB = c + e; }
                }
            }
        }
#pragma unroll
        for (int o = LPR >> 1; o > 0; o >>= 1) {
            const float oa = __shfl_xor_sync(kFullMask, bestA, o), ob = __shfl_xor_sync(kFullMask, bestB, o);
            const int ia = __shfl_xor_sync(kFullMask, argA, o), ib = __shfl_xor_sync(kFullMask, argB, o);
            if (oa > bestA || (oa == bestA && ia < argA)) { bestA = oa; argA = ia; }
            if (ob > bestB || (ob == bestB && ib < argB)) { bestB = ob; argB = ib; }
        }
        if (gl == 0) emit_candidate(p, rowA, xa, argA);
        if (gl == (LPR > 1 ? 1 : 0) && okB) emit_candidate(p, rowB, xb, argB);
    }
}

// ---------------------------------------------------------------------------
// Bulk-async variant (C % 4 == 0, C <= 128): the class-logit map is streamed through shared
// memory by the TMA unit — cp.async.bulk of 64 consecutive rows (64*C*4 B, contiguous in
// HBM) + their 64 location logits per stage, completion signalled on an mbarrier — in a
// ring of kStages stages per CTA, persistent CTAs striding over the chunks.  Bytes in flight
// are set by the ring (2 CTAs x 4 stages x 20 KB per SM at C = 80), not by what the compiler
// keeps in registers, and every byte is read from HBM exactly once.  Consumers: 4 lanes per
// row, conflict-free LDS.128, first-argmax as above.
// ---------------------------------------------------------------------------
constexpr int kChunkRows = 64;             // rows per ring stage of the default variant == rows one pass of a 256-thread CTA covers
                                           // (4 lanes per row); small scans use 32-row stages on 128-thread CTAs (see the entry point)

__device__ __forceinline__ uint32_t smem_u32(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Streamed exactly once: tag the lines evict-first so the scan does not push the L2-resident working set of the
// concurrently running kernels (anchor tables, selections, candidate and positive lists) out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Candidates found while streaming are only *staged* in shared memory (row, logit, class, raw
// box): the global atomic that allocates the output slot and the dependent stores would put a
// ~2 us round trip on the critical path of every 64-row chunk.  The stage list is flushed by
// the whole CTA, all candidates in parallel, when it runs full and at the end.
constexpr int kStageCap = 256;

struct StagedCand {
    int row_lo, row_hi;      // 64-bit row index
    float x;
    int arg;
};

// One warp turns up to 32 staged entries (one per lane) into candidates: no block-level synchronisation inside.  Entries
// passed the conservative logit pre-filter only; the exact test sigmoid(x) > thr (ref :113) is made here.
// `entry`: this lane's staged entry or nullptr; all 32 lanes of the warp must call.
// Programmatic dependent launch (sm_90+): the scan only READS the maps until its first flush, so a launch made with
// cudaLaunchAttributeProgrammaticStreamSerialization may start streaming while the previous kernel of the stream (the
// NMS of the lane's previous step, or the previous scan in a back-to-back loop) is still draining; everything that
// touches the candidate lists / counters waits for that kernel first.  Both instructions are no-ops in a normal launch,
// which is how the scan is launched: the overlap was measured and does not shorten the pipelined step (DESIGN.md).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_prior_grids() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename T = float>
__device__ __forceinline__ void flush_staged(const DenseDecodeParams &p, const StagedCand *entry)
{
    pdl_wait_prior_grids();
    const int lane = threadIdx.x & 31;
    const bool small = (int64_t)p.batch * p.A < (1ll << 31);
    __syncwarp();
    {
        StagedCand c;
        c.row_lo = c.row_hi = c.arg = 0; c.x = 0.f;
        if (entry != nullptr) c = *entry;
        const float s = entry != nullptr ? round_to<T>(sigmoid_f(c.x)) : 0.f;
        const bool have = entry != nullptr && s > p.score_thr;
        const int64_t row = have ? (((int64_t)c.row_hi << 32) | (unsigned)c.row_lo) : 0;
        const int b = small ? (int)((unsigned)row / (unsigned)p.A) : (int)(row / p.A);
        const int a = (int)(row - (int64_t)b * p.A);
        // everything that does not depend on the output slot first: the raw box is only needed for candidates (2 % of
        // the locations at cfg1; its line was prefetched into L2 when the candidate was staged), and the decode
        // arithmetic runs while the slot atomic below is in flight — at the end of the kernel this chain is the tail
        float4 raw = make_float4(0.f, 0.f, 0.f, 0.f), off = raw, sc = raw;
        if (have) {
            if constexpr (sizeof(T) == 4) raw = __ldcs(reinterpret_cast<const float4 *>(p.box_raw) + row);
            else raw = ldf4(reinterpret_cast<const T *>(p.box_raw) + 4 * row);
            off = __ldg(p.offsets + a);
            sc = __ldg(p.scales + a);
        }
        // one returning atomic per (warp, image) instead of one per candidate: neighbours in the list come from
        // the same 64-row chunk, i.e. almost always the same image (same-address atomics serialise in L2)
        const unsigned act = __ballot_sync(kFullMask, have);
        int slot = 0;
        if (have) {
            const unsigned peers = __match_any_sync(act, b);
            const int leader = __ffs(peers) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(p.cand_count + b, __popc(peers));
            base = __shfl_sync(peers, base, leader);
            slot = base + __popc(peers & ((1u << lane) - 1u));
        }
        const float4 box = make_float4((off.x + sc.x * round_to<T>(expf(raw.x))) * p.img_w, (off.y + sc.y * round_to<T>(expf(raw.y))) * p.img_h,
                                       (off.z + sc.z * round_to<T>(expf(raw.z))) * p.img_w, (off.w + sc.w * round_to<T>(expf(raw.w))) * p.img_h);
        if (have && slot < p.cap) {
            const int64_t o = (int64_t)b * p.cap + slot;
            p.cand_key[o] = ((unsigned long long)__float_as_uint(s) << 32) | (unsigned long long)(0xffffffffu - (unsigned)a);
            p.cand_box[o] = box;
            p.cand_cls[o] = c.arg;
        }
    }
    __syncwarp();
}

// T: element type of the three maps.  Half maps put ROWS x C x 2 bytes into a stage (half the HBM traffic); a lane then
// owns 16-byte vectors of EIGHT logits (VPL counts those).
template <int VPL, bool EXACT, int ROWS = kChunkRows, typename T = float>     // ROWS per stage; the CTA has 4 * ROWS threads
__global__ void __launch_bounds__(4 * ROWS) k_dense_decode_tma(DenseDecodeParams p, int stages, int n_chunks)
{
    constexpr int kPerVec = 16 / (int)sizeof(T);
    constexpr int kWarps = 4 * ROWS / 32;
    extern __shared__ __align__(128) unsigned char s_ring[];
    __shared__ StagedCand s_list[kWarps * 32];                    // one 32-entry segment per warp: no atomics to append
    __shared__ int s_seg_count[kWarps];
    static_assert(kStageCap == 256 && kWarps <= 8, "at most 8 warps x 32 staged candidates");
    const int tid = threadIdx.x, gl = tid & 3, r = tid >> 2, lane = tid & 31, warp = tid >> 5;
    int n_staged = 0;                                             // this warp's segment fill (warp-uniform)
    const int C4 = p.C / kPerVec;                                  // 16-byte vectors per row
    const int64_t rows = (int64_t)p.batch * p.A;
    // per stage: 64 rows of class logits — ONE bulk copy per stage.  The location logit of a row is a 4-byte
    // coalesced load one chunk ahead (one lane per row), the raw box is read for candidates only (flush_staged):
    // small bulk copies cost the TMA unit as much as big ones (measured with tools/micro/read_bw.cu: a ring of
    // single 21 KB copies reaches the 6.3 TB/s read ceiling, the former 3-copy stage did not).
    const uint32_t stage_bytes = (uint32_t)ROWS * (uint32_t)p.C * (uint32_t)sizeof(T);
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_ring + (size_t)stages * stage_bytes);

    const uint64_t policy = l2_evict_first_policy();
    auto issue = [&](int stage, int chunk) {                      // one elected thread
        const int64_t row0 = (int64_t)chunk * ROWS;
        const int64_t n = rows - row0 < ROWS ? rows - row0 : ROWS;
        const uint32_t cb = (uint32_t)n * (uint32_t)p.C * (uint32_t)sizeof(T);
        mbar_expect_tx(bars + stage, cb);
        bulk_g2s(s_ring + (size_t)stage * stage_bytes, reinterpret_cast<const T *>(p.cls) + row0 * p.C, cb, bars + stage, policy);
    };

    pdl_launch_dependents();
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) mbar_init(bars + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0)
        for (int s = 0; s < stages; ++s) {
            const int c = blockIdx.x + s * gridDim.x;
            if (c < n_chunks) issue(s, c);
        }

    // sigmoid(x) > thr is monotone in x: compare logits against the smallest logit whose sigmoid passes
    const float x_thr = p.logit_thr;
    auto load_loc = [&](int chunk) -> float {                     // lane gl == 0 of every row group
        const int64_t row = (int64_t)chunk * ROWS + r;
        if (!(gl == 0 && chunk < n_chunks && row < rows)) return -CUDART_INF_F;
        if constexpr (sizeof(T) == 4) return __ldcs(p.loc + row);
        else return ldf(reinterpret_cast<const T *>(p.loc) + row);
    };
    float x_next = load_loc((int)blockIdx.x);
    int s = 0;                                                    // ring slot and its phase, carried (no k % stages,
    uint32_t phase = 0;                                           // k / stages: a runtime divisor costs ~35 instructions)
    for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const float x = x_next;
        x_next = load_loc(c + (int)gridDim.x);                    // in flight while this chunk is consumed
        mbar_wait(bars + s, phase);
        const unsigned char *base = s_ring + (size_t)s * stage_bytes;
        const int64_t row = (int64_t)c * ROWS + r;
        const bool ok = row < rows;
        // first arg-max of the row in two cheap steps: the row maximum (max tree + 2 shuffles), then the
        // lowest class index whose logit equals it (reverse predicated scan + 2 shuffles); half the
        // instructions of a running (value, index) comparison.  NaN logits never win (as before).
        float m = -CUDART_INF_F;
        int arg = 0x7fffffff;
        if constexpr (sizeof(T) == 4) {
            const float4 *src = reinterpret_cast<const float4 *>(base) + r * C4;
            float4 q[VPL];
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
                const int v = gl + 4 * i;
                if (EXACT || v < C4) {
                    q[i] = src[v];
                    m = fmaxf(m, fmaxf(fmaxf(q[i].x, q[i].y), fmaxf(q[i].z, q[i].w)));
                }
            }
            m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 1));
            m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 2));
#pragma unroll
            for (int i = VPL - 1; i >= 0; --i) {
                const int v = gl + 4 * i;
                if (EXACT || v < C4) {
                    if (q[i].w == m) arg = 4 * v + 3;
                    if (q[i].z == m) arg = 4 * v + 2;
                    if (q[i].y == m) arg = 4 * v + 1;
                    if (q[i].x == m) arg = 4 * v;
                }
            }
        } else {
            const uint4 *src = reinterpret_cast<const uint4 *>(base) + r * C4;
            float q[VPL][8];
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
                const int v = gl + 4 * i;
                if (EXACT || v < C4) {
                    const uint4 u = src[v];
                    const unsigned w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float2 f;
                        if constexpr (std::is_same<T, __half>::value) f = __half22float2(*reinterpret_cast<const __half2 *>(&w4[e]));
                        else f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w4[e]));
                        q[i][2 * e] = f.x; q[i][2 * e + 1] = f.y;
                        m = fmaxf(m, fmaxf(f.x, f.y));
                    }
                }
            }
            m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 1));
            m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 2));
#pragma unroll
            for (int i = VPL - 1; i >= 0; --i) {
                const int v = gl + 4 * i;
                if (EXACT || v < C4) {
#pragma unroll
                    for (int e = 7; e >= 0; --e)
                        if (q[i][e] == m) arg = 8 * v + e;
                }
            }
        }
        arg = min(arg, __shfl_xor_sync(kFullMask, arg, 1));
        arg = min(arg, __shfl_xor_sync(kFullMask, arg, 2));
        if (arg == 0x7fffffff) arg = 0;                           // all-NaN row
        // Anything on a candidate's path delays the barrier below and with it the refill of this stage (a chunk has a
        // candidate 3 times out of 4 at cfg1): only the logit pre-filter, a ballot and one shared-memory store stay in
        // the loop (no atomic: the warp owns its segment and carries the fill count in a register); the sigmoid test,
        // the slot atomic, the box decode and the stores happen in flush_staged.
        const bool staged = gl == 0 && ok && x >= x_thr;
        const unsigned sm = __ballot_sync(kFullMask, staged);
        if (staged) {
            StagedCand sc;
            sc.row_lo = (int)(row & 0xffffffff); sc.row_hi = (int)(row >> 32);
            sc.x = x; sc.arg = arg;
            s_list[warp * 32 + n_staged + __popc(sm & ((1u << lane) - 1u))] = sc;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const T *>(p.box_raw) + 4 * row));      // read at flush time
        }
        n_staged += __popc(sm);
        __syncthreads();                                          // every lane is done with stage s
        if (tid == 0) {
            const int next = c + stages * gridDim.x;
            if (next < n_chunks) issue(s, next);
        }
        if (n_staged > 32 - 8) {                                  // warp-uniform: the segment could overflow next chunk
            flush_staged<T>(p, lane < n_staged ? s_list + warp * 32 + lane : nullptr);
            n_staged = 0;
        }
        if (++s == stages) { s = 0; phase ^= 1u; }
    }
    // What is left (a handful per warp at cfg1) is flushed by the CTA as ONE list: every CTA of the grid ends at the
    // same time, and 8 slot atomics per CTA on the 64 per-image counters queue up at the L2 — one or two do not.
    if (lane == 0) s_seg_count[warp] = n_staged;
    __syncthreads();
    int total = 0, mine_seg = -1, mine_idx = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        const int cnt = s_seg_count[w];
        if (mine_seg < 0 && tid < total + cnt) { mine_seg = w; mine_idx = tid - total; }
        total += cnt;
    }
    if ((tid & ~31) < total)                                       // warp-uniform: this warp has entries of the merged list
        flush_staged<T>(p, tid < total ? s_list + mine_seg * 32 + mine_idx : nullptr);
}

// ---------------------------------------------------------------------------
// Candidate-first variant.  score = sigmoid(loc) does not depend on the class logits
// (ref :113,:117), so only the rows that pass the threshold need their C class logits and
// their raw box: the kernel streams the location map (4 B per location, coalesced), and
// gathers 4C+16 B per *candidate*.  Same outputs as the dense variants (the lists are
// unordered in both).  Compulsory traffic 4*A + cand*(4C+16+28) per image — 30x less than
// the dense scan at 2 % candidates; it loses to the TMA stream once most rows pass.
//
// One warp per block of 32 consecutive rows.  Lane = row for the threshold test and the slot
// allocation (one returning atomic per (warp, image)); then the candidates are taken four
// at a time by the warp's four 8-lane groups: lane j of a group loads float4s j, j+8, ...
// of the class row (128 contiguous bytes per group and load), first-argmax = row maximum
// (3 shuffles) then lowest index equal to it (3 shuffles), like the TMA consumer.
// VEC = 4: 16-byte loads (C % 4 == 0, aligned); VEC = 1: any C.
// ---------------------------------------------------------------------------
// HOST: the class / box maps are pinned host memory read in place over PCIe (rows of at most 32 16-byte vectors): a
// candidate's class row is ONE warp instruction (lane v = vector v; up to R candidates of the block in flight), its raw box
// is requested together with it (one round trip, not two back to back), first-argmax over the warp.  Own instantiation: the
// device-memory kernel keeps its registers.  PCIe reads are bounded by outstanding requests, not bytes
// (tools/micro/host_gather_bw.cu), and element loads of half maps would be 2-byte requests.
template <int VEC, typename T = float, bool HOST = false>     // T: element type of the three maps (VEC == 4 needs T == float)
__global__ void __launch_bounds__(256) k_candidate_decode(DenseDecodeParams p)
{
    const T *t_loc = reinterpret_cast<const T *>(p.loc), *t_cls = reinterpret_cast<const T *>(p.cls);
    const T *t_box = reinterpret_cast<const T *>(p.box_raw);
    const int lane = threadIdx.x & 31, gq = lane >> 3, gl = lane & 7;
    const int64_t rows = (int64_t)p.batch * p.A;
    const int64_t n_blocks = (rows + 31) >> 5;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int CV = p.C / VEC;                                      // vectors per row (VEC == 1: CV == C)
    for (int64_t blk = warp0; blk < n_blocks; blk += n_warps) {
        const int64_t row = (blk << 5) + lane;
        const bool in = row < rows;
        const float x = in ? ldf(t_loc + row) : -CUDART_INF_F;
        float s = 0.f;
        bool cand = false;
        if (in && x >= p.logit_thr) { s = round_to<T>(sigmoid_f(x)); cand = s > p.score_thr; }
        const unsigned m = __ballot_sync(kFullMask, cand);
        if (m == 0u) continue;
        const int b = !in ? 0 : (rows < (1ll << 31) ? (int)((unsigned)row / (unsigned)p.A) : (int)(row / p.A));
        const int a = in ? (int)(row - (int64_t)b * p.A) : 0;
        int slot = 0;
        if (cand) {                                                // the atomic's round trip overlaps the row gathers
            const unsigned peers = __match_any_sync(m, b);
            const int leader = __ffs(peers) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(p.cand_count + b, __popc(peers));
            base = __shfl_sync(peers, base, leader);
            slot = base + __popc(peers & ((1u << lane) - 1u));
        }
        const int first = __ffs(m) - 1;
        if constexpr (HOST) {
            constexpr int N = Vec16<T>::N, R = N == 4 ? 4 : 2;
            const int CVW = p.C / N;                               // <= 32 (launcher)
            for (unsigned rem = m; rem != 0u;) {                   // R candidates per pass: requests first, then the reductions
                int src[R], cnt = 0;
                float q[R][N];
                float4 raw[R];
#pragma unroll
                for (int k = 0; k < R; ++k) {
                    src[k] = first;
                    if (rem != 0u) { src[k] = __ffs(rem) - 1; rem &= rem - 1u; ++cnt; }
                    const int64_t crow = (blk << 5) + src[k];
                    raw[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (k < cnt && lane < CVW) ld_vec16(t_cls + crow * p.C + lane * N, q[k]);
                    else {
#pragma unroll
                        for (int e = 0; e < N; ++e) q[k][e] = -CUDART_INF_F;
                    }
                    if (k < cnt && lane == 0) raw[k] = ldf4(t_box + 4 * crow);
                }
#pragma unroll
                for (int k = 0; k < R; ++k) {
                    if (k >= cnt) continue;                        // warp-uniform
                    float best = -CUDART_INF_F;
                    int arg = 0x7fffffff;
#pragma unroll
                    for (int e = 0; e < N; ++e)
                        if (q[k][e] > best) { best = q[k][e]; arg = lane * N + e; }       // ascending index inside the lane: first max
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const float ob = __shfl_xor_sync(kFullMask, best, o);
                        const int oa = __shfl_xor_sync(kFullMask, arg, o);
                        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
                    }
                    if (arg == 0x7fffffff) arg = 0;                // all -inf / NaN row: same convention as below
                    const float cs = __shfl_sync(kFullMask, s, src[k]);
                    const int ca = __shfl_sync(kFullMask, a, src[k]), cb = __shfl_sync(kFullMask, b, src[k]);
                    const int cslot = __shfl_sync(kFullMask, slot, src[k]);
                    if (lane == 0 && cslot < p.cap) {
                        const float4 off = __ldg(p.offsets + ca), sc = __ldg(p.scales + ca);
                        const int64_t o = (int64_t)cb * p.cap + cslot;
                        p.cand_key[o] = ((unsigned long long)__float_as_uint(cs) << 32) | (unsigned long long)(0xffffffffu - (unsigned)ca);
                        p.cand_box[o] = make_float4((off.x + sc.x * round_to<T>(expf(raw[k].x))) * p.img_w, (off.y + sc.y * round_to<T>(expf(raw[k].y))) * p.img_h,
                                                    (off.z + sc.z * round_to<T>(expf(raw[k].z))) * p.img_w, (off.w + sc.w * round_to<T>(expf(raw[k].w))) * p.img_h);
                        p.cand_cls[o] = arg;
                    }
                }
            }
        } else
        for (unsigned rem = m; rem != 0u;) {                       // four candidates per pass: peel the four lowest set bits
            int src = first;                                       // lane that owns this group's candidate
            bool have = false;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (rem != 0u) {
                    if (gq == k) { src = __ffs(rem) - 1; have = true; }
                    rem &= rem - 1u;
                }
            }
            const int64_t crow = (blk << 5) + src;
            float best = -CUDART_INF_F;
            int arg = 0x7fffffff;
            if (VEC == 4) {
                const float4 *src4 = reinterpret_cast<const float4 *>(p.cls) + crow * CV;
                for (int v0 = 0; v0 < CV; v0 += 32) {              // 4 loads in flight per lane and pass
                    float4 q[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int v = v0 + gl + 8 * i;
                        q[i] = (have && v < CV) ? __ldcs(src4 + v) : make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int c = 4 * (v0 + gl + 8 * i);
                        const float e[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (e[k] > best) { best = e[k]; arg = c + k; }     // ascending index inside the lane: first max
                    }
                }
            } else {
                const T *srow = t_cls + crow * p.C;
                for (int c = gl; c < (have ? p.C : 0); c += 8) {
                    const float e = ldf(srow + c);
                    if (e > best) { best = e; arg = c; }
                }
            }
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) {                      // inside the 8-lane group
                const float ob = __shfl_xor_sync(kFullMask, best, o);
                const int oa = __shfl_xor_sync(kFullMask, arg, o);
                if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
            }
            // -inf rows (arg still unset when every logit is -inf or NaN): first index whose logit equals the
            // maximum is 0 for an all -inf row; NaN never wins — same convention as the dense variants
            if (arg == 0x7fffffff) arg = 0;
            const float cs = __shfl_sync(kFullMask, s, src);
            const int ca = __shfl_sync(kFullMask, a, src), cb = __shfl_sync(kFullMask, b, src);
            const int cslot = __shfl_sync(kFullMask, slot, src);
            if (have && gl == 0 && cslot < p.cap) {
                const float4 raw = ldf4(t_box + 4 * crow);
                const float4 off = __ldg(p.offsets + ca), sc = __ldg(p.scales + ca);
                const int64_t o = (int64_t)cb * p.cap + cslot;
                p.cand_key[o] = ((unsigned long long)__float_as_uint(cs) << 32) | (unsigned long long)(0xffffffffu - (unsigned)ca);
                p.cand_box[o] = make_float4((off.x + sc.x * round_to<T>(expf(raw.x))) * p.img_w, (off.y + sc.y * round_to<T>(expf(raw.y))) * p.img_h,
                                            (off.z + sc.z * round_to<T>(expf(raw.z))) * p.img_w, (off.w + sc.w * round_to<T>(expf(raw.w))) * p.img_h);
                p.cand_cls[o] = arg;
            }
        }
    }
}

__global__ void k_zero_i32(int32_t *p, int n)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = 0;
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_topk(const float *loc_logits, int batch, int64_t num_anchors, int k, int64_t *idx,
                            float *top_logits, void *stream)
{
    return sihl_od_topk_t(loc_logits, SIHL_OD_F32, batch, num_anchors, k, idx, top_logits, stream);
}

extern "C" int sihl_od_topk_t(const void *loc_logits, int map_dtype, int batch, int64_t num_anchors, int k, int64_t *idx,
                              float *top_logits, void *stream)
{
    SIHL_CHECK_ARG(loc_logits && idx && top_logits, "NULL argument");
    SIHL_CHECK_ARG(k >= 1 && k <= kTopkMaxK, "k=%d outside 1..%d", k, kTopkMaxK);
    SIHL_CHECK_ARG(num_anchors >= k && num_anchors < (1ll << 30),
                   "selected index k out of range: k=%d > %lld locations (torch.topk raises in the reference)", k,
                   (long long)num_anchors);
    if (batch <= 0) return SIHL_OD_OK;
    int kp = 1;
    while (kp < k) kp <<= 1;
    SIHL_DISPATCH_DTYPE(map_dtype, (k_topk<T><<<batch, kTopkThreads, 0, (cudaStream_t)stream>>>(
                                       reinterpret_cast<const T *>(loc_logits), (int)num_anchors, k, kp, idx, top_logits)));
    SIHL_CHECK_LAUNCH("k_topk");
    return SIHL_OD_OK;
}

extern "C" int sihl_od_decode_rows(const float *top_logits, const int64_t *idx, int batch, int k,
                                   const float *cls_rows, int num_classes, const float *box_rows,
                                   const float *offsets, const float *scales, int img_w, int img_h,
                                   int64_t *num_instances, float *scores, int64_t *classes, float *boxes, void *stream)
{
    return sihl_od_decode_rows_t(top_logits, idx, batch, k, cls_rows, num_classes, box_rows, SIHL_OD_F32, offsets, scales, img_w,
                                 img_h, num_instances, scores, classes, boxes, stream);
}

extern "C" int sihl_od_decode_rows_t(const float *top_logits, const int64_t *idx, int batch, int k,
                                     const void *cls_rows, int num_classes, const void *box_rows, int map_dtype,
                                     const float *offsets, const float *scales, int img_w, int img_h,
                                     int64_t *num_instances, float *scores, int64_t *classes, float *boxes, void *stream)
{
    SIHL_CHECK_ARG(top_logits && idx && cls_rows && box_rows && offsets && scales, "NULL input");
    SIHL_CHECK_ARG(num_instances && scores && classes && boxes, "NULL output");
    SIHL_CHECK_ARG(k >= 1 && num_classes >= 1 && img_w > 0 && img_h > 0, "bad sizes");
    if (batch <= 0) return SIHL_OD_OK;
    SIHL_CHECK_ARG((reinterpret_cast<uintptr_t>(box_rows) & 15u) == 0, "box_rows must be 16-byte aligned");
    SIHL_DISPATCH_DTYPE(map_dtype, (k_decode_rows<T><<<batch, 256, 0, (cudaStream_t)stream>>>(
        top_logits, idx, k, reinterpret_cast<const T *>(cls_rows), num_classes, reinterpret_cast<const T *>(box_rows),
        reinterpret_cast<const float4 *>(offsets), reinterpret_cast<const float4 *>(scales), (float)img_w, (float)img_h,
        num_instances, scores, classes, boxes)));
    SIHL_CHECK_LAUNCH("k_decode_rows");
    return SIHL_OD_OK;
}

// Argument checks, optional counter zeroing and the parameter block shared by the dense and the
// candidate-first decode.  Returns 1 when there is nothing to do (batch == 0).
static int decode_prologue(const float *loc_logits, const float *cls_logits, const float *box_raw, int batch,
                           int64_t num_anchors, int num_classes, const float *offsets, const float *scales,
                           int img_w, int img_h, float score_thr, int32_t *cand_count, int64_t cand_capacity,
                           uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts, cudaStream_t st,
                           DenseDecodeParams *out, int *nothing)
{
    *nothing = 0;
    SIHL_CHECK_ARG(loc_logits && cls_logits && box_raw && offsets && scales, "NULL input");
    SIHL_CHECK_ARG(cand_count && cand_key && cand_box && cand_cls, "NULL output");
    SIHL_CHECK_ARG(batch >= 0 && num_anchors > 0 && num_anchors < (1ll << 30) && num_classes >= 1 && cand_capacity >= 1,
                   "bad sizes");
    SIHL_CHECK_ARG(img_w > 0 && img_h > 0, "image size %dx%d", img_w, img_h);
    SIHL_CHECK_ARG(score_thr >= 0.f, "score_thr=%f must be >= 0 (scores are sigmoid outputs)", (double)score_thr);
    if (batch == 0) { *nothing = 1; return SIHL_OD_OK; }
    if (zero_counts) {
        k_zero_i32<<<(batch + 255) / 256, 256, 0, st>>>(cand_count, batch);
        SIHL_CHECK_LAUNCH("k_zero_i32");
    }
    DenseDecodeParams &p = *out;
    p.loc = loc_logits; p.cls = cls_logits; p.box_raw = box_raw; p.batch = batch; p.A = (int)num_anchors; p.C = num_classes;
    p.offsets = reinterpret_cast<const float4 *>(offsets); p.scales = reinterpret_cast<const float4 *>(scales);
    p.img_w = (float)img_w; p.img_h = (float)img_h; p.score_thr = score_thr;
    {   // logit(thr) minus a safety margin: only saves the exp for the bulk of the rows
        const double t = (double)score_thr;
        p.logit_thr = (t <= 0.0) ? -HUGE_VALF : (t >= 1.0 ? HUGE_VALF : (float)(log(t / (1.0 - t)) - 1e-3 * (1.0 + fabs(log(t / (1.0 - t))))));
    }
    p.cand_count = cand_count; p.cap = cand_capacity;
    p.cand_key = reinterpret_cast<unsigned long long *>(cand_key); p.cand_box = reinterpret_cast<float4 *>(cand_box);
    p.cand_cls = cand_cls;
    return SIHL_OD_OK;
}

extern "C" int sihl_od_dense_decode(const float *loc_logits, const float *cls_logits, const float *box_raw, int batch,
                                    int64_t num_anchors, int num_classes, const float *offsets, const float *scales,
                                    int img_w, int img_h, float score_thr, int32_t *cand_count, int64_t cand_capacity,
                                    uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                                    void *stream)
{
    return sihl_od_dense_decode_t(loc_logits, cls_logits, box_raw, SIHL_OD_F32, batch, num_anchors, num_classes, offsets, scales,
                                  img_w, img_h, score_thr, cand_count, cand_capacity, cand_key, cand_box, cand_cls, zero_counts,
                                  stream);
}

// Half maps: the TMA ring with 2-byte elements (C % 8 == 0, C <= 256, 16-byte aligned maps).
template <typename T>
static int launch_decode_tma_half(const DenseDecodeParams &p, int64_t rows, int num_classes, cudaStream_t st)
{
    const int cv = num_classes / 8;
    const int vpl = (cv + 3) / 4;
    const bool exact = vpl * 4 == cv;
    int rows_per_stage = kChunkRows, stages = 2, ctas_per_sm = 2;
    if ((rows + kChunkRows - 1) / kChunkRows < (int64_t)16 * kNumSMs * 2) { rows_per_stage = 32; stages = 2; ctas_per_sm = 3; }
    else { stages = 4; }                                   // half-size stages: twice as many keep the same bytes in flight
    const size_t stage_bytes = (size_t)rows_per_stage * num_classes * sizeof(T);
    const size_t smem = stages * stage_bytes + stages * sizeof(uint64_t);
    const int n_chunks = (int)((rows + rows_per_stage - 1) / rows_per_stage);
    int blocks = kNumSMs * ctas_per_sm;
    if (blocks > n_chunks) blocks = n_chunks;
#define SIHL_DH_LAUNCH(KERN, THREADS)                                                                             \
    do {                                                                                                          \
        auto kern = KERN;                                                                                         \
        int rc = cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),  \
                             "cudaFuncSetAttribute(k_dense_decode_tma)");                                         \
        if (rc) return rc;                                                                                        \
        kern<<<blocks, THREADS, smem, st>>>(p, stages, n_chunks);                                                 \
        SIHL_CHECK_LAUNCH("k_dense_decode_tma (half maps)");                                                      \
    } while (0)
#define SIHL_DH(VPL)                                                                                              \
    do {                                                                                                          \
        if (rows_per_stage == 64) {                                                                               \
            if (exact) SIHL_DH_LAUNCH((k_dense_decode_tma<VPL, true, 64, T>), 256);                               \
            else SIHL_DH_LAUNCH((k_dense_decode_tma<VPL, false, 64, T>), 256);                                    \
        } else {                                                                                                  \
            if (exact) SIHL_DH_LAUNCH((k_dense_decode_tma<VPL, true, 32, T>), 128);                               \
            else SIHL_DH_LAUNCH((k_dense_decode_tma<VPL, false, 32, T>), 128);                                    \
        }                                                                                                         \
    } while (0)
    switch (vpl) {
        case 1: SIHL_DH(1); break;
        case 2: SIHL_DH(2); break;
        case 3: SIHL_DH(3); break;
        case 4: SIHL_DH(4); break;
        default: SIHL_DH(8); break;
    }
#undef SIHL_DH
#undef SIHL_DH_LAUNCH
    return SIHL_OD_OK;
}

extern "C" int sihl_od_dense_decode_t(const void *loc_logits_v, const void *cls_logits_v, const void *box_raw_v, int map_dtype,
                                      int batch, int64_t num_anchors, int num_classes, const float *offsets,
                                      const float *scales, int img_w, int img_h, float score_thr, int32_t *cand_count,
                                      int64_t cand_capacity, uint64_t *cand_key, float *cand_box, int32_t *cand_cls,
                                      int zero_counts, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const float *loc_logits = reinterpret_cast<const float *>(loc_logits_v), *cls_logits = reinterpret_cast<const float *>(cls_logits_v);
    const float *box_raw = reinterpret_cast<const float *>(box_raw_v);
    DenseDecodeParams p;
    int nothing = 0;
    int rc0 = decode_prologue(loc_logits, cls_logits, box_raw, batch, num_anchors, num_classes, offsets, scales, img_w, img_h,
                              score_thr, cand_count, cand_capacity, cand_key, cand_box, cand_cls, zero_counts, st, &p, &nothing);
    if (rc0 || nothing) return rc0;
    if (map_dtype != SIHL_OD_F32) {
        SIHL_CHECK_ARG(map_dtype == SIHL_OD_F16 || map_dtype == SIHL_OD_BF16, "map dtype code %d", map_dtype);
        const bool ok = num_classes % 8 == 0 && num_classes <= 256 && (int64_t)batch * num_anchors >= 4 * kChunkRows &&
                        ((reinterpret_cast<uintptr_t>(cls_logits_v) | reinterpret_cast<uintptr_t>(box_raw_v)) & 15u) == 0;
        SIHL_CHECK_ARG(ok, "the dense scan of half maps needs C %% 8 == 0, C <= 256, >= 256 rows and 16-byte aligned maps "
                           "(C=%d): use sihl_od_candidate_decode_t", num_classes);
        // scores are sigmoid() rounded to the map type and may cross the threshold from below: widen the pre-filter
        if (p.logit_thr > -HUGE_VALF && p.logit_thr < HUGE_VALF) p.logit_thr -= 0.05f * (1.f + fabsf(p.logit_thr));
        const int64_t rows_h = (int64_t)batch * num_anchors;
        if (map_dtype == SIHL_OD_F16) return launch_decode_tma_half<__half>(p, rows_h, num_classes, st);
        return launch_decode_tma_half<__nv_bfloat16>(p, rows_h, num_classes, st);
    }
    const int64_t rows = (int64_t)batch * num_anchors;
    const bool aligned = (num_classes % 4 == 0) && ((reinterpret_cast<uintptr_t>(cls_logits) & 15u) == 0) &&
                         ((reinterpret_cast<uintptr_t>(box_raw) & 15u) == 0);
    const int c4 = num_classes / 4;
    const bool loc_aligned = (reinterpret_cast<uintptr_t>(loc_logits) & 15u) == 0;
    if (aligned && loc_aligned && c4 <= 32 && rows >= 4 * kChunkRows) {
        const int vpl = (c4 + 3) / 4;
        const bool exact = vpl * 4 == c4;
        // 2 stages x 2 CTAs per SM of 64-row stages: measured on B200 the kernel is already at the HBM roof with ~87 KB
        // in flight per SM (3 and 4 stages give the same 32 us), and the smaller ring leaves ~120 KB of shared
        // memory per SM to the kernels of the other chain / the neighbouring step running concurrently.
        // SMALL scans (fewer than ~16 such stages per CTA: the 1024^2 / batch 8 crowd config has 9) are dominated by
        // ring start-up, the last partial round and the end-of-kernel flush: they take 32-row stages on 128-thread
        // CTAs, 3 per SM with 2 stages each — half as long work items (5 % instead of 10 % imbalance in the last round)
        // and 1.5x the CTAs.  Measured at crowd (profiles/r02_decode_sweep_crowd.json): 18.5 us with the cfg1 ring,
        // 14.1 us with this one (14.0-14.5 us for every 32-row ring with >= 3 CTAs per SM; this is the one with the
        // smallest shared-memory footprint, 60 KB per SM).
        const int stages = 2;
        int rows_per_stage = kChunkRows, ctas_per_sm = 2;
        if ((rows + kChunkRows - 1) / kChunkRows < (int64_t)16 * kNumSMs * 2) { rows_per_stage = 32; ctas_per_sm = 3; }
        const size_t stage_bytes = (size_t)rows_per_stage * num_classes * 4;
        const size_t smem = stages * stage_bytes + stages * sizeof(uint64_t);
        const int n_chunks = (int)((rows + rows_per_stage - 1) / rows_per_stage);
        int blocks = kNumSMs * ctas_per_sm;
        if (blocks > n_chunks) blocks = n_chunks;
#define SIHL_DT_LAUNCH(KERN, THREADS)                                                                             \
    do {                                                                                                          \
        auto kern = KERN;                                                                                         \
        int rc = cuda_status(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),  \
                             "cudaFuncSetAttribute(k_dense_decode_tma)");                                         \
        if (rc) return rc;                                                                                        \
        kern<<<blocks, THREADS, smem, st>>>(p, stages, n_chunks);                                                 \
        SIHL_CHECK_LAUNCH("k_dense_decode_tma");                                                                  \
    } while (0)
#define SIHL_DT(VPL)                                                                                              \
    do {                                                                                                          \
        if (rows_per_stage == 64) {                                                                               \
            if (exact) SIHL_DT_LAUNCH((k_dense_decode_tma<VPL, true, 64>), 256);                                  \
            else SIHL_DT_LAUNCH((k_dense_decode_tma<VPL, false, 64>), 256);                                       \
        } else {                                                                                                  \
            if (exact) SIHL_DT_LAUNCH((k_dense_decode_tma<VPL, true, 32>), 128);                                  \
            else SIHL_DT_LAUNCH((k_dense_decode_tma<VPL, false, 32>), 128);                                       \
        }                                                                                                         \
    } while (0)
        switch (vpl) {
            case 1: SIHL_DT(1); break;
            case 2: SIHL_DT(2); break;
            case 3: SIHL_DT(3); break;
            case 4: SIHL_DT(4); break;
            case 5: SIHL_DT(5); break;
            case 6: SIHL_DT(6); break;
            case 7: SIHL_DT(7); break;
            default: SIHL_DT(8); break;
        }
#undef SIHL_DT
#undef SIHL_DT_LAUNCH
    } else if (aligned && c4 <= 32 * 8) {
        // 4 lanes per row up to C = 128, a full warp per row beyond; grid = 4 resident CTAs per SM
        const int lpr = c4 <= 32 ? 4 : 32;
        int64_t blocks = (rows * lpr / 2 + 255) / 256;
        const int64_t cap = (int64_t)kNumSMs * 4;
        if (blocks > cap) blocks = cap;
        const dim3 grid((unsigned)(blocks < 1 ? 1 : blocks));
        const int vpl = (c4 + lpr - 1) / lpr;
        const bool exact = vpl * lpr == c4;
#define SIHL_DD(LPR, VPL)                                                                    \
    if (exact) k_dense_decode_v4<LPR, VPL, true><<<grid, 256, 0, st>>>(p);                   \
    else k_dense_decode_v4<LPR, VPL, false><<<grid, 256, 0, st>>>(p)
        if (lpr == 4) {
            switch (vpl) {
                case 1: SIHL_DD(4, 1); break;
                case 2: SIHL_DD(4, 2); break;
                case 3: SIHL_DD(4, 3); break;
                case 4: SIHL_DD(4, 4); break;
                case 5: SIHL_DD(4, 5); break;
                case 6: SIHL_DD(4, 6); break;
                case 7: SIHL_DD(4, 7); break;
                default: SIHL_DD(4, 8); break;
            }
        } else {
            switch (vpl) {
                case 2: SIHL_DD(32, 2); break;
                case 3: SIHL_DD(32, 3); break;
                case 4: SIHL_DD(32, 4); break;
                case 5: SIHL_DD(32, 5); break;
                case 6: SIHL_DD(32, 6); break;
                case 7: SIHL_DD(32, 7); break;
                default: SIHL_DD(32, 8); break;
            }
        }
#undef SIHL_DD
    } else {
        int64_t blocks = (rows * 8 + 255) / 256;
        const int64_t cap = (int64_t)kNumSMs * 8;          // 8 resident CTAs of 256 threads per SM
        if (blocks > cap) blocks = cap;
        const dim3 grid((unsigned)(blocks < 1 ? 1 : blocks));
        k_dense_decode<0><<<grid, 256, 0, st>>>(p);
    }
    SIHL_CHECK_LAUNCH("k_dense_decode");
    return SIHL_OD_OK;
}

extern "C" int sihl_od_candidate_decode(const float *loc_logits, const float *cls_logits, const float *box_raw, int batch,
                                        int64_t num_anchors, int num_classes, const float *offsets, const float *scales,
                                        int img_w, int img_h, float score_thr, int32_t *cand_count, int64_t cand_capacity,
                                        uint64_t *cand_key, float *cand_box, int32_t *cand_cls, int zero_counts,
                                        void *stream)
{
    return sihl_od_candidate_decode_t(loc_logits, cls_logits, box_raw, SIHL_OD_F32, batch, num_anchors, num_classes, offsets,
                                      scales, img_w, img_h, score_thr, cand_count, cand_capacity, cand_key, cand_box, cand_cls,
                                      zero_counts, stream);
}

extern "C" int sihl_od_candidate_decode_t(const void *loc_logits_v, const void *cls_logits_v, const void *box_raw_v, int map_dtype,
                                          int batch, int64_t num_anchors, int num_classes, const float *offsets,
                                          const float *scales, int img_w, int img_h, float score_thr, int32_t *cand_count,
                                          int64_t cand_capacity, uint64_t *cand_key, float *cand_box, int32_t *cand_cls,
                                          int zero_counts, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    const float *loc_logits = reinterpret_cast<const float *>(loc_logits_v), *cls_logits = reinterpret_cast<const float *>(cls_logits_v);
    const float *box_raw = reinterpret_cast<const float *>(box_raw_v);
    DenseDecodeParams p;
    int nothing = 0;
    int rc0 = decode_prologue(loc_logits, cls_logits, box_raw, batch, num_anchors, num_classes, offsets, scales, img_w, img_h,
                              score_thr, cand_count, cand_capacity, cand_key, cand_box, cand_cls, zero_counts, st, &p, &nothing);
    if (rc0 || nothing) return rc0;
    const int64_t rows = (int64_t)batch * num_anchors;
    const int64_t row_blocks = (rows + 31) / 32;                   // one warp per 32 rows, 8 warps per CTA
    int64_t blocks = (row_blocks + 7) / 8;
    const int64_t cap = (int64_t)kNumSMs * 6;                      // 40 registers: 6 resident CTAs of 256 threads per SM
    if (blocks > cap) blocks = cap;
    const bool vec = (num_classes % 4 == 0) && ((reinterpret_cast<uintptr_t>(cls_logits) & 15u) == 0);
    SIHL_CHECK_ARG((reinterpret_cast<uintptr_t>(box_raw) & 15u) == 0, "box_raw must be 16-byte aligned");
    bool host = false;                                             // pinned host maps (zero-copy)
    {
        const void *host_ok_maps[2] = {cls_logits_v, box_raw_v};
        for (const void *map : host_ok_maps) {       // pageable host memory would fault in the kernel: refuse it here
            cudaPointerAttributes attr;
            if (cudaPointerGetAttributes(&attr, map) != cudaSuccess) { (void)cudaGetLastError(); continue; }
            SIHL_CHECK_ARG(attr.type != cudaMemoryTypeUnregistered,
                           "box_raw / cls_logits must be device memory or PINNED host memory (got a pageable host pointer)");
            if (map == cls_logits_v) host = attr.type == cudaMemoryTypeHost;
        }
        // the whole-row reads need 16-byte rows of at most 32 vectors
        const size_t row_bytes = (size_t)num_classes * (map_dtype == SIHL_OD_F32 ? 4 : 2);
        host = host && row_bytes % 16 == 0 && row_bytes <= 32 * 16 && (reinterpret_cast<uintptr_t>(cls_logits_v) & 15u) == 0;
    }
    if (map_dtype == SIHL_OD_F32) {
        if (host) k_candidate_decode<4, float, true><<<(unsigned)blocks, 256, 0, st>>>(p);
        else if (vec) k_candidate_decode<4><<<(unsigned)blocks, 256, 0, st>>>(p);
        else k_candidate_decode<1><<<(unsigned)blocks, 256, 0, st>>>(p);
    } else {
        // half maps: the score is sigmoid() ROUNDED to the map type (what the reference's `.sigmoid()` returns under
        // autocast), which can cross the threshold from below: widen the conservative logit pre-filter accordingly
        if (p.logit_thr > -HUGE_VALF && p.logit_thr < HUGE_VALF) p.logit_thr -= 0.05f * (1.f + fabsf(p.logit_thr));
        if (host) SIHL_DISPATCH_DTYPE(map_dtype, (k_candidate_decode<1, T, true><<<(unsigned)blocks, 256, 0, st>>>(p)));
        else SIHL_DISPATCH_DTYPE(map_dtype, (k_candidate_decode<1, T><<<(unsigned)blocks, 256, 0, st>>>(p)));
    }
    SIHL_CHECK_LAUNCH("k_candidate_decode");
    return SIHL_OD_OK;
}
