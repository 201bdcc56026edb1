
// od_loss.cu — positive-row losses of the detection head over dense maps, and the loss finalize
// (SURVEY.md §8 a5-a10).  The compact-row forward and backward of the drop-in head's training
// step are in od_train.cu.
//
//   k_pos_loss_tiles  ref :187-208 (+ torchvision ciou_loss.py)   gather-bound, (16+4C) B / positive
//   k_loss_finalize   ref :163-172, :180, :197, :208, :210        5 scalars
//
// Sums are accumulated per thread in fp32 over a handful of elements, then in fp64
// through warp shuffles, one shared-memory hop and one atomicAdd per CTA and term.
#include "od_common.cuh"
#include "od_pos.cuh"

namespace sihl {

// Positive-row losses straight from the per-tile lists k_assign_resolve leaves behind (dense
// maps only).  Work items are 32-row chunks of those lists, published by k_assign_resolve in
// pos_chunks (count in sums[7]): coarse-level tiles hold several hundred positives, fine-level
// tiles a handful, so chunking the lists balances the CTAs and no CTA ever starts empty.  One CTA
// of 128 threads takes one chunk per round, 4 (or 8) lanes per row.  No compaction, no host
// round trip; the class-logit row was prefetched into L2 by k_assign_resolve.
// The last CTA to finish may also fold k_loss_finalize in (single-GPU case).
constexpr int kPosTileThreads = 128;

struct PosTileParams {
    const int32_t *pos_chunks; const int32_t *tile_pos_rows; const int2 *tile_pos_aux; int n_tiles; int num_anchors;
    const float4 *offsets; const float4 *scales; float img_w, img_h;
    const float4 *gt_boxes; const int64_t *gt_classes; const int32_t *gt_offsets;
    int host_rows;                                                        // the maps live in pinned host memory
    const void *box_raw; const void *cls; int num_classes; int cls_vec4;   // element type T of the kernel template;
    double *sums;                                                         // cls_vec4: rows are read 16 bytes at a time
    float *losses; unsigned *done_counter;       // optional fused finalize
};

// optional fused cross-GPU exchange of the sums (od_exchange.cu): world > 1, peer[r] = rank r's region
struct ExchangeParams {
    int world, rank;
    unsigned long long *const *peer;             // device array [world]
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// All-reduce (sum) of the 8 partial sums across the GPUs of the node, by the last CTA of the loss kernel:
// thread q pushes this rank's sums into rank q's region (plain stores over NVLink, then a release store of the
// step number), waits for rank q's push into the local region, and 8 threads add the W contributions in rank
// order.  A peer that never shows up (a crashed rank) ends the wait after the region's timeout (word 18W+1 in ns,
// sihl_od_exchange_set_timeout; 0 = the 120 s default — long enough for a rank stalled by a dataloader, a checkpoint
// or first-step lazy initialisation) with NaN sums instead of a hang, AND records the step in the region's sticky
// error word (18W+2), which the host reads with sihl_od_exchange_status: a late peer is reported, not only NaN-ed.
__device__ __noinline__ void exchange_sums(unsigned long long *const *peer, int W, int rank, double *sums,
                                           double *s_in /* shared [8] */)
{
    const int tid = threadIdx.x;
    __shared__ unsigned long long s_step;
    __shared__ int s_timeout;
    unsigned long long *mine = peer[rank];
    if (tid == 0) {
        s_step = ++mine[18 * W];                                   // this GPU's step counter (only this CTA touches it)
        s_timeout = 0;
    }
    if (tid < SIHL_OD_NUM_SUMS) s_in[tid] = reinterpret_cast<volatile double *>(sums)[tid];
    __syncthreads();
    const unsigned long long step = s_step;
    const int parity = (int)(step & 1ull);
    if (tid < W) {
        unsigned long long *theirs = peer[tid];
        double *dst = reinterpret_cast<double *>(theirs) + ((size_t)parity * W + rank) * SIHL_OD_NUM_SUMS;
#pragma unroll
        for (int i = 0; i < SIHL_OD_NUM_SUMS; ++i) dst[i] = s_in[i];
        // the release store orders THIS thread's eight stores above before the flag at system scope: no separate
        // (and, over NVLink, microsecond-expensive) __threadfence_system() is needed
        st_release_sys(theirs + 16 * W + parity * W + rank, step);
        const unsigned long long *flag = mine + 16 * W + parity * W + tid;
        const unsigned long long t0 = global_timer_ns();
        unsigned long long limit = *reinterpret_cast<volatile unsigned long long *>(mine + 18 * W + 1);
        if (limit == 0ull) limit = 120000000000ull;
        while (ld_acquire_sys(flag) != step) {
            if (global_timer_ns() - t0 > limit) {
                s_timeout = 1;
                atomicCAS(mine + 18 * W + 2, 0ull, step);            // sticky: the first step that timed out
                break;
            }
            __nanosleep(64);
        }
    }
    __syncthreads();
    if (tid < SIHL_OD_NUM_SUMS) {
        const volatile double *src = reinterpret_cast<volatile double *>(mine) + (size_t)parity * W * SIHL_OD_NUM_SUMS;
        double total = 0.0;
        for (int r = 0; r < W; ++r) total += src[r * SIHL_OD_NUM_SUMS + tid];
        sums[tid] = s_timeout ? CUDART_NAN : total;
    }
    __syncthreads();
}

// Row statistics of a class-logit row of type T by 4 lanes with 16-byte loads (C * sizeof(T) % 16 == 0, aligned rows).
template <typename T>
__device__ __forceinline__ void row_softmax_stats4t(const T *__restrict__ z, int C, int gl, float *m_out, float *s_out)
{
    constexpr int N = Vec16<T>::N;
    const int CV = C / N;
    float m = -CUDART_INF_F;
    for (int v = gl; v < CV; v += 4) {
        float q[N];
        ld_vec16(z + v * N, q);
#pragma unroll
        for (int e = 0; e < N; ++e) m = fmaxf(m, q[e]);
    }
    m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 2));
    m = fmaxf(m, __shfl_xor_sync(kFullMask, m, 1));
    float s = 0.f;
    for (int v = gl; v < CV; v += 4) {
        float q[N];
        ld_vec16(z + v * N, q);
#pragma unroll
        for (int e = 0; e < N; ++e) s += __expf(q[e] - m);
    }
    s += __shfl_xor_sync(kFullMask, s, 2);
    s += __shfl_xor_sync(kFullMask, s, 1);
    *m_out = m;
    *s_out = s;
}

// q[i] for a run-time i with the array kept in registers (a compare-and-assign loop is turned back into a local-memory
// index by the compiler): log2(N) rounds of halving selects.
template <int N>
__device__ __forceinline__ float pick_reg(const float (&q)[N], int i)
{
    float a[N];
#pragma unroll
    for (int e = 0; e < N; ++e) a[e] = q[e];
#pragma unroll
    for (int h = N / 2; h >= 1; h >>= 1) {
        const bool hi = (i & h) != 0;
#pragma unroll
        for (int e = 0; e < h; ++e) a[e] = hi ? a[e + h] : a[e];
    }
    return a[0];
}

// The same with 8 lanes per row: every load instruction covers 128 contiguous bytes of a row.  For maps in device memory
// this is no better than 4 lanes; for maps left in PINNED HOST memory (read in place over PCIe) the request size is what
// counts: the link runs out of read tags long before it runs out of bandwidth, and 128-byte reads need half as many.
template <typename T>
__device__ __forceinline__ void row_softmax_stats8t(const T *__restrict__ z, int C, int gl, float *m_out, float *s_out)
{
    constexpr int N = Vec16<T>::N;
    const int CV = C / N;
    float m = -CUDART_INF_F;
    for (int v = gl; v < CV; v += 8) {
        float q[N];
        ld_vec16(z + v * N, q);
#pragma unroll
        for (int e = 0; e < N; ++e) m = fmaxf(m, q[e]);
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
    float s = 0.f;
    for (int v = gl; v < CV; v += 8) {
        float q[N];
        ld_vec16(z + v * N, q);
#pragma unroll
        for (int e = 0; e < N; ++e) s += __expf(q[e] - m);
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    *m_out = m;
    *s_out = s;
}

// EXCHANGE: the last CTA all-reduces the sums over peer memory before it finalizes (multi-GPU); T: map element type
// HOST: the class / box maps live in pinned host memory and the rows are read in place over PCIe (own instantiation, so
// that nothing of it touches the register budget or the schedule of the device-memory kernel)
template <bool EXCHANGE, typename T = float, bool HOST = false>
__global__ void __launch_bounds__(kPosTileThreads, 8) k_pos_loss_tiles(PosTileParams p, ExchangeParams x)
{
    const int host_rows = HOST ? p.host_rows : 0;
    const T *t_cls = reinterpret_cast<const T *>(p.cls), *t_box = reinterpret_cast<const T *>(p.box_raw);
    __shared__ double s_red[2 * 32];
    __shared__ bool s_last;
    const int tid = threadIdx.x;
    // the first descriptor is fetched together with the list length (stale entries are harmless: they are
    // only used when blockIdx.x < n_chunks)
    // pos_chunks == NULL: a shard without a single image still takes part in the exchange (it pushes its zero sums)
    int desc = p.pos_chunks != nullptr ? __ldg(p.pos_chunks + blockIdx.x) : 0;
    const int n_chunks = p.pos_chunks != nullptr ? (int)p.sums[7] : 0;
    const int A = p.num_anchors;
    float acc_box = 0.f, acc_cls = 0.f;
    if (p.cls == nullptr || p.cls_vec4) {
        // WARP per chunk (the common case: class rows readable 16 bytes at a time).  Lane = row for everything that is
        // per row — list entry, gt / class target, the whole CIoU term (all 32 lanes busy, where a CTA per chunk kept
        // 96 of 128 threads idle through the ~300-instruction box loss) and the final cross-entropy — and 4 lanes per
        // row, 8 rows per pass, for the class-row statistics.  One dependent chain per chunk (descriptor -> list
        // entries -> targets + rows), four chunks in flight per CTA.
        const int lane = tid & 31, warp = tid >> 5;
        constexpr int kWarps = kPosTileThreads / 32;
        const int gl4 = lane & 3, grp8 = lane >> 2;
        for (int w = (int)blockIdx.x * kWarps + warp; w < n_chunks; w += (int)gridDim.x * kWarps) {
            const int d = (w == (int)blockIdx.x && warp == 0) ? desc : __ldg(p.pos_chunks + w);
            const int slot = d >> 10, r_begin = ((d >> 6) & 15) * 32, n = (d & 63) + 1;
            const int b = slot / p.n_tiles;
            const bool mine = lane < n;
            const int32_t flat = __ldg(p.tile_pos_rows + (int64_t)slot * kTile + r_begin + (mine ? lane : 0));
            const int2 ga = __ldg(p.tile_pos_aux + (int64_t)slot * kTile + r_begin + (mine ? lane : 0));
            const float wgt = __int_as_float(ga.y);
            // host-resident maps: the raw box is REQUESTED here and USED after the class rows have been requested too —
            // one PCIe round trip per chunk instead of two back to back (the sums do not depend on the order)
            const bool do_box = p.box_raw != nullptr && mine;
            float4 raw = make_float4(0.f, 0.f, 0.f, 0.f);
            if (do_box) raw = ldf4(t_box + 4 * (int64_t)flat);
            if (!HOST && do_box) {
                const int a = flat - b * A;
                acc_box += wgt * pos_box_loss(raw, __ldg(p.offsets + a), __ldg(p.scales + a),
                                              __ldg(p.gt_boxes + ga.x), p.img_w, p.img_h);                  // ref :197
            }
            if (p.cls != nullptr) {
                const int64_t tgt64 = __ldg(p.gt_classes + ga.x);
                const bool tgt_ok = tgt64 >= 0 && tgt64 < p.num_classes;   // out-of-range label: NaN loss, no foreign read
                float my_m = 0.f, my_se = 1.f, my_zt = 0.f;
                if (host_rows == 2) {
                    // WHOLE ROW PER WARP INSTRUCTION (host-resident rows of at most 32 16-byte vectors): lane v loads
                    // vector v, R rows in flight per warp, and the row crosses the bus ONCE — the statistics and the
                    // target's logit come from registers.  tools/micro/host_gather_bw.cu: 48.8 GB/s of the link's 55
                    // for 320-byte rows, against 37-45 GB/s for 8 lanes x 16 B.
                    constexpr int N = Vec16<T>::N, R = N == 4 ? 4 : 2;
                    const int CV = p.num_classes / N;
                    const int tgt_i = tgt_ok ? (int)tgt64 : 0;
                    for (int r0 = 0; r0 < n; r0 += R) {                    // n is warp-uniform
                        float q[R][N];
#pragma unroll
                        for (int k = 0; k < R; ++k) {
                            const int r = r0 + k;
                            const int32_t rflat = __shfl_sync(kFullMask, flat, r < n ? r : 0);
                            if (lane < CV && r < n) ld_vec16(t_cls + (int64_t)rflat * p.num_classes + lane * N, q[k]);
                            else {
#pragma unroll
                                for (int e = 0; e < N; ++e) q[k][e] = -CUDART_INF_F;
                            }
                        }
#pragma unroll
                        for (int k = 0; k < R; ++k) {
                            const int r = r0 + k;
                            if (r >= n) continue;                          // warp-uniform
                            float m = q[k][0];
#pragma unroll
                            for (int e = 1; e < N; ++e) m = fmaxf(m, q[k][e]);
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
                            float se = 0.f;
                            if (lane < CV) {
#pragma unroll
                                for (int e = 0; e < N; ++e) se += __expf(q[k][e] - m);
                            }
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(kFullMask, se, o);
                            const int t = __shfl_sync(kFullMask, tgt_i, r);
                            const float zt = __shfl_sync(kFullMask, pick_reg<N>(q[k], t & (N - 1)), t / N);
                            if (lane == r) { my_m = m; my_se = se; my_zt = zt; }
                        }
                    }
                } else if (host_rows) {                                  // 8 lanes per row, 4 rows per pass (see row_softmax_stats8t)
                    const int gl8 = lane & 7, grp4 = lane >> 3;
#pragma unroll
                    for (int pass = 0; pass < 8; ++pass) {
                        if (pass * 4 >= n) break;                          // warp-uniform
                        const int r = pass * 4 + grp4;
                        const int32_t rflat = __shfl_sync(kFullMask, flat, r < n ? r : 0);
                        float m, se;
                        row_softmax_stats8t<T>(t_cls + (int64_t)rflat * p.num_classes, p.num_classes, gl8, &m, &se);
                        const float m_r = __shfl_sync(kFullMask, m, 8 * (lane & 3)), se_r = __shfl_sync(kFullMask, se, 8 * (lane & 3));
                        if ((lane >> 2) == pass) { my_m = m_r; my_se = se_r; }
                    }
                } else
#pragma unroll
                for (int pass = 0; pass < 4; ++pass) {
                    if (pass * 8 >= n) break;                              // warp-uniform
                    const int r = pass * 8 + grp8;
                    const int32_t rflat = __shfl_sync(kFullMask, flat, r < n ? r : 0);
                    float m, se;
                    if constexpr (sizeof(T) == 4)
                        row_softmax_stats4v<true>(reinterpret_cast<const float *>(p.cls) + (int64_t)rflat * p.num_classes,
                                                  p.num_classes, gl4, &m, &se);
                    else
                        row_softmax_stats4t<T>(t_cls + (int64_t)rflat * p.num_classes, p.num_classes, gl4, &m, &se);
                    // hand the statistics of row r to lane r (its group sits at lanes 4 * (r & 7) .. + 3 of this pass)
                    const float m_r = __shfl_sync(kFullMask, m, 4 * (lane & 7)), se_r = __shfl_sync(kFullMask, se, 4 * (lane & 7));
                    if ((lane >> 3) == pass) { my_m = m_r; my_se = se_r; }
                }
                if (mine) {
                    if (host_rows != 2) my_zt = ldf(t_cls + (int64_t)flat * p.num_classes + (tgt_ok ? (int)tgt64 : 0));
                    const float ce = (logf(my_se) + my_m) - my_zt;
                    acc_cls += wgt * (tgt_ok ? ce : CUDART_NAN_F);                                          // ref :208
                }
            }
            if (HOST && do_box) {
                const int a = flat - b * A;
                acc_box += wgt * pos_box_loss(raw, __ldg(p.offsets + a), __ldg(p.scales + a),
                                              __ldg(p.gt_boxes + ga.x), p.img_w, p.img_h);                  // ref :197
            }
        }
    } else {
    const int lpr = 8;                                            // lanes per positive row (element loads, any C)
    const int gl = tid & (lpr - 1), grp = tid / lpr, ngrp = kPosTileThreads / lpr;
    for (int w = blockIdx.x; w < n_chunks; w += gridDim.x) {
        if (w != (int)blockIdx.x) desc = __ldg(p.pos_chunks + w);
        const int slot = desc >> 10, r_begin = ((desc >> 6) & 15) * 32, n = (desc & 63) + 1;
        const int b = slot / p.n_tiles;
        const int32_t *rows = p.tile_pos_rows + (int64_t)slot * kTile + r_begin;
        const int2 *aux = p.tile_pos_aux + (int64_t)slot * kTile + r_begin;
        if (p.cls != nullptr) {
            for (int r0 = 0; r0 < n; r0 += ngrp) {                // class loss: one round with 4 lanes per row
                const int r = r0 + grp;
                const bool ok = r < n;
                const int64_t flat = __ldg(rows + (ok ? r : 0));
                const int2 ga = __ldg(aux + (ok ? r : 0));
                const int64_t tgt64 = __ldg(p.gt_classes + ga.x);
                const bool tgt_ok = tgt64 >= 0 && tgt64 < p.num_classes;   // out-of-range label: NaN loss, no foreign read
                const int tgt = tgt_ok ? (int)tgt64 : 0;
                float m, se;
                if constexpr (sizeof(T) == 4) {
                    const float *zf = reinterpret_cast<const float *>(p.cls) + flat * p.num_classes;
                    if (p.cls_vec4) row_softmax_stats4v<true>(zf, p.num_classes, gl, &m, &se);
                    else row_softmax_stats8<true>(zf, p.num_classes, gl, &m, &se);
                } else {
                    const T *zt = t_cls + flat * p.num_classes;
                    if (p.cls_vec4) {
                        row_softmax_stats4t<T>(zt, p.num_classes, gl, &m, &se);
                    } else {                                       // 8 lanes, element loads
                        m = -CUDART_INF_F;
                        for (int c = gl; c < p.num_classes; c += 8) m = fmaxf(m, ldf(zt + c));
#pragma unroll
                        for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
                        se = 0.f;
                        for (int c = gl; c < p.num_classes; c += 8) se += __expf(ldf(zt + c) - m);
#pragma unroll
                        for (int o = 4; o > 0; o >>= 1) se += __shfl_xor_sync(kFullMask, se, o);
                    }
                }
                if (ok && gl == 0) {
                    const float ce = (logf(se) + m) - ldf(t_cls + flat * p.num_classes + tgt);
                    acc_cls += __int_as_float(ga.y) * (tgt_ok ? ce : CUDART_NAN_F);         // ref :208
                }
            }
        }
        if (p.box_raw != nullptr && tid < n) {                    // box loss: one lane per row (a chunk has <= 32 rows)
            const int64_t flat = __ldg(rows + tid);
            const int2 ga = __ldg(aux + tid);
            const int a = (int)(flat - (int64_t)b * A);
            acc_box += __int_as_float(ga.y) * pos_box_loss(ldf4(t_box + 4 * flat), __ldg(p.offsets + a), __ldg(p.scales + a),
                                                           __ldg(p.gt_boxes + ga.x), p.img_w, p.img_h);      // ref :197
        }
    }
    }
    double v[2] = {acc_box, acc_cls};
    const int slot_idx[2] = {4, 5};
    block_accumulate<2>(v, s_red, p.sums, slot_idx);
    if (p.losses != nullptr) {                                    // last CTA out computes the five losses
        if (tid == 0) {
            __threadfence();
            s_last = atomicAdd(p.done_counter, 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (EXCHANGE) {
            if (s_last) {                                         // block-uniform: the whole CTA takes part
                __threadfence();
                exchange_sums(x.peer, x.world, x.rank, p.sums, s_red);
            }
        }
        if (s_last && tid == 0) {
            __threadfence();
            finalize_losses(const_cast<const double *>(reinterpret_cast<volatile double *>(p.sums)), p.losses);
            *p.done_counter = 0u;
        }
    }
}

__global__ void k_loss_finalize(const double *__restrict__ sums, float *__restrict__ losses)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) finalize_losses(sums, losses);
}

}  // namespace sihl

using namespace sihl;

extern "C" int sihl_od_loss_finalize(const double *sums, float *losses, void *stream)
{
    SIHL_CHECK_ARG(sums && losses, "NULL argument");
    k_loss_finalize<<<1, 32, 0, (cudaStream_t)stream>>>(sums, losses);
    SIHL_CHECK_LAUNCH("k_loss_finalize");
    return SIHL_OD_OK;
}

extern "C" int sihl_od_pos_loss_tiles(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                                      const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                                      const float *offsets, const float *scales, int img_w, int img_h,
                                      const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                                      const float *box_raw, const float *cls_logits, int num_classes, double *sums,
                                      float *losses, uint32_t *done_counter, void *stream)
{
    return sihl_od_pos_loss_tiles_exchange(pos_chunks, tile_pos_rows, tile_pos_aux, batch, num_anchors, offsets, scales, img_w,
                                           img_h, gt_boxes, gt_classes, gt_offsets, box_raw, cls_logits, num_classes, sums,
                                           losses, done_counter, nullptr, 1, 0, stream);
}

extern "C" int sihl_od_pos_loss_tiles_exchange(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                                               const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                                               const float *offsets, const float *scales, int img_w, int img_h,
                                               const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                                               const float *box_raw, const float *cls_logits, int num_classes, double *sums,
                                               float *losses, uint32_t *done_counter, void *const *peer_regions, int world,
                                               int rank, void *stream)
{
    return sihl_od_pos_loss_tiles_exchange_t(pos_chunks, tile_pos_rows, tile_pos_aux, batch, num_anchors, offsets, scales, img_w,
                                             img_h, gt_boxes, gt_classes, gt_offsets, box_raw, cls_logits, SIHL_OD_F32,
                                             num_classes, sums, losses, done_counter, peer_regions, world, rank, stream);
}

extern "C" int sihl_od_pos_loss_tiles_exchange_t(const int32_t *pos_chunks, const int32_t *tile_pos_rows,
                                                 const int32_t *tile_pos_aux, int batch, int64_t num_anchors,
                                                 const float *offsets, const float *scales, int img_w, int img_h,
                                                 const float *gt_boxes, const int64_t *gt_classes, const int32_t *gt_offsets,
                                                 const void *box_raw, const void *cls_logits, int map_dtype, int num_classes,
                                                 double *sums, float *losses, uint32_t *done_counter,
                                                 void *const *peer_regions, int world, int rank, void *stream)
{
    (void)gt_offsets;
    SIHL_CHECK_ARG(world >= 1 && world <= SIHL_OD_MAX_PEERS && rank >= 0 && rank < world, "world=%d rank=%d", world, rank);
    SIHL_CHECK_ARG(world == 1 || (peer_regions != nullptr && losses != nullptr),
                   "the fused exchange needs the peer regions and the fused finalize (losses, done_counter)");
    SIHL_CHECK_ARG(batch >= 0 && num_anchors >= 0 && num_anchors < (1ll << 30), "bad sizes");
    const bool empty_shard = (int64_t)batch * ((num_anchors + kTile - 1) / kTile) == 0;
    SIHL_CHECK_ARG(sums && (empty_shard || (pos_chunks && tile_pos_rows && tile_pos_aux)), "NULL argument");
    SIHL_CHECK_ARG(box_raw == nullptr || (offsets && scales && img_w > 0 && img_h > 0),
                   "box loss needs offsets, scales and the image size");
    SIHL_CHECK_ARG(cls_logits == nullptr || num_classes > 0, "class loss needs num_classes");
    SIHL_CHECK_ARG((losses == nullptr) == (done_counter == nullptr), "losses and done_counter go together");
    const int n_tiles = (int)((num_anchors + kTile - 1) / kTile);
    const int64_t n_slots = (int64_t)batch * n_tiles;
    // an empty shard has nothing to add, but with peers it must still push its (zero) sums and step number:
    // returning here would leave every other rank waiting for it until the timeout
    if (n_slots == 0 && world == 1) return SIHL_OD_OK;
    PosTileParams p;
    p.pos_chunks = n_slots == 0 ? nullptr : pos_chunks; p.tile_pos_rows = tile_pos_rows; p.tile_pos_aux = reinterpret_cast<const int2 *>(tile_pos_aux);
    p.n_tiles = n_tiles; p.num_anchors = (int)num_anchors;
    p.offsets = reinterpret_cast<const float4 *>(offsets); p.scales = reinterpret_cast<const float4 *>(scales);
    p.img_w = (float)img_w; p.img_h = (float)img_h;
    p.gt_boxes = reinterpret_cast<const float4 *>(gt_boxes); p.gt_classes = gt_classes; p.gt_offsets = gt_offsets;
    p.box_raw = box_raw; p.cls = cls_logits; p.num_classes = num_classes;
    const int esz = map_dtype == SIHL_OD_F32 ? 4 : 2;
    p.cls_vec4 = (((size_t)num_classes * esz) % 16 == 0) && ((reinterpret_cast<uintptr_t>(cls_logits) & 15u) == 0);
    SIHL_CHECK_ARG(box_raw == nullptr || (reinterpret_cast<uintptr_t>(box_raw) & (4 * esz - 1)) == 0, "box_raw rows must be aligned");
    p.sums = sums; p.losses = losses; p.done_counter = done_counter;
    p.host_rows = 0;
    const void *host_ok_maps[2] = {cls_logits, box_raw};
    for (const void *map : host_ok_maps) {               // pageable host memory would fault in the kernel: refuse it here
        cudaPointerAttributes attr;
        if (map == nullptr) continue;
        if (cudaPointerGetAttributes(&attr, map) != cudaSuccess) { (void)cudaGetLastError(); continue; }
        SIHL_CHECK_ARG(attr.type != cudaMemoryTypeUnregistered,
                       "box_raw / cls_logits must be device memory or PINNED host memory (got a pageable host pointer)");
        if (map == cls_logits) p.host_rows = attr.type == cudaMemoryTypeHost;
    }
    if (!p.cls_vec4) p.host_rows = 0;
    // pinned host maps (zero-copy) take wider row reads: 2 = whole row per warp instruction (rows of at most 32
    // vectors), 1 = 8 lanes x 16 B
    if (p.host_rows && (size_t)num_classes * esz <= 32 * 16) p.host_rows = 2;
    ExchangeParams x;
    x.world = world; x.rank = rank;
    x.peer = reinterpret_cast<unsigned long long *const *>(peer_regions);
    // persistent grid: up to 12 CTAs of 128 threads per SM, never more than the chunk-list capacity
    int64_t blocks = n_slots * (kTile / 32);
    // 6 persistent CTAs per SM (2-3 chunks each at cfg1), not the 12 the launch bounds allow: every CTA ends with two
    // fp64 atomics on one 64-byte line + the completion ticket, and ~1800 of those serialise in one L2 slice.  Measured
    // in the cfg1 pipeline (same box A/B): 12 -> 41.6 / 28.2 us per step (dense / candidate-first), 6 -> 40.8 / 25.6,
    // 4 -> 40.6 / 26.0.
    const int64_t cap = (int64_t)kNumSMs * 6;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (p.host_rows) {
        if (world > 1) SIHL_DISPATCH_DTYPE(map_dtype, (k_pos_loss_tiles<true, T, true><<<(unsigned)blocks, kPosTileThreads, 0, (cudaStream_t)stream>>>(p, x)));
        else SIHL_DISPATCH_DTYPE(map_dtype, (k_pos_loss_tiles<false, T, true><<<(unsigned)blocks, kPosTileThreads, 0, (cudaStream_t)stream>>>(p, x)));
    } else if (world > 1) SIHL_DISPATCH_DTYPE(map_dtype, (k_pos_loss_tiles<true, T><<<(unsigned)blocks, kPosTileThreads, 0, (cudaStream_t)stream>>>(p, x)));
    else SIHL_DISPATCH_DTYPE(map_dtype, (k_pos_loss_tiles<false, T><<<(unsigned)blocks, kPosTileThreads, 0, (cudaStream_t)stream>>>(p, x)));
    SIHL_CHECK_LAUNCH("k_pos_loss_tiles");
    return SIHL_OD_OK;
}
