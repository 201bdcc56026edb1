// Row N4 (SURVEY.md §8f): the step BEFORE the hot path — the head's per-location MLP towers
// (ref src/sihl/heads/object_detection.py:51-61 builds four torchvision ``ops.MLP(256 -> [256]*4 + [out],
// norm_layer=LayerNorm, activation_layer=SiLU)``; :116 / :121 / :175 apply them to every location).  One tower layer is
//
//     hidden:  y = SiLU(LayerNorm(x W^T + b) * gamma + beta)     x [M,256] bf16, W [256,256] bf16, y [M,256] bf16
//     output:  y = x W^T + b                                     W [n,256] bf16 (n = 1, 4, num_classes), y [M,n] fp32
//
// and this is the one GEMM-shaped piece of the head, so it is the one place the 5th-generation tensor cores are used:
//
//   * W stays resident in shared memory for the life of the (persistent, one-per-SM) CTA — four 64-column K chunks in
//     the 128-byte-swizzled K-major layout `tcgen05.mma` reads through a shared-memory descriptor;
//   * x row tiles (128 rows x 64 columns = 16 KB) stream through a TMA ring (`cp.async.bulk.tensor.2d`, hardware
//     swizzle, mbarrier completion); rows past M are zero-filled by the TMA unit;
//   * one elected thread issues 16 `tcgen05.mma.cta_group::1.kind::f16` (M=128, N, K=16) per tile into one of two
//     TMEM accumulator stages (2 x N fp32 columns), `tcgen05.commit` releases ring slots / publishes the accumulator;
//   * sixteen epilogue warps (hidden layers; four for the narrow output layers) — four per TMEM lane quarter, thread =
//     row, 64 columns each — read their slice of the accumulator ONCE with `tcgen05.ld` into registers (which frees the
//     TMEM stage for the tile after next at once), add the bias, take the slice's sum and centred sum of squares,
//     combine the four slices of a row through one shared-memory exchange per tile (parallel-variance formula),
//     normalise, apply SiLU as h + h*tanh(h) (h = z/2: one MUFU op per element), round to bf16, and store.  The
//     arithmetic is packed fp32x2 (FADD2 / FMUL2 / FFMA2).  Stores: a thread's 128-byte piece of its row is 4 x 4
//     transposed inside the lane quad (SHFL.BFLY) so that every 256-bit store instruction of a warp writes 8 complete
//     128-byte lines instead of touching 32 (L1 wavefronts per tile: 512 instead of 2 048; measured 9.0k -> 7.6k
//     cycles per tile).
//
// A hidden layer reads 512 B and writes 512 B per location for 131 kFLOP: at M = 545 600 (640^2, batch 64) that is
// 559 MB and 71.5 GFLOP per layer — HBM-bound at ~87 us, a third of what the unfused Linear + LayerNorm + SiLU kernels
// move; measured 124 us (4.5 TB/s, 577 TFLOP/s): what is left is the epilogue's MIO work per tile (MUFU, LDS, stores),
// see DESIGN.md.  Every wait is bounded: a pipeline bug traps instead of hanging the GPU.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>

#include "../../include/sihl_od.h"

namespace {

constexpr int kK = 256;                       // in_features of every tower layer (the reference's num_channels default)
constexpr int kBlockM = 128;                  // rows per tile = TMEM lanes
constexpr int kChunkK = 64;                   // bf16 per 128-byte swizzle row
constexpr int kChunks = kK / kChunkK;         // 4
constexpr int kUmmaK = 16;                    // K per tcgen05.mma (bf16)
constexpr int kXStageBytes = kBlockM * 128;   // one ring slot: 128 rows x 128 B
constexpr int kThreads = 576;                 // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-17: epilogue
constexpr int kParts = 4;                     // epilogue warps per TMEM lane quarter of a hidden layer
constexpr int kPartCols = 64;                 // columns each of them owns (held in registers for the whole epilogue)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: ~2 s of polling, then trap (a launch failure the host sees) — never a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int what) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("sihl_od_mlp: barrier wait timed out (block %d thread %d wait-site %d parity %u)\n", blockIdx.x, threadIdx.x, what, parity);
            __trap();
        }
    }
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n"
        ".reg .b32 rx;\n"
        ".reg .pred px;\n"
        "elect.sync rx|px, %1;\n"
        "@px mov.s32 %0, 1;\n"
        "}\n"
        : "+r"(pred)
        : "r"(0xFFFFFFFFu));
    return pred != 0;
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, both operands K-major bf16, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Shared-memory matrix descriptor: K-major tile of 128-byte rows, 128-byte swizzle, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t sw128_kmajor_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);     // start address, 16-byte units        bits [0,14)
    d |= static_cast<uint64_t>(1) << 16;                     // leading byte offset (unused here)   bits [16,30)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;             // stride byte offset: 8 rows x 128 B  bits [32,46)
    d |= static_cast<uint64_t>(1) << 46;                     // descriptor version (Blackwell)      bits [46,48)
    d |= static_cast<uint64_t>(2) << 61;                     // SWIZZLE_128B                        bits [61,64)
    return d;
}
// Instruction descriptor of kind::f16: fp32 accumulator, bf16 A and B, both K-major, shape 128 x N.
template <int N>
__host__ __device__ constexpr uint32_t idesc_bf16_f32() {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(kBlockM >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&v)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]), "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]),
          "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]),
          "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]),
          "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

// ---- packed fp32x2 arithmetic (sm_100: two fp32 lanes per instruction) and small epilogue helpers ----------------------
__device__ __forceinline__ uint64_t pack2(uint32_t lo, uint32_t hi) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ uint64_t pack2f(float lo, float hi) { return pack2(__float_as_uint(lo), __float_as_uint(hi)); }
__device__ __forceinline__ float lo_of(uint64_t v) { return __uint_as_float(static_cast<uint32_t>(v)); }
__device__ __forceinline__ float hi_of(uint64_t v) { return __uint_as_float(static_cast<uint32_t>(v >> 32)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float tanh_fast(float x) { float r; asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ uint32_t bf16x2_of(uint64_t v) {
    const __nv_bfloat162 b = __floats2bfloat162_rn(lo_of(v), hi_of(v));
    return *reinterpret_cast<const uint32_t*>(&b);
}
__device__ __forceinline__ void st_global_256(void* dst, const uint32_t* v) {      // one full 32-byte sector per lane
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]),
                 "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }   // the sixteen epilogue warps only

__host__ __device__ constexpr int tmem_stage_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : 256; }

template <int N>
struct MlpSmem {
    static constexpr int kStages = (N == 256) ? 5 : 8;      // N == 256: W takes 128 KB of the 227
    static constexpr int kWBytes = kChunks * N * 128;
    static constexpr int kRingBytes = kStages * kXStageBytes;
    static constexpr int kParamBytes = 3 * N * 4 + 2 * 2 * kParts * kBlockM * 4;   // bias, gamma/2, beta/2 + two row-statistics exchange buffers
    static constexpr int kBarBytes = (2 * kStages + 1 + 4) * 8 + 16;
    static constexpr int kTotal = 1024 /* alignment slack */ + kWBytes + kRingBytes + kParamBytes + kBarBytes;
};

struct MlpParams {
    const float* bias;
    const float* gamma;      // hidden layers only
    const float* beta;       // hidden layers only
    void* out;               // hidden: bf16 [M,N]; output layer: fp32 [M,out_cols]
    long long M;
    int n_tiles;
    int out_cols;
    float eps;
    float* row_stats;               // kHidden, optional: [M,2] = (mean, rstd) of every row's LayerNorm, kept for the backward
    void* pre_out;                  // kHiddenPre: bf16 [M,N] = x W^T + bias, the pre-activation, kept for the backward
    long long rows_per_image;       // kLinear: see the row formula above
    long long out_rows_per_image;
    long long out_row_offset;
};

// MODE kHidden:  bias + LayerNorm + SiLU -> bf16 [M,N]   (N == 256; the towers' hidden layers)
// MODE kOutF32:  bias                    -> fp32 [M,out_cols], out_cols <= N   (the towers' last Linear)
// MODE kLinear:  bias                    -> bf16 rows of N == 256, row m written at
//                (m / rows_per_image) * out_rows_per_image + out_row_offset + m % rows_per_image   (the laterals: 1x1 conv
//                with the BatchNorm folded in, each level landing in its slice of the concatenated [B, A, 256] features)
// MODE kHiddenPre: kHidden that also stores the pre-activation (bf16) -> the training backward does not recompute it
constexpr int kHidden = 0, kOutF32 = 1, kLinear = 2, kHiddenPre = 3;
template <int N, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
k_mlp_layer(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const MlpParams p) {
    using L = MlpSmem<N>;
    constexpr bool HIDDEN = MODE == kHidden || MODE == kHiddenPre;
    constexpr bool WIDE = MODE != kOutF32;                // sixteen epilogue warps, bf16 rows of 256
    static_assert(!WIDE || N == 256, "the wide epilogue is built for 256 output columns");
    constexpr int S = L::kStages;
    constexpr int kStageCols = tmem_stage_cols(N);
    constexpr int kTmemCols = 2 * kStageCols;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // the swizzle atoms need 1024-byte alignment
    uint8_t* sW = base;                                   // 4 chunks x [N rows x 128 B], swizzled by the TMA unit
    uint8_t* sX = sW + L::kWBytes;                        // ring of [128 rows x 128 B] slots
    float* sBias = reinterpret_cast<float*>(sX + L::kRingBytes);
    float* sGamma = sBias + N;
    float* sBeta = sGamma + N;
    float* sStat = sBeta + N;                             // [tile parity][sum | M2][part][row]
    uint64_t* full = reinterpret_cast<uint64_t*>(sStat + 2 * 2 * kParts * kBlockM);
    uint64_t* empty = full + S;
    uint64_t* w_full = empty + S;
    uint64_t* t_full = w_full + 1;                        // [2] accumulator stage ready for the epilogue
    uint64_t* t_empty = t_full + 2;                       // [2] accumulator stage drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < N; i += kThreads) {
        sBias[i] = p.bias[i];
        sGamma[i] = HIDDEN ? 0.5f * p.gamma[i] : 1.f;     // the 1/2 of SiLU's tanh form folded in (exact)
        sBeta[i] = HIDDEN ? 0.5f * p.beta[i] : 0.f;
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(w_full, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], WIDE ? 4 * kParts : 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {                                      // TMEM: one warp allocates and later frees
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (elect_one()) {
            mbar_expect_tx(w_full, L::kWBytes);
            for (int c = 0; c < kChunks; ++c) tma_load_2d(&map_w, w_full, sW + c * (N * 128), c * kChunkK, 0);
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
                for (int c = 0; c < kChunks; ++c, ++it) {
                    const uint32_t s = it % S, ph = (it / S) & 1;
                    mbar_wait(&empty[s], ph ^ 1, 0);
                    mbar_expect_tx(&full[s], kXStageBytes);
                    tma_load_2d(&map_x, &full[s], sX + s * kXStageBytes, c * kChunkK, tile * kBlockM);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one()) {
            constexpr uint32_t idesc = idesc_bf16_f32<N>();
            mbar_wait(w_full, 0, 1);
            uint32_t it = 0, t = 0;
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
                const uint32_t as = t & 1, aph = (t >> 1) & 1;
                mbar_wait(&t_empty[as], aph ^ 1, 2);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * kStageCols;
                for (int c = 0; c < kChunks; ++c, ++it) {
                    const uint32_t s = it % S, ph = (it / S) & 1;
                    mbar_wait(&full[s], ph, 3);
                    tc_fence_after();
                    const uint32_t a_base = smem_u32(sX + s * kXStageBytes);
                    const uint32_t b_base = smem_u32(sW + c * (N * 128));
#pragma unroll
                    for (int k = 0; k < kChunkK / kUmmaK; ++k) {
                        tc_mma_bf16(d_tmem, sw128_kmajor_desc(a_base + k * (kUmmaK * 2)), sw128_kmajor_desc(b_base + k * (kUmmaK * 2)), idesc,
                                    static_cast<uint32_t>((c | k) != 0));
                    }
                    tc_commit(&empty[s]);                 // ring slot free once these MMAs have read it
                }
                tc_commit(&t_full[as]);                   // accumulator complete
            }
        }
    } else if (WIDE || warp < 6) {
        // ===== epilogue: warp w may touch TMEM lanes 32*(w%4) .. +31; thread = row.  Hidden layers: sixteen warps, the
        // four warps of a lane quarter own 64 columns each, read them from TMEM ONCE into registers (which frees the
        // accumulator stage at once) and exchange their partial row statistics through shared memory; the arithmetic
        // is packed fp32x2 (FADD2 / FMUL2 / FFMA2: two columns per issue slot). =====
        const int quarter = warp & 3;
        const int part = (warp - 2) >> 2;
        const int row = quarter * 32 + lane;
        uint32_t t = 0;
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++t) {
            const uint32_t as = t & 1, aph = (t >> 1) & 1;
            mbar_wait(&t_full[as], aph, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * kStageCols;
            const long long grow = static_cast<long long>(tile) * kBlockM + row;
            if constexpr (WIDE) {
                const int cbase = part * kPartCols;
                // store: a thread holds one 128-byte line of its row as four 32-byte pieces.  Written as they are, a
                // warp-wide 32-byte store touches 32 different lines (32 L1 wavefronts); a 4 x 4 transpose of the pieces
                // inside every lane quad (two butterfly steps of SHFL.BFLY) makes lanes 4g..4g+3 hold the four pieces
                // of ONE row, so each store instruction writes 8 complete lines.
                auto store_rows = [&](uint32_t (&pk)[kPartCols / 2], __nv_bfloat16* out, bool mapped) {
                    const bool b0 = lane & 1, b1 = lane & 2;
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
#pragma unroll
                        for (int j = 0; j < 4; j += 2) {                   // step 1: partner lane ^ 1 swaps pieces (j, j+1)
                            const uint32_t send = b0 ? pk[8 * j + r] : pk[8 * (j + 1) + r];
                            const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 1);
                            if (b0) pk[8 * j + r] = recv; else pk[8 * (j + 1) + r] = recv;
                        }
#pragma unroll
                        for (int j = 0; j < 2; ++j) {                      // step 2: partner lane ^ 2 swaps pieces (j, j+2)
                            const uint32_t send = b1 ? pk[8 * j + r] : pk[8 * (j + 2) + r];
                            const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 2);
                            if (b1) pk[8 * j + r] = recv; else pk[8 * (j + 2) + r] = recv;
                        }
                    }
                    // now piece k of this lane = columns [16 q, 16 q + 16) (q = lane & 3) of row (lane & ~3) + k
                    const long long qrow = static_cast<long long>(tile) * kBlockM + quarter * 32 + (lane & ~3);
                    __nv_bfloat16* obase = out + cbase + 16 * (lane & 3);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const long long m = qrow + k;
                        if (m < p.M) {
                            long long orow_k = m;
                            if (mapped) {
                                const long long img = m / p.rows_per_image;
                                orow_k = img * p.out_rows_per_image + p.out_row_offset + (m - img * p.rows_per_image);
                            }
                            st_global_256(obase + orow_k * N, pk + 8 * k);
                        }
                    }
                };
                if constexpr (MODE == kHiddenPre) {
                    // first pass over the accumulator: v = bf16(x W^T + bias), the pre-activation the backward needs.  The
                    // accumulator is read from TMEM again below rather than kept: 64 more live registers would spill, the
                    // second tcgen05.ld costs a few hundred cycles, and the TMEM stage is not needed before tile t + 2.
                    uint32_t v0[kPartCols];
                    tmem_ld64(taddr + cbase, v0);
                    uint32_t pk0[kPartCols / 2];
#pragma unroll
                    for (int j = 0; j < kPartCols; j += 4) {
                        const ulonglong2 b4 = *reinterpret_cast<const ulonglong2*>(&sBias[cbase + j]);
                        pk0[j >> 1] = bf16x2_of(add2(pack2(v0[j], v0[j + 1]), b4.x));
                        pk0[(j >> 1) + 1] = bf16x2_of(add2(pack2(v0[j + 2], v0[j + 3]), b4.y));
                    }
                    store_rows(pk0, reinterpret_cast<__nv_bfloat16*>(p.pre_out), false);
                }
                uint32_t v[kPartCols];
                tmem_ld64(taddr + cbase, v);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&t_empty[as]);              // the accumulator stage is free for tile t + 2
                uint64_t x[kPartCols / 2];
                // statistics of the thread's own 64 columns: x = acc + bias, sum, then the sum of squares about the
                // LOCAL mean (two passes over registers, no synchronisation in between)
                uint64_t s2a = 0, s2b = 0;
#pragma unroll
                for (int j = 0; j < kPartCols; j += 4) {
                    const ulonglong2 b4 = *reinterpret_cast<const ulonglong2*>(&sBias[cbase + j]);
                    x[j >> 1] = add2(pack2(v[j], v[j + 1]), b4.x);
                    x[(j >> 1) + 1] = add2(pack2(v[j + 2], v[j + 3]), b4.y);
                    s2a = add2(s2a, x[j >> 1]);
                    s2b = add2(s2b, x[(j >> 1) + 1]);
                }
                uint32_t packed[kPartCols / 2];
                if constexpr (HIDDEN) {
                const float sum_p = (lo_of(s2a) + hi_of(s2a)) + (lo_of(s2b) + hi_of(s2b));
                const float mean_p = sum_p * (1.f / kPartCols);
                const uint64_t mean_p2 = pack2f(mean_p, mean_p);
                uint64_t q2a = 0, q2b = 0;
#pragma unroll
                for (int j = 0; j < kPartCols / 2; j += 2) {
                    const uint64_t d0 = sub2(x[j], mean_p2), d1 = sub2(x[j + 1], mean_p2);
                    q2a = fma2(d0, d0, q2a);
                    q2b = fma2(d1, d1, q2b);
                }
                // one exchange per tile (buffers alternate with the tile parity): the four column slices of a row are
                // combined with the parallel-variance formula  M2 = sum_q [ M2_q + n_q (mean_q - mean)^2 ]
                float* stat = sStat + (t & 1) * (2 * kParts * kBlockM);
                stat[(0 * kParts + part) * kBlockM + row] = sum_p;
                stat[(1 * kParts + part) * kBlockM + row] = (lo_of(q2a) + hi_of(q2a)) + (lo_of(q2b) + hi_of(q2b));
                epi_sync();
                float sums[kParts], mean = 0.f, m2 = 0.f;
#pragma unroll
                for (int q = 0; q < kParts; ++q) {
                    sums[q] = stat[(0 * kParts + q) * kBlockM + row];
                    mean += sums[q];
                    m2 += stat[(1 * kParts + q) * kBlockM + row];
                }
                mean *= (1.f / N);
#pragma unroll
                for (int q = 0; q < kParts; ++q) {
                    const float dm = sums[q] * (1.f / kPartCols) - mean;
                    m2 = __fmaf_rn(dm * dm, static_cast<float>(kPartCols), m2);
                }
                const float rstd = 1.f / sqrtf(m2 * (1.f / N) + p.eps);
                if (p.row_stats != nullptr && part == 0 && grow < p.M)
                    *reinterpret_cast<float2*>(p.row_stats + 2 * grow) = make_float2(mean, rstd);
                const uint64_t mean2 = pack2f(mean, mean);
                const uint64_t rstd2 = pack2f(rstd, rstd);
                // normalise, SiLU, round to bf16: the thread's 64 columns are one 128-byte line of the output row
#pragma unroll
                for (int j = 0; j < kPartCols; j += 4) {
                    const ulonglong2 g4 = *reinterpret_cast<const ulonglong2*>(&sGamma[cbase + j]);     // gamma / 2
                    const ulonglong2 e4 = *reinterpret_cast<const ulonglong2*>(&sBeta[cbase + j]);      // beta / 2
                    // h = SiLU argument / 2;  SiLU(z) = z * sigmoid(z) = h + h * tanh(h): one MUFU op per element
                    const uint64_t h0 = fma2(mul2(sub2(x[j >> 1], mean2), rstd2), g4.x, e4.x);
                    const uint64_t h1 = fma2(mul2(sub2(x[(j >> 1) + 1], mean2), rstd2), g4.y, e4.y);
                    const uint64_t y0 = fma2(h0, pack2f(tanh_fast(lo_of(h0)), tanh_fast(hi_of(h0))), h0);
                    const uint64_t y1 = fma2(h1, pack2f(tanh_fast(lo_of(h1)), tanh_fast(hi_of(h1))), h1);
                    packed[j >> 1] = bf16x2_of(y0);
                    packed[(j >> 1) + 1] = bf16x2_of(y1);
                }
                } else {
#pragma unroll
                    for (int j = 0; j < kPartCols / 2; ++j) packed[j] = bf16x2_of(x[j]);       // kLinear: bias only
                }
                store_rows(packed, reinterpret_cast<__nv_bfloat16*>(p.out), MODE == kLinear);
                continue;                                              // t_empty was signalled right after the load
            } else {
                uint32_t v[16];
                float* orow = reinterpret_cast<float*>(p.out) + grow * p.out_cols;
                const bool vec4 = (p.out_cols & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15u) == 0;
#pragma unroll 1
                for (int c0 = 0; c0 < N; c0 += 16) {
                    if (c0 >= p.out_cols) break;                                   // padded columns: nothing to write
                    tmem_ld16(taddr + c0, v);
                    if (grow < p.M) {
                        if (vec4) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4)
                                if (c0 + j < p.out_cols)
                                    *reinterpret_cast<float4*>(orow + c0 + j) =
                                        make_float4(__uint_as_float(v[j]) + sBias[c0 + j], __uint_as_float(v[j + 1]) + sBias[c0 + j + 1],
                                                    __uint_as_float(v[j + 2]) + sBias[c0 + j + 2], __uint_as_float(v[j + 3]) + sBias[c0 + j + 3]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (c0 + j < p.out_cols) orow[c0 + j] = __uint_as_float(v[j]) + sBias[c0 + j];
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_empty[as]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// NCHW fp32 feature map -> rows of channels in bf16: x [B, C, HW] -> y [B * HW, C] (the A operand of the lateral GEMM).
// 64 x 64 tiles through shared memory: reads coalesced along HW, 16-byte writes coalesced along C.  HBM-bound (6 B / element).
__global__ void __launch_bounds__(256) k_nchw_to_rows_bf16(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, long long HW) {
    __shared__ float tile[64][65];
    const long long hw0 = static_cast<long long>(blockIdx.x) * 64;
    const int c0 = blockIdx.y * 64;
    const float* xb = x + static_cast<long long>(blockIdx.z) * C * HW;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;                 // 64 x 4
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const int c = ty + 4 * r;
        tile[c][tx] = (hw0 + tx < HW) ? xb[static_cast<long long>(c0 + c) * HW + hw0 + tx] : 0.f;
    }
    __syncthreads();
    const int chunk = threadIdx.x & 7, rr = threadIdx.x >> 3;               // 8 chunks of 8 channels x 32 rows per pass
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        const int h = rr + 32 * pass;
        if (hw0 + h < HW) {
            uint32_t w4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const __nv_bfloat162 b2 = __floats2bfloat162_rn(tile[chunk * 8 + 2 * q][h], tile[chunk * 8 + 2 * q + 1][h]);
                w4[q] = *reinterpret_cast<const uint32_t*>(&b2);
            }
            __nv_bfloat16* dst = y + (static_cast<long long>(blockIdx.z) * HW + hw0 + h) * C + c0 + chunk * 8;
            *reinterpret_cast<uint4*>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
        }
    }
}

// Backward of LayerNorm + SiLU for the towers' training path, lane = 8 columns.
//   n = (v - mean) rstd, z = n gamma + beta, dz = dy * SiLU'(z), dn = dz gamma,
//   dv = rstd (dn - mean_j(dn) - n mean_j(dn n));  column sums of dz n, dz, dv = d gamma, d beta, d bias
// v is the layer's pre-activation (x W^T + b in bf16: kept by the forward, MODE kHiddenPre, or recomputed by the linear mode
// of the layer kernel), (mean, rstd) come from the forward.  Every CTA writes its partial column sums to partials[blockIdx.x][3][256] (summed by the caller:
// deterministic, no atomics).  HBM-bound: 2 x 512 B read + 512 B written per row.
//
// RANK1: the layer is the tower's LAST hidden layer and the Linear behind it has ONE output (the location and the IoU
// tower, ref :56, :60), so the upstream gradient is the outer product dy[m,:] = bf16(dout[m]) * w_out[:] (rounded to bf16
// like the library GEMM it replaces would): read as 4 B per row + one weight row instead of a materialised [M,256] matrix.
constexpr int kBwdWarps = 8;
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// The rows are streamed through a shared-memory ring by the TMA unit.  The register-staged design this replaced (one warp
// per row, two rows' loads in flight per warp) held ~106 registers per thread, so two CTAs = 16 warps fit on an SM and every
// warp's loads were exposed once per iteration: measured 200 us per [537 600, 256] layer = 4.1 TB/s for 825 MB.  Here the
// TMA unit keeps kRingStages x 32 rows of v and dy (one contiguous cp.async.bulk each, completion on an mbarrier) in
// flight per CTA regardless of what the warps hold in registers; the eight warps take 4 rows each per stage (lane = 8 columns, conflict-free LDS.128) and hand the stage back through an
// `empty` mbarrier; thread 0 refills a stage at the top of the next iteration (a ninth, dedicated producer warp would cap
// the kernel at 96 registers per thread and spill).  Row statistics (8 B per row) and, RANK1, dout (4 B per row) are plain broadcast loads one
// stage ahead.  Same arithmetic, and the same row -> (CTA, warp) order for both variants of RANK1, so they stay bit-equal.
constexpr int kRingRows = 32;
constexpr int kRingStages = 3;
constexpr int kRingThreads = kBwdWarps * 32;
constexpr int kRingArrBytes = kRingRows * kK * 2;                           // 16 KB: 32 rows of one operand
template <bool RANK1> __host__ __device__ constexpr int ring_stage_bytes() { return RANK1 ? kRingArrBytes : 2 * kRingArrBytes; }
template <bool RANK1> __host__ __device__ constexpr int ring_smem_bytes() { return kRingStages * ring_stage_bytes<RANK1>() + 2 * kRingStages * 8 + 128; }
static_assert(kRingStages * kRingArrBytes >= kBwdWarps * 3 * kK * 4, "the final reduction reuses the ring");

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}

template <bool RANK1>
__global__ void __launch_bounds__(kRingThreads, 2) k_mlp_hidden_bwd_ring(const __nv_bfloat16* __restrict__ v, const __nv_bfloat16* __restrict__ dy,
                                                                          const float* __restrict__ dout, const __nv_bfloat16* __restrict__ w_out,
                                                                          const float* __restrict__ row_stats, const float* __restrict__ gamma,
                                                                          const float* __restrict__ beta, long long M, __nv_bfloat16* __restrict__ dv,
                                                                          float* __restrict__ partials) {
    extern __shared__ uint8_t ring_raw[];
    uint8_t* ring = ring_raw + ((128u - (smem_u32(ring_raw) & 127u)) & 127u);
    constexpr int kStageBytes = ring_stage_bytes<RANK1>();
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + kRingStages * kStageBytes);
    uint64_t* empty = full + kRingStages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_chunks = static_cast<int>((M + kRingRows - 1) / kRingRows);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kRingStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kBwdWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int c0 = lane * 8;
    uint64_t acc_g2[4], acc_b2[4], acc_v2[4];                    // columns (c0 + 2q, c0 + 2q + 1)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc_g2[q] = acc_b2[q] = acc_v2[q] = 0ull;

    auto issue = [&](int stage, int c) {                         // thread 0 only
        const long long row0 = static_cast<long long>(c) * kRingRows;
        const uint32_t bytes = static_cast<uint32_t>((M - row0 < kRingRows ? M - row0 : kRingRows) * kK * 2);
        mbar_expect_tx(&full[stage], RANK1 ? bytes : 2 * bytes);
        bulk_g2s(ring + stage * kStageBytes, v + row0 * kK, bytes, &full[stage]);
        if constexpr (!RANK1) bulk_g2s(ring + stage * kStageBytes + kRingArrBytes, dy + row0 * kK, bytes, &full[stage]);
    };
    if (threadIdx.x == 0)
        for (int st0 = 0; st0 < kRingStages; ++st0) {
            const long long c = static_cast<long long>(blockIdx.x) + static_cast<long long>(st0) * gridDim.x;
            if (c < n_chunks) issue(st0, static_cast<int>(c));
        }
    {
        // ===== consumers: warp w owns rows 4w .. 4w+3 of every stage =====
        constexpr int kWarpRows = kRingRows / kBwdWarps;         // 4
        uint64_t g2[4], be2[4], wo2[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            g2[q] = pack2f(gamma[c0 + 2 * q], gamma[c0 + 2 * q + 1]);
            be2[q] = pack2f(beta[c0 + 2 * q], beta[c0 + 2 * q + 1]);
            wo2[q] = RANK1 ? pack2f(__bfloat162float(w_out[c0 + 2 * q]), __bfloat162float(w_out[c0 + 2 * q + 1])) : 0ull;
        }
        float2 st_next[kWarpRows];
        float dc_next[kWarpRows];
        auto load_side = [&](int c) {                           // broadcast loads (every lane the same address), one stage ahead
#pragma unroll
            for (int r = 0; r < kWarpRows; ++r) {
                const long long row = static_cast<long long>(c) * kRingRows + warp * kWarpRows + r;
                const bool ok = c < n_chunks && row < M;
                st_next[r] = ok ? *reinterpret_cast<const float2*>(row_stats + 2 * row) : make_float2(0.f, 0.f);
                dc_next[r] = (RANK1 && ok) ? bf16_round(dout[row]) : 0.f;
            }
        };
        load_side(blockIdx.x);
        int s = 0, rs = -1;                                      // rs: the stage consumed last iteration, to be refilled
        uint32_t ph = 0, rph = 0;
        for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
            if (threadIdx.x == 0 && rs >= 0) {
                const long long cn = static_cast<long long>(c) + static_cast<long long>(kRingStages - 1) * gridDim.x;
                if (cn < n_chunks) {
                    mbar_wait(&empty[rs], rph, 20);              // all eight warps have read it
                    issue(rs, static_cast<int>(cn));
                }
            }
            float2 st[kWarpRows];
            float dcol[kWarpRows];
#pragma unroll
            for (int r = 0; r < kWarpRows; ++r) { st[r] = st_next[r]; dcol[r] = dc_next[r]; }
            load_side(c + static_cast<int>(gridDim.x));
            mbar_wait(&full[s], ph, 21);
            const uint8_t* sv = ring + s * kStageBytes + (warp * kWarpRows) * (kK * 2) + lane * 16;
            const long long row_base = static_cast<long long>(c) * kRingRows + warp * kWarpRows;
            // two rows at a time, in lockstep: the two rows' arithmetic and their 2 x 2 x 5 reduction shuffles are independent
            // instruction streams the scheduler can interleave (16 consumer warps per SM: the kernel is bound by issue
            // latency, not by the 825 MB it moves)
#pragma unroll
            for (int r0 = 0; r0 < kWarpRows; r0 += 2) {
                if (row_base + r0 >= M) break;                   // warp-uniform: both rows past M
                // packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2: columns 2q, 2q+1 per instruction), as in the forward epilogue
                uint64_t n[2][4], dn[2][4], s1[2] = {0ull, 0ull}, s2[2] = {0ull, 0ull};
                bool live[2];
                const uint64_t half2 = pack2f(0.5f, 0.5f), one2 = pack2f(1.f, 1.f);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = r0 + h;
                    live[h] = row_base + r < M;                  // a row past M holds stale shared memory: contributes exact zeros
                    const uint4 v4 = *reinterpret_cast<const uint4*>(sv + r * (kK * 2));
                    uint4 d4 = make_uint4(0, 0, 0, 0);
                    if constexpr (!RANK1) d4 = *reinterpret_cast<const uint4*>(sv + kRingArrBytes + r * (kK * 2));
                    const uint32_t vw[4] = {v4.x, v4.y, v4.z, v4.w}, dw[4] = {d4.x, d4.y, d4.z, d4.w};
                    const uint64_t mean2 = pack2f(st[r].x, st[r].x), rstd2 = pack2f(st[r].y, st[r].y), dcol2 = pack2f(dcol[r], dcol[r]);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        // bf16 -> fp32 is a 16-bit shift: (low half << 16, high half & 0xffff0000)
                        uint64_t vv = pack2(vw[q] << 16, vw[q] & 0xffff0000u);
                        uint64_t dd;
                        if constexpr (RANK1) {
                            const uint32_t rounded = bf16x2_of(mul2(dcol2, wo2[q]));                  // bf16(bf16(dout) * w_out), like the GEMM
                            dd = pack2(rounded << 16, rounded & 0xffff0000u);
                        } else {
                            dd = pack2(dw[q] << 16, dw[q] & 0xffff0000u);
                        }
                        if (!live[h]) { vv = 0ull; dd = 0ull; }
                        n[h][q] = mul2(sub2(vv, mean2), rstd2);
                        const uint64_t z = fma2(n[h][q], g2[q], be2[q]);
                        const uint64_t hz = mul2(z, half2);
                        const uint64_t sg = fma2(half2, pack2f(tanh_fast(lo_of(hz)), tanh_fast(hi_of(hz))), half2);   // sigmoid(z), one MUFU op each
                        const uint64_t dz = mul2(dd, mul2(sg, fma2(z, sub2(one2, sg), one2)));                        // dy * SiLU'(z)
                        acc_g2[q] = fma2(dz, n[h][q], acc_g2[q]);
                        acc_b2[q] = add2(acc_b2[q], dz);
                        dn[h][q] = mul2(dz, g2[q]);
                        s1[h] = add2(s1[h], dn[h][q]);
                        s2[h] = fma2(dn[h][q], n[h][q], s2[h]);
                    }
                }
                float r1[2], r2[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) { r1[h] = lo_of(s1[h]) + hi_of(s1[h]); r2[h] = lo_of(s2[h]) + hi_of(s2[h]); }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        r1[h] += __shfl_xor_sync(0xffffffffu, r1[h], o);
                        r2[h] += __shfl_xor_sync(0xffffffffu, r2[h], o);
                    }
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int r = r0 + h;
                    const float a = r1[h] * (1.f / kK), b = r2[h] * (1.f / kK);
                    const uint64_t a2 = pack2f(a, a), nb2 = pack2f(-b, -b), rstd2 = pack2f(st[r].y, st[r].y);
                    uint32_t ow[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint64_t o2 = mul2(rstd2, fma2(n[h][q], nb2, sub2(dn[h][q], a2)));      // rstd (dn - a - n b)
                        acc_v2[q] = add2(acc_v2[q], o2);
                        ow[q] = bf16x2_of(o2);
                    }
                    if (live[h]) *reinterpret_cast<uint4*>(dv + (row_base + r) * kK + c0) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);               // this warp has read its rows of the stage
            rs = s; rph = ph;
            if (++s == kRingStages) { s = 0; ph ^= 1; }
        }
    }
    __syncthreads();                                             // every stage consumed: the ring is free for the reduction
    float* red = reinterpret_cast<float*>(ring);                 // [warp][3][256]
    {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            *reinterpret_cast<float2*>(&red[(warp * 3 + 0) * kK + c0 + 2 * q]) = make_float2(lo_of(acc_g2[q]), hi_of(acc_g2[q]));
            *reinterpret_cast<float2*>(&red[(warp * 3 + 1) * kK + c0 + 2 * q]) = make_float2(lo_of(acc_b2[q]), hi_of(acc_b2[q]));
            *reinterpret_cast<float2*>(&red[(warp * 3 + 2) * kK + c0 + 2 * q]) = make_float2(lo_of(acc_v2[q]), hi_of(acc_v2[q]));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * kK; i += kRingThreads) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += red[w * 3 * kK + i];
        partials[static_cast<long long>(blockIdx.x) * 3 * kK + i] = t;
    }
}

// bf16 -> fp32 of a contiguous array (the gradient handed back to the fp32 laterals): 16-byte loads, 2 x 16-byte stores.
__global__ void __launch_bounds__(256) k_bf16_to_f32(const uint4* __restrict__ src, float4* __restrict__ dst, long long n_vec8) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec8; i += stride) {
        const uint4 w = src[i];
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.y));
        const float2 c = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.z));
        const float2 d = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.w));
        dst[2 * i] = make_float4(a.x, a.y, b.x, b.y);
        dst[2 * i + 1] = make_float4(c.x, c.y, d.x, d.y);
    }
}

// ---- training path of the laterals (1x1 conv + batch-statistics BatchNorm over rows [M,256]) ---------------------------------
// Backward of the BatchNorm, reductions over ROWS (per channel): one warp per row, lane = 8 channels, register
// accumulators, per-CTA partials.
//   pass 1 (k_bn_bwd_colsums): partials[cta][0][c] = sum_m dz[m,c], partials[cta][1][c] = sum_m dz[m,c] n[m,c]
//   pass 2 (k_bn_bwd_apply):   dy[m,c] = scale[c] (dz[m,c] - mean_dz[c] - n[m,c] mean_dzn[c])
// n = (y - mean) invstd is the normalised conv output (recomputed by the caller with the linear mode of the layer kernel).
// dz may be a slice of a larger [B, rows_out, 256] tensor (one level of the concatenated features' gradient): row m of the
// level is row (m / rows_per_image) * dz_rows_per_image + dz_row_offset + m % rows_per_image of dz — read in place, no copy.
struct RowMap {
    unsigned rows_per_image;
    long long src_rows_per_image, src_row_offset;
    __device__ __forceinline__ long long operator()(long long m) const {
        const unsigned img = static_cast<unsigned>(m) / rows_per_image;              // M < 2^31 (checked by the caller)
        return static_cast<long long>(img) * src_rows_per_image + src_row_offset + (static_cast<unsigned>(m) - img * rows_per_image);
    }
};
__global__ void __launch_bounds__(kBwdWarps * 32) k_bn_bwd_colsums(const __nv_bfloat16* __restrict__ dz, const RowMap map, const __nv_bfloat16* __restrict__ n,
                                                                    long long M, float* __restrict__ partials) {
    __shared__ float red[kBwdWarps][2][kK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = lane * 8;
    float a0[8], a1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) a0[j] = a1[j] = 0.f;
    const long long stride = static_cast<long long>(gridDim.x) * kBwdWarps;
    for (long long row = static_cast<long long>(blockIdx.x) * kBwdWarps + warp; row < M; row += stride) {
        const uint4 d4 = *reinterpret_cast<const uint4*>(dz + map(row) * kK + c0);
        const uint4 n4 = *reinterpret_cast<const uint4*>(n + row * kK + c0);
        const uint32_t dw[4] = {d4.x, d4.y, d4.z, d4.w}, nw[4] = {n4.x, n4.y, n4.z, n4.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 df = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&dw[q]));
            const float2 nf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&nw[q]));
            a0[2 * q] += df.x; a0[2 * q + 1] += df.y;
            a1[2 * q] = __fmaf_rn(df.x, nf.x, a1[2 * q]); a1[2 * q + 1] = __fmaf_rn(df.y, nf.y, a1[2 * q + 1]);
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { red[warp][0][c0 + j] = a0[j]; red[warp][1][c0 + j] = a1[j]; }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * kK; i += kBwdWarps * 32) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += red[w][i / kK][i % kK];
        partials[static_cast<long long>(blockIdx.x) * 2 * kK + i] = t;
    }
}

__global__ void __launch_bounds__(256) k_bn_bwd_apply(const __nv_bfloat16* __restrict__ dz, const RowMap map, const __nv_bfloat16* __restrict__ n,
                                                       const float* __restrict__ scale, const float* __restrict__ mean_dz,
                                                       const float* __restrict__ mean_dzn, long long M, __nv_bfloat16* __restrict__ dy) {
    const int lane = threadIdx.x & 31;
    const int c0 = lane * 8;
    float sc[8], m0[8], m1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = scale[c0 + j]; m0[j] = mean_dz[c0 + j]; m1[j] = mean_dzn[c0 + j]; }
    const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    for (long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); row < M; row += warps) {
        const uint4 d4 = *reinterpret_cast<const uint4*>(dz + map(row) * kK + c0);
        const uint4 n4 = *reinterpret_cast<const uint4*>(n + row * kK + c0);
        const uint32_t dw[4] = {d4.x, d4.y, d4.z, d4.w}, nw[4] = {n4.x, n4.y, n4.z, n4.w};
        uint32_t ow[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 df = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&dw[q]));
            const float2 nf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&nw[q]));
            const float o0 = sc[2 * q] * (df.x - m0[2 * q] - nf.x * m1[2 * q]);
            const float o1 = sc[2 * q + 1] * (df.y - m0[2 * q + 1] - nf.y * m1[2 * q + 1]);
            const __nv_bfloat162 p2 = __floats2bfloat162_rn(o0, o1);
            ow[q] = *reinterpret_cast<const uint32_t*>(&p2);
        }
        *reinterpret_cast<uint4*>(dy + row * kK + c0) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
}

// Column sums of bf16 rows [M,256] in fp32 (the first moment of a lateral's input, see sihl_od_lateral_linear's training
// notes): per-CTA partials [gridDim.x][256], summed by the caller (deterministic).  HBM-bound, 512 B per row.
__global__ void __launch_bounds__(kBwdWarps * 32) k_rows_colsum(const __nv_bfloat16* __restrict__ x, long long M, float* __restrict__ partials) {
    __shared__ float red[kBwdWarps][kK];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = lane * 8;
    float a[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = 0.f;
    const long long stride = static_cast<long long>(gridDim.x) * kBwdWarps * 4;
    for (long long row0 = (static_cast<long long>(blockIdx.x) * kBwdWarps + warp) * 4; row0 < M; row0 += stride) {
        uint4 r4[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) r4[r] = row0 + r < M ? *reinterpret_cast<const uint4*>(x + (row0 + r) * kK + c0) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const uint32_t w[4] = {r4[r].x, r4[r].y, r4[r].z, r4[r].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[q]));
                a[2 * q] += f.x; a[2 * q + 1] += f.y;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[warp][c0 + j] = a[j];
    __syncthreads();
    for (int i = threadIdx.x; i < kK; i += kBwdWarps * 32) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += red[w][i];
        partials[static_cast<long long>(blockIdx.x) * kK + i] = t;
    }
}

// rows of channels in bf16 -> NCHW fp32: y [B*HW, C] -> x [B, C, HW] (the gradient handed back to the neck).
__global__ void __launch_bounds__(256) k_rows_to_nchw_f32(const __nv_bfloat16* __restrict__ y, float* __restrict__ x, int C, long long HW) {
    __shared__ float tile[64][65];                                           // [hw][c]
    const long long hw0 = static_cast<long long>(blockIdx.x) * 64;
    const int c0 = blockIdx.y * 64;
    const int chunk = threadIdx.x & 7, rr = threadIdx.x >> 3;               // 8 chunks of 8 channels x 32 rows per pass
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        const int h = rr + 32 * pass;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (hw0 + h < HW) w = *reinterpret_cast<const uint4*>(y + (static_cast<long long>(blockIdx.z) * HW + hw0 + h) * C + c0 + chunk * 8);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ww[q]));
            tile[h][chunk * 8 + 2 * q] = f.x;
            tile[h][chunk * 8 + 2 * q + 1] = f.y;
        }
    }
    __syncthreads();
    float* xb = x + static_cast<long long>(blockIdx.z) * C * HW;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;                 // 64 x 4
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const int c = ty + 4 * r;
        if (hw0 + tx < HW) xb[static_cast<long long>(c0 + c) * HW + hw0 + tx] = tile[tx][c];
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult status;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &status) != cudaSuccess || status != cudaDriverEntryPointSuccess)
            ptr = nullptr;
        return reinterpret_cast<EncodeTiledFn>(ptr);
    }();
    return fn;
}

// [rows, 256] bf16 row-major matrix, read in boxes of box_rows x 64 columns (128 B) with the 128-byte swizzle.
bool make_map(CUtensorMap* map, const void* ptr, unsigned long long rows, unsigned box_rows) {
    EncodeTiledFn fn = encode_tiled();
    if (!fn) return false;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(kK), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(kK) * 2};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(kChunkK), box_rows};
    const cuuint32_t elem[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int sm_count() {
    static int n = [] {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) v = 0;
        return v;
    }();
    return n;
}

template <int N, int MODE>
int launch_layer(const void* x, long long M, const void* w, const MlpParams& p_in, cudaStream_t stream) {
    using L = MlpSmem<N>;
    // per launch: the attribute belongs to the current device's context, and a process may drive several
    if (cudaFuncSetAttribute(k_mlp_layer<N, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal) != cudaSuccess) return SIHL_OD_ECUDA;
    CUtensorMap map_x, map_w;
    if (!make_map(&map_x, x, static_cast<unsigned long long>(M), kBlockM) || !make_map(&map_w, w, N, N)) return SIHL_OD_ECUDA;
    MlpParams p = p_in;
    p.M = M;
    p.n_tiles = static_cast<int>((M + kBlockM - 1) / kBlockM);
    const int sms = sm_count();
    if (sms <= 0) return SIHL_OD_ECUDA;
    const int grid = p.n_tiles < sms ? p.n_tiles : sms;
    k_mlp_layer<N, MODE><<<grid, kThreads, L::kTotal, stream>>>(map_x, map_w, p);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

// The kernel writes partials[gridDim.x][3][256]; any partial_rows in [1, 8 x SMs] is a valid grid.
template <bool RANK1>
int launch_hidden_bwd(const void* v, const void* dy, const float* dout, const void* w_out, const float* row_stats, const float* gamma,
                             const float* beta, int64_t M, void* dv, float* partials, int partial_rows, cudaStream_t st) {
    if (cudaFuncSetAttribute(k_mlp_hidden_bwd_ring<RANK1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ring_smem_bytes<RANK1>()) != cudaSuccess)
        return SIHL_OD_ECUDA;
    k_mlp_hidden_bwd_ring<RANK1><<<partial_rows, kRingThreads, ring_smem_bytes<RANK1>(), st>>>(
        static_cast<const __nv_bfloat16*>(v), static_cast<const __nv_bfloat16*>(dy), dout, static_cast<const __nv_bfloat16*>(w_out), row_stats, gamma,
        beta, M, static_cast<__nv_bfloat16*>(dv), partials);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

extern "C" {

SIHL_OD_API int sihl_od_mlp_hidden(const void* x_bf16, int64_t M, int channels, const void* w_bf16, const float* bias, const float* gamma,
                                   const float* beta, float eps, void* y_bf16, void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL) return SIHL_OD_EINVAL;
    if (M == 0) return SIHL_OD_OK;
    if (!x_bf16 || !w_bf16 || !bias || !gamma || !beta || !y_bf16 || !aligned16(x_bf16) || !aligned16(w_bf16) || !aligned16(y_bf16))
        return SIHL_OD_EINVAL;
    MlpParams p{};
    p.bias = bias; p.gamma = gamma; p.beta = beta; p.out = y_bf16; p.eps = eps; p.out_cols = kK;
    return launch_layer<256, kHidden>(x_bf16, M, w_bf16, p, static_cast<cudaStream_t>(stream));
}

SIHL_OD_API int sihl_od_mlp_hidden_train(const void* x_bf16, int64_t M, int channels, const void* w_bf16, const float* bias, const float* gamma,
                                         const float* beta, float eps, void* y_bf16, float* row_stats, void* v_bf16, void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL) return SIHL_OD_EINVAL;
    if (M == 0) return SIHL_OD_OK;
    if (!x_bf16 || !w_bf16 || !bias || !gamma || !beta || !y_bf16 || !row_stats || !aligned16(x_bf16) || !aligned16(w_bf16) || !aligned16(y_bf16) ||
        (reinterpret_cast<uintptr_t>(row_stats) & 7u) || !aligned16(v_bf16))
        return SIHL_OD_EINVAL;
    MlpParams p{};
    p.bias = bias; p.gamma = gamma; p.beta = beta; p.out = y_bf16; p.eps = eps; p.out_cols = kK; p.row_stats = row_stats; p.pre_out = v_bf16;
    if (v_bf16 != nullptr) return launch_layer<256, kHiddenPre>(x_bf16, M, w_bf16, p, static_cast<cudaStream_t>(stream));
    return launch_layer<256, kHidden>(x_bf16, M, w_bf16, p, static_cast<cudaStream_t>(stream));
}

SIHL_OD_API int sihl_od_bf16_to_f32(const void* src_bf16, int64_t n, float* dst, void* stream) {
    if (n < 0 || (n & 7) != 0) return SIHL_OD_EINVAL;
    if (n == 0) return SIHL_OD_OK;
    if (!src_bf16 || !dst || !aligned16(src_bf16) || !aligned16(dst)) return SIHL_OD_EINVAL;
    const int sms = sm_count();
    if (sms <= 0) return SIHL_OD_ECUDA;
    k_bf16_to_f32<<<sms * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const uint4*>(src_bf16), reinterpret_cast<float4*>(dst), n / 8);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

SIHL_OD_API int sihl_od_mlp_bwd_partial_rows(void) { const int sms = sm_count(); return sms > 0 ? 8 * sms : 0; }

SIHL_OD_API int sihl_od_mlp_hidden_bwd_partial_rows(void) { const int sms = sm_count(); return sms > 0 ? 2 * sms : 0; }

SIHL_OD_API int sihl_od_mlp_hidden_bwd(const void* v_bf16, const void* dy_bf16, const float* row_stats, const float* gamma, const float* beta, int64_t M,
                                       int channels, void* dv_bf16, float* partials, int partial_rows, void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL || partial_rows <= 0 || partial_rows > sihl_od_mlp_bwd_partial_rows()) return SIHL_OD_EINVAL;
    if (!partials || !gamma || !beta) return SIHL_OD_EINVAL;
    if (M > 0 && (!v_bf16 || !dy_bf16 || !row_stats || !dv_bf16 || !aligned16(v_bf16) || !aligned16(dy_bf16) || !aligned16(dv_bf16) ||
                  (reinterpret_cast<uintptr_t>(row_stats) & 7u)))
        return SIHL_OD_EINVAL;
    return launch_hidden_bwd<false>(v_bf16, dy_bf16, nullptr, nullptr, row_stats, gamma, beta, M, dv_bf16, partials, partial_rows,
                                    static_cast<cudaStream_t>(stream));
}

SIHL_OD_API int sihl_od_mlp_hidden_bwd_rank1(const void* v_bf16, const float* dout, const void* w_out_bf16, const float* row_stats, const float* gamma,
                                             const float* beta, int64_t M, int channels, void* dv_bf16, float* partials, int partial_rows,
                                             void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL || partial_rows <= 0 || partial_rows > sihl_od_mlp_bwd_partial_rows()) return SIHL_OD_EINVAL;
    if (!partials || !gamma || !beta || !w_out_bf16) return SIHL_OD_EINVAL;
    if (M > 0 && (!v_bf16 || !dout || !row_stats || !dv_bf16 || !aligned16(v_bf16) || !aligned16(dv_bf16) ||
                  (reinterpret_cast<uintptr_t>(row_stats) & 7u) || (reinterpret_cast<uintptr_t>(dout) & 3u)))
        return SIHL_OD_EINVAL;
    return launch_hidden_bwd<true>(v_bf16, nullptr, dout, w_out_bf16, row_stats, gamma, beta, M, dv_bf16, partials, partial_rows,
                                   static_cast<cudaStream_t>(stream));
}

SIHL_OD_API int sihl_od_mlp_out(const void* x_bf16, int64_t M, int channels, const void* w_bf16, const float* bias, int n_pad, int out_cols,
                                float* y, void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL || out_cols < 1 || out_cols > n_pad) return SIHL_OD_EINVAL;
    if (n_pad != 16 && n_pad != 32 && n_pad != 64 && n_pad != 96 && n_pad != 128 && n_pad != 256) return SIHL_OD_EINVAL;
    if (M == 0) return SIHL_OD_OK;
    if (!x_bf16 || !w_bf16 || !bias || !y || !aligned16(x_bf16) || !aligned16(w_bf16)) return SIHL_OD_EINVAL;
    MlpParams p{};
    p.bias = bias; p.out = y; p.out_cols = out_cols;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (n_pad) {
        case 16: return launch_layer<16, kOutF32>(x_bf16, M, w_bf16, p, st);
        case 32: return launch_layer<32, kOutF32>(x_bf16, M, w_bf16, p, st);
        case 64: return launch_layer<64, kOutF32>(x_bf16, M, w_bf16, p, st);
        case 96: return launch_layer<96, kOutF32>(x_bf16, M, w_bf16, p, st);
        case 128: return launch_layer<128, kOutF32>(x_bf16, M, w_bf16, p, st);
        default: return launch_layer<256, kOutF32>(x_bf16, M, w_bf16, p, st);
    }
}

SIHL_OD_API int sihl_od_lateral_rows(const float* x_nchw, int batch, int channels, int64_t hw, void* rows_bf16, void* stream) {
    if (batch < 0 || channels <= 0 || (channels & 63) != 0 || hw < 0 || batch > 65535) return SIHL_OD_EINVAL;
    if (batch == 0 || hw == 0) return SIHL_OD_OK;
    if (!x_nchw || !rows_bf16 || !aligned16(rows_bf16)) return SIHL_OD_EINVAL;
    const dim3 grid(static_cast<unsigned>((hw + 63) / 64), static_cast<unsigned>(channels / 64), static_cast<unsigned>(batch));
    k_nchw_to_rows_bf16<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x_nchw, static_cast<__nv_bfloat16*>(rows_bf16), channels, hw);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

SIHL_OD_API int sihl_od_rows_to_nchw(const void* rows_bf16, int batch, int channels, int64_t hw, float* x_nchw, void* stream) {
    if (batch < 0 || channels <= 0 || (channels & 63) != 0 || hw < 0 || batch > 65535) return SIHL_OD_EINVAL;
    if (batch == 0 || hw == 0) return SIHL_OD_OK;
    if (!rows_bf16 || !x_nchw || !aligned16(rows_bf16)) return SIHL_OD_EINVAL;
    const dim3 grid(static_cast<unsigned>((hw + 63) / 64), static_cast<unsigned>(channels / 64), static_cast<unsigned>(batch));
    k_rows_to_nchw_f32<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(rows_bf16), x_nchw, channels, hw);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

static bool row_map_ok(int64_t M, int64_t rows_per_image, int64_t src_rows_per_image, int64_t src_row_offset) {
    return M <= 0x7FFFFF00LL && rows_per_image > 0 && rows_per_image <= 0x7FFFFF00LL && src_rows_per_image >= rows_per_image && src_row_offset >= 0 &&
           src_row_offset + rows_per_image <= src_rows_per_image && M % rows_per_image == 0;
}

SIHL_OD_API int sihl_od_bn_bwd_colsums_map(const void* dz_bf16, int64_t rows_per_image, int64_t dz_rows_per_image, int64_t dz_row_offset,
                                           const void* n_bf16, int64_t M, int channels, float* partials, int partial_rows, void* stream) {
    if (channels != kK || M < 0 || partial_rows <= 0 || partial_rows != sihl_od_mlp_bwd_partial_rows() || !partials) return SIHL_OD_EINVAL;
    if (M > 0 && (!dz_bf16 || !n_bf16 || !aligned16(dz_bf16) || !aligned16(n_bf16) || !row_map_ok(M, rows_per_image, dz_rows_per_image, dz_row_offset)))
        return SIHL_OD_EINVAL;
    const RowMap map{static_cast<unsigned>(M > 0 ? rows_per_image : 1), dz_rows_per_image, dz_row_offset};
    k_bn_bwd_colsums<<<partial_rows, kBwdWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(dz_bf16), map, static_cast<const __nv_bfloat16*>(n_bf16), M, partials);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

SIHL_OD_API int sihl_od_bn_bwd_colsums(const void* dz_bf16, const void* n_bf16, int64_t M, int channels, float* partials, int partial_rows,
                                       void* stream) {
    return sihl_od_bn_bwd_colsums_map(dz_bf16, M > 0 ? M : 1, M > 0 ? M : 1, 0, n_bf16, M, channels, partials, partial_rows, stream);
}

SIHL_OD_API int sihl_od_bn_bwd_apply_map(const void* dz_bf16, int64_t rows_per_image, int64_t dz_rows_per_image, int64_t dz_row_offset,
                                         const void* n_bf16, const float* scale, const float* mean_dz, const float* mean_dzn, int64_t M, int channels,
                                         void* dy_bf16, void* stream) {
    if (channels != kK || M < 0) return SIHL_OD_EINVAL;
    if (M == 0) return SIHL_OD_OK;
    if (!dz_bf16 || !n_bf16 || !scale || !mean_dz || !mean_dzn || !dy_bf16 || !aligned16(dz_bf16) || !aligned16(n_bf16) || !aligned16(dy_bf16) ||
        !row_map_ok(M, rows_per_image, dz_rows_per_image, dz_row_offset))
        return SIHL_OD_EINVAL;
    const int sms = sm_count();
    if (sms <= 0) return SIHL_OD_ECUDA;
    const RowMap map{static_cast<unsigned>(rows_per_image), dz_rows_per_image, dz_row_offset};
    k_bn_bwd_apply<<<sms * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(dz_bf16), map,
                                                                          static_cast<const __nv_bfloat16*>(n_bf16), scale, mean_dz, mean_dzn, M,
                                                                          static_cast<__nv_bfloat16*>(dy_bf16));
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

SIHL_OD_API int sihl_od_bn_bwd_apply(const void* dz_bf16, const void* n_bf16, const float* scale, const float* mean_dz, const float* mean_dzn,
                                     int64_t M, int channels, void* dy_bf16, void* stream) {
    return sihl_od_bn_bwd_apply_map(dz_bf16, M > 0 ? M : 1, M > 0 ? M : 1, 0, n_bf16, scale, mean_dz, mean_dzn, M, channels, dy_bf16, stream);
}

SIHL_OD_API int sihl_od_rows_colsum(const void* rows_bf16, int64_t M, int channels, float* partials, int partial_rows, void* stream) {
    if (channels != kK || M < 0 || partial_rows <= 0 || partial_rows != sihl_od_mlp_bwd_partial_rows() || !partials) return SIHL_OD_EINVAL;
    if (M > 0 && (!rows_bf16 || !aligned16(rows_bf16))) return SIHL_OD_EINVAL;
    k_rows_colsum<<<partial_rows, kBwdWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(rows_bf16), M, partials);
    return cudaGetLastError() == cudaSuccess ? SIHL_OD_OK : SIHL_OD_ECUDA;
}

SIHL_OD_API int sihl_od_lateral_linear(const void* rows_bf16, int64_t M, int channels, const void* w_bf16, const float* bias, int64_t rows_per_image,
                                       int64_t out_rows_per_image, int64_t out_row_offset, void* y_bf16, void* stream) {
    if (channels != kK || M < 0 || M > 0x7FFFFF00LL || rows_per_image <= 0 || out_rows_per_image < rows_per_image || out_row_offset < 0 ||
        out_row_offset + rows_per_image > out_rows_per_image)
        return SIHL_OD_EINVAL;
    if (M == 0) return SIHL_OD_OK;
    if (!rows_bf16 || !w_bf16 || !bias || !y_bf16 || !aligned16(rows_bf16) || !aligned16(w_bf16) || !aligned16(y_bf16)) return SIHL_OD_EINVAL;
    MlpParams p{};
    p.bias = bias; p.out = y_bf16; p.out_cols = kK;
    p.rows_per_image = rows_per_image; p.out_rows_per_image = out_rows_per_image; p.out_row_offset = out_row_offset;
    return launch_layer<256, kLinear>(rows_bf16, M, w_bf16, p, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
