// od_common.cuh — shared device helpers for libsihl_b200 (sm_100a only).
//
// Arithmetic contract: every kernel that produces values compared bit-for-bit
// with torch-CUDA eager (anchors, CIoU, decoded boxes, sigmoid) is compiled with
// -fmad=false -prec-div=true -prec-sqrt=true and never --use_fast_math, so each
// source operator is one IEEE fp32 operation, in the operator order of the
// torch / torchvision eager code (SURVEY.md §7.1).  Fused multiply-adds appear
// only where torch's own kernels have them, written explicitly (__fmaf_rn).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/sihl_od.h"
#include "od_math.h"

namespace sihl {

void set_error(const char *fmt, ...);
int cuda_status(cudaError_t e, const char *what);

#define SIHL_CHECK_ARG(cond, ...)                          \
    do {                                                   \
        if (!(cond)) {                                     \
            ::sihl::set_error(__VA_ARGS__);                \
            return SIHL_OD_EINVAL;                         \
        }                                                  \
    } while (0)

#define SIHL_CHECK_LAUNCH(what)                                              \
    do {                                                                     \
        int _rc = ::sihl::cuda_status(cudaGetLastError(), what);             \
        if (_rc) return _rc;                                                 \
    } while (0)

constexpr int kNumSMs = 148;          // B200
constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kTile = 512;            // anchors per CTA of k_assign_resolve == capacity of one tile's positive list

// v rounded up to a multiple of 256 bytes: the alignment of every array carved out of a workspace.
size_t round_up_256(size_t v);

// The class / box maps may be device memory or pinned host memory read in place over PCIe; pageable host memory would
// fault in the kernel.  Returns SIHL_OD_EINVAL (error text set) when a map is pageable host memory, SIHL_OD_OK
// otherwise, and sets *cls_host to whether cls_logits is pinned host memory.  A NULL map is skipped.
int classify_maps(const void *cls_logits, const void *box_raw, bool *cls_host);

struct LevelTable {                   // passed by value as a kernel parameter
    int n;
    int h[SIHL_OD_MAX_LEVELS];
    int w[SIHL_OD_MAX_LEVELS];
    int base[SIHL_OD_MAX_LEVELS + 1]; // first anchor index of each level
};

// Head-output maps may arrive in half precision (the reference trains with precision="16-mixed",
// ref examples/object_detection.py:294, and upcasts inside its autocast-off blocks, ref :178,:195,:206):
// kernels templated on the map type load T and upcast in registers — no fp32 copy of the map is ever made.
// The dtype codes are SIHL_OD_F32 / _F16 / _BF16 of include/sihl_od.h.
template <typename T> __device__ __forceinline__ float ldf(const T *p);
template <> __device__ __forceinline__ float ldf<float>(const float *p) { return __ldg(p); }
template <> __device__ __forceinline__ float ldf<__half>(const __half *p) { return __half2float(__ldg(p)); }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16 *p) { return __bfloat162float(__ldg(p)); }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// v rounded to T and back (what an ATen op "run in the input dtype" returns for a half input)
template <typename T> __device__ __forceinline__ float round_to(float v);
template <> __device__ __forceinline__ float round_to<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_to<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float round_to<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// four consecutive elements (a raw box) as float4
template <typename T> __device__ __forceinline__ float4 ldf4(const T *p);
template <> __device__ __forceinline__ float4 ldf4<float>(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
template <> __device__ __forceinline__ float4 ldf4<__half>(const __half *p)
{
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <> __device__ __forceinline__ float4 ldf4<__nv_bfloat16>(const __nv_bfloat16 *p)
{
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.x)), b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
template <typename T> __device__ __forceinline__ void stf4(T *p, float4 v);
template <> __device__ __forceinline__ void stf4<float>(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }
template <> __device__ __forceinline__ void stf4<__half>(__half *p, float4 v)
{
    uint2 u;
    *reinterpret_cast<__half2 *>(&u.x) = __floats2half2_rn(v.x, v.y);
    *reinterpret_cast<__half2 *>(&u.y) = __floats2half2_rn(v.z, v.w);
    *reinterpret_cast<uint2 *>(p) = u;
}
template <> __device__ __forceinline__ void stf4<__nv_bfloat16>(__nv_bfloat16 *p, float4 v)
{
    uint2 u;
    *reinterpret_cast<__nv_bfloat162 *>(&u.x) = __floats2bfloat162_rn(v.x, v.y);
    *reinterpret_cast<__nv_bfloat162 *>(&u.y) = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2 *>(p) = u;
}

// 16 bytes of a row (4 floats / 8 halfs) as floats; p must be 16-byte aligned.
template <typename T> struct Vec16 { static constexpr int N = 16 / (int)sizeof(T); };
template <typename T> __device__ __forceinline__ void ld_vec16(const T *p, float (&out)[Vec16<T>::N]);
template <> __device__ __forceinline__ void ld_vec16<float>(const float *p, float (&out)[4])
{
    const float4 q = __ldg(reinterpret_cast<const float4 *>(p));
    out[0] = q.x; out[1] = q.y; out[2] = q.z; out[3] = q.w;
}
template <> __device__ __forceinline__ void ld_vec16<__half>(const __half *p, float (&out)[8])
{
    const uint4 u = __ldg(reinterpret_cast<const uint4 *>(p));
    const unsigned w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));
        out[2 * i] = f.x; out[2 * i + 1] = f.y;
    }
}
template <> __device__ __forceinline__ void ld_vec16<__nv_bfloat16>(const __nv_bfloat16 *p, float (&out)[8])
{
    const uint4 u = __ldg(reinterpret_cast<const uint4 *>(p));
    const unsigned w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w[i]));
        out[2 * i] = f.x; out[2 * i + 1] = f.y;
    }
}
template <typename T> __device__ __forceinline__ void st_vec16(T *p, const float (&v)[Vec16<T>::N]);
template <> __device__ __forceinline__ void st_vec16<float>(float *p, const float (&v)[4])
{
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void st_vec16<__half>(__half *p, const float (&v)[8])
{
    uint4 u;
    unsigned *w = reinterpret_cast<unsigned *>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) *reinterpret_cast<__half2 *>(&w[i]) = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4 *>(p) = u;
}
template <> __device__ __forceinline__ void st_vec16<__nv_bfloat16>(__nv_bfloat16 *p, const float (&v)[8])
{
    uint4 u;
    unsigned *w = reinterpret_cast<unsigned *>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) *reinterpret_cast<__nv_bfloat162 *>(&w[i]) = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4 *>(p) = u;
}

// Run `stmt` with the alias T bound to the C++ type of dtype code `code`; returns SIHL_OD_EINVAL on a bad code.
#define SIHL_DISPATCH_DTYPE(code, ...)                                                           \
    do {                                                                                         \
        if ((code) == SIHL_OD_F32) { using T = float; __VA_ARGS__; }                             \
        else if ((code) == SIHL_OD_F16) { using T = __half; __VA_ARGS__; }                       \
        else if ((code) == SIHL_OD_BF16) { using T = __nv_bfloat16; __VA_ARGS__; }               \
        else { ::sihl::set_error("map dtype code %d is not one of f32/f16/bf16", (int)(code)); return SIHL_OD_EINVAL; } \
    } while (0)

__device__ __forceinline__ Box4 to_box(float4 b) { return Box4{b.x, b.y, b.z, b.w}; }

// Order-preserving map fp32 -> uint32 (ascending) and its inverse.
__device__ __forceinline__ unsigned f2ord(float f)
{
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// IoU of two xyxy boxes with the operator order of torchvision's CPU nms kernel
// (torchvision/csrc/ops/cpu/nms_kernel.cpp: ovr = inter / (iarea + areas[j] - inter)),
// areas as (x2 - x1) * (y2 - y1).  NaN when both boxes have zero area.
__device__ __forceinline__ float box_iou(float4 a, float area_a, float4 b, float area_b)
{
    const float w = fmaxf(0.f, fminf(a.z, b.z) - fmaxf(a.x, b.x));
    const float h = fmaxf(0.f, fminf(a.w, b.w) - fmaxf(a.y, b.y));
    const float inter = w * h;
    return inter / ((area_a + area_b) - inter);
}

// The overlap a greedy NMS compares with its threshold: kIoU is torchvision's nms (box_iou), kDIoU is DIoU-NMS
// (od_math.h diou_pair).  A compile-time kind: the kernels of each kind are separate instantiations.
constexpr int kIoU = 0;
constexpr int kDIoU = 1;

// The suppression test of a kept box a against a later box b: overlap > thr (false for a NaN overlap).
template <int KIND>
__device__ __forceinline__ bool overlap_gt(float4 a, float area_a, float4 b, float area_b, float thr)
{
    static_assert(KIND == kIoU || KIND == kDIoU, "overlap kind");
    if (KIND == kDIoU) return diou_pair(to_box(a), area_a, to_box(b), area_b) > thr;
    return box_iou(a, area_a, b, area_b) > thr;
}

// Shared-memory address and mbarrier set-up of the TMA rings (od_infer.cu, od_mlp.cu).
__device__ __forceinline__ uint32_t smem_u32(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFullMask, v, o));
    return v;
}

// binary_cross_entropy_with_logits term (od_math.h bce_logits) for the fused resolve pass, where it is 13 % of the
// kernel's instructions: log1p(e^-|x|) with y = e^-|x| from ex2.approx and, for y < 0.223 (|x| > 1.5: all but a
// handful of the locations of a detection head whose location logits sit around -5), the alternating series
// y - y^2/2 + ... - y^8/8 (truncation <= y^8/9 = 7e-7 relative) in 8 FMAs; the exact libdevice path otherwise.
// The location loss is held to 1e-5 relative (north_star), not to bit equality; sihl_od_train_loss keeps the
// libdevice form.
__device__ __forceinline__ float bce_logits_fast(float x, float t)
{
    const float ax = fabsf(x);
    const float y = __expf(-ax);
    float l;
    if (y < 0.223f) {
        float q = -0.125f;
        q = __fmaf_rn(q, y, 0.14285714285714285f);
        q = __fmaf_rn(q, y, -0.16666666666666666f);
        q = __fmaf_rn(q, y, 0.2f);
        q = __fmaf_rn(q, y, -0.25f);
        q = __fmaf_rn(q, y, 0.33333333333333333f);
        q = __fmaf_rn(q, y, -0.5f);
        q = __fmaf_rn(q, y, 1.f);
        l = q * y;
    } else {
        l = log1pf(expf(-ax));
    }
    return (1.f - t) * x + (fmaxf(-x, 0.f) + l);
}

// Block-wide sum of NV doubles per thread -> atomicAdd into dst[slot[i]] by one thread.
// red: shared double[NV * 32].
template <int NV>
__device__ __forceinline__ void block_accumulate(double (&v)[NV], double *red, double *dst, const int (&slot)[NV])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) red[i * 32 + warp] = v[i];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            double x = lane < nwarps ? red[i * 32 + lane] : 0.0;
            x = warp_sum(x);
            if (lane == 0 && x != 0.0) atomicAdd(dst + slot[i], x);
        }
    }
    __syncthreads();
}


// Block-wide sum of NV floats per thread (each the sum of a handful of elements): fp32 inside a warp,
// fp64 across warps and into dst[slot[i]] — one shared-memory hop, one atomicAdd per CTA and term.
// red: shared double[NV * 32].
template <int NV>
__device__ __forceinline__ void block_accumulate_f(float (&v)[NV], double *red, double *dst, const int (&slot)[NV])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) red[i * 32 + warp] = (double)v[i];
    }
    __syncthreads();
    // lane i of warp 0 finishes term i: a handful of fp64 adds, then one atomicAdd per CTA and term
    if (warp == 0 && lane < NV) {
        double x = 0.0;
        for (int w = 0; w < nwarps; ++w) x += red[lane * 32 + w];
        int sl = 0;
#pragma unroll
        for (int i = 0; i < NV; ++i)
            if (lane == i) sl = slot[i];
        if (x != 0.0) atomicAdd(dst + sl, x);
    }
}

}  // namespace sihl
