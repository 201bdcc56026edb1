// od_api.cu — version + thread-local error text of the C ABI (include/sihl_od.h), and the host helpers of od_common.cuh.
#include <cstdarg>
#include <cstdio>
#include <initializer_list>

#include "od_common.cuh"

namespace sihl {

static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int cuda_status(cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return SIHL_OD_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return SIHL_OD_ECUDA;
}

size_t round_up_256(size_t v) { return (v + 255) & ~(size_t)255; }

int classify_maps(const void *cls_logits, const void *box_raw, bool *cls_host)
{
    *cls_host = false;
    for (const void *map : {cls_logits, box_raw}) {
        cudaPointerAttributes attr;
        if (map == nullptr) continue;
        if (cudaPointerGetAttributes(&attr, map) != cudaSuccess) { (void)cudaGetLastError(); continue; }
        SIHL_CHECK_ARG(attr.type != cudaMemoryTypeUnregistered,
                       "box_raw / cls_logits must be device memory or PINNED host memory (got a pageable host pointer)");
        if (map == cls_logits) *cls_host = attr.type == cudaMemoryTypeHost;
    }
    return SIHL_OD_OK;
}

}  // namespace sihl

extern "C" int sihl_od_version(void) { return 102; }   // 0.1.2

extern "C" const char *sihl_od_last_error_string(void) { return sihl::g_error; }
