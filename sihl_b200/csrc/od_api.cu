// od_api.cu — version + thread-local error text of the C ABI (include/sihl_od.h).
#include <cstdarg>
#include <cstdio>

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

}  // namespace sihl

extern "C" int sihl_od_version(void) { return 102; }   // 0.1.2

extern "C" const char *sihl_od_last_error_string(void) { return sihl::g_error; }
