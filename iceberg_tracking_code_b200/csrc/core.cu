// Library-wide pieces of libibt.so: version, error strings, last CUDA error (thread local).
#include "common.cuh"
#include <stdio.h>

namespace ibt {

static thread_local char g_last_error[512] = "";

void set_last_error(cudaError_t e, const char *where)
{
    snprintf(g_last_error, sizeof(g_last_error), "%s: %s (%s)", where ? where : "?", cudaGetErrorString(e),
             cudaGetErrorName(e));
}

} // namespace ibt

IBT_API int ibt_version(void) { return 104; }     /* major * 100 + minor */

IBT_API const char *ibt_error_string(int code)
{
    switch (code) {
    case IBT_OK: return "ok";
    case IBT_E_INVALID: return "invalid argument";
    case IBT_E_CUDA: return "CUDA error (see ibt_last_cuda_error)";
    case IBT_E_WORKSPACE: return "workspace too small";
    case IBT_E_CAPACITY: return "output capacity too small";
    case IBT_E_UNSUPPORTED: return "unsupported input";
    default: return "unknown error code";
    }
}

IBT_API const char *ibt_last_cuda_error(void) { return ibt::g_last_error; }
