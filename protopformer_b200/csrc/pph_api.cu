// Library-level entry points: version, last-error string, device query.
#include <stdarg.h>
#include <stdlib.h>

#include "pph_common.cuh"

namespace pph {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace pph

extern "C" int pph_version(void) { return PPH_VERSION; }

extern "C" const char* pph_last_error_string(void) { return pph::g_err; }

extern "C" int pph_sm_count(void) {
    int dev = 0, n = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) {
        pph::set_error("pph_sm_count: %s", cudaGetErrorString(e));
        return -(int)e;
    }
    return n;
}
