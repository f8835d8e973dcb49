// msw_capi.cu -- version / error entry points of the C ABI (include/msw_b200.h), and the host helpers the
// kernels' launchers share (SM count, tensor-map encoder).
#include "../../include/msw_b200.h"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <execinfo.h>
#include <signal.h>
#include <stdarg.h>
#include <stdio.h>
#include <unistd.h>

namespace msw {

static thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char *what)
{
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    cudaGetLastError();   // clear the sticky-less error state
    return -(int)e;
}

int sm_count()
{
    static thread_local int cached_dev = -1, cached_sms = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        cached_dev = dev;
        cached_sms = sms;
    }
    return cached_sms;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn()
{
    static const EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

bool tensor_map_encoder_available() { return encode_tiled_fn() != nullptr; }

CUresult encode_tiled(CUtensorMap *map, CUtensorMapDataType dtype, cuuint32_t rank, const void *base,
                      const cuuint64_t *dims, const cuuint64_t *strides, const cuuint32_t *box,
                      CUtensorMapSwizzle swizzle)
{
    static const cuuint32_t elem_strides[5] = {1, 1, 1, 1, 1};     // rank <= 5
    const EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return CUDA_ERROR_NOT_SUPPORTED;
    return fn(map, dtype, rank, const_cast<void *>(base), dims, strides, box, elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE,
              swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

}  // namespace msw

extern "C" int msw_version(void) { return MSW_VERSION; }
extern "C" const char *msw_last_error(void) { return msw::g_err; }
extern "C" int msw_words_per_board(int32_t H, int32_t W)
{
    if (H < 1 || W < 1 || W > 32 || (long long)H * W > MSW_MAX_CELLS) return 0;
    return (H * W + 31) / 32;
}

// Development aid (not part of the ABI in include/msw_b200.h): print a native backtrace on SIGSEGV.
static void msw_segv_handler(int sig)
{
    void *frames[64];
    const int n = backtrace(frames, 64);
    const char msg[] = "\n[msw] SIGSEGV, native backtrace:\n";
    if (write(2, msg, sizeof(msg) - 1) < 0) {}
    backtrace_symbols_fd(frames, n, 2);
    signal(sig, SIG_DFL);
    raise(sig);
}
extern "C" void msw_debug_segv_backtrace(void) { signal(SIGSEGV, msw_segv_handler); }
