// tq_capi.cu -- process-wide plumbing behind the C ABI (include/tq_b200.h):
// thread-local error text, launch accounting, device properties.
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "tq_common.cuh"

namespace tq {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int check_launch(const char *what)
{
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(TQ_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return TQ_OK;
}

int check_encoding(int enc)
{
    if (enc != TQ_ENC_HESE && enc != TQ_ENC_BINARY && enc != TQ_ENC_BOOTH)
        return fail(TQ_ERR_INVALID, "unknown term encoding %d (TQ_ENC_HESE, TQ_ENC_BINARY or TQ_ENC_BOOTH)", enc);
    return TQ_OK;
}

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int num_sms()
{
    // one entry per device; B200 reports 148
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

}  // namespace tq

extern "C" int tq_version(void) { return TQ_VERSION; }
extern "C" const char *tq_last_error(void) { return tq::g_err; }
extern "C" uint64_t tq_launch_count(void) { return tq::g_launches.load(std::memory_order_relaxed); }
