// tq_capi.cu -- process-wide plumbing behind the C ABI (include/tq_b200.h):
// thread-local error text, launch accounting, device properties, the fused encoders' quantiser check.
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

int next_quant(NextQuant &q, const void *out_codes, float sf, int bits, int terms, int enc, int max_bits, bool need_fast)
{
    if (check_encoding(enc) != TQ_OK) return TQ_ERR_INVALID;
    if (out_codes) {
        if (!(sf > 0.0f) || !(sf < INFINITY)) return fail(TQ_ERR_INVALID, "next_sf must be positive and finite");
        if (bits < 1 || bits > max_bits) return fail(TQ_ERR_UNSUPPORTED, "fused encode supports 1..%d bits", max_bits);
        if (terms < 0) return fail(TQ_ERR_INVALID, "next_terms must be >= 0");
        if (need_fast && !fast_div_ok(sf))
            return fail(TQ_ERR_UNSUPPORTED, "fused encode needs 2^-30 <= next_sf <= 2^30 (got %g): encode with tq_tr_encode_codes instead", (double)sf);
    }
    q.write_codes = out_codes ? 1 : 0;
    q.sf = out_codes ? sf : 1.0f;
    q.bits = out_codes ? bits : 1;
    q.terms = terms;
    q.enc = enc;
    q.fastdiv = fast_div_ok(q.sf) ? 1 : 0;
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
