// tq_calib.cu -- calibration and accounting kernels that surround the TR op in
// tr_layer.py, each replacing a Python/torch loop with one pass over the data:
//
//   tq_hist_accumulate   tr_layer.py:91-94   hist_bins += torch.histc(x, 8192, -50, 50)
//   tq_mse_profile       tr_layer.py:43-54   2048 scale factors x 8192 bins, argmin of the
//                                            histogram-weighted squared error (2048 launches
//                                            + 2048 host syncs in the reference)
//   tq_hese_term_count   tr_layer.py:57-63   per-element Python loop over every weight
#include "tq_common.cuh"

namespace tq {

// ---- histogram ---------------------------------------------------------------------------
// torch.histc (CUDA) bins with  bin = (int)((x - lo) * nbins / (hi - lo))  in fp32, clamps
// bin == nbins to the last bin and ignores x outside [lo, hi] (NaN included).
__device__ __forceinline__ int hist_bin(float v, float lo, float hi, int nbins)
{
    if (!(v >= lo && v <= hi)) return -1;
    const float t = __fmul_rn(__fsub_rn(v, lo), (float)nbins);
    int bin = (int)__fdiv_rn(t, __fsub_rn(hi, lo));
    if (bin == nbins) bin -= 1;
    return bin;
}

constexpr int HIST_THREADS = 512;

template <typename Tin>
__global__ void __launch_bounds__(HIST_THREADS)
hist_count_kernel(const Tin *__restrict__ x, int64_t n, uint32_t *__restrict__ counts, int nbins,
                  float lo, float hi)
{
    extern __shared__ uint32_t sh[];
    for (int i = threadIdx.x; i < nbins; i += HIST_THREADS) sh[i] = 0u;
    __syncthreads();

    constexpr int VEC = 16 / sizeof(Tin);
    const int64_t nvec = ((reinterpret_cast<uintptr_t>(x) & 15u) == 0) ? n / VEC : 0;
    const Vec<Tin, VEC> *vx = reinterpret_cast<const Vec<Tin, VEC> *>(x);
    for (int64_t i = (int64_t)blockIdx.x * HIST_THREADS + threadIdx.x; i < nvec;
         i += (int64_t)gridDim.x * HIST_THREADS) {
        const int4 raw = __ldcs(reinterpret_cast<const int4 *>(vx + i));
        Vec<Tin, VEC> v;
        memcpy(&v, &raw, 16);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const int b = hist_bin(Elem<Tin>::to_f32(v.v[e]), lo, hi, nbins);
            if (b >= 0) atomicAdd(&sh[b], 1u);
        }
    }
    for (int64_t i = nvec * VEC + (int64_t)blockIdx.x * HIST_THREADS + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * HIST_THREADS) {
        const int b = hist_bin(Elem<Tin>::to_f32(x[i]), lo, hi, nbins);
        if (b >= 0) atomicAdd(&sh[b], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += HIST_THREADS)
        if (sh[i]) atomicAdd(&counts[i], sh[i]);
}

__global__ void hist_finalize_kernel(float *__restrict__ hist, uint32_t *__restrict__ counts, int nbins)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nbins) {
        hist[i] += (float)counts[i];        // one rounding per call, like hist_bins += histc(...)
        counts[i] = 0u;                     // scratch is left zeroed for the next call
    }
}

// ---- fused calibration sweep ----------------------------------------------------------------
constexpr int MSE_THREADS = 256;

__global__ void __launch_bounds__(MSE_THREADS)
mse_profile_kernel(const float *__restrict__ hist, const float *__restrict__ x, int nbins,
                   const float *__restrict__ sfs, int bits, int terms, int enc, double *__restrict__ errs)
{
    const int s = blockIdx.x;
    const float sf = sfs[s];
    const Quant k = make_quant(sf, (float)((1u << bits) - 1u));
    double acc = 0.0;
    for (int b = threadIdx.x; b < nbins; b += MSE_THREADS) {
        const float xv = x[b];
        uint32_t neg;
        const uint32_t q = quantize_any<float, false>(xv, k, false, neg);
        int code = elem_code(q, enc, terms);
        code = neg ? -code : code;
        const float xh = __fmul_rn((float)code, sf);
        const float d = __fsub_rn(xv, xh);                 // (x - xh)
        const float t = __fmul_rn(hist[b], __fmul_rn(d, d));  // hist * (..)**2, fp32 per op
        acc += (double)t;
    }
    __shared__ double red[MSE_THREADS];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int w = MSE_THREADS / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) errs[s] = red[0];
}

// first index of the minimum of (float)errs -- torch.argmin(torch.Tensor(errs)) (tr_layer.py:53)
__global__ void __launch_bounds__(1024)
argmin_kernel(const double *__restrict__ errs, int nsf, int *__restrict__ argmin)
{
    __shared__ float bv[1024];
    __shared__ int bi[1024];
    float best = INFINITY;
    int idx = 0x7FFFFFFF;
    for (int i = threadIdx.x; i < nsf; i += 1024) {
        const float e = (float)errs[i];
        if (idx == 0x7FFFFFFF || e < best) { best = e; idx = i; }   // i ascends: first minimum wins
    }
    bv[threadIdx.x] = best;
    bi[threadIdx.x] = idx;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
            const float e = bv[threadIdx.x + w];
            const int i = bi[threadIdx.x + w];
            if (i != 0x7FFFFFFF &&
                (bi[threadIdx.x] == 0x7FFFFFFF || e < bv[threadIdx.x] ||
                 (e == bv[threadIdx.x] && i < bi[threadIdx.x]))) {
                bv[threadIdx.x] = e;
                bi[threadIdx.x] = i;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *argmin = bi[0];
}

// ---- term count ---------------------------------------------------------------------------------
template <typename Tin>
__global__ void __launch_bounds__(256)
term_count_kernel(const Tin *__restrict__ w, int64_t n, float sf, float inv_sf, int recip, int enc,
                  unsigned long long *__restrict__ count)
{
    unsigned long long local = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const float v = Elem<Tin>::to_f32(w[i]);
        const float r = recip ? __fmul_rn(v, inv_sf) : __fdiv_rn(v, sf);
        const int k = __float2int_rz(r);                      // .int(): toward zero
        const uint32_t m = (uint32_t)(k < 0 ? -(long long)k : (long long)k);
        uint32_t T, N;
        term_masks(m, enc, T, N);
        local += (unsigned)__popc(T);
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xFFFFFFFFu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, local);
}

// ---- on-device check of the hoisted-reciprocal divide against div.rn.f32 ---------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x)
{
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

__global__ void selftest_division_kernel(uint64_t n, uint32_t seed, unsigned long long *mismatch)
{
    unsigned long long bad = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t h1 = mix32((uint32_t)i ^ seed), h2 = mix32((uint32_t)(i >> 32) + h1 + 0x9e3779b9u);
        // sf: random mantissa, exponent uniformly in [2^-30, 2^30]
        const int es = (int)(h1 % 61u) - 30;
        float sf = __uint_as_float(((uint32_t)(es + 127) << 23) | (h2 & 0x7FFFFFu));
        sf = fminf(sf, 1073741824.0f);
        // a: any non-negative float bit pattern (zero, denormals, huge, inf included), or a
        // near-half-integer multiple of sf (the quantiser's rounding boundaries)
        const uint32_t h3 = mix32(h2 ^ 0x85ebca6bu);
        float a;
        if (h3 & 1u) {
            a = fmaxf(__uint_as_float(mix32(h3) & 0x7FFFFFFFu), 0.0f);
        } else {
            const float kk = (float)((h3 >> 1) & 0x3FFu) * 0.5f;
            a = __uint_as_float(__float_as_uint(kk * sf) + ((h3 >> 12) & 3u) - 1u);
            a = fmaxf(fabsf(a), 0.0f);
        }
        const Quant k = make_quant(sf, 65535.0f);
        const uint32_t qa = quantize_f32<true>(a, k);
        const uint32_t qb = quantize_f32<false>(a, k);
        bad += (qa != qb);
        // in the range where the quotient matters the divide itself must agree bit for bit
        if (a >= 1e-24f && a <= 1.4e14f) {
            bad += (__float_as_uint(div_rn_nonneg<true>(a, k)) != __float_as_uint(div_rn_nonneg<false>(a, k)));
        }
    }
    if (bad) atomicAdd(mismatch, bad);
}

static int grid_cap(int64_t items, int threads, int per_sm)
{
    const int64_t need = (items + threads - 1) / threads;
    const int64_t cap = (int64_t)num_sms() * per_sm;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace tq

using namespace tq;

extern "C" int tq_hist_accumulate(const void *x, int dtype, int64_t n, float *hist,
                                  uint32_t *counts_scratch, int nbins, float lo, float hi,
                                  void *stream)
{
    if (n < 0 || nbins < 1 || nbins > 12288) return fail(TQ_ERR_INVALID, "nbins must be in [1, 12288]");
    if (!hist || !counts_scratch || (!x && n)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (!(hi > lo)) return fail(TQ_ERR_INVALID, "empty histogram range");
    cudaStream_t s = (cudaStream_t)stream;
    if (n > 0) {
        const size_t smem = (size_t)nbins * sizeof(uint32_t);
        const int grid = grid_cap((n + 3) / 4, HIST_THREADS, 2);
        switch (dtype) {
            case TQ_F32:
                hist_count_kernel<float><<<grid, HIST_THREADS, smem, s>>>((const float *)x, n, counts_scratch, nbins, lo, hi);
                break;
            case TQ_BF16:
                hist_count_kernel<__nv_bfloat16><<<grid, HIST_THREADS, smem, s>>>((const __nv_bfloat16 *)x, n, counts_scratch, nbins, lo, hi);
                break;
            case TQ_F16:
                hist_count_kernel<__half><<<grid, HIST_THREADS, smem, s>>>((const __half *)x, n, counts_scratch, nbins, lo, hi);
                break;
            default: return fail(TQ_ERR_UNSUPPORTED, "histogram supports f32/bf16/f16 inputs");
        }
        count_launch();
        int rc = check_launch("hist_count_kernel");
        if (rc != TQ_OK) return rc;
    }
    hist_finalize_kernel<<<(nbins + 255) / 256, 256, 0, s>>>(hist, counts_scratch, nbins);
    count_launch();
    return check_launch("hist_finalize_kernel");
}

extern "C" int tq_mse_profile(const float *hist, const float *x, int nbins, const float *sfs,
                              int nsf, int bits, int terms, double *errs, int *argmin,
                              void *stream)
{
    return tq_mse_profile_enc(hist, x, nbins, sfs, nsf, bits, terms, TQ_ENC_HESE, errs, argmin, stream);
}

extern "C" int tq_mse_profile_enc(const float *hist, const float *x, int nbins, const float *sfs,
                                  int nsf, int bits, int terms, int encoding, double *errs, int *argmin,
                                  void *stream)
{
    if (check_encoding(encoding) != TQ_OK) return TQ_ERR_INVALID;
    if (!hist || !x || !sfs || !errs || !argmin) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (nbins < 1 || nsf < 1) return fail(TQ_ERR_INVALID, "empty sweep");
    if (bits < 1 || bits > TQ_MAX_BITS || terms < 0) return fail(TQ_ERR_INVALID, "bad bits/terms");
    cudaStream_t s = (cudaStream_t)stream;
    mse_profile_kernel<<<nsf, MSE_THREADS, 0, s>>>(hist, x, nbins, sfs, bits, terms, encoding, errs);
    count_launch();
    int rc = check_launch("mse_profile_kernel");
    if (rc != TQ_OK) return rc;
    argmin_kernel<<<1, 1024, 0, s>>>(errs, nsf, argmin);
    count_launch();
    return check_launch("argmin_kernel");
}

extern "C" int tq_hese_term_count(const void *w, int dtype, int64_t n, float sf, unsigned flags,
                                  unsigned long long *count, void *stream)
{
    return tq_term_count(w, dtype, n, sf, TQ_ENC_HESE, flags, count, stream);
}

extern "C" int tq_term_count(const void *w, int dtype, int64_t n, float sf, int encoding, unsigned flags,
                             unsigned long long *count, void *stream)
{
    if (check_encoding(encoding) != TQ_OK) return TQ_ERR_INVALID;
    if (!count || (!w && n)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (!(sf > 0.0f)) return fail(TQ_ERR_INVALID, "sf must be positive");
    if (n <= 0) return TQ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int recip = (flags & TQ_FLAG_RECIP_DIV) ? 1 : 0;
    const float inv = 1.0f / sf;
    const int grid = grid_cap(n, 256, 8);
    switch (dtype) {
        case TQ_F32:
            term_count_kernel<float><<<grid, 256, 0, s>>>((const float *)w, n, sf, inv, recip, encoding, count);
            break;
        case TQ_BF16:
            term_count_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16 *)w, n, sf, inv, recip, encoding, count);
            break;
        default: return fail(TQ_ERR_UNSUPPORTED, "term count supports f32/bf16 inputs");
    }
    count_launch();
    return check_launch("term_count_kernel");
}

extern "C" int tq_selftest_division(uint64_t n, uint32_t seed, unsigned long long *mismatch,
                                    void *stream)
{
    if (!mismatch) return fail(TQ_ERR_INVALID, "NULL pointer");
    selftest_division_kernel<<<num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(n, seed, mismatch);
    count_launch();
    return check_launch("selftest_division_kernel");
}
