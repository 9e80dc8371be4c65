// tq_loss.cu -- per-token negative log-likelihood straight from the logits, in one read of them.
//
//   loss[r] = logsumexp(x[r, 0:cols]) - x[r, target[r]]      (= -log_softmax(x[r])[target[r]])
//
// The language model's perplexity needs one float per token from a [T*B, V] decoder output.  torch.log_softmax writes a
// second [T*B, V] tensor for nll_loss to pick one value per row from; this pass reads the decoder output once, in place
// (row stride ld >= cols, so linear_codes' padded [M, Op] output needs no slice copy), and writes only the loss.
//
// Layout.  A row is reduced by one CTA, or by a cluster of C = 2 / 4 / 8 CTAs when there are too few rows to fill the
// GPU; CTA c of the cluster takes the c-th contiguous share of the row's 16-byte-aligned body.  Each thread reads 4
// float4 per step (16 values; 128-bit streaming loads, lanes adjacent) and folds them into its running (max m, sum s of
// exp(x - m)): the chunk maximum, the rescale of s by exp(m_old - m_new) and a pairwise sum of the 16 exponentials.  The
// 0-3 scalars before the body and the 0-3 after it are one value each for the first threads of rank 0.  The block then
// takes the exact maximum M of every thread's m (and of the cluster's CTAs through distributed shared memory), rescales
// each s to M and adds them in a fixed tree (warp butterfly, then the 16 warp sums, then the cluster's CTAs in rank
// order).  Every sum has one order for a given (rows, cols, ld, row alignment): runs and graph replays are bit-identical.
//
// Special values follow torch.log_softmax + nll_loss: -inf entries add 0; a NaN anywhere, a +inf anywhere (inf - inf in
// torch) and an all -inf row give NaN.  A target outside [0, cols) gives NaN too: targets are data, not a reason to fault.
//
// Accuracy (accurate expf / logf, never __expf).  First order, relative to S = sum exp(x - M): expf 2 ulp (4u, u = 2^-24)
// per term, the rounding of x - M (u * (M - x), at most u * ln(cols) in the softmax-weighted mean), the 16-term pairwise
// sum (4u), per later step of a thread one fma that rescales and adds (4u for the factor's expf + u), the rescale to M
// (5u) and the block tree (9u + log2 C).  A thread of the 2800 x 33,278 decoder output takes at most 6 steps (5 body
// steps and one scalar), so |dS / S| <= (8 + 25 + 14 + 10.4) u = 57.4 u = 3.4e-6, and with logf (1 ulp) and the two
// final roundings |d loss| <= 3.7e-6 * max(loss, 1).  Each further step of a longer row adds 5u.
#include <cooperative_groups.h>

#include "tq_common.cuh"

namespace cg = cooperative_groups;

namespace tq {
namespace {

constexpr int NLL_THREADS = 512;
constexpr int NLL_WARPS = NLL_THREADS / 32;
constexpr int NLL_VEC = 4;                                   // float4 loads per thread per step: 16 values
constexpr int64_t NLL_STEP4 = (int64_t)NLL_THREADS * NLL_VEC;   // float4 a CTA reads per step
constexpr int NLL_MAX_CLUSTER = 8;                           // the portable cluster size

struct NllParams {
    const float *x;
    const int64_t *target;
    float *loss;
    int64_t rows, cols, ld;
};

// fold N values into (m, s): m' = max(m, v), s' = s * exp(m - m') + sum exp(v - m').  A shift of 0 while everything
// so far is -inf keeps -inf entries at exp(-inf) = 0 instead of exp(-inf - -inf) = NaN; a NaN value reaches s through
// its exponential (fmaxf drops it from the maximum) and stays there.
template <int N>
__device__ __forceinline__ void absorb(float &m, float &s, const float (&v)[N])
{
    float cm = v[0];
#pragma unroll
    for (int j = 1; j < N; ++j) cm = fmaxf(cm, v[j]);
    const float mn = fmaxf(m, cm);
    const float shift = mn == -INFINITY ? 0.0f : mn;
    float e[N];
#pragma unroll
    for (int j = 0; j < N; ++j) e[j] = expf(v[j] - shift);
#pragma unroll
    for (int w = N / 2; w >= 1; w /= 2)
#pragma unroll
        for (int j = 0; j < w; ++j) e[j] = e[j] + e[j + w];
    s = __fmaf_rn(s, expf(m - shift), e[0]);
    m = mn;
}

__global__ void __launch_bounds__(NLL_THREADS, 2) log_softmax_nll_kernel(const NllParams p)
{
    __shared__ float red_m[NLL_WARPS], red_s[NLL_WARPS];
    __shared__ float part_m, part_s;                         // this CTA's share, read by the cluster through DSMEM
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t nclusters = gridDim.x / C;

    for (int64_t r = blockIdx.x / C; r < p.rows; r += nclusters) {
        const float *row = p.x + r * p.ld;
        float xt = NAN;                                      // x[r, target]: fetched first, used last
        if (rank == 0 && tid == 0) {
            const int64_t t = p.target[r];
            if (t >= 0 && t < p.cols) xt = row[t];
        }
        const int64_t head = min(p.cols, (int64_t)(((16u - ((uintptr_t)row & 15u)) & 15u) >> 2));
        const int64_t n4 = (p.cols - head) >> 2;
        const int64_t tail = p.cols - head - 4 * n4;
        const int64_t b0 = n4 * rank / C, b1 = n4 * (rank + 1) / C;
        const float4 *body = reinterpret_cast<const float4 *>(row + head);

        float m = -INFINITY, s = 0.0f;
        if (rank == 0 && tid < head + tail) {
            const float v[1] = {row[tid < head ? tid : 4 * n4 + tid]};
            absorb(m, s, v);
        }
        for (int64_t i = b0 + tid; i < b1; i += NLL_STEP4) {
            float v[4 * NLL_VEC];
#pragma unroll
            for (int j = 0; j < NLL_VEC; ++j) {
                const int64_t k = i + (int64_t)j * NLL_THREADS;
                const float4 q = k < b1 ? __ldcs(body + k) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
                v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
            }
            absorb(m, s, v);
        }

        // the row's maximum: exact, so its order does not matter
        float M = m;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
        if (lane == 0) red_m[warp] = M;
        __syncthreads();
#pragma unroll
        for (int w = 0; w < NLL_WARPS; ++w) M = fmaxf(M, red_m[w]);
        if (C > 1) {
            if (tid == 0) part_m = M;
            cluster.sync();
            for (int c = 0; c < C; ++c) M = fmaxf(M, *cluster.map_shared_rank(&part_m, c));
        }
        // every s rescaled to M, then one fixed tree
        const float shift = M == -INFINITY ? 0.0f : M;
        float S = s * expf(m - shift);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) S = S + __shfl_xor_sync(0xffffffffu, S, o);
        if (lane == 0) red_s[warp] = S;
        __syncthreads();
        if (tid == 0) {
            float w4[NLL_WARPS];
#pragma unroll
            for (int w = 0; w < NLL_WARPS; ++w) w4[w] = red_s[w];
#pragma unroll
            for (int w = NLL_WARPS / 2; w >= 1; w /= 2)
#pragma unroll
                for (int j = 0; j < w; ++j) w4[j] = w4[j] + w4[j + w];
            S = w4[0];
            part_s = S;
        }
        if (C > 1) {
            cluster.sync();                                  // every part_s written
            if (rank == 0 && tid == 0) {
                float cs[NLL_MAX_CLUSTER];                   // C is a power of two: the tree over C ranks
#pragma unroll
                for (int c = 0; c < NLL_MAX_CLUSTER; ++c) cs[c] = c < C ? *cluster.map_shared_rank(&part_s, c) : 0.0f;
#pragma unroll
                for (int w = NLL_MAX_CLUSTER / 2; w >= 1; w /= 2)
#pragma unroll
                    for (int j = 0; j < w; ++j)
                        if (j + w < C) cs[j] = cs[j] + cs[j + w];
                S = cs[0];
            }
            cluster.sync();                                  // no CTA reuses or releases its parts while they are read
        }
        if (rank == 0 && tid == 0) {
            // M = -inf: every entry -inf (or NaN); M = +inf: inf - inf.  A NaN anywhere has made S NaN.
            p.loss[r] = isfinite(M) ? (M - xt) + logf(S) : NAN;
        }
    }
}

// ---- combine of the decoder's loss partials (tq_linear_codes_nll / tq_linear_planes_i8_nll, tq_gemm.cu) ----------------
// The conv epilogue leaves, per row r, `slots` (max m_p, sum s_p of exp(x - m_p)) partials at part[p * M + r] and the
// target logit at xt[r].  A CTA takes 32 rows: warp w reads slots w, w + 8, ... of all 32 rows (lane = row, coalesced),
// the row maximum M is taken exactly, every s_p is rescaled to it and summed in fp64, in a fixed order (per warp by
// slot, then the eight warps in a tree), so the result is bit-identical for any grid and under graph replay.  fp64
// makes the combine's own error negligible (~2^-53 per step): the loss error is that of the epilogue's fp32 partials.
constexpr int CMB_ROWS = 32, CMB_WARPS = 8;

__global__ void __launch_bounds__(CMB_ROWS * CMB_WARPS)
nll_combine_kernel(const float2 *__restrict__ part, const float *__restrict__ xt, const int64_t *__restrict__ target,
                   float *__restrict__ loss, int M, int slots, int V)
{
    __shared__ float sm[CMB_WARPS][CMB_ROWS];
    __shared__ double ss[CMB_WARPS][CMB_ROWS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * CMB_ROWS + lane;
    const bool live = r < M;
    float m = -INFINITY;
    if (live)
        for (int p = warp; p < slots; p += CMB_WARPS) m = fmaxf(m, __ldg(&part[(int64_t)p * M + r].x));
    sm[warp][lane] = m;
    __syncthreads();
    float Mx = sm[0][lane];
#pragma unroll
    for (int w = 1; w < CMB_WARPS; ++w) Mx = fmaxf(Mx, sm[w][lane]);
    const double shift = Mx == -INFINITY ? 0.0 : (double)Mx;  // all -inf: every s_p is 0 (exp(-inf) = 0, not NaN)
    double S = 0.0;
    if (live)
        for (int p = warp; p < slots; p += CMB_WARPS) {
            const float2 q = __ldg(&part[(int64_t)p * M + r]);
            S += (double)q.y * exp((double)q.x - shift);    // exact difference; a NaN s_p makes S NaN
        }
    ss[warp][lane] = S;
    __syncthreads();
    if (warp == 0 && live) {
        double w8[CMB_WARPS];
#pragma unroll
        for (int w = 0; w < CMB_WARPS; ++w) w8[w] = ss[w][lane];
#pragma unroll
        for (int w = CMB_WARPS / 2; w >= 1; w /= 2)
#pragma unroll
            for (int j = 0; j < w; ++j) w8[j] = w8[j] + w8[j + w];
        const int64_t t = target[r];
        // M = -inf: every logit -inf; M = +inf: inf - inf; a target outside [0, V) has no logit (its slot is stale)
        loss[r] = (isfinite(Mx) && t >= 0 && t < V) ? (float)(((double)Mx - (double)xt[r]) + log(w8[0])) : NAN;
    }
}

}  // namespace

int nll_combine(const float2 *part, const float *xt, const int64_t *target, float *loss, int M, int slots, int V,
                cudaStream_t s)
{
    nll_combine_kernel<<<(unsigned)((M + CMB_ROWS - 1) / CMB_ROWS), CMB_ROWS * CMB_WARPS, 0, s>>>(part, xt, target, loss, M,
                                                                                                 slots, V);
    count_launch();
    return check_launch("nll_combine_kernel");
}

}  // namespace tq

using namespace tq;

extern "C" int tq_log_softmax_nll(const float *logits, int64_t rows, int64_t cols, int64_t ld, const int64_t *targets,
                                  float *loss, void *stream)
{
    if (!logits || !targets || !loss) return fail(TQ_ERR_INVALID, "NULL pointer");
    if ((((uintptr_t)logits | (uintptr_t)loss) & 3u) || ((uintptr_t)targets & 7u))
        return fail(TQ_ERR_INVALID, "logits / loss must be 4-byte aligned (fp32), targets 8-byte aligned (int64)");
    if (rows < 1 || cols < 1 || ld < cols)
        return fail(TQ_ERR_INVALID, "rows = %lld, cols = %lld, ld = %lld: need rows >= 1, cols >= 1, ld >= cols",
                    (long long)rows, (long long)cols, (long long)ld);
    if (ld > INT64_MAX / (int64_t)sizeof(float) / rows)
        return fail(TQ_ERR_INVALID, "rows * ld = %lld x %lld floats overflows int64", (long long)rows, (long long)ld);

    // one CTA per row when the rows fill two CTAs per SM; otherwise split each row over a cluster, as long as every CTA
    // keeps at least one full step of the row
    const int sms = num_sms();
    int C = 1;
    while (C < NLL_MAX_CLUSTER && rows * C < 2 * (int64_t)sms && cols / (2 * C) >= 4 * NLL_STEP4) C *= 2;
    const int64_t nclusters = rows < (int64_t)1 << 20 ? rows : (int64_t)1 << 20;

    NllParams p;
    p.x = logits; p.target = targets; p.loss = loss;
    p.rows = rows; p.cols = cols; p.ld = ld;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(nclusters * C));
    cfg.blockDim = dim3(NLL_THREADS);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, log_softmax_nll_kernel, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(TQ_ERR_CUDA, "log_softmax_nll_kernel (%lld clusters of %d CTAs): %s", (long long)nclusters, C,
                    cudaGetErrorString(e));
    }
    count_launch();
    return check_launch("log_softmax_nll_kernel");
}
