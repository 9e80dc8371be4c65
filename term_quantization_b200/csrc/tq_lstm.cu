// tq_lstm.cu -- the recurrence of one LSTM layer, all T steps in one persistent cooperative kernel.
//
//   gates_t = (gin[t] + bias) + h_{t-1} . W_hh^T          (torch gate order i, f, g, o; fp32)
//   c_t = sigmoid(f) * c_{t-1} + sigmoid(i) * tanh(g),  h_t = sigmoid(o) * tanh(c_t),  y[t] = h_t
//
// Layout.  CTA x owns the hidden units [x*U, x*U + U) and keeps their 4U rows of W_hh in shared memory for the whole
// sequence (row 4u + gate).  Every step it stages h_{t-1} in tiles of BT batch rows, as many as fit next to the weights
// (68 for the 650-unit language model on a B200), and each warp computes, for one unit and 8 batch
// rows, the 32 dot products of the unit's four gate rows with those 8 hidden vectors: lane l sums k = l, l + 32, ...
// in order, then a 31-shuffle transpose reduction leaves the complete sum of (gate, row) = (l / 8, l % 8) in lane l.
// Every sum is therefore taken in one fixed order, so eager runs and graph replays are bit-identical.  The cell
// update runs in the lane that owns the batch row; c stays in `cn` (each (b, unit) is owned by one thread for the whole
// sequence).  Steps are separated by a grid-wide barrier, which needs every CTA resident at once: the launch is
// cooperative (cudaLaunchAttributeCooperative), sized against cudaOccupancyMaxActiveBlocksPerMultiprocessor.
//
// h_{t-1} is read with ld.global.cg: it was written by other SMs during the previous step and must come from L2, never
// from a line this SM's L1 might hold from before the write.
#include <cooperative_groups.h>

#include "tq_common.cuh"

namespace cg = cooperative_groups;

namespace tq {
namespace {

constexpr int LSTM_THREADS = 512;                         // 16 warps: 110 registers, no spills
constexpr int LSTM_WARPS = LSTM_THREADS / 32;
constexpr int LSTM_NB = 8;                                   // batch rows per warp task (4 gates x 8 rows = 32 sums)
constexpr size_t LSTM_GATE_SMEM = (size_t)LSTM_WARPS * 32 * sizeof(float);

struct LstmParams {
    const float *gin, *bias, *w_hh, *h0, *c0;
    float *y, *hn, *cn;
    int T, B, H, U, BT;
};

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// dst[0, n) = src[0, n) through L2 (ld.global.cg), 16-byte loads with 8 in flight per thread when src is 16-byte aligned
// (dst always is): every CTA reads the whole of h_{t-1} each step, so this copy is latency-bound unless it is batched
__device__ __forceinline__ void stage_rows(float *dst, const float *src, int n)
{
    int i = threadIdx.x;
    if (((uintptr_t)src & 15u) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        const int n4 = n >> 2;
        for (; i + 7 * LSTM_THREADS < n4; i += 8 * LSTM_THREADS) {
            float4 r[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = __ldcg(s4 + i + j * LSTM_THREADS);
#pragma unroll
            for (int j = 0; j < 8; ++j) d4[i + j * LSTM_THREADS] = r[j];
        }
        for (; i < n4; i += LSTM_THREADS) d4[i] = __ldcg(s4 + i);
        i = 4 * n4 + threadIdx.x;
    }
    for (; i < n; i += LSTM_THREADS) dst[i] = __ldcg(src + i);
}

__global__ void __launch_bounds__(LSTM_THREADS, 1) lstm_recurrence_kernel(const LstmParams p)
{
    extern __shared__ __align__(16) float smem[];
    const int H = p.H, B = p.B, U = p.U;
    float *ws = smem;                                        // [4U][H]
    float *hs = ws + (size_t)4 * U * H;                      // [BT][H]
    float *gs = hs + (size_t)p.BT * H;                       // [warps][32]
    const int j0 = blockIdx.x * U;
    const int nu = min(U, H - j0);
    for (int i = threadIdx.x; i < 4 * nu * H; i += LSTM_THREADS) {
        const int r = i / H, k = i - r * H;
        ws[i] = p.w_hh[(size_t)((r & 3) * H + j0 + (r >> 2)) * H + k];
    }
    cg::grid_group grid = cg::this_grid();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lgate = lane >> 3, lrow = lane & 7;            // the (gate, row) whose sum lane ends up holding
    float *gw = gs + warp * 32;

    for (int t = 0; t < p.T; ++t) {
        const float *hprev = t == 0 ? p.h0 : p.y + (size_t)(t - 1) * B * H;
        const float *cprev = t == 0 ? p.c0 : p.cn;
        const float *gin_t = p.gin + (size_t)t * B * 4 * H;
        float *y_t = p.y + (size_t)t * B * H;
        for (int b0 = 0; b0 < B; b0 += p.BT) {
            const int nb = min(p.BT, B - b0);
            __syncthreads();                                 // the previous tile's readers are done (and ws is loaded)
            stage_rows(hs, hprev + (size_t)b0 * H, nb * H);
            __syncthreads();
            const int ngroups = (nb + LSTM_NB - 1) / LSTM_NB;
            for (int task = warp; task < nu * ngroups; task += LSTM_WARPS) {
                const int u = task / ngroups, jb = (task - u * ngroups) * LSTM_NB;
                const int nbg = min(LSTM_NB, nb - jb);
                const int unit = j0 + u;
                const int b = b0 + jb + lrow;
                const bool mine = lrow < nbg;
                float pre = 0.0f;
                if (mine) {
                    pre = gin_t[(size_t)b * 4 * H + lgate * H + unit];
                    if (p.bias) pre = pre + p.bias[lgate * H + unit];
                }
                // the cell state of the row this lane updates, fetched before the products hide its latency
                const float cold = lrow < nbg && lane < LSTM_NB ? cprev[(size_t)b * H + unit] : 0.0f;
                const float *w = ws + (size_t)4 * u * H;
                int hrow[LSTM_NB];                           // rows past the tile repeat its last row (sums discarded)
#pragma unroll
                for (int j = 0; j < LSTM_NB; ++j) hrow[j] = (jb + min(j, nbg - 1)) * H;
                float v[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = 0.0f;
                for (int k = lane; k < H; k += 32) {
                    float wk[4], hk[LSTM_NB];
#pragma unroll
                    for (int g = 0; g < 4; ++g) wk[g] = w[g * H + k];
#pragma unroll
                    for (int j = 0; j < LSTM_NB; ++j) hk[j] = hs[hrow[j] + k];
#pragma unroll
                    for (int g = 0; g < 4; ++g)
#pragma unroll
                        for (int j = 0; j < LSTM_NB; ++j) v[g * LSTM_NB + j] = __fmaf_rn(wk[g], hk[j], v[g * LSTM_NB + j]);
                }
                // transpose reduction: after the step with offset n, slot i of lane l holds index i + (l & n ? n : 0) (summed
                // with its partner's); after the last step slot 0 of lane l holds the whole sum of index l
#pragma unroll
                for (int n = 16; n >= 1; n >>= 1) {
                    const bool upper = (lane & n) != 0;
#pragma unroll
                    for (int i = 0; i < n; ++i) {
                        const float send = upper ? v[i] : v[i + n];
                        const float keep = upper ? v[i + n] : v[i];
                        v[i] = __fadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, n));
                    }
                }
                gw[lane] = __fadd_rn(pre, v[0]);
                __syncwarp();
                if (lane < nbg) {
                    const size_t o = (size_t)b * H + unit;          // lane < 8: b is this lane's own batch row
                    const float ig = sigmoid_f(gw[lane]), fg = sigmoid_f(gw[8 + lane]);
                    const float gg = tanhf(gw[16 + lane]), og = sigmoid_f(gw[24 + lane]);
                    const float c = __fmaf_rn(fg, cold, __fmul_rn(ig, gg));
                    const float h = __fmul_rn(og, tanhf(c));
                    p.cn[o] = c;
                    y_t[o] = h;
                    if (t == p.T - 1) p.hn[o] = h;
                }
                __syncwarp();
            }
        }
        grid.sync();                                         // h_t complete (and visible) before anyone reads it
    }
}

struct LstmLaunch {
    int U, blocks, BT;
    size_t smem;
};

// shared memory of a CTA holding the gate rows of U units and a tile of BT hidden rows
size_t lstm_smem(int H, int U, int BT) { return ((size_t)4 * U + BT) * H * sizeof(float) + LSTM_GATE_SMEM; }

// U = ceil(H / SMs) units per CTA (one CTA per SM at most); the rows must fit together with at least one hidden row
bool lstm_fits(int H, int sms, size_t smem_optin) { return lstm_smem(H, (H + sms - 1) / sms, 1) <= smem_optin; }

int lstm_max_hidden(int sms, size_t smem_optin)
{
    int best = 0;
    for (int H = 1; H <= 65536; ++H)
        if (lstm_fits(H, sms, smem_optin)) best = H;
    return best;
}

}  // namespace
}  // namespace tq

using namespace tq;

extern "C" int tq_lstm_recurrence(const float *gin, const float *bias, const float *w_hh, const float *h0, const float *c0,
                                  float *y, float *hn, float *cn, int T, int B, int H, void *stream)
{
    if (!gin || !w_hh || !h0 || !c0 || !y || !hn || !cn) return fail(TQ_ERR_INVALID, "NULL pointer");
    const uintptr_t addr = (uintptr_t)gin | (uintptr_t)bias | (uintptr_t)w_hh | (uintptr_t)h0 | (uintptr_t)c0 |
                           (uintptr_t)y | (uintptr_t)hn | (uintptr_t)cn;
    if (addr & 3u) return fail(TQ_ERR_INVALID, "pointers must be 4-byte aligned (fp32 tensors)");
    if (T < 1 || B < 1 || H < 1) return fail(TQ_ERR_INVALID, "T = %d, B = %d, H = %d: each must be at least 1", T, B, H);
    if ((int64_t)B * 4 * H > INT32_MAX) return fail(TQ_ERR_INVALID, "B * 4H = %lld exceeds 2^31 - 1", (long long)B * 4 * H);
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return fail(TQ_ERR_CUDA, "tq_lstm_recurrence: cannot read the device's shared-memory limit");
    const int sms = num_sms();
    if (!lstm_fits(H, sms, (size_t)optin))
        return fail(TQ_ERR_UNSUPPORTED, "H = %d: the 4 x %d gate rows per CTA and one hidden row need %zu bytes of shared memory, "
                    "%d are available (largest H on this device: %d)", H, (H + sms - 1) / sms,
                    lstm_smem(H, (H + sms - 1) / sms, 1), optin, lstm_max_hidden(sms, (size_t)optin));
    LstmLaunch L;
    L.U = (H + sms - 1) / sms;
    L.blocks = (H + L.U - 1) / L.U;
    const size_t fixed = lstm_smem(H, L.U, 0);
    const size_t rows = ((size_t)optin - fixed) / ((size_t)H * sizeof(float));
    L.BT = (int)(rows < (size_t)B ? rows : (size_t)B);
    L.smem = lstm_smem(H, L.U, L.BT);
    if (L.smem > 48 * 1024 &&
        cudaFuncSetAttribute(lstm_recurrence_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(lstm_recurrence_kernel)");
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lstm_recurrence_kernel, LSTM_THREADS, L.smem) != cudaSuccess)
        return check_launch("cudaOccupancyMaxActiveBlocksPerMultiprocessor(lstm_recurrence_kernel)");
    if ((int64_t)per_sm * sms < L.blocks)
        return fail(TQ_ERR_UNSUPPORTED, "lstm_recurrence_kernel: %d CTAs cannot all be resident (%d per SM x %d SMs)",
                    L.blocks, per_sm, sms);

    LstmParams p;
    p.gin = gin; p.bias = bias; p.w_hh = w_hh; p.h0 = h0; p.c0 = c0;
    p.y = y; p.hn = hn; p.cn = cn;
    p.T = T; p.B = B; p.H = H; p.U = L.U; p.BT = L.BT;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)L.blocks);
    cfg.blockDim = dim3(LSTM_THREADS);
    cfg.dynamicSmemBytes = L.smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, lstm_recurrence_kernel, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(TQ_ERR_CUDA, "lstm_recurrence_kernel (cooperative launch of %d CTAs): %s", L.blocks, cudaGetErrorString(e));
    }
    count_launch();
    return check_launch("lstm_recurrence_kernel");
}
