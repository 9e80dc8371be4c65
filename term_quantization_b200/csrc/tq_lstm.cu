// tq_lstm.cu -- the recurrence of one RNN layer (LSTM, GRU, or vanilla RNN with tanh / ReLU), all T steps in one
// persistent cooperative kernel, recurrence_kernel<Cell>.  Torch's gate order and formulas, fp32:
//
//   LSTM (G = 4 gates i, f, g, o):  a = (gin[t] + bias) + h_{t-1} . W_hh^T
//       c_t = sigmoid(f) * c_{t-1} + sigmoid(i) * tanh(g),  h_t = sigmoid(o) * tanh(c_t)
//   GRU (G = 3 gates r, z, n; gin = W_ih x + b_ih):
//       r = sigmoid((gin_r + b_hr) + W_hr . h),  z = sigmoid((gin_z + b_hz) + W_hz . h)
//       n = tanh(gin_n + r * (b_hn + W_hn . h)),  h_t = n + z * (h_{t-1} - n)      (= (1 - z) n + z h_{t-1})
//   RNN (G = 1; gin = W_ih x):  h_t = act((gin + bias) + W_hh . h),  act = tanh or ReLU (NaN stays NaN, as torch.relu)
//   y[t] = h_t
//
// Layout.  CTA x owns the hidden units [x*U, x*U + U) and keeps their G*U rows of W_hh in shared memory for the whole
// sequence (row G*u + gate).  Every step it stages h_{t-1} in tiles of BT batch rows, as many as fit next to the weights
// (68 for the 650-unit LSTM language model on a B200).  A warp task is one unit and NB = 32 / G batch rows (LSTM 4 x 8,
// GRU 3 x 10 with 2 idle slots, RNN 1 x 32): lane l sums the products of the unit's G gate rows with those NB hidden
// vectors over k = l, l + 32, ... in order, then a 31-shuffle transpose reduction leaves the complete sum of
// (gate, row) = (l / NB, l % NB) in lane l (lanes G*NB.. hold sums of zeros).  Every sum is therefore taken in one fixed
// order, so eager runs and graph replays are bit-identical.  The cell update runs in the lane that owns the batch row;
// the LSTM's c stays in `cn` (each (b, unit) is owned by one thread for the whole sequence), the GRU reads h_{t-1} of its
// row from the staged tile.  Steps are separated by a grid-wide barrier, which needs every CTA resident at once: the
// launch is cooperative (cudaLaunchAttributeCooperative), sized against cudaOccupancyMaxActiveBlocksPerMultiprocessor.
//
// h_{t-1} is read with ld.global.cg: it was written by other SMs during the previous step and must come from L2, never
// from a line this SM's L1 might hold from before the write.
//
// Tensor-memory tier (recurrence_kernel<Cell, true>).  When the G*U gate rows do not fit in shared memory next to one
// hidden row (above H = 1404 / 1628 / 2812 for LSTM / GRU / RNN on a B200), units [0, NT) of each CTA keep their rows in
// the SM's 256 KB of tensor memory instead and units [NT, U) stay in shared memory.  tcgen05.ld.32x32b lets warp w reach
// only TMEM lanes 32 (w % 4) .. +31, so TMEM unit u belongs to quarter q = u % 4, slot s = u / 4: lane 32 q + l holds the
// unit's weights for k = 32 m + l at column s * C + G m + gate (C = G * ceil(H / 32) rounded up to whole loads, zeros past
// H).  One tcgen05.ld of 16 columns (LSTM: 4 m x 4 gates, RNN: 16 m; GRU adds an .x8 for 8 m x 3 gates) gives wk[G] for
// several consecutive m.  Only the source of wk[g] changes: every lane still sums k = l, l + 32, ... in increasing k with
// the same FMAs and the same transpose reduction follows, so a unit's results do not depend on where its rows live.
// Scheduling: the tasks of quarter q's TMEM units run round-robin on the four warps w with w % 4 == q; the tasks of the
// shared-memory units then run round-robin on all sixteen warps.  The CTA (one per SM) allocates all 512 columns at kernel
// start, relinquishes the permit and deallocates after the last step; the kernel has no other way out.  NT is the most
// units TMEM holds (4 * floor(512 / C)), at most U, which also frees shared memory for more hidden rows per tile.  Below
// the old bound the launch is the shared-memory-only instance recurrence_kernel<Cell, false>, the same code as before.
//
// Test switch (environment, read on every call):
//   TQ_RECURRENCE_TMEM_UNITS=n   n units per CTA in TMEM (clamped to what TMEM holds and to U), at any H; 0 is the
//                                shared-memory-only instance.  Pins the TMEM path bit for bit against shared memory.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

#include "tq_common.cuh"

namespace cg = cooperative_groups;

namespace tq {
namespace {

constexpr int LSTM_THREADS = 512;                         // 16 warps, no spills in any cell's instance
constexpr int LSTM_WARPS = LSTM_THREADS / 32;
constexpr size_t LSTM_GATE_SMEM = (size_t)LSTM_WARPS * 32 * sizeof(float);

enum Cell { CELL_LSTM, CELL_GRU, CELL_RNN_TANH, CELL_RNN_RELU };

__host__ __device__ constexpr int cell_gates(int cell) { return cell == CELL_LSTM ? 4 : cell == CELL_GRU ? 3 : 1; }

constexpr int TMEM_COLS = 512;

// m values (k = 32 m + lane) per TMEM load: 16 columns (LSTM, RNN), 16 + 8 (GRU)
__host__ __device__ constexpr int tmem_chunk(int G) { return G == 4 ? 4 : G == 3 ? 8 : 16; }

// TMEM columns of one unit: G per m, the m range rounded up to whole loads
__host__ __device__ constexpr int tmem_unit_cols(int G, int H)
{
    return G * (((H + 31) / 32 + tmem_chunk(G) - 1) / tmem_chunk(G) * tmem_chunk(G));
}

// units per CTA whose rows TMEM holds: 4 quarters x floor(512 / columns per unit)
constexpr int tmem_units_max(int G, int H) { return 4 * (TMEM_COLS / tmem_unit_cols(G, H)); }

// floats of the gate rows in shared memory, rounded up to 16 bytes: the hidden tile behind them takes float4 stores
__host__ __device__ constexpr size_t gate_row_floats(int G, int U, int H)
{
    return G % 4 == 0 ? (size_t)G * U * H : ((size_t)G * U * H + 3) & ~(size_t)3;
}

struct LstmParams {
    const float *gin, *bias, *w_hh, *h0, *c0;                // GRU: bias = b_hh; c0 / cn: LSTM only
    float *y, *hn, *cn;
    int T, B, H, U, BT;
    int NT;                                                  // units per CTA in TMEM (tier instance only)
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

// ReLU as torch.relu: a NaN stays NaN (fmaxf would drop it)
__device__ __forceinline__ float relu_f(float x) { return x < 0.0f ? 0.0f : x; }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 16 (+ 8 when N = 24) consecutive columns of this warp's 32 TMEM lanes, one column per register
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&r)[N])
{
    static_assert(N == 16 || N == 24, "TMEM loads of 16 or 24 columns");
    uint32_t *u = reinterpret_cast<uint32_t *>(r);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, "
                 "%14, %15}, [%16];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                   "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr));
    if constexpr (N == 24)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(u[16]), "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]),
                       "=r"(u[23])
                     : "r"(taddr + 16));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const float (&r)[N])
{
    static_assert(N == 16 || N == 24, "TMEM stores of 16 or 24 columns");
    const uint32_t *u = reinterpret_cast<const uint32_t *>(r);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, "
                 "%14, %15, %16};"
                 ::"r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]),
                   "r"(u[8]), "r"(u[9]), "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
                 : "memory");
    if constexpr (N == 24)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                     ::"r"(taddr + 16), "r"(u[16]), "r"(u[17]), "r"(u[18]), "r"(u[19]), "r"(u[20]), "r"(u[21]),
                       "r"(u[22]), "r"(u[23])
                     : "memory");
}

template <int CELL, bool TIER>
__global__ void __launch_bounds__(LSTM_THREADS, 1) recurrence_kernel(const LstmParams p)
{
    constexpr int G = cell_gates(CELL), NB = 32 / G;        // gates per unit, batch rows per warp task
    constexpr int MC = tmem_chunk(G);                        // m values per TMEM load
    extern __shared__ __align__(16) float smem[];
    const int H = p.H, B = p.B, U = p.U;
    float *ws = smem;                                        // [G (U - NT)][H]
    float *hs = ws + gate_row_floats(G, TIER ? U - p.NT : U, H);   // [BT][H], 16-byte aligned
    float *gs = hs + (size_t)p.BT * H;                       // [warps][32]
    const int j0 = blockIdx.x * U;
    const int nu = min(U, H - j0);
    const int nt = TIER ? min(p.NT, nu) : 0;                 // units [0, nt) in TMEM, [nt, nu) in shared memory
    for (int i = threadIdx.x; i < G * (nu - nt) * H; i += LSTM_THREADS) {
        const int r = i / H, k = i - r * H;
        ws[i] = p.w_hh[(size_t)((int)((unsigned)r % G) * H + j0 + nt + (int)((unsigned)r / G)) * H + k];
    }
    cg::grid_group grid = cg::this_grid();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lgate = lane / NB, lrow = lane % NB;           // the (gate, row) whose sum lane ends up holding
    float *gw = gs + warp * 32;

    // TMEM: this warp's quarter q = warp % 4, its lanes 32 q .. +31, and the nq TMEM units (u = q + 4 s) of that quarter
    const int KC = (H + 31) >> 5, UC = tmem_unit_cols(G, H);
    const int q = warp & 3, nq = nt > q ? (nt - q + 3) >> 2 : 0;
    uint32_t tmem_base = 0, tmem = 0;
    if constexpr (TIER) {
        if (warp == 0) {                                     // gs is free until the first task: it receives the address
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"((uint32_t)__cvta_generic_to_shared(gs)), "r"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem_base = *reinterpret_cast<volatile uint32_t *>(gs);
        tmem = tmem_base + ((uint32_t)(32 * q) << 16);
        // the quarter's four warps fill its slots a load-sized chunk at a time, zeros past H
        const int nchunks = UC / (G * MC);
        for (int c = warp >> 2; c < nq * nchunks; c += 4) {
            const int s = c / nchunks, m0 = (c - s * nchunks) * MC;
            const int unit = j0 + q + 4 * s;
            float r[G * MC];
#pragma unroll
            for (int j = 0; j < G * MC; ++j) {
                const int k = (m0 + j / G) * 32 + lane;
                r[j] = k < H ? p.w_hh[(size_t)((j % G) * H + unit) * H + k] : 0.0f;
            }
            tmem_st(tmem + s * UC + m0 * G, r);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncthreads();                                     // every quarter's rows are in TMEM, gs is read
        tc_fence_after();
    }

    for (int t = 0; t < p.T; ++t) {
        const float *hprev = t == 0 ? p.h0 : p.y + (size_t)(t - 1) * B * H;
        const float *cprev = t == 0 ? p.c0 : p.cn;
        const float *gin_t = p.gin + (size_t)t * B * G * H;
        float *y_t = p.y + (size_t)t * B * H;
        for (int b0 = 0; b0 < B; b0 += p.BT) {
            const int nb = min(p.BT, B - b0);
            __syncthreads();                                 // the previous tile's readers are done (and ws is loaded)
            stage_rows(hs, hprev + (size_t)b0 * H, nb * H);
            __syncthreads();
            const int ngroups = (nb + NB - 1) / NB;
            // the shared-memory-only instance keeps its own copy of the task: sharing the tier's body changed its address
            // code, and the RNN's recurrence at 650 units lost 10 %; this way the four instances keep their SASS
            if constexpr (!TIER) {
                for (int task = warp; task < nu * ngroups; task += LSTM_WARPS) {
                    const int u = task / ngroups, jb = (task - u * ngroups) * NB;
                    const int nbg = min(NB, nb - jb);
                    const int unit = j0 + u;
                    const int b = b0 + jb + lrow;
                    const bool mine = lgate < G && lrow < nbg;
                    float pre = 0.0f;
                    if (mine) {
                        // the GRU's n gate adds gin_n only after the reset gate scaled W_hn . h + b_hn
                        if (CELL != CELL_GRU || lgate != 2) pre = gin_t[(size_t)b * G * H + lgate * H + unit];
                        if (p.bias) pre = pre + p.bias[lgate * H + unit];
                    }
                    // what the cell update needs besides the gates (the LSTM's cell state, the GRU's gin_n), fetched
                    // before the products hide its latency
                    float aux = 0.0f;
                    if (CELL == CELL_LSTM) aux = lrow < nbg && lane < NB ? cprev[(size_t)b * H + unit] : 0.0f;
                    if (CELL == CELL_GRU) aux = lrow < nbg && lane < NB ? gin_t[(size_t)b * G * H + 2 * H + unit] : 0.0f;
                    const float *w = ws + (size_t)G * u * H;
                    int hrow[NB];                                // rows past the tile repeat its last row (sums discarded)
#pragma unroll
                    for (int j = 0; j < NB; ++j) hrow[j] = (jb + min(j, nbg - 1)) * H;
                    float v[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = 0.0f;
                    for (int k = lane; k < H; k += 32) {
                        float wk[G], hk[NB];
#pragma unroll
                        for (int g = 0; g < G; ++g) wk[g] = w[g * H + k];
#pragma unroll
                        for (int j = 0; j < NB; ++j) hk[j] = hs[hrow[j] + k];
#pragma unroll
                        for (int g = 0; g < G; ++g)
#pragma unroll
                            for (int j = 0; j < NB; ++j) v[g * NB + j] = __fmaf_rn(wk[g], hk[j], v[g * NB + j]);
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
                        const size_t o = (size_t)b * H + unit;          // lane < NB: b is this lane's own batch row
                        float h;
                        if constexpr (CELL == CELL_LSTM) {
                            const float ig = sigmoid_f(gw[lane]), fg = sigmoid_f(gw[8 + lane]);
                            const float gg = tanhf(gw[16 + lane]), og = sigmoid_f(gw[24 + lane]);
                            const float c = __fmaf_rn(fg, aux, __fmul_rn(ig, gg));
                            h = __fmul_rn(og, tanhf(c));
                            p.cn[o] = c;
                        } else if constexpr (CELL == CELL_GRU) {
                            const float rg = sigmoid_f(gw[lane]), zg = sigmoid_f(gw[NB + lane]);
                            const float ng = tanhf(__fadd_rn(aux, __fmul_rn(rg, gw[2 * NB + lane])));
                            h = __fmaf_rn(zg, __fsub_rn(hs[(size_t)(jb + lane) * H + unit], ng), ng);
                        } else {
                            h = CELL == CELL_RNN_TANH ? tanhf(gw[lane]) : relu_f(gw[lane]);
                        }
                        y_t[o] = h;
                        if (t == p.T - 1) p.hn[o] = h;
                    }
                    __syncwarp();
                }
            } else {
                // one warp task: unit u with batch rows jb .. jb + NB of the tile, its gate rows at w (shared memory) or at
                // TMEM column address ta
                auto task = [&](const int u, const int jb, const float *w, const uint32_t ta, auto from_tmem) {
                    const int nbg = min(NB, nb - jb);
                    const int unit = j0 + u;
                    const int b = b0 + jb + lrow;
                    const bool mine = lgate < G && lrow < nbg;
                    float pre = 0.0f;
                    if (mine) {
                        // the GRU's n gate adds gin_n only after the reset gate scaled W_hn . h + b_hn
                        if (CELL != CELL_GRU || lgate != 2) pre = gin_t[(size_t)b * G * H + lgate * H + unit];
                        if (p.bias) pre = pre + p.bias[lgate * H + unit];
                    }
                    // what the cell update needs besides the gates (the LSTM's cell state, the GRU's gin_n), fetched
                    // before the products hide its latency
                    float aux = 0.0f;
                    if (CELL == CELL_LSTM) aux = lrow < nbg && lane < NB ? cprev[(size_t)b * H + unit] : 0.0f;
                    if (CELL == CELL_GRU) aux = lrow < nbg && lane < NB ? gin_t[(size_t)b * G * H + 2 * H + unit] : 0.0f;
                    int hrow[NB];                                // rows past the tile repeat its last row (sums discarded)
#pragma unroll
                    for (int j = 0; j < NB; ++j) hrow[j] = (jb + min(j, nbg - 1)) * H;
                    float v[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = 0.0f;
                    if constexpr (!decltype(from_tmem)::value) {
                        for (int k = lane; k < H; k += 32) {
                            float wk[G], hk[NB];
#pragma unroll
                            for (int g = 0; g < G; ++g) wk[g] = w[g * H + k];
#pragma unroll
                            for (int j = 0; j < NB; ++j) hk[j] = hs[hrow[j] + k];
#pragma unroll
                            for (int g = 0; g < G; ++g)
#pragma unroll
                                for (int j = 0; j < NB; ++j) v[g * NB + j] = __fmaf_rn(wk[g], hk[j], v[g * NB + j]);
                        }
                    } else {
                        // the same products in the same order, wk[g] out of TMEM: MC consecutive m per load
                        for (int m0 = 0; m0 < KC; m0 += MC) {
                            float wc[G * MC];
                            tmem_ld(ta + m0 * G, wc);
#pragma unroll
                            for (int mm = 0; mm < MC; ++mm) {
                                const int k = (m0 + mm) * 32 + lane;
                                if (k < H) {
                                    float hk[NB];
#pragma unroll
                                    for (int j = 0; j < NB; ++j) hk[j] = hs[hrow[j] + k];
#pragma unroll
                                    for (int g = 0; g < G; ++g)
#pragma unroll
                                        for (int j = 0; j < NB; ++j)
                                            v[g * NB + j] = __fmaf_rn(wc[mm * G + g], hk[j], v[g * NB + j]);
                                }
                            }
                        }
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
                        const size_t o = (size_t)b * H + unit;          // lane < NB: b is this lane's own batch row
                        float h;
                        if constexpr (CELL == CELL_LSTM) {
                            const float ig = sigmoid_f(gw[lane]), fg = sigmoid_f(gw[8 + lane]);
                            const float gg = tanhf(gw[16 + lane]), og = sigmoid_f(gw[24 + lane]);
                            const float c = __fmaf_rn(fg, aux, __fmul_rn(ig, gg));
                            h = __fmul_rn(og, tanhf(c));
                            p.cn[o] = c;
                        } else if constexpr (CELL == CELL_GRU) {
                            const float rg = sigmoid_f(gw[lane]), zg = sigmoid_f(gw[NB + lane]);
                            const float ng = tanhf(__fadd_rn(aux, __fmul_rn(rg, gw[2 * NB + lane])));
                            h = __fmaf_rn(zg, __fsub_rn(hs[(size_t)(jb + lane) * H + unit], ng), ng);
                        } else {
                            h = CELL == CELL_RNN_TANH ? tanhf(gw[lane]) : relu_f(gw[lane]);
                        }
                        y_t[o] = h;
                        if (t == p.T - 1) p.hn[o] = h;
                    }
                    __syncwarp();
                };
                for (int i = warp >> 2; i < nq * ngroups; i += 4) {
                    const int s = i / ngroups;
                    task(q + 4 * s, (i - s * ngroups) * NB, nullptr, tmem + s * UC, std::true_type{});
                }
                for (int i = warp; i < (nu - nt) * ngroups; i += LSTM_WARPS) {
                    const int r = i / ngroups;
                    task(nt + r, (i - r * ngroups) * NB, ws + (size_t)G * r * H, 0u, std::false_type{});
                }
            }
        }
        grid.sync();                                         // h_t complete (and visible) before anyone reads it
    }

    if constexpr (TIER) {                                    // every CTA releases its columns: the kernel has no other exit
        tc_fence_before();
        __syncthreads();
        if (warp == 0)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// shared memory of a CTA holding the G gate rows of U units and a tile of BT hidden rows
size_t recurrence_smem(int G, int H, int U, int BT)
{
    return (gate_row_floats(G, U, H) + (size_t)BT * H) * sizeof(float) + LSTM_GATE_SMEM;
}

// units per CTA whose rows go to TMEM: none while all U fit in shared memory next to one hidden row (the
// shared-memory-only instance), otherwise as many as TMEM holds
int recurrence_tmem_units(int G, int H, int U, size_t smem_optin)
{
    return recurrence_smem(G, H, U, 1) <= smem_optin ? 0 : std::min(U, tmem_units_max(G, H));
}

// U = ceil(H / SMs) units per CTA (one CTA per SM at most); the rows of the units TMEM does not hold must fit in shared
// memory together with at least one hidden row
bool recurrence_fits(int G, int H, int sms, size_t smem_optin)
{
    const int U = (H + sms - 1) / sms;
    return recurrence_smem(G, H, U - recurrence_tmem_units(G, H, U, smem_optin), 1) <= smem_optin;
}

// the one statement of the hidden-size bound: the refusals below and tq_recurrence_max_hidden report it
int recurrence_max_hidden(int G, int sms, size_t smem_optin)
{
    int best = 0;
    for (int H = 1; H <= 65536; ++H)
        if (recurrence_fits(G, H, sms, smem_optin)) best = H;
    return best;
}

int smem_optin(int *optin)
{
    int dev = 0;
    return cudaGetDevice(&dev) == cudaSuccess &&
           cudaDeviceGetAttribute(optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess;
}

const char *const KERNEL_NAME[] = {"lstm_recurrence_kernel", "gru_recurrence_kernel", "rnn_tanh_recurrence_kernel",
                                   "rnn_relu_recurrence_kernel"};

// the checks and launch every cell shares; p holds the operands, T, B and H
template <int CELL>
int launch_recurrence(const char *entry, LstmParams p, uintptr_t addr, void *stream)
{
    constexpr int G = cell_gates(CELL);
    const char *kname = KERNEL_NAME[CELL];
    const int T = p.T, B = p.B, H = p.H;
    if (addr & 3u) return fail(TQ_ERR_INVALID, "pointers must be 4-byte aligned (fp32 tensors)");
    if (T < 1 || B < 1 || H < 1) return fail(TQ_ERR_INVALID, "T = %d, B = %d, H = %d: each must be at least 1", T, B, H);
    if ((int64_t)B * G * H > INT32_MAX)
        return fail(TQ_ERR_INVALID, "B * %dH = %lld exceeds 2^31 - 1", G, (long long)B * G * H);
    int optin = 0;
    if (!smem_optin(&optin)) return fail(TQ_ERR_CUDA, "%s: cannot read the device's shared-memory limit", entry);
    const int sms = num_sms();
    p.U = (H + sms - 1) / sms;
    if (!recurrence_fits(G, H, sms, (size_t)optin)) {
        const int nt = recurrence_tmem_units(G, H, p.U, (size_t)optin);
        return fail(TQ_ERR_UNSUPPORTED, "H = %d: %d units per CTA, %d of them in tensor memory; the %d x %d gate rows of the "
                    "rest and one hidden row need %zu bytes of shared memory, %d are available (largest H on this device: "
                    "%d)", H, p.U, nt, G, p.U - nt, recurrence_smem(G, H, p.U - nt, 1), optin,
                    recurrence_max_hidden(G, sms, (size_t)optin));
    }
    p.NT = recurrence_tmem_units(G, H, p.U, (size_t)optin);
    if (const char *env = getenv("TQ_RECURRENCE_TMEM_UNITS"))
        p.NT = std::max(0, std::min(atoi(env), std::min(p.U, tmem_units_max(G, H))));
    if (recurrence_smem(G, H, p.U - p.NT, 1) > (size_t)optin)
        return fail(TQ_ERR_UNSUPPORTED, "H = %d: TQ_RECURRENCE_TMEM_UNITS=%d leaves %d units per CTA in shared memory, more "
                    "than fit", H, p.NT, p.U - p.NT);
    void (*const kernel)(LstmParams) = p.NT ? recurrence_kernel<CELL, true> : recurrence_kernel<CELL, false>;
    const int blocks = (H + p.U - 1) / p.U;
    const size_t fixed = recurrence_smem(G, H, p.U - p.NT, 0);
    const size_t rows = ((size_t)optin - fixed) / ((size_t)H * sizeof(float));
    p.BT = (int)(rows < (size_t)B ? rows : (size_t)B);
    const size_t smem = recurrence_smem(G, H, p.U - p.NT, p.BT);
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return fail(TQ_ERR_CUDA, "cudaFuncSetAttribute(%s): %s", kname, cudaGetErrorString(cudaGetLastError()));
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, LSTM_THREADS, smem) != cudaSuccess)
        return fail(TQ_ERR_CUDA, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(%s): %s", kname,
                    cudaGetErrorString(cudaGetLastError()));
    if ((int64_t)per_sm * sms < blocks)
        return fail(TQ_ERR_UNSUPPORTED, "%s: %d CTAs cannot all be resident (%d per SM x %d SMs)", kname, blocks, per_sm, sms);

    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(LSTM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(TQ_ERR_CUDA, "%s (cooperative launch of %d CTAs): %s", kname, blocks, cudaGetErrorString(e));
    }
    count_launch();
    return check_launch(kname);
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
    const LstmParams p = {gin, bias, w_hh, h0, c0, y, hn, cn, T, B, H, 0, 0, 0};
    return launch_recurrence<CELL_LSTM>("tq_lstm_recurrence", p, addr, stream);
}

extern "C" int tq_gru_recurrence(const float *gin, const float *b_hh, const float *w_hh, const float *h0, float *y,
                                 float *hn, int T, int B, int H, void *stream)
{
    if (!gin || !w_hh || !h0 || !y || !hn) return fail(TQ_ERR_INVALID, "NULL pointer");
    const uintptr_t addr = (uintptr_t)gin | (uintptr_t)b_hh | (uintptr_t)w_hh | (uintptr_t)h0 | (uintptr_t)y |
                           (uintptr_t)hn;
    const LstmParams p = {gin, b_hh, w_hh, h0, nullptr, y, hn, nullptr, T, B, H, 0, 0, 0};
    return launch_recurrence<CELL_GRU>("tq_gru_recurrence", p, addr, stream);
}

extern "C" int tq_rnn_recurrence(const float *gin, const float *bias, const float *w_hh, const float *h0, float *y,
                                 float *hn, int T, int B, int H, int relu, void *stream)
{
    if (!gin || !w_hh || !h0 || !y || !hn) return fail(TQ_ERR_INVALID, "NULL pointer");
    const uintptr_t addr = (uintptr_t)gin | (uintptr_t)bias | (uintptr_t)w_hh | (uintptr_t)h0 | (uintptr_t)y |
                           (uintptr_t)hn;
    const LstmParams p = {gin, bias, w_hh, h0, nullptr, y, hn, nullptr, T, B, H, 0, 0, 0};
    return relu ? launch_recurrence<CELL_RNN_RELU>("tq_rnn_recurrence", p, addr, stream)
                : launch_recurrence<CELL_RNN_TANH>("tq_rnn_recurrence", p, addr, stream);
}

extern "C" int tq_recurrence_max_hidden(int gates)
{
    if (gates != 1 && gates != 3 && gates != 4)
        return fail(TQ_ERR_INVALID, "gates = %d: 4 (LSTM), 3 (GRU) or 1 (RNN)", gates), -1;
    int optin = 0;
    if (!smem_optin(&optin)) return fail(TQ_ERR_CUDA, "tq_recurrence_max_hidden: cannot read the device's shared-memory limit"), -1;
    return recurrence_max_hidden(gates, num_sms(), (size_t)optin);
}
