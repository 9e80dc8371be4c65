// tq_encode.cu -- term-reveal encode-and-truncate kernels for B200 (sm_100a).
//
// Replaces tr_cuda_kernel (kernels/tr_cuda_kernel.cu:58-125): that kernel launches one
// thread per ELEMENT of which 1/g do work, keeps 8.3 KB of term lists per thread in local
// memory and uses scalar strided accesses.  Here the term list never exists: a value's
// terms are two bit masks (term_masks), and "the alpha largest terms of the group" is a
// cut level p* found by counting set bits -- every term above p* survives, at p* the first
// r values (lowest channel first) keep theirs, everything below is dropped.
//
// Three kernels:
//   tr_elem_kernel    g == 1 (every activation, tr_layer.py:97-98).  A pure stream:
//                     128-bit loads/stores, 4 vectors in flight per thread, persistent grid
//                     sized to the SM count.  For bits <= 12 the whole quantised-value ->
//                     output map is a 2^(bits+1)-entry table in shared memory built once per
//                     CTA, so the per-element work is divide, round, one LDS.
//   tr_group_kernel   g in {2,4,8,16,32}, fp32 (weights, tr_layer.py:120,148,178,185):
//                     one thread owns one group in registers, popc-based binary search for
//                     the cut level; vector loads when groups are contiguous (WH == 1).
//   tr_generic_kernel anything else (odd g, tail groups, fp64/bf16/f16 groups, misaligned
//                     pointers): same selection rule, plain loops.
//
// HBM traffic is the algorithmic minimum: each element is read once and written once.
#include <cstdlib>
#include <type_traits>

#include "tq_common.cuh"

namespace tq {

struct EncParams {
    float sf;
    float maxv;      // 2^bits - 1
    int bits;
    int alpha;       // budget per group (g == 1: terms per value)
    int enc;
    int relu;
    int fastdiv;     // 2^-30 <= sf <= 2^30: hoisted-reciprocal divide is exact (tq_common.cuh)
};

// =========================================================================================
// g == 1 : elementwise stream
// =========================================================================================
constexpr int ELEM_THREADS = 256;

template <typename Tin, typename Tout, bool DEQ, bool FAST>
__device__ __forceinline__ Tout elem_out_compute(Tin xin, const EncParams &p, const Quant &k, bool &ovf)
{
    uint32_t neg;
    const uint32_t q = quantize_any<Tin, FAST>(xin, k, p.relu != 0, neg);
    int code = elem_code(q, p.enc, p.alpha);
    code = neg ? -code : code;
    if constexpr (DEQ) {
        return dequant<Tout>(code, p.sf);
    } else {
        return pack_code<Tout>(code, ovf);
    }
}

// table entry: the final output bit pattern (<= 32 bit) for index q | neg << bits.  Integer
// codes narrower than 32 bit carry "did not fit" in bit 31.
template <typename Tout, bool DEQ>
__device__ __forceinline__ uint32_t lut_entry(uint32_t idx, const EncParams &p)
{
    if constexpr (sizeof(Tout) > 4) {
        return 0u;                                   // fp64 never takes the table path
    } else {
        const uint32_t q = idx & ((1u << p.bits) - 1u);
        const uint32_t neg = idx >> p.bits;
        int code = elem_code(q, p.enc, p.alpha);
        code = neg ? -code : code;
        uint32_t b = 0u;
        if constexpr (DEQ) {
            const Tout o = dequant<Tout>(code, p.sf);
            memcpy(&b, &o, sizeof(Tout));
        } else {
            bool ov = false;
            const Tout o = pack_code<Tout>(code, ov);
            memcpy(&b, &o, sizeof(Tout));
            if (sizeof(Tout) < 4 && ov) b |= 0x80000000u;
        }
        return b;
    }
}

template <typename Tout>
__device__ __forceinline__ Tout lut_decode(uint32_t e)
{
    Tout o;
    if constexpr (sizeof(Tout) > 4) o = Tout(0);
    else memcpy(&o, &e, sizeof(Tout));
    return o;
}

template <typename Tin, typename Tout, bool DEQ, bool FAST, int ELEM_UNROLL>
__global__ void __launch_bounds__(ELEM_THREADS)
tr_elem_kernel(const Tin *__restrict__ in, Tout *__restrict__ out, int64_t n, EncParams p,
               int use_lut, int *__restrict__ overflow)
{
    constexpr int VEC = 16 / sizeof(Tin);
    using VIn = Vec<Tin, VEC>;
    using VOut = Vec<Tout, VEC>;
    extern __shared__ uint32_t lut[];
    bool ovf = false;
    const Quant k = make_quant(p.sf, p.maxv);
    const bool relu = p.relu != 0;
    const int bits = p.bits;

    if (use_lut) {
        const uint32_t entries = 2u << p.bits;
        for (uint32_t i = threadIdx.x; i < entries; i += ELEM_THREADS) lut[i] = lut_entry<Tout, DEQ>(i, p);
        __syncthreads();
    }

    const int64_t nvec = n / VEC;
    const int64_t chunk = (int64_t)ELEM_THREADS * ELEM_UNROLL;
    const int64_t nchunks = (nvec + chunk - 1) / chunk;
    const VIn *vin = reinterpret_cast<const VIn *>(in);
    VOut *vout = reinterpret_cast<VOut *>(out);

    for (int64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
        const int64_t v0 = c * chunk + threadIdx.x;
        VIn x[ELEM_UNROLL];
#pragma unroll
        for (int u = 0; u < ELEM_UNROLL; ++u) {
            const int64_t vi = v0 + (int64_t)u * ELEM_THREADS;
            if (vi < nvec) {
                const int4 raw = __ldcs(reinterpret_cast<const int4 *>(vin + vi));
                memcpy(&x[u], &raw, 16);
            }
        }
#pragma unroll
        for (int u = 0; u < ELEM_UNROLL; ++u) {
            const int64_t vi = v0 + (int64_t)u * ELEM_THREADS;
            if (vi < nvec) {
                VOut y;
                if (use_lut) {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        uint32_t neg;
                        const uint32_t q = quantize_any<Tin, FAST>(x[u].v[e], k, relu, neg);
                        const uint32_t ent = lut[q | (neg << bits)];
                        if (!DEQ && sizeof(Tout) < 4) ovf |= (ent >> 31) != 0u;
                        y.v[e] = lut_decode<Tout>(ent);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) y.v[e] = elem_out_compute<Tin, Tout, DEQ, FAST>(x[u].v[e], p, k, ovf);
                }
                vout[vi] = y;
            }
        }
    }

    // ragged tail (n % VEC elements), one thread
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (int64_t i = nvec * VEC; i < n; ++i) out[i] = elem_out_compute<Tin, Tout, DEQ, FAST>(in[i], p, k, ovf);
    }
    if (!DEQ && ovf && overflow) atomicExch(overflow, 1);
}

// =========================================================================================
// g in {2,4,8,16,32}, fp32 : one thread per group, registers only
// =========================================================================================
constexpr int GROUP_THREADS = 128;

// number of terms at level >= p over the group; W packs two 16-bit term masks per word
template <int NW>
__device__ __forceinline__ int count_at_or_above(const uint32_t (&W)[NW], int p)
{
    const uint32_t m = ((0xFFFFu << p) & 0xFFFFu) * 0x00010001u;
    int c = 0;
#pragma unroll
    for (int i = 0; i < NW; ++i) c += __popc(W[i] & m);
    return c;
}

constexpr int GROUP_LUT_MAX_BITS = 12;          // 2^bits entries of (T | N << 16) in shared memory: 16 KB at most

// LAYOUT 0: groups strided by WH in global memory (large planes: consecutive threads take consecutive wh, coalesced);
// LAYOUT 1: contiguous groups (WH == 1): 128-bit loads / stores per group;
// LAYOUT 2: small planes (conv weights, WH = kh * kw = 9, 25, 49: the reference's real weight layout, tr_layer.py:117-120):
//           a block of G * WH consecutive elements holds exactly WH complete groups, so a CTA copies whole blocks into
//           shared memory with coalesced 128-bit loads, every thread picks its group out of shared memory (stride WH,
//           conflict-free across the threads of a warp), writes the result back in place, and the tile leaves with
//           coalesced 128-bit stores.  The strided variant touches ~8 sectors per warp load on such tensors (1.1 TB/s).
template <int G, int LAYOUT, typename Tout, bool DEQ, bool FAST>
__global__ void __launch_bounds__(GROUP_THREADS)
tr_group_kernel(const float *__restrict__ in, Tout *__restrict__ out,
                int64_t B, int64_t C, int64_t WH, EncParams p, int use_lut, int lut_bytes, int *__restrict__ overflow)
{
    constexpr bool CONTIG = LAYOUT == 1;
    static_assert(G >= 2 && G <= 32 && (G & (G - 1)) == 0, "G must be a power of two");
    constexpr int NW = G / 2;
    extern __shared__ uint32_t tn_lut[];            // q -> T | N << 16 (term presence / negative-term masks)
    const Quant k = make_quant(p.sf, p.maxv);
    const int64_t CG = C / G;                       // caller guarantees C % G == 0
    const int64_t total = B * CG * WH;
    bool ovf = false;
    if (use_lut == 2) {
        // 16-byte entries: bytes 0..11 = number of terms of q at level >= 0..11 (cumulative from the top), word 3 =
        // T | N << 16.  Adding the entries of a group gives its term count at EVERY level at once.
        for (uint32_t q = threadIdx.x; q < (1u << p.bits); q += GROUP_THREADS) {
            uint32_t T, N;
            term_masks(q, p.enc, T, N);
            uint32_t w[3] = {0u, 0u, 0u};
#pragma unroll
            for (int lvl = 0; lvl < 12; ++lvl) w[lvl >> 2] |= (uint32_t)__popc(T >> lvl) << (8 * (lvl & 3));
            reinterpret_cast<uint4 *>(tn_lut)[q] = make_uint4(w[0], w[1], w[2], T | (N << 16));
        }
        __syncthreads();
    } else if (use_lut) {
        for (uint32_t q = threadIdx.x; q < (1u << p.bits); q += GROUP_THREADS) {
            uint32_t T, N;
            term_masks(q, p.enc, T, N);
            tn_lut[q] = T | (N << 16);
        }
        __syncthreads();
    }
    const uint32_t lut_base = (uint32_t)__cvta_generic_to_shared(tn_lut);

    // quantise the g values of one group, find the cut level of its term budget, rebuild the surviving codes
    auto select = [&](const float (&x)[G], Tout (&y)[G]) {
        uint32_t tn[G];                              // T | N << 16 | sign << 31   (T, N < 2^15)
        const bool relu = p.relu != 0;
        int pc, r;
        bool cut;
        const int alpha = p.alpha, bits = p.bits;
        if (use_lut == 2) {
            // group term counts at every level from one 16-byte lookup + 3 adds per value (bytes cannot carry: <= 7
            // terms per value, G <= 16); the levels whose count exceeds alpha are 0..pc, so pc = (#such levels) - 1
            uint32_t S0 = 0u, S1 = 0u, S2 = 0u;
#pragma unroll
            for (int j = 0; j < G; ++j) {
                uint32_t neg;
                const uint32_t q = quantize_any<float, FAST>(x[j], k, relu, neg);
                uint32_t a0, a1, a2, e;
                asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(e) : "r"(lut_base + q * 16u));
                S0 += a0; S1 += a1; S2 += a2;
                tn[j] = e | (neg << 31);
            }
            const uint32_t K = (uint32_t)(127 - alpha) * 0x01010101u;          // byte > alpha  <=>  bit 7 of byte + 127 - alpha
            const int nlev = __popc((S0 + K) & 0x80808080u) + __popc((S1 + K) & 0x80808080u) + __popc((S2 + K) & 0x80808080u);
            cut = nlev > 0;
            pc = cut ? nlev - 1 : 0;
            const int idx = pc + 1;                                             // count at levels > pc
            const uint32_t w = idx < 4 ? S0 : (idx < 8 ? S1 : S2);
            const int above = idx >= 12 ? 0 : (int)((w >> (8 * (idx & 3))) & 0xFFu);
            r = alpha - above;
        } else {
            uint32_t W[NW];                              // two T masks per word, for the counting probes
            if (use_lut) {                               // one branch per group, one LDS per value (32-bit shared address)
#pragma unroll
                for (int j = 0; j < G; ++j) {
                    uint32_t neg;
                    const uint32_t q = quantize_any<float, FAST>(x[j], k, relu, neg);
                    uint32_t e;
                    asm("ld.shared.u32 %0, [%1];" : "=r"(e) : "r"(lut_base + q * 4u));
                    if (j & 1) W[j >> 1] |= e << 16; else W[j >> 1] = e & 0xFFFFu;
                    tn[j] = e | (neg << 31);
                }
            } else {
#pragma unroll
                for (int j = 0; j < G; ++j) {
                    uint32_t neg;
                    const uint32_t q = quantize_any<float, FAST>(x[j], k, relu, neg);
                    uint32_t T, N;
                    term_masks(q, p.enc, T, N);
                    const uint32_t e = T | (N << 16);
                    if (j & 1) W[j >> 1] |= e << 16; else W[j >> 1] = e & 0xFFFFu;
                    tn[j] = e | (neg << 31);
                }
            }
            // cut level: largest pc with (#terms at level >= pc) > alpha; none -> keep everything.
            // Branch-free (selects, no divergence between the groups of a warp): 4-probe binary search over levels 0..15.
            cut = count_at_or_above<NW>(W, 0) > alpha;
            pc = 0;
#pragma unroll
            for (int step = 8; step >= 1; step >>= 1) {
                const int cand = pc + step;
                const int c = count_at_or_above<NW>(W, cand);
                pc = (cand <= bits && c > alpha) ? cand : pc;
            }
            r = alpha - count_at_or_above<NW>(W, pc + 1);                       // (pc + 1 == 16 -> empty mask -> 0)
        }
        const uint32_t cutbit = cut ? (1u << pc) : 0u;
        const uint32_t himask = cut ? (0xFFFFu & ~((2u << pc) - 1u)) : 0xFFFFu;

        int cnt = 0;
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const uint32_t e = tn[j];
            const uint32_t at = (e & cutbit) != 0u ? 1u : 0u;       // a term at the cut level: the first r of the group keep it
            const uint32_t K = (e & himask) | ((at != 0u && cnt < r) ? cutbit : 0u);
            cnt += (int)at;
            const int v = (int)K - 2 * (int)(K & (e >> 16) & 0x7FFFu);
            const int code = ((int)e < 0) ? -v : v;
            if constexpr (DEQ) y[j] = dequant<Tout>(code, p.sf);
            else y[j] = pack_code<Tout>(code, ovf);
        }
    };

    if constexpr (LAYOUT == 2) {
        // tile = nb blocks of G * WH floats = nb * WH groups (nb * WH <= GROUP_THREADS); fp32 in, fp32 out only
        float *tile = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(tn_lut) + lut_bytes);
        const int wh_i = (int)WH, blk_elems = G * wh_i;
        const int nb_max = GROUP_THREADS / wh_i;
        const int64_t n_blocks = B * CG;
        const int64_t n_tiles = (n_blocks + nb_max - 1) / nb_max;
        for (int64_t tix = blockIdx.x; tix < n_tiles; tix += gridDim.x) {
            const int64_t blk0 = tix * nb_max;
            const int nb = (int)((n_blocks - blk0) < nb_max ? (n_blocks - blk0) : nb_max);
            const int elems = nb * blk_elems;                     // a multiple of 4 (G >= 4) and 16-byte aligned in memory
            const float *src = in + blk0 * blk_elems;
            float *dst = reinterpret_cast<float *>(out) + blk0 * blk_elems;
            for (int i = threadIdx.x * 4; i < elems; i += GROUP_THREADS * 4)
                *reinterpret_cast<int4 *>(tile + i) = __ldcs(reinterpret_cast<const int4 *>(src + i));
            __syncthreads();
            if ((int)threadIdx.x < nb * wh_i) {
                const int blk = (int)threadIdx.x / wh_i, wh = (int)threadIdx.x % wh_i;
                float *gp = tile + blk * blk_elems + wh;
                float x[G];
#pragma unroll
                for (int j = 0; j < G; ++j) x[j] = gp[j * wh_i];
                Tout y[G];
                select(x, y);
#pragma unroll
                for (int j = 0; j < G; ++j) gp[j * wh_i] = (float)y[j];
            }
            __syncthreads();
            for (int i = threadIdx.x * 4; i < elems; i += GROUP_THREADS * 4)
                __stcs(reinterpret_cast<int4 *>(dst + i), *reinterpret_cast<const int4 *>(tile + i));
            __syncthreads();
        }
    }
    if constexpr (LAYOUT == 1 && G >= 4 && (sizeof(Tout) * G) % 16 == 0) {
        // contiguous groups, 128-bit accesses: the NEXT group of this thread is requested before the current one is
        // encoded (registers as a second buffer), which doubles the bytes in flight per SM at the same occupancy --
        // with one group per thread in flight the kernel sat at ~32 KB per SM, short of what HBM latency x bandwidth asks
        constexpr int NV = (G * 4) / 16, NVO = (int)(sizeof(Tout) * G) / 16;
        const int64_t step = (int64_t)gridDim.x * GROUP_THREADS;
        int64_t t = (int64_t)blockIdx.x * GROUP_THREADS + threadIdx.x;
        int4 cur[NV], nxt[NV];
        if (t < total) {
#pragma unroll
            for (int v = 0; v < NV; ++v) cur[v] = __ldcs(reinterpret_cast<const int4 *>(in + t * G) + v);
        }
        while (t < total) {
            const int64_t tn = t + step;
            if (tn < total) {
#pragma unroll
                for (int v = 0; v < NV; ++v) nxt[v] = __ldcs(reinterpret_cast<const int4 *>(in + tn * G) + v);
            }
            float x[G];
#pragma unroll
            for (int v = 0; v < NV; ++v) memcpy(&x[v * 4], &cur[v], 16);
            Tout y[G];
            select(x, y);
            int4 *dst = reinterpret_cast<int4 *>(out + t * G);
#pragma unroll
            for (int v = 0; v < NVO; ++v) {
                int4 raw;
                memcpy(&raw, reinterpret_cast<const char *>(y) + 16 * v, 16);
                __stcs(dst + v, raw);
            }
#pragma unroll
            for (int v = 0; v < NV; ++v) cur[v] = nxt[v];
            t = tn;
        }
    } else
    if constexpr (LAYOUT != 2)
    for (int64_t t = (int64_t)blockIdx.x * GROUP_THREADS + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * GROUP_THREADS) {
        int64_t base, stride;
        if (CONTIG) {
            base = t * G;
            stride = 1;
        } else {
            const int64_t wh = t % WH;
            const int64_t bc = t / WH;              // = b * CG + cg
            base = bc * G * WH + wh;
            stride = WH;
        }

        float x[G];
        if (CONTIG) {
            constexpr int NV = (G * 4) / 16 ? (G * 4) / 16 : 1;
            if constexpr (G >= 4) {
                const int4 *src = reinterpret_cast<const int4 *>(in + base);
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const int4 raw = __ldcs(src + v);
                    memcpy(&x[v * 4], &raw, 16);
                }
            } else {
                const float2 raw = __ldcs(reinterpret_cast<const float2 *>(in + base));
                x[0] = raw.x; x[1] = raw.y;
            }
        } else {
#pragma unroll
            for (int j = 0; j < G; ++j) x[j] = __ldg(in + base + j * stride);
        }

        Tout y[G];
        select(x, y);
        constexpr int OUT_BYTES = (int)sizeof(Tout) * G;
        if (CONTIG && OUT_BYTES % 16 == 0) {
            int4 *dst = reinterpret_cast<int4 *>(out + base);
#pragma unroll
            for (int v = 0; v < OUT_BYTES / 16; ++v) {
                int4 raw;
                memcpy(&raw, reinterpret_cast<const char *>(y) + 16 * v, 16);
                dst[v] = raw;
            }
        } else if (CONTIG && OUT_BYTES == 8) {
            int2 raw;
            memcpy(&raw, y, 8);
            *reinterpret_cast<int2 *>(out + base) = raw;
        } else if (CONTIG && OUT_BYTES == 4) {
            int raw;
            memcpy(&raw, y, 4);
            *reinterpret_cast<int *>(out + base) = raw;
        } else {
#pragma unroll
            for (int j = 0; j < G; ++j) out[base + j * stride] = y[j];
        }
    }
    if (!DEQ && ovf && overflow) atomicExch(overflow, 1);
}

// =========================================================================================
// generic fallback: any g <= 32, any dtype, tail groups, any alignment
// =========================================================================================
template <typename Tin, typename Tout, bool DEQ>
__global__ void __launch_bounds__(128)
tr_generic_kernel(const Tin *__restrict__ in, Tout *__restrict__ out,
                  int64_t B, int64_t C, int64_t WH, int g, EncParams p, int *__restrict__ overflow)
{
    const int64_t CG = (C + g - 1) / g;
    const int64_t total = B * CG * WH;
    bool ovf = false;
    const Quant k = make_quant(p.sf, p.maxv);
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t wh = t % WH;
        const int64_t bc = t / WH;
        const int64_t cg = bc % CG;
        const int64_t b = bc / CG;
        const int n = (int)((cg * g + g <= C) ? g : (C - cg * g));   // tail group: C % g values
        const int64_t base = (b * C + cg * g) * WH + wh;

        uint32_t T[TQ_MAX_GROUP], N[TQ_MAX_GROUP];
        uint32_t negmask = 0u;
        for (int j = 0; j < n; ++j) {
            uint32_t neg;
            const uint32_t q = quantize_any<Tin, false>(in[base + (int64_t)j * WH], k, p.relu != 0, neg);
            negmask |= neg << j;
            term_masks(q, p.enc, T[j], N[j]);
        }
        // walk levels from the top until the budget runs out
        int rem = p.alpha, pc = -1, r = 0;
        for (int lvl = p.bits; lvl >= 0; --lvl) {
            int c = 0;
            for (int j = 0; j < n; ++j) c += (T[j] >> lvl) & 1u;
            if (c > rem) { pc = lvl; r = rem; break; }
            rem -= c;
        }
        const uint32_t cutbit = pc >= 0 ? (1u << pc) : 0u;
        const uint32_t himask = pc >= 0 ? ~((cutbit << 1) - 1u) : 0xFFFFFFFFu;
        int cnt = 0;
        for (int j = 0; j < n; ++j) {
            uint32_t K = T[j] & himask;
            if (T[j] & cutbit) { if (cnt < r) K |= cutbit; ++cnt; }
            int v = (int)K - 2 * (int)(K & N[j]);
            v = ((negmask >> j) & 1u) ? -v : v;
            const int64_t idx = base + (int64_t)j * WH;
            if constexpr (DEQ) out[idx] = dequant<Tout>(v, p.sf);
            else out[idx] = pack_code<Tout>(v, ovf);
        }
    }
    if (!DEQ && ovf && overflow) atomicExch(overflow, 1);
}

// =========================================================================================
// host dispatch
// =========================================================================================
static int grid_for(int64_t work_items, int threads, int ctas_per_sm)
{
    const int64_t need = (work_items + threads - 1) / threads;
    const int64_t cap = (int64_t)num_sms() * ctas_per_sm;
    return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

template <typename Tin, typename Tout, bool DEQ>
static int launch_elem(const void *in, void *out, int64_t n, const EncParams &p, int *overflow,
                       cudaStream_t s)
{
    constexpr int VEC = 16 / sizeof(Tin);
    static const int tune_unroll = getenv("TQ_ELEM_UNROLL") ? atoi(getenv("TQ_ELEM_UNROLL")) : 4;
    static const int tune_ctas = getenv("TQ_ELEM_CTAS") ? atoi(getenv("TQ_ELEM_CTAS")) : 16;   // > resident: waves balance the two dies
    const int unroll = tune_unroll == 8 ? 8 : (tune_unroll == 2 ? 2 : 4);
    const int use_lut = (p.bits <= 12 && sizeof(Tout) <= 4 && n >= 4096) ? 1 : 0;
    const size_t smem = use_lut ? (size_t)(2u << p.bits) * sizeof(uint32_t) : 0;
    const int64_t chunks = (n / VEC + ELEM_THREADS * unroll - 1) / (ELEM_THREADS * unroll);
    int grid = (int)(chunks < 1 ? 1 : chunks);
    const int cap = num_sms() * tune_ctas;
    if (grid > cap) grid = cap;
#define TQ_LAUNCH_E(FD, UN)                                                                     \
    tr_elem_kernel<Tin, Tout, DEQ, FD, UN><<<grid, ELEM_THREADS, smem, s>>>(                    \
        (const Tin *)in, (Tout *)out, n, p, use_lut, overflow)
    if (!p.fastdiv) TQ_LAUNCH_E(false, 4);
    else if (unroll == 8) TQ_LAUNCH_E(true, 8);
    else if (unroll == 2) TQ_LAUNCH_E(true, 2);
    else TQ_LAUNCH_E(true, 4);
#undef TQ_LAUNCH_E
    count_launch();
    return check_launch("tr_elem_kernel");
}

template <typename Tout, bool DEQ>
static int launch_group_f32(const void *in, void *out, int64_t B, int64_t C, int64_t WH, int g,
                            const EncParams &p, int *overflow, cudaStream_t s)
{
    const int64_t total = B * (C / g) * WH;
    const int grid = grid_for(total, GROUP_THREADS, 16);
    const bool contig = (WH == 1);
    // the term-mask table pays for itself once a CTA has a few thousand values to encode
    int use_lut = (p.bits <= GROUP_LUT_MAX_BITS && total * g >= (int64_t)grid * (8 << p.bits)) ? 1 : 0;
    // 16-byte entries (cumulative term counts per level): bits <= 10 (levels 0..10 in 12 bytes, 16 KB); alpha <= 127
    // keeps the compare trick inside a byte.  Pays for g <= 8 (measured: g=8 4.18 -> 4.55 TB/s, g=4 3.45 -> 3.91);
    // at g = 16 the six popcount probes are amortised over 16 values and the 4-byte table wins (4.59 vs 3.93 TB/s)
    static const bool no_lut16 = getenv("TQ_GROUP_NO_LUT16") != nullptr;
    if (use_lut && !no_lut16 && p.bits <= 10 && g <= 8 && p.alpha <= 127) use_lut = 2;
    const size_t lut_bytes = use_lut == 2 ? ((size_t)16 << p.bits) : (use_lut ? (sizeof(uint32_t) << p.bits) : 0);
    // small planes (conv weights): staged through shared memory.  fp32 -> fp32, g >= 4 (blocks of g * WH floats stay
    // 16-byte aligned), whole tensor 16-byte aligned
    // MEASURED (B200, 9-bit, g = 8): slower than the strided variant, whose sector over-fetch is absorbed by L1 --
    // OIHW 512x512x3x3: 735 vs 965 GB/s, 2048x1024x3x3: 2.5 vs 3.5 TB/s (three barriers per 4 KB tile, the term table
    // rebuilt per CTA for ~4 tiles of work).  Kept as an opt-in experiment (TQ_GROUP_STAGED=1); weights are term-revealed
    // once per model conversion, not per forward.
    static const bool want_staged = getenv("TQ_GROUP_STAGED") != nullptr;
    const bool staged = want_staged && !contig && DEQ && std::is_same<Tout, float>::value && WH <= 64 && g >= 4 &&
                        (((uintptr_t)in | (uintptr_t)out) & 15u) == 0;
    size_t smem = lut_bytes;
    int grid_l = grid;
    if (staged) {
        const int nb_max = GROUP_THREADS / (int)WH;
        smem += (size_t)nb_max * g * WH * sizeof(float);
        const int64_t n_tiles = (B * (C / g) + nb_max - 1) / nb_max;
        const int64_t cap = (int64_t)num_sms() * 8;
        grid_l = (int)(n_tiles < cap ? n_tiles : cap);
        if (use_lut && total * g < (int64_t)grid_l * (8 << p.bits)) { use_lut = 0; smem -= lut_bytes; }
    }
    if (smem > 48 * 1024) return fail(TQ_ERR_UNSUPPORTED, "internal: grouped kernel shared memory");
    const int lutb = (int)(use_lut ? lut_bytes : 0);
#define TQ_LAUNCH_GF(GG, LY, FD)                                                                \
    tr_group_kernel<GG, LY, Tout, DEQ, FD><<<grid_l, GROUP_THREADS, smem, s>>>(                 \
        (const float *)in, (Tout *)out, B, C, WH, p, use_lut, lutb, overflow)
#define TQ_LAUNCH_G(GG)                                                                         \
    case GG:                                                                                    \
        if (contig) { if (p.fastdiv) TQ_LAUNCH_GF(GG, 1, true); else TQ_LAUNCH_GF(GG, 1, false); }          \
        else if (staged && GG >= 4) { if (p.fastdiv) TQ_LAUNCH_GF(GG, (GG >= 4 ? 2 : 0), true); else TQ_LAUNCH_GF(GG, (GG >= 4 ? 2 : 0), false); } \
        else        { if (p.fastdiv) TQ_LAUNCH_GF(GG, 0, true); else TQ_LAUNCH_GF(GG, 0, false); }          \
        break;
    switch (g) {
        TQ_LAUNCH_G(2)
        TQ_LAUNCH_G(4)
        TQ_LAUNCH_G(8)
        TQ_LAUNCH_G(16)
        TQ_LAUNCH_G(32)
        default: return fail(TQ_ERR_INVALID, "internal: group kernel called with g=%d", g);
    }
#undef TQ_LAUNCH_G
#undef TQ_LAUNCH_GF
    count_launch();
    return check_launch("tr_group_kernel");
}

template <typename Tin, typename Tout, bool DEQ>
static int launch_generic(const void *in, void *out, int64_t B, int64_t C, int64_t WH, int g,
                          const EncParams &p, int *overflow, cudaStream_t s)
{
    const int64_t total = B * ((C + g - 1) / g) * WH;
    const int grid = grid_for(total, 128, 8);
    tr_generic_kernel<Tin, Tout, DEQ><<<grid, 128, 0, s>>>((const Tin *)in, (Tout *)out, B, C, WH, g, p, overflow);
    count_launch();
    return check_launch("tr_generic_kernel");
}

static bool aligned16(const void *a, const void *b)
{
    return (((uintptr_t)a | (uintptr_t)b) & 15u) == 0;
}

static int validate(const void *in, const void *out, int64_t B, int64_t C, int64_t WH, float sf,
                    int bits, int g, int alpha, int enc, EncParams &p, unsigned flags)
{
    if (B < 0 || C < 0 || WH < 0) return fail(TQ_ERR_INVALID, "negative dimension");
    if ((!in || !out) && B * C * WH > 0) return fail(TQ_ERR_INVALID, "NULL tensor pointer");
    if (!(sf > 0.0f) || !(sf < INFINITY)) return fail(TQ_ERR_INVALID, "sf must be positive and finite (got %g)", (double)sf);
    if (bits < 1 || bits > TQ_MAX_BITS) return fail(TQ_ERR_INVALID, "bitwidth must be in [1, %d] (got %d)", TQ_MAX_BITS, bits);
    if (g < 1 || g > TQ_MAX_GROUP) return fail(TQ_ERR_INVALID, "group_size must be in [1, %d] (got %d)", TQ_MAX_GROUP, g);
    if (alpha < 0) return fail(TQ_ERR_INVALID, "num_keep_terms must be >= 0 (got %d)", alpha);
    if (enc < 0 || enc > 2) return fail(TQ_ERR_INVALID, "unknown encoding %d", enc);
    p.sf = sf;
    p.maxv = (float)((1u << bits) - 1u);
    p.bits = bits;
    p.alpha = alpha;
    p.enc = enc;
    p.relu = (flags & TQ_FLAG_RELU) ? 1 : 0;
    p.fastdiv = fast_div_ok(sf) && !(flags & TQ_FLAG_EXACT_DIV) ? 1 : 0;
    return TQ_OK;
}

template <typename Tin, typename Tout, bool DEQ>
static int dispatch(const void *in, void *out, int64_t B, int64_t C, int64_t WH, int g,
                    const EncParams &p, int *overflow, cudaStream_t s)
{
    const int64_t n = B * C * WH;
    if (n == 0) return TQ_OK;
    if (g == 1) {
        // groups of one: the (B, C, WH) structure is irrelevant, stream the flat tensor
        if (aligned16(in, out)) return launch_elem<Tin, Tout, DEQ>(in, out, n, p, overflow, s);
        return launch_generic<Tin, Tout, DEQ>(in, out, 1, n, 1, 1, p, overflow, s);
    }
    // register-resident fast path: fp32 in, fp32 / int8 / int16 out, power-of-two groups
    if constexpr (std::is_same<Tin, float>::value &&
                  (DEQ || std::is_same<Tout, int8_t>::value || std::is_same<Tout, int16_t>::value)) {
        const bool pow2 = (g & (g - 1)) == 0;
        if (pow2 && C % g == 0 && p.bits <= 15 && (WH != 1 || aligned16(in, out)))
            return launch_group_f32<Tout, DEQ>(in, out, B, C, WH, g, p, overflow, s);
    }
    return launch_generic<Tin, Tout, DEQ>(in, out, B, C, WH, g, p, overflow, s);
}

}  // namespace tq

using namespace tq;

extern "C" int tq_tr_encode(const void *in, void *out, int dtype, int64_t B, int64_t C, int64_t WH,
                            float sf, int bits, int g, int alpha, int encoding, unsigned flags,
                            void *stream)
{
    EncParams p;
    int rc = validate(in, out, B, C, WH, sf, bits, g, alpha, encoding, p, flags);
    if (rc != TQ_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    switch (dtype) {
        case TQ_F32:  return dispatch<float, float, true>(in, out, B, C, WH, g, p, nullptr, s);
        case TQ_F64:  return dispatch<double, double, true>(in, out, B, C, WH, g, p, nullptr, s);
        case TQ_BF16: return dispatch<__nv_bfloat16, __nv_bfloat16, true>(in, out, B, C, WH, g, p, nullptr, s);
        case TQ_F16:  return dispatch<__half, __half, true>(in, out, B, C, WH, g, p, nullptr, s);
        default: return fail(TQ_ERR_INVALID, "unknown dtype %d", dtype);
    }
}

template <typename Tin>
static int encode_codes_t(const void *in, void *codes, int code_dtype, int64_t B, int64_t C,
                          int64_t WH, int g, const EncParams &p, int *overflow, cudaStream_t s)
{
    switch (code_dtype) {
        case TQ_I8:  return dispatch<Tin, int8_t, false>(in, codes, B, C, WH, g, p, overflow, s);
        case TQ_U8:  return dispatch<Tin, uint8_t, false>(in, codes, B, C, WH, g, p, overflow, s);
        case TQ_I16: return dispatch<Tin, int16_t, false>(in, codes, B, C, WH, g, p, overflow, s);
        case TQ_I32: return dispatch<Tin, int32_t, false>(in, codes, B, C, WH, g, p, overflow, s);
        case TQ_F16C: return dispatch<Tin, __half, false>(in, codes, B, C, WH, g, p, overflow, s);
        default: return fail(TQ_ERR_INVALID, "unknown code dtype %d", code_dtype);
    }
}

extern "C" int tq_tr_encode_codes(const void *in, void *codes, int dtype, int code_dtype,
                                  int64_t B, int64_t C, int64_t WH, float sf, int bits, int g,
                                  int alpha, int encoding, unsigned flags, int *overflow,
                                  void *stream)
{
    EncParams p;
    int rc = validate(in, codes, B, C, WH, sf, bits, g, alpha, encoding, p, flags);
    if (rc != TQ_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    switch (dtype) {
        case TQ_F32:  return encode_codes_t<float>(in, codes, code_dtype, B, C, WH, g, p, overflow, s);
        case TQ_BF16: return encode_codes_t<__nv_bfloat16>(in, codes, code_dtype, B, C, WH, g, p, overflow, s);
        case TQ_F16:
        case TQ_F64:  return fail(TQ_ERR_UNSUPPORTED, "integer codes are produced from f32 or bf16 inputs only");
        default: return fail(TQ_ERR_INVALID, "unknown dtype %d", dtype);
    }
}
