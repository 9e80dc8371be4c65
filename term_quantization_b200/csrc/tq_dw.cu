// tq_dw.cu -- the memory-bound layers of the depthwise CNNs (BASELINE.json configs[3], MobileNet-V2) on term codes.
//
// The reference wraps a depthwise conv like any other (cnn_models/__init__.py:52-65 gives it the "effectively
// unquantised" weight setting (16, 1, 16)), so per forward it runs: TR encode of the input (tr_layer.py:96-99, g = 1) ->
// cuDNN fp32 depthwise conv on the dequantised values -> BatchNorm -> ReLU6, and the next wrapped conv encodes the
// result again: five passes over the activation.  Here ONE kernel reads the input's fp16 term codes (written by the
// producing conv's epilogue), accumulates the 9 taps in int32 (|a| <= 2^bits, |w| <= 2^15: |acc| < 2^29, exact),
// applies t = float(acc) * (sf_x * sf_w) (+ bias), fma(t, bn_a, bn_b), ReLU / ReLU6, and writes the fp16 term codes of
// the consumer's quantiser (and / or the fp32 value).  Algorithmic bytes: 2 B read + 2 B written per element.
//
// Mapping: NHWC.  A tile = TH x TW output pixels x 64 channels of one image; its (TH*s+2) x (TW*s+2) x 64 input codes
// are staged into shared memory by ONE tiled 4-D TMA load (cp.async.bulk.tensor; the halo outside the image arrives as
// zeros: padding costs nothing), double-buffered so that the load of tile i+1 overlaps the arithmetic of tile i.  One
// thread = 8 channels (one 128-bit shared-memory read per input pixel) x DW_PIX consecutive output pixels of a row, the
// 3 x ((DW_PIX-1)*s+3) input pixels read once and reused across the outputs; weights (int32 [9][C]) and the
// (q, sign) -> code table sit in shared memory; outputs leave as 128-bit stores, 128 contiguous bytes per 8 threads.
// The first version of this kernel read its inputs with per-thread global loads and was latency-bound (5.9 ms per
// MobileNet-V2 forward at batch 512 for 4.7 GB of algorithmic traffic); see DESIGN.md.
#include <cuda.h>

#include "tq_common.cuh"

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
namespace tq {
EncodeTiledFn encode_tiled();           // tq_gemm.cu
}

namespace tq {

constexpr int DW_PIX = 4;

struct DwParams {
    int N, H, W, C, Ho, Wo, stride;
    float scale;
    const float *bias, *bn_a, *bn_b;
    int relu;                   // 0 none, 1 ReLU, 2 ReLU6
    int write_f32;
    NextQuant nq;
};

// activation shared by the epilogues of this file
__device__ __forceinline__ float apply_act(float t, int relu)
{
    if (relu) t = fmaxf(t, 0.0f);
    if (relu == 2) t = fminf(t, 6.0f);
    return t;
}

struct DwTile {
    int th, tw;                 // output pixels per tile
    int tiles_h, tiles_w, cblocks;
    int in_h, in_w;             // input pixels per tile (with halo)
    int stage_bytes;
    int unsigned_act;           // input codes are known to lie in [0, 1023] (post-ReLU): integer extraction without cvt
};

__device__ __forceinline__ uint32_t dw_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint4 dw_lds128(uint32_t saddr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}

// STRIDE 1 | 2; CB = channels per tile (64, or 32 for channel counts that are odd multiples of 32: no idle lanes);
// UNSIGNED: input codes lie in [0, 1023] (post-ReLU): integer extraction without cvt; FAST: hoisted-reciprocal quantiser
template <int STRIDE, int CB, bool UNSIGNED, bool FAST>
__global__ void __launch_bounds__(256, 2)
depthwise3x3_codes_kernel(const __grid_constant__ CUtensorMap tmIn, const int32_t *__restrict__ wgt,
                          float *__restrict__ out_f32, __half *__restrict__ out_codes, DwParams p, DwTile tl)
{
    extern __shared__ __align__(128) uint8_t dw_smem[];
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(dw_smem) + 127) & ~uintptr_t(127));
    uint8_t *stage0 = base;                                                     // 2 x [in_h][in_w][64] fp16
    int32_t *sw = reinterpret_cast<int32_t *>(base + 2 * tl.stage_bytes);       // [9][C]
    __half *lut = reinterpret_cast<__half *>(sw + 9 * p.C);                     // (q, sign) -> code
    uint64_t *full = reinterpret_cast<uint64_t *>(reinterpret_cast<uint8_t *>(lut) + code_table_bytes(p.nq.bits));
    for (int i = threadIdx.x; i < 9 * p.C; i += blockDim.x) sw[i] = wgt[i];
    if (p.nq.write_codes) {
        for (uint32_t i = threadIdx.x; i < (2u << p.nq.bits); i += blockDim.x) {
            const int code = elem_code(i & ((1u << p.nq.bits) - 1u), p.nq.enc, p.nq.terms);
            lut[i] = __int2half_rn((i >> p.nq.bits) ? -code : code);
        }
    }
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dw_smem_u32(&full[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dw_smem_u32(&full[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmIn) : "memory");
    }
    __syncthreads();
    const Quant nq = make_quant(p.nq);
    const int tiles_per_img = tl.tiles_h * tl.tiles_w * tl.cblocks;
    const int64_t total = (int64_t)p.N * tiles_per_img;

    auto issue = [&](int64_t tile, int stage) {             // one thread: TMA the input box of `tile` into `stage`
        const int cb = (int)(tile % tl.cblocks);
        const int64_t r = tile / tl.cblocks;
        const int tw = (int)(r % tl.tiles_w), th = (int)((r / tl.tiles_w) % tl.tiles_h), n = (int)(r / ((int64_t)tl.tiles_w * tl.tiles_h));
        const uint32_t bar = dw_smem_u32(&full[stage]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)tl.stage_bytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
            ::"r"(dw_smem_u32(stage0 + stage * tl.stage_bytes)), "l"(&tmIn), "r"(bar), "r"(cb * CB), "r"(tw * tl.tw * STRIDE - 1),
              "r"(th * tl.th * STRIDE - 1), "r"(n) : "memory");
    };

    constexpr int IN_PIX = (DW_PIX - 1) * STRIDE + 3;
    const int groups_w = tl.tw / DW_PIX;
    constexpr int C8 = CB / 8;                              // 8-channel blocks per tile
    const int items = tl.th * groups_w * C8;                // (row, 4-pixel group, 8-channel block) of a tile
    const uint32_t sw_addr = dw_smem_u32(sw);
    int stage = 0;
    uint32_t phases = 0u;                                   // bit s = parity to wait for on stage s
    if (threadIdx.x == 0 && (int64_t)blockIdx.x < total) issue(blockIdx.x, 0);
    for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int64_t next = tile + gridDim.x;
        if (threadIdx.x == 0 && next < total) issue(next, stage ^ 1);      // (stage ^ 1 was released by the barrier below)
        {   // wait for this tile's box
            const uint32_t bar = dw_smem_u32(&full[stage]);
            asm volatile(
                "{\n\t"
                ".reg .pred P1;\n\t"
                "DW_WAIT:\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
                "@P1 bra DW_DONE;\n\t"
                "bra DW_WAIT;\n\t"
                "DW_DONE:\n\t"
                "}" ::"r"(bar), "r"((phases >> stage) & 1u) : "memory");
            phases ^= 1u << stage;
        }
        const int cb = (int)(tile % tl.cblocks);
        const int64_t r = tile / tl.cblocks;
        const int twi = (int)(r % tl.tiles_w), thi = (int)((r / tl.tiles_w) % tl.tiles_h), n = (int)(r / ((int64_t)tl.tiles_w * tl.tiles_h));
        const uint32_t sin = dw_smem_u32(stage0 + stage * tl.stage_bytes);
        for (int item = threadIdx.x; item < items; item += blockDim.x) {
            const int c8 = item % C8;
            const int gw = (item / C8) % groups_w, row = (item / C8) / groups_w;
            const int ch = cb * CB + c8 * 8;
            const int ho = thi * tl.th + row, wo0 = twi * tl.tw + gw * DW_PIX;
            if (ch >= p.C || ho >= p.Ho || wo0 >= p.Wo) continue;
            int acc[DW_PIX][8];
#pragma unroll
            for (int j = 0; j < DW_PIX; ++j)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[j][c] = 0;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                int wrow[3][8];
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const uint4 w0 = dw_lds128(sw_addr + (uint32_t)((dy * 3 + dx) * p.C + ch) * 4u);
                    const uint4 w1 = dw_lds128(sw_addr + (uint32_t)((dy * 3 + dx) * p.C + ch + 4) * 4u);
                    wrow[dx][0] = w0.x; wrow[dx][1] = w0.y; wrow[dx][2] = w0.z; wrow[dx][3] = w0.w;
                    wrow[dx][4] = w1.x; wrow[dx][5] = w1.y; wrow[dx][6] = w1.z; wrow[dx][7] = w1.w;
                }
                const uint32_t rowp = sin + (uint32_t)(((row * STRIDE + dy) * tl.in_w + gw * DW_PIX * STRIDE) * CB + c8 * 8) * 2u;
#pragma unroll
                for (int px = 0; px < IN_PIX; ++px) {
                    const uint4 raw = dw_lds128(rowp + (uint32_t)px * (CB * 2));
                    const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
                    int v[8];
                    if constexpr (UNSIGNED) {
                        // integer codes 0..1023 held in fp16: x + 1024 is exact and its mantissa field IS the integer
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            __half2 x2 = *reinterpret_cast<const __half2 *>(&rw[h]);
                            x2 = __hadd2(x2, __half2half2(__ushort_as_half((unsigned short)0x6400)));   // 1024.0
                            const uint32_t b = *reinterpret_cast<const uint32_t *>(&x2);
                            v[2 * h] = (int)(b & 0x3FFu);
                            v[2 * h + 1] = (int)((b >> 16) & 0x3FFu);
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 8; ++c) v[c] = __half2int_rn(__ushort_as_half((unsigned short)(rw[c >> 1] >> (16 * (c & 1)))));
                    }
#pragma unroll
                    for (int j = 0; j < DW_PIX; ++j) {
                        const int dx = px - j * STRIDE;              // compile-time after unrolling
                        if (dx < 0 || dx > 2) continue;
#pragma unroll
                        for (int c = 0; c < 8; ++c) acc[j][c] += v[c] * wrow[dx][c];
                    }
                }
            }
            // epilogue: float(acc) * scale (+ bias) -> fma(BN) -> activation -> fp32 and / or term codes
            float ba[8], bb[8], bs[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                ba[c] = p.bn_a ? __ldg(p.bn_a + ch + c) : 1.0f;
                bb[c] = p.bn_b ? __ldg(p.bn_b + ch + c) : 0.0f;
                bs[c] = p.bias ? __ldg(p.bias + ch + c) : 0.0f;
            }
#pragma unroll
            for (int j = 0; j < DW_PIX; ++j) {
                const int wo = wo0 + j;
                if (wo >= p.Wo) break;
                const int64_t o = (((int64_t)n * p.Ho + ho) * p.Wo + wo) * p.C + ch;
                float tv[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float x = __fmul_rn(__int2float_rn(acc[j][c]), p.scale);
                    if (p.bias) x = __fadd_rn(x, bs[c]);
                    if (p.bn_a) x = __fmaf_rn(x, ba[c], bb[c]);
                    tv[c] = apply_act(x, p.relu);
                }
                if (p.write_f32) {
                    reinterpret_cast<float4 *>(out_f32 + o)[0] = make_float4(tv[0], tv[1], tv[2], tv[3]);
                    reinterpret_cast<float4 *>(out_f32 + o)[1] = make_float4(tv[4], tv[5], tv[6], tv[7]);
                }
                if (p.nq.write_codes) {
                    uint32_t hc[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const uint32_t neg = __float_as_uint(tv[c]) >> 31;
                        const uint32_t qi = quantize_f32<FAST>(tv[c], nq);
                        hc[c] = __half_as_ushort(lut[qi | (neg << p.nq.bits)]);
                    }
                    *reinterpret_cast<uint4 *>(out_codes + o) =
                        make_uint4(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16), hc[4] | (hc[5] << 16), hc[6] | (hc[7] << 16));
                }
            }
        }
        __syncthreads();                                    // every thread is done with `stage`: it may be refilled
        stage ^= 1;
    }
}

// fp32 NHWC -> (+ bias[c]) -> fma(x, a[c], b[c]) -> activation -> fp32 and / or fp16 term codes: the tail of an unwrapped first conv
// (cnn_models/__init__.py:34-36) fused with the first wrapped layer's LinearQuantize (tr_layer.py:96-99).
__global__ void __launch_bounds__(256)
bn_act_encode_kernel(const float *__restrict__ x, float *__restrict__ out_f32, __half *__restrict__ out_codes, int64_t n4, int C,
                     DwParams p)
{
    extern __shared__ __align__(128) uint8_t dw_smem[];
    __half *lut = reinterpret_cast<__half *>(dw_smem);
    if (p.nq.write_codes) {
        for (uint32_t i = threadIdx.x; i < (2u << p.nq.bits); i += blockDim.x) {
            const int code = elem_code(i & ((1u << p.nq.bits) - 1u), p.nq.enc, p.nq.terms);
            lut[i] = __int2half_rn((i >> p.nq.bits) ? -code : code);
        }
        __syncthreads();
    }
    const Quant nq = make_quant(p.nq);
    const int c4n = C >> 2;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n4; t += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(t % c4n);
        const float4 v = __ldg(reinterpret_cast<const float4 *>(x) + t);
        float tv[4] = {v.x, v.y, v.z, v.w};
        if (p.bias) {                                   // the conv's own bias: one fp32 add, as cuDNN / torch apply it
            const float4 bi = __ldg(reinterpret_cast<const float4 *>(p.bias) + c4);
            tv[0] = __fadd_rn(tv[0], bi.x); tv[1] = __fadd_rn(tv[1], bi.y);
            tv[2] = __fadd_rn(tv[2], bi.z); tv[3] = __fadd_rn(tv[3], bi.w);
        }
        if (p.bn_a) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(p.bn_a) + c4);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(p.bn_b) + c4);
            tv[0] = __fmaf_rn(tv[0], a.x, b.x); tv[1] = __fmaf_rn(tv[1], a.y, b.y);
            tv[2] = __fmaf_rn(tv[2], a.z, b.z); tv[3] = __fmaf_rn(tv[3], a.w, b.w);
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) tv[e] = apply_act(tv[e], p.relu);
        if (p.write_f32) reinterpret_cast<float4 *>(out_f32)[t] = make_float4(tv[0], tv[1], tv[2], tv[3]);
        if (p.nq.write_codes) {
            uint32_t hc[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t neg = __float_as_uint(tv[e]) >> 31;
                const uint32_t qi = p.nq.fastdiv ? quantize_f32<true>(tv[e], nq) : quantize_f32<false>(tv[e], nq);
                hc[e] = __half_as_ushort(lut[qi | (neg << p.nq.bits)]);
            }
            reinterpret_cast<uint2 *>(out_codes)[t] = make_uint2(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16));
        }
    }
}

// Max-pool on fp16 NHWC tensors (term codes between the convs of the VGG-style stacks: for g = 1 the truncated code is
// monotone in the value, so pooling the codes equals encoding the pooled values).  One thread = 8 channels (16 bytes) of
// one output pixel; window positions outside the map are skipped (torch's -inf padding).  Memory-bound.
__global__ void __launch_bounds__(256)
maxpool2d_f16_kernel(const uint4 *__restrict__ x, uint4 *__restrict__ y, int N, int H, int W, int C8, int Ho, int Wo,
                     int k, int stride, int pad)
{
    const int64_t total = (int64_t)N * Ho * Wo * C8;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c8 = (int)(t % C8);
        const int64_t pix = t / C8;
        const int wo = (int)(pix % Wo), ho = (int)((pix / Wo) % Ho), n = (int)(pix / ((int64_t)Wo * Ho));
        const __half2 ninf = __half2half2(__ushort_as_half((unsigned short)0xFC00u));
        __half2 m0 = ninf, m1 = ninf, m2 = ninf, m3 = ninf;
        for (int dy = 0; dy < k; ++dy) {
            const int h = ho * stride - pad + dy;
            if (h < 0 || h >= H) continue;
            for (int dx = 0; dx < k; ++dx) {
                const int w = wo * stride - pad + dx;
                if (w < 0 || w >= W) continue;
                const uint4 v = __ldcs(x + (((int64_t)n * H + h) * W + w) * C8 + c8);
                m0 = __hmax2(m0, *reinterpret_cast<const __half2 *>(&v.x));
                m1 = __hmax2(m1, *reinterpret_cast<const __half2 *>(&v.y));
                m2 = __hmax2(m2, *reinterpret_cast<const __half2 *>(&v.z));
                m3 = __hmax2(m3, *reinterpret_cast<const __half2 *>(&v.w));
            }
        }
        uint4 o;
        o.x = *reinterpret_cast<const uint32_t *>(&m0); o.y = *reinterpret_cast<const uint32_t *>(&m1);
        o.z = *reinterpret_cast<const uint32_t *>(&m2); o.w = *reinterpret_cast<const uint32_t *>(&m3);
        y[t] = o;
    }
}

// =============================================================================================
// First conv of the VGG-style / depthwise CNNs (3x3, 3 input channels, never wrapped: cnn_models/__init__.py:34-36) on the
// CUDA cores in fp32, with its bias, BatchNorm, ReLU / ReLU6 and the first wrapped layer's LinearQuantize in the same
// kernel: the fp32 map (1.6 GB for VGG-16 at batch 128) is never written unless asked for.  27 FMAs per output in a fixed
// order (filter row, filter column, channel), bias added after the sum as cuDNN does.
// One thread = 8 output channels x 8 pixels (64 accumulators); a warp = COUT/8 channel groups x PGW = 256/COUT pixel
// groups; pixel j of group pg is column j * PGW + pg of the tile, so the lanes of a warp read ADJACENT input pixels
// (bank-conflict free for both strides: 3 or 6 floats apart) and a 16-byte store instruction writes PGW adjacent pixels
// x COUT channels = 512 contiguous bytes.  Operands come from shared memory as broadcasts (the lanes of a pixel group
// share the input value, the lanes of a channel group the weights).
// =============================================================================================
struct FirstConvParams {
    int N, H, W, Ho, Wo, stride;
    const float *bias, *bn_a, *bn_b;
    int relu, write_f32;
    NextQuant nq;
};

template <int COUT, int STRIDE, bool FAST>
__global__ void __launch_bounds__(256, 2)
first_conv3x3_kernel(const float *__restrict__ x, const float *__restrict__ wgt, float *__restrict__ out_f32,
                     __half *__restrict__ out_codes, FirstConvParams p)
{
    constexpr int CG = COUT / 8;                 // channel groups per warp
    constexpr int PGW = 32 / CG;                 // pixel groups (of 8 pixels) per warp
    constexpr int TW = PGW * 8, TH = 8;          // output tile of a CTA: one row per warp
    constexpr int IW = (TW - 1) * STRIDE + 3, IH = (TH - 1) * STRIDE + 3;
    extern __shared__ __align__(128) uint8_t dw_smem[];
    float *sw = reinterpret_cast<float *>(dw_smem);                 // [27][COUT]
    float *sin = sw + 27 * COUT;                                    // [IH][IW][3]
    __half *lut = reinterpret_cast<__half *>(sin + ((IH * IW * 3 + 3) & ~3));
    for (int i = threadIdx.x; i < 27 * COUT; i += 256) sw[i] = wgt[i];
    if (p.nq.write_codes) {
        for (uint32_t i = threadIdx.x; i < (2u << p.nq.bits); i += 256) {
            const int code = elem_code(i & ((1u << p.nq.bits) - 1u), p.nq.enc, p.nq.terms);
            lut[i] = __int2half_rn((i >> p.nq.bits) ? -code : code);
        }
    }
    const Quant nq = make_quant(p.nq);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cg = lane % CG, pg = lane / CG;
    const int tiles_w = (p.Wo + TW - 1) / TW, tiles_h = (p.Ho + TH - 1) / TH;
    const int64_t total = (int64_t)p.N * tiles_h * tiles_w;
    for (int64_t tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int tw = (int)(tile % tiles_w), th = (int)((tile / tiles_w) % tiles_h), n = (int)(tile / ((int64_t)tiles_w * tiles_h));
        const int h_in0 = th * TH * STRIDE - 1, w_in0 = tw * TW * STRIDE - 1;
        __syncthreads();                                            // the previous tile's reads of `sin` are done
        for (int hi = warp; hi < IH; hi += 8) {                     // a tile row is IW * 3 contiguous floats of the image row
            const int h = h_in0 + hi;
            const bool row_in = h >= 0 && h < p.H;
            const float *src = x + (((int64_t)n * p.H + (row_in ? h : 0)) * p.W + w_in0) * 3;
            const int k_lo = w_in0 < 0 ? -w_in0 * 3 : 0, k_hi = (p.W - w_in0) * 3;      // floats of the row that exist
            for (int k = lane; k < IW * 3; k += 32)
                sin[hi * IW * 3 + k] = (row_in && k >= k_lo && k < k_hi) ? __ldg(src + k) : 0.0f;
        }
        __syncthreads();
        float acc[8][8];                                            // [pixel][channel]
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[j][c] = 0.0f;
        const float *in0 = sin + ((warp * STRIDE) * IW + pg * STRIDE) * 3;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int sx = 0; sx < 3; ++sx) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float4 w0 = *reinterpret_cast<const float4 *>(sw + ((r * 3 + sx) * 3 + c) * COUT + cg * 8);
                    const float4 w1 = *reinterpret_cast<const float4 *>(sw + ((r * 3 + sx) * 3 + c) * COUT + cg * 8 + 4);
                    const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float v = in0[(r * IW + j * PGW * STRIDE + sx) * 3 + c];
#pragma unroll
                        for (int k = 0; k < 8; ++k) acc[j][k] = __fmaf_rn(v, wv[k], acc[j][k]);
                    }
                }
            }
        }
        const int ho = th * TH + warp;
        if (ho >= p.Ho) continue;
        float ba[8], bb[8], bs[8];                                  // (loaded per tile: 24 registers less across the FMA loop)
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            ba[c] = p.bn_a ? __ldg(p.bn_a + cg * 8 + c) : 1.0f;
            bb[c] = p.bn_b ? __ldg(p.bn_b + cg * 8 + c) : 0.0f;
            bs[c] = p.bias ? __ldg(p.bias + cg * 8 + c) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int wo = tw * TW + j * PGW + pg;
            if (wo >= p.Wo) break;
            const int64_t o = (((int64_t)n * p.Ho + ho) * p.Wo + wo) * COUT + cg * 8;
            float tv[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float t = acc[j][c];
                if (p.bias) t = __fadd_rn(t, bs[c]);
                if (p.bn_a) t = __fmaf_rn(t, ba[c], bb[c]);
                tv[c] = apply_act(t, p.relu);
            }
            if (p.write_f32) {
                reinterpret_cast<float4 *>(out_f32 + o)[0] = make_float4(tv[0], tv[1], tv[2], tv[3]);
                reinterpret_cast<float4 *>(out_f32 + o)[1] = make_float4(tv[4], tv[5], tv[6], tv[7]);
            }
            if (p.nq.write_codes) {
                uint32_t hc[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint32_t neg = __float_as_uint(tv[c]) >> 31;
                    const uint32_t qi = quantize_f32<FAST>(tv[c], nq);
                    hc[c] = __half_as_ushort(lut[qi | (neg << p.nq.bits)]);
                }
                *reinterpret_cast<uint4 *>(out_codes + o) =
                    make_uint4(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16), hc[4] | (hc[5] << 16), hc[6] | (hc[7] << 16));
            }
        }
    }
}

}  // namespace tq

using namespace tq;

extern "C" int tq_depthwise3x3_codes(const void *act_codes, const int32_t *wgt_codes, float *out_f32, void *out_codes,
                                     const float *bias, const float *bn_a, const float *bn_b, int N, int H, int W, int C,
                                     int stride, float scale, int relu, int act_unsigned, float next_sf, int next_bits,
                                     int next_terms, void *stream)
{
    return tq_depthwise3x3_codes_enc(act_codes, wgt_codes, out_f32, out_codes, bias, bn_a, bn_b, N, H, W, C, stride, scale,
                                     relu, act_unsigned, next_sf, next_bits, next_terms, TQ_ENC_HESE, stream);
}

extern "C" int tq_depthwise3x3_codes_enc(const void *act_codes, const int32_t *wgt_codes, float *out_f32, void *out_codes,
                                         const float *bias, const float *bn_a, const float *bn_b, int N, int H, int W, int C,
                                         int stride, float scale, int relu, int act_unsigned, float next_sf, int next_bits,
                                         int next_terms, int next_enc, void *stream)
{
    DwParams p{};
    int rc = next_quant(p.nq, out_codes, next_sf, next_bits, next_terms, next_enc, FP16_CODE_MAX_BITS, false);
    if (rc != TQ_OK) return rc;
    if (!act_codes || !wgt_codes || (!out_f32 && !out_codes)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (N < 1 || H < 1 || W < 1 || C < 8 || C % 8) return fail(TQ_ERR_INVALID, "bad shape (C must be a multiple of 8)");
    if (stride != 1 && stride != 2) return fail(TQ_ERR_UNSUPPORTED, "depthwise 3x3: stride 1 or 2");
    if ((bn_a == nullptr) != (bn_b == nullptr)) return fail(TQ_ERR_INVALID, "bn_a and bn_b go together");
    if (relu < 0 || relu > 2) return fail(TQ_ERR_INVALID, "relu: 0 none, 1 ReLU, 2 ReLU6");
    if ((((uintptr_t)act_codes | (uintptr_t)wgt_codes | (uintptr_t)out_f32 | (uintptr_t)out_codes) & 15u) != 0)
        return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    p.N = N; p.H = H; p.W = W; p.C = C; p.stride = stride;
    p.Ho = (H + 2 - 3) / stride + 1;
    p.Wo = (W + 2 - 3) / stride + 1;
    p.scale = scale; p.bias = bias; p.bn_a = bn_a; p.bn_b = bn_b; p.relu = relu;
    p.write_f32 = out_f32 ? 1 : 0;
    // tile: TW a multiple of DW_PIX; small maps take small tiles (a 7x7 map in a 8x16 tile would idle 62 % of the lanes)
    DwTile tl{};
    tl.tw = p.Wo > 8 ? 16 : 8;
    tl.th = p.Ho > 4 ? 8 : 4;
    if (stride == 2 && tl.tw == 16) tl.th = 4;              // (2*4+2) x (2*16+2) x 128 B = 43.5 KB per stage
    tl.tiles_w = (p.Wo + tl.tw - 1) / tl.tw;
    tl.tiles_h = (p.Ho + tl.th - 1) / tl.th;
    const int cbsz = (C % 64 == 0) ? 64 : 32;               // odd multiples of 32 (and 8/16/24-channel maps): half-width tiles
    // a 32-channel tile of 8 x 16 pixels is only 128 work items for 256 threads (ncu: 44 % of the stall samples at the
    // end-of-tile barrier): twice the rows where the stage still fits (stride 1)
    if (cbsz == 32 && stride == 1 && tl.th == 8 && p.Ho > 8) { tl.th = 16; tl.tiles_h = (p.Ho + tl.th - 1) / tl.th; }
    tl.cblocks = (C + cbsz - 1) / cbsz;
    tl.in_w = tl.tw * stride + 2;
    tl.in_h = tl.th * stride + 2;
    tl.stage_bytes = (tl.in_h * tl.in_w * cbsz * 2 + 127) & ~127;
    tl.unsigned_act = act_unsigned ? 1 : 0;
    CUtensorMap tm;
    {
        cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
        cuuint32_t box[4] = {(cuuint32_t)cbsz, (cuuint32_t)tl.in_w, (cuuint32_t)tl.in_h, 1};
        cuuint32_t one[4] = {1, 1, 1, 1};
        CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void *>(act_codes), dims, strides, box, one,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled(depthwise input) failed: %d", (int)r);
    }
    const size_t smem = 128 + 2 * (size_t)tl.stage_bytes + (size_t)9 * C * 4 + code_table_bytes(p.nq.bits) + 64;
    if (smem > 220 * 1024) return fail(TQ_ERR_UNSUPPORTED, "depthwise conv: %d channels do not fit shared memory", C);
    const int64_t total = (int64_t)N * tl.tiles_h * tl.tiles_w * tl.cblocks;
    // persistent CTAs: as many as fit per SM by shared memory (the tile loop double-buffers its own loads)
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm > 2) per_sm = 2;                             // __launch_bounds__(256, 2)
    if (per_sm < 1) per_sm = 1;
    int64_t blocks = (int64_t)num_sms() * per_sm;
    if (blocks > total) blocks = total;
    typedef void (*Kern)(const CUtensorMap, const int32_t *, float *, __half *, DwParams, DwTile);
    // [stride - 1][CB == 32][unsigned][fast]
    static const Kern table[2][2][2][2] = {
        {{{depthwise3x3_codes_kernel<1, 64, false, false>, depthwise3x3_codes_kernel<1, 64, false, true>},
          {depthwise3x3_codes_kernel<1, 64, true, false>, depthwise3x3_codes_kernel<1, 64, true, true>}},
         {{depthwise3x3_codes_kernel<1, 32, false, false>, depthwise3x3_codes_kernel<1, 32, false, true>},
          {depthwise3x3_codes_kernel<1, 32, true, false>, depthwise3x3_codes_kernel<1, 32, true, true>}}},
        {{{depthwise3x3_codes_kernel<2, 64, false, false>, depthwise3x3_codes_kernel<2, 64, false, true>},
          {depthwise3x3_codes_kernel<2, 64, true, false>, depthwise3x3_codes_kernel<2, 64, true, true>}},
         {{depthwise3x3_codes_kernel<2, 32, false, false>, depthwise3x3_codes_kernel<2, 32, false, true>},
          {depthwise3x3_codes_kernel<2, 32, true, false>, depthwise3x3_codes_kernel<2, 32, true, true>}}}};
    const int i_cb = cbsz == 32 ? 1 : 0, i_un = tl.unsigned_act, i_fast = p.nq.fastdiv;
    Kern kern = table[stride - 1][i_cb][i_un][i_fast];
    static bool attr_set[16][64] = {{false}};
    const int kidx = ((stride - 1) * 2 + i_cb) * 4 + i_un * 2 + i_fast;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_set[kidx][dev]) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(depthwise3x3_codes_kernel)");
        attr_set[kidx][dev] = true;
    }
    kern<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(tm, wgt_codes, out_f32, (__half *)out_codes, p, tl);
    count_launch();
    return check_launch("depthwise3x3_codes_kernel");
}

extern "C" int tq_bn_act_encode(const float *x, const float *bias, const float *bn_a, const float *bn_b, float *out_f32,
                                void *out_codes, int64_t npix, int C, int relu, float next_sf, int next_bits, int next_terms,
                                void *stream)
{
    return tq_bn_act_encode_enc(x, bias, bn_a, bn_b, out_f32, out_codes, npix, C, relu, next_sf, next_bits, next_terms,
                                TQ_ENC_HESE, stream);
}

extern "C" int tq_bn_act_encode_enc(const float *x, const float *bias, const float *bn_a, const float *bn_b, float *out_f32,
                                    void *out_codes, int64_t npix, int C, int relu, float next_sf, int next_bits,
                                    int next_terms, int next_enc, void *stream)
{
    DwParams p{};
    const int rc = next_quant(p.nq, out_codes, next_sf, next_bits, next_terms, next_enc, FP16_CODE_MAX_BITS, false);
    if (rc != TQ_OK) return rc;
    if (!x || (!out_f32 && !out_codes)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (npix < 0 || C < 4 || C % 4) return fail(TQ_ERR_INVALID, "bad shape (C must be a multiple of 4)");
    if ((bn_a == nullptr) != (bn_b == nullptr)) return fail(TQ_ERR_INVALID, "bn_a and bn_b go together");
    if (relu < 0 || relu > 2) return fail(TQ_ERR_INVALID, "relu: 0 none, 1 ReLU, 2 ReLU6");
    if ((((uintptr_t)x | (uintptr_t)bias | (uintptr_t)bn_a | (uintptr_t)bn_b | (uintptr_t)out_f32 | (uintptr_t)out_codes) & 15u) != 0)
        return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    if (npix == 0) return TQ_OK;
    p.C = C; p.bias = bias; p.bn_a = bn_a; p.bn_b = bn_b; p.relu = relu; p.write_f32 = out_f32 ? 1 : 0;
    const int64_t n4 = npix * (C / 4);
    int64_t blocks = (n4 + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    if (blocks > cap) blocks = cap;
    const size_t smem = out_codes ? code_table_bytes(p.nq.bits) : 0;
    bn_act_encode_kernel<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(x, out_f32, (__half *)out_codes, n4, C, p);
    count_launch();
    return check_launch("bn_act_encode_kernel");
}

extern "C" int tq_maxpool2d_f16(const void *x_f16, void *y_f16, int N, int H, int W, int C, int k, int stride, int pad,
                                void *stream)
{
    if (!x_f16 || !y_f16) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (N < 1 || H < 1 || W < 1 || C < 8 || C % 8) return fail(TQ_ERR_INVALID, "bad shape (C must be a multiple of 8)");
    if (k < 1 || k > 7 || stride < 1 || pad < 0 || 2 * pad > k) return fail(TQ_ERR_INVALID, "bad pooling window");
    if ((((uintptr_t)x_f16 | (uintptr_t)y_f16) & 15u) != 0) return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    const int Ho = (H + 2 * pad - k) / stride + 1, Wo = (W + 2 * pad - k) / stride + 1;      // floor mode
    if (Ho < 1 || Wo < 1) return fail(TQ_ERR_INVALID, "empty output");
    const int64_t total = (int64_t)N * Ho * Wo * (C / 8);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 32;
    if (blocks > cap) blocks = cap;
    maxpool2d_f16_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const uint4 *)x_f16, (uint4 *)y_f16, N, H, W, C / 8, Ho, Wo,
                                                                        k, stride, pad);
    count_launch();
    return check_launch("maxpool2d_f16_kernel");
}

template <int COUT, int STRIDE>
static int launch_first_conv(const float *x, const float *wgt, float *out_f32, void *out_codes, const FirstConvParams &p,
                             cudaStream_t s)
{
    constexpr int CGN = COUT / 8, TW = (32 / CGN) * 8, TH = 8;
    constexpr int IW = (TW - 1) * STRIDE + 3, IH = (TH - 1) * STRIDE + 3;
    const size_t smem = (size_t)27 * COUT * 4 + (size_t)((IH * IW * 3 + 3) & ~3) * 4 + (p.nq.write_codes ? code_table_bytes(p.nq.bits) : 0);
    const int64_t tiles = (int64_t)p.N * ((p.Ho + TH - 1) / TH) * ((p.Wo + TW - 1) / TW);
    const int64_t cap = (int64_t)num_sms() * 2;
    const int grid = (int)(tiles < cap ? tiles : cap);
    auto kern = p.nq.fastdiv ? first_conv3x3_kernel<COUT, STRIDE, true> : first_conv3x3_kernel<COUT, STRIDE, false>;
    if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(first_conv3x3_kernel)");
    kern<<<grid, 256, smem, s>>>(x, wgt, out_f32, (__half *)out_codes, p);
    count_launch();
    return check_launch("first_conv3x3_kernel");
}

extern "C" int tq_first_conv3x3_fused(const float *x, const float *wgt, const float *bias, const float *bn_a, const float *bn_b,
                                      float *out_f32, void *out_codes, int N, int H, int W, int Cout, int stride, int relu,
                                      float next_sf, int next_bits, int next_terms, void *stream)
{
    return tq_first_conv3x3_fused_enc(x, wgt, bias, bn_a, bn_b, out_f32, out_codes, N, H, W, Cout, stride, relu, next_sf,
                                      next_bits, next_terms, TQ_ENC_HESE, stream);
}

extern "C" int tq_first_conv3x3_fused_enc(const float *x, const float *wgt, const float *bias, const float *bn_a,
                                          const float *bn_b, float *out_f32, void *out_codes, int N, int H, int W, int Cout,
                                          int stride, int relu, float next_sf, int next_bits, int next_terms, int next_enc,
                                          void *stream)
{
    FirstConvParams p{};
    const int rc = next_quant(p.nq, out_codes, next_sf, next_bits, next_terms, next_enc, FP16_CODE_MAX_BITS, false);
    if (rc != TQ_OK) return rc;
    if (!x || !wgt || (!out_f32 && !out_codes)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (N < 1 || H < 1 || W < 1) return fail(TQ_ERR_INVALID, "bad shape");
    if (Cout != 32 && Cout != 64) return fail(TQ_ERR_UNSUPPORTED, "first conv: Cout must be 32 or 64, got %d", Cout);
    if (stride != 1 && stride != 2) return fail(TQ_ERR_UNSUPPORTED, "first conv: stride 1 or 2");
    if ((bn_a == nullptr) != (bn_b == nullptr)) return fail(TQ_ERR_INVALID, "bn_a and bn_b go together");
    if (relu < 0 || relu > 2) return fail(TQ_ERR_INVALID, "relu: 0 none, 1 ReLU, 2 ReLU6");
    if ((((uintptr_t)out_f32 | (uintptr_t)out_codes) & 15u) != 0 || (((uintptr_t)x | (uintptr_t)wgt) & 3u) != 0)
        return fail(TQ_ERR_INVALID, "outputs must be 16-byte aligned");
    p.N = N; p.H = H; p.W = W; p.stride = stride;
    p.Ho = (H + 2 - 3) / stride + 1; p.Wo = (W + 2 - 3) / stride + 1;                // pad 1
    p.bias = bias; p.bn_a = bn_a; p.bn_b = bn_b; p.relu = relu; p.write_f32 = out_f32 ? 1 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (Cout == 64) return stride == 1 ? launch_first_conv<64, 1>(x, wgt, out_f32, out_codes, p, s) : launch_first_conv<64, 2>(x, wgt, out_f32, out_codes, p, s);
    return stride == 1 ? launch_first_conv<32, 1>(x, wgt, out_f32, out_codes, p, s) : launch_first_conv<32, 2>(x, wgt, out_f32, out_codes, p, s);
}
