// tq_pool.cu -- fused tail of the (unquantised) stem of the CNNs in cnn_models/:
//   BatchNorm (per-channel affine) -> ReLU -> MaxPool 3x3 / stride 2 / pad 1 -> fp32 NHWC output
//   + fp16 term codes of that output for the first wrapped conv (tr_layer.py:96-99 fused in).
// torchvision's ResNet runs these as three passes over the largest activation of the network
// (N x 64 x 112 x 112 fp32 = 822 MB at batch 256) plus a TR-encode pass over the pooled tensor; here
// the conv output is read once and the pooled tensor / its codes are written once.
// Memory-bound: algorithmic bytes = 4*N*H*W*C (read) + 4*N*Ho*Wo*C (write) + 2*N*Ho*Wo*C (codes).
#include <cuda.h>

#include "tq_common.cuh"

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
namespace tq {
EncodeTiledFn encode_tiled();           // tq_gemm.cu
}

namespace tq {

struct PoolParams {
    int N, H, W, C, Ho, Wo;
    int relu;
    NextQuant nq;
};

__global__ void __launch_bounds__(256)
bn_relu_maxpool3x3s2_kernel(const float *__restrict__ x, const float *__restrict__ bn_a,
                            const float *__restrict__ bn_b, float *__restrict__ out,
                            __half *__restrict__ codes, PoolParams p)
{
    extern __shared__ __half lut[];
    if (p.nq.write_codes) {
        for (uint32_t i = threadIdx.x; i < (2u << p.nq.bits); i += blockDim.x) {
            const int code = elem_code(i & ((1u << p.nq.bits) - 1u), p.nq.enc, p.nq.terms);
            lut[i] = __int2half_rn((i >> p.nq.bits) ? -code : code);
        }
        __syncthreads();
    }
    const Quant nq = make_quant(p.nq);
    const int c4n = p.C >> 2;
    const int64_t total = (int64_t)p.N * p.Ho * p.Wo * c4n;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(t % c4n);
        const int64_t pix = t / c4n;
        const int wo = (int)(pix % p.Wo), ho = (int)((pix / p.Wo) % p.Ho), n = (int)(pix / ((int64_t)p.Wo * p.Ho));
        const float4 a = __ldg(reinterpret_cast<const float4 *>(bn_a) + c4);
        const float4 b = __ldg(reinterpret_cast<const float4 *>(bn_b) + c4);
        float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const int h = ho * 2 - 1 + dy;
            if (h < 0 || h >= p.H) continue;
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
                const int w = wo * 2 - 1 + dx;
                if (w < 0 || w >= p.W) continue;
                const float4 v = __ldg(reinterpret_cast<const float4 *>(x + (((int64_t)n * p.H + h) * p.W + w) * p.C) + c4);
                m.x = fmaxf(m.x, __fmaf_rn(v.x, a.x, b.x));
                m.y = fmaxf(m.y, __fmaf_rn(v.y, a.y, b.y));
                m.z = fmaxf(m.z, __fmaf_rn(v.z, a.z, b.z));
                m.w = fmaxf(m.w, __fmaf_rn(v.w, a.w, b.w));
            }
        }
        if (p.relu) { m.x = fmaxf(m.x, 0.f); m.y = fmaxf(m.y, 0.f); m.z = fmaxf(m.z, 0.f); m.w = fmaxf(m.w, 0.f); }
        reinterpret_cast<float4 *>(out)[t] = m;
        if (p.nq.write_codes) {
            const float vv[4] = {m.x, m.y, m.z, m.w};
            uint32_t hc[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t neg = __float_as_uint(vv[e]) >> 31;
                const uint32_t q = p.nq.fastdiv ? quantize_f32<true>(vv[e], nq) : quantize_f32<false>(vv[e], nq);
                hc[e] = __half_as_ushort(lut[q | (neg << p.nq.bits)]);
            }
            reinterpret_cast<uint2 *>(codes)[t] = make_uint2(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16));
        }
    }
}

// Tiled variant: TMA drops the (2 PR + 1) x (2 PC + 1) x 64-channel input box of PR x PC pooled pixels into shared memory
// (double-buffered: the next box lands while this one is pooled; positions outside the map arrive as zeros and are masked
// in the window loop, since the padding of a max-pool is -inf).  Each input value crosses L2 -> SM 1.17 times (PR = 4,
// PC = 7: 1.2 times) instead of the 2.25 times of the kernel above, whose row overlap between CTAs is served by L2 (8.4 TB/s
// through L2 for 4.4 TB/s of algorithmic bytes).  A first tiled version with ordinary loads + barriers between the load and
// the pooling phase was 2x SLOWER than the simple kernel (0.56 vs 0.26 ms): no overlap, little memory parallelism.
// KW: horizontal window (stride 2, pad 1 for KW = 3; stride 1, no padding for KW = 1).  KW = 1 pools the row maxima the
// stem conv writes (tq_stem_conv7x7s2_rowmax): only the vertical 3 / 2 / 1 window is left, on half the bytes.
constexpr int PT_PR = 4, PT_CB = 64, PT_IH = 2 * PT_PR + 1;
constexpr int PT_STAGES = 3;                    // boxes in flight or in use per CTA (3 x 34.6 KB: two CTAs per SM)
constexpr int PT_THREADS = PT_PR * 7 * (PT_CB / 4);       // one (pooled pixel, 4 channels) item per thread and tile (KW = 3): 448
template <int KW> struct PoolTile {
    static constexpr int SW = KW == 3 ? 2 : 1, PAD = KW / 2;
    static constexpr int PC = KW == 3 ? 7 : 14;             // pooled columns per tile: a ~34 KB input box either way
    static constexpr int IW = SW * (PC - 1) + KW;
    static constexpr int STAGE_BYTES = PT_IH * IW * PT_CB * 4;
};

template <int KW>
__global__ void __launch_bounds__(PT_THREADS, 2)
bn_relu_maxpool3x3s2_tiled_kernel(const __grid_constant__ CUtensorMap tmIn, const float *__restrict__ bn_a,
                                  const float *__restrict__ bn_b, float *__restrict__ out,
                                  __half *__restrict__ codes, PoolParams p)
{
    using T = PoolTile<KW>;
    constexpr int PT_PC = T::PC, PT_IW = T::IW, PT_STAGE_BYTES = T::STAGE_BYTES;
    extern __shared__ __align__(128) uint8_t pool_smem[];
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(pool_smem) + 127) & ~uintptr_t(127));
    __half *lut = reinterpret_cast<__half *>(base + PT_STAGES * PT_STAGE_BYTES);
    uint64_t *full = reinterpret_cast<uint64_t *>(base + PT_STAGES * PT_STAGE_BYTES + code_table_bytes(p.nq.bits));
    if (p.nq.write_codes) {
        for (uint32_t i = threadIdx.x; i < (2u << p.nq.bits); i += blockDim.x) {
            const int code = elem_code(i & ((1u << p.nq.bits) - 1u), p.nq.enc, p.nq.terms);
            lut[i] = __int2half_rn((i >> p.nq.bits) ? -code : code);
        }
    }
    auto s32 = [](const void *q) { return (uint32_t)__cvta_generic_to_shared(q); };
    if (threadIdx.x == 0) {
        for (int i = 0; i < PT_STAGES; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(s32(&full[i])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmIn) : "memory");
    }
    __syncthreads();
    const Quant nq = make_quant(p.nq);
    const int cblocks = (p.C + PT_CB - 1) / PT_CB, tiles_w = (p.Wo + PT_PC - 1) / PT_PC, tiles_h = (p.Ho + PT_PR - 1) / PT_PR;
    const int64_t total = (int64_t)p.N * tiles_h * tiles_w * cblocks;
    const int C4 = p.C >> 2;
    constexpr int c4n = PT_CB / 4;
    auto issue = [&](int64_t t, int stage) {
        const int cb = (int)(t % cblocks);
        const int64_t r = t / cblocks;
        const int tw = (int)(r % tiles_w), th = (int)((r / tiles_w) % tiles_h), n = (int)(r / ((int64_t)tiles_w * tiles_h));
        const uint32_t bar = s32(&full[stage]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)PT_STAGE_BYTES) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
            ::"r"(s32(base + stage * PT_STAGE_BYTES)), "l"(&tmIn), "r"(bar), "r"(cb * PT_CB), "r"(tw * PT_PC * T::SW - T::PAD),
              "r"(th * PT_PR * 2 - 1), "r"(n) : "memory");
    };
    int stage = 0;
    uint32_t phases = 0u;
    if (threadIdx.x == 0)
        for (int i = 0; i < PT_STAGES - 1; ++i)
            if ((int64_t)blockIdx.x + (int64_t)i * gridDim.x < total) issue(blockIdx.x + (int64_t)i * gridDim.x, i);
    for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
        const int64_t next = t + (int64_t)(PT_STAGES - 1) * gridDim.x;
        // (the stage before this one was released by the barrier at the end of the previous iteration)
        if (threadIdx.x == 0 && next < total) issue(next, (stage + PT_STAGES - 1) % PT_STAGES);
        {
            const uint32_t bar = s32(&full[stage]);
            asm volatile(
                "{\n\t"
                ".reg .pred P1;\n\t"
                "PT_WAIT:\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
                "@P1 bra PT_DONE;\n\t"
                "bra PT_WAIT;\n\t"
                "PT_DONE:\n\t"
                "}" ::"r"(bar), "r"((phases >> stage) & 1u) : "memory");
            phases ^= 1u << stage;
        }
        const int cb = (int)(t % cblocks);
        const int64_t r = t / cblocks;
        const int tw = (int)(r % tiles_w), th = (int)((r / tiles_w) % tiles_h), n = (int)(r / ((int64_t)tiles_w * tiles_h));
        const int h0 = th * PT_PR * 2 - 1, w0 = tw * PT_PC * T::SW - T::PAD;
        const float4 *tile = reinterpret_cast<const float4 *>(base + stage * PT_STAGE_BYTES);
        for (int o = threadIdx.x; o < PT_PR * PT_PC * c4n; o += blockDim.x) {
            const int c4 = o % c4n, pw = (o / c4n) % PT_PC, ph = o / (c4n * PT_PC);
            const int ho = th * PT_PR + ph, wo = tw * PT_PC + pw;
            const int cg = cb * c4n + c4;
            if (ho >= p.Ho || wo >= p.Wo || cg >= C4) continue;
            const float4 a = __ldg(reinterpret_cast<const float4 *>(bn_a) + cg);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(bn_b) + cg);
            const float ninf = -INFINITY;
            float4 m = make_float4(ninf, ninf, ninf, ninf);
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const int h = h0 + 2 * ph + dy;
                if (h < 0 || h >= p.H) continue;
#pragma unroll
                for (int dx = 0; dx < KW; ++dx) {
                    const int w = w0 + T::SW * pw + dx;
                    if (w < 0 || w >= p.W) continue;
                    const float4 v = tile[((2 * ph + dy) * PT_IW + T::SW * pw + dx) * c4n + c4];
                    m.x = fmaxf(m.x, __fmaf_rn(v.x, a.x, b.x));
                    m.y = fmaxf(m.y, __fmaf_rn(v.y, a.y, b.y));
                    m.z = fmaxf(m.z, __fmaf_rn(v.z, a.z, b.z));
                    m.w = fmaxf(m.w, __fmaf_rn(v.w, a.w, b.w));
                }
            }
            if (p.relu) { m.x = fmaxf(m.x, 0.f); m.y = fmaxf(m.y, 0.f); m.z = fmaxf(m.z, 0.f); m.w = fmaxf(m.w, 0.f); }
            const int64_t oi = (((int64_t)n * p.Ho + ho) * p.Wo + wo) * C4 + cg;
            reinterpret_cast<float4 *>(out)[oi] = m;
            if (p.nq.write_codes) {
                const float vv[4] = {m.x, m.y, m.z, m.w};
                uint32_t hc[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const uint32_t neg = __float_as_uint(vv[e]) >> 31;
                    const uint32_t q = p.nq.fastdiv ? quantize_f32<true>(vv[e], nq) : quantize_f32<false>(vv[e], nq);
                    hc[e] = __half_as_ushort(lut[q | (neg << p.nq.bits)]);
                }
                reinterpret_cast<uint2 *>(codes)[oi] = make_uint2(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16));
            }
        }
        __syncthreads();                                    // every thread is done with `stage`: it may be refilled
        stage = stage + 1 == PT_STAGES ? 0 : stage + 1;
    }
}

}  // namespace tq

using namespace tq;

namespace {

// the checks and parameters both entry points share; Ho = pooled rows, Wo = pooled columns
int pool_params(PoolParams &p, const float *x, const float *bn_a, const float *bn_b, float *out, void *out_codes, int N,
                int H, int W, int C, int Wo, int relu, float next_sf, int next_bits, int next_terms, int next_enc)
{
    if (!x || !bn_a || !bn_b || !out) return fail(TQ_ERR_INVALID, "NULL pointer");
    p = PoolParams{};
    const int rc = next_quant(p.nq, out_codes, next_sf, next_bits, next_terms, next_enc, FP16_CODE_MAX_BITS, false);
    if (rc != TQ_OK) return rc;
    if (N < 1 || H < 1 || W < 1 || C < 4 || C % 4) return fail(TQ_ERR_INVALID, "bad shape (C must be a multiple of 4)");
    if ((((uintptr_t)x | (uintptr_t)bn_a | (uintptr_t)bn_b | (uintptr_t)out | (uintptr_t)out_codes) & 15u) != 0)
        return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    p.N = N; p.H = H; p.W = W; p.C = C;
    p.Ho = (H + 2 - 3) / 2 + 1;
    p.Wo = Wo;
    p.relu = relu ? 1 : 0;
    return TQ_OK;
}

template <int KW>
int launch_tiled(EncodeTiledFn enc, const float *x, const float *bn_a, const float *bn_b, float *out, void *out_codes,
                 const PoolParams &p, void *stream)
{
    using T = PoolTile<KW>;
    const int N = p.N, H = p.H, W = p.W, C = p.C;
    CUtensorMap tm;
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
    cuuint32_t box[4] = {(cuuint32_t)PT_CB, (cuuint32_t)T::IW, (cuuint32_t)PT_IH, 1};
    cuuint32_t one[4] = {1, 1, 1, 1};
    CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float *>(x), dims, strides, box, one,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled(pool input) failed: %d", (int)r);
    const size_t smem_t = PT_STAGES * (size_t)T::STAGE_BYTES + code_table_bytes(p.nq.bits) + 64 + 128;
    static bool attr_done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        if (cudaFuncSetAttribute(bn_relu_maxpool3x3s2_tiled_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(bn_relu_maxpool3x3s2_tiled_kernel)");
        attr_done[dev] = true;
    }
    const int64_t tiles = (int64_t)N * ((p.Ho + PT_PR - 1) / PT_PR) * ((p.Wo + T::PC - 1) / T::PC) * ((C + PT_CB - 1) / PT_CB);
    const int64_t capt = (int64_t)num_sms() * 2;
    bn_relu_maxpool3x3s2_tiled_kernel<KW><<<(int)(tiles < capt ? tiles : capt), PT_THREADS, smem_t, (cudaStream_t)stream>>>(
        tm, bn_a, bn_b, out, (__half *)out_codes, p);
    count_launch();
    return check_launch("bn_relu_maxpool3x3s2_tiled_kernel");
}

}  // namespace

extern "C" int tq_bn_relu_maxpool_encode_enc(const float *x, const float *bn_a, const float *bn_b, float *out,
                                             void *out_codes, int N, int H, int W, int C, int relu,
                                             float next_sf, int next_bits, int next_terms, int next_enc, void *stream)
{
    PoolParams p;
    int rc = pool_params(p, x, bn_a, bn_b, out, out_codes, N, H, W, C, (W + 2 - 3) / 2 + 1, relu, next_sf, next_bits, next_terms,
                         next_enc);
    if (rc != TQ_OK) return rc;
    // tiled TMA variant for 64-channel blocks on maps of at least one 4 x 14 tile; TQ_POOL_TILED=0 keeps the
    // one-thread-per-output kernel
    static const int tiled_env = getenv("TQ_POOL_TILED") ? atoi(getenv("TQ_POOL_TILED")) : 1;
    if (tiled_env && C % PT_CB == 0 && p.Ho >= PT_PR && p.Wo >= PoolTile<3>::PC) {
        EncodeTiledFn enc = encode_tiled();
        if (enc) return launch_tiled<3>(enc, x, bn_a, bn_b, out, out_codes, p, stream);
    }
    const int64_t total = (int64_t)N * p.Ho * p.Wo * (C / 4);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    if (blocks > cap) blocks = cap;
    const size_t smem = out_codes ? code_table_bytes(p.nq.bits) : 0;
    bn_relu_maxpool3x3s2_kernel<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(
        x, bn_a, bn_b, out, (__half *)out_codes, p);
    count_launch();
    return check_launch("bn_relu_maxpool3x3s2_kernel");
}

extern "C" int tq_bn_relu_maxpool_encode(const float *x, const float *bn_a, const float *bn_b, float *out,
                                         void *out_codes, int N, int H, int W, int C, int relu,
                                         float next_sf, int next_bits, int next_terms, void *stream)
{
    return tq_bn_relu_maxpool_encode_enc(x, bn_a, bn_b, out, out_codes, N, H, W, C, relu, next_sf, next_bits, next_terms,
                                         TQ_ENC_HESE, stream);
}

extern "C" int tq_bn_relu_maxpool_encode_rowmax_enc(const float *x, const float *bn_a, const float *bn_b, float *out,
                                                    void *out_codes, int N, int H, int W, int C, int relu,
                                                    float next_sf, int next_bits, int next_terms, int next_enc, void *stream)
{
    // x: [N, H, W, C] row maxima (W = pooled columns); the vertical 3 / 2 / 1 window is all that is left
    PoolParams p;
    int rc = pool_params(p, x, bn_a, bn_b, out, out_codes, N, H, W, C, W, relu, next_sf, next_bits, next_terms, next_enc);
    if (rc != TQ_OK) return rc;
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    return launch_tiled<1>(enc, x, bn_a, bn_b, out, out_codes, p, stream);
}

extern "C" int tq_bn_relu_maxpool_encode_rowmax(const float *x, const float *bn_a, const float *bn_b, float *out,
                                                void *out_codes, int N, int H, int W, int C, int relu,
                                                float next_sf, int next_bits, int next_terms, void *stream)
{
    return tq_bn_relu_maxpool_encode_rowmax_enc(x, bn_a, bn_b, out, out_codes, N, H, W, C, relu, next_sf, next_bits,
                                                next_terms, TQ_ENC_HESE, stream);
}


// =============================================================================================
// uint8 images -> normalised bf16: what torchvision's ToTensor + Normalize compute on the host in fp32
// (util.py:12-27: x = u8 / 255, then (x - mean[c]) / std[c]), rounded to the bf16 the fused engine consumes.
// Lets a batch cross PCIe as 1 byte per value instead of 2 (bf16) or 4 (the reference's fp32 loader, util.py:54).
// =============================================================================================
namespace tq {

__global__ void __launch_bounds__(256)
u8_normalize_bf16_kernel(const uint8_t *__restrict__ x, __nv_bfloat16 *__restrict__ y, int64_t npix4,
                         float m0, float m1, float m2, float s0, float s1, float s2)
{
    // 4 pixels (12 bytes in, 24 bytes out) per thread: channel of byte k is k % 3
    const float mean[3] = {m0, m1, m2}, sd[3] = {s0, s1, s2};
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < npix4; t += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(x) + t * 3;
        const uint32_t w[3] = {__ldg(src), __ldg(src + 1), __ldg(src + 2)};
        __align__(8) __nv_bfloat16 out[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            const float v = __fdiv_rn((float)((w[k >> 2] >> (8 * (k & 3))) & 0xFFu), 255.0f);
            out[k] = __float2bfloat16_rn(__fdiv_rn(__fsub_rn(v, mean[k % 3]), sd[k % 3]));
        }
        uint2 *dst = reinterpret_cast<uint2 *>(y + t * 12);
        dst[0] = reinterpret_cast<const uint2 *>(out)[0];
        dst[1] = reinterpret_cast<const uint2 *>(out)[1];
        dst[2] = reinterpret_cast<const uint2 *>(out)[2];
    }
}

}  // namespace tq

extern "C" int tq_u8_normalize_bf16(const void *x_u8, void *y_bf16, int64_t npix, const float *mean3, const float *std3,
                                    void *stream)
{
    if (!x_u8 || !y_bf16 || !mean3 || !std3) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (npix < 0 || npix % 4 != 0) return fail(TQ_ERR_INVALID, "pixel count must be a multiple of 4");
    if ((((uintptr_t)x_u8 & 3u) | ((uintptr_t)y_bf16 & 7u)) != 0) return fail(TQ_ERR_INVALID, "pointers must be 4 / 8-byte aligned");
    for (int c = 0; c < 3; ++c)
        if (!(std3[c] > 0.0f)) return fail(TQ_ERR_INVALID, "std must be positive");
    if (npix == 0) return TQ_OK;
    const int64_t n4 = npix / 4;
    int64_t blocks = (n4 + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    if (blocks > cap) blocks = cap;
    u8_normalize_bf16_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const uint8_t *)x_u8, (__nv_bfloat16 *)y_bf16, n4,
                                                                          mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2]);
    count_launch();
    return check_launch("u8_normalize_bf16_kernel");
}
