// tq_gemm.cu -- the contraction that consumes term-revealed operands, on tcgen05 tensor cores.
//
// Reference: tr_layer.py:126 / :154 feed the DEQUANTISED fp32 activations and weights to cuDNN /
// cuBLAS.  Here the operands are the integer term codes themselves (tq_tr_encode_codes) and the scale
// sf_x * sf_w is applied once in the epilogue to the EXACT integer accumulator.  Two operand kinds:
//
//   KIND 0  codes held as fp16 (every |code| <= 2048 is exact in an 11-bit significand), multiplied with
//           tcgen05.mma kind::f16 into fp32 accumulators in TMEM.  All products (<= 2^17) and all partial
//           sums below 2^24 are exact integers in fp32.  The contract is STATIC: the caller passes
//           acc_groups = G only after proving, from the weights alone (tq_conv_weight_l1), that every
//           partial sum of every one of the G channel-block chunks of K stays below 2^24 for ANY
//           activation codes in [0, act_max] (or [-act_max, act_max]); each chunk then accumulates into
//           its own TMEM accumulator and the epilogue adds the G exact integers in int32.
//   KIND 1  codes split into signed 8-bit planes (v = 16 * hi + lo, hi = v >> 4, lo = v & 15), multiplied
//           with tcgen05.mma kind::i8 into s32 accumulators in TMEM: one accumulator per plane-pair
//           weight (hi*hi, hi*lo + lo*hi, lo*lo), recombined with shifts in int32 in the epilogue.
//           Exact for every input (|acc| < 2^31 is checked from the shapes): the unconditional engine.
//
// In both kinds the epilogue sees the int32 accumulator of an integer conv and computes
// t = float(acc) * scale (one RN conversion, exact below 2^24, and one RN multiply).
//
// Implicit GEMM, NHWC activations, [R*S][Cout][Cin] weights:
//   M tile  = a box of  nbox x hbox x wbox  output pixels (<= 128 rows), fetched per filter tap
//             (r, s) by ONE tiled 4-D TMA load at offset (h0*stride + r - pad, w0*stride + s - pad)
//             with element strides = conv stride; out-of-image pixels arrive as zeros (padding
//             is free), so there is no im2col buffer and no index arithmetic on the SMs.
//   K loop  = taps x 64-channel blocks; each stage holds a 128x64 A tile and a BLOCK_N x 64 B
//             tile, both K-major with the 128-byte swizzle TMA and UMMA agree on.
//   N tile  = BLOCK_N output channels; two accumulator stages in TMEM so the epilogue of tile i
//             overlaps the MMAs of tile i+1.
// Warp roles (640 threads, persistent CTAs, one per SM): warp 0 TMA producer (one thread), warp 1 MMA
// issuer (one thread), warp 2 TMEM allocator, warps 4-19 four epilogue groups of four warps: group
// (a, h) drains column half h of every second tile (TMEM -> registers -> fused tail -> swizzled smem ->
// TMA store).
//
// CTA pairs (template argument CG = 2, the streamed-weight halo mode on maps with at least one pair of tiles per TPC): two
// CTAs of a cluster run ONE tcgen05.mma.cta_group::2 of M = 256, each holding the halo box of its own M tile and half of
// the weight tile -- see the helpers below and DESIGN.md section 6.  Small maps (7x7) use a packed halo: several
// whole images per tile with shared zero padding.
//
// Measurement / experiment switches (environment, read once; none is needed in normal use):
//   TQ_CONV_PAIR=0 / TQ_CONV_PAIR3=1           single CTAs everywhere / CTA pairs also for the resident-weight halo mode
//   TQ_CONV_NO_PACKED                          no packed halo for small maps (per-tap streaming instead)
//   TQ_CONV_HALO_SLACK=n                       percent of extra tiles a halo tiling may cost (default 16)
//   -DTQ_CONV_TRACE (tools/conv_trace.sh)      debug build: per-role cycle accounting printed by two CTAs per launch
//   TQ_CONV_SKIP_EPI / _SKIP_MMA / _SKIP_TMA   run without the epilogue / the MMAs / the TMA loads (results are garbage;
//                                              SKIP_TMA=2 / 4 in the streamed-weight halo mode: no weight / no halo loads):
//                                              isolates which pipeline paces a layer (tools/conv_microbench.py)
//   TQ_CONV_STAGES=n, TQ_CONV_ASTAGES=n        cap the stage ring / set the halo-buffer ring depth (MODE 4)
//   TQ_CONV_WBOX / TQ_CONV_HBOX                force the pixel box of MODE 0 tiles
//   TQ_CONV_NO_PROG / _NO_HALO / _NO_HALO4     fall back from resident weights / halo loads to per-tap streaming
//   TQ_CONV_N256=1                             BLOCK_N = 256 tiles where Cout % 256 == 0 (slower on ResNet shapes)
//   TQ_CONV_HALO_BASEOFF=1                     set the UMMA descriptor base-offset field in halo mode (WRONG results:
//                                              kept as the record of how the swizzle was found to be address-based)
#ifdef TQ_CONV_TRACE
#include <cstdio>
#endif
#include <cuda.h>

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <vector>

#include "tq_common.cuh"

namespace tq {

constexpr int GM_BLOCK_M = 128;
constexpr int GM_ROW_BYTES = 128;               // one K block = one 128-byte swizzle row: 64 fp16 or 128 s8 channels
constexpr int GM_BLOCK_K = 64;                  // fp16 elements per K block (KIND 0)
constexpr int GM_THREADS = 640;                 // 4 control warps + 4 epilogue groups of 4 warps
constexpr int GM_A_BYTES = GM_BLOCK_M * GM_ROW_BYTES;
constexpr int GM_I8_SHIFT = 4;                  // s8 planes: v = (hi << 4) + lo

struct ConvGeom {
    int N, H, W, C, Cout, R, S, stride, pad, Ho, Wo;
    int wbox, hbox, nbox;                       // output pixels per M tile
    int hw;                                     // pixels per MMA row group: wbox, or wbox + S - 1 in halo mode
    int step_w, step_h, off_w, off_h;           // tile origin in output pixels: (tw * step_w + off_w, th * step_h + off_h)
    int pool, pool_p, pool_q;                   // fused 3x3/s2/p1 max-pool (stem): pooled pixels per tile
    int halo, halo_baseoff;                     // halo mode (MODE 3); whether to set the descriptor's base-offset field
    int img_h1;                                 // packed halo (small maps, several images per tile): H + 1 box rows per image, else 0
    int pair;                                   // MODE 4 on CTA pairs (cta_group::2): two M tiles per MMA, half a weight tile per CTA
    int tiles_w, tiles_h, tiles_n;              // M tiles along w, h, image
    int m_tiles, n_tiles, kc_blocks;
    int a_tx_bytes;                             // bytes one A box deposits
    float scale;
    // shared-memory carve-up (runtime, 1024-byte aligned regions)
    int a_stages, a_stage_bytes;                 // MODE 4: ring of halo buffers (at bstat_off) beside the weight-tile ring
    int stages, stage_bytes, ring_off, bstat_off, epi_off, epi_group_bytes, epi_codes_off, lut_off, bar_off, smem_total;
    // "program" mode for small layers (Cout <= BLOCK_N, all weights resident in shared memory): the K loop is
    // a table of A loads, each followed by 1-2 MMAs against stationary B tiles into an accumulator group
    int prog_steps, nb_tiles, n_groups;
    // exact-accumulator contract (see the file header).  KIND 0: n_groups = K chunks of kcpg channel blocks each, summed
    // as integers when acc_int.  KIND 1: planes_a x planes_w signed 8-bit planes (stacked along the image / tap
    // dimension of the operand tensors), plane pair (pa, pw) accumulates into group pa + pw; kblk = channels per block.
    int kcpg, acc_int, planes_a, planes_w, kblk;
    int b_rows;                                 // rows of a resident weight tile when it is not BLOCK_N (MODE 2: 128)
    int dbg_skip_epilogue;      // profiling aid (TQ_CONV_SKIP_EPI=1): drain accumulators without storing
    int dbg_skip_mma, dbg_skip_tma;   // TQ_CONV_SKIP_MMA / TQ_CONV_SKIP_TMA: isolate the load and the MMA pipelines
    // MODE 2 step table, one packed word per (A plane, filter row), planes stacked along N (coordinate
    // n0 + plane * N):   n_mma | b_tile0 << 4 | group0 << 8 | b_tile1 << 12 | group1 << 16
    uint32_t prog_mma[16];
    // fused epilogue (all optional):  t = acc*scale (+bias) ; t = fma(t, bn_a, bn_b) ; t += residual ;
    // t = max(t, 0) ; fp32 tile out (TMA store) ; fp16 term codes of t for the next layer (TMA store)
    const float *bias, *bn_a, *bn_b, *residual;
    int relu, relu6, write_f32;                 // relu6: additionally clamp at 6 (ReLU6 of the depthwise CNNs)
    NextQuant nq;
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap *map, uint64_t *bar, void *dst, int c0, int c1, int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap *map, uint64_t *bar, void *dst, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// one lane of a converged warp (the rest of the warp stays converged around the asm that follows)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xFFFFFFFF;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
template <int KIND>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    if constexpr (KIND == 1) umma_i8(tmem_d, desc_a, desc_b, idesc, accumulate);
    else umma_f16(tmem_d, desc_a, desc_b, idesc, accumulate);
}
// ---- CTA pair (cta_group::2): two CTAs of a cluster on one TPC run ONE tcgen05.mma of M = 256 -- each supplies the A rows
// of its own M tile and HALF of the B tile (N / 2 rows), so per CTA the weight traffic from L2 and the B reads from shared
// memory are halved.  The leader (cluster rank 0) issues every MMA and commit; loads of both CTAs complete on the leader's
// barriers, commits arrive on the same barrier of both CTAs.
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// loads into this CTA's shared memory whose bytes complete on a barrier of either CTA of the pair
__device__ __forceinline__ void tma_load_4d_pair(const CUtensorMap *map, uint32_t bar_cluster, void *dst, int c0, int c1, int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(const CUtensorMap *map, uint32_t bar_cluster, void *dst, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives (once the MMAs issued so far have retired) on the same barrier of BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// -DTQ_CONV_TRACE (debug builds only, tools/conv_trace.sh): per-role cycle accounting with clock64, printed by two CTAs
#ifdef TQ_CONV_TRACE
#define TR_DECL(n) long long trc[n] = {}
#define TR(slot, ...) do { const long long _t = clock64(); __VA_ARGS__; trc[slot] += clock64() - _t; } while (0)
#define TR_T0(name) const long long name = clock64()
#define TR_SINCE(slot, name) trc[slot] += clock64() - name
#else
#define TR_DECL(n)
#define TR(slot, ...) do { __VA_ARGS__; } while (0)
#define TR_T0(name)
#define TR_SINCE(slot, name)
#endif

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tma_store_4d(const CUtensorMap *map, const void *src, int c0, int c1, int c2, int c3)
{
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void cp_async16(void *dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// K-major, 128-byte swizzle: rows of 128 B, 8-row atoms 1024 B apart (SBO), LBO unused,
// descriptor version 1 (sm_100), layout type 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

constexpr int GM_LUT_MAX_BITS = 10;             // fused next-layer encode: code_table_bytes(bits) in smem
constexpr int GM_MAX_STAGES = 8;
constexpr int GM_EPI_GROUPS = 4;                // (accumulator stage, column half)
constexpr int GM_EPI_F32_BYTES = 16384;         // per epilogue group: [128][32] fp32 staging (output tile / residual tile)
constexpr int GM_EPI_CODE_BYTES = 8192;         // per epilogue group: [128][32] fp16 code staging
constexpr int GM_SMEM_BUDGET = 227 * 1024;

// ---- epilogue arithmetic (per 32-column chunk of one accumulator row) -------------------------
// FULL = all 32 channels of the chunk exist (c0 + 32 <= Cout): no per-channel guards, parameter loads with
// immediate offsets
template <bool FULL>
__device__ __forceinline__ void epi_affine(float (&t)[32], const ConvGeom &g, int c0)
{
    if (g.bias) {
        const float4 *bp = reinterpret_cast<const float4 *>(g.bias + c0);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            if (FULL || c0 + j < g.Cout) {
                const float4 b = __ldg(bp + (j >> 2));
                t[j] = __fadd_rn(t[j], b.x); t[j + 1] = __fadd_rn(t[j + 1], b.y);
                t[j + 2] = __fadd_rn(t[j + 2], b.z); t[j + 3] = __fadd_rn(t[j + 3], b.w);
            }
        }
    }
    if (g.bn_a) {
        const float4 *ap = reinterpret_cast<const float4 *>(g.bn_a + c0);
        const float4 *bp = reinterpret_cast<const float4 *>(g.bn_b + c0);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            if (FULL || c0 + j < g.Cout) {
                const float4 a = __ldg(ap + (j >> 2));
                const float4 b = __ldg(bp + (j >> 2));
                t[j] = __fmaf_rn(t[j], a.x, b.x); t[j + 1] = __fmaf_rn(t[j + 1], a.y, b.y);
                t[j + 2] = __fmaf_rn(t[j + 2], a.z, b.z); t[j + 3] = __fmaf_rn(t[j + 3], a.w, b.w);
            }
        }
    }
}

// residual add (the staging tile holds the residual), ReLU, fp32 tile and / or term codes into the staging tiles.
// RELU: the values are >= 0 afterwards, so the encode needs neither |x| nor the sign half of the table.
// Written as PHASES over the 32 values of the chunk, each behind ONE uniform branch (ncu, round 2: with the flags tested
// inside the per-4-value loop the chunk cost 37 SASS instructions per value against ~12 of arithmetic).  The fused
// encode always uses the hoisted-reciprocal divide: the host refuses next_sf outside [2^-30, 2^30] (check_conv_args).
// Table lookup: after the two round-down adds the quantised value sits in the mantissa of t = 2^23 + q, i.e.
// bits = 0x4B000000 + q, so the byte address of entry (q | sign << bits) is 2 * bits + const: one IMAD + one LDS.
__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr)
{
    uint16_t v;
    asm("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(saddr));      // the table is read-only after the prologue barrier
    return v;
}

template <bool RELU>
__device__ __forceinline__ void epi_stage(float (&t)[32], const ConvGeom &g, uint8_t *st_f32, uint8_t *st_codes, int row,
                                          bool has_res, const __half *lut, const Quant &nq)
{
    const uint32_t sw128 = (uint32_t)(row & 7);             // 16B piece index ^= row % 8
    const uint32_t sw64 = (uint32_t)((row >> 1) & 3);       // 16B piece index ^= (row / 2) % 4
    uint8_t *frow = st_f32 + row * 128, *crow = st_codes + row * 64;
    if (has_res) {                                          // rows / channels outside the tensor arrive as zeros
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 r = *reinterpret_cast<const float4 *>(frow + (((uint32_t)(j >> 2) ^ sw128) << 4));
            t[j] = __fadd_rn(t[j], r.x); t[j + 1] = __fadd_rn(t[j + 1], r.y);
            t[j + 2] = __fadd_rn(t[j + 2], r.z); t[j + 3] = __fadd_rn(t[j + 3], r.w);
        }
    }
    if (RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) t[j] = fmaxf(t[j], 0.0f);          // NaN -> 0
        if (g.relu6) {
#pragma unroll
            for (int j = 0; j < 32; ++j) t[j] = fminf(t[j], 6.0f);
        }
    }
    if (g.write_f32) {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4 *>(frow + (((uint32_t)(j >> 2) ^ sw128) << 4)) = make_float4(t[j], t[j + 1], t[j + 2], t[j + 3]);
    }
    if (g.nq.write_codes) {
        // entry address = lut + 2 * (q | sign << bits), q = bits(t) - 0x4B000000
        const uint32_t lut_s = smem_u32(lut) - 2u * 0x4B000000u;
        const uint32_t sign_off = 2u << g.nq.bits;          // byte offset of the negative half of the table
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
            uint32_t hc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float x = t[j + e];
                float r;
                if (RELU) r = div_rn_nonneg<true>(x, nq);               // already >= 0 and not NaN
                else r = div_rn_nonneg<true>(fmaxf(fabsf(x), 0.0f), nq);
                r = fminf(r, nq.maxv);
                float q = __fadd_rd(r, 0.5f);
                q = __fadd_rd(q, 8388608.0f);
                uint32_t addr = __float_as_uint(q) * 2u + lut_s;
                if (!RELU) addr += (__float_as_uint(x) >> 31) * sign_off;
                hc[e] = lds_u16(addr);
            }
            *reinterpret_cast<uint4 *>(crow + (((uint32_t)(j >> 3) ^ sw64) << 4)) =
                make_uint4(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16), hc[4] | (hc[5] << 16), hc[6] | (hc[7] << 16));
        }
    }
}

// MODE 0: A and B tiles stream through the stage ring.  MODE 1: all weight tiles resident in shared memory
// (tile = filter tap, one 64-channel block), only A streams.  MODE 2 (the hi/lo stem conv): resident weights,
// one halo load per A plane (x_hi, x_lo) covering all R filter rows, and a step table naming, per
// (plane, filter row), one or two MMA groups = (resident weight tile, accumulator group).
// MODE 3: resident weights + ONE halo load per tile (stride-1 convs): the box of (hbox+R-1) x (wbox+S-1)
// input pixels lands once in shared memory and filter tap (r, s) is the same buffer read from row
// r * (wbox+S-1) + s on: MMA row m is halo row start + m, i.e. output pixel (m / hw, m % hw), of which the
// columns m % hw >= wbox are junk and dropped by the epilogue.  A traffic per tile falls from R*S boxes to one.
// MODE 4: halo mode for layers whose weights do not fit shared memory (Cout > 64 or several 64-channel blocks):
// a ring of halo buffers (one load per tile and channel block) and a ring of streamed weight tiles (one per
// filter tap and channel block), each with its own full / empty barriers.
// RELU: the epilogue's ReLU flag as a compile-time constant (the encode after a ReLU needs no sign handling; a
// run-time branch would duplicate the staging code inside one kernel and cost instruction-cache misses).
// KIND: 0 = fp16 codes, kind::f16, fp32 accumulators; 1 = s8 planes, kind::i8, s32 accumulators (MODE 0 only).
// CG: 1 = one CTA per tile; 2 = CTA pair (MODE 4 only): the pair takes two M tiles of the same N tile, see the helpers above.
template <int BLOCK_N, int MODE, bool RELU, int KIND, int CG = 1>
__global__ void __launch_bounds__(GM_THREADS, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmD,
                      const __grid_constant__ CUtensorMap tmR, const __grid_constant__ ConvGeom g)
{
    static_assert(KIND == 0 || MODE == 0, "the s8-plane engine streams both operands (MODE 0)");
    static_assert(CG == 1 || ((MODE == 4 || MODE == 3) && KIND == 0), "the CTA pair runs the halo modes");
    // MODE 2 (hi/lo stem conv): a resident weight tile stacks the hi plane (rows 0..63) on the lo plane (rows 64..127) and
    // ONE N = 128 MMA computes x * w_hi into accumulator columns [c, c + 64) and x * w_lo into [c + 64, c + 128): 64 cycles
    // instead of two N = 64 MMAs at 57 each.  The epilogue's view stays BLOCK_N = 64 output channels, four column groups.
    constexpr int MMA_N = MODE == 2 ? 2 * BLOCK_N : BLOCK_N;
    constexpr int B_BYTES = MMA_N * GM_ROW_BYTES;
    const int STAGES = g.stages;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *ring = smem + g.ring_off;              // STAGES x (A tile [+ B tile when streaming])
    uint8_t *bstat = smem + g.bstat_off;            // stationary B tiles (program mode)
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + g.bar_off);
    uint64_t *empty_bar = full_bar + GM_MAX_STAGES;
    uint64_t *tfull_bar = empty_bar + GM_MAX_STAGES;    // [3] accumulator ready
    uint64_t *tempty_bar = tfull_bar + 3;               // [3] accumulator drained
    uint64_t *bfull_bar = tempty_bar + 3;               // stationary weights landed
    uint64_t *res_bar = bfull_bar + 1;                  // [4] residual tile landed in an epilogue group's staging
    uint64_t *afull_bar = res_bar + GM_EPI_GROUPS;      // [4] MODE 4: halo buffer landed / consumed
    uint64_t *aempty_bar = afull_bar + 4;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(aempty_bar + 4);
    constexpr bool prog = MODE >= 1 && MODE <= 3;       // weights resident in shared memory
    const int acc_cols = g.n_groups * BLOCK_N;          // TMEM columns of one accumulator stage

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Tile walk.  CG 1: CTA b takes tiles b, b + grid, ...; tile = m_tile * n_tiles + n_tile.  CG 2: pair p = b / 2 takes
    // "super tiles" p, p + grid / 2, ...; super tile = (m_tile / 2) * n_tiles + n_tile and CTA rank r of the pair owns
    // m_tile = 2 * (super / n_tiles) + r.  With an odd number of M tiles the last one has no partner: the partner CTA runs
    // a tile whose image index is out of range -- its TMA loads are zero-filled and its TMA stores dropped.
    const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
    const int tile_first = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_step = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int total_tiles = CG == 2 ? ((g.m_tiles + 1) / 2) * g.n_tiles : g.m_tiles * g.n_tiles;
    auto m_tile_of = [&](int tile) { return CG == 2 ? 2 * (tile / g.n_tiles) + (int)cta_rank : tile / g.n_tiles; };
    const int kblocks = g.R * g.S * g.kc_blocks * (KIND == 1 ? g.planes_a * g.planes_w : 1);
    // accumulator stages in TMEM: three when they fit the 512 columns (the MMA issuer may then run two tiles ahead of
    // an epilogue that holds its accumulator until the last chunk is in registers), else two; a tile with four K chunks
    // (or three plane-pair accumulators) of 128 columns owns all of TMEM and runs with ONE stage: its MMAs start when
    // the previous tile's accumulators are in registers
    const int ACC_STAGES = 3 * acc_cols <= 512 ? 3 : (2 * acc_cols <= 512 ? 2 : 1);
    uint32_t TMEM_COLS = 32;                            // power of two >= the accumulator stages
    while (TMEM_COLS < (uint32_t)(ACC_STAGES * acc_cols)) TMEM_COLS <<= 1;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
        if (g.write_f32) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmC) : "memory");
        if (g.nq.write_codes) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmD) : "memory");
        if (g.residual) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmR) : "memory");
    }
    __half *lut = reinterpret_cast<__half *>(smem + g.lut_off);
    if (g.nq.write_codes) {
        // (q, sign) -> fp16 term code of the consumer's quantiser, as in tr_elem_kernel
        for (uint32_t i = threadIdx.x; i < (2u << g.nq.bits); i += GM_THREADS) {
            int code = elem_code(i & ((1u << g.nq.bits) - 1u), g.nq.enc, g.nq.terms);
            lut[i] = __int2half_rn((i >> g.nq.bits) ? -code : code);
        }
    }
    if (MODE == 4 && g.img_h1) {
        // packed halo: the rows after each box (read by the taps of the last image's last pixels: its bottom padding)
        // are never written by TMA -- zero them once, for the tensor cores' (async-proxy) reads
        const int tail = g.a_stage_bytes - g.a_tx_bytes;
        for (int i = threadIdx.x * 16; i < g.a_stages * tail; i += GM_THREADS * 16)
            *reinterpret_cast<uint4 *>(bstat + (i / tail) * g.a_stage_bytes + g.a_tx_bytes + (i % tail)) = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async();
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        mbar_init(bfull_bar, 1);
        // an accumulator stage is drained by two epilogue groups (256 threads); with a single stage all four groups
        // drain every tile (a quarter of the columns each)
        // (CTA pair: the leader's barrier also collects the partner's epilogue threads)
        for (int i = 0; i < 3; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], (ACC_STAGES == 1 ? 512 : 256) * CG); }
        for (int i = 0; i < GM_EPI_GROUPS; ++i) mbar_init(&res_bar[i], 1);
        for (int i = 0; i < 4; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if constexpr (CG == 2) {                            // the same warp of both CTAs, same destination offset
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all();              // the partner's barriers are initialised before anything arrives on them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        // ONE thread runs the whole loop: no elect / reconvergence instructions per stage -- the per-stage
        // latency of this loop (and of the MMA loop below) bounds the kernel when a stage holds only ~230
        // cycles of tensor work (BLOCK_N = 64), see DESIGN.md section 6.
        if (elect_one()) {
            int stage = 0;
            uint32_t phase = 0;
            uint8_t *sdst = ring;
            if constexpr (prog && CG == 2) {                // this CTA's half of every resident tile, counted on the leader's barrier
                const uint32_t bfull0 = mapa_u32(smem_u32(bfull_bar), 0);
                if (cta_rank == 0) mbar_expect_tx(bfull_bar, (uint32_t)(g.nb_tiles * B_BYTES));
                for (int t = 0; t < g.nb_tiles; ++t)
                    tma_load_3d_pair(&tmB, bfull0, bstat + t * (B_BYTES / 2), 0, (int)cta_rank * (BLOCK_N / 2), t);
            } else if constexpr (prog) {                    // all weights once: they stay resident
                mbar_expect_tx(bfull_bar, (uint32_t)(g.nb_tiles * B_BYTES));
                for (int t = 0; t < g.nb_tiles; ++t) tma_load_3d(&tmB, bfull_bar, bstat + t * B_BYTES, 0, 0, t);
            }
            if constexpr (MODE == 4 && CG == 2) {
                // CTA pair: this CTA's halo box and its half (rows cta_rank * 64 ..) of every weight tile, TWO filter taps
                // per ring stage (eight MMAs per hand-shake).  All bytes complete on the LEADER's full barriers, which the
                // leader arms with the byte count of both CTAs; a slot is free when the leader's multicast commit has
                // arrived on this CTA's own empty barrier.
                constexpr uint32_t B_HALF = (uint32_t)B_BYTES / 2;
                const int kcb = g.kc_blocks, taps = g.R * g.S, a_stages = g.a_stages;
                const uint32_t full0 = mapa_u32(smem_u32(full_bar), 0), afull0 = mapa_u32(smem_u32(afull_bar), 0);
                int as = 0, bs = 0;
                uint32_t aph = 0, bph = 0;
                TR_DECL(4);
                TR_T0(tp0);
                // The halo box of step (tile, kc) + 1 is requested BEFORE the weight tiles of step (tile, kc): its buffer (a ring
                // of three) was last read two steps ago, so the request never waits, and the box has a whole step to land.
                auto load_halo = [&](int tile, int kc) {
                    const int m_tile = m_tile_of(tile);
                    const int tw = m_tile % g.tiles_w, th = (m_tile / g.tiles_w) % g.tiles_h, tn = m_tile / (g.tiles_w * g.tiles_h);
                    TR(0, mbar_wait(&aempty_bar[as], aph ^ 1u));
                    if (cta_rank == 0) mbar_expect_tx(&afull_bar[as], 2u * (uint32_t)g.a_tx_bytes);
                    tma_load_4d_pair(&tmA, afull0 + 8u * (uint32_t)as, bstat + as * g.a_stage_bytes, kc * GM_BLOCK_K,
                                     tw * g.step_w - g.pad, th * g.step_h - g.pad, tn * g.nbox);     // stride 1
                    if (++as == a_stages) { as = 0; aph ^= 1u; }
                };
                const bool ahead = a_stages >= 3;
                if (ahead && tile_first < total_tiles) load_halo(tile_first, 0);
                for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
                    const int n_tile = tile % g.n_tiles;
                    const int nb0 = n_tile * BLOCK_N + (int)cta_rank * (BLOCK_N / 2);
                    for (int kc = 0; kc < kcb; ++kc) {
                        if (!ahead) load_halo(tile, kc);
                        else if (kc + 1 < kcb) load_halo(tile, kc + 1);
                        else if (tile + tile_step < total_tiles) load_halo(tile + tile_step, 0);
                        for (int tap = 0; tap < taps; tap += 2) {
                            const int nt = taps - tap >= 2 ? 2 : 1;
                            TR(1, mbar_wait(&empty_bar[bs], bph ^ 1u));
                            if (cta_rank == 0) mbar_expect_tx(&full_bar[bs], 2u * (uint32_t)nt * B_HALF);
                            for (int j = 0; j < nt; ++j)
                                tma_load_3d_pair(&tmB, full0 + 8u * (uint32_t)bs, ring + bs * g.stage_bytes + j * (int)B_HALF,
                                                 kc * GM_BLOCK_K, nb0, tap + j);
                            if (++bs == STAGES) { bs = 0; bph ^= 1u; }
                        }
                    }
                }
#ifdef TQ_CONV_TRACE
                TR_SINCE(2, tp0);
                if (blockIdx.x == 0 || blockIdx.x == 101)
                    printf("cta %3d producer (pair): total %lld, wait halo-empty %lld, wait weight-empty %lld\n", blockIdx.x, trc[2], trc[0], trc[1]);
#endif
            } else if constexpr (MODE == 4) {
                const int kcb = g.kc_blocks, taps = g.R * g.S, a_stages = g.a_stages;
                int as = 0, bs = 0;
                uint32_t aph = 0, bph = 0;
                TR_DECL(4);
                TR_T0(tp0);
                for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
                    const int n_tile = tile % g.n_tiles, m_tile = m_tile_of(tile);
                    const int tw = m_tile % g.tiles_w, th = (m_tile / g.tiles_w) % g.tiles_h, tn = m_tile / (g.tiles_w * g.tiles_h);
                    const int w_in0 = tw * g.step_w - g.pad, h_in0 = th * g.step_h - g.pad;     // stride 1
                    const int nb0 = n_tile * BLOCK_N;
                    for (int kc = 0; kc < kcb; ++kc) {
                        TR(0, mbar_wait(&aempty_bar[as], aph ^ 1u));
                        if (g.dbg_skip_tma == 4) {                      // TQ_CONV_SKIP_TMA=4: no halo loads (isolation run)
                            mbar_arrive(&afull_bar[as]);
                        } else {
                        mbar_expect_tx(&afull_bar[as], (uint32_t)g.a_tx_bytes);
                        tma_load_4d(&tmA, &afull_bar[as], bstat + as * g.a_stage_bytes, kc * GM_BLOCK_K, w_in0, h_in0, tn * g.nbox);
                        }
                        if (++as == a_stages) { as = 0; aph ^= 1u; }
                        for (int tap = 0; tap < taps; ++tap) {
                            TR(1, mbar_wait(&empty_bar[bs], bph ^ 1u));
                            if (g.dbg_skip_tma == 2) {                  // TQ_CONV_SKIP_TMA=2: no weight loads (isolation run)
                                mbar_arrive(&full_bar[bs]);
                            } else {
                            mbar_expect_tx(&full_bar[bs], (uint32_t)B_BYTES);
                            tma_load_3d(&tmB, &full_bar[bs], ring + bs * B_BYTES, kc * GM_BLOCK_K, nb0, tap);
                            }
                            if (++bs == STAGES) { bs = 0; bph ^= 1u; }
                        }
                    }
                }
#ifdef TQ_CONV_TRACE
                TR_SINCE(2, tp0);
                if (blockIdx.x == 0 || blockIdx.x == 100)
                    printf("cta %3d producer: total %lld, wait halo-empty %lld, wait weight-empty %lld\n", blockIdx.x, trc[2], trc[0], trc[1]);
#endif
            } else if constexpr (MODE == 3 && CG == 2) {
                // CTA pair, resident weights: one halo box per tile and CTA, completing on the leader's full barrier
                const uint32_t full0 = mapa_u32(smem_u32(full_bar), 0);
                for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
                    const int m_tile = m_tile_of(tile);
                    const int tw = m_tile % g.tiles_w, th = (m_tile / g.tiles_w) % g.tiles_h, tn = m_tile / (g.tiles_w * g.tiles_h);
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2u * (uint32_t)g.a_tx_bytes);
                    tma_load_4d_pair(&tmA, full0 + 8u * (uint32_t)stage, sdst, 0, tw * g.step_w - g.pad, th * g.step_h - g.pad, tn * g.nbox);
                    sdst += g.stage_bytes;
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; sdst = ring; }
                }
            } else {
            const int steps = MODE == 3 ? g.kc_blocks : (MODE == 2 ? g.prog_steps / g.R : (prog ? g.prog_steps : kblocks));
            const int S = MODE == 3 ? 1 : g.S, kc_blocks = g.kc_blocks, stage_bytes = g.stage_bytes;
            const uint32_t tx_bytes = (uint32_t)g.a_tx_bytes + (prog ? 0u : (uint32_t)B_BYTES);
            const bool skip_tma = g.dbg_skip_tma != 0;
            for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
                const int n_tile = tile % g.n_tiles, m_tile = m_tile_of(tile);
                const int tw = m_tile % g.tiles_w, th = (m_tile / g.tiles_w) % g.tiles_h, tn = m_tile / (g.tiles_w * g.tiles_h);
                const int w_in0 = (tw * g.step_w + g.off_w) * g.stride - g.pad, h_in0 = (th * g.step_h + g.off_h) * g.stride - g.pad, n0 = tn * g.nbox;
                const int nb0 = n_tile * BLOCK_N;
                int r = 0, sx = 0, kc = 0;                  // tap (r, sx), channel block kc
                int pa = 0, pw = 0;                         // KIND 1: operand planes of this step (pa outer, pw inner)
                const int kblk = g.kblk, taps_all = g.R * g.S;
                for (int st = 0; st < steps; ++st) {
                    int cc, cw, ch, cn, bt;
                    if constexpr (MODE == 2) {
                        cw = w_in0; ch = h_in0; cc = 0; cn = n0 + st * g.N;   // plane st: rows h_in0 .. h_in0 + hbox + R - 2
                        bt = 0;
                    } else {
                        cw = w_in0 + sx; ch = h_in0 + r; cc = kc * kblk; cn = n0; bt = r * S + sx;
                        if constexpr (KIND == 1) { cn += pa * g.N; bt += pw * taps_all; }   // planes stacked along image / tap
                    }
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    if (skip_tma) mbar_arrive(&full_bar[stage]);
                    else {
                        mbar_expect_tx(&full_bar[stage], tx_bytes);
                        tma_load_4d(&tmA, &full_bar[stage], sdst, cc, cw, ch, cn);
                        if constexpr (!prog) tma_load_3d(&tmB, &full_bar[stage], sdst + GM_A_BYTES, cc, nb0, bt);
                    }
                    sdst += stage_bytes;
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; sdst = ring; }
                    if (++kc == kc_blocks) {
                        kc = 0;
                        if constexpr (KIND == 1) {            // tap outermost, then plane pair, then channel block
                            if (++pw == g.planes_w) { pw = 0; if (++pa == g.planes_a) { pa = 0; if (++sx == S) { sx = 0; ++r; } } }
                        } else {
                            if (++sx == S) { sx = 0; ++r; }
                        }
                    }
                }
            }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        // ONE thread issues every tcgen05.mma / tcgen05.commit (see the producer's note).
        // instruction descriptor: both operands K-major, N = BLOCK_N, M = 128;  KIND 0: D = F32 (bits 4-5 = 1),
        // A = B = F16 (0);  KIND 1: D = S32 (2), A = B = signed 8-bit (a_format bits 7-9 = 1, b_format bits 10-12 = 1)
        constexpr uint32_t IDESC = (KIND == 1 ? ((2u << 4) | (1u << 7) | (1u << 10)) : (1u << 4)) |
                                   ((uint32_t)(MMA_N >> 3) << 17) | ((uint32_t)(GM_BLOCK_M >> 4) << 24);
        constexpr uint64_t DESC_HI = ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
        if (elect_one() && cta_rank == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            const uint32_t a_lo0 = ((smem_u32(ring) & 0x3FFFFu) >> 4) | (1u << 16);      // descriptor low words
            const uint32_t b_lo0 = ((smem_u32(bstat) & 0x3FFFFu) >> 4) | (1u << 16);
            const uint32_t a_step = (uint32_t)g.stage_bytes >> 4;
            uint32_t a_lo = a_lo0;
            const int steps = prog ? g.prog_steps : kblocks;
            const bool skip_mma = g.dbg_skip_mma != 0;
            uint32_t pw = MODE == 2 ? g.prog_mma[0] : 0u;
            int as4 = 0;                                    // MODE 4: halo ring position
            uint32_t aph4 = 0;
            if constexpr (prog) {
                mbar_wait(bfull_bar, 0);
                tc_fence_after();
            }
            TR_DECL(6);
            TR_T0(ti0);
            for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
                TR(0, mbar_wait(&tempty_bar[acc], acc_phase ^ 1u));
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * acc_cols);
                if constexpr (MODE == 4 && CG == 2) {
                    // leader of the CTA pair: M = 256 (both CTAs' tiles), two taps per stage, multicast commits
                    constexpr uint32_t IDESC2 = (1u << 4) | ((uint32_t)(MMA_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
                    constexpr uint32_t B_HALF16 = (uint32_t)(B_BYTES / 2) >> 4;
                    const int taps = g.R * g.S, S = g.S, kcb = g.kc_blocks;
                    const uint32_t row_step = (uint32_t)g.hw * 8u;
                    int kin = 0;
                    uint32_t td = tmem_d;
                    for (int kc = 0; kc < kcb; ++kc) {
                        TR(1, mbar_wait(&afull_bar[as4], aph4));
                        tc_fence_after();
                        uint32_t a_row = b_lo0 + (uint32_t)as4 * ((uint32_t)g.a_stage_bytes >> 4);
                        int sx = 0;
                        for (int tap = 0; tap < taps; tap += 2) {
                            const int nt = taps - tap >= 2 ? 2 : 1;
                            TR(2, mbar_wait(&full_bar[stage], phase));
                            tc_fence_after();
                            for (int j = 0; j < nt; ++j) {
                                const uint64_t da = DESC_HI | (a_row + (uint32_t)sx * 8u);
                                const uint64_t db = DESC_HI | (a_lo + (uint32_t)j * B_HALF16);
#pragma unroll
                                for (int k = 0; k < GM_ROW_BYTES / 32; ++k)
                                    umma_f16_pair(td, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC2, (kin | (tap + j) | k) != 0 ? 1u : 0u);
                                if (++sx == S) { sx = 0; a_row += row_step; }
                            }
                            umma_commit_pair(&empty_bar[stage]);        // both CTAs' halves of the stage are free
                            a_lo += a_step;
                            if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                        }
                        umma_commit_pair(&aempty_bar[as4]);
                        if (++as4 == g.a_stages) { as4 = 0; aph4 ^= 1u; }
                        if (++kin == g.kcpg) { kin = 0; td += BLOCK_N; }
                    }
                } else if constexpr (MODE == 4) {
                    const int taps = g.R * g.S, S = g.S, kcb = g.kc_blocks;
                    const uint32_t row_step = (uint32_t)g.hw * 8u;      // one halo row of pixels, in 16-byte units
                    int kin = 0;                                        // channel block within the K chunk
                    uint32_t td = tmem_d;                               // accumulator of the current K chunk
                    for (int kc = 0; kc < kcb; ++kc) {
                        TR(1, mbar_wait(&afull_bar[as4], aph4));
                        tc_fence_after();
                        uint32_t a_row = b_lo0 + (uint32_t)as4 * ((uint32_t)g.a_stage_bytes >> 4);   // halo ring lives at bstat
                        int sx = 0;
                        for (int tap = 0; tap < taps; ++tap) {
                            TR(2, mbar_wait(&full_bar[stage], phase));
                            tc_fence_after();
                            const uint64_t da = DESC_HI | (a_row + (uint32_t)sx * 8u);
                            const uint64_t db = DESC_HI | a_lo;         // weight-tile ring (stage_bytes = B_BYTES)
                            if (!skip_mma) {
#pragma unroll
                                for (int k = 0; k < GM_ROW_BYTES / 32; ++k)
                                    umma<KIND>(td, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC, (kin | tap | k) != 0 ? 1u : 0u);
                            }
                            umma_commit(&empty_bar[stage]);             // weight tile consumed
                            a_lo += a_step;
                            if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                            if (++sx == S) { sx = 0; a_row += row_step; }
                        }
                        umma_commit(&aempty_bar[as4]);                  // halo buffer consumed
                        if (++as4 == g.a_stages) { as4 = 0; aph4 ^= 1u; }
                        if (++kin == g.kcpg) { kin = 0; td += BLOCK_N; }   // next K chunk: next accumulator group
                    }
                } else if constexpr (MODE == 3 && CG == 2) {
                    // leader of the CTA pair: M = 256 (both CTAs' tiles), every tap against the pair's resident half tiles
                    constexpr uint32_t IDESC2 = (1u << 4) | ((uint32_t)(MMA_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
                    const int taps = g.R * g.S, S = g.S;
                    const uint32_t row_step = (uint32_t)g.hw * 8u;
                    TR(2, mbar_wait(&full_bar[stage], phase));
                    tc_fence_after();
                    uint32_t a_row = a_lo, b_lo = b_lo0;
                    int s = 0;
                    for (int tap = 0; tap < taps; ++tap) {
                        const uint64_t da = DESC_HI | (a_row + (uint32_t)s * 8u);
                        const uint64_t db = DESC_HI | b_lo;
#pragma unroll
                        for (int k = 0; k < GM_ROW_BYTES / 32; ++k)
                            umma_f16_pair(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC2, (tap | k) != 0 ? 1u : 0u);
                        b_lo += (uint32_t)(B_BYTES / 2) >> 4;
                        if (++s == S) { s = 0; a_row += row_step; }
                    }
                    umma_commit_pair(&empty_bar[stage]);
                    a_lo += a_step;
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                } else if constexpr (MODE == 3) {
                    const int taps = g.R * g.S, S = g.S, kcb = g.kc_blocks;
                    const uint32_t row_step = (uint32_t)g.hw * 8u;      // one halo row of pixels, in 16-byte units
                    for (int kc = 0; kc < kcb; ++kc) {
                        TR(2, mbar_wait(&full_bar[stage], phase));
                        tc_fence_after();
                        uint32_t a_row = a_lo, b_lo = b_lo0 + (uint32_t)kc * (uint32_t)(B_BYTES >> 4);
                        int s = 0;
                        for (int tap = 0; tap < taps; ++tap) {
                            const uint32_t a_tap = a_row + (uint32_t)s * 8u;
                            uint64_t da = DESC_HI | a_tap;
                            if (g.halo_baseoff) da |= (uint64_t)((a_tap >> 3) & 7u) << 49;
                            const uint64_t db = DESC_HI | b_lo;
                            if (!skip_mma) {
#pragma unroll
                                for (int k = 0; k < GM_ROW_BYTES / 32; ++k)
                                    umma<KIND>(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC, (kc | tap | k) != 0 ? 1u : 0u);
                            }
                            b_lo += (uint32_t)kcb * (uint32_t)(B_BYTES >> 4);
                            if (++s == S) { s = 0; a_row += row_step; }
                        }
                        umma_commit(&empty_bar[stage]);
                        a_lo += a_step;
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                    }
                } else if constexpr (MODE != 2) {
                    uint32_t b_lo = b_lo0;                              // MODE 1: resident tile of this step
                    // accumulator group of a step.  KIND 0: K chunk = kc / kcpg (kc is the fastest index of the step
                    // order); a group's first MMA is the one of tap 0, first block of the chunk.  KIND 1: plane pair
                    // (pa, pw) -> group pa + pw; within a tap the pairs run (0,0) (0,1) (1,0) (1,1), so a group is
                    // first written by the pair with pa == 0 or pw == planes_w - 1 (of tap 0, channel block 0).
                    int kc = 0, kin = 0, tap0 = 1, pa = 0, pw = 0;
                    uint32_t grp = 0;
                    for (int st = 0; st < steps; ++st) {
                        TR(2, mbar_wait(&full_bar[stage], phase));
                        tc_fence_after();
                        const uint64_t da = DESC_HI | a_lo;
                        const uint64_t db = DESC_HI | (MODE == 1 ? b_lo : a_lo + (uint32_t)(GM_A_BYTES >> 4));
                        uint32_t fresh;                                 // 1: this step's first MMA overwrites the accumulator
                        if constexpr (KIND == 1) {
                            grp = (uint32_t)(pa + pw);
                            fresh = (tap0 && kc == 0 && (pa == 0 || pw == g.planes_w - 1)) ? 1u : 0u;
                        } else {
                            fresh = (tap0 && kin == 0) ? 1u : 0u;
                        }
                        const uint32_t td = tmem_d + grp * BLOCK_N;
                        if (!skip_mma) {
#pragma unroll
                            for (int k = 0; k < GM_ROW_BYTES / 32; ++k)   // UMMA_K = 32 bytes (16 fp16 / 32 s8) = +2 in the address field
                                umma<KIND>(td, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC, (k != 0 || !fresh) ? 1u : 0u);
                        }
                        umma_commit(&empty_bar[stage]);                 // frees the smem stage when the MMAs retire
                        a_lo += a_step;
                        b_lo += (uint32_t)(B_BYTES >> 4);
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                        if constexpr (KIND == 1) {
                            if (++kc == g.kc_blocks) {
                                kc = 0;
                                if (++pw == g.planes_w) { pw = 0; if (++pa == g.planes_a) { pa = 0; tap0 = 0; } }
                            }
                        } else {
                            ++kin; ++kc;
                            if (kin == g.kcpg) { kin = 0; ++grp; }
                            if (kc == g.kc_blocks) { kc = 0; kin = 0; grp = 0; tap0 = 0; }
                        }
                    }
                } else {
                    uint32_t started = 0;                               // accumulator groups already written in this tile
                    const int R = g.R, planes = steps / R;
                    const uint32_t row_step = (uint32_t)g.hw * 8u;      // one row of the pixel box, in 16-byte units
                    int st = 0;
                    for (int pl = 0; pl < planes; ++pl) {
                        TR(2, mbar_wait(&full_bar[stage], phase));
                        tc_fence_after();
                        uint32_t a_row = a_lo;
                        for (int r = 0; r < R; ++r, ++st, a_row += row_step) {
                            const uint32_t cur = pw;
                            pw = g.prog_mma[st + 1 < steps ? st + 1 : 0];
                            const uint64_t da = DESC_HI | a_row;
                            const uint32_t g0 = (cur >> 8) & 0xFu;
                            const uint64_t db = DESC_HI | (b_lo0 + ((cur >> 4) & 0xFu) * (uint32_t)(B_BYTES >> 4));
                            const uint32_t first = ((started >> g0) & 1u) ^ 1u;
                            started |= 1u << g0;
                            if (!skip_mma) {
#pragma unroll
                                for (int k = 0; k < GM_BLOCK_K / 16; ++k)
                                    umma_f16(tmem_d + g0 * BLOCK_N, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), IDESC,
                                             (k != 0 || !first) ? 1u : 0u);
                            }
                            if ((cur & 0xFu) == 2u) {
                                const uint32_t g1 = (cur >> 16) & 0xFu;
                                const uint64_t db1 = DESC_HI | (b_lo0 + ((cur >> 12) & 0xFu) * (uint32_t)(B_BYTES >> 4));
                                const uint32_t first1 = ((started >> g1) & 1u) ^ 1u;
                                started |= 1u << g1;
                                if (!skip_mma) {
#pragma unroll
                                    for (int k = 0; k < GM_BLOCK_K / 16; ++k)
                                        umma_f16(tmem_d + g1 * BLOCK_N, da + (uint64_t)(2 * k), db1 + (uint64_t)(2 * k), IDESC,
                                                 (k != 0 || !first1) ? 1u : 0u);
                                }
                            }
                        }
                        umma_commit(&empty_bar[stage]);
                        a_lo += a_step;
                        if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
                    }
                }
                if constexpr (CG == 2) umma_commit_pair(&tfull_bar[acc]);
                else umma_commit(&tfull_bar[acc]);                      // accumulator complete
                if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
            }
#ifdef TQ_CONV_TRACE
            TR_SINCE(3, ti0);
            if (blockIdx.x == 0 || blockIdx.x == 100)
                printf("cta %3d issuer: total %lld, wait acc-empty %lld, wait halo-full %lld, wait stage-full %lld\n", blockIdx.x, trc[3], trc[0], trc[1], trc[2]);
#endif
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ============ epilogue: TMEM -> registers -> swizzled smem -> TMA store ============
        // Four groups of four warps.  Group (a, h) drains column half h of accumulator stage a (every second
        // tile of this CTA), in chunks of 32 columns: 16 epilogue warps keep enough arithmetic in flight to hide
        // the TMEM / shared-memory / barrier latencies, and each group owns its staging tiles, so the only wait
        // on a TMA store is for the group's own previous chunk, placed after the arithmetic.
        // The residual tile is fetched by TMA into the fp32 staging tile (coalesced, asynchronous), updated in
        // place and stored back out by TMA.
        const int grp = (warp - 4) >> 2;                        // 0..3
        const int pair = grp >> 1, half = grp & 1;               // the pair takes every second tile of this CTA
        const int ew = warp & 3;                                // TMEM lanes 32*ew .. 32*ew+31
        const int mrow = ew * 32 + lane;                        // accumulator row = TMEM lane
        // staging row of this accumulator row: dense (hbox x wbox) pixel order; in halo mode the columns
        // mrow % hw >= wbox are junk and write nothing
        // (packed halo: box row y = image y / (H + 1), pixel row y % (H + 1) < H; the staging tile is [image][h][w])
        const int my = mrow / g.hw, mx = mrow % g.hw;
        const int row = g.img_h1 ? (my / g.img_h1) * (g.wbox * g.hbox) + (my % g.img_h1) * g.wbox + mx : my * g.wbox + mx;
        const bool row_live = g.img_h1 ? (mx < g.wbox && (my % g.img_h1) < g.hbox && (my / g.img_h1) < g.nbox) : (mx < g.wbox && row < 128);
        const bool store_thread = (ew == 0 && lane == 0);
        uint8_t *st_f32 = smem + g.epi_off + grp * g.epi_group_bytes;   // [128][32] fp32, 128B swizzle
        uint8_t *st_codes = st_f32 + g.epi_codes_off;                   // [128][32] fp16,  64B swizzle
        const Quant nq = make_quant(g.nq);
        const bool has_res = g.residual != nullptr;
        // With two or three accumulator stages the pairs alternate tiles and group (pair, half) takes half of the columns.
        // With ONE stage (a tile's accumulator groups fill tensor memory) consecutive completions of the same barrier
        // cannot be told apart by two waiters that skip every second one, so all four groups take EVERY tile, a quarter
        // of the columns each (which also drains the accumulator four-wide before the next tile's MMAs may start).
        const bool single = ACC_STAGES == 1;
        const int CHUNKS = single ? BLOCK_N / 128 : BLOCK_N / 64;   // 32-column chunks per group and tile
        const uint32_t res_bytes = (uint32_t)(g.wbox * g.hbox * g.nbox) * 128u;
        uint32_t res_phase = 0;
        int it = 0;
        // "this thread's share of accumulator stage a is in registers": on the MMA issuer's barrier (the pair leader's)
        const uint32_t tempty0 = CG == 2 ? mapa_u32(smem_u32(tempty_bar), 0) : 0u;
        auto release_acc = [&](int a) {
            if (CG == 2 && cta_rank != 0) mbar_arrive_cluster(tempty0 + 8u * (uint32_t)a);
            else mbar_arrive(&tempty_bar[a]);
        };
        TR_DECL(8);
        TR_T0(te0);
        // Tile coordinates and the accumulator stage advance by carries, not by the seven run-time integer divisions per
        // tile the plain decode costs every epilogue thread (~150 of the ~950 instructions per 32-column chunk).
        const int n_tiles = g.n_tiles, tiles_w = g.tiles_w, tiles_h = g.tiles_h;
        int n_tile = tile_first % n_tiles;
        int tw, th, tn;
        {
            const int m0 = m_tile_of(tile_first);
            tw = m0 % tiles_w; th = (m0 / tiles_w) % tiles_h; tn = m0 / (tiles_w * tiles_h);
        }
        const int step_n = tile_step % n_tiles, step_m = (tile_step / n_tiles) * CG;       // M tiles per loop step (before the carry)
        const int s_w = step_m % tiles_w, s_h = (step_m / tiles_w) % tiles_h, s_n = step_m / (tiles_w * tiles_h);
        const int u_w = CG % tiles_w, u_h = (CG / tiles_w) % tiles_h, u_n = CG / (tiles_w * tiles_h);   // the carry out of n_tile
        auto add_m = [&](int dw, int dh, int dn) {
            tw += dw;
            int c = tw >= tiles_w ? 1 : 0;
            tw -= c ? tiles_w : 0;
            th += dh + c;
            c = th >= tiles_h ? 1 : 0;
            th -= c ? tiles_h : 0;
            tn += dn + c;
        };
        int acc = 0;                                                  // accumulator stage of this tile and its use parity
        uint32_t acc_phase = 0;
        auto next_tile = [&]() {
            n_tile += step_n;
            const bool carry = n_tile >= n_tiles;
            n_tile -= carry ? n_tiles : 0;
            add_m(s_w, s_h, s_n);
            if (carry) add_m(u_w, u_h, u_n);
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
        };
        for (int tile = tile_first; tile < total_tiles; tile += tile_step, ++it, next_tile()) {
            if (!single && (it & 1) != pair) continue;
            const int w0 = tw * g.wbox, h0 = th * g.hbox, n0 = tn * g.nbox;

            if (g.dbg_skip_epilogue) {
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                tc_fence_before();
                release_acc(acc);
                continue;
            }
#pragma unroll 1
            for (int cc = 0; cc < CHUNKS; ++cc) {
                const int col0 = (single ? grp * (BLOCK_N / 4) : half * (BLOCK_N / 2)) + cc * 32;   // column of the tile
                const int c0 = n_tile * BLOCK_N + col0;                     // output channel
                const bool chunk_live = c0 < g.Cout;
                // (a) residual tile -> fp32 staging (needs the staging tile free: the previous store has read it)
                if (has_res && store_thread && chunk_live) {
                    bulk_wait_read0();
                    mbar_expect_tx(&res_bar[grp], res_bytes);
                    tma_load_4d(&tmR, &res_bar[grp], st_f32, c0, w0, h0, n0);
                }
                if (cc == 0) {
                    TR(0, mbar_wait(&tfull_bar[acc], acc_phase));
                    tc_fence_after();
                }
                if (!chunk_live) {                               // channels beyond Cout (uniform over the group)
                    if (cc == CHUNKS - 1) {
                        tc_fence_before();
                        release_acc(acc);
                    }
                    continue;
                }
                float t[32];
                TR_T0(tl0);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    uint32_t v[16];
                    const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * acc_cols + col0 + hh * 16);
                    tmem_ld_32x32b_x16(tcol, v);
                    // Accumulator groups.  Exact integer accumulators (K chunks of a kind::f16 conv: fp32 values holding
                    // integers below 2^24; kind::i8 plane pairs: s32) are combined in int32 -- chunks added, plane pairs by
                    // Horner with the plane shift ((hi*hi << 4) + hi*lo + lo*hi) << 4) + lo*lo -- and converted to fp32
                    // ONCE (RN).  The hi/lo planes of the fp32 stem conv are summed in fp32 RN.  All in place in v[].
                    const bool as_int = KIND == 1 || g.acc_int != 0;
                    if (g.n_groups > 1) {
                        if (KIND == 0 && as_int) {
#pragma unroll
                            for (int e = 0; e < 16; ++e) v[e] = (uint32_t)__float2int_rn(__uint_as_float(v[e]));
                        }
                        for (int gi = 1; gi < g.n_groups; ++gi) {
                            uint32_t u[16];
                            tmem_ld_32x32b_x16(tcol + (uint32_t)(gi * BLOCK_N), u);
#pragma unroll
                            for (int e = 0; e < 16; ++e) {
                                if (KIND == 1) v[e] = (v[e] << GM_I8_SHIFT) + u[e];
                                else if (as_int) v[e] += (uint32_t)__float2int_rn(__uint_as_float(u[e]));
                                else v[e] = __float_as_uint(__fadd_rn(__uint_as_float(v[e]), __uint_as_float(u[e])));
                            }
                        }
                    }
                    if (KIND == 1 || (as_int && g.n_groups > 1)) {
#pragma unroll
                        for (int e = 0; e < 16; ++e) v[e] = __float_as_uint(__int2float_rn((int)v[e]));
                    }
#pragma unroll
                    for (int e = 0; e < 16; ++e) t[hh * 16 + e] = __fmul_rn(__uint_as_float(v[e]), g.scale);
                }
                if (cc == CHUNKS - 1) {                          // this group's share of the accumulator is in registers
                    tc_fence_before();
                    release_acc(acc);
                }
                TR_SINCE(1, tl0);
                TR_T0(tq0);
                if constexpr (MODE == 2) {
                    if (g.pool == 2) {
                        // ---- horizontal half of the 3x3 / stride 2 / pad 1 max-pool (two-pass stem) ----
                        // The tile is 4 conv rows x 32 conv columns (31 used, consecutive tiles overlapping by one
                        // column): warp ew holds conv row ew, lane x its column x.  Output q (lane 2 ql) is the max of
                        // the RAW conv sums of lanes 2 ql, 2 ql + 1, 2 ql + 2 (conv columns 2q-1, 2q, 2q+1; a column outside
                        // the conv map is left out), taken with two shuffles per value: no staging of the conv values, so
                        // the epilogue adds almost nothing to the shared-memory traffic of the MMAs.  The weights carry
                        // sign(bn_a) (see the pooled mode below), so tq_bn_relu_maxpool_encode_rowmax takes the vertical
                        // max and applies the affine after it.
                        const int Q = g.pool_q, ql = lane >> 1, q = tw * Q + ql;
                        const bool left = q > 0, right = 2 * q + 1 < g.Wo;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float c = __shfl_down_sync(0xFFFFFFFFu, t[j], 1);
                            const float r = __shfl_down_sync(0xFFFFFFFFu, t[j], 2);
                            const float m = right ? fmaxf(c, r) : c;
                            t[j] = left ? fmaxf(t[j], m) : m;
                        }
                        TR_SINCE(2, tq0);
                        TR_T0(tq2);
                        // the row-max staging tile ([4 * Q][32] fp32) is free once this group's previous TMA store has read it
                        if (store_thread) bulk_wait_read0();
                        epi_bar_sync(1 + grp);
                        TR_SINCE(4, tq2);
                        TR_T0(tq3);
                        if (!(lane & 1) && ql < Q) {
                            const int o = ew * Q + ql;
                            uint8_t *orow = st_f32 + o * 128;
                            const uint32_t sw = (uint32_t)(o & 7);
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4 *>(orow + (((uint32_t)(j >> 2) ^ sw) << 4)) =
                                    make_float4(t[j], t[j + 1], t[j + 2], t[j + 3]);
                        }
                        TR_SINCE(5, tq3);
                        fence_proxy_async();
                        epi_bar_sync(1 + grp);
                        if (store_thread) {
                            tma_store_4d(&tmC, st_f32, c0, tw * Q, th * g.hbox, n0);
                            bulk_commit();
                        }
                        TR_SINCE(6, tq0);
                        continue;
                    }
                    if (g.pool) {
                        // ---- fused BatchNorm + ReLU + 3x3 / stride 2 / pad 1 max-pool + next-layer encode (stem) ----
                        // The tile is the (2P+1) x (2Q+1) box of conv pixels under P x Q pooled pixels.  The RAW conv
                        // sums are staged; the pooling threads take the window maximum out of shared memory (window
                        // positions outside the conv output are replaced by the centre, which always exists) and only
                        // then apply fma(., bn_a, bn_b), ReLU and the encode -- once per pooled value instead of once
                        // per conv value.  max commutes with the affine because bn_a >= 0 here: the host folds
                        // sign(bn_a) into the weights of the channel (exact: products and truncated sums negate
                        // exactly), so max_i fma(x_i, a, b) = fma(max_i(sign(a) x_i), |a|, b).
                        // (the conv staging tile is never read by TMA; the previous tile's pooling reads of it
                        // finished before that tile's last group barrier)
                        {
                            uint8_t *frow = st_f32 + mrow * 128;
                            const uint32_t sw = (uint32_t)(mrow & 7);
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4 *>(frow + (((uint32_t)(j >> 2) ^ sw) << 4)) =
                                    make_float4(t[j], t[j + 1], t[j + 2], t[j + 3]);
                        }
                        epi_bar_sync(1 + grp);
                        TR_SINCE(2, tq0);
                        TR_T0(tq1);
                        uint8_t *st_pool = st_codes, *st_pcodes = st_codes + 4096;   // [P*Q][32] fp32 / fp16 tiles
                        const int pp = mrow >> 2, cb = mrow & 3;                     // pooled pixel, 8-channel block
                        float pv[8];
                        const bool pool_thread = pp < g.pool_p * g.pool_q;
                        if (pool_thread) {
                            const int pl = pp / g.pool_q, ql = pp % g.pool_q;
                            // conv pixel of window position (dy, dx): (2 (p0 + pl) - 1 + dy, 2 (q0 + ql) - 1 + dx)
                            const int oh0 = 2 * (th * g.pool_p + pl) - 1, ow0 = 2 * (tw * g.pool_q + ql) - 1;
                            int rowoff[3], coloff[3];
#pragma unroll
                            for (int d = 0; d < 3; ++d) {
                                rowoff[d] = (2 * pl + (((unsigned)(oh0 + d) < (unsigned)g.Ho) ? d : 1)) * g.hw;
                                coloff[d] = 2 * ql + (((unsigned)(ow0 + d) < (unsigned)g.Wo) ? d : 1);
                            }
                            float4 m0 = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY), m1 = m0;
#pragma unroll
                            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                                for (int dx = 0; dx < 3; ++dx) {
                                    const int mm = rowoff[dy] + coloff[dx];
                                    const uint32_t sw = (uint32_t)(mm & 7);
                                    const float4 a = *reinterpret_cast<const float4 *>(st_f32 + mm * 128 + (((uint32_t)(2 * cb) ^ sw) << 4));
                                    const float4 b = *reinterpret_cast<const float4 *>(st_f32 + mm * 128 + (((uint32_t)(2 * cb + 1) ^ sw) << 4));
                                    m0.x = fmaxf(m0.x, a.x); m0.y = fmaxf(m0.y, a.y); m0.z = fmaxf(m0.z, a.z); m0.w = fmaxf(m0.w, a.w);
                                    m1.x = fmaxf(m1.x, b.x); m1.y = fmaxf(m1.y, b.y); m1.z = fmaxf(m1.z, b.z); m1.w = fmaxf(m1.w, b.w);
                                }
                            pv[0] = m0.x; pv[1] = m0.y; pv[2] = m0.z; pv[3] = m0.w; pv[4] = m1.x; pv[5] = m1.y; pv[6] = m1.z; pv[7] = m1.w;
                            const int c8 = c0 + 8 * cb;
                            if (c8 < g.Cout) {                                        // Cout % 8 == 0
                                const float4 a0 = __ldg(reinterpret_cast<const float4 *>(g.bn_a + c8));
                                const float4 a1 = __ldg(reinterpret_cast<const float4 *>(g.bn_a + c8 + 4));
                                const float4 b0 = __ldg(reinterpret_cast<const float4 *>(g.bn_b + c8));
                                const float4 b1 = __ldg(reinterpret_cast<const float4 *>(g.bn_b + c8 + 4));
                                const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                                const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    pv[e] = __fmaf_rn(pv[e], av[e], bv[e]);
                                    if (RELU) pv[e] = fmaxf(pv[e], 0.0f);
                                }
                            }
                        }
                        // the pooled staging tiles are free once this group's previous TMA store has read them
                        TR_SINCE(3, tq1);
                        TR_T0(tq2);
                        if (store_thread) bulk_wait_read0();
                        epi_bar_sync(1 + grp);
                        TR_SINCE(4, tq2);
                        TR_T0(tq3);
                        if (pool_thread) {
                            const uint32_t psw = (uint32_t)(pp & 7);
                            *reinterpret_cast<float4 *>(st_pool + pp * 128 + (((uint32_t)(2 * cb) ^ psw) << 4)) = make_float4(pv[0], pv[1], pv[2], pv[3]);
                            *reinterpret_cast<float4 *>(st_pool + pp * 128 + (((uint32_t)(2 * cb + 1) ^ psw) << 4)) = make_float4(pv[4], pv[5], pv[6], pv[7]);
                            if (g.nq.write_codes) {
                                uint32_t hc[8];
#pragma unroll
                                for (int e = 0; e < 8; ++e) {
                                    uint32_t idx;
                                    if (RELU) idx = g.nq.fastdiv ? quantize_f32_nonneg<true>(pv[e], nq) : quantize_f32_nonneg<false>(pv[e], nq);
                                    else idx = (g.nq.fastdiv ? quantize_f32<true>(pv[e], nq) : quantize_f32<false>(pv[e], nq)) |
                                               ((__float_as_uint(pv[e]) >> 31) << g.nq.bits);
                                    hc[e] = __half_as_ushort(lut[idx]);
                                }
                                *reinterpret_cast<uint4 *>(st_pcodes + pp * 64 + (((uint32_t)cb ^ (uint32_t)((pp >> 1) & 3)) << 4)) =
                                    make_uint4(hc[0] | (hc[1] << 16), hc[2] | (hc[3] << 16), hc[4] | (hc[5] << 16), hc[6] | (hc[7] << 16));
                            }
                        }
                        TR_SINCE(5, tq3);
                        fence_proxy_async();
                        epi_bar_sync(1 + grp);
                        if (store_thread) {
                            tma_store_4d(&tmC, st_pool, c0, tw * g.pool_q, th * g.pool_p, n0);
                            if (g.nq.write_codes) tma_store_4d(&tmD, st_pcodes, c0, tw * g.pool_q, th * g.pool_p, n0);
                            bulk_commit();
                        }
                        TR_SINCE(6, tq0);
                        continue;
                    }
                }
                TR(2, if (c0 + 32 <= g.Cout) epi_affine<true>(t, g, c0); else epi_affine<false>(t, g, c0));
                // (b) staging: with a residual it already holds this chunk's residual tile; otherwise the previous
                //     store of this group must have finished reading it before it is overwritten
                TR_T0(tw0);
                if (has_res) {
                    mbar_wait(&res_bar[grp], res_phase);
                } else {
                    if (store_thread) bulk_wait_read0();
                    epi_bar_sync(1 + grp);
                }
                TR_SINCE(3, tw0);
                TR(4, if (row_live) epi_stage<RELU>(t, g, st_f32, st_codes, row, has_res, lut, nq));
                if (has_res) res_phase ^= 1u;
                // (c) staging complete: hand it to the async proxy and store
                TR_T0(ts0);
                fence_proxy_async();
                epi_bar_sync(1 + grp);
                if (store_thread) {
                    if (g.write_f32) tma_store_4d(&tmC, st_f32, c0, w0, h0, n0);
                    if (g.nq.write_codes) tma_store_4d(&tmD, st_codes, c0, w0, h0, n0);
                    bulk_commit();
                }
                TR_SINCE(5, ts0);
            }
        }
#ifdef TQ_CONV_TRACE
        TR_SINCE(7, te0);
        if ((blockIdx.x == 0 || blockIdx.x == 100) && store_thread && grp < 2)
            printf("cta %3d epilogue group %d: total %lld, wait acc-full %lld, tmem+combine %lld, affine %lld, wait staging %lld, stage %lld, "
                   "sync+store %lld, pooled tail %lld  (pooled stem: the four middle slots are raw staging + sync, window max + affine, store wait + sync, "
                   "pooled tile + encode)\n", blockIdx.x, grp, trc[7], trc[0], trc[1], trc[2], trc[3], trc[4], trc[5], trc[6]);
#endif
        if (store_thread) bulk_wait0();
    }

    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all();              // neither CTA leaves while the pair's MMAs may touch its memories
    else __syncthreads();
    if (warp == 2) {
        if constexpr (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled()          // shared with tq_dw.cu
{
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    });
    return fn;
}

// choose the pixel box (wbox, hbox, nbox), product <= 128, that needs the fewest M tiles
static void pick_box(ConvGeom &g)
{
    long best = -1;
    static const int force_w = getenv("TQ_CONV_WBOX") ? atoi(getenv("TQ_CONV_WBOX")) : 0;
    static const int force_h = getenv("TQ_CONV_HBOX") ? atoi(getenv("TQ_CONV_HBOX")) : 0;
    for (int wb = 1; wb <= g.Wo && wb <= 128; ++wb) {
        if (wb * g.stride > 256) break;
        if (force_w && wb != force_w && force_w <= g.Wo) continue;
        for (int hb = 1; hb <= g.Ho && wb * hb <= 128; ++hb) {
            if (hb * g.stride > 256) break;
            if (force_h && hb != force_h && force_h <= g.Ho && force_w * force_h <= 128) continue;
            int nb = 1;
            if (wb == g.Wo && hb == g.Ho) nb = 128 / (wb * hb) < g.N ? 128 / (wb * hb) : g.N;
            if (nb < 1) nb = 1;
            const long tiles = (long)((g.Wo + wb - 1) / wb) * ((g.Ho + hb - 1) / hb) * ((g.N + nb - 1) / nb);
            if (best < 0 || tiles < best || (tiles == best && wb > g.wbox)) {
                best = tiles;
                g.wbox = wb; g.hbox = hb; g.nbox = nb;
            }
        }
    }
    g.tiles_w = (g.Wo + g.wbox - 1) / g.wbox;
    g.tiles_h = (g.Ho + g.hbox - 1) / g.hbox;
    g.tiles_n = (g.N + g.nbox - 1) / g.nbox;
    g.m_tiles = g.tiles_w * g.tiles_h * g.tiles_n;
    g.a_tx_bytes = g.wbox * g.hbox * g.nbox * GM_ROW_BYTES;
}

// halo mode: the pixel box (wbox x hbox, one image) whose rows, laid out (wbox + S - 1) pixels apart, fit
// 128 accumulator rows; fewest tiles first, then the smallest halo
static bool pick_box_halo(ConvGeom &g)
{
    long best = -1, best_halo = 0;
    int bw = 0, bh = 0;
    for (int wb = 1; wb <= g.Wo; ++wb) {
        const int hw = wb + g.S - 1;
        if (hw > 128 || hw > 256) break;
        int hb = 128 / hw;
        if (hb > g.Ho) hb = g.Ho;
        if (hb < 1 || hb + g.R - 1 > 256) continue;
        const long tiles = (long)((g.Wo + wb - 1) / wb) * ((g.Ho + hb - 1) / hb) * g.N;
        const long halo = (long)hw * (hb + g.R - 1);
        if (best < 0 || tiles < best || (tiles == best && halo < best_halo)) { best = tiles; best_halo = halo; bw = wb; bh = hb; }
    }
    if (best < 0) return false;
    g.wbox = bw; g.hbox = bh; g.nbox = 1;
    g.hw = bw + g.S - 1;
    g.tiles_w = (g.Wo + bw - 1) / bw;
    g.tiles_h = (g.Ho + bh - 1) / bh;
    g.tiles_n = g.N;
    g.m_tiles = g.tiles_w * g.tiles_h * g.tiles_n;
    g.a_tx_bytes = g.hw * (bh + g.R - 1) * GM_ROW_BYTES;
    return true;
}

// carve shared memory: [stationary B][stage ring][2 x epilogue staging][LUT][barriers]
static int plan_smem(ConvGeom &g, int block_n)
{
    const int b_bytes = (g.b_rows > 0 ? g.b_rows : block_n) * GM_ROW_BYTES;   // (MODE 2 stacks hi | lo: 2 * block_n rows per tile)
    const bool prog = g.prog_steps > 0;
    g.stage_bytes = GM_A_BYTES + (prog ? 0 : b_bytes);
    if (g.halo) g.stage_bytes = (g.a_tx_bytes + 1023) & ~1023;
    g.bstat_off = 0;
    g.ring_off = prog ? g.nb_tiles * (g.pair ? b_bytes / 2 : b_bytes) : 0;     // (a pair CTA keeps half of every resident tile)
    if (g.halo && !prog) {                          // MODE 4: [halo ring][weight-tile ring]
        g.a_stage_bytes = (g.a_tx_bytes + 1023) & ~1023;
        if (g.img_h1) g.a_stage_bytes = (g.a_tx_bytes + ((g.R - 1) * g.hw + g.S) * GM_ROW_BYTES + 1023) & ~1023;   // + the zero tail
        static const int a_stages_env = getenv("TQ_CONV_ASTAGES") ? atoi(getenv("TQ_CONV_ASTAGES")) : 0;
        // single CTAs, measured: 2 halo buffers + a deeper weight ring win.  CTA pairs: 3, so that the next box is requested a
        // whole step ahead (see the producer)
        g.a_stages = a_stages_env >= 2 && a_stages_env <= 4 ? a_stages_env : (g.pair ? 3 : 2);
        g.stage_bytes = b_bytes;
        g.ring_off = g.a_stages * g.a_stage_bytes;
    }
    // epilogue staging per group: fp32 tile only if an fp32 tile is written or a residual is read, code tile only
    // if codes are written -- what is not needed goes to the stage ring
    g.epi_codes_off = (g.write_f32 || g.residual) ? GM_EPI_F32_BYTES : 0;
    g.epi_group_bytes = g.epi_codes_off + ((g.nq.write_codes || g.pool == 1) ? GM_EPI_CODE_BYTES : 0);
    const int epi_bytes = GM_EPI_GROUPS * g.epi_group_bytes;
    const int fixed = g.ring_off + epi_bytes + (int)code_table_bytes(GM_LUT_MAX_BITS) + 1024 /* barriers */ + 1024 /* align */;
    int stages = (GM_SMEM_BUDGET - fixed) / g.stage_bytes;
    if (stages > GM_MAX_STAGES) stages = GM_MAX_STAGES;
    static const int cap = getenv("TQ_CONV_STAGES") ? atoi(getenv("TQ_CONV_STAGES")) : GM_MAX_STAGES;
    if (stages > cap && cap >= 2) stages = cap;
    if (stages < 2) return fail(TQ_ERR_UNSUPPORTED, "shared memory budget: %d resident weight tiles do not fit", g.nb_tiles);
    g.stages = stages;
    g.epi_off = g.ring_off + stages * g.stage_bytes;
    g.lut_off = g.epi_off + epi_bytes;
    g.bar_off = g.lut_off + (int)code_table_bytes(GM_LUT_MAX_BITS);
    g.smem_total = g.bar_off + 1024 + 1024;
    return TQ_OK;
}

template <int BLOCK_N, int MODE, int KIND = 0, int CG = 1>
static int launch_conv_mode(const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmC,
                            const CUtensorMap &tmD, const CUtensorMap &tmR, ConvGeom &g, cudaStream_t s)
{
    static const bool skip_epi = getenv("TQ_CONV_SKIP_EPI") != nullptr;
    g.dbg_skip_epilogue = skip_epi ? 1 : 0;
    static const bool skip_mma = getenv("TQ_CONV_SKIP_MMA") != nullptr;
    static const int skip_tma = getenv("TQ_CONV_SKIP_TMA") ? atoi(getenv("TQ_CONV_SKIP_TMA")) : 0;
    g.dbg_skip_mma = skip_mma ? 1 : 0;
    g.dbg_skip_tma = skip_tma;
    auto kern = g.relu ? conv_igemm_kernel<BLOCK_N, MODE, true, KIND, CG> : conv_igemm_kernel<BLOCK_N, MODE, false, KIND, CG>;
    static bool attr_set[2][64] = {{false}};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_set[g.relu ? 1 : 0][dev]) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GM_SMEM_BUDGET) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(conv_igemm_kernel)");
        attr_set[g.relu ? 1 : 0][dev] = true;
    }
    if constexpr (CG == 2) {
        // one cluster of two CTAs per TPC; as many pairs as fit the device at once (at most one per two SMs)
        const int supers = ((g.m_tiles + 1) / 2) * g.n_tiles;
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(GM_THREADS); cfg.dynamicSmemBytes = (size_t)g.smem_total; cfg.stream = s;
        cfg.attrs = attr; cfg.numAttrs = 1;
        static int max_pairs[2][64] = {{0}};
        int &mp = max_pairs[g.relu ? 1 : 0][dev >= 0 && dev < 64 ? dev : 0];
        if (mp == 0) {
            cfg.gridDim = dim3((unsigned)(num_sms() & ~1));
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) { (void)cudaGetLastError(); n = num_sms() / 2; }
            mp = n < num_sms() / 2 ? n : num_sms() / 2;
        }
        const int pairs = supers < mp ? supers : mp;
        cfg.gridDim = dim3((unsigned)(2 * pairs));
        cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmC, tmD, tmR, g);
        count_launch();
        if (e != cudaSuccess) return fail(TQ_ERR_CUDA, "conv_igemm_kernel (CTA pairs): %s", cudaGetErrorString(e));
        return check_launch("conv_igemm_kernel");
    } else {
        const int total = g.m_tiles * g.n_tiles;
        const int grid = total < num_sms() ? total : num_sms();
        kern<<<grid, GM_THREADS, g.smem_total, s>>>(tmA, tmB, tmC, tmD, tmR, g);
        count_launch();
        return check_launch("conv_igemm_kernel");
    }
}

// which kernel instance runs a planned conv
enum ConvVariant { CV_NONE = 0, CV_64_M0, CV_64_M1, CV_64_M2, CV_64_M3, CV_64_M3_PAIR, CV_128_M0, CV_128_M4, CV_128_M4_PAIR, CV_256_M0, CV_I8_64, CV_I8_128 };

// general_prog: the step table (prog_mma) is in use; otherwise resident weights are tile = tap
static int pick_variant(ConvGeom &g, int block_n, int kind, bool general_prog, ConvVariant &v)
{
    if (g.n_groups < 1) g.n_groups = 1;
    if (g.n_groups * block_n > 512) return fail(TQ_ERR_UNSUPPORTED, "accumulator groups exceed tensor memory");
    if (g.kcpg < 1) g.kcpg = g.kc_blocks;
    int rc = plan_smem(g, block_n);
    if (rc != TQ_OK) return rc;
    if (kind == 1) {
        if (g.prog_steps != 0 || g.halo || block_n == 256) return fail(TQ_ERR_UNSUPPORTED, "s8-plane engine: streaming mode only");
        v = block_n == 64 ? CV_I8_64 : CV_I8_128;
        return TQ_OK;
    }
    if (g.prog_steps == 0 && g.halo) {
        if (block_n != 128) return fail(TQ_ERR_UNSUPPORTED, "streamed-weight halo mode is built for BLOCK_N = 128 only");
        v = g.pair ? CV_128_M4_PAIR : CV_128_M4;
        return TQ_OK;
    }
    if (g.prog_steps == 0) { v = block_n == 64 ? CV_64_M0 : (block_n == 128 ? CV_128_M0 : CV_256_M0); return TQ_OK; }
    if (block_n != 64) return fail(TQ_ERR_UNSUPPORTED, "resident-weight mode is built for BLOCK_N = 64 only");
    v = general_prog ? CV_64_M2 : (g.halo ? (g.pair ? CV_64_M3_PAIR : CV_64_M3) : CV_64_M1);
    return TQ_OK;
}

static int launch_variant(ConvVariant v, const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmC,
                          const CUtensorMap &tmD, const CUtensorMap &tmR, ConvGeom &g, cudaStream_t s)
{
    switch (v) {
    case CV_64_M0: return launch_conv_mode<64, 0>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_64_M1: return launch_conv_mode<64, 1>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_64_M2: return launch_conv_mode<64, 2>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_64_M3: return launch_conv_mode<64, 3>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_64_M3_PAIR: return launch_conv_mode<64, 3, 0, 2>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_128_M0: return launch_conv_mode<128, 0>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_128_M4: return launch_conv_mode<128, 4>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_128_M4_PAIR: return launch_conv_mode<128, 4, 0, 2>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_256_M0: return launch_conv_mode<256, 0>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_I8_64: return launch_conv_mode<64, 0, 1>(tmA, tmB, tmC, tmD, tmR, g, s);
    case CV_I8_128: return launch_conv_mode<128, 0, 1>(tmA, tmB, tmC, tmD, tmR, g, s);
    default: return fail(TQ_ERR_UNSUPPORTED, "no kernel variant");
    }
}

// ---- plan cache -------------------------------------------------------------------------------
// Planning a conv (tile search, shared-memory carve-up, five cuTensorMapEncodeTiled calls) costs tens of
// microseconds on the host; a model calls the same (pointers, shape, epilogue) conv every forward, so finished
// plans are kept per argument tuple.  Tensor maps hold device ADDRESSES, not contents: a plan stays valid for
// as long as the caller reuses the same buffers, and any other argument tuple simply plans again.
struct ConvArgs {
    const void *act, *wgt, *out_f32, *out_codes, *bias, *bn_a, *bn_b, *residual;
    int kind, N, H, W, C, Cout, R, S, stride, pad, relu, acc_groups, planes_a, planes_w, device;
    float scale;
    NextQuant nq;
};
struct ConvPlan {
    ConvArgs key;
    ConvGeom g;
    CUtensorMap tmA, tmB, tmC, tmD, tmR;
    ConvVariant variant;
};
static std::mutex g_plan_mu;
static std::vector<ConvPlan> g_plans[64];        // small open hash: bucket = hash % 64
static size_t g_plan_count = 0;

static uint64_t hash_args(const ConvArgs &a)
{
    const unsigned char *p = reinterpret_cast<const unsigned char *>(&a);
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < sizeof(ConvArgs); ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

static int encode_map(EncodeTiledFn enc, CUtensorMap *tm, CUtensorMapDataType dt, int esize, const void *base,
                      int rank, const cuuint64_t *dims, const cuuint32_t *box, const cuuint32_t *estr, const char *what,
                      CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B)
{
    cuuint64_t strides[4];
    cuuint64_t acc = (cuuint64_t)esize;
    for (int i = 0; i < rank - 1; ++i) { acc *= dims[i]; strides[i] = acc; }
    CUresult r = enc(tm, dt, (cuuint32_t)rank, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled(%s) failed: %d", what, (int)r);
    return TQ_OK;
}

// Plans one conv: tile shape, operand-movement mode, shared-memory carve-up, tensor maps.  kind 0: act / wgt are fp16
// codes ([N,H,W,C], [R*S][Cout][C]) and acc_groups K chunks accumulate apart.  kind 1: act / wgt are s8 planes
// ([PA][N][H][W][C], [PW][R*S][Cout][C]).
static int plan_conv(const ConvArgs &a, ConvPlan &pl)
{
    const int N = a.N, H = a.H, W = a.W, C = a.C, Cout = a.Cout, R = a.R, S = a.S, stride = a.stride, pad = a.pad;
    const int kind = a.kind;
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");

    ConvGeom g{};
    g.N = N; g.H = H; g.W = W; g.C = C; g.Cout = Cout; g.R = R; g.S = S; g.stride = stride; g.pad = pad;
    g.Ho = (H + 2 * pad - R) / stride + 1;
    g.Wo = (W + 2 * pad - S) / stride + 1;
    if (g.Ho < 1 || g.Wo < 1) return fail(TQ_ERR_INVALID, "empty output");
    g.scale = a.scale;
    g.kblk = kind == 1 ? GM_ROW_BYTES : GM_BLOCK_K;
    g.kc_blocks = (C + g.kblk - 1) / g.kblk;
    g.planes_a = kind == 1 ? a.planes_a : 1;
    g.planes_w = kind == 1 ? a.planes_w : 1;
    pick_box(g);
    g.hw = g.wbox;
    // N tile.  At N = 128 the operand reads from shared memory (A 4 KB + B 4 KB per 64-cycle MMA) plus the TMA writes
    // of the next stage ask for twice the 128 B/cycle of shared-memory bandwidth (DESIGN.md section 6); N = 256 halves
    // the A share, but on the ResNet shapes it loses more than it gains: 48 KB stages leave 2-3 ring stages beside the
    // epilogue staging tiles and 512 tiles are 3.46 waves of 148 CTAs (measured: 14x14 / 7x7 layers 5-13 % slower,
    // only the residual-without-codes layer 8 % faster).  Opt-in: TQ_CONV_N256=1.
    static const int n256 = getenv("TQ_CONV_N256") ? atoi(getenv("TQ_CONV_N256")) : 0;
    const int block_n = Cout <= 64 ? 64 : ((n256 && kind == 0 && a.acc_groups == 1 && Cout % 256 == 0) ? 256 : 128);
    g.n_tiles = (Cout + block_n - 1) / block_n;
    g.bias = (const float *)a.bias; g.bn_a = (const float *)a.bn_a; g.bn_b = (const float *)a.bn_b;
    g.residual = (const float *)a.residual;
    g.relu = a.relu ? 1 : 0;
    g.relu6 = a.relu == 2 ? 1 : 0;
    g.write_f32 = a.out_f32 ? 1 : 0;
    g.nq = a.nq;
    // accumulator groups
    if (kind == 1) {
        g.n_groups = g.planes_a + g.planes_w - 1;
        g.kcpg = g.kc_blocks;
        g.acc_int = 1;
    } else {
        if (a.acc_groups < 1 || g.kc_blocks % a.acc_groups != 0)
            return fail(TQ_ERR_INVALID, "acc_groups = %d must divide the %d 64-channel blocks of C", a.acc_groups, g.kc_blocks);
        g.n_groups = a.acc_groups;
        g.kcpg = g.kc_blocks / a.acc_groups;
        g.acc_int = a.acc_groups > 1 ? 1 : 0;
    }
    // one accumulator stage (more than 256 columns per tile) is drained by four epilogue groups of 32 columns: N = 128 only
    if (g.n_groups * block_n > 512 || (2 * g.n_groups * block_n > 512 && block_n != 128))
        return fail(TQ_ERR_UNSUPPORTED, "%d accumulator groups of %d columns exceed tensor memory", g.n_groups, block_n);
    // small layers: every weight tile stays resident in shared memory and the K loop is a table of A loads
    const int taps = R * S * g.kc_blocks;
    static const bool no_prog = getenv("TQ_CONV_NO_PROG") != nullptr;
    if (kind == 0 && g.n_groups == 1 && !no_prog && Cout <= 64 && taps <= 12) {
        g.prog_steps = taps;
        g.nb_tiles = taps;
        // stride-1 filters wider than 1x1 on maps big enough to fill the tile: one halo load per tile
        static const bool no_halo = getenv("TQ_CONV_NO_HALO") != nullptr;
        // The UMMA 128-byte swizzle is a function of the absolute shared-memory address (as TMA's is for a
        // 1024-byte aligned box), so a descriptor may start at any 128-byte row of a swizzled buffer with the
        // base-offset field left 0 (measured: with base offset = (addr >> 7) & 7 the results are wrong).
        static const bool halo_baseoff = getenv("TQ_CONV_HALO_BASEOFF") ? atoi(getenv("TQ_CONV_HALO_BASEOFF")) != 0 : false;
        if (!no_halo && g.kc_blocks == 1 && stride == 1 && R * S > 1) {
            ConvGeom h = g;
            // (halo tiles are a little less dense -- up to TQ_CONV_HALO_SLACK percent more tiles are accepted: one box per
            // tile instead of R*S is worth more than that.  Measured on VGG-16's 224x224 64 -> 64 layer, 14 % more tiles:
            // 0.740 -> 0.621 ms)
            static const int slack = getenv("TQ_CONV_HALO_SLACK") ? atoi(getenv("TQ_CONV_HALO_SLACK")) : 16;
            if (pick_box_halo(h) && (long)h.m_tiles * 100 <= (long)g.m_tiles * (100 + slack)) {
                g = h;
                g.halo = 1;
                g.halo_baseoff = halo_baseoff ? 1 : 0;
                // CTA pairs (opt-in, TQ_CONV_PAIR3=1): N = 64 MMAs are bound by shared-memory operand reads (A 4 KB + B 2 KB per
                // 32-cycle MMA); with half of every weight tile per CTA it is 4 + 1 KB.  Measured: the 56x56 64 -> 64 layer with
                // an fp32-only epilogue 0.0756 -> 0.0569 ms (1040 TFLOP/s), but NO change inside ResNet-18 / VGG-16, where
                // these layers also encode their output and the epilogue's instruction issue (30 per value) is what bounds
                // them -- so single CTAs stay the default.
                static const int pair3_env = getenv("TQ_CONV_PAIR3") ? atoi(getenv("TQ_CONV_PAIR3")) : 0;
                static const int pair_env3 = getenv("TQ_CONV_PAIR") ? atoi(getenv("TQ_CONV_PAIR")) : 1;
                if (pair3_env && pair_env3 && !g.halo_baseoff && Cout % 16 == 0 && ((g.m_tiles + 1) / 2) * g.n_tiles >= num_sms() / 2) g.pair = 1;
            }
        }
    }

    g.step_w = g.wbox; g.step_h = g.hbox; g.off_w = 0; g.off_h = 0;
    // streamed-weight halo mode (MODE 4): stride-1 filters wider than 1x1 on maps that fill the tile
    static const bool no_halo4 = getenv("TQ_CONV_NO_HALO4") != nullptr;
    // Packed halo for small maps (7x7): images are laid out W + 1 pixels per row and H + 1 rows apart -- the zero column
    // left of a row is also the right padding of the row above, the zero row above an image also the bottom padding of
    // the image before it -- so one TMA box of (W + 1) x (H + 1) x nbox pixels (origin (-1, -1)) is the halo of nbox whole
    // images, and filter tap (r, s) is that buffer read from row r * (W + 1) + s on.  MMA row m = image m / ((W+1)(H+1)),
    // pixel ((m / (W+1)) % (H+1), m % (W+1)); the rows with pixel row H or column W are junk.
    static const bool no_packed = getenv("TQ_CONV_NO_PACKED") != nullptr;
    if (kind == 0 && !no_halo4 && !no_packed && g.prog_steps == 0 && !g.halo && block_n == 128 && stride == 1 && R == 3 && S == 3 &&
        pad == 1 && N >= 2 && 2 * (W + 1) * (H + 1) <= 128) {
        const int per = (W + 1) * (H + 1);
        g.wbox = W; g.hbox = H; g.nbox = 128 / per < N ? 128 / per : N;
        g.hw = W + 1; g.img_h1 = H + 1;
        g.tiles_w = g.tiles_h = 1; g.tiles_n = (N + g.nbox - 1) / g.nbox; g.m_tiles = g.tiles_n;
        g.a_tx_bytes = g.nbox * per * GM_ROW_BYTES;
        g.step_w = g.wbox; g.step_h = g.hbox;
        g.halo = 1;
        static const int pair_env = getenv("TQ_CONV_PAIR") ? atoi(getenv("TQ_CONV_PAIR")) : 1;
        if (pair_env && ((g.m_tiles + 1) / 2) * g.n_tiles >= num_sms() / 2) g.pair = 1;
    }
    if (kind == 0 && !no_halo4 && g.prog_steps == 0 && !g.halo && block_n == 128 && stride == 1 && R * S > 1) {
        ConvGeom h = g;
        static const int slack4 = getenv("TQ_CONV_HALO_SLACK") ? atoi(getenv("TQ_CONV_HALO_SLACK")) : 16;
        if (pick_box_halo(h) && (long)h.m_tiles * 100 <= (long)g.m_tiles * (100 + slack4)) {
            h.step_w = h.wbox; h.step_h = h.hbox;
            g = h;
            g.halo = 1;
            // CTA pairs (cta_group::2) when there are enough tiles to keep every pair busy: per CTA half the weight
            // traffic from L2 and 6 KB instead of 8 KB of operand reads per MMA.  TQ_CONV_PAIR=0 keeps single CTAs.
            static const int pair_env = getenv("TQ_CONV_PAIR") ? atoi(getenv("TQ_CONV_PAIR")) : 1;
            if (pair_env && ((g.m_tiles + 1) / 2) * g.n_tiles >= num_sms() / 2) g.pair = 1;
        }
    }
    const CUtensorMapDataType op_dt = kind == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const int op_es = kind == 1 ? 1 : 2;
    int rc;
    {   // activations: (C, W, H, planes * N); box spans wbox*stride x hbox*stride pixels, element strides = conv stride
        cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)(g.planes_a * N)};
        cuuint32_t box[4] = {(cuuint32_t)g.kblk, (cuuint32_t)(g.wbox * stride), (cuuint32_t)(g.hbox * stride), (cuuint32_t)g.nbox};
        if (g.halo) { box[1] = (cuuint32_t)g.hw; box[2] = (cuuint32_t)(g.hbox + R - 1); }
        if (g.img_h1) { box[2] = (cuuint32_t)g.img_h1; box[3] = (cuuint32_t)g.nbox; }
        cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
        if ((rc = encode_map(enc, &pl.tmA, op_dt, op_es, a.act, 4, dims, box, estr, "activations")) != TQ_OK) return rc;
    }
    {   // weights: (C, Cout, planes * R*S), one K block of one tap per tile
        if (g.prog_steps > 0 && g.kc_blocks != 1) { g.halo = 0; g.pair = 0; g.prog_steps = 0; g.nb_tiles = 0; }   // (program mode: one block per tap)
        cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)Cout, (cuuint64_t)(g.planes_w * R * S)};
        cuuint32_t box[3] = {(cuuint32_t)g.kblk, (cuuint32_t)(g.pair ? block_n / 2 : block_n), 1};   // (a pair CTA loads half a tile)
        cuuint32_t estr[3] = {1, 1, 1};
        if ((rc = encode_map(enc, &pl.tmB, op_dt, op_es, a.wgt, 3, dims, box, estr, "weights")) != TQ_OK) return rc;
    }
    cuuint64_t odims[4] = {(cuuint64_t)Cout, (cuuint64_t)g.Wo, (cuuint64_t)g.Ho, (cuuint64_t)N};
    cuuint32_t one[4] = {1, 1, 1, 1};
    cuuint32_t obox[4] = {32, (cuuint32_t)g.wbox, (cuuint32_t)g.hbox, (cuuint32_t)g.nbox};
    // fp32 output tile: 32 channels (128 B) x pixel box; fp16 code tile: 32 channels (64 B, 64-byte swizzle);
    // residual tile: same box as the fp32 output tile.  Unused maps still have to be valid objects.
    pl.tmC = pl.tmA; pl.tmD = pl.tmA; pl.tmR = pl.tmA;
    if (a.out_f32 && (rc = encode_map(enc, &pl.tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.out_f32, 4, odims, obox, one, "fp32 output")) != TQ_OK) return rc;
    if (a.out_codes && (rc = encode_map(enc, &pl.tmD, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, a.out_codes, 4, odims, obox, one, "code output",
                                        CU_TENSOR_MAP_SWIZZLE_64B)) != TQ_OK) return rc;
    if (a.residual && (rc = encode_map(enc, &pl.tmR, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.residual, 4, odims, obox, one, "residual")) != TQ_OK) return rc;
    if ((rc = pick_variant(g, block_n, kind, false, pl.variant)) != TQ_OK) return rc;
    pl.g = g;
    pl.key = a;
    return TQ_OK;
}

static int run_conv(ConvArgs &a, cudaStream_t s)
{
    int dev = 0;
    cudaGetDevice(&dev);
    a.device = dev;
    const uint64_t h = hash_args(a);
    static const bool no_cache = getenv("TQ_CONV_NO_PLAN_CACHE") != nullptr;
    ConvPlan pl;
    bool hit = false;
    if (!no_cache) {
        std::lock_guard<std::mutex> lk(g_plan_mu);
        for (const ConvPlan &c : g_plans[h & 63])
            if (memcmp(&c.key, &a, sizeof(ConvArgs)) == 0) { pl = c; hit = true; break; }
    }
    if (!hit) {
        int rc = plan_conv(a, pl);
        if (rc != TQ_OK) return rc;
        if (!no_cache) {
            std::lock_guard<std::mutex> lk(g_plan_mu);
            if (g_plan_count >= 4096) { for (auto &b : g_plans) b.clear(); g_plan_count = 0; }
            g_plans[h & 63].push_back(pl);
            ++g_plan_count;
        }
    }
    return launch_variant(pl.variant, pl.tmA, pl.tmB, pl.tmC, pl.tmD, pl.tmR, pl.g, s);
}

// checks the arguments and fills nq; the fused encode only has the hoisted-reciprocal divide (tq_common.cuh)
static int check_conv_args(NextQuant &nq, const void *act, const void *wgt, const void *out_f32, const void *out_codes,
                           const void *bias, const void *bn_a, const void *bn_b, const void *residual, int N, int H, int W,
                           int C, int Cout, int R, int S, int stride, int pad, float next_sf, int next_bits, int next_terms,
                           int next_enc, int c_align)
{
    const int rc = next_quant(nq, out_codes, next_sf, next_bits, next_terms, next_enc, GM_LUT_MAX_BITS, true);
    if (rc != TQ_OK) return rc;
    if (!act || !wgt || (!out_f32 && !out_codes)) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (N < 1 || H < 1 || W < 1 || C < 1 || Cout < 1 || R < 1 || S < 1 || stride < 1 || pad < 0)
        return fail(TQ_ERR_INVALID, "bad convolution geometry");
    if (C % c_align != 0) return fail(TQ_ERR_UNSUPPORTED, "input channels must be a multiple of %d (16-byte TMA rows), got %d", c_align, C);
    if (Cout % 4 != 0) return fail(TQ_ERR_UNSUPPORTED, "output channels must be a multiple of 4, got %d", Cout);
    if (out_codes && Cout % 8 != 0) return fail(TQ_ERR_UNSUPPORTED, "code output needs Cout %% 8 == 0, got %d", Cout);
    if ((bn_a == nullptr) != (bn_b == nullptr)) return fail(TQ_ERR_INVALID, "bn_a and bn_b go together");
    if ((((uintptr_t)act | (uintptr_t)wgt | (uintptr_t)out_f32 | (uintptr_t)out_codes | (uintptr_t)bias |
          (uintptr_t)bn_a | (uintptr_t)bn_b | (uintptr_t)residual) & 15u) != 0)
        return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    return TQ_OK;
}

}  // namespace tq

using namespace tq;

extern "C" int tq_conv2d_codes_fused(const void *act, const void *wgt, float *out_f32, void *out_codes,
                                     const float *bias, const float *bn_a, const float *bn_b,
                                     const float *residual, int N, int H, int W, int C, int Cout, int R, int S,
                                     int stride, int pad, float scale, int relu, float next_sf, int next_bits,
                                     int next_terms, int acc_groups, void *stream)
{
    return tq_conv2d_codes_fused_enc(act, wgt, out_f32, out_codes, bias, bn_a, bn_b, residual, N, H, W, C, Cout, R, S, stride,
                                     pad, scale, relu, next_sf, next_bits, next_terms, TQ_ENC_HESE, acc_groups, stream);
}

extern "C" int tq_conv2d_codes_fused_enc(const void *act, const void *wgt, float *out_f32, void *out_codes,
                                         const float *bias, const float *bn_a, const float *bn_b,
                                         const float *residual, int N, int H, int W, int C, int Cout, int R, int S,
                                         int stride, int pad, float scale, int relu, float next_sf, int next_bits,
                                         int next_terms, int next_enc, int acc_groups, void *stream)
{
    ConvArgs a;
    memset(&a, 0, sizeof(a));                       // (padding bytes take part in the cache key)
    int rc = check_conv_args(a.nq, act, wgt, out_f32, out_codes, bias, bn_a, bn_b, residual, N, H, W, C, Cout, R, S, stride, pad,
                             next_sf, next_bits, next_terms, next_enc, 8);
    if (rc != TQ_OK) return rc;
    a.act = act; a.wgt = wgt; a.out_f32 = out_f32; a.out_codes = out_codes; a.bias = bias; a.bn_a = bn_a; a.bn_b = bn_b;
    a.residual = residual;
    a.kind = 0; a.N = N; a.H = H; a.W = W; a.C = C; a.Cout = Cout; a.R = R; a.S = S; a.stride = stride; a.pad = pad;
    a.relu = relu == 2 ? 2 : (relu ? 1 : 0);
    a.acc_groups = acc_groups < 1 ? 1 : acc_groups; a.planes_a = 1; a.planes_w = 1;
    a.scale = scale;
    return run_conv(a, (cudaStream_t)stream);
}

extern "C" int tq_conv2d_codes_f16(const void *act, const void *wgt, const float *bias, float *out,
                                   int N, int H, int W, int C, int Cout, int R, int S, int stride, int pad,
                                   float scale, int acc_groups, void *stream)
{
    if (!out) return fail(TQ_ERR_INVALID, "NULL pointer");
    return tq_conv2d_codes_fused(act, wgt, out, nullptr, bias, nullptr, nullptr, nullptr, N, H, W, C, Cout, R, S,
                                 stride, pad, scale, 0, 1.0f, 1, 0, acc_groups, stream);
}

extern "C" int tq_conv2d_planes_i8(const void *act_planes, const void *wgt_planes, int planes_a, int planes_w,
                                   float *out_f32, void *out_codes, const float *bias, const float *bn_a,
                                   const float *bn_b, const float *residual, int N, int H, int W, int C, int Cout,
                                   int R, int S, int stride, int pad, float scale, int relu, float next_sf,
                                   int next_bits, int next_terms, int act_max, int wgt_max, void *stream)
{
    return tq_conv2d_planes_i8_enc(act_planes, wgt_planes, planes_a, planes_w, out_f32, out_codes, bias, bn_a, bn_b, residual,
                                   N, H, W, C, Cout, R, S, stride, pad, scale, relu, next_sf, next_bits, next_terms,
                                   TQ_ENC_HESE, act_max, wgt_max, stream);
}

extern "C" int tq_conv2d_planes_i8_enc(const void *act_planes, const void *wgt_planes, int planes_a, int planes_w,
                                       float *out_f32, void *out_codes, const float *bias, const float *bn_a,
                                       const float *bn_b, const float *residual, int N, int H, int W, int C, int Cout,
                                       int R, int S, int stride, int pad, float scale, int relu, float next_sf,
                                       int next_bits, int next_terms, int next_enc, int act_max, int wgt_max, void *stream)
{
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    int rc = check_conv_args(a.nq, act_planes, wgt_planes, out_f32, out_codes, bias, bn_a, bn_b, residual, N, H, W, C, Cout, R,
                             S, stride, pad, next_sf, next_bits, next_terms, next_enc, 16);
    if (rc != TQ_OK) return rc;
    if (planes_a < 1 || planes_a > 2 || planes_w < 1 || planes_w > 2) return fail(TQ_ERR_INVALID, "1 or 2 planes per operand");
    // int32 accumulators: |acc| <= K * act_max * wgt_max (the caller's bounds on |code|: 2^bits by construction of the
    // term codes; what one / two planes can hold caps them)
    const int acap = planes_a == 2 ? 2047 : 127, wcap = planes_w == 2 ? 2047 : 127;
    if (act_max < 1 || act_max > acap || wgt_max < 1 || wgt_max > wcap)
        return fail(TQ_ERR_INVALID, "act_max / wgt_max must lie in 1..%d / 1..%d for %d / %d planes", acap, wcap, planes_a, planes_w);
    if ((double)C * R * S * (double)act_max * (double)wgt_max >= 2147483648.0)
        return fail(TQ_ERR_UNSUPPORTED, "K = %d with |a| <= %d, |w| <= %d can overflow an int32 accumulator", C * R * S, act_max, wgt_max);
    a.act = act_planes; a.wgt = wgt_planes; a.out_f32 = out_f32; a.out_codes = out_codes; a.bias = bias; a.bn_a = bn_a;
    a.bn_b = bn_b; a.residual = residual;
    a.kind = 1; a.N = N; a.H = H; a.W = W; a.C = C; a.Cout = Cout; a.R = R; a.S = S; a.stride = stride; a.pad = pad;
    a.relu = relu == 2 ? 2 : (relu ? 1 : 0);
    a.acc_groups = 1; a.planes_a = planes_a; a.planes_w = planes_w;
    a.scale = scale;
    return run_conv(a, (cudaStream_t)stream);
}

// ---- operand planes and the static accumulator bound ------------------------------------------------
namespace tq {

// fp16 integer codes -> signed 8-bit planes: code = 16 * hi + lo, hi = code >> 4 (floor), lo = code & 15.
// planes == 1: the code itself as s8 (the caller knows |code| <= 127; a code outside sets *overflow).
__global__ void __launch_bounds__(256)
codes_to_planes_kernel(const __half *__restrict__ codes, int8_t *__restrict__ planes, int64_t n8, int64_t plane_stride,
                       int nplanes, int *__restrict__ overflow)
{
    bool ovf = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(codes) + i);      // 8 codes
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t hi[2] = {0u, 0u}, lo[2] = {0u, 0u};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int c = __half2int_rn(__ushort_as_half((unsigned short)(w[e >> 1] >> (16 * (e & 1)))));
            int h, l;
            if (nplanes == 2) { h = c >> GM_I8_SHIFT; l = c & ((1 << GM_I8_SHIFT) - 1); }
            else { h = c; l = 0; }
            ovf |= (h < -128 || h > 127);
            hi[e >> 2] |= (uint32_t)(h & 0xFF) << (8 * (e & 3));
            lo[e >> 2] |= (uint32_t)(l & 0xFF) << (8 * (e & 3));
        }
        reinterpret_cast<uint2 *>(planes)[i] = make_uint2(hi[0], hi[1]);
        if (nplanes == 2) reinterpret_cast<uint2 *>(planes + plane_stride)[i] = make_uint2(lo[0], lo[1]);
    }
    if (ovf && overflow) atomicExch(overflow, 1);
}

// per (output channel, 64-channel block): sum of the positive and of the negative weight codes over all taps
__global__ void __launch_bounds__(128)
weight_l1_kernel(const __half *__restrict__ wgt, int RS, int Cout, int C, int kcb, long long *__restrict__ pos, long long *__restrict__ neg)
{
    const int co = blockIdx.x, kb = blockIdx.y;
    long long p = 0, m = 0;
    const int c0 = kb * GM_BLOCK_K, c1 = min(C, c0 + GM_BLOCK_K);
    for (int t = threadIdx.x; t < RS * (c1 - c0); t += blockDim.x) {
        const int tap = t / (c1 - c0), c = c0 + t % (c1 - c0);
        const int v = __half2int_rn(wgt[((int64_t)tap * Cout + co) * C + c]);
        if (v > 0) p += v; else m -= v;
    }
    __shared__ long long sp[128], sm[128];
    sp[threadIdx.x] = p; sm[threadIdx.x] = m;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sp[threadIdx.x] += sp[threadIdx.x + o]; sm[threadIdx.x] += sm[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { pos[(int64_t)co * kcb + kb] = sp[0]; neg[(int64_t)co * kcb + kb] = sm[0]; }
}

}  // namespace tq

extern "C" int tq_codes_to_planes(const void *codes_f16, void *planes_s8, int64_t n, int planes, int *overflow, void *stream)
{
    if (!codes_f16 || !planes_s8) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (n < 0 || n % 8 != 0) return fail(TQ_ERR_INVALID, "element count must be a multiple of 8");
    if (planes != 1 && planes != 2) return fail(TQ_ERR_INVALID, "1 or 2 planes");
    if ((((uintptr_t)codes_f16 | (uintptr_t)planes_s8) & 15u) != 0) return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    if (n == 0) return TQ_OK;
    int64_t blocks = (n / 8 + 255) / 256;
    if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
    codes_to_planes_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const __half *)codes_f16, (int8_t *)planes_s8, n / 8, n,
                                                                        planes, overflow);
    count_launch();
    return check_launch("codes_to_planes_kernel");
}

extern "C" int tq_conv_weight_l1(const void *wgt_f16, int RS, int Cout, int C, long long *pos, long long *neg, void *stream)
{
    if (!wgt_f16 || !pos || !neg) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (RS < 1 || Cout < 1 || C < 1) return fail(TQ_ERR_INVALID, "bad weight shape");
    const int kcb = (C + GM_BLOCK_K - 1) / GM_BLOCK_K;
    weight_l1_kernel<<<dim3((unsigned)Cout, (unsigned)kcb), 128, 0, (cudaStream_t)stream>>>((const __half *)wgt_f16, RS, Cout, C, kcb, pos, neg);
    count_launch();
    return check_launch("weight_l1_kernel");
}


// =============================================================================================
// Unquantised stem conv (7x7 / stride 2 / pad 3 on 3 channels -- the first conv of the CNNs in
// cnn_models/, never wrapped: cnn_models/__init__.py:34-36) on the same tensor-core kernel.
//
//   * space-to-depth: with the image padded by 3 and folded 2x2 into 16 channels ((dr, ds, c), c
//     padded 3 -> 4) the conv is a 4x4 / stride-1 conv without padding:  r = 2R + dr, s = 2S + ds.
//   * for one filter row R the four taps S = 0..3 x 16 channels are 64 CONTIGUOUS fp16 of the
//     folded image, so the A operand of a k-block is a tensor map whose inner dimension is that
//     64-element window and whose next dimension (output column) advances by 16 elements: the
//     windows overlap, TMA does the im2col.
//   * fp32 accuracy from fp16 tensor cores: x = x_hi + x_lo, w = w_hi + w_lo (fp16 each) and
//     acc = x_hi*w_hi + x_hi*w_lo + x_lo*w_hi in the fp32 TMEM accumulator (the dropped lo*lo
//     term is 2^-22 relative, below the rounding noise of an fp32 FMA chain of length 147).
// =============================================================================================
namespace tq {

// uint8 images: ToTensor + Normalize as torchvision computes them on the host in fp32 (util.py:12-27: x = u8 / 255, then
// (x - mean[c]) / std[c], each one IEEE operation), rounded to bf16 -- exactly what tq_u8_normalize_bf16 writes -- folded
// straight into the fp16 planes (a bf16 value is an fp16 value down to 2^-14)
struct StemNorm { float mean[3], sd[3]; };
__device__ __forceinline__ float stem_pixel(uint8_t v, int c, const StemNorm &nm)
{
    const float t = __fdiv_rn((float)v, 255.0f);
    return __bfloat162float(__float2bfloat16_rn(__fdiv_rn(__fsub_rn(t, nm.mean[c]), nm.sd[c])));
}
template <typename T> __device__ __forceinline__ float stem_pixel(T v, int, const StemNorm &) { return Elem<T>::to_f32(v); }

template <typename Tin, bool LO>
__global__ void __launch_bounds__(256)
stem_prepare_kernel(const Tin *__restrict__ x, __half *__restrict__ x2, int N, int H, int W, int Hs, int Ws, StemNorm nm)
{
    // one thread per folded pixel (n, hs, ws): 16 halves hi (+ 16 halves lo for fp32 input; bf16 / fp16
    // images are fp16-exact down to 2^-14, below that the residue is < 2^-25 absolute and is dropped)
    // uint8 images: the 3 x 256 possible normalised values once per CTA (two IEEE divisions each), then one lookup per value
    __shared__ __half norm_lut[std::is_same<Tin, uint8_t>::value ? 768 : 1];
    if constexpr (std::is_same<Tin, uint8_t>::value) {
        for (int i = threadIdx.x; i < 768; i += blockDim.x) norm_lut[i] = __float2half_rn(stem_pixel((uint8_t)(i & 255), i >> 8, nm));
        __syncthreads();
    }
    const int64_t total = (int64_t)N * Hs * Ws;
    const int64_t plane = total * 16;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int ws = (int)(t % Ws), hs = (int)((t / Ws) % Hs), n = (int)(t / ((int64_t)Ws * Hs));
        __align__(16) __half hi[16], lo[16];
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const int h = 2 * hs + (d >> 1) - 3, w = 2 * ws + (d & 1) - 3;
            const bool in = h >= 0 && h < H && w >= 0 && w < W;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if constexpr (std::is_same<Tin, uint8_t>::value) {
                    hi[d * 4 + c] = (in && c < 3) ? norm_lut[c * 256 + (int)x[(((int64_t)n * H + h) * W + w) * 3 + c]] : __float2half_rn(0.0f);
                } else {
                    float v = 0.0f;
                    if (in && c < 3) v = stem_pixel(x[(((int64_t)n * H + h) * W + w) * 3 + c], c, nm);
                    const __half vh = __float2half_rn(v);
                    hi[d * 4 + c] = vh;
                    if (LO) lo[d * 4 + c] = __float2half_rn(v - __half2float(vh));
                }
            }
        }
        uint4 *dh = reinterpret_cast<uint4 *>(x2 + t * 16);
        dh[0] = reinterpret_cast<const uint4 *>(hi)[0]; dh[1] = reinterpret_cast<const uint4 *>(hi)[1];
        if constexpr (LO) {
            uint4 *dl = reinterpret_cast<uint4 *>(x2 + plane + t * 16);
            dl[0] = reinterpret_cast<const uint4 *>(lo)[0]; dl[1] = reinterpret_cast<const uint4 *>(lo)[1];
        }
    }
}

}  // namespace tq

// (image dtype of the uint8 entry point inside stem_impl: the public TQ_U8 is a CODE dtype and shares its value with TQ_F16)
constexpr int STEM_U8 = 100;

// pool = 0: out = conv (fp32 [N, H/2, W/2, Cout]).  pool = 1: out = maxpool3x3s2p1(relu?(fma(conv, bn_a, bn_b)))
// (fp32 [N, Hp, Wp, Cout]) and, if out_codes, its fp16 term codes for the next layer's quantiser.  pool = 2: out = the
// max of conv columns 2q-1, 2q, 2q+1 of every conv row (fp32 [N, H/2, Wp, Cout]), the horizontal half of the pool.
static int stem_impl(const void *x, int x_dtype, void *x2_scratch, const void *w2, float *out, void *out_codes,
                     const float *bn_a, const float *bn_b, int relu, int pool, float next_sf, int next_bits,
                     int next_terms, int next_enc, int N, int H, int W, int Cout, void *stream, const float *mean3 = nullptr,
                     const float *std3 = nullptr)
{
    // the quantiser is checked before the fold pass below is launched: a refused call enqueues nothing (only the pooled
    // stem passes out_codes)
    ConvGeom g{};
    int rc = next_quant(g.nq, out_codes, next_sf, next_bits, next_terms, next_enc, GM_LUT_MAX_BITS, false);
    if (rc != TQ_OK) return rc;
    if (!x || !x2_scratch || !w2 || !out) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (x_dtype != TQ_F32 && x_dtype != TQ_BF16 && x_dtype != TQ_F16 && x_dtype != STEM_U8)
        return fail(TQ_ERR_UNSUPPORTED, "stem conv input must be fp32, bf16, fp16 or uint8");
    StemNorm nm{};
    if (x_dtype == STEM_U8) {
        if (!mean3 || !std3) return fail(TQ_ERR_INVALID, "uint8 images need mean3 / std3");
        for (int c = 0; c < 3; ++c) {
            if (!(std3[c] > 0.0f)) return fail(TQ_ERR_INVALID, "std must be positive");
            nm.mean[c] = mean3[c]; nm.sd[c] = std3[c];
        }
    }
    const bool lo_plane = x_dtype == TQ_F32;
    if (N < 1 || H < 2 || W < 2 || (H & 1) || (W & 1)) return fail(TQ_ERR_INVALID, "H and W must be even");
    if (Cout < 4 || Cout % 4) return fail(TQ_ERR_UNSUPPORTED, "Cout must be a multiple of 4");
    if ((((uintptr_t)x2_scratch | (uintptr_t)w2 | (uintptr_t)out) & 15u) != 0)
        return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cudaStream_t s = (cudaStream_t)stream;
    const int Ho = H / 2, Wo = W / 2, Hs = Ho + 3, Ws = Wo + 3;

    {   // fold + split the image: fp32 NHWC3 -> fp16 [2][N][Hs][Ws][16]
        const int64_t total = (int64_t)N * Hs * Ws;
        int64_t blocks = (total + 255) / 256;
        if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
        if (x_dtype == TQ_F32)
            stem_prepare_kernel<float, true><<<(int)blocks, 256, 0, s>>>((const float *)x, (__half *)x2_scratch, N, H, W, Hs, Ws, nm);
        else if (x_dtype == TQ_BF16)
            stem_prepare_kernel<__nv_bfloat16, false><<<(int)blocks, 256, 0, s>>>((const __nv_bfloat16 *)x, (__half *)x2_scratch, N, H, W, Hs, Ws, nm);
        else if (x_dtype == STEM_U8)
            stem_prepare_kernel<uint8_t, false><<<(int)blocks, 256, 0, s>>>((const uint8_t *)x, (__half *)x2_scratch, N, H, W, Hs, Ws, nm);
        else
            stem_prepare_kernel<__half, false><<<(int)blocks, 256, 0, s>>>((const __half *)x, (__half *)x2_scratch, N, H, W, Hs, Ws, nm);
        count_launch();
        if ((rc = check_launch("stem_prepare_kernel")) != TQ_OK) return rc;
    }

    g.N = N; g.H = Hs; g.W = Wo; g.C = 64; g.Cout = Cout; g.R = 4; g.S = 1; g.stride = 1; g.pad = 0;
    g.Ho = Ho; g.Wo = Wo;
    g.scale = 1.0f;
    g.kc_blocks = 1;
    int Hp = 0, Wp = 0;
    if (!pool) {
        if (!pick_box_halo(g)) return fail(TQ_ERR_UNSUPPORTED, "stem conv: no tile shape");
        g.step_w = g.wbox; g.step_h = g.hbox;
    } else if (pool == 2) {
        // row-max tile: 4 conv rows x 32 conv columns (one warp per row, see the epilogue) -> 4 x Q row maxima, Q <= 15
        Wp = (Wo - 1) / 2 + 1;
        g.pool = 2;
        g.pool_q = Wp < 15 ? Wp : 15;
        g.wbox = 32; g.hbox = Ho < 4 ? Ho : 4; g.nbox = 1;
        g.step_w = 2 * g.pool_q; g.step_h = g.hbox; g.off_w = -1; g.off_h = 0;
        g.tiles_w = (Wp + g.pool_q - 1) / g.pool_q; g.tiles_h = (Ho + g.hbox - 1) / g.hbox; g.tiles_n = N;
        g.m_tiles = g.tiles_w * g.tiles_h * g.tiles_n;
    } else {
        // pooled tile P x Q over the (2P+1) x (2Q+1) conv pixels it needs (<= 128 accumulator rows): fewest tiles
        Hp = (Ho + 2 - 3) / 2 + 1; Wp = (Wo + 2 - 3) / 2 + 1;
        long best = -1;
        for (int P = 1; P <= Hp && 2 * P + 1 <= 128; ++P)
            for (int Q = 1; Q <= Wp && (2 * P + 1) * (2 * Q + 1) <= 128; ++Q) {
                const long tiles = (long)((Hp + P - 1) / P) * ((Wp + Q - 1) / Q);
                if (best < 0 || tiles < best || (tiles == best && Q > g.pool_q)) { best = tiles; g.pool_p = P; g.pool_q = Q; }
            }
        g.pool = 1;
        g.wbox = 2 * g.pool_q + 1; g.hbox = 2 * g.pool_p + 1; g.nbox = 1;
        g.step_w = 2 * g.pool_q; g.step_h = 2 * g.pool_p; g.off_w = -1; g.off_h = -1;
        g.tiles_w = (Wp + g.pool_q - 1) / g.pool_q; g.tiles_h = (Hp + g.pool_p - 1) / g.pool_p; g.tiles_n = N;
        g.m_tiles = g.tiles_w * g.tiles_h * g.tiles_n;
        g.a_tx_bytes = g.wbox * g.hbox * GM_BLOCK_K * 2;
        if (g.pool_p * g.pool_q > 32) return fail(TQ_ERR_UNSUPPORTED, "pooled tile too large");
        g.bn_a = bn_a; g.bn_b = bn_b; g.relu = relu ? 1 : 0;
    }
    g.hw = g.wbox;
    const int block_n = Cout <= 64 ? 64 : 128;
    g.n_tiles = (Cout + block_n - 1) / block_n;
    g.write_f32 = 1;
    // program: per image plane (x_hi, and x_lo for fp32 images) ONE halo load covering the four folded filter rows; per
    // filter row R one N = 128 MMA group against the resident tile R = [w_hi (rows 0..63) ; w_lo (rows 64..127)]: columns
    // [c, c+64) of the accumulator receive x * w_hi, [c+64, c+128) x * w_lo.  Rows 0-1 and rows 2-3 accumulate apart
    // (c = 0 / 128): tensor-core accumulation truncates, so fewer steps per accumulator = less bias, and the small lo
    // products live apart from the large ones; the four 64-column groups are summed once, in fp32 RN, in the epilogue.
    // TQ_STEM_SPLIT=0: all four filter rows into ONE accumulator pair (2 column groups, half the TMEM reads of the
    // epilogue, three accumulator stages) at the price of 16 instead of 8 truncating accumulation steps
    static const int split_rows = getenv("TQ_STEM_SPLIT") ? atoi(getenv("TQ_STEM_SPLIT")) : 1;
    g.prog_steps = lo_plane ? 8 : 4; g.nb_tiles = 4; g.n_groups = split_rows ? 4 : 2; g.b_rows = 128;
    for (uint32_t R = 0; R < 4; ++R) {
        g.prog_mma[R] = 1u | (R << 4) | (((R < 2 || !split_rows) ? 0u : 2u) << 8);
        g.prog_mma[4 + R] = g.prog_mma[R];                  // x_lo against the same tiles (x_lo * w_lo is 2^-22: harmless)
    }

    CUtensorMap tmA, tmB, tmC, tmD;
    {   // overlapping windows: inner 64 elements, output column advances by one folded pixel (16 elements)
        cuuint64_t dims[4] = {64, (cuuint64_t)Wo, (cuuint64_t)Hs, (cuuint64_t)((lo_plane ? 2 : 1) * N)};
        cuuint64_t strides[3] = {32, (cuuint64_t)Ws * 32, (cuuint64_t)Hs * Ws * 32};
        cuuint32_t box[4] = {64, (cuuint32_t)g.wbox, (cuuint32_t)(g.hbox + g.R - 1), 1};   // all R filter rows at once
        cuuint32_t one[4] = {1, 1, 1, 1};
        g.a_tx_bytes = g.wbox * (g.hbox + g.R - 1) * GM_BLOCK_K * 2;
        g.halo = 1;                                         // (stage size follows a_tx_bytes)
        CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x2_scratch, dims, strides, box, one,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(TQ_ERR_CUDA, "cuTensorMapEncodeTiled(stem windows) failed: %d", (int)r);
    }
    {
        cuuint64_t dims[3] = {64, 128, 4};
        cuuint32_t box[3] = {64, 128, 1};
        cuuint32_t one[3] = {1, 1, 1};
        if ((rc = encode_map(enc, &tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w2, 3, dims, box, one, "stem weights")) != TQ_OK) return rc;
    }
    tmD = tmA;
    if (!pool) {
        cuuint64_t odims[4] = {(cuuint64_t)Cout, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)N};
        cuuint32_t box[4] = {32, (cuuint32_t)g.wbox, (cuuint32_t)g.hbox, (cuuint32_t)g.nbox};
        cuuint32_t one[4] = {1, 1, 1, 1};
        if ((rc = encode_map(enc, &tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, 4, odims, box, one, "stem output")) != TQ_OK) return rc;
    } else if (pool == 2) {
        cuuint64_t odims[4] = {(cuuint64_t)Cout, (cuuint64_t)Wp, (cuuint64_t)Ho, (cuuint64_t)N};
        cuuint32_t box[4] = {32, (cuuint32_t)g.pool_q, (cuuint32_t)g.hbox, 1};
        cuuint32_t one[4] = {1, 1, 1, 1};
        if ((rc = encode_map(enc, &tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, 4, odims, box, one, "stem row maxima")) != TQ_OK) return rc;
    } else {
        cuuint64_t odims[4] = {(cuuint64_t)Cout, (cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)N};
        cuuint32_t box[4] = {32, (cuuint32_t)g.pool_q, (cuuint32_t)g.pool_p, 1};
        cuuint32_t one[4] = {1, 1, 1, 1};
        if ((rc = encode_map(enc, &tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, 4, odims, box, one, "pooled output")) != TQ_OK) return rc;
        if (out_codes && (rc = encode_map(enc, &tmD, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, out_codes, 4, odims, box, one,
                                          "pooled codes", CU_TENSOR_MAP_SWIZZLE_64B)) != TQ_OK) return rc;
    }
    if (g.nbox != 1) return fail(TQ_ERR_UNSUPPORTED, "stem conv expects images of at least 128 output pixels");
    if (block_n != 64) return fail(TQ_ERR_UNSUPPORTED, "stem conv supports Cout <= 64");
    g.kblk = GM_BLOCK_K; g.kcpg = 1; g.planes_a = g.planes_w = 1; g.acc_int = 0;   // hi/lo groups are summed in fp32
    ConvVariant variant = CV_NONE;
    if ((rc = pick_variant(g, 64, 0, true, variant)) != TQ_OK) return rc;
    return launch_variant(variant, tmA, tmB, tmC, tmD, tmA, g, s);
}

extern "C" int tq_stem_conv7x7s2_dt(const void *x, int x_dtype, void *x2_scratch, const void *w2, float *out,
                                    int N, int H, int W, int Cout, void *stream)
{
    return stem_impl(x, x_dtype, x2_scratch, w2, out, nullptr, nullptr, nullptr, 0, 0, 1.0f, 1, 0, TQ_ENC_HESE, N, H, W, Cout, stream);
}

extern "C" int tq_stem_conv7x7s2_pool(const void *x, int x_dtype, void *x2_scratch, const void *w2,
                                      const float *bn_a, const float *bn_b, int relu, float *out, void *out_codes,
                                      int N, int H, int W, int Cout, float next_sf, int next_bits, int next_terms,
                                      void *stream)
{
    return tq_stem_conv7x7s2_pool_enc(x, x_dtype, x2_scratch, w2, bn_a, bn_b, relu, out, out_codes, N, H, W, Cout, next_sf,
                                      next_bits, next_terms, TQ_ENC_HESE, stream);
}

extern "C" int tq_stem_conv7x7s2_pool_enc(const void *x, int x_dtype, void *x2_scratch, const void *w2,
                                          const float *bn_a, const float *bn_b, int relu, float *out, void *out_codes,
                                          int N, int H, int W, int Cout, float next_sf, int next_bits, int next_terms,
                                          int next_enc, void *stream)
{
    if (!bn_a || !bn_b) return fail(TQ_ERR_INVALID, "NULL pointer");
    if (Cout % 8) return fail(TQ_ERR_UNSUPPORTED, "Cout must be a multiple of 8");
    if ((((uintptr_t)bn_a | (uintptr_t)bn_b | (uintptr_t)out_codes) & 15u) != 0) return fail(TQ_ERR_INVALID, "pointers must be 16-byte aligned");
    return stem_impl(x, x_dtype, x2_scratch, w2, out, out_codes, bn_a, bn_b, relu, 1, next_sf, next_bits, next_terms,
                     next_enc, N, H, W, Cout, stream);
}

extern "C" int tq_stem_conv7x7s2_u8(const void *x_u8, const float *mean3, const float *std3, void *x2_scratch, const void *w2,
                                    float *out, int N, int H, int W, int Cout, void *stream)
{
    return stem_impl(x_u8, STEM_U8, x2_scratch, w2, out, nullptr, nullptr, nullptr, 0, 0, 1.0f, 1, 0, TQ_ENC_HESE, N, H, W, Cout, stream,
                     mean3, std3);
}

extern "C" int tq_stem_conv7x7s2_rowmax(const void *x, int x_dtype, void *x2_scratch, const void *w2, float *out,
                                        int N, int H, int W, int Cout, void *stream)
{
    return stem_impl(x, x_dtype, x2_scratch, w2, out, nullptr, nullptr, nullptr, 0, 2, 1.0f, 1, 0, TQ_ENC_HESE, N, H, W, Cout, stream);
}

extern "C" int tq_stem_conv7x7s2_u8_rowmax(const void *x_u8, const float *mean3, const float *std3, void *x2_scratch,
                                           const void *w2, float *out, int N, int H, int W, int Cout, void *stream)
{
    return stem_impl(x_u8, STEM_U8, x2_scratch, w2, out, nullptr, nullptr, nullptr, 0, 2, 1.0f, 1, 0, TQ_ENC_HESE, N, H, W, Cout, stream,
                     mean3, std3);
}

extern "C" int tq_stem_conv7x7s2(const float *x, void *x2_scratch, const void *w2, float *out,
                                 int N, int H, int W, int Cout, void *stream)
{
    return tq_stem_conv7x7s2_dt(x, TQ_F32, x2_scratch, w2, out, N, H, W, Cout, stream);
}
