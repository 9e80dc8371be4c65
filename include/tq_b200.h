/*
 * tq_b200.h -- C ABI of libtq_b200.so: the B200 (sm_100a) implementation of the
 * term-quantization hot path of BradMcDanel/term-quantization.
 *
 * This is the drop-in boundary.  Every entry point takes plain device pointers,
 * explicit sizes and the caller's CUDA stream; none takes a torch type.  The
 * reference exposes this path through one pybind11 function,
 *
 *     at::Tensor tr(const at::Tensor input, const float sf, const int32_t bitwidth,
 *                   const int32_t group_size, const int32_t num_keep_terms)
 *                                                    (kernels/tr_cuda.cpp:20-28)
 *
 * whose launcher (kernels/tr_cuda_kernel.cu:128-160) reads B = size(0),
 * C = size(1), W*H = size(2)*size(3) and launches tr_cuda_kernel on the legacy
 * default stream.  tq_tr_encode() below is what that binding calls instead; the
 * remaining entry points replace the Python/torch loops that surround it in
 * tr_layer.py (cited per function).  INTEGRATION.md shows the binding a
 * maintainer of the reference would add.
 *
 * All functions are asynchronous on `stream` (a cudaStream_t passed as void*,
 * NULL = legacy default stream), run on the current CUDA device, never
 * synchronise, and return TQ_OK or an error code; tq_last_error() returns a
 * thread-local message for the last failure.  There is no CPU fallback.
 */
#ifndef TQ_B200_H
#define TQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TQ_VERSION 201

/* status codes */
#define TQ_OK               0
#define TQ_ERR_INVALID      1   /* bad argument (range, NULL pointer, sf <= 0 ...)   */
#define TQ_ERR_UNSUPPORTED  2   /* valid in principle but not implemented            */
#define TQ_ERR_CUDA         3   /* launch or runtime failure, see tq_last_error()    */

/* element types of the floating tensors (reference dispatches float/double only,
 * kernels/tr_cuda_kernel.cu:146; bf16/f16 are upcast to fp32 and then identical) */
#define TQ_F32   0
#define TQ_F64   1
#define TQ_BF16  2
#define TQ_F16   3

/* element types of integer code tensors */
#define TQ_I8    0   /* saturating is an error: caller must know |code| <= 127 */
#define TQ_I16   1
#define TQ_I32   2
#define TQ_U8    3   /* for ReLU-ed activations, |code| <= 255                 */
#define TQ_F16C  4   /* integer codes stored as fp16 values (exact for |code| <= 2048):
                        the operand format of tq_conv2d_codes_f16                 */

/* term encodings.  The reference kernel implements HESE only
 * (kernels/tr_cuda_kernel.cu:29-55); BINARY (bit_utils.py:63-73) and radix-2
 * BOOTH (verilog/booth_encoder.v:57-78) are additions with the same selection rule.
 * For every encoding the truncated code of q in [0, 2^bits - 1] satisfies |code| <= 2^bits
 * (BINARY: <= 2^bits - 1) and is non-decreasing in q (DESIGN.md section 3).  Every fused
 * entry point below encodes with HESE; its _enc twin takes the encoding (`next_enc`,
 * after the term budget) and returns TQ_ERR_INVALID for any other value before it
 * launches anything. */
#define TQ_ENC_HESE    0
#define TQ_ENC_BINARY  1
#define TQ_ENC_BOOTH   2

/* flags */
#define TQ_FLAG_RELU       1u  /* clamp negative inputs to +0 before quantising (fused ReLU,
                                  verilog/relu_quantizer.v:119-137 pipeline order)        */
#define TQ_FLAG_RECIP_DIV  2u  /* tq_hese_term_count: w * (1/sf) instead of w / sf -- what
                                  torch's CUDA `tensor / python_float` computes            */

#define TQ_FLAG_EXACT_DIV  4u  /* tq_tr_encode*: force the per-element div.rn.f32 variant even
                                  when the hoisted-reciprocal divide applies (testing)     */

/* limits (reference: MAX_GROUP_SIZE 32, kernels/tr_cuda_kernel.cu:9) */
#define TQ_MAX_GROUP   32
#define TQ_MAX_BITS    16

int         tq_version(void);
const char *tq_last_error(void);
/* number of kernels this library has launched in this process (bench.py gpu_launches) */
uint64_t    tq_launch_count(void);

/*
 * Term-reveal a (B, C, WH) tensor: uniform-quantise every element to
 * q = min(round_half_up(|x|/sf), 2^bits-1), expand q into signed power-of-two
 * terms, keep the `alpha` largest terms of every group of `g` consecutive
 * channels (fixed b and wh, element stride WH; ties -> lowest channel), sum the
 * survivors and write sign(x) * sum * sf in the input dtype.
 * Replaces tr_cuda() (kernels/tr_cuda_kernel.cu:58-160) bit for bit wherever the
 * reference is defined.  Where it is not (C % g != 0: race + out-of-bounds,
 * SURVEY 8a-3) the tail group holds the C % g real channels and the full budget,
 * i.e. the reference's result on a zero-padded tensor.
 *   1 <= g <= 32, 1 <= bits <= 16, alpha >= 0, sf > 0 and finite.
 * in and out may alias exactly (in-place) but not partially.
 */
int tq_tr_encode(const void *in, void *out, int dtype,
                 int64_t B, int64_t C, int64_t WH,
                 float sf, int bits, int g, int alpha,
                 int encoding, unsigned flags, void *stream);

/*
 * Same selection, but writes the signed integer code (sign(x) * sum of surviving
 * terms, |code| <= 2^bits) instead of the dequantised value: the operand format of
 * the integer conv/linear (tr_layer.py:126,154 computed on integers).  A code that
 * does not fit code_dtype sets *overflow (device int, may be NULL) to 1 and is
 * written saturated.
 */
int tq_tr_encode_codes(const void *in, void *codes, int dtype, int code_dtype,
                       int64_t B, int64_t C, int64_t WH,
                       float sf, int bits, int g, int alpha,
                       int encoding, unsigned flags, int *overflow, void *stream);

/*
 * hist[b] += number of x in bin b, with torch.histc's CUDA binning
 * (tr_layer.py:92: torch.histc(x, 8192, -50, 50)); hist is float32[nbins] on the
 * device.  Elements are counted exactly in counts_scratch (uint32, left zeroed again on
 * return) and added to hist with one fp32 rounding per bin per call.
 */
int tq_hist_accumulate(const void *x, int dtype, int64_t n,
                       float *hist, uint32_t *counts_scratch /* nbins, zeroed once by the caller */,
                       int nbins, float lo, float hi, void *stream);

/*
 * Fused calibration sweep (tr_layer.py:43-54): for every scale factor sfs[s],
 * errs[s] = sum_b hist[b] * (x[b] - tr(x[b]; sfs[s], bits, g=1, terms))^2, each
 * elementwise op rounded to fp32 as torch does, the sum in fp64; *argmin = index
 * of the first minimum of (float)errs.  All pointers are device pointers;
 * (errs: nsf doubles).  Two launches instead of 2048 launches + 2048 host syncs.
 */
int tq_mse_profile(const float *hist, const float *x, int nbins,
                   const float *sfs, int nsf, int bits, int terms,
                   double *errs, int *argmin, void *stream);
/* the same sweep with tr(x[b]) in the given TQ_ENC_* encoding */
int tq_mse_profile_enc(const float *hist, const float *x, int nbins,
                       const float *sfs, int nsf, int bits, int terms, int encoding,
                       double *errs, int *argmin, void *stream);

/*
 * *count += sum_i len(hese(int(w[i] / sf)))  (tr_layer.py:57-63, the per-element
 * Python loop of compute_compressed_hese); count is a device uint64.
 */
int tq_hese_term_count(const void *w, int dtype, int64_t n, float sf, unsigned flags,
                       unsigned long long *count, void *stream);
/* the same count for any TQ_ENC_* encoding: *count += sum_i (number of terms of int(w[i] / sf)) */
int tq_term_count(const void *w, int dtype, int64_t n, float sf, int encoding, unsigned flags,
                  unsigned long long *count, void *stream);

/*
 * Convolution on term codes with tcgen05 tensor cores (replaces the cuDNN fp32 conv under
 * TRConv2dLayer.forward, tr_layer.py:124-126, computed on the integer codes instead of the
 * dequantised values):
 *     acc[n,ho,wo,co] = sum_{r,s,ci} act[n, ho*stride+r-pad, wo*stride+s-pad, ci] * wgt[r*S+s, co, ci]     (int32, exact)
 *     out             = float(acc) * scale (+ bias[co])
 * act  fp16 NHWC [N,H,W,C] holding integer codes (TQ_F16C), C % 8 == 0
 * wgt  fp16 [R*S][Cout][C] holding integer codes, Cout % 4 == 0
 * out  fp32 NHWC [N,Ho,Wo,Cout]; bias fp32 [Cout] or NULL; scale = sf_x * sf_w.  groups = 1, dilation = 1.
 *
 * EXACTNESS CONTRACT (kind::f16 MMAs accumulate in fp32, exact for integers below 2^24).  The K dimension is
 * cut into acc_groups chunks of (C / 64) / acc_groups consecutive 64-channel blocks (all taps); every chunk
 * accumulates in its own tensor-memory accumulator and the epilogue adds the chunks in int32.  The result is
 * the exact int32 accumulator if, for every output channel and every chunk,
 *     act_max * max(sum of positive weight codes, sum of negative weight codes) < 2^24
 * (non-negative activations <= act_max; for signed activations use the sum of |w|): no partial sum of such a
 * chunk can leave the exact range whatever the activations are.  tq_conv_weight_l1() returns those sums; the
 * caller passes the smallest acc_groups that satisfies the bound (acc_groups must divide C / 64 and
 * acc_groups * min(128, roundup64(Cout)) <= 512 tensor-memory columns).  Weights that cannot be proven go to
 * tq_conv2d_planes_i8(), which is exact for every input.  The Python layer (conv_codes.plan_weight) does this
 * per layer at pack time and refuses to run an unproven layer on this entry point.
 */
int tq_conv2d_codes_f16(const void *act, const void *wgt, const float *bias, float *out,
                        int N, int H, int W, int C, int Cout, int R, int S, int stride, int pad,
                        float scale, int acc_groups, void *stream);

/*
 * Same contraction with the layer's whole tail fused into the epilogue (verilog/systolic_dla_top.v
 * pipeline order: accumulate -> ReLU/requantise -> encode -> truncate; tr_layer.py:124-126 plus the
 * BatchNorm / residual / ReLU that follow a conv in the CNNs of cnn_models/):
 *     t = float(acc) * scale (+ bias[co]);  t = fma(t, bn_a[co], bn_b[co]);  t += residual[n,ho,wo,co];
 *     t = max(t, 0) if relu (relu = 2: ReLU6, t = min(max(t, 0), 6));  out_f32 = t;
 *     out_codes = term code of t under the consumer's quantiser
 *     (next_sf, next_bits <= 10, next_terms; g = 1, HESE; _enc: next_enc) stored as fp16 NHWC.
 * Every step is optional (NULL pointer / relu = 0); at least one of out_f32, out_codes is given.
 * Every step is one IEEE fp32 operation in this order, so the result is reproducible bit for bit on a CPU
 * (oracle/fused_emul.py).  Outputs are written with TMA stores from swizzled shared memory (fully coalesced,
 * clipped at the tensor edge).
 */
int tq_conv2d_codes_fused(const void *act, const void *wgt, float *out_f32, void *out_codes,
                          const float *bias, const float *bn_a, const float *bn_b, const float *residual,
                          int N, int H, int W, int C, int Cout, int R, int S, int stride, int pad,
                          float scale, int relu, float next_sf, int next_bits, int next_terms,
                          int acc_groups, void *stream);
int tq_conv2d_codes_fused_enc(const void *act, const void *wgt, float *out_f32, void *out_codes,
                              const float *bias, const float *bn_a, const float *bn_b, const float *residual,
                              int N, int H, int W, int C, int Cout, int R, int S, int stride, int pad,
                              float scale, int relu, float next_sf, int next_bits, int next_terms, int next_enc,
                              int acc_groups, void *stream);

/*
 * The same fused conv on SIGNED 8-BIT OPERAND PLANES with tcgen05.mma kind::i8 and int32 accumulators in
 * tensor memory: exact for every input (the north star's "tcgen05 int8 implicit-GEMM ... int32 accumulators").
 * A code v (|v| <= 2047) is split as v = 16 * hi + lo with hi = v >> 4 (arithmetic) and lo = v & 15; an operand
 * whose codes all fit -128..127 is a single plane.
 *   act_planes  int8 [planes_a][N][H][W][C]   (plane 0 = hi or the code itself, plane 1 = lo), C % 16 == 0
 *   wgt_planes  int8 [planes_w][R*S][Cout][C]
 * Plane pair (pa, pw) accumulates into TMEM accumulator pa + pw; the epilogue recombines them by Horner's rule
 * with the plane shift in int32 and continues exactly as tq_conv2d_codes_fused.  act_max / wgt_max are the caller's
 * bounds on |code| (2^bits by construction of the term codes); C * R * S * act_max * wgt_max < 2^31 is required.
 * tq_codes_to_planes() produces the planes from fp16 codes.  The output codes are HESE; _enc: next_enc.
 */
int tq_conv2d_planes_i8(const void *act_planes, const void *wgt_planes, int planes_a, int planes_w,
                        float *out_f32, void *out_codes, const float *bias, const float *bn_a,
                        const float *bn_b, const float *residual, int N, int H, int W, int C, int Cout,
                        int R, int S, int stride, int pad, float scale, int relu, float next_sf,
                        int next_bits, int next_terms, int act_max, int wgt_max, void *stream);
int tq_conv2d_planes_i8_enc(const void *act_planes, const void *wgt_planes, int planes_a, int planes_w,
                            float *out_f32, void *out_codes, const float *bias, const float *bn_a,
                            const float *bn_b, const float *residual, int N, int H, int W, int C, int Cout,
                            int R, int S, int stride, int pad, float scale, int relu, float next_sf,
                            int next_bits, int next_terms, int next_enc, int act_max, int wgt_max, void *stream);

/* fp16 integer codes (n elements, n % 8 == 0) -> `planes` signed 8-bit planes of n bytes each, plane p at
 * planes_s8 + p * n.  planes = 1 stores the code itself; a value that does not fit sets *overflow (device int,
 * may be NULL) to 1. */
int tq_codes_to_planes(const void *codes_f16, void *planes_s8, int64_t n, int planes, int *overflow, void *stream);

/* Static accumulator bound of a packed weight (see the exactness contract above): for every output channel co
 * and every 64-channel block kb, pos[co * kcb + kb] = sum of the positive codes of wgt[:, co, 64 kb .. 64 kb + 63]
 * over all taps and neg[...] = minus the sum of the negative ones (kcb = ceil(C / 64); device int64 arrays). */
int tq_conv_weight_l1(const void *wgt_f16, int RS, int Cout, int C, long long *pos, long long *neg, void *stream);

/*
 * Fused tail of the unquantised stem (torchvision ResNet: bn1 -> relu -> maxpool(3, 2, 1), then
 * the first wrapped conv's LinearQuantize, tr_layer.py:96-99): x fp32 NHWC [N,H,W,C] ->
 * out fp32 NHWC [N,Ho,Wo,C] = maxpool3x3s2p1(relu(fma(x, bn_a, bn_b))) and, if out_codes != NULL,
 * the fp16 term codes of `out` under (next_sf, next_bits <= 11, next_terms; HESE, _enc: next_enc).  C % 4 == 0.
 */
int tq_bn_relu_maxpool_encode(const float *x, const float *bn_a, const float *bn_b, float *out,
                              void *out_codes, int N, int H, int W, int C, int relu,
                              float next_sf, int next_bits, int next_terms, void *stream);
int tq_bn_relu_maxpool_encode_enc(const float *x, const float *bn_a, const float *bn_b, float *out,
                                  void *out_codes, int N, int H, int W, int C, int relu,
                                  float next_sf, int next_bits, int next_terms, int next_enc, void *stream);

/*
 * The unquantised stem conv of the CNNs (7x7, stride 2, pad 3, 3 input channels, no bias;
 * torchvision resnet `conv1`, left in fp32 by the reference: cnn_models/__init__.py:34-36) on the
 * tensor-core kernel with fp32-level accuracy (hi/lo fp16 operand pairs, fp32 accumulation).
 *   x          fp32 NHWC [N, H, W, 3] (H, W even)
 *   x2_scratch 2 * N * (H/2+3) * (W/2+3) * 16 fp16 of scratch (folded hi / lo image planes)
 *   w2         fp16 [4][128][64]: tile R = filter row R of the 8x8-padded kernel folded 2x2 (64 = 4 taps x (2x2x4)
 *              folded channels); rows 0..Cout-1 of a tile hold the fp16 hi plane of the weights, rows 64..64+Cout-1
 *              the lo plane (w = hi + lo), the rest zeros (conv_codes.pack_stem_weight builds it); Cout <= 64
 *   out        fp32 NHWC [N, H/2, W/2, Cout]
 */
int tq_stem_conv7x7s2(const float *x, void *x2_scratch, const void *w2, float *out,
                      int N, int H, int W, int Cout, void *stream);
/* Same with the image dtype given (TQ_F32, TQ_BF16 or TQ_F16).  16-bit images are exact in the fp16 hi
 * plane (down to 2^-14; smaller magnitudes lose < 2^-25 absolute), so the lo image plane and its MMAs are
 * skipped: x2_scratch then needs N * (H/2+3) * (W/2+3) * 16 fp16. */
int tq_stem_conv7x7s2_dt(const void *x, int x_dtype, void *x2_scratch, const void *w2, float *out,
                         int N, int H, int W, int Cout, void *stream);

/*
 * The same conv on uint8 NHWC images [N][H][W][3] with ToTensor + Normalize folded in: the value convolved is
 * bf16(((u8 / 255) - mean3[c]) / std3[c]) -- what tq_u8_normalize_bf16 writes, each step one fp32 IEEE operation as
 * torchvision computes it on the host (util.py:12-27) -- so a batch crosses PCIe as one byte per value and no
 * normalised image is ever materialised.  mean3 / std3 are HOST arrays of 3 floats.
 */
int tq_stem_conv7x7s2_u8(const void *x_u8, const float *mean3, const float *std3, void *x2_scratch, const void *w2,
                         float *out, int N, int H, int W, int Cout, void *stream);
/*
 * The whole unquantised stem in one tensor-core kernel: conv 7x7/s2/p3 -> per-channel affine (BatchNorm) ->
 * ReLU (if relu) -> max-pool 3x3/s2/p1 -> fp32 NHWC [N, Hp, Wp, Cout] (Hp = (H/2 - 1)/2 + 1) and, if out_codes,
 * the fp16 term codes of that tensor for the first wrapped conv's quantiser (tr_layer.py:96-99; HESE, _enc: next_enc).  Each tile
 * computes the (2P+1) x (2Q+1) conv pixels under P x Q pooled pixels, so the conv output (822 MB at batch 256)
 * never reaches HBM.  Same values as tq_stem_conv7x7s2_dt followed by tq_bn_relu_maxpool_encode.
 * CONTRACT: bn_a >= 0.  The pooling takes the window maximum of the raw conv sums and applies the affine once
 * per pooled value; a channel with a negative slope is handled by the caller folding sign(bn_a) into that
 * channel's weights and passing |bn_a| (conv_codes.pack_stem_weight(w, bn_a) / stem_conv_pool do this): negation
 * of a channel's weights negates its sums exactly, and max_i fma(x_i, a, b) = fma(max_i(sign(a) x_i), |a|, b).
 */
int tq_stem_conv7x7s2_pool(const void *x, int x_dtype, void *x2_scratch, const void *w2,
                           const float *bn_a, const float *bn_b, int relu, float *out, void *out_codes,
                           int N, int H, int W, int Cout, float next_sf, int next_bits, int next_terms,
                           void *stream);
int tq_stem_conv7x7s2_pool_enc(const void *x, int x_dtype, void *x2_scratch, const void *w2,
                               const float *bn_a, const float *bn_b, int relu, float *out, void *out_codes,
                               int N, int H, int W, int Cout, float next_sf, int next_bits, int next_terms,
                               int next_enc, void *stream);

/*
 * The stem in two passes that split the 3x3/s2/p1 max-pool by axis, so that only half of the conv map crosses HBM:
 *   tq_stem_conv7x7s2_rowmax (x_dtype TQ_F32, TQ_BF16 or TQ_F16) / tq_stem_conv7x7s2_u8_rowmax (uint8 images as in
 *   tq_stem_conv7x7s2_u8) write out = fp32 NHWC [N, H/2, Wp, Cout] (Wp = (W/2 - 1)/2 + 1), the RAW conv sums maxed
 *   over conv columns 2q-1, 2q, 2q+1 of each conv row (columns outside the map excluded);
 *   tq_bn_relu_maxpool_encode_rowmax takes that tensor as x [N, H, W, C] (H = conv rows, W = pooled columns,
 *   C % 4 == 0) and writes out fp32 NHWC [N, (H - 1)/2 + 1, W, C] = relu(fma(max over rows 2p-1, 2p, 2p+1, bn_a,
 *   bn_b)) and its fp16 codes as tq_bn_relu_maxpool_encode does.
 * Together: the same values as tq_stem_conv7x7s2_dt followed by tq_bn_relu_maxpool_encode.
 * CONTRACT: as for tq_stem_conv7x7s2_pool, the max is taken before the affine, so bn_a >= 0: the caller folds
 * sign(bn_a) into the channel's weights and passes |bn_a| (conv_codes.stem_pool_operands).
 */
int tq_stem_conv7x7s2_rowmax(const void *x, int x_dtype, void *x2_scratch, const void *w2, float *out,
                             int N, int H, int W, int Cout, void *stream);
int tq_stem_conv7x7s2_u8_rowmax(const void *x_u8, const float *mean3, const float *std3, void *x2_scratch,
                                const void *w2, float *out, int N, int H, int W, int Cout, void *stream);
int tq_bn_relu_maxpool_encode_rowmax(const float *x, const float *bn_a, const float *bn_b, float *out,
                                     void *out_codes, int N, int H, int W, int C, int relu,
                                     float next_sf, int next_bits, int next_terms, void *stream);
int tq_bn_relu_maxpool_encode_rowmax_enc(const float *x, const float *bn_a, const float *bn_b, float *out,
                                         void *out_codes, int N, int H, int W, int C, int relu,
                                         float next_sf, int next_bits, int next_terms, int next_enc, void *stream);

/*
 * Depthwise 3x3 conv (pad 1, stride 1 or 2) on term codes, the memory-bound layer of the depthwise CNNs
 * (BASELINE.json configs[3]; wrapped by the reference with the (16, 1, 16) weight setting, cnn_models/__init__.py:52-65,
 * and run as TR encode -> cuDNN fp32 conv -> BatchNorm -> ReLU6, tr_layer.py:124-126):
 *     acc[n,ho,wo,c] = sum_{r,s} act[n, ho*stride+r-1, wo*stride+s-1, c] * wgt[r*3+s, c]        (int32, exact)
 *     t = float(acc) * scale (+ bias[c]);  t = fma(t, bn_a[c], bn_b[c]);  relu: 0 none, 1 ReLU, 2 ReLU6;
 *     out_f32 = t and / or out_codes = fp16 term code of t under (next_sf, next_bits <= 11, next_terms), g = 1, HESE
 *     (_enc: next_enc).
 * act fp16 NHWC [N,H,W,C] integer codes, wgt int32 [9][C] integer codes (|a| <= 2^11, |w| <= 2^16), C % 8 == 0.
 * act_unsigned != 0: the caller guarantees 0 <= act <= 1023 (the output of a ReLU under a quantiser of <= 9 bits), which
 * lets the kernel extract the integers without conversion instructions.  Input tiles (with their zero halo) are staged
 * into shared memory by TMA.  Algorithmic bytes: 2 B read + 2 B (codes) / 4 B (fp32) written per element.
 */
int tq_depthwise3x3_codes(const void *act_codes, const int32_t *wgt_codes, float *out_f32, void *out_codes,
                          const float *bias, const float *bn_a, const float *bn_b, int N, int H, int W, int C,
                          int stride, float scale, int relu, int act_unsigned, float next_sf, int next_bits,
                          int next_terms, void *stream);
int tq_depthwise3x3_codes_enc(const void *act_codes, const int32_t *wgt_codes, float *out_f32, void *out_codes,
                              const float *bias, const float *bn_a, const float *bn_b, int N, int H, int W, int C,
                              int stride, float scale, int relu, int act_unsigned, float next_sf, int next_bits,
                              int next_terms, int next_enc, void *stream);

/*
 * Tail of an unwrapped conv (the first conv of every CNN, cnn_models/__init__.py:34-36) fused with the first wrapped
 * layer's LinearQuantize (tr_layer.py:96-99): x fp32 [npix][C] -> + bias (the conv's own bias, one fp32 add, when the
 * conv ran without it; may be NULL) -> fma(x, bn_a, bn_b) -> activation (relu as above) -> out_f32 and / or fp16 term
 * codes (HESE; _enc: next_enc).  C % 4 == 0.
 */
int tq_bn_act_encode(const float *x, const float *bias, const float *bn_a, const float *bn_b, float *out_f32,
                     void *out_codes, int64_t npix, int C, int relu, float next_sf, int next_bits, int next_terms,
                     void *stream);
int tq_bn_act_encode_enc(const float *x, const float *bias, const float *bn_a, const float *bn_b, float *out_f32,
                         void *out_codes, int64_t npix, int C, int relu, float next_sf, int next_bits, int next_terms,
                         int next_enc, void *stream);

/*
 * The unwrapped first conv of the VGG-style / depthwise CNNs (cnn_models/__init__.py:34-36: nn.Conv2d(3, Cout, 3, stride,
 * padding=1), Cout 32 or 64, stride 1 or 2) in fp32 on the CUDA cores, fused with what follows it: + bias, BatchNorm
 * affine, ReLU / ReLU6 and the first wrapped layer's LinearQuantize (tr_layer.py:96-99).  x fp32 NHWC [N][H][W][3],
 * wgt fp32 [3][3][3][Cout] (filter row, filter column, input channel, output channel); sums run in that order, one
 * fmaf per term, bias added after the sum.  out_f32 and / or fp16 term codes (HESE; _enc: next_enc), NHWC.  An fp32
 * conv: it equals cuDNN's up to the summation order, not bit for bit.
 */
int tq_first_conv3x3_fused(const float *x, const float *wgt, const float *bias, const float *bn_a, const float *bn_b,
                           float *out_f32, void *out_codes, int N, int H, int W, int Cout, int stride, int relu,
                           float next_sf, int next_bits, int next_terms, void *stream);
int tq_first_conv3x3_fused_enc(const float *x, const float *wgt, const float *bias, const float *bn_a, const float *bn_b,
                               float *out_f32, void *out_codes, int N, int H, int W, int Cout, int stride, int relu,
                               float next_sf, int next_bits, int next_terms, int next_enc, void *stream);

/*
 * nn.MaxPool2d(k, stride, pad) (floor mode, no dilation) on an fp16 NHWC tensor: the term codes between the convs of
 * the VGG-style stacks (cnn_models/__init__.py wraps the convs, the pools stay: for g = 1 the truncated code is monotone
 * in the non-negative value, so pooling codes == encoding pooled values).  C % 8 == 0.
 */
int tq_maxpool2d_f16(const void *x_f16, void *y_f16, int N, int H, int W, int C, int k, int stride, int pad,
                     void *stream);

/*
 * uint8 NHWC images [npix][3] -> normalised bf16 [npix][3]: ((u8 / 255) - mean[c]) / std[c], each step one fp32 IEEE
 * operation as torchvision's ToTensor + Normalize compute it on the host (util.py:12-27), then rounded to bf16 -- the
 * image dtype of the fused engine.  mean3 / std3 are HOST arrays of 3 floats.  npix % 4 == 0.
 */
int tq_u8_normalize_bf16(const void *x_u8, void *y_bf16, int64_t npix, const float *mean3, const float *std3,
                         void *stream);

/*
 * The recurrence of one unidirectional LSTM layer (nn.LSTM, torch gate order i, f, g, o), all T steps in ONE launch of a
 * persistent cooperative kernel (the step-wise loop tr_layer.py:174-195 runs as cuDNN calls, or as ~11 torch kernels per step):
 *     gates = (gin[t] + bias) + h_{t-1} . w_hh^T;  c_t = sig(f) * c_{t-1} + sig(i) * tanh(g);  h_t = sig(o) * tanh(c_t)
 *   gin  fp32 [T][B][4H], the input projection of every step (W_ih x_t, without bias)
 *   bias fp32 [4H] (b_ih + b_hh) or NULL;  w_hh fp32 [4H][H] row-major (nn.LSTM's weight_hh_l*);  h0, c0 fp32 [B][H]
 *   y    fp32 [T][B][H] = h_t;  hn, cn fp32 [B][H] = h_T, c_T
 * fp32 FFMA with one fixed summation order per dot product (bit-identical from run to run), sig(x) = 1 / (1 + expf(-x)),
 * accurate expf / tanhf.  Each CTA keeps the 4 gate rows of ceil(H / SMs) hidden units in shared memory; H is refused
 * (TQ_ERR_UNSUPPORTED) when those rows and one hidden row exceed the device's opt-in shared memory per block (B200:
 * H <= 1404).  All pointers 4-byte aligned, no output may alias an input; T, B, H >= 1.  The grid-wide barrier between steps
 * relies on a cooperative launch, so the whole grid is resident by construction.
 */
int tq_lstm_recurrence(const float *gin, const float *bias, const float *w_hh, const float *h0, const float *c0,
                       float *y, float *hn, float *cn, int T, int B, int H, void *stream);

/*
 * The same persistent recurrence for the other cells of nn.GRU / nn.RNN (one unidirectional layer, torch's gate order
 * and formulas), the same kernel template, numerics, layout and refusals as tq_lstm_recurrence:
 *   GRU (gates r, z, n):  gin fp32 [T][B][3H] = W_ih x_t + b_ih;  b_hh fp32 [3H] or NULL;  w_hh fp32 [3H][H]
 *       r = sig(gin_r + b_hr + W_hr h),  z = sig(gin_z + b_hz + W_hz h),  n = tanh(gin_n + r * (W_hn h + b_hn)),
 *       h_t = n + z * (h_{t-1} - n)
 *   RNN:  gin fp32 [T][B][H] = W_ih x_t;  bias fp32 [H] (b_ih + b_hh) or NULL;  w_hh fp32 [H][H]
 *       h_t = act(gin + bias + W_hh h),  act = relu ? ReLU (a NaN stays NaN, as torch.relu) : tanh
 *   h0 fp32 [B][H];  y fp32 [T][B][H] = h_t;  hn fp32 [B][H] = h_T
 * Each CTA keeps the G gate rows (G = 3 / 1) of ceil(H / SMs) units in shared memory, so the bound on H grows as G
 * shrinks (B200: GRU H <= 1628, RNN H <= 2812).  TQ_ERR_INVALID for NULL or misaligned pointers, T, B or H below 1 and
 * B * G * H above 2^31 - 1; TQ_ERR_UNSUPPORTED (the message names the largest H) above the bound; all before any launch.
 */
int tq_gru_recurrence(const float *gin, const float *b_hh, const float *w_hh, const float *h0, float *y, float *hn,
                      int T, int B, int H, void *stream);
int tq_rnn_recurrence(const float *gin, const float *bias, const float *w_hh, const float *h0, float *y, float *hn,
                      int T, int B, int H, int relu, void *stream);

/* Largest H the recurrence of a cell with `gates` gate rows per unit (4 LSTM, 3 GRU, 1 RNN) takes on the current
 * device; -1 (TQ_ERR_INVALID / TQ_ERR_CUDA in tq_last_error) for another gate count or an unreadable device. */
int tq_recurrence_max_hidden(int gates);

/*
 * Per-row negative log-likelihood of a target class, read straight from the logits (one pass, no log-probability tensor):
 *     loss[r] = logsumexp(logits[r][0:cols]) - logits[r][targets[r]]  = -log_softmax(logits[r])[targets[r]]
 *   logits  fp32 [rows][ld] (row stride ld >= cols elements: a padded GEMM output is read in place, its pad ignored)
 *   targets int64 [rows];  loss fp32 [rows]
 * fp32 with accurate expf / logf and one fixed summation order per row (bit-identical from run to run and under graph
 * replay).  Special values as torch.log_softmax + nll_loss: -inf entries add 0, a NaN or +inf in the row and an all -inf
 * row give NaN.  A target outside [0, cols) gives a NaN loss for its row (no fault).  logits and loss 4-byte aligned,
 * targets 8-byte aligned, rows, cols >= 1, ld >= cols, rows * ld * 4 bytes within int64; otherwise TQ_ERR_INVALID before
 * any launch.
 */
int tq_log_softmax_nll(const float *logits, int64_t rows, int64_t cols, int64_t ld, const int64_t *targets, float *loss,
                       void *stream);

/*
 * The same per-row loss straight from a linear layer on term codes, without writing its output (the language model's
 * decoder): logits[r][c] = float(exact int32 accumulator) * scale (+ bias[c]), bit for bit the values
 * tq_conv2d_codes_fused(_enc) / tq_conv2d_planes_i8(_enc) write for the 1 x M image (N = 1, H = 1, W = M, C = K,
 * Cout = Op, 1x1 filter, no BatchNorm / residual / ReLU), and
 *     loss[r] = logsumexp(logits[r][0:V]) - logits[r][targets[r]]
 *   x_codes  fp16 [M][K] codes (K % 8 == 0) / x_planes int8 [planes_a][M][K] (K % 16 == 0)
 *   wgt      fp16 [1][Op][K] packed weight codes / wgt_planes int8 [planes_w][1][Op][K]; Op % 4 == 0
 *   bias     fp32 [Op] or NULL; rows [V, Op) of the weight and bias are padding, never part of any loss
 *   targets  int64 [M];  loss fp32 [M]
 *   workspace, workspace_bytes >= tq_linear_nll_workspace_bytes(M, Op): the caller's, per call (under stream capture
 *   it comes from the graph's memory pool like every other buffer; the library keeps none)
 * acc_groups, planes, act_max, wgt_max: as the conv entry points (the exactness contract above).  The decoder's
 * epilogue keeps, per row and 32-column chunk, a running (max, sum exp(x - max)) over the live columns c < V with
 * ex2.approx of fl(fl(x - max) * log2 e), writes one pair per row and column slice of an N tile (no fp32 tile, no codes,
 * no TMA store) and the target logit, and a second kernel rescales the pairs to the row maximum and adds them in fp64
 * in a fixed order.  The result is within 4e-6 * max(|ref|, 1) of an fp64 logsumexp - gather of the same logits and
 * bit-identical from run to run, for any grid and under graph replay.  Special values and out-of-range targets as
 * tq_log_softmax_nll (NaN, no fault).  TQ_ERR_INVALID before any launch: NULL or misaligned pointers (operands and bias
 * 16-byte, targets 8-byte, loss 4-byte, workspace 16-byte aligned), M < 1, V < 1, V > Op, sizes that overflow int64,
 * a workspace that is too small; TQ_ERR_UNSUPPORTED for a plan outside the streaming single-CTA conv variants.
 */
int64_t tq_linear_nll_workspace_bytes(int64_t M, int64_t Op);   /* -1 for M < 1, Op < 1 or sizes beyond int64 */
int tq_linear_codes_nll(const void *x_codes, const void *wgt, int64_t M, int K, int Op, int V, float scale,
                        const float *bias, int acc_groups, const int64_t *targets, float *loss, void *workspace,
                        int64_t workspace_bytes, void *stream);
int tq_linear_planes_i8_nll(const void *x_planes, const void *wgt_planes, int planes_a, int planes_w, int64_t M, int K,
                            int Op, int V, float scale, const float *bias, int act_max, int wgt_max,
                            const int64_t *targets, float *loss, void *workspace, int64_t workspace_bytes, void *stream);

/*
 * Device self-test: quantises n pseudo-random (a, sf) pairs (sf in [2^-30, 2^30], a over all
 * non-negative floats and the quantiser's rounding boundaries) with the hoisted-reciprocal
 * divide and with div.rn.f32 and adds the number of disagreements to *mismatch (device).
 */
int tq_selftest_division(uint64_t n, uint32_t seed, unsigned long long *mismatch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TQ_B200_H */
