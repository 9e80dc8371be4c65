"""CPU emulation of the FUSED arithmetic (csrc/tq_gemm.cu epilogue), bit for bit.

TEST INFRASTRUCTURE ONLY (see oracle/tq_oracle.py).  The fused engine replaces, per wrapped conv, the
reference's  TR encode -> fp32 conv -> BatchNorm -> (+ residual) -> ReLU  (tr_layer.py:124-126 inside a
torchvision BasicBlock) by ONE kernel whose every step is a single IEEE fp32 operation on an exact integer
accumulator.  That chain is reproducible on a CPU without any tolerance, which no float convolution is:

    acc   = sum_k a_k * w_k            exact integer (here: fp64 convolution of integer tensors, < 2^53)
    t     = fl32(acc) * scale          RN conversion (exact below 2^24), RN multiply;  scale = fl32(sf_x) * fl32(sf_w)
    t     = t + bias[co]               RN add                     (if the conv has a bias)
    t     = fmaf(t, bn_a[co], bn_b[co])  one rounding             (if a BatchNorm follows)
    t     = t + residual               RN add                     (block output)
    t     = fmaxf(t, 0)                (if a ReLU follows: NaN -> +0, -0 -> +0, see relu_f32())
    codes = tr(t; next_sf, bits, g=1, terms)   oracle.tr: the reference's quantise / HESE / truncate

`run_resnet_chain` chains this over every BasicBlock of a ResNet exactly as fused.FusedResNet does.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import tq_oracle as O


def encode(x_nhwc, quant):
    """fp32 [N,H,W,C] -> int32 term codes under quant = (sf, bits, terms), g = 1 (tr_layer.py:96-99)."""
    sf, bits, terms = quant
    x = np.ascontiguousarray(x_nhwc, dtype=np.float32)
    _, codes = O.tr(x.reshape(1, -1, 1, 1), sf, bits, 1, terms, return_codes=True)
    return codes.reshape(x.shape)


def conv_exact(codes_nhwc, w_codes, ks, stride, pad):
    """Exact integer convolution: int codes [N,H,W,C] x [R*S, Cout, C] -> float64 [N,Ho,Wo,Cout] holding integers."""
    R, S = ks
    RS, Cout, C = w_codes.shape
    w = torch.from_numpy(np.asarray(w_codes, dtype=np.float64)).view(R, S, Cout, C).permute(2, 3, 0, 1).contiguous()
    a = torch.from_numpy(np.asarray(codes_nhwc, dtype=np.float64)).permute(0, 3, 1, 2).contiguous()
    acc = F.conv2d(a, w, None, stride, pad).permute(0, 2, 3, 1).contiguous().numpy()
    assert float(np.abs(acc).max(initial=0.0)) < 2.0 ** 31, "int32 accumulator overflow"
    return acc


def fused_conv(codes_nhwc, conv, residual=None, relu=False, next_quant=None):
    """One fused conv.  conv: dict(w=[R*S,Cout,C] int codes, ks, stride, pad, scale (python float of an fp32),
    bias=None|[Cout], bn=None|(a, b)).  Returns (t fp32 [N,Ho,Wo,Cout], codes int32 or None)."""
    acc = conv_exact(codes_nhwc, conv["w"], conv["ks"], conv["stride"], conv["pad"])
    t = acc.astype(np.float32) * np.float32(conv["scale"])
    if conv.get("bias") is not None:
        t = t + np.asarray(conv["bias"], dtype=np.float32)
    if conv.get("bn") is not None:
        t = O.fma_channels(t, conv["bn"][0], conv["bn"][1])
    if residual is not None:
        t = t + np.asarray(residual, dtype=np.float32)
    if relu:
        t = relu_f32(t)
    t = np.ascontiguousarray(t, dtype=np.float32)
    return t, (encode(t, next_quant) if next_quant is not None else None)


def relu_f32(t):
    """fmaxf(t, 0) as the fused epilogues compute it (DESIGN.md section 3): an IEEE maxNum drops a NaN operand, so
    NaN -> +0 (where torch.relu keeps the NaN), and -0 -> +0."""
    t = np.asarray(t, dtype=np.float32)
    return np.where(t > 0, t, np.float32(0.0)).astype(np.float32)


def maxpool_f32_nan_dropped(x_nhwc, k, stride, pad):
    """The fused max-pools on an fp32 NHWC map: a running fmaxf from -inf, so a NaN is ignored and a window holding
    only NaN (or nothing but padding) yields -inf, where torch's max_pool2d propagates the NaN."""
    x = np.asarray(x_nhwc, dtype=np.float32)
    x = np.where(np.isnan(x), np.float32(-np.inf), x)
    return maxpool_nhwc(x, k, stride, pad).astype(np.float32)


def run_resnet_chain(blocks, stem_out):
    """blocks: list of (conv1, conv2, down-or-None) dicts, each with a 'quant' = (sf, bits, terms) of its input
    quantiser; stem_out: fp32 [N,H,W,C] -- the tensor that reaches layer1 (after the unquantised stem, which is
    outside the TQ path: cnn_models/__init__.py:34-36).  Returns the fp32 [N,h,w,C'] output of the last block."""
    cur = np.ascontiguousarray(stem_out, dtype=np.float32)
    for c1, c2, down in blocks:
        identity = cur if down is None else fused_conv(encode(cur, down["quant"]), down)[0]
        _, mid = fused_conv(encode(cur, c1["quant"]), c1, relu=True, next_quant=c2["quant"])
        cur, _ = fused_conv(mid, c2, residual=identity, relu=True)
    return cur


def _act(t, relu):
    if relu:
        t = relu_f32(t)
    if relu in ("relu6", 2):
        t = np.minimum(t, np.float32(6.0))
    return t


def fused_conv_act(codes_nhwc, conv, residual=None, relu=False, next_quant=None):
    """fused_conv with the activation given as False / True / 'relu6' (the depthwise CNNs clamp at 6)."""
    acc = conv_exact(codes_nhwc, conv["w"], conv["ks"], conv["stride"], conv["pad"])
    t = acc.astype(np.float32) * np.float32(conv["scale"])
    if conv.get("bias") is not None:
        t = t + np.asarray(conv["bias"], dtype=np.float32)
    if conv.get("bn") is not None:
        t = O.fma_channels(t, conv["bn"][0], conv["bn"][1])
    if residual is not None:
        t = t + np.asarray(residual, dtype=np.float32)
    t = np.ascontiguousarray(_act(t, relu), dtype=np.float32)
    return t, (encode(t, next_quant) if next_quant is not None else None)


def depthwise_exact(codes_nhwc, w9c, stride):
    """Exact depthwise 3x3 / pad 1 conv: int codes [N,H,W,C] x int [9, C] -> float64 [N,Ho,Wo,C] holding integers."""
    C = w9c.shape[1]
    w = torch.from_numpy(np.asarray(w9c, dtype=np.float64)).t().contiguous().view(C, 1, 3, 3)
    a = torch.from_numpy(np.asarray(codes_nhwc, dtype=np.float64)).permute(0, 3, 1, 2).contiguous()
    acc = F.conv2d(a, w, None, stride, 1, 1, C).permute(0, 2, 3, 1).contiguous().numpy()
    assert float(np.abs(acc).max(initial=0.0)) < 2.0 ** 31
    return acc


def fused_depthwise(codes_nhwc, dw, relu=False, next_quant=None):
    """tq_depthwise3x3_codes on the CPU: exact int32 accumulator -> fl32 * scale (+ bias) -> fmaf BN -> activation."""
    acc = depthwise_exact(codes_nhwc, dw["w"], dw["stride"])
    t = acc.astype(np.float32) * np.float32(dw["scale"])
    if dw.get("bias") is not None:
        t = t + np.asarray(dw["bias"], dtype=np.float32)
    if dw.get("bn") is not None:
        t = O.fma_channels(t, dw["bn"][0], dw["bn"][1])
    t = np.ascontiguousarray(_act(t, relu), dtype=np.float32)
    return t, (encode(t, next_quant) if next_quant is not None else None)


def run_mobilenet_chain(desc, stem_codes):
    """desc = fused.FusedMobileNet.chain_description(); stem_codes: int codes [N,H,W,C] reaching the first block (the
    unwrapped stem conv + BN + ReLU6 + first encode are outside the chain).  Returns the fp32 output of the last 1x1
    conv (+ BN + ReLU6), i.e. the tensor the average pool reads."""
    codes = np.asarray(stem_codes).astype(np.int32)
    cur = None
    blocks = desc["blocks"]
    for i, (expand, dw, proj, use_res) in enumerate(blocks):
        h = codes
        if expand is not None:
            _, h = fused_conv_act(h, expand, relu="relu6", next_quant=dw["quant"])
        _, h = fused_depthwise(h, dw, relu="relu6", next_quant=proj["quant"])
        nxt = blocks[i + 1] if i + 1 < len(blocks) else None
        nq = (nxt[0] or nxt[1])["quant"] if nxt is not None else desc["last"]["quant"]
        cur, codes = fused_conv_act(h, proj, residual=cur if use_res else None, relu=False, next_quant=nq)
    out, _ = fused_conv_act(codes, desc["last"], relu="relu6")
    return out


def maxpool_nhwc(x, k, stride, pad):
    """nn.MaxPool2d(k, stride, pad) (floor mode) on an NHWC array (integer codes or fp32): -inf padding."""
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).permute(0, 3, 1, 2)
    return F.max_pool2d(t, k, stride, pad).permute(0, 2, 3, 1).contiguous().numpy()


def run_vgg_chain(stages, stem_codes):
    """stages = fused.FusedVGG.chain_description(); stem_codes: int codes [N,H,W,C] reaching the first wrapped conv (the
    unwrapped first conv + BN + ReLU + first encode are outside the chain).  Every conv is the exact integer conv of the
    codes -> fl32 * scale (+ bias) -> fmaf BN -> ReLU -> the next quantiser's codes; max-pools act on the codes
    (monotone for g = 1) or, after the last conv, on the fp32 map.  Returns the fp32 map the average pool reads."""
    codes = np.asarray(stem_codes).astype(np.int32)
    out = None
    for i, st in enumerate(stages):
        if st[0] == "conv":
            _, conv, relu = st
            nxt = next((s[1]["quant"] for s in stages[i + 1:] if s[0] == "conv"), None)
            out, codes = fused_conv(codes, conv, relu=relu, next_quant=nxt)
            if nxt is not None:
                out = None
        else:
            _, k, stride, pad = st
            if codes is not None:
                codes = maxpool_nhwc(codes, k, stride, pad).astype(np.int32)
            else:
                out = maxpool_nhwc(out, k, stride, pad).astype(np.float32)
    return out
