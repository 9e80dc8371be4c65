"""Convolution / linear on term codes with the tcgen05 kernel (csrc/tq_gemm.cu).

`conv2d_codes` is the raw op (fp16 NHWC codes in, fp32 NHWC out).  `pack_conv_weight` turns a
term-revealed OIHW weight into the [R*S][Cout][Cin] fp16 code tensor the kernel reads."""
import torch

from . import _lib
from . import tr_cuda


def pack_conv_weight(w, w_sf, weight_bits, group_size, num_terms):
    """Term-reveal an (O, I, kh, kw) fp32 weight (groups along I, tr_layer.py:117-120) and
    return its integer codes as fp16 [kh*kw, O, I]."""
    codes = tr_cuda.tr_codes(w.detach().contiguous(), w_sf, weight_bits, group_size, num_terms,
                             dtype=torch.int16)
    O, I, kh, kw = codes.shape
    return codes.permute(2, 3, 0, 1).reshape(kh * kw, O, I).to(torch.float16).contiguous()


# ---- exact-accumulator contract -------------------------------------------------------------------------
# The kind::f16 kernel accumulates in fp32: exact only below 2^24.  Whether a layer can run on it is PROVEN here
# from its weight codes alone, for every possible activation (include/tq_b200.h, "EXACTNESS CONTRACT"): a chunk
# of K whose activations lie in [0, act_max] has every partial sum inside
# [-act_max * sum(w-), +act_max * sum(w+)].  A layer that cannot be proven with the accumulator groups tensor
# memory offers runs on the kind::i8 plane engine (int32 accumulators, exact for every input).

EXACT_LIMIT = 1 << 24


def _quant_args(next_quant):
    """(sf, bits, terms, TQ_ENC_*) of a consumer's quantiser given as (sf, bits, terms) -- HESE -- or
    (sf, bits, terms, encoding name); None: no codes are written."""
    if not next_quant:
        return 1.0, 1, 0, _lib.ENC_HESE
    if len(next_quant) not in (3, 4):
        raise ValueError(f"next_quant must be (sf, bits, terms) or (sf, bits, terms, encoding), got {next_quant!r}")
    enc = _lib.encoding_id(next_quant[3]) if len(next_quant) == 4 else _lib.ENC_HESE
    return next_quant[0], next_quant[1], next_quant[2], enc


def _ptr(t):
    """Device address of an optional tensor argument (None: NULL)."""
    return t.data_ptr() if t is not None else None


def _relu_code(relu):
    """Activation of the fused epilogues: False / 0 none, True / 1 ReLU, 'relu6' / 2 ReLU6."""
    if relu in ("relu6", 2):
        return 2
    return 1 if relu else 0


class WeightPlan:
    """How one packed weight [R*S, Cout, C] runs exactly: engine 'f16' with `groups` K chunks, or 'i8' with the
    signed 8-bit planes of the weight codes.  Built once per weight by `plan_weight`."""

    def __init__(self, engine, groups, bound, act_max, signed, wgt, planes=None, planes_w=0, wgt_max=0):
        self.engine, self.groups, self.bound, self.act_max, self.signed = engine, groups, bound, act_max, signed
        self.wgt, self.planes, self.planes_w, self.wgt_max = wgt, planes, planes_w, wgt_max

    def __repr__(self):
        return (f"WeightPlan({self.engine}, groups={self.groups}, bound={self.bound:.3e}, act_max={self.act_max}, "
                f"signed={self.signed}, planes_w={self.planes_w})")


def weight_l1(wgt):
    """(pos, neg): int64 [Cout, ceil(C/64)] sums of the positive / negative weight codes per output channel and
    64-channel block over all taps (tq_conv_weight_l1)."""
    RS, Cout, C = wgt.shape
    kcb = (C + 63) // 64
    pos = torch.empty((Cout, kcb), dtype=torch.int64, device=wgt.device)
    neg = torch.empty_like(pos)
    with torch.cuda.device(wgt.device):
        rc = _lib.lib().tq_conv_weight_l1(wgt.data_ptr(), RS, Cout, C, pos.data_ptr(), neg.data_ptr(),
                                          torch.cuda.current_stream(wgt.device).cuda_stream)
    _lib.check(rc)
    return pos, neg


def codes_to_planes(codes, planes):
    """fp16 integer codes (any shape, numel % 8 == 0) -> int8 [planes, *shape]: plane 0 = code >> 4 and plane 1 =
    code & 15, or the code itself for planes == 1 (raises if a code does not fit)."""
    if codes.dtype != torch.float16 or not codes.is_contiguous() or not codes.is_cuda:
        raise RuntimeError("codes_to_planes expects a contiguous fp16 CUDA tensor")
    out = torch.empty((planes,) + tuple(codes.shape), dtype=torch.int8, device=codes.device)
    ovf = torch.zeros(1, dtype=torch.int32, device=codes.device)
    with torch.cuda.device(codes.device):
        rc = _lib.lib().tq_codes_to_planes(codes.data_ptr(), out.data_ptr(), codes.numel(), planes, ovf.data_ptr(),
                                           torch.cuda.current_stream(codes.device).cuda_stream)
    _lib.check(rc)
    return out, ovf


def _planes_needed(max_abs_code):
    if max_abs_code <= 127:
        return 1
    if max_abs_code <= 2047:
        return 2
    raise NotImplementedError(f"codes up to {max_abs_code} do not fit two signed 8-bit planes")


def plan_weight(wgt, act_max, signed_act=False, engine="auto"):
    """Static exactness proof for a packed weight `wgt` (fp16 codes [R*S, Cout, C]) under activations in
    [0, act_max] (or [-act_max, act_max] when signed_act).  engine: 'auto' (kind::f16 with the fewest accumulator
    groups that can be proven, else the kind::i8 plane engine), 'f16' (raise if it cannot be proven), 'i8'."""
    if wgt.dtype != torch.float16 or wgt.dim() != 3 or not wgt.is_contiguous():
        raise RuntimeError("plan_weight expects a contiguous fp16 [R*S, Cout, C] code tensor")
    RS, Cout, C = wgt.shape
    bound = float("inf")
    if engine in ("auto", "f16"):
        pos, neg = weight_l1(wgt)
        kcb = pos.shape[1]
        block_n = 64 if Cout <= 64 else 128
        for groups in (1, 2, 4, 8):
            if kcb % groups or groups * block_n > (512 if block_n == 128 else 256):   # tensor-memory columns (tq_gemm.cu)
                continue
            p = pos.view(Cout, groups, kcb // groups).sum(2)
            n = neg.view(Cout, groups, kcb // groups).sum(2)
            worst = (p + n) if signed_act else torch.maximum(p, n)
            b = float(act_max) * float(worst.max().item())
            bound = min(bound, b)
            if b < EXACT_LIMIT:
                return WeightPlan("f16", groups, b, act_max, signed_act, wgt)
        if engine == "f16":
            raise NotImplementedError(
                f"kind::f16 conv: cannot prove exact fp32 accumulation for this weight (best bound {bound:.3e} >= 2^24 "
                f"with act_max = {act_max}); use the kind::i8 plane engine (engine='i8' / 'auto')")
    if C % 16:
        raise NotImplementedError("kind::i8 plane engine needs C % 16 == 0")
    wmax = int(wgt.abs().max().item())
    pw = _planes_needed(wmax)
    planes, ovf = codes_to_planes(wgt, pw)
    if int(ovf.item()):
        raise RuntimeError("weight codes do not fit their planes")
    return WeightPlan("i8", 1, bound, act_max, signed_act, wgt, planes=planes, planes_w=pw, wgt_max=max(wmax, 1))


def _cached_plan(wgt, act_max, signed_act, engine):
    """The plan of `wgt` for the raw ops called without plan=.  It is kept on the weight tensor itself, so it lives
    exactly as long as the weight: a CUDA graph that captured a call keeps the weight alive and with it the int8 planes
    the i8 engine reads.  An in-place change of the weight (a new _version) replaces the plan."""
    plans = wgt.__dict__.setdefault("_tq_plans", {})
    key = (int(act_max), bool(signed_act), engine)
    stamp = (wgt.data_ptr(), wgt._version, tuple(wgt.shape))
    hit = plans.get(key)
    if hit is None or hit[0] != stamp:
        hit = plans[key] = (stamp, plan_weight(wgt, act_max, signed_act, engine))
    return hit[1]


def _run_conv(act, plan, out, codes, bias, bn, residual, N, H, W, C, Cout, R, S, stride, pad, scale, relu, sf, bits,
              terms, enc, act_planes=None):
    stream = torch.cuda.current_stream(act.device).cuda_stream
    with torch.cuda.device(act.device):
        if plan.engine == "f16":
            rc = _lib.lib().tq_conv2d_codes_fused_enc(
                act.data_ptr(), plan.wgt.data_ptr(), _ptr(out), _ptr(codes), _ptr(bias),
                _ptr(bn[0]) if bn else None, _ptr(bn[1]) if bn else None, _ptr(residual),
                N, H, W, C, Cout, R, S, stride, pad, float(scale), _relu_code(relu), float(sf), int(bits),
                int(terms), enc, int(plan.groups), stream)
        else:
            if act_planes is None:
                pa = _planes_needed(plan.act_max)
                act_planes, _ = codes_to_planes(act, pa)
            rc = _lib.lib().tq_conv2d_planes_i8_enc(
                act_planes.data_ptr(), plan.planes.data_ptr(), act_planes.shape[0], plan.planes_w, _ptr(out), _ptr(codes),
                _ptr(bias), _ptr(bn[0]) if bn else None, _ptr(bn[1]) if bn else None, _ptr(residual),
                N, H, W, C, Cout, R, S, stride, pad, float(scale), _relu_code(relu), float(sf), int(bits), int(terms),
                enc, int(plan.act_max), int(plan.wgt_max), stream)
    _lib.check(rc)


def conv2d_codes(act, wgt, bias, kernel_size, stride, pad, scale, out=None, *, act_max=512, signed_act=False,
                 engine="auto", plan=None):
    """act: fp16 [N, H, W, C] codes with |code| <= act_max (non-negative unless signed_act); wgt: fp16
    [R*S, Cout, C] codes; returns fp32 [N, Ho, Wo, Cout] = float(exact int32 accumulator) * scale (+ bias).
    The engine is chosen by the static proof of `plan_weight` (cached per weight tensor)."""
    if not (act.is_cuda and wgt.is_cuda and act.dtype == torch.float16 and wgt.dtype == torch.float16):
        raise RuntimeError("conv2d_codes expects fp16 CUDA code tensors")
    if not (act.is_contiguous() and wgt.is_contiguous()):
        raise RuntimeError("conv2d_codes expects contiguous NHWC activations and packed weights")
    N, H, W, C = act.shape
    R, S = kernel_size
    RS, Cout, C2 = wgt.shape
    if RS != R * S or C2 != C:
        raise RuntimeError("weight / activation shape mismatch")
    Ho = (H + 2 * pad - R) // stride + 1
    Wo = (W + 2 * pad - S) // stride + 1
    if out is None:
        out = torch.empty((N, Ho, Wo, Cout), dtype=torch.float32, device=act.device)
    if plan is None:
        plan = _cached_plan(wgt, act_max, signed_act, engine)
    _run_conv(act, plan, out, None, bias, None, None, N, H, W, C, Cout, R, S, stride, pad, scale, False, 1.0, 1, 0,
              _lib.ENC_HESE)
    return out


def conv2d_codes_fused(act, wgt, kernel_size, stride, pad, scale, *, bias=None, bn=None, residual=None,
                       relu=False, want_f32=True, next_quant=None, act_max=512, signed_act=False, engine="auto",
                       plan=None):
    """Conv on codes with the fused tail (see tq_conv2d_codes_fused in include/tq_b200.h).

    bn = (a, b) fp32 [Cout] per-channel affine applied as fma(t, a, b); residual fp32
    [N, Ho, Wo, Cout]; next_quant = (sf, bits, terms) of the consumer's LinearQuantize (HESE), or
    (sf, bits, terms, encoding) for a consumer with another term encoding.
    Returns (out_f32 or None, out_codes or None)."""
    N, H, W, C = act.shape
    R, S = kernel_size
    RS, Cout, C2 = wgt.shape
    if act.dtype != torch.float16 or wgt.dtype != torch.float16 or RS != R * S or C2 != C:
        raise RuntimeError("conv2d_codes_fused: bad operands")
    Ho = (H + 2 * pad - R) // stride + 1
    Wo = (W + 2 * pad - S) // stride + 1
    out = torch.empty((N, Ho, Wo, Cout), dtype=torch.float32, device=act.device) if want_f32 else None
    codes = torch.empty((N, Ho, Wo, Cout), dtype=torch.float16, device=act.device) if next_quant else None
    if residual is not None and (residual.shape != (N, Ho, Wo, Cout) or not residual.is_contiguous()
                                 or residual.dtype != torch.float32):
        raise RuntimeError("residual must be a contiguous fp32 [N, Ho, Wo, Cout] tensor")
    sf, bits, terms, enc = _quant_args(next_quant)
    if plan is None:
        plan = _cached_plan(wgt, act_max, signed_act, engine)
    _run_conv(act, plan, out, codes, bias, bn, residual, N, H, W, C, Cout, R, S, stride, pad, scale, relu, sf, bits, terms,
              enc)
    return out, codes


def pack_linear_weight(w, w_sf):
    """Term-revealed (out, in) fp32 weight (an integer multiple of w_sf) -> fp16 codes [1, out_pad, in_pad] for the conv
    kernel run as a GEMM (1x1 conv over a 1 x M "image"): `in` padded to a multiple of 16 with zero codes (TMA rows are
    16 bytes; 650 -> 656 for the LSTM), `out` to a multiple of 4.  Returns (packed, fp32 w_sf)."""
    sf32 = torch.tensor(w_sf, dtype=torch.float32).item()
    codes = torch.round(w.detach() / sf32)
    if not torch.equal(codes * sf32, w.detach()):
        raise RuntimeError("weight is not an integer multiple of w_sf any more")
    O, I = codes.shape
    Op, Ip = (O + 3) // 4 * 4, (I + 15) // 16 * 16
    packed = torch.zeros((1, Op, Ip), dtype=torch.float16, device=w.device)
    packed[0, :O, :I] = codes.to(torch.float16)
    return packed, sf32


def linear_codes(x_codes, wgt, scale, *, bias=None, out_features=None, plan=None, act_max=512, signed_act=True,
                 engine="auto"):
    """x_codes fp16 [M, K] integer codes times packed weight codes [1, out_pad, K_pad] (pack_linear_weight):
    float(exact int32 accumulator) * scale (+ bias) -> fp32 [M, out_features].  The GEMM runs on the tcgen05 conv
    kernel as a 1x1 conv over a 1 x M image; the engine (kind::f16 with proven K chunks / kind::i8 planes) comes from
    `plan_weight`."""
    if x_codes.dtype != torch.float16 or x_codes.dim() != 2:
        raise RuntimeError("linear_codes expects fp16 [M, K] codes")
    M, K = x_codes.shape
    _, Op, Kp = wgt.shape
    if K > Kp:
        raise RuntimeError("weight / activation shape mismatch")
    if K != Kp:
        xp = torch.zeros((M, Kp), dtype=torch.float16, device=x_codes.device)
        xp[:, :K] = x_codes
        x_codes = xp
    bias_p = bias
    if bias is not None and bias.numel() != Op:
        bias_p = torch.zeros(Op, dtype=torch.float32, device=wgt.device)
        bias_p[:bias.numel()] = bias.detach().float()
    out = conv2d_codes(x_codes.contiguous().view(1, 1, M, Kp), wgt, bias_p, (1, 1), 1, 0, scale, plan=plan, act_max=act_max,
                       signed_act=signed_act, engine=engine).view(M, Op)
    n = out_features if out_features is not None else Op
    return out if n == Op else out[:, :n]


def linear_codes_nll(x_codes, wgt, scale, targets, *, bias=None, out_features=None, plan=None, act_max=512,
                     signed_act=True, engine="auto"):
    """Per-row negative log-likelihood of `targets` under the logits linear_codes(x_codes, wgt, scale, bias=bias,
    out_features=out_features, ...) would return, without writing them (tq_linear_codes_nll / tq_linear_planes_i8_nll):
    the decoder's epilogue reduces each row's (max, sum exp) over the first out_features columns and picks the target
    logit, and a small kernel combines the partials.  Same operands, plan and engines as linear_codes; targets int64 [M]
    on the same device.  Returns fp32 [M] = logsumexp(logits[r]) - logits[r, targets[r]], within 4e-6 * max(|ref|, 1)
    of fp64 over the same logits; a target outside [0, out_features) gives NaN for its row."""
    if x_codes.dtype != torch.float16 or wgt.dtype != torch.float16 or targets.dtype != torch.int64:
        raise RuntimeError(f"linear_codes_nll expects fp16 codes and weights and int64 targets, got {x_codes.dtype}, "
                           f"{wgt.dtype} and {targets.dtype}")
    if x_codes.dim() != 2 or wgt.dim() != 3 or wgt.shape[0] != 1 or targets.dim() != 1 \
            or targets.shape[0] != x_codes.shape[0]:
        raise ValueError(f"linear_codes_nll expects codes [M, K], a packed weight [1, Op, Kp] and targets [M], got "
                         f"{tuple(x_codes.shape)}, {tuple(wgt.shape)} and {tuple(targets.shape)}")
    M, K = x_codes.shape
    _, Op, Kp = wgt.shape
    V = out_features if out_features is not None else Op
    if M < 1 or K > Kp or not 1 <= V <= Op:
        raise ValueError(f"linear_codes_nll: M = {M}, K = {K} against Kp = {Kp}, out_features = {V} against Op = {Op}: "
                         f"need M >= 1, K <= Kp and 1 <= out_features <= Op")
    if not targets.is_contiguous() or not wgt.is_contiguous():
        raise ValueError("linear_codes_nll expects contiguous targets and a contiguous packed weight")
    if bias is not None and (bias.dtype != torch.float32 or bias.dim() != 1 or bias.numel() not in (V, Op)):
        raise ValueError(f"linear_codes_nll expects an fp32 bias of out_features or Op entries, got {bias.dtype} "
                         f"{tuple(bias.shape)}")
    devs = {t.device for t in (x_codes, wgt, targets) + ((bias,) if bias is not None else ())}
    if len(devs) != 1 or not x_codes.is_cuda:
        raise RuntimeError(f"linear_codes_nll expects every tensor on one CUDA device, got {sorted(map(str, devs))}")
    if K != Kp or not x_codes.is_contiguous():
        xp = torch.zeros((M, Kp), dtype=torch.float16, device=x_codes.device)
        xp[:, :K] = x_codes
        x_codes = xp
    if bias is not None and bias.numel() != Op:
        bp = torch.zeros(Op, dtype=torch.float32, device=wgt.device)
        bp[:bias.numel()] = bias
        bias = bp
    elif bias is not None:
        bias = bias.contiguous()
    if plan is None:
        plan = _cached_plan(wgt, act_max, signed_act, engine)
    L = _lib.lib()
    ws_bytes = int(L.tq_linear_nll_workspace_bytes(M, Op))
    if ws_bytes < 0:
        raise ValueError(f"linear_codes_nll: M = {M} rows of Op = {Op} columns overflow the workspace size")
    workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=x_codes.device)     # per call (graph pool under capture)
    loss = torch.empty(M, dtype=torch.float32, device=x_codes.device)
    stream = torch.cuda.current_stream(x_codes.device).cuda_stream
    with torch.cuda.device(x_codes.device):
        if plan.engine == "f16":
            rc = L.tq_linear_codes_nll(x_codes.data_ptr(), plan.wgt.data_ptr(), M, Kp, Op, V, float(scale), _ptr(bias),
                                       int(plan.groups), targets.data_ptr(), loss.data_ptr(), workspace.data_ptr(),
                                       ws_bytes, stream)
        else:
            act_planes, _ = codes_to_planes(x_codes, _planes_needed(plan.act_max))
            rc = L.tq_linear_planes_i8_nll(act_planes.data_ptr(), plan.planes.data_ptr(), act_planes.shape[0],
                                           plan.planes_w, M, Kp, Op, V, float(scale), _ptr(bias), int(plan.act_max),
                                           int(plan.wgt_max), targets.data_ptr(), loss.data_ptr(), workspace.data_ptr(),
                                           ws_bytes, stream)
    _lib.check(rc)
    return loss


def pack_depthwise_weight(w, w_sf):
    """Term-revealed depthwise weight (C, 1, 3, 3) fp32 (already an integer multiple of w_sf) -> int32 [9, C] codes."""
    if w.dim() != 4 or w.shape[1] != 1 or tuple(w.shape[2:]) != (3, 3):
        raise NotImplementedError("depthwise packing expects a (C, 1, 3, 3) weight")
    sf32 = torch.tensor(w_sf, dtype=torch.float32).item()
    codes = torch.round(w.detach() / sf32)
    if not torch.equal(codes * sf32, w.detach()):
        raise RuntimeError("depthwise weight is not an integer multiple of w_sf any more")
    return codes.view(w.shape[0], 9).t().contiguous().to(torch.int32), sf32


def depthwise3x3_codes(act, wgt, stride, scale, *, bias=None, bn=None, relu=False, want_f32=False, next_quant=None,
                       act_unsigned=False):
    """Depthwise 3x3 / pad 1 conv on fp16 codes [N, H, W, C] with int32 weight codes [9, C]: exact int32 accumulator,
    then the fused tail (tq_depthwise3x3_codes).  act_unsigned: the codes are known to lie in [0, 1023] (post-ReLU
    input under a quantiser of at most 9 bits).  Returns (out_f32 or None, out_codes or None)."""
    if act.dtype != torch.float16 or not act.is_contiguous() or wgt.dtype != torch.int32 or not wgt.is_contiguous():
        raise RuntimeError("depthwise3x3_codes expects contiguous fp16 NHWC codes and int32 [9, C] weights")
    N, H, W, C = act.shape
    if tuple(wgt.shape) != (9, C):
        raise RuntimeError("weight / activation shape mismatch")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty((N, Ho, Wo, C), dtype=torch.float32, device=act.device) if want_f32 else None
    codes = torch.empty((N, Ho, Wo, C), dtype=torch.float16, device=act.device) if next_quant else None
    sf, bits, terms, enc = _quant_args(next_quant)
    with torch.cuda.device(act.device):
        rc = _lib.lib().tq_depthwise3x3_codes_enc(
            act.data_ptr(), wgt.data_ptr(), _ptr(out), _ptr(codes), _ptr(bias), _ptr(bn[0]) if bn else None,
            _ptr(bn[1]) if bn else None, N, H, W, C, stride, float(scale), _relu_code(relu), int(bool(act_unsigned)),
            float(sf), int(bits), int(terms), enc, torch.cuda.current_stream(act.device).cuda_stream)
    _lib.check(rc)
    return out, codes


def pack_first_conv_weight(w_oihw):
    """(Cout, 3, 3, 3) conv weight -> fp32 [3][3][3][Cout] (filter row, filter column, input channel, output channel)."""
    if w_oihw.dim() != 4 or w_oihw.shape[1:] != (3, 3, 3):
        raise RuntimeError("pack_first_conv_weight expects a (Cout, 3, 3, 3) weight")
    return w_oihw.detach().float().permute(2, 3, 1, 0).contiguous()


def first_conv3x3_fused(x_nhwc, w_packed, stride=1, bias=None, bn=None, relu=False, want_f32=False, next_quant=None):
    """nn.Conv2d(3, Cout, 3, stride, padding=1) in fp32 on an fp32 NHWC [N, H, W, 3] tensor, fused with + bias,
    BatchNorm affine, ReLU / ReLU6 and the next quantiser (tq_first_conv3x3_fused).  Returns (out fp32 or None,
    fp16 term codes or None), both [N, Ho, Wo, Cout]."""
    if x_nhwc.dtype != torch.float32 or not x_nhwc.is_contiguous() or not x_nhwc.is_cuda or x_nhwc.shape[-1] != 3:
        raise RuntimeError("first_conv3x3_fused expects a contiguous fp32 CUDA [N, H, W, 3] tensor")
    N, H, W, _ = x_nhwc.shape
    Cout = w_packed.shape[-1]
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty((N, Ho, Wo, Cout), dtype=torch.float32, device=x_nhwc.device) if want_f32 else None
    codes = torch.empty((N, Ho, Wo, Cout), dtype=torch.float16, device=x_nhwc.device) if next_quant else None
    if out is None and codes is None:
        raise RuntimeError("first_conv3x3_fused: nothing to compute (want_f32 or next_quant)")
    sf, bits, terms, enc = _quant_args(next_quant)
    for t in (bias, bn[0] if bn else None, bn[1] if bn else None):
        if t is not None and (t.dtype != torch.float32 or t.numel() != Cout or not t.is_contiguous() or t.device != x_nhwc.device):
            raise RuntimeError("first_conv3x3_fused: bias / bn must be contiguous fp32 [Cout] tensors on the input's device")
    with torch.cuda.device(x_nhwc.device):
        rc = _lib.lib().tq_first_conv3x3_fused_enc(
            x_nhwc.data_ptr(), w_packed.data_ptr(), _ptr(bias), _ptr(bn[0]) if bn else None, _ptr(bn[1]) if bn else None,
            _ptr(out), _ptr(codes), N, H, W, Cout, int(stride), _relu_code(relu), float(sf), int(bits), int(terms), enc,
            torch.cuda.current_stream(x_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, codes


def maxpool_codes(codes_nhwc, kernel_size, stride=None, padding=0):
    """nn.MaxPool2d(kernel_size, stride, padding) (floor mode) on fp16 NHWC term codes (tq_maxpool2d_f16)."""
    k = kernel_size if isinstance(kernel_size, int) else kernel_size[0]
    st = k if stride is None else (stride if isinstance(stride, int) else stride[0])
    pd = padding if isinstance(padding, int) else padding[0]
    if codes_nhwc.dtype != torch.float16 or not codes_nhwc.is_contiguous() or not codes_nhwc.is_cuda:
        raise RuntimeError("maxpool_codes expects a contiguous fp16 CUDA [N, H, W, C] tensor")
    N, H, W, C = codes_nhwc.shape
    Ho, Wo = (H + 2 * pd - k) // st + 1, (W + 2 * pd - k) // st + 1
    out = torch.empty((N, Ho, Wo, C), dtype=torch.float16, device=codes_nhwc.device)
    with torch.cuda.device(codes_nhwc.device):
        rc = _lib.lib().tq_maxpool2d_f16(codes_nhwc.data_ptr(), out.data_ptr(), N, H, W, C, k, st, pd,
                                         torch.cuda.current_stream(codes_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out


def bn_act_encode(x_nhwc, bn=None, relu=False, want_f32=False, next_quant=None, bias=None):
    """fp32 [..., C] -> (+ bias) -> fma(x, a, b) -> activation -> fp32 and / or fp16 term codes (tq_bn_act_encode)."""
    if x_nhwc.dtype != torch.float32 or not x_nhwc.is_contiguous() or not x_nhwc.is_cuda:
        raise RuntimeError("bn_act_encode expects a contiguous fp32 CUDA tensor with channels last")
    C = x_nhwc.shape[-1]
    out = torch.empty_like(x_nhwc) if want_f32 else None
    codes = torch.empty(x_nhwc.shape, dtype=torch.float16, device=x_nhwc.device) if next_quant else None
    sf, bits, terms, enc = _quant_args(next_quant)
    with torch.cuda.device(x_nhwc.device):
        if bias is not None and (bias.dtype != torch.float32 or bias.numel() != C or not bias.is_contiguous() or bias.device != x_nhwc.device):
            raise RuntimeError("bn_act_encode: bias must be a contiguous fp32 [C] tensor on the input's device")
        rc = _lib.lib().tq_bn_act_encode_enc(
            x_nhwc.data_ptr(), _ptr(bias), _ptr(bn[0]) if bn else None, _ptr(bn[1]) if bn else None, _ptr(out), _ptr(codes),
            x_nhwc.numel() // C, C, _relu_code(relu), float(sf), int(bits), int(terms), enc,
            torch.cuda.current_stream(x_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, codes


def bn_relu_maxpool_encode(x_nhwc, bn, relu=True, next_quant=None, rowmax=False):
    """maxpool3x3/s2/p1(relu(fma(x, a, b))) on an fp32 [N, H, W, C] tensor, plus the fp16 term
    codes of the result for the first wrapped conv.  Returns (out [N, Ho, Wo, C], codes or None).
    rowmax=True: x is [N, H, Wo, C], the row maxima stem_conv7x7s2(..., rowmax=True) writes (the horizontal half of the
    pool already taken, bn from stem_pool_operands); only the vertical window is left (tq_bn_relu_maxpool_encode_rowmax)."""
    if x_nhwc.dtype != torch.float32 or not x_nhwc.is_contiguous() or not x_nhwc.is_cuda:
        raise RuntimeError("bn_relu_maxpool_encode expects a contiguous fp32 CUDA [N, H, W, C] tensor")
    N, H, W, C = x_nhwc.shape
    Ho, Wo = (H - 1) // 2 + 1, (W if rowmax else (W - 1) // 2 + 1)
    out = torch.empty((N, Ho, Wo, C), dtype=torch.float32, device=x_nhwc.device)
    codes = torch.empty((N, Ho, Wo, C), dtype=torch.float16, device=x_nhwc.device) if next_quant else None
    sf, bits, terms, enc = _quant_args(next_quant)
    L = _lib.lib()
    fn = L.tq_bn_relu_maxpool_encode_rowmax_enc if rowmax else L.tq_bn_relu_maxpool_encode_enc
    with torch.cuda.device(x_nhwc.device):
        rc = fn(
            x_nhwc.data_ptr(), bn[0].data_ptr(), bn[1].data_ptr(), out.data_ptr(),
            codes.data_ptr() if codes is not None else None, N, H, W, C, int(bool(relu)),
            float(sf), int(bits), int(terms), enc, torch.cuda.current_stream(x_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, codes


def pack_stem_weight(w, channel_sign=None):
    """(Cout, 3, 7, 7) fp32 -> fp16 [4][128][64] for tq_stem_conv7x7s2: the kernel padded to 8x8 and
    folded 2x2 (r = 2R + dr, s = 2S + ds), tile R holding (S, dr, ds, c) with c padded to 4; rows 0..Cout-1 of a tile are
    the fp16 hi plane, rows 64..64+Cout-1 the lo plane (w = w_hi + w_lo), so that one N = 128 MMA multiplies by both.
    `channel_sign` (+1 / -1 per output channel) is folded into the weights (the one-kernel stem pools before the
    BatchNorm affine and needs non-negative slopes: see stem_conv_pool)."""
    Cout, Cin, kh, kw = w.shape
    if (Cin, kh, kw) != (3, 7, 7) or Cout > 64:
        raise NotImplementedError("stem conv packing expects a (Cout <= 64, 3, 7, 7) weight")
    w8 = torch.zeros(Cout, 4, 8, 8, dtype=torch.float32, device=w.device)
    w8[:, :3, :7, :7] = w.detach().float()
    if channel_sign is not None:
        w8 = w8 * channel_sign.view(-1, 1, 1, 1).to(w8)
    # [co, c, R, dr, S, ds] -> [R, co, S, dr, ds, c]
    w2 = w8.view(Cout, 4, 4, 2, 4, 2).permute(2, 0, 4, 3, 5, 1).reshape(4, Cout, 64)
    hi = w2.half()
    lo = (w2 - hi.float()).half()
    out = torch.zeros(4, 128, 64, dtype=torch.float16, device=w.device)
    out[:, :Cout] = hi
    out[:, 64:64 + Cout] = lo
    return out.contiguous()


_STEM_DTYPES = {torch.float32: _lib.TQ_F32, torch.bfloat16: _lib.TQ_BF16, torch.float16: _lib.TQ_F16}


def _stem_out_w(W, rowmax):
    """Columns of the stem conv's output: W/2 conv columns, or the (W/2 - 1) // 2 + 1 row maxima."""
    return (W // 2 - 1) // 2 + 1 if rowmax else W // 2


def stem_conv7x7s2(x_nhwc, w2, scratch=None, cout=None, rowmax=False):
    """fp32 / bf16 / fp16 [N, H, W, 3] -> fp32 [N, H/2, W/2, Cout] (7x7 / stride 2 / pad 3, no bias).
    rowmax=True: fp32 [N, H/2, Wp, Cout] (Wp = (W/2 - 1) // 2 + 1), the max of conv columns 2q-1, 2q, 2q+1 of each conv
    row -- the horizontal half of the stem's 3x3/s2/p1 max-pool (tq_stem_conv7x7s2_rowmax), for
    bn_relu_maxpool_encode(..., rowmax=True); `w2` then comes from stem_pool_operands (the pool runs before the affine)."""
    if x_nhwc.dtype not in _STEM_DTYPES or not x_nhwc.is_contiguous() or x_nhwc.shape[-1] != 3:
        raise RuntimeError("stem_conv7x7s2 expects a contiguous fp32 / bf16 / fp16 [N, H, W, 3] tensor")
    N, H, W, _ = x_nhwc.shape
    Cout = cout if cout is not None else 64
    need = (2 if x_nhwc.dtype == torch.float32 else 1) * N * (H // 2 + 3) * (W // 2 + 3) * 16
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty(need, dtype=torch.float16, device=x_nhwc.device)
    out = torch.empty((N, H // 2, _stem_out_w(W, rowmax), Cout), dtype=torch.float32, device=x_nhwc.device)
    fn = _lib.lib().tq_stem_conv7x7s2_rowmax if rowmax else _lib.lib().tq_stem_conv7x7s2_dt
    with torch.cuda.device(x_nhwc.device):
        rc = fn(x_nhwc.data_ptr(), _STEM_DTYPES[x_nhwc.dtype], scratch.data_ptr(),
                                             w2.data_ptr(), out.data_ptr(), N, H, W, Cout,
                                             torch.cuda.current_stream(x_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, scratch


def stem_conv7x7s2_u8(x_u8_nhwc, mean, std, w2, scratch=None, cout=None, rowmax=False):
    """uint8 [N, H, W, 3] images -> fp32 [N, H/2, W/2, Cout]: ToTensor + Normalize (rounded to bf16, exactly what
    inference.normalize_u8 produces) folded into the stem conv's fold pass (tq_stem_conv7x7s2_u8).
    rowmax: as for stem_conv7x7s2 (tq_stem_conv7x7s2_u8_rowmax)."""
    import ctypes
    if x_u8_nhwc.dtype != torch.uint8 or not x_u8_nhwc.is_contiguous() or not x_u8_nhwc.is_cuda or x_u8_nhwc.shape[-1] != 3:
        raise RuntimeError("stem_conv7x7s2_u8 expects a contiguous uint8 CUDA [N, H, W, 3] tensor")
    N, H, W, _ = x_u8_nhwc.shape
    Cout = cout if cout is not None else 64
    need = N * (H // 2 + 3) * (W // 2 + 3) * 16
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty(need, dtype=torch.float16, device=x_u8_nhwc.device)
    out = torch.empty((N, H // 2, _stem_out_w(W, rowmax), Cout), dtype=torch.float32, device=x_u8_nhwc.device)
    m = (ctypes.c_float * 3)(*mean)
    s = (ctypes.c_float * 3)(*std)
    fn = _lib.lib().tq_stem_conv7x7s2_u8_rowmax if rowmax else _lib.lib().tq_stem_conv7x7s2_u8
    with torch.cuda.device(x_u8_nhwc.device):
        rc = fn(x_u8_nhwc.data_ptr(), ctypes.cast(m, ctypes.c_void_p), ctypes.cast(s, ctypes.c_void_p),
                                             scratch.data_ptr(), w2.data_ptr(), out.data_ptr(), N, H, W, Cout,
                                             torch.cuda.current_stream(x_u8_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, scratch


def stem_pool_operands(w, bn):
    """Operands of the one-kernel stem for a (Cout, 3, 7, 7) weight and BatchNorm affine (a, b): the kernel pools
    the raw conv sums and applies the affine once per pooled value, which needs a >= 0, so sign(a) moves into the
    channel's weights (exact) and |a| is passed.  Returns (w2_signed, (|a|, b))."""
    a, b = bn
    sign = torch.where(a < 0, -torch.ones_like(a), torch.ones_like(a))
    return pack_stem_weight(w, sign), (a.abs().contiguous(), b.contiguous())


def stem_conv_pool(x_nhwc, w2, bn, relu=True, next_quant=None, scratch=None):
    # (Cout = number of BatchNorm channels: the packed weight tile is always 128 rows)
    """The whole stem in one launch: maxpool3x3/s2/p1(relu(fma(conv7x7s2(x), a, b))) -> fp32
    [N, Hp, Wp, Cout] plus the fp16 term codes of the result (next_quant = (sf, bits, terms[, encoding])).
    Same values as stem_conv7x7s2 followed by bn_relu_maxpool_encode; the conv output never reaches HBM.
    `w2`, `bn` must come from stem_pool_operands (sign of the slope folded into the weights, bn[0] >= 0).
    Returns (out, codes or None, scratch)."""
    if x_nhwc.dtype not in _STEM_DTYPES or not x_nhwc.is_contiguous() or x_nhwc.shape[-1] != 3:
        raise RuntimeError("stem_conv_pool expects a contiguous fp32 / bf16 / fp16 [N, H, W, 3] tensor")
    N, H, W, _ = x_nhwc.shape
    Cout = bn[0].numel()
    need = (2 if x_nhwc.dtype == torch.float32 else 1) * N * (H // 2 + 3) * (W // 2 + 3) * 16
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty(need, dtype=torch.float16, device=x_nhwc.device)
    Hp, Wp = (H // 2 - 1) // 2 + 1, (W // 2 - 1) // 2 + 1
    out = torch.empty((N, Hp, Wp, Cout), dtype=torch.float32, device=x_nhwc.device)
    codes = torch.empty((N, Hp, Wp, Cout), dtype=torch.float16, device=x_nhwc.device) if next_quant else None
    sf, bits, terms, enc = _quant_args(next_quant)
    with torch.cuda.device(x_nhwc.device):
        rc = _lib.lib().tq_stem_conv7x7s2_pool_enc(
            x_nhwc.data_ptr(), _STEM_DTYPES[x_nhwc.dtype], scratch.data_ptr(), w2.data_ptr(),
            bn[0].data_ptr(), bn[1].data_ptr(), int(bool(relu)), out.data_ptr(),
            codes.data_ptr() if codes is not None else None, N, H, W, Cout, float(sf), int(bits), int(terms), enc,
            torch.cuda.current_stream(x_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out, codes, scratch


# gate rows per hidden unit of each RNNModel cell: the recurrence kernel keeps this many rows of W_hh per unit
RECURRENCE_GATES = {"LSTM": 4, "GRU": 3, "RNN_TANH": 1, "RNN_RELU": 1}


def recurrence_max_hidden(cell, device=None):
    """Largest hidden size the recurrence kernel of `cell` ('LSTM', 'GRU', 'RNN_TANH' or 'RNN_RELU') takes on `device`:
    each CTA keeps the gate rows of ceil(H / SMs) units on chip, as many units as fit in the SM's tensor memory
    (4 * floor(512 / (gates * ceil(H / 32))) once shared memory alone is not enough) and the rest in shared memory next
    to one hidden row and 2 KB of gate scratch (B200: LSTM 2048, GRU 2304, RNN 4096).  The library computes it
    (tq_recurrence_max_hidden), the same number its refusals name."""
    if cell not in RECURRENCE_GATES:
        raise ValueError(f"unknown recurrent cell {cell!r}: expected one of {', '.join(RECURRENCE_GATES)}")
    with torch.cuda.device(device if device is not None else torch.cuda.current_device()):
        n = _lib.lib().tq_recurrence_max_hidden(RECURRENCE_GATES[cell])
    if n < 0:
        raise _lib.TQError(f"tq_b200: {_lib.lib().tq_last_error().decode('utf-8', 'replace')}")
    return n


def lstm_max_hidden(device=None):
    """Largest hidden size tq_lstm_recurrence takes on `device` (recurrence_max_hidden('LSTM'))."""
    return recurrence_max_hidden("LSTM", device)


def _recurrence_shapes(name, gates, gin, bias, w_hh, h0, c0=None):
    """The checks every recurrence wrapper makes before the library is reached; returns (T, B, H)."""
    ts = [t for t in (gin, bias, w_hh, h0, c0) if t is not None]
    if any(not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() for t in ts):
        raise RuntimeError(f"{name} expects contiguous fp32 CUDA tensors")
    if any(t.device != gin.device for t in ts):
        raise RuntimeError(f"{name}: every tensor must be on the same device")
    gh = f"{gates}H" if gates > 1 else "H"
    if gin.dim() != 3 or w_hh.dim() != 2:
        raise RuntimeError(f"{name} expects gin [T, B, {gh}] and w_hh [{gh}, H]")
    T, B, G = gin.shape
    H = w_hh.shape[1]
    if G != gates * H or tuple(w_hh.shape) != (gates * H, H) or tuple(h0.shape) != (B, H) \
            or (c0 is not None and tuple(c0.shape) != (B, H)) or (bias is not None and tuple(bias.shape) != (gates * H,)):
        raise RuntimeError(f"{name}: shapes gin {tuple(gin.shape)}, w_hh {tuple(w_hh.shape)}, h0 {tuple(h0.shape)}, "
                           + (f"c0 {tuple(c0.shape)}, " if c0 is not None else "")
                           + f"bias {None if bias is None else tuple(bias.shape)} do not agree")
    return T, B, H


def lstm_recurrence(gin, bias, w_hh, h0, c0):
    """All T steps of one LSTM layer in one launch (tq_lstm_recurrence): gin fp32 [T, B, 4H] (W_ih x_t, torch gate order
    i, f, g, o), bias fp32 [4H] (b_ih + b_hh) or None, w_hh fp32 [4H, H], h0 / c0 fp32 [B, H].
    Returns (y [T, B, H], hn [B, H], cn [B, H]), fp32 with a fixed summation order."""
    T, B, H = _recurrence_shapes("lstm_recurrence", 4, gin, bias, w_hh, h0, c0)
    y = torch.empty((T, B, H), dtype=torch.float32, device=gin.device)
    hn = torch.empty((B, H), dtype=torch.float32, device=gin.device)
    cn = torch.empty((B, H), dtype=torch.float32, device=gin.device)
    with torch.cuda.device(gin.device):
        rc = _lib.lib().tq_lstm_recurrence(gin.data_ptr(), bias.data_ptr() if bias is not None else None, w_hh.data_ptr(),
                                           h0.data_ptr(), c0.data_ptr(), y.data_ptr(), hn.data_ptr(), cn.data_ptr(),
                                           T, B, H, torch.cuda.current_stream(gin.device).cuda_stream)
    _lib.check(rc)
    return y, hn, cn


def gru_recurrence(gin, b_hh, w_hh, h0):
    """All T steps of one GRU layer in one launch (tq_gru_recurrence): gin fp32 [T, B, 3H] (W_ih x_t + b_ih, torch gate
    order r, z, n), b_hh fp32 [3H] or None, w_hh fp32 [3H, H], h0 fp32 [B, H].  b_hn stays inside the reset gate's
    product: n = tanh(gin_n + r * (W_hn h + b_hn)).  Returns (y [T, B, H], hn [B, H]), fp32 with a fixed summation
    order."""
    T, B, H = _recurrence_shapes("gru_recurrence", 3, gin, b_hh, w_hh, h0)
    y = torch.empty((T, B, H), dtype=torch.float32, device=gin.device)
    hn = torch.empty((B, H), dtype=torch.float32, device=gin.device)
    with torch.cuda.device(gin.device):
        rc = _lib.lib().tq_gru_recurrence(gin.data_ptr(), b_hh.data_ptr() if b_hh is not None else None, w_hh.data_ptr(),
                                          h0.data_ptr(), y.data_ptr(), hn.data_ptr(), T, B, H,
                                          torch.cuda.current_stream(gin.device).cuda_stream)
    _lib.check(rc)
    return y, hn


def rnn_recurrence(gin, bias, w_hh, h0, nonlinearity):
    """All T steps of one vanilla RNN layer in one launch (tq_rnn_recurrence): h_t = act(gin[t] + bias + W_hh h_{t-1})
    with gin fp32 [T, B, H] (W_ih x_t), bias fp32 [H] (b_ih + b_hh) or None, w_hh fp32 [H, H], h0 fp32 [B, H] and
    nonlinearity 'tanh' or 'relu' (a NaN stays NaN, as torch.relu).  Returns (y [T, B, H], hn [B, H]), fp32 with a
    fixed summation order."""
    if nonlinearity not in ("tanh", "relu"):
        raise ValueError(f"rnn_recurrence: nonlinearity {nonlinearity!r} is neither 'tanh' nor 'relu'")
    T, B, H = _recurrence_shapes("rnn_recurrence", 1, gin, bias, w_hh, h0)
    y = torch.empty((T, B, H), dtype=torch.float32, device=gin.device)
    hn = torch.empty((B, H), dtype=torch.float32, device=gin.device)
    with torch.cuda.device(gin.device):
        rc = _lib.lib().tq_rnn_recurrence(gin.data_ptr(), bias.data_ptr() if bias is not None else None, w_hh.data_ptr(),
                                          h0.data_ptr(), y.data_ptr(), hn.data_ptr(), T, B, H,
                                          int(nonlinearity == "relu"), torch.cuda.current_stream(gin.device).cuda_stream)
    _lib.check(rc)
    return y, hn


def log_softmax_nll(logits, targets):
    """Per-row negative log-likelihood in one read of the logits (tq_log_softmax_nll): loss[r] =
    logsumexp(logits[r]) - logits[r, targets[r]], i.e. nll_loss(log_softmax(logits), targets, reduction='none') without
    the log-probability tensor.  logits: fp32 CUDA [rows, cols] whose last dimension is contiguous, any row stride >= cols
    (a column slice of a padded GEMM output is read in place); targets: int64 [rows] on the same device.  Returns fp32
    [rows].  A target outside [0, cols) gives NaN for its row (nll_loss would raise; ignore_index is not special here)."""
    if logits.dtype != torch.float32 or targets.dtype != torch.int64:
        raise RuntimeError(f"log_softmax_nll expects fp32 logits and int64 targets, got {logits.dtype} and {targets.dtype}")
    if logits.dim() != 2 or targets.dim() != 1 or targets.shape[0] != logits.shape[0]:
        raise ValueError(f"log_softmax_nll expects logits [rows, cols] and targets [rows], got {tuple(logits.shape)} and "
                         f"{tuple(targets.shape)}")
    rows, cols = logits.shape
    if rows < 1 or cols < 1:
        raise ValueError(f"log_softmax_nll: empty logits {tuple(logits.shape)}")
    ld = logits.stride(0) if rows > 1 else cols              # a single row's stride is arbitrary
    if (cols > 1 and logits.stride(1) != 1) or ld < cols:
        raise ValueError(f"log_softmax_nll expects rows of contiguous logits with a row stride >= cols, got strides "
                         f"{logits.stride()} for {tuple(logits.shape)}")
    if not targets.is_contiguous():
        raise ValueError("log_softmax_nll expects contiguous targets")
    if not logits.is_cuda or not targets.is_cuda or logits.device != targets.device:
        raise RuntimeError(f"log_softmax_nll expects logits and targets on one CUDA device, got {logits.device} and "
                           f"{targets.device}")
    loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
    with torch.cuda.device(logits.device):
        rc = _lib.lib().tq_log_softmax_nll(logits.data_ptr(), rows, cols, ld, targets.data_ptr(), loss.data_ptr(),
                                           torch.cuda.current_stream(logits.device).cuda_stream)
    _lib.check(rc)
    return loss
