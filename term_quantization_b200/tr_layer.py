"""Drop-in for the reference module ``tr_layer`` (tr_layer.py:1-201).

Same public names, constructor signatures and attributes:

    LinearQuantize(data_bits, data_terms)                        tr_layer.py:78-104
    TRConv2dLayer / TRLinearLayer / TRLSTMLayer(layer, data_bits=8, data_terms=4,
        weight_bits=8, group_size=1, num_terms=8)                tr_layer.py:106-201
    set_tr_tracking(model, tracking)                             tr_layer.py:66-76
    mse_profile(hist, minv, maxv, bit_width, terms)              tr_layer.py:43-54
    hese(number), compute_compressed_hese(w, sf, weight_terms)   tr_layer.py:9-41, 57-63

Addition: every one of them except ``hese`` takes a keyword-only ``encoding`` ('hese', the
reference's and the default, 'binary' or 'booth'): the term representation of a TR layer's
weights and of its input quantiser, fixed for the layer's life.

What changed underneath: every ``tr_cuda.tr`` call lands in the sm_100a kernels of
libtq_b200.so; the tracking-mode ``torch.histc`` + add is one fused histogram pass; the
calibration sweep (2048 launches + 2048 syncs per layer in the reference) is one fused kernel;
``compute_compressed_hese`` is a device-side popcount reduction instead of a Python loop over
every weight.  There is no CPU path.

Reference quirks are kept by default (``STRICT_REFERENCE = True``): TRLinearLayer.forward
feeds the *unquantised* input to the linear (tr_layer.py:152-154), TRLSTMLayer only term-reveals
layer 0 and leaves ``w_sf`` at the hh value (tr_layer.py:174-186).  Set
``tr_layer.STRICT_REFERENCE = False`` to have TRLinearLayer use the quantised input.
"""
import math

import torch
import torch.nn as nn

from . import _lib
from . import tr_cuda

STRICT_REFERENCE = True

__all__ = ["hese", "mse_profile", "compute_compressed_hese", "set_tr_tracking", "use_tensor_cores", "LinearQuantize",
           "TRConv2dLayer", "TRLinearLayer", "TRLSTMLayer", "tr_cuda", "STRICT_REFERENCE"]


def hese(number):
    """Signed power-of-two terms of an integer under HESE, smallest magnitude first
    (same list as tr_layer.py:9-41): an isolated 1-bit stays +2^i, a run of ones [lo..hi]
    becomes -2^lo, +2^(hi+1); everything is negated for negative numbers."""
    number = int(number)
    sign = -1 if number < 0 else 1
    q = abs(number)
    out, i = [], 0
    while q >> i:
        if not (q >> i) & 1:
            i += 1
            continue
        lo = i
        while (q >> i) & 1:
            i += 1
        if i - lo == 1:
            out.append(sign * (1 << lo))
        else:
            out.append(-sign * (1 << lo))
            out.append(sign * (1 << i))
    return out


def mse_profile(hist, minv, maxv, bit_width, terms, *, encoding="hese"):
    """Scale factor minimising the histogram-weighted squared error of g=1 term quantisation
    (tr_layer.py:43-54).  Same grid (linspace(minv, maxv, len(hist)) on the device), same 2048
    candidates, same first-minimum rule; one fused sweep on the device."""
    enc = _lib.encoding_id(encoding)
    dev = hist.device if hist.is_cuda else torch.device("cuda")
    hist = hist.to(device=dev, dtype=torch.float32).contiguous()
    x = torch.linspace(minv, maxv, len(hist)).to(dev)
    sfs_t = torch.linspace(1e-8, maxv, 2048)
    sfs = sfs_t.tolist()
    sfs_d = sfs_t.to(dev)
    errs = torch.empty(len(sfs), dtype=torch.float64, device=dev)
    argmin = torch.empty(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.lib().tq_mse_profile_enc(hist.data_ptr(), x.data_ptr(), len(hist), sfs_d.data_ptr(),
                                           len(sfs), int(bit_width), int(terms), enc, errs.data_ptr(),
                                           argmin.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc)
    return sfs[int(argmin.item())]


def compute_compressed_hese(w, sf, weight_terms, *, encoding="hese"):
    """Parameter bits of a HESE-compressed weight tensor (tr_layer.py:57-63):
    (ceil(log2(weight_terms)) + 2) bits per surviving term.  ``encoding`` counts the terms of
    that encoding instead."""
    enc = _lib.encoding_id(encoding)
    exp_bits = math.ceil(math.log2(weight_terms))
    bit_width = exp_bits + 2          # 1 for sign, 1 for barrier
    w = w.detach()
    if not w.is_cuda:
        raise RuntimeError("w must be a CUDA tensor")
    w = w.contiguous()
    count = torch.zeros(1, dtype=torch.int64, device=w.device)
    dt = {torch.float32: _lib.TQ_F32, torch.bfloat16: _lib.TQ_BF16}[w.dtype]
    with torch.cuda.device(w.device):
        # `w / sf` with a Python float on a CUDA tensor is w * (1/sf) inside torch
        rc = _lib.lib().tq_term_count(w.data_ptr(), dt, w.numel(), float(sf), enc,
                                      _lib.FLAG_RECIP_DIV, count.data_ptr(),
                                      torch.cuda.current_stream(w.device).cuda_stream)
    _lib.check(rc)
    return bit_width * int(count.item())


def use_tensor_cores(model, enable=True, engine="auto"):
    """Switch every supported TRConv2dLayer of `model` to the tcgen05 code-domain conv.
    engine: 'auto' (kind::f16 where exact fp32 accumulation is proven from the weights, else the kind::i8 plane
    engine), 'f16' (raise for an unprovable layer) or 'i8'.
    Returns (switched, skipped) where skipped is a list of (module name, reason)."""
    switched, skipped = [], []
    for name, layer in model.named_modules():
        if isinstance(layer, TRConv2dLayer):
            why = layer.tensor_core_blocker() if enable else None
            if why is None:
                try:
                    layer.use_tensor_cores(enable, engine)
                    switched.append(name)
                except NotImplementedError as e:      # no engine can run this layer exactly (e.g. unprovable and C % 16 != 0)
                    layer.use_tensor_cores(False)
                    skipped.append((name, str(e)))
            else:
                skipped.append((name, why))
        elif isinstance(layer, (TRLinearLayer, TRLSTMLayer)):
            try:
                layer.use_tensor_cores(enable, engine)
                switched.append(name)
            except NotImplementedError as e:
                skipped.append((name, str(e)))
    return switched, skipped


def set_tr_tracking(model, tracking):
    """Switch every TR layer between histogram tracking and quantised inference
    (tr_layer.py:66-76); leaving tracking runs the calibration sweep."""
    for layer in list(model.modules()):
        if isinstance(layer, (TRLinearLayer, TRLSTMLayer, TRConv2dLayer)):
            layer.tracking(tracking)
    return model


class LinearQuantize(nn.Module):
    """Activation quantiser (tr_layer.py:78-104).  While ``tracking`` it accumulates an
    8192-bin histogram over [-50, 50] and passes the input through; afterwards it
    term-reveals the flattened activation with g = 1 and ``data_terms`` terms per value of
    ``encoding``."""

    def __init__(self, data_bits, data_terms, *, encoding="hese"):
        super().__init__()
        _lib.encoding_id(encoding)
        self.encoding = encoding
        self.sf = 1
        self.num_bins = 8192
        self.minv = -50
        self.maxv = 50
        self.register_buffer("hist_bins", torch.zeros(self.num_bins))
        self.tracking = True
        self.data_bits = data_bits
        self.data_terms = data_terms
        self._scratch = None

    def _track(self, x):
        xc = x.detach().contiguous()
        if xc.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise RuntimeError(f"LinearQuantize tracking: unsupported input dtype {xc.dtype} (fp32 / bf16 / fp16)")
        # the kernel adds fp32 counts into hist_bins through a raw pointer: after model.half() / .to(other device)
        # the buffer would be too small or live on another GPU, so it is brought back first (counts stay exact
        # in fp32 up to 2^24 per bin per call)
        if self.hist_bins.dtype != torch.float32 or self.hist_bins.device != xc.device:
            self.hist_bins = self.hist_bins.to(device=xc.device, dtype=torch.float32)
        if not self.hist_bins.is_contiguous() or self.hist_bins.numel() != self.num_bins:
            raise RuntimeError("LinearQuantize.hist_bins must be a contiguous fp32 tensor of num_bins elements")
        if self._scratch is None or self._scratch.device != xc.device:
            self._scratch = torch.zeros(self.num_bins, dtype=torch.int32, device=xc.device)
        dt = tr_cuda._DTYPES[xc.dtype]
        with torch.cuda.device(xc.device):
            rc = _lib.lib().tq_hist_accumulate(
                xc.data_ptr(), dt, xc.numel(), self.hist_bins.data_ptr(), self._scratch.data_ptr(),
                self.num_bins, float(self.minv), float(self.maxv),
                torch.cuda.current_stream(xc.device).cuda_stream)
        _lib.check(rc)

    def forward(self, x):
        if self.tracking:
            if not x.is_cuda:
                raise RuntimeError("input must be a CUDA tensor")
            self._track(x)
            return x
        dims = x.shape
        flat = x.contiguous().view(1, -1, 1, 1)          # tr_layer.py:97
        flat = tr_cuda.tr(flat, self.sf, self.data_bits, 1, self.data_terms, encoding=self.encoding)
        return flat.view(*dims)

    def finish_tracking(self):
        self.sf = mse_profile(self.hist_bins, self.minv, self.maxv, self.data_bits, self.data_terms,
                              encoding=self.encoding)
        self.tracking = False


class _TRBase(nn.Module):
    def _setup(self, device, data_bits, data_terms, weight_bits, group_size, num_terms, encoding):
        _lib.encoding_id(encoding)
        self.encoding = encoding
        self.data_bits = data_bits
        self.data_terms = data_terms
        self.input_quant = LinearQuantize(data_bits, data_terms, encoding=encoding).to(device)
        self.group_size = group_size
        self.num_terms = num_terms
        self.weight_bits = weight_bits

    def _reveal_weight(self, w):
        """w_sf = max|w| / 2^(bits-1) then tr over groups of input channels
        (tr_layer.py:117-121).  Sets self.w_sf, returns the new Parameter."""
        self.w_sf = w.abs().max().item() / 2 ** (self.weight_bits - 1)
        wq = tr_cuda.tr(w.detach().contiguous(), self.w_sf, self.weight_bits, self.group_size,
                        self.num_terms, encoding=self.encoding)
        return nn.Parameter(wq)

    def tracking(self, tracking):
        if not tracking:
            self.input_quant.finish_tracking()
        else:
            self.input_quant.tracking = True


class TRConv2dLayer(_TRBase):
    """Conv2d on term-revealed weights and activations (tr_layer.py:106-132).

    Default forward = the reference's: dequantised activations into the stock fp32 conv.
    After ``use_tensor_cores()`` the same layer computes on the integer term codes with the
    tcgen05 kernel (csrc/tq_gemm.cu): activations are encoded to fp16 codes in NHWC, weights
    are the packed codes of the already term-revealed ``conv.weight``, the exact integer
    accumulator is scaled by ``sf_x * w_sf`` (+ bias) in the epilogue, and the result comes
    back as a channels_last fp32 tensor."""

    def __init__(self, conv_layer, data_bits=8, data_terms=4, weight_bits=8, group_size=1,
                 num_terms=8, *, encoding="hese"):
        super().__init__()
        self._setup(conv_layer.weight.device, data_bits, data_terms, weight_bits, group_size,
                    num_terms, encoding)
        conv_layer.weight = self._reveal_weight(conv_layer.weight)
        self.conv = conv_layer
        # packed operands of the tensor-core path: a NON-PERSISTENT buffer, so that .to(device) / .cuda() move it with
        # the module while state_dict stays the reference's; rebuilt whenever conv.weight or w_sf changed
        self.register_buffer("_tc_weight", None, persistent=False)
        self._tc_plan = None
        self._tc_key = None

    def tensor_core_blocker(self):
        """None if the tcgen05 path supports this layer, else the reason it does not."""
        c = self.conv
        if not isinstance(c, nn.Conv2d) or type(c) is not nn.Conv2d:
            return "not a plain nn.Conv2d"
        if c.groups != 1:
            return "grouped/depthwise conv"
        if c.dilation != (1, 1):
            return "dilated conv"
        if c.stride[0] != c.stride[1] or c.padding[0] != c.padding[1] or isinstance(c.padding, str):
            return "asymmetric stride/padding"
        if c.padding_mode != "zeros":
            return "non-zero padding mode"
        if c.in_channels % 8 or c.out_channels % 4:
            return "channel counts must be multiples of 8 (in) and 4 (out)"
        if self.weight_bits > 10 or self.data_bits > 10:
            return "codes above 2^10 fit neither fp16 codes with a provable fp32 accumulator nor two 8-bit planes"
        if c.weight.dtype != torch.float32:
            return "fp32 weights only"
        return None

    def _weight_key(self):
        w = self.conv.weight
        return (w.data_ptr(), w._version, w.device, float(self.w_sf), int(self.data_bits))

    def use_tensor_cores(self, enable=True, engine="auto"):
        """Pack the term-revealed weight for the tcgen05 conv and PROVE how it can run exactly
        (conv_codes.plan_weight): kind::f16 with as many K-chunk accumulators as the static bound
        act_max * max(sum w+, sum w-) < 2^24 needs, else the kind::i8 plane engine.  engine='f16' raises for a layer
        that cannot be proven, engine='i8' forces the plane engine."""
        if not enable:
            self._tc_weight = None
            self._tc_plan = None
            self._tc_key = None
            return self
        why = self.tensor_core_blocker()
        if why is not None:
            raise NotImplementedError(f"tcgen05 conv path: {why}")
        from . import conv_codes
        w = self.conv.weight.detach()
        sf32 = torch.tensor(self.w_sf, dtype=torch.float32).item()       # what the binding saw
        codes = torch.round(w / sf32)
        if not torch.equal(codes * sf32, w):
            raise RuntimeError("conv.weight is not an integer multiple of w_sf any more")
        O, I, kh, kw = codes.shape
        self._tc_weight = codes.permute(2, 3, 0, 1).reshape(kh * kw, O, I).to(torch.float16).contiguous()
        self._tc_wsf32 = sf32
        self._tc_engine = engine
        # activation codes reach 2^data_bits (HESE rounds 2^bits - 1 up); they are signed unless a ReLU precedes the
        # layer, which the layer cannot know: the proof assumes signed activations (sum of |w|) -- fused executors
        # that know the input is post-ReLU re-plan with signed_act=False (fused._Conv)
        self._tc_plan = conv_codes.plan_weight(self._tc_weight, 1 << self.data_bits, signed_act=True, engine=engine)
        self._tc_key = self._weight_key()
        return self

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        tcw = getattr(self, "_tc_weight", None)
        if tcw is not None and (self._tc_plan is None or self._tc_plan.wgt is not tcw):
            # moved / cast with the module: the plan holds device pointers of the old tensors
            self.use_tensor_cores(True, getattr(self, "_tc_engine", "auto"))
        return out

    def _forward_tensor_cores(self, x):
        from . import conv_codes
        if self._tc_key != self._weight_key():                           # load_state_dict / re-reveal since packing
            self.use_tensor_cores(True, getattr(self, "_tc_engine", "auto"))
        c = self.conv
        q = self.input_quant
        x_nhwc = x.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1)   # physical NHWC view
        codes = tr_cuda.tr_codes(x_nhwc.view(1, -1, 1, 1), q.sf, q.data_bits, 1, q.data_terms,
                                 dtype=torch.float16, encoding=q.encoding).view(x_nhwc.shape)
        sfx32 = torch.tensor(float(q.sf), dtype=torch.float32)
        scale = (sfx32 * torch.tensor(self._tc_wsf32, dtype=torch.float32)).item()   # fp32 product
        out = conv_codes.conv2d_codes(codes, self._tc_weight, c.bias, c.kernel_size, c.stride[0],
                                      c.padding[0], scale, plan=self._tc_plan)
        return out.permute(0, 3, 1, 2)                                   # NCHW shape, channels_last memory

    def forward(self, x):
        if self._tc_weight is not None and not self.input_quant.tracking:
            return self._forward_tensor_cores(x)
        return self.conv(self.input_quant(x))


class TRLinearLayer(_TRBase):
    """Linear on term-revealed weights (tr_layer.py:134-160).

    Default forward = the reference's, quirk included: with STRICT_REFERENCE the quantised input is discarded and the
    float linear runs on the raw input (tr_layer.py:152-154), so there is no integer contraction to run.  After
    ``use_tensor_cores()`` the layer computes what the wrapper evidently intends -- linear(q(x)) -- on the integer term
    codes with the tcgen05 kernel (exact int32 accumulator, sf_x * w_sf and the bias in the epilogue)."""

    def __init__(self, linear_layer, data_bits=8, data_terms=4, weight_bits=8, group_size=1,
                 num_terms=8, *, encoding="hese"):
        super().__init__()
        self._setup(linear_layer.weight.device, data_bits, data_terms, weight_bits, group_size,
                    num_terms, encoding)
        linear_layer.weight = self._reveal_weight(linear_layer.weight)
        self.linear = linear_layer
        self.register_buffer("_tc_weight", None, persistent=False)
        self._tc_plan = None

    def use_tensor_cores(self, enable=True, engine="auto"):
        if not enable:
            self._tc_weight, self._tc_plan = None, None
            return self
        from . import conv_codes
        if self.data_bits > 10 or self.weight_bits > 10:
            raise NotImplementedError("tcgen05 linear path: codes above 2^10")
        self._tc_weight, self._tc_wsf32 = conv_codes.pack_linear_weight(self.linear.weight, self.w_sf)
        self._tc_engine = engine
        self._tc_plan = conv_codes.plan_weight(self._tc_weight, 1 << self.data_bits, signed_act=True, engine=engine)
        self._tc_key = (self.linear.weight.data_ptr(), self.linear.weight._version, float(self.w_sf))
        return self

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        tcw = getattr(self, "_tc_weight", None)
        if tcw is not None and (self._tc_plan is None or self._tc_plan.wgt is not tcw):
            self.use_tensor_cores(True, getattr(self, "_tc_engine", "auto"))
        return out

    def _forward_tensor_cores(self, x):
        from . import conv_codes
        if self._tc_key != (self.linear.weight.data_ptr(), self.linear.weight._version, float(self.w_sf)):
            self.use_tensor_cores(True, getattr(self, "_tc_engine", "auto"))
        q = self.input_quant
        lead = x.shape[:-1]
        x2 = x.contiguous().view(-1, x.shape[-1])
        codes = tr_cuda.tr_codes(x2.view(1, -1, 1, 1), q.sf, q.data_bits, 1, q.data_terms, dtype=torch.float16,
                                 encoding=q.encoding).view(x2.shape)
        scale = (torch.tensor(float(q.sf), dtype=torch.float32) * torch.tensor(self._tc_wsf32, dtype=torch.float32)).item()
        out = conv_codes.linear_codes(codes, self._tc_weight, scale, bias=self.linear.bias,
                                      out_features=self.linear.out_features, plan=self._tc_plan)
        return out.reshape(*lead, self.linear.out_features)

    def forward(self, x):
        if self._tc_weight is not None and not self.input_quant.tracking:
            return self._forward_tensor_cores(x)
        if STRICT_REFERENCE:
            # tr_layer.py:152-154 quantises x and then ignores the result; only the histogram
            # side effect of tracking mode is observable, so that is all that is kept.
            if self.input_quant.tracking:
                self.input_quant(x)
            return self.linear(x)
        return self.linear(self.input_quant(x))


class TRLSTMLayer(_TRBase):
    """nn.LSTM whose layer-0 weights are term-revealed; emb, h0 and c0 share one input
    quantiser (tr_layer.py:162-201).

    Default forward = the reference's: quantised emb / h0 / c0 into the stock cuDNN LSTM.  After
    ``use_tensor_cores()`` the one integer contraction the layer contains -- layer 0's input projection
    W_ih . q(emb_t) for all T x B tokens at once (the recurrent products see fp32 hidden states after t = 0) -- runs on
    the tcgen05 kernel on term codes (exact int32 accumulators, K = 650 zero-padded to 656), layer 0's recurrence is
    evaluated step by step on that projection, and the remaining layers stay on cuDNN."""

    def __init__(self, lstm_layer, data_bits=8, data_terms=4, weight_bits=8, group_size=1,
                 num_terms=8, *, encoding="hese"):
        super().__init__()
        self._setup(lstm_layer.weight_ih_l0.device, data_bits, data_terms, weight_bits, group_size,
                    num_terms, encoding)
        lstm_layer.weight_ih_l0 = self._reveal_weight(lstm_layer.weight_ih_l0)
        self.w_sf_ih = self.w_sf                                                 # (w_sf itself ends up as hh's, like the reference)
        lstm_layer.weight_hh_l0 = self._reveal_weight(lstm_layer.weight_hh_l0)   # w_sf := hh's
        self.lstm = lstm_layer
        self.lstm.flatten_parameters()
        self.register_buffer("_tc_weight", None, persistent=False)
        self._tc_plan = None

    def use_tensor_cores(self, enable=True, engine="auto"):
        if not enable:
            self._tc_weight, self._tc_plan = None, None
            return self
        from . import conv_codes
        m = self.lstm
        if not isinstance(m, nn.LSTM) or m.bidirectional or m.batch_first or m.proj_size != 0:
            raise NotImplementedError("tcgen05 LSTM path: unidirectional, time-major nn.LSTM without projections")
        self._tc_weight, self._tc_wsf32 = conv_codes.pack_linear_weight(m.weight_ih_l0, self.w_sf_ih)
        self._tc_engine = engine
        self._tc_plan = conv_codes.plan_weight(self._tc_weight, 1 << self.data_bits, signed_act=True, engine=engine)
        return self

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        tcw = getattr(self, "_tc_weight", None)
        if tcw is not None and (self._tc_plan is None or self._tc_plan.wgt is not tcw):
            self.use_tensor_cores(True, getattr(self, "_tc_engine", "auto"))
        return out

    def input_projection(self, emb):
        """W_ih . q(emb) for every token, [T, B, 4H] fp32 = float(exact int32 accumulator) * (sf_x * w_sf_ih)."""
        from . import conv_codes
        q = self.input_quant
        T, B, I = emb.shape
        codes = tr_cuda.tr_codes(emb.contiguous().view(1, -1, 1, 1), q.sf, q.data_bits, 1, q.data_terms,
                                 dtype=torch.float16, encoding=q.encoding).view(T * B, I)
        scale = (torch.tensor(float(q.sf), dtype=torch.float32) * torch.tensor(self._tc_wsf32, dtype=torch.float32)).item()
        g = conv_codes.linear_codes(codes, self._tc_weight, scale, out_features=4 * self.lstm.hidden_size, plan=self._tc_plan)
        return g.view(T, B, -1)

    def _forward_tensor_cores(self, emb, hidden):
        m = self.lstm
        h0, c0 = (self.input_quant(h) for h in hidden)                           # shared quantiser (tr_layer.py:193-194)
        gin = self.input_projection(emb)
        bias = (m.bias_ih_l0 + m.bias_hh_l0) if m.bias else None
        w_hh_t = m.weight_hh_l0.t()
        h, c = h0[0], c0[0]
        outs = []
        for t in range(gin.shape[0]):                                            # layer 0: i, f, g, o (torch gate order)
            gates = torch.addmm(gin[t] if bias is None else gin[t] + bias, h, w_hh_t)
            i, f, g, o = gates.chunk(4, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
            h = torch.sigmoid(o) * torch.tanh(c)
            outs.append(h)
        y = torch.stack(outs)
        hn, cn = [h], [c]
        if m.num_layers > 1:                                                     # upper layers: cuDNN, unchanged weights
            per = 4 if m.bias else 2
            y, h_up, c_up = torch._VF.lstm(y, (h0[1:].contiguous(), c0[1:].contiguous()), m._flat_weights[per:], m.bias,
                                           m.num_layers - 1, 0.0, False, False, False)
            hn.append(h_up)
            cn.append(c_up)
            return y, (torch.cat([hn[0].unsqueeze(0), h_up]), torch.cat([cn[0].unsqueeze(0), c_up]))
        return y, (h.unsqueeze(0), c.unsqueeze(0))

    def forward(self, emb, hidden):
        if self._tc_weight is not None and not self.input_quant.tracking and not self.lstm.training:
            return self._forward_tensor_cores(emb, hidden)
        embq = self.input_quant(emb)
        hidden_qs = tuple(self.input_quant(h) for h in hidden)
        return self.lstm(embq, hidden_qs)
