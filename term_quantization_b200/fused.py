"""Fused execution of a TQ-converted ResNet (torchvision BasicBlock or Bottleneck topology).

The reference runs, per wrapped conv: TR encode -> cuDNN conv -> BatchNorm -> ReLU (-> add) as
separate passes over fp32 activations (tr_layer.py:124-126 inside torchvision's BasicBlock).
Here each conv is ONE launch of the tcgen05 kernel whose epilogue applies the BatchNorm affine,
the residual add and the ReLU, and emits the fp16 term codes the *next* conv consumes
(the accumulate -> ReLU/requantise -> encode -> truncate order of verilog/systolic_dla_top.v).
fp32 activations are materialised only where the graph needs them (block outputs, which feed
the next residual add).  The stem (first conv, never wrapped: cnn_models/__init__.py:34-36) stays
unquantised fp32 arithmetic but also runs on the tensor cores (hi/lo fp16 operand pairs, fp32
accumulate: conv_codes.stem_conv7x7s2; `stem="cudnn"` keeps cuDNN's fp32 conv); the row half of its max-pool
runs in the conv's epilogue, BatchNorm + ReLU + the column half + first encode in one pass.  Global average pool and the classifier stay on PyTorch.

Numerics: every conv's accumulator is the exact int32 accumulator of the integer contraction -- by a static proof
from the weight codes (kind::f16 MMAs with K-chunk accumulators) or on the kind::i8 plane engine
(conv_codes.plan_weight; include/tq_b200.h "EXACTNESS CONTRACT") -- and every step of the epilogue is one IEEE fp32
operation (fl32(acc) * scale, fmaf(t, a, b) with a = weight * rsqrt(var + eps), b = fmaf(-mean, a, bias), + residual,
ReLU, the reference's quantise / HESE / truncate), so the whole chain is reproduced bit for bit by
oracle/fused_emul.py on a CPU (tests/test_layers_gpu.py).  Against the reference's own float path (cuDNN fp32 conv and
BatchNorm, 1-2 ulp from fmaf) a value sitting on a quantisation boundary can round differently.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import conv_codes, tr_cuda, tr_layer


def _bn_affine(bn):
    with torch.no_grad():
        a = bn.weight * torch.rsqrt(bn.running_var + bn.eps)
        b = torch.addcmul(bn.bias, -bn.running_mean, a)
    return a.float().contiguous(), b.float().contiguous()


def _quant_key(layer):
    """(sf, bits, terms) of a HESE quantiser, (sf, bits, terms, encoding) of any other: the `next_quant` of the fused
    epilogues, and the key under which the executors keep the codes of one tensor per quantiser."""
    q = layer.input_quant
    key = (float(q.sf), int(q.data_bits), int(q.data_terms))
    return key if q.encoding == "hese" else key + (q.encoding,)


class _Conv:
    """Packed operands of one TRConv2dLayer + the BatchNorm that follows it, and the exactness plan of its
    contraction (conv_codes.plan_weight).  `post_relu`: the executor guarantees non-negative input codes, which
    halves the static accumulator bound (only one sign of the weights can pile up)."""

    def __init__(self, layer, bn, post_relu=True, engine="auto"):
        why = layer.tensor_core_blocker()
        if why is not None:
            raise NotImplementedError(f"fused path: {why}")
        if layer.input_quant.tracking:
            raise RuntimeError("calibrate the model (set_tr_tracking(model, False)) before fusing")
        if layer._tc_weight is None or layer._tc_key != layer._weight_key():
            layer.use_tensor_cores(True, engine)
        self.layer = layer
        self.w = layer._tc_weight
        self.plan = conv_codes.plan_weight(self.w, 1 << int(layer.input_quant.data_bits), signed_act=not post_relu,
                                           engine=engine)
        self.quant = _quant_key(layer)
        sfx32 = torch.tensor(self.quant[0], dtype=torch.float32)
        self.scale = (sfx32 * torch.tensor(layer._tc_wsf32, dtype=torch.float32)).item()
        self.bias = layer.conv.bias
        self.bn = _bn_affine(bn) if bn is not None else None
        c = layer.conv
        self.ks, self.stride, self.pad = c.kernel_size, c.stride[0], c.padding[0]

    def check_fresh(self):
        """The packed weight, scale and quantiser are snapshots: refuse to run on stale ones (re-calibration,
        load_state_dict, .to(device) after fusing)."""
        layer = self.layer
        if layer._tc_weight is not self.w or layer._tc_key != layer._weight_key() or _quant_key(layer) != self.quant:
            raise RuntimeError("the wrapped model changed after fusing (weights, device or scale factors): "
                               "build the fused executor again")

    def __call__(self, codes, residual=None, relu=False, want_f32=True, next_quant=None):
        return conv_codes.conv2d_codes_fused(codes, self.w, self.ks, self.stride, self.pad, self.scale,
                                             bias=self.bias, bn=self.bn, residual=residual, relu=relu,
                                             want_f32=want_f32, next_quant=next_quant, plan=self.plan)


class FusedResNet(nn.Module):
    """Wraps a calibrated, TQ-converted torchvision ResNet built from BasicBlocks (resnet18 / 34) or Bottlenecks
    (resnet50 / 101 / 152, wide_resnet50_2 / 101_2: any base_width, groups 1, no dilation).

    Per BasicBlock: conv1 (BN + ReLU, emits conv2's codes) and conv2 (BN + identity + ReLU, writes the fp32 block
    output and the next block's codes).  Per Bottleneck (stride on the 3x3 conv, torchvision v1.5): conv1 1x1 and
    conv2 3x3/s codes to codes with BN + ReLU, conv3 1x1 with BN + identity + ReLU writing the fp32 block output and
    the next block's codes.  The downsample (1x1/s conv + BN) goes from codes to the fp32 identity.  A ResNeXt
    (grouped conv2), a dilated stage or a downsample that is not a wrapped conv is refused with NotImplementedError
    before anything is launched."""

    def __init__(self, model, stem="tcgen05", engine="auto"):
        """engine: how each conv's exact accumulator is obtained ('auto' | 'f16' | 'i8', conv_codes.plan_weight).
        stem: 'tcgen05' (stem conv on the tensor cores with the horizontal half of the max-pool in its epilogue, then the
        vertical half + BN + ReLU + first encode in one pass: the conv map crosses HBM at half size), 'tcgen05_pool' (the whole stem -- conv, BatchNorm, ReLU, max-pool, first encode -- in ONE
        tensor-core kernel, pooling in the conv epilogue: the 822 MB conv output never reaches HBM; bit-identical, but its
        pooled epilogue makes it 0.53 ms), or 'cudnn' (cuDNN's fp32 conv)."""
        super().__init__()
        if stem not in ("tcgen05", "tcgen05_pool", "cudnn"):
            raise ValueError("stem must be 'tcgen05', 'tcgen05_pool' or 'cudnn'")
        self.stem_mode = stem
        # the whole topology is checked before any _Conv is built: packing and planning a weight launches kernels
        plan = []                                     # per block: ([(conv, bn) of the body], (conv, bn) of the downsample | None)
        for stage in (model.layer1, model.layer2, model.layer3, model.layer4):
            for blk in stage:
                if hasattr(blk, "conv3") and hasattr(blk, "bn3"):
                    body = [(blk.conv1, blk.bn1), (blk.conv2, blk.bn2), (blk.conv3, blk.bn3)]
                elif hasattr(blk, "conv2") and hasattr(blk, "bn2"):
                    body = [(blk.conv1, blk.bn1), (blk.conv2, blk.bn2)]
                else:
                    raise NotImplementedError("FusedResNet expects TQ-converted BasicBlocks or Bottlenecks")
                if not all(isinstance(c, tr_layer.TRConv2dLayer) for c, _ in body):
                    raise NotImplementedError("FusedResNet expects TQ-converted BasicBlocks or Bottlenecks")
                down = None
                if blk.downsample is not None:
                    if not isinstance(blk.downsample[0], tr_layer.TRConv2dLayer):
                        raise NotImplementedError("downsample conv must be a TRConv2dLayer")
                    down = (blk.downsample[0], blk.downsample[1])
                for c, _ in body + ([down] if down else []):
                    why = c.tensor_core_blocker()     # ResNeXt: 'grouped/depthwise conv'; dilated stages: 'dilated conv'
                    if why is not None:
                        raise NotImplementedError(f"fused path: {why}")
                plan.append((body, down))
        self.model = model.to(memory_format=torch.channels_last).eval()
        # every conv input of a BasicBlock or Bottleneck chain is the output of a ReLU (block input / the body convs'
        # outputs), so every _Conv takes the one-sided (post_relu) bound
        self.blocks = [tuple(_Conv(c, bn, engine=engine) for c, bn in body)
                       + ((_Conv(*down, engine=engine) if down else None),) for body, down in plan]
        mp = model.maxpool
        self.fuse_stem = (isinstance(mp, nn.MaxPool2d) and mp.kernel_size in (3, (3, 3)) and mp.stride in (2, (2, 2))
                          and mp.padding in (1, (1, 1)) and mp.dilation in (1, (1, 1)) and not mp.ceil_mode
                          and model.conv1.out_channels % 8 == 0 and self.blocks[0][0].quant[1] <= 10)
        self.stem_bn = _bn_affine(model.bn1)
        c1 = model.conv1
        self.stem_w = None
        if (stem != "cudnn" and self.fuse_stem and tuple(c1.weight.shape[1:]) == (3, 7, 7) and c1.stride == (2, 2)
                and c1.padding == (3, 3) and c1.dilation == (1, 1) and c1.groups == 1 and c1.bias is None
                and c1.out_channels <= 64):
            # both tensor-core stems pool the raw conv sums and apply the BatchNorm affine after: sign(slope) goes into
            # the weights, |slope| into stem_bn_pool (conv_codes.stem_pool_operands)
            self.stem_w, self.stem_bn_pool = conv_codes.stem_pool_operands(c1.weight, self.stem_bn)
        # (no stem scratch is kept here: each stem call allocates its folded image, so that under CUDA-graph capture it
        # comes from that graph's private pool, and a later, larger call cannot free memory a captured graph still writes)

    @staticmethod
    def _encode(x_nhwc, quant):
        sf, bits, terms = quant[:3]
        return tr_cuda.tr_codes(x_nhwc.view(1, -1, 1, 1), sf, bits, 1, terms, dtype=torch.float16,
                                encoding=quant[3] if len(quant) == 4 else "hese").view(x_nhwc.shape)

    def chain_description(self):
        """The fused chain as plain data (integer weight codes, fp32 scale, BatchNorm affine, quantiser per conv), one
        (conv1, conv2, down) tuple per BasicBlock and one (conv1, conv2, conv3, down) tuple per Bottleneck (down: None
        without a downsample): what a CPU emulation needs to reproduce the block outputs bit for bit
        (oracle/fused_emul.run_resnet_chain for BasicBlocks)."""
        def d(c):
            if c is None:
                return None
            return {"w": c.w.cpu().numpy().astype("int32"), "ks": tuple(c.ks), "stride": c.stride, "pad": c.pad,
                    "scale": c.scale, "bias": None if c.bias is None else c.bias.detach().float().cpu().numpy(),
                    "bn": None if c.bn is None else (c.bn[0].cpu().numpy(), c.bn[1].cpu().numpy()),
                    "quant": c.quant, "engine": c.plan.engine, "groups": c.plan.groups}
        return [tuple(d(c) for c in blk) for blk in self.blocks]

    @torch.no_grad()
    def forward_u8(self, x_u8_nhwc, mean, std):
        """uint8 [N, H, W, 3] images (1 byte per value over PCIe): ToTensor + Normalize happen inside the stem's fold
        pass when the two-launch tensor-core stem runs; otherwise the images are normalised first (same values)."""
        H, W = x_u8_nhwc.shape[1], x_u8_nhwc.shape[2]
        if (self.fuse_stem and self.stem_w is not None and self.stem_mode != "tcgen05_pool" and H % 2 == 0 and W % 2 == 0
                and (H // 2) * (W // 2) >= 128):
            return self.forward(x_u8_nhwc, u8_norm=(tuple(mean), tuple(std)))
        from . import inference
        return self.forward(inference.normalize_u8(x_u8_nhwc, mean, std))

    def forward(self, x, capture=None, u8_norm=None):
        """x: [N, 3, H, W] images, fp32 or bf16 / fp16 (16-bit images are used as they are: the values the
        reference would see after `images.float()`), any memory format (channels_last avoids a copy).
        capture: optional dict that receives 'stem' (the fp32 NHWC tensor reaching layer1) and 'final' (the
        last block's fp32 NHWC output) -- the two ends of the chain the CPU emulation checks.
        u8_norm: (mean, std) when x is a uint8 [N, H, W, 3] batch (see forward_u8)."""
        m = self.model
        if not torch.cuda.is_current_stream_capturing():
            for blk in self.blocks:
                for c in blk:
                    if c is not None:
                        c.check_fresh()
        if u8_norm is not None:
            # uint8 NHWC batch: normalisation inside the fold pass of the two-launch tensor-core stem (forward_u8 checked)
            q0 = self.blocks[0][0].quant
            y, _ = conv_codes.stem_conv7x7s2_u8(x, u8_norm[0], u8_norm[1], self.stem_w, cout=m.conv1.out_channels, rowmax=True)
            cur, c0 = conv_codes.bn_relu_maxpool_encode(y, self.stem_bn_pool, relu=True, next_quant=q0, rowmax=True)
            codes = {q0: c0}
        elif self.fuse_stem:
            x = x.contiguous(memory_format=torch.channels_last)
            # stem conv (never wrapped, fp32 arithmetic), then bn1 + relu + maxpool + first encode in one pass
            q0 = self.blocks[0][0].quant
            if self.stem_w is not None and x.shape[2] % 2 == 0 and x.shape[3] % 2 == 0 \
                    and (x.shape[2] // 2) * (x.shape[3] // 2) >= 128:
                if self.stem_mode == "tcgen05_pool":
                    # conv + bn1 + relu + maxpool + first encode: one tensor-core kernel
                    cur, c0, _ = conv_codes.stem_conv_pool(x.permute(0, 2, 3, 1), self.stem_w, self.stem_bn_pool, relu=True,
                                                           next_quant=q0)
                else:
                    # conv + row max of the pool window, then column max + bn1 + relu + first encode
                    y, _ = conv_codes.stem_conv7x7s2(x.permute(0, 2, 3, 1), self.stem_w, cout=m.conv1.out_channels,
                                                     rowmax=True)
                    cur, c0 = conv_codes.bn_relu_maxpool_encode(y, self.stem_bn_pool, relu=True, next_quant=q0, rowmax=True)
            else:
                y = m.conv1(x.float()).permute(0, 2, 3, 1)
                cur, c0 = conv_codes.bn_relu_maxpool_encode(y, self.stem_bn, relu=True, next_quant=q0)
            codes = {q0: c0}                             # quantiser -> fp16 codes of `cur`
        else:
            x = x.contiguous(memory_format=torch.channels_last)
            x = m.maxpool(m.relu(m.bn1(m.conv1(x.float()))))
            cur = x.permute(0, 2, 3, 1)                  # fp32 [N, H, W, C], contiguous
            codes = {}
        if capture is not None:
            capture["stem"] = cur
        for i, (*body, down) in enumerate(self.blocks):
            def get(q):
                if q not in codes:
                    codes[q] = self._encode(cur, q)
                return codes[q]
            identity = cur if down is None else down(get(down.quant), want_f32=True)[0]
            # conv1 (and a Bottleneck's conv2): codes to the next body conv's codes, BN + ReLU in the epilogue
            mid = get(body[0].quant)
            for c, c_next in zip(body[:-1], body[1:]):
                _, mid = c(mid, relu=True, want_f32=False, next_quant=c_next.quant)
            nxt = self.blocks[i + 1][0].quant if i + 1 < len(self.blocks) else None
            cur, out_codes = body[-1](mid, residual=identity, relu=True, want_f32=True, next_quant=nxt)
            codes = {nxt: out_codes} if nxt is not None else {}
        if capture is not None:
            capture["final"] = cur
        y = cur.permute(0, 3, 1, 2)                      # NCHW shape, channels_last memory
        return m.fc(torch.flatten(m.avgpool(y), 1))


def _first_conv_ok(c):
    """Is this unwrapped first conv one tq_first_conv3x3_fused runs (3 -> 32 / 64 channels, 3x3, pad 1, stride 1 / 2)?"""
    return (c.in_channels == 3 and c.out_channels in (32, 64) and c.kernel_size == (3, 3) and c.padding == (1, 1)
            and c.stride in ((1, 1), (2, 2)) and c.dilation == (1, 1) and c.groups == 1 and c.weight.dtype == torch.float32)


def _square(pool):
    """nn.MaxPool2d with one window size / stride / padding for both axes (what tq_maxpool2d_f16 takes)."""
    def one(v):
        return v if isinstance(v, int) else (v[0] if v[0] == v[1] else None)
    k, s, p = one(pool.kernel_size), one(pool.stride if pool.stride is not None else pool.kernel_size), one(pool.padding)
    return k is not None and s is not None and p is not None and k <= 7 and 2 * p <= k


class FusedVGG(nn.Module):
    """Fused execution of a TQ-converted torchvision VGG (`features` = conv [-> BatchNorm] -> ReLU [-> MaxPool 2x2]
    chains; BASELINE.json configs[2]).  Every wrapped conv is one launch of the tcgen05 kernel with bias,
    BatchNorm affine and ReLU in the epilogue, emitting directly the fp16 term codes of the NEXT wrapped conv's
    quantiser.  Max-pooling runs on those codes: for g = 1 the truncated code of every encoding (HESE, binary, Booth) is
    a monotone non-decreasing function of the (post-ReLU, non-negative) value, so maxpool(code(x)) == code(maxpool(x))
    exactly and no fp32 activation is materialised between the first and the last conv (tests/test_oracle.py and
    tests/test_encodings_host.py check the monotonicity exhaustively).  The first conv (never wrapped, cnn_models/__init__.py:34-36) stays on cuDNN fp32."""

    def __init__(self, model):
        super().__init__()
        self.model = model.to(memory_format=torch.channels_last).eval()
        mods = list(model.features.children())
        if not isinstance(mods[0], nn.Conv2d) or isinstance(mods[0], tr_layer.TRConv2dLayer):
            raise NotImplementedError("FusedVGG expects an unwrapped first conv")
        self.stages = []                     # (kind, payload): 'torch' module | 'conv' (_Conv, relu) | 'pool' module
        i = 0
        post_relu = False                    # is the tensor reaching the next conv the output of a ReLU (or a pool of one)?
        while i < len(mods):
            m = mods[i]
            if isinstance(m, nn.ReLU):
                post_relu = True
            elif not isinstance(m, nn.MaxPool2d) and not isinstance(m, tr_layer.TRConv2dLayer):
                post_relu = False
            if isinstance(m, tr_layer.TRConv2dLayer):
                bn = None
                relu = False
                j = i + 1
                if j < len(mods) and isinstance(mods[j], nn.BatchNorm2d):
                    bn = mods[j]
                    j += 1
                if j < len(mods) and isinstance(mods[j], nn.ReLU):
                    relu = True
                    j += 1
                self.stages.append(("conv", (_Conv(m, bn, post_relu=post_relu), relu)))
                post_relu = relu
                i = j
            elif isinstance(m, nn.MaxPool2d):
                if m.dilation not in (1, (1, 1)) or m.ceil_mode:
                    raise NotImplementedError("FusedVGG: unsupported max-pool")
                self.stages.append(("pool", m))
                i += 1
            else:
                self.stages.append(("torch", m))
                i += 1
        self.first_tr = next(k for k, (kind, _) in enumerate(self.stages) if kind == "conv")
        if any(kind == "torch" for kind, _ in self.stages[self.first_tr:]):
            raise NotImplementedError("FusedVGG: unexpected module after the first wrapped conv")
        # every conv but the last must be followed (through pools) by a conv and end in a ReLU (pooling on codes)
        convs = [k for k, (kind, _) in enumerate(self.stages) if kind == "conv"]
        for k in convs[:-1]:
            if not self.stages[k][1][1]:
                raise NotImplementedError("FusedVGG: conv without ReLU before a quantiser")

    def chain_description(self):
        """The stages after the first wrapped conv's quantiser as plain data for oracle/fused_emul.run_vgg_chain:
        ('conv', dict, relu) and ('pool', kernel, stride, padding)."""
        out = []
        for kind, payload in self.stages[self.first_tr:]:
            if kind == "conv":
                c, relu = payload
                out.append(("conv", {"w": c.w.cpu().numpy().astype("int32"), "ks": tuple(c.ks), "stride": c.stride, "pad": c.pad,
                                     "scale": c.scale, "bias": None if c.bias is None else c.bias.detach().float().cpu().numpy(),
                                     "bn": None if c.bn is None else (c.bn[0].cpu().numpy(), c.bn[1].cpu().numpy()),
                                     "quant": c.quant, "engine": c.plan.engine, "groups": c.plan.groups}, bool(relu)))
            else:
                one = lambda v: v if isinstance(v, int) else v[0]   # noqa: E731
                out.append(("pool", one(payload.kernel_size), one(payload.stride if payload.stride is not None else payload.kernel_size),
                            one(payload.padding)))
        return out

    @torch.no_grad()
    def forward(self, x, capture=None):
        """capture: optional dict that receives 'stem_codes' (the fp16 codes reaching the first wrapped conv) and 'final'
        (the fp32 NHWC map the average pool reads) -- the two ends of the chain the CPU emulation checks."""
        m = self.model
        if not torch.cuda.is_current_stream_capturing():
            for kind, payload in self.stages:
                if kind == "conv":
                    payload[0].check_fresh()
        x = x.float().contiguous(memory_format=torch.channels_last)
        convs = [k for k, (kind, _) in enumerate(self.stages) if kind == "conv"]
        q0 = self.stages[convs[0]][1][0].quant
        stem = [mod for _, mod in self.stages[:self.first_tr]]
        if (len(stem) == 3 and isinstance(stem[0], nn.Conv2d) and isinstance(stem[1], nn.BatchNorm2d)
                and isinstance(stem[2], nn.ReLU) and stem[0].out_channels % 4 == 0):
            # unwrapped first conv on cuDNN fp32; its BatchNorm + ReLU + the first wrapped conv's encode in ONE pass
            # (tq_bn_act_encode) instead of three passes over the largest activation of the network
            # (the conv's bias rides along as one fp32 add in that pass: torch would add it in a pass of its own over
            # the 1.6 GB map)
            c0 = stem[0]
            if getattr(self, "_stem_bn", None) is None:
                self._stem_bn = _bn_affine(stem[1])
            bias0 = None if c0.bias is None else c0.bias.detach().float().contiguous()
            if _first_conv_ok(c0):
                # 3 -> 32 / 64 channels, 3x3, pad 1: conv + bias + BN + ReLU + encode in ONE kernel of the library (fp32 on
                # the CUDA cores); the fp32 map -- 1.6 GB at batch 128 -- is never written
                if getattr(self, "_stem_w", None) is None:
                    self._stem_w = conv_codes.pack_first_conv_weight(c0.weight)
                _, codes = conv_codes.first_conv3x3_fused(x.permute(0, 2, 3, 1), self._stem_w, c0.stride[0], bias0, self._stem_bn,
                                                          relu=True, next_quant=q0)
            else:
                y = F.conv2d(x, c0.weight, None, c0.stride, c0.padding, c0.dilation, c0.groups).permute(0, 2, 3, 1).contiguous()
                _, codes = conv_codes.bn_act_encode(y, self._stem_bn, relu=True, next_quant=q0, bias=bias0)
        else:
            for mod in stem:                                      # any other stem: module by module on torch
                x = mod(x)
            codes = FusedResNet._encode(x.permute(0, 2, 3, 1), q0)                  # NHWC fp16 codes
        if capture is not None:
            capture["stem_codes"] = codes
        out = None
        for k in range(self.first_tr, len(self.stages)):
            kind, payload = self.stages[k]
            if kind == "conv":
                conv, relu = payload
                nxt = next((self.stages[j][1][0].quant for j in range(k + 1, len(self.stages))
                            if self.stages[j][0] == "conv"), None)
                if nxt is not None:
                    _, codes = conv(codes, relu=relu, want_f32=False, next_quant=nxt)
                else:
                    out, _ = conv(codes, relu=relu, want_f32=True)
                    codes = None
            else:                                                   # max-pool: on the codes (exact), or on the last fp32 map
                if codes is not None and codes.shape[-1] % 8 == 0 and _square(payload):
                    codes = conv_codes.maxpool_codes(codes, payload.kernel_size, payload.stride, payload.padding)
                    continue
                t = codes if codes is not None else out
                t = payload(t.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
                if codes is not None:
                    codes = t.contiguous()
                else:
                    out = t.contiguous()
        if capture is not None:
            capture["final"] = out
        y = out.permute(0, 3, 1, 2)
        return m.classifier(torch.flatten(m.avgpool(y), 1))


class _Depthwise:
    """Packed operands of a wrapped depthwise 3x3 conv (the reference's (16, 1, 16) setting) + its BatchNorm."""

    def __init__(self, layer, bn):
        c = layer.conv
        if not (c.groups == c.in_channels == c.out_channels and c.kernel_size == (3, 3) and c.padding == (1, 1)
                and c.stride in ((1, 1), (2, 2)) and c.dilation == (1, 1) and c.in_channels % 8 == 0):
            raise NotImplementedError("fused depthwise path: 3x3 / pad 1 / stride 1 or 2 depthwise convs with C % 8 == 0")
        if layer.input_quant.tracking:
            raise RuntimeError("calibrate the model (set_tr_tracking(model, False)) before fusing")
        if layer.data_bits > 11 or layer.weight_bits > 16:
            raise NotImplementedError("fused depthwise path: int32 accumulator needs data_bits <= 11, weight_bits <= 16")
        self.layer = layer
        self.w, wsf32 = conv_codes.pack_depthwise_weight(c.weight, layer.w_sf)
        self.quant = _quant_key(layer)
        self.scale = (torch.tensor(self.quant[0], dtype=torch.float32) * torch.tensor(wsf32, dtype=torch.float32)).item()
        self.bias = c.bias
        self.bn = _bn_affine(bn) if bn is not None else None
        self.stride = c.stride[0]

    def __call__(self, codes, relu=False, want_f32=False, next_quant=None, post_relu=False):
        return conv_codes.depthwise3x3_codes(codes, self.w, self.stride, self.scale, bias=self.bias, bn=self.bn, relu=relu,
                                             want_f32=want_f32, next_quant=next_quant,
                                             act_unsigned=post_relu and self.quant[1] <= 9)


class FusedMobileNet(nn.Module):
    """Fused execution of a TQ-converted torchvision MobileNet-V2 (BASELINE.json configs[3]).

    Per InvertedResidual block: the 1x1 expand and project convs run on the tcgen05 kernel (BatchNorm, ReLU6, residual
    add and the NEXT layer's term encode in the epilogue) and the depthwise 3x3 conv -- the memory-bound layer -- is one
    kernel from fp16 codes to fp16 codes (tq_depthwise3x3_codes: int32 accumulator, BatchNorm, ReLU6, encode).  The only
    fp32 activations that reach HBM are the block outputs a later residual add needs.  The reference runs every one of
    these layers as TR encode -> cuDNN conv -> BatchNorm -> ReLU6 over fp32 tensors (tr_layer.py:124-126).  The first
    conv (never wrapped, cnn_models/__init__.py:34-36) stays on cuDNN fp32; its BatchNorm + ReLU6 + first encode are one
    pass (tq_bn_act_encode).  Average pool and classifier stay on PyTorch."""

    def __init__(self, model, engine="auto"):
        super().__init__()
        from torchvision.models.mobilenetv2 import InvertedResidual
        self.model = model.to(memory_format=torch.channels_last).eval()
        feats = list(model.features.children())
        stem = list(feats[0].children())
        if not (isinstance(stem[0], nn.Conv2d) and not isinstance(stem[0], tr_layer.TRConv2dLayer)
                and isinstance(stem[1], nn.BatchNorm2d) and isinstance(stem[2], nn.ReLU6)):
            raise NotImplementedError("FusedMobileNet expects an unwrapped conv-BN-ReLU6 stem")
        self.stem_conv, self.stem_bn = stem[0], _bn_affine(stem[1])
        self.blocks = []                                    # (expand | None, depthwise, project, use_res)
        post_relu = True                                    # the stem ends in ReLU6
        for blk in feats[1:-1]:
            if not isinstance(blk, InvertedResidual):
                raise NotImplementedError("FusedMobileNet expects InvertedResidual blocks")
            mods = list(blk.conv.children())
            expand = None
            if len(mods) == 4:                              # Conv2dNormActivation(expand), Conv2dNormActivation(dw), conv, bn
                e = list(mods[0].children())
                expand = _Conv(e[0], e[1], post_relu=post_relu, engine=engine)
                mods = mods[1:]
            d = list(mods[0].children())
            dw = _Depthwise(d[0], d[1])
            proj = _Conv(mods[1], mods[2], post_relu=True, engine=engine)      # its input is the depthwise ReLU6 output
            self.blocks.append((expand, dw, proj, blk.use_res_connect))
            post_relu = False                               # block outputs are linear (no activation after the projection)
        last = list(feats[-1].children())
        self.last = _Conv(last[0], last[1], post_relu=False, engine=engine)

    def chain_description(self):
        """Plain data for oracle/fused_emul.run_mobilenet_chain."""
        def conv(c):
            if c is None:
                return None
            return {"w": c.w.cpu().numpy().astype("int32"), "ks": tuple(c.ks), "stride": c.stride, "pad": c.pad,
                    "scale": c.scale, "bias": None if c.bias is None else c.bias.detach().float().cpu().numpy(),
                    "bn": None if c.bn is None else (c.bn[0].cpu().numpy(), c.bn[1].cpu().numpy()),
                    "quant": c.quant, "engine": c.plan.engine, "groups": c.plan.groups}

        def dwd(d):
            return {"w": d.w.cpu().numpy(), "stride": d.stride, "scale": d.scale,
                    "bias": None if d.bias is None else d.bias.detach().float().cpu().numpy(),
                    "bn": None if d.bn is None else (d.bn[0].cpu().numpy(), d.bn[1].cpu().numpy()), "quant": d.quant}
        return {"blocks": [(conv(e), dwd(d), conv(p), bool(r)) for e, d, p, r in self.blocks], "last": conv(self.last)}

    @torch.no_grad()
    def forward(self, x, capture=None):
        m = self.model
        if not torch.cuda.is_current_stream_capturing():
            for expand, dw, proj, _ in self.blocks:
                for c in (expand, proj):
                    if c is not None:
                        c.check_fresh()
                if _quant_key(dw.layer) != dw.quant:
                    raise RuntimeError("the wrapped model was re-calibrated after fusing: build the fused executor again")
            self.last.check_fresh()
        x = x.contiguous(memory_format=torch.channels_last)
        first = self.blocks[0][0] or self.blocks[0][1]
        c0 = self.stem_conv
        if _first_conv_ok(c0):
            # conv 3 -> 32 (3x3 / stride 2) + BN + ReLU6 + the first wrapped layer's encode in one kernel of the library
            if getattr(self, "_stem_w", None) is None:
                self._stem_w = conv_codes.pack_first_conv_weight(c0.weight)
            bias0 = None if c0.bias is None else c0.bias.detach().float().contiguous()
            _, codes = conv_codes.first_conv3x3_fused(x.float().permute(0, 2, 3, 1), self._stem_w, c0.stride[0], bias0,
                                                      self.stem_bn, relu="relu6", next_quant=first.quant)
        else:
            y = c0(x.float()).permute(0, 2, 3, 1)                               # fp32 NHWC (channels_last memory)
            _, codes = conv_codes.bn_act_encode(y.contiguous(), self.stem_bn, relu="relu6", next_quant=first.quant)
        if capture is not None:
            capture["stem_codes"] = codes
        cur = None                                                              # fp32 block output, when a residual needs it
        for i, (expand, dw, proj, use_res) in enumerate(self.blocks):
            h = codes
            if expand is not None:
                _, h = expand(h, relu="relu6", want_f32=False, next_quant=dw.quant)
            _, h = dw(h, relu="relu6", next_quant=proj.quant, post_relu=True)   # its input: ReLU6 of the expand conv / stem
            nxt = self.blocks[i + 1] if i + 1 < len(self.blocks) else None
            nq = ((nxt[0] or nxt[1]).quant if nxt is not None else self.last.quant)
            need_f32 = nxt is not None and nxt[3]                               # the next block adds this output back
            cur, codes = proj(h, residual=cur if use_res else None, relu=False, want_f32=need_f32, next_quant=nq)
        out, _ = self.last(codes, relu="relu6", want_f32=True)
        if capture is not None:
            capture["final"] = out
        y = out.permute(0, 3, 1, 2)
        return m.classifier(torch.flatten(nn.functional.adaptive_avg_pool2d(y, (1, 1)), 1))


def _param_key(t):
    return None if t is None else (t.data_ptr(), t._version, t.device)


class _FusedLanguageModel(nn.Module):
    """What FusedLSTM and FusedRNN share: the TRLinearLayer decoder on term codes (its input codes, linear_codes for
    forward, linear_codes_nll for nll, the padded bias and scale), the staleness checks, and forward / nll around the
    cell-specific _recurrence(input, hidden) -> (y [T, B, H] of the last layer, hidden state out).  A subclass
    switches the decoder to its tensor-core path (use_tensor_cores) before it calls _init_decoder and sets _key."""

    def _init_decoder(self):
        dec = self.model.decoder
        self.dec_scale = (torch.tensor(float(dec.input_quant.sf), dtype=torch.float32)
                          * torch.tensor(dec._tc_wsf32, dtype=torch.float32)).item()
        # the decoder bias padded to the packed weight's rows once, so that linear_codes allocates nothing next to its output
        _, out_pad, _ = dec._tc_weight.shape
        self.dec_bias = None
        if dec.linear.bias is not None:
            self.dec_bias = torch.zeros(out_pad, dtype=torch.float32, device=dec.linear.bias.device)
            self.dec_bias[:dec.linear.out_features] = dec.linear.bias.detach()

    def _decoder_snapshot(self):
        dec = self.model.decoder
        return [_param_key(dec.linear.weight), _param_key(dec.linear.bias), float(dec.w_sf), dec._tc_weight,
                _quant_key(dec)]

    def check_fresh(self):
        """Weights, packed operands and scale factors are snapshots: refuse stale ones (load_state_dict, in-place
        updates, .to(device), re-calibration after fusing) and a model switched back to training or tracking."""
        if self.training or self.model.training:
            raise RuntimeError(f"{type(self).__name__} runs inference only: call .eval() first")
        if any(q.tracking for q in self._quantisers()):
            raise RuntimeError("the wrapped model is tracking (calibrating) again: finish the calibration and build the "
                               "fused executor again")
        key = self._snapshot()
        if any(a is not b if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor) else a != b
               for a, b in zip(key, self._key)):
            raise RuntimeError("the wrapped model changed after fusing (weights, device or scale factors): "
                               "build the fused executor again")

    def _decoder_codes(self, input, hidden):
        """The chain forward and nll share: the recurrence, then the decoder's input quantiser.  Returns (the decoder's
        fp16 input codes [T*B, Kp] at the packed weight's width, so that the decoder copies nothing; the hidden state
        out; y).  The recurrence's temporaries are gone before the decoder runs."""
        if not torch.cuda.is_current_stream_capturing():
            self.check_fresh()
        dec = self.model.decoder
        y, hidden = self._recurrence(input, hidden)
        T, B, H = y.shape
        q = dec.input_quant
        codes = torch.zeros((T * B, dec._tc_weight.shape[2]), dtype=torch.float16, device=y.device)
        codes[:, :H] = tr_cuda.tr_codes(y.view(1, -1, 1, 1), q.sf, q.data_bits, 1, q.data_terms, dtype=torch.float16,
                                        encoding=q.encoding).view(T * B, H)
        return codes, hidden, y

    def _decoded(self, input, hidden):
        """_decoder_codes, then the decoder's linear(q(y)) on term codes.  Returns (decoded [T*B, ntoken] fp32, a column
        slice of the decoder's padded output; the hidden state out; y; the decoder's fp16 input codes [T*B, H])."""
        codes, hidden, y = self._decoder_codes(input, hidden)
        dec = self.model.decoder
        decoded = conv_codes.linear_codes(codes, dec._tc_weight, self.dec_scale, bias=self.dec_bias,
                                          out_features=dec.linear.out_features, plan=dec._tc_plan)
        return decoded, hidden, y, codes[:, :y.shape[2]]

    @torch.no_grad()
    def forward(self, input, hidden, capture=None):
        """input: int64 [T, B] tokens; hidden: the hidden state RNNModel.forward takes.  capture: optional dict that
        receives 'y' (the last layer's fp32 output [T, B, H]), 'codes' (the decoder's fp16 input codes [T*B, H]) and
        'decoded' (the decoder's fp32 output before log_softmax)."""
        decoded, hidden, y, codes = self._decoded(input, hidden)
        if capture is not None:
            capture["y"], capture["codes"], capture["decoded"] = y, codes, decoded
        return F.log_softmax(decoded, dim=1), hidden

    @torch.no_grad()
    def nll(self, input, targets, hidden):
        """Per-token negative log-likelihood of `targets` (int64 [T*B], the next tokens in forward's row order) under
        the model: the chain of forward up to the decoder's input codes, then the decoder with the loss epilogue
        (conv_codes.linear_codes_nll), which reduces each row of logits inside the decoder and never writes them.
        Equals nll_loss(forward(input, hidden)[0], targets, reduction='none') within 4e-6 * max(|ref|, 1) of fp64 over
        the decoder output, without allocating any [T*B, ntoken] tensor.  Returns (loss fp32 [T*B], the hidden state
        out); a target outside [0, ntoken) gives NaN for its token."""
        T, B = input.shape
        name = type(self).__name__
        if targets.dtype != torch.int64 or targets.dim() != 1 or targets.shape[0] != T * B:
            raise ValueError(f"{name}.nll expects int64 targets [T*B] = [{T * B}], got {targets.dtype} "
                             f"{tuple(targets.shape)}")
        if targets.device != input.device:
            raise RuntimeError(f"{name}.nll: targets on {targets.device}, tokens on {input.device}")
        codes, hidden, _ = self._decoder_codes(input, hidden)
        dec = self.model.decoder
        loss = conv_codes.linear_codes_nll(codes, dec._tc_weight, self.dec_scale, targets, bias=self.dec_bias,
                                           out_features=dec.linear.out_features, plan=dec._tc_plan)
        return loss, hidden


class FusedLSTM(_FusedLanguageModel):
    """Fused execution of a calibrated, TQ-converted RNNModel('LSTM', ...) (BASELINE.json configs[4]): an nn.Embedding
    encoder, a TRLSTMLayer rnn and a TRLinearLayer decoder.  forward(input, hidden) -> (log_probs [T*B, ntoken], (hn, cn))
    follows RNNModel.forward, so a bptt loop carries the hidden state across chunks unchanged.

    Chain: embedding gather -> the rnn's shared quantiser on h0 / c0 -> layer 0's exact integer input projection on
    tcgen05 (TRLSTMLayer.input_projection) -> tq_lstm_recurrence (all T steps in one persistent kernel) -> for every
    upper layer an fp32 GEMM y . W_ih^T (torch.mm: true fp32 unless torch.backends.cuda.matmul.allow_tf32 is set; those
    weights are not term-revealed, as in the reference) and the recurrence kernel -> the decoder's linear(q(y)) on term
    codes (exact int32 accumulator, scale and bias in the epilogue) -> log_softmax.  Building the executor switches the rnn and decoder layers to their tensor-core paths (use_tensor_cores).
    The recurrence is fp32 with a fixed summation order: bit-identical from run to run and under CUDA-graph replay, within
    1e-5 of an fp64 recurrence, not bit-comparable with cuDNN or the step-wise loop of TRLSTMLayer.

    nll(input, targets, hidden) runs the same chain up to the decoder's input codes and ends in the decoder with the loss
    epilogue (conv_codes.linear_codes_nll): the per-token loss for perplexity, with neither the [T*B, ntoken] logits nor
    the log-probabilities ever written."""

    def __init__(self, model):
        super().__init__()
        rnn, dec = getattr(model, "rnn", None), getattr(model, "decoder", None)
        if getattr(model, "rnn_type", None) != "LSTM" or not isinstance(rnn, tr_layer.TRLSTMLayer) \
                or not isinstance(getattr(model, "encoder", None), nn.Embedding):
            raise NotImplementedError("FusedLSTM expects a TQ-converted RNNModel('LSTM', ...): nn.Embedding encoder, "
                                      "TRLSTMLayer rnn (GRU and vanilla RNN models run on FusedRNN)")
        m = rnn.lstm
        if type(m) is not nn.LSTM or m.bidirectional or m.batch_first or m.proj_size != 0:
            raise NotImplementedError("FusedLSTM: unidirectional, time-major nn.LSTM without projections only "
                                      f"(bidirectional={m.bidirectional}, batch_first={m.batch_first}, proj_size={m.proj_size})")
        if not isinstance(dec, tr_layer.TRLinearLayer) or dec.linear.in_features != m.hidden_size:
            raise NotImplementedError("FusedLSTM expects a TRLinearLayer decoder over the LSTM's hidden state")
        for name, p in m.named_parameters():
            if p.dtype != torch.float32 or not p.is_cuda:
                raise NotImplementedError(f"FusedLSTM: fp32 CUDA parameters only ({name} is {p.dtype} on {p.device})")
        hmax = conv_codes.lstm_max_hidden(m.weight_hh_l0.device)
        if m.hidden_size > hmax:
            raise NotImplementedError(f"FusedLSTM: hidden size {m.hidden_size} exceeds what the recurrence kernel keeps in "
                                      f"shared and tensor memory on this device (H <= {hmax})")
        if rnn.input_quant.tracking or dec.input_quant.tracking:
            raise RuntimeError("calibrate the model (set_tr_tracking(model, False)) before fusing")
        if model.training:
            raise RuntimeError("FusedLSTM runs inference only: call model.eval() first")
        dec.use_tensor_cores()                       # raises before any launch when the decoder's codes do not fit
        rnn.use_tensor_cores()
        self.model = model
        self.layers = []                             # per layer: (w_ih or None for layer 0, w_hh, combined bias or None)
        with torch.no_grad():
            for l in range(m.num_layers):
                bias = None
                if m.bias:
                    bias = (getattr(m, f"bias_ih_l{l}") + getattr(m, f"bias_hh_l{l}")).contiguous()
                self.layers.append((None if l == 0 else getattr(m, f"weight_ih_l{l}"), getattr(m, f"weight_hh_l{l}"), bias))
        self._init_decoder()
        self._key = self._snapshot()
        self.train(False)

    def _quantisers(self):
        return self.model.rnn.input_quant, self.model.decoder.input_quant

    def _snapshot(self):
        rnn = self.model.rnn
        return [[_param_key(p) for p in rnn.lstm.parameters()], _param_key(self.model.encoder.weight), float(rnn.w_sf_ih),
                rnn._tc_weight, _quant_key(rnn)] + self._decoder_snapshot()

    def _recurrence(self, input, hidden):
        """Embedding, the shared quantiser on h0 / c0, then every layer's input projection and recurrence kernel.
        Returns (y [T, B, H] of the last layer, (hn, cn) [layers, B, H])."""
        model = self.model
        rnn = model.rnn
        h0, c0 = (rnn.input_quant(h) for h in hidden)                 # the shared quantiser (tr_layer.py:193-194)
        T, B = input.shape
        hn, cn = [], []
        y = None
        for l, (w_ih, w_hh, bias) in enumerate(self.layers):
            if l == 0:
                gin = rnn.input_projection(model.encoder(input))       # (the embedding is freed with the projection)
            else:
                gin = torch.mm(y.view(T * B, -1), w_ih.t()).view(T, B, -1)
            y, h, c = conv_codes.lstm_recurrence(gin, bias, w_hh, h0[l].contiguous(), c0[l].contiguous())
            del gin                                                     # before the next layer's projection is allocated
            hn.append(h)
            cn.append(c)
        return y, (torch.stack(hn), torch.stack(cn))


class FusedRNN(_FusedLanguageModel):
    """Fused execution of a calibrated, TQ-converted RNNModel('GRU' | 'RNN_TANH' | 'RNN_RELU', ...): an nn.Embedding
    encoder, an nn.GRU / nn.RNN rnn and a TRLinearLayer decoder.  forward(input, hidden) -> (log_probs [T*B, ntoken], hn)
    follows RNNModel.forward with its single hidden tensor [layers, B, H].

    As in the reference, only the decoder is a TR layer: the recurrent weights are not term-revealed and h0 is not
    quantised.  Chain: embedding gather -> per layer an fp32 GEMM x . W_ih^T (+ b_ih for the GRU; torch.mm / addmm, true
    fp32 unless torch.backends.cuda.matmul.allow_tf32 is set) and the recurrence kernel (conv_codes.gru_recurrence /
    rnn_recurrence: all T steps in one persistent launch) -> the decoder's linear(q(y)) on term codes -> log_softmax, or
    the decoder's loss epilogue for nll, exactly as FusedLSTM.  The recurrence is fp32 with a fixed summation order:
    bit-identical from run to run and under CUDA-graph replay, within 1e-5 of an fp64 recurrence, not bit-comparable
    with cuDNN."""

    def __init__(self, model):
        super().__init__()
        kind = getattr(model, "rnn_type", None)
        rnn, dec = getattr(model, "rnn", None), getattr(model, "decoder", None)
        if kind == "LSTM":
            raise NotImplementedError("FusedRNN runs GRU and vanilla RNN models: use FusedLSTM for RNNModel('LSTM', ...)")
        cls = {"GRU": nn.GRU, "RNN_TANH": nn.RNN, "RNN_RELU": nn.RNN}.get(kind)
        if cls is None or type(rnn) is not cls or not isinstance(getattr(model, "encoder", None), nn.Embedding):
            raise NotImplementedError("FusedRNN expects a TQ-converted RNNModel('GRU' | 'RNN_TANH' | 'RNN_RELU', ...): "
                                      "nn.Embedding encoder, nn.GRU / nn.RNN rnn")
        self.nonlinearity = None if kind == "GRU" else kind.split("_")[1].lower()
        if cls is nn.RNN and rnn.nonlinearity != self.nonlinearity:
            raise NotImplementedError(f"FusedRNN: an {kind} model with a {rnn.nonlinearity} nn.RNN")
        if rnn.bidirectional or rnn.batch_first:
            raise NotImplementedError("FusedRNN: unidirectional, time-major recurrences only "
                                      f"(bidirectional={rnn.bidirectional}, batch_first={rnn.batch_first})")
        if not isinstance(dec, tr_layer.TRLinearLayer) or dec.linear.in_features != rnn.hidden_size:
            raise NotImplementedError(f"FusedRNN expects a TRLinearLayer decoder over the {kind}'s hidden state")
        for name, p in rnn.named_parameters():
            if p.dtype != torch.float32 or not p.is_cuda:
                raise NotImplementedError(f"FusedRNN: fp32 CUDA parameters only ({name} is {p.dtype} on {p.device})")
        hmax = conv_codes.recurrence_max_hidden(kind, rnn.weight_hh_l0.device)
        if rnn.hidden_size > hmax:
            raise NotImplementedError(f"FusedRNN: hidden size {rnn.hidden_size} exceeds what the {kind} recurrence kernel "
                                      f"keeps in shared and tensor memory on this device (H <= {hmax})")
        if dec.input_quant.tracking:
            raise RuntimeError("calibrate the model (set_tr_tracking(model, False)) before fusing")
        if model.training:
            raise RuntimeError("FusedRNN runs inference only: call model.eval() first")
        dec.use_tensor_cores()                       # raises before any launch when the decoder's codes do not fit
        self.model = model
        self.cell = kind
        # per layer: (w_ih, the bias folded into the input GEMM or None, w_hh, the kernel's bias or None).  The GRU's
        # b_hn multiplies with the reset gate, so b_ih goes into the GEMM and b_hh to the kernel; an RNN adds both.
        self.layers = []
        with torch.no_grad():
            for l in range(rnn.num_layers):
                w_ih, w_hh = getattr(rnn, f"weight_ih_l{l}"), getattr(rnn, f"weight_hh_l{l}")
                b_gemm = b_rec = None
                if rnn.bias:
                    b_ih, b_hh = getattr(rnn, f"bias_ih_l{l}"), getattr(rnn, f"bias_hh_l{l}")
                    if kind == "GRU":
                        b_gemm, b_rec = b_ih, b_hh
                    else:
                        b_rec = (b_ih + b_hh).contiguous()
                self.layers.append((w_ih, b_gemm, w_hh, b_rec))
        self._init_decoder()
        self._key = self._snapshot()
        self.train(False)

    def _quantisers(self):
        return (self.model.decoder.input_quant,)

    def _snapshot(self):
        return [[_param_key(p) for p in self.model.rnn.parameters()],
                _param_key(self.model.encoder.weight)] + self._decoder_snapshot()

    def _recurrence(self, input, hidden):
        """Embedding, then every layer's input GEMM and recurrence kernel.  Returns (y [T, B, H] of the last layer,
        hn [layers, B, H])."""
        T, B = input.shape
        y = self.model.encoder(input)
        hn = []
        for l, (w_ih, b_gemm, w_hh, b_rec) in enumerate(self.layers):
            x = y.view(T * B, -1)
            gin = (torch.mm(x, w_ih.t()) if b_gemm is None else torch.addmm(b_gemm, x, w_ih.t())).view(T, B, -1)
            del x, y                                                    # the layer input, before the kernel's output
            if self.nonlinearity is None:
                y, h = conv_codes.gru_recurrence(gin, b_rec, w_hh, hidden[l].contiguous())
            else:
                y, h = conv_codes.rnn_recurrence(gin, b_rec, w_hh, hidden[l].contiguous(), self.nonlinearity)
            del gin                                                     # before the next layer's GEMM is allocated
            hn.append(h)
        return y, torch.stack(hn)
