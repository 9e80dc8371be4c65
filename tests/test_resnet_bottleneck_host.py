"""Bottleneck ResNets on the fused engine, the host side: the driver's model list, the conversion of ResNet-50, and the
CPU emulation of a Bottleneck chain.

`run_resnet_chain` is the bit-exact CPU emulation of fused.FusedResNet for both block types, built on the per-conv
arithmetic of oracle/fused_emul.py (exact integer conv -> fl32 -> * scale -> fmaf BN -> + residual -> ReLU -> codes).
tests/test_resnet_bottleneck_gpu.py checks the fused chain against it.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import fused_emul
from oracle import tq_oracle as O


def run_resnet_chain(blocks, stem_out):
    """blocks = fused.FusedResNet.chain_description(): (conv1, conv2, down) per BasicBlock -- oracle/fused_emul's own
    run_resnet_chain -- or (conv1, conv2, conv3, down) per Bottleneck.  In a Bottleneck conv1 and conv2 go from codes to
    the next conv's codes with BN + ReLU, and conv3 adds the identity (the block input, or the downsample's fp32 output)
    before its ReLU.  Codes come from fused_emul.encode, so an encoding-aware encode installed there is followed.
    Returns the fp32 [N, h, w, C'] output of the last block."""
    if all(len(b) == 3 for b in blocks):
        return fused_emul.run_resnet_chain(blocks, stem_out)
    cur = np.ascontiguousarray(stem_out, dtype=np.float32)
    for blk in blocks:
        *body, down = blk
        identity = cur if down is None else fused_emul.fused_conv(fused_emul.encode(cur, down["quant"]), down)[0]
        h = fused_emul.encode(cur, body[0]["quant"])
        for c, c_next in zip(body[:-1], body[1:]):
            _, h = fused_emul.fused_conv(h, c, relu=True, next_quant=c_next["quant"])
        cur, _ = fused_emul.fused_conv(h, body[-1], residual=identity, relu=True)
    return cur


def test_driver_takes_the_deeper_resnets():
    from term_quantization_b200 import cnn_models, evaluate_cnn
    assert cnn_models.model_names() == ['alexnet', 'vgg16_bn', 'resnet18', 'efficientnet_b0', 'mobilenet_v2']
    for arch in ("resnet34", "resnet50", "resnet101", "resnet152", "wide_resnet50_2"):
        assert callable(getattr(cnn_models, arch))
        # the parser accepts the name; main() then stops for want of a CUDA device (or runs, on a GPU machine)
        with pytest.raises(SystemExit) as e:
            evaluate_cnn.main(["-a", arch, "--help"])
        assert e.value.code == 0
    with pytest.raises(SystemExit) as e:
        evaluate_cnn.main(["-a", "resnext50_32x4d", "--quick"])
    assert e.value.code == 2                                     # argparse: invalid choice


def test_resnet50_conversion_wraps_52_convs(monkeypatch):
    """Every conv but the stem of ResNet-50 (16 Bottlenecks x 3 + 4 downsamples) becomes a TRConv2dLayer with the
    reference's (9, 8, 12) setting; the stem keeps the 'unquantised' (16, 1, 16) entry and is not wrapped."""
    from torchvision.models import resnet50
    from term_quantization_b200 import cnn_models, tr_layer
    seen = []

    def tr(x, sf, bits, g, alpha, **_):                          # weights as they are: only the settings matter here
        seen.append((bits, g, alpha))
        return x.detach().clone()
    monkeypatch.setattr(tr_layer.tr_cuda, "tr", tr)
    net = resnet50(weights=None)
    params = cnn_models.static_conv_layer_settings(net, 9, 8, 12)
    assert len(params) == 53 and params[0] == (16, 1, 16) and all(p == (9, 8, 12) for p in params[1:])
    q = cnn_models.convert_model(net, params, 9, 3)
    layers = [m for m in q.modules() if isinstance(m, tr_layer.TRConv2dLayer)]
    assert len(layers) == 52 and not isinstance(q.conv1, tr_layer.TRConv2dLayer)
    assert seen == [(9, 8, 12)] * 52
    assert all((m.data_bits, m.data_terms, m.weight_bits, m.group_size, m.num_terms) == (9, 3, 9, 8, 12) for m in layers)
    assert all(isinstance(b.conv3, tr_layer.TRConv2dLayer) for s in (q.layer1, q.layer2, q.layer3, q.layer4) for b in s)
    assert sum(b.downsample is not None and isinstance(b.downsample[0], tr_layer.TRConv2dLayer)
               for s in (q.layer1, q.layer2, q.layer3, q.layer4) for b in s) == 4


def _conv(rng, cin, cout, ks, stride, sf_in, with_bn=True):
    pad = ks // 2
    w = rng.integers(-40, 41, (ks * ks, cout, cin)).astype(np.int32)
    bn = (rng.uniform(0.5, 1.5, cout).astype(np.float32), rng.normal(0, 0.2, cout).astype(np.float32)) if with_bn else None
    return {"w": w, "ks": (ks, ks), "stride": stride, "pad": pad, "scale": float(np.float32(1.3e-4)), "bias": None,
            "bn": bn, "quant": (sf_in, 9, 3)}


def fma32(t, a, b):
    """fmaf(t, a, b) per channel in fp64: t * a is exact there, the sum is rounded to odd (TwoSum error, then the last bit
    forced to 1 when inexact), so the final rounding to fp32 is the single rounding of the exact t * a + b."""
    p = t.astype(np.float64) * a.astype(np.float64)
    b = np.broadcast_to(b.astype(np.float64), p.shape)
    s = p + b
    bb = s - p
    err = (p - (s - bb)) + (b - bb)
    even = (s.view(np.uint64) & 1) == 0
    s = np.where((err != 0) & even, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def _straight(blocks, x):
    """The same chain written out directly: fp64 integer conv of the codes, then every epilogue step rounded to fp32 one
    operation at a time (the BatchNorm as one fused multiply-add: fma32), codes from oracle.tr."""
    def codes(t, q):
        _, c = O.tr(np.ascontiguousarray(t, np.float32).reshape(1, -1, 1, 1), q[0], q[1], 1, q[2], return_codes=True)
        return c.reshape(t.shape).astype(np.float64)

    def conv(c_in, c, res=None, relu=True):
        R, S = c["ks"]
        w = torch.from_numpy(c["w"].astype(np.float64)).view(R, S, *c["w"].shape[1:]).permute(2, 3, 0, 1)
        acc = torch.nn.functional.conv2d(torch.from_numpy(c_in).permute(0, 3, 1, 2), w, None, c["stride"], c["pad"])
        acc = acc.permute(0, 2, 3, 1).numpy()
        t = (acc.astype(np.float32) * np.float32(c["scale"])).astype(np.float32)
        if c["bn"] is not None:
            t = fma32(t, c["bn"][0], c["bn"][1])
        if res is not None:
            t = (t + res).astype(np.float32)
        return np.where(t > 0, t, np.float32(0)).astype(np.float32) if relu else t

    cur = x
    for c1, c2, c3, down in blocks:
        identity = cur if down is None else conv(codes(cur, down["quant"]), down, relu=False)
        h = conv(codes(cur, c1["quant"]), c1)
        h = conv(codes(h, c2["quant"]), c2)
        cur = conv(codes(h, c3["quant"]), c3, res=identity)
    return cur


def test_bottleneck_emulation_equals_a_straight_composition():
    """Two hand-made Bottlenecks (one with a 1x1/s2 downsample and the stride on the 3x3 conv, one with the identity
    shortcut) on a 2 x 9 x 7 map: run_resnet_chain on the 4-tuples equals the composition written out above, bit for
    bit; the 3-tuple path is oracle/fused_emul's own."""
    rng = np.random.default_rng(5)
    x = np.maximum(rng.normal(0, 1, (2, 9, 7, 16)), 0).astype(np.float32)
    sf = lambda v: float(np.float32(v))                                 # noqa: E731
    b1 = (_conv(rng, 16, 8, 1, 1, sf(0.01)), _conv(rng, 8, 8, 3, 2, sf(0.02)), _conv(rng, 8, 32, 1, 1, sf(0.015)),
          _conv(rng, 16, 32, 1, 2, sf(0.01)))
    b2 = (_conv(rng, 32, 8, 1, 1, sf(0.03)), _conv(rng, 8, 8, 3, 1, sf(0.02)), _conv(rng, 8, 32, 1, 1, sf(0.02)), None)
    blocks = [b1, b2]
    got = run_resnet_chain(blocks, x)
    want = _straight(blocks, x)
    assert got.shape == (2, 5, 4, 32) and got.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (got > 0).mean() > 0.2                                        # the chain is not all zeros after the ReLUs
    basic = [(b1[0], _conv(rng, 8, 16, 3, 1, sf(0.02)), None)]
    assert np.array_equal(run_resnet_chain(basic, x), fused_emul.run_resnet_chain(basic, x))
