"""The stem with its 3x3/s2/p1 max-pool split by axis: the conv epilogue takes the max over the window's columns
(stem_conv7x7s2(..., rowmax=True)), the pool pass the max over its rows plus BatchNorm, ReLU and the first encode
(bn_relu_maxpool_encode(..., rowmax=True)).  Both must equal the full-map stem conv followed by bn_relu_maxpool_encode
bit for bit: the fp32 pooled map and the fp16 codes."""
import pytest
import torch

pytestmark = pytest.mark.gpu

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16, "u8": torch.uint8}


def _images(shape, dtype, g):
    N, H, W = shape
    if dtype == torch.uint8:
        return torch.randint(0, 256, (N, H, W, 3), device="cuda", dtype=torch.uint8, generator=g)
    return torch.randn(N, H, W, 3, device="cuda", generator=g).to(dtype).contiguous()


def _check(x, w, bn, relu):
    from term_quantization_b200 import conv_codes
    cout = w.shape[0]

    def stem(w2, rowmax):
        if x.dtype == torch.uint8:
            return conv_codes.stem_conv7x7s2_u8(x, MEAN, STD, w2, cout=cout, rowmax=rowmax)[0]
        return conv_codes.stem_conv7x7s2(x, w2, cout=cout, rowmax=rowmax)[0]

    y = stem(conv_codes.pack_stem_weight(w), False)
    want, _ = conv_codes.bn_relu_maxpool_encode(y, bn, relu=relu)
    nq = (float(want.abs().max()) / 512, 9, 3)
    want, want_codes = conv_codes.bn_relu_maxpool_encode(y, bn, relu=relu, next_quant=nq)
    del y
    w2s, bns = conv_codes.stem_pool_operands(w, bn)          # sign of the slope folded into the weights
    rows = stem(w2s, True)
    N, H, W = x.shape[:3]
    assert rows.shape == (N, H // 2, (W // 2 - 1) // 2 + 1, cout)
    got, codes = conv_codes.bn_relu_maxpool_encode(rows, bns, relu=relu, next_quant=nq, rowmax=True)
    assert got.shape == want.shape
    assert torch.equal(got, want), float((got - want).abs().max())
    assert torch.equal(codes, want_codes)
    got2, none = conv_codes.bn_relu_maxpool_encode(rows, bns, relu=relu, rowmax=True)
    assert none is None and torch.equal(got2, want)


def _operands(cout, g):
    w = torch.randn(cout, 3, 7, 7, device="cuda", generator=g) * 0.1
    a = torch.randn(cout, device="cuda", generator=g)
    a[::5] = 0.0                                               # zero slopes beside negative and positive ones
    b = torch.randn(cout, device="cuda", generator=g)
    return w, (a, b)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("shape", [(3, 224, 224), (2, 64, 96), (2, 50, 38), (1, 226, 222)])
def test_rowmax_stem_equals_full_map_stem(dtype, shape):
    g = torch.Generator(device="cuda").manual_seed(5)
    x = _images(shape, DTYPES[dtype], g)
    w, bn = _operands(64, g)
    for relu in (True, False):
        _check(x, w, bn, relu)


def test_rowmax_stem_narrow_channels():
    """Cout = 32: half of the pool pass's 64-channel box lies beyond the tensor."""
    g = torch.Generator(device="cuda").manual_seed(6)
    w, bn = _operands(32, g)
    _check(_images((2, 64, 96), torch.bfloat16, g), w, bn, True)


@pytest.mark.parametrize("dtype", ["bf16", "u8"])
def test_rowmax_stem_full_batch(dtype):
    g = torch.Generator(device="cuda").manual_seed(7)
    w, bn = _operands(64, g)
    _check(_images((256, 224, 224), DTYPES[dtype], g), w, bn, True)


def test_fused_resnet_logits_equal_full_map_stem(monkeypatch):
    """FusedResNet on the bench's seeded model: the logits of the row-max stem equal those of the full-map stem conv
    followed by bn_relu_maxpool_encode (the same executor with the two stem calls swapped for the full-map pair), for
    bf16 and uint8 images."""
    import bench
    from term_quantization_b200 import conv_codes, fused, inference
    model = bench.build_tq_resnet18("cuda")
    g = torch.Generator(device="cuda").manual_seed(1234)
    images = torch.randn(16, 3, 224, 224, device="cuda", generator=g).bfloat16()
    inference.calibrate(model, [images.float()])
    f = fused.FusedResNet(model.to(memory_format=torch.channels_last))
    x8 = torch.randint(0, 256, (16, 224, 224, 3), device="cuda", dtype=torch.uint8, generator=g)
    with torch.no_grad():
        got, got8 = f(images), f.forward_u8(x8, MEAN, STD)
        w_plain = conv_codes.pack_stem_weight(model.conv1.weight)
        conv, conv_u8, pool = conv_codes.stem_conv7x7s2, conv_codes.stem_conv7x7s2_u8, conv_codes.bn_relu_maxpool_encode
        monkeypatch.setattr(conv_codes, "stem_conv7x7s2",
                            lambda x, w2, scratch=None, cout=None, rowmax=False: conv(x, w_plain, scratch, cout))
        monkeypatch.setattr(conv_codes, "stem_conv7x7s2_u8",
                            lambda x, m, s, w2, scratch=None, cout=None, rowmax=False: conv_u8(x, m, s, w_plain, scratch, cout))
        monkeypatch.setattr(conv_codes, "bn_relu_maxpool_encode",
                            lambda y, bn, relu=True, next_quant=None, rowmax=False: pool(y, f.stem_bn, relu, next_quant))
        want, want8 = f(images), f.forward_u8(x8, MEAN, STD)
    assert torch.equal(got, want)
    assert torch.equal(got8, want8)
