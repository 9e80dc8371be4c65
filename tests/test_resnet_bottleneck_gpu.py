"""Bottleneck ResNets (ResNet-50 / 101 / 152, wide ResNet-50-2) on fused.FusedResNet.

The chain is pinned bit for bit to its CPU emulation (test_resnet_bottleneck_host.run_resnet_chain, on
oracle/fused_emul.py's per-conv arithmetic) for every engine and encoding; ragged shapes and the wide network against the
layer-by-layer tensor-core path; graph replay, the uint8 front end and the staleness checks as for BasicBlocks; and the
networks the engine does not run (ResNeXt, dilated stages) refused before any launch, so that select_engine falls back.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

from test_encodings_host import emul_encode
from test_resnet_bottleneck_host import run_resnet_chain

pytestmark = pytest.mark.gpu

CL = torch.channels_last
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


@pytest.fixture(autouse=True)
def _fp32_math(monkeypatch):
    # the float parts (classifier, the layer-by-layer path's BatchNorm) stay true fp32
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)


def _randomise_bn(model, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for mod in model.modules():
            if isinstance(mod, nn.BatchNorm2d):
                n = mod.num_features
                mod.running_mean.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)
                mod.running_var.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.weight.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.bias.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)


def _tq(arch, seed=0, encoding="hese", calib=None, **kw):
    """Random-init torchvision model with randomised BatchNorm statistics, TQ-converted at the benchmarked setting
    (9-bit, g=8, alpha=12, 3 data terms) and calibrated on `calib` when given."""
    import torchvision
    from term_quantization_b200 import cnn_models, inference
    torch.manual_seed(seed)
    base = getattr(torchvision.models, arch)(weights=None, **kw).cuda().eval()
    _randomise_bn(base, seed)
    q = cnn_models.convert_model(base, cnn_models.static_conv_layer_settings(base, 9, 8, 12), 9, 3, encoding=encoding)
    if calib is not None:
        inference.calibrate(q, [calib.float()])
    return q


def _images(n, h, w, seed):
    return torch.randn(n, 3, h, w, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))


def _bit_equal(got, want):
    return got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("engine", ["auto", "i8"])
def test_fused_resnet50_bit_exact_against_cpu_emulation(engine):
    """ResNet-50 at 224^2, batch 2, non-trivial BatchNorm statistics: 16 Bottlenecks (3 launches each) and 4
    downsamples.  The last block's output EQUALS the CPU emulation of the chain bit for bit, and the logits agree with
    an fp64 classifier on the emulated features within 1e-5 relative."""
    from term_quantization_b200 import fused
    x = _images(2, 224, 224, 3).bfloat16()
    q = _tq("resnet50", calib=x).to(memory_format=CL)
    f = fused.FusedResNet(q, engine=engine)
    cap = {}
    with torch.no_grad():
        logits = f(x, capture=cap)
    desc = f.chain_description()
    assert len(desc) == 16 and all(len(b) == 4 for b in desc) and sum(b[3] is not None for b in desc) == 4
    used = sorted({(c["engine"], c["groups"]) for blk in desc for c in blk if c is not None})
    print(f"resnet50 {engine}: engines (engine, accumulator groups) {used}")
    if engine == "auto":
        # as in ResNet-18, the K = 4608 3x3 convs of layer4 need K-chunk accumulators for the static proof
        assert all(e in ("f16", "i8") for e, _ in used) and max(g for e, g in used if e == "f16") >= 2, used
    else:
        assert used == [("i8", 1)]
    emu = run_resnet_chain(desc, cap["stem"].cpu().numpy())
    got = cap["final"].cpu().numpy()
    assert _bit_equal(got, emu), f"{int((got != emu).sum())} of {got.size} block outputs differ"
    feat = torch.from_numpy(emu).double().mean(dim=(1, 2))
    want = feat @ q.fc.weight.detach().double().cpu().t() + q.fc.bias.detach().double().cpu()
    rel = float((logits.double().cpu() - want).abs().max()) / float(want.abs().max())
    print(f"resnet50 {engine}: block outputs bit-exact, logits vs fp64 classifier on the emulated features {rel:.2e}")
    assert rel < 1e-5


@pytest.mark.parametrize("enc", ["hese", "binary", "booth"])
def test_fused_resnet50_encodings_match_emulation(enc, monkeypatch):
    """Every term encoding through the Bottleneck chain at 96^2: the emulation encodes with each layer's encoding."""
    from oracle import fused_emul
    from term_quantization_b200 import fused
    monkeypatch.setattr(fused_emul, "encode", emul_encode)
    x = _images(2, 96, 96, 4).bfloat16()
    q = _tq("resnet50", seed=2, encoding=enc, calib=x).to(memory_format=CL)
    f = fused.FusedResNet(q)
    desc = f.chain_description()
    assert all(c is None or (c["quant"][3] if len(c["quant"]) == 4 else "hese") == enc for blk in desc for c in blk)
    cap = {}
    with torch.no_grad():
        f(x, capture=cap)
    emu = run_resnet_chain(desc, cap["stem"].cpu().numpy())
    got = cap["final"].cpu().numpy()
    assert _bit_equal(got, emu), (enc, int((got != emu).sum()))


@pytest.mark.parametrize("arch,wrapped", [("resnet50", 52), ("wide_resnet50_2", 52), ("resnet152", 154)])
def test_fused_bottleneck_ragged_shape_against_layer_by_layer(arch, wrapped):
    """Batch 3 at 160 x 192 (40 x 48 ... 5 x 6 maps, partial tiles everywhere): the same logits as the layer-by-layer
    tensor-core path up to the fused BatchNorm's 1-2 ulp; the three stem variants agree.  wide_resnet50_2's 3x3 convs
    reach K = 9216; every wrapped conv of these networks has an exact engine (none is refused)."""
    from term_quantization_b200 import fused, tr_layer
    x = _images(3, 160, 192, 8)
    q = _tq(arch, seed=1, calib=x).to(memory_format=CL)
    with torch.no_grad():
        switched, skipped = tr_layer.use_tensor_cores(q)
        assert len(switched) == wrapped and not skipped, skipped
        unfused = q(x.contiguous(memory_format=CL))
        fa = fused.FusedResNet(q)
        a = fa(x)
        b = fused.FusedResNet(q, stem="tcgen05_pool")(x)
        c = fused.FusedResNet(q, stem="cudnn")(x)
    plan = [(blk[1]["w"].shape[0] * blk[1]["w"].shape[2], blk[1]["engine"], blk[1]["groups"]) for blk in fa.chain_description()]
    print(f"{arch}: conv2 (K, engine, groups) per block {plan}")
    scale = float(unfused.abs().max())
    assert torch.equal(a, b)
    assert float((a - c).abs().max()) / scale < 2e-2
    assert float((a - unfused).abs().max()) / scale < 2e-2
    assert float((a.argmax(1) == unfused.argmax(1)).float().mean()) >= 2 / 3


def test_fused_resnet50_graph_replay_u8_and_staleness():
    """ShardedInference(cuda_graphs=True) replays equal eager bit for bit on fresh batches in one buffer; forward_u8
    equals the bf16 path on the same normalised images; load_state_dict or a re-calibration after fusing is refused."""
    from term_quantization_b200 import fused, inference
    calib = _images(2, 96, 128, 1)
    q = _tq("resnet50", seed=3, calib=calib).to(memory_format=CL)
    f = fused.FusedResNet(q)
    batches = [_images(2, 96, 128, s).contiguous(memory_format=CL).bfloat16() for s in (11, 12, 13)]
    with torch.no_grad():
        want = [f(b).clone() for b in batches]
    assert not torch.equal(want[0], want[1])
    runner = inference.ShardedInference(f, "cuda", cuda_graphs=True)
    buf = torch.empty_like(batches[0])
    for b, w in zip(batches, want):
        buf.copy_(b)
        got = runner.forward(buf)
        assert torch.equal(got, w), float((got - w).abs().max())
    assert len(runner._graphs) == 1

    x8 = torch.randint(0, 256, (2, 96, 128, 3), device="cuda", dtype=torch.uint8,
                       generator=torch.Generator(device="cuda").manual_seed(5))
    with torch.no_grad():
        assert torch.equal(f.forward_u8(x8, MEAN, STD), f(inference.normalize_u8(x8, MEAN, STD)))
        assert torch.equal(inference.U8Frontend(f)(x8), f(inference.normalize_u8(x8)))

    q.load_state_dict(q.state_dict())
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f(batches[0])
    f = fused.FusedResNet(q)
    with torch.no_grad():
        f(batches[0])
    inference.calibrate(q, [4 * calib.contiguous(memory_format=CL)])     # a new calibration sweep: new scale factors
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f(batches[0])


@pytest.mark.parametrize("arch,kw,why", [("resnext50_32x4d", {}, "grouped"),
                                         ("resnet50", {"replace_stride_with_dilation": [False, True, True]}, "dilated")])
def test_unsupported_bottleneck_networks_refused_before_any_launch(arch, kw, why):
    from term_quantization_b200 import _lib, evaluate_cnn, fused
    q = _tq(arch, calib=_images(2, 64, 64, 2), **kw).to(memory_format=CL)
    n0 = _lib.launch_count()
    with pytest.raises(NotImplementedError, match=why):
        fused.FusedResNet(q)
    assert _lib.launch_count() == n0
    with pytest.raises(NotImplementedError, match="no fused executor"):
        evaluate_cnn.select_engine(q, "fused")
    assert evaluate_cnn.select_engine(q, "auto") is q               # the layer-by-layer tcgen05 path


def test_uncalibrated_bottleneck_network_raises():
    from term_quantization_b200 import _lib, fused
    q = _tq("resnet50").to(memory_format=CL)
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="calibrate the model"):
        fused.FusedResNet(q)
    assert _lib.launch_count() == n0


def test_non_tr_downsample_refused():
    from term_quantization_b200 import fused
    q = _tq("resnet50", calib=_images(2, 64, 64, 2)).to(memory_format=CL)
    conv = q.layer2[0].downsample[0]
    q.layer2[0].downsample[0] = conv.conv                          # the plain nn.Conv2d inside the wrapper
    with pytest.raises(NotImplementedError, match="downsample conv must be a TRConv2dLayer"):
        fused.FusedResNet(q)


def _wrapped_macs(arch):
    import torchvision
    m = getattr(torchvision.models, arch)(weights=None).eval()
    macs = []

    def hook(mod, inp, out):
        kh, kw = mod.weight.shape[2:]
        macs.append(out.nelement() * (mod.in_channels // mod.groups) * kh * kw)
    hs = [c.register_forward_hook(hook) for c in m.modules() if isinstance(c, nn.Conv2d)]
    with torch.no_grad():
        m(torch.zeros(1, 3, 224, 224))
    for h in hs:
        h.remove()
    return sum(macs[1:])                                           # the first conv is never wrapped


def test_evaluate_cnn_driver_runs_resnet50_fused(tmp_path):
    """evaluate_cnn -a resnet50 on synthetic data: the float path and the fused engine count the same term-pair
    multiplications, 3 data terms * (alpha / g = 1.5) * the wrapped convs' MACs."""
    from term_quantization_b200 import evaluate_cnn
    res = {}
    for engine in ("float", "fused"):
        res[engine] = evaluate_cnn.main(["-a", "resnet50", "-b", "16", "--images", "32", "--quick", "--engine", engine,
                                         "--out-file", str(tmp_path / f"{engine}.json")])
        assert len(res[engine]["tr-data3"]["accs"]) == 1
    macs = _wrapped_macs("resnet50")
    print("resnet50 wrapped-conv MACs per image:", macs)
    assert res["float"]["tr-data3"]["tmacs"] == res["fused"]["tr-data3"]["tmacs"]
    assert abs(res["float"]["tr-data3"]["tmacs"][0] / (3 * 1.5 * macs) - 1) < 1e-6
