"""Binary and Booth term encodings on every fused kernel, every fused executor, the layers, calibration and drivers.

Each check runs for both encodings against the CPU emulation (tests/test_encodings_host.emul_encode on oracle.tr, which
takes the encoding), bit for bit.  Every kernel check also asserts that some case of its grid gives codes that differ
from HESE's, so a kernel that ignored the encoding could not pass, and that with 'hese' the `_enc` entry points equal
the original ones.
"""
import ctypes

import numpy as np
import pytest
import torch

from test_encodings_host import emul_encode, emul_mse_profile, emul_term_count
from test_fused_encoders_gpu import ACTS, FAST_SFS, check_f32, hard_values, sample_ks, terms_for

pytestmark = pytest.mark.gpu

ENCS = ("binary", "booth")


@pytest.fixture(autouse=True)
def encoding_aware_emulation(monkeypatch):
    """oracle/fused_emul encodes with HESE only; the chains here follow each layer's (sf, bits, terms, encoding).  The
    float paths the layers are compared with stay true fp32 (no TF32)."""
    from oracle import fused_emul
    monkeypatch.setattr(fused_emul, "encode", emul_encode)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)


def check_codes(got, want_f32, quant, what):
    want = emul_encode(np.asarray(want_f32, dtype=np.float32), quant)
    got = got.cpu().numpy().astype(np.int32)
    if not np.array_equal(got, want):
        i = int(np.flatnonzero(got.ravel() != want.ravel())[0])
        raise AssertionError(f"{what}: codes differ at {i}: value {np.asarray(want_f32).ravel()[i]!r} "
                             f"got {got.ravel()[i]} want {want.ravel()[i]}")
    return not np.array_equal(want, emul_encode(np.asarray(want_f32, dtype=np.float32), quant[:3]))


# index of `next_enc` in the argument list of each _enc entry point: dropping it gives the original entry point's
# (conv_codes calls the _enc entry points for every encoding; the originals remain for C callers)
_ENC_ARG = {"tq_conv2d_codes_fused_enc": 22, "tq_conv2d_planes_i8_enc": 24, "tq_stem_conv7x7s2_pool_enc": 16,
            "tq_bn_relu_maxpool_encode_enc": 13, "tq_bn_relu_maxpool_encode_rowmax_enc": 13,
            "tq_depthwise3x3_codes_enc": 18, "tq_bn_act_encode_enc": 12, "tq_first_conv3x3_fused_enc": 16}


class _ViaOriginalEntryPoints:
    """Stands in for libtq_b200 inside conv_codes: every _enc entry point called with TQ_ENC_HESE goes to its original
    entry point, the encoding dropped."""

    def __init__(self, L):
        self._L = L

    def __getattr__(self, name):
        if name not in _ENC_ARG:
            return getattr(self._L, name)
        fn, old = getattr(self._L, name), getattr(self._L, name[:-len("_enc")])
        k = _ENC_ARG[name]
        assert fn.argtypes[:k] + fn.argtypes[k + 1:] == old.argtypes and fn.argtypes[k] is ctypes.c_int, name

        def call(*args):
            assert args[k] == 0, name                    # TQ_ENC_HESE
            return old(*args[:k], *args[k + 1:])
        return call


@pytest.fixture
def hese_vs_original(monkeypatch):
    """run(fn) -> (outputs of fn through the _enc entry points with TQ_ENC_HESE, outputs through the original ones)."""
    from term_quantization_b200 import _lib, conv_codes

    class Shim:
        def __getattr__(self, name):
            return getattr(_lib, name)

        def lib(self):
            return _ViaOriginalEntryPoints(_lib.lib())

    def run(fn):
        new = fn()
        with monkeypatch.context() as m:
            m.setattr(conv_codes, "_lib", Shim())
            old = fn()
        return new, old
    return run


def _same(a, b):
    a = [t for t in (a if isinstance(a, tuple) else (a,)) if torch.is_tensor(t)]
    b = [t for t in (b if isinstance(b, tuple) else (b,)) if torch.is_tensor(t)]
    return len(a) == len(b) and all(torch.equal(x.view(torch.uint8) if x.dtype == torch.float32 else x,
                                                y.view(torch.uint8) if y.dtype == torch.float32 else y)
                                    for x, y in zip(a, b))


def _fill(values, n):
    return np.resize(values, n).astype(np.float32)


def _chunks(values, chunk):
    return [_fill(values[j * chunk:(j + 1) * chunk], chunk) for j in range(-(-values.size // chunk))]


SFS = FAST_SFS + (2.0 ** -31,)


# ---- 1. every fused encoder at the hard values --------------------------------------------------------------------

@pytest.mark.parametrize("enc", ENCS)
def test_bn_act_and_pools_hard_values(enc, hese_vs_original):
    from oracle import fused_emul
    from term_quantization_b200 import conv_codes
    differs = {"bn_act": False, "pool": False, "pool_tiled": False, "pool_rowmax": False}
    for bits in range(1, 12):
        for sf in SFS:
            hv = hard_values(sf, bits)
            x = torch.from_numpy(_fill(hv, -(-hv.size // 8) * 8).reshape(-1, 8)).cuda()
            for terms in terms_for(bits):
                act = ACTS[(bits + terms) % 3]
                quant = (sf, bits, terms, enc)
                out, codes = conv_codes.bn_act_encode(x, None, act, True, quant)
                want = fused_emul._act(x.cpu().numpy(), act)
                check_f32(out, want, ("bn_act", quant, act))
                differs["bn_act"] |= check_codes(codes, want, quant, ("bn_act", quant, act))
            for kind, (C, W, rowmax) in (("pool", (8, 9, False)), ("pool_tiled", (64, 27, False)),
                                         ("pool_rowmax", (64, 14, True))):
                Wo = W if rowmax else (W - 1) // 2 + 1
                Ho = max(5, -(-hv.size // (Wo * C)))                      # every hard value in its own window
                m = np.full((1, 2 * Ho - 1, W, C), -np.inf, np.float32)
                cols = slice(None) if rowmax else slice(0, None, 2)
                m[0, 0::2, cols, :] = _fill(hv, Ho * Wo * C).reshape(Ho, Wo, C)
                pooled = fused_emul.maxpool_f32_nan_dropped(m, *(((3, 1), (2, 1), (1, 0)) if rowmax else (3, 2, 1)))
                bn = (torch.ones(C, device="cuda"), torch.full((C,), -0.0, device="cuda"))
                xt = torch.from_numpy(m).cuda()
                for terms in terms_for(bits):
                    quant = (sf, bits, terms, enc)
                    out, codes = conv_codes.bn_relu_maxpool_encode(xt, bn, relu=True, next_quant=quant, rowmax=rowmax)
                    want = fused_emul._act(pooled, True)
                    check_f32(out, want, (kind, quant))
                    differs[kind] |= check_codes(codes, want, quant, (kind, quant))
    assert all(differs.values()), differs
    x = torch.from_numpy(_fill(hard_values(0.25, 9), 4096).reshape(-1, 64)).cuda()
    xm = x.view(1, 8, 8, 64)
    bn = (torch.ones(64, device="cuda"), torch.zeros(64, device="cuda"))
    for quant in ((0.25, 9, 3, "hese"), (0.25, 11, 1, "hese")):
        assert _same(*hese_vs_original(lambda: conv_codes.bn_act_encode(x, bn, True, True, quant)))
        for rowmax in (False, True):
            assert _same(*hese_vs_original(lambda: conv_codes.bn_relu_maxpool_encode(xm, bn, next_quant=quant, rowmax=rowmax)))


@pytest.mark.parametrize("enc", ENCS)
def test_depthwise_first_conv_stem_hard_values(enc, hese_vs_original):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    differs = {"depthwise": False, "first_conv": False, "stem_pool": False}
    C = 192
    wgt = torch.randint(-100, 101, (9, C), device="cuda", dtype=torch.int32, generator=torch.Generator("cuda").manual_seed(1))
    dw_act = torch.zeros((1, 5, 7, C), dtype=torch.float16, device="cuda")
    img = torch.zeros((1, 5, 9, 3), device="cuda")
    fw = conv_codes.pack_first_conv_weight(torch.randn(64, 3, 3, 3, device="cuda"))
    stem_x = torch.zeros((1, 32, 32, 3), device="cuda")
    stem_w = conv_codes.pack_stem_weight(torch.zeros(64, 3, 7, 7, device="cuda"))
    i = 0
    for bits in range(1, 12):
        for sf in SFS:
            for terms in terms_for(bits):
                quant = (sf, bits, terms, enc)
                act, stride = ACTS[i % 3], 1 + i % 2
                i += 1
                for bv in _chunks(hard_values(sf, bits, sample_ks(bits)), C):
                    b = torch.from_numpy(bv).cuda()
                    out, codes = conv_codes.depthwise3x3_codes(dw_act, wgt, stride, 0.75, bn=(torch.ones(C, device="cuda"), b),
                                                               relu=act, want_f32=True, next_quant=quant,
                                                               act_unsigned=bool(i % 4 < 2))
                    want = fused_emul._act(O.fma_channels(np.zeros(out.shape, np.float32), np.ones(C, np.float32), bv), act)
                    check_f32(out, want, ("depthwise", quant))
                    differs["depthwise"] |= check_codes(codes, want, quant, ("depthwise", quant))
                for bv in _chunks(hard_values(sf, bits, sample_ks(bits)), 64):
                    b = torch.from_numpy(bv).cuda()
                    ones = torch.ones(64, device="cuda")
                    out, codes = conv_codes.first_conv3x3_fused(img, fw, stride, bn=(ones, b), relu=act, want_f32=True,
                                                                next_quant=quant)
                    want = fused_emul._act(O.fma_channels(np.zeros(out.shape, np.float32), np.ones(64, np.float32), bv), act)
                    check_f32(out, want, ("first conv", quant))
                    differs["first_conv"] |= check_codes(codes, want, quant, ("first conv", quant))
                    if bits <= 10:
                        out, codes, _ = conv_codes.stem_conv_pool(stem_x, stem_w, (ones, b), relu=act is True,
                                                                  next_quant=quant)
                        want = fused_emul._act(O.fma_channels(np.zeros(out.shape, np.float32), np.ones(64, np.float32), bv),
                                               act is True)
                        check_f32(out, want, ("stem pool", quant))
                        differs["stem_pool"] |= check_codes(codes, want, quant, ("stem pool", quant))
    assert all(differs.values()), differs
    ones = torch.ones(64, device="cuda")
    b = torch.from_numpy(_fill(hard_values(0.25, 9), 64)).cuda()
    for quant in ((0.25, 9, 3, "hese"), (0.25, 9, 1, "hese")):
        assert _same(*hese_vs_original(lambda: conv_codes.depthwise3x3_codes(
            dw_act, wgt, 2, 0.75, bn=(torch.ones(C, device="cuda"), torch.from_numpy(_fill(hard_values(0.25, 9), C)).cuda()),
            relu=True, want_f32=True, next_quant=quant)))
        assert _same(*hese_vs_original(lambda: conv_codes.first_conv3x3_fused(img, fw, 1, bn=(ones, b), want_f32=True,
                                                                              next_quant=quant)))
        assert _same(*hese_vs_original(lambda: conv_codes.stem_conv_pool(stem_x, stem_w, (ones, b), next_quant=quant)[:2]))


CONV_GEOMS = {
    # N, H, W, C, Cout, k, stride, pad
    "mode3_halo": (2, 56, 56, 64, 64, 3, 1, 1),
    "mode1_resident": (2, 28, 28, 64, 64, 3, 2, 1),
    "mode0_streamed": (2, 56, 56, 64, 128, 1, 2, 0),
    "mode4_halo_streamed": (3, 28, 28, 128, 128, 3, 1, 1),
    "cta_pairs": (41, 28, 28, 128, 128, 3, 1, 1),
    "packed_halo": (151, 7, 7, 128, 256, 3, 1, 1),
}


@pytest.mark.parametrize("engine", ["f16", "i8"])
@pytest.mark.parametrize("geom", list(CONV_GEOMS))
def test_conv_epilogue_hard_values(geom, engine, hese_vs_original):
    from oracle import fused_emul
    from term_quantization_b200 import conv_codes
    N, H, W, C, Cout, k, stride, pad = CONV_GEOMS[geom]
    wgt = torch.randint(-8, 9, (k * k, Cout, C), device="cuda", generator=torch.Generator("cuda").manual_seed(C)).half()
    plan = conv_codes.plan_weight(wgt, 512, engine=engine)
    act = torch.zeros((N, H, W, C), dtype=torch.float16, device="cuda")
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    shape = (N, Ho, Wo, Cout)
    bn = (torch.ones(Cout, device="cuda"), torch.zeros(Cout, device="cuda"))
    differs = False
    i = 0
    for bits in (1, 2, 3, 6, 9, 10):
        sf = FAST_SFS[i % 4]
        hv = hard_values(sf, bits)
        rt = torch.from_numpy(_fill(hv, N * Ho * Wo * Cout).reshape(shape)).cuda()
        for terms in (0, 1, 2, bits):
            relu = ACTS[i % 3]
            i += 1
            for enc in ENCS:
                quant = (sf, bits, terms, enc)
                out, codes = conv_codes.conv2d_codes_fused(act, wgt, (k, k), stride, pad, 1.0, bn=bn, residual=rt,
                                                           relu=relu, next_quant=quant, plan=plan)
                want_v = fused_emul._act(np.float32(0.0) + hv, relu)
                check_f32(out, np.resize(want_v, shape), (geom, engine, quant))
                got = codes.cpu().numpy().astype(np.int32)
                want = np.resize(emul_encode(want_v, quant), shape)
                assert np.array_equal(got, want), (geom, engine, quant, int((got != want).sum()))
                differs |= not np.array_equal(want, np.resize(emul_encode(want_v, quant[:3]), shape))
    assert differs
    for quant in ((0.25, 9, 3, "hese"), (0.0371, 6, 1, "hese")):
        rt = torch.from_numpy(_fill(hard_values(quant[0], quant[1]), N * Ho * Wo * Cout).reshape(shape)).cuda()
        assert _same(*hese_vs_original(lambda: conv_codes.conv2d_codes_fused(
            act, wgt, (k, k), stride, pad, 1.0, bn=bn, residual=rt, relu=True, next_quant=quant, plan=plan)))


@pytest.mark.parametrize("engine", ["f16", "i8"])
def test_conv_plan_cache_tells_encodings_apart(engine):
    """Two calls with the same buffers and shapes that differ only in the output encoding must not share a cached plan
    (the encoding is part of the plan key): codes after codes, each equal to its own encoding's emulation."""
    from term_quantization_b200 import _lib, conv_codes
    N, H, W, C, Cout = 2, 14, 14, 64, 64
    wgt = torch.randint(-8, 9, (9, Cout, C), device="cuda", generator=torch.Generator("cuda").manual_seed(3)).half()
    plan = conv_codes.plan_weight(wgt, 512, engine=engine)
    act = torch.zeros((N, H, W, C), dtype=torch.float16, device="cuda")
    if engine == "i8":
        act, _ = conv_codes.codes_to_planes(act, 1)
    res = torch.from_numpy(_fill(hard_values(0.25, 9), N * H * W * Cout).reshape(N, H, W, Cout)).cuda()
    bn = (torch.ones(Cout, device="cuda"), torch.zeros(Cout, device="cuda"))
    out = torch.empty((N, H, W, Cout), device="cuda")
    codes = torch.empty((N, H, W, Cout), dtype=torch.float16, device="cuda")
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    seen = {}
    for enc in ("hese", "booth", "binary", "hese", "booth"):
        e = _lib.ENCODINGS[enc]
        geom = (N, H, W, C, Cout, 3, 3, 1, 1, 1.0, 1, 0.25, 9, 1)
        if engine == "f16":
            rc = L.tq_conv2d_codes_fused_enc(act.data_ptr(), wgt.data_ptr(), out.data_ptr(), codes.data_ptr(), None,
                                             bn[0].data_ptr(), bn[1].data_ptr(), res.data_ptr(), *geom, e, plan.groups, stream)
        else:
            rc = L.tq_conv2d_planes_i8_enc(act.data_ptr(), plan.planes.data_ptr(), 1, plan.planes_w, out.data_ptr(),
                                           codes.data_ptr(), None, bn[0].data_ptr(), bn[1].data_ptr(), res.data_ptr(),
                                           *geom, e, 127, plan.wgt_max, stream)
        _lib.check(rc)
        from oracle import fused_emul
        want = emul_encode(fused_emul.relu_f32(np.float32(0.0) + res.cpu().numpy()), (0.25, 9, 1, enc))
        got = codes.cpu().numpy().astype(np.int32)
        assert np.array_equal(got, want), (engine, enc, int((got != want).sum()))
        seen[enc] = got
    assert not np.array_equal(seen["hese"], seen["booth"]) and not np.array_equal(seen["hese"], seen["binary"])


# ---- 2. fused executors against the CPU emulation ---------------------------------------------------------------

def _tq(arch, enc, seed=0):
    import torchvision
    from term_quantization_b200 import cnn_models
    from test_graph_pipeline_gpu import _randomise_bn
    torch.manual_seed(seed)
    base = getattr(torchvision.models, arch)(weights=None).cuda().eval()
    _randomise_bn(base, seed)
    return cnn_models.convert_model(base, cnn_models.static_conv_layer_settings(base, 9, 8, 12), 9, 3, encoding=enc)


@pytest.mark.parametrize("enc", ENCS)
def test_fused_resnet18_chain_matches_emulation(enc):
    from oracle import fused_emul
    from term_quantization_b200 import fused, inference
    x = torch.randn(2, 3, 96, 128, device="cuda", generator=torch.Generator("cuda").manual_seed(3)).bfloat16()
    q = _tq("resnet18", enc)
    inference.calibrate(q, [x.float()])
    q = q.to(memory_format=torch.channels_last)
    stems = {}
    for stem, engine in (("tcgen05", "f16"), ("tcgen05", "i8"), ("tcgen05_pool", "auto"), ("cudnn", "auto")):
        f = fused.FusedResNet(q, stem=stem, engine="auto" if engine == "f16" else engine)
        desc = f.chain_description()
        assert all(c is None or len(c["quant"]) == 4 and c["quant"][3] == enc for blk in desc for c in blk)
        if engine == "i8":
            assert {c["engine"] for blk in desc for c in blk if c} == {"i8"}
        cap = {}
        with torch.no_grad():
            logits = f(x, capture=cap)
        emu = fused_emul.run_resnet_chain(desc, cap["stem"].cpu().numpy())
        got = cap["final"].cpu().numpy()
        assert np.array_equal(got.view(np.uint32), emu.view(np.uint32)), (enc, stem, engine, int((got != emu).sum()))
        stems[(stem, engine)] = logits
    assert torch.equal(stems[("tcgen05", "f16")], stems[("tcgen05", "i8")])
    assert torch.equal(stems[("tcgen05", "f16")], stems[("tcgen05_pool", "auto")])
    # the stem's own codes: the one-kernel stem, the row-max pair and a fresh encode of its output agree
    from term_quantization_b200 import conv_codes
    f = fused.FusedResNet(q)
    q0 = f.blocks[0][0].quant
    xc = x.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1)
    out_a, codes_a, _ = conv_codes.stem_conv_pool(xc, f.stem_w, f.stem_bn_pool, relu=True, next_quant=q0)
    y, _ = conv_codes.stem_conv7x7s2(xc, f.stem_w, cout=64, rowmax=True)
    out_b, codes_b = conv_codes.bn_relu_maxpool_encode(y, f.stem_bn_pool, relu=True, next_quant=q0, rowmax=True)
    assert torch.equal(out_a, out_b) and torch.equal(codes_a, codes_b)
    assert np.array_equal(codes_a.cpu().numpy().astype(np.int32), emul_encode(out_a.cpu().numpy(), q0))


@pytest.mark.parametrize("enc", ENCS)
def test_fused_vgg16_and_mobilenet_chains_match_emulation(enc):
    from oracle import fused_emul
    from term_quantization_b200 import fused, inference
    x = torch.randn(2, 3, 64, 96, device="cuda", generator=torch.Generator("cuda").manual_seed(14))
    q = _tq("vgg16_bn", enc, seed=9)
    inference.calibrate(q, [x])
    f = fused.FusedVGG(q.to(memory_format=torch.channels_last))
    cap = {}
    with torch.no_grad():
        f(x, capture=cap)
    stages = f.chain_description()
    q0 = f.stages[f.first_tr][1][0].quant
    assert q0[3] == enc and sum(s[0] == "pool" for s in stages) == 5
    want = fused_emul.run_vgg_chain(stages, cap["stem_codes"].cpu().numpy().astype(np.int32))
    got = cap["final"].cpu().numpy()
    assert got.shape == want.shape and np.array_equal(got, want), (enc, float(np.abs(got - want).max()))

    x = torch.randn(2, 3, 96, 128, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    q = _tq("mobilenet_v2", enc, seed=5)
    inference.calibrate(q, [x])
    f = fused.FusedMobileNet(q)
    cap = {}
    with torch.no_grad():
        f(x, capture=cap)
    emu = fused_emul.run_mobilenet_chain(f.chain_description(), cap["stem_codes"].cpu().numpy())
    final = cap["final"].cpu().numpy()
    assert np.array_equal(final, emu), (enc, int((final != emu).sum()))
    # the first conv's codes, from its own fp32 output
    first = f.blocks[0][0] or f.blocks[0][1]
    from term_quantization_b200 import conv_codes
    out, codes = conv_codes.first_conv3x3_fused(x.permute(0, 2, 3, 1).contiguous(), f._stem_w, 2,
                                                None if f.stem_conv.bias is None else f.stem_conv.bias.detach().float(),
                                                f.stem_bn, relu="relu6", want_f32=True, next_quant=first.quant)
    assert torch.equal(codes, cap["stem_codes"])
    assert np.array_equal(codes.cpu().numpy().astype(np.int32), emul_encode(out.cpu().numpy(), first.quant))


# ---- 3. layer by layer: tensor cores against the float path -----------------------------------------------------

@pytest.mark.parametrize("enc", ENCS)
def test_tensor_core_layers_match_float_path(enc):
    import torch.nn as nn
    from term_quantization_b200 import tr_cuda, tr_layer
    g = torch.Generator("cuda").manual_seed(2)
    torch.manual_seed(0)
    conv = tr_layer.TRConv2dLayer(nn.Conv2d(64, 64, 3, padding=1).cuda(), 9, 3, 9, 8, 12, encoding=enc)
    x = torch.relu(torch.randn(4, 64, 20, 20, device="cuda", generator=g))
    with torch.no_grad():
        conv(x)
        tr_layer.set_tr_tracking(conv, False)
        ref = conv(x)
        conv.use_tensor_cores()
        got = conv(x)
    assert float((got - ref).abs().max()) <= 2e-6 * float(ref.abs().max()) * (64 * 9) ** 0.5
    lin = tr_layer.TRLinearLayer(nn.Linear(784, 512).cuda(), 6, 6, 4, 8, 12, encoding=enc)
    x = torch.randn(256, 784, device="cuda", generator=g)
    with torch.no_grad():
        lin(x)
        tr_layer.set_tr_tracking(lin, False)
        ref = lin.linear(lin.input_quant(x))
        lin.use_tensor_cores()
        got = lin(x)
    assert float((got - ref).abs().max()) <= 2e-6 * float(ref.abs().max()) * 784 ** 0.5
    # 2 data terms: a binding budget, under which binary, Booth and HESE codes differ (with 8 terms on 8-bit data
    # neither binary nor HESE truncates anything and all three give q itself)
    L = tr_layer.TRLSTMLayer(nn.LSTM(650, 650, 1).cuda().eval(), 8, 2, 8, 8, 12, encoding=enc)
    emb = torch.randn(35, 8, 650, device="cuda", generator=g) * 0.1
    hid = tuple(torch.randn(1, 8, 650, device="cuda", generator=g) * 0.1 for _ in range(2))
    with torch.no_grad():
        L(emb, hid)
        tr_layer.set_tr_tracking(L, False)
        L.use_tensor_cores()
        q = L.input_quant
        codes = tr_cuda.tr_codes(emb.view(1, -1, 1, 1), q.sf, 8, 1, 2, dtype=torch.int32, encoding=enc).view(-1, 650)
        hese = tr_cuda.tr_codes(emb.view(1, -1, 1, 1), q.sf, 8, 1, 2, dtype=torch.int32).view(-1, 650)
        wc = torch.round(L.lstm.weight_ih_l0 / np.float32(L.w_sf_ih))
        acc = codes.double() @ wc.double().t()
        scale = np.float32(q.sf) * np.float32(L.w_sf_ih)
        assert torch.equal(L.input_projection(emb).view(-1, 2600), acc.float() * scale)
    assert not torch.equal(codes, hese)


# ---- 4. calibration and the parameter-bit count -------------------------------------------------------------------

@pytest.mark.parametrize("enc", ENCS)
def test_mse_profile_and_term_count(enc):
    from oracle import tq_oracle as O
    from term_quantization_b200 import tr_cuda, tr_layer
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.relu(torch.randn(200000, device="cuda", generator=g)) * 2.5
    hist = torch.histc(x, 8192, -50, 50)
    grid = torch.linspace(-50, 50, 8192)
    sfs = torch.linspace(1e-8, 50, 2048)
    for bits, terms in ((8, 3), (6, 2), (4, 1)):
        sf = tr_layer.mse_profile(hist, -50, 50, bits, terms, encoding=enc)
        idx, errs = emul_mse_profile(hist.cpu().numpy(), grid.numpy(), sfs.numpy(), bits, terms, enc)
        assert sf == sfs.tolist()[idx], (enc, bits, terms)
        xg = grid.cuda()
        lo, hi = max(idx - 8, 0), min(idx + 9, 2048)
        ref = [(hist * (xg - tr_cuda.tr(xg.view(-1, 1, 1, 1), s, bits, 1, terms, encoding=enc).view(-1)) ** 2).sum()
               for s in sfs.tolist()[lo:hi]]
        assert lo + int(torch.argmin(torch.Tensor(ref))) == idx
        np.testing.assert_allclose(torch.Tensor(ref).numpy(), errs[lo:hi], rtol=2e-5)
    w = torch.randn(40, 96, device="cuda", generator=g) * 0.1
    sf = w.abs().max().item() / 128
    wq = tr_cuda.tr(w, sf, 8, 8, 12, encoding=enc)
    want = emul_term_count(wq.cpu().numpy(), sf, enc)
    assert tr_layer.compute_compressed_hese(wq, sf, 12, encoding=enc) == (int(np.ceil(np.log2(12))) + 2) * want
    assert emul_term_count(wq.cpu().numpy(), sf, "hese") == sum(len(tr_layer.hese(v)) for v in (wq / sf).int().view(-1).tolist())
    assert want != emul_term_count(wq.cpu().numpy(), sf, "hese")
    assert O.ENC_HESE == 0


# ---- 5. graph replay ---------------------------------------------------------------------------------------------

def test_booth_resnet_graph_replay_equals_eager():
    from term_quantization_b200 import fused, inference
    from test_graph_pipeline_gpu import _replay_equals_eager
    calib = torch.randn(4, 3, 96, 128, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    q = _tq("resnet18", "booth")
    inference.calibrate(q, [calib])
    f = fused.FusedResNet(q.to(memory_format=torch.channels_last))
    assert "booth" in f.blocks[0][0].quant
    _replay_equals_eager(f, "bf16", 3)
    _replay_equals_eager(inference.U8Frontend(f), "uint8", 3)


# ---- 6. drivers -------------------------------------------------------------------------------------------------

def test_drivers_take_the_encoding(tmp_path):
    from term_quantization_b200 import evaluate_cnn, evaluate_lstm, evaluate_mlp
    res = {}
    for engine in ("float", "auto"):
        res[engine] = evaluate_cnn.main(["-a", "resnet18", "-b", "16", "--images", "32", "--quick", "--engine", engine,
                                         "--encoding", "booth", "--out-file", str(tmp_path / f"{engine}.json")])
        assert len(res[engine]["tr-data3"]["accs"]) == 1
    assert res["float"]["tr-data3"]["tmacs"] == res["auto"]["tr-data3"]["tmacs"]
    res = evaluate_mlp.main(["--wb", "8", "--wt", "12", "--db", "8", "--dt", "4", "--gs", "8", "--samples", "512",
                             "--encoding", "binary"])
    assert len(res["accs"]) == 1 and res["param_bits"][0] > 0
    res = evaluate_lstm.main(["--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--emsize", "64",
                              "--nhid", "64", "--tokens", "1500", "--encoding", "binary"])
    assert len(res["ppls"]) == 1 and np.isfinite(res["ppls"][0])


# ---- 7. refusal ------------------------------------------------------------------------------------------------

def test_bad_encoding_is_refused_before_any_launch():
    from term_quantization_b200 import _lib, conv_codes
    L = _lib.lib()
    dev = "cuda"
    x = torch.zeros((1, 8, 14, 64), device=dev)
    bn = (torch.ones(64, device=dev), torch.zeros(64, device=dev))
    codes = torch.empty((1, 8, 14, 64), dtype=torch.float16, device=dev)
    cact = torch.zeros((1, 8, 8, 64), dtype=torch.float16, device=dev)
    cw = torch.ones((9, 64, 64), dtype=torch.float16, device=dev)
    s = torch.cuda.current_stream().cuda_stream
    n0 = _lib.launch_count()
    for bad in (-1, 3, 99):
        calls = [
            lambda: L.tq_conv2d_codes_fused_enc(cact.data_ptr(), cw.data_ptr(), None, codes.data_ptr(), None, None, None, None,
                                                1, 8, 8, 64, 64, 3, 3, 1, 1, 1.0, 1, 0.5, 8, 3, bad, 1, s),
            lambda: L.tq_bn_act_encode_enc(x.data_ptr(), None, None, None, None, codes.data_ptr(), 112, 64, 1, 0.5, 8, 3, bad, s),
            lambda: L.tq_bn_relu_maxpool_encode_enc(x.data_ptr(), bn[0].data_ptr(), bn[1].data_ptr(), x.data_ptr(),
                                                    None, 1, 8, 14, 64, 1, 0.5, 8, 3, bad, s),
            lambda: L.tq_mse_profile_enc(x.data_ptr(), x.data_ptr(), 64, x.data_ptr(), 4, 8, 3, bad, x.data_ptr(),
                                         x.data_ptr(), s),
            lambda: L.tq_term_count(x.data_ptr(), 0, 64, 0.5, bad, 0, x.data_ptr(), s),
        ]
        for call in calls:
            assert call() == _lib.TQ_ERR_INVALID
            assert "encoding" in L.tq_last_error().decode()
        for quant in ((0.5, 8, 3, "csd"), (0.5, 8, 3, 2)):
            with pytest.raises(ValueError):
                conv_codes.bn_act_encode(x, bn, next_quant=quant)
            with pytest.raises(ValueError):
                conv_codes.conv2d_codes_fused(cact, cw, (3, 3), 1, 1, 1.0, next_quant=quant)
    assert _lib.launch_count() == n0
