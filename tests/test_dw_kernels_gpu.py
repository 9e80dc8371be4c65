"""The kernels of csrc/tq_dw.cu at every template instance the host can pick, on real data, against plain CPU references.

Depthwise 3x3 on codes (`depthwise3x3_codes_kernel<STRIDE, CB, UNSIGNED, FAST>`, 16 instances).  The host picks
CB = 64 channels per tile when C % 64 == 0 and 32 otherwise, UNSIGNED = act_unsigned, FAST = the consumer's sf lies in
[2^-30, 2^30] (or no codes are written), and the tile from the output size; `dw_plan` below restates that rule.  The
cases cross every instance with every tile class: 8- and 16-pixel-wide tiles, 4-, 8- and 16-row tiles, widths that
leave a partial 4-pixel group, ragged channel blocks (C = 40, 72, 136), 32-channel boxes wider than an 8/16/24-channel
tensor, 1x1 and 2x3 maps, and maps with three or more tiles per persistent CTA, so both stages of the double buffer turn
over.  The codes are signed in [-2^11, 2^11] or, for UNSIGNED, in [0, 1023] (the documented limit), half of them zero;
the weights lie in [-2^15, 2^15], some cases at the extremes so that |acc| passes 2^24.  The fp32 output must equal the
exact integer accumulator (fp64 grouped conv of integers, oracle/fused_emul.depthwise_exact) followed by the fp32
epilogue of fused_emul.fused_depthwise bit for bit, and the codes must equal oracle.tr of that value in the consumer's
encoding.

First conv (`first_conv3x3_kernel<COUT, STRIDE, FAST>`, 8 instances): output widths at and around the tile width
TW = 8 * 32 / (COUT / 8), 1-pixel-wide and 1-pixel-high images, five images per launch so that tiles cross images.  The
image sits inside a buffer whose head and tail are NaN, so a read before its first or past its last pixel poisons an
output.  fp32 against an fp64 conv (the 2e-6 of test_layers_gpu), codes exactly against oracle.tr of the kernel's own
fp32 output.

bn_act_encode on channel counts that are multiples of 4 but not of 8, and the fp16 max-pool on codes over every window,
stride and padding it accepts, both exactly.

Which instance every case reaches is asserted from the restated host rule, and the rule itself is checked against the
kernel names a profiler sees launched.
"""
import collections
import itertools
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import bits_equal
from test_encodings_host import emul_encode

pytestmark = pytest.mark.gpu

B200_SMS = 148
ENCS = ("hese", "binary", "booth")
ACTS = (False, True, "relu6")
EPILOGUES = ("plain", "bias", "bn", "bias+bn")
BITS = (9, 4, 11, 6, 8, 1, 10, 3, 7, 5, 2)
FAST_LO, FAST_HI = 2.0 ** -30, 2.0 ** 30
SLOW_SFS = (2.0 ** -31, 2.0 ** -36, 2.0 ** 31, 2.0 ** 36)


def _cdiv(a, b):
    return -(-a // b)


def _terms(i, bits):
    return (bits + 2, 3, 1, bits, 0, 2)[i % 6]


def _fast(quant):
    """FAST of the kernel the host picks: the hoisted-reciprocal divide is exact for 2^-30 <= sf <= 2^30; without codes
    the quantiser is the neutral sf = 1."""
    return quant is None or FAST_LO <= float(np.float32(quant[0])) <= FAST_HI


def _sf_and_magnitude(i, fast, bits):
    """(sf, M): the consumer's scale factor and the magnitude the case's values are scaled to, so that the codes use the
    whole range of the quantiser on both sides of the fast-divide range (and saturate in part)."""
    if fast:
        M = 8.0                                                  # ReLU6 clamps part of the values
        return float(np.float32(M / 2 ** bits * (0.37, 1.0, 2.9)[i % 3])), M
    sf = SLOW_SFS[i % len(SLOW_SFS)]
    return sf, sf * 2 ** bits * 0.7


def _check_f32(got, want, what):
    got = got.cpu().numpy()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not bits_equal(got, want):
        bad = np.flatnonzero(got.view(np.uint32).ravel() != want.view(np.uint32).ravel())
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size} of {got.size} fp32 outputs differ, first at "
                             f"{tuple(int(v) for v in np.unravel_index(i, got.shape))}: "
                             f"got {got.ravel()[i]!r} want {want.ravel()[i]!r}")


def _check_codes(got, want, what):
    got = got.cpu().numpy().astype(np.int32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got.ravel() != want.ravel())
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size} of {got.size} codes differ, first at "
                             f"{tuple(int(v) for v in np.unravel_index(i, got.shape))}: "
                             f"got {got.ravel()[i]} want {want.ravel()[i]}")


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---- depthwise: the host rule, restated -------------------------------------------------------------------------

DwCase = collections.namedtuple("DwCase", "N H W C stride unsigned epi act fast enc bits terms extreme seed")


def dw_plan(case, sms=B200_SMS):
    """What tq_depthwise3x3_codes_enc launches for this case: the kernel instance (STRIDE, CB, UNSIGNED, FAST), the
    tile (rows, columns), the tile count and the number of persistent CTAs."""
    s = case.stride
    Ho, Wo = (case.H - 1) // s + 1, (case.W - 1) // s + 1
    cb = 64 if case.C % 64 == 0 else 32
    tw = 16 if Wo > 8 else 8
    th = 8 if Ho > 4 else 4
    if s == 2 and tw == 16:
        th = 4
    if cb == 32 and s == 1 and th == 8 and Ho > 8:
        th = 16
    tiles = case.N * _cdiv(Ho, th) * _cdiv(Wo, tw) * _cdiv(case.C, cb)
    stage = ((th * s + 2) * (tw * s + 2) * cb * 2 + 127) & ~127
    table = ((2 << case.bits) * 2 + 15) & ~15
    smem = 128 + 2 * stage + 9 * case.C * 4 + table + 64
    per_sm = min(2, max(1, (227 * 1024) // (smem + 1024)))
    return {"instance": (s, cb, case.unsigned, case.fast), "tile": (th, tw), "tiles": tiles, "per_sm": per_sm,
            "ctas": min(tiles, sms * per_sm)}


# (rows, columns) of the tiles the host rule can pick, per (stride, CB)
DW_TILES = {(1, 64): {(4, 8), (4, 16), (8, 8), (8, 16)},
            (1, 32): {(4, 8), (4, 16), (8, 8), (8, 16), (16, 8), (16, 16)},
            (2, 64): {(4, 8), (8, 8), (4, 16)},
            (2, 32): {(4, 8), (8, 8), (4, 16)}}
# four or more channel counts of each CB (64: C % 64 == 0); among the 32-channel ones ragged last blocks (40, 72, 136)
# and tensors narrower than the 32-channel box (8, 16, 24)
DW_CHANNELS = (8, 16, 24, 32, 40, 64, 72, 96, 128, 136, 192, 960)
# (Ho, Wo): every tile of DW_TILES, full and partial tiles, a partial 4-pixel group
DW_OUT = ((1, 1), (2, 3), (4, 8), (4, 9), (5, 16), (6, 5), (8, 17), (9, 8), (16, 16), (17, 33))
DW_FLAGS = ((False, True), (True, True), (False, False), (True, False))          # (unsigned, fast)


def _dw_case(i, N, Ho, Wo, C, stride, unsigned, fast, extreme=False, par=0):
    """stride 2 takes both input parities that give the same output size (2Ho - 1 and 2Ho rows)."""
    H = (Ho - 1) * stride + 1 + (stride == 2 and par % 2)
    W = (Wo - 1) * stride + 1 + (stride == 2 and (par // 2) % 2)
    bits = BITS[i % len(BITS)]
    return DwCase(N, H, W, C, stride, unsigned, EPILOGUES[i % 4], ACTS[(i // 4) % 3], fast, ENCS[(i // 12) % 3], bits,
                  _terms(i, bits), extreme, 1000 + i)


def _dw_cases():
    cases = []
    for stride in (1, 2):
        seen = collections.Counter()
        for C in DW_CHANNELS:
            cb = 64 if C % 64 == 0 else 32
            ci = seen[cb]                     # the four (unsigned, fast) turn with the channel count: every output
            seen[cb] += 1                     # size meets every instance
            for j, (Ho, Wo) in enumerate(DW_OUT):
                i = len(cases)
                unsigned, fast = DW_FLAGS[(ci + j) % 4]
                N = 3 if i % 2 and C < 960 else 1
                cases.append(_dw_case(i, N, Ho, Wo, C, stride, unsigned, fast, extreme=(i % 7 == 3), par=j))
    # every CTA of the persistent grid runs at least three tiles: both stages of the double buffer are refilled
    for C, stride, Ho, Wo, unsigned in ((8, 1, 16, 16, False), (64, 1, 4, 8, False), (24, 2, 4, 8, True),
                                        (64, 2, 4, 8, False)):
        one = _dw_case(len(cases), 1, Ho, Wo, C, stride, unsigned, True)
        plan = dw_plan(one)
        cases.append(one._replace(N=_cdiv(3 * B200_SMS * plan["per_sm"], plan["tiles"])))
    # a seeded random tail
    rng = np.random.default_rng(20261022)
    for _ in range(40):
        i = len(cases)
        cases.append(_dw_case(i, int(rng.integers(1, 4)), int(rng.integers(1, 21)), int(rng.integers(1, 41)),
                              int(rng.choice(DW_CHANNELS)), int(rng.integers(1, 3)), bool(rng.integers(0, 2)),
                              bool(rng.integers(0, 2)), extreme=bool(rng.integers(0, 5) == 0), par=int(rng.integers(0, 4))))
    return cases


DW_CASES = _dw_cases()
DW_MANY_TILES = DW_CASES[2 * len(DW_CHANNELS) * len(DW_OUT):][:4]


def _dw_id(c):
    return (f"s{c.stride}-C{c.C}-N{c.N}-{c.H}x{c.W}-{'u' if c.unsigned else 's'}-{c.epi}-{c.act or 'noact'}-"
            f"{'fast' if c.fast else 'slow'}-{c.enc}-b{c.bits}t{c.terms}{'-ext' if c.extreme else ''}")


def _dw_codes(rng, shape, unsigned, extreme):
    """fp16-exact integer codes, half of them zero, with the ends of the range planted."""
    if unsigned:
        hi, ends = 1023, (0, 1, 512, 1022, 1023)
        a = rng.choice(np.array([1022, 1023]), shape) if extreme else rng.integers(0, hi + 1, shape)
    else:
        hi, ends = 2048, (-2048, -2047, -1, 1, 2047, 2048)
        a = rng.choice(np.array([-2048, -2047, 2047, 2048]), shape) if extreme else rng.integers(-hi, hi + 1, shape)
    a = np.where(rng.random(shape) < 0.5, 0, a).reshape(-1)
    pick = rng.choice(a.size, size=min(a.size, 4 * len(ends)), replace=False)
    a[pick] = np.resize(np.array(ends), pick.size)
    return a.reshape(shape).astype(np.int32)


def _dw_setup(case):
    """Device operands of the case and its CPU reference (fp32 output, codes)."""
    from oracle import fused_emul
    rng = np.random.default_rng(case.seed)
    codes = _dw_codes(rng, (case.N, case.H, case.W, case.C), case.unsigned, case.extreme)
    if case.extreme:
        w = rng.choice(np.array([-32768, -32767, 32767, 32768]), (9, case.C))
    else:
        w = rng.integers(-32768, 32769, (9, case.C))
    w = w.astype(np.int32)
    sf, M = _sf_and_magnitude(case.seed, case.fast, case.bits)
    acc = fused_emul.depthwise_exact(codes, w, case.stride)
    scale = float(np.float32(M / max(float(np.abs(acc).max()), 1.0)))
    bias = (rng.standard_normal(case.C) * M / 4).astype(np.float32) if "bias" in case.epi else None
    bn = None
    if "bn" in case.epi:
        bn = ((rng.uniform(0.5, 1.5, case.C) * rng.choice([-1.0, 1.0], case.C)).astype(np.float32),
              (rng.standard_normal(case.C) * M / 4).astype(np.float32))
    quant = (sf, case.bits, case.terms, case.enc)
    dw = {"w": w, "stride": case.stride, "scale": scale, "bias": bias, "bn": bn}
    t_ref, _ = fused_emul.fused_depthwise(codes, dw, relu=case.act)
    dev = {"act": torch.from_numpy(codes.astype(np.float16)).cuda(), "wgt": torch.from_numpy(w).cuda(),
           "stride": case.stride, "scale": scale, "relu": case.act, "act_unsigned": case.unsigned,
           "bias": None if bias is None else torch.from_numpy(bias).cuda(),
           "bn": None if bn is None else tuple(torch.from_numpy(v).cuda() for v in bn)}
    return dev, quant, t_ref, emul_encode(t_ref, quant)


def _dw_run(dev, **kw):
    from term_quantization_b200 import conv_codes
    return conv_codes.depthwise3x3_codes(dev["act"], dev["wgt"], dev["stride"], dev["scale"], bias=dev["bias"],
                                         bn=dev["bn"], relu=dev["relu"], act_unsigned=dev["act_unsigned"], **kw)


@pytest.mark.parametrize("case", DW_CASES, ids=[f"d{i:03d}-{_dw_id(c)}" for i, c in enumerate(DW_CASES)])
def test_depthwise_against_exact_reference(case):
    dev, quant, t_ref, c_ref = _dw_setup(case)
    plan = dw_plan(case, _sms())
    what = (_dw_id(case), "instance", plan["instance"], "tile", plan["tile"])
    assert _fast(quant) == case.fast, what
    out, codes = _dw_run(dev, want_f32=True, next_quant=quant)
    _check_f32(out, t_ref, what)
    _check_codes(codes, c_ref, what)
    none, codes2 = _dw_run(dev, next_quant=quant)                               # codes only
    assert none is None
    _check_codes(codes2, c_ref, what + ("codes only",))
    out3, none = _dw_run(dev, want_f32=True)                                    # fp32 only (FAST: the neutral quantiser)
    assert none is None
    _check_f32(out3, t_ref, what + ("fp32 only",))


def test_depthwise_many_tile_cases_loop_every_cta():
    """The cases sized for the persistent grid give every CTA at least three tiles on this device."""
    for case in DW_MANY_TILES:
        plan = dw_plan(case, _sms())
        assert plan["tiles"] >= 3 * plan["ctas"], (_dw_id(case), plan)


# ---- first conv ------------------------------------------------------------------------------------------------

FcCase = collections.namedtuple("FcCase", "N H W cout stride fast bias bn act enc bits terms seed")


def fc_tile_width(cout):
    return 8 * 32 // (cout // 8)


def fc_instance(case):
    return (case.cout, case.stride, case.fast)


def _fc_cases():
    cases = []
    for cout, stride, fast in itertools.product((32, 64), (1, 2), (True, False)):
        TW = fc_tile_width(cout)
        outs = [((7, 8, 9)[(j + len(cases)) % 3], wo) for j, wo in enumerate((TW - 1, TW, TW + 1, 2 * TW + 1))]
        shapes = []
        for j, (Ho, Wo) in enumerate(outs):                     # both input parities that give the output (stride 2)
            shapes.append(((Ho - 1) * stride + 1 + (stride == 2 and j % 2),
                           (Wo - 1) * stride + 1 + (stride == 2 and (j // 2) % 2)))
        shapes += [(1, (TW + 1) * stride), (9, 1), (1, 1)]       # 1-pixel-high and 1-pixel-wide images
        for H, W in shapes:
            i = len(cases)
            bits = BITS[i % len(BITS)]
            cases.append(FcCase(5, H, W, cout, stride, fast, bool(i % 2), bool((i // 2) % 2), ACTS[i % 3], ENCS[i % 3],
                                bits, _terms(i, bits), 2000 + i))
    return cases


FC_CASES = _fc_cases()


def _fc_id(c):
    return (f"co{c.cout}-s{c.stride}-{c.H}x{c.W}-{'fast' if c.fast else 'slow'}-{'bias' if c.bias else 'nobias'}-"
            f"{'bn' if c.bn else 'nobn'}-{c.act or 'noact'}-{c.enc}-b{c.bits}t{c.terms}")


def _fc_setup(case):
    """Device operands (the image inside a NaN-bordered buffer), the fp64 reference and the quantiser."""
    from term_quantization_b200 import conv_codes
    rng = np.random.default_rng(case.seed)
    mag = 1.0 if case.fast else (2.0 ** -40, 2.0 ** 40)[case.seed % 2]
    x = (rng.standard_normal((case.N, case.H, case.W, 3)) * mag).astype(np.float32)
    w = (rng.standard_normal((case.cout, 3, 3, 3)) * 0.2).astype(np.float32)
    bias = (rng.standard_normal(case.cout) * mag * 0.5).astype(np.float32) if case.bias else None
    a = (rng.uniform(0.5, 1.5, case.cout) * rng.choice([-1.0, 1.0], case.cout)).astype(np.float32)
    b = (rng.standard_normal(case.cout) * mag).astype(np.float32)
    ref = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2).double(), torch.from_numpy(w).double(),
                   None if bias is None else torch.from_numpy(bias).double(), case.stride, 1).permute(0, 2, 3, 1)
    if case.bn:
        ref = ref * torch.from_numpy(a).double() + torch.from_numpy(b).double()
    if case.act:
        ref = ref.clamp(min=0)
    if case.act == "relu6":
        ref = ref.clamp(max=6)
    if case.fast:
        sf = float(np.float32(max(float(ref.abs().max()), 1e-3) / 2 ** case.bits * (0.37, 1.0, 2.9)[case.seed % 3]))
    else:
        sf = (2.0 ** -36, 2.0 ** 36)[case.seed % 2] / 2 ** case.bits
        sf = max(sf, 2.0 ** 31) if mag > 1 else min(sf, 2.0 ** -31)
    # dead borders: a read before the first or past the last pixel of the image reads NaN
    n = x.size
    border = 6 * (case.W + 2) + 65
    buf = torch.full((border + n + border,), float("nan"), device="cuda")
    buf[border:border + n] = torch.from_numpy(x.reshape(-1)).cuda()
    dev = {"x": buf[border:border + n].view(x.shape), "w": conv_codes.pack_first_conv_weight(torch.from_numpy(w).cuda()),
           "stride": case.stride, "relu": case.act,
           "bias": None if bias is None else torch.from_numpy(bias).cuda(),
           "bn": (torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) if case.bn else None}
    return dev, (sf, case.bits, case.terms, case.enc), ref


def _fc_run(dev, **kw):
    from term_quantization_b200 import conv_codes
    return conv_codes.first_conv3x3_fused(dev["x"], dev["w"], dev["stride"], dev["bias"], dev["bn"], relu=dev["relu"],
                                          **kw)


@pytest.mark.parametrize("case", FC_CASES, ids=[f"f{i:02d}-{_fc_id(c)}" for i, c in enumerate(FC_CASES)])
def test_first_conv_against_fp64_and_oracle_codes(case):
    dev, quant, ref = _fc_setup(case)
    what = (_fc_id(case), "instance", fc_instance(case))
    assert _fast(quant) == case.fast, what
    out, codes = _fc_run(dev, want_f32=True, next_quant=quant)
    assert tuple(out.shape) == tuple(ref.shape), what
    assert bool(torch.isfinite(out).all()), what + ("non-finite output: a read outside the image",)
    err = float((out.double().cpu() - ref).abs().max()) / max(float(ref.abs().max()), float(np.finfo(np.float32).tiny))
    assert err < 2e-6, what + (err,)
    got = out.cpu().numpy()
    c_ref = emul_encode(got, quant)
    _check_codes(codes, c_ref, what)
    none, codes2 = _fc_run(dev, next_quant=quant)                               # codes only
    assert none is None
    _check_codes(codes2, c_ref, what + ("codes only",))
    out3, none = _fc_run(dev, want_f32=True)                                    # fp32 only
    assert none is None
    _check_f32(out3, got, what + ("fp32 only",))


# ---- bn_act_encode: C a multiple of 4, not of 8 --------------------------------------------------------------------

@pytest.mark.parametrize("C", [4, 12, 20, 36])
def test_bn_act_encode_quarter_channel_blocks(C):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    rng = np.random.default_rng(C)
    i = 0
    for epi in EPILOGUES:
        for act in ACTS:
            N, H, W = ((1, 1, 1), (1, 3, 7), (3, 5, 3), (5, 7, 9))[i % 4]           # odd pixel counts
            fast = i % 3 != 2
            bits = BITS[i % len(BITS)]
            sf, M = _sf_and_magnitude(i, fast, bits)
            quant = (sf, bits, _terms(i, bits), ENCS[i % 3])
            i += 1
            x = (rng.standard_normal((N, H, W, C)) * M / 2).astype(np.float32)
            bias = (rng.standard_normal(C) * M / 4).astype(np.float32) if "bias" in epi else None
            a = (rng.uniform(0.5, 1.5, C) * rng.choice([-1.0, 1.0], C)).astype(np.float32)
            b = (rng.standard_normal(C) * M / 4).astype(np.float32)
            t = x if bias is None else x + bias
            if "bn" in epi:
                t = O.fma_channels(t, a, b)
            want = np.ascontiguousarray(fused_emul._act(t, act), dtype=np.float32)
            bn = (torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) if "bn" in epi else None
            bias_t = None if bias is None else torch.from_numpy(bias).cuda()
            xt = torch.from_numpy(x).cuda()
            what = ("bn_act_encode", (N, H, W, C), epi, act, quant)
            assert _fast(quant) == fast
            out, codes = conv_codes.bn_act_encode(xt, bn, act, True, quant, bias=bias_t)
            _check_f32(out, want, what)
            c_ref = emul_encode(want, quant)
            _check_codes(codes, c_ref, what)
            none, codes2 = conv_codes.bn_act_encode(xt, bn, act, False, quant, bias=bias_t)
            assert none is None
            _check_codes(codes2, c_ref, what + ("codes only",))
            out3, none = conv_codes.bn_act_encode(xt, bn, act, True, None, bias=bias_t)
            assert none is None
            _check_f32(out3, want, what + ("fp32 only",))


# ---- the max-pool on fp16 codes --------------------------------------------------------------------------------

@pytest.mark.parametrize("k", range(1, 8))
def test_maxpool_codes_every_window(k):
    """Every stride 1..3 and padding 0..k/2 of the window k x k, on the smallest map that still gives one output (the
    window reaches into the padding on every side; all codes negative, so a zero standing in for the padding shows) and
    on a larger map with a ragged right and bottom edge; codes up to +-2^11."""
    from term_quantization_b200 import conv_codes
    rng = np.random.default_rng(k)
    for stride in (1, 2, 3):
        for pad in range(k // 2 + 1):
            for C in (8, 24, 136):
                small = max(1, k - 2 * pad)
                for N, H, W, negative in ((1, small, small, True), (2, small + stride + 1, small + 2 * stride, False)):
                    shape = (N, H, W, C)
                    if negative:
                        x = -rng.integers(1, 2049, shape)
                    else:
                        x = rng.integers(-2048, 2049, shape)
                        flat = x.reshape(-1)
                        pick = rng.choice(flat.size, size=min(flat.size, 8), replace=False)
                        flat[pick] = np.resize(np.array([-2048, 2048]), pick.size)
                    x = x.astype(np.float32)
                    want = F.max_pool2d(torch.from_numpy(x).permute(0, 3, 1, 2), k, stride, pad).permute(0, 2, 3, 1)
                    got = conv_codes.maxpool_codes(torch.from_numpy(x).half().cuda(), k, stride, pad)
                    what = ("maxpool", shape, k, stride, pad)
                    assert tuple(got.shape) == tuple(want.shape), what
                    assert torch.equal(got.float().cpu(), want), what + (
                        int((got.float().cpu() != want).sum()), "differ")


# ---- which instances the cases reach ---------------------------------------------------------------------------

DW_INSTANCES = set(itertools.product((1, 2), (64, 32), (False, True), (False, True)))
FC_INSTANCES = set(itertools.product((32, 64), (1, 2), (False, True)))


def test_every_kernel_instance_is_checked():
    """By the restated host rule, the checked cases reach all 16 depthwise and all 8 first-conv instances, and each
    depthwise instance meets every tile shape its stride and channel block allow."""
    dw = collections.Counter(dw_plan(c)["instance"] for c in DW_CASES)
    fc = collections.Counter(fc_instance(c) for c in FC_CASES)
    print(f"depthwise instances checked: {len(set(dw) & DW_INSTANCES)}/16", dict(sorted(dw.items())))
    print(f"first-conv instances checked: {len(set(fc) & FC_INSTANCES)}/8", dict(sorted(fc.items())))
    assert set(dw) == DW_INSTANCES
    assert set(fc) == FC_INSTANCES
    tiles = collections.defaultdict(set)
    for c in DW_CASES:
        p = dw_plan(c)
        tiles[p["instance"]].add(p["tile"])
    for inst in DW_INSTANCES:
        assert tiles[inst] == DW_TILES[inst[:2]], (inst, sorted(tiles[inst]))
    # ragged channel blocks and boxes wider than the tensor, signed and unsigned, both strides
    for s, u in itertools.product((1, 2), (False, True)):
        assert {c.C for c in DW_CASES if c.stride == s and c.unsigned == u} >= {8, 16, 24, 40, 72, 136}, (s, u)


_DW_NAME = re.compile(r"depthwise3x3_codes_kernel\s*<\s*(\d+)\s*,\s*(\d+)\s*,\s*(true|false)\s*,\s*(true|false)\s*>")
_DW_MANGLED = re.compile(r"depthwise3x3_codes_kernelILi(\d+)ELi(\d+)ELb([01])ELb([01])E")
_FC_NAME = re.compile(r"first_conv3x3_kernel\s*<\s*(\d+)\s*,\s*(\d+)\s*,\s*(true|false)\s*>")
_FC_MANGLED = re.compile(r"first_conv3x3_kernelILi(\d+)ELi(\d+)ELb([01])E")


def _flag(s):
    return s in ("true", "1")


def _launched(prof):
    """(depthwise instances, first-conv instances) launched inside the profiler, with multiplicity."""
    dw, fc = collections.Counter(), collections.Counter()
    for ev in prof.key_averages():
        m = _DW_NAME.search(ev.key) or _DW_MANGLED.search(ev.key)
        if m:
            dw[(int(m[1]), int(m[2]), _flag(m[3]), _flag(m[4]))] += ev.count
        m = _FC_NAME.search(ev.key) or _FC_MANGLED.search(ev.key)
        if m:
            fc[(int(m[1]), int(m[2]), _flag(m[3]))] += ev.count
    return dw, fc


def test_restated_host_rule_matches_the_launched_kernels():
    """One representative case of every instance runs under torch.profiler: the kernel names launched must be exactly
    the instances dw_plan / fc_instance predict, once each."""
    from torch.profiler import ProfilerActivity, profile
    dw_reps = {}
    for c in DW_CASES:
        dw_reps.setdefault(dw_plan(c)["instance"], c)
    fc_reps = {}
    for c in FC_CASES:
        fc_reps.setdefault(fc_instance(c), c)
    dw_ops = [(inst, _dw_setup(c)) for inst, c in sorted(dw_reps.items())]
    fc_ops = [(inst, _fc_setup(c)) for inst, c in sorted(fc_reps.items())]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, (dev, quant, _, _) in dw_ops:
            _dw_run(dev, want_f32=True, next_quant=quant)
        for _, (dev, quant, _) in fc_ops:
            _fc_run(dev, want_f32=True, next_quant=quant)
        torch.cuda.synchronize()
    dw, fc = _launched(prof)
    print("depthwise launched:", dict(sorted(dw.items())))
    print("first conv launched:", dict(sorted(fc.items())))
    assert dw == collections.Counter(inst for inst, _ in dw_ops)
    assert fc == collections.Counter(inst for inst, _ in fc_ops)
    assert set(dw) == DW_INSTANCES and set(fc) == FC_INSTANCES
