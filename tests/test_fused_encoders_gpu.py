"""The term encoder inside every fused epilogue, pinned to the oracle at the values where an encoder goes wrong.

Each fused kernel ends by encoding its value for the next layer's quantiser:  q = min(round_half_up(|x| / sf),
2^bits - 1) -> HESE -> keep the `terms` largest terms, one lookup in a (q, sign) -> code table.  The quantiser, its
checks and the table are shared (csrc/tq_common.cuh); each kernel has its own per-value loop (csrc/tq_gemm.cu: conv
epilogue and one-kernel stem pool; csrc/tq_pool.cu: the pool passes; csrc/tq_dw.cu: depthwise, bn_act_encode, first
conv).  Here the value that reaches the encoder is made equal to a set of
hard values -- every rounding tie (k + 1/2) sf with its neighbours one and two ulps away, the saturation edge, zeros of
both signs, subnormals, infinities and NaN -- and both the fp32 output and the codes must equal the CPU emulation
(oracle/fused_emul.py, oracle/tq_oracle.c) bit for bit, across bit widths, term budgets (binding or not), scale factors
on both sides of the fast-divide range [2^-30, 2^30], and activations.

NaN (DESIGN.md section 3): ReLU and max-pool are fmaxf, which drops a NaN operand; a NaN reaching the encoder encodes
as 0.  The GPU's NaN payload is canonical, so NaNs are compared as NaN, every other value by its bits.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import bits_equal

pytestmark = pytest.mark.gpu

FAST_SFS = (0.25, 0.0371, 2.0 ** -30, 2.0 ** 30)
SLOW_SFS = (2.0 ** -31, 2.0 ** 31, 1e-38, 3e38)        # __fdiv_rn everywhere except the conv, which refuses them
ALL_SFS = FAST_SFS + SLOW_SFS
ACTS = (False, True, "relu6")


def hard_values(sf, bits, ks=None):
    """fp32 values that sit on the edges of the quantiser (sf, bits), both signs: 0, the smallest subnormal, every
    tie fl32((k + 1/2) sf) for k in 0..2^bits (or the given ks) with its +-1 and +-2 ulp neighbours, the saturation
    edge (2^bits - 1/2) sf +- ulps, 2^bits sf, 1e30, FLT_MAX, inf and NaN."""
    sf64 = float(np.float32(sf))
    ks = np.arange(2 ** bits + 1) if ks is None else np.asarray(sorted(set(ks)))
    with np.errstate(over="ignore"):                      # beyond FLT_MAX: inf, which is a hard value too
        ties = ((ks + 0.5) * sf64).astype(np.float32)    # exact in fp64, one rounding to fp32
        edge = (2 ** bits - 0.5) * sf64
        base = np.array([*ties, edge, 2 ** bits * sf64]).astype(np.float32)
    up1 = np.nextafter(base, np.float32(np.inf))
    up2 = np.nextafter(up1, np.float32(np.inf))
    dn1 = np.nextafter(base, np.float32(0))
    dn2 = np.nextafter(dn1, np.float32(0))
    special = np.array([0.0, np.float32(2.0 ** -149), 1e30, np.finfo(np.float32).max, np.inf, np.nan], dtype=np.float32)
    v = np.concatenate([special, base, up1, up2, dn1, dn2]).astype(np.float32)
    v = np.concatenate([v, -v])
    _, first = np.unique(v.view(np.uint32), return_index=True)
    return np.ascontiguousarray(v[np.sort(first)])


def sample_ks(bits):
    """The ties a per-channel injection (Cout <= 64 values per launch) covers: both ends and the middle of the range."""
    top = 2 ** bits
    return [k for k in (0, 1, 2, 3, top // 2 - 1, top // 2, top - 2, top - 1, top) if 0 <= k <= top]


def terms_for(bits):
    return sorted({0, 1, 2, 3, bits, bits + 2})


def _oracle_codes(x, sf, bits, terms):
    from oracle import fused_emul
    return fused_emul.encode(np.asarray(x, dtype=np.float32).reshape(-1), (sf, bits, terms)).reshape(np.shape(x))


def _canon(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return np.where(np.isnan(a), np.float32(np.nan), a)


def _first_diff(got, want):
    bad = np.flatnonzero(_canon(got).view(np.uint32).ravel() != _canon(want).view(np.uint32).ravel())
    i = int(bad[0]) if bad.size else -1
    return f"{bad.size} differ, first at {i}: got {got.ravel()[i]!r} want {want.ravel()[i]!r}" if bad.size else ""


def check_f32(got, want, what):
    got = got.cpu().numpy() if torch.is_tensor(got) else got
    assert bits_equal(_canon(got), _canon(want)), (what, _first_diff(got, want))


def check_codes(got, want_f32, quant, what, want=None):
    """got: the kernel's fp16 codes; want: the oracle's codes of want_f32 (computed here unless given)."""
    want = _oracle_codes(want_f32, *quant) if want is None else want
    got = got.cpu().numpy().astype(np.int32)
    if not np.array_equal(got, want):
        i = int(np.flatnonzero(got.ravel() != want.ravel())[0])
        raise AssertionError(f"{what}: codes differ at {i}: value {np.asarray(want_f32).ravel()[i]!r} "
                             f"got {got.ravel()[i]} want {want.ravel()[i]}")


def _fill(values, n):
    """values cycled to n entries (with at least one full copy when n >= len(values))."""
    return np.resize(values, n).astype(np.float32)


# ---- bn_act_encode: the value is the input ---------------------------------------------------------------------

def _bn_act(x, C, variant, act, quant):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    dev = "cuda"
    xt = torch.from_numpy(x.reshape(-1, C)).to(dev)
    # bias = -0 and bn = (1, -0) leave every value (-0 included) unchanged: the paths run, the values stay hard
    bias = torch.full((C,), -0.0, device=dev) if variant & 1 else None
    bn = (torch.ones(C, device=dev), torch.full((C,), -0.0, device=dev)) if variant & 2 else None
    want = x.reshape(-1, C)
    if bias is not None:
        want = want + np.float32(-0.0)
    if bn is not None:
        want = O.fma_channels(want, np.ones(C, np.float32), np.full(C, -0.0, np.float32))
    want = fused_emul._act(want, act)
    out, codes = conv_codes.bn_act_encode(xt, bn, act, True, quant, bias=bias)
    what = ("bn_act_encode", quant, variant, act)
    check_f32(out, want, what)
    check_codes(codes, want, quant, what)
    none, codes2 = conv_codes.bn_act_encode(xt, bn, act, False, quant, bias=bias)
    assert none is None and torch.equal(codes2, codes), what


@pytest.mark.parametrize("bits", range(1, 12))
def test_bn_act_encode_hard_values(bits):
    i = 0
    for sf in ALL_SFS:
        hv = hard_values(sf, bits)
        x = _fill(hv, -(-hv.size // 8) * 8)
        for terms in terms_for(bits):
            for act in ACTS:
                _bn_act(x, 8, i % 4, act, (sf, bits, terms))
                i += 1


# ---- the pools: a map whose every window holds one hard value (and -inf) ------------------------------------

def _pool_case(values, C, Wo, rowmax):
    """[1, H, W, C] map: hard values on the even rows (and, for the 3x3 window, even columns), which belong to exactly
    one pooling window each; -inf elsewhere."""
    per_row = Wo * C
    Ho = max(4, -(-values.size // per_row))
    H, W = 2 * Ho - 1, (Wo if rowmax else 2 * Wo - 1)
    x = np.full((1, H, W, C), -np.inf, dtype=np.float32)
    v = _fill(values, Ho * per_row).reshape(Ho, Wo, C)
    if rowmax:
        x[0, 0::2, :, :] = v
    else:
        x[0, 0::2, 0::2, :] = v
    return x


POOL_KINDS = {"simple": (20, 7, False), "tiled": (64, 14, False), "rowmax": (64, 14, True)}


@pytest.mark.parametrize("kind", list(POOL_KINDS))
@pytest.mark.parametrize("bits", range(1, 12))
def test_pool_encode_hard_values(bits, kind):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    C, Wo, rowmax = POOL_KINDS[kind]
    a, b = np.ones(C, np.float32), np.full(C, -0.0, np.float32)        # fma(v, 1, -0) == v, -0 included
    bn = (torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda())
    window = ((3, 1), (2, 1), (1, 0)) if rowmax else (3, 2, 1)
    for sf in ALL_SFS:
        x = _pool_case(hard_values(sf, bits), C, Wo, rowmax)
        pooled = fused_emul.maxpool_f32_nan_dropped(O.fma_channels(x, a, b), *window)
        xt = torch.from_numpy(x).cuda()
        for terms in terms_for(bits):
            for relu in (False, True):
                quant = (sf, bits, terms)
                want = fused_emul._act(pooled, relu)
                out, codes = conv_codes.bn_relu_maxpool_encode(xt, bn, relu=relu, next_quant=quant, rowmax=rowmax)
                what = (kind, quant, relu)
                check_f32(out, want, what)
                check_codes(codes, want, quant, what)


# ---- depthwise: zero activations, the BatchNorm shift per channel is the hard value --------------------------------

def _per_channel_chunks(values, chunk):
    n = -(-values.size // chunk)
    return [_fill(values[j * chunk:(j + 1) * chunk], chunk) for j in range(n)]


@pytest.mark.parametrize("bits", range(1, 12))
def test_depthwise_hard_values(bits):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    C = 960
    g = torch.Generator(device="cuda").manual_seed(bits)
    wgt = torch.randint(-100, 101, (9, C), device="cuda", generator=g, dtype=torch.int32)
    act = {s: torch.zeros((1, 5, 7, C), dtype=torch.float16, device="cuda") for s in (1, 2)}
    ones = torch.ones(C, device="cuda")
    i = 0
    for sf in ALL_SFS:
        for terms in terms_for(bits):
            quant = (sf, bits, terms)
            stride, act_fn, unsigned = 1 + i % 2, ACTS[i % 3], bool((i // 2) % 2)
            i += 1
            for bv in _per_channel_chunks(hard_values(sf, bits), C):
                b = torch.from_numpy(bv).cuda()
                out, codes = conv_codes.depthwise3x3_codes(act[stride], wgt, stride, 0.75, bn=(ones, b), relu=act_fn,
                                                           want_f32=True, next_quant=quant, act_unsigned=unsigned)
                t = O.fma_channels(np.zeros(out.shape, np.float32), np.ones(C, np.float32), bv)   # fma(+0, 1, b)
                want = fused_emul._act(t, act_fn)
                what = ("depthwise", quant, stride, act_fn, unsigned)
                check_f32(out, want, what)
                check_codes(codes, want, quant, what)
                none, codes2 = conv_codes.depthwise3x3_codes(act[stride], wgt, stride, 0.75, bn=(ones, b), relu=act_fn,
                                                             next_quant=quant, act_unsigned=unsigned)
                assert none is None and torch.equal(codes2, codes), what


# ---- first conv: zero image, the BatchNorm shift per output channel is the hard value --------------------------------

@pytest.mark.parametrize("bits", range(1, 12))
def test_first_conv_hard_values(bits):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    g = torch.Generator(device="cuda").manual_seed(100 + bits)
    x = torch.zeros((1, 5, 9, 3), device="cuda")
    i = 0
    for cout in (64, 32):
        wp = conv_codes.pack_first_conv_weight(torch.randn(cout, 3, 3, 3, device="cuda", generator=g))
        ones = torch.ones(cout, device="cuda")
        for sf in ALL_SFS:
            for terms in terms_for(bits):
                quant = (sf, bits, terms)
                stride, act_fn = 1 + i % 2, ACTS[i % 3]
                i += 1
                for bv in _per_channel_chunks(hard_values(sf, bits, sample_ks(bits)), cout):
                    b = torch.from_numpy(bv).cuda()
                    out, codes = conv_codes.first_conv3x3_fused(x, wp, stride, bn=(ones, b), relu=act_fn, want_f32=True,
                                                                next_quant=quant)
                    t = O.fma_channels(np.zeros(out.shape, np.float32), np.ones(cout, np.float32), bv)
                    want = fused_emul._act(t, act_fn)
                    what = ("first conv", cout, quant, stride, act_fn)
                    check_f32(out, want, what)
                    check_codes(codes, want, quant, what)
                    none, codes2 = conv_codes.first_conv3x3_fused(x, wp, stride, bn=(ones, b), relu=act_fn, next_quant=quant)
                    assert none is None and torch.equal(codes2, codes), what


# ---- one-kernel stem: zero image and zero weights, so the pooled conv is +0 and the output is fma(0, 1, b) = b ---------

@pytest.mark.parametrize("bits", range(1, 11))
def test_stem_conv_pool_hard_values(bits):
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    x = torch.zeros((1, 32, 32, 3), device="cuda")
    i = 0
    for cout in (64, 32):
        w2 = conv_codes.pack_stem_weight(torch.zeros(cout, 3, 7, 7, device="cuda"))
        ones = torch.ones(cout, device="cuda")
        for sf in ALL_SFS:
            for terms in terms_for(bits):
                for relu in (False, True):
                    quant = (sf, bits, terms)
                    i += 1
                    for bv in _per_channel_chunks(hard_values(sf, bits, sample_ks(bits)), cout):
                        b = torch.from_numpy(bv).cuda()
                        out, codes, _ = conv_codes.stem_conv_pool(x, w2, (ones, b), relu=relu, next_quant=quant)
                        t = O.fma_channels(np.zeros(out.shape, np.float32), np.ones(cout, np.float32), bv)
                        want = fused_emul._act(t, relu)
                        what = ("stem pool", cout, quant, relu)
                        check_f32(out, want, what)
                        check_codes(codes, want, quant, what)


# ---- the conv epilogue on both engines: zero activations, bn = (1, 0), the residual is the hard value ------------------

CONV_GEOMS = {
    # N, H, W, C, Cout, k, stride, pad
    "mode3_halo": (2, 56, 56, 64, 64, 3, 1, 1),
    "mode1_resident": (2, 28, 28, 64, 64, 3, 2, 1),
    "mode0_streamed": (2, 56, 56, 64, 128, 1, 2, 0),
    "mode4_halo_streamed": (3, 28, 28, 128, 128, 3, 1, 1),
    "ragged": (1, 9, 13, 72, 72, 3, 1, 1),
    "cta_pairs": (41, 28, 28, 128, 128, 3, 1, 1),
    "packed_halo": (151, 7, 7, 128, 256, 3, 1, 1),
}
CONV_BITS = (1, 2, 3, 6, 8, 9, 10)


@pytest.mark.parametrize("engine", ["f16", "i8"])
@pytest.mark.parametrize("geom", list(CONV_GEOMS))
def test_conv_epilogue_hard_values(geom, engine):
    from oracle import fused_emul
    from term_quantization_b200 import conv_codes
    N, H, W, C, Cout, k, stride, pad = CONV_GEOMS[geom]
    if engine == "i8" and C % 16:
        pytest.skip("the kind::i8 plane engine needs C % 16 == 0")
    g = torch.Generator(device="cuda").manual_seed(sum(CONV_GEOMS[geom]))
    wgt = torch.randint(-8, 9, (k * k, Cout, C), device="cuda", generator=g).half().contiguous()
    plan = conv_codes.plan_weight(wgt, 512, engine=engine)
    act = torch.zeros((N, H, W, C), dtype=torch.float16, device="cuda")
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    bn = (torch.ones(Cout, device="cuda"), torch.zeros(Cout, device="cuda"))
    i = 0
    for bits in CONV_BITS:
        for terms in sorted({0, 1, 3, bits}):
            sf = FAST_SFS[i % 4]
            relu = ACTS[i % 3]
            i += 1
            quant = (sf, bits, terms)
            hv = hard_values(sf, bits)
            shape = (N, Ho, Wo, Cout)
            rt = torch.from_numpy(_fill(hv, N * Ho * Wo * Cout).reshape(shape)).cuda()
            out, codes = conv_codes.conv2d_codes_fused(act, wgt, (k, k), stride, pad, 1.0, bn=bn, residual=rt, relu=relu,
                                                       next_quant=quant, plan=plan)
            want_v = fused_emul._act(np.float32(0.0) + hv, relu)                  # t = fma(+0, 1, 0) + residual
            want = _fill(want_v, rt.numel()).reshape(shape)                       # (the residual map cycles hv)
            what = (geom, engine, quant, relu)
            check_f32(out, want, what)
            check_codes(codes, want, quant, what, want=np.resize(_oracle_codes(want_v, *quant), shape))
            none, codes2 = conv_codes.conv2d_codes_fused(act, wgt, (k, k), stride, pad, 1.0, bn=bn, residual=rt,
                                                         relu=relu, want_f32=False, next_quant=quant, plan=plan)
            assert none is None and torch.equal(codes2, codes), what


# ---- the row-max pool pass on its own against torch --------------------------------------------------------------

@pytest.mark.parametrize("C", [4, 8, 20, 32, 64, 96, 128, 192])
def test_rowmax_pool_against_torch(C):
    """tq_bn_relu_maxpool_encode_rowmax: max over rows (3,1)/(2,1)/(1,0) of fma(x, a, b), ReLU, encode; against
    torch's max_pool2d of the CPU fma, with NaN / inf sprinkled in (NaN dropped by the max, see the module doc)."""
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    rng = np.random.default_rng(C)
    a = rng.standard_normal(C).astype(np.float32)
    a[::3] = 0.0                                                    # zero slopes beside negative and positive ones
    b = rng.standard_normal(C).astype(np.float32)
    bn = (torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda())
    i = 0
    for rows in (1, 2, 3, 7, 8, 9, 112):
        for cols in (1, 13, 14, 15, 28, 56):
            N, relu = (1, 3)[i % 2], bool((i // 2) % 2)
            i += 1
            x = (rng.standard_normal((N, rows, cols, C)) * 3).astype(np.float32)
            flat = x.reshape(-1)
            pick = rng.choice(flat.size, size=max(1, flat.size // 97), replace=False)
            flat[pick] = rng.choice(np.array([np.nan, np.inf, -np.inf], np.float32), size=pick.size)
            y = O.fma_channels(x, a, b)
            ref = F.max_pool2d(torch.from_numpy(np.where(np.isnan(y), np.float32(-np.inf), y)).permute(0, 3, 1, 2),
                               (3, 1), (2, 1), (1, 0)).permute(0, 2, 3, 1).numpy()
            want = fused_emul._act(ref, relu)
            finite = np.abs(want[np.isfinite(want)])
            quant = (max(float(finite.max(initial=0.0)), 1e-3) / 512, 9, 3)
            out, codes = conv_codes.bn_relu_maxpool_encode(torch.from_numpy(x).cuda(), bn, relu=relu, next_quant=quant,
                                                           rowmax=True)
            what = ("rowmax", N, rows, cols, C, relu)
            assert tuple(out.shape) == want.shape, what
            check_f32(out, want, what)
            check_codes(codes, want, quant, what)


# ---- refusals: Python exceptions, no launch ---------------------------------------------------------------------

def _refused(call, prep_launches=0, raises=(ValueError, NotImplementedError)):
    """call raises before its kernel is launched; prep_launches: kernels the Python wrapper runs before the refusing
    C entry point (the kind::i8 engine splits the activations into planes first)."""
    from term_quantization_b200 import _lib
    n0 = _lib.launch_count()
    with pytest.raises(raises):
        call()
    assert _lib.launch_count() - n0 <= prep_launches


def test_fused_encoders_refuse_bad_quantisers():
    from term_quantization_b200 import conv_codes
    dev = "cuda"
    x = torch.zeros((1, 8, 14, 64), device=dev)
    bn = (torch.ones(64, device=dev), torch.zeros(64, device=dev))
    dw_act = torch.zeros((1, 4, 4, 64), dtype=torch.float16, device=dev)
    dw_w = torch.zeros((9, 64), dtype=torch.int32, device=dev)
    img = torch.zeros((1, 8, 8, 3), device=dev)
    fw = conv_codes.pack_first_conv_weight(torch.zeros(64, 3, 3, 3, device=dev))
    stem_x = torch.zeros((1, 32, 32, 3), device=dev)
    stem_w = conv_codes.pack_stem_weight(torch.zeros(64, 3, 7, 7, device=dev))
    cact = torch.zeros((1, 8, 8, 64), dtype=torch.float16, device=dev)
    cw = torch.ones((9, 64, 64), dtype=torch.float16, device=dev)
    plans = {e: conv_codes.plan_weight(cw, 512, engine=e) for e in ("f16", "i8")}
    kernels = {
        "pool": (11, lambda q: conv_codes.bn_relu_maxpool_encode(x, bn, next_quant=q)),
        "pool_rowmax": (11, lambda q: conv_codes.bn_relu_maxpool_encode(x, bn, next_quant=q, rowmax=True)),
        "depthwise": (11, lambda q: conv_codes.depthwise3x3_codes(dw_act, dw_w, 1, 1.0, next_quant=q)),
        "bn_act_encode": (11, lambda q: conv_codes.bn_act_encode(x, bn, next_quant=q)),
        "first_conv": (11, lambda q: conv_codes.first_conv3x3_fused(img, fw, 1, bn=bn, next_quant=q)),
        "stem_pool": (10, lambda q: conv_codes.stem_conv_pool(stem_x, stem_w, bn, next_quant=q)),
    }
    for e, plan in plans.items():
        kernels["conv_" + e] = (10, lambda q, plan=plan: conv_codes.conv2d_codes_fused(cact, cw, (3, 3), 1, 1, 1.0, relu=True,
                                                                                       next_quant=q, plan=plan))
    for name, (max_bits, call) in kernels.items():
        call((0.5, max_bits, 3))                                     # the largest bit width runs
        torch.cuda.synchronize()
        prep = 1 if name == "conv_i8" else 0
        for bits in (0, max_bits + 1, 12):
            _refused(lambda: call((0.5, bits, 3)), prep)
        _refused(lambda: call((0.5, 8, -1)), prep, ValueError)       # a bad argument (TQ_ERR_INVALID) everywhere
        for sf in (0.0, -1.0, float("inf"), float("nan")):
            _refused(lambda: call((sf, 8, 3)), prep)
        if name.startswith("conv_"):
            lo = float(np.nextafter(np.float32(2.0 ** -30), np.float32(0)))
            hi = float(np.nextafter(np.float32(2.0 ** 30), np.float32(np.inf)))
            for sf in (lo, hi) + SLOW_SFS:
                _refused(lambda: call((sf, 8, 3)), prep)
            call((2.0 ** -30, 8, 3))
            call((2.0 ** 30, 8, 3))
