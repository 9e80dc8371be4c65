"""CPU tests that pin oracle/ (our restatement) to the reference: golden vectors generated
from the reference kernel body, the live reference shim when present, and bit_utils.py."""
import numpy as np
import pytest

from conftest import bits_equal, golden_cases
from oracle import tq_oracle as O


def test_golden_vectors_match_restatement():
    cases = golden_cases()
    assert len(cases) >= 40
    for x, sf, bits, g, alpha, y in cases:
        assert bits_equal(O.tr(x, sf, bits, g, alpha), y), (x.shape, bits, g, alpha)


def test_survey_hand_table():
    # SURVEY section 4: figures/term-reveal.png example under HESE
    out = O.tr(np.array([[3.2, 0.15, 0.7]], dtype=np.float32), 0.05, 8, 3, 4)
    assert np.array_equal(out, np.array([[64, 4, 14]], dtype=np.float32) * np.float32(0.05))
    v = np.array([[127, -127, 3, -6, 11, 0, 27, 255]], dtype=np.float32)
    assert O.tr(v, 1.0, 8, 8, 12).tolist() == [[127, -128, 4, -6, 12, 0, 28, 256]]
    assert O.tr(v, 1.0, 8, 8, 16).tolist() == [[127, -127, 3, -6, 11, 0, 27, 256]]
    # round-half-up with the 0.5 added in double (kernels/tr_cuda_kernel.cu:22)
    assert O.quantize(0.49999997, 1.0, 8) == 0
    assert O.quantize(0.5, 1.0, 8) == 1
    assert O.quantize(2.5, 1.0, 8) == 3
    assert O.quantize(1e9, 1.0, 8) == 255
    assert O.quantize(float("inf"), 1.0, 8) == 255
    assert O.quantize(float("nan"), 1.0, 8) == 0


def test_terms_identities_exhaustive():
    for enc in (O.ENC_HESE, O.ENC_BINARY, O.ENC_BOOTH):
        for q in range(1 << 12):
            p, n = O.terms(q, enc)
            assert p & n == 0 and p - n == q
    # HESE never uses more terms than binary or Booth
    for q in range(1 << 12):
        h = sum(bin(m).count("1") for m in O.terms(q, O.ENC_HESE))
        assert h <= bin(q).count("1")
        assert h <= sum(bin(m).count("1") for m in O.terms(q, O.ENC_BOOTH))


def _py_hese(number):
    """Window scan of bit_utils.py:10-44 restated on integers (terms, largest first)."""
    out, i = [], number.bit_length() - 1
    while i >= 0:
        b0 = (number >> (i - 1)) & 1 if i > 0 else 0
        b1 = (number >> i) & 1
        b2 = (number >> (i + 1)) & 1
        if (b2, b1, b0) == (0, 1, 0):
            out.append(1 << i)
            i -= 1
        elif (b2, b1, b0) == (0, 1, 1):
            out.append(1 << (i + 1))
        elif (b2, b1, b0) == (1, 1, 0):
            out.append(-(1 << i))
        i -= 1
    return out


def test_terms_match_bit_utils_scan():
    for q in range(1, 1 << 13):
        p, n = O.terms(q)
        mine = sorted([1 << i for i in range(32) if (p >> i) & 1] +
                      [-(1 << i) for i in range(32) if (n >> i) & 1], key=lambda t: -abs(t))
        assert mine == _py_hese(q), q


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (no /root/reference)")
def test_restatement_equals_reference_body_random():
    rng = np.random.default_rng(7)
    for g in (1, 2, 4, 8, 16, 32):
        for bits in (3, 6, 8, 9, 12, 16):
            x = (rng.standard_normal((3, 64, 3, 3)) * rng.uniform(0.1, 3)).astype(np.float32)
            sf = float(np.abs(x).max() / 2 ** (bits - 1))
            alpha = int(rng.integers(0, 3 * g + 2))
            assert bits_equal(O.ref_tr(x, sf, bits, g, alpha), O.tr(x, sf, bits, g, alpha))
            xd = x.astype(np.float64)
            assert bits_equal(O.ref_tr(xd, sf, bits, g, alpha), O.tr(xd, sf, bits, g, alpha))


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (no /root/reference)")
def test_encoder_equals_reference_exhaustive_17bit():
    for q in range(0, 1 << 17, 1):
        p, n = O.terms(q)
        mine = sorted([1 << i for i in range(32) if (p >> i) & 1] +
                      [-(1 << i) for i in range(32) if (n >> i) & 1], key=lambda t: -abs(t))
        assert mine == O.ref_hese_terms(float(q), 1.0, 17), q


def test_tail_group_is_zero_padding():
    # SURVEY 8a-3: C % g != 0 is defined as the reference on a zero-padded tensor
    rng = np.random.default_rng(3)
    x = rng.standard_normal((4, 650)).astype(np.float32)
    xp = np.zeros((4, 656), dtype=np.float32)
    xp[:, :650] = x
    sf = float(np.abs(x).max() / 128)
    assert bits_equal(O.tr(x, sf, 8, 8, 12), O.tr(xp, sf, 8, 8, 12)[:, :650].copy())
    if O.have_ref():
        assert bits_equal(O.tr(x, sf, 8, 8, 12), O.ref_tr(xp, sf, 8, 8, 12)[:, :650].copy())


def test_relu_and_codes():
    x = np.array([[-3.0, 2.0, -0.2, 7.0]], dtype=np.float32)
    out, codes = O.tr(x, 1.0, 8, 1, 8, relu=True, return_codes=True)
    assert out.tolist() == [[0, 2, 0, 7]] and codes.tolist() == [[0, 2, 0, 7]]
    out, codes = O.tr(x, 1.0, 8, 1, 1, return_codes=True)
    assert codes.tolist() == [[-4, 2, 0, 8]]
    assert not np.signbit(out[0, 2])          # small negative -> +0.0 like the reference


def test_hist_and_mse_profile_and_counts():
    x = np.array([-50.0, 50.0, 0.0, 49.999, -60.0, 61.0, 0.0061], dtype=np.float32)
    h = O.hist(x, np.zeros(8192, dtype=np.float32), -50, 50)
    assert h.sum() == 5 and h[0] == 1 and h[8191] == 2 and h[4096] == 2
    # mse_profile (tr_layer.py:43-54): a histogram concentrated at one value picks an sf
    # that represents that value exactly
    grid = np.linspace(-50, 50, 8192, dtype=np.float32)
    hb = np.zeros(8192, dtype=np.float32)
    hb[6000] = 10
    sfs = np.linspace(1e-8, 50, 2048, dtype=np.float32)
    idx, errs = O.mse_profile(hb, grid, sfs, 8, 3)
    assert errs[idx] == errs.min() and errs[idx] < 1e-3
    # compute_compressed_hese (tr_layer.py:57-63): 3 = 4-1 (2 terms), 5 = 4+1 (2), 7 = 8-1 (2), 0
    assert O.hese_term_count(np.array([3, -5, 7, 0, 8], dtype=np.float32), 1.0) == 7


def test_gemm_i32():
    rng = np.random.default_rng(0)
    a = rng.integers(-256, 257, size=(5, 33)).astype(np.int16)
    w = rng.integers(-128, 129, size=(7, 33)).astype(np.int16)
    assert np.array_equal(O.gemm_i32(a, w), a.astype(np.int64) @ w.astype(np.int64).T)


def test_truncated_hese_code_is_monotone_in_q():
    """For g = 1 the sum of the k largest HESE terms is a non-decreasing function of the quantised value (and the
    quantised value of the input), so a max-pool commutes with the encode of non-negative activations:
    maxpool(code(x)) == code(maxpool(x)).  fused.FusedVGG pools on the fp16 codes because of this."""
    for bits in (4, 6, 8, 9, 10):
        q = np.arange(0, 2 ** bits, dtype=np.float32).reshape(1, -1, 1, 1)
        for k in range(1, 7):
            _, codes = O.tr(q, 1.0, bits, 1, k, return_codes=True)
            assert np.all(np.diff(codes.reshape(-1)) >= 0), (bits, k)


def _enc_golden():
    import os
    from conftest import ROOT
    return np.load(os.path.join(ROOT, "tests", "golden", "enc_golden.npz"))


def test_binary_encoding_pinned_to_reference_expand_binary_bits():
    """TQ_ENC_BINARY against bit_utils.expand_binary_bits (bit_utils.py:63-73) run from the reference's text
    (tests/golden/make_golden_encodings.py): the oracle's quantised value and binary term set are the
    reference's MSB-first bit planes, and keeping the k most significant terms keeps the first k set planes."""
    z = _enc_golden()
    W, sf, bits, planes = z["bin_W"], float(z["bin_sf"]), int(z["bin_bits"]), z["bin_planes"]
    q_ref = (planes.astype(np.int64) << np.arange(bits - 1, -1, -1)).sum(1)
    for w, q, row in zip(W[:600], q_ref[:600], planes[:600]):
        assert O.quantize(abs(float(w)), sf, bits + 1) == q          # reference does not clip: give the quantiser room
        p, n = O.terms(int(q), O.ENC_BINARY)
        assert n == 0 and p == q
    x = W.reshape(1, -1, 1, 1)
    for k in (1, 2, 3, bits + 1):
        _, codes = O.tr(x, sf, bits + 1, 1, k, encoding=O.ENC_BINARY, return_codes=True)
        first_k = (np.cumsum(planes, axis=1) <= k) & (planes > 0)
        want = (first_k.astype(np.int64) << np.arange(bits - 1, -1, -1)).sum(1) * np.where(W < 0, -1, 1)
        assert np.array_equal(codes.reshape(-1), want)


def test_booth_encoding_pinned_to_verilog_truth_table():
    """TQ_ENC_BOOTH against verilog/booth_encoder.v:57-78 clocked bit-serially over every 12-bit value
    (tests/golden/make_golden_encodings.py): same positive / negative digit masks."""
    z = _enc_golden()
    for q, P, N in zip(z["booth_q"], z["booth_P"], z["booth_N"]):
        assert O.terms(int(q), O.ENC_BOOTH) == (int(P), int(N)), q


@pytest.mark.parametrize("bits", range(1, 12))
def test_fused_encoder_hard_values_hit_every_class(bits):
    """The hard values of tests/test_fused_encoders_gpu.py really contain, for every (sf, bits) it uses, a tie that
    rounds up, its lower neighbour rounding down, saturated codes of both signs, NaN (-> 0), zeros of both signs and
    the smallest subnormal: the GPU comparisons cannot quietly turn trivial."""
    from test_fused_encoders_gpu import ALL_SFS, hard_values, _oracle_codes
    for sf in ALL_SFS:
        x = hard_values(sf, bits)
        sf32 = np.float32(sf)
        q = np.array([O.quantize(v, sf32, bits) for v in x])
        with np.errstate(over="ignore"):
            r = np.abs(x) / sf32                                       # fp32 IEEE divide, as the kernels compute it
        tie = np.flatnonzero(np.isfinite(r) & (r == np.floor(r) + np.float32(0.5)) & (r < 2 ** bits - 1))
        assert tie.size, (sf, bits, "no exact tie below saturation")
        ups = [i for i in tie if q[i] == int(r[i]) + 1]
        assert ups, (sf, bits, "no tie rounds up")
        lows = [i for i in ups if O.quantize(np.nextafter(x[i], np.float32(0)), sf32, bits) == int(r[i])
                and np.nextafter(x[i], np.float32(0)) in x]
        assert lows, (sf, bits, "no tie's lower neighbour (in the set) rounds down")
        codes = _oracle_codes(x, sf, bits, bits)                       # budget not binding: saturation shows
        sat = int(_oracle_codes(np.array([np.inf], np.float32), sf, bits, bits)[0])
        assert sat > 0 and (codes == sat).any() and (codes == -sat).any(), (sf, bits, "saturated codes of both signs")
        nan = np.isnan(x)
        assert nan.any() and (codes[nan] == 0).all() and (_oracle_codes(x, sf, bits, 0) == 0).all()
        assert (x == 0).sum() == 2 and np.signbit(x[x == 0]).sum() == 1                  # +0 and -0
        assert (np.abs(x) == np.float32(2.0 ** -149)).sum() == 2
