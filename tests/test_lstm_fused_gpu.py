"""The LSTM recurrence kernel (tq_lstm_recurrence: all T steps of a layer in one cooperative launch) and the fused
language-model executor built on it (fused.FusedLSTM), on the GPU.

Numerics contract: the recurrence is fp32 with one fixed summation order.  It is not bit-comparable with cuDNN or with
the step-wise torch loop, so it is held to an fp64 recurrence on the same inputs at 1e-5 * max(|ref|, 1); eager calls
and CUDA-graph replays are bit-identical; the decoder stays an exact integer contraction of the codes it is given."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

ENCS = ["hese", "binary", "booth"]


@pytest.fixture(autouse=True)
def _fp32_math():
    # cuDNN's LSTM (the tcgen05 path's upper layers) and the fused path's upper-layer GEMM stay true fp32
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _within(a, b):
    err = float((a.double() - b.double()).abs().max())
    assert err <= 1e-5 * max(float(b.abs().max()), 1.0), err


def _ref_recurrence(gin, bias, w, h0, c0):
    """fp64 recurrence in torch gate order i, f, g, o."""
    W, h, c = w.double(), h0.double(), c0.double()
    b = bias.double() if bias is not None else 0.0
    ys = []
    for t in range(gin.shape[0]):
        z = gin[t].double() + b + h @ W.t()
        i, f, g, o = z.chunk(4, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        ys.append(h)
    return torch.stack(ys), h, c


def _operands(T, B, H, bias, gen, saturate=False):
    s = 1.0 / H ** 0.5
    gin = torch.randn(T, B, 4 * H, device="cuda", generator=gen) * 0.5
    if saturate:
        # gates around +-30: sigmoid / tanh saturate, and c grows by about one per step (i = f = 1, g = +1 on every
        # unit); the output gate keeps random signs
        gin = torch.sign(gin) * 30.0
        gin[:, :, :3 * H] = 30.0
    w = (torch.rand(4 * H, H, device="cuda", generator=gen) * 2 - 1) * s
    b = (torch.rand(4 * H, device="cuda", generator=gen) * 2 - 1) * s if bias else None
    h0 = torch.randn(B, H, device="cuda", generator=gen) * 0.3
    c0 = torch.randn(B, H, device="cuda", generator=gen) * 0.3
    return gin, b, w, h0, c0


# 1 / 7 / 33 units: one unit per CTA; 301: 3 units per CTA and a last CTA with one; 650 (the language model): 5 units on
# each of 130 CTAs; 1024: 7 units per CTA, the last with 2, and at B = 128 the hidden rows are staged in 5 tiles
CASES = [(1, 1, 1, True), (2, 3, 1, False), (35, 80, 1, True), (1, 128, 7, True), (35, 3, 7, False), (2, 1, 33, True),
         (35, 128, 33, False), (2, 80, 301, True), (35, 1, 650, True), (1, 80, 650, False), (35, 80, 650, True),
         (2, 128, 650, True), (35, 3, 1024, True), (2, 128, 1024, False), (35, 128, 1024, True), (35, 80, 1024, True)]


@pytest.mark.parametrize("T,B,H,bias", CASES)
def test_recurrence_against_fp64(T, B, H, bias):
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(T * 10007 + B * 101 + H)
    args = _operands(T, B, H, bias, gen)
    y, hn, cn = conv_codes.lstm_recurrence(*args)
    ry, rh, rc = _ref_recurrence(*args)
    assert y.shape == (T, B, H) and hn.shape == (B, H) and cn.shape == (B, H)
    for a, b in ((y, ry), (hn, rh), (cn, rc)):
        _within(a, b)
    assert torch.equal(hn, y[-1])


@pytest.mark.parametrize("H", [7, 650])
def test_recurrence_saturating_gates(H):
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(H)
    args = _operands(35, 80, H, True, gen, saturate=True)
    y, hn, cn = conv_codes.lstm_recurrence(*args)
    ry, rh, rc = _ref_recurrence(*args)
    assert float(rc.abs().max()) > 30                        # c really grew
    for a, b in ((y, ry), (hn, rh), (cn, rc)):
        _within(a, b)


def test_recurrence_eager_and_replay_bit_identical():
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(7)
    args = _operands(35, 80, 650, True, gen)
    first = conv_codes.lstm_recurrence(*args)
    second = conv_codes.lstm_recurrence(*args)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        conv_codes.lstm_recurrence(*args)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = conv_codes.lstm_recurrence(*args)
    graph.replay()
    torch.cuda.synchronize()
    for a, b, c in zip(first, second, out):
        assert torch.equal(a, b) and torch.equal(a, c)


# ---- the executor ---------------------------------------------------------------------------------------------

def _lm(enc="hese", H=650, layers=2, ntoken=None, seed=0, T=35, B=80, data_bits=8, kind="LSTM"):
    """A calibrated TQ RNNModel (the bench's settings: wb 8, g 8, alpha 12, db 8, 8 data terms) with a non-zero decoder
    bias, its calibration tokens and a random hidden state."""
    from term_quantization_b200 import evaluate_lstm, tr_layer
    from term_quantization_b200.lstm_models.model import RNNModel
    ntoken = ntoken or evaluate_lstm.NTOKENS
    torch.manual_seed(seed)
    base = RNNModel(kind, ntoken, H, H, layers, 0.5, True).cuda().eval()
    base.decoder.bias.data.uniform_(-0.1, 0.1)
    q = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), data_bits, 8,
                                    encoding=enc)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    tokens = torch.randint(ntoken, (T, B), device="cuda", generator=g)
    hidden = tuple(torch.randn(layers, B, H, device="cuda", generator=g) * 0.3 for _ in range(2))
    if kind == "LSTM":
        with torch.no_grad():
            q(tokens, hidden)
            tr_layer.set_tr_tracking(q, False)
    return q, tokens, hidden


def _tc_and_fused(q):
    from term_quantization_b200 import fused, tr_layer
    q_tc = copy.deepcopy(q)
    tr_layer.use_tensor_cores(q_tc)
    return q_tc, fused.FusedLSTM(copy.deepcopy(q))


def _q(y, quant):
    """sign(y) * q: the quantised integer before the term encoding (binary with a budget that never binds)."""
    from term_quantization_b200 import tr_cuda
    return tr_cuda.tr_codes(y.contiguous().view(1, -1, 1, 1), quant.sf, quant.data_bits, 1, quant.data_bits + 2,
                            dtype=torch.int32, encoding="binary").view(y.shape)


@pytest.mark.parametrize("enc", ENCS)
def test_executor_against_tensor_core_path(enc):
    from term_quantization_b200 import tr_cuda
    q, tokens, hidden = _lm(enc)
    q_tc, f = _tc_and_fused(q)
    seen = {}
    hook = q_tc.decoder.register_forward_hook(lambda m, i, o: seen.update(x=i[0]))
    cap = {}
    with torch.no_grad():
        out_tc, (h_tc, c_tc) = q_tc(tokens, hidden)
        out_f, (h_f, c_f) = f(tokens, hidden, capture=cap)
    hook.remove()
    y_tc = seen["x"]
    assert out_f.shape == out_tc.shape == (35 * 80, q.ntoken) and h_f.shape == h_tc.shape == (2, 80, 650)
    for a, b in ((h_f, h_tc), (c_f, c_tc), (cap["y"], y_tc)):
        _within(a, b)
    # decoder input codes: equal wherever the two paths quantise to the same integer; elsewhere the fp32 values sit on
    # either side of a rounding boundary (k - 1/2) * sf
    dq = f.model.decoder.input_quant
    codes_tc = tr_cuda.tr_codes(y_tc.contiguous().view(1, -1, 1, 1), dq.sf, dq.data_bits, 1, dq.data_terms,
                                dtype=torch.float16, encoding=dq.encoding).view(-1, 650)
    q_f, q_t = _q(cap["y"], dq).view(-1, 650), _q(y_tc, dq).view(-1, 650)
    same = q_f == q_t
    assert torch.equal(cap["codes"][same], codes_tc[same])
    diff = ~same
    assert int(diff.sum()) <= 1e-2 * diff.numel()
    if diff.any():
        a, b = q_f[diff].abs(), q_t[diff].abs()
        assert int((a - b).abs().max()) == 1 and not bool(((q_f[diff] * q_t[diff]) < 0).any())
        edge = torch.maximum(a, b).double() - 0.5
        sf32 = float(np.float32(dq.sf))
        r_f = cap["y"].reshape(-1, 650)[diff].double().abs() / sf32
        r_t = y_tc.reshape(-1, 650)[diff].double().abs() / sf32
        lo, hi = torch.minimum(r_f, r_t), torch.maximum(r_f, r_t)
        assert bool((lo <= edge + 1e-4).all()) and bool((hi >= edge - 1e-4).all())
    # the decoder is exact: float(int32 GEMM of the codes it was given) * scale + bias, bit for bit
    dec = f.model.decoder
    wsf = np.float32(dec.w_sf)
    wc = torch.round(dec.linear.weight / wsf)
    assert torch.equal(wc * wsf, dec.linear.weight)
    acc = cap["codes"].double() @ wc.double().t()
    scale = float(np.float32(dq.sf) * wsf)
    assert torch.equal(cap["decoded"], acc.float() * scale + dec.linear.bias)
    assert torch.equal(out_f, torch.log_softmax(cap["decoded"], dim=1))


def test_executor_graph_replay_equals_eager():
    from term_quantization_b200 import evaluate_lstm
    q, tokens, hidden = _lm("hese")
    _, f = _tc_and_fused(q)
    g = torch.Generator(device="cuda").manual_seed(99)
    tok = tokens.clone()
    hid = tuple(h.clone() for h in hidden)
    with torch.no_grad():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                f(tok, hid)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out, (h, c) = f(tok, hid)
        seen = []
        for _ in range(3):
            tok.copy_(torch.randint(evaluate_lstm.NTOKENS, tok.shape, device="cuda", generator=g))
            for t in hid:
                t.copy_(torch.randn(t.shape, device="cuda", generator=g) * 0.3)
            graph.replay()
            got = (out.clone(), h.clone(), c.clone())
            want_out, (want_h, want_c) = f(tok, hid)
            for a, b in zip(got, (want_out, want_h, want_c)):
                assert torch.equal(a, b), float((a - b).abs().max())
            seen.append(got)
    for k in range(3):
        assert all(not torch.equal(seen[i][k], seen[j][k]) for i in range(3) for j in range(i))


def test_executor_carries_hidden_state_across_chunks():
    q, tokens, hidden = _lm("hese")
    q_tc, f = _tc_and_fused(q)
    g = torch.Generator(device="cuda").manual_seed(5)
    chunks = [tokens, torch.randint(q.ntoken, tokens.shape, device="cuda", generator=g)]
    h_tc = h_f = hidden
    with torch.no_grad():
        for x in chunks:
            out_tc, h_tc = q_tc(x, h_tc)
            out_f, h_f = f(x, h_f)
            for a, b in zip(h_f, h_tc):
                _within(a, b)
    # the log-probabilities of the second chunk agree as closely as the decoder's quantiser allows
    assert float((out_f - out_tc).abs().mean()) < 1e-3


def test_driver_fused_engine_matches_tcgen05():
    from term_quantization_b200 import evaluate_lstm
    args = ["--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--emsize", "64", "--nhid", "64",
            "--tokens", "1500"]
    tc = evaluate_lstm.main(args + ["--engine", "tcgen05"])
    fu = evaluate_lstm.main(args + ["--engine", "fused"])
    assert abs(fu["ppls"][0] - tc["ppls"][0]) <= 1e-4 * tc["ppls"][0], (fu["ppls"], tc["ppls"])
    assert fu["tmacs"] == tc["tmacs"] and fu["param_bits"] == tc["param_bits"]


# ---- refusals ---------------------------------------------------------------------------------------------------

def test_kernel_refuses_before_any_launch():
    from term_quantization_b200 import _lib, conv_codes
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(1 << 20, device="cuda")
    p = buf.data_ptr()
    hmax = conv_codes.lstm_max_hidden()
    n0 = _lib.launch_count()
    bad = [
        (None, None, p, p, p, p, p, p, 1, 1, 8),             # NULL gin
        (p, None, None, p, p, p, p, p, 1, 1, 8),             # NULL w_hh
        (p, None, p, p, p, p, p, None, 1, 1, 8),             # NULL cn
        (p + 2, None, p, p, p, p, p, p, 1, 1, 8),            # misaligned gin
        (p, p + 1, p, p, p, p, p, p, 1, 1, 8),               # misaligned bias
        (p, None, p, p, p, p + 6, p, p, 1, 1, 8),            # misaligned y
        (p, None, p, p, p, p, p, p, 0, 1, 8),                # T < 1
        (p, None, p, p, p, p, p, p, 1, 0, 8),                # B < 1
        (p, None, p, p, p, p, p, p, 1, 1, 0),                # H < 1
        (p, None, p, p, p, p, p, p, 1, 1, -5),
    ]
    for a in bad:
        assert L.tq_lstm_recurrence(*a, s) == _lib.TQ_ERR_INVALID, a
    rc = L.tq_lstm_recurrence(p, None, p, p, p, p, p, p, 1, 1, hmax + 1, s)
    assert rc == _lib.TQ_ERR_UNSUPPORTED and f"largest H on this device: {hmax}" in L.tq_last_error().decode()
    assert _lib.launch_count() == n0
    with pytest.raises(RuntimeError):
        conv_codes.lstm_recurrence(torch.zeros(1, 1, 8, device="cuda"), None, torch.zeros(8, 2, device="cuda"),
                                   torch.zeros(1, 3, device="cuda"), torch.zeros(1, 2, device="cuda"))
    with pytest.raises(RuntimeError):
        conv_codes.lstm_recurrence(torch.zeros(1, 1, 8, device="cuda").double(), None, torch.zeros(8, 2, device="cuda"),
                                   torch.zeros(1, 2, device="cuda"), torch.zeros(1, 2, device="cuda"))
    assert _lib.launch_count() == n0
    # at the bound it runs
    gen = torch.Generator(device="cuda").manual_seed(1)
    args = _operands(2, 2, hmax, True, gen)
    y, hn, cn = conv_codes.lstm_recurrence(*args)
    ry, rh, rc = _ref_recurrence(*args)
    _within(y, ry)


def test_executor_refusals():
    from term_quantization_b200 import _lib, fused, tr_layer, conv_codes
    cases = []
    q, tokens, hidden = _lm("hese", H=32, ntoken=100, T=5, B=4)
    cases.append(("uncalibrated", _lm("hese", H=32, ntoken=100, kind="LSTM", T=5, B=4)[0]))
    tr_layer.set_tr_tracking(cases[-1][1], True)
    tr = copy.deepcopy(q).train()
    cases.append(("training", tr))
    for kind in ("GRU", "RNN_TANH"):
        m, _, _ = _lm("hese", H=32, ntoken=100, kind=kind, T=5, B=4)
        cases.append((kind, m))
    from term_quantization_b200 import evaluate_lstm
    from term_quantization_b200.lstm_models.model import RNNModel
    for kw in ({"bidirectional": True}, {"batch_first": True}, {"proj_size": 16}):
        base = RNNModel("LSTM", 100, 32, 32, 1, 0.0, False).cuda().eval()
        base.rnn = nn.LSTM(32, 32, 1, **kw).cuda().eval()
        m = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8)
        tr_layer.set_tr_tracking(m, False)
        cases.append((str(kw), m))
    m11, _, _ = _lm("hese", H=32, ntoken=100, T=5, B=4, data_bits=11)          # decoder codes above 2^10
    cases.append(("decoder bits", m11))
    hmax = conv_codes.lstm_max_hidden()
    big = RNNModel("LSTM", 100, 16, hmax + 1, 1, 0.0, False).cuda().eval()
    big = evaluate_lstm.convert_model(big, evaluate_lstm.static_lstm_layer_settings(big, 8, 8, 12), 8, 8)
    tr_layer.set_tr_tracking(big, False)
    cases.append(("H above the bound", big))
    n0 = _lib.launch_count()
    for what, m in cases:
        with pytest.raises((RuntimeError, NotImplementedError)):
            fused.FusedLSTM(m)
            pytest.fail(what)
    assert _lib.launch_count() == n0
    # stale weights, a model switched back to training, re-calibration after fusing
    f = fused.FusedLSTM(q)
    with torch.no_grad():
        f(tokens, hidden)
        q.rnn.lstm.weight_hh_l1.mul_(1.0)
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f(tokens, hidden)
    f = fused.FusedLSTM(q)
    f.train()
    with pytest.raises(RuntimeError, match="inference only"):
        f(tokens, hidden)
    f.eval()
    sf = q.rnn.input_quant.sf
    tr_layer.set_tr_tracking(q, True)
    n1 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="tracking"):
        f(tokens, hidden)
    assert _lib.launch_count() == n1
    q.rnn.input_quant.hist_bins.zero_()
    q.rnn.input_quant(torch.randn(100000, device="cuda") * 5)          # a histogram of much wider activations
    tr_layer.set_tr_tracking(q, False)
    assert q.rnn.input_quant.sf != sf
    n1 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f(tokens, hidden)
    assert _lib.launch_count() == n1
