"""The GRU and vanilla-RNN recurrence kernels (tq_gru_recurrence, tq_rnn_recurrence: the LSTM's persistent cooperative
kernel instantiated for 3 and 1 gates) and the fused executor built on them (fused.FusedRNN), on the GPU.

Numerics contract, as for the LSTM: fp32 with one fixed summation order, held to an fp64 recurrence on the same inputs
at 1e-5 * max(|ref|, 1); eager calls, side streams and CUDA-graph replays are bit-identical; the decoder stays an exact
integer contraction of the codes it is given, and nll agrees with nll_loss over forward's log-probabilities."""
import copy
import gc

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

CELLS = ["GRU", "RNN_TANH", "RNN_RELU"]
ENCS = ["hese", "binary", "booth"]
GATES = {"GRU": 3, "RNN_TANH": 1, "RNN_RELU": 1}


@pytest.fixture(autouse=True)
def _fp32_math():
    # cuDNN's GRU / RNN (the tcgen05 path) and the fused path's input GEMMs stay true fp32
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _within(a, b, tol=1e-5):
    err = float((a.double() - b.double()).abs().max())
    assert err <= tol * max(float(b.abs().max()), 1.0), err


def _run(cell, gin, bias, w, h0):
    from term_quantization_b200 import conv_codes
    if cell == "GRU":
        return conv_codes.gru_recurrence(gin, bias, w, h0)
    return conv_codes.rnn_recurrence(gin, bias, w, h0, cell.split("_")[1].lower())


def _ref(cell, gin, bias, w, h0):
    """fp64 recurrence with torch's formulas (GRU gate order r, z, n; b_hn inside the reset gate's product)."""
    W, h = w.double(), h0.double()
    b = bias.double() if bias is not None else torch.zeros(w.shape[0], dtype=torch.float64, device=w.device)
    ys = []
    for t in range(gin.shape[0]):
        gi = gin[t].double()
        gh = h @ W.t() + b
        if cell == "GRU":
            ir, iz, i_n = gi.chunk(3, dim=1)
            hr, hz, h_n = gh.chunk(3, dim=1)
            r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
            n = torch.tanh(i_n + r * h_n)
            h = (1 - z) * n + z * h
        else:
            h = torch.tanh(gi + gh) if cell == "RNN_TANH" else torch.relu(gi + gh)
        ys.append(h)
    return torch.stack(ys), h


def _operands(cell, T, B, H, bias, gen, saturate=False):
    G = GATES[cell]
    s = 1.0 / H ** 0.5
    gin = torch.randn(T, B, G * H, device="cuda", generator=gen) * 0.5
    if saturate:
        gin = torch.sign(gin) * 30.0                         # every gate pre-activation around +-30
    w = (torch.rand(G * H, H, device="cuda", generator=gen) * 2 - 1) * s
    b = (torch.rand(G * H, device="cuda", generator=gen) * 2 - 1) * s if bias else None
    h0 = torch.randn(B, H, device="cuda", generator=gen) * 0.3
    return gin, b, w, h0


# the LSTM test's grid: 1 / 7 / 33 units: one unit per CTA; 301: 3 units per CTA and a last CTA with one; 650: 5 units on
# each of 130 CTAs; 1024: 7 units per CTA, the last with 2; B = 128 with H = 1024 stages the hidden rows in several tiles
CASES = [(1, 1, 1, True), (2, 3, 1, False), (35, 80, 1, True), (1, 128, 7, True), (35, 3, 7, False), (2, 1, 33, True),
         (35, 128, 33, False), (2, 80, 301, True), (35, 1, 650, True), (1, 80, 650, False), (35, 80, 650, True),
         (2, 128, 650, True), (35, 3, 1024, True), (2, 128, 1024, False), (35, 128, 1024, True), (35, 80, 1024, True)]


@pytest.mark.parametrize("cell", CELLS)
@pytest.mark.parametrize("T,B,H,bias", CASES)
def test_recurrence_against_fp64(cell, T, B, H, bias):
    gen = torch.Generator(device="cuda").manual_seed(T * 10007 + B * 101 + H)
    args = _operands(cell, T, B, H, bias, gen)
    y, hn = _run(cell, *args)
    ry, rh = _ref(cell, *args)
    assert y.shape == (T, B, H) and hn.shape == (B, H)
    _within(y, ry)
    _within(hn, rh)
    assert torch.equal(hn, y[-1])


@pytest.mark.parametrize("cell", CELLS)
def test_recurrence_hidden_rows_in_many_tiles(cell):
    # H = 2048 (RNN) / 1536 (GRU): few hidden rows fit next to the weights, so B = 80 takes several tiles per step
    from term_quantization_b200 import conv_codes
    H = min(2048 if GATES[cell] == 1 else 1536, conv_codes.recurrence_max_hidden(cell))
    gen = torch.Generator(device="cuda").manual_seed(H)
    args = _operands(cell, 3, 80, H, True, gen)
    y, hn = _run(cell, *args)
    ry, rh = _ref(cell, *args)
    _within(y, ry)
    _within(hn, rh)


@pytest.mark.parametrize("cell", CELLS)
@pytest.mark.parametrize("H", [7, 650])
def test_recurrence_saturating_gates(cell, H):
    gen = torch.Generator(device="cuda").manual_seed(H + 1)
    args = _operands(cell, 35, 80, H, True, gen, saturate=True)
    y, hn = _run(cell, *args)
    ry, rh = _ref(cell, *args)
    if cell == "RNN_RELU":
        assert float(ry.abs().max()) > 30                    # the ReLU RNN's state really grew
    _within(y, ry)
    _within(hn, rh)


def test_relu_recurrence_keeps_nan():
    gen = torch.Generator(device="cuda").manual_seed(11)
    gin, b, w, h0 = _operands("RNN_RELU", 6, 80, 650, True, gen)
    gin[2, 5, 17] = float("nan")                             # row 5 is NaN from step 2 on, every other row stays finite
    gin[0, 9, 3] = -float("nan")
    y, hn = _run("RNN_RELU", gin, b, w, h0)
    ry, rh = _ref("RNN_RELU", gin, b, w, h0)
    assert bool(torch.isnan(ry).any()) and not bool(torch.isnan(ry).all())
    assert torch.equal(torch.isnan(y), torch.isnan(ry)) and torch.equal(torch.isnan(hn), torch.isnan(rh))
    ok = ~torch.isnan(ry)
    _within(y[ok], ry[ok])


@pytest.mark.parametrize("cell", CELLS)
def test_recurrence_eager_side_stream_and_replay_bit_identical(cell):
    gen = torch.Generator(device="cuda").manual_seed(7)
    args = _operands(cell, 35, 80, 650, True, gen)
    first = _run(cell, *args)
    second = _run(cell, *args)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        on_side = _run(cell, *args)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _run(cell, *args)
    graph.replay()
    torch.cuda.synchronize()
    for a, b, c, d in zip(first, second, on_side, out):
        assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(a, d)


# ---- the executor ---------------------------------------------------------------------------------------------

def _lm(kind, enc="hese", H=650, layers=2, ntoken=None, seed=0, T=35, B=80, data_bits=8, calibrate=True):
    """A calibrated TQ RNNModel(kind) (the bench's settings: wb 8, g 8, alpha 12, db 8, 8 data terms; only the decoder
    is wrapped) with a non-zero decoder bias, its tokens, next tokens and a random hidden state."""
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
    targets = torch.randint(ntoken, (T * B,), device="cuda", generator=g)
    hidden = torch.randn(layers, B, H, device="cuda", generator=g) * 0.3
    if kind == "LSTM":
        hidden = (hidden, hidden.clone())
    if calibrate:
        with torch.no_grad():
            q(tokens, hidden)
            tr_layer.set_tr_tracking(q, False)
    return q, tokens, targets, hidden


def _q(y, quant):
    """sign(y) * q: the quantised integer before the term encoding (binary with a budget that never binds)."""
    from term_quantization_b200 import tr_cuda
    return tr_cuda.tr_codes(y.contiguous().view(1, -1, 1, 1), quant.sf, quant.data_bits, 1, quant.data_bits + 2,
                            dtype=torch.int32, encoding="binary").view(y.shape)


@pytest.mark.parametrize("enc", ENCS)
@pytest.mark.parametrize("cell", CELLS)
def test_executor_against_tensor_core_path(cell, enc):
    from term_quantization_b200 import fused, tr_cuda, tr_layer
    q, tokens, _, hidden = _lm(cell, enc)
    q_tc = copy.deepcopy(q)
    tr_layer.use_tensor_cores(q_tc)
    f = fused.FusedRNN(copy.deepcopy(q))
    seen = {}
    hook = q_tc.decoder.register_forward_hook(lambda m, i, o: seen.update(x=i[0]))
    cap = {}
    with torch.no_grad():
        out_tc, h_tc = q_tc(tokens, hidden)
        out_f, h_f = f(tokens, hidden, capture=cap)
    hook.remove()
    y_tc = seen["x"]
    assert out_f.shape == out_tc.shape == (35 * 80, q.ntoken) and h_f.shape == h_tc.shape == (2, 80, 650)
    _within(h_f, h_tc)
    _within(cap["y"], y_tc)
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


@pytest.mark.parametrize("cell", CELLS)
def test_executor_nll_against_nll_loss_of_forward(cell):
    from term_quantization_b200 import fused
    q, tokens, targets, hidden = _lm(cell)
    f = fused.FusedRNN(q)
    g = torch.Generator(device="cuda").manual_seed(3)
    chunks = [(tokens, targets), (torch.randint(q.ntoken, tokens.shape, device="cuda", generator=g),
                                  torch.randint(q.ntoken, targets.shape, device="cuda", generator=g))]
    hf = hn = hidden
    with torch.no_grad():
        for x, t in chunks:                                   # the hidden state carried across two bptt chunks
            out, hf = f(x, hf)
            loss, hn = f.nll(x, t, hn)
            assert loss.shape == (35 * 80,) and loss.dtype == torch.float32
            _within(loss, F.nll_loss(out, t, reduction="none"), tol=4e-6)
            assert torch.equal(hn, hf)


@pytest.mark.parametrize("cell", CELLS)
def test_executor_nll_peak_memory_and_graph_replay(cell):
    from term_quantization_b200 import evaluate_lstm, fused
    T, B = 35, 80
    q, tokens, targets, hidden = _lm(cell, T=T, B=B)
    f = fused.FusedRNN(q)
    V = q.ntoken
    with torch.no_grad():
        f.nll(tokens, targets, hidden)                        # plans, cuBLAS workspace, module loads
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = f.nll(tokens, targets, hidden)
        torch.cuda.synchronize()
        rise = torch.cuda.max_memory_allocated() - base
        del out
        assert rise < T * B * V * 4 / 8, (rise, T * B * V * 4 / 8)

        g = torch.Generator(device="cuda").manual_seed(99)
        tok, tgt, hid = tokens.clone(), targets.clone(), hidden.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                f.nll(tok, tgt, hid)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss, h = f.nll(tok, tgt, hid)
        for _ in range(2):
            tok.copy_(torch.randint(evaluate_lstm.NTOKENS, tok.shape, device="cuda", generator=g))
            tgt.copy_(torch.randint(evaluate_lstm.NTOKENS, tgt.shape, device="cuda", generator=g))
            hid.copy_(torch.randn(hid.shape, device="cuda", generator=g) * 0.3)
            graph.replay()
            got = (loss.clone(), h.clone())
            want = f.nll(tok, tgt, hid)
            for a, b in zip(got, want):
                assert torch.equal(a, b), float((a - b).abs().max())


@pytest.mark.parametrize("cell", CELLS)
def test_driver_fused_engine_matches_tcgen05(cell):
    from term_quantization_b200 import evaluate_lstm
    args = ["--model", cell, "--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--emsize", "64",
            "--nhid", "64", "--tokens", "1500"]
    tc = evaluate_lstm.main(args + ["--engine", "tcgen05"])
    fu = evaluate_lstm.main(args + ["--engine", "fused"])
    assert abs(fu["ppls"][0] - tc["ppls"][0]) <= 1e-4 * tc["ppls"][0], (fu["ppls"], tc["ppls"])
    assert fu["tmacs"] == tc["tmacs"] and fu["param_bits"] == tc["param_bits"]


# ---- refusals ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cell", CELLS)
def test_kernel_refuses_before_any_launch(cell):
    from term_quantization_b200 import _lib, conv_codes
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(1 << 20, device="cuda")
    p = buf.data_ptr()
    hmax = conv_codes.recurrence_max_hidden(cell)
    assert hmax == L.tq_recurrence_max_hidden(GATES[cell])
    assert hmax > conv_codes.lstm_max_hidden()
    if cell == "GRU":
        call = lambda gin, b, w, h0, y, hn, T, B, H: L.tq_gru_recurrence(gin, b, w, h0, y, hn, T, B, H, s)  # noqa: E731
    else:
        relu = int(cell == "RNN_RELU")
        call = lambda gin, b, w, h0, y, hn, T, B, H: L.tq_rnn_recurrence(gin, b, w, h0, y, hn, T, B, H, relu, s)  # noqa: E731
    n0 = _lib.launch_count()
    bad = [
        (None, None, p, p, p, p, 1, 1, 8),                   # NULL gin
        (p, None, None, p, p, p, 1, 1, 8),                   # NULL w_hh
        (p, None, p, None, p, p, 1, 1, 8),                   # NULL h0
        (p, None, p, p, None, p, 1, 1, 8),                   # NULL y
        (p, None, p, p, p, None, 1, 1, 8),                   # NULL hn
        (p + 2, None, p, p, p, p, 1, 1, 8),                  # misaligned gin
        (p, p + 1, p, p, p, p, 1, 1, 8),                     # misaligned bias
        (p, None, p, p, p + 6, p, 1, 1, 8),                  # misaligned y
        (p, None, p, p, p, p, 0, 1, 8),                      # T < 1
        (p, None, p, p, p, p, 1, 0, 8),                      # B < 1
        (p, None, p, p, p, p, 1, 1, 0),                      # H < 1
        (p, None, p, p, p, p, 1, 1, -5),
        (p, None, p, p, p, p, 1, (1 << 31) // (GATES[cell] * 8) + 1, 8),   # B * G * H above 2^31 - 1
    ]
    for a in bad:
        assert call(*a) == _lib.TQ_ERR_INVALID, a
    assert call(p, None, p, p, p, p, 1, 1, hmax + 1) == _lib.TQ_ERR_UNSUPPORTED
    assert f"largest H on this device: {hmax}" in L.tq_last_error().decode()
    assert L.tq_recurrence_max_hidden(2) == -1
    assert _lib.launch_count() == n0
    z = lambda *s: torch.zeros(*s, device="cuda")  # noqa: E731
    G = GATES[cell]
    for args in ((z(1, 1, G * 2), None, z(G * 2, 2), z(1, 3)),                    # h0 of the wrong width
                 (z(1, 1, G * 2).double(), None, z(G * 2, 2), z(1, 2)),           # fp64
                 (z(1, 1, G * 2), z(G * 2 + 1), z(G * 2, 2), z(1, 2)),            # bias of the wrong length
                 (z(1, 1, G * 4)[:, :, ::2], None, z(G * 2, 2), z(1, 2)),         # not contiguous
                 (z(1, 1, G * 2), None, z(G * 2, 2).cpu(), z(1, 2))):             # mixed devices
        with pytest.raises(RuntimeError):
            _run(cell, *args)
    with pytest.raises(ValueError):
        conv_codes.rnn_recurrence(z(1, 1, 2), None, z(2, 2), z(1, 2), "sigmoid")
    with pytest.raises(ValueError):
        conv_codes.recurrence_max_hidden("LSTMP")
    assert _lib.launch_count() == n0
    # at the bound it runs
    gen = torch.Generator(device="cuda").manual_seed(1)
    args = _operands(cell, 2, 2, hmax, True, gen)
    y, hn = _run(cell, *args)
    ry, rh = _ref(cell, *args)
    _within(y, ry)
    _within(hn, rh)


def test_executor_refusals():
    import torch.nn as nn
    from term_quantization_b200 import _lib, conv_codes, evaluate_lstm, fused, tr_layer
    from term_quantization_b200.lstm_models.model import RNNModel
    small = dict(H=32, ntoken=100, T=5, B=4)
    cases = [("uncalibrated", _lm("GRU", calibrate=False, **small)[0]),
             ("training", copy.deepcopy(_lm("GRU", **small)[0]).train()),
             ("LSTM", _lm("LSTM", **small)[0]),
             ("decoder bits", _lm("RNN_TANH", data_bits=11, **small)[0])]       # decoder codes above 2^10
    for kind, kw in (("GRU", {"bidirectional": True}), ("RNN_RELU", {"batch_first": True})):
        base = RNNModel(kind, 100, 32, 32, 1, 0.0, False).cuda().eval()
        cls = nn.GRU if kind == "GRU" else nn.RNN
        extra = {} if kind == "GRU" else {"nonlinearity": "relu"}
        base.rnn = cls(32, 32, 1, **kw, **extra).cuda().eval()
        m = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8)
        tr_layer.set_tr_tracking(m, False)
        cases.append((str(kw), m))
    half = _lm("GRU", **small)[0]
    half.rnn.half()
    cases.append(("fp16 parameters", half))
    for cell in CELLS:
        hmax = conv_codes.recurrence_max_hidden(cell)
        big = RNNModel(cell, 100, 16, hmax + 1, 1, 0.0, False).cuda().eval()
        big = evaluate_lstm.convert_model(big, evaluate_lstm.static_lstm_layer_settings(big, 8, 8, 12), 8, 8)
        tr_layer.set_tr_tracking(big, False)
        cases.append((f"{cell} H above the bound", big))
    n0 = _lib.launch_count()
    for what, m in cases:
        with pytest.raises((RuntimeError, NotImplementedError)):
            fused.FusedRNN(m)
            pytest.fail(what)
    with pytest.raises(NotImplementedError, match="FusedLSTM"):
        fused.FusedRNN(cases[2][1])
    assert _lib.launch_count() == n0
    # stale weights, a model switched back to training, re-calibration after fusing
    q, tokens, targets, hidden = _lm("GRU", **small)
    f = fused.FusedRNN(q)
    with torch.no_grad():
        f(tokens, hidden)
        q.rnn.weight_hh_l1.mul_(1.0)
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f(tokens, hidden)
    assert _lib.launch_count() == n0
    f = fused.FusedRNN(q)
    n0 = _lib.launch_count()
    with pytest.raises(ValueError, match="int64 targets"):
        f.nll(tokens, targets[:-1], hidden)
    f.train()
    with pytest.raises(RuntimeError, match="inference only"):
        f.nll(tokens, targets, hidden)
    f.eval()
    sf = q.decoder.input_quant.sf
    tr_layer.set_tr_tracking(q, True)
    with pytest.raises(RuntimeError, match="tracking"):
        f(tokens, hidden)
    assert _lib.launch_count() == n0
    q.decoder.input_quant.hist_bins.zero_()
    q.decoder.input_quant(torch.randn(100000, device="cuda") * 5)          # a histogram of much wider activations
    tr_layer.set_tr_tracking(q, False)
    assert q.decoder.input_quant.sf != sf
    n0 = _lib.launch_count()
    with pytest.raises(RuntimeError, match="changed after fusing"):
        f.nll(tokens, targets, hidden)
    assert _lib.launch_count() == n0
