"""The recurrence kernel's tensor-memory tier (recurrence_kernel<Cell, true> in tq_lstm.cu): above the hidden size whose
W_hh rows fit in shared memory, part of each CTA's gate rows live in TMEM.  Only the source of each weight changes, so
the tier is pinned bit for bit to the shared-memory path (TQ_RECURRENCE_TMEM_UNITS forces units into TMEM at any H),
held to an fp64 recurrence above the old bound, and run through the executors and the driver at the word-language-model
example's large configuration (emsize = nhid = 1500, tied)."""
import copy
import gc

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

CELLS = ["LSTM", "GRU", "RNN_TANH", "RNN_RELU"]
GATES = {"LSTM": 4, "GRU": 3, "RNN_TANH": 1, "RNN_RELU": 1}
ENV = "TQ_RECURRENCE_TMEM_UNITS"


@pytest.fixture(autouse=True)
def _fp32_math():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _within(a, b, tol=1e-5):
    err = float((a.double() - b.double()).abs().max())
    assert err <= tol * max(float(b.abs().max()), 1.0), err


def _smem_only_bound(cell):
    """Largest H whose gate rows all fit in shared memory next to one hidden row (the bound before the TMEM tier)."""
    props = torch.cuda.get_device_properties(0)
    G, sms, optin = GATES[cell], props.multi_processor_count, props.shared_memory_per_block_optin
    best = 0
    for H in range(1, 8193):
        U = (H + sms - 1) // sms
        rows = G * U * H if G % 4 == 0 else (G * U * H + 3) & ~3
        if (rows + H) * 4 + 2048 <= optin:
            best = H
    return best


def _operands(cell, T, B, H, gen, saturate=False):
    G = GATES[cell]
    s = 1.0 / H ** 0.5
    gin = torch.randn(T, B, G * H, device="cuda", generator=gen) * 0.5
    if saturate:
        gin = torch.sign(gin) * 30.0                         # every gate pre-activation around +-30
    w = (torch.rand(G * H, H, device="cuda", generator=gen) * 2 - 1) * s
    b = (torch.rand(G * H, device="cuda", generator=gen) * 2 - 1) * s
    h0 = torch.randn(B, H, device="cuda", generator=gen) * 0.3
    if cell == "LSTM":
        return gin, b, w, h0, torch.randn(B, H, device="cuda", generator=gen) * 0.3
    return gin, b, w, h0


def _run(cell, *args):
    from term_quantization_b200 import conv_codes
    if cell == "LSTM":
        return conv_codes.lstm_recurrence(*args)
    if cell == "GRU":
        return conv_codes.gru_recurrence(*args)
    return conv_codes.rnn_recurrence(*args, cell.split("_")[1].lower())


def _ref(cell, gin, bias, w, h0, c0=None):
    """fp64 recurrence with torch's formulas and gate orders."""
    W, h, b = w.double(), h0.double(), bias.double()
    c = c0.double() if c0 is not None else None
    ys = []
    for t in range(gin.shape[0]):
        gi, gh = gin[t].double(), h @ W.t() + b
        if cell == "LSTM":
            i, f, g, o = (gi + gh).chunk(4, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
            h = torch.sigmoid(o) * torch.tanh(c)
        elif cell == "GRU":
            ir, iz, i_n = gi.chunk(3, dim=1)
            hr, hz, h_n = gh.chunk(3, dim=1)
            r, z = torch.sigmoid(ir + hr), torch.sigmoid(iz + hz)
            n = torch.tanh(i_n + r * h_n)
            h = (1 - z) * n + z * h
        else:
            h = torch.tanh(gi + gh) if cell == "RNN_TANH" else torch.relu(gi + gh)
        ys.append(h)
    return (torch.stack(ys), h) + ((c,) if cell == "LSTM" else ())


# ---- the tier against shared memory, bit for bit ---------------------------------------------------------------

# 1 / 7 / 33: one unit per CTA; 301: 3 per CTA and a last CTA with one; 650: 5 per CTA; 1024: 7 per CTA, the last with
# 2, and B = 128 stages the hidden rows in several tiles.  1 unit in TMEM: quarter 0 holds one unit, the others stay
# in shared memory; the maximum (clamped to U): every unit in TMEM, quarters with one and two units
BIT_CASES = [(3, 80, 1), (3, 80, 7), (3, 80, 33), (3, 80, 301), (3, 80, 650), (2, 128, 1024)]


@pytest.mark.parametrize("cell", CELLS)
@pytest.mark.parametrize("T,B,H", BIT_CASES)
def test_tmem_units_bit_identical_to_shared_memory(cell, T, B, H, monkeypatch):
    gen = torch.Generator(device="cuda").manual_seed(H * 7 + B)
    args = _operands(cell, T, B, H, gen)
    outs = []
    for n in (0, 1, 1 << 20):
        monkeypatch.setenv(ENV, str(n))
        outs.append(_run(cell, *args))
    for other in outs[1:]:
        for a, b in zip(outs[0], other):
            assert torch.equal(a, b), float((a - b).abs().max())
    _within(outs[0][0], _ref(cell, *args)[0])


# ---- above the old bound, against fp64 -----------------------------------------------------------------------

def _large_sizes(cell):
    from term_quantization_b200 import conv_codes
    hs = {_smem_only_bound(cell) + 1, 1500, conv_codes.recurrence_max_hidden(cell)}
    if cell != "LSTM":
        hs.add(2048)
    return sorted(hs)


@pytest.mark.parametrize("cell", CELLS)
def test_above_old_bound_against_fp64(cell):
    for H in _large_sizes(cell):
        T = 35 if H == 1500 else 4
        gen = torch.Generator(device="cuda").manual_seed(H)
        args = _operands(cell, T, 80, H, gen)
        out = _run(cell, *args)
        ref = _ref(cell, *args)
        assert out[0].shape == (T, 80, H)
        for a, b in zip(out, ref):
            _within(a, b)
        assert torch.equal(out[1], out[0][-1])


@pytest.mark.parametrize("cell", CELLS)
def test_saturating_gates_at_1500(cell):
    gen = torch.Generator(device="cuda").manual_seed(3)
    args = _operands(cell, 35, 80, 1500, gen, saturate=True)
    out = _run(cell, *args)
    ref = _ref(cell, *args)
    if cell == "RNN_RELU":
        assert float(ref[0].abs().max()) > 30
    for a, b in zip(out, ref):
        _within(a, b)


def test_relu_keeps_nan_at_1500():
    gen = torch.Generator(device="cuda").manual_seed(11)
    gin, b, w, h0 = _operands("RNN_RELU", 6, 80, 1500, gen)
    gin[2, 5, 17] = float("nan")
    gin[0, 9, 3] = -float("nan")
    y, hn = _run("RNN_RELU", gin, b, w, h0)
    ry, rh = _ref("RNN_RELU", gin, b, w, h0)
    assert bool(torch.isnan(ry).any()) and not bool(torch.isnan(ry).all())
    assert torch.equal(torch.isnan(y), torch.isnan(ry)) and torch.equal(torch.isnan(hn), torch.isnan(rh))
    ok = ~torch.isnan(ry)
    _within(y[ok], ry[ok])


@pytest.mark.parametrize("cell", CELLS)
def test_graph_replay_equals_eager_at_1500(cell):
    gen = torch.Generator(device="cuda").manual_seed(7)
    args = _operands(cell, 35, 80, 1500, gen)
    eager = _run(cell, *args)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _run(cell, *args)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _run(cell, *args)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, out):
        assert torch.equal(a, b)


def test_tmem_released_for_the_next_tcgen05_kernel():
    """Layer 0, layer 1, then the decoder on the same stream, as FusedLSTM runs them: both tiered launches and the
    tcgen05 GEMM after them allocate TMEM, so each must find it released."""
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(5)
    a0 = _operands("LSTM", 35, 80, 1500, gen)
    a1 = _operands("LSTM", 35, 80, 1500, gen)
    r0 = _run("LSTM", *a0)
    r1 = _run("LSTM", *a1)
    M, K, V = 35 * 80, 1504, 1000
    x = torch.randint(-8, 9, (M, K), device="cuda", generator=gen).half()
    w = torch.randint(-8, 9, (1, V, K), device="cuda", generator=gen).half()
    plan = conv_codes.plan_weight(w, 512, signed_act=True)
    logits = conv_codes.linear_codes(x, w, 0.5, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(logits, (x.double() @ w[0].double().t()).float() * 0.5)
    for out, args in ((r0, a0), (r1, a1)):
        for a, b in zip(out, _ref("LSTM", *args)):
            _within(a, b)


# ---- executors and the driver at 1500 / 2048 -------------------------------------------------------------------

def _lm(kind, H, T=35, B=80, seed=0):
    from term_quantization_b200 import evaluate_lstm, tr_layer
    from term_quantization_b200.lstm_models.model import RNNModel
    torch.manual_seed(seed)
    base = RNNModel(kind, evaluate_lstm.NTOKENS, H, H, 2, 0.5, True).cuda().eval()
    base.decoder.bias.data.uniform_(-0.1, 0.1)
    q = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    tokens = torch.randint(evaluate_lstm.NTOKENS, (T, B), device="cuda", generator=g)
    targets = torch.randint(evaluate_lstm.NTOKENS, (T * B,), device="cuda", generator=g)
    hidden = torch.randn(2, B, H, device="cuda", generator=g) * 0.3
    if kind == "LSTM":
        hidden = (hidden, torch.randn(2, B, H, device="cuda", generator=g) * 0.3)
    with torch.no_grad():
        q(tokens, hidden)
        tr_layer.set_tr_tracking(q, False)
    return q, tokens, targets, hidden


@pytest.mark.parametrize("kind,H", [("LSTM", 1500), ("GRU", 2048)])
def test_executor_forward_and_nll(kind, H):
    from term_quantization_b200 import fused, tr_layer
    q, tokens, targets, hidden = _lm(kind, H)
    q_tc = copy.deepcopy(q)
    tr_layer.use_tensor_cores(q_tc)
    f = (fused.FusedLSTM if kind == "LSTM" else fused.FusedRNN)(copy.deepcopy(q))
    seen = {}
    hook = q_tc.decoder.register_forward_hook(lambda m, i, o: seen.update(x=i[0]))
    cap = {}
    with torch.no_grad():
        out_tc, h_tc = q_tc(tokens, hidden)
        out_f, h_f = f(tokens, hidden, capture=cap)
    hook.remove()
    assert out_f.shape == out_tc.shape == (35 * 80, q.ntoken)
    for a, b in zip(h_f if kind == "LSTM" else (h_f,), h_tc if kind == "LSTM" else (h_tc,)):
        _within(a, b)
    _within(cap["y"], seen["x"])
    # the decoder is exact on the codes it was given
    dec = f.model.decoder
    wsf = np.float32(dec.w_sf)
    wc = torch.round(dec.linear.weight / wsf)
    acc = cap["codes"].double() @ wc.double().t()
    scale = float(np.float32(dec.input_quant.sf) * wsf)
    assert torch.equal(cap["decoded"], acc.float() * scale + dec.linear.bias)
    assert float((out_f - out_tc).abs().mean()) < 1e-3

    V = q.ntoken
    with torch.no_grad():
        loss, hn = f.nll(tokens, targets, hidden)
        _within(loss, F.nll_loss(out_f, targets, reduction="none"), tol=4e-6)
        for a, b in zip(hn if kind == "LSTM" else (hn,), h_f if kind == "LSTM" else (h_f,)):
            assert torch.equal(a, b)
        del out_f, out_tc, cap, seen
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = f.nll(tokens, targets, hidden)
        torch.cuda.synchronize()
        rise = torch.cuda.max_memory_allocated() - base
        del out
    # no [T*B, V] tensor, not even in fp16: what rises is the step's own buffers (at 1500 the LSTM's gin [T*B, 4H] fp32
    # alone is 67 MB)
    assert rise < 35 * 80 * V * 2 * 0.75, rise


def test_driver_fused_engine_matches_tcgen05_at_1500():
    from term_quantization_b200 import evaluate_lstm
    args = ["--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--emsize", "1500", "--nhid", "1500",
            "--tokens", "3000"]
    tc = evaluate_lstm.main(args + ["--engine", "tcgen05"])
    fu = evaluate_lstm.main(args + ["--engine", "fused"])
    assert abs(fu["ppls"][0] - tc["ppls"][0]) <= 1e-4 * tc["ppls"][0], (fu["ppls"], tc["ppls"])
    assert fu["tmacs"] == tc["tmacs"] and fu["param_bits"] == tc["param_bits"]


# ---- refusals ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cell", CELLS)
def test_refusal_above_the_new_bound(cell):
    from term_quantization_b200 import _lib, conv_codes
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(1 << 20, device="cuda")
    p = buf.data_ptr()
    hmax = conv_codes.recurrence_max_hidden(cell)
    assert hmax > _smem_only_bound(cell)
    n0 = _lib.launch_count()
    for H in (hmax + 1, hmax + 100, 2 * hmax):
        if cell == "LSTM":
            rc = L.tq_lstm_recurrence(p, None, p, p, p, p, p, p, 1, 1, H, s)
        elif cell == "GRU":
            rc = L.tq_gru_recurrence(p, None, p, p, p, p, 1, 1, H, s)
        else:
            rc = L.tq_rnn_recurrence(p, None, p, p, p, p, 1, 1, H, int(cell == "RNN_RELU"), s)
        assert rc == _lib.TQ_ERR_UNSUPPORTED, H
        assert f"largest H on this device: {hmax}" in L.tq_last_error().decode()
    with pytest.raises(NotImplementedError, match=f"largest H on this device: {hmax}"):
        _run(cell, *_operands(cell, 1, 1, hmax + 1, torch.Generator(device="cuda").manual_seed(0)))
    assert _lib.launch_count() == n0
    for H in (hmax - 1, hmax):
        gen = torch.Generator(device="cuda").manual_seed(H)
        args = _operands(cell, 2, 2, H, gen)
        for a, b in zip(_run(cell, *args), _ref(cell, *args)):
            _within(a, b)
