"""The decoder's loss epilogue (tq_linear_codes_nll / tq_linear_planes_i8_nll, conv_codes.linear_codes_nll) and
FusedLSTM.nll built on it, on the GPU.

Numerics contract: loss[r] = logsumexp(x[r, :V]) - x[r, t[r]] over the fp32 logits x that linear_codes writes for the
same operands, held to an fp64 logsumexp - gather of those logits at 4e-6 * max(|ref|, 1) per row.  First order,
relative to S = sum exp(x - max) (u = 2^-24): each term is ex2.approx (2 ulp, 4u) of fl(fl(x - m) * log2 e), whose two
roundings and the rounding of log2 e move the exponent by at most 3u (M - x) in natural units, M the row maximum; the
rescales of a term on its way to M (chunk maximum -> tile maximum in fp32, then -> M in fp64) add up to the same M - x,
so weighted by each term's share of S they stay below 3u * sum p (M - x) <= 3u ln V (31.2u at V = 33,278); the 32-term
pairwise sum of a chunk (5u); the one fma that rescales and adds the second chunk of a tile (ex2 4u + 2u).  The combine
runs in fp64 (exact differences, ~2^-53 per step) and rounds once.  Together 46u = 2.8e-6 relative in S, i.e. absolute
in log S, plus u * |loss| for the final rounding: below 2.9e-6 * max(|loss|, 1).  Eager calls, side streams and
CUDA-graph replays are bit-identical."""
import gc

import pytest
import torch

pytestmark = pytest.mark.gpu

BOUND = 4e-6
ACT_MAX = 512


@pytest.fixture(autouse=True)
def _fp32_math():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _ref(x, t):
    xd = x.double()
    return torch.logsumexp(xd, 1) - xd.gather(1, t[:, None])[:, 0]


def _within(got, ref):
    err = (got.double() - ref).abs()
    lim = BOUND * ref.abs().clamp(min=1.0)
    bad = ~(err <= lim)
    assert not bool(bad.any()), (int(bad.sum()), float((err / lim).max()))


_WEIGHTS = {}


def _operands(M, V, K, with_bias, extra_pad):
    """Codes [M, K] in [-300, 300] (act_max 512, two s8 planes on the i8 engine), a packed weight [1, Op, Kp] with codes
    in [-20, 20] whose pad rows [V, Op) hold large non-zero codes, and a bias whose pad entries are large too: a pad
    column that leaked into a loss would dominate it.  Op = V rounded up to 4, plus 4 more rows when extra_pad."""
    key = (V, K, with_bias, extra_pad)
    if key not in _WEIGHTS:
        g = torch.Generator(device="cuda").manual_seed(V * 7919 + K)
        Op = (V + 3) // 4 * 4 + (4 if extra_pad else 0)
        Kp = (K + 15) // 16 * 16
        w = torch.randint(-20, 21, (1, Op, Kp), device="cuda", generator=g).half()
        w[:, :, K:] = 0
        w[:, V:, :K] = 20
        b = None
        if with_bias:
            b = torch.rand(Op, device="cuda", generator=g) * 2 - 1
            b[V:] = 100.0
        _WEIGHTS.clear()
        _WEIGHTS[key] = (w, b)
    w, b = _WEIGHTS[key]
    g = torch.Generator(device="cuda").manual_seed(M * 31 + V + K)
    x = torch.randint(-300, 301, (M, K), device="cuda", generator=g).half()
    scale = 8.0 / (300 * 20 * K ** 0.5)                        # logits of a few units, the largest tens
    return x, w, b, scale


def _targets(M, V, gen):
    """0, V - 1, then both sides of every 32-column chunk boundary below V (N tiles of 64 / 128 / 256 columns and their
    column slices), cycling over the rows; random where the list has run out."""
    bnd = torch.tensor([0, V - 1] + [c for k in range(32, V, 32) for c in (k - 1, k)], device="cuda")
    t = torch.randint(V, (M,), device="cuda", generator=gen)
    n = min(M, 2 * bnd.numel())
    t[:n] = bnd[torch.arange(n, device="cuda") % bnd.numel()]
    return t


def _plan(w, engine, groups=None):
    from term_quantization_b200 import conv_codes
    if groups is not None:                                   # K chunks forced (the codes are small enough for any)
        return conv_codes.WeightPlan("f16", groups, 0.0, ACT_MAX, True, w)
    return conv_codes.plan_weight(w, ACT_MAX, signed_act=True, engine=engine)


def _check(M, V, K, with_bias, engine, extra_pad, groups=None):
    from term_quantization_b200 import conv_codes
    x, w, b, scale = _operands(M, V, K, with_bias, extra_pad)
    plan = _plan(w, engine, groups)
    assert plan.engine == engine
    gen = torch.Generator(device="cuda").manual_seed(M + 3 * V)
    t = _targets(M, V, gen)
    logits = conv_codes.linear_codes(x, w, scale, bias=b, out_features=V, plan=plan)
    got = conv_codes.linear_codes_nll(x, w, scale, t, bias=b, out_features=V, plan=plan)
    assert got.shape == (M,) and got.dtype == torch.float32
    _within(got, _ref(logits, t))


@pytest.mark.parametrize("engine", ["f16", "i8"])
@pytest.mark.parametrize("with_bias", [False, True])
@pytest.mark.parametrize("K", [16, 656])
@pytest.mark.parametrize("V", [1, 2, 31, 32, 33, 127, 128, 129, 4097, 33278])
@pytest.mark.parametrize("M", [1, 3, 127, 128, 129, 2800])
def test_against_fp64(M, V, K, with_bias, engine):
    _check(M, V, K, with_bias, engine, extra_pad=not with_bias)


@pytest.mark.parametrize("groups", [2, 4])
@pytest.mark.parametrize("V", [33, 129, 4097, 33278])
@pytest.mark.parametrize("M", [3, 2800])
def test_f16_k_chunk_groups(M, V, groups):
    """K = 256: four 64-channel blocks in 2 or 4 accumulator groups (4 x 128 columns fill tensor memory: one accumulator
    stage drained by all four epilogue groups, four column slices per N tile)."""
    if V <= 64 and groups == 4:
        pytest.skip("N = 64 tiles take at most 4 groups of 64 columns in two stages; covered by groups = 2")
    _check(M, V, 256, True, "f16", extra_pad=True, groups=groups)


def test_padding_never_counts():
    """Pad rows of the packed weight and pad entries of the bias that would dominate every row if they leaked."""
    from term_quantization_b200 import conv_codes
    M, V, K = 300, 130, 64
    x, w, b, scale = _operands(M, V, K, True, True)
    w = w.clone()
    w[:, V:, :] = 20
    b = b.clone()
    b[V:] = 1e4
    t = _targets(M, V, torch.Generator(device="cuda").manual_seed(5))
    for engine in ("f16", "i8"):
        plan = _plan(w, engine)
        logits = conv_codes.linear_codes(x, w, scale, bias=b, plan=plan)
        assert float(logits[:, V:].min()) > 1e3
        got = conv_codes.linear_codes_nll(x, w, scale, t, bias=b, out_features=V, plan=plan)
        _within(got, _ref(logits[:, :V], t))


@pytest.mark.parametrize("engine", ["f16", "i8"])
@pytest.mark.parametrize("M,V", [(2800, 33278), (3, 33278), (129, 4097), (7, 33)])
def test_eager_side_stream_and_graph_replay_bit_identical(M, V, engine):
    from term_quantization_b200 import conv_codes
    x, w, b, scale = _operands(M, V, 656, True, False)
    plan = _plan(w, engine)
    x = x.clone()
    t = _targets(M, V, torch.Generator(device="cuda").manual_seed(17))

    def run():
        return conv_codes.linear_codes_nll(x, w, scale, t, bias=b, out_features=V, plan=plan)
    first, second = run(), run()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        on_side = run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(first, second) and torch.equal(first, on_side) and torch.equal(first, out)
    x.copy_(torch.flip(x, (0,)))                              # a replay reads the inputs as they are now
    t.copy_(torch.flip(t, (0,)))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, run())
    if M > 1:
        assert not torch.equal(out, first)


@pytest.mark.parametrize("engine", ["f16", "i8"])
def test_out_of_range_targets_give_nan_in_their_rows(engine):
    from term_quantization_b200 import conv_codes
    M, V = 400, 4097
    x, w, b, scale = _operands(M, V, 656, True, True)
    plan = _plan(w, engine)
    t = _targets(M, V, torch.Generator(device="cuda").manual_seed(23))
    bad = t.clone()
    rows = [0, 5, 127, 128, 399]
    for i, r in enumerate(rows):
        bad[r] = [-1, V, V + 3, -(1 << 40), 1 << 40][i]        # V .. Op - 1 are pad columns: no logit either
    got = conv_codes.linear_codes_nll(x, w, scale, bad, bias=b, out_features=V, plan=plan)
    nan = torch.zeros(M, dtype=torch.bool, device="cuda")
    nan[rows] = True
    assert torch.equal(torch.isnan(got), nan)
    logits = conv_codes.linear_codes(x, w, scale, bias=b, out_features=V, plan=plan)
    _within(got[~nan], _ref(logits, t)[~nan])


# ---- refusals ---------------------------------------------------------------------------------------------------

def test_c_entries_refuse_before_any_launch():
    from term_quantization_b200 import _lib
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    M, K, Op, V = 64, 64, 132, 130
    ws = int(L.tq_linear_nll_workspace_bytes(M, Op))
    assert ws > 0
    assert L.tq_linear_nll_workspace_bytes(0, Op) < 0 and L.tq_linear_nll_workspace_bytes(M, 0) < 0
    assert L.tq_linear_nll_workspace_bytes(1 << 40, 1 << 30) < 0
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    n0 = _lib.launch_count()
    big = 1 << 62
    # (x, w, M, K, Op, V, bias, targets, loss, workspace, workspace_bytes)
    good = [p, p, M, K, Op, V, p, p, p, p, ws]
    edits = [
        {0: None}, {1: None}, {7: None}, {8: None}, {9: None},            # NULL operands / targets / loss / workspace
        {0: p + 8}, {1: p + 4}, {6: p + 4}, {7: p + 4}, {8: p + 2}, {9: p + 8},   # misaligned
        {2: 0}, {2: -5}, {5: 0}, {5: -1}, {5: Op + 1},                   # M < 1, V < 1, V > Op
        {10: ws - 1}, {10: 0},                                          # workspace too small
        {2: big}, {2: 1 << 31},                                         # sizes beyond int64 / int rows
    ]
    for e in edits:
        a = list(good)
        for i, v in e.items():
            a[i] = v
        x, w, m, k, op, v, bias, tg, loss, wk, wb = a
        assert L.tq_linear_codes_nll(x, w, m, k, op, v, 1.0, bias, 1, tg, loss, wk, wb, s) == _lib.TQ_ERR_INVALID, e
        assert L.tq_linear_planes_i8_nll(x, w, 2, 1, m, k, op, v, 1.0, bias, 512, 20, tg, loss, wk, wb, s) \
            == _lib.TQ_ERR_INVALID, e
    assert _lib.launch_count() == n0


def test_python_refusals_before_any_launch():
    from term_quantization_b200 import conv_codes, _lib
    x, w, b, scale = _operands(8, 130, 64, True, False)
    t = torch.zeros(8, dtype=torch.int64, device="cuda")
    conv_codes.linear_codes_nll(x, w, scale, t, bias=b, out_features=130)      # plans and module loads
    n0 = _lib.launch_count()
    cases = [
        dict(x_codes=x.float()), dict(wgt=w.float()), dict(targets=t.int()),    # dtypes
        dict(x_codes=x[0]), dict(targets=t[:7]), dict(targets=t.view(8, 1)), dict(wgt=w[0]),   # shapes
        dict(out_features=0), dict(out_features=133), dict(x_codes=torch.zeros(0, 64, dtype=torch.float16, device="cuda"),
                                                             targets=t[:0]),
        dict(targets=torch.zeros(16, dtype=torch.int64, device="cuda")[::2]),  # non-contiguous targets
        dict(bias=b.double()), dict(bias=b[:100]),
        dict(x_codes=x.cpu()), dict(targets=t.cpu()), dict(bias=b.cpu()),     # host tensors
    ]
    for c in cases:
        kw = dict(x_codes=x, wgt=w, scale=scale, targets=t, bias=b, out_features=130)
        kw.update(c)
        with pytest.raises((RuntimeError, ValueError)):
            conv_codes.linear_codes_nll(kw.pop("x_codes"), kw.pop("wgt"), kw.pop("scale"), kw.pop("targets"), **kw)
    assert _lib.launch_count() == n0


# ---- the executor ---------------------------------------------------------------------------------------------

def _lm(enc="hese", H=650, layers=2, ntoken=None, seed=0, T=35, B=80):
    from term_quantization_b200 import evaluate_lstm, tr_layer
    from term_quantization_b200.lstm_models.model import RNNModel
    ntoken = ntoken or evaluate_lstm.NTOKENS
    torch.manual_seed(seed)
    base = RNNModel("LSTM", ntoken, H, H, layers, 0.5, True).cuda().eval()
    base.decoder.bias.data.uniform_(-0.1, 0.1)
    q = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8, encoding=enc)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    tokens = torch.randint(ntoken, (T, B), device="cuda", generator=g)
    targets = torch.randint(ntoken, (T * B,), device="cuda", generator=g)
    hidden = tuple(torch.randn(layers, B, H, device="cuda", generator=g) * 0.3 for _ in range(2))
    with torch.no_grad():
        q(tokens, hidden)
        tr_layer.set_tr_tracking(q, False)
    return q, tokens, targets, hidden


@pytest.mark.parametrize("enc", ["hese", "binary", "booth"])
def test_executor_nll_against_fp64_of_forward(enc):
    from term_quantization_b200 import fused
    q, tokens, targets, hidden = _lm(enc)
    f = fused.FusedLSTM(q)
    g = torch.Generator(device="cuda").manual_seed(3)
    chunks = [(tokens, targets), (torch.randint(q.ntoken, tokens.shape, device="cuda", generator=g),
                                  torch.randint(q.ntoken, targets.shape, device="cuda", generator=g))]
    hf = hn = hidden
    with torch.no_grad():
        for x, t in chunks:                                   # the hidden state carried across two bptt chunks
            cap = {}
            _, hf = f(x, hf, capture=cap)
            loss, hn = f.nll(x, t, hn)
            assert loss.shape == (35 * 80,) and loss.dtype == torch.float32
            _within(loss, _ref(cap["decoded"], t))
            assert torch.equal(hn[0], hf[0]) and torch.equal(hn[1], hf[1])


def test_executor_graph_replay_equals_eager():
    from term_quantization_b200 import evaluate_lstm, fused
    q, tokens, targets, hidden = _lm("hese")
    f = fused.FusedLSTM(q)
    g = torch.Generator(device="cuda").manual_seed(99)
    tok, tgt = tokens.clone(), targets.clone()
    hid = tuple(h.clone() for h in hidden)
    with torch.no_grad():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                f.nll(tok, tgt, hid)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss, (h, c) = f.nll(tok, tgt, hid)
        for _ in range(2):
            tok.copy_(torch.randint(evaluate_lstm.NTOKENS, tok.shape, device="cuda", generator=g))
            tgt.copy_(torch.randint(evaluate_lstm.NTOKENS, tgt.shape, device="cuda", generator=g))
            for t in hid:
                t.copy_(torch.randn(t.shape, device="cuda", generator=g) * 0.3)
            graph.replay()
            got = (loss.clone(), h.clone(), c.clone())
            want_loss, (want_h, want_c) = f.nll(tok, tgt, hid)
            for a, b in zip(got, (want_loss, want_h, want_c)):
                assert torch.equal(a, b), float((a - b).abs().max())


def test_executor_peak_memory_below_an_eighth_of_the_logits():
    from term_quantization_b200 import fused
    T, B = 35, 80
    q, tokens, targets, hidden = _lm("hese", T=T, B=B)
    f = fused.FusedLSTM(q)
    V = q.ntoken
    assert V == 33278
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
