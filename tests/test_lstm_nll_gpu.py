"""The one-pass log-softmax + NLL kernel (tq_log_softmax_nll) and FusedLSTM.nll built on it, on the GPU.

Numerics contract: loss[r] = logsumexp(x[r]) - x[r, t[r]] in fp32 with accurate expf / logf and one fixed summation order.
It is held to an fp64 logsumexp - gather of the same logits at 4e-6 * max(|ref|, 1) per row.  First order, relative to
S = sum exp(x - max) (u = 2^-24): expf's 2 ulp per term (4u); the rounding of x - max (at most u * ln(cols) in the
softmax-weighted mean, 10.4u at 33,278 columns); a 16-term pairwise sum (4u); per later step of a thread one fma that
rescales and adds (5u, at most 5 such steps at these sizes); the rescale to the row maximum (5u) and the block tree (9u):
57.4u = 3.4e-6.  logf (1 ulp) and the two final roundings add at most 4u * loss, so the error stays below
3.7e-6 * max(loss, 1).  Eager calls and CUDA-graph replays are bit-identical."""
import gc

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ENCS = ["hese", "binary", "booth"]
BOUND = 4e-6


@pytest.fixture(autouse=True)
def _fp32_math():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _ref(x, t):
    """fp64 logsumexp - gather (targets in range)."""
    xd = x.double()
    return torch.logsumexp(xd, 1) - xd.gather(1, t[:, None])[:, 0]


def _within(got, ref):
    err = (got.double() - ref).abs()
    lim = BOUND * ref.abs().clamp(min=1.0)
    bad = ~(err <= lim)
    assert not bool(bad.any()), (int(bad.sum()), float((err / lim).max()))


SCALES = [1e-3, 0.1, 1.0, 10.0, 80.0]


def _logits(rows, cols, layout, gen):
    """fp32 [rows, cols] with uniform values in [-scale, scale], the scale cycling over SCALES by row; layout 'dense'
    (ld = cols), 'padded' (ld = cols rounded up to 4 as in linear_codes' output, or cols + 4; the pad holds NaN, which
    must never be read) or 'shifted' (the first row starts one float past a 16-byte boundary and ld = cols + 1, so rows
    start at every alignment)."""
    ld = {"dense": cols, "padded": (cols + 3) // 4 * 4 if cols % 4 else cols + 4, "shifted": cols + 1}[layout]
    off = 1 if layout == "shifted" else 0
    buf = torch.full((rows * ld + off,), float("nan"), device="cuda")
    x = buf[off:].view(rows, ld)[:, :cols]
    scale = torch.tensor([SCALES[(r + cols) % len(SCALES)] for r in range(rows)], device="cuda")
    x.copy_((torch.rand(rows, cols, device="cuda", generator=gen) * 2 - 1) * scale[:, None])
    return x


def _targets(rows, cols, gen):
    t = torch.randint(cols, (rows,), device="cuda", generator=gen)
    t[0] = 0
    t[-1] = cols - 1
    return t


@pytest.mark.parametrize("layout", ["dense", "padded", "shifted"])
@pytest.mark.parametrize("cols", [1, 2, 31, 32, 33, 4097, 33278])
@pytest.mark.parametrize("rows", [1, 3, 2800])
def test_kernel_against_fp64(rows, cols, layout):
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(rows * 100003 + cols)
    x = _logits(rows, cols, layout, gen)
    t = _targets(rows, cols, gen)
    if layout == "padded" and cols == 33278:
        assert x.stride(0) == 33280                            # linear_codes' real Op for the 33,278-word decoder
    got = conv_codes.log_softmax_nll(x, t)
    assert got.shape == (rows,) and got.dtype == torch.float32
    _within(got, _ref(x, t))


@pytest.mark.parametrize("cols", [1, 2, 33, 4097, 33278])
def test_constant_rows(cols):
    from term_quantization_b200 import conv_codes
    vals = torch.tensor([-80.0, -1e-3, 0.0, 3.5, 80.0], device="cuda")
    x = vals[:, None].expand(-1, cols).contiguous()
    for t in (torch.zeros(5, dtype=torch.int64, device="cuda"), torch.full((5,), cols - 1, device="cuda")):
        got = conv_codes.log_softmax_nll(x, t)
        _within(got, _ref(x, t))
        _within(got, torch.full((5,), float(torch.tensor(float(cols)).double().log()), device="cuda").double())


@pytest.mark.parametrize("rows,cols", [(3, 33), (3, 33278), (600, 4097), (600, 33278)])
def test_special_values_follow_torch(rows, cols):
    """NaN, +-inf, an all -inf row and out-of-range targets against log_softmax + nll_loss.  (rows, cols) = (3, 33278)
    splits each row over a cluster of CTAs, the others give each row one CTA."""
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(rows + cols)
    x = torch.randn(rows, cols, device="cuda", generator=gen) * 3
    t = torch.randint(cols, (rows,), device="cuda", generator=gen)
    last = cols - 1
    # row 0: a NaN; row 1: +inf; row 2: some -inf entries (one at the target), finite elsewhere
    x[0, cols // 2] = float("nan")
    x[1, last] = float("inf")
    x[2, ::3] = float("-inf")
    t[2] = 0
    if rows > 3:
        x[3, :] = float("-inf")                               # all -inf
        x[4, 1::2] = float("-inf")                            # -inf next to finite values, target finite
        t[4] = 0
        x[5, 0] = float("nan")
        x[5, 1] = float("inf")
        x[6, :] = float("-inf")
        x[6, last] = 2.0                                      # one finite entry: the loss is 0 or +inf
        t[6] = last
        x[7, :] = x[6, :]
        t[7] = 0
    valid = torch.ones(rows, dtype=torch.bool, device="cuda")
    bad_t = t.clone()
    if rows > 9:
        bad_t[8], bad_t[9] = -1, cols                          # out of range
        valid[8:10] = False
    got = conv_codes.log_softmax_nll(x, bad_t)
    want = F.nll_loss(torch.log_softmax(x, 1), t, reduction="none")
    want[~valid] = float("nan")
    assert torch.equal(torch.isnan(got), torch.isnan(want)), (torch.isnan(got).nonzero(), torch.isnan(want).nonzero())
    inf = torch.isinf(want)
    assert torch.equal(torch.isinf(got), inf) and torch.equal(got[inf], want[inf])
    fin = torch.isfinite(want)
    assert bool(fin.sum() >= rows - 10)
    with torch.no_grad():
        xd = x.double()
        ref = torch.logsumexp(xd, 1) - xd.gather(1, t[:, None])[:, 0]
    _within(got[fin], ref[fin])


@pytest.mark.parametrize("rows,cols,ld", [(2800, 33278, 33280), (3, 33278, 33278), (1, 4097, 4097), (7, 33, 35)])
def test_eager_and_graph_replay_bit_identical(rows, cols, ld):
    from term_quantization_b200 import conv_codes
    gen = torch.Generator(device="cuda").manual_seed(11)
    x = (torch.randn(rows, ld, device="cuda", generator=gen) * 5)[:, :cols]
    t = torch.randint(cols, (rows,), device="cuda", generator=gen)
    first = conv_codes.log_softmax_nll(x, t)
    second = conv_codes.log_softmax_nll(x, t)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        conv_codes.log_softmax_nll(x, t)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = conv_codes.log_softmax_nll(x, t)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(first, second) and torch.equal(first, out)
    x.mul_(0.5)                                               # a replay reads the inputs as they are now
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, conv_codes.log_softmax_nll(x, t))


# ---- the executor ---------------------------------------------------------------------------------------------

def _lm(enc="hese", H=650, layers=2, ntoken=None, seed=0, T=35, B=80):
    """A calibrated TQ RNNModel (wb 8, g 8, alpha 12, db 8, 8 data terms) with a non-zero decoder bias, its calibration
    tokens, next-token targets and a random hidden state."""
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


@pytest.mark.parametrize("enc", ENCS)
def test_nll_against_forward(enc):
    from term_quantization_b200 import fused
    q, tokens, targets, hidden = _lm(enc)
    f = fused.FusedLSTM(q)
    g = torch.Generator(device="cuda").manual_seed(3)
    chunks = [(tokens, targets), (torch.randint(q.ntoken, tokens.shape, device="cuda", generator=g),
                                  torch.randint(q.ntoken, targets.shape, device="cuda", generator=g))]
    hf = hn = hidden
    with torch.no_grad():
        for x, t in chunks:                                   # the hidden state carried across two bptt chunks
            logp, hf = f(x, hf)
            want = F.nll_loss(logp, t, reduction="none")
            loss, hn = f.nll(x, t, hn)
            assert loss.shape == (35 * 80,) and loss.dtype == torch.float32
            _within(loss, want.double())
            assert torch.equal(hn[0], hf[0]) and torch.equal(hn[1], hf[1])


def test_nll_against_fp64_of_the_decoder_output():
    from term_quantization_b200 import fused
    q, tokens, targets, hidden = _lm("hese")
    f = fused.FusedLSTM(q)
    cap = {}
    with torch.no_grad():
        f(tokens, hidden, capture=cap)
        loss, _ = f.nll(tokens, targets, hidden)
    assert cap["decoded"].stride(0) == 33280                  # read in place from the padded decoder output
    _within(loss, _ref(cap["decoded"], targets))


def test_nll_graph_replay_equals_eager():
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
        seen = []
        for _ in range(3):
            tok.copy_(torch.randint(evaluate_lstm.NTOKENS, tok.shape, device="cuda", generator=g))
            tgt.copy_(torch.randint(evaluate_lstm.NTOKENS, tgt.shape, device="cuda", generator=g))
            for t in hid:
                t.copy_(torch.randn(t.shape, device="cuda", generator=g) * 0.3)
            graph.replay()
            got = (loss.clone(), h.clone(), c.clone())
            want_loss, (want_h, want_c) = f.nll(tok, tgt, hid)
            for a, b in zip(got, (want_loss, want_h, want_c)):
                assert torch.equal(a, b), float((a - b).abs().max())
            seen.append(got)
    assert all(not torch.equal(seen[i][0], seen[j][0]) for i in range(3) for j in range(i))


def test_nll_allocates_no_vocabulary_wide_tensor():
    from term_quantization_b200 import fused
    T, B = 35, 80
    q, tokens, targets, hidden = _lm("hese", T=T, B=B)
    f = fused.FusedLSTM(q)
    V = q.ntoken

    def with_log_probs():
        return F.nll_loss(f(tokens, hidden)[0], targets, reduction="none")

    def one_pass():
        return f.nll(tokens, targets, hidden)[0]

    def rise(fn):
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fn()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        del out
        return peak

    with torch.no_grad():
        with_log_probs(), one_pass()                            # plans, cuBLAS workspace, module loads
        a, b = rise(with_log_probs), rise(one_pass)
    assert a - b >= T * B * V * 4, (a, b, T * B * V * 4)


def test_driver_fused_engine_scores_with_nll():
    """The perplexity itself is pinned to the tcgen05 engine by test_driver_fused_engine_matches_tcgen05."""
    import math
    from term_quantization_b200 import evaluate_lstm, fused
    args = ["--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--emsize", "64", "--nhid", "64",
            "--tokens", "1500"]
    calls = []
    orig = fused.FusedLSTM.nll

    def counted(self, *a):
        calls.append(1)
        return orig(self, *a)
    fused.FusedLSTM.nll = counted
    try:
        fu = evaluate_lstm.main(args + ["--engine", "fused"])
    finally:
        fused.FusedLSTM.nll = orig
    assert len(calls) == -(-(1500 // 10 - 1) // 35)            # one call per bptt chunk of the scored pass
    assert math.isfinite(fu["ppls"][0])


# ---- refusals ---------------------------------------------------------------------------------------------------

def test_kernel_refuses_before_any_launch():
    from term_quantization_b200 import _lib, conv_codes
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(1 << 16, device="cuda")
    p = buf.data_ptr()
    n0 = _lib.launch_count()
    big = 1 << 62
    bad = [
        (None, 4, 8, 8, p, p),                                # NULL logits
        (p, 4, 8, 8, None, p),                                # NULL targets
        (p, 4, 8, 8, p, None),                                # NULL loss
        (p + 2, 4, 8, 8, p, p),                               # misaligned logits
        (p, 4, 8, 8, p + 4, p),                               # targets not 8-byte aligned
        (p, 4, 8, 8, p, p + 1),                               # misaligned loss
        (p, 0, 8, 8, p, p),                                   # rows < 1
        (p, -3, 8, 8, p, p),
        (p, 4, 0, 8, p, p),                                   # cols < 1
        (p, 4, 8, 7, p, p),                                   # ld < cols
        (p, 4, big, big, p, p),                               # rows * ld overflows int64
        (p, big, 8, 8, p, p),
    ]
    for a in bad:
        assert L.tq_log_softmax_nll(*a, s) == _lib.TQ_ERR_INVALID, a
    assert _lib.launch_count() == n0
    x = torch.zeros(4, 10, device="cuda")
    t = torch.zeros(4, dtype=torch.int64, device="cuda")
    cases = [
        (x.double(), t), (x, t.int()),                        # dtypes
        (x.cpu(), t), (x, t.cpu()), (x.cpu(), t.cpu()),       # host tensors / mismatched devices
        (torch.zeros(64, device="cuda").as_strided((4, 10), (8, 1)), t),   # ld < cols
        (x, t[:3]), (x, torch.zeros(4, 1, dtype=torch.int64, device="cuda")),   # target length
    ]
    if torch.cuda.device_count() > 1:
        cases.append((x, t.to("cuda:1")))
    for logits, targets in cases:
        with pytest.raises((RuntimeError, ValueError)):
            conv_codes.log_softmax_nll(logits, targets)
    assert _lib.launch_count() == n0


def test_executor_nll_refusals():
    from term_quantization_b200 import _lib, fused, tr_layer
    q, tokens, targets, hidden = _lm("hese", H=32, ntoken=100, T=5, B=4)
    f = fused.FusedLSTM(q)
    with torch.no_grad():
        f.nll(tokens, targets, hidden)
        n0 = _lib.launch_count()
        for bad in (targets.int(), targets[:-1], targets.view(5, 4), targets.cpu(), targets.float()):
            with pytest.raises((RuntimeError, ValueError)):
                f.nll(tokens, bad, hidden)
        assert _lib.launch_count() == n0
        f.train()
        with pytest.raises(RuntimeError, match="inference only"):
            f.nll(tokens, targets, hidden)
        f.eval()
        q.rnn.lstm.weight_hh_l0.mul_(1.0)                     # stale weights
        with pytest.raises(RuntimeError, match="changed after fusing"):
            f.nll(tokens, targets, hidden)
        assert _lib.launch_count() == n0
        f = fused.FusedLSTM(q)
        tr_layer.set_tr_tracking(q, True)
        n1 = _lib.launch_count()
        with pytest.raises(RuntimeError, match="tracking"):
            f.nll(tokens, targets, hidden)
        assert _lib.launch_count() == n1
