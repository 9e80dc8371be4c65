"""Binary and Booth term encodings above the raw op: the facts the fused engines rely on, checked exhaustively on the
oracle, and the Python surface (layers, model conversion, drivers) refusing what it cannot run.

The CPU emulation of an encoding-aware chain is defined here on top of oracle.tr (which takes the encoding):
`emul_encode` is oracle/fused_emul.encode for a quantiser (sf, bits, terms) -- HESE -- or (sf, bits, terms, encoding),
the `next_quant` form of term_quantization_b200.conv_codes.  tests/test_encodings_gpu.py installs it in fused_emul so
that the chain emulations there follow each layer's encoding.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import tq_oracle as O

ENC_IDS = {"hese": O.ENC_HESE, "binary": O.ENC_BINARY, "booth": O.ENC_BOOTH}


def emul_encode(x_nhwc, quant):
    """fp32 array -> int32 term codes under quant = (sf, bits, terms[, encoding]), g = 1."""
    sf, bits, terms = quant[:3]
    enc = ENC_IDS[quant[3]] if len(quant) == 4 else O.ENC_HESE
    x = np.ascontiguousarray(x_nhwc, dtype=np.float32)
    _, codes = O.tr(x.reshape(1, -1, 1, 1), sf, bits, 1, terms, encoding=enc, return_codes=True)
    return codes.reshape(x.shape)


def emul_mse_profile(hist_bins, x, sfs, bits, terms, encoding):
    """tq_mse_profile_enc on the CPU: errs[s] = sum_b hist[b] * (x[b] - tr(x[b]; sfs[s]))^2 with every elementwise op
    rounded to fp32 and the sum in fp64; returns (first index of the minimum of fp32(errs), errs)."""
    hist_bins = np.asarray(hist_bins, dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    errs = np.empty(len(sfs), dtype=np.float64)
    for s, sf in enumerate(np.asarray(sfs, dtype=np.float32)):
        xh = O.tr(x.reshape(1, -1, 1, 1), float(sf), bits, 1, terms, encoding=ENC_IDS[encoding]).reshape(-1)
        d = (x - xh).astype(np.float32)
        errs[s] = np.sum((hist_bins * (d * d).astype(np.float32)).astype(np.float32), dtype=np.float64)
    return int(np.argmin(errs.astype(np.float32))), errs


def emul_term_count(w, sf, encoding):
    """tq_term_count with TQ_FLAG_RECIP_DIV: sum over w of the number of terms of int(w * fl32(1 / sf))."""
    w = np.ascontiguousarray(w, dtype=np.float32).ravel()
    inv = np.float32(1.0) / np.float32(sf)
    ints = np.trunc((w * inv).astype(np.float32)).astype(np.int64)
    total = 0
    for v in ints.tolist():
        p, n = O.terms(abs(v), ENC_IDS[encoding])
        total += bin(p).count("1") + bin(n).count("1")
    return total


@pytest.mark.parametrize("encoding", list(ENC_IDS))
def test_truncated_code_is_bounded_and_monotone(encoding):
    """For every bit width 1..11 and term budget 0..bits+2 the truncated code of q = 0 .. 2^bits - 1 is non-decreasing
    in q (max-pooling codes == encoding the pooled value) and |code| <= 2^bits (binary: 2^bits - 1), the bound the
    fp16 code stores, the i8 planes and the accumulator proofs assume."""
    for bits in range(1, 12):
        q = np.arange(2 ** bits, dtype=np.float32)
        top = 2 ** bits - (encoding == "binary")
        for terms in range(bits + 3):
            codes = emul_encode(q, (1.0, bits, terms, encoding))
            assert np.all(np.diff(codes) >= 0), (encoding, bits, terms, np.flatnonzero(np.diff(codes) < 0)[:4])
            assert codes.min() >= 0 and codes.max() <= top, (encoding, bits, terms, codes.max())
            neg = emul_encode(-q, (1.0, bits, terms, encoding))
            assert np.array_equal(neg, -codes)


def test_encodings_differ_where_the_tests_need_them_to():
    """Booth codes can exceed HESE's (q = 2^(bits-1) is +2^bits - 2^(bits-1); one term keeps 2^bits), and binary keeps
    fewer high bits than HESE under a binding budget: a GPU test that compares against these codes can tell them apart."""
    q = np.arange(2 ** 9, dtype=np.float32)
    hese = emul_encode(q, (1.0, 9, 1))
    for enc in ("binary", "booth"):
        assert not np.array_equal(emul_encode(q, (1.0, 9, 1, enc)), hese), enc
    assert emul_encode(np.float32([256.0]), (1.0, 9, 1, "booth"))[0] == 512
    assert emul_encode(np.float32([256.0]), (1.0, 9, 1))[0] == 256


def test_emul_encode_hese_tuples_agree():
    from oracle import fused_emul
    rng = np.random.default_rng(0)
    x = (rng.standard_normal((2, 5, 7, 16)) * 3).astype(np.float32)
    for bits, terms in ((9, 3), (6, 2), (4, 8)):
        want = fused_emul.encode(x, (0.0371, bits, terms))
        assert np.array_equal(emul_encode(x, (0.0371, bits, terms)), want)
        assert np.array_equal(emul_encode(x, (0.0371, bits, terms, "hese")), want)


def test_unknown_encodings_are_refused():
    from term_quantization_b200 import _lib, cnn_models, conv_codes, evaluate_cnn, evaluate_lstm, evaluate_mlp, tr_layer
    for bad in ("HESE", "csd", "", None, 0, 2):
        with pytest.raises(ValueError, match="unknown term encoding"):
            _lib.encoding_id(bad)
    conv = nn.Conv2d(8, 8, 3)
    with pytest.raises(ValueError):
        tr_layer.LinearQuantize(8, 3, encoding="csd")
    for cls, mod in ((tr_layer.TRConv2dLayer, conv), (tr_layer.TRLinearLayer, nn.Linear(8, 8)),
                     (tr_layer.TRLSTMLayer, nn.LSTM(8, 8))):
        with pytest.raises(ValueError):
            cls(mod, 8, 3, 8, 1, 8, encoding="csd")
    net = nn.Sequential(nn.Conv2d(3, 8, 3), nn.Conv2d(8, 8, 3))
    with pytest.raises(ValueError):
        cnn_models.convert_model(net, [(8, 1, 8)] * 2, 8, 3, encoding="csd")
    with pytest.raises(ValueError):
        tr_layer.mse_profile(torch.zeros(8192), -50, 50, 8, 3, encoding="csd")
    with pytest.raises(ValueError):
        tr_layer.compute_compressed_hese(torch.zeros(4), 1.0, 8, encoding="csd")
    with pytest.raises(ValueError):
        conv_codes._quant_args((0.5, 8, 3, "csd"))
    with pytest.raises(ValueError):
        conv_codes._quant_args((0.5, 8))
    assert conv_codes._quant_args((0.5, 8, 3)) == (0.5, 8, 3, _lib.ENC_HESE)
    assert conv_codes._quant_args((0.5, 8, 3, "booth")) == (0.5, 8, 3, _lib.ENC_BOOTH)
    for main in (evaluate_cnn.main, evaluate_mlp.main, evaluate_lstm.main):
        with pytest.raises(SystemExit) as e:
            main(["--encoding", "csd"])
        assert e.value.code == 2                 # argparse: refused before any device work


@pytest.fixture
def cpu_tr(monkeypatch):
    """tr_cuda.tr replaced by the oracle on CPU tensors, recording the encoding of every call."""
    from term_quantization_b200 import tr_layer
    seen = []

    def tr(x, sf, bits, g, alpha, *, encoding="hese", **_):
        seen.append(encoding)
        return torch.from_numpy(O.tr(x.detach().numpy(), sf, bits, g, alpha, encoding=ENC_IDS[encoding]))
    monkeypatch.setattr(tr_layer.tr_cuda, "tr", tr)
    return seen


def test_convert_model_sets_every_layer_encoding(cpu_tr):
    from term_quantization_b200 import cnn_models, tr_layer
    torch.manual_seed(0)
    net = nn.Sequential(nn.Conv2d(3, 16, 3), nn.ReLU(), nn.Conv2d(16, 16, 3), nn.BatchNorm2d(16),
                        nn.Conv2d(16, 32, 1), nn.Conv2d(32, 32, 3, groups=32))
    params = cnn_models.static_conv_layer_settings(net, 9, 8, 12)
    hese = cnn_models.convert_model(net, params, 9, 3)
    assert set(cpu_tr) == {"hese"}
    cpu_tr.clear()
    booth = cnn_models.convert_model(net, params, 9, 3, encoding="booth")
    assert set(cpu_tr) == {"booth"} and len(cpu_tr) == 3
    layers = [m for m in booth.modules() if isinstance(m, tr_layer.TRConv2dLayer)]
    assert len(layers) == 3
    assert all(m.encoding == "booth" and m.input_quant.encoding == "booth" for m in layers)
    assert all(m.encoding == "hese" for m in hese.modules() if isinstance(m, tr_layer.TRConv2dLayer))
    assert list(booth.state_dict()) == list(hese.state_dict())
    # the weights are revealed in the layer's encoding (Booth and HESE differ on this random weight)
    w_b, w_h = booth[2].conv.weight.detach(), hese[2].conv.weight.detach()
    sf = booth[2].w_sf
    want = O.tr(net[2].weight.detach().numpy(), sf, 9, 8, 12, encoding=O.ENC_BOOTH)
    assert np.array_equal(w_b.numpy(), want) and not torch.equal(w_b, w_h)


def test_layer_drivers_pass_the_encoding(cpu_tr):
    from term_quantization_b200 import evaluate_lstm, evaluate_mlp, tr_layer
    from term_quantization_b200.lstm_models.model import RNNModel
    from term_quantization_b200.train_mlp import MNISTMLP
    torch.manual_seed(0)
    mlp = evaluate_mlp.replace_linear_layers(MNISTMLP(), [(8, 8, 12)] * 3, 8, 3, encoding="binary")
    lins = [m for m in mlp.modules() if isinstance(m, tr_layer.TRLinearLayer)]
    assert len(lins) == 3 and all(m.encoding == "binary" == m.input_quant.encoding for m in lins)
    rnn = RNNModel("LSTM", 50, 16, 16, 2, 0.0, False)
    q = evaluate_lstm.convert_model(rnn, evaluate_lstm.static_lstm_layer_settings(rnn, 8, 8, 12), 8, 3, encoding="booth")
    wrapped = [m for m in q.modules() if isinstance(m, (tr_layer.TRLSTMLayer, tr_layer.TRLinearLayer))]
    assert len(wrapped) == 2 and all(m.encoding == "booth" for m in wrapped)
    assert set(cpu_tr) == {"binary", "booth"}
