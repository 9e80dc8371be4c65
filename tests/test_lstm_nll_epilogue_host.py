"""CPU checks of the decoder's loss-epilogue interface (conv_codes.linear_codes_nll): the refusals that need no device,
all raised before the library is reached."""
import pytest
import torch


@pytest.fixture
def no_library(monkeypatch):
    """Any call into libtq_b200 fails the test: every case below must be refused before it."""
    from term_quantization_b200 import _lib

    def reached():
        pytest.fail("linear_codes_nll reached the library")
    monkeypatch.setattr(_lib, "lib", reached)


def _ops(M=4, K=16, Op=12):
    return (torch.zeros(M, K, dtype=torch.float16), torch.zeros(1, Op, K, dtype=torch.float16),
            torch.zeros(M, dtype=torch.int64))


def _call(x, w, t, **kw):
    from term_quantization_b200 import conv_codes
    return conv_codes.linear_codes_nll(x, w, 0.5, t, **kw)


def test_refuses_wrong_dtypes(no_library):
    x, w, t = _ops()
    for a, b, c in ((x.float(), w, t), (x, w.float(), t), (x, w, t.int()), (x, w, t.float()), (x.to(torch.int8), w, t)):
        with pytest.raises(RuntimeError, match="fp16 codes and weights and int64 targets"):
            _call(a, b, c)


def test_refuses_bad_shapes(no_library):
    x, w, t = _ops()
    cases = [
        (x[0], w, t, {}),                                     # codes not 2-D
        (x, w[0], t, {}),                                     # weight not [1, Op, Kp]
        (x, torch.zeros(2, 12, 16, dtype=torch.float16), t, {}),
        (x, w, t[:3], {}),                                    # target length
        (x, w, t.view(4, 1), {}),
        (torch.zeros(0, 16, dtype=torch.float16), w, t[:0], {}),   # no rows
        (torch.zeros(4, 32, dtype=torch.float16), w, t, {}),  # K > Kp
        (x, w, t, {"out_features": 0}),                       # V < 1
        (x, w, t, {"out_features": 13}),                      # V > Op
        (x, w, torch.zeros(8, dtype=torch.int64)[::2], {}),   # non-contiguous targets
        (x, w, t, {"bias": torch.zeros(12, dtype=torch.float64)}),
        (x, w, t, {"bias": torch.zeros(7)}),                  # neither out_features nor Op entries
        (x, w, t, {"bias": torch.zeros(3, 4)}),
    ]
    for a, b, c, kw in cases:
        with pytest.raises(ValueError):
            _call(a, b, c, **kw)


def test_refuses_host_tensors(no_library):
    x, w, t = _ops()
    with pytest.raises(RuntimeError, match="CUDA"):
        _call(x, w, t)
    with pytest.raises(RuntimeError, match="CUDA"):
        _call(x, w, t, bias=torch.zeros(10), out_features=10)
