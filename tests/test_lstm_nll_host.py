"""CPU checks of the one-pass log-softmax + NLL interface (conv_codes.log_softmax_nll): the refusals that need no device,
all raised before the library is reached."""
import pytest
import torch


@pytest.fixture
def no_library(monkeypatch):
    """Any call into libtq_b200 fails the test: every case below must be refused before it."""
    from term_quantization_b200 import _lib

    def reached():
        pytest.fail("log_softmax_nll reached the library")
    monkeypatch.setattr(_lib, "lib", reached)


def test_refuses_wrong_dtypes(no_library):
    from term_quantization_b200 import conv_codes
    x, t = torch.zeros(4, 10), torch.zeros(4, dtype=torch.int64)
    for logits, targets in ((x.double(), t), (x.half(), t), (x, t.int()), (x, t.float())):
        with pytest.raises(RuntimeError, match="fp32 logits and int64 targets"):
            conv_codes.log_softmax_nll(logits, targets)


def test_refuses_bad_shapes_and_strides(no_library):
    from term_quantization_b200 import conv_codes
    t4 = torch.zeros(4, dtype=torch.int64)
    base = torch.zeros(4, 16)
    cases = [
        (torch.zeros(40), t4),                                # not 2-D
        (torch.zeros(2, 4, 10), t4),
        (torch.zeros(4, 10), torch.zeros(3, dtype=torch.int64)),   # wrong target length
        (torch.zeros(4, 10), torch.zeros(4, 1, dtype=torch.int64)),
        (torch.zeros(4, 0), t4),                              # no columns
        (torch.zeros(0, 10), torch.zeros(0, dtype=torch.int64)),
        (base.t()[:4], t4),                                   # last dimension not contiguous
        (base.as_strided((4, 10), (8, 1)), t4),               # row stride 8 < 10 columns
        (torch.zeros(4, 10), torch.zeros(8, dtype=torch.int64)[::2]),   # non-contiguous targets
    ]
    for logits, targets in cases:
        with pytest.raises(ValueError):
            conv_codes.log_softmax_nll(logits, targets)


def test_refuses_host_tensors(no_library):
    from term_quantization_b200 import conv_codes
    with pytest.raises(RuntimeError, match="CUDA"):
        conv_codes.log_softmax_nll(torch.zeros(4, 10), torch.zeros(4, dtype=torch.int64))
    # a padded row stride is accepted up to the device check
    with pytest.raises(RuntimeError, match="CUDA"):
        conv_codes.log_softmax_nll(torch.zeros(4, 12)[:, :10], torch.zeros(4, dtype=torch.int64))
