"""CPU checks of the fused LSTM executor's interface: the driver's --engine choices and refusals that need no device."""
import pytest
import torch
import torch.nn as nn


def test_evaluate_lstm_refuses_an_unknown_engine():
    from term_quantization_b200 import evaluate_lstm
    with pytest.raises(SystemExit) as e:
        evaluate_lstm.main(["--wb", "8", "--wt", "12", "--db", "8", "--dt", "8", "--gs", "8", "--engine", "cudnn"])
    assert e.value.code == 2


@pytest.mark.parametrize("kind", ["GRU", "RNN_TANH", "RNN_RELU"])
def test_fused_lstm_refuses_other_recurrences(kind):
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    with pytest.raises(NotImplementedError, match="LSTM"):
        fused.FusedLSTM(RNNModel(kind, 50, 16, 16, 2, 0.0, False).eval())


def test_fused_lstm_refuses_an_unconverted_model():
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    with pytest.raises(NotImplementedError, match="TRLSTMLayer"):
        fused.FusedLSTM(RNNModel("LSTM", 50, 16, 16, 2, 0.0, False).eval())


def test_lstm_recurrence_refuses_host_tensors():
    from term_quantization_b200 import conv_codes
    z = torch.zeros
    with pytest.raises(RuntimeError, match="CUDA"):
        conv_codes.lstm_recurrence(z(2, 3, 16), None, z(16, 4), z(3, 4), z(3, 4))
