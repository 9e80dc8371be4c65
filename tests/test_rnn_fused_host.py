"""CPU checks of the fused GRU / vanilla-RNN executor's interface: refusals that need no device."""
import pytest
import torch
import torch.nn as nn


def test_fused_rnn_points_lstm_models_to_fused_lstm():
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    with pytest.raises(NotImplementedError, match="FusedLSTM"):
        fused.FusedRNN(RNNModel("LSTM", 50, 16, 16, 2, 0.0, False).eval())


@pytest.mark.parametrize("kind", ["GRU", "RNN_TANH", "RNN_RELU"])
def test_fused_rnn_refuses_an_unconverted_model(kind):
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    with pytest.raises(NotImplementedError, match="TRLinearLayer"):
        fused.FusedRNN(RNNModel(kind, 50, 16, 16, 2, 0.0, False).eval())


@pytest.mark.parametrize("kw", [{"bidirectional": True}, {"batch_first": True}])
def test_fused_rnn_refuses_bidirectional_and_batch_first(kw):
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    m = RNNModel("GRU", 50, 16, 16, 1, 0.0, False).eval()
    m.rnn = nn.GRU(16, 16, 1, **kw)
    with pytest.raises(NotImplementedError, match="unidirectional"):
        fused.FusedRNN(m)


def test_fused_rnn_refuses_a_cell_that_does_not_match_the_model():
    from term_quantization_b200 import fused
    from term_quantization_b200.lstm_models.model import RNNModel
    m = RNNModel("RNN_RELU", 50, 16, 16, 1, 0.0, False).eval()
    m.rnn = nn.RNN(16, 16, 1, nonlinearity="tanh")
    with pytest.raises(NotImplementedError, match="tanh"):
        fused.FusedRNN(m)
    m.rnn = nn.GRU(16, 16, 1)
    with pytest.raises(NotImplementedError, match="nn.GRU / nn.RNN"):
        fused.FusedRNN(m)


def test_recurrences_refuse_host_tensors_and_unknown_cells():
    from term_quantization_b200 import conv_codes
    z = torch.zeros
    with pytest.raises(RuntimeError, match="CUDA"):
        conv_codes.gru_recurrence(z(2, 3, 12), None, z(12, 4), z(3, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        conv_codes.rnn_recurrence(z(2, 3, 4), None, z(4, 4), z(3, 4), "tanh")
    with pytest.raises(ValueError, match="nonlinearity"):
        conv_codes.rnn_recurrence(z(2, 3, 4), None, z(4, 4), z(3, 4), "sigmoid")
    with pytest.raises(ValueError, match="cell"):
        conv_codes.recurrence_max_hidden("LSTMP")
    assert set(conv_codes.RECURRENCE_GATES) == {"LSTM", "GRU", "RNN_TANH", "RNN_RELU"}
