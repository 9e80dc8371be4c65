"""Term-pair multiplication counters for the TR layers (mirror of profile_model.py:8-64).

ops of a TR conv / linear = data_terms' * (alpha' / g) * MACs with data_terms' =
min(data_terms, data_bits) and alpha' = min(alpha, weight_bits) when g == 1; convs are counted
only for C_in > 3 and groups == 1 (profile_model.py:25); linear layers also count parameter
bits -- numel * bits for g == 1, else the compressed size in the layer's term encoding (device popcount reduction
instead of the reference's per-element Python loop, tr_layer.py:57-63).  Counts land in the
wrapped child's float32 buffer like the reference."""
import torch
import torch.nn as nn

from . import thop, tr_layer

try:
    from efficientnet_pytorch.utils import Conv2dStaticSamePadding
except ImportError:  # not in this image
    Conv2dStaticSamePadding = None


def _term_pairs(m, macs):
    weight_terms = min(m.num_terms, m.weight_bits) if m.group_size == 1 else m.num_terms
    data_terms = min(m.data_terms, m.data_bits)
    return data_terms * (weight_terms / m.group_size) * macs


def tr_conv2d_ops(m, x, y):
    x = x[0]
    kh, kw = m.conv.weight.shape[2:]
    macs = y.nelement() * (m.conv.in_channels // m.conv.groups * kh * kw)
    if x.shape[1] > 3 and m.conv.groups == 1:
        m.conv.total_ops += torch.Tensor([int(_term_pairs(m, macs))])


def tr_linear_ops(m, x, y):
    macs = y.nelement() * m.linear.in_features
    m.linear.total_ops += torch.Tensor([int(_term_pairs(m, macs))])
    if m.group_size == 1:
        weight_bits = m.linear.weight.nelement() * m.weight_bits
    else:
        weight_bits = tr_layer.compute_compressed_hese(m.linear.weight, m.w_sf, m.weight_bits, encoding=m.encoding)
    m.linear.total_params += torch.Tensor([int(weight_bits)])


def tr_lstm_ops(m, x, y):
    # the reference counts nothing for the LSTM itself (profile_model.py:48-49)
    return None


_ZERO_COUNTED = (nn.Conv2d, nn.BatchNorm2d, nn.Linear, nn.AvgPool2d, nn.AdaptiveAvgPool2d)     # inner / free layers


def get_model_ops(model, inputs):
    """(term-pair multiplications, parameter bits) of one forward of `model` on `inputs`."""
    counters = {layer_type: thop.count_hooks.zero_ops for layer_type in _ZERO_COUNTED}
    if Conv2dStaticSamePadding is not None:
        counters[Conv2dStaticSamePadding] = thop.count_hooks.zero_ops
    counters.update({tr_layer.TRConv2dLayer: tr_conv2d_ops, tr_layer.TRLinearLayer: tr_linear_ops,
                     tr_layer.TRLSTMLayer: tr_lstm_ops})
    return thop.profile(model, inputs=inputs, custom_ops=counters)
