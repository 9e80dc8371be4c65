"""Model zoo glue and conv-layer replacement (mirror of cnn_models/__init__.py:18-70).

Semantics kept from the reference: the first conv of a network is never wrapped
(cnn_models/__init__.py:34-36); the first conv, grouped/depthwise convs and any conv whose
module name contains 'se' get the "effectively unquantised" setting (16, 1, 16)
(:52-65); per-layer settings are (weight_bits, group_size, weight_terms) tuples.

efficientnet_b0 needs the third-party ``efficientnet_pytorch`` package, which is not in this
image; it is resolved lazily so everything else works without it.
"""
from copy import deepcopy

import torch.nn as nn
from torchvision.models import alexnet, mobilenet_v2, resnet18, vgg16_bn  # noqa: F401
# deeper ResNets beyond the reference's list: BasicBlock resnet34 and the Bottleneck networks (fused.FusedResNet runs all)
from torchvision.models import resnet34, resnet50, resnet101, resnet152, wide_resnet50_2  # noqa: F401

from .. import _lib
from ..tr_layer import TRConv2dLayer

try:  # optional, exactly as optional as in the image
    from efficientnet_pytorch import EfficientNet
    from efficientnet_pytorch.utils import Conv2dStaticSamePadding
    _CONV_TYPES = (nn.Conv2d, Conv2dStaticSamePadding)
except ImportError:  # pragma: no cover
    EfficientNet = None
    _CONV_TYPES = (nn.Conv2d,)


def model_names():
    return ['alexnet', 'vgg16_bn', 'resnet18', 'efficientnet_b0', 'mobilenet_v2']


def resnet_names():
    """The ResNets exported here besides the reference's resnet18 (evaluate_cnn -a takes them too)."""
    return ['resnet34', 'resnet50', 'resnet101', 'resnet152', 'wide_resnet50_2']


def efficientnet_b0(pretrained=True):
    if EfficientNet is None:
        raise ImportError("efficientnet_b0 needs the efficientnet_pytorch package")
    if pretrained:
        return EfficientNet.from_pretrained('efficientnet-b0')
    return EfficientNet.from_name('efficientnet-b0')


def is_conv_layer(layer):
    return isinstance(layer, _CONV_TYPES)


def _conv_layers(model):
    return [(name, layer) for name, layer in model.named_modules() if is_conv_layer(layer)]


def _parent_of(model, name):
    parent = model
    keys = name.split('.')
    for k in keys[:-1]:
        parent = parent._modules[k]
    return parent, keys[-1]


def replace_conv_layers(model, tr_params, data_bits, data_terms, *, encoding='hese'):
    """Swap every conv but the first for a TRConv2dLayer, in named_modules order; `encoding` is the term encoding
    ('hese', 'binary' or 'booth') of every wrapped layer."""
    _lib.encoding_id(encoding)
    for idx, (name, layer) in enumerate(_conv_layers(model)):
        if idx == 0:
            continue
        weight_bits, group_size, weight_terms = tr_params[idx]
        parent, key = _parent_of(model, name)
        parent._modules[key] = TRConv2dLayer(layer, data_bits, data_terms, weight_bits,
                                             group_size, weight_terms, encoding=encoding)
    return model


def static_conv_layer_settings(model, weight_bits, group_size, num_terms):
    stats = []
    for idx, (name, layer) in enumerate(_conv_layers(model)):
        if idx == 0 or layer.groups > 1 or 'se' in name:
            stats.append((16, 1, 16))
        else:
            stats.append((weight_bits, group_size, num_terms))
    return stats


def convert_model(model, tr_params, data_bits, data_terms, *, encoding='hese'):
    # the conversion rewrites weights in place, so work on a copy (refuse a bad encoding before copying)
    _lib.encoding_id(encoding)
    return replace_conv_layers(deepcopy(model), tr_params, data_bits, data_terms, encoding=encoding)
