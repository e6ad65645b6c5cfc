"""Reference model of the whole attention-augmented DenseNet, built from torch ops only.  TEST INFRASTRUCTURE ONLY.

The reference's DenseNet (models/attn_aug_conv.py:448-517) with the ImageNet stem: torchvision's ``_DenseBlock``, Transitions
``norm`` (InstanceNorm2d) -> ``relu`` -> ``conv`` (``RefAAConv``: the oracle's ``aaconv_forward_sequential``), ``norm5`` and a
Linear classifier.  It shares no code with ``chexpert_b200``, has the reference's state_dict names (an ``aadensenet121``
state_dict loads strictly), and runs in whatever dtype it is cast to -- float64 is the parity reference of the training step.
Pinned by tests/test_oracle.py against the reference's own tiny-DenseNet fixture (tests/golden/tiny_densenet*.npz).
"""
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F
from torchvision.models.densenet import _DenseBlock

from .aaconv_oracle import AAConvShape, aaconv_forward_sequential, derive_transition_attn


class RefAAConv(nn.Module):
    """AAConv2d(3 x 3, stride 2) of a Transition: bias-free Conv2d parameter holders ``conv`` / ``in_proj_qkv`` / ``out_proj`` and
    ``key_rel_h`` / ``key_rel_w``, registered in the reference's order; forward is aaconv_forward_sequential."""

    def __init__(self, cin, cout, dk, dv, nh, relative, dims):
        super().__init__()
        self.shape = AAConvShape(cin, cout, 3, 2, dk, dv, nh, relative, tuple(dims))
        self.conv = nn.Conv2d(cin, cout - dv, 3, 2, 1, bias=False) if cout > dv else None
        self.in_proj_qkv = nn.Conv2d(cin, 2 * dk + dv, 1, 2, bias=False)
        self.out_proj = nn.Conv2d(dv, dv, 1, bias=False)
        if relative:
            self.key_rel_h = nn.Parameter(torch.zeros(dk // nh, 2 * dims[0] - 1))
            self.key_rel_w = nn.Parameter(torch.zeros(dk // nh, 2 * dims[1] - 1))

    def forward(self, x):
        return aaconv_forward_sequential(x, dict(self.named_parameters()), self.shape)


class RefDenseNet(nn.Module):
    def __init__(self, growth_rate, block_config, num_init_features, attn_params, image_size, num_classes=5, bn_size=4):
        super().__init__()
        feats = OrderedDict([('conv0', nn.Conv2d(3, num_init_features, 7, 2, 3, bias=False)),
                             ('norm0', nn.BatchNorm2d(num_init_features)), ('relu0', nn.ReLU(inplace=True)),
                             ('pool0', nn.MaxPool2d(3, 2, 1))])
        dims = image_size[0] // 4, image_size[1] // 4           # the attention maps follow the stem's /4 and every stage's /2
        width = num_init_features
        for i, n in enumerate(block_config):
            feats[f'denseblock{i + 1}'] = _DenseBlock(n, width, bn_size, growth_rate, 0.0)
            width += n * growth_rate
            if i != len(block_config) - 1:
                dk, dv, d = derive_transition_attn(width // 2, {**attn_params, 'input_dims': dims})
                feats[f'transition{i + 1}'] = nn.Sequential(OrderedDict([
                    ('norm', nn.InstanceNorm2d(width)), ('relu', nn.ReLU()),
                    ('conv', RefAAConv(width, width // 2, dk, dv, attn_params['nh'], attn_params['relative'], d))]))
                width //= 2
            dims = dims[0] // 2, dims[1] // 2
        feats['norm5'] = nn.BatchNorm2d(width)
        self.features = nn.Sequential(feats)
        self.classifier = nn.Linear(width, num_classes)

    def forward(self, x):
        return self.classifier(F.adaptive_avg_pool2d(F.relu(self.features(x)), 1).flatten(1))


def ref_aadensenet121(image_size=(320, 320), num_classes=5):
    """The reference's aadensenet121 (chexpert.py:474-476)."""
    return RefDenseNet(32, (6, 12, 24, 16), 64, {'k': 0.2, 'v': 0.1, 'nh': 8, 'relative': True}, image_size, num_classes)
