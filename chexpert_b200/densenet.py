"""Host-side wiring of the attention-augmented DenseNet121 around the B200 AAConv2d.

The wiring lives here (SURVEY.md section 8, rows a13-a15): which dk/dv/input_dims each Transition gets, the
InstanceNorm -> ReLU -> AAConv2d(3x3, stride 2) sequence, and the weight initialisation, so that a checkpoint written
by the reference (``features.transition{1,2,3}.conv.{conv,in_proj_qkv,out_proj}.weight``, ``...key_rel_h/w``;
chexpert.py:90-123,504-518) loads strictly into this model and vice versa.  The dense blocks are torchvision's
(``_DenseBlock``), exactly as in the reference (models/attn_aug_conv.py:13,479); they are outside the hot path.

    reference                                   here
    models/attn_aug_conv.py:411-446 _Transition -> transition()
    models/attn_aug_conv.py:448-517 DenseNet    -> DenseNet
    chexpert.py:474-476 'aadensenet121'         -> aadensenet121()
    chexpert.py:24 torchvision densenet121      -> densenet121()  (Transitions: BNTransition with fused_transition)
"""
from collections import OrderedDict


import torch
import torch.nn as nn
import torch.nn.functional as F
from torchvision.models.densenet import _DenseBlock, _DenseLayer

from .aaconv import AAConv2d
from .fused_bn import (bn_relu, tap_bn_relu, tap_bn_relu_cl, bn_relu_cl, cl_ok, slice_layout, _is_cl, bn_relu_eval, eval_ok,
                       eval_cl_ok, _fused_ok, pool_ok, bn_relu_pool, bn_relu_pool_eval, module_bn, _alias, _strided_ok)
from .gradcam import grad_cam


def transition_attn_dims(num_output_features, attn_params):
    """dk, dv, (H, W) of the AAConv2d in one Transition (models/attn_aug_conv.py:416-427)."""
    nh = attn_params['nh']
    dk = max(20 * nh, int((attn_params['k'] * num_output_features // nh) * nh))
    dv = int((attn_params['v'] * num_output_features // nh) * nh)
    dims = attn_params['input_dims'][0] // 2, attn_params['input_dims'][1] // 2   # attention runs on the strided map
    return dk, dv, dims


class AATransition(nn.Sequential):
    """InstanceNorm2d -> ReLU -> AAConv2d(3x3, stride 2) with the reference's child names ``norm`` / ``relu`` / ``conv``
    (models/attn_aug_conv.py:436-440), so state_dicts are interchangeable.

    ``fused_prologue=True`` (SURVEY.md section 8 row f1): on CUDA the InstanceNorm statistics, the normalisation and the ReLU
    run inside the AAConv2d kernels (one statistics pass + the operand pack forward; one fused adjoint pass backward) instead
    of as two separate torch modules; ``norm`` and ``relu`` stay as (parameter-free) children and define eps.
    ``forward(x, out_total=C)`` makes the AAConv2d epilogues write into the first channels of the next dense block's
    (B, C, H, W) feature buffer (row f3)."""

    def __init__(self, num_input_features, num_output_features, attn_params, precision=None, fused_prologue=False):
        super().__init__()
        dk, dv, dims = transition_attn_dims(num_output_features, attn_params)
        self.add_module('norm', nn.InstanceNorm2d(num_input_features))          # affine=False, no running stats (:438)
        self.add_module('relu', nn.ReLU(inplace=True))
        self.add_module('conv', AAConv2d(num_input_features, num_output_features, 3, 2, dk, dv, attn_params['nh'],
                                         attn_params['relative'], dims, precision=precision))
        self.fused_prologue = bool(fused_prologue)

    def forward(self, x, out_total=None):
        if self.fused_prologue and x.is_cuda and not self.norm.affine and not self.norm.track_running_stats:
            return self.conv(x, out_total=out_total, fused_in=self.norm.eps)
        return self.conv(self.relu(self.norm(x)), out_total=out_total)


def transition(num_input_features, num_output_features, attn_params=None, precision=None, fused_prologue=False):
    """Sequential with the reference's child names: norm, relu, conv (+ pool for the plain variant)."""
    if attn_params is None:   # stock DenseNet transition (models/attn_aug_conv.py:429-434)
        return nn.Sequential(OrderedDict([
            ('norm', nn.BatchNorm2d(num_input_features)),
            ('relu', nn.ReLU(inplace=True)),
            ('conv', nn.Conv2d(num_input_features, num_output_features, kernel_size=1, stride=1, bias=False)),
            ('pool', nn.AvgPool2d(kernel_size=2, stride=2)),
        ]))
    return AATransition(num_input_features, num_output_features, attn_params, precision, fused_prologue)


# ------------------------------------------------------------------------------------------------
# pre-allocated DenseBlock feature buffer (SURVEY.md section 8 row f3)
# ------------------------------------------------------------------------------------------------
class _Adopt(torch.autograd.Function):
    """init_features -> the first channels of the block's buffer (copied unless they were produced there)."""

    @staticmethod
    def forward(ctx, init, buf):
        c0 = init.shape[1]
        view = _alias(buf, 0, c0)
        if init.data_ptr() != view.data_ptr() or init.stride() != view.stride():
            view.copy_(init)
        return view

    @staticmethod
    def backward(ctx, g):
        return g, None


class _Append(torch.autograd.Function):
    """[features so far | new_features]: the concatenation of torchvision's block (densenet.py:48,120-124) without the copy of
    everything that came before -- only the layer's own `growth_rate` channels are written, next to the rest."""

    @staticmethod
    def forward(ctx, prev, new, buf):
        c = prev.shape[1]
        ctx.c = c
        _alias(buf, c, c + new.shape[1]).copy_(new)
        return _alias(buf, 0, c + new.shape[1])

    @staticmethod
    def backward(ctx, g):
        return g[:, :ctx.c], g[:, ctx.c:], None


def _to_nhwc(g):
    """The gradient of a channel slice of an NCHW buffer as a dense channels-last tensor (for a convolution's backward)."""
    if g.is_cuda and _strided_ok(g, aligned=True):
        return slice_layout(g, torch.empty(g.shape, device=g.device, dtype=g.dtype, memory_format=torch.channels_last), to_nchw=False)
    return g.contiguous(memory_format=torch.channels_last)


class _AppendCL(torch.autograd.Function):
    """_Append for channels-last new features: they are transposed into their channel slice of the NCHW buffer (one tiled kernel),
    and the slice of the buffer gradient is transposed back to NHWC for conv2's backward."""

    @staticmethod
    def forward(ctx, prev, new, buf):
        c, k = prev.shape[1], new.shape[1]
        ctx.c = c
        slice_layout(new.detach(), _alias(buf, c, c + k), to_nchw=True)
        return _alias(buf, 0, c + k)

    @staticmethod
    def backward(ctx, g):
        return g[:, :ctx.c], _to_nhwc(g[:, ctx.c:]), None


class _ToBuffer(torch.autograd.Function):
    """A channels-last (B, Cout, H, W) tensor -> channels [0, Cout) of a new (B, out_total, H, W) NCHW feature buffer, which the next
    BufferedDenseBlock adopts without a copy; backward hands the slice's gradient back channels-last (as _AppendCL does)."""

    @staticmethod
    def forward(ctx, z, out_total):
        B, C, H, W = z.shape
        buf = torch.empty(B, out_total, H, W, device=z.device, dtype=z.dtype)
        view = _alias(buf, 0, C)
        slice_layout(z.detach(), view, to_nchw=True)
        ctx.mark_non_differentiable(buf)
        return view, buf

    @staticmethod
    def backward(ctx, g, _gbuf):
        return _to_nhwc(g), None


def _append(feats, new, buf, slice_ok):
    """[feats | new] in buf: a channels-last `new` is transposed into its slice when ``slice_ok`` (see BufferedDenseBlock.forward),
    anything else is copied."""
    if slice_ok and _is_cl(new):
        return _AppendCL.apply(feats, new, buf)
    return _Append.apply(feats, new.contiguous(), buf)


class BNTransition(nn.Sequential):
    """torchvision's ``_Transition`` (BatchNorm2d -> ReLU -> Conv2d 1x1 -> AvgPool2d(2), densenet.py:98-104) with its child names
    ``norm`` / ``relu`` / ``conv`` / ``pool``, so state_dicts are interchangeable, and a fused route on CUDA.

    There the BatchNorm + ReLU + 2x2 average run as one kernel (fused_bn.bn_relu_pool) that reads the finished feature buffer once
    and writes the pooled operand channels-last; the 1x1 convolution (cuDNN, as in the dense layers) then runs on a quarter of the
    pixels -- the pool and the per-pixel linear convolution commute.  In training the kernel reuses the block's shared BatchNorm
    statistics (``x.bn_stats``, set by BufferedDenseBlock), so only the block's last layer's channels are reduced again.
    ``forward(x, out_total=C)`` writes the result into channels [0, Cout) of a new (B, C, H/2, W/2) buffer, attached as
    ``.feature_buffer`` for the next block to adopt.

    The fused route is taken in training on CUDA, and in eval mode with autograd off when ``fused_eval``; C and Cout multiples of 4,
    H and W >= 2, (H/2)(W/2) a multiple of 4 and four-element alignment are required (fused_bn.pool_ok).  Anything else -- CPU, eval
    with grad enabled (Grad-CAM), a shape past those limits -- runs the four modules unchanged (the norm through fused_bn.module_bn,
    so that a num_batches_tracked which TrainStep bumps is not bumped twice)."""

    def __init__(self, num_input_features, num_output_features, fused_eval=False):
        super().__init__(OrderedDict([
            ('norm', nn.BatchNorm2d(num_input_features)),
            ('relu', nn.ReLU(inplace=True)),
            ('conv', nn.Conv2d(num_input_features, num_output_features, kernel_size=1, stride=1, bias=False)),
            ('pool', nn.AvgPool2d(kernel_size=2, stride=2)),
        ]))
        self.fused_eval = bool(fused_eval)

    def _fused(self, x):
        if x.dim() != 4 or not (self.training or self.fused_eval) or not pool_ok(self.norm, x):
            return False
        H, W = x.shape[2:]
        return self.conv.out_channels % 4 == 0 and ((H // 2) * (W // 2)) % 4 == 0      # aaconv_slice_layout into the next buffer

    def forward(self, x, out_total=None):
        if not self._fused(x):
            return self.pool(self.conv(self.relu(module_bn(self.norm, x))))
        if self.training:
            p = bn_relu_pool(self.norm, x, getattr(x, 'bn_stats', None))
        else:
            p = bn_relu_pool_eval(self.norm, x)
        z = F.conv2d(p, self.conv.weight).contiguous(memory_format=torch.channels_last)
        y, buf = _ToBuffer.apply(z, int(out_total or z.shape[1]))
        y.feature_buffer = buf
        return y


class BufferedDenseBlock(nn.ModuleDict):
    """torchvision's ``_DenseBlock`` (same ``denselayer%d`` children, parameters and arithmetic; the reference uses it at
    models/attn_aug_conv.py:479-482) over ONE pre-allocated (B, C_in + n * growth, H, W) feature buffer: layer i reads channels
    [0, c_i) of the buffer and writes its output behind them, so the per-layer ``torch.cat`` (O(layers^2) copy traffic and
    saved activations) disappears.  If ``init_features`` already lives in such a buffer (an AAConv2d called with ``out_total``),
    it is adopted without a copy.  The gradient of the concatenated features is accumulated along the chain
    (one add per layer over contiguous tensors) instead of per (producer, consumer) pair.

    ``fused_eval=True``: in eval mode on CUDA with autograd off, every norm -> relu pair runs as relu(BatchNorm2d eval) through
    fused_bn.bn_relu_eval (running statistics; the same layout plan as training: NCHW prefix -> NHWC for conv1, NHWC -> NHWC for
    conv2).  Anything else -- training, grad enabled (e.g. Grad-CAM), CPU -- takes the path below unchanged."""

    def __init__(self, num_layers, num_input_features, bn_size, growth_rate, drop_rate, fused_eval=False):
        super().__init__()
        for i in range(num_layers):
            self.add_module('denselayer%d' % (i + 1),
                            _DenseLayer(num_input_features + i * growth_rate, growth_rate=growth_rate, bn_size=bn_size,
                                        drop_rate=drop_rate))
        self.num_input_features, self.growth_rate, self.num_layers = num_input_features, growth_rate, num_layers
        self.out_channels = num_input_features + num_layers * growth_rate
        self.inner_channels_last = True   # False: NCHW inside the layers, the route taken when slice_ok / cl_ok fail
        self.fused_eval = bool(fused_eval)

    def _forward_eval(self, feats, buf, slice_ok):
        """Inference through the eval-mode BatchNorm + ReLU kernels (no stats buffer: the running statistics are all they read)."""
        for layer in self.values():
            norm1, norm2 = layer.norm1, layer.norm2
            if self.inner_channels_last and slice_ok and eval_cl_ok(norm1, feats):
                z = layer.conv1(bn_relu_eval(norm1, feats, out_cl=True))
                y2 = bn_relu_eval(norm2, z, out_cl=True) if eval_cl_ok(norm2, z) else bn_relu_eval(norm2, z)
                new = layer.conv2(y2).to(buf.dtype)
            else:
                new = layer.conv2(bn_relu_eval(norm2, layer.conv1(bn_relu_eval(norm1, feats)))).to(buf.dtype)
            feats = _append(feats, new, buf, slice_ok)
        return feats

    def forward(self, init_features):
        B, C0, H, W = init_features.shape
        buf = getattr(init_features, 'feature_buffer', None)
        if (buf is None or tuple(buf.shape) != (B, self.out_channels, H, W) or buf.dtype != init_features.dtype
                or not buf.is_contiguous() or buf.data_ptr() != init_features.data_ptr()):
            buf = torch.empty(B, self.out_channels, H, W, dtype=init_features.dtype, device=init_features.device)
        feats = _Adopt.apply(init_features, buf)
        # every layer's features are a channel prefix of buf (the same strides and start): whether aaconv_slice_layout can write the
        # growth channels of channels-last layers into the buffer holds for the whole block
        slice_ok = buf.is_cuda and self.growth_rate % 4 == 0 and (H * W) % 4 == 0 and _strided_ok(feats, aligned=True)
        if self.fused_eval and all(eval_ok(layer.norm1, feats) and eval_ok(layer.norm2, feats) for layer in self.values()):
            return self._forward_eval(feats, buf, slice_ok)
        # per-(channel, sample) plane statistics of the buffer, shared by the norm1 of every layer: layer i only reduces the channels
        # layer i-1 has not seen (its own 32 new ones); the first layer reduces the block's input channels
        stats = torch.empty(2 * B * self.out_channels, device=buf.device, dtype=torch.float32) if buf.is_cuda else None
        valid = 0
        shared = stats is not None          # every norm1 reduced its new channels into `stats` (the fused kernels ran)
        for layer in self.values():
            # norm -> relu pairs: fused strided kernels in training on CUDA (chexpert_b200.fused_bn), the torch modules otherwise
            c = feats.shape[1]
            if (self.inner_channels_last and slice_ok and layer.drop_rate == 0 and torch.is_grad_enabled() and feats.requires_grad
                    and cl_ok(layer.norm1, feats)):
                # The two convolutions of the layer run channels-last (cuDNN's tensor-core kernels are NHWC; with NCHW tensors it
                # transposes every operand of every fprop / dgrad / wgrad itself: 21 % of the step in the round-2 profile).  The
                # layout change rides on the BatchNorm + ReLU passes (csrc/bn_cl.cu); the buffer itself stays NCHW.
                feats, y1 = tap_bn_relu_cl(layer.norm1, feats, (stats, valid))
                z = layer.conv1(y1)
                if _is_cl(z) and cl_ok(layer.norm2, z):
                    new = layer.conv2(bn_relu_cl(layer.norm2, z))
                else:
                    new = layer.conv2(bn_relu(layer.norm2, z.contiguous()))
                valid = c
                feats = _append(feats, new.to(buf.dtype), buf, slice_ok)
                continue
            # norm1 taps the concatenated features: backward adds its dx into the gradient of the concatenation in place
            shared = shared and _fused_ok(layer.norm1, feats)
            feats, y1 = tap_bn_relu(layer.norm1, feats, None if stats is None else (stats, valid))
            new = layer.conv2(bn_relu(layer.norm2, layer.conv1(y1)))
            valid = c
            if layer.drop_rate > 0:
                new = F.dropout(new, p=layer.drop_rate, training=self.training)
            feats = _Append.apply(feats, new.to(buf.dtype), buf)
        if shared:
            # the statistics of channels [0, valid) of the output are in `stats`: a BNTransition reduces only the last layer's channels
            feats.bn_stats = (stats, valid)
        return feats


class DenseNet(nn.Module):
    """DenseNet with attention-augmented transitions; constructor of models/attn_aug_conv.py:452-453 plus
    ``precision`` ('fp32' | 'bf16') for the AAConv2d kernels.  Unlike the reference, ``attn_params`` is not mutated.
    With ``attn_params=None`` it is torchvision's DenseNet (same state_dict); ``fused_transition=True`` with ``feature_buffer=True``
    then builds BNTransition (fused BatchNorm + ReLU + pool kernel) in place of the module Transition."""

    def __init__(self, growth_rate=32, block_config=(6, 12, 24, 16), num_init_features=64, bn_size=4, drop_rate=0,
                 num_classes=1000, attn_params=None, precision=None, feature_buffer=False, fused_prologue=False, fused_eval=False,
                 fused_transition=False):
        super().__init__()
        self.feature_buffer = bool(feature_buffer)
        self.fused_eval = bool(fused_eval)
        attn = dict(attn_params) if attn_params is not None else None
        if len(block_config) == 4:    # ImageNet stem: /4 before the first block (:460-468)
            stem = [('conv0', nn.Conv2d(3, num_init_features, kernel_size=7, stride=2, padding=3, bias=False)),
                    ('norm0', nn.BatchNorm2d(num_init_features)),
                    ('relu0', nn.ReLU(inplace=True)),
                    ('pool0', nn.MaxPool2d(kernel_size=3, stride=2, padding=1))]
            if attn is not None:
                attn['input_dims'] = attn['input_dims'][0] // 4, attn['input_dims'][1] // 4
        else:                         # CIFAR stem (:470-474)
            stem = [('conv0', nn.Conv2d(3, num_init_features, kernel_size=5, stride=1, padding=2, bias=False)),
                    ('norm0', nn.BatchNorm2d(num_init_features)),
                    ('relu0', nn.ReLU(inplace=True))]
        self.features = nn.Sequential(OrderedDict(stem))
        width = num_init_features
        for i, num_layers in enumerate(block_config):
            block = (BufferedDenseBlock(num_layers, width, bn_size, growth_rate, drop_rate, fused_eval) if feature_buffer else
                     _DenseBlock(num_layers=num_layers, num_input_features=width, bn_size=bn_size, growth_rate=growth_rate,
                                 drop_rate=drop_rate))
            self.features.add_module(f'denseblock{i + 1}', block)
            width += num_layers * growth_rate
            if i != len(block_config) - 1:
                if attn is None and feature_buffer and fused_transition:
                    trans = BNTransition(width, width // 2, fused_eval)
                else:
                    trans = transition(width, width // 2, attn, precision, fused_prologue)
                self.features.add_module(f'transition{i + 1}', trans)
                width //= 2
            if attn is not None:      # every stage halves the map the next transition's attention sees (:491-493)
                attn['input_dims'] = attn['input_dims'][0] // 2, attn['input_dims'][1] // 2
        self.features.add_module('norm5', nn.BatchNorm2d(width))
        self.classifier = nn.Linear(width, num_classes)
        for m in self.modules():      # :503-510 -- includes the three Conv2d parameter holders of every AAConv2d
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Linear):
                nn.init.constant_(m.bias, 0)

    def _bn_relu(self, bn, x):
        """Stem norm0 -> relu0 and norm5 -> F.relu: the eval-mode kernel when fused_eval asks for it and it applies (eval mode, CUDA,
        autograd off), the training-mode kernels / the module otherwise."""
        if self.fused_eval and eval_ok(bn, x):
            return bn_relu_eval(bn, x)
        return bn_relu(bn, x)

    def _norm5_input(self, x):
        """-> the input of features.norm5: the last dense block's output (with feature_buffer, its whole buffer)."""
        mods = list(self.features.children())[:-1]                  # norm5 is the last child
        if not self.feature_buffer:
            for m in mods:
                x = m(x)
            return x
        skip = False
        for i, m in enumerate(mods):
            if skip:
                skip = False
                continue
            nxt = mods[i + 1] if i + 1 < len(mods) else None
            if isinstance(m, (AATransition, BNTransition)) and isinstance(nxt, BufferedDenseBlock):
                x = m(x, out_total=nxt.out_channels)      # the Transition writes into the next block's buffer
            elif isinstance(m, nn.BatchNorm2d) and isinstance(nxt, nn.ReLU):
                x = self._bn_relu(m, x)                   # stem: norm0 -> relu0 as one fused op (grid (C, B) instead of one CTA per channel)
                skip = True
            else:
                x = m(x)
        return x

    def _norm5_relu(self, x):
        """relu(features.norm5(x)): norm5 followed by forward()'s F.relu."""
        if not self.feature_buffer:
            return F.relu(self.features.norm5(x), inplace=True)
        return self._bn_relu(self.features.norm5, x)

    def _features(self, x):
        """-> relu(features(x)) (models/attn_aug_conv.py:513-514).  Without feature_buffer model.features runs as the module it is,
        so hooks on it keep firing."""
        if not self.feature_buffer:
            return F.relu(self.features(x), inplace=True)
        return self._norm5_relu(self._norm5_input(x))

    def _head(self, f):
        return self.classifier(F.adaptive_avg_pool2d(f, (1, 1)).flatten(1))

    def forward(self, x):
        return self._head(self._features(x))

    def forward_grad_cam(self, x, size=None):
        """-> (logits, maps): the logits of forward(x) and Grad-CAM of every class at model.features' output (the layer the reference
        hooks, chexpert.py:260-361), computed in closed form by gradcam.grad_cam from norm5's input -- no backward pass.  maps: fp32
        (B, K, h, w) at the feature map's resolution, or (B, K, size, size) upsampled bilinearly when `size` is given.
        Inference only: eval mode, CUDA, autograd off, and a norm5 the eval kernels take (fused_bn.eval_ok); anything else raises."""
        if self.training:
            raise RuntimeError('forward_grad_cam runs in eval mode only (call model.eval()): Grad-CAM here uses the running statistics')
        if torch.is_grad_enabled():
            raise RuntimeError('forward_grad_cam runs with autograd off (torch.no_grad()): its gradient is computed in closed form')
        if not x.is_cuda:
            raise RuntimeError('forward_grad_cam runs on CUDA only; there is no CPU fallback')
        h = self._norm5_input(x)
        if not eval_ok(self.features.norm5, h):
            raise RuntimeError('forward_grad_cam needs an affine norm5 with fp32 parameters and running statistics and an fp32 / bf16 '
                               'feature map of at most 65535 samples')
        logits = self._head(self._norm5_relu(h))
        cam, up = grad_cam(h, self.features.norm5, self.classifier, size)
        return logits, cam if up is None else up

    def attn_layers(self):
        """The AAConv2d modules the visualise path hooks (chexpert.py:478)."""
        return [m for m in self.modules() if isinstance(m, AAConv2d)]


def aadensenet121(num_classes=5, input_dims=(320, 320), precision=None, feature_buffer=False, fused_prologue=False, fused_eval=False):
    """The model behind ``--model aadensenet121`` (chexpert.py:474-476); ``input_dims`` is the image size.
    ``feature_buffer`` / ``fused_prologue``: the B200 execution options of rows f3 / f1 (same parameters, same state_dict).
    ``fused_eval``: inference of the feature-buffer model (eval mode, CUDA, autograd off) runs its BatchNorm + ReLU pairs through
    the eval-mode kernels (fused_bn.bn_relu_eval); it has no effect without ``feature_buffer`` and adds no parameters."""
    return DenseNet(32, (6, 12, 24, 16), 64, num_classes=num_classes,
                    attn_params={'k': 0.2, 'v': 0.1, 'nh': 8, 'relative': True, 'input_dims': tuple(input_dims)},
                    precision=precision, feature_buffer=feature_buffer, fused_prologue=fused_prologue, fused_eval=fused_eval)


def densenet121(num_classes=5, feature_buffer=False, fused_transition=False, fused_eval=False):
    """The model behind ``--model densenet121`` (chexpert.py:24): torchvision's densenet121 -- same 727 state_dict keys and shapes,
    6,958,981 parameters at 5 classes, so torchvision's state_dict (e.g. ImageNet-initialised weights with the classifier replaced)
    loads strictly.  ``feature_buffer`` / ``fused_eval``: the dense-block execution options of aadensenet121;
    ``fused_transition`` (with ``feature_buffer``): the Transitions run as BNTransition.  None of them adds parameters."""
    return DenseNet(32, (6, 12, 24, 16), 64, num_classes=num_classes, attn_params=None, feature_buffer=feature_buffer,
                    fused_eval=fused_eval, fused_transition=fused_transition)


def build_model(arch, num_classes=5, size=320, precision=None, feature_buffer=False, fused=False, fused_eval=False):
    """aadensenet121 or the reference's baseline densenet121 by name.  ``fused``: aadensenet121's fused_prologue / densenet121's
    fused_transition (fused BatchNorm + ReLU + pool Transitions); ``size`` and ``precision`` only concern aadensenet121's AAConv2d."""
    if arch == 'aadensenet121':
        return aadensenet121(num_classes, (size, size), precision=precision, feature_buffer=feature_buffer, fused_prologue=fused,
                             fused_eval=fused_eval)
    if arch == 'densenet121':
        return densenet121(num_classes, feature_buffer=feature_buffer, fused_transition=fused, fused_eval=fused_eval)
    raise ValueError(f"arch must be 'aadensenet121' or 'densenet121', got {arch!r}")


def conv_weight_plan(model):
    """[(name, conv, channels_last)] for the nn.Conv2d modules of `model` that cuDNN runs: all but the parameter holders of the
    AAConv2d modules, whose fp32 weights the library's kernels read.  channels_last: a k x k convolution of a BufferedDenseBlock whose
    layers run channels-last (inner_channels_last) sees NHWC activations, so its weight is kept channels-last too, or cuDNN would
    transpose it on every call.  1 x 1 weights are the same bytes in both formats; the stem's convolution stays NCHW."""
    own = {id(p) for m in model.modules() if isinstance(m, AAConv2d) for p in m.parameters()}
    cl = {id(m) for b in model.modules() if isinstance(b, BufferedDenseBlock) and b.inner_channels_last for m in b.modules()}
    return [(name, m, id(m) in cl and m.weight.shape[2] * m.weight.shape[3] > 1) for name, m in model.named_modules()
            if isinstance(m, nn.Conv2d) and id(m.weight) not in own]
