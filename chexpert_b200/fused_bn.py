"""BatchNorm2d (training mode) + ReLU as one op that reads its input through a batch stride -- the normalisation of a channel
slice of the pre-allocated DenseBlock feature buffer (SURVEY.md section 8 row f3; torchvision densenet.py:36-41 under
models/attn_aug_conv.py:479-482).  Parameters, buffers and the arithmetic are nn.BatchNorm2d's (same state_dict, same running
statistics update); eval mode and CPU tensors go through the module's own forward.  bn_relu_eval is the eval-mode counterpart
(running statistics, no backward) that the dense blocks take only when asked to (DenseNet(fused_eval=True)) and autograd is off.
bn_relu_pool / bn_relu_pool_eval add the 2x2 average pool of torchvision's Transition (densenet.BNTransition).
"""
import ctypes

import torch
import torch.nn.functional as F

from . import _lib
from .aaconv import _ptr, _stream

_DT = {torch.float32: _lib.FP32, torch.bfloat16: _lib.BF16}


def _aligned(t):
    return t.data_ptr() % (4 * t.element_size()) == 0


def _strided_ok(t, aligned=False):
    """(B, C, H, W) with dense (C, H, W) inside every sample: a contiguous tensor or a channel slice of the feature buffer.
    ``aligned``: the start and the batch stride on four-element boundaries too (the vectorised kernels' accesses)."""
    B, C, H, W = t.shape
    return (t.stride(3) == 1 and t.stride(2) == W and t.stride(1) == H * W and t.stride(0) >= C * H * W
            and (not aligned or (t.stride(0) % 4 == 0 and _aligned(t))))


def _input_ok(x):
    """A CUDA fp32 / bf16 (B, C, H, W) tensor with at most 65535 samples."""
    return x.is_cuda and x.dim() == 4 and x.dtype in _DT and x.shape[0] <= 65535


def _module_ok(bn):
    """An affine BatchNorm2d with running statistics (and a momentum when it is training) whose weight, bias and running statistics
    are contiguous fp32: the kernels read and update them through float pointers."""
    if not (bn.affine and bn.track_running_stats and (bn.momentum is not None or not bn.training)):
        return False
    w, b, m, v = bn.weight, bn.bias, bn.running_mean, bn.running_var
    return (m is not None and w.dtype == b.dtype == m.dtype == v.dtype == torch.float32
            and w.is_contiguous() and b.is_contiguous() and m.is_contiguous() and v.is_contiguous())


def _bump(bn):
    if bn.num_batches_tracked is not None and not getattr(bn, '_nbt_batched', False):   # TrainStep bumps all counters in one launch
        bn.num_batches_tracked.add_(1)


def _alias(t, c0=0, c1=None):
    """Channels [c0, c1) (default: all) of the (B, C, H, W) tensor t over the same memory, with its own autograd identity and
    version counter: later writes into other channels of the same feature buffer must not invalidate what an op saved."""
    c1 = t.shape[1] if c1 is None else c1
    return torch.empty(0, dtype=t.dtype, device=t.device).set_(t.untyped_storage(), t.storage_offset() + c0 * t.stride(1),
                                                               (t.shape[0], c1 - c0, *t.shape[2:]), t.stride())


def _block_stats(lib, stats, x):
    """-> (plane statistics buffer, n_valid) for x.  ``stats = (buffer, n_valid)``: plane statistics shared along a dense block --
    channels [0, n_valid) of x were already reduced into `buffer` by the previous layer (channel-major (C_total, B) float2: a
    prefix is a valid (C, B) table).  Without it, or when it is too small for x: a fresh workspace with nothing valid."""
    B, C = x.shape[0], x.shape[1]
    if stats is not None and stats[0].numel() * 4 >= 8 * B * C:
        return stats[0], min(int(stats[1]), C)
    return torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C) // 4, device=x.device, dtype=torch.float32), 0


def _stats_nchw(lib, xs, pst, valid):
    """Reduces channels [valid, C) of xs into pst (aaconv_bn_stats_nchw) -> (G, bpb): the batch-group split of its partials."""
    B, C, H, W = xs.shape
    G, bpb = ctypes.c_int(0), ctypes.c_int(0)
    _lib.check(lib.aaconv_bn_stats_nchw(_ptr(xs), _DT[xs.dtype], B, C, H * W, xs.stride(0), _ptr(pst), valid, ctypes.byref(G),
                                        ctypes.byref(bpb), _stream()), 'aaconv_bn_stats_nchw')
    return G.value, bpb.value


def _grad_wb(ctx, xs):
    """Empty fp32 (dweight, dbias), None where autograd does not ask for one."""
    C, need = xs.shape[1], ctx.needs_input_grad
    return (torch.empty(C, device=xs.device, dtype=torch.float32) if need[1] else None,
            torch.empty(C, device=xs.device, dtype=torch.float32) if need[2] else None)


def _accumulates(g, xs, aligned=False):
    """The gradient g of the concatenation can take dx in place: xs's dtype and shape, dense samples."""
    return g is not None and g.dtype == xs.dtype and g.shape == xs.shape and _strided_ok(g, aligned)


class _BNReLU(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps, stats=None):
        lib = _lib.load()
        B, C, H, W = x.shape
        xs = x.detach()
        w, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        with torch.cuda.device(x.device):
            y = torch.empty(B, C, H, W, device=x.device, dtype=x.dtype)
            saved = torch.empty(C, 2, device=x.device, dtype=torch.float32)
            ws, valid = _block_stats(lib, stats, x)
            _lib.check(lib.aaconv_bn_relu_forward(_ptr(xs), _DT[x.dtype], B, C, H * W, xs.stride(0), _ptr(w), _ptr(b),
                                                  _ptr(running_mean), _ptr(running_var), float(momentum), float(eps), _ptr(y),
                                                  _ptr(saved), _ptr(ws), valid, _stream()), 'aaconv_bn_relu_forward')
        ctx.save_for_backward(xs, saved, w, b)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        xs, saved, w, b = ctx.saved_tensors
        B, C, H, W = xs.shape
        g = dy.detach().to(xs.dtype).contiguous()
        with torch.cuda.device(xs.device):
            dx = torch.empty(B, C, H, W, device=xs.device, dtype=xs.dtype) if ctx.needs_input_grad[0] else None
            dw, db = _grad_wb(ctx, xs)
            ws = torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C), device=xs.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_backward(_ptr(xs), _DT[xs.dtype], B, C, H * W, xs.stride(0), _ptr(g), _ptr(saved), _ptr(w),
                                                   _ptr(b), _ptr(dx), _ptr(dw), _ptr(db), _ptr(ws), _stream()), 'aaconv_bn_relu_backward')
        return dx, dw, db, None, None, None, None, None


class _TapBNReLU(torch.autograd.Function):
    """(feats, relu(bn(feats))) for the concatenated features of a dense block: the first output IS the input (handed on to the
    next layer's concatenation), so that backward sees both consumers' gradients at once and ADDS this layer's dx into the
    gradient of the concatenation in place (aaconv_bn_relu_backward_acc) -- instead of a dense dx and autograd's own add."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps, stats=None):
        y = _BNReLU.forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps, stats)
        return _alias(x), y

    @staticmethod
    def backward(ctx, g_feats, dy):
        if dy is None:
            return g_feats, None, None, None, None, None, None, None
        xs, saved, w, b = ctx.saved_tensors
        if not (ctx.needs_input_grad[0] and _accumulates(g_feats, xs)):
            dx, dw, db = _BNReLU.backward(ctx, dy)[:3]
            if g_feats is not None and dx is not None:
                dx = dx + g_feats
            elif dx is None:
                dx = g_feats
            return dx, dw, db, None, None, None, None, None
        lib = _lib.load()
        B, C, H, W = xs.shape
        g = dy.detach().to(xs.dtype).contiguous()
        with torch.cuda.device(xs.device):
            dw, db = _grad_wb(ctx, xs)
            ws = torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C), device=xs.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_backward_acc(_ptr(xs), _DT[xs.dtype], B, C, H * W, xs.stride(0), _ptr(g), _ptr(saved), _ptr(w),
                                                       _ptr(b), _ptr(g_feats), g_feats.stride(0), _ptr(dw), _ptr(db), _ptr(ws),
                                                       _stream()), 'aaconv_bn_relu_backward_acc')
        return g_feats, dw, db, None, None, None, None, None


def _fused_ok(bn, x):
    return bn.training and _input_ok(x) and _module_ok(bn) and _strided_ok(x)


def module_bn(bn, x):
    """bn(x) through the module's own arithmetic, for the paths that do not run the fused kernels.  A counter that TrainStep bumps
    itself (``_nbt_batched``) must not be bumped again by nn.BatchNorm2d.forward: for a training-mode module with a momentum that
    forward is F.batch_norm with the module's buffers and parameters, plus the bump, so F.batch_norm is called without it."""
    if getattr(bn, '_nbt_batched', False) and bn.training and bn.track_running_stats and bn.momentum is not None:
        return F.batch_norm(x, bn.running_mean, bn.running_var, bn.weight, bn.bias, True, bn.momentum, bn.eps)
    return bn(x)


def tap_bn_relu(bn, x, stats=None):
    """-> (x handed on, relu(bn(x))): bn_relu for an input that has a second consumer (the concatenation of a dense block)."""
    if not (_fused_ok(bn, x) and torch.is_grad_enabled() and x.requires_grad):
        return x, bn_relu(bn, x, stats)
    _bump(bn)
    return _TapBNReLU.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.momentum, bn.eps, stats)


def bn_relu(bn, x, stats=None):
    """relu(bn(x)) for an nn.BatchNorm2d `bn`; the fused strided kernels when it is training on CUDA, the modules otherwise.
    ``stats = (float32 buffer of >= 2*B*C elements, n_valid_channels)`` shares the per-plane statistics between the layers of a
    dense block (see aaconv_bn_relu_forward)."""
    if not _fused_ok(bn, x):
        return F.relu(module_bn(bn, x), inplace=True)
    _bump(bn)
    return _BNReLU.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.momentum, bn.eps, stats)


# ------------------------------------------------------------------------------------------------
# channels-last side of a dense layer (csrc/bn_cl.cu): the convolutions see NHWC tensors, the feature buffer stays NCHW
# ------------------------------------------------------------------------------------------------
_CL = torch.channels_last


def _is_cl(t):
    return t.dim() == 4 and t.is_contiguous(memory_format=_CL)


CL_MAX_C = 4096   # channels of an NHWC input the statistics kernel keeps in registers (csrc/bn_cl.cu, CL_MAX_C)


def cl_ok(bn, x):
    """The channels-last kernels cover training-mode BatchNorm2d on CUDA with C and H*W multiples of 4, and at most CL_MAX_C
    channels when x itself is channels-last."""
    if not (bn.training and _input_ok(x) and _module_ok(bn)):
        return False
    B, C, H, W = x.shape
    return C % 4 == 0 and (H * W) % 4 == 0 and (C <= CL_MAX_C or not _is_cl(x))


class _TapBNReLUCL(torch.autograd.Function):
    """_TapBNReLU with an NHWC output: x = channel prefix of the NCHW feature buffer -> (x handed on, relu(bn(x)) channels-last);
    backward takes the NHWC gradient and adds dx into the NCHW gradient of the concatenation in place."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps, stats):
        lib = _lib.load()
        B, C, H, W = x.shape
        xs = x.detach()
        w, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        with torch.cuda.device(x.device):
            y = torch.empty((B, C, H, W), device=x.device, dtype=x.dtype, memory_format=_CL)
            saved = torch.empty(C, 2, device=x.device, dtype=torch.float32)
            pst, valid = _block_stats(lib, stats, x)
            ws = torch.empty(lib.aaconv_bn_relu_cl_workspace_bytes(B, C, H * W), device=x.device, dtype=torch.uint8)
            G, bpb = _stats_nchw(lib, xs, pst, valid)
            _lib.check(lib.aaconv_bn_relu_cl_forward(_ptr(xs), _DT[x.dtype], B, C, H * W, 0, xs.stride(0), _ptr(w), _ptr(b),
                                                     _ptr(running_mean), _ptr(running_var), float(momentum), float(eps), _ptr(y), _ptr(saved),
                                                     _ptr(ws), _ptr(pst), G, bpb, _stream()), 'aaconv_bn_relu_cl_forward')
        ctx.save_for_backward(xs, saved, w, b)
        return _alias(xs), y

    @staticmethod
    def backward(ctx, g_feats, dy):
        xs, saved, w, b = ctx.saved_tensors
        if dy is None:
            return g_feats, None, None, None, None, None, None, None
        lib = _lib.load()
        B, C, H, W = xs.shape
        g = dy.detach().to(xs.dtype).contiguous(memory_format=_CL)
        acc = _accumulates(g_feats, xs, aligned=True)
        with torch.cuda.device(xs.device):
            dx = g_feats if acc else torch.empty(B, C, H, W, device=xs.device, dtype=xs.dtype)
            dw, db = _grad_wb(ctx, xs)
            ws = torch.empty(lib.aaconv_bn_relu_cl_workspace_bytes(B, C, H * W), device=xs.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_cl_backward(_ptr(xs), _DT[xs.dtype], B, C, H * W, 0, xs.stride(0), _ptr(g), _ptr(saved), _ptr(w),
                                                      _ptr(b), _ptr(dx), dx.stride(0), int(acc), _ptr(dw), _ptr(db), _ptr(ws), _stream()),
                       'aaconv_bn_relu_cl_backward')
        if not acc and g_feats is not None:
            dx = dx + g_feats
        return dx, dw, db, None, None, None, None, None


class _BNReLUCL(torch.autograd.Function):
    """relu(bn(x)) for a channels-last x (the bottleneck between conv1 and conv2), channels-last out."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps):
        lib = _lib.load()
        B, C, H, W = x.shape
        xs = x.detach()
        w, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        with torch.cuda.device(x.device):
            y = torch.empty((B, C, H, W), device=x.device, dtype=x.dtype, memory_format=_CL)
            saved = torch.empty(C, 2, device=x.device, dtype=torch.float32)
            ws = torch.empty(lib.aaconv_bn_relu_cl_workspace_bytes(B, C, H * W), device=x.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_cl_forward(_ptr(xs), _DT[x.dtype], B, C, H * W, 1, C * H * W, _ptr(w), _ptr(b), _ptr(running_mean),
                                                     _ptr(running_var), float(momentum), float(eps), _ptr(y), _ptr(saved), _ptr(ws), None, 0, 0,
                                                     _stream()), 'aaconv_bn_relu_cl_forward')
        ctx.save_for_backward(xs, saved, w, b)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        xs, saved, w, b = ctx.saved_tensors
        B, C, H, W = xs.shape
        g = dy.detach().to(xs.dtype).contiguous(memory_format=_CL)
        with torch.cuda.device(xs.device):
            dx = torch.empty((B, C, H, W), device=xs.device, dtype=xs.dtype, memory_format=_CL) if ctx.needs_input_grad[0] else None
            dw, db = _grad_wb(ctx, xs)
            ws = torch.empty(lib.aaconv_bn_relu_cl_workspace_bytes(B, C, H * W), device=xs.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_cl_backward(_ptr(xs), _DT[xs.dtype], B, C, H * W, 1, C * H * W, _ptr(g), _ptr(saved), _ptr(w), _ptr(b),
                                                      _ptr(dx), C * H * W, 0, _ptr(dw), _ptr(db), _ptr(ws), _stream()),
                       'aaconv_bn_relu_cl_backward')
        return dx, dw, db, None, None, None, None


def tap_bn_relu_cl(bn, x, stats=None):
    _bump(bn)
    return _TapBNReLUCL.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.momentum, bn.eps, stats)


def bn_relu_cl(bn, x):
    _bump(bn)
    return _BNReLUCL.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.momentum, bn.eps)


# ------------------------------------------------------------------------------------------------
# eval mode (running statistics): aaconv_bn_relu_eval, inference only -- no autograd, no backward
# ------------------------------------------------------------------------------------------------
def eval_ok(bn, x):
    """relu(bn(x)) may run through bn_relu_eval: an eval-mode, affine BatchNorm2d with fp32 running statistics, a CUDA tensor in
    fp32 / bf16, and no autograd graph being recorded (the eval kernels have no backward)."""
    return not bn.training and not torch.is_grad_enabled() and _input_ok(x) and _module_ok(bn)


def eval_cl_ok(bn, x):
    """bn_relu_eval(bn, x, out_cl=True) is supported: C and H*W multiples of 4, x a channels-last tensor of at most CL_MAX_C channels
    or an NCHW tensor with dense samples, both aligned for four-element accesses."""
    if not eval_ok(bn, x):
        return False
    B, C, H, W = x.shape
    return (C % 4 == 0 and (H * W) % 4 == 0
            and ((_is_cl(x) and C <= CL_MAX_C and _aligned(x)) or _strided_ok(x, aligned=True)))


def bn_relu_eval(bn, x, out_cl=False):
    """relu(bn(x)) for an eval-mode nn.BatchNorm2d from its running statistics (which are read, never written; num_batches_tracked is
    not touched).  x: an NCHW tensor with dense samples (e.g. a channel prefix of the feature buffer) or a channels-last tensor;
    -> a new tensor, channels-last when `out_cl` (see eval_cl_ok for when that is supported), contiguous NCHW otherwise."""
    if not x.is_cuda:
        raise RuntimeError('fused_bn.bn_relu_eval runs on CUDA only; there is no CPU fallback')
    if not eval_ok(bn, x):
        raise RuntimeError('fused_bn.bn_relu_eval needs an eval-mode affine BatchNorm2d with fp32 parameters and running statistics, '
                           'an fp32 / bf16 4-d input with B <= 65535, and autograd off (the eval kernels have no backward)')
    if out_cl and not eval_cl_ok(bn, x):
        raise RuntimeError('fused_bn.bn_relu_eval: channels-last output needs C and H*W multiples of 4, four-element alignment and '
                           f'at most {CL_MAX_C} channels for a channels-last input')
    x_is_cl = not _strided_ok(x) and _is_cl(x)
    if not x_is_cl and not _strided_ok(x):
        x = x.contiguous()
    if x_is_cl and not out_cl:                 # no NHWC -> NCHW variant
        x, x_is_cl = x.contiguous(), False
    lib = _lib.load()
    B, C, H, W = x.shape
    w, b = bn.weight.detach(), bn.bias.detach()
    with torch.cuda.device(x.device):
        y = torch.empty((B, C, H, W), device=x.device, dtype=x.dtype, memory_format=_CL if out_cl else torch.contiguous_format)
        _lib.check(lib.aaconv_bn_relu_eval(_ptr(x), _DT[x.dtype], B, C, H * W, int(x_is_cl), C * H * W if x_is_cl else x.stride(0),
                                           _ptr(w), _ptr(b), _ptr(bn.running_mean), _ptr(bn.running_var), float(bn.eps), _ptr(y),
                                           int(out_cl), _stream()), 'aaconv_bn_relu_eval')
    return y


# ------------------------------------------------------------------------------------------------
# BatchNorm2d + ReLU + AvgPool2d(2) of torchvision's Transition (csrc/bn_cl.cu, pool_* kernels): the pool runs ahead of the 1x1
# convolution, on the channels-last operand the convolution reads
# ------------------------------------------------------------------------------------------------
def pool_ok(bn, x):
    """bn_relu_pool (bn training) / bn_relu_pool_eval (bn in eval mode, autograd off: see eval_ok) take x: a CUDA fp32 / bf16
    (B, C, H, W) tensor with dense samples (e.g. a dense block's feature buffer), C a multiple of 4, H and W >= 2, and x and its
    batch stride aligned for four-element accesses."""
    if not ((bn.training or not torch.is_grad_enabled()) and _input_ok(x) and _module_ok(bn) and _strided_ok(x, aligned=True)):
        return False
    B, C, H, W = x.shape
    return C % 4 == 0 and H >= 2 and W >= 2


class _BNReLUPool(torch.autograd.Function):
    """P = avgpool2(relu(bn(x))) channels-last (B, C, H // 2, W // 2) for a training-mode BatchNorm2d; backward takes dP
    channels-last and returns dx for every pixel of x."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, momentum, eps, stats):
        lib = _lib.load()
        B, C, H, W = x.shape
        xs = x.detach()
        w, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        with torch.cuda.device(x.device):
            y = torch.empty((B, C, H // 2, W // 2), device=x.device, dtype=x.dtype, memory_format=_CL)
            saved = torch.empty(C, 2, device=x.device, dtype=torch.float32)
            pst, valid = _block_stats(lib, stats, x)
            G, bpb = _stats_nchw(lib, xs, pst, valid)
            _lib.check(lib.aaconv_bn_relu_pool_forward(_ptr(xs), _DT[x.dtype], B, C, H, W, xs.stride(0), 1, _ptr(w), _ptr(b),
                                                       _ptr(running_mean), _ptr(running_var), float(momentum), float(eps), _ptr(y),
                                                       _ptr(saved), _ptr(pst), G, bpb, _stream()), 'aaconv_bn_relu_pool_forward')
        ctx.save_for_backward(xs, saved, w, b)
        return y

    @staticmethod
    def backward(ctx, dP):
        lib = _lib.load()
        xs, saved, w, b = ctx.saved_tensors
        B, C, H, W = xs.shape
        g = dP.detach().to(xs.dtype).contiguous(memory_format=_CL)
        with torch.cuda.device(xs.device):
            dx = torch.empty(B, C, H, W, device=xs.device, dtype=xs.dtype) if ctx.needs_input_grad[0] else None
            dw, db = _grad_wb(ctx, xs)
            ws = torch.empty(lib.aaconv_bn_relu_pool_workspace_bytes(B, C, H, W), device=xs.device, dtype=torch.uint8)
            _lib.check(lib.aaconv_bn_relu_pool_backward(_ptr(xs), _DT[xs.dtype], B, C, H, W, xs.stride(0), _ptr(g), _ptr(saved), _ptr(w),
                                                        _ptr(b), _ptr(dx), C * H * W, 0, _ptr(dw), _ptr(db), _ptr(ws), _stream()),
                       'aaconv_bn_relu_pool_backward')
        return dx, dw, db, None, None, None, None, None


def bn_relu_pool(bn, x, stats=None):
    """avgpool2(relu(bn(x))) as a channels-last (B, C, H // 2, W // 2) tensor for a training-mode nn.BatchNorm2d `bn` (batch statistics
    over all H x W pixels, running statistics and num_batches_tracked updated as the module does).  ``stats = (float32 buffer of
    >= 2*B*C elements, n_valid_channels)``: a dense block's shared plane statistics (see bn_relu).  See pool_ok for what x may be."""
    if not (bn.training and pool_ok(bn, x)):
        raise RuntimeError('fused_bn.bn_relu_pool needs a training-mode affine BatchNorm2d with fp32 parameters and running statistics '
                           'and a CUDA fp32 / bf16 input with dense samples, C a multiple of 4, H and W >= 2, aligned for four-element '
                           'accesses')
    _bump(bn)
    return _BNReLUPool.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.momentum, bn.eps, stats)


def bn_relu_pool_eval(bn, x):
    """bn_relu_pool for an eval-mode nn.BatchNorm2d under no_grad: the running statistics are read, never written; no backward."""
    if bn.training or not pool_ok(bn, x):
        raise RuntimeError('fused_bn.bn_relu_pool_eval needs an eval-mode affine BatchNorm2d with fp32 parameters and running '
                           'statistics, autograd off and a CUDA fp32 / bf16 input with dense samples, C a multiple of 4, H and W >= 2, '
                           'aligned for four-element accesses')
    lib = _lib.load()
    B, C, H, W = x.shape
    with torch.cuda.device(x.device):
        y = torch.empty((B, C, H // 2, W // 2), device=x.device, dtype=x.dtype, memory_format=_CL)
        _lib.check(lib.aaconv_bn_relu_pool_forward(_ptr(x), _DT[x.dtype], B, C, H, W, x.stride(0), 0, _ptr(bn.weight), _ptr(bn.bias),
                                                   _ptr(bn.running_mean), _ptr(bn.running_var), 0.0, float(bn.eps), _ptr(y), None, None,
                                                   0, 0, _stream()), 'aaconv_bn_relu_pool_forward')
    return y


def slice_layout(src, dst, to_nchw):
    """Channel-slice layout change through the C ABI: src NHWC dense -> dst NCHW (batch stride) when to_nchw, else the reverse."""
    lib = _lib.load()
    nchw, cl = (dst, src) if to_nchw else (src, dst)
    B, C, H, W = nchw.shape
    with torch.cuda.device(src.device):
        _lib.check(lib.aaconv_slice_layout(_ptr(src), _ptr(dst), _DT[src.dtype], B, C, H * W, nchw.stride(0), int(to_nchw), _stream()),
                   'aaconv_slice_layout')
    return dst
