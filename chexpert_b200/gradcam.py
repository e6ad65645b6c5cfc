"""Grad-CAM at features.norm5 on the device (the data part of grad_cam / visualize, chexpert.py:260-361; SURVEY.md section 2 row 9).

The head of both models is norm5 -> relu -> global average pool -> Linear, so the gradient of each logit with respect to the output
of model.features has a closed form, and Grad-CAM (Selvaraju et al. 2017) at that layer needs no backward pass.  One call of
aaconv_grad_cam (csrc/cam.cu) computes it from norm5's input X (the last dense block's output, e.g. its whole feature buffer):

    A = norm5(X) (eval mode),  m_k = #{p : A_k[p] > 0},  n = h * w
    cam[b, c] = relu(sum_k classifier.weight[c, k] * m_k / n^2 * A_k)              (B, K, h, w)
    up = F.interpolate(cam, (size, size), mode='bilinear', align_corners=False)      (B, K, size, size), when size is given

DenseNet.forward_grad_cam and evaluate.Predictor.grad_cam run it after the logits.  Colour maps, overlays and other plotting are
out of scope (DESIGN.md section 8).
"""
import torch

from . import _lib
from .aaconv import _ptr, _stream
from .fused_bn import _DT, _module_ok, _strided_ok


def grad_cam(x, norm5, classifier, size=None):
    """x: norm5's input, a CUDA fp32 / bf16 (B, C, h, w) tensor with dense samples (a batch stride wider than C*h*w is fine);
    norm5: the eval-mode nn.BatchNorm2d; classifier: the nn.Linear that follows the pool.  -> (cam, up): fp32 (B, K, h, w) and
    (B, K, size, size), up None without `size`.  There is no CPU fallback; the kernel's limits (C <= 4096, h*w <= 4096, K <= 64,
    size <= 4096) raise a RuntimeError that names them."""
    if not x.is_cuda:
        raise RuntimeError('gradcam.grad_cam runs on CUDA only; there is no CPU fallback')
    if x.dim() != 4 or x.dtype not in _DT or not _strided_ok(x):
        raise RuntimeError(f'gradcam.grad_cam takes an fp32 / bf16 (B, C, h, w) tensor with dense samples, got {x.dtype} '
                           f'{tuple(x.shape)} with strides {x.stride()}')
    B, C, h, w = x.shape
    if norm5.training or not _module_ok(norm5) or norm5.num_features != C or norm5.weight.device != x.device:
        raise RuntimeError(f'gradcam.grad_cam needs an eval-mode affine BatchNorm2d of {C} channels with fp32 parameters and running '
                           f'statistics on {x.device}')
    W = classifier.weight.detach()
    if W.dim() != 2 or W.shape[1] != C or W.dtype != torch.float32 or not W.is_contiguous() or W.device != x.device:
        raise RuntimeError(f'gradcam.grad_cam needs a classifier weight (K, {C}) fp32 contiguous on {x.device}, got {W.dtype} '
                           f'{tuple(W.shape)} on {W.device}')
    K = W.shape[0]
    if size is not None and (isinstance(size, bool) or not isinstance(size, int)):
        raise RuntimeError(f'gradcam.grad_cam: size must be an int or None, got {size!r}')
    lib = _lib.load()
    with torch.cuda.device(x.device):
        cam = torch.empty(B, K, h, w, device=x.device, dtype=torch.float32)
        up = None if size is None else torch.empty(B, K, size, size, device=x.device, dtype=torch.float32)
        ws = torch.empty(B * C, device=x.device, dtype=torch.int32)
        _lib.check(lib.aaconv_grad_cam(_ptr(x), _DT[x.dtype], B, C, h, w, x.stride(0), _ptr(norm5.weight), _ptr(norm5.bias),
                                       _ptr(norm5.running_mean), _ptr(norm5.running_var), float(norm5.eps), _ptr(W), K, _ptr(cam),
                                       _ptr(up), 0 if size is None else size, _ptr(ws), _stream()), 'aaconv_grad_cam')
    return cam, up
