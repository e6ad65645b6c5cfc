"""CPU oracle for the AAConv2d hot path.  TEST INFRASTRUCTURE ONLY.

This file restates, on the CPU, the algorithm of the reference's attention-augmented
convolution and loss so that the CUDA path can be checked against it.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import it; the product package ``chexpert_b200`` never does.

Parity pinning: the reference ships no golden vectors or numeric tests for this path
(SURVEY.md section 4), so the oracle is pinned by differential execution against the reference
module itself: ``oracle/gen_golden.py`` imports ``/root/reference/models/attn_aug_conv.py``
(in the authoring container), runs it on seeded inputs and commits inputs/outputs/grads under
``tests/golden/``; ``tests/test_oracle.py`` checks every function below against those fixtures.

What each function follows (paths relative to /root/reference):

* ``derive_transition_attn``      models/attn_aug_conv.py:416-427
* ``out_hw``                      models/attn_aug_conv.py:34-35 (conv arithmetic of nn.Conv2d)
* ``rel_to_abs_shift``            models/attn_aug_conv.py:43-53
* ``relative_logits_axis``        models/attn_aug_conv.py:55-63
* ``aaconv_forward_sequential``   models/attn_aug_conv.py:65-97 (same op order; used as the CPU timing port)
* ``aaconv_forward_closed``       closed form of models/attn_aug_conv.py:75-86 (SURVEY.md section 8a, row a6)
* ``aaconv_backward_closed``      hand-derived adjoint of :65-97 (the reference relies on autograd)
* ``aaconv_backward_closed_by_head`` the same, one head at a time (bounded memory for L = 4096, BASELINE config 4)
* ``bce_with_logits``             chexpert.py:530,160 (train) and :205,144 (eval)
* ``uones_targets``               dataset.py:20-25,139,142
* ``ensemble_mean`` / ``auroc``   chexpert.py:233 and :130-135
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

# dataset.py:20-23 -- the 14 CSV label columns, and dataset.py:25 -- the 5 competition columns.
ALL_LABELS = ['No Finding', 'Enlarged Cardiomediastinum', 'Cardiomegaly', 'Lung Opacity', 'Lung Lesion',
              'Edema', 'Consolidation', 'Pneumonia', 'Atelectasis', 'Pneumothorax', 'Pleural Effusion',
              'Pleural Other', 'Fracture', 'Support Devices']
COMPETITION_LABELS = ['Atelectasis', 'Cardiomegaly', 'Consolidation', 'Edema', 'Pleural Effusion']
COMPETITION_INDEX = [ALL_LABELS.index(n) for n in COMPETITION_LABELS]  # [8, 2, 6, 5, 10]


@dataclass
class AAConvShape:
    """Static description of one AAConv2d instance (constructor arguments of attn_aug_conv.py:20)."""
    in_channels: int
    out_channels: int
    kernel_size: int
    stride: int
    dk: int
    dv: int
    nh: int
    relative: bool
    input_dims: tuple  # (H, W) of the OUTPUT (post-stride) map
    padding: int | None = None
    dilation: int = 1

    @property
    def dkh(self):
        return self.dk // self.nh

    @property
    def dvh(self):
        return self.dv // self.nh

    @property
    def pad(self):
        return self.padding if self.padding else self.kernel_size // 2


def derive_transition_attn(num_output_features: int, attn_params: dict):
    """dk, dv, input_dims of the AAConv2d inside a DenseNet transition (attn_aug_conv.py:416-427)."""
    nh = attn_params['nh']
    dk = max(20 * nh, int((attn_params['k'] * num_output_features // nh) * nh))
    dv = int((attn_params['v'] * num_output_features // nh) * nh)
    dims = attn_params['input_dims'][0] // 2, attn_params['input_dims'][1] // 2
    return dk, dv, dims


def out_hw(hin, win, k, stride, pad, dil=1):
    ho = (hin + 2 * pad - dil * (k - 1) - 1) // stride + 1
    wo = (win + 2 * pad - dil * (k - 1) - 1) // stride + 1
    return ho, wo


def init_params(shape: AAConvShape, seed: int = 0, dtype=torch.float32, kaiming: bool = True):
    """Parameters with the shapes of attn_aug_conv.py:34-41 and the init of :503-510 / :40-41."""
    g = torch.Generator().manual_seed(seed)
    s = shape
    p = {}

    def conv_w(co, ci, k):
        w = torch.randn(co, ci, k, k, generator=g, dtype=torch.float64)
        if kaiming:  # kaiming_normal_, fan_in, gain sqrt(2)
            w = w * math.sqrt(2.0 / (ci * k * k))
        else:       # nn.Conv2d default is kaiming_uniform(a=sqrt5); only the scale matters for tests
            w = w * math.sqrt(1.0 / (3 * ci * k * k))
        return w.to(dtype)

    if s.out_channels > s.dv:
        p['conv.weight'] = conv_w(s.out_channels - s.dv, s.in_channels, s.kernel_size)
    p['in_proj_qkv.weight'] = conv_w(2 * s.dk + s.dv, s.in_channels, 1)
    p['out_proj.weight'] = conv_w(s.dv, s.dv, 1)
    if s.relative:
        H, W = s.input_dims
        p['key_rel_h'] = (s.dk ** -0.5 + torch.randn(s.dkh, 2 * H - 1, generator=g, dtype=torch.float64)).to(dtype)
        p['key_rel_w'] = (s.dk ** -0.5 + torch.randn(s.dkh, 2 * W - 1, generator=g, dtype=torch.float64)).to(dtype)
    return p


# ----------------------------------------------------------------------------------------------
# sequential restatement (op order of the reference forward; autograd-capable; CPU timing port)
# ----------------------------------------------------------------------------------------------

def rel_to_abs_shift(t):
    """(B, G, L, 2L-1) relative-indexed -> (B, G, L, L) absolute-indexed: out[i, j] = t[i, j - i + L - 1].

    Same skewing device as attn_aug_conv.py:43-53: append one column, flatten the last two axes,
    append L-1 more entries, refold with rows of length 2L-1 and keep the top-right L x L block.
    """
    B, G, L, _ = t.shape
    t = F.pad(t, (0, 1)).flatten(2)
    t = F.pad(t, (0, L - 1)).reshape(B, G, L + 1, 2 * L - 1)
    return t[:, :, :L, L - 1:]


def relative_logits_axis(q, rel_k):
    """q (B, nh, A, Lx, dkh), rel_k (dkh, 2Lx-1) -> (B, nh, A, A', Lx, Lx) broadcast over A' (:55-63)."""
    B, nh, A, Lx, _ = q.shape
    r = torch.matmul(q, rel_k).reshape(B, nh * A, Lx, 2 * Lx - 1)
    r = rel_to_abs_shift(r)
    return r.reshape(B, nh, A, 1, Lx, Lx).expand(-1, -1, -1, A, -1, -1)


def aaconv_forward_sequential(x, p, s: AAConvShape, return_weights=False):
    """Forward in the reference's op order (attn_aug_conv.py:65-97).  Differentiable by autograd."""
    qkv = F.conv2d(x, p['in_proj_qkv.weight'], stride=s.stride)
    q, k, v = qkv.split([s.dk, s.dk, s.dv], dim=1)
    B, _, H, W = qkv.shape
    fq = q.reshape(B, s.nh, s.dkh, H * W) * s.dkh ** -0.5
    fk = k.reshape(B, s.nh, s.dkh, H * W)
    fv = v.reshape(B, s.nh, s.dvh, H * W)
    logits = torch.matmul(fq.transpose(2, 3), fk)
    if s.relative:
        q5 = fq.reshape(B, s.nh, s.dkh, H, W).permute(0, 1, 3, 4, 2)
        wl = relative_logits_axis(q5, p['key_rel_w'])
        hl = relative_logits_axis(q5.transpose(2, 3), p['key_rel_h'])
        wl = wl.permute(0, 1, 2, 4, 3, 5).reshape(B, s.nh, H * W, H * W)
        hl = hl.permute(0, 1, 4, 2, 5, 3).reshape(B, s.nh, H * W, H * W)
        logits = logits + (hl + wl)
    weights = F.softmax(logits, -1)
    a = torch.matmul(weights, fv.transpose(2, 3)).transpose(2, 3).reshape(B, -1, H, W)
    a = F.conv2d(a, p['out_proj.weight'])
    if 'conv.weight' in p:
        c = F.conv2d(x, p['conv.weight'], stride=s.stride, padding=s.pad, dilation=s.dilation)
        a = torch.cat([c, a], dim=1)
    return (a, weights) if return_weights else a


# ----------------------------------------------------------------------------------------------
# closed form (fp64 tie-breaker) and explicit backward
# ----------------------------------------------------------------------------------------------

def _project_qkv(x, p, s):
    xs = x[:, :, ::s.stride, ::s.stride]
    B, _, H, W = xs.shape
    qkv = torch.einsum('oc,bchw->bohw', p['in_proj_qkv.weight'][:, :, 0, 0], xs)
    q = qkv[:, :s.dk].reshape(B, s.nh, s.dkh, H * W) * s.dkh ** -0.5
    k = qkv[:, s.dk:2 * s.dk].reshape(B, s.nh, s.dkh, H * W)
    v = qkv[:, 2 * s.dk:].reshape(B, s.nh, s.dvh, H * W)
    return xs, q, k, v, H, W


def _rel_index(n, device):
    i = torch.arange(n, device=device)
    return i[None, :] - i[:, None] + n - 1  # [query coord, key coord] -> relative slot


def closed_logits(q, k, p, s, H, W):
    """logit[b,n,(y,x),(y',x')] = q.k + q.key_rel_w[:, x'-x+W-1] + q.key_rel_h[:, y'-y+H-1]."""
    B = q.shape[0]
    logits = torch.einsum('bndq,bndk->bnqk', q, k)
    if s.relative:
        rw = torch.einsum('bndq,dr->bnqr', q, p['key_rel_w']).reshape(B, s.nh, H, W, 2 * W - 1)
        rh = torch.einsum('bndq,dr->bnqr', q, p['key_rel_h']).reshape(B, s.nh, H, W, 2 * H - 1)
        ix = _rel_index(W, q.device)  # [x, x']
        iy = _rel_index(H, q.device)  # [y, y']
        aw = torch.gather(rw, 4, ix[None, None, None].expand(B, s.nh, H, W, W))      # [b,n,y,x,x']
        ah = torch.gather(rh, 4, iy[None, None, :, None, :].expand(B, s.nh, H, W, H))  # [b,n,y,x,y']
        logits = logits.reshape(B, s.nh, H, W, H, W) + aw[:, :, :, :, None, :] + ah[:, :, :, :, :, None]
        logits = logits.reshape(B, s.nh, H * W, H * W)
    return logits


def aaconv_forward_closed(x, p, s: AAConvShape, return_weights=False, return_state=False):
    xs, q, k, v, H, W = _project_qkv(x, p, s)
    B = x.shape[0]
    P = torch.softmax(closed_logits(q, k, p, s, H, W), dim=-1)
    O = torch.einsum('bnqk,bndk->bndq', P, v)                 # per-head attention output
    pre = O.reshape(B, s.dv, H, W)
    a = torch.einsum('oc,bchw->bohw', p['out_proj.weight'][:, :, 0, 0], pre)
    if 'conv.weight' in p:
        c = F.conv2d(x, p['conv.weight'], stride=s.stride, padding=s.pad, dilation=s.dilation)
        a = torch.cat([c, a], dim=1)
    if return_state:
        return a, dict(xs=xs, q=q, k=k, v=v, P=P, O=O, H=H, W=W)
    return (a, P) if return_weights else a


def aaconv_backward_closed(x, p, s: AAConvShape, dy):
    """Explicit adjoint (SURVEY.md section 8a 'Backward contract').  Returns dict of grads."""
    y, st = aaconv_forward_closed(x, p, s, return_state=True)
    xs, q, k, v, P, O, H, W = (st[n] for n in ('xs', 'q', 'k', 'v', 'P', 'O', 'H', 'W'))
    B = x.shape[0]
    g = {}
    nconv = s.out_channels - s.dv if 'conv.weight' in p else 0
    dya = dy[:, nconv:]
    Wo = p['out_proj.weight'][:, :, 0, 0]
    g['out_proj.weight'] = torch.einsum('bohw,bchw->oc', dya, O.reshape(B, s.dv, H, W))[:, :, None, None]
    dO = torch.einsum('oc,bohw->bchw', Wo, dya).reshape(B, s.nh, s.dvh, H * W)
    dV = torch.einsum('bnqk,bndq->bndk', P, dO)
    dP = torch.einsum('bndq,bndk->bnqk', dO, v)
    delta = (dP * P).sum(-1, keepdim=True)
    dS = P * (dP - delta)
    dq = torch.einsum('bnqk,bndk->bndq', dS, k)
    dk = torch.einsum('bnqk,bndq->bndk', dS, q)
    if s.relative:
        dS6 = dS.reshape(B, s.nh, H, W, H, W)
        dAw = dS6.sum(4)                              # [b,n,y,x,x']  summed over key rows
        dAh = dS6.sum(5)                              # [b,n,y,x,y']  summed over key columns
        ix = _rel_index(W, x.device)
        iy = _rel_index(H, x.device)
        dRw = torch.zeros(B, s.nh, H, W, 2 * W - 1, dtype=x.dtype, device=x.device).scatter_add_(
            4, ix[None, None, None].expand(B, s.nh, H, W, W), dAw)
        dRh = torch.zeros(B, s.nh, H, W, 2 * H - 1, dtype=x.dtype, device=x.device).scatter_add_(
            4, iy[None, None, :, None, :].expand(B, s.nh, H, W, H), dAh)
        dRw = dRw.reshape(B, s.nh, H * W, -1)
        dRh = dRh.reshape(B, s.nh, H * W, -1)
        g['key_rel_w'] = torch.einsum('bndq,bnqr->dr', q, dRw)
        g['key_rel_h'] = torch.einsum('bndq,bnqr->dr', q, dRh)
        dq = dq + torch.einsum('dr,bnqr->bndq', p['key_rel_w'], dRw) + torch.einsum('dr,bnqr->bndq', p['key_rel_h'], dRh)
    dqkv = torch.cat([(dq * s.dkh ** -0.5).reshape(B, s.dk, H, W), dk.reshape(B, s.dk, H, W),
                      dV.reshape(B, s.dv, H, W)], dim=1)
    g['in_proj_qkv.weight'] = torch.einsum('bohw,bchw->oc', dqkv, xs)[:, :, None, None]
    dx = torch.zeros_like(x)
    dx[:, :, ::s.stride, ::s.stride] += torch.einsum('oc,bohw->bchw', p['in_proj_qkv.weight'][:, :, 0, 0], dqkv)
    if nconv:
        dyc = dy[:, :nconv]
        g['conv.weight'] = torch.nn.grad.conv2d_weight(x, p['conv.weight'].shape, dyc, stride=s.stride,
                                                       padding=s.pad, dilation=s.dilation)
        dx = dx + torch.nn.grad.conv2d_input(x.shape, p['conv.weight'], dyc, stride=s.stride,
                                             padding=s.pad, dilation=s.dilation)
    g['x'] = dx
    return y, g


def aaconv_backward_closed_by_head(x, p, s: AAConvShape, dy, return_weights_head=None):
    """Same adjoint as ``aaconv_backward_closed`` evaluated one head at a time, so that only one (B, L, L) block of
    logits / probabilities / dS is alive at once: the L = 4096 case (512-px Transition 1, BASELINE config 4) then needs
    ~1 GB per block in fp64 instead of 8 x that.  Returns (y, grads[, P of head `return_weights_head`])."""
    xs, q, k, v, H, W = _project_qkv(x, p, s)
    B, L = x.shape[0], H * W
    nconv = s.out_channels - s.dv if 'conv.weight' in p else 0
    Wo = p['out_proj.weight'][:, :, 0, 0]
    dya = dy[:, nconv:]
    dO_all = torch.einsum('oc,bohw->bchw', Wo, dya).reshape(B, s.nh, s.dvh, L)
    O = torch.zeros(B, s.nh, s.dvh, L, dtype=x.dtype, device=x.device)
    dq, dk, dV = torch.zeros_like(q), torch.zeros_like(k), torch.zeros_like(v)
    g = {}
    if s.relative:
        g['key_rel_w'] = torch.zeros_like(p['key_rel_w'])
        g['key_rel_h'] = torch.zeros_like(p['key_rel_h'])
        ix, iy = _rel_index(W, x.device), _rel_index(H, x.device)
    keep = None
    one = AAConvShape(s.in_channels, s.out_channels, s.kernel_size, s.stride, s.dkh, s.dvh, 1, s.relative, s.input_dims,
                      s.padding, s.dilation)
    for n in range(s.nh):
        qn, kn, vn, dOn = q[:, n:n + 1], k[:, n:n + 1], v[:, n:n + 1], dO_all[:, n:n + 1]
        P = torch.softmax(closed_logits(qn, kn, p, one, H, W), dim=-1)
        if return_weights_head == n:
            keep = P[:, 0].clone()
        O[:, n:n + 1] = torch.einsum('bnqk,bndk->bndq', P, vn)
        dV[:, n:n + 1] = torch.einsum('bnqk,bndq->bndk', P, dOn)
        dP = torch.einsum('bndq,bndk->bnqk', dOn, vn)
        dS = P * (dP - (dP * P).sum(-1, keepdim=True))
        del dP
        dqn = torch.einsum('bnqk,bndk->bndq', dS, kn)
        dk[:, n:n + 1] = torch.einsum('bnqk,bndq->bndk', dS, qn)
        if s.relative:
            dS6 = dS.reshape(B, 1, H, W, H, W)
            dAw, dAh = dS6.sum(4), dS6.sum(5)
            dRw = torch.zeros(B, 1, H, W, 2 * W - 1, dtype=x.dtype, device=x.device).scatter_add_(4, ix[None, None, None].expand(B, 1, H, W, W), dAw)
            dRh = torch.zeros(B, 1, H, W, 2 * H - 1, dtype=x.dtype, device=x.device).scatter_add_(
                4, iy[None, None, :, None, :].expand(B, 1, H, W, H), dAh)
            dRw, dRh = dRw.reshape(B, 1, L, -1), dRh.reshape(B, 1, L, -1)
            g['key_rel_w'] += torch.einsum('bndq,bnqr->dr', qn, dRw)
            g['key_rel_h'] += torch.einsum('bndq,bnqr->dr', qn, dRh)
            dqn = dqn + torch.einsum('dr,bnqr->bndq', p['key_rel_w'], dRw) + torch.einsum('dr,bnqr->bndq', p['key_rel_h'], dRh)
        dq[:, n:n + 1] = dqn
        del dS, P
    a = torch.einsum('oc,bchw->bohw', Wo, O.reshape(B, s.dv, H, W))
    g['out_proj.weight'] = torch.einsum('bohw,bchw->oc', dya, O.reshape(B, s.dv, H, W))[:, :, None, None]
    dqkv = torch.cat([(dq * s.dkh ** -0.5).reshape(B, s.dk, H, W), dk.reshape(B, s.dk, H, W), dV.reshape(B, s.dv, H, W)], dim=1)
    g['in_proj_qkv.weight'] = torch.einsum('bohw,bchw->oc', dqkv, xs)[:, :, None, None]
    dx = torch.zeros_like(x)
    dx[:, :, ::s.stride, ::s.stride] += torch.einsum('oc,bohw->bchw', p['in_proj_qkv.weight'][:, :, 0, 0], dqkv)
    if nconv:
        dyc = dy[:, :nconv]
        c = F.conv2d(x, p['conv.weight'], stride=s.stride, padding=s.pad, dilation=s.dilation)
        a = torch.cat([c, a], dim=1)
        g['conv.weight'] = torch.nn.grad.conv2d_weight(x, p['conv.weight'].shape, dyc, stride=s.stride, padding=s.pad,
                                                       dilation=s.dilation)
        dx = dx + torch.nn.grad.conv2d_input(x.shape, p['conv.weight'], dyc, stride=s.stride, padding=s.pad, dilation=s.dilation)
    g['x'] = dx
    return (a, g, keep) if return_weights_head is not None else (a, g)


def aaconv_autograd(x, p, s: AAConvShape, dy, fn=aaconv_forward_sequential):
    """Forward + autograd backward of ``fn``; returns (y, grads) with the same keys as the closed form."""
    x = x.detach().clone().requires_grad_(True)
    pp = {n: t.detach().clone().requires_grad_(True) for n, t in p.items()}
    y = fn(x, pp, s)
    y.backward(dy)
    g = {n: t.grad for n, t in pp.items()}
    g['x'] = x.grad
    return y.detach(), g


class SequentialAAConv2d(torch.nn.Module):
    """nn.Module wrapper over ``aaconv_forward_sequential`` -- the timed CPU port of the reference module."""

    def __init__(self, shape: AAConvShape, params: dict):
        super().__init__()
        self.shape = shape
        self.params_ = torch.nn.ParameterDict({n.replace('.', '__'): torch.nn.Parameter(t.clone()) for n, t in params.items()})

    def forward(self, x):
        p = {n.replace('__', '.'): t for n, t in self.params_.items()}
        return aaconv_forward_sequential(x, p, self.shape)


# ----------------------------------------------------------------------------------------------
# loss, labels, metrics
# ----------------------------------------------------------------------------------------------

def bce_with_logits(z, t):
    """Element losses (B, C) = max(z,0) - z t + log1p(exp(-|z|))  (nn.BCEWithLogitsLoss(reduction='none'))."""
    return torch.clamp(z, min=0) - z * t + torch.log1p(torch.exp(-z.abs()))


def bce_train_loss(z, t):
    """chexpert.py:160 -- sum over classes, mean over batch.  Returns (loss, dloss/dz)."""
    el = bce_with_logits(z, t)
    return el.sum(1).mean(0), (torch.sigmoid(z) - t) / z.shape[0]


def uones_targets(raw14):
    """Raw CheXpert labels (N,14) in {nan,-1,0,1} -> (N,5) float targets: blank->0 (dataset.py:139),
    uncertain -1 -> 1 (dataset.py:142), competition columns in the order of dataset.py:25."""
    t = torch.as_tensor(raw14, dtype=torch.float32)[:, COMPETITION_INDEX].clone()
    t[torch.isnan(t)] = 0.0
    t[t == -1] = 1.0
    return t


def ensemble_mean(list_of_logits):
    """chexpert.py:233 -- mean of raw logits over checkpoints."""
    return torch.stack(list_of_logits, dim=2).mean(2)


def auroc_per_class(logits, targets):
    """chexpert.py:130-135 -- sklearn roc_curve + auc per class on raw logits."""
    from sklearn.metrics import roc_curve, auc
    out = []
    for i in range(logits.shape[1]):
        fpr, tpr, _ = roc_curve(np.asarray(targets[:, i]), np.asarray(logits[:, i]))
        out.append(float(auc(fpr, tpr)))
    return out


# ----------------------------------------------------------------------------------------------
# work model (SURVEY.md section 8d)
# ----------------------------------------------------------------------------------------------

def algorithmic_flops_fwd(B, s: AAConvShape):
    H, W = s.input_dims
    L = H * W
    nconv = max(s.out_channels - s.dv, 0)
    dense = 2 * B * L * (s.kernel_size ** 2 * s.in_channels * nconv + s.in_channels * (2 * s.dk + s.dv) + s.dv ** 2)
    rel = s.dkh * ((2 * W - 1) + (2 * H - 1)) if s.relative else 0
    attn = 2 * B * s.nh * L * (L * s.dkh + rel + L * s.dvh)
    return dense + attn
