"""Shared helpers for the parity tests (fixtures -> oracle shapes/params)."""
import glob
import os

import numpy as np
import torch

from oracle import aaconv_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
PARAM_NAMES = ('conv.weight', 'in_proj_qkv.weight', 'out_proj.weight', 'key_rel_h', 'key_rel_w')


def golden_cases(tag):
    return sorted(os.path.basename(f)[len('aaconv_'):-len(f'_{tag}.npz')]
                  for f in glob.glob(os.path.join(GOLDEN, f'aaconv_*_{tag}.npz')))


def load_fixture(stem):
    """tests/golden/<stem>.npz together with its parts <stem>.part*.npz -> {name: array}.  A fixture whose arrays would make one
    file larger than 1 MB is stored split across such parts; the arrays themselves are the generator's, unchanged."""
    z = {}
    for f in [os.path.join(GOLDEN, stem + '.npz')] + sorted(glob.glob(os.path.join(GOLDEN, stem + '.part*.npz'))):
        with np.load(f) as part:
            z.update((k, part[k]) for k in part.files)
    return z


def load_case(name, tag):
    z = np.load(os.path.join(GOLDEN, f'aaconv_{name}_{tag}.npz'))
    B, Cin, Hin, Win, Cout, ks, st, dk, dv, nh, rel = (int(v) for v in z['cfg'])
    H, W = (Hin - 1) // st + 1, (Win - 1) // st + 1
    shape = O.AAConvShape(Cin, Cout, ks, st, dk, dv, nh, bool(rel), (H, W))
    params = {n: torch.from_numpy(z['p.' + n]) for n in PARAM_NAMES if 'p.' + n in z.files}
    grads = {n: torch.from_numpy(z['g.' + n]) for n in PARAM_NAMES if 'g.' + n in z.files}
    grads['x'] = torch.from_numpy(z['gx'])
    t = {k: torch.from_numpy(z[k]) for k in ('x', 'dy', 'y', 'weights')}
    return shape, params, grads, t


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def autocast_reference(s, p, x, dy):
    """The reference op sequence (oracle port of attn_aug_conv.py:65-97) executed by PyTorch itself in bf16
    (torch.autocast) on the GPU: the calibration for what bf16 arithmetic can deliver on these inputs.
    -> dict with 'y', 'x' (grad) and the parameter-gradient names."""
    prm = {k: v.float().cuda().requires_grad_(True) for k, v in p.items()}
    xc = x.float().cuda().requires_grad_(True)
    with torch.autocast('cuda', dtype=torch.bfloat16):
        y = O.aaconv_forward_sequential(xc, prm, s)
    y.float().backward(dy.float().cuda())
    out = {'y': y.float().detach(), 'x': xc.grad}
    out.update({k: v.grad for k, v in prm.items()})
    return out
