"""Generate tests/golden/transition_*.npz by executing the UNMODIFIED reference `_Transition`
(InstanceNorm2d -> ReLU -> AAConv2d 3x3 stride 2; /root/reference/models/attn_aug_conv.py:409-446) in the authoring container.

Run:  PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden_transition.py
Each fixture holds a seeded PRE-norm input x (dense-block-like features: per-channel offsets and scales, both signs), the
parameters, the reference forward output, dy, and autograd's gradients for x and every parameter -- what the fused
InstanceNorm + ReLU prologue of chexpert_b200 (SURVEY.md section 8 row f1) is checked against.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, '/root/reference/models')
import attn_aug_conv as ref  # noqa: E402  (the reference itself)

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '..', 'tests', 'golden')

# name -> (B, Cin, Hin, Win, k, v)      Cout = Cin // 2 as in DenseNet (attn_aug_conv.py:485-488); nh = 8, relative
CASES = {
    'even16':    (2, 32, 16, 16, 0.5, 0.5),
    'nonsquare': (3, 64, 12, 20, 0.2, 0.25),
}


def run_case(name, cfg, dtype):
    B, Cin, Hin, Win, k, v = cfg
    torch.manual_seed(sum(map(ord, name)) + 17)
    attn = {'k': k, 'v': v, 'nh': 8, 'relative': True, 'input_dims': (Hin, Win)}
    with contextlib.redirect_stdout(io.StringIO()):
        m = ref._Transition(Cin, Cin // 2, attn)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Conv2d):
            torch.nn.init.kaiming_normal_(mod.weight)
    m = m.to(dtype)
    x = (torch.randn(B, Cin, Hin, Win, dtype=dtype) * (0.5 + torch.rand(1, Cin, 1, 1, dtype=dtype) * 2)
         + torch.randn(1, Cin, 1, 1, dtype=dtype)).requires_grad_(True)
    y = m(x)
    dy = torch.randn_like(y)
    y.backward(dy)
    c = m.conv
    rec = {'cfg': np.array([B, Cin, Hin, Win, Cin // 2, c.dk, c.dv, c.nh]), 'x': x.detach().numpy(), 'dy': dy.numpy(),
           'y': y.detach().numpy(), 'gx': x.grad.numpy()}
    for n, p in m.named_parameters():
        rec['p.' + n] = p.detach().numpy()
        rec['g.' + n] = p.grad.numpy()
    return rec


def main():
    for name, cfg in CASES.items():
        for dtype, tag in ((torch.float64, 'f64'),):
            rec = run_case(name, cfg, dtype)
            # the inputs (x, dy, parameters) go to a second part so that no file exceeds 1 MB (tests/helpers.py: load_fixture)
            inputs = {k: v for k, v in rec.items() if k in ('x', 'dy') or k.startswith('p.')}
            np.savez_compressed(os.path.join(OUT, f'transition_{name}_{tag}.npz'), **{k: v for k, v in rec.items() if k not in inputs})
            np.savez_compressed(os.path.join(OUT, f'transition_{name}_{tag}.part2.npz'), **inputs)
            print(name, tag, {k: v.shape for k, v in rec.items()})


if __name__ == '__main__':
    main()
