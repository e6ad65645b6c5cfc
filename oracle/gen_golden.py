"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (authoring container only).

Run:  PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden.py
Needs /root/reference (read-only).  The produced fixtures are committed; nothing on the GPU box
reads /root/reference.  Each fixture holds seeded inputs, parameters, the reference forward output,
the softmax weights the reference stashes on the module, and autograd gradients for dy.
"""
import json
import os
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, '/root/reference/models')
import attn_aug_conv as ref  # noqa: E402  (the reference itself)

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '..', 'tests', 'golden')

# name -> (B, Cin, Hin, Win, Cout, ksize, stride, dk, dv, nh, relative)
CASES = {
    'nonsquare_s2':   (2, 12, 10, 14, 24, 3, 2, 16, 8, 4, True),
    'square_s1_k1':   (1, 8, 6, 6, 16, 1, 1, 8, 4, 2, True),
    'norel_s2':       (2, 10, 8, 8, 20, 3, 2, 8, 4, 4, False),
    'heads8_dkh20':   (1, 32, 12, 12, 40, 3, 2, 160, 8, 8, True),
    'attn_only':      (1, 6, 8, 10, 8, 3, 2, 8, 8, 2, True),     # out_channels <= dv -> conv branch is None
    'dvh3_odd_in':    (2, 16, 9, 11, 48, 3, 2, 16, 24, 8, True),  # odd input extent, dvh = 3
}


def run_case(name, cfg, dtype):
    B, Cin, Hin, Win, Cout, ks, st, dk, dv, nh, rel = cfg
    H = (Hin - 1) // st + 1
    W = (Win - 1) // st + 1
    torch.manual_seed(sum(map(ord, name)))
    m = ref.AAConv2d(Cin, Cout, ks, st, dk, dv, nh, rel, (H, W))
    for mod in m.modules():
        if isinstance(mod, torch.nn.Conv2d):
            torch.nn.init.kaiming_normal_(mod.weight)
    m = m.to(dtype)
    x = torch.relu(torch.randn(B, Cin, Hin, Win, dtype=dtype)).requires_grad_(True)
    y = m(x)
    dy = torch.randn_like(y)
    y.backward(dy)
    rec = {'cfg': np.array([B, Cin, Hin, Win, Cout, ks, st, dk, dv, nh, int(rel)]),
           'x': x.detach().numpy(), 'dy': dy.numpy(), 'y': y.detach().numpy(),
           'weights': m.weights.detach().numpy(), 'gx': x.grad.numpy()}
    for n, p in m.named_parameters():
        rec['p.' + n] = p.detach().numpy()
        rec['g.' + n] = p.grad.numpy()
    return rec


def main():
    os.makedirs(OUT, exist_ok=True)
    for name, cfg in CASES.items():
        for dtype, tag in ((torch.float64, 'f64'), (torch.float32, 'f32')):
            rec = run_case(name, cfg, dtype)
            np.savez_compressed(os.path.join(OUT, f'aaconv_{name}_{tag}.npz'), **rec)
            print(name, tag, {k: v.shape for k, v in rec.items() if k in ('x', 'y', 'weights')})

    # rel_to_abs golden (attn_aug_conv.py:43-53) on a tiny tensor
    m = ref.AAConv2d(4, 8, 3, 1, 4, 4, 2, True, (3, 3))
    t = torch.arange(2 * 3 * 5 * 9, dtype=torch.float64).reshape(2, 3, 5, 9)
    np.savez_compressed(os.path.join(OUT, 'rel_to_abs.npz'), t=t.numpy(), out=m.rel_to_abs(t).numpy())

    # loss golden: nn.BCEWithLogitsLoss(reduction='none') + .sum(1).mean(0)   (chexpert.py:530,160)
    g = torch.Generator().manual_seed(7)
    z = (4 * torch.randn(16, 5, generator=g)).requires_grad_(True)
    z.data[0, 0] = 60.0
    z.data[1, 1] = -60.0
    t = (torch.rand(16, 5, generator=g) < 0.3).float()
    el = torch.nn.BCEWithLogitsLoss(reduction='none')(z, t)
    loss = el.sum(1).mean(0)
    loss.backward()
    np.savez_compressed(os.path.join(OUT, 'bce.npz'), z=z.detach().numpy(), t=t.numpy(), el=el.detach().numpy(),
                        loss=loss.detach().numpy(), gz=z.grad.numpy())

    # model-level anchors: state_dict keys/shapes + transition hyper-parameters + parameter count
    import contextlib
    import io
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        torch.manual_seed(0)
        net = ref.DenseNet(32, (6, 12, 24, 16), 64, num_classes=5,
                           attn_params={'k': 0.2, 'v': 0.1, 'nh': 8, 'relative': True, 'input_dims': (320, 320)})
    meta = {'n_params': sum(p.numel() for p in net.parameters()),
            'state_dict': {k: list(v.shape) for k, v in net.state_dict().items()},
            'transition_prints': buf.getvalue().strip().split('\n'),
            'transitions': {}}
    for i in (1, 2, 3):
        c = getattr(net.features, f'transition{i}').conv
        meta['transitions'][str(i)] = {'dk': c.dk, 'dv': c.dv, 'nh': c.nh, 'relative': c.relative,
                                       'key_rel_h': list(c.key_rel_h.shape), 'key_rel_w': list(c.key_rel_w.shape),
                                       'repr': c.extra_repr()}
    # tiny whole-model forward/backward anchor (64x64 input keeps the fixture small)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        tiny = ref.DenseNet(16, (2, 2, 2, 2), 32, num_classes=5,
                            attn_params={'k': 0.5, 'v': 0.5, 'nh': 8, 'relative': True, 'input_dims': (64, 64)})
    g = torch.Generator().manual_seed(1)
    xin = ((torch.rand(2, 1, 64, 64, generator=g) - 0.5330) / 0.0349).expand(-1, 3, -1, -1).contiguous()
    tgt = (torch.rand(2, 5, generator=g) < 0.3).float()
    tiny.train()
    out = tiny(xin)
    loss = torch.nn.BCEWithLogitsLoss(reduction='none')(out, tgt).sum(1).mean(0)
    loss.backward()
    rec = {'x': xin.numpy(), 't': tgt.numpy(), 'out': out.detach().numpy(), 'loss': loss.detach().numpy()}
    for k, v in tiny.named_parameters():
        if 'transition' in k or k.startswith('classifier'):
            rec['g.' + k] = v.grad.numpy()
    np.savez_compressed(os.path.join(OUT, 'tiny_densenet.npz'), **rec)
    # the state_dict is a second part so that no file exceeds 1 MB (tests/helpers.py: load_fixture)
    np.savez_compressed(os.path.join(OUT, 'tiny_densenet.part2.npz'), **{'sd.' + k: v.numpy() for k, v in tiny.state_dict().items()})
    with open(os.path.join(OUT, 'aadensenet121_meta.json'), 'w') as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print('n_params', meta['n_params'])


if __name__ == '__main__':
    main()
