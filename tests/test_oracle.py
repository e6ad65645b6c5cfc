"""The oracle vs the committed outputs of the reference module (tests/golden, made by oracle/gen_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import aaconv_oracle as O
from oracle import model_oracle as M
from tests.helpers import GOLDEN, golden_cases, load_case, load_fixture, rel_err


def test_rel_to_abs_matches_reference():
    z = np.load(os.path.join(GOLDEN, 'rel_to_abs.npz'))
    out = O.rel_to_abs_shift(torch.from_numpy(z['t']))
    assert torch.equal(out, torch.from_numpy(z['out']))
    # index law the CUDA kernels rely on: out[i, j] = t[i, j - i + L - 1]
    t = torch.from_numpy(z['t'])
    L = t.shape[2]
    for i in range(L):
        for j in range(L):
            assert torch.equal(out[..., i, j], t[..., i, j - i + L - 1])


@pytest.mark.parametrize('name', golden_cases('f64'))
def test_forward_f64(name):
    s, p, g, t = load_case(name, 'f64')
    y_seq, w_seq = O.aaconv_forward_sequential(t['x'], p, s, return_weights=True)
    y_cl, w_cl = O.aaconv_forward_closed(t['x'], p, s, return_weights=True)
    for y, w in ((y_seq, w_seq), (y_cl, w_cl)):
        assert rel_err(y, t['y']) < 1e-12
        assert rel_err(w, t['weights']) < 1e-12


@pytest.mark.parametrize('name', golden_cases('f64'))
def test_backward_f64(name):
    s, p, g, t = load_case(name, 'f64')
    _, g_cl = O.aaconv_backward_closed(t['x'], p, s, t['dy'])
    _, g_ad = O.aaconv_autograd(t['x'], p, s, t['dy'])
    assert set(g_cl) == set(g) == set(g_ad)
    for n in g:
        assert rel_err(g_cl[n], g[n]) < 1e-11, n
        assert rel_err(g_ad[n], g[n]) < 1e-11, n


@pytest.mark.parametrize('name', golden_cases('f64'))
def test_backward_by_head_f64(name):
    """The bounded-memory (one head at a time) adjoint used for the L = 4096 GPU test is the same function."""
    s, p, g, t = load_case(name, 'f64')
    y, g_h, w0 = O.aaconv_backward_closed_by_head(t['x'], p, s, t['dy'], return_weights_head=s.nh - 1)
    assert rel_err(y, t['y']) < 1e-12
    assert rel_err(w0, t['weights'][:, s.nh - 1]) < 1e-12
    assert set(g_h) == set(g)
    for n in g:
        assert rel_err(g_h[n], g[n]) < 1e-11, n


@pytest.mark.parametrize('name', golden_cases('f32'))
def test_forward_backward_f32(name):
    s, p, g, t = load_case(name, 'f32')
    y, g_ad = O.aaconv_autograd(t['x'], p, s, t['dy'])
    assert rel_err(y, t['y']) < 1e-5
    for n in g:
        assert rel_err(g_ad[n], g[n]) < 1e-4, n


def test_bce_golden():
    z = np.load(os.path.join(GOLDEN, 'bce.npz'))
    zz, t = torch.from_numpy(z['z']), torch.from_numpy(z['t'])
    el = O.bce_with_logits(zz, t)
    loss, gz = O.bce_train_loss(zz, t)
    # ATen's fp32 kernel loses relative precision on tiny element losses (cancellation; abs err ~4e-7);
    # the restated formula is closer to the fp64 value, so compare with an absolute floor.
    assert torch.allclose(el, torch.from_numpy(z['el']), rtol=1e-5, atol=2e-6)
    el64 = O.bce_with_logits(zz.double(), t.double())
    assert torch.allclose(el.double(), el64, rtol=1e-6, atol=1e-6)
    assert torch.allclose(loss, torch.from_numpy(z['loss']), rtol=1e-6)
    assert torch.allclose(gz, torch.from_numpy(z['gz']), rtol=1e-5, atol=1e-8)


def test_uones_selection():
    nan = float('nan')
    raw = torch.tensor([[0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13.],
                        [nan] * 14,
                        [-1.] * 14,
                        [1, nan, -1, 0, 1, 0, nan, 1, -1, 0, 1, nan, 0, 1]])
    t = O.uones_targets(raw)
    assert O.COMPETITION_INDEX == [8, 2, 6, 5, 10]
    assert t[0].tolist() == [8, 2, 6, 5, 10]
    assert t[1].tolist() == [0] * 5
    assert t[2].tolist() == [1] * 5
    assert t[3].tolist() == [1, 1, 0, 0, 1]


def test_transition_hyperparameters_and_flops():
    meta = json.load(open(os.path.join(GOLDEN, 'aadensenet121_meta.json')))
    attn = {'k': 0.2, 'v': 0.1, 'nh': 8, 'relative': True, 'input_dims': (80, 80)}
    want = {1: (160, 8, (40, 40)), 2: (160, 24, (20, 20)), 3: (160, 48, (10, 10))}
    dims = (80, 80)
    for i, cout in ((1, 128), (2, 256), (3, 512)):
        attn['input_dims'] = dims
        dk, dv, d = O.derive_transition_attn(cout, attn)
        assert (dk, dv, d) == want[i]
        assert meta['transitions'][str(i)]['dk'] == dk and meta['transitions'][str(i)]['dv'] == dv
        assert meta['transitions'][str(i)]['key_rel_h'] == [dk // 8, 2 * d[0] - 1]
        dims = d
    assert meta['n_params'] == 12534381
    # SURVEY.md section 8d table
    t1 = O.AAConvShape(256, 128, 3, 2, 160, 8, 8, True, (40, 40))
    t2 = O.AAConvShape(512, 256, 3, 2, 160, 24, 8, True, (20, 20))
    t3 = O.AAConvShape(1024, 512, 3, 2, 160, 48, 8, True, (10, 10))
    assert abs(O.algorithmic_flops_fwd(16, t1) / 1e9 - 33.515) < 2e-3
    assert abs(O.algorithmic_flops_fwd(16, t2) / 1e9 - 17.048) < 2e-3
    assert abs(O.algorithmic_flops_fwd(16, t3) / 1e9 - 14.983) < 2e-3


def test_ensemble_mean_and_auroc():
    g = torch.Generator().manual_seed(0)
    outs = [torch.randn(20, 5, generator=g) for _ in range(3)]
    m = O.ensemble_mean(outs)
    assert torch.allclose(m, (outs[0] + outs[1] + outs[2]) / 3, atol=1e-6)
    t = torch.zeros(20, 5)
    t[::2] = 1
    perfect = t * 2 - 1
    assert O.auroc_per_class(perfect, t) == [1.0] * 5


# The reference model (oracle/model_oracle.py) in float64 against the reference's own fp32 forward / backward of the tiny DenseNet.
# The fixture is fp32, so its rounding is the floor: measured 2.2e-6 (logits, of max), 4.4e-8 (loss) and 1.7e-5 (worst of the 17
# gradients, transition2.conv.key_rel_h, of its max).  The gates sit ~5x above those; a wrong wiring (a missed stem /4, a swapped
# dk / dv, a Transition without its InstanceNorm) moves the logits by O(1).
TINY_OUT_TOL, TINY_LOSS_TOL, TINY_GRAD_TOL = 1e-5, 2e-7, 1e-4


def test_reference_model_reproduces_the_tiny_densenet_fixture():
    z = load_fixture('tiny_densenet')
    m = M.RefDenseNet(16, (2, 2, 2, 2), 32, {'k': 0.5, 'v': 0.5, 'nh': 8, 'relative': True}, (64, 64))
    m.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith('sd.')}, strict=True)
    m = m.double().train()
    out = m(torch.from_numpy(z['x']).double())
    loss = O.bce_with_logits(out, torch.from_numpy(z['t']).double()).sum(1).mean(0)
    loss.backward()
    assert rel_err(out.detach(), torch.from_numpy(z['out'])) < TINY_OUT_TOL
    assert rel_err(loss.detach(), torch.from_numpy(z['loss'])) < TINY_LOSS_TOL
    grads = {k: p.grad for k, p in m.named_parameters()}
    names = [k[2:] for k in z if k.startswith('g.')]
    assert len(names) == 17 and set(names) <= set(grads)
    for k in names:
        assert rel_err(grads[k], torch.from_numpy(z['g.' + k])) < TINY_GRAD_TOL, k


def test_reference_aadensenet121_has_the_models_state_dict():
    """The 320-px reference and chexpert_b200's aadensenet121: the same state_dict keys in the same order, the shapes of the
    reference's own model (tests/golden/aadensenet121_meta.json), and strict loads both ways."""
    from chexpert_b200.densenet import aadensenet121
    meta = json.load(open(os.path.join(GOLDEN, 'aadensenet121_meta.json')))
    ref, ours = M.ref_aadensenet121((320, 320)).state_dict(), aadensenet121(5, (320, 320)).state_dict()
    assert list(ref) == list(ours) and set(ref) == set(meta['state_dict'])
    for k, v in ref.items():
        assert list(v.shape) == list(ours[k].shape) == meta['state_dict'][k], k
    assert sum(v.numel() for k, v in ref.items() if not k.endswith(('running_mean', 'running_var', 'num_batches_tracked'))) \
        == meta['n_params']
    M.ref_aadensenet121((320, 320)).load_state_dict(ours, strict=True)
    aadensenet121(5, (320, 320)).load_state_dict(ref, strict=True)
