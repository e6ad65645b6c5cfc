"""GPU parity: the CUDA path, called through the module / C ABI, against the oracle and the reference fixtures."""
import numpy as np
import os
import pytest
import torch

from oracle import aaconv_oracle as O
from tests.helpers import (FP32_TOL, GOLDEN, _bf16_grad_close, _bf16_output_close, _fp32_close, autocast_reference, golden_cases,
                           load_case, load_fixture, rel_err, rel_l2)

pytestmark = pytest.mark.gpu

def _module(s, p, precision):
    import chexpert_b200 as cb
    m = cb.AAConv2d(s.in_channels, s.out_channels, s.kernel_size, s.stride, s.dk, s.dv, s.nh, s.relative,
                    s.input_dims, precision=precision)
    m.load_state_dict({k: v.float() for k, v in p.items()}, strict=True)
    return m.cuda()


@pytest.mark.parametrize('name', golden_cases('f64'))
def test_fp32_matches_reference_fixture(name):
    s, p, g, t = load_case(name, 'f64')
    m = _module(s, p, 'fp32')
    x = t['x'].float().cuda().requires_grad_(True)
    y, w = m(x, return_attn=True)
    y.backward(t['dy'].float().cuda())
    _fp32_close(y, t['y'], 'y')
    _fp32_close(w, t['weights'], 'weights')
    _fp32_close(x.grad, g['x'], 'dx')
    for n, prm in m.named_parameters():
        _fp32_close(prm.grad, g[n], n)


@pytest.mark.parametrize('tag,shape,B,hin', [
    ('T3', O.AAConvShape(1024, 512, 3, 2, 160, 48, 8, True, (10, 10)), 2, 20),
    ('T2', O.AAConvShape(512, 256, 3, 2, 160, 24, 8, True, (20, 20)), 1, 40),
    ('T1', O.AAConvShape(256, 128, 3, 2, 160, 8, 8, True, (40, 40)), 1, 80),
])
def test_fp32_transition_shapes_vs_oracle(tag, shape, B, hin):
    p = O.init_params(shape, seed=0)
    g0 = torch.Generator().manual_seed(1)
    x = torch.relu(torch.randn(B, shape.in_channels, hin, hin, generator=g0))
    dy = torch.randn(B, shape.out_channels, *shape.input_dims, generator=g0)
    y_ref, g_ref = O.aaconv_backward_closed(x.double(), {k: v.double() for k, v in p.items()}, shape, dy.double())
    m = _module(shape, p, 'fp32')
    xc = x.cuda().requires_grad_(True)
    y = m(xc)
    y.backward(dy.cuda())
    _fp32_close(y, y_ref, 'y')
    _fp32_close(xc.grad, g_ref['x'], 'dx')
    for n, prm in m.named_parameters():
        _fp32_close(prm.grad, g_ref[n], n)


def test_weights_are_opt_in_and_rows_sum_to_one():
    s, p, g, t = load_case('nonsquare_s2', 'f64')
    m = _module(s, p, 'fp32')
    x = t['x'].float().cuda()
    with torch.no_grad():
        m(x)
        assert m.weights is None                      # never materialised by default
        m.store_weights = True
        m(x)
    B, nh = x.shape[0], s.nh
    H, W = s.input_dims
    assert m.weights.shape == (B, nh, H * W, H * W)
    # read contract of the visualise path (chexpert.py:383-387)
    v = m.weights.data[0].reshape(m.nh, H, W, H, W)
    assert torch.allclose(v.sum((-1, -2)), torch.ones(nh, H, W, device='cuda'), atol=1e-5)


def test_needs_input_grad_is_honoured():
    s, p, g, t = load_case('heads8_dkh20', 'f64')
    m = _module(s, p, 'fp32')
    for prm in m.parameters():
        prm.requires_grad_(False)
    m.key_rel_w.requires_grad_(True)
    x = t['x'].float().cuda()
    y = m(x)
    y.backward(t['dy'].float().cuda())
    assert m.in_proj_qkv.weight.grad is None and m.conv.weight.grad is None
    assert rel_err(m.key_rel_w.grad.cpu(), g['key_rel_w']) < FP32_TOL


def test_unsupported_bf16_shape_names_the_limit():
    """ADVICE r1: shapes outside the tensor-core kernels must fail with the real reason, not 'NULL buffer'."""
    import chexpert_b200 as cb
    m = cb.AAConv2d(16, 160, 3, 2, 16, 128, 8, False, (4, 4), precision='bf16').cuda()    # dv/nh = 16 > 14
    with pytest.raises(RuntimeError, match='dv/nh'):
        m(torch.randn(1, 16, 8, 8, device='cuda'))


def test_shape_mismatch_raises():
    import chexpert_b200 as cb
    m = cb.AAConv2d(8, 16, 3, 2, 8, 4, 2, True, (4, 4)).cuda()
    with pytest.raises(RuntimeError):
        m(torch.randn(1, 8, 10, 10, device='cuda'))    # 5x5 map vs input_dims 4x4
    with pytest.raises(RuntimeError):
        m(torch.randn(1, 7, 8, 8, device='cuda'))


def test_bce_kernel_matches_reference_fixture():
    import chexpert_b200 as cb
    z = np.load(os.path.join(GOLDEN, 'bce.npz'))
    zz = torch.from_numpy(z['z']).cuda().requires_grad_(True)
    t = torch.from_numpy(z['t']).cuda()
    el = cb.BCEWithLogitsLoss('none')(zz, t)
    assert torch.allclose(el.cpu(), torch.from_numpy(z['el']), rtol=1e-5, atol=2e-6)
    loss = cb.BCEWithLogitsLoss('train')(zz, t)
    loss.backward()
    assert torch.allclose(loss.cpu(), torch.from_numpy(z['loss']), rtol=1e-5)
    assert torch.allclose(zz.grad.cpu(), torch.from_numpy(z['gz']), rtol=1e-4, atol=1e-7)
    # reference usage: element losses then .sum(1).mean(0) through autograd  (chexpert.py:160)
    zz.grad = None
    cb.BCEWithLogitsLoss('none')(zz, t).sum(1).mean(0).backward()
    assert torch.allclose(zz.grad.cpu(), torch.from_numpy(z['gz']), rtol=1e-4, atol=1e-7)


def test_bce_raw_uones_labels():
    import chexpert_b200 as cb
    g = torch.Generator().manual_seed(3)
    raw = torch.tensor([float('nan'), -1.0, 0.0, 1.0])[torch.randint(0, 4, (16, 14), generator=g)]
    z = torch.randn(16, 5, generator=g)
    t = O.uones_targets(raw)
    want, _ = O.bce_train_loss(z, t)
    got = cb.BCEWithLogitsLoss('train', raw_labels=True)(z.cuda(), raw.cuda())
    assert torch.allclose(got.cpu(), want, rtol=1e-5)


def _bf16_case(s, p, x, dy, y_ref, g_ref, w_ref=None):
    m = _module(s, p, 'bf16')
    xc = x.float().cuda().requires_grad_(True)
    if w_ref is not None:
        y, w = m(xc, return_attn=True)
    else:
        y, w = m(xc), None
    y.backward(dy.float().cuda())
    ac = autocast_reference(s, p, x, dy)
    _bf16_output_close(y, y_ref, 'y', ac['y'])
    if w is not None:
        _bf16_output_close(w, w_ref, 'weights')
    _bf16_grad_close(xc.grad, g_ref['x'], ac['x'], 'dx')
    for n, prm in m.named_parameters():
        _bf16_grad_close(prm.grad, g_ref[n], ac[n], n)


@pytest.mark.parametrize('name', golden_cases('f64'))
def test_bf16_matches_reference_fixture(name):
    s, p, g, t = load_case(name, 'f64')
    _bf16_case(s, p, t['x'], t['dy'], t['y'], g, t['weights'])


@pytest.mark.parametrize('tag,shape,B,hin', [
    ('T3', O.AAConvShape(1024, 512, 3, 2, 160, 48, 8, True, (10, 10)), 4, 20),
    ('T2', O.AAConvShape(512, 256, 3, 2, 160, 24, 8, True, (20, 20)), 2, 40),
    ('T1', O.AAConvShape(256, 128, 3, 2, 160, 8, 8, True, (40, 40)), 1, 80),
])
def test_bf16_transition_shapes_vs_oracle(tag, shape, B, hin):
    p = O.init_params(shape, seed=0)
    g0 = torch.Generator().manual_seed(1)
    x = torch.relu(torch.randn(B, shape.in_channels, hin, hin, generator=g0))
    dy = torch.randn(B, shape.out_channels, *shape.input_dims, generator=g0)
    y_ref, g_ref = O.aaconv_backward_closed(x.double(), {k: v.double() for k, v in p.items()}, shape, dy.double())
    _bf16_case(shape, p, x, dy, y_ref, g_ref)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_L4096_vs_oracle(precision):
    """BASELINE config 4 (512-px input: Transition-1 attention over L = 64 x 64 = 4096 positions, key_rel_* 20 x 127) against the
    oracle evaluated one head at a time (oracle.aaconv_backward_closed_by_head, fp64; B = 1 and Cin = 64 bound the CPU time,
    the attention geometry -- 8 heads, dkh 20, dvh 1, 33 q-tiles x 64 key tiles per head -- is the full-size one).  Checks y, the
    returned attention map of the last head, dx and all five parameter gradients."""
    shape = O.AAConvShape(64, 128, 3, 2, 160, 8, 8, True, (64, 64))
    p = O.init_params(shape, seed=0)
    g0 = torch.Generator().manual_seed(1)
    x = torch.relu(torch.randn(1, 64, 128, 128, generator=g0))
    dy = torch.randn(1, 128, 64, 64, generator=g0)
    y_ref, g_ref, w_ref = O.aaconv_backward_closed_by_head(x.double(), {k: v.double() for k, v in p.items()}, shape, dy.double(),
                                                           return_weights_head=7)
    m = _module(shape, p, precision)
    xc = x.cuda().requires_grad_(True)
    y, w = m(xc, return_attn=True)
    y.backward(dy.cuda())
    assert w.shape == (1, 8, 4096, 4096)
    if precision == 'fp32':
        _fp32_close(y, y_ref, 'y')
        _fp32_close(w[:, 7], w_ref, 'weights[head 7]')
        _fp32_close(xc.grad, g_ref['x'], 'dx')
        for n, prm in m.named_parameters():
            _fp32_close(prm.grad, g_ref[n], n)
    else:
        ac = autocast_reference(shape, p, x, dy)
        _bf16_output_close(y, y_ref, 'y', ac['y'])
        _bf16_output_close(w[:, 7], w_ref, 'weights[head 7]')
        _bf16_grad_close(xc.grad, g_ref['x'], ac['x'], 'dx')
        for n, prm in m.named_parameters():
            _bf16_grad_close(prm.grad, g_ref[n], ac[n], n)


def test_full_size_T1_properties_bf16():
    """BASELINE size (B=16, 256ch, 80x80): size-independent properties instead of an O(L^2) oracle run --
    batch independence (sample b of the batched call == the same sample run alone, bit for bit: no cross-sample
    coupling, no atomics-order dependence) and linearity of backward in dy."""
    shape = O.AAConvShape(256, 128, 3, 2, 160, 8, 8, True, (40, 40))
    p = O.init_params(shape, seed=0)
    m = _module(shape, p, 'bf16')
    g0 = torch.Generator().manual_seed(5)
    x = torch.relu(torch.randn(16, 256, 80, 80, generator=g0)).cuda()
    dy = torch.randn(16, 128, 40, 40, generator=g0).cuda()
    xa = x.clone().requires_grad_(True)
    ya = m(xa)
    ya.backward(dy)
    gw = m.key_rel_w.grad.clone()
    m.zero_grad()
    xb = x[3:4].clone().requires_grad_(True)
    yb = m(xb)
    yb.backward(dy[3:4])
    assert torch.equal(ya[3:4], yb)
    assert torch.equal(xa.grad[3:4], xb.grad)
    assert torch.isfinite(ya).all() and torch.isfinite(xa.grad).all()
    m.zero_grad()
    xc = x.clone().requires_grad_(True)
    m(xc).backward(2.0 * dy)
    assert torch.allclose(xc.grad, 2.0 * xa.grad, rtol=1e-2, atol=1e-4)
    assert rel_err(m.key_rel_w.grad, 2.0 * gw) < 2e-2


@pytest.mark.parametrize('B,H', [(3, 48), (9, 24), (2, 64)])
def test_persistent_attention_kernels_many_items_per_cta(B, H):
    """The small-value-width attention kernels are persistent: one CTA walks several (batch, head, tile) items and keeps
    its barrier rings running across them.  Shapes with > 148 items and 1 / 2 / 3 operand atoms (H = 24 / 48 / 64),
    bf16 against the fp32 kernels (themselves gated against the oracle above): an item-boundary protocol error shows up
    as a launch failure or as garbage in the later items."""
    shape = O.AAConvShape(64, 64, 3, 2, 160, 8, 8, True, (H, H))
    p = O.init_params(shape, seed=3)
    g0 = torch.Generator().manual_seed(9)
    x = torch.relu(torch.randn(B, 64, 2 * H, 2 * H, generator=g0)).cuda()
    dy = torch.randn(B, 64, H, H, generator=g0).cuda()
    res = {}
    for precision in ('fp32', 'bf16'):
        m = _module(shape, p, precision)
        xc = x.clone().requires_grad_(True)
        y = m(xc)
        y.backward(dy)
        torch.cuda.synchronize()
        res[precision] = [y.detach(), xc.grad] + [q.grad for q in m.parameters()]
    for a, b in zip(res['bf16'], res['fp32']):
        assert torch.isfinite(a).all()
        assert rel_l2(a, b) < 3e-2, rel_l2(a, b)


def test_tiny_densenet_matches_reference_fixture():
    """Whole-model anchor: the reference DenseNet(16,(2,2,2,2),32, k=v=0.5) forward/backward on one batch
    (fixture written by oracle/gen_golden.py), fp32 kernels, strict state_dict load."""
    from chexpert_b200.densenet import DenseNet
    import chexpert_b200 as cb
    torch.backends.cudnn.allow_tf32 = False          # the dense blocks are torch/cuDNN: keep them in true fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    z = load_fixture('tiny_densenet')
    m = DenseNet(16, (2, 2, 2, 2), 32, num_classes=5,
                 attn_params={'k': 0.5, 'v': 0.5, 'nh': 8, 'relative': True, 'input_dims': (64, 64)}, precision='fp32')
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z if k.startswith('sd.')}
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    out = m(torch.from_numpy(z['x']).cuda())
    loss = cb.BCEWithLogitsLoss('train')(out, torch.from_numpy(z['t']).cuda())
    loss.backward()
    assert torch.allclose(out.cpu(), torch.from_numpy(z['out']), rtol=1e-3, atol=1e-4)
    assert torch.allclose(loss.cpu(), torch.from_numpy(z['loss']), rtol=1e-4)
    for k, prm in m.named_parameters():
        if 'g.' + k in z:
            assert rel_err(prm.grad.cpu(), torch.from_numpy(z['g.' + k])) < 2e-3, k


def test_train_step_cuda_graph_matches_eager():
    """chexpert_b200.train.TrainStep(cuda_graph=True) replays the captured forward / loss / backward / SGD step: the loss
    sequence must follow the eager one (same kernels, same order; cuDNN may pick another algorithm under capture)."""
    from chexpert_b200.train import TrainStep, synthetic_batch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    x, t = synthetic_batch(4, size=64, seed=5, device='cuda')
    losses = {}
    for mode in (False, True):
        ts = TrainStep('cuda', size=64, precision='fp32', lr=2e-4, cuda_graph=mode, seed=0)
        losses[mode] = torch.stack([ts(x, t) for _ in range(6)]).cpu()
        if mode:
            assert ts._graph is not None and ts.graph_launches > 0
    assert torch.isfinite(losses[True]).all()
    # cuDNN's backward kernels are not run-to-run deterministic and training amplifies the difference step by step
    assert torch.allclose(losses[True][:4], losses[False][:4], rtol=5e-3, atol=1e-3), (losses[True], losses[False])
    assert torch.allclose(losses[True], losses[False], rtol=3e-2, atol=1e-3), (losses[True], losses[False])
    assert float(losses[False][-1]) != float(losses[False][0])       # the steps really update the weights


def test_stress_512px_persistent_kernels_bitwise_stable():
    """VERDICT r1 #8: the persistent attention kernels keep hand-maintained mbarrier phase invariants across work items; a
    violated invariant shows up as an intermittent launch failure or garbage in later items.  200 forward + backward passes at
    the 512-px geometry (L = 4096: 33 query tiles x 8 heads x 2 images = 528 items on 148 CTAs, 3 operand atoms), every result
    bit-identical to the first."""
    shape = O.AAConvShape(64, 128, 3, 2, 160, 8, 8, True, (64, 64))
    p = O.init_params(shape, seed=2)
    m = _module(shape, p, 'bf16')
    g0 = torch.Generator().manual_seed(4)
    x = torch.relu(torch.randn(2, 64, 128, 128, generator=g0)).cuda().requires_grad_(True)
    dy = torch.randn(2, 128, 64, 64, generator=g0).cuda()
    first = None
    for it in range(200):
        m.zero_grad(set_to_none=True)
        x.grad = None
        y = m(x)
        y.backward(dy)
        cur = [y.detach(), x.grad] + [q.grad for q in m.parameters()]
        if first is None:
            torch.cuda.synchronize()
            first = [t.clone() for t in cur]
            assert all(torch.isfinite(t).all() for t in first)
        elif it % 20 == 19 or it == 199:
            for a, b in zip(cur, first):
                assert torch.equal(a, b), f'iteration {it}: result differs from the first pass'
    torch.cuda.synchronize()
