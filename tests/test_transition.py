"""SURVEY.md section 8 rows f1 / f3 and the typed boundary:
  * the fused InstanceNorm2d + ReLU prologue (and its fused adjoint) against fixtures written by the UNMODIFIED reference
    `_Transition` (models/attn_aug_conv.py:409-446; oracle/gen_golden_transition.py),
  * the pre-allocated DenseBlock feature buffer against torchvision's `_DenseBlock` (CPU) and the AAConv2d epilogue writing
    straight into it (`out_total`),
  * bf16 activations at the boundary (x / dx / y in bf16, as under autocast) against the fp32 boundary.
"""
import glob
import os

import pytest
import torch

from tests.helpers import GOLDEN, load_fixture, rel_err, rel_l2

CASES = sorted(os.path.basename(f)[len('transition_'):-len('_f64.npz')] for f in glob.glob(os.path.join(GOLDEN, 'transition_*_f64.npz')))


def _load(name):
    z = load_fixture(f'transition_{name}_f64')
    B, Cin, Hin, Win, Cout, dk, dv, nh = (int(v) for v in z['cfg'])
    return z, (B, Cin, Hin, Win, Cout, dk, dv, nh)


def _transition(z, cfg, precision, fused):
    from chexpert_b200.densenet import AATransition
    B, Cin, Hin, Win, Cout, dk, dv, nh = cfg
    # k, v chosen by the fixture generator are recovered from dk / dv only through the module's own derivation: build directly
    attn = {'k': 0.0, 'v': dv / Cout, 'nh': nh, 'relative': True, 'input_dims': (Hin, Win)}
    m = AATransition(Cin, Cout, attn, precision=precision, fused_prologue=fused)
    assert (m.conv.dk, m.conv.dv) == (dk, dv)
    sd = {k[2:]: torch.from_numpy(z[k]).float() for k in z if k.startswith('p.')}
    m.load_state_dict(sd, strict=True)        # same keys as the reference _Transition: conv.conv.weight, conv.key_rel_h, ...
    return m.cuda()


# ------------------------------------------------------------------------------------------------ CPU
def test_buffered_dense_block_equals_torchvision_block():
    from torchvision.models.densenet import _DenseBlock
    from chexpert_b200.densenet import BufferedDenseBlock
    torch.manual_seed(0)
    a = _DenseBlock(4, 16, 4, 8, 0.0)
    b = BufferedDenseBlock(4, 16, 4, 8, 0.0)
    assert list(a.state_dict()) == list(b.state_dict())
    b.load_state_dict(a.state_dict(), strict=True)
    x = torch.randn(3, 16, 9, 7)
    for train in (True, False):
        a.train(train), b.train(train)
        xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        ya, yb = a(xa), b(xb)
        assert yb.is_contiguous() and yb.shape == ya.shape
        assert torch.allclose(ya, yb, rtol=1e-5, atol=1e-6)
        g = torch.randn_like(ya)
        a.zero_grad(), b.zero_grad()
        ya.backward(g), yb.backward(g)
        assert torch.allclose(xa.grad, xb.grad, rtol=1e-4, atol=1e-5)
        for (n, p), (_, q) in zip(a.named_parameters(), b.named_parameters()):
            assert rel_err(q.grad, p.grad) < 1e-5, n


def test_buffered_block_adopts_a_producer_buffer_without_copy():
    from chexpert_b200.densenet import BufferedDenseBlock
    torch.manual_seed(1)
    b = BufferedDenseBlock(2, 8, 4, 4, 0.0).eval()
    buf = torch.zeros(2, 16, 5, 5)
    init = buf[:, :8]
    init.copy_(torch.randn(2, 8, 5, 5))
    init.feature_buffer = buf
    with torch.no_grad():
        out = b(init)
    assert out.data_ptr() == buf.data_ptr()                        # the block worked inside the producer's buffer
    with torch.no_grad():
        want = b(init.clone())                                     # no buffer attached: allocates and copies
    assert torch.equal(out, want)


def test_model_options_keep_state_dict_and_function():
    from chexpert_b200.densenet import DenseNet
    kw = dict(growth_rate=8, block_config=(2, 2), num_init_features=16, num_classes=5, attn_params=None)
    torch.manual_seed(0)
    a = DenseNet(**kw)
    torch.manual_seed(0)
    b = DenseNet(feature_buffer=True, **kw)
    assert list(a.state_dict()) == list(b.state_dict())
    b.load_state_dict(a.state_dict(), strict=True)
    x = torch.randn(2, 3, 16, 16)
    assert torch.allclose(a(x), b(x), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize('name', CASES)
@pytest.mark.parametrize('fused', [False, True])
def test_transition_fp32_matches_reference_fixture(name, fused):
    z, cfg = _load(name)
    m = _transition(z, cfg, 'fp32', fused)
    x = torch.from_numpy(z['x']).float().cuda().requires_grad_(True)
    y = m(x)
    y.backward(torch.from_numpy(z['dy']).float().cuda())
    tol = 1e-4
    assert rel_err(y.detach().cpu(), torch.from_numpy(z['y'])) < tol
    assert rel_err(x.grad.cpu(), torch.from_numpy(z['gx'])) < tol
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu(), torch.from_numpy(z['g.' + n])) < tol, n


@pytest.mark.gpu
@pytest.mark.parametrize('name', CASES)
@pytest.mark.parametrize('io', ['fp32', 'bf16'])
def test_transition_fused_bf16_matches_reference_fixture(name, io):
    """bf16 tensor-core mode with the fused prologue; io = bf16 feeds bf16 activations (as under autocast): x / dx / y in bf16."""
    z, cfg = _load(name)
    m = _transition(z, cfg, 'bf16', True)
    dt = torch.bfloat16 if io == 'bf16' else torch.float32
    x = torch.from_numpy(z['x']).to(dt).cuda().requires_grad_(True)
    y = m(x)
    assert y.dtype == dt and x.dtype == dt
    y.backward(torch.from_numpy(z['dy']).to(dt).cuda())
    assert x.grad.dtype == dt
    assert rel_l2(y.detach().float().cpu(), torch.from_numpy(z['y'])) < 2e-2
    assert torch.allclose(y.detach().float().cpu().double(), torch.from_numpy(z['y']), rtol=3e-2, atol=3e-2)
    assert rel_l2(x.grad.float().cpu(), torch.from_numpy(z['gx'])) < 4e-2
    for n, p in m.named_parameters():
        assert rel_l2(p.grad.cpu(), torch.from_numpy(z['g.' + n])) < 4e-2, n


@pytest.mark.gpu
@pytest.mark.parametrize('precision,dt', [('fp32', torch.float32), ('bf16', torch.float32), ('bf16', torch.bfloat16)])
def test_epilogue_writes_into_the_feature_buffer(precision, dt):
    """`out_total`: y lands in the first Cout channels of a (B, Ctot, H, W) buffer, bit-identical to the dense call, the rest of
    the buffer untouched by the kernels; gradients unchanged."""
    import chexpert_b200 as cb
    torch.manual_seed(3)
    m = cb.AAConv2d(64, 32, 3, 2, 160, 8, 8, True, (12, 10), precision=precision).cuda()
    x = torch.relu(torch.randn(2, 64, 24, 20, device='cuda')).to(dt)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ya = m(xa)
    yb = m(xb, out_total=80)
    buf = yb.feature_buffer
    assert tuple(buf.shape) == (2, 80, 12, 10) and buf.dtype == dt and yb.data_ptr() == buf.data_ptr()
    assert torch.equal(ya, yb)
    dy = torch.randn_like(ya)
    ya.backward(dy)
    ga = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    yb.backward(dy)
    assert torch.equal(xa.grad, xb.grad)
    for a, p in zip(ga, m.parameters()):
        assert torch.equal(a, p.grad)


@pytest.mark.gpu
def test_tiny_densenet_buffered_fused_matches_reference_fixture():
    """Whole-model anchor with BOTH options on: the reference DenseNet(16,(2,2,2,2),32) fixture (oracle/gen_golden.py), fp32."""
    from chexpert_b200.densenet import DenseNet
    import chexpert_b200 as cb
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    z = load_fixture('tiny_densenet')
    m = DenseNet(16, (2, 2, 2, 2), 32, num_classes=5,
                 attn_params={'k': 0.5, 'v': 0.5, 'nh': 8, 'relative': True, 'input_dims': (64, 64)}, precision='fp32',
                 feature_buffer=True, fused_prologue=True)
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


@pytest.mark.gpu
def test_train_step_options_follow_the_plain_step():
    """TrainStep(buffered=True, fused_prologue=True) under autocast (bf16 activations at the AAConv2d boundary) tracks the plain
    configuration's loss sequence."""
    from chexpert_b200.train import TrainStep, synthetic_batch
    x, t = synthetic_batch(4, size=64, seed=5, device='cuda')
    losses = {}
    for opt in (False, True):
        ts = TrainStep('cuda', size=64, precision='bf16', lr=2e-4, seed=0, buffered=opt, fused_prologue=opt)
        losses[opt] = torch.stack([ts(x, t) for _ in range(5)]).cpu()
    assert torch.isfinite(losses[True]).all()
    assert torch.allclose(losses[True], losses[False], rtol=5e-2, atol=5e-3), (losses[True], losses[False])


@pytest.mark.gpu
@pytest.mark.parametrize('dt,tol', [(torch.float32, 2e-5), (torch.bfloat16, 2e-2)])
def test_fused_bn_relu_on_a_buffer_slice_matches_torch(dt, tol):
    """chexpert_b200.fused_bn.bn_relu (training mode) on a strided channel slice of a feature buffer against
    nn.BatchNorm2d + ReLU on the contiguous copy: output, running statistics, dx, dweight, dbias."""
    from chexpert_b200.fused_bn import bn_relu
    torch.manual_seed(0)
    B, Ctot, C, H, W = 5, 48, 24, 9, 7
    buf = (torch.randn(B, Ctot, H, W, device='cuda') * 2 + 0.5).to(dt)
    ref = torch.nn.BatchNorm2d(C).cuda()
    ours = torch.nn.BatchNorm2d(C).cuda()
    with torch.no_grad():
        ref.weight.uniform_(0.5, 1.5), ref.bias.uniform_(-0.5, 0.5)
    ours.load_state_dict(ref.state_dict())
    xa = buf[:, :C].clone().float().requires_grad_(True)                 # contiguous fp32 reference input
    xb = buf[:, :C].detach().requires_grad_(True)                         # the strided slice itself
    assert not xb.is_contiguous()
    ya = torch.relu(ref(xa))
    yb = bn_relu(ours, xb)
    assert yb.dtype == dt and yb.is_contiguous()
    scale = float(ya.abs().max())
    assert float((ya - yb.float()).abs().max()) < tol * scale
    assert torch.allclose(ours.running_mean, ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(ours.running_var, ref.running_var, rtol=1e-4, atol=1e-5)
    assert int(ours.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    g = torch.randn_like(ya)
    ya.backward(g)
    yb.backward(g.to(dt))
    assert float((xa.grad - xb.grad.float()).abs().max()) < tol * float(xa.grad.abs().max()) * 2
    assert rel_err(ours.weight.grad, ref.weight.grad) < tol and rel_err(ours.bias.grad, ref.bias.grad) < tol
    ours.eval(), ref.eval()                                               # eval mode goes through the module itself
    assert torch.allclose(bn_relu(ours, xb.detach()).float(), torch.relu(ref(xa.detach())), rtol=tol, atol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize('dt,tol', [(torch.float32, 2e-5), (torch.bfloat16, 2e-2)])
@pytest.mark.parametrize('geom', [(5, 96, 40, 6, 10), (16, 160, 96, 10, 10), (3, 64, 64, 12, 8)])
def test_channels_last_bn_relu_kernels_match_torch(dt, tol, geom):
    """csrc/bn_cl.cu through chexpert_b200.fused_bn: (a) tap_bn_relu_cl -- NCHW channel prefix of a feature buffer in, NHWC out, dx added
    in place into an NCHW gradient; (b) bn_relu_cl -- NHWC in, NHWC out; (c) the slice transposes.  Against nn.BatchNorm2d + ReLU in
    fp32 on contiguous copies: outputs, running statistics, dx (incl. the accumulation), dweight, dbias."""
    from chexpert_b200.fused_bn import bn_relu_cl, slice_layout, tap_bn_relu_cl
    torch.manual_seed(1)
    B, Ctot, C, H, W = geom
    buf = (torch.randn(B, Ctot, H, W, device='cuda') * 2 + 0.5).to(dt)

    def pair():
        ref, ours = torch.nn.BatchNorm2d(C).cuda(), torch.nn.BatchNorm2d(C).cuda()
        with torch.no_grad():
            ref.weight.uniform_(0.5, 1.5), ref.bias.uniform_(-0.5, 0.5)
        ours.load_state_dict(ref.state_dict())
        return ref, ours

    # ---- (a) NCHW prefix -> NHWC, gradient accumulated into a strided NCHW tensor ----
    ref, ours = pair()
    xa = buf[:, :C].clone().float().requires_grad_(True)
    xb = buf[:, :C].detach().requires_grad_(True)
    ya = torch.relu(ref(xa))
    stats = torch.empty(2 * B * Ctot, device='cuda', dtype=torch.float32)
    fb, yb = tap_bn_relu_cl(ours, xb, (stats, 0))
    assert yb.is_contiguous(memory_format=torch.channels_last) and fb.data_ptr() == xb.data_ptr()
    scale = float(ya.detach().abs().max())
    assert float((ya - yb.float()).abs().max()) < tol * scale
    assert torch.allclose(ours.running_mean, ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(ours.running_var, ref.running_var, rtol=1e-4, atol=1e-5)
    g = torch.randn_like(ya)
    gbuf = torch.randn(B, Ctot, H, W, device='cuda').to(dt)               # gradient of the whole buffer; the prefix gets dx added
    g_prefix0 = gbuf[:, :C].float().clone()
    ya.backward(g)
    torch.autograd.backward([fb, yb], [gbuf[:, :C], g.to(dt).contiguous(memory_format=torch.channels_last)])
    want = xa.grad + g_prefix0
    assert float((want - gbuf[:, :C].float()).abs().max()) < tol * float(want.abs().max()) * 2      # accumulated in place
    assert float((want - xb.grad.float()).abs().max()) < tol * float(want.abs().max()) * 2
    assert rel_err(ours.weight.grad, ref.weight.grad) < tol and rel_err(ours.bias.grad, ref.bias.grad) < tol

    # ---- (b) NHWC -> NHWC ----
    ref, ours = pair()
    xc = buf[:, :C].clone().float().requires_grad_(True)
    xd = buf[:, :C].detach().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    yc = torch.relu(ref(xc))
    yd = bn_relu_cl(ours, xd)
    assert yd.is_contiguous(memory_format=torch.channels_last)
    assert float((yc - yd.float()).abs().max()) < tol * float(yc.abs().max())
    assert torch.allclose(ours.running_mean, ref.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(ours.running_var, ref.running_var, rtol=1e-4, atol=1e-5)
    yc.backward(g)
    yd.backward(g.to(dt).contiguous(memory_format=torch.channels_last))
    assert float((xc.grad - xd.grad.float()).abs().max()) < tol * float(xc.grad.abs().max()) * 2
    assert rel_err(ours.weight.grad, ref.weight.grad) < tol and rel_err(ours.bias.grad, ref.bias.grad) < tol

    # ---- (c) slice transposes: NHWC -> NCHW slice of the buffer and back, bit exact ----
    k = 32
    new = torch.randn(B, k, H, W, device='cuda').to(dt).contiguous(memory_format=torch.channels_last)
    tgt = torch.zeros(B, Ctot, H, W, device='cuda', dtype=dt)
    slice_layout(new, tgt[:, 8:8 + k], to_nchw=True)
    assert torch.equal(tgt[:, 8:8 + k], new) and float(tgt[:, :8].abs().max()) == 0 and float(tgt[:, 8 + k:].abs().max()) == 0
    back = torch.empty_like(new)
    slice_layout(tgt[:, 8:8 + k], back, to_nchw=False)
    assert back.is_contiguous(memory_format=torch.channels_last) and torch.equal(back, new)
