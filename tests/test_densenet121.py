"""The reference's baseline model, torchvision's densenet121, on the fused path: densenet121(), the BatchNorm + ReLU + AvgPool2d(2)
Transition kernels (aaconv_bn_relu_pool_forward / _backward, csrc/bn_cl.cu) against float64, BNTransition, and TrainStep /
Predictor with arch='densenet121'.

The kernel data and gates are those of tests/test_bn_kernels.py (training) and tests/test_inference.py (eval), imported from
there.  The training reference is theirs too: BatchNorm + ReLU + pool backward is BatchNorm + ReLU backward with the source-pixel
gradient dy = dP / 4 spread over each 2 x 2 window and 0 on a dropped odd row / column; the pooled output is avg_pool2d of the
reference y.
"""
import ctypes
import types

import pytest
import torch
import torch.nn.functional as F
import torchvision

from chexpert_b200 import _lib, densenet, fused_bn
from chexpert_b200.aaconv import _ptr, _stream
from tests.test_bn_kernels import (EPS, MOM, Ref, _gen, check_elem, check_running, check_stats, check_wb,
                                   dx_allowance, feature_buffer, features, grad_out, make_bn, ties)
from tests.test_inference import _bf16_ulp, eval_bn, eval_features
from tests.test_inference import reference as eval_reference

CL = torch.channels_last
N_PARAMS = 6958981            # torchvision.models.densenet121(num_classes=5)


# ------------------------------------------------------------------------------------------------ CPU: the model
def _pair(seed=0, **kw):
    torch.manual_seed(seed)
    tv = torchvision.models.densenet121(num_classes=5)
    ours = densenet.densenet121(5, **kw)
    return tv, ours


def test_densenet121_has_torchvisions_state_dict():
    tv, ours = _pair()
    a, b = tv.state_dict(), ours.state_dict()
    assert list(a) == list(b) and len(a) == 727
    assert all(a[k].shape == b[k].shape for k in a)
    assert sum(p.numel() for p in ours.parameters()) == sum(p.numel() for p in tv.parameters()) == N_PARAMS
    ours.load_state_dict(a, strict=True)
    tv.load_state_dict(b, strict=True)
    for kw in ({'feature_buffer': True}, {'feature_buffer': True, 'fused_transition': True, 'fused_eval': True}):
        assert list(densenet.densenet121(5, **kw).state_dict()) == list(a)


def test_densenet121_forward_and_backward_are_torchvisions_on_cpu():
    """Without the new keywords the model is torchvision's network op for op: same logits and gradients, bit for bit."""
    tv, ours = _pair()
    ours.load_state_dict(tv.state_dict(), strict=True)
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    ya, yb = tv(x), ours(x)
    assert torch.equal(ya, yb)
    g = torch.randn(ya.shape, generator=torch.Generator().manual_seed(2))
    ya.backward(g)
    yb.backward(g)
    for (n, pa), pb in zip(tv.named_parameters(), ours.parameters()):
        assert torch.equal(pa.grad, pb.grad), n
    for (n, ba), bb in zip(tv.named_buffers(), ours.buffers()):
        assert torch.equal(ba, bb), n


def test_module_transition_unless_fused_transition_is_asked_for():
    for kw in ({'feature_buffer': True}, {'fused_transition': True}):
        m = densenet.DenseNet(32, (6, 12, 24, 16), 64, num_classes=5, attn_params=None, **kw)
        t = m.features.transition1
        assert type(t) is torch.nn.Sequential and list(dict(t.named_children())) == ['norm', 'relu', 'conv', 'pool']
    m = densenet.densenet121(5, feature_buffer=True, fused_transition=True)
    assert all(isinstance(getattr(m.features, f'transition{i}'), densenet.BNTransition) for i in (1, 2, 3))


def test_bn_transition_on_cpu_is_the_module_path():
    torch.manual_seed(0)
    ref = torchvision.models.densenet._Transition(64, 32)
    t = densenet.BNTransition(64, 32, fused_eval=True)
    t.load_state_dict(ref.state_dict(), strict=True)
    x = torch.randn(2, 64, 9, 8, generator=torch.Generator().manual_seed(1))
    assert torch.equal(t(x, out_total=48), ref(x))
    t.eval(), ref.eval()
    with torch.no_grad():
        assert torch.equal(t(x), ref(x))


def test_module_fallbacks_leave_a_batched_counter_alone():
    """TrainStep(buffered=True) bumps every num_batches_tracked once per step itself (one foreach add, `_nbt_batched`).  Where
    bn_relu, tap_bn_relu and BNTransition run the modules (here: on the CPU; on the GPU for inputs the kernels do not take) the norm
    must not count the batch a second time, and must otherwise be the module's own arithmetic, bit for bit."""
    x = torch.randn(2, 64, 9, 8, generator=torch.Generator().manual_seed(1))
    torch.manual_seed(0)
    ref = torchvision.models.densenet._Transition(64, 32)
    t = densenet.BNTransition(64, 32)
    t.load_state_dict(ref.state_dict(), strict=True)
    t.norm._nbt_batched = True
    pairs = [('BNTransition', ref(x), t(x, out_total=48), ref.norm, t.norm)]
    for name, fn in (('bn_relu', fused_bn.bn_relu), ('tap_bn_relu', lambda bn, v: fused_bn.tap_bn_relu(bn, v)[1])):
        a = torch.nn.BatchNorm2d(64)
        with torch.no_grad():
            a.weight.uniform_(0.5, 1.5), a.bias.uniform_(-0.5, 0.5)
        b = torch.nn.BatchNorm2d(64)
        b.load_state_dict(a.state_dict())
        b._nbt_batched = True
        pairs.append((name, F.relu(a(x)), fn(b, x), a, b))
    for name, want, got, a, b in pairs:
        assert torch.equal(got, want), name
        assert torch.equal(b.running_mean, a.running_mean) and torch.equal(b.running_var, a.running_var), name
        assert int(a.num_batches_tracked) == 1 and int(b.num_batches_tracked) == 0, (name, int(b.num_batches_tracked))


# ------------------------------------------------------------------------------------------------ GPU: the kernels against float64
def _dt(dtype):
    return _lib.FP32 if dtype == torch.float32 else _lib.BF16


def spread(dP, H, W):
    """dP (B, C, H // 2, W // 2) -> the source-pixel gradient of the 2 x 2 mean: dP / 4 on every window pixel, 0 on a dropped odd
    row / column."""
    B, C, Hp, Wp = dP.shape
    dy = torch.zeros(B, C, H, W, device=dP.device, dtype=torch.float64)
    dy[:, :, :2 * Hp, :2 * Wp] = dP.double().repeat_interleave(2, 2).repeat_interleave(2, 3) / 4
    return dy


def stats_nchw(xs, dtype, B, C, H, W, pst, valid):
    G, bpb = ctypes.c_int(0), ctypes.c_int(0)
    _lib.check(_lib.load().aaconv_bn_stats_nchw(_ptr(xs), _dt(dtype), B, C, H * W, xs.stride(0), _ptr(pst), valid, ctypes.byref(G),
                                                ctypes.byref(bpb), _stream()), 'aaconv_bn_stats_nchw')
    return G.value, bpb.value


def pool_forward(xs, bn, y, saved, pst, G, bpb, training=1):
    B, C, H, W = xs.shape
    return _lib.load().aaconv_bn_relu_pool_forward(_ptr(xs), _dt(xs.dtype), B, C, H, W, xs.stride(0), training, _ptr(bn.weight),
                                                   _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var), MOM, EPS, _ptr(y),
                                                   _ptr(saved), _ptr(pst), G, bpb, _stream())


def pool_backward(xs, dP, saved, bn, dx, acc, dw, db):
    lib = _lib.load()
    B, C, H, W = xs.shape
    ws = torch.empty(lib.aaconv_bn_relu_pool_workspace_bytes(B, C, H, W), device='cuda', dtype=torch.uint8)
    return lib.aaconv_bn_relu_pool_backward(_ptr(xs), _dt(xs.dtype), B, C, H, W, xs.stride(0), _ptr(dP), _ptr(saved), _ptr(bn.weight),
                                            _ptr(bn.bias), _ptr(dx), 0 if dx is None else dx.stride(0), acc, _ptr(dw), _ptr(db),
                                            _ptr(ws), _stream())


def run_train(x, bn, dP, acc):
    """Two forward calls (the running statistics move twice) and one backward of the kernels on x, read as the channel prefix of a
    wider feature buffer; dx written or added into the prefix of a wider gradient buffer.  Checks that P is written in full and
    nothing past it, and that the feature buffer and the gradient channels behind the input are untouched.
    -> (P in (B, C, H', W') layout, saved, dx, the gradient that was there before (acc) or None, dweight, dbias)."""
    B, C, H, W = x.shape
    n = B * C * (H // 2) * (W // 2)
    buf = feature_buffer(x)
    keep = buf.clone()
    xs = buf[:, :C]
    pst = torch.empty(2 * B * C, device='cuda', dtype=torch.float32)
    saved = torch.empty(C, 2, device='cuda', dtype=torch.float32)
    for _ in range(2):
        y = torch.full((n + 64,), float('nan'), device='cuda', dtype=x.dtype)
        G, bpb = stats_nchw(xs, x.dtype, B, C, H, W, pst, 0)
        _lib.check(pool_forward(xs, bn, y, saved, pst, G, bpb), 'aaconv_bn_relu_pool_forward')
    torch.cuda.synchronize()
    assert bool(torch.isnan(y[n:]).all()), 'P: written past its end'
    P = y[:n].view(B, H // 2, W // 2, C).permute(0, 3, 1, 2)
    gbuf = feature_buffer(grad_out(B, C, H, W, x.dtype, 7), seed=98)
    g0 = gbuf.clone()
    dw, db = torch.empty(C, device='cuda'), torch.empty(C, device='cuda')
    _lib.check(pool_backward(xs, dP.contiguous(memory_format=CL), saved, bn, gbuf[:, :C], int(acc), dw, db), 'aaconv_bn_relu_pool_backward')
    torch.cuda.synchronize()
    assert torch.equal(buf, keep), 'the feature buffer changed'
    assert torch.equal(gbuf[:, C:], g0[:, C:]), 'gradient channels behind the input changed'
    return P, saved, gbuf[:, :C], (g0[:, :C] if acc else None), dw, db


def two_step_running(ref, rm0, rv0):
    """The running statistics after two updates with the same batch (nn.BatchNorm2d: momentum, unbiased variance)."""
    unb = ref.var * (ref.n / (ref.n - 1))
    rm1, rv1 = (1 - MOM) * rm0.double() + MOM * ref.mean, (1 - MOM) * rv0.double() + MOM * unb
    return types.SimpleNamespace(var=ref.var, rm=(1 - MOM) * rm1 + MOM * ref.mean, rv=(1 - MOM) * rv1 + MOM * unb)


def check_train(what, x, bn, dP, acc):
    B, C, H, W = x.shape
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    ref = Ref(x, bn.weight, bn.bias, spread(dP, H, W), rm0, rv0)
    tie = ties(ref)
    P, saved, dx, base, dw, db = run_train(x, bn, dP, acc)
    check_elem(f'{what} P', P, F.avg_pool2d(ref.y, 2), x.dtype)
    check_elem(f'{what} dx', dx, ref.dx if base is None else ref.dx + base.double(), x.dtype, skip=tie, allow=dx_allowance(ref, tie))
    check_stats(what, saved, ref)
    check_running(what, bn, two_step_running(ref, rm0, rv0))
    check_wb(what, dw, db, ref, tie)
    d = dx.double() - (0 if base is None else base.double())     # the dropped row / column has g = 0 but gets the mean terms of dx
    assert (H % 2 == 0 or float(d[:, :, -1].abs().max()) > 0) and (W % 2 == 0 or float(d[:, :, :, -1].abs().max()) > 0), what


def check_eval_pool(what, got, x, bn):
    """The gates of test_inference.check_eval on the 2 x 2 means: the per-channel fp32 bound of the affine map holds for each
    term, and the three adds and the quarter round once more each (half a bound on top); bf16 rounds the fp32 mean once."""
    ref, _, bound = eval_reference(x, bn)
    ref, bound = F.avg_pool2d(ref, 2), 1.5 * bound
    got = got.double()
    assert torch.isfinite(got).all(), f'{what}: non-finite values'
    if x.dtype == torch.float32:
        err, lim = (got - ref).abs(), bound.expand_as(ref)
    else:
        r16 = ref.to(torch.bfloat16).double()
        err, lim = (got - r16).abs(), torch.maximum(_bf16_ulp(r16), _bf16_ulp(got)) + bound
    ratio = float((err / lim.clamp_min(1e-300)).max())
    print(f'{what}: worst error {ratio:.3g} of its bound')
    assert bool((err <= lim).all()), f'{what}: {int((err > lim).sum())} elements over the gate (worst {ratio:.3g})'


# (name, B, C, H, W): the three Transitions of densenet121 at B = 16, 320 px, and the edges
GEOMETRIES = [
    ('transition1', 16, 256, 80, 80),       # G = 16 statistics groups of one plane
    ('transition2', 16, 512, 40, 40),       # G = 4: groups of 5 / 5 / 5 / 1 planes
    ('transition3', 16, 1024, 20, 20),      # G = 1
    ('odd_15x17', 4, 64, 15, 17),           # a dropped row and a dropped column
    ('batch1', 1, 64, 20, 20),
    ('batch17', 17, 36, 40, 40),            # last group of 2 planes, a channel tile of 36 of 64
]
CASES = [pytest.param(B, C, H, W, id=name) for name, B, C, H, W in GEOMETRIES]
DTYPES = [pytest.param(torch.float32, id='fp32'), pytest.param(torch.bfloat16, id='bf16')]


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('acc', [False, True], ids=['write', 'accumulate'])
@pytest.mark.parametrize('B,C,H,W', CASES)
def test_bn_relu_pool_train_matches_float64(B, C, H, W, acc, dtype):
    x = features(B, C, H, W, dtype, 1)
    dP = grad_out(B, C, H // 2, W // 2, dtype, 2)
    check_train(f'{B}x{C}x{H}x{W} {dtype} {"acc" if acc else "write"}', x, make_bn(C, 3), dP, acc)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('B,C,H,W', CASES)
def test_bn_relu_pool_eval_matches_float64(B, C, H, W, dtype):
    bn = eval_bn(C, 3)
    x = eval_features(B, C, H, W, bn, dtype, 1)
    buf = feature_buffer(x)
    keep, stats = buf.clone(), [t.clone() for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    n = B * C * (H // 2) * (W // 2)
    y = torch.full((n + 64,), float('nan'), device='cuda', dtype=dtype)
    _lib.check(pool_forward(buf[:, :C], bn, y, None, None, 0, 0, training=0), 'aaconv_bn_relu_pool_forward')
    torch.cuda.synchronize()
    assert bool(torch.isnan(y[n:]).all()) and torch.equal(buf, keep)
    assert all(torch.equal(a, b) for a, b in zip((bn.running_mean, bn.running_var, bn.num_batches_tracked), stats))
    P = y[:n].view(B, H // 2, W // 2, C).permute(0, 3, 1, 2)
    check_eval_pool(f'eval {B}x{C}x{H}x{W} {dtype}', P, x, bn)
    with torch.no_grad():                    # the Python route: the same bits, channels-last
        yp = fused_bn.bn_relu_pool_eval(bn, buf[:, :C])
    assert yp.is_contiguous(memory_format=CL) and torch.equal(yp, P)


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['misaligned', 'c_not_multiple_of_4', 'h1'])
def test_bn_relu_pool_rejects_what_it_does_not_support(case):
    """Each limit is refused with a message naming it, and fused_bn.pool_ok says no, so BNTransition runs the modules."""
    lib = _lib.load()
    B, C, H, W, offset = {'misaligned': (4, 64, 8, 8, 1), 'c_not_multiple_of_4': (4, 66, 8, 8, 0), 'h1': (4, 64, 1, 8, 0)}[case]
    bn = make_bn(C, 3)
    x = features(B, C, H, W, torch.float32, 1)
    buf = feature_buffer(x, offset=offset)
    xs = buf[:, :C]
    pst = torch.empty(2 * B * C, device='cuda')
    saved = torch.empty(C, 2, device='cuda')
    y = torch.empty(B * C * max(H // 2, 1) * (W // 2), device='cuda')
    G, bpb = stats_nchw(xs, torch.float32, B, C, H, W, pst, 0)
    assert pool_forward(xs, bn, y, saved, pst, G, bpb) == -1
    msg = lib.aaconv_last_error().decode()
    want = 'aligned for four-element accesses' if case == 'misaligned' else 'C a multiple of 4, H and W >= 2'
    assert want in msg, msg
    assert pool_backward(xs, y, saved, bn, None, 0, None, None) == -1
    assert want in lib.aaconv_last_error().decode()
    assert not fused_bn.pool_ok(bn, xs)
    with pytest.raises(RuntimeError, match='multiple of 4'):
        fused_bn.bn_relu_pool(bn, xs)


@pytest.mark.gpu
def test_shared_block_statistics_are_read_not_recomputed():
    """Channels below stats_valid_channels take their statistics from the block's buffer: shifting one entry of channel 5 moves
    channel 5's output and no other; channels at or above it are reduced here, so their entries are overwritten."""
    B, C, H, W = 16, 64, 40, 40
    x = features(B, C, H, W, torch.float32, 1)
    buf = feature_buffer(x)
    xs = buf[:, :C]
    pst = torch.empty(2 * B * C, device='cuda')
    stats_nchw(xs, torch.float32, B, C, H, W, pst, 0)                  # the block's reduction of every channel
    G, _ = stats_nchw(xs, torch.float32, B, C, H, W, pst, C)            # layout: (mean, M2) of group g of channel c at [c * G + g]
    assert G == 4
    outs = []
    for shift in (False, True):
        p = pst.clone()
        if shift:
            p.view(-1, 2)[5 * G, 0] += 1.0                              # group 0's mean of channel 5
            p.view(-1, 2)[40 * G, 0] += 1.0                             # channel 40 >= valid: recomputed, the shift vanishes
        bn = make_bn(C, 3)
        y = torch.empty(B, C, H // 2, W // 2, device='cuda', memory_format=CL)
        G, bpb = stats_nchw(xs, torch.float32, B, C, H, W, p, 32)
        _lib.check(pool_forward(xs, bn, y, torch.empty(C, 2, device='cuda'), p, G, bpb), 'aaconv_bn_relu_pool_forward')
        outs.append(y)
    moved = (outs[0] != outs[1]).flatten(2).any(2).any(0)
    assert moved.nonzero().flatten().tolist() == [5], moved.nonzero().flatten().tolist()


# ------------------------------------------------------------------------------------------------ GPU: module, model, steps
@pytest.fixture
def no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def rel(a, b):
    """max |a - b| over max |b| (the whole-tensor gate of the model tests, as tests/helpers.rel_err)."""
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


# Module-level gates.  fp32 against float64: a gradient within 2e-3 of its tensor's largest entry (the tiny-DenseNet anchor of
# tests/test_gpu_parity.py); y and the running statistics, one layer deep, within 1e-4.
GRAD_TOL, OUT_TOL = 2e-3, 1e-4
# Model-level gates.  Through densenet121's 58 BatchNorm layers at 64 px (B = 4: 16 elements per channel in the last block) the fp32
# error against float64 is set by the network's conditioning, not by one kernel: a parameter gradient that is a sum of terms of both
# signs (e.g. the stem's BatchNorm weight) can carry several percent of its largest entry in ANY fp32 evaluation.  So each tensor of
# the fused model is gated against the error of torchvision's own fp32 model on the same GPU and data: at most CTL_FACTOR times it,
# or GRAD_TOL / OUT_TOL where that is larger.
CTL_FACTOR = 3.0


def gate_vs_control(what, ours, ctl, ref, tol):
    """Per tensor: rel(ours, ref) <= max(tol, CTL_FACTOR * rel(ctl, ref)); prints the worst tensor."""
    worst = ('', 0.0, 0.0)
    for n in ref:
        e, ec = rel(ours[n], ref[n]), rel(ctl[n], ref[n])
        if e / max(tol, CTL_FACTOR * ec) > worst[1] / max(tol, CTL_FACTOR * worst[2]) or not worst[0]:
            worst = (n, e, ec)
        assert e <= max(tol, CTL_FACTOR * ec), f'{what} {n}: {e:.3g} of max, torchvision fp32 {ec:.3g}'
    print(f'{what}: worst {worst[0]} {worst[1]:.3g} of max (torchvision fp32: {worst[2]:.3g})')


@pytest.mark.gpu
@pytest.mark.parametrize('B,C,H,W', [(16, 256, 80, 80), (4, 64, 15, 17)], ids=['transition1', 'odd_15x17'])
def test_bn_transition_matches_torchvision_in_float64(B, C, H, W, no_tf32):
    torch.manual_seed(0)
    ref = torchvision.models.densenet._Transition(C, C // 2).cuda().double()
    t = densenet.BNTransition(C, C // 2).cuda()
    with torch.no_grad():
        bn = make_bn(C, 3)
        ref.norm.load_state_dict(bn.state_dict())
    t.load_state_dict(ref.state_dict())
    x = features(B, C, H, W, torch.float32, 1)
    xb = feature_buffer(x)[:, :C].detach().requires_grad_(True)
    y = t(xb, out_total=C // 2 + 16)
    assert y.feature_buffer.shape == (B, C // 2 + 16, H // 2, W // 2) and y.data_ptr() == y.feature_buffer.data_ptr()
    assert int(t.norm.num_batches_tracked) == 1
    xr = x.double().requires_grad_(True)
    yr = ref(xr)
    g = grad_out(B, C // 2, H // 2, W // 2, torch.float32, 2)
    y.backward(g)
    yr.backward(g.double())
    checks = [('y', y, yr), ('dx', xb.grad, xr.grad), ('conv.weight', t.conv.weight.grad, ref.conv.weight.grad),
              ('norm.weight', t.norm.weight.grad, ref.norm.weight.grad), ('norm.bias', t.norm.bias.grad, ref.norm.bias.grad),
              ('running_mean', t.norm.running_mean, ref.norm.running_mean), ('running_var', t.norm.running_var, ref.norm.running_var)]
    for name, got, want in checks:
        e = rel(got, want)
        print(f'BNTransition {B}x{C}x{H}x{W} {name}: {e:.3g} of max')
        assert e < (OUT_TOL if name in ('y', 'running_mean', 'running_var') else GRAD_TOL), (name, e)


def _models(seed=0):
    torch.manual_seed(seed)
    tv = torchvision.models.densenet121(num_classes=5)
    with torch.no_grad():               # non-trivial running statistics for the eval comparison
        for m in tv.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.uniform_(-0.5, 0.5)
                m.running_var.uniform_(0.5, 2.0)
    return tv


def _train_once(model, x, t, loss_fn):
    loss = loss_fn(model(x.to(next(model.parameters()).dtype)).double(), t)
    loss.backward()
    return (loss.detach(), {n: p.grad for n, p in model.named_parameters()},
            {n: b for n, b in model.named_buffers() if b.dtype.is_floating_point})


@pytest.mark.gpu
def test_fused_densenet121_matches_torchvision_in_float64(no_tf32, monkeypatch):
    """densenet121(feature_buffer, fused_transition) in fp32 against torchvision's densenet121 in float64, same state_dict, B = 4 at
    64 px: train-mode loss, every parameter gradient and the running statistics (gated against torchvision's fp32 model, see
    CTL_FACTOR); then eval logits with fused_eval.  The per-launch profile shows the pooled kernels once per Transition in forward
    and in backward, and every Transition read its block's statistics."""
    from chexpert_b200.loss import BCEWithLogitsLoss
    sd = _models().state_dict()
    ref = _models().cuda().double().train()
    ctl = _models().cuda().train()
    ours = densenet.densenet121(5, feature_buffer=True, fused_transition=True, fused_eval=True).cuda()
    ours.load_state_dict(sd)
    calls = []
    fn = densenet.bn_relu_pool
    monkeypatch.setattr(densenet, 'bn_relu_pool', lambda bn, x, stats=None: calls.append(stats is not None) or fn(bn, x, stats))
    x = torch.randn(4, 3, 64, 64, generator=_gen(1), device='cuda')
    t = (torch.rand(4, 5, generator=_gen(2), device='cuda') < 0.3).double()
    loss_fn = lambda z, tt: torch.nn.functional.binary_cross_entropy_with_logits(z, tt, reduction='none').sum(1).mean(0)  # noqa: E731
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    out = ours(x)
    torch.cuda.synchronize()
    fwd = [n for n, _ in _lib.profile_end()]
    loss = BCEWithLogitsLoss('train').cuda()(out, t.float())
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    loss.backward()
    torch.cuda.synchronize()
    bwd = [n for n, _ in _lib.profile_end()]
    assert calls == [True, True, True], calls                # every Transition reused its block's statistics
    assert fwd.count('bn_pool_apply') == 3, fwd
    assert bwd.count('bn_pool_bwd_reduce') == 3 and bwd.count('bn_pool_bwd_dx') == 3, bwd
    loss_r, g_r, b_r = _train_once(ref, x, t, loss_fn)
    loss_c, g_c, b_c = _train_once(ctl, x, t, loss_fn)
    e, ec = rel(loss.detach(), loss_r), rel(loss_c, loss_r)
    print(f'loss {float(loss):.7f}, float64 {float(loss_r):.7f}, torchvision fp32 {float(loss_c):.7f}')
    assert e <= max(OUT_TOL, CTL_FACTOR * ec), (e, ec)
    gate_vs_control('gradient', {n: p.grad for n, p in ours.named_parameters()}, g_c, g_r, GRAD_TOL)
    gate_vs_control('running statistics', {n: b for n, b in ours.named_buffers() if b.dtype.is_floating_point}, b_c, b_r, OUT_TOL)
    assert all(int(b) == 1 for n, b in ours.named_buffers() if n.endswith('num_batches_tracked'))
    # eval: fused_eval runs the eval kernels (autograd off) against the float64 model in eval mode on the same state_dict
    ours2 = densenet.densenet121(5, feature_buffer=True, fused_transition=True, fused_eval=True).cuda().eval()
    ours2.load_state_dict(sd)
    ref.load_state_dict(sd)
    calls.clear()
    ev = fused_bn.bn_relu_pool_eval
    n_eval = []
    monkeypatch.setattr(densenet, 'bn_relu_pool_eval', lambda bn, x: n_eval.append(1) or ev(bn, x))
    with torch.no_grad():
        e = rel(ours2(x), ref.eval()(x.double()))
    print(f'eval logits: {e:.3g} of max')
    assert e < OUT_TOL and len(n_eval) == 3 and not calls


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_train_step_densenet121(precision, no_tf32, monkeypatch):
    """TrainStep(arch='densenet121', buffered, fused_prologue, cuda_graph): the replayed steps match the eager steps, and three eager
    steps track torchvision's model trained in float64 by the same loss and optimizer -- gated, as above, against the plain
    TrainStep (torchvision's modules) in the same precision.  Parameters are compared by their updates over the three steps, all
    tensors together in L2: a zero-initialised BatchNorm bias holds nothing but its update, so a per-tensor gate would measure the
    amplified rounding of a few small sums."""
    from chexpert_b200.train import TrainStep, synthetic_batch
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)      # no run-to-run differences from cuDNN's atomics
    x, t = synthetic_batch(4, size=64, seed=5, device='cuda')
    kw = dict(size=64, precision=precision, lr=1e-3, seed=0, arch='densenet121')
    fused = TrainStep('cuda', buffered=True, fused_prologue=True, cuda_graph=True, graph_after=2, **kw)
    assert isinstance(fused.model.features.transition1, densenet.BNTransition)
    eager = TrainStep('cuda', buffered=True, fused_prologue=True, cuda_graph=False, **kw)
    plain = TrainStep('cuda', buffered=False, fused_prologue=False, cuda_graph=False, **kw)
    p0 = {n: p.detach().double().clone() for n, p in eager.model.named_parameters()}
    tv = torchvision.models.densenet121(num_classes=5).cuda().double()
    tv.load_state_dict(eager.model.state_dict())
    opt = torch.optim.SGD(tv.parameters(), lr=1e-3, momentum=0.9, nesterov=True)
    lf, le, lp, lt = [], [], [], []
    for _ in range(4):                  # two eager steps, the capture, a replay
        lf.append(float(fused(x, t)))
    for _ in range(3):
        le.append(float(eager(x, t)))
        lp.append(float(plain(x, t)))
        opt.zero_grad()
        loss = eager.loss_fn(tv(x.double()).float(), t)
        loss.backward()
        opt.step()
        lt.append(float(loss))
    assert fused._graph is not None
    print(f'{precision}: graph {lf}, eager {le}, plain {lp}, torchvision float64 {lt}')
    # graph against eager: the same kernels in the same order -- the gates of tests/test_gpu_parity.py::test_train_step_cuda_graph_matches_eager
    assert all(abs(a - b) <= 5e-3 * abs(b) + 1e-3 for a, b in zip(lf, le)), (lf, le)
    tol = GRAD_TOL if precision == 'fp32' else 2e-2      # bf16: autocast rounds every dense-block activation to 8 bits
    for a, c, r in zip(le, lp, lt):
        assert abs(a - r) <= max(tol * abs(r), CTL_FACTOR * abs(c - r)), (le, lp, lt)

    def update(m):
        return torch.cat([(p.detach().double() - p0[n]).flatten() for n, p in m.named_parameters()])
    du, dc, dr = update(eager.model), update(plain.model), update(tv)
    e, ec = float((du - dr).norm() / dr.norm()), float((dc - dr).norm() / dr.norm())
    print(f'{precision}: parameter updates {e:.3g} of their L2 norm (plain TrainStep: {ec:.3g})')
    assert e <= max(tol, CTL_FACTOR * ec), (e, ec)


@pytest.mark.gpu
@pytest.mark.parametrize('channels_last', [False, True], ids=['nchw', 'channels_last'])
def test_train_step_densenet121_counts_each_batch_once(channels_last):
    """TrainStep(buffered=True) bumps every num_batches_tracked itself, so the BatchNorms that run as modules must not bump it again.
    At 288 px transition3 sees 18 x 18 maps: their 9 x 9 pool is past the fused route's limit ((H/2)(W/2) a multiple of 4), so it
    runs the four modules; with channels_last the stem's conv0 writes a channels-last map, which norm0 takes through the module."""
    from chexpert_b200.train import TrainStep, synthetic_batch
    ts = TrainStep('cuda', size=288, precision='bf16', lr=1e-3, seed=0, arch='densenet121', buffered=True, fused_prologue=True,
                   channels_last=channels_last)
    t3 = ts.model.features.transition3
    assert isinstance(t3, densenet.BNTransition) and not t3._fused(torch.empty(2, 1024, 18, 18, device='cuda'))
    x, t = synthetic_batch(2, size=288, seed=5, device='cuda')
    for _ in range(2):
        ts(x, t)
    counts = {n: int(m.num_batches_tracked) for n, m in ts.model.named_modules() if isinstance(m, torch.nn.BatchNorm2d)}
    assert len(counts) == 121 and all(c == 2 for c in counts.values()), {n: c for n, c in counts.items() if c != 2}


@pytest.mark.gpu
@pytest.mark.parametrize('autocast', [False, True], ids=['fp32', 'bf16_autocast'])
def test_predictor_densenet121(autocast, no_tf32):
    """Predictor(arch='densenet121') against predict_logits of the torchvision model on two checkpoints: one capture serves both,
    and the last batch of 42 = 16 + 16 + 10 images is padded.  Gates: fp32 as the eval logits above; bf16 autocast those of
    tests/test_inference.py::test_predictor_bf16_autocast_matches_reference (rtol 2e-2, atol 1e-2)."""
    from chexpert_b200.evaluate import Predictor, predict_logits, synthetic_radiographs_u8
    images = synthetic_radiographs_u8(42, 320, seed=3)
    p = Predictor(5, 320, batch_size=16, autocast=autocast, arch='densenet121')
    for seed in (0, 1):
        tv = _models(seed).cuda()
        p.load_state_dict(tv.state_dict())
        got = p(images)
        want = predict_logits(tv, images, 16)
        print(f'Predictor densenet121 autocast={autocast} checkpoint {seed}: {rel(got, want):.3g} of max')
        if autocast:
            assert torch.allclose(got, want, rtol=2e-2, atol=1e-2), float((got - want).abs().max())
        else:
            assert rel(got, want) < OUT_TOL
    assert p.captures == 1
