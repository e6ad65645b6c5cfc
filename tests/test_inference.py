"""Inference through the fused dense-block path: the eval-mode BatchNorm2d + ReLU kernel (aaconv_bn_relu_eval, csrc/bn_cl.cu and
csrc/bn_relu.cu) against float64, BufferedDenseBlock / DenseNet with fused_eval, and chexpert_b200.evaluate.Predictor against the
reference logits of tests/golden/eval_ensemble.npz.

Kernel data: running_mean = 64 + randn per channel, running_var log-uniform over [1e-3, 1e2], weight with negative entries and one
zero, bias in [-0.5, 0.5], x = running_mean + sqrt(running_var) * randn.  So every channel's pre-activation straddles zero, and the
affine map y = x s + t (s = w / sqrt(var + eps), t = b - mean s) cancels two terms of up to |64 s| against each other.
"""
import json
import os

import numpy as np
import pytest
import torch

from chexpert_b200 import _lib, densenet, fused_bn
from chexpert_b200.aaconv import _ptr, _stream
from tests.helpers import GOLDEN

EPS = 1e-5
CL = torch.channels_last
ZERO_W = 3              # the channel whose weight is exactly 0 (y = relu(bias) there)

# ---- gates ----
# fp32: s, t and the fma are each rounded once in fp32 (s: IEEE sqrt and division, t: a product and a sum), so the error of
# x s + t is a few ulps of the terms it adds up: per channel, 1e-6 (~8 ulps) of max(|x s| + |mean s| + |bias|) over the channel.
FP32_REL = 1e-6
# bf16: the kernel computes in fp32 and rounds once to bf16.  The float64 value rounded to bf16 may differ from the kernel's by one
# bf16 ulp (the two fall on either side of a rounding boundary), plus the fp32 error above where the fp32 value has moved (near
# zero after the cancellation, the fp32 bound can exceed a bf16 ulp).
# Near ties (both dtypes): an element whose float64 pre-activation lies within the fp32 bound of zero may come out as 0 -- the
# ReLU can land on either side; the gate |got - ref| <= bound admits exactly that, since |ref| <= |pre| <= bound there.


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def eval_bn(C, seed):
    """Eval-mode BatchNorm2d with the running statistics and affine parameters described in the module docstring."""
    g = _gen(seed)
    bn = torch.nn.BatchNorm2d(C, eps=EPS).cuda().eval()
    with torch.no_grad():
        bn.running_mean.copy_(64 + torch.randn(C, generator=g, device='cuda'))
        bn.running_var.copy_(10 ** (-3 + 5 * torch.rand(C, generator=g, device='cuda')))
        sign = torch.where(torch.rand(C, generator=g, device='cuda') < 0.3, -1.0, 1.0)
        bn.weight.copy_(sign * (0.25 + torch.rand(C, generator=g, device='cuda')))
        bn.weight[min(ZERO_W, C - 1)] = 0
        bn.bias.copy_(torch.rand(C, generator=g, device='cuda') - 0.5)
        bn.num_batches_tracked.fill_(7)
    return bn


def eval_features(B, C, H, W, bn, dtype, seed):
    g = _gen(seed)
    m, s = bn.running_mean.double()[None, :, None, None], bn.running_var.double().sqrt()[None, :, None, None]
    return (m + s * torch.randn(B, C, H, W, generator=g, device='cuda', dtype=torch.float64)).to(dtype)


def reference(x, bn):
    """float64 relu(BatchNorm2d eval) of x's values -> (y, pre-activation, per-channel fp32 error bound)."""
    x64 = x.double()
    w, b = bn.weight.double()[None, :, None, None], bn.bias.double()[None, :, None, None]
    m, v = bn.running_mean.double()[None, :, None, None], bn.running_var.double()[None, :, None, None]
    s = w / (v + EPS).sqrt()
    pre = (x64 - m) * s + b
    scale = (x64 * s).abs().amax((0, 2, 3), keepdim=True) + (m * s).abs() + b.abs()
    return pre.clamp_min(0), pre, FP32_REL * scale


def _bf16_ulp(v):
    """Spacing of bf16 numbers at |v| (8 significant bits); 0 at 0."""
    a = v.abs().clamp_min(1e-30)
    return torch.where(v == 0, torch.zeros_like(v), torch.exp2(torch.floor(torch.log2(a)) - 7))


def check_eval(what, got, x, bn):
    """The gates above; `got` in (B, C, H, W) logical layout, x the input's values."""
    ref, pre, bound = reference(x, bn)
    got = got.double()
    assert torch.isfinite(got).all(), f'{what}: non-finite values'
    if x.dtype == torch.float32:
        err, lim = (got - ref).abs(), bound.expand_as(ref)
    else:
        r16 = ref.to(torch.bfloat16).double()
        err, lim = (got - r16).abs(), torch.maximum(_bf16_ulp(r16), _bf16_ulp(got)) + bound
    ratio = float((err / lim.clamp_min(1e-300)).max())
    print(f'{what}: worst error {ratio:.3g} of its bound, {int((pre.abs() <= bound).sum())} near-ties')
    bad = err > lim
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f'{what}: {int(bad.sum())} elements over the gate (worst {ratio:.3g}), first at {i}: '
                             f'got {float(got[i]):.9g}, want {float(ref[i]):.9g}, pre-activation {float(pre[i]):.9g}')


def wide_buffer(x, extra=8, offset=0, seed=99):
    """(B, C + extra, H, W) buffer whose first C channels are x, its storage `offset` elements into the allocation."""
    B, C, H, W = x.shape
    flat = torch.empty(offset + B * (C + extra) * H * W, device='cuda', dtype=x.dtype)
    buf = flat[offset:].view(B, C + extra, H, W)
    buf[:, C:] = torch.randn(B, extra, H, W, generator=_gen(seed), device='cuda').to(x.dtype)
    buf[:, :C] = x
    return buf


def _call(xs, x_is_cl, xbs, bn, y, y_is_cl, dtype, B, C, HW):
    lib = _lib.load()
    return lib.aaconv_bn_relu_eval(_ptr(xs), _lib.FP32 if dtype == torch.float32 else _lib.BF16, B, C, HW, x_is_cl, xbs,
                                   _ptr(bn.weight), _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var), EPS, _ptr(y),
                                   y_is_cl, _stream())


PAIRS = {'nchw_nchw': (0, 0), 'nchw_nhwc': (0, 1), 'nhwc_nhwc': (1, 1)}


def run_abi(pair, x, bn, offset=0):
    """aaconv_bn_relu_eval on x (NCHW pairs: read as the channel prefix of a wider buffer) into a NaN-filled y with a NaN margin.
    -> y in logical (B, C, H, W) layout.  Checks: y written in full and nothing past it, the input buffer and the BatchNorm's
    buffers unchanged."""
    x_is_cl, y_is_cl = PAIRS[pair]
    B, C, H, W = x.shape
    n = B * C * H * W
    if x_is_cl:
        src = x.contiguous(memory_format=CL)
        xs, xbs = src, C * H * W
    else:
        src = wide_buffer(x, offset=offset)
        xs, xbs = src[:, :C], src.stride(0)
    keep = src.clone()
    stats = [t.clone() for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    y = torch.full((n + 64,), float('nan'), device='cuda', dtype=x.dtype)
    _lib.check(_call(xs, x_is_cl, xbs, bn, y, y_is_cl, x.dtype, B, C, H * W), 'aaconv_bn_relu_eval')
    torch.cuda.synchronize()
    assert bool(torch.isnan(y[n:]).all()), 'y: written past its end'
    assert torch.equal(src, keep), 'the input changed'
    assert all(torch.equal(a, b) for a, b in zip((bn.running_mean, bn.running_var, bn.num_batches_tracked), stats)), \
        'running statistics changed'
    return y[:n].view(B, H, W, C).permute(0, 3, 1, 2) if y_is_cl else y[:n].view(B, C, H, W)


# (name, B, C, H, W): aadensenet121's BatchNorm geometries at B = 16, 320 px, and the edges
GEOMETRIES = [
    ('stem_norm0', 16, 64, 160, 160),
    ('block1_norm1_first', 16, 64, 80, 80), ('block1_norm1_last', 16, 224, 80, 80), ('block1_norm2', 16, 128, 80, 80),
    ('block2_norm1_first', 16, 128, 40, 40), ('block2_norm1_last', 16, 480, 40, 40), ('block2_norm2', 16, 128, 40, 40),
    ('block3_norm1_first', 16, 256, 20, 20), ('block3_norm1_last', 16, 992, 20, 20), ('block3_norm2', 16, 128, 20, 20),
    ('block4_norm1_first', 16, 512, 10, 10), ('block4_norm1_last', 16, 992, 10, 10), ('block4_norm2', 16, 128, 10, 10),
    ('norm5', 16, 1024, 10, 10),
    ('batch1', 1, 64, 10, 10),
    ('c36_partial_tile', 16, 36, 40, 40),          # one channel tile of 36 of 64
]
CASES = [pytest.param(B, C, H, W, pair, id=f'{name}-{pair}') for name, B, C, H, W in GEOMETRIES for pair in PAIRS]
DTYPES = [pytest.param(torch.float32, id='fp32'), pytest.param(torch.bfloat16, id='bf16')]


# ------------------------------------------------------------------------------------------------ CPU
def test_reference_is_torch_eval_batch_norm_in_float64():
    class _Bn:
        pass
    g = torch.Generator().manual_seed(0)
    B, C, H, W = 3, 5, 4, 6
    bn = _Bn()
    bn.weight, bn.bias = torch.randn(C, generator=g), torch.randn(C, generator=g)
    bn.running_mean, bn.running_var = 64 + torch.randn(C, generator=g), torch.rand(C, generator=g) + 1e-3
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 3 + 64
    want = torch.relu(torch.nn.functional.batch_norm(x, bn.running_mean.double(), bn.running_var.double(), bn.weight.double(),
                                                     bn.bias.double(), False, 0.1, EPS))
    assert torch.allclose(reference(x, bn)[0], want, rtol=1e-12, atol=1e-10)


def test_predictor_has_no_cpu_fallback():
    from chexpert_b200.evaluate import Predictor
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        Predictor(device='cpu')


def test_fused_eval_model_has_the_reference_state_dict():
    meta = json.load(open(os.path.join(GOLDEN, 'aadensenet121_meta.json')))
    for fb in (False, True):
        m = densenet.aadensenet121(5, (320, 320), feature_buffer=fb, fused_eval=True)
        assert m.fused_eval
        sd = m.state_dict()
        assert set(sd) == set(meta['state_dict'])
        assert all(list(sd[k].shape) == list(v) for k, v in meta['state_dict'].items())


def _tiny(fused_eval, seed=0):
    torch.manual_seed(seed)
    m = densenet.DenseNet(growth_rate=8, block_config=(2, 3), num_init_features=16, num_classes=5, feature_buffer=True,
                          fused_eval=fused_eval)
    for mod in m.modules():           # non-trivial running statistics
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.uniform_(-0.5, 0.5)
            mod.running_var.uniform_(0.5, 2.0)
    return m


def _forbid_eval_kernel(monkeypatch):
    def boom(*a, **k):
        raise AssertionError('bn_relu_eval was called')
    monkeypatch.setattr(densenet, 'bn_relu_eval', boom)
    monkeypatch.setattr(fused_bn, 'bn_relu_eval', boom)


def test_fused_eval_leaves_cpu_inference_on_the_module_path(monkeypatch):
    _forbid_eval_kernel(monkeypatch)
    x = torch.randn(2, 3, 16, 16, generator=torch.Generator().manual_seed(1))
    plain, fused = _tiny(False).eval(), _tiny(True).eval()
    with torch.no_grad():
        assert torch.equal(fused(x), plain(x))


# ------------------------------------------------------------------------------------------------ GPU: the kernel against float64
@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('B,C,H,W,pair', CASES)
def test_bn_relu_eval_matches_float64(B, C, H, W, pair, dtype):
    bn = eval_bn(C, 3)
    x = eval_features(B, C, H, W, bn, dtype, 1)
    y = run_abi(pair, x, bn)
    check_eval(f'{pair} {B}x{C}x{H}x{W} {dtype}', y, x, bn)
    # the Python route gives the same bits and leaves num_batches_tracked alone
    xin = x.contiguous(memory_format=CL) if PAIRS[pair][0] else wide_buffer(x)[:, :C]
    with torch.no_grad():
        yp = fused_bn.bn_relu_eval(bn, xin, out_cl=bool(PAIRS[pair][1]))
    assert yp.is_contiguous(memory_format=CL if PAIRS[pair][1] else torch.contiguous_format)
    assert torch.equal(yp, y) and int(bn.num_batches_tracked) == 7


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('case', ['hw49', 'misaligned'])
def test_tiled_variants_reject_what_only_nchw_serves(case, dtype):
    """H*W = 49 and a slice one element off four-element alignment: both tiled variants refuse with a message naming the
    condition, fused_bn.eval_cl_ok says no, and NCHW -> NCHW serves them (checked against float64)."""
    B, C, H, W, offset = (16, 32, 7, 7, 0) if case == 'hw49' else (16, 64, 20, 20, 1)
    bn = eval_bn(C, 3)
    x = eval_features(B, C, H, W, bn, dtype, 1)
    buf = wide_buffer(x, offset=offset)
    y = torch.empty(B * C * H * W, device='cuda', dtype=dtype)
    for x_is_cl, xs in ((0, buf[:, :C]), (1, x.contiguous(memory_format=CL) if case == 'hw49' else buf[:, :C])):
        if case == 'misaligned' and x_is_cl:
            continue                                       # a dense NHWC tensor of its own is always aligned
        code = _call(xs, x_is_cl, xs.stride(0) if not x_is_cl else C * H * W, bn, y, 1, dtype, B, C, H * W)
        assert code == -1
        msg = _lib.load().aaconv_last_error().decode()
        assert ('multiples of 4' if case == 'hw49' else 'aligned for four-element accesses') in msg, msg
    with torch.no_grad():
        assert not fused_bn.eval_cl_ok(bn, buf[:, :C])
    check_eval(f'{case} nchw_nchw {dtype}', run_abi('nchw_nchw', x, bn, offset=offset), x, bn)


@pytest.mark.gpu
def test_bn_relu_eval_rejects_what_it_does_not_support():
    lib = _lib.load()
    bn = eval_bn(4100, 3)
    x = torch.zeros(2, 4100, 4, 4, device='cuda').contiguous(memory_format=CL)
    y = torch.empty_like(x)
    assert _call(x, 1, 4100 * 16, bn, y, 1, torch.float32, 2, 4100, 16) == -1
    assert 'at most 4096 channels' in lib.aaconv_last_error().decode()
    assert _call(x, 1, 4100 * 16, bn, y, 0, torch.float32, 2, 4100, 16) == -1          # no NHWC -> NCHW variant
    assert 'needs an NHWC output' in lib.aaconv_last_error().decode()
    with torch.no_grad():
        assert not fused_bn.eval_cl_ok(bn, x)
        check_eval('4100 channels via nchw', fused_bn.bn_relu_eval(bn, x), x, bn)         # Python: an NCHW copy, NCHW -> NCHW
    bn.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match='eval-mode'):
        fused_bn.bn_relu_eval(bn, x)


# ------------------------------------------------------------------------------------------------ GPU: block and model
@pytest.fixture
def no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _counting(monkeypatch, calls):
    fn = densenet.bn_relu_eval

    def wrapped(bn, x, out_cl=False):
        key = ('nhwc' if fused_bn._is_cl(x) and not fused_bn._strided_ok(x) else 'nchw') + ('->nhwc' if out_cl else '->nchw')
        calls[key] = calls.get(key, 0) + 1
        return fn(bn, x, out_cl)
    monkeypatch.setattr(densenet, 'bn_relu_eval', wrapped)


@pytest.mark.gpu
@pytest.mark.parametrize('route,B,C0,H,W', [('channels_last', 16, 128, 40, 40), ('nchw', 16, 128, 40, 40), ('hw49', 4, 64, 7, 7)])
def test_fused_eval_block_matches_torchvision_in_float64(route, B, C0, H, W, no_tf32, monkeypatch):
    """Three layers of BufferedDenseBlock(fused_eval=True) in eval mode under no_grad against torchvision's _DenseBlock in eval
    mode in float64 on the same state_dict.  'nchw' turns the channels-last plan off; at 7 x 7 the plan cannot apply."""
    from torchvision.models.densenet import _DenseBlock
    args = (3, C0, 4, 32, 0.0)
    torch.manual_seed(0)
    a = _DenseBlock(*args).cuda().double().eval()
    for i, m in enumerate(x for x in a.modules() if isinstance(x, torch.nn.BatchNorm2d)):
        bn = eval_bn(m.num_features, 10 + i)
        with torch.no_grad():         # running statistics near the data below (mean ~0.5, var ~1): an O(1) pre-activation
            bn.running_mean.uniform_(-0.5, 1.0)
            bn.running_var.uniform_(0.3, 3.0)
        m.load_state_dict(bn.double().state_dict())
    b = densenet.BufferedDenseBlock(*args, fused_eval=True).cuda().eval()
    b.load_state_dict(a.state_dict())
    b.inner_channels_last = route != 'nchw'
    calls = {}
    _counting(monkeypatch, calls)
    x = torch.randn(B, C0, H, W, generator=_gen(1), device='cuda') + 0.5
    with torch.no_grad():
        yb = b(x)
        ya = a(x.double())
    err = float((yb.double() - ya).abs().max() / ya.abs().max())
    print(f'{route}: block y {err:.3g} of max, calls {calls}')
    assert err < 1e-4, err
    want = {'nchw->nhwc': 3, 'nhwc->nhwc': 3} if route == 'channels_last' else {'nchw->nchw': 6}
    assert calls == want


@pytest.mark.gpu
def test_fused_eval_is_opt_in(no_tf32, monkeypatch):
    """fused_eval=False in eval mode, and fused_eval=True with grad enabled, never reach bn_relu_eval; in the latter the input
    gradient still matches the plain model's."""
    x = torch.randn(4, 3, 16, 16, generator=_gen(2), device='cuda')
    plain, fused = _tiny(False).cuda().eval(), _tiny(True).cuda().eval()
    with torch.no_grad():
        y_fused_nograd = fused(x)           # the eval kernels run here ...
    calls = {}
    _counting(monkeypatch, calls)
    with torch.no_grad():
        fused(x)
    assert sum(calls.values()) == 2 + 2 * 5        # stem, norm5 and the two BatchNorms of each of the 5 dense layers
    _forbid_eval_kernel(monkeypatch)               # ... and nowhere below
    with torch.no_grad():
        y_plain = plain(x)
    assert torch.allclose(y_fused_nograd, y_plain, rtol=1e-4, atol=1e-5)
    # grad enabled: both models run the same module path.  cuDNN's default backward-data algorithms may sum in a different order
    # from call to call (atomics), which moves gradient elements near zero by more than any per-element rtol; with deterministic
    # algorithms the two backward passes are the same computation, and the gate is relative to the largest gradient
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)
    xp, xf = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    yp, yf = plain(xp), fused(xf)
    g = torch.randn(yp.shape, generator=_gen(3), device='cuda')
    yp.backward(g)
    yf.backward(g)
    ey = float((yf - yp).abs().max() / yp.abs().max())
    eg = float((xf.grad - xp.grad).abs().max() / xp.grad.abs().max())
    print(f'grad enabled: y {ey:.3g}, dx {eg:.3g} of max')
    assert ey < 1e-6 and eg < 1e-6, (ey, eg)


# ------------------------------------------------------------------------------------------------ GPU: Predictor
FIX = os.path.join(GOLDEN, 'eval_ensemble.npz')


@pytest.fixture(scope='module')
def gold():
    return np.load(FIX)


@pytest.fixture(scope='module')
def eval_set():
    from chexpert_b200.evaluate import synthetic_radiographs_u8, synthetic_eval_targets
    return synthetic_radiographs_u8(234, 320, seed=3), synthetic_eval_targets(234, seed=4)


def _state_dicts(n, precision):
    out = []
    for s in range(n):
        torch.manual_seed(s)
        out.append(densenet.aadensenet121(5, (320, 320), precision=precision).state_dict())
    return out


def _auroc(z, t):
    from chexpert_b200 import evaluate as E
    return E.auroc_per_class(z.cuda(), t.cuda()).cpu().double().numpy()


def _ensemble(gold, eval_set, precision, autocast, n):
    from chexpert_b200 import evaluate as E
    p = E.Predictor(5, 320, precision=precision, batch_size=16, autocast=autocast)
    res = E.evaluate_ensemble(p, _state_dicts(n, precision), eval_set[0], eval_set[1])
    assert p.captures == 1
    return res


@pytest.mark.gpu
def test_predictor_fp32_matches_reference(gold, eval_set, no_tf32):
    """The gates of test_eval.py::test_ensemble_eval_fp32_matches_reference (3 checkpoints)."""
    n = min(3, gold['per_model'].shape[0])
    res = _ensemble(gold, eval_set, 'fp32', None, n)
    want = torch.from_numpy(gold['per_model'][:n])
    got = res['per_model'].cpu()
    spread, err = float(want.std(1).min()), float((got - want).abs().max())
    print(f'Predictor fp32: max logit error {err:.3g}, spread {spread:.3g}')
    assert err < 5e-4 * max(1.0, float(want.abs().max())) and err < 0.05 * spread, (err, spread)
    for i in range(n):
        np.testing.assert_allclose(_auroc(got[i], eval_set[1]), gold['auroc_per_model'][i], rtol=0, atol=1e-3)
    ref_loss = torch.nn.BCEWithLogitsLoss(reduction='none')
    el = torch.stack([ref_loss(z, eval_set[1]) for z in want], 2).mean(2).mean(0)
    np.testing.assert_allclose(res['loss'].cpu().numpy(), el.numpy(), rtol=2e-4, atol=2e-5)


def _bf16_gates(gold, eval_set, res, what, auroc_gates=True):
    n = gold['per_model'].shape[0]
    want = torch.from_numpy(gold['per_model'])
    got = res['per_model'].cpu()
    d = np.abs(res['auroc'].cpu().double().numpy() - gold['auroc_mean'])
    dm = np.abs(np.stack([_auroc(got[i], eval_set[1]) for i in range(n)]) - gold['auroc_per_model'])
    print(f'{what}: max logit error {float((got - want).abs().max()):.3g}; ensemble AUROC |diff| per class {d}; '
          f'per-checkpoint AUROC |diff| max {dm.max():.3g} mean {dm.mean():.3g}')
    assert torch.allclose(got, want, rtol=2e-2, atol=1e-2), float((got - want).abs().max())
    np.testing.assert_allclose(res['outputs'].cpu().numpy(), gold['mean'], rtol=2e-2, atol=1e-2)
    if auroc_gates:
        assert d.max() < 2e-3 and d.mean() < 1e-3, d
        assert dm.max() < 4e-3 and dm.mean() < 1e-3, dm


@pytest.mark.gpu
def test_predictor_bf16_matches_reference(gold, eval_set, no_tf32):
    """The gates of test_eval.py::test_ensemble_eval_bf16_auroc (all 10 checkpoints): bf16 AAConv2d kernels, fp32 dense blocks."""
    _bf16_gates(gold, eval_set, _ensemble(gold, eval_set, 'bf16', False, gold['per_model'].shape[0]), 'Predictor bf16')


@pytest.mark.gpu
def test_predictor_bf16_autocast_matches_reference(gold, eval_set, no_tf32):
    """bf16 with the dense blocks under autocast (bf16 activations and weights, opt-in): logits within rtol 2e-2 / atol 1e-2 of the
    reference.  Measured on a B200 it misses the bf16 mode's AUROC gates (ensemble up to 3.6e-3 per class, against 2e-3), which is why
    Predictor does not use autocast unless asked; the deltas are printed, not gated."""
    _bf16_gates(gold, eval_set, _ensemble(gold, eval_set, 'bf16', True, gold['per_model'].shape[0]), 'Predictor bf16 autocast',
                auroc_gates=False)


@pytest.mark.gpu
def test_predictor_graph_replays_the_eager_step_bit_for_bit(eval_set):
    from chexpert_b200.evaluate import Predictor
    images = eval_set[0][:32]
    sds = _state_dicts(2, 'bf16')
    pe, pg = Predictor(cuda_graph=False), Predictor(cuda_graph=True)
    pe.load_state_dict(sds[0])
    pg.load_state_dict(sds[0])
    pg(images)                                    # two eager warm-up batches
    assert pg.captures == 0
    full = pg(images)                             # capture at the first batch, then replays
    assert pg.captures == 1
    assert torch.equal(full, pe(images))
    pg(images[:16])                               # the static input now holds images 0..15
    ragged = pg(images[16:26])                    # rows 10..15 of the replayed batch: images 10..15, sliced off
    assert ragged.shape == (10, 5) and torch.equal(ragged, full[16:26])
    pe.load_state_dict(sds[1])
    pg.load_state_dict(sds[1])
    again = pg(images)
    assert pg.captures == 1
    assert torch.equal(again, pe(images)) and not torch.equal(again, full)
