"""Grad-CAM at features.norm5 (chexpert_b200/gradcam.py, csrc/cam.cu, DenseNet.forward_grad_cam, Predictor.grad_cam).

CPU: the closed form the kernel computes equals torch.autograd Grad-CAM, in float64, on small DenseNets of both kinds; the
forward_grad_cam refusals.  GPU: the kernel against the float64 closed form at the models' norm5 geometries and the edges, its
upsampling against F.interpolate, its limits, determinism; Predictor.grad_cam against float64 autograd Grad-CAM on the module path,
gated against PyTorch's own fp32 / autocast execution of it, and its CUDA graphs.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from chexpert_b200 import _lib, densenet, fused_bn
from chexpert_b200.aaconv import _ptr, _stream
from oracle.model_oracle import RefDenseNet, ref_aadensenet121


# ------------------------------------------------------------------------------------------------ references
def closed_form(x, norm5, W):
    """float64 Grad-CAM at norm5's output from its input x: (cam, pre-ReLU map).  `mask` of A > 0 is computed here unless given."""
    return closed_form_masked(x, norm5, W, None)


def _affine64(x, norm5):
    w, b = norm5.weight.double(), norm5.bias.double()
    m, v = norm5.running_mean.double(), norm5.running_var.double()
    s = w / (v + norm5.eps).sqrt()
    t = b - m * s
    return x.double() * s[None, :, None, None] + t[None, :, None, None], s, t


def closed_form_masked(x, norm5, W, mask):
    A, _, _ = _affine64(x, norm5)
    n = A.shape[2] * A.shape[3]
    mk = (A > 0 if mask is None else mask).double().sum((2, 3))                      # (B, C)
    alpha = W.double()[None] * mk[:, None, :] / (n * n)                             # (B, K, C)
    pre = torch.einsum('bkc,bchw->bkhw', alpha, A)
    return pre.clamp_min(0), pre, alpha, A


def autograd_grad_cam(model, x, classes):
    """Grad-CAM as a user computes it today: a forward hook on model.features captures its output (the model goes on with a clone:
    DenseNet._features applies an in-place ReLU to it), autograd.grad of each class's summed logit.  -> (logits, (B, K, h, w))."""
    store = {}

    def hook(m, i, o):
        store['A'] = o
        return o.clone()
    h = model.features.register_forward_hook(hook)
    try:
        with torch.enable_grad():
            xx = x.detach().requires_grad_(True)         # the hooked tensor needs a graph behind it
            z = model(xx)
            A = store['A']
            maps = []
            for c in range(classes):
                g, = torch.autograd.grad(z[:, c].sum(), A, retain_graph=True)
                alpha = g.mean((2, 3), keepdim=True)
                maps.append(torch.relu((alpha * A).sum(1)))
    finally:
        h.remove()
    return z.detach(), torch.stack(maps, 1).detach()


def _random_stats(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                C = m.num_features
                m.running_mean.copy_(torch.randn(C, generator=g) * 0.3)
                m.running_var.copy_(0.5 + torch.rand(C, generator=g))
                m.weight.copy_(torch.randn(C, generator=g))
                m.bias.copy_(torch.randn(C, generator=g) * 0.5)
        model.classifier.weight.copy_(torch.randn(model.classifier.weight.shape, generator=g))
        model.classifier.weight[2] = 0                       # class 2: no weight, its map must be 0
        model.classifier.bias.copy_(torch.randn(model.classifier.bias.shape, generator=g) + 1)


def _small(kind):
    torch.manual_seed(0)
    if kind == 'attention':
        m, size = RefDenseNet(16, (2, 2), 32, {'k': 0.2, 'v': 0.1, 'nh': 2, 'relative': True}, (48, 48)), 48
    else:
        m, size = densenet.DenseNet(growth_rate=8, block_config=(2, 3), num_init_features=16, num_classes=5), 12
    _random_stats(m, 1)
    return m.double().eval(), torch.randn(3, 3, size, size, generator=torch.Generator().manual_seed(2), dtype=torch.float64)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize('kind', ['attention', 'plain'])
def test_closed_form_is_autograd_grad_cam(kind):
    model, x = _small(kind)
    store = {}
    h = model.features.norm5.register_forward_pre_hook(lambda m, i: store.__setitem__('X', i[0].detach().clone()))
    try:
        logits, want = autograd_grad_cam(model, x, 5)
    finally:
        h.remove()
    got, pre, _, A = closed_form(store['X'], model.features.norm5, model.classifier.weight)
    assert bool((A < 0).any()) and bool((A > 0).any())
    assert float(want.abs().max()) > 0
    torch.testing.assert_close(got, want, rtol=1e-10, atol=1e-12 * float(want.abs().max()))
    assert bool((got[:, 2] == 0).all()) and bool((want[:, 2] == 0).all())
    with torch.no_grad():                                # the classifier bias moves the logits, not the maps
        model.classifier.bias.add_(3.0)
    logits2, want2 = autograd_grad_cam(model, x, 5)
    assert not torch.allclose(logits2, logits)
    torch.testing.assert_close(want2, want, rtol=1e-12, atol=0)


def test_forward_grad_cam_refusals():
    model = densenet.DenseNet(growth_rate=8, block_config=(2, 3), num_init_features=16, num_classes=5)
    x = torch.randn(2, 3, 12, 12)
    with torch.no_grad(), pytest.raises(RuntimeError, match='eval mode only'):
        model.train().forward_grad_cam(x)
    model.eval()
    with pytest.raises(RuntimeError, match='autograd off'):
        model.forward_grad_cam(x)
    with torch.no_grad(), pytest.raises(RuntimeError, match='CUDA only'):
        model.forward_grad_cam(x)


def test_grad_cam_binding_refuses_cpu_tensors():
    from chexpert_b200.gradcam import grad_cam
    bn, lin = torch.nn.BatchNorm2d(8).eval(), torch.nn.Linear(8, 5)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        grad_cam(torch.randn(2, 8, 4, 4), bn, lin)


# ------------------------------------------------------------------------------------------------ GPU: the kernel
EPS = 1e-5
# (name, C, h, w, S): norm5 of both archs at 320 / 512 px (10 x 10, 16 x 16), densenet121 at 227 px (7 x 7), the 64 x 64 map of a
# 2048-px input, 1 x 1 and an odd 3 x 5
GEOMS = [('norm5_320', 1024, 10, 10, 320), ('norm5_512', 1024, 16, 16, 512), ('densenet121_227', 1024, 7, 7, 227),
         ('map64', 1024, 64, 64, 256), ('map1x1', 1024, 1, 1, 16), ('odd3x5', 200, 3, 5, 37)]
BK = [(1, 1), (16, 5), (17, 14)]
DTYPES = {'fp32': torch.float32, 'bf16': torch.bfloat16}


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def eval_norm5(C, seed):
    """Eval-mode BatchNorm2d whose pre-activation straddles zero in every channel (running_mean 64 + randn, log-uniform variance,
    weights of both signs and one zero) -- the data of tests/test_inference.py."""
    g = _gen(seed)
    bn = torch.nn.BatchNorm2d(C, eps=EPS).cuda().eval()
    with torch.no_grad():
        bn.running_mean.copy_(64 + torch.randn(C, generator=g, device='cuda'))
        bn.running_var.copy_(10 ** (-3 + 5 * torch.rand(C, generator=g, device='cuda')))
        sign = torch.where(torch.rand(C, generator=g, device='cuda') < 0.3, -1.0, 1.0)
        bn.weight.copy_(sign * (0.25 + torch.rand(C, generator=g, device='cuda')))
        bn.weight[min(3, C - 1)] = 0
        bn.bias.copy_(torch.rand(C, generator=g, device='cuda') - 0.5)
    return bn


def features(B, C, h, w, bn, dtype, seed, extra=0):
    """(B, C, h, w) of `dtype`, the first C channels of a (B, C + extra, h, w) buffer when extra > 0."""
    g = _gen(seed)
    m, s = bn.running_mean.double()[None, :, None, None], bn.running_var.double().sqrt()[None, :, None, None]
    x = (m + s * torch.randn(B, C, h, w, generator=g, device='cuda', dtype=torch.float64)).to(dtype)
    if not extra:
        return x
    buf = torch.randn(B, C + extra, h, w, generator=g, device='cuda').to(dtype)
    buf[:, :C] = x
    return buf[:, :C]


def classifier_weight(K, C, seed):
    W = torch.randn(K, C, generator=_gen(seed), device='cuda') / C ** 0.5
    if K > 1:
        W[1] = 0                                          # a class without weight: its map is 0
    return W


GUARD = 64


def run_kernel(x, bn, W, S=None, expect=0):
    """aaconv_grad_cam into NaN-filled outputs with NaN guard bands on both sides -> (code, cam, up)."""
    B, C, h, w = x.shape
    K = W.shape[0]
    cam_buf = torch.full((2 * GUARD + B * K * h * w,), float('nan'), device='cuda')
    up_buf = torch.full((2 * GUARD + B * K * S * S,), float('nan'), device='cuda') if S else None
    ws = torch.empty(B * C, device='cuda', dtype=torch.int32)
    lib = _lib.load()
    code = lib.aaconv_grad_cam(_ptr(x), _lib.BF16 if x.dtype == torch.bfloat16 else _lib.FP32, B, C, h, w, x.stride(0), _ptr(bn.weight),
                               _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var), EPS, _ptr(W), K,
                               _ptr(cam_buf[GUARD:]), _ptr(up_buf[GUARD:]) if S else None, S or 0, _ptr(ws), _stream())
    if code:
        return code, None, None
    torch.cuda.synchronize()
    for what, buf in (('cam', cam_buf), ('up', up_buf)):
        if buf is not None:
            assert bool(buf[:GUARD].isnan().all()) and bool(buf[-GUARD:].isnan().all()), f'{what}: written outside its extent'
            assert not bool(buf[GUARD:-GUARD].isnan().any()), f'{what}: not written in full'
    cam = cam_buf[GUARD:-GUARD].view(B, K, h, w)
    up = up_buf[GUARD:-GUARD].view(B, K, S, S) if S else None
    return code, cam, up


@pytest.mark.gpu
@pytest.mark.parametrize('layout', ['dense', 'strided'])
@pytest.mark.parametrize('dtype', list(DTYPES))
@pytest.mark.parametrize('B,K', BK)
@pytest.mark.parametrize('name,C,h,w,S', GEOMS)
def test_kernel_matches_float64_closed_form(name, C, h, w, S, B, K, dtype, layout):
    bn = eval_norm5(C, 3)
    x = features(B, C, h, w, bn, DTYPES[dtype], 1, extra=8 if layout == 'strided' else 0)
    W = classifier_weight(K, C, 5)
    keep = [t.clone() for t in (x, bn.weight, bn.bias, bn.running_mean, bn.running_var, W)]
    code, cam, up = run_kernel(x, bn, W, S)
    assert code == 0, _lib.load().aaconv_last_error().decode()
    assert all(torch.equal(a, b) for a, b in zip((x, bn.weight, bn.bias, bn.running_mean, bn.running_var, W), keep)), 'an input changed'
    # the zero set of the eval kernel on the same input, so that near-ties take the kernel's side
    with torch.no_grad():
        mask = fused_bn.bn_relu_eval(bn, x) > 0
    ref, pre, alpha, A = closed_form_masked(x, bn, W, mask)
    # per element: fp32 rounding of the affine (cancellation of |x s| against |mean s|) and of the C-term sum, relative to the
    # magnitudes that enter them
    _, s, t = _affine64(x, bn)
    mag = x.double().abs() * s.abs()[None, :, None, None] + t.abs()[None, :, None, None] + A.abs()
    bound = 2e-5 * torch.einsum('bkc,bchw->bkhw', alpha.abs(), mag) + 1e-30
    err = (cam.double() - ref).abs()
    worst = float((err / bound).max())
    print(f'{name} B={B} K={K} {dtype} {layout}: worst error {worst:.3g} of its bound, max map {float(ref.abs().max()):.3g}')
    assert worst <= 1.0, worst
    if K > 1:
        assert bool((cam[:, 1] == 0).all())
    want_up = F.interpolate(cam, size=(S, S), mode='bilinear', align_corners=False)
    e_up = float((up - want_up).abs().max())
    assert e_up <= 1e-6 * float(want_up.abs().max()) + 1e-30, e_up


@pytest.mark.gpu
def test_kernel_is_deterministic_and_per_image():
    C, h, w, K, S = 1024, 10, 10, 5, 320
    bn = eval_norm5(C, 3)
    x = features(16, C, h, w, bn, torch.float32, 1)
    W = classifier_weight(K, C, 5)
    _, cam1, up1 = run_kernel(x, bn, W, S)
    _, cam2, up2 = run_kernel(x, bn, W, S)
    assert torch.equal(cam1, cam2) and torch.equal(up1, up2)
    perm = torch.randperm(16, generator=torch.Generator().manual_seed(0)).cuda()
    _, cam3, up3 = run_kernel(x[perm].contiguous(), bn, W, S)
    assert torch.equal(cam3, cam1[perm]) and torch.equal(up3, up1[perm])
    _, cam4, up4 = run_kernel(x[5:6].contiguous(), bn, W, S)
    assert torch.equal(cam4, cam1[5:6]) and torch.equal(up4, up1[5:6])


@pytest.mark.gpu
def test_kernel_rejects_what_it_does_not_support():
    lib = _lib.load()
    bn = eval_norm5(4097, 3)
    W = classifier_weight(65, 4097, 5)
    x = torch.zeros(2, 4097, 65, 65, device='cuda')
    cam = torch.empty(2 * 65 * 65 * 65 * 65, device='cuda')
    up = torch.empty(2 * 65 * 4097 * 4, device='cuda')
    ws = torch.empty(2 * 4097, device='cuda', dtype=torch.int32)

    def call(B=2, C=1024, h=10, w=10, K=5, S=320, xbs=None, dtype=_lib.FP32, xp=None, up_=up):
        return lib.aaconv_grad_cam(xp if xp is not None else _ptr(x), dtype, B, C, h, w, C * h * w if xbs is None else xbs,
                                   _ptr(bn.weight), _ptr(bn.bias), _ptr(bn.running_mean), _ptr(bn.running_var), EPS, _ptr(W), K,
                                   _ptr(cam), _ptr(up_) if up_ is not None else None, S, _ptr(ws), _stream())
    cases = [
        (dict(C=4097), 'C 4097 outside [1, 4096]'), (dict(C=0), 'C 0 outside [1, 4096]'),
        (dict(h=65, w=64), 'h*w at most 4096 (64 x 64)'), (dict(h=0), 'h*w at most 4096'),
        (dict(K=0), 'K 0 outside [1, 64] classes'), (dict(K=65), 'K 65 outside [1, 64] classes'),
        (dict(S=0), 'S 0 outside [1, 4096]'), (dict(S=4097), 'S 4097 outside [1, 4096]'),
        (dict(B=0), 'B 0 outside [1, 65535]'), (dict(B=65536), 'B 65536 outside [1, 65535]'),
        (dict(xbs=1024 * 100 - 1), 'x_batch_stride 102399 below C*h*w'),
        (dict(dtype=2), 'neither fp32 nor bf16'),
        (dict(xp=torch.empty(16, dtype=torch.uint8, device='cuda').data_ptr() + 2), 'aligned to its 4-byte element'),
    ]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        text = lib.aaconv_last_error().decode()
        assert msg in text, (kw, text)
    assert call(S=0, up_=None) == 0                              # without `up` S is not read
    assert call(C=4096, h=64, w=64, K=64, S=4) == 0              # every limit itself is accepted
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ GPU: model and Predictor
@pytest.fixture
def no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _state_dict(arch, seed):
    """aadensenet121 seed 0 is checkpoint 0 of tests/golden/eval_ensemble.npz; densenet121 is seed-initialised the same way."""
    torch.manual_seed(seed)
    return densenet.build_model(arch, 5, 320, 'bf16').state_dict()


def _module_model(arch, sd):
    m = ref_aadensenet121((320, 320)) if arch == 'aadensenet121' else densenet.densenet121(5)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


def _ref_maps(model, x, dtype, autocast=False):
    m = model.to(dtype)
    with torch.autocast('cuda', dtype=torch.bfloat16, enabled=autocast):
        logits, cam = autograd_grad_cam(m, x.to(dtype), 5)
    up = F.interpolate(cam.double(), size=(320, 320), mode='bilinear', align_corners=False)
    return logits.double(), up


def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max())


# (Predictor precision, autocast, control): PyTorch's own execution the case is gated against
MODES = {'fp32': ('fp32', False), 'bf16': ('bf16', False), 'bf16_autocast': ('bf16', True)}
VS_CONTROL = 4.0


@pytest.mark.gpu
@pytest.mark.parametrize('mode', list(MODES))
@pytest.mark.parametrize('arch', ['aadensenet121', 'densenet121'])
def test_predictor_grad_cam_matches_float64_autograd(arch, mode, no_tf32):
    """Predictor.grad_cam over 16 synthetic radiographs against float64 autograd Grad-CAM on the module path (same checkpoint),
    upsampled to 320 px in float64.  Gate: its max error (relative to the largest map value) within VS_CONTROL times that of the
    control -- the same autograd Grad-CAM run by PyTorch in fp32 (fp32 mode) or under bf16 autocast (bf16 modes) -- plus 1e-4."""
    from chexpert_b200.evaluate import Predictor, normalise_u8, synthetic_radiographs_u8
    precision, autocast = MODES[mode]
    sd = _state_dict(arch, 0)
    images = synthetic_radiographs_u8(16, 320, seed=3)
    p = Predictor(5, 320, precision=precision, batch_size=16, autocast=autocast, cuda_graph=False, arch=arch)
    p.load_state_dict(sd)
    logits, maps = p.grad_cam(images)
    assert logits.shape == (16, 5) and maps.shape == (16, 5, 320, 320) and maps.dtype == torch.float32
    assert torch.equal(logits, p(images))
    x = normalise_u8(images.cuda())
    model = _module_model(arch, sd)
    z64, want = _ref_maps(model, x, torch.float64)
    _, ctrl = _ref_maps(model, x, torch.float32, autocast=mode != 'fp32')
    e_ours, e_ctrl = _rel(maps, want), _rel(ctrl, want)
    e_logits = float((logits.double() - z64).abs().max())
    print(f'{arch} {mode}: maps error {e_ours:.3g} of max, control {e_ctrl:.3g}, ratio {e_ours / e_ctrl:.3g}; '
          f'logits error {e_logits:.3g}')
    assert e_ours <= VS_CONTROL * e_ctrl + 1e-4, (e_ours, e_ctrl)


@pytest.mark.gpu
def test_forward_grad_cam_without_feature_buffer(no_tf32):
    """The module-path densenet121 (no feature buffer): forward_grad_cam's logits are forward's, its maps the closed form of what
    norm5 reads, and a hook on model.features still fires in forward."""
    sd = _state_dict('densenet121', 0)
    model = _module_model('densenet121', sd)
    from chexpert_b200.evaluate import normalise_u8, synthetic_radiographs_u8
    x = normalise_u8(synthetic_radiographs_u8(4, 320, seed=3).cuda())
    seen, store = [], {}
    h1 = model.features.register_forward_hook(lambda m, i, o: seen.append(1))
    h2 = model.features.norm5.register_forward_pre_hook(lambda m, i: store.__setitem__('X', i[0].clone()))
    with torch.no_grad():
        z = model(x)
        logits, cam = model.forward_grad_cam(x)
    h1.remove()
    h2.remove()
    assert len(seen) == 1 and torch.equal(logits, z)
    with torch.no_grad():
        mask = fused_bn.bn_relu_eval(model.features.norm5, store['X']) > 0
    ref = closed_form_masked(store['X'], model.features.norm5, model.classifier.weight, mask)[0]
    assert _rel(cam, ref) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize('arch', ['aadensenet121', 'densenet121'])
def test_predictor_grad_cam_graphs(arch):
    """Each input form's Grad-CAM graph replays the eager step bit for bit, with a ragged tail and one capture across
    load_state_dict; raw radiographs give what their host-preprocessed uint8 crops give; a batch costs __call__'s launches plus the
    three Grad-CAM launches."""
    from chexpert_b200.evaluate import Predictor
    from tests.test_radiograph_prep import host_u8, raw_set
    raw = raw_set(32, 1)
    u8 = torch.stack([host_u8(i, 320) for i in raw])
    sds = [_state_dict(arch, s) for s in (0, 1)]
    pe = Predictor(5, 320, batch_size=16, cuda_graph=False, arch=arch)
    pg = Predictor(5, 320, batch_size=16, cuda_graph=True, arch=arch)
    for p in (pe, pg):
        p.load_state_dict(sds[0])
    want_z, want_m = pe.grad_cam(u8)
    rz, rm = pe.grad_cam(raw)
    assert torch.equal(rz, want_z) and torch.equal(rm, want_m)
    for form in (u8, raw):
        captures = pg.captures
        z, m = pg.grad_cam(form)                           # two eager warm-up batches
        assert pg.captures == captures
        assert torch.equal(z, want_z) and torch.equal(m, want_m)
        z, m = pg.grad_cam(form)                           # capture at the first batch, then a replay
        assert pg.captures == captures + 1
        assert torch.equal(z, want_z) and torch.equal(m, want_m)
        pg.grad_cam(form[:16])                             # the static input now holds images 0..15
        z, m = pg.grad_cam(form[16:26])                    # a ragged batch: rows 10..15 replay images 10..15, sliced off
        assert z.shape == (10, 5) and m.shape == (10, 5, 320, 320)
        assert torch.equal(z, want_z[16:26]) and torch.equal(m, want_m[16:26])
    assert torch.equal(pg(u8), want_z) and pg.captures == 2   # __call__ keeps its own paths: warm-up ...
    assert torch.equal(pg(u8), want_z) and pg.captures == 3   # ... and capture
    pe.load_state_dict(sds[1])
    pg.load_state_dict(sds[1])
    want_z1, want_m1 = pe.grad_cam(u8)
    assert not torch.equal(want_m1, want_m)
    for form in (u8, raw):
        z, m = pg.grad_cam(form)
        assert torch.equal(z, want_z1) and torch.equal(m, want_m1)
    assert pg.captures == 3
    pg(raw)
    pg(raw)
    assert pg.captures == 4

    def launches(fn):
        _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
        fn()
        torch.cuda.synchronize()
        return sorted(name for name, _ in _lib.profile_end())
    pg(raw)
    pg(raw)
    assert pg.captures == 4
    for form in (u8[:20], raw[:20]):
        call, cam = launches(lambda: pe(form)), launches(lambda: pe.grad_cam(form))
        extra = list(cam)
        for name in call:
            extra.remove(name)
        assert sorted(extra) == sorted(['grad_cam_count', 'grad_cam_map', 'grad_cam_upsample'] * 2), extra   # two batches
        assert launches(lambda: pg(form)) == launches(lambda: pg.grad_cam(form))   # replays: the same host launches (prep for raw)
