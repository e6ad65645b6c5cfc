"""The dense-block BatchNorm2d (training) + ReLU kernels (csrc/bn_relu.cu, csrc/bn_cl.cu) and the Transition's fused
InstanceNorm2d + ReLU prologue (csrc/prologue.cu) against float64 references written out with plain torch ops.

The host code derives the kernels' work split from (B, C, HW): groups of `bpb` batch planes (G groups, the last one possibly
smaller), reduction segments of the channels-last kernels (hundreds per channel at 80x80), channel tiles of 64.  The cases below
are aadensenet121's own BatchNorm geometries at B = 16, 320 px (stem norm0, the first and last norm1 of every dense block, the
norm2 bottleneck at every map size, norm5) plus the edges of that split.  The data gives every sample and every channel its own
offset, so group means differ by O(1): a group partial with a wrong element count, a dropped partial or a mixed-up segment moves
the statistics far past the gates, which i.i.d. data would hide.
"""
import ctypes
import math

import pytest
import torch

from chexpert_b200 import _lib, densenet, fused_bn
from chexpert_b200.aaconv import _ptr, _stream

EPS, MOM = 1e-5, 0.1
CL = torch.channels_last
BIG, CONST = 1, 2          # channel 64 + randn (cancellation in the variance), channel constant over the batch (variance 0)

# ---- gates (per channel, relative to that channel's largest |reference| unless said otherwise) ----
# fp32 y and dx: the kernels sum in fp32 over groups and segments of at most a few hundred elements per thread, so x^ and the
# gradient means carry relative errors of order 1e-6; 2e-5 leaves a margin of about ten.
TOL32 = 2e-5
# saved / running statistics: rstd and running var relative; mean within TOL_STAT of the channel's standard deviation
# sqrt(var + eps).  A channel whose |mean| is far above its standard deviation (BIG: 64 against 1) holds its fp32 mean only to
# an ulp of |mean| per rounded step of the Chan merge, so MEAN_ULPS ulps of |mean| are allowed on top.
TOL_STAT = 1e-5
MEAN_ULPS = 8 * 2.0 ** -24
# bf16 y and dx: computed in fp32 and rounded once to bf16.  bf16 keeps 8 significant bits, so half an ulp is up to 2^-8 of the
# value (just above a power of two); the fp32 error before the rounding goes into the 1e-4 max|ref| term.
#   |got - ref| <= 2^-8 |ref| + 1e-4 max|ref|
BF16_REL, BF16_ABS = 2.0 ** -8, 1e-4
# dweight / dbias: relative to the largest |reference| over all channels.  dy and x both have per-sample offsets, so both sums
# grow like n and their fp32 summation error stays near 1e-6 of it.
TOL_W = 1e-5
# ReLU near ties: the kernel's mask comes from an fp32 pre-activation, the reference's from float64.  Elements with
# |w x^ + b| < TIE may fall on either side; they leave the elementwise dx check (and must be fewer than TIE_FRAC of the
# elements) and widen their channel's dw / db bound by sum |dy| (1 + |x^|).  A tie on the other side also moves the channel's
# sums (sum g, sum g x^) and through them dx = k (g - sum g / n - x^ sum g x^ / n) at every other element of the channel, by up to
# k / n (sum |dy| + |x^| sum |dy x^|) over the ties (tie_allowance): at n = 1600 (10x10, B = 16) one tie moves a whole channel's dx
# by some 1e-4 of its max, above TOL32.
TIE, TIE_FRAC = 1e-5, 1e-4


# ------------------------------------------------------------------------------------------------ data and reference
def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _unif(shape, lo, hi, g):
    return lo + (hi - lo) * torch.rand(shape, generator=g, device='cuda', dtype=torch.float64)


def features(B, C, H, W, dtype, seed):
    """x[b, c] = off_b + off_c + s_c * randn (off_b in +-2, off_c in +-4, s_c in [0.5, 3]); channel BIG = 64 + randn, channel
    CONST = 0 everywhere.  (Any other constant has a mean that is not exact in fp32, and rstd = eps^-1/2 ~ 316 amplifies its
    rounding in y past the fp32 gate.)"""
    g = _gen(seed)
    x = (_unif((B, 1, 1, 1), -2, 2, g) + _unif((1, C, 1, 1), -4, 4, g)
         + _unif((1, C, 1, 1), 0.5, 3, g) * torch.randn(B, C, H, W, generator=g, device='cuda', dtype=torch.float64))
    x[:, BIG] = 64 + torch.randn(B, H, W, generator=g, device='cuda', dtype=torch.float64)
    x[:, CONST] = 0
    return x.to(dtype)


def grad_out(B, C, H, W, dtype, seed):
    """dy with a per-sample offset (so sum dy and sum dy x^ grow like n, not like sqrt(n))."""
    g = _gen(seed)
    return (_unif((B, 1, 1, 1), -1, 1, g) + torch.randn(B, C, H, W, generator=g, device='cuda', dtype=torch.float64)).to(dtype)


def make_bn(C, seed, nbt_batched=False):
    g = _gen(seed)
    bn = torch.nn.BatchNorm2d(C, eps=EPS, momentum=MOM).cuda()
    with torch.no_grad():
        sign = torch.where(torch.rand(C, generator=g, device='cuda') < 0.25, -1.0, 1.0)
        bn.weight.copy_(sign * (0.5 + torch.rand(C, generator=g, device='cuda')))
        bn.bias.copy_(torch.rand(C, generator=g, device='cuda') - 0.5)
        bn.bias[CONST] = 0.3                       # x^ = 0 there: a clear ReLU mask
        bn.running_mean.copy_(torch.randn(C, generator=g, device='cuda'))
        bn.running_var.copy_(0.5 + torch.rand(C, generator=g, device='cuda'))
    if nbt_batched:
        bn._nbt_batched = True
    return bn


class Ref:
    """Batch-statistics BatchNorm + ReLU in float64: mean, biased variance, relu((x - mean) rsqrt(var + eps) w + b); dx, dw, db by
    autograd on that graph; running statistics with the unbiased factor n / (n - 1)."""

    def __init__(self, x, w, b, dy=None, rm0=None, rv0=None):
        B, C, H, W = x.shape
        self.n = n = B * H * W
        x64 = x.detach().double().requires_grad_(dy is not None)
        w64 = w.detach().double().requires_grad_(dy is not None)
        b64 = b.detach().double().requires_grad_(dy is not None)
        mean = x64.mean((0, 2, 3))
        var = ((x64 - mean[None, :, None, None]) ** 2).mean((0, 2, 3))
        rstd = (var + EPS).rsqrt()
        xh = (x64 - mean[None, :, None, None]) * rstd[None, :, None, None]
        pre = xh * w64[None, :, None, None] + b64[None, :, None, None]
        y = torch.relu(pre)
        if dy is not None:
            y.backward(dy.double())
            self.dx, self.dw, self.db = x64.grad, w64.grad, b64.grad
            self.dy = dy.double()
        self.y, self.xh, self.pre = y.detach(), xh.detach(), pre.detach()
        self.mean, self.var, self.rstd = mean.detach(), var.detach(), rstd.detach()
        self.k = (w64.detach() * self.rstd).abs()                     # |d dx / d g|
        if rm0 is not None:
            self.rm = (1 - MOM) * rm0.double() + MOM * self.mean
            self.rv = (1 - MOM) * rv0.double() + MOM * self.var * (n / (n - 1))


def ties(ref):
    t = ref.pre.abs() < TIE
    print(f'{int(t.sum())} near-ties in {t.numel()} elements')
    assert int(t.sum()) < TIE_FRAC * t.numel(), f'{int(t.sum())} near-ties in {t.numel()} elements'
    return t


def tie_allowance(k, n, dy, xh, tie, dims):
    """What the ties (`tie`, reduced over `dims` with n elements each) can move dx by elsewhere in their reduction set, for
    dx = k (g - mean g - x^ mean g x^): k / n (sum |dy| + |x^| sum |dy x^|) over the ties (see TIE)."""
    s1 = (dy.abs() * tie).sum(dims, keepdim=True)
    s2 = (dy.abs() * xh.abs() * tie).sum(dims, keepdim=True)
    return k / n * (s1 + xh.abs() * s2)


def dx_allowance(ref, tie):
    return tie_allowance(ref.k[None, :, None, None], ref.n, ref.dy, ref.xh, tie, (0, 2, 3))


# ------------------------------------------------------------------------------------------------ gates
def _per_channel_max(t):
    return t.abs().amax((0, 2, 3))[None, :, None, None]


def check_elem(what, got, ref, dtype, skip=None, allow=None):
    """Elementwise gate, (B, C, H, W) logical layout, bound per channel (see TOL32 / BF16_REL); `skip`: elements left out,
    `allow`: added to the bound (near ties, see TIE)."""
    got, ref = got.detach().double(), ref.detach().double()
    assert got.shape == ref.shape, what
    assert torch.isfinite(got).all(), f'{what}: non-finite values'
    scale = _per_channel_max(ref)
    bound = TOL32 * scale if dtype == torch.float32 else BF16_REL * ref.abs() + BF16_ABS * scale
    if allow is not None:
        bound = bound + allow
    err = (got - ref).abs()
    if skip is not None:
        err = err.masked_fill(skip, 0.0)
    ratio = float((err / bound.clamp_min(1e-300)).max())
    print(f'{what}: worst error {ratio:.3g} of its bound')
    bad = err > bound
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f'{what}: {int(bad.sum())} elements over the gate (worst {ratio:.3g} of it), first at {i}: '
                             f'got {float(got[i]):.9g}, want {float(ref[i]):.9g}')


def check_stats(what, saved, ref):
    """saved (C, 2) = (mean, rstd) against the float64 statistics."""
    mean, rstd = saved[:, 0].double(), saved[:, 1].double()
    tol_m = TOL_STAT * (ref.var + EPS).sqrt() + MEAN_ULPS * ref.mean.abs()
    em, er = (mean - ref.mean).abs() / tol_m, (rstd - ref.rstd).abs() / (TOL_STAT * ref.rstd)
    print(f'{what}: saved mean {float(em.max()):.3g}, rstd {float(er.max()):.3g} of their bounds')
    assert float(em.max()) <= 1, f'{what}: saved mean off in channel {int(em.argmax())} ({float(em.max()):.3g} of the gate)'
    assert float(er.max()) <= 1, f'{what}: saved rstd off in channel {int(er.argmax())} ({float(er.max()):.3g} of the gate)'


def check_running(what, bn, ref):
    tol_m = TOL_STAT * (ref.var + EPS).sqrt() + MEAN_ULPS * ref.rm.abs()
    em = (bn.running_mean.double() - ref.rm).abs() / tol_m
    ev = (bn.running_var.double() - ref.rv).abs() / (TOL_STAT * ref.rv)
    print(f'{what}: running mean {float(em.max()):.3g}, running var {float(ev.max()):.3g} of their bounds')
    assert float(em.max()) <= 1, f'{what}: running mean off in channel {int(em.argmax())} ({float(em.max()):.3g} of the gate)'
    assert float(ev.max()) <= 1, f'{what}: running var off in channel {int(ev.argmax())} ({float(ev.max()):.3g} of the gate)'


def check_wb(what, dw, db, ref, tie):
    widen = (ref.dy.abs() * (1 + ref.xh.abs()) * tie).sum((0, 2, 3))
    for name, got, want in (('dweight', dw, ref.dw), ('dbias', db, ref.db)):
        bound = TOL_W * want.abs().max() + widen
        err = (got.double() - want).abs()
        print(f'{what}: {name} {float((err / bound).max()):.3g} of its bound')
        assert bool((err <= bound).all()), f'{what}: {name} off in channel {int((err / bound).argmax())}'


# ------------------------------------------------------------------------------------------------ the paths
def feature_buffer(x, extra=8, offset=0, seed=99):
    """(B, C + extra, H, W) buffer in x's dtype whose first C channels are x; its storage starts `offset` elements into an
    allocation (offset 1: no four-element alignment)."""
    B, C, H, W = x.shape
    flat = torch.empty(offset + B * (C + extra) * H * W, device='cuda', dtype=x.dtype)
    buf = flat[offset:].view(B, C + extra, H, W)
    buf[:, C:] = torch.randn(B, extra, H, W, generator=_gen(seed), device='cuda').to(x.dtype)
    buf[:, :C] = x
    return buf


def run_path(path, x, bn, dy, offset=0):
    """One forward + backward of `path` on x; -> (y, gradient as the path leaves it, what was there before (or None), saved).
    The feature buffer must be untouched, and so must the gradient channels behind the layer's input."""
    B, C, H, W = x.shape
    if path == 'cl':
        xl = x.contiguous(memory_format=CL).requires_grad_(True)
        y = fused_bn.bn_relu_cl(bn, xl)
        saved = y.grad_fn.saved_tensors[1].clone()
        y.backward(dy.contiguous(memory_format=CL))
        assert y.is_contiguous(memory_format=CL) and xl.grad.is_contiguous(memory_format=CL)
        return y, xl.grad, None, saved
    buf = feature_buffer(x, offset=offset)
    keep = buf.clone()
    xb = buf[:, :C].detach().requires_grad_(True)
    if path == 'nchw':
        y = fused_bn.bn_relu(bn, xb)
        saved = y.grad_fn.saved_tensors[1].clone()
        y.backward(dy)
        assert torch.equal(buf, keep), 'the feature buffer changed'
        return y, xb.grad, None, saved
    tap = {'tap': fused_bn.tap_bn_relu, 'tap_cl': fused_bn.tap_bn_relu_cl}[path]
    fb, y = tap(bn, xb)
    assert fb.data_ptr() == xb.data_ptr()
    saved = y.grad_fn.saved_tensors[1].clone()
    gbuf = feature_buffer(grad_out(B, C, H, W, x.dtype, 7), offset=offset, seed=98)
    g0 = gbuf.clone()
    torch.autograd.backward([fb, y], [gbuf[:, :C], dy.contiguous(memory_format=CL) if path == 'tap_cl' else dy])
    assert torch.equal(buf, keep), 'the feature buffer changed'
    assert torch.equal(gbuf[:, C:], g0[:, C:]), 'gradient channels behind the input changed'
    return y, gbuf[:, :C], g0[:, :C], saved          # checked against g0 + dx: the accumulation happened in place


def check_path(what, path, x, dy, bn, offset=0):
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    ref = Ref(x, bn.weight, bn.bias, dy, rm0, rv0)
    tie = ties(ref)
    y, dx, base, saved = run_path(path, x, bn, dy, offset)
    assert y.dtype == x.dtype and dx.dtype == x.dtype
    check_elem(f'{what} y', y, ref.y, x.dtype)
    check_elem(f'{what} dx', dx, ref.dx if base is None else ref.dx + base.double(), x.dtype, skip=tie,
               allow=dx_allowance(ref, tie))
    check_stats(what, saved, ref)
    check_running(what, bn, ref)
    assert int(bn.num_batches_tracked) == 1
    check_wb(what, bn.weight.grad, bn.bias.grad, ref, tie)


# (name, B, C, H, W, paths).  nchw = bn_relu (plain dx), tap = tap_bn_relu (dx added into the buffer gradient), tap_cl =
# tap_bn_relu_cl (NCHW prefix -> NHWC), cl = bn_relu_cl (NHWC -> NHWC).
GEOMETRIES = [
    ('stem_norm0', 16, 64, 160, 160, ('nchw',)),                    # G = 16 groups of one plane
    ('block1_norm1_first', 16, 64, 80, 80, ('tap', 'tap_cl')),      # G = 16; 1600 backward partials per channel
    ('block1_norm1_last', 16, 224, 80, 80, ('tap', 'tap_cl')),      # last channel tile 32 wide
    ('block1_norm2', 16, 128, 80, 80, ('cl', 'nchw')),              # 582 segments of 176 rows, the last one 144
    ('block2_norm1_first', 16, 128, 40, 40, ('tap', 'tap_cl')),     # bpb = 5, G = 4: groups of 5 / 5 / 5 / 1 planes
    ('block2_norm1_last', 16, 480, 40, 40, ('tap', 'tap_cl')),
    ('block2_norm2', 16, 128, 40, 40, ('cl', 'nchw')),              # 534 segments of 48 rows, the last one 16
    ('block3_norm1_first', 16, 256, 20, 20, ('tap', 'tap_cl')),     # G = 1 from here on
    ('block3_norm1_last', 16, 992, 20, 20, ('tap', 'tap_cl')),
    ('block3_norm2', 16, 128, 20, 20, ('cl', 'nchw')),
    ('block4_norm1_first', 16, 512, 10, 10, ('tap', 'tap_cl')),
    ('block4_norm1_last', 16, 992, 10, 10, ('tap', 'tap_cl')),
    ('block4_norm2', 16, 128, 10, 10, ('cl', 'nchw')),
    ('norm5', 16, 1024, 10, 10, ('nchw',)),
    ('hw49_two_groups', 200, 32, 7, 7, ('nchw', 'tap')),            # scalar path, G = 2 with a last group of 33 planes
    ('c36_partial_tile', 16, 36, 40, 40, ('nchw', 'tap', 'tap_cl', 'cl')),
    ('batch1', 1, 64, 10, 10, ('nchw', 'tap', 'tap_cl', 'cl')),
    ('batch17', 17, 128, 40, 40, ('nchw', 'tap', 'tap_cl', 'cl')),  # last group of 2 planes
]
CASES = [pytest.param(B, C, H, W, path, id=f'{name}-{path}') for name, B, C, H, W, paths in GEOMETRIES for path in paths]
DTYPES = [pytest.param(torch.float32, id='fp32'), pytest.param(torch.bfloat16, id='bf16')]


# ------------------------------------------------------------------------------------------------ CPU: the reference itself
def test_reference_matches_torch_batch_norm_in_float64():
    B, C, H, W = 3, 5, 4, 6
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 3 + 1
    w, b = torch.rand(C, generator=g, dtype=torch.float64) + 0.5, torch.rand(C, generator=g, dtype=torch.float64) - 0.5
    dy = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    rm0, rv0 = torch.randn(C, dtype=torch.float64), torch.rand(C, dtype=torch.float64) + 0.5
    ref = Ref(x, w, b, dy, rm0, rv0)
    xt, wt, bt = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    rm, rv = rm0.clone(), rv0.clone()
    yt = torch.relu(torch.nn.functional.batch_norm(xt, rm, rv, wt, bt, True, MOM, EPS))
    yt.backward(dy)
    for got, want in ((ref.y, yt), (ref.dx, xt.grad), (ref.dw, wt.grad), (ref.db, bt.grad), (ref.rm, rm), (ref.rv, rv)):
        assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------ GPU: every path, every geometry
@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('B,C,H,W,path', CASES)
def test_bn_relu_paths_match_float64(B, C, H, W, path, dtype):
    x, dy = features(B, C, H, W, dtype, 1), grad_out(B, C, H, W, dtype, 2)
    check_path(f'{path} {B}x{C}x{H}x{W} {dtype}', path, x, dy, make_bn(C, 3))


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('path', ['nchw', 'tap'])
def test_misaligned_input_takes_the_scalar_path(path, dtype):
    """x one element past four-element alignment: unit = 1 although HW % 4 == 0 (the gradient buffer is misaligned alike)."""
    B, C, H, W = 17, 64, 20, 20
    x, dy = features(B, C, H, W, dtype, 1), grad_out(B, C, H, W, dtype, 2)
    check_path(f'misaligned {path} {dtype}', path, x, dy, make_bn(C, 3), offset=1)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('tap', ['tap', 'tap_cl'])
@pytest.mark.parametrize('g_feats', ['none', 'misaligned', 'channels_last'])
def test_tap_backward_fallbacks(tap, g_feats, dtype):
    """The backward of the tap ops when the gradient of the concatenation is missing or cannot be accumulated into in place: a
    dense dx (bn_bwd_dx / t_bwd_dx without accumulation), plus the given gradient."""
    B, C, H, W = 17, 36, 40, 40
    x, dy = features(B, C, H, W, dtype, 1), grad_out(B, C, H, W, dtype, 2)
    bn = make_bn(C, 3)
    ref = Ref(x, bn.weight, bn.bias, dy)
    tie = ties(ref)
    xb = feature_buffer(x)[:, :C].detach().requires_grad_(True)
    fn, fwd = {'tap': (fused_bn._TapBNReLU, fused_bn.tap_bn_relu), 'tap_cl': (fused_bn._TapBNReLUCL, fused_bn.tap_bn_relu_cl)}[tap]
    _, y = fwd(bn, xb)
    gf = None
    if g_feats != 'none':
        g = grad_out(B, C, H, W, dtype, 7)
        gf = (torch.empty(B * C * H * W + 1, device='cuda', dtype=dtype)[1:].view(B, C, H, W) if g_feats == 'misaligned'
              else torch.empty_like(g, memory_format=CL))
        gf.copy_(g)
        assert gf.data_ptr() % (4 * gf.element_size()) != 0 or not gf.is_contiguous()
    g_keep = None if gf is None else gf.clone()
    dyy = dy.contiguous(memory_format=CL) if tap == 'tap_cl' else dy
    dx, dw, db = fn.backward(y.grad_fn, gf, dyy)[:3]           # y.grad_fn is the op's ctx
    if gf is not None:
        if tap == 'tap' and g_feats == 'misaligned':
            assert dx is gf                                      # the NCHW tap accumulates in place through scalar accesses
        else:
            assert dx.data_ptr() != gf.data_ptr() and torch.equal(gf, g_keep)
    want = ref.dx if gf is None else ref.dx + g_keep.double()
    allow = dx_allowance(ref, tie)
    if gf is not None and dx is not gf and dtype == torch.bfloat16:
        allow = allow + BF16_REL * ref.dx.abs()      # dx is rounded to bf16 before the add, which rounds again
    check_elem(f'{tap} fallback ({g_feats}) dx', dx, want, dtype, skip=tie, allow=allow)
    check_wb(f'{tap} fallback ({g_feats})', dw, db, ref, tie)


# ------------------------------------------------------------------------------------------------ GPU: running statistics
@pytest.mark.gpu
@pytest.mark.parametrize('nbt_batched', [False, True])
@pytest.mark.parametrize('B,C,H,W,path', [(17, 128, 40, 40, 'tap_cl'), (16, 64, 10, 10, 'tap'), (1, 64, 10, 10, 'nchw'),
                                          (16, 128, 10, 10, 'cl')])
def test_running_statistics_over_two_calls(B, C, H, W, path, nbt_batched):
    bn = make_bn(C, 3, nbt_batched)
    for call in (1, 2):
        x, dy = features(B, C, H, W, torch.float32, 10 + call), grad_out(B, C, H, W, torch.float32, 20 + call)
        ref = Ref(x, bn.weight, bn.bias, None, bn.running_mean.clone(), bn.running_var.clone())
        bn.weight.grad = bn.bias.grad = None
        run_path(path, x, bn, dy)
        check_running(f'{path} call {call}', bn, ref)
        assert int(bn.num_batches_tracked) == (0 if nbt_batched else call)


# ------------------------------------------------------------------------------------------------ GPU: statistics shared along a block
def _groups(x):
    """(G, bpb) of the shared partial buffer for x, as the library reports them (no channel is reduced: valid == C)."""
    lib, B, C, H, W = _lib.load(), *x.shape
    G, bpb = ctypes.c_int(0), ctypes.c_int(0)
    ws = torch.empty(2 * B * C, device='cuda', dtype=torch.float32)
    _lib.check(lib.aaconv_bn_stats_nchw(_ptr(x), _lib.FP32 if x.dtype == torch.float32 else _lib.BF16, B, C, H * W, x.stride(0),
                                        _ptr(ws), C, ctypes.byref(G), ctypes.byref(bpb), _stream()), 'aaconv_bn_stats_nchw')
    return G.value, bpb.value


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('tap', ['tap', 'tap_cl'])
@pytest.mark.parametrize('B,C0,H,W', [(16, 128, 40, 40), (16, 256, 20, 20)])
def test_dense_block_shares_statistics(B, C0, H, W, tap, dtype):
    """Layer i of a dense block normalises channels [0, c_i) of the buffer and reduces only [c_{i-1}, c_i): the rest comes from
    the partials layer i-1 left in the block's stats buffer.  Every layer must still match the float64 reference on its prefix;
    and a shifted channel-0 partial (layout c * G + group, float2 (mean, M2)) must move the next layer's channel 0."""
    n, k = 3, 32
    buf = features(B, C0 + n * k, H, W, dtype, 5)
    stats = torch.empty(2 * B * buf.shape[1], device='cuda', dtype=torch.float32)
    fwd = {'tap': fused_bn.tap_bn_relu, 'tap_cl': fused_bn.tap_bn_relu_cl}[tap]
    G = _groups(buf)[0]
    valid = 0
    for i in range(n + 1):
        c = C0 + i * k
        bn = make_bn(c, 30 + i)
        ref = Ref(buf[:, :c], bn.weight, bn.bias, None, bn.running_mean.clone(), bn.running_var.clone())
        _, y = fwd(bn, buf[:, :c].detach().requires_grad_(True), (stats, valid))
        saved = y.grad_fn.saved_tensors[1]
        if i < n:
            check_elem(f'layer {i} y', y, ref.y, dtype)
            check_stats(f'layer {i}', saved, ref)
            check_running(f'layer {i}', bn, ref)
            if i == n - 1:
                stats.view(-1, 2)[:G, 0] += 5 * float(ref.var[0].sqrt())     # channel 0's group means, as the next layer reads them
        else:                                                                   # the control: only channel 0 moves, and far
            check_elem(f'layer {i} y, channels 1..', y[:, 1:], ref.y[:, 1:], dtype)
            moved = float((y[:, 0].double() - ref.y[:, 0]).abs().max() / ref.y[:, 0].abs().max())
            assert moved > 0.1, f'channel 0 ignored the shared partials (moved {moved:.3g} of its max)'
            assert abs(float(saved[0, 0]) - float(ref.mean[0]) - 5 * float(ref.var[0].sqrt())) < 1e-3 * float(ref.var[0].sqrt())
        valid = c


# ------------------------------------------------------------------------------------------------ GPU: the C ABI's outputs
def _nan(n, dtype, margin=64):
    return torch.full((n + margin,), float('nan'), device='cuda', dtype=dtype)


def _margin_nan(t, n, what):
    assert bool(torch.isnan(t[n:]).all()), f'{what}: written past its end'


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('side', ['nchw', 'tap_cl', 'cl'])
def test_abi_writes_exactly_its_outputs(side, dtype):
    """Through the C ABI with CUDA tensors: y, saved, dx, dw and db are pre-filled with NaN and carry a NaN margin; every element
    must be written (and right), nothing behind; the feature buffer is not written; the accumulating backward leaves the gradient
    channels [C, Ctot) bit-identical."""
    lib = _lib.load()
    dt = _lib.FP32 if dtype == torch.float32 else _lib.BF16
    B, C, H, W = 17, 36, 40, 40
    HW, n = H * W, B * C * H * W
    x, dy = features(B, C, H, W, dtype, 1), grad_out(B, C, H, W, dtype, 2)
    bn = make_bn(C, 3)
    w, b = bn.weight.detach(), bn.bias.detach()
    ref = Ref(x, w, b, dy, bn.running_mean.clone(), bn.running_var.clone())
    tie = ties(ref)
    buf = feature_buffer(x)
    keep = buf.clone()
    xs = buf[:, :C]
    y, saved = _nan(n, dtype), _nan(2 * C, torch.float32)
    st = _stream()
    if side == 'nchw':
        ws = torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C) // 4, device='cuda', dtype=torch.float32)
        _lib.check(lib.aaconv_bn_relu_forward(_ptr(xs), dt, B, C, HW, xs.stride(0), _ptr(w), _ptr(b), _ptr(bn.running_mean),
                                              _ptr(bn.running_var), MOM, EPS, _ptr(y), _ptr(saved), _ptr(ws), 0, st), 'forward')
        y_nchw = y[:n].view(B, C, H, W)
    else:
        ws = torch.empty(lib.aaconv_bn_relu_cl_workspace_bytes(B, C, HW), device='cuda', dtype=torch.uint8)
        if side == 'tap_cl':
            pst = torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C) // 4, device='cuda', dtype=torch.float32)
            G, bpb = ctypes.c_int(0), ctypes.c_int(0)
            _lib.check(lib.aaconv_bn_stats_nchw(_ptr(xs), dt, B, C, HW, xs.stride(0), _ptr(pst), 0, ctypes.byref(G), ctypes.byref(bpb),
                                                st), 'stats')
            _lib.check(lib.aaconv_bn_relu_cl_forward(_ptr(xs), dt, B, C, HW, 0, xs.stride(0), _ptr(w), _ptr(b), _ptr(bn.running_mean),
                                                     _ptr(bn.running_var), MOM, EPS, _ptr(y), _ptr(saved), _ptr(ws), _ptr(pst),
                                                     G.value, bpb.value, st), 'cl forward')
        else:
            xs = x.contiguous(memory_format=CL)
            _lib.check(lib.aaconv_bn_relu_cl_forward(_ptr(xs), dt, B, C, HW, 1, C * HW, _ptr(w), _ptr(b), _ptr(bn.running_mean),
                                                     _ptr(bn.running_var), MOM, EPS, _ptr(y), _ptr(saved), _ptr(ws), None, 0, 0, st),
                       'cl forward')
        y_nchw = y[:n].view(B, H, W, C).permute(0, 3, 1, 2)
    _margin_nan(y, n, 'y')
    _margin_nan(saved, 2 * C, 'saved')
    assert torch.equal(buf, keep), 'the feature buffer changed'
    check_elem(f'{side} abi y', y_nchw, ref.y, dtype)
    check_stats(f'{side} abi', saved[:2 * C].view(C, 2), ref)
    check_running(f'{side} abi', bn, ref)

    dy_in = dy if side == 'nchw' else dy.contiguous(memory_format=CL)
    for acc in ((0, 1) if side != 'cl' else (0,)):
        dw, db = _nan(C, torch.float32), _nan(C, torch.float32)
        if acc:
            gbuf = feature_buffer(grad_out(B, C, H, W, dtype, 7), seed=98)
            g0 = gbuf.clone()
            dx, dbs = gbuf, gbuf.stride(0)
        else:
            dx, dbs = _nan(n, dtype), C * HW
        if side == 'nchw':
            wsb = torch.empty(lib.aaconv_bn_relu_workspace_bytes(B, C), device='cuda', dtype=torch.uint8)
            if acc:
                _lib.check(lib.aaconv_bn_relu_backward_acc(_ptr(xs), dt, B, C, HW, xs.stride(0), _ptr(dy_in), _ptr(saved), _ptr(w),
                                                           _ptr(b), _ptr(dx), dbs, _ptr(dw), _ptr(db), _ptr(wsb), st), 'backward acc')
            else:
                _lib.check(lib.aaconv_bn_relu_backward(_ptr(xs), dt, B, C, HW, xs.stride(0), _ptr(dy_in), _ptr(saved), _ptr(w), _ptr(b),
                                                       _ptr(dx), _ptr(dw), _ptr(db), _ptr(wsb), st), 'backward')
        else:
            x_is_cl = int(side == 'cl')
            _lib.check(lib.aaconv_bn_relu_cl_backward(_ptr(xs), dt, B, C, HW, x_is_cl, C * HW if x_is_cl else xs.stride(0), _ptr(dy_in),
                                                      _ptr(saved), _ptr(w), _ptr(b), _ptr(dx), dbs, acc, _ptr(dw), _ptr(db), _ptr(ws),
                                                      st), 'cl backward')
        assert torch.equal(buf, keep), 'the feature buffer changed'
        _margin_nan(dw, C, 'dweight')
        _margin_nan(db, C, 'dbias')
        check_wb(f'{side} abi acc={acc}', dw[:C], db[:C], ref, tie)
        if acc:
            assert torch.equal(gbuf[:, C:], g0[:, C:]), 'gradient channels behind the input changed'
            check_elem(f'{side} abi dx (accumulated)', gbuf[:, :C], ref.dx + g0[:, :C].double(), dtype, skip=tie,
                       allow=dx_allowance(ref, tie))
        else:
            _margin_nan(dx, n, 'dx')
            got = dx[:n].view(B, H, W, C).permute(0, 3, 1, 2) if side == 'cl' else dx[:n].view(B, C, H, W)
            check_elem(f'{side} abi dx', got, ref.dx, dtype, skip=tie, allow=dx_allowance(ref, tie))


# ------------------------------------------------------------------------------------------------ GPU: NHWC channel limit
@pytest.mark.gpu
def test_bn_relu_cl_at_4096_channels_matches_float64():
    B, C, H, W = 2, 4096, 4, 4
    x, dy = features(B, C, H, W, torch.float32, 1), grad_out(B, C, H, W, torch.float32, 2)
    check_path('cl 4096 channels', 'cl', x, dy, make_bn(C, 3))


@pytest.mark.gpu
@pytest.mark.parametrize('C', [4100, 8192])
def test_bn_relu_cl_rejects_more_than_4096_channels(C):
    """cl_stats keeps a thread's segment means in registers for at most 4 x 4 x 256 channels; beyond that the channels-last
    kernels refuse an NHWC input, and cl_ok sends such a tensor to the NCHW kernels."""
    x = features(2, C, 4, 4, torch.float32, 1).contiguous(memory_format=CL).requires_grad_(True)
    bn = make_bn(C, 3)
    assert not fused_bn.cl_ok(bn, x)
    assert fused_bn.cl_ok(bn, x.detach().contiguous())                  # the NCHW-input kernels have no channel limit
    assert fused_bn.cl_ok(make_bn(4096, 3), x.detach()[:, :4096].contiguous(memory_format=CL))
    with pytest.raises(RuntimeError, match='at most 4096 channels'):
        fused_bn.bn_relu_cl(bn, x)


@pytest.mark.gpu
@pytest.mark.parametrize('which', ['module', 'running_stats', 'weight_bias'])
def test_route_predicates_refuse_a_batchnorm_that_is_not_fp32(which):
    """The kernels read weight and bias and read or update the running statistics through float pointers, so every route predicate
    refuses a BatchNorm2d with bf16 parameters or running statistics (e.g. after model.to(torch.bfloat16)): such a module takes the
    module path.  Only the predicates run here; no kernel is launched."""
    B, C, H, W = 4, 64, 8, 8
    x = torch.empty(B, C, H, W, device='cuda', dtype=torch.bfloat16)
    xl = torch.empty(B, C, H, W, device='cuda', dtype=torch.bfloat16, memory_format=CL)

    def routes(bn):
        bn.train()
        ok = [fused_bn._fused_ok(bn, x), fused_bn.cl_ok(bn, x), fused_bn.cl_ok(bn, xl), fused_bn.pool_ok(bn, x)]
        bn.eval()
        with torch.no_grad():
            ok += [fused_bn.eval_ok(bn, x), fused_bn.eval_cl_ok(bn, x), fused_bn.eval_cl_ok(bn, xl), fused_bn.pool_ok(bn, x)]
        return ok
    assert all(routes(torch.nn.BatchNorm2d(C).cuda()))                  # fp32: every route takes it
    bn = torch.nn.BatchNorm2d(C)
    if which == 'module':
        bn.to(torch.bfloat16)
    elif which == 'running_stats':
        bn.running_mean, bn.running_var = bn.running_mean.bfloat16(), bn.running_var.bfloat16()
    else:
        bn.weight.data, bn.bias.data = bn.weight.data.bfloat16(), bn.bias.data.bfloat16()
    assert not any(routes(bn.cuda())), routes(bn)


@pytest.fixture
def no_tf32():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _kernel_grad_mask(y):
    """The ReLU mask the backward kernels of a BatchNorm + ReLU op apply: fmaf(w, x^, b) > 0 with x^ = (x - mean) * rstd in fp32
    from the saved statistics.  (w x^ is exact in float64, so the sign of w x^ + b there is the sign of the fma.)"""
    xs, saved, w, b = y.grad_fn.saved_tensors
    xh = (xs.float() - saved[:, 0][None, :, None, None]) * saved[:, 1][None, :, None, None]
    return w.double()[None, :, None, None] * xh.double() + b.double()[None, :, None, None] > 0


def _recording(monkeypatch, name, calls, masks):
    """Wrap densenet.<name> (a BatchNorm + ReLU op) to count its calls and keep the ReLU mask of its backward."""
    fn = getattr(densenet, name)

    def wrapped(*a, **k):
        calls[name] = calls.get(name, 0) + 1
        out = fn(*a, **k)
        masks.append(_kernel_grad_mask(out[1] if isinstance(out, tuple) else out))
        return out
    monkeypatch.setattr(densenet, name, wrapped)


class _ReLUWithTies(torch.nn.Module):
    """ReLU for the float64 reference whose mask follows the block under test where |pre-activation| < TIE: there the fp32 and
    float64 masks may legitimately differ (as may the kernel's forward and backward masks, from two fp32 formulas), and one
    element on the other side moves a whole pixel of the input gradient."""

    def __init__(self, mask32):
        super().__init__()
        self.mask32 = mask32

    def forward(self, pre):
        tie = pre.abs() < TIE
        assert int(tie.sum()) < TIE_FRAC * tie.numel()
        return pre * torch.where(tie, self.mask32, pre > 0)


def _block_against_torchvision(block_args, x, inner_cl, monkeypatch, watch, tol=1e-4):
    from torchvision.models.densenet import _DenseBlock
    torch.manual_seed(0)
    a = _DenseBlock(*block_args).cuda().double().train()
    for m in a.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.load_state_dict(make_bn(m.num_features, m.num_features).double().state_dict())
    b = densenet.BufferedDenseBlock(*block_args).cuda().train()
    b.load_state_dict(a.state_dict())
    b.inner_channels_last = inner_cl
    calls, masks = {}, []
    for name in watch:
        _recording(monkeypatch, name, calls, masks)
    xb = x.clone().requires_grad_(True)
    yb = b(xb)
    assert len(masks) == 2 * len(a)                            # norm1 -> relu1 and norm2 -> relu2 of every layer, in order
    for i, layer in enumerate(a.values()):
        layer.relu1, layer.relu2 = _ReLUWithTies(masks[2 * i]), _ReLUWithTies(masks[2 * i + 1])
    xa = x.double().requires_grad_(True)
    ya = a(xa)
    dy = grad_out(*ya.shape, torch.float32, 2)
    ya.backward(dy.double())
    yb.backward(dy)

    def check(what, got, want):
        err = (got.double() - want).abs()
        r = float(err.max() / want.abs().max())
        print(f'block {what}: {r:.3g} of max')
        assert r < tol, f'{what}: {r:.3g} of max at {tuple(int(v) for v in (err == err.max()).nonzero()[0])}'
    check('y', yb, ya)
    check('dx', xb.grad, xa.grad)
    for (name, p), (_, q) in zip(a.named_parameters(), b.named_parameters()):
        check(name, q.grad, p.grad)
    for (name, p), (_, q) in zip(a.named_buffers(), b.named_buffers()):
        check(name, q, p.double())
    return calls


@pytest.mark.gpu
@pytest.mark.parametrize('inner_cl', [True, False])
def test_buffered_block_matches_torchvision_in_float64(inner_cl, no_tf32, monkeypatch):
    """The first three layers of block 2 (B = 16, 40x40, 128 input channels): BufferedDenseBlock against torchvision's
    _DenseBlock in float64 on the same state_dict; outputs, input gradient, every parameter gradient, running statistics."""
    x = features(16, 128, 40, 40, torch.float32, 1)
    calls = _block_against_torchvision((3, 128, 4, 32, 0.0), x, inner_cl, monkeypatch,
                                       ('tap_bn_relu_cl', 'tap_bn_relu', 'bn_relu_cl', 'bn_relu'))
    want = {'tap_bn_relu_cl': 3, 'bn_relu_cl': 3} if inner_cl else {'tap_bn_relu': 3, 'bn_relu': 3}
    assert calls == want


@pytest.mark.gpu
def test_buffered_block_sends_wide_bottlenecks_to_the_nchw_kernels(no_tf32, monkeypatch):
    """bn_size * growth = 4100 bottleneck channels: norm2 cannot take the NHWC kernels and runs bn_relu on an NCHW copy."""
    x = features(2, 8, 4, 4, torch.float32, 1)
    calls = _block_against_torchvision((1, 8, 1025, 4, 0.0), x, True, monkeypatch, ('tap_bn_relu_cl', 'bn_relu_cl', 'bn_relu'))
    assert calls == {'tap_bn_relu_cl': 1, 'bn_relu': 1}


# ------------------------------------------------------------------------------------------------ GPU: Transition prologue
def _instance_norm_relu64(x):
    m = x.mean((2, 3), keepdim=True)
    v = ((x - m) ** 2).mean((2, 3), keepdim=True)
    return torch.relu((x - m) * (v + EPS).rsqrt()), (x - m) * (v + EPS).rsqrt()


@pytest.mark.gpu
@pytest.mark.parametrize('precision,dtype,H,W', [('fp32', torch.float32, 80, 80), ('fp32', torch.float32, 40, 40),
                                                 ('fp32', torch.float32, 20, 20), ('bf16', torch.bfloat16, 34, 34)])
def test_fused_prologue_matches_float64_instance_norm(precision, dtype, H, W, no_tf32):
    """AATransition(fused_prologue=True) against the unfused module fed relu(instance_norm(x)) computed in float64; the reference
    dx is the float64 adjoint of InstanceNorm o ReLU applied to the unfused module's input gradient.  Both sides run the same
    AAConv2d kernels, so the difference isolates in_stats / in_relu_bwd.  34 x 34 in bf16: planes of 1156 = 4 mod 8 elements
    start alternately on and off 16-byte boundaries, so in_stats mixes its vector and scalar loops."""
    from chexpert_b200.densenet import AATransition
    B, Cin, Cout = 2, 64, 32
    attn = {'k': 0.0, 'v': 0.25, 'nh': 8, 'relative': True, 'input_dims': (H, W)}
    torch.manual_seed(0)
    fused = AATransition(Cin, Cout, attn, precision=precision, fused_prologue=True).cuda()
    plain = AATransition(Cin, Cout, attn, precision=precision, fused_prologue=False).cuda()
    plain.load_state_dict(fused.state_dict())
    g = _gen(4)
    x = (_unif((B, Cin, 1, 1), -3, 3, g) + _unif((B, Cin, 1, 1), 0.5, 2, g)
         * torch.randn(B, Cin, H, W, generator=g, device='cuda', dtype=torch.float64)).to(dtype)
    x64 = x.double().requires_grad_(True)
    u64, xh64 = _instance_norm_relu64(x64)
    u = u64.detach().to(dtype).requires_grad_(True)
    y_ref = plain.conv(u)
    dy = grad_out(*y_ref.shape, dtype, 5)
    y_ref.backward(dy)
    u64.backward(u.grad.double())
    xf = x.clone().requires_grad_(True)
    y = fused(xf)
    y.backward(dy)
    tie = xh64.detach().abs() < TIE
    assert int(tie.sum()) < TIE_FRAC * tie.numel()
    rstd = ((x64.detach() - x64.detach().mean((2, 3), keepdim=True)) ** 2).mean((2, 3), keepdim=True).add(EPS).rsqrt()
    allow = tie_allowance(rstd, H * W, u.grad.double(), xh64.detach(), tie, (2, 3))
    # fp32: 1e-5 of max, both sides run the same kernels.  bf16: the packed operand is bf16(relu(x^)) on both sides, from an fp32 x^
    # on one and a float64 x^ on the other; a rare rounding flip of one operand (2^-8 of it) moves an output by ~1e-4 of max, and the
    # outputs are bf16 themselves: 2^-8 |ref| + 1e-3 max.
    for what, got, want, skip in (('y', y, y_ref, None), ('dx', xf.grad, x64.grad, tie)):
        got, want = got.detach().double(), want.detach().double()
        err = (got - want).abs()
        bound = 1e-5 * want.abs().max() if precision == 'fp32' else 2.0 ** -8 * want.abs() + 1e-3 * want.abs().max()
        if skip is not None:
            err, bound = err.masked_fill(skip, 0.0), bound + allow
        print(f'prologue {precision} {H}x{W} {what}: worst {float((err / bound).max()):.3g} of its bound')
        assert bool((err <= bound).all()), what
