"""Every dispatch route of the bf16 AAConv2d path against the float64 oracle, with the kernels each case ran asserted.

The bf16 path is a chain of shape-dependent choices (operand builder, attention kernel family and template, out_proj
adjoint, tcgen05 or FFMA GEMMs, wgrad, "direct" dq, dgrad residue classes, boundary conversions).  Each case below is a
geometry picked to land on one combination; the library's per-launch profile (_lib.profile_begin / profile_end) records
which kernels really ran, so a case that drifts onto another route fails here instead of silently testing something else.
The same cases also run in fp32 mode against the same reference.

Template instances share a kernel name in the profile; the comment on each case gives the instance its geometry selects
(computed from the host predicates: attn_cc.cu cc_attn_fwd / launch_bwd_cc, aug_ops.cu rel_bwd, gemm_tc.cu tc_wgrad_supported).
"""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import aaconv_oracle as O
from tests.helpers import _bf16_grad_close, _bf16_output_close, _fp32_close, autocast_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'chexpert_b200', 'csrc')

# one entry per decision of the bf16 path: option -> kernels that run only on that option
DECISIONS = {
    'builder': {'tc': ('aug_build_tc',), 'mma': ('aug_build_fwd',)},
    'attention': {'cc': ('attn_fwd_cc', 'attn_bwd_dkv_cc', 'attn_bwd_dq_cc'),
                  'tc': ('attn_fwd_tc', 'attn_bwd_dkv_tc', 'attn_bwd_dq_tc')},
    'out_bwd': {'patch': ('out_bwd_patch', 'out_w_reduce'),
                'data': ('out_bwd_data_patch', 'out_bwd_weight_f32', 'splitk_reduce')},
    'gemm': {'tc': ('pack_wf', 'conv_qkv_fprop_tc', 'pack_nhwc_bf16', 'pack_wd', 'conv_qkv_dgrad_tc'),
             'ffma': ('conv_fwd_f32', 'qkv_fwd_f32', 'conv_bwd_data_f32', 'qkv_bwd_data_f32')},
    'wgrad': {'tc': ('conv_qkv_wgrad_tc', 'wgrad_reduce'),
              'ffma': ('conv_bwd_weight_f32', 'qkv_bwd_weight_f32', 'splitk_reduce')},
    'dq': {'direct_tc': ('rel_bwd_tc', 'rel_bwd_reduce'), 'direct': ('rel_bwd', 'rel_bwd_reduce'),
           'split': ('aug_rel_weight_grad', 'splitk_reduce', 'aug_bwd_dq')},
}


class Case:
    """One geometry and the option it takes at each decision.  fp32_rejects: text of the error the fp32 path raises instead
    (its attention backward tile outgrows a block's shared memory on rows of 128 pixels and more); fp32 mode then checks
    that the call is rejected with that message."""

    def __init__(self, cid, B, cin, hin, win, cout, k, s, dk, dv, nh, routes, extra=(), seed=0, fp32_rejects=None):
        self.id, self.B, self.hin, self.win, self.fp32_rejects = cid, B, hin, win, fp32_rejects
        H, W = (hin - 1) // s + 1, (win - 1) // s + 1
        self.shape = O.AAConvShape(cin, cout, k, s, dk, dv, nh, True, (H, W))
        self.L = H * W
        self.routes, self.seed = routes, seed
        must, must_not = set(extra), set()
        for dec, opt in routes.items():
            for o, names in DECISIONS[dec].items():
                (must if o == opt else must_not).update(names)
        if routes['gemm'] == 'tc' and routes['dq'] == 'split':
            must.add('pack_dqkv')             # the non-direct dq / dk / dv are packed for the GEMMs by a separate pass
        self.must, self.must_not = must, must_not - must


R = dict
CASES = {c.id: c for c in [
    # 512-px Transition 2: 32x32 is no builder size; dv/nh 3 -> tc attention (KATOMS 2), out_bwd_data_patch;
    # rel_bwd<5, 3> pipelined on the direct path
    Case('T2_512', 2, 512, 64, 64, 256, 3, 2, 160, 24, 8,
         R(builder='mma', attention='tc', out_bwd='data', gemm='tc', wgrad='tc', dq='direct')),
    # 512-px Transition 3: rel_bwd<2, 3>, tc attention with dv/nh 6
    Case('T3_512', 2, 1024, 32, 32, 512, 3, 2, 160, 48, 8,
         R(builder='mma', attention='tc', out_bwd='data', gemm='tc', wgrad='tc', dq='direct')),
    # attn_*_cc<2, 2>, out_bwd_patch<8, 2>, tcgen05 builder and rel_bwd_tc with dv/nh 2
    Case('dvh2_cc_k2', 1, 256, 80, 80, 128, 3, 2, 160, 16, 8,
         R(builder='tc', attention='cc', out_bwd='patch', gemm='tc', wgrad='tc', dq='direct_tc')),
    # out_bwd_patch<8, 2> next to the mma.sync builder and rel_bwd<1, 3>; attn_*_cc<1, 2> at nh = 8
    Case('dvh2_nh8_small', 2, 32, 12, 12, 40, 3, 2, 160, 16, 8,
         R(builder='mma', attention='cc', out_bwd='patch', gemm='tc', wgrad='tc', dq='direct')),
    # attn_*_cc<3, 1> with KD = 156 > 152 -> the OUTW_MAX dQa staging; out_bwd_patch<8, 1>; tcgen05 GEMMs at W = 128;
    # 2W - 1 = 255 rules out the direct dq; non-square relative tables
    Case('w128_outw_max', 1, 16, 16, 256, 48, 3, 2, 160, 8, 8,
         R(builder='mma', attention='cc', out_bwd='patch', gemm='tc', wgrad='tc', dq='split'), fp32_rejects='shared memory'),
    # the same map with dv/nh 2: the dK/dV kernel of attn_*_cc<3, 2> needs more shared memory than a block can have, so the
    # tc attention kernels run it (out_bwd_patch<8, 2> next to them)
    Case('dvh2_katoms3', 1, 16, 16, 256, 48, 3, 2, 160, 16, 8,
         R(builder='mma', attention='tc', out_bwd='patch', gemm='tc', wgrad='tc', dq='split'), fp32_rejects='shared memory'),
    # W = 130: FFMA conv / qkv GEMMs and wgrad; tc attention at KATOMS 3 (L % 4 = 2)
    Case('ffma_gemm', 2, 8, 6, 260, 16, 3, 2, 8, 4, 2,
         R(builder='mma', attention='tc', out_bwd='data', gemm='ffma', wgrad='ffma', dq='split'), fp32_rejects='shared memory'),
    # 288-px Transition 3: tcgen05 fprop / dgrad, FFMA wgrad (no multiple of W = 9 within 128 is a multiple of 16)
    Case('T3_288', 2, 1024, 18, 18, 512, 3, 2, 160, 48, 8,
         R(builder='mma', attention='tc', out_bwd='data', gemm='tc', wgrad='ffma', dq='split')),
    # dv/nh 1 on the tc attention kernels (L = 90), out_bwd_patch<8, 1>, direct rel_bwd<2, 3>
    Case('dvh1_tc', 2, 64, 18, 20, 64, 3, 2, 160, 8, 8,
         R(builder='mma', attention='tc', out_bwd='patch', gemm='tc', wgrad='tc', dq='direct')),
    # dk/nh 27: rel_bwd<2, 4> not pipelined (L * dk/nh = 1350 is not a multiple of 4); tc attention with out_bwd_patch<8, 2>
    Case('dkh27', 3, 32, 10, 20, 48, 3, 2, 216, 16, 8,
         R(builder='mma', attention='tc', out_bwd='patch', gemm='tc', wgrad='tc', dq='direct')),
    # dk/nh 32 (the limit): rel_bwd<3, 4> pipelined, attn_*_cc<2, 2>
    Case('dkh32_cc', 2, 64, 48, 48, 64, 3, 2, 256, 16, 8,
         R(builder='mma', attention='cc', out_bwd='patch', gemm='tc', wgrad='tc', dq='direct')),
    # 1x1 conv, stride 2: only input-pixel class (0, 0) has taps; the other three are unpaired classes written by zero_class
    Case('k1_s2', 2, 16, 13, 12, 32, 1, 2, 16, 8, 4,
         R(builder='mma', attention='tc', out_bwd='data', gemm='tc', wgrad='tc', dq='direct'), extra=('zero_class',)),
]}

# kernels the bf16 path can launch that no case above is expected to run
EXCLUDED = {
    'out_fwd_f32': 'fp32 path only (the bf16 path applies out_proj in out_proj_fwd)',
    'out_bwd_data_f32': 'fp32 path only (the bf16 path fuses it into out_bwd_patch / out_bwd_data_patch)',
    'rel_weight_grad_f32': 'fp32 path only (the bf16 path uses rel_bwd / aug_rel_weight_grad)',
}
# kernels every bf16 case runs; boundary variants add their own below
ALWAYS = ('out_proj_fwd',)
BOUNDARY = ('in_stats', 'pack_nhwc_bf16_in_relu', 'in_relu_apply', 'in_relu_bwd', 'dx_convert')


def _boundary_kernels(case, x_bf16, fused):
    """Kernels of the typed boundary / fused InstanceNorm + ReLU prologue (bf16_path.cu) for one variant."""
    gemm, wgrad = case.routes['gemm'] == 'tc', case.routes['wgrad'] == 'tc'
    ks = set()
    if fused:
        ks |= {'in_stats', 'in_relu_bwd'}
        if gemm:
            ks.add('pack_nhwc_bf16_in_relu')
    if (fused or x_bf16) and not (gemm and wgrad):
        ks.add('in_relu_apply')              # an FFMA stage reads x itself: fp32 copy of the (normalised) input
    if x_bf16 and not fused and not gemm:
        ks.add('dx_convert')                 # the FFMA dgrad writes fp32; tcgen05 dgrad writes a bf16 dx directly
    return ks


# ------------------------------------------------------------------------------------------------
# inputs, float64 reference (cached per case and variant), autocast calibration
# ------------------------------------------------------------------------------------------------
IN_EPS = 1e-5
_REF = {}


def _inputs(case):
    s = case.shape
    g = torch.Generator().manual_seed(100 + case.seed)
    x = torch.relu(torch.randn(case.B, s.in_channels, case.hin, case.win, generator=g))
    dy = torch.randn(case.B, s.out_channels, *s.input_dims, generator=g)
    return O.init_params(s, seed=case.seed), x, dy


def _prologue(x):
    return torch.relu(F.instance_norm(x, eps=IN_EPS))


def _autograd_ref(s, p, x, dy, fused, dtype, want_w):
    """forward_sequential (with the fused prologue in front) differentiated by autograd -> y, grads, weights"""
    xx = x.to(dtype).requires_grad_(True)
    pp = {k: v.to(dtype).requires_grad_(True) for k, v in p.items()}
    y, w = O.aaconv_forward_sequential(_prologue(xx) if fused else xx, pp, s, return_weights=True)
    y.backward(dy.to(dtype))
    g = {k: v.grad for k, v in pp.items()}
    g['x'] = xx.grad
    return y.detach(), g, (w.detach() if want_w else None)


def reference(case, x_bf16=False, fused=False):
    """-> (params, x, dy, y_ref, g_ref, w_ref or None, autocast dict); float64 on the GPU, returned on the CPU."""
    key = (case.id, x_bf16, fused)
    if key in _REF:
        return _REF[key]
    s = case.shape
    p, x, dy = _inputs(case)
    if x_bf16:                            # the kernels see the rounded input (and y, hence dy, is bf16 there too):
        x, dy = x.bfloat16().float(), dy.bfloat16().float()      # rounding those is not kernel error
    want_w = case.L <= 1600
    dev = torch.device('cuda')
    pd = {k: v.to(dev, torch.float64) for k, v in p.items()}
    if fused:
        y_ref, g_ref, w_ref = _autograd_ref(s, pd, x.to(dev), dy.to(dev), True, torch.float64, want_w)
        prm = {k: v.float().to(dev).requires_grad_(True) for k, v in p.items()}
        xc = x.to(dev).requires_grad_(True)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            ya = O.aaconv_forward_sequential(_prologue(xc), prm, s)
        ya.float().backward(dy.to(dev))
        ac = {'y': ya.float().detach(), 'x': xc.grad}
        ac.update({k: v.grad for k, v in prm.items()})
    else:
        y_ref, g_ref = O.aaconv_backward_closed(x.to(dev, torch.float64), pd, s, dy.to(dev, torch.float64))
        w_ref = O.aaconv_forward_closed(x.to(dev, torch.float64), pd, s, return_weights=True)[1] if want_w else None
        ac = autocast_reference(s, p, x, dy)
    cpu = lambda t: None if t is None else t.detach().cpu()      # noqa: E731
    out = (p, x, dy, cpu(y_ref), {k: cpu(v) for k, v in g_ref.items()}, cpu(w_ref), {k: cpu(v) for k, v in ac.items()})
    del y_ref, g_ref, w_ref
    _REF[key] = out
    return out


def _module(case, p, precision):
    import chexpert_b200 as cb
    s = case.shape
    m = cb.AAConv2d(s.in_channels, s.out_channels, s.kernel_size, s.stride, s.dk, s.dv, s.nh, s.relative, s.input_dims,
                    precision=precision)
    m.load_state_dict({k: v.float() for k, v in p.items()}, strict=True)
    return m.cuda()


def _run(case, precision, x_bf16=False, fused=False, profile=True):
    """forward + backward of the CUDA module -> (y, weights, dx, {param: grad}, kernel names in launch order)"""
    from chexpert_b200 import _lib
    p, x, dy, *_ = reference(case, x_bf16, fused)
    m = _module(case, p, precision)
    xc = x.cuda().to(torch.bfloat16 if x_bf16 else torch.float32).requires_grad_(True)
    torch.cuda.synchronize()
    if profile:
        _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    try:
        y, w = m(xc, return_attn=case.L <= 1600, fused_in=IN_EPS if fused else None)
        y.backward(dy.cuda().to(y.dtype))
    finally:
        ran = [n for n, _ in _lib.profile_end()] if profile else []
    torch.cuda.synchronize()
    return y.detach(), w, xc.grad, {n: q.grad for n, q in m.named_parameters()}, ran


def _check_route(case, ran, precision, x_bf16=False, fused=False):
    ran_set = set(ran)
    if precision == 'fp32':
        bf16_only = set().union(*(n for dec in DECISIONS.values() for o, n in dec.items())) - set(DECISIONS['gemm']['ffma']) \
            - set(DECISIONS['wgrad']['ffma']) - {'splitk_reduce', 'out_bwd_weight_f32'}
        assert 'attn_fwd_f32' in ran_set and not (ran_set & bf16_only), f'{case.id} fp32: ran {sorted(ran_set)}'
        return
    bnd = _boundary_kernels(case, x_bf16, fused)
    must = set(case.must) | set(ALWAYS) | bnd
    must_not = (set(case.must_not) | set(BOUNDARY)) - must
    if case.L <= 1600:
        must.add('aug_weights_bf16')
    missing, extra = sorted(must - ran_set), sorted(must_not & ran_set)
    assert not missing and not extra, (f'{case.id} (x_bf16={x_bf16}, fused={fused}) is on another route: '
                                       f'missing {missing}, unexpected {extra}; ran {sorted(ran_set)}')


def _check_values(case, precision, y, w, dx, grads, x_bf16=False, fused=False, only=None):
    p, x, dy, y_ref, g_ref, w_ref, ac = reference(case, x_bf16, fused)
    names = list(g_ref) if only is None else only
    if precision == 'fp32':
        _fp32_close(y, y_ref, 'y')
        if w is not None:
            _fp32_close(w, w_ref, 'weights')
        for n in names:
            _fp32_close(dx if n == 'x' else grads[n], g_ref[n], n)
        return
    _bf16_output_close(y, y_ref, 'y', ac['y'])
    if w is not None:
        _bf16_output_close(w, w_ref, 'weights')
    for n in names:
        _bf16_grad_close(dx if n == 'x' else grads[n], g_ref[n], ac[n], n)


# ------------------------------------------------------------------------------------------------
# 1. one case per route, bf16 and fp32, against float64; the profile names the route
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
@pytest.mark.parametrize('cid', list(CASES))
@pytest.mark.gpu
def test_route_matches_oracle(cid, precision):
    case = CASES[cid]
    if precision == 'fp32' and case.fp32_rejects:
        with pytest.raises(RuntimeError, match=case.fp32_rejects):
            _run(case, precision, profile=False)
        return
    y, w, dx, grads, ran = _run(case, precision)
    _check_route(case, ran, precision)
    _check_values(case, precision, y, w, dx, grads)


# boundary variants: fp32 / bf16 x, with and without the fused InstanceNorm + ReLU prologue, on an FFMA-GEMM geometry and on
# one with tcgen05 GEMMs but an FFMA wgrad (the two consumers of the fp32 copy of x).  In fp32 mode a bf16 x is converted in
# Python before the kernels and y / dx come back rounded to bf16, which no 1e-4 gate can hold: that mode runs fp32 x only.
BOUNDARY_VARIANTS = [(cid, prec, xb, fu) for cid in ('ffma_gemm', 'T3_288') for xb in (False, True) for fu in (False, True)
                     for prec in ('bf16', 'fp32') if not (prec == 'fp32' and (xb or CASES[cid].fp32_rejects)) and (xb or fu)]


@pytest.mark.parametrize('cid,precision,x_bf16,fused', BOUNDARY_VARIANTS)
@pytest.mark.gpu
def test_boundary_variant_matches_oracle(cid, precision, x_bf16, fused):
    case = CASES[cid]
    y, w, dx, grads, ran = _run(case, precision, x_bf16, fused)
    assert y.dtype == dx.dtype == (torch.bfloat16 if x_bf16 else torch.float32)
    _check_route(case, ran, precision, x_bf16, fused)
    _check_values(case, precision, y, w, dx, grads, x_bf16, fused)


# ------------------------------------------------------------------------------------------------
# 2. contracts: backward twice on one saved block, partial gradients, batch independence
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cid', ['T2_512', 'dvh2_cc_k2', 'w128_outw_max'])
@pytest.mark.gpu
def test_backward_twice_is_bit_identical(cid):
    """The saved block is patched in place by backward (the backward-only columns of Qa) and the direct path clears its
    packed dq/dk/dv operand first: a retained graph must give the same gradients on the second call, bit for bit."""
    case = CASES[cid]
    p, x, dy, *_ = reference(case)
    m = _module(case, p, 'bf16')
    xc = x.cuda().requires_grad_(True)
    y = m(xc)
    res = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        xc.grad = None
        y.backward(dy.cuda(), retain_graph=True)
        torch.cuda.synchronize()
        res.append([xc.grad.clone()] + [q.grad.clone() for q in m.parameters()])
    for (n, _), a, b in zip([('x', None)] + list(m.named_parameters()), *res):
        assert torch.equal(a, b), f'{cid}: second backward changed {n}'


PARTIAL = {'x_frozen': ('conv.weight', 'in_proj_qkv.weight', 'out_proj.weight', 'key_rel_h', 'key_rel_w'),
           'key_rel_w_only': ('key_rel_w',), 'qkv_only': ('in_proj_qkv.weight',)}


@pytest.mark.parametrize('which', list(PARTIAL))
@pytest.mark.parametrize('cid', ['dvh2_cc_k2', 'w128_outw_max'])
@pytest.mark.gpu
def test_partial_gradients_bf16(cid, which):
    """Gradients that are not requested are not written (NULL members of aaconv_param_grads) and come back None; the
    requested ones still meet the gate."""
    case = CASES[cid]
    p, x, dy, *_ = reference(case)
    m = _module(case, p, 'bf16')
    want = PARTIAL[which]
    for n, q in m.named_parameters():
        q.requires_grad_(n in want)
    y = m(x.cuda())
    y.backward(dy.cuda())
    y = y.detach()
    grads = {n: q.grad for n, q in m.named_parameters()}
    for n, g in grads.items():
        assert (g is None) == (n not in want), f'{cid}: {n} requested={n in want} but grad is {"None" if g is None else "set"}'
    _check_values(case, 'bf16', y, None, None, grads, only=list(want))


@pytest.mark.parametrize('cid', ['T2_512', 'dvh2_cc_k2'])
@pytest.mark.gpu
def test_batch_independence_bf16(cid):
    """Sample b of a batched call equals the same sample run alone, bit for bit (y and dx)."""
    case = CASES[cid]
    s = case.shape
    p = O.init_params(s, seed=case.seed)
    m = _module(case, p, 'bf16')
    g = torch.Generator().manual_seed(7)
    x = torch.relu(torch.randn(3, s.in_channels, case.hin, case.win, generator=g)).cuda()
    dy = torch.randn(3, s.out_channels, *s.input_dims, generator=g).cuda()
    xa = x.clone().requires_grad_(True)
    ya = m(xa)
    ya.backward(dy)
    xb = x[1:2].clone().requires_grad_(True)
    yb = m(xb)
    yb.backward(dy[1:2])
    assert torch.equal(ya[1:2], yb)
    assert torch.equal(xa.grad[1:2], xb.grad)


# ------------------------------------------------------------------------------------------------
# 3. the route table covers every kernel the bf16 path can launch (no GPU needed)
# ------------------------------------------------------------------------------------------------
ROUTE_SOURCES = ('attn_cc.cu', 'attn_tc.cu', 'attn_tc_bwd.cu', 'aug_ops.cu', 'aug_tc.cu', 'gemm_tc.cu', 'prologue.cu',
                 'fp32_gemms.cu')


def launched_kernel_names():
    names = set()
    for f in ROUTE_SOURCES:
        src = open(os.path.join(CSRC, f)).read()
        for call in re.findall(r'(?:AACONV_LAUNCH_OK|launch_simt_gemm|\.flush)\(([^;]*?)\)\s*;', src, re.S):
            names.update(re.findall(r'"(\w+)"', call))
    return names


def test_route_table_covers_every_bf16_kernel():
    names = launched_kernel_names()
    assert {'attn_fwd_cc', 'conv_qkv_fprop_tc', 'conv_qkv_dgrad_tc', 'conv_fwd_f32', 'dx_convert', 'in_relu_bwd'} <= names
    expected = set(ALWAYS) | set(BOUNDARY) | {'aug_weights_bf16'}
    for c in CASES.values():
        expected |= c.must
    uncovered = sorted(names - expected - set(EXCLUDED))
    assert not uncovered, f'kernels with no route case and no EXCLUDED entry: {uncovered}'
    assert not (set(EXCLUDED) & expected), f'excluded yet expected by a case: {sorted(set(EXCLUDED) & expected)}'
    stale = sorted(set(EXCLUDED) - names)
    assert not stale, f'EXCLUDED names no longer launched: {stale}'
    for dec in DECISIONS.values():                  # every option of every decision is taken by some case
        for names_ in dec.values():
            assert set(names_) <= expected
