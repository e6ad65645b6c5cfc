"""aadensenet121's training step as bench.py times it -- TrainStep('cuda', size=320, buffered=True, fused_prologue=True): bf16
weight shadows, the batched num_batches_tracked bump, the fused dense-block and Transition kernels, the BCE kernel, SGD, and the
CUDA graph with its re-capture on an lr change -- against the float64 reference model of oracle/model_oracle.py (torch ops only,
no chexpert_b200 code) run on the GPU from the same state_dict and batch, with the reference's loss (U-Ones targets,
BCE-with-logits summed over classes, averaged over the batch) and optimizer.

Gates: rel = max |ours - reference| / max |reference| per tensor (tests/test_densenet121.gate_vs_control), or the relative L2
over all gradients together, at most CTL_FACTOR (bf16 L2: BF16_L2_VS_CONTROL) times the error of a control -- the same reference
model run by PyTorch in the step's own precision (fp32 with TF32 off, or fp32 parameters under torch.autocast(bf16)) -- or a floor
where that is larger: fp32 GRAD_TOL / OUT_TOL of tests/test_densenet121.py, bf16 BF16_REL_TO_MAX / BF16_REL_L2 of tests/helpers.py.

Measured on a B200 (1000 W), B = 16 at 320 px.  On this i.i.d.-noise batch the single-step gradients are ill-conditioned in any
precision: the fp32 control is up to 2.4e-2 of max off float64 (transition3.conv.conv.weight) and 8.1e-3 in L2; the bf16 control
up to 0.93 of max (denseblock3.denselayer5.norm2.weight) and 0.73 in L2.  The step sits at the controls' level: fp32 L2 9.1e-3,
bf16 L2 0.731; bf16 per tensor at most 0.59 of its gate; running statistics at most 0.07 (fp32) and 0.46 (bf16) of theirs.  The
fp32 gradients are gated in L2 only: their per-tensor ratio to the fp32 control has a median of 1.0-1.2 in every block, but the
ratio of two error draws of that size has a tail -- 12 of 370 tensors (8 of them in denseblock4, whose 10 x 10 maps hold 1600
elements per channel) are over 3x, the worst 8.9x (denseblock4.denselayer11.conv2.weight, 3.2e-2 against 3.6e-3).  No float64
gate can see two bf16 shadow gradients swapped (0.86 in L2 against the control's 0.73): shadow_mismatches checks the shadows
exactly instead.
"""
import pytest
import torch
import torch.nn as nn

from chexpert_b200 import _lib
from chexpert_b200.densenet import AATransition, BufferedDenseBlock
from chexpert_b200.train import TrainStep, synthetic_batch
from oracle import aaconv_oracle as O
from oracle.model_oracle import ref_aadensenet121
from tests.helpers import BF16_REL_L2, BF16_REL_TO_MAX, BF16_RTOL
from tests.test_densenet121 import CTL_FACTOR, GRAD_TOL, OUT_TOL, no_tf32, rel  # noqa: F401  (no_tf32 is a fixture)

pytestmark = pytest.mark.gpu

SIZE = 320
DTYPE = {'f64': torch.float64, 'fp32': torch.float32, 'autocast': torch.float32}
STATS = ('running_mean', 'running_var')
# bf16, gradients or parameter updates of all tensors together in relative L2: at most this times the autocast control's error.
# Summed over 12.5 M elements that ratio is stable where the per-tensor one is not: measured on a B200 (1000 W) 0.997 for one
# step (0.731 against 0.733) and 0.998 over six steps (0.563 against 0.564).  At CTL_FACTOR it would let all-zero gradients or
# updates (1.0) pass against controls that far off float64; at 1.25 it does not.
BF16_L2_VS_CONTROL = 1.25


@pytest.fixture
def deterministic(monkeypatch):
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)      # no run-to-run differences from cuDNN's atomics


def reference_model(sd, mode):
    """The reference aadensenet121 on the GPU from state_dict `sd`: 'f64' the float64 reference, 'fp32' the fp32 control, 'autocast'
    the bf16 control (fp32 parameters, run under torch.autocast(bf16) by reference_loss)."""
    m = ref_aadensenet121((SIZE, SIZE))
    m.load_state_dict(sd, strict=True)
    return m.to('cuda', DTYPE[mode]).train()


def reference_loss(m, mode, x, raw):
    dt = DTYPE[mode]
    with torch.autocast('cuda', dtype=torch.bfloat16, enabled=mode == 'autocast'):
        z = m(x.to(dt))
    return O.bce_with_logits(z.to(dt), O.uones_targets(raw.cpu()).to('cuda', dt)).sum(1).mean(0)


def snapshot(model):
    return {n: t.detach().double().clone() for n, t in model.state_dict().items() if t.dtype.is_floating_point}


def gate(ours, ctl, ref, floor):
    """-> [(rel / its limit, name, rel, the control's rel)] for every tensor of `ref`, worst first.  Limit: max(floor,
    CTL_FACTOR * the control's rel)."""
    rows = []
    for n in ref:
        e, ec = rel(ours[n], ref[n]), rel(ctl[n], ref[n])
        rows.append((e / max(floor, CTL_FACTOR * ec), n, e, ec))
    return sorted(rows, reverse=True)


def check(what, rows):
    ratio, n, e, ec = rows[0]
    print(f'{what}: worst {n}: {e:.3g} of max, control {ec:.3g}; {ratio:.3g} of its gate')
    bad = [r for r in rows if r[0] > 1]
    assert not bad, f'{what}: {len(bad)} tensors over the gate: ' + '; '.join(f'{n} {e:.3g} (control {ec:.3g})' for _, n, e, ec in bad[:5])


def rel_l2_all(ours, ref):
    num = sum(float(((ours[n].double() - ref[n].double()) ** 2).sum()) for n in ref)
    return (num / sum(float((ref[n].double() ** 2).sum()) for n in ref)) ** 0.5


# ------------------------------------------------------------------------------------------------ one step, B = 16 at 320 px
B1, LR1 = 16, 1e-3
CONFIGS = {'bf16': dict(precision='bf16'), 'bf16_channels_last': dict(precision='bf16', channels_last=True),
           'fp32': dict(precision='fp32')}


@pytest.fixture(scope='module')
def reference_step():
    """-> step(sd, x, raw, mode): (loss, gradients, running-statistic changes) of one reference step from state_dict `sd`, computed
    once per mode for the module's tests (every config starts from TrainStep(seed=0)'s state_dict) and released after them."""
    cache = {}

    def step(sd, x, raw, mode):
        cache.setdefault('sd', {k: v.clone() for k, v in sd.items()})
        assert all(torch.equal(sd[k], cache['sd'][k]) for k in sd), 'TrainStep(seed=0) starts from another state_dict'
        if mode not in cache:
            m = reference_model(sd, mode)
            loss = reference_loss(m, mode, x, raw)
            loss.backward()
            grads = {n: p.grad.detach() for n, p in m.named_parameters()}
            stats = {n: b.detach().double() - sd[n].double() for n, b in m.named_buffers() if n.endswith(STATS)}
            cache[mode] = (loss.detach(), grads, stats)
            del m, loss
        return cache[mode]

    yield step
    cache.clear()
    torch.cuda.empty_cache()


def one_step(config):
    """-> (TrainStep after one eager call on B1 images, its loss, the state_dict before the call, the batch, the launch names)."""
    ts = TrainStep('cuda', size=SIZE, lr=LR1, seed=0, buffered=True, fused_prologue=True, **CONFIGS[config])
    x, raw = synthetic_batch(B1, size=SIZE, seed=5, device='cuda')
    sd = {k: v.detach().clone() for k, v in ts.model.state_dict().items()}
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    loss = ts(x, raw)
    torch.cuda.synchronize()
    return ts, loss, sd, x, raw, [n for n, _ in _lib.profile_end()]


def sgd_gradients(ts):
    """The gradient SGD read: a first nesterov step stores it as the momentum buffer (and adds 0.9 x it to .grad in place)."""
    return {n: ts.opt.state[p]['momentum_buffer'] for n, p in ts.model.named_parameters()}


def shadow_mismatches(ts, sd, grads):
    """The bf16 weight shadows of TrainStep, checked exactly after one step: shadow i is the pre-step master weight named
    _sh_names[i] cast to bf16, that master is _sh_params[i], and the gradient SGD read for it is shadow i's gradient cast to fp32,
    bit for bit.  -> the names for which any of that fails.  In bf16 this, not a float64 gate, is what catches a mis-ordered cast,
    functional_call mapping or copy-back: the bf16 gradients of the dense-block weights are 0.7-0.8 of max off float64 in
    PyTorch's own autocast execution of the reference, so swapping two of them stays inside any gate calibrated on it."""
    bad = []
    for name, p, sh in zip(ts._sh_names, ts._sh_params, ts._sh):
        if not (ts.model.get_parameter(name) is p and torch.equal(sh.detach(), sd[name].to(torch.bfloat16))
                and torch.equal(grads[name], sh.grad.float())):
            bad.append(name)
    return bad


@pytest.mark.parametrize('config', list(CONFIGS))
def test_one_step_matches_float64(config, reference_step, no_tf32, deterministic):
    """One eager call of the benchmarked configuration: num_batches_tracked of every BatchNorm2d; from the per-launch profile, the
    kernels the layer plan implies; the SGD update against the gradient; the loss and the running statistics of every BatchNorm2d
    (their change over the step) against the float64 reference; every parameter's gradient as SGD read it, in relative L2 over all
    of them, and in bf16 per tensor as well; in bf16 the weight shadows exactly (shadow_mismatches).  Each of the two checks must
    reject the gradients of two same-shape dense-block weights swapped -- in bf16 the shadow check, in fp32 the L2 gate."""
    ts, loss, sd, x, raw, names = one_step(config)
    bf16 = ts.autocast
    bns = {n: m for n, m in ts.model.named_modules() if isinstance(m, nn.BatchNorm2d)}
    layers = [layer for m in ts.model.modules() if isinstance(m, BufferedDenseBlock) for layer in m.values()]
    transitions = [m for m in ts.model.modules() if isinstance(m, AATransition) and m.fused_prologue]

    # TrainStep counts each batch once, on every BatchNorm2d (its own foreach add; no module path may add a second)
    counts = {n: int(m.num_batches_tracked) for n, m in bns.items()}
    assert len(bns) == 2 + 2 * len(layers)                     # norm0, norm5, norm1 / norm2 of every dense layer
    assert all(c == 1 for c in counts.values()), {n: c for n, c in counts.items() if c != 1}
    # the route: every dense layer's norm1 runs the NCHW-prefix -> NHWC tile kernel and its norm2 the NHWC -> NHWC kernel
    # (csrc/bn_cl.cu), every Transition the fused InstanceNorm prologue, the loss the BCE kernel -- a silent fall-back fails here
    route = {k: names.count(k) for k in ('bn_t_apply', 'bn_cl_apply', 'in_stats', 'bce')}
    assert route == {'bn_t_apply': len(layers), 'bn_cl_apply': len(layers), 'in_stats': len(transitions), 'bce': 1}, route
    assert len(layers) == 58 and len(transitions) == 3

    grads = sgd_gradients(ts)
    a, b = 'features.denseblock1.denselayer1.conv2.weight', 'features.denseblock1.denselayer2.conv2.weight'
    assert grads[a].shape == grads[b].shape == (32, 128, 3, 3)
    swapped = dict(grads, **{a: grads[b], b: grads[a]})          # what a mis-ordered copy-back of two shadow gradients gives
    if bf16:
        assert len(ts._sh) == 2 * len(layers) + 1                   # conv0 and both convolutions of every dense layer
        assert shadow_mismatches(ts, sd, grads) == []
        assert shadow_mismatches(ts, sd, swapped) == [a, b]
        assert shadow_mismatches(ts, dict(sd, **{a: sd[b], b: sd[a]}), grads) == [a, b]     # ... of two shadow casts
    # the update: p1 = p0 - lr (g + 0.9 g), each step of which rounds once in fp32
    for n, p in ts.model.named_parameters():
        g, p0, p1 = grads[n].double(), sd[n].double(), p.detach().double()
        err = (p1 - (p0 - LR1 * 1.9 * g)).abs()
        lim = 2.0 ** -23 * p1.abs() + 2.0 ** -21 * LR1 * 1.9 * g.abs()
        assert bool((err <= lim).all()), f'SGD update of {n}: {float((err - lim).max()):.3g} over fp32 rounding'

    stats = {n: b.detach().double() - sd[n].double() for n, b in ts.model.named_buffers() if n.endswith(STATS)}
    assert len(stats) == 2 * len(bns)
    loss_r, g_r, s_r = reference_step(sd, x, raw, 'f64')
    loss_c, g_c, s_c = reference_step(sd, x, raw, 'autocast' if bf16 else 'fp32')
    assert set(grads) == set(g_r) and set(stats) == set(s_r)
    e, ec = rel(loss, loss_r), rel(loss_c, loss_r)
    print(f'{config}: loss {float(loss):.7f}, float64 {float(loss_r):.7f}, control {float(loss_c):.7f}')
    assert e <= max(BF16_RTOL if bf16 else OUT_TOL, CTL_FACTOR * ec), (e, ec)
    check(f'{config} running statistics', gate(stats, s_c, s_r, BF16_REL_TO_MAX if bf16 else OUT_TOL))
    if bf16:
        check(f'{config} gradients', gate(grads, g_c, g_r, BF16_REL_TO_MAX))
    floor, factor = (BF16_REL_L2, BF16_L2_VS_CONTROL) if bf16 else (GRAD_TOL, CTL_FACTOR)
    e, ec = rel_l2_all(grads, g_r), rel_l2_all(g_c, g_r)
    print(f'{config}: gradients {e:.3g} in relative L2 (control {ec:.3g})')
    assert e <= max(floor, factor * ec), (e, ec)
    e_swap = rel_l2_all(swapped, g_r)
    print(f'{config}: with {a} and {b} swapped, {e_swap:.3g} in relative L2; against the control: '
          f'{rel_l2_all(grads, g_c):.3g} (swapped {rel_l2_all(swapped, g_c):.3g})')
    if not bf16:
        assert e_swap > max(floor, factor * ec)


# ------------------------------------------------------------------------------------------------ six steps, graph and re-capture
B2, LR2, GRAPH_TOL = 4, 1e-3, 1e-2


def test_graph_recapture_and_six_steps_match_float64(no_tf32, deterministic):
    """bf16 TrainStep with cuda_graph=True (graph_after=2) and with cuda_graph=False, and the float64 reference with its autocast
    control trained by SGD(lr, momentum 0.9, nesterov), all four under MultiStepLR(milestones=[4], gamma=0.1), 6 calls at B = 4:
    the capture happens at call 3 and the lr drop after call 4 forces a re-capture at call 5.

    Graph against eager: the losses, and the parameters and running statistics after 6 steps (their changes, in relative L2 at
    GRAPH_TOL).  Eager against the reference: the losses and the parameter updates over the 6 steps, in L2, gated against the
    control as tests/test_densenet121.py::test_train_step_densenet121 does.  num_batches_tracked is 6 everywhere.

    A missed re-capture would replay steps 5 and 6 at the old lr: 10x the eager run's updates of those steps, p6 - p4, so the graph
    run would end 9 (p6 - p4) away from the eager one.  With the momentum buffers of 4 steps behind them, steps 5 and 6 at lr / 10
    are ~7.5 % of the whole update (nesterov step sizes 1.9, 2.71, 3.44, 4.10 before the drop, 4.69 and 5.22 after it, for a steady
    gradient), so that distance is ~0.68 of the update norm: ~70x GRAPH_TOL.  The test measures it and asserts it exceeds 10x."""
    kw = dict(size=SIZE, precision='bf16', lr=LR2, seed=0, buffered=True, fused_prologue=True)
    graph = TrainStep('cuda', cuda_graph=True, graph_after=2, **kw)
    eager = TrainStep('cuda', cuda_graph=False, **kw)
    x, raw = synthetic_batch(B2, size=SIZE, seed=6, device='cuda')
    sd = {k: v.detach().clone() for k, v in eager.model.state_dict().items()}
    assert all(torch.equal(v, sd[k]) for k, v in graph.model.state_dict().items())
    runs = {}
    for ts in (graph, eager):
        ts.sched = torch.optim.lr_scheduler.MultiStepLR(ts.opt, [4], gamma=0.1)
    for mode in ('f64', 'autocast'):
        m = reference_model(sd, mode)
        opt = torch.optim.SGD(m.parameters(), lr=LR2, momentum=0.9, nesterov=True)
        runs[mode] = (m, opt, torch.optim.lr_scheduler.MultiStepLR(opt, [4], gamma=0.1))
    p0 = snapshot(eager.model)
    losses = {k: [] for k in ('graph', 'eager', 'f64', 'autocast')}
    graphs = []
    for call in range(1, 7):
        losses['graph'].append(float(graph(x, raw)))
        graphs.append(graph._graph)
        losses['eager'].append(float(eager(x, raw)))
        if call == 4:
            p4 = snapshot(eager.model)
        for mode, (m, opt, sched) in runs.items():
            opt.zero_grad(set_to_none=True)
            loss = reference_loss(m, mode, x, raw)
            loss.backward()
            opt.step()
            sched.step()
            losses[mode].append(float(loss))
    print('losses', {k: [round(v, 6) for v in vs] for k, vs in losses.items()})

    # capture at call 3, replay at call 4, re-capture at call 5 at the dropped lr
    assert graphs[0] is None and graphs[1] is None and graphs[2] is not None and graphs[3] is graphs[2]
    assert graphs[4] is not graphs[3] and graphs[5] is graphs[4]
    assert graph._graph_lr == [pytest.approx(LR2 * 0.1, rel=1e-12)]
    for ts in (graph, eager):
        counts = {n: int(m.num_batches_tracked) for n, m in ts.model.named_modules() if isinstance(m, nn.BatchNorm2d)}
        assert all(c == 6 for c in counts.values()), {n: c for n, c in counts.items() if c != 6}

    # graph against eager: the gates of tests/test_gpu_parity.py::test_train_step_cuda_graph_matches_eager on the losses
    lg, le = torch.tensor(losses['graph']), torch.tensor(losses['eager'])
    assert torch.allclose(lg[:4], le[:4], rtol=5e-3, atol=1e-3) and torch.allclose(lg, le, rtol=3e-2, atol=1e-3), (lg, le)
    pg, p6 = snapshot(graph.model), snapshot(eager.model)
    delta = lambda a, b, keys: {k: a[k] - b[k] for k in keys}      # noqa: E731
    pn = [n for n, _ in eager.model.named_parameters()]
    sn = [n for n in p6 if n.endswith(STATS)]
    e_p = rel_l2_all(delta(pg, p0, pn), delta(p6, p0, pn))
    e_s = rel_l2_all(delta(pg, p0, sn), delta(p6, p0, sn))
    missed = 9 * rel_l2_all(delta(p4, p0, pn), delta(p6, p0, pn))       # 9 |p6 - p4| / |p6 - p0|
    print(f'graph vs eager after 6 steps: parameter updates {e_p:.3g}, running statistics {e_s:.3g} in relative L2; '
          f'a missed re-capture would be {missed:.3g}')
    assert e_p <= GRAPH_TOL and e_s <= GRAPH_TOL, (e_p, e_s)
    assert missed > 10 * GRAPH_TOL, missed

    # eager against the float64 reference, gated by the autocast control (test_train_step_densenet121's bf16 tolerance as the floor).
    # Measured on a B200 (1000 W): updates 0.563 of their L2 norm off float64, control 0.564, ours against the control 0.441;
    # graph against eager 0 and 0 (bit-identical), a missed re-capture 0.518.
    tol = 2e-2
    for a, c, r in zip(losses['eager'], losses['autocast'], losses['f64']):
        assert abs(a - r) <= max(tol * abs(r), CTL_FACTOR * abs(c - r)), losses
    pr = {n: p.detach().double() for n, p in runs['f64'][0].named_parameters()}
    pc = {n: p.detach().double() for n, p in runs['autocast'][0].named_parameters()}
    du, dr, dc = delta(p6, p0, pn), delta(pr, p0, pn), delta(pc, p0, pn)
    e, ec = rel_l2_all(du, dr), rel_l2_all(dc, dr)
    print(f'parameter updates over 6 steps: {e:.3g} of their L2 norm (autocast control {ec:.3g}); against the control '
          f'{rel_l2_all(du, dc):.3g}; zero updates would be 1')
    assert e <= max(tol, BF16_L2_VS_CONTROL * ec), (e, ec)
