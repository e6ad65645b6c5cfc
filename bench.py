#!/usr/bin/env python
"""bench.py -- AAConv2d fwd+bwd throughput on B200 (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision bf16|fp32] [--shape T1|T2|T3|T1_512] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference algorithm's CPU port on the host cores

A step = one forward + backward of the AAConv2d module at the Transition-1 shape (B=16 per GPU, 256 ch,
80x80 -> 40x40, 8 heads, dk=160, dv=8) on synthetic relu(randn) input (SURVEY.md section 8d), through the
public nn.Module / autograd.Function (which calls the C ABI).  Under torchrun (N>1) every rank runs its own
batch (weak scaling) and the parameter gradients are all-reduced over NCCL inside the step.

Prints ONE JSON line on rank 0.  `value` = algorithmic TFLOP/s (fwd+bwd = 3 x fwd, SURVEY.md 8d), inputs
resident in HBM; `e2e` = same with pinned-host x/dy copied in and y + parameter grads copied out each step.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPES = {  # name -> (Cin, Hin, Cout, dk, dv)   (SURVEY.md section 8 table)
    'T1': (256, 80, 128, 160, 8),
    'T2': (512, 40, 256, 160, 24),
    'T3': (1024, 20, 512, 160, 48),
    'T1_512': (256, 128, 128, 160, 8),
}


def flops_fwd(B, cin, hin, cout, dk, dv, nh=8, ks=3):
    H = W = hin // 2
    L = H * W
    dkh, dvh = dk // nh, dv // nh
    dense = 2 * B * L * (ks * ks * cin * (cout - dv) + cin * (2 * dk + dv) + dv * dv)
    attn = 2 * B * nh * L * (L * dkh + dkh * ((2 * W - 1) + (2 * H - 1)) + L * dvh)
    return dense + attn


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return j['bf16_tflops'], j['hbm_gbs'], 'measured'
    return 1590.0, 6650.0, 'fallback'


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap',
                     nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: 'hw_power_brake'}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report nothing rather than fail the bench
            self.reasons.add(f'nvml_unavailable:{type(e).__name__}')

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


DUMP_ELEMENTS = 15 << 20      # float32 elements written by --dump-outputs in all: 60 MiB


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each tensor of `arrays` (name -> tensor) as out_dir/<name>.npy in float32.  The smaller tensors are written
    whole, in their shape; a tensor beyond its share of DUMP_ELEMENTS is written as a flat sample at a fixed set of flat indices
    (torch.randperm seeded with 0, sorted), the same for every run with the same arguments, so two builds compare element for
    element."""
    os.makedirs(out_dir, exist_ok=True)
    left, todo = DUMP_ELEMENTS, sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(todo):
        cap = left // (len(todo) - i)
        a = t.detach().float().cpu()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + '.npy'), a.numpy())
        left -= a.numel()


def cpu_port(shape, B, steps, warmup, threads):
    """The reference algorithm (oracle port of attn_aug_conv.py:65-97 + autograd) on the host cores."""
    from oracle import aaconv_oracle as O
    cin, hin, cout, dk, dv = SHAPES[shape]
    s = O.AAConvShape(cin, cout, 3, 2, dk, dv, 8, True, (hin // 2, hin // 2))
    torch.set_num_threads(threads)
    m = O.SequentialAAConv2d(s, O.init_params(s, seed=0))
    g = torch.Generator().manual_seed(0)
    x = torch.relu(torch.randn(B, cin, hin, hin, generator=g)).requires_grad_(True)
    dy = torch.randn(B, cout, hin // 2, hin // 2, generator=torch.Generator().manual_seed(1))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        m.zero_grad(set_to_none=True)
        x.grad = None
        m(x).backward(dy)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times)


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores, same config / metric / unit as our arm (B = 16 per step)."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cin, hin, cout, dk, dv = SHAPES[args.shape]
    B = args.ref_batch
    W = min(args.warmup, 1)
    K = args.steps if args.ref_max_steps is None else min(args.steps, args.ref_max_steps)   # ~0.8 s per B=16 step on 16 threads
    sec = cpu_port(args.shape, B, K, W, threads)
    tf = 3 * flops_fwd(B, cin, hin, cout, dk, dv) / sec / 1e12
    line = {'impl': 'reference', 'metric': 'aaconv_fwd_bwd_tflops', 'value': tf, 'unit': 'TFLOP/s', 'n_gpus': args.gpus,
            'steps': K, 'warmup': W, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'AAConv2d {args.shape} fwd+bwd (configs[1])', 'shape': args.shape, 'batch_per_gpu': args.batch,
                       'cin': cin, 'hin': hin, 'cout': cout, 'dk': dk, 'dv': dv, 'nh': 8, 'precision': 'fp32 (reference arithmetic)',
                       'sample_batch_per_step': B},
            'cpu_baseline': {'value': tf, 'unit': 'TFLOP/s', 'cores': threads, 'kind': 'port',
                             'sample': f'oracle.SequentialAAConv2d (reference op order, torch CPU fp32) {args.shape} B={B} '
                                       f'fwd+bwd x{K}'},
            'e2e': {'value': tf, 'unit': 'TFLOP/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


class Ctx:
    """Process / device context shared by the measurements of one bench.py run."""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.world = int(os.environ.get('WORLD_SIZE', 1))
        self.rank = int(os.environ.get('RANK', 0))
        self.local = int(os.environ.get('LOCAL_RANK', 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        if self.world > 1:
            # the model step captures its bucket all-reduces in a CUDA graph: no watchdog aborts while collectives are captured
            os.environ.setdefault('TORCH_NCCL_ASYNC_ERROR_HANDLING', '0')
            dist.init_process_group('nccl', device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return list(vals)
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()


def measure_model(ctx, args, K, W, cuda_graph, sampler=None, dump_dir=None):
    """configs[2]: whole-model data-parallel training step of aadensenet121 (chexpert.py:152-165) on synthetic radiographs:
    forward, BCE loss, backward with the bucketed NCCL gradient all-reduce, SGD-nesterov.  -> dict (rank 0 uses it).
    `dump_dir`: the loss of the last timed step and the parameters it left go there (dump_outputs)."""
    from chexpert_b200 import _lib
    from chexpert_b200.train import TrainStep, synthetic_batch
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    B = args.batch
    ts = TrainStep(dev, size=args.size, precision=args.precision, cuda_graph=cuda_graph, channels_last=args.channels_last,
                   buffered=not args.no_feature_buffer, fused_prologue=not args.no_fused_prologue)
    xh, th = synthetic_batch(B, size=args.size, seed=1000 + rank)
    xh, th = xh.pin_memory(), th.pin_memory()
    x, t = xh.to(dev), th.to(dev)
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def timed(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    def e2e_step():
        xd = xh.to(dev, non_blocking=True)
        td = th.to(dev, non_blocking=True)
        loss_host.copy_(ts(xd, td), non_blocking=True)

    for _ in range(W):
        ts(x, t)
    ctx.barrier()
    l0 = _lib.launch_count()
    last = {}
    ms = timed(lambda: last.update(loss=ts(x, t)), K)
    launches = _lib.launch_count() - l0
    if cuda_graph:          # replays do not pass through the host-side launch counter: count what one replay holds
        launches = ts.graph_launches * K
    if dump_dir and rank == 0:      # before the steps below overwrite the captured graph's output and the parameters
        last.update(('param_' + n.replace('.', '_'), p) for n, p in ts.model.named_parameters())
        dump_outputs(dump_dir, last)
    ctx.barrier()
    for _ in range(2):
        e2e_step()
    ctx.barrier()
    ms_e2e = timed(e2e_step, K)
    ctx.barrier()
    ms, ms_e2e = ctx.max_over_ranks(ms, ms_e2e)
    out = {'images_per_s': B * world / (ms * 1e-3), 'ms_per_step': ms, 'steps': K, 'warmup': W, 'n_gpus': world,
           'batch_per_gpu': B, 'image': args.size, 'precision': args.precision, 'cuda_graph': bool(cuda_graph),
           'feature_buffer': not args.no_feature_buffer, 'fused_prologue': not args.no_fused_prologue,
           'bucket_mb': 25.0, 'allreduce_bytes': ts.buckets.nbytes if ts.buckets is not None else 0,
           'n_buckets': len(ts.buckets.buckets) if ts.buckets is not None else 0,
           'e2e_images_per_s': B * world / (ms_e2e * 1e-3), 'e2e_ms_per_step': ms_e2e,
           'h2d_bytes_per_step': xh.numel() * 4 + th.numel() * 4, 'd2h_bytes_per_step': 4,
           'aaconv_launches': launches, 'loss': float(loss_host)}
    ts.release()
    ctx.barrier()
    return out


def run_model(args):
    """--workload model: the model measurement alone, as its own JSON line (images/s)."""
    ctx = Ctx(args)
    W, K = max(args.warmup, 3), args.steps
    sampler = ClockSampler(ctx.local)
    sampler.start()
    m = measure_model(ctx, args, K, W, args.cuda_graph, dump_dir=args.dump_outputs)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if ctx.rank == 0:
        line = {'metric': 'aadensenet121_train_images_per_s', 'value': m['images_per_s'], 'unit': 'images/s', 'n_gpus': ctx.world,
                'steps': K, 'warmup': W, 'ms_per_step': m['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic',
                'config': {'workload': 'aadensenet121 training step (configs[2])', 'batch_per_gpu': args.batch, 'image': args.size,
                           'precision': args.precision, 'optimizer': 'SGD nesterov momentum 0.9', 'parallelism': f'dp{ctx.world}',
                           'cuda_graph': bool(args.cuda_graph), 'feature_buffer': m['feature_buffer'], 'fused_prologue': m['fused_prologue'],
                           'l2': 'activations of one step (>> 126 MB) stream through L2; no explicit flush',
                           'dense_blocks': 'torch/cuDNN dense layers under torch.autocast(bf16), as the reference wires them'},
                'e2e': {'value': m['e2e_images_per_s'], 'unit': 'images/s', 'ms_per_step': m['e2e_ms_per_step'],
                        'h2d_bytes_per_step': m['h2d_bytes_per_step'], 'd2h_bytes_per_step': 4},
                'gpu_launches': m['aaconv_launches'], 'clocks': sampler.summary(), 'roofline': None, 'model': m}
        print(json.dumps(line), flush=True)
    finish(ctx, args.cuda_graph)


def finish(ctx, captured_nccl):
    sys.stdout.flush()
    if ctx.world > 1:
        ctx.barrier()
        if captured_nccl:        # process-group teardown after captured NCCL work has been seen to hang: leave without it
            os._exit(0)
        ctx.dist.destroy_process_group()


def ncu_traffic(kernel):
    """dram bytes per launch of `kernel` from the committed summary of this build's own `ncu --set full` capture
    (profiles/ncu_dram_bytes.json, written by tools/ncu_traffic.py from the .ncu-rep raw page); None if absent."""
    p = os.path.join(ROOT, 'profiles', 'ncu_dram_bytes.json')
    if not os.path.exists(p):
        return None, None
    j = json.load(open(p))
    return j.get('kernels', {}).get(kernel), j.get('source')


def measure_layer(ctx, args, shape, K, W, want_e2e=True, sampler=None, dump_dir=None):
    # args.io_dtype: element type of x / dy / y at the module boundary ('fp32' as the reference module, or 'bf16' = the
    # activations torch.autocast hands the Transition in the bf16 training configuration, configs[2])
    """One AAConv2d forward + backward at a Transition shape through the public nn.Module (configs[1]).  -> dict.
    `dump_dir`: y, dx and the (all-reduced) parameter gradients of the last timed step go there (dump_outputs)."""
    import chexpert_b200 as cb
    from chexpert_b200 import _lib
    dev, world, rank, dist = ctx.dev, ctx.world, ctx.rank, ctx.dist
    cin, hin, cout, dk, dv = SHAPES[shape]
    B = args.batch
    H = hin // 2

    torch.manual_seed(0)
    m = cb.AAConv2d(cin, cout, 3, 2, dk, dv, 8, True, (H, H), precision=args.precision)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Conv2d):
            torch.nn.init.kaiming_normal_(mod.weight)
    m = m.to(dev)
    params = [p for p in m.parameters()]
    g = torch.Generator().manual_seed(1000 + rank)
    io_t = torch.bfloat16 if (args.io_dtype == 'bf16' and args.precision == 'bf16') else torch.float32
    x_host = torch.relu(torch.randn(B, cin, hin, hin, generator=g)).to(io_t).pin_memory()
    dy_host = torch.randn(B, cout, H, H, generator=g).to(io_t).pin_memory()
    x = x_host.to(dev).requires_grad_(True)
    dy = dy_host.to(dev)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def step(xin, dyin):
        """-> y and the all-reduced parameter gradients (one flat tensor; None on one GPU, where p.grad is the result)."""
        for p in params:
            p.grad = None
        xin.grad = None
        y = m(xin)
        y.backward(dyin)
        flat = None
        if world > 1:   # data-parallel exchange step: one bucket with every parameter gradient of the module, averaged by NCCL
            flat = torch.cat([p.grad.reshape(-1) for p in params])
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
        return y, flat

    def timed(fn, n):
        """n calls, each bracketed by its own CUDA events on the current stream; L2 flushed in between."""
        evs = []
        for _ in range(n):
            if not args.no_flush:
                flush_buf.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / n   # ms

    for _ in range(W):
        step(x, dy)
    ctx.barrier()
    l0 = _lib.launch_count()
    last = {}
    t_wall = time.perf_counter()
    ms = timed(lambda: last.update(out=step(x, dy)), K)
    ctx.barrier()
    t_wall = time.perf_counter() - t_wall
    launches = _lib.launch_count() - l0
    if dump_dir and rank == 0:
        y, flat = last['out']
        grads = ([p.grad for p in params] if flat is None else
                 [g.view_as(p) for g, p in zip(flat.split([p.numel() for p in params]), params)])
        outs = {'y': y, 'grad_x': x.grad}
        outs.update(('grad_' + n.replace('.', '_'), g) for (n, _), g in zip(m.named_parameters(), grads))
        dump_outputs(dump_dir, outs)
    out = {'shape': shape, 'ms': ms, 'launches': launches, 't_wall': t_wall, 'h2d': 0, 'd2h': 0, 'ms_e2e': None,
           'io_dtype': 'bf16' if io_t == torch.bfloat16 else 'fp32'}

    if want_e2e:
        # end-to-end: pinned host buffers in, y + parameter grads out, every step.  The way a training loop feeds a GPU: the
        # uploads of step k+1 on a copy stream while step k computes, results read back on a third stream from double-buffered
        # device staging.  Every step's H2D and D2H copies are inside the timed region; they overlap compute.
        y_host = torch.empty(B, cout, H, H, dtype=io_t).pin_memory()
        g_host = [torch.empty(p.shape).pin_memory() for p in params]
        up, down = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        xbuf = [torch.empty_like(x) for _ in range(2)]
        dybuf = [torch.empty_like(dy) for _ in range(2)]
        ystage = [torch.empty(B, cout, H, H, device=dev, dtype=io_t) for _ in range(2)]
        gstage = [[torch.empty_like(p) for p in params] for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]       # upload into input buffer i finished
        freed = [torch.cuda.Event() for _ in range(2)]       # compute on input buffer i finished
        staged = [torch.cuda.Event() for _ in range(2)]      # results of a step are in staging buffer i
        drained = [torch.cuda.Event() for _ in range(2)]     # staging buffer i has been read back
        state = {'k': 0, 'n': 0}

        def upload(i):
            with torch.cuda.stream(up):
                up.wait_event(freed[i])
                xbuf[i].copy_(x_host, non_blocking=True)
                dybuf[i].copy_(dy_host, non_blocking=True)
                ready[i].record(up)

        def e2e_step():
            cur = torch.cuda.current_stream(dev)
            k = state['k']
            i = k & 1
            if k == 0:
                upload(i)
            if k + 1 < state['n']:
                upload(i ^ 1)                                # next step's inputs travel while this step computes
            cur.wait_event(ready[i])
            y, _ = step(xbuf[i].detach().requires_grad_(True), dybuf[i])
            freed[i].record(cur)
            cur.wait_event(drained[i])
            ystage[i].copy_(y.detach())
            for gs, p in zip(gstage[i], params):
                gs.copy_(p.grad)
            staged[i].record(cur)
            with torch.cuda.stream(down):
                down.wait_event(staged[i])
                y_host.copy_(ystage[i], non_blocking=True)
                for gh, gs in zip(g_host, gstage[i]):
                    gh.copy_(gs, non_blocking=True)
                drained[i].record(down)
            state['k'] = k + 1

        def e2e_timed(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            state['k'], state['n'] = 0, n
            torch.cuda.synchronize()
            cur = torch.cuda.current_stream(dev)
            for ev in freed + drained:
                ev.record(cur)
            a.record()
            for _ in range(n):
                e2e_step()
            cur.wait_stream(down)                            # the last read-back is part of the region
            cur.wait_stream(up)
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n

        e2e_timed(3)
        ctx.barrier()
        out['ms_e2e'] = e2e_timed(K)
        ctx.barrier()
        out['h2d'] = x_host.numel() * x_host.element_size() + dy_host.numel() * dy_host.element_size()
        out['d2h'] = y_host.numel() * y_host.element_size() + sum(t.numel() * 4 for t in g_host)

    out['ms'], e2e_max = ctx.max_over_ranks(out['ms'], out['ms_e2e'] or 0.0)
    if want_e2e:
        out['ms_e2e'] = e2e_max

    # per-kernel device times (own start/stop CUDA events around every launch) of three extra steps: dominant-kernel roofline
    ctx.barrier()
    if not args.no_flush:
        flush_buf.zero_()
    torch.cuda.synchronize()
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        step(x, dy)
    torch.cuda.synchronize()
    agg = {}
    for name, t in _lib.profile_end():
        a = agg.setdefault(name, [0.0, 0])
        a[0] += t
        a[1] += 1
    out['kernels'] = {n: {'ms_total_per_step': v[0] / 3, 'launches_per_step': v[1] / 3} for n, v in agg.items()}
    out['flops'] = 3 * flops_fwd(B, cin, hin, cout, dk, dv)
    return out


def roofline_of(layer, args, clocks, world):
    """Dominant kernel of a measured layer against the tensor peak (+ the MUFU.EX2 floor for the attention kernels)."""
    kern = layer['kernels']
    if not kern:
        return None
    cin, hin, cout, dk, dv = SHAPES[layer['shape']]
    B, H = args.batch, hin // 2
    L = H * H
    nh, dkh, dvh = 8, dk // 8, dv // 8
    peak_tf, peak_gbs, how = peaks()
    top = max(kern.items(), key=lambda kv: kv[1]['ms_total_per_step'])
    attn_f = 2 * B * nh * L * (L * dkh + dkh * (4 * H - 2) + L * dvh)
    dense = 2 * B * L * (9 * cin * (cout - dv) + cin * (2 * dk + dv))
    # algorithmic flops per launch (DESIGN.md section 4); recompute is not counted
    work = {'attn_fwd': attn_f, 'attn_bwd_dq': attn_f, 'attn_bwd_dkv': attn_f,
            'conv_qkv_fprop': dense, 'conv_qkv_dgrad': dense, 'conv_qkv_wgrad': dense}
    key = next((k for k in sorted(work, key=len, reverse=True) if top[0].startswith(k)), None)
    nl = max(top[1]['launches_per_step'], 1.0)
    dur = top[1]['ms_total_per_step'] * 1e-3 / nl
    ach = work[key] / dur / 1e12 if key else None
    # every score is exponentiated once per attention kernel: the MUFU.EX2 floor (15.9 ex2/clk/SM measured,
    # tools/mufu_bench.cu) is the binding roofline of the attention kernels, reported beside the tensor one
    exps = B * nh * L * L if top[0].startswith('attn_') else 0
    clk = (clocks['sm_mhz'] or 1965) * 1e6
    traffic, src = ncu_traffic(top[0]) if (layer['shape'] == 'T1' and B == 16) else (None, None)
    return {'kernel': top[0], 'bound': 'tensor', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s',
            'frac': (ach / peak_tf) if ach else None, 'traffic': traffic, 'traffic_source': src,
            'peak_source': how, 'ms_per_step': top[1]['ms_total_per_step'], 'launches_per_step': top[1]['launches_per_step'],
            'us_per_launch': dur * 1e6, 'mufu_exp_per_launch': exps,
            'mufu_floor_us': exps / (148 * 15.9 * clk) * 1e6 if exps else None,
            'mufu_frac': (exps / (148 * 15.9 * clk)) / dur if exps else None,
            'module_frac_of_bf16_peak': layer['flops'] / (layer['ms'] * 1e-3) / 1e12 / peak_tf}


def parity_note():
    """Measured bf16-mode parity figures of this build (profiles/parity_bf16.json, written by the GPU test run) -- printed in the
    line because one of them is a documented exception to north_star (see DESIGN.md section 7)."""
    p = os.path.join(ROOT, 'profiles', 'parity_bf16.json')
    return json.load(open(p)) if os.path.exists(p) else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', default=os.environ.get('AACONV_BENCH_PRECISION', 'bf16'), choices=['bf16', 'fp32'])
    ap.add_argument('--io-dtype', default='bf16', choices=['bf16', 'fp32'],
                    help="element type of x / dy / y at the AAConv2d boundary in bf16 mode: 'bf16' = autocast activations (what the "
                         "Transition receives in bf16 training, configs[2]); 'fp32' = the reference module's own tensors")
    ap.add_argument('--shape', default='T1', choices=list(SHAPES))
    ap.add_argument('--batch', type=int, default=16)
    ap.add_argument('--ref-batch', type=int, default=16, help='per-step batch of the CPU reference arm (same config as ours)')
    ap.add_argument('--ref-max-steps', type=int, default=None,
                    help='optional cap on the timed steps of the CPU reference arm (default: --steps, ~0.8 s each at B=16)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-flush', action='store_true')
    ap.add_argument('--no-model', action='store_true', help='skip the whole-model training measurement (`model` field)')
    ap.add_argument('--no-shapes', action='store_true', help='skip the T2 / T3 / T1_512 rows (`shapes` field; N = 1 only)')
    ap.add_argument('--model-eager', action='store_true', help='`model` field: eager step instead of the CUDA-graph replay')
    ap.add_argument('--no-feature-buffer', action='store_true',
                    help='model: torchvision dense blocks (torch.cat, torch BatchNorm) instead of the pre-allocated feature buffer with '
                         'fused strided BN + ReLU')
    ap.add_argument('--no-fused-prologue', action='store_true', help='model: nn.InstanceNorm2d + ReLU instead of the fused prologue')
    ap.add_argument('--workload', default='layer', choices=['layer', 'model'],
                    help="layer: AAConv2d fwd+bwd microbench (configs[1], the headline) plus `shapes` and `model` fields; model: the "
                         "aadensenet121 training step alone (configs[2]: batch 16/GPU, 320x320, SGD-nesterov, gradient all-reduce)")
    ap.add_argument('--size', type=int, default=320)
    ap.add_argument('--channels-last', action='store_true', help='model workload: channels_last memory format for the dense blocks')
    ap.add_argument('--cuda-graph', action='store_true', help='model workload: capture the whole training step in a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed to DIR/<name>.npy (float32; layer: y, grad_x and the parameter '
                         'gradients, model: loss and the updated parameters); inputs are seeded, so runs with the same arguments '
                         'compare output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
    if args.impl == 'reference':
        return run_reference(args)
    if args.workload == 'model':
        return run_model(args)

    ctx = Ctx(args)
    W, K = max(args.warmup, 3), args.steps
    sampler = ClockSampler(ctx.local)
    sampler.start()
    layer = measure_layer(ctx, args, args.shape, K, W, want_e2e=True, dump_dir=args.dump_outputs)
    other = None                                     # the same layer through the other boundary element type (reported beside)
    if args.precision == 'bf16' and ctx.world == 1:
        keep = args.io_dtype
        args.io_dtype = 'fp32' if keep == 'bf16' else 'bf16'
        other = measure_layer(ctx, args, args.shape, K, 3, want_e2e=True)
        args.io_dtype = keep
    shapes = {}
    if ctx.world == 1 and not args.no_shapes:
        for sh in ('T2', 'T3', 'T1_512'):
            if sh != args.shape:
                shapes[sh] = measure_layer(ctx, args, sh, K, 3, want_e2e=False)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.summary()
    model = None
    graph = not args.model_eager
    if not args.no_model:
        try:
            model = measure_model(ctx, args, K, max(W, 4), cuda_graph=graph)
        except Exception as e:   # the headline layer numbers are still printed
            model = {'error': f'{type(e).__name__}: {e}'[:300]}

    if ctx.rank == 0:
        cin, hin, cout, dk, dv = SHAPES[args.shape]
        world, B = ctx.world, args.batch
        f_tot = layer['flops']
        peak_tf, peak_gbs, how = peaks()
        tf = f_tot * world / (layer['ms'] * 1e-3) / 1e12
        srows = {}
        for sh, r in shapes.items():
            rf = roofline_of(r, args, clocks, 1)
            srows[sh] = {'ms_per_step': r['ms'], 'tflops': r['flops'] / (r['ms'] * 1e-3) / 1e12,
                         'frac_of_bf16_peak': r['flops'] / (r['ms'] * 1e-3) / 1e12 / peak_tf, 'launches_per_step': r['launches'] / K,
                         'dominant_kernel': rf['kernel'] if rf else None, 'dominant_us': rf['us_per_launch'] if rf else None,
                         'dominant_frac': rf['frac'] if rf else None}
        line = {'metric': 'aaconv_fwd_bwd_tflops', 'value': tf, 'unit': 'TFLOP/s', 'n_gpus': world, 'steps': K, 'warmup': W,
                'ms_per_step': layer['ms'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic',
                'config': {'workload': f'AAConv2d {args.shape} fwd+bwd (configs[1])', 'shape': args.shape,
                           'batch_per_gpu': B, 'cin': cin, 'hin': hin, 'cout': cout, 'dk': dk, 'dv': dv, 'nh': 8,
                           'precision': args.precision, 'boundary_dtype': layer['io_dtype'], 'l2': 'flushed between timed steps (256 MiB memset)' if not args.no_flush else 'not flushed',
                           'gflop_per_step_per_gpu': f_tot / 1e9, 'wall_s_timed_region': layer['t_wall'],
                           'tolerance': 'bf16 mode: outputs rtol 2e-2 / atol 1e-2 on >= 99.9 % of elements; gradients by relative L2 <= 3e-2, '
                                        '<= 4e-2 of max-abs and <= 2.5x torch.autocast (DESIGN.md section 7) -- a substitute for a fixed atol'},
                'e2e': {'value': f_tot * world / (layer['ms_e2e'] * 1e-3) / 1e12, 'unit': 'TFLOP/s', 'ms_per_step': layer['ms_e2e'],
                        'h2d_bytes_per_step': layer['h2d'], 'd2h_bytes_per_step': layer['d2h'],
                        'boundary_dtype': layer['io_dtype'],
                        'pipeline': 'pinned host buffers; upload of step k+1 and read-back of step k on side streams overlap compute'},
                'gpu_launches': layer['launches'], 'clocks': clocks, 'roofline': roofline_of(layer, args, clocks, world),
                'kernels': layer['kernels'], 'shapes': srows, 'model': model, 'parity': parity_note()}
        if other is not None:
            line['other_boundary'] = {'boundary_dtype': other['io_dtype'], 'ms_per_step': other['ms'],
                                      'value': f_tot / (other['ms'] * 1e-3) / 1e12, 'e2e_ms_per_step': other['ms_e2e'],
                                      'e2e_value': f_tot / (other['ms_e2e'] * 1e-3) / 1e12, 'h2d_bytes_per_step': other['h2d'],
                                      'd2h_bytes_per_step': other['d2h']}
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            cb_B = args.ref_batch
            sec = cpu_port(args.shape, cb_B, 3, 1, threads)
            line['cpu_baseline'] = {'value': 3 * flops_fwd(cb_B, cin, hin, cout, dk, dv) / sec / 1e12, 'unit': 'TFLOP/s',
                                    'cores': threads, 'kind': 'port',
                                    'sample': f'oracle.SequentialAAConv2d {args.shape} B={cb_B} fwd+bwd, 1 warm-up + 3 timed'}
        print(json.dumps(line), flush=True)
    finish(ctx, captured_nccl=(model is not None and graph))


if __name__ == '__main__':
    main()
