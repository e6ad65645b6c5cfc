"""Training and inference throughput of the reference's baseline model, torchvision's densenet121, at batch 16 and 320 px.

    python tools/densenet121_bench.py [--out DIR] [--precisions bf16,fp32] [--steps 20] [--warmup 4] [--rounds 2]

The arms, all from the same seeded state_dict:
    torchvision  (a) torchvision's modules: densenet121() without options, which is torchvision.models.densenet121 op for op
                     (tests/test_densenet121.py checks them bit for bit on CPU); for inference torchvision.models.densenet121 itself
    buffered     (b) densenet121(feature_buffer=True): the fused dense blocks, module Transitions
    fused        (c) densenet121(feature_buffer=True, fused_transition=True): the fused BatchNorm + ReLU + pool Transitions as well
Training: train.TrainStep(arch='densenet121', cuda_graph=True) on one synthetic batch, images/s over --steps replayed steps after
--warmup steps (two eager, the capture, replays).  Inference: evaluate.Predictor(arch='densenet121') with its CUDA graph; for (a)
and (b) the same Predictor runs torchvision's model / the fused model with module Transitions.  'bf16' is bf16 autocast in both
(TrainStep: bf16 weight shadows; Predictor: autocast=True, bf16 weights for every arm); 'fp32' has TF32 off.  Times come from CUDA
events; the arms alternate within every round.  Also printed: the largest difference of the training losses and of the logits
between arm (a) and the others, and the card's name and power limit from the same run.  Prints one JSON object, and writes it to
DIR/densenet121_bench.json with --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torchvision

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from chexpert_b200 import evaluate as E                   # noqa: E402
from chexpert_b200.densenet import BNTransition          # noqa: E402
from chexpert_b200.train import TrainStep, synthetic_batch  # noqa: E402

SIZE, BATCH = 320, 16
ARMS = ('torchvision', 'buffered', 'fused')


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return info


def timed(fn, steps):
    """-> (seconds per call over `steps` calls, CUDA events), and what the last call returned."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / steps, out


def train_steps(precision):
    kw = dict(size=SIZE, precision=precision, lr=1e-3, seed=0, arch='densenet121', cuda_graph=True)
    return {'torchvision': TrainStep('cuda', buffered=False, fused_prologue=False, **kw),
            'buffered': TrainStep('cuda', buffered=True, fused_prologue=False, **kw),
            'fused': TrainStep('cuda', buffered=True, fused_prologue=True, **kw)}


def predictors(precision, sd):
    autocast = precision == 'bf16'
    ps = {a: E.Predictor(5, SIZE, batch_size=BATCH, autocast=autocast, arch='densenet121') for a in ARMS}
    for m in ps['buffered'].model.modules():            # module Transitions in the fused-eval model
        if isinstance(m, BNTransition):
            m.fused_eval = False
    tv = torchvision.models.densenet121(num_classes=5)
    tv.load_state_dict(sd)
    tv.requires_grad_(False)
    if autocast:
        for m in tv.modules():
            if isinstance(m, torch.nn.Conv2d):
                m.weight.data = m.weight.data.to(torch.bfloat16)
    ps['torchvision'].model = tv.cuda().eval()
    for a in ('buffered', 'fused'):
        ps[a].load_state_dict(sd)
    return ps


def run(precision, steps, warmup, rounds):
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    x, t = synthetic_batch(BATCH, size=SIZE, seed=5, device='cuda')
    res = {'precision': precision, 'train_images_per_s': {a: [] for a in ARMS}, 'infer_images_per_s': {a: [] for a in ARMS}}
    ts = train_steps(precision)
    sd = {k: v.detach().cpu() for k, v in ts['torchvision'].model.state_dict().items()}
    losses = {a: [float(ts[a](x, t)) for _ in range(warmup)] for a in ARMS}      # eager, capture, replays: the same losses compared
    for _ in range(rounds):
        for a in ARMS:
            sec, _ = timed(lambda: ts[a](x, t), steps)
            res['train_images_per_s'][a].append(BATCH / sec)
    res['train_losses'] = losses
    res['max_loss_diff_vs_torchvision'] = {a: max(abs(u - v) for u, v in zip(losses[a], losses['torchvision'])) for a in ARMS[1:]}
    del ts
    torch.cuda.empty_cache()
    images = E.synthetic_radiographs_u8(BATCH * 4, SIZE, seed=3)
    ps = predictors(precision, sd)
    logits = {a: ps[a](images) for a in ARMS}          # two eager batches, the capture, a replay
    dev = images[:BATCH].cuda()
    for _ in range(rounds):
        for a in ARMS:
            sec, _ = timed(lambda: ps[a](dev), steps)
            res['infer_images_per_s'][a].append(BATCH / sec)
    res['max_logit_diff_vs_torchvision'] = {a: float((logits[a] - logits['torchvision']).abs().max()) for a in ARMS[1:]}
    res['captures'] = {a: ps[a].captures for a in ARMS}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--precisions', default='bf16,fp32')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=4)
    ap.add_argument('--rounds', type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('densenet121_bench.py measures on a CUDA device; none is available')
    if args.warmup < 4:
        raise SystemExit('--warmup must be >= 4: two eager steps, the capture and one replay')
    out = {'card': card(), 'batch': BATCH, 'size': SIZE, 'steps': args.steps, 'warmup': args.warmup,
           'results': [run(p, args.steps, args.warmup, args.rounds) for p in args.precisions.split(',')]}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'densenet121_bench.json'), 'w') as f:
            f.write(s)


if __name__ == '__main__':
    main()
