"""Inference throughput of aadensenet121 at 320 px: today's evaluation against the fused dense-block Predictor.

    python tools/infer_bench.py --out DIR [--batches 16,64] [--precisions bf16,fp32] [--seconds 1.0] [--rounds 3]

The arms, each fed the same host uint8 images (4 batches per call) and the same seeded checkpoint:
    plain      evaluate.predict_logits on aadensenet121()                                     (today's evaluation)
    buffered   evaluate.predict_logits on aadensenet121(feature_buffer=True, fused_prologue=True)
    eager      evaluate.Predictor(cuda_graph=False)
    graph      evaluate.Predictor(cuda_graph=True)
    graph_autocast  evaluate.Predictor(cuda_graph=True, autocast=True)                            (bf16 only)
'bf16' is precision='bf16': the AAConv2d kernels in bf16; the dense blocks stay fp32 in every arm but graph_autocast, which runs
them under bf16 autocast (opt-in: it misses the bf16 mode's AUROC gate, see DESIGN.md).  Every arm is warmed up at its shape, then timed
with CUDA events over windows of at least --seconds each; the arms alternate within every round.  Also measured: the wall time of
the 10-checkpoint x 234-image evaluate_ensemble with the plain model and with a Predictor, and the largest logit difference between
the plain arm and every other arm on the same images.  Writes DIR/infer_bench.json and prints it; the card's name and power limit come
from the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from chexpert_b200 import evaluate as E          # noqa: E402
from chexpert_b200.densenet import aadensenet121  # noqa: E402

SIZE = 320


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return info


def checkpoint(seed, precision, **kw):
    torch.manual_seed(seed)
    return aadensenet121(5, (SIZE, SIZE), precision=precision, **kw)


def arms(precision, bs, sd):
    plain = checkpoint(0, precision).cuda().eval()
    buffered = checkpoint(0, precision, feature_buffer=True, fused_prologue=True).cuda().eval()
    plain.load_state_dict(sd)
    buffered.load_state_dict(sd)
    eager = E.Predictor(5, SIZE, precision=precision, batch_size=bs, cuda_graph=False)
    graph = E.Predictor(5, SIZE, precision=precision, batch_size=bs, cuda_graph=True)
    eager.load_state_dict(sd)
    graph.load_state_dict(sd)
    fns = {'plain': lambda im: E.predict_logits(plain, im, bs), 'buffered': lambda im: E.predict_logits(buffered, im, bs),
           'eager': eager, 'graph': graph}
    if precision == 'bf16':
        fns['graph_autocast'] = E.Predictor(5, SIZE, precision=precision, batch_size=bs, cuda_graph=True, autocast=True)
        fns['graph_autocast'].load_state_dict(sd)
    return fns


def window(fn, images, seconds):
    """-> (images per second, calls) over one window of at least `seconds`, timed with CUDA events."""
    t0 = time.perf_counter()
    fn(images)
    torch.cuda.synchronize()
    reps = max(1, int(seconds / max(time.perf_counter() - t0, 1e-4)) + 1)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn(images)
    stop.record()
    stop.synchronize()
    return reps * images.shape[0] / (start.elapsed_time(stop) / 1e3), reps


def throughput(precisions, batches, seconds, rounds, sd):
    out = []
    for precision in precisions:
        for bs in batches:
            images = E.synthetic_radiographs_u8(4 * bs, SIZE, seed=5)
            fns = arms(precision, bs, sd)
            logits = {}
            for name, fn in fns.items():          # warm-up: every arm at its shape (the graph arm captures here)
                for _ in range(3):
                    logits[name] = fn(images)
            torch.cuda.synchronize()
            rates = {name: [] for name in fns}
            for _ in range(rounds):
                for name, fn in fns.items():
                    rates[name].append(window(fn, images, seconds)[0])
            row = {'precision': precision, 'batch': bs, 'images_per_call': images.shape[0],
                   'images_per_s': {n: sorted(r)[len(r) // 2] for n, r in rates.items()},
                   'images_per_s_rounds': rates,
                   'max_abs_logit_diff_plain_vs': {n: float((logits['plain'] - logits[n]).abs().max()) for n in fns if n != 'plain'},
                   'graph_captures': fns['graph'].captures}
            row['speedup_vs_plain'] = {n: r / row['images_per_s']['plain'] for n, r in row['images_per_s'].items()}
            print(json.dumps(row), flush=True)
            out.append(row)
            del fns
            torch.cuda.empty_cache()
    return out


def ensemble(precisions, n_ckpt, sds):
    images, targets = E.synthetic_radiographs_u8(234, SIZE, seed=3), E.synthetic_eval_targets(234, seed=4)
    out = []
    for precision in precisions:
        model = checkpoint(0, precision).cuda()
        preds = [('predictor', E.Predictor(5, SIZE, precision=precision, batch_size=16))]
        if precision == 'bf16':
            preds.append(('predictor_autocast', E.Predictor(5, SIZE, precision=precision, batch_size=16, autocast=True)))
        times = {name: [] for name, _ in [('plain', model)] + preds}
        res = {}
        for _ in range(2):                       # the Predictor's first run includes its warm-up batches and the capture
            for name, m in [('plain', model)] + preds:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res[name] = E.evaluate_ensemble(m, sds[:n_ckpt], images, targets)
                torch.cuda.synchronize()
                times[name].append(time.perf_counter() - t0)
        row = {'precision': precision, 'checkpoints': n_ckpt, 'images': 234, 'wall_s_first_run': {k: v[0] for k, v in times.items()},
               'wall_s_second_run': {k: v[1] for k, v in times.items()},
               'max_abs_logit_diff_plain_vs': {n: float((res['plain']['per_model'] - res[n]['per_model']).abs().max()) for n, _ in preds},
               'auroc': {n: r['auroc'].tolist() for n, r in res.items()},
               'predictor_captures': {n: p.captures for n, p in preds}}
        print(json.dumps(row), flush=True)
        out.append(row)
        del model, preds
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', required=True, help='directory for infer_bench.json')
    ap.add_argument('--batches', default='16,64')
    ap.add_argument('--precisions', default='bf16,fp32')
    ap.add_argument('--seconds', type=float, default=1.0, help='least timed work per arm and round')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--checkpoints', type=int, default=10, help='checkpoints of the ensemble timing (0: skip it)')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('infer_bench.py measures on a CUDA device; none is available')
    os.makedirs(a.out, exist_ok=True)
    precisions, batches = a.precisions.split(','), [int(b) for b in a.batches.split(',')]
    info = card()
    print(json.dumps(info), flush=True)
    sds = [checkpoint(s, 'fp32').state_dict() for s in range(max(1, a.checkpoints))]
    result = {'card': info, 'size': SIZE, 'tf32': {'cudnn': torch.backends.cudnn.allow_tf32,
                                                   'matmul': torch.backends.cuda.matmul.allow_tf32},
              'throughput': throughput(precisions, batches, a.seconds, a.rounds, sds[0]),
              'ensemble': ensemble(precisions, a.checkpoints, sds) if a.checkpoints > 0 else []}
    with open(os.path.join(a.out, 'infer_bench.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps({'card': info['name'], 'throughput': [(r['precision'], r['batch'], r['images_per_s']) for r in result['throughput']],
                      'ensemble': [(r['precision'], r['wall_s_second_run']) for r in result['ensemble']]}))


if __name__ == '__main__':
    main()
