"""The input side of training and inference: the reference's host transform (PIL, DataLoader workers) against the device kernel
(chexpert_b200.preprocess, csrc/prep.cu).

    python tools/prep_bench.py --out DIR [--steps 30] [--launches 200]

Two geometry mixes of B = 16 raw 8-bit radiographs: 'small' (CheXpert-small-like, 320 x 390 and 390 x 320: the resize is an
identity, only the crop runs) and 'full' (full-resolution-like, 2320 x 2828, 2828 x 2320, 3000 x 2500 and 2500 x 3000).
    kernel      prepare() per batch, CUDA events over --launches launches that rotate over 8 batches with 8 separate outputs (a working
                set of 8 x (input + 19.7 MB output), larger than the 126 MB L2 for both mixes); bytes = input pixels + fp32 output,
                GB/s against that
    host_pil    Resize(320) + CenterCrop(320) + ToTensor + Normalize + 3-channel expand (the reference transform) on every host core
                through a process pool, as DataLoader workers run it; images/s over the pool's wall time
    predictor   aadensenet121 bf16 Predictor (CUDA graph), 64 raw host images per call: the device path (pack, upload, prep, model)
                against host PIL in the pool to uint8 crops followed by today's uint8 path; images/s, each arm timed on its own
    train_e2e   TrainStep (bf16, buffered, fused prologue, CUDA graph) at B = 16: a pinned raw Radiographs batch per step against the
                pinned fp32 x that bench.py's e2e copies; images/s
Writes DIR/prep_bench.json and prints it; the card's name and power limit come from the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SIZE, B = 320, 16
MIXES = {'small': [(320, 390), (390, 320)], 'full': [(2320, 2828), (2828, 2320), (3000, 2500), (2500, 3000)]}


def radiographs(mix, n, seed):
    """n deterministic radiograph-like images of the mix (smooth content plus noise; any content costs the same)."""
    rng = np.random.default_rng(seed)
    shapes = MIXES[mix]
    out = []
    for i in range(n):
        h, w = shapes[i % len(shapes)]
        coarse = rng.integers(60, 200, (h // 64 + 1, w // 64 + 1)).astype(np.int16)
        base = np.repeat(np.repeat(coarse, 64, 0), 64, 1)[:h, :w]
        out.append(np.clip(base + rng.integers(-8, 9, (h, w), dtype=np.int16), 0, 255).astype(np.uint8))
    return out


# ---- host side: process-pool workers ----------------------------------------------------------------------------------
_IMAGES = {}


def _pil_job(job):
    """Worker: the reference transform over `reps` passes of the mix's images (made once per worker).  mode 'float' -> count;
    mode 'u8' -> the uint8 crops (what the Predictor's uint8 path takes)."""
    import torchvision.transforms as T
    from PIL import Image
    torch.set_num_threads(1)          # as in a DataLoader worker: one worker per core, no intra-op thread pools on top
    mix, n, seed, reps, mode = job
    key = (mix, n, seed)
    if key not in _IMAGES:
        _IMAGES[key] = [Image.fromarray(a, 'L') for a in radiographs(mix, n, seed)]
    crop = T.Compose([T.Resize(SIZE), T.CenterCrop(SIZE)])
    full = T.Compose([crop, T.ToTensor(), T.Normalize([0.5330], [0.0349]), T.Lambda(lambda x: x.expand(3, -1, -1))])
    if mode == 'u8':
        return np.stack([np.asarray(crop(im)) for im in _IMAGES[key]])
    for _ in range(reps):
        for im in _IMAGES[key]:
            full(im)
    return reps * n


def host_pil(pool, workers, mix, reps):
    jobs = [(mix, len(MIXES[mix]), 100 + w, reps, 'float') for w in range(workers)]
    list(pool.map(_pil_job, [(m, n, s, 1, md) for m, n, s, _, md in jobs]))        # warm: images made, modules imported
    t0 = time.perf_counter()
    done = sum(pool.map(_pil_job, jobs))
    dt = time.perf_counter() - t0
    return {'workers': workers, 'images': done, 'seconds': dt, 'images_per_s': done / dt}


def host_u8(pool, workers, mix, n, seed):
    """n images of the mix as uint8 crops, produced by the pool (the images are split over the workers by seed)."""
    per = -(-n // workers)
    parts = list(pool.map(_pil_job, [(mix, per, seed + w, 1, 'u8') for w in range(workers)]))
    return torch.from_numpy(np.concatenate(parts)[:n])


def raw_images(workers, mix, n, seed):
    per = -(-n // workers)
    out = []
    for w in range(workers):
        out += radiographs(mix, per, seed + w)
    return out[:n]


# ---- device side ------------------------------------------------------------------------------------------------------
def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return info


def events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def kernel(mix, launches):
    from chexpert_b200.preprocess import pack_radiographs, prepare
    rads = [pack_radiographs(radiographs(mix, B, 200 + r), SIZE).to('cuda') for r in range(8)]
    outs = [torch.empty(B, 3, SIZE, SIZE, device='cuda') for _ in rads]
    for r, o in zip(rads, outs):
        prepare(r, out=o)
    torch.cuda.synchronize()
    ms = events(lambda i: prepare(rads[i % 8], out=outs[i % 8]), launches)
    in_bytes, out_bytes = rads[0].pixels.numel(), outs[0].numel() * 4
    return {'ms_per_batch': ms, 'input_bytes': in_bytes, 'output_bytes': out_bytes,
            'gb_per_s': (in_bytes + out_bytes) / (ms * 1e-3) / 1e9, 'images_per_s': B / (ms * 1e-3)}


def predictor(pool, workers, mix, n, reps):
    from chexpert_b200.evaluate import Predictor
    p = Predictor(5, SIZE, precision='bf16', batch_size=B)
    raw = raw_images(workers, mix, n, 300)
    u8 = host_u8(pool, workers, mix, n, 300)
    for _ in range(3):                                  # warm-up: both paths captured
        want, got = p(u8), p(raw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        p(raw)
    torch.cuda.synchronize()
    t_dev = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        p(host_u8(pool, workers, mix, n, 300))
    torch.cuda.synchronize()
    t_host = (time.perf_counter() - t0) / reps
    return {'images_per_call': n, 'device_prep_images_per_s': n / t_dev, 'host_pil_then_u8_images_per_s': n / t_host,
            'captures': p.captures, 'logits_equal': bool(torch.equal(want, got))}


def train_e2e(steps):
    from chexpert_b200.preprocess import pack_radiographs
    from chexpert_b200.train import TrainStep, synthetic_batch
    ts = TrainStep('cuda', size=SIZE, precision='bf16', cuda_graph=True, buffered=True, fused_prologue=True)
    xh, th = synthetic_batch(B, size=SIZE, seed=1000)
    xh, th = xh.pin_memory(), th.pin_memory()
    x, t = xh.cuda(), th.cuda()
    for _ in range(3):
        ts(x, t)
    arms = {'fp32_x': lambda: ts(xh.to('cuda', non_blocking=True), th.to('cuda', non_blocking=True))}
    for mix in MIXES:
        rad = pack_radiographs(radiographs(mix, B, 400), SIZE)
        arms['raw_' + mix] = lambda rad=rad: ts(rad, th.to('cuda', non_blocking=True))
    out = {}
    for _ in range(2):                                   # two rounds, arms alternating
        for name, fn in arms.items():
            for _ in range(2):
                fn()
            ms = events(lambda i: fn(), steps)
            out.setdefault(name, []).append(B / (ms * 1e-3))
    res = {name: {'images_per_s': max(r), 'rounds': r} for name, r in out.items()}
    res['h2d_bytes_per_step'] = {'fp32_x': xh.numel() * 4,
                                 **{'raw_' + m: sum(h * w for h, w in MIXES[m] * (B // len(MIXES[m]))) for m in MIXES}}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--launches', type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('prep_bench.py measures on a CUDA device; none found')
    os.makedirs(args.out, exist_ok=True)
    workers = os.cpu_count()
    res = {'card': card(), 'host_cpus': workers, 'batch': B, 'size': SIZE,
           'mixes': {m: [list(s) for s in v] for m, v in MIXES.items()}}
    import multiprocessing as mp
    with ProcessPoolExecutor(workers, mp_context=mp.get_context('spawn')) as pool:
        res['host_pil'] = {m: host_pil(pool, workers, m, 2000 if m == 'small' else 16) for m in MIXES}
        print(json.dumps(res['host_pil']), flush=True)
        res['kernel'] = {m: kernel(m, args.launches) for m in MIXES}
        print(json.dumps(res['kernel']), flush=True)
        res['predictor'] = {m: predictor(pool, workers, m, 64, 5) for m in MIXES}
        print(json.dumps(res['predictor']), flush=True)
    res['train_e2e'] = train_e2e(args.steps)
    print(json.dumps(res['train_e2e']), flush=True)
    with open(os.path.join(args.out, 'prep_bench.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
