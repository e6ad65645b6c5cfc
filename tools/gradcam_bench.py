"""Grad-CAM on the fused inference path (Predictor.grad_cam, csrc/cam.cu) against what a user can do without it.

    python tools/gradcam_bench.py --out DIR [--batches 8] [--launches 400]

At 320 px, for aadensenet121 and densenet121, batch 16 and 64, precision fp32 and bf16 (bf16 AAConv2d kernels, fp32 dense blocks:
the Predictor's default), over `--batches` batches of synthetic radiographs (uint8, on the device):
    call        Predictor.__call__ (CUDA graph): logits only
    grad_cam    Predictor.grad_cam (CUDA graph): the same logits and (N, 5, 320, 320) Grad-CAM maps
    module      the module path as it runs today: the model (no feature buffer) in eval mode with autograd on, a forward hook on
                model.features (the output captured, the model going on with a clone), autograd.grad of each of the 5 classes' summed
                logits, alpha = mean gradient, relu(sum alpha * A), F.interpolate to 320 px
Each arm: ms per batch and images/s from a host clock around a synchronised loop, after two warm-up calls.
    kernel      aaconv_grad_cam alone at B = 16 and 64 (norm5 input (B, 1024, 10, 10) fp32 and bf16, K = 5, S = 320), --launches
                calls that rotate over 8 input / output sets (a working set larger than the 126 MB L2): CUDA events around the whole
                loop (us_per_call_stream: includes the host's ctypes calls between launches), and the library's per-launch event
                pairs (us_per_kernel, us_device: the kernels' own device time); bytes = the input read once + cam and upsampled maps
                written, GB/s against the device time
Writes DIR/gradcam_bench.json and prints it; the card's name and power limit come from the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from chexpert_b200 import evaluate as E          # noqa: E402
from chexpert_b200.densenet import build_model   # noqa: E402
from chexpert_b200 import _lib                   # noqa: E402
from chexpert_b200.aaconv import _ptr, _stream   # noqa: E402

SIZE, K = 320, 5


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return info


def timed(fn, n_batches, bs):
    fn()
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {'ms_per_batch': round(1e3 * dt / n_batches, 3), 'images_per_s': round(n_batches * bs / dt, 1)}


def module_grad_cam(model, x):
    store = {}

    def hook(m, i, o):
        store['A'] = o
        return o.clone()
    h = model.features.register_forward_hook(hook)
    try:
        z = model(x)
        A = store['A']
        maps = []
        for c in range(K):
            g, = torch.autograd.grad(z[:, c].sum(), A, retain_graph=c < K - 1)
            maps.append(torch.relu((g.mean((2, 3), keepdim=True) * A).sum(1)))
    finally:
        h.remove()
    return z.detach(), F.interpolate(torch.stack(maps, 1).detach(), size=(SIZE, SIZE), mode='bilinear', align_corners=False)


def arms(arch, precision, bs, n_batches, images):
    torch.manual_seed(0)
    sd = build_model(arch, K, SIZE, precision).state_dict()
    p = E.Predictor(K, SIZE, precision=precision, batch_size=bs, arch=arch)
    p.load_state_dict(sd)
    out = {'call': timed(lambda: p(images), n_batches, bs), 'grad_cam': timed(lambda: p.grad_cam(images), n_batches, bs)}
    model = build_model(arch, K, SIZE, precision).cuda().eval()
    model.load_state_dict(sd)

    def module():
        for i in range(0, images.shape[0], bs):
            module_grad_cam(model, E.normalise_u8(images[i:i + bs]))
    out['module'] = timed(module, n_batches, bs)
    del p, model
    torch.cuda.empty_cache()
    return out


def kernel(bs, dtype, launches):
    C, h, w = 1024, 10, 10
    norm5 = torch.nn.BatchNorm2d(C).cuda().eval()
    W = torch.randn(K, C, device='cuda')
    lib = _lib.load()
    # 8 input / output sets, preallocated: the working set exceeds the L2
    sets = [(torch.randn(bs, C, h, w, device='cuda').to(dtype), torch.empty(bs, K, h, w, device='cuda'),
             torch.empty(bs, K, SIZE, SIZE, device='cuda'), torch.empty(bs * C, device='cuda', dtype=torch.int32)) for _ in range(8)]
    nbytes = bs * C * h * w * sets[0][0].element_size() + bs * K * h * w * 4 + bs * K * SIZE * SIZE * 4

    def run(i):
        x, cam, up, ws = sets[i % 8]
        _lib.check(lib.aaconv_grad_cam(_ptr(x), _lib.BF16 if dtype == torch.bfloat16 else _lib.FP32, bs, C, h, w, x.stride(0),
                                       _ptr(norm5.weight), _ptr(norm5.bias), _ptr(norm5.running_mean), _ptr(norm5.running_var),
                                       norm5.eps, _ptr(W), K, _ptr(cam), _ptr(up), SIZE, _ptr(ws), _stream()), 'aaconv_grad_cam')
    for i in range(16):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    us = 1e3 * e0.elapsed_time(e1) / launches
    # the same calls with the library's per-launch event pairs: device time of each kernel, without the host's gaps between calls
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    for i in range(launches):
        run(i)
    torch.cuda.synchronize()
    per = {}
    for name, ms in _lib.profile_end(4 * launches):
        per[name] = per.get(name, 0.0) + 1e3 * ms / launches
    dev = sum(per.values())
    return {'us_per_call_stream': round(us, 2), 'us_per_kernel': {k: round(v, 2) for k, v in per.items()}, 'us_device': round(dev, 2),
            'bytes': nbytes, 'GB_per_s_device': round(nbytes / dev / 1e3, 1), 'working_set_MB': round(8 * (nbytes + bs * C * 4) / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--batches', type=int, default=8)
    ap.add_argument('--launches', type=int, default=400)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'gradcam_bench needs a CUDA device'
    torch.backends.cudnn.benchmark = False
    res = {'card': card(), 'size': SIZE, 'batches': a.batches, 'arms': {}, 'kernel': {}}
    for bs in (16, 64):
        images = E.synthetic_radiographs_u8(bs * a.batches, SIZE, seed=3).cuda()
        for arch in ('aadensenet121', 'densenet121'):
            for precision in ('bf16', 'fp32'):
                key = f'{arch}/{precision}/B{bs}'
                res['arms'][key] = arms(arch, precision, bs, a.batches, images)
                print(key, res['arms'][key], flush=True)
        for dt, dtype in (('fp32', torch.float32), ('bf16', torch.bfloat16)):
            res['kernel'][f'{dt}/B{bs}'] = kernel(bs, dtype, a.launches)
            print('kernel', dt, bs, res['kernel'][f'{dt}/B{bs}'], flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'gradcam_bench.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
