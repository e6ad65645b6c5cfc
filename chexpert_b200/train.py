"""One data-parallel training step of aadensenet121, the way chexpert.py:152-165 runs it, on synthetic
radiograph-shaped batches (SURVEY.md section 8d, configs 1/3/4).

    model(x) -> BCE-with-logits on the 5 competition classes, sum over classes, mean over batch (chexpert.py:160,530)
    -> backward -> [bucketed all-reduce over ranks] -> SGD(momentum 0.9, nesterov) + MultiStepLR (chexpert.py:479-480)

The loop around it (tqdm, tensorboard, checkpoint tracker, periodic eval; chexpert.py:167-193) is outside the hot
path and not rebuilt; `TrainStep` is what bench.py times and what a user's own loop would call per batch.
"""
import contextlib
import os

import torch
import torch.distributed as dist

from . import _lib
from .dataparallel import GradientBuckets
from .densenet import build_model, conv_weight_plan
from .loss import BCEWithLogitsLoss

# dataset normalisation constants of the reference transform (chexpert.py:70-72)
PIXEL_MEAN, PIXEL_STD = 0.5330, 0.0349


def synthetic_batch(batch, size=320, seed=0, device='cpu', raw_labels=True):
    """Radiograph-shaped synthetic input: one-channel U[0,1] image normalised and replicated to 3 channels
    (chexpert.py:64-72), labels either raw 14-wide rows in {nan,-1,0,1} (dataset.py:20-23) or (B,5) {0,1} targets."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(batch, 1, size, size, generator=g)
    x = ((u - PIXEL_MEAN) / PIXEL_STD).expand(-1, 3, -1, -1).contiguous()
    if raw_labels:
        vals = torch.tensor([float('nan'), -1.0, 0.0, 1.0])
        idx = torch.multinomial(torch.tensor([0.55, 0.10, 0.15, 0.20]), batch * 14, replacement=True, generator=g)
        t = vals[idx].reshape(batch, 14)
    else:
        t = (torch.rand(batch, 5, generator=g) < 0.3).float()
    return x.to(device), t.to(device)


class TrainStep:
    """Owns model, loss kernel, optimizer, scheduler and (when world > 1) the gradient buckets."""

    def __init__(self, device, size=320, precision='bf16', lr=1e-4, raw_labels=True, bucket_mb=25.0, seed=0,
                 autocast=True, channels_last=False, cuda_graph=False, graph_after=2, buffered=False, fused_prologue=False,
                 batched_casts=True, arch='aadensenet121'):
        torch.manual_seed(seed)
        self.device = torch.device(device)
        # arch (densenet.build_model): 'aadensenet121' or the reference's baseline 'densenet121'; the optimizer is the same for both
        self.model = build_model(arch, 5, size, precision, feature_buffer=buffered, fused=fused_prologue).to(self.device)
        if channels_last:
            self.model = self.model.to(memory_format=torch.channels_last)
        self.loss_fn = BCEWithLogitsLoss('train', raw_labels=raw_labels).to(self.device)
        self.opt = torch.optim.SGD(self.model.parameters(), lr=lr, momentum=0.9, nesterov=True)
        self.sched = torch.optim.lr_scheduler.MultiStepLR(self.opt, [40000, 60000])
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        # the dense blocks are torch/cuDNN (outside the hot path); bf16 autocast only decides THEIR arithmetic
        self.autocast = bool(autocast and precision == 'bf16' and self.device.type == 'cuda')
        # cuda_graph: after `graph_after` eager steps (they create the momentum buffers and warm cuDNN up) the whole step --
        # forward, loss, backward, bucket all-reduces, optimizer -- is captured once and replayed: the ~3000 small launches
        # of the 120-layer dense blocks stop being bound by the Python / launch rate.  Re-captured when the lr changes.
        # Multi-rank: the bucket all-reduces are captured too.  That needs the thread-local capture mode (NCCL's watchdog
        # thread polls events during the capture; the default global mode hung at 2 GPUs) and, at exit, the graph has to go
        # before the process group (release()).
        # batched_casts: under autocast every cuDNN convolution casts its fp32 weight to bf16 in forward and its bf16 weight
        # gradient back to fp32 in backward -- ~360 three-microsecond kernels per step (9 % of the captured step).  Same
        # arithmetic, two launches: all conv weights are cast at once into bf16 shadows (torch._foreach_copy_), the model runs
        # on the shadows (torch.func.functional_call), and the shadows' gradients are cast back at once.
        # the fused BN+ReLU path bumps num_batches_tracked itself (118 one-element kernels per step): one foreach launch instead
        self._nbt = []
        if buffered and self.device.type == 'cuda':
            for m in self.model.modules():
                if isinstance(m, torch.nn.BatchNorm2d) and m.num_batches_tracked is not None:
                    m._nbt_batched = True
                    self._nbt.append(m.num_batches_tracked)
        self._sh = None
        if batched_casts and self.autocast:
            self._setup_shadows()
        # Gradient exchange.  On CUDA: fresh gradients, packed (one multi-tensor copy per ~25 MB bucket) and all-reduced (NCCL, averaged)
        # AFTER backward.  Measured on 2 and 8 B200s under the CUDA graph: communication under backward is slower here --
        # AACONV_DP_OVERLAP=1 (one hook per bucket, GradientBuckets(overlap='bucket')) 2504 images/s vs 2777 at 2 GPUs, the
        # per-parameter hook variant (overlap=True: 360 small accumulate kernels per step) 7.03x vs 7.62x at 8 GPUs in the first
        # session: the ~0.5 ms all-reduce costs the concurrent convolutions more than it hides.
        mode = True if self.device.type != 'cuda' else ('bucket' if os.environ.get('AACONV_DP_OVERLAP', '0') == '1' else False)
        srcs = dict(zip(self._sh_params, self._sh)) if self._sh is not None else None
        # The bucket hooks create the AccumulateGrad nodes of their tensors at registration, and such a node keeps the stream it was
        # created under: registered under the default stream they would make it wait on the capturing stream during the graph capture
        # (cudaErrorStreamCaptureImplicit).  So with bucket hooks EVERY step -- eager, capture, replay -- runs on one side stream.
        self._stream = torch.cuda.Stream(self.device) if (self.world > 1 and mode == 'bucket') else None
        with torch.cuda.stream(self._stream) if self._stream is not None else contextlib.nullcontext():
            self.buckets = (GradientBuckets(self.model, bucket_mb=bucket_mb, overlap=mode, grad_sources=srcs if mode == 'bucket' else None)
                            if self.world > 1 else None)
        self._bucket_sources = self.buckets is not None and mode == 'bucket' and self._sh is not None
        self.cuda_graph = bool(cuda_graph and self.device.type == 'cuda')
        self.graph_after = graph_after
        self._calls = 0
        self._graph = None
        self._graph_lr = None
        self.graph_launches = 0
        self.model.train()

    def _setup_shadows(self):
        plan = conv_weight_plan(self.model)
        self._sh_names, self._sh_params = [n + '.weight' for n, _, _ in plan], [m.weight for _, m, _ in plan]
        # The weights the plan keeps channels-last are the fp32 MASTER weights themselves (values, state_dict and optimizer are
        # layout-agnostic): with a contiguous master and a channels-last shadow torch._foreach_copy_ fell back to one strided copy
        # kernel per tensor (1.1 ms per step in the profile).
        for _, m, cl in plan:
            if cl:
                m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
        self._sh = [torch.empty_like(p, dtype=torch.bfloat16).requires_grad_(True) for p in self._sh_params]   # preserve_format: strides of p
        self._sh_grads = [torch.empty_like(p) for p in self._sh_params]          # fp32, static: what the optimizer / buckets read

    def _step(self, x, target):
        if self.buckets is not None:
            self.buckets.reset()
        else:
            self.opt.zero_grad(set_to_none=True)
        if self._nbt:
            torch._foreach_add_(self._nbt, 1)
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=self.autocast):
            if self._sh is not None:
                with torch.no_grad():
                    torch._foreach_copy_(self._sh, self._sh_params)
                for t in self._sh:
                    t.grad = None
                out = torch.func.functional_call(self.model, dict(zip(self._sh_names, self._sh)), (x,))
            else:
                out = self.model(x)
        loss = self.loss_fn(out.float(), target)
        loss.backward()
        if self._sh is not None and not self._bucket_sources:      # (bucket hooks pack the shadows' gradients themselves)
            with torch.no_grad():
                torch._foreach_copy_(self._sh_grads, [t.grad for t in self._sh])
            for p, g in zip(self._sh_params, self._sh_grads):
                p.grad = g
        if self.buckets is not None:
            self.buckets.finish()
        self.opt.step()
        return loss.detach()

    def _capture(self, x, target):
        self._sx, self._st = x.clone(), target.clone()
        torch.cuda.synchronize(self.device)
        self._graph = torch.cuda.CUDAGraph()
        if self.buckets is None:
            self.opt.zero_grad(set_to_none=True)
        n0 = _lib.launch_count()
        mode = 'thread_local' if self.world > 1 else 'global'   # NCCL's watchdog thread polls events during the capture
        with torch.cuda.graph(self._graph, stream=self._stream, capture_error_mode=mode):
            self._sloss = self._step(self._sx, self._st)
        self.graph_launches = _lib.launch_count() - n0      # kernels of libaaconv_b200 inside one replay
        self._graph_lr = [g['lr'] for g in self.opt.param_groups]

    def release(self):
        """Drop the captured graph (call before dist.destroy_process_group())."""
        self._graph = None
        self._sloss = self._sx = self._st = None
        if self.device.type == 'cuda':
            torch.cuda.synchronize(self.device)

    def __call__(self, x, target):
        """-> loss (0-dim device tensor; no host sync, unlike loss.item() at chexpert.py:167)."""
        if self._stream is None:
            return self._call(x, target)
        cur = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(cur)
        with torch.cuda.stream(self._stream):
            loss = self._call(x, target)
        cur.wait_stream(self._stream)
        return loss

    def _call(self, x, target):
        self._calls += 1
        if not self.cuda_graph or self._calls <= self.graph_after:
            loss = self._step(x, target)
        else:
            if self._graph is None or self._graph_lr != [g['lr'] for g in self.opt.param_groups]:
                self._capture(x, target)
            self._sx.copy_(x, non_blocking=True)
            self._st.copy_(target, non_blocking=True)
            self._graph.replay()
            loss = self._sloss.clone()       # the static tensor is overwritten by the next replay
        self.sched.step()
        return loss
