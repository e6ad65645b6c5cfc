"""Data-parallel training plumbing: one process per GPU, batch sharded across ranks, gradients averaged over the ranks after
backward as flat buckets, one all-reduce per bucket.

The reference is single-process / single-device (chexpert.py:38,453); this is the one new subsystem SURVEY.md
section 8(e) asks for.  The batch dimension is the only shard: every AAConv2d kernel runs unsharded on its rank.

Design (deliberately small, no torch DDP wrapper):
  * parameters are laid out, in REVERSE registration order (the order backward produces gradients), into flat
    fp32 buckets of ~``bucket_mb``;
  * autograd writes fresh gradients; ``finish()`` packs each bucket with one multi-tensor copy, all-reduces it as a mean
    over the global batch (the reference's ``.mean(0)``, chexpert.py:160) and points every ``p.grad`` at its slice of the
    bucket.  There is no per-parameter accumulate kernel (360 small launches per step for aadensenet121, ~1 ms under a CUDA
    graph); the price is an all-reduce that is not hidden under backward (~0.2 ms for 50 MB over NVLink 5 at 8 GPUs);
  * every rank issues the all-reduces in the same bucket order, whichever parameters received a gradient on it.
Works with the gloo backend on CPU, which is how tests/ covers world_size 2 without GPUs.
"""
import torch
import torch.distributed as dist


class GradientBuckets:
    """Averages the gradients of ``module``'s trainable parameters over the ranks of ``process_group``.

    One step is ``reset()``, one or more ``backward()`` calls, ``finish()``, then the optimizer step.  Gradients of several
    ``backward()`` calls in one step add up in ``.grad`` as usual, and ``finish()`` exchanges their sum once."""

    def __init__(self, module, bucket_mb=25.0, process_group=None, broadcast_from=0):
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.params = [p for p in module.parameters() if p.requires_grad]
        if not self.params:
            raise ValueError('module has no trainable parameters')
        if self.world > 1 and broadcast_from is not None:   # identical replicas before the first step
            for t in list(module.parameters()) + list(module.buffers()):
                dist.broadcast(t.data, broadcast_from, group=process_group)
        cap = max(1, int(bucket_mb * (1 << 20) / 4))
        self.buckets = []          # (flat tensor, [params])
        self._view = {}
        cur, cur_n = [], 0
        for p in reversed(self.params):
            if cur and cur_n + p.numel() > cap:
                self._seal(cur)
                cur, cur_n = [], 0
            cur.append(p)
            cur_n += p.numel()
        if cur:
            self._seal(cur)
        self.reset()

    def _seal(self, params):
        dev = params[0].device
        flat = torch.zeros(sum(p.numel() for p in params), dtype=torch.float32, device=dev)
        off = 0
        for p in params:
            if p.dtype != torch.float32 or p.device != dev:
                raise ValueError('GradientBuckets expects fp32 master parameters on one device')
            # the view has the parameter's own (dense) strides -- channels-last conv weights included -- so that packing its
            # gradient is part of one multi-tensor copy instead of a strided copy of its own
            seg = flat[off:off + p.numel()]
            self._view[p] = seg.view_as(p) if p.is_contiguous() else seg.as_strided(p.shape, p.stride())
            off += p.numel()
        self.buckets.append((flat, params))

    def reset(self):
        """Drop the gradients (replaces optimizer.zero_grad(set_to_none=True)) and arm the step."""
        for p in self.params:
            p.grad = None
        self._armed = True

    def finish(self):
        """Average the gradients over the ranks.  Call once after backward(), before optimizer.step()."""
        if not self._armed:
            raise RuntimeError('GradientBuckets: finish() called twice, or without reset() since the last finish() -- the '
                               'gradients are already averaged; call reset() at the start of every step')
        avg = dist.ReduceOp.AVG if (self.world > 1 and dist.get_backend(self.group) == 'nccl') else None
        for flat, params in self.buckets:
            views = [self._view[p] for p in params]
            have = [(v, p.grad) for v, p in zip(views, params) if p.grad is not None]
            for v, p in zip(views, params):
                if p.grad is None:
                    v.zero_()                 # parameter without a gradient on this rank contributes zeros
            if have:
                torch._foreach_copy_([v for v, _ in have], [g for _, g in have])
            if self.world > 1:
                if avg is not None:
                    dist.all_reduce(flat, op=avg, group=self.group)
                else:
                    dist.all_reduce(flat, group=self.group)
                    flat.div_(self.world)
            for v, p in zip(views, params):
                p.grad = v
        self._armed = False

    @property
    def nbytes(self):
        return sum(f.numel() * 4 for f, _ in self.buckets)
