"""Evaluation side of the hot path (SURVEY.md section 8d config 5, row f4): batched inference, the 10-checkpoint
ensemble (mean of raw logits, chexpert.py:217-236), per-class AUROC (chexpert.py:130-135) and the attention maps the
visualise path reads (chexpert.py:365,383-387).

    reference                                        here
    chexpert.py:196-214  evaluate_single_model   ->  predict_logits
    chexpert.py:217-236  evaluate_ensemble       ->  evaluate_ensemble  (mean + AUROC + element losses run on the device
                                                     through the C ABI: aaconv_ensemble_mean / aaconv_auroc / BCE kernel)
    chexpert.py:130-146  compute_metrics         ->  auroc_per_class
    chexpert.py:363-397  vis_attn (data part)    ->  attention_maps
    chexpert.py:260-361  grad_cam (data part)    ->  Predictor.grad_cam  (closed form at norm5, aaconv_grad_cam; see gradcam.py)

No sklearn, no host round trip per batch; plotting is out of scope (DESIGN.md section 8).
"""
import ctypes

import torch
import torch.nn.functional as F

from . import _lib
from .aaconv import AAConv2d, _ptr, _stream
from .densenet import build_model, conv_weight_plan
from .loss import BCEWithLogitsLoss
from .preprocess import Radiographs, pack_radiographs, prepare

PIXEL_MEAN, PIXEL_STD = 0.5330, 0.0349        # chexpert.py:70-72


def synthetic_radiographs_u8(n, size=320, seed=3):
    """Deterministic radiograph-shaped 8-bit images (n, size, size): a smooth per-image background, two dark 'lung'
    lobes whose position / extent / depth vary per image, a bright mediastinum band and sensor noise.  Unlike i.i.d.
    noise, images differ globally, so a network's logits spread across the set and AUROC is a meaningful check.
    Quantised to uint8 like the JPEGs the reference loads (dataset.py:101), which also absorbs last-ulp differences
    between hosts."""
    g = torch.Generator().manual_seed(seed)
    coarse = torch.rand(n, 1, 5, 5, generator=g)
    base = F.interpolate(coarse, size=(size, size), mode='bilinear', align_corners=True)[:, 0]
    par = torch.rand(n, 10, generator=g)
    noise = torch.randn(n, size, size, generator=g)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, size), torch.linspace(-1, 1, size), indexing='ij')
    yy, xx = yy[None], xx[None]

    def p(i, lo, hi):
        return (lo + (hi - lo) * par[:, i])[:, None, None]
    lobe = lambda cx, cy, sx, sy: torch.exp(-(((xx - cx) / sx) ** 2 + ((yy - cy) / sy) ** 2))   # noqa: E731
    lungs = lobe(-p(0, 0.3, 0.5), p(1, -0.2, 0.1), p(2, 0.2, 0.35), p(3, 0.4, 0.7)) \
        + lobe(p(4, 0.3, 0.5), p(5, -0.2, 0.1), p(6, 0.2, 0.35), p(3, 0.4, 0.7))
    spine = torch.exp(-(xx / 0.08) ** 2)
    img = p(7, 0.35, 0.6) + 0.25 * (base - 0.5) - p(8, 0.15, 0.4) * lungs + p(9, 0.05, 0.2) * spine + 0.02 * noise
    return (img.clamp(0, 1) * 255).round().to(torch.uint8)


def normalise_u8(img_u8):
    """uint8 (n, H, W) -> float (n, 3, H, W): /255, Normalize(mean, std), grey -> 3 channels (chexpert.py:68-72)."""
    x = (img_u8.float() / 255.0 - PIXEL_MEAN) / PIXEL_STD
    return x[:, None].expand(-1, 3, -1, -1).contiguous()


def synthetic_eval_targets(n, seed=4, p=0.3):
    """(n, 5) Bernoulli(p) targets, re-drawn until every class has both values (else AUROC is undefined)."""
    g = torch.Generator().manual_seed(seed)
    while True:
        t = (torch.rand(n, 5, generator=g) < p).float()
        if bool(((t.sum(0) > 0) & (t.sum(0) < n)).all()):
            return t


@torch.no_grad()
def predict_logits(model, images_u8, batch_size=16, device='cuda'):
    """Raw logits (N, 5) of `model` (eval mode) over uint8 images, batch by batch (chexpert.py:196-214); the last batch
    may be ragged (234 = 14 x 16 + 10)."""
    model.eval()
    outs = []
    for i in range(0, images_u8.shape[0], batch_size):
        x = normalise_u8(images_u8[i:i + batch_size].to(device, non_blocking=True))
        outs.append(model(x).float())
    return torch.cat(outs, 0)


def ensemble_mean(stacked_logits):
    """(n_models, N, C) device tensor -> (N, C) mean over checkpoints (chexpert.py:233)."""
    if not stacked_logits.is_cuda:
        raise RuntimeError('chexpert_b200.evaluate runs on CUDA only; there is no CPU fallback')
    lib = _lib.load()
    z = stacked_logits.detach().float().contiguous()
    M, N, C = z.shape
    with torch.cuda.device(z.device):
        out = torch.empty(N, C, device=z.device, dtype=torch.float32)
        _lib.check(lib.aaconv_ensemble_mean(_ptr(z), M, N, C, _ptr(out), _stream()), 'aaconv_ensemble_mean')
    return out


def auroc_per_class(logits, targets):
    """(N, C) logits, (N, C) {0,1} targets on the device -> (C,) AUROC (chexpert.py:130-135), NaN where undefined."""
    if not logits.is_cuda:
        raise RuntimeError('chexpert_b200.evaluate runs on CUDA only; there is no CPU fallback')
    lib = _lib.load()
    z = logits.detach().float().contiguous()
    t = targets.detach().to(device=z.device, dtype=torch.float32).contiguous()
    N, C = z.shape
    if tuple(t.shape) != (N, C):
        raise RuntimeError(f'targets {tuple(t.shape)} do not match logits {(N, C)}')
    with torch.cuda.device(z.device):
        ws = torch.empty(lib.aaconv_auroc_workspace_bytes(C), device=z.device, dtype=torch.uint8)
        out = torch.empty(C, device=z.device, dtype=torch.float32)
        _lib.check(lib.aaconv_auroc(_ptr(z), _ptr(t), N, C, _ptr(out), _ptr(ws), _stream()), 'aaconv_auroc')
    return out


class Predictor:
    """Inference counterpart of train.TrainStep: uint8 images (N, H, W), on the host or the device -> (N, num_classes) float32 logits
    on the device, with the arithmetic of predict_logits (normalise_u8, then the model in eval mode under no_grad).

    The model is aadensenet121(feature_buffer=True, fused_prologue=True, fused_eval=True): the dense blocks write into one feature
    buffer, the Transitions' InstanceNorm + ReLU run inside the AAConv2d kernels, and every BatchNorm + ReLU runs through the
    eval-mode kernels with the dense layers' convolutions channels-last.  Only uint8 images cross PCIe.

    ``autocast=True`` (opt-in; None or False: off) runs the torch/cuDNN layers under bf16 autocast.  The stem and dense-block
    convolution weights are then kept in bf16 inside this model (the dense blocks' k x k weights channels-last), so no per-call cast
    kernels run; load_state_dict converts the fp32 checkpoint values as it copies them.  AAConv2d and BatchNorm parameters stay fp32
    (the kernels read fp32).  Measured on a B200 over the 10 seed-initialised checkpoints of tests/golden/eval_ensemble.npz, autocast
    keeps the logits within rtol 2e-2 / atol 1e-2 of the fp32 reference (max error 0.012) but misses the bf16 mode's AUROC gate: up to
    3.6e-3 per class on the ensemble, against 2e-3.  So it is not the default, even for precision='bf16': without it the dense blocks
    stay fp32, as in predict_logits.

    ``cuda_graph``: after WARMUP eager batches (cuDNN picks its algorithms) one graph of the whole step at ``batch_size`` is
    captured and replayed.  A ragged last batch is padded to ``batch_size`` (samples are independent in eval mode) and sliced.
    load_state_dict writes parameters and buffers in place, so one capture serves every checkpoint of an ensemble;
    ``captures`` counts the captures made.  Raw radiographs (any sizes, see __call__) have a graph of their own, captured the same
    way from a static prepared (batch_size, 3, S, S) input onward; the prep launch runs before each replay, so batches of any
    geometries replay it.

    ``grad_cam(images)`` returns the same logits together with Grad-CAM maps of every class at the model's input size
    (DenseNet.forward_grad_cam); each input form has a graph of its own for it, captured the same way.

    ``arch='densenet121'``: the reference's baseline, torchvision's densenet121, as densenet121(feature_buffer=True,
    fused_transition=True, fused_eval=True) -- its Transitions' BatchNorm + ReLU + pool run through the eval-mode pooled kernel."""

    WARMUP = 2

    def __init__(self, num_classes=5, size=320, precision='bf16', batch_size=16, device='cuda', autocast=False, cuda_graph=True,
                 arch='aadensenet121'):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('chexpert_b200.evaluate.Predictor runs on CUDA only; there is no CPU fallback')
        self.num_classes, self.size, self.batch_size = num_classes, size, int(batch_size)
        self.autocast = bool(autocast)
        model = build_model(arch, num_classes, size, precision, feature_buffer=True, fused=True, fused_eval=True)
        model.requires_grad_(False)
        for _, m, cl in conv_weight_plan(model):
            m.weight.data = m.weight.data.to(torch.bfloat16 if self.autocast else torch.float32,
                                             memory_format=torch.channels_last if cl else torch.contiguous_format)
        self.model = model.to(self.device).eval()
        self.cuda_graph = bool(cuda_graph)
        self._warm = {'u8': 0, 'raw': 0, 'u8_cam': 0, 'raw_cam': 0}
        self._graphs = {}                   # input path -> (graph, static logits)
        self._sx = self._rx = None          # static inputs: uint8 (batch_size, S, S); prepared float (batch_size, 3, S, S)
        self.captures = 0

    def load_state_dict(self, state_dict):
        """Strict, in place (a reference checkpoint loads unchanged); a captured graph stays valid."""
        with torch.no_grad():
            self.model.load_state_dict(state_dict, strict=True)

    def _forward(self, u8, cam=False):
        return self._model_forward(normalise_u8(u8), cam)

    def _model_forward(self, x, cam=False):
        """-> logits, or (logits, Grad-CAM maps at the input size) when `cam`."""
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=self.autocast, cache_enabled=False):
            if not cam:
                return self.model(x).float()
            logits, maps = self.model.forward_grad_cam(x, self.size)
            return logits.float(), maps

    def _run(self, path, forward, sx, n):
        """forward(sx), each output sliced to [:n]: eager for the first WARMUP batches of this input path, then through the path's
        graph, captured once."""
        def head(y):
            return tuple(t[:n] for t in y) if isinstance(y, tuple) else y[:n]
        if path not in self._graphs:
            if self._warm[path] < self.WARMUP:
                self._warm[path] += 1
                return head(forward(sx))
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                sy = forward(sx)
            self._graphs[path] = (graph, sy)
            self.captures += 1
        graph, sy = self._graphs[path]
        graph.replay()
        return head(sy)

    def _batch(self, chunk, cam=False):
        n = chunk.shape[0]
        if not self.cuda_graph:
            return self._forward(chunk.to(self.device, non_blocking=True), cam)
        if self._sx is None:
            self._sx = torch.zeros(self.batch_size, *chunk.shape[1:], dtype=torch.uint8, device=self.device)
        self._sx[:n].copy_(chunk, non_blocking=True)       # rows [n, batch_size) keep earlier images: padding, sliced off below
        return self._run('u8_cam' if cam else 'u8', lambda sx: self._forward(sx, cam), self._sx, n)

    def _raw_batch(self, rad, cam=False):
        """Radiographs on the device -> logits: one prep launch, then the model from the prepared tensor onward."""
        n = len(rad)
        if not self.cuda_graph:
            return self._model_forward(prepare(rad), cam)
        if self._rx is None:
            self._rx = torch.zeros(self.batch_size, 3, self.size, self.size, dtype=torch.float32, device=self.device)
        prepare(rad, out=self._rx[:n])                      # rows [n, batch_size): padding, as in _batch
        return self._run('raw_cam' if cam else 'raw', lambda rx: self._model_forward(rx, cam), self._rx, n)

    def _predict(self, images, cam):
        raw = isinstance(images, (Radiographs, list, tuple))
        if not raw and (images.dtype != torch.uint8 or images.dim() != 3):
            raise RuntimeError(f'Predictor takes uint8 (N, H, W) images, got {images.dtype} {tuple(images.shape)}')
        if isinstance(images, Radiographs) and images.size != self.size:
            raise RuntimeError(f'Radiographs packed for size {images.size}, this Predictor takes {self.size}')
        with torch.cuda.device(self.device):
            if isinstance(images, Radiographs):
                images = images.to(self.device)
            N = len(images)
            out = torch.empty(N, self.num_classes, device=self.device, dtype=torch.float32)
            maps = torch.empty(N, self.num_classes, self.size, self.size, device=self.device, dtype=torch.float32) if cam else None
            for i in range(0, N, self.batch_size):
                chunk = images[i:i + self.batch_size]
                if isinstance(chunk, Radiographs):
                    y = self._raw_batch(chunk, cam)
                elif raw:
                    y = self._raw_batch(pack_radiographs(chunk, self.size).to(self.device), cam)
                else:
                    y = self._batch(chunk, cam)
                if cam:
                    y, m = y
                    maps[i:i + m.shape[0]].copy_(m)
                out[i:i + y.shape[0]].copy_(y)
            return out, maps

    @torch.no_grad()
    def __call__(self, images):
        """-> (N, num_classes) float32 logits on the device, batch by batch, from either
        - uint8 (N, S, S) images already at the model's size, on the host or the device, normalised by normalise_u8; or
        - raw radiographs of any sizes: a list of 2-D uint8 host images (packed and uploaded batch by batch), or a
          preprocess.Radiographs of side S (uploaded whole if on the host).  preprocess.prepare runs the reference's
          Resize(S) + CenterCrop(S) + normalisation on the device, one launch per batch; its CUDA graph starts after it."""
        return self._predict(images, cam=False)[0]

    @torch.no_grad()
    def grad_cam(self, images):
        """-> (logits (N, num_classes), maps (N, num_classes, S, S)), both float32 on the device, from the inputs __call__ takes.
        The logits are __call__'s, bit for bit; maps[:, c] is Grad-CAM of class c at model.features' output (the layer the reference
        hooks, chexpert.py:260-361), upsampled bilinearly to the input size S (DenseNet.forward_grad_cam, gradcam.py).  Each input
        form has a graph of its own for this step."""
        return self._predict(images, cam=True)


@torch.no_grad()
def evaluate_ensemble(model, state_dicts, images_u8, targets, batch_size=16, device='cuda'):
    """The reference's ensemble evaluation (chexpert.py:217-236): every checkpoint's state_dict is loaded strictly into
    `model`, its logits and element losses over the whole set are kept, the ensemble output / loss are their means over the
    checkpoints (chexpert.py:233-234; note mean-of-losses, not loss-of-mean); metrics as compute_metrics (chexpert.py:130-146)
    minus the plotting inputs.  -> dict(outputs, per_model, auroc, loss).
    `model` may be a Predictor; it then runs on its own device with its own batch size (`batch_size` / `device` are not used),
    and `images_u8` may also be raw radiographs (see Predictor.__call__): a list is packed and uploaded once for all checkpoints."""
    if isinstance(model, Predictor):
        device = model.device
        if isinstance(images_u8, (list, tuple)):
            images_u8 = pack_radiographs(images_u8, model.size).to(device)
    t = targets.to(device)
    loss_fn = BCEWithLogitsLoss('none').to(device)
    per_model, losses = [], []
    for sd in state_dicts:
        if isinstance(model, Predictor):
            model.load_state_dict(sd)
            per_model.append(model(images_u8))
            losses.append(loss_fn(per_model[-1], t))
            continue
        model.load_state_dict(sd, strict=True)
        per_model.append(predict_logits(model, images_u8, batch_size, device))
        losses.append(loss_fn(per_model[-1], t))       # element losses of THIS checkpoint (chexpert.py:205,229-231)
    stacked = torch.stack(per_model, 0)
    outputs = ensemble_mean(stacked)                    # chexpert.py:233
    el = ensemble_mean(torch.stack(losses, 0))          # chexpert.py:234: mean over checkpoints of the element losses
    return {'outputs': outputs, 'per_model': stacked, 'auroc': auroc_per_class(outputs, t), 'loss': el.mean(0)}


@torch.no_grad()
def attention_maps(model, x):
    """Softmax maps of every AAConv2d for a batch, shaped like the visualise path reshapes them
    (chexpert.py:383-387): list of (B, nh, H, W, H, W)."""
    layers = [m for m in model.modules() if isinstance(m, AAConv2d)]
    old = [m.store_weights for m in layers]
    for m in layers:
        m.store_weights = True
    try:
        model(x)
        maps = []
        for m in layers:
            B, nh, L, _ = m.weights.shape
            H = m.key_rel_h.shape[1] // 2 + 1 if m.relative else int(round(L ** 0.5))
            W = L // H
            maps.append(m.weights.reshape(B, nh, H, W, H, W))
            m.weights = None
    finally:
        for m, o in zip(layers, old):
            m.store_weights = o
    return maps
