"""The reference's input transform on the device (chexpert_b200/preprocess.py, csrc/prep.cu) against the host path it replaces:
torchvision's Resize(S) + CenterCrop(S) on a PIL 'L' image, then evaluate.normalise_u8 on the device -- bit for bit, at mixed
geometries in one launch and one by one, and through Predictor, evaluate_ensemble and TrainStep."""
import numpy as np
import pytest
import torch
import torchvision.transforms as T
from PIL import Image

from chexpert_b200 import _lib
from chexpert_b200.evaluate import normalise_u8, synthetic_radiographs_u8
from chexpert_b200.preprocess import MAX_SIDE, pack_radiographs, prepare, resized_geometry


def host_u8(img, size):
    """The reference's PIL path up to the uint8 crop: (S, S) uint8."""
    pil = T.CenterCrop(size)(T.Resize(size)(Image.fromarray(np.asarray(img), 'L')))
    return torch.from_numpy(np.array(pil))


def host_input(images, size):
    """What the host path feeds the model: normalise_u8 of the PIL crops, on the device."""
    return normalise_u8(torch.stack([host_u8(img, size) for img in images]).cuda())


# (h, w) per model side S: identity, upscales, downscales of full-resolution sizes, extreme aspect ratios, 1 x 1, odd / prime sides,
# round-half-even crop offsets (640 x 782 -> 320 x 391: 35.5 -> 36; 640 x 786 -> 320 x 393: 36.5 -> 36) and the largest side
GEOMETRIES = {
    320: [(320, 390), (390, 320), (320, 320), (200, 250), (1, 1), (40, 1500), (1500, 40), (2828, 2320), (2320, 2828),
          (3000, 4000), (4096, 3072), (640, 782), (640, 786), (782, 640), (331, 467), (997, 1009), (521, 389), (13, 7919),
          (7919, 13), (1, 977), (977, 1), (319, 321), (321, 319), (2, 3), (MAX_SIDE, MAX_SIDE), (MAX_SIDE, 613), (613, MAX_SIDE)]
    + [tuple(int(v) for v in hw) for hw in np.random.default_rng(7).integers(1, 3000, (21, 2))],
    512: [(320, 390), (390, 320), (512, 512), (2828, 2320), (1, 1), (40, 1500), (1021, 769), (4093, 3079)],
    227: [(227, 300), (300, 227), (1000, 1000), (2828, 2320), (41, 43)],
}


def content(h, w, kind, seed):
    if kind == 0:
        return np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)
    if kind == 1:
        return ((np.indices((h, w)).sum(0) % 2) * 255).astype(np.uint8)
    side = max(h, w)
    if side > 1024:      # smooth radiograph-like content, bilinearly enlarged past the generator's practical size
        small = synthetic_radiographs_u8(1, 512, seed=seed)[0].numpy()
        return np.array(Image.fromarray(small, 'L').resize((w, h), Image.BILINEAR))
    return synthetic_radiographs_u8(1, side, seed=seed)[0, :h, :w].numpy()


def cases(size):
    return [content(h, w, i % 3, i) for i, (h, w) in enumerate(GEOMETRIES[size])]


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize('size', [320, 512])
def test_geometry_is_torchvisions(size):
    """resized size == torchvision's Resize(S) on a PIL image; crop offsets == CenterCrop(S) of an image whose pixels hold their
    own index"""
    sizes = [(640, 782), (640, 786), (782, 640), (786, 640), (320, 390), (390, 320), (1, 1), (40, 1500), (2828, 2320), (7, 101),
             (size, size), (size + 1, size + 3), (997, 1009)]
    rad = pack_radiographs([np.zeros(s, np.uint8) for s in sizes], size)
    g = rad.geometry.tolist()
    for (h, w), row in zip(sizes, g):
        rw, rh = T.Resize(size)(Image.new('L', (w, h))).size
        idx = np.arange(rh * rw, dtype=np.int32).reshape(rh, rw)
        corner = int(np.asarray(T.CenterCrop(size)(Image.fromarray(idx, 'I')))[0, 0])
        assert row[1:7] == [h, w, rh, rw, corner // rw, corner % rw], ((h, w), row)
    assert [r[0] for r in g] == list(np.cumsum([0] + [h * w for h, w in sizes[:-1]]))
    assert rad.max_side == 2828 and len(rad) == len(sizes) and rad.pixels.numel() == sum(h * w for h, w in sizes)
    assert resized_geometry(640, 782, 320) == (320, 391, 0, 36) and resized_geometry(640, 786, 320) == (320, 393, 0, 36)


def test_pack_copies_the_pixels():
    imgs = [torch.randint(0, 256, (5, 7), dtype=torch.uint8), np.arange(12, dtype=np.uint8).reshape(3, 4)[:, ::-1],
            torch.randint(0, 256, (9, 4), dtype=torch.uint8).t()]
    rad = pack_radiographs(imgs, 16)
    for img, (off, h, w, *_) in zip(imgs, rad.geometry.tolist()):
        assert torch.equal(rad.pixels[off:off + h * w].view(h, w), torch.as_tensor(np.ascontiguousarray(img)))
    part = rad[1:3]
    assert len(part) == 2 and part.pixels is rad.pixels and part.geometry.tolist() == rad.geometry[1:3].tolist()


@pytest.mark.parametrize('images, size, message', [
    ([np.zeros((5, 5), np.float32)], 320, 'must be uint8'),
    ([torch.zeros(5, 5, dtype=torch.int16)], 320, 'must be uint8'),
    ([torch.zeros(5, 5, 3, dtype=torch.uint8)], 320, 'must be 2-D'),
    ([], 320, 'at least 1 image'),
    ([torch.zeros(0, 5, dtype=torch.uint8)], 320, 'at least 1 pixel'),
    ([np.zeros((5, 0), np.uint8)], 320, 'at least 1 pixel'),
    ([torch.zeros(MAX_SIDE + 1, 2, dtype=torch.uint8)], 320, f'MAX_SIDE = {MAX_SIDE}'),
    ([torch.zeros(2, MAX_SIDE + 1, dtype=torch.uint8)], 320, f'MAX_SIDE = {MAX_SIDE}'),
    ([torch.zeros(5, 5, dtype=torch.uint8)], 8, 'MIN_SIZE, MAX_SIZE'),
    ([torch.zeros(5, 5, dtype=torch.uint8)], 4096, 'MIN_SIZE, MAX_SIZE'),
    (torch.zeros(2, 5, 5, dtype=torch.uint8), 320, 'sequence of 2-D images'),
    (['not an image'], 320, 'torch.Tensor or numpy array'),
], ids=['float32', 'int16', '3d', 'empty', 'zero_h', 'zero_w', 'tall', 'wide', 'size_small', 'size_large', 'one_array', 'str'])
def test_pack_rejects(images, size, message):
    with pytest.raises((ValueError, TypeError), match=message.replace('[', r'\[').replace('(', r'\(')):
        pack_radiographs(images, size)


def test_prepare_needs_cuda():
    rad = pack_radiographs([torch.zeros(5, 5, dtype=torch.uint8)], 16)
    with pytest.raises(RuntimeError, match='CUDA only'):
        prepare(rad)


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize('size', [320, 512, 227])
def test_prepare_is_bit_identical_to_pil_and_normalise_u8(size):
    images = cases(size)
    want = host_input(images, size)
    rad = pack_radiographs(images, size).to('cuda')
    n0 = _lib.launch_count()
    got = prepare(rad)                                       # every geometry of this size in one launch
    assert _lib.launch_count() - n0 == 1
    assert got.shape == (len(images), 3, size, size) and got.is_contiguous()
    bad = [GEOMETRIES[size][i] for i in range(len(images)) if not torch.equal(got[i], want[i])]
    assert not bad, f'differs from the PIL path at {bad}'
    out = torch.full((1, 3, size, size), float('nan'), device='cuda')
    for i, img in enumerate(images):                         # B = 1, into a caller's tensor
        prepare(pack_radiographs([img], size).to('cuda'), out=out)
        assert torch.equal(out[0], want[i]), GEOMETRIES[size][i]


def raw_set(n, seed):
    """n raw radiographs of CheXpert-like mixed sizes: the small set's 320-px short side and larger downscales."""
    rng = np.random.default_rng(seed)
    shapes = [(320, 390), (390, 320), (700, 560), (1210, 1000), (320, 320), (413, 389)]
    return [content(*shapes[int(rng.integers(len(shapes)))], 2, seed * 100 + i) for i in range(n)]


def _state_dict(arch, seed):
    from chexpert_b200 import densenet
    torch.manual_seed(seed)
    return densenet.build_model(arch, 5, 320, 'bf16').state_dict()


@pytest.mark.gpu
@pytest.mark.parametrize('arch', ['aadensenet121', 'densenet121'])
def test_predictor_takes_raw_radiographs(arch):
    """Logits from a raw list == logits from the host-preprocessed uint8 tensor, eager and under the graph, with a ragged tail
    (21 = 16 + 5); a second batch set of other geometries replays the raw path's graph without a new capture; the uint8 path keeps
    its own graph.  Under the graph a call costs one prep launch per batch."""
    from chexpert_b200.evaluate import Predictor
    raw, other = raw_set(21, 1), raw_set(19, 2)
    u8, u8_other = torch.stack([host_u8(i, 320) for i in raw]), torch.stack([host_u8(i, 320) for i in other])
    sd = _state_dict(arch, 0)
    pe = Predictor(5, 320, precision='bf16', batch_size=16, cuda_graph=False, arch=arch)
    pe.load_state_dict(sd)
    assert torch.equal(pe(raw), pe(u8))
    pg = Predictor(5, 320, precision='bf16', batch_size=16, cuda_graph=True, arch=arch)
    pg.load_state_dict(sd)
    want_eager = pg(u8)                                      # two eager warm-up batches of the uint8 path
    want = pg(u8)                                            # its capture
    assert pg.captures == 1
    assert torch.equal(pg(raw), want_eager)                  # the raw path's two warm-up batches
    assert pg.captures == 1
    assert torch.equal(pg(raw), want) and pg.captures == 2   # its capture, at the first batch of this call
    n0 = _lib.launch_count()
    got_other = pg(other)
    assert _lib.launch_count() - n0 == 2                     # replays: only the two prep launches are enqueued from the host
    assert pg.captures == 2
    assert torch.equal(got_other, pg(u8_other)) and pg.captures == 2
    rad = pack_radiographs(raw, 320)                         # a packed host batch, uploaded whole and sliced per batch
    assert torch.equal(pg(rad), want) and torch.equal(pg(rad.to('cuda')), want) and pg.captures == 2


@pytest.mark.gpu
def test_evaluate_ensemble_takes_raw_radiographs():
    from chexpert_b200.evaluate import Predictor, evaluate_ensemble, synthetic_eval_targets
    raw = raw_set(20, 3)
    u8 = torch.stack([host_u8(i, 320) for i in raw])
    t = synthetic_eval_targets(20, seed=4)
    sds = [_state_dict('aadensenet121', s) for s in (0, 1)]
    p = Predictor(5, 320, precision='bf16', batch_size=8)
    want, got = evaluate_ensemble(p, sds, u8, t), evaluate_ensemble(p, sds, raw, t)
    for k in ('outputs', 'per_model', 'auroc', 'loss'):
        assert torch.equal(got[k], want[k]), k


@pytest.mark.gpu
def test_train_step_takes_radiographs(monkeypatch):
    """TrainStep(buffered, fused_prologue, bf16, cuda_graph after 2 eager steps): Radiographs give the losses and parameters of the
    host-preprocessed float x bit for bit over two eager steps, the capture and two replays; a replay costs one prep launch."""
    from chexpert_b200.train import TrainStep, synthetic_batch
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)      # no run-to-run differences from cuDNN's atomics
    kw = dict(size=320, precision='bf16', lr=1e-3, seed=0, buffered=True, fused_prologue=True, cuda_graph=True, graph_after=2)
    a, b = TrainStep('cuda', **kw), TrainStep('cuda', **kw)
    _, target = synthetic_batch(2, size=320, seed=5, device='cuda')
    batches = [raw_set(2, 10 + i) for i in range(5)]
    for i, images in enumerate(batches):
        rad = pack_radiographs(images, 320)
        n0 = _lib.launch_count()
        la = a(rad, target)
        if i == 4:
            assert _lib.launch_count() - n0 == 1
        lb = b(host_input(images, 320), target)
        assert torch.equal(la, lb), (i, float(la), float(lb))
    assert a._graph is not None
    for (n, p), q in zip(a.model.named_parameters(), b.model.parameters()):
        assert torch.equal(p, q), n
