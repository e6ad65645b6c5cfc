"""The reference's input transform on the device (chexpert.py:64-79, SURVEY.md section 2 row 8):

    Resize(S) -> CenterCrop(S) -> ToTensor -> Normalize(0.5330, 0.0349) -> grey to 3 channels

for decoded 8-bit grayscale radiographs of any size.  Only the bytes cross PCIe; one kernel launch per batch
(aaconv_radiograph_prep, csrc/prep.cu) writes the fp32 (B, 3, S, S) model input, bit-identical to torchvision's PIL path
(transforms.Resize(S) bilinear, transforms.CenterCrop(S) on a PIL 'L' image) followed by evaluate.normalise_u8 on the device.

    r = pack_radiographs(images, 320).to('cuda')     # host: validate, geometry, one pinned buffer; then an async upload
    x = prepare(r)                                   # device: (B, 3, 320, 320) float32
"""
import numpy as np
import torch

from . import _lib
from .aaconv import _ptr, _stream

MAX_SIDE = 8192                  # longest input side the kernel takes
MIN_SIZE, MAX_SIZE = 16, 2048    # model input sides S the kernel takes
MAX_BATCH = 65535                # images per launch (grid y)


def resized_geometry(h, w, size):
    """(resized h, resized w, crop top, crop left) of torchvision's Resize(size) then CenterCrop(size) on an (h, w) image: the
    short side becomes `size`, the long side int(size * long / short) in Python float arithmetic (_compute_resized_output_size);
    the crop offsets are int(round((resized - size) / 2.0)), round half to even (center_crop)."""
    short, long = (w, h) if w <= h else (h, w)
    new_long = int(size * long / short)
    rh, rw = (new_long, size) if w <= h else (size, new_long)
    return rh, rw, int(round((rh - size) / 2.0)), int(round((rw - size) / 2.0))


class Radiographs:
    """A packed batch of 8-bit grayscale images: `pixels` (total_bytes,) uint8, each image's rows back to back, and `geometry`
    (B, 8) int64 rows (byte offset, h, w, resized h, resized w, crop top, crop left, 0) for model input side `size`.
    `max_side` bounds every h and w.  Built by pack_radiographs; batches of it are views (same pixel buffer, a row range of the
    geometry table, whose offsets stay absolute)."""

    def __init__(self, pixels, geometry, size, max_side):
        self.pixels, self.geometry, self.size, self.max_side = pixels, geometry, int(size), int(max_side)

    def __len__(self):
        return self.geometry.shape[0]

    @property
    def device(self):
        return self.pixels.device

    def to(self, device):
        """Both buffers on `device`, copied with non_blocking=True (asynchronous from the pinned host buffers)."""
        device = torch.device(device)
        if self.pixels.device == device and self.geometry.device == device:
            return self
        return Radiographs(self.pixels.to(device, non_blocking=True), self.geometry.to(device, non_blocking=True), self.size,
                           self.max_side)

    def __getitem__(self, index):
        if not isinstance(index, slice) or index.step not in (None, 1):
            raise TypeError('Radiographs takes contiguous slices only')
        g = self.geometry[index]
        if g.shape[0] == 0:
            raise IndexError(f'empty slice {index} of {len(self)} radiographs')
        return Radiographs(self.pixels, g, self.size, self.max_side)


def _as_u8_image(img, i):
    if isinstance(img, np.ndarray):
        if img.dtype != np.uint8:
            raise ValueError(f'image {i}: dtype {img.dtype}, radiographs must be uint8 (8-bit grayscale)')
        img = torch.from_numpy(np.ascontiguousarray(img))
    elif not isinstance(img, torch.Tensor):
        raise TypeError(f'image {i}: expected a torch.Tensor or numpy array, got {type(img).__name__}')
    if img.dtype != torch.uint8:
        raise ValueError(f'image {i}: dtype {img.dtype}, radiographs must be uint8 (8-bit grayscale)')
    if img.ndim != 2:
        raise ValueError(f'image {i}: shape {tuple(img.shape)}, radiographs must be 2-D (H, W) grayscale')
    if img.device.type != 'cpu':
        raise ValueError(f'image {i}: on {img.device}, pack_radiographs takes host images')
    h, w = img.shape
    if h < 1 or w < 1:
        raise ValueError(f'image {i}: shape {(h, w)}, both sides must be at least 1 pixel')
    if h > MAX_SIDE or w > MAX_SIDE:
        raise ValueError(f'image {i}: shape {(h, w)}, sides are limited to MAX_SIDE = {MAX_SIDE} pixels')
    return img


def pack_radiographs(images, size):
    """Sequence of 2-D uint8 host images (torch tensors or numpy arrays, any sizes) -> Radiographs for model input side `size`:
    one flat uint8 buffer and the geometry table, both pinned when CUDA is available.  Everything is validated here, before
    any byte reaches the kernel."""
    if isinstance(size, bool) or not isinstance(size, int) or not MIN_SIZE <= size <= MAX_SIZE:
        raise ValueError(f'size {size!r}: the model input side must be an int in [MIN_SIZE, MAX_SIZE] = [{MIN_SIZE}, {MAX_SIZE}]')
    if isinstance(images, (torch.Tensor, np.ndarray)):
        raise TypeError('pack_radiographs takes a sequence of 2-D images (a list), not one array')
    images = [_as_u8_image(img, i) for i, img in enumerate(images)]
    if not images:
        raise ValueError('pack_radiographs: empty list, a batch needs at least 1 image')
    if len(images) > MAX_BATCH:
        raise ValueError(f'pack_radiographs: {len(images)} images, a batch is limited to MAX_BATCH = {MAX_BATCH}')
    rows, off = [], 0
    for img in images:
        h, w = img.shape
        rows.append((off, h, w, *resized_geometry(h, w, size), 0))
        off += h * w
    pin = torch.cuda.is_available()
    pixels = torch.empty(off, dtype=torch.uint8, pin_memory=pin)
    for (o, h, w, *_), img in zip(rows, images):
        pixels[o:o + h * w].view(h, w).copy_(torch.as_tensor(img))
    geometry = torch.tensor(rows, dtype=torch.int64)
    if pin:
        geometry = geometry.pin_memory()
    return Radiographs(pixels, geometry, size, max(max(r[1], r[2]) for r in rows))


def prepare(radiographs, out=None):
    """Radiographs on a CUDA device -> (B, 3, S, S) float32 model input there, in one launch on the current stream.  `out`: a
    contiguous float32 (B, 3, S, S) tensor on that device to write into (a static input of a CUDA graph, say)."""
    r = radiographs
    dev = r.pixels.device
    if dev.type != 'cuda' or r.geometry.device != dev:
        raise RuntimeError('prepare runs on CUDA only (move the batch with Radiographs.to(device)); there is no CPU fallback')
    B, S = len(r), r.size
    if out is None:
        out = torch.empty(B, 3, S, S, device=dev, dtype=torch.float32)
    elif out.dtype != torch.float32 or out.device != dev or tuple(out.shape) != (B, 3, S, S) or not out.is_contiguous():
        raise RuntimeError(f'out must be a contiguous float32 {(B, 3, S, S)} tensor on {dev}, got {out.dtype} '
                           f'{tuple(out.shape)} on {out.device}')
    lib = _lib.load()
    with torch.cuda.device(dev):
        _lib.check(lib.aaconv_radiograph_prep(_ptr(r.pixels), r.pixels.numel(), _ptr(r.geometry), B, r.max_side, S, _ptr(out),
                                              _stream()), 'aaconv_radiograph_prep')
    return out
