"""Training-time augmentation on the GPU (row N4): the reference's loader chain (``__main__.py:153-176``: pad_resize ->
ColorJitter(saturation=0.2, brightness=0.1) -> RandomCrop -> random flips, the same draw for image and label,
``dataset.py:171-179``) as one fused gather kernel over a device-resident dataset (``in_memory=True`` in the reference).
``draw_params`` makes the random draws with the distributions of the torchvision transforms; ``augment_batch`` applies
them to a stack of equally sized sources, ``augment_ragged`` to a ``DeviceDataset`` of processed images of any size up to
the target -- including the odd size differences, where ``pad_resize`` ends with Pillow's bilinear resize
(csrc/augment.cu)."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .dataset import make_dataset, pil_loader

PARAM_DTYPE = np.dtype([('src', '<i4'), ('x0', '<i4'), ('y0', '<i4'), ('hflip', '<i4'), ('vflip', '<i4'), ('order', '<i4'),
                        ('brightness', '<f4'), ('saturation', '<f4')])


def draw_params(rng, batch, n_sources, crop, target_hw=(1024, 1024), saturation=0.2, brightness=0.1, sources=None):
    """rng: numpy Generator.  ColorJitter draws each factor uniformly in [max(0, 1 - v), 1 + v] and applies the two
    ops in random order; RandomCrop draws the offset uniformly; each flip has probability 0.5 (torchvision transforms)."""
    p = np.zeros(batch, dtype=PARAM_DTYPE)
    p['src'] = rng.integers(0, n_sources, batch) if sources is None else np.asarray(sources)
    p['x0'] = rng.integers(0, target_hw[1] - crop + 1, batch)
    p['y0'] = rng.integers(0, target_hw[0] - crop + 1, batch)
    p['hflip'] = rng.random(batch) < 0.5
    p['vflip'] = rng.random(batch) < 0.5
    p['order'] = rng.integers(0, 2, batch)
    p['brightness'] = rng.uniform(max(0.0, 1 - brightness), 1 + brightness, batch) if brightness > 0 else 0.0
    p['saturation'] = rng.uniform(max(0.0, 1 - saturation), 1 + saturation, batch) if saturation > 0 else 0.0
    return p


def augment_batch(images, duals, params, crop, target_hw=(1024, 1024)):
    """images u8 CUDA [M,Hs,Ws,3]; duals u8 CUDA [M,Hs,Ws] (0/127/255) or None; params: structured array (PARAM_DTYPE).
    Returns (u8 [B,crop,crop,3], u8 class map [B,crop,crop] or None) on the device -- what Trainer.step consumes."""
    lib = _lib.load()
    if not images.is_cuda or images.dtype != torch.uint8 or images.dim() != 4 or images.shape[3] != 3:
        raise RuntimeError('augment_batch: images must be a CUDA u8 tensor [M,Hs,Ws,3]')
    images = images.contiguous()
    M, Hs, Ws, _ = images.shape
    if duals is not None:
        if not duals.is_cuda or duals.dtype != torch.uint8 or tuple(duals.shape) != (M, Hs, Ws):
            raise RuntimeError('augment_batch: duals must be a CUDA u8 tensor [M,Hs,Ws]')
        duals = duals.contiguous()
    params = np.ascontiguousarray(params, dtype=PARAM_DTYPE)
    B = params.shape[0]
    if B == 0 or params['src'].min() < 0 or params['src'].max() >= M:
        raise RuntimeError('augment_batch: source index out of range')
    if (params['x0'].min() < 0 or params['y0'].min() < 0 or params['x0'].max() + crop > target_hw[1]
            or params['y0'].max() + crop > target_hw[0]):
        raise RuntimeError('augment_batch: crop window outside the padded image')
    with torch.cuda.device(images.device):
        pd = torch.from_numpy(params.view(np.uint8).reshape(B, -1).copy()).to(images.device)
        out = torch.empty((B, crop, crop, 3), dtype=torch.uint8, device=images.device)
        cls = torch.empty((B, crop, crop), dtype=torch.uint8, device=images.device) if duals is not None else None
        _lib.check(lib.nbc_augment_batch(C.c_void_p(images.data_ptr()), C.c_void_p(duals.data_ptr() if duals is not None else 0),
                                         M, Hs, Ws, target_hw[0], target_hw[1], crop, C.c_void_p(pd.data_ptr()), B,
                                         C.c_void_p(out.data_ptr()), C.c_void_p(cls.data_ptr() if cls is not None else 0),
                                         C.c_void_p(torch.cuda.current_stream(images.device).cuda_stream)), 'nbc_augment_batch')
    return out, cls


# ---- ragged sources: the full pad_resize ---------------------------------------------------------------------------
def pil_bilinear_table(n_in, n_out):
    """Pillow's BILINEAR coefficients for an ``n_in -> n_out`` axis (Resample.c precompute_coeffs +
    normalize_coeffs_8bpc), restated in float64 with the C code's operations in its order: row i = (first input index,
    three fixed-point weights with 22 fraction bits).  Only ``n_in = n_out + 1`` is used (pad_resize of an odd
    difference), which never needs more than three taps."""
    scale = float(n_in) / float(n_out)
    filterscale = max(scale, 1.0)
    support = 1.0 * filterscale
    ss = 1.0 / filterscale
    out = np.zeros((n_out, 4), dtype=np.int32)
    for xx in range(n_out):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), n_in) - xmin
        k = []
        for x in range(xmax):
            t = abs((x + xmin - center + 0.5) * ss)
            k.append(1.0 - t if t < 1.0 else 0.0)
        ww = 0.0
        for v in k:                                      # the C loop's left-to-right float64 sum
            ww += v
        k = [v / ww if ww != 0.0 else v for v in k]
        fixed = [int(-0.5 + v * (1 << 22)) if v < 0 else int(0.5 + v * (1 << 22)) for v in k]
        while len(fixed) > 3 and fixed[-1] == 0:
            fixed.pop()
        if len(fixed) > 3:
            raise ValueError('pil_bilinear_table: %d -> %d needs more than three taps' % (n_in, n_out))
        out[xx, 0] = xmin
        out[xx, 1:1 + len(fixed)] = fixed
    return out


def resize_tables(target_hw):
    """int32 [target_h + target_w, 4]: the (target + 1 -> target) table of the H axis, then of the W axis."""
    return np.concatenate([pil_bilinear_table(target_hw[0] + 1, target_hw[0]), pil_bilinear_table(target_hw[1] + 1, target_hw[1])])


def label_classes(duals):
    """Class map of dual label images as the reference's loader makes it: ToTensor (v / 255 in f32), * 2, round half to
    even (dataset.py:184-193)."""
    lut = np.rint(np.arange(256, dtype=np.float32) / np.float32(255) * np.float32(2)).astype(np.uint8)
    return lut[duals]


class DeviceDataset:
    """A labelled dataset resident on one GPU: processed images of any size in one canvas.

    images u8 [M,Hc,Wc,3], duals u8 [M,Hc,Wc] (what the augmentation reads), classes u8 [M,Hc,Wc] (the dual's class map,
    what validation compares against), dims int32 [M,2] (height, width) on the device; ``sizes`` is the same on the host,
    ``label_pixels`` the number of pixels of each item whose class is not 0 (for ``utils.get_splits``), ``wood_types`` and
    ``fnames`` follow the dataset order.  Rows and columns outside an item's size are zero and never read."""

    def __init__(self, images, duals, wood_types, device='cuda:0', fnames=None):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('DeviceDataset: a CUDA device is required (no CPU path)')
        M = len(images)
        if M == 0 or len(duals) != M or len(wood_types) != M:
            raise RuntimeError('DeviceDataset: one dual image and one wood type per image, at least one image')
        self.sizes = np.zeros((M, 2), dtype=np.int32)
        for m, (img, dual) in enumerate(zip(images, duals)):
            if img.ndim != 3 or img.shape[2] != 3 or img.dtype != np.uint8 or dual is None or dual.shape != img.shape[:2]:
                raise RuntimeError('DeviceDataset: item %d needs a u8 [H,W,3] image and a u8 [H,W] dual of the same size' % m)
            self.sizes[m] = img.shape[:2]
        Hc, Wc = (int(v) for v in self.sizes.max(0))
        self.wood_types = list(wood_types)
        self.fnames = list(fnames) if fnames is not None else ['%d' % m for m in range(M)]
        self.label_pixels = np.zeros(M, dtype=np.int64)
        with torch.cuda.device(self.device):
            self.images = torch.zeros((M, Hc, Wc, 3), dtype=torch.uint8, device=self.device)
            self.duals = torch.zeros((M, Hc, Wc), dtype=torch.uint8, device=self.device)
            self.classes = torch.zeros((M, Hc, Wc), dtype=torch.uint8, device=self.device)
            for m, (img, dual) in enumerate(zip(images, duals)):
                h, w = self.sizes[m]
                cls = label_classes(dual)
                self.label_pixels[m] = int(np.count_nonzero(cls))
                self.images[m, :h, :w] = torch.from_numpy(np.array(img, dtype=np.uint8)).to(self.device)
                self.duals[m, :h, :w] = torch.from_numpy(np.array(dual, dtype=np.uint8)).to(self.device)
                self.classes[m, :h, :w] = torch.from_numpy(cls).to(self.device)
            self.dims = torch.from_numpy(self.sizes.copy()).to(self.device)
        self._tables = {}

    def __len__(self):
        return len(self.wood_types)

    def split_items(self):
        """What ``utils.get_splits(dataset, label_pixels=ds.label_pixels)`` iterates: (_, _, fname, wood_type)."""
        return [(None, None, f, w) for f, w in zip(self.fnames, self.wood_types)]

    def tables(self, target_hw):
        key = tuple(int(v) for v in target_hw)
        if key not in self._tables:
            with torch.cuda.device(self.device):
                self._tables[key] = torch.from_numpy(resize_tables(key)).to(self.device)
        return self._tables[key]


def load_dataset(root, device='cuda:0', items=None):
    """``samples/<wood>/*`` and ``duals/<wood>/*`` of a labelled folder in ``dataset.make_dataset`` order, decoded on the
    host (RGB and L) and copied once to ``device``.  Every sample needs its dual image.  ``items`` (optional): indices
    into that order; only those items are loaded, in the order given."""
    entries = make_dataset(root)
    items = entries if items is None else [entries[int(i)] for i in items]
    if not items:
        raise RuntimeError('load_dataset: no images under %s/samples' % root)
    missing = [f for _, t, f, _ in items if not t]
    if missing:
        raise RuntimeError('load_dataset: %d samples have no dual image under %s/duals (first: %s)' % (len(missing), root, missing[0]))
    images = [pil_loader(p) for p, _, _, _ in items]
    duals = [pil_loader(t, grayscale=True) for _, t, _, _ in items]
    return DeviceDataset(images, duals, [w for _, _, _, w in items], device, fnames=[f for _, _, f, _ in items])


def augment_ragged(ds, params, crop, target_hw=(1024, 1024)):
    """``augment_batch`` over a ``DeviceDataset``: params index its items, every item is pad_resize'd to ``target_hw``
    (reflect padding, plus Pillow's bilinear resize on an axis with an odd difference).  Returns (u8 [B,crop,crop,3],
    u8 class map [B,crop,crop]) on the device."""
    lib = _lib.load()
    params = np.ascontiguousarray(params, dtype=PARAM_DTYPE)
    B = params.shape[0]
    M, Hc, Wc, _ = ds.images.shape
    if B == 0 or params['src'].min() < 0 or params['src'].max() >= M:
        raise RuntimeError('augment_ragged: source index out of range')
    if (params['x0'].min() < 0 or params['y0'].min() < 0 or params['x0'].max() + crop > target_hw[1]
            or params['y0'].max() + crop > target_hw[0]):
        raise RuntimeError('augment_ragged: crop window outside the padded image')
    dev = ds.device
    with torch.cuda.device(dev):
        tables = ds.tables(target_hw)
        pd = torch.from_numpy(params.view(np.uint8).reshape(B, -1).copy()).to(dev)
        out = torch.empty((B, crop, crop, 3), dtype=torch.uint8, device=dev)
        cls = torch.empty((B, crop, crop), dtype=torch.uint8, device=dev)
        _lib.check(lib.nbc_augment_ragged(C.c_void_p(ds.images.data_ptr()), C.c_void_p(ds.duals.data_ptr()), M, Hc, Wc,
                                          C.c_void_p(ds.dims.data_ptr()), int(target_hw[0]), int(target_hw[1]),
                                          C.c_void_p(tables.data_ptr()), crop, C.c_void_p(pd.data_ptr()), B,
                                          C.c_void_p(out.data_ptr()), C.c_void_p(cls.data_ptr()),
                                          C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), 'nbc_augment_ragged')
    return out, cls
