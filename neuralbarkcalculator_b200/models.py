"""Host-side mirror of the hot-path pieces of the reference's ``models.py``.

Same public names and arguments as the reference -- ``fcn_resnet50``, ``SimpleSegmentationModel``, ``FCNHead``,
``trim_black``, ``Preprocessor``, ``NeuralBarkCalculator`` -- and the same 326-key torchvision ``state_dict`` layout,
so a checkpoint trained with the reference loads with ``strict=True``.  The modules only *hold* the parameters:
``forward`` hands them to the native plan in ``libnbc.so`` (hand-written sm_100a kernels); nothing here computes with
torch ops and nothing runs on the CPU."""
import csv
import os
import warnings
from concurrent.futures import ThreadPoolExecutor
from os.path import join

import numpy as np
import torch
import torch.nn as nn
from PIL import Image
from torchvision.models import resnet
from torchvision.models._utils import IntermediateLayerGetter

from . import ops
from .dataset import RegressionDatasetFolder, make_dataset, pil_loader, read_bmp_pixels


# 16-bit storage format of activations / packed weights of the predict path.  fp16: same tcgen05 rate as bf16, 3 more
# mantissa bits -- the format that meets the parity bar against the reference's f32 forward (argmax agreement >= 99.9 %,
# percentages within 0.1 pp; profiles/r02_parity.md); stores saturate at +-65504 and a plan whose BN-folded weights do not
# fit the fp16 range is refused (use 'bf16', which has the f32 exponent range and 8x the rounding error).
DEFAULT_PRECISION = 'fp16'


class FCNHead(nn.Sequential):
    """Parameter container with the layout of models.py:113-124 (conv3x3, BN, ReLU, Dropout, conv1x1+bias)."""

    def __init__(self, in_channels, channels, dropout=0.1):
        inter_channels = in_channels // 4
        super().__init__(nn.Conv2d(in_channels, inter_channels, 3, padding=1, bias=False),
                         nn.BatchNorm2d(inter_channels), nn.ReLU(), nn.Dropout(dropout),
                         nn.Conv2d(inter_channels, channels, 1))


class SimpleSegmentationModel(nn.Module):
    """models.py:27-43.  ``forward(x f32 [N,3,H,W] normalised) -> f32 logits [N,3,H,W]`` (a Tensor, not a dict)."""

    def __init__(self, backbone, classifier, mean=None, std=None):
        super().__init__()
        self.backbone = backbone
        self.classifier = classifier
        self._plan = None
        self._plan_key = None
        self._mean = list(mean) if mean is not None else [0.0, 0.0, 0.0]
        self._std = list(std) if std is not None else [1.0, 1.0, 1.0]
        self._precision = DEFAULT_PRECISION

    # -- native plan management ------------------------------------------------------------------------------
    # The plan holds BN-folded 16-bit copies of the weights, so it must be rebuilt when they change.  Everything that
    # replaces or moves parameters through the nn.Module API invalidates it (load_state_dict, .to / .cuda / .half / .float
    # via _apply); the per-call check is O(1) -- two sentinel tensors' (data_ptr, version).  In-place edits that bypass
    # the version counter (``p.data.copy_()``) need an explicit ``invalidate_plan()``.
    def invalidate_plan(self):
        self._plan = None
        self._plan_key = None

    def load_state_dict(self, *args, **kwargs):
        self.invalidate_plan()
        return super().load_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self.invalidate_plan()
        return super()._apply(fn, *args, **kwargs)

    def _state_key(self):
        first, last = self.backbone.conv1.weight, self.classifier[4].bias
        return (first.data_ptr(), first._version, last.data_ptr(), last._version)

    def native_plan(self):
        """Build (or reuse) the nbc_plan holding the BN-folded 16-bit weights for the current parameters."""
        key = self._state_key()
        if self._plan is None or key != self._plan_key:
            sd = self.state_dict(keep_vars=True)
            tensors = list(sd.values())
            if len(tensors) != 326:
                raise RuntimeError('unexpected state_dict layout: %d tensors' % len(tensors))
            dev = tensors[0].device
            if dev.type != 'cuda':
                raise RuntimeError('model is on %s: move it to a CUDA device (no CPU path)' % dev)
            self._plan = ops.Plan(tensors, self._mean, self._std, dev, self._precision)
            self._plan_key = key
        return self._plan

    def set_normalisation(self, mean, std):
        """mean/std used when the plan is fed u8 images (``forward_u8``); models.py:208-209, 233-237."""
        self._mean, self._std = list(mean), list(std)
        self._plan = None

    def set_precision(self, precision):
        """16-bit storage format of activations / packed weights on the tensor cores: 'fp16' (default, see
        DEFAULT_PRECISION) or 'bf16' (same speed, 8x the rounding error, f32 exponent range)."""
        if precision not in ('bf16', 'fp16'):
            raise ValueError("precision must be 'bf16' or 'fp16'")
        if precision != self._precision:
            self._precision = precision
            self._plan = None

    def _check_eval(self):
        if self.training:
            raise NotImplementedError(
                'the module forward is the inference path; call .eval().  Training (train-mode BatchNorm, dropout, backward, '
                'Adam, NCCL all-reduce) runs natively through neuralbarkcalculator_b200.train.Trainer -- there is '
                'deliberately no torch-autograd fallback.')

    def forward(self, x):
        self._check_eval()
        low = self.native_plan().forward(x.float())
        return ops.upsample_bicubic(low, tuple(x.shape[-2:]))

    # -- fused entry points used by NeuralBarkCalculator ------------------------------------------------------------
    def lowres_logits_u8(self, images_u8):
        """u8 NHWC [N,H,W,3] -> f32 [N,3,h,w]; ToTensor + Normalize happen in the stem kernel."""
        self._check_eval()
        return self.native_plan().forward(images_u8)

    def predict_mask_u8(self, images_u8):
        """u8 NHWC images -> u8 class mask [N,H,W] = argmax(bicubic(logits)) without materialising the logits."""
        low = self.lowres_logits_u8(images_u8)
        return ops.upsample_argmax(low, (images_u8.shape[1], images_u8.shape[2]))


_DUAL_LUT = np.array([0, 127, 255] + [0] * 253, dtype=np.uint8)


def fcn_resnet50(pretrained=True, dropout=0.1):
    """models.py:127-139.  ``pretrained=True`` needs torchvision's ImageNet weights (a download)."""
    weights = None
    if pretrained:
        weights = resnet.ResNet50_Weights.IMAGENET1K_V1
    backbone = resnet.resnet50(weights=weights, replace_stride_with_dilation=[False, True, True])
    backbone = IntermediateLayerGetter(backbone, return_layers={'layer4': 'out'})
    return SimpleSegmentationModel(backbone, FCNHead(2048, 3, dropout))


def trim_black(image):
    """models.py:157-166 on a CUDA u8 [H,W,3] tensor; returns the kept rows (a view-sized copy)."""
    out, fl = ops.trim_u8(image)
    first, last = fl.tolist()
    return out[:(last - first) * image.shape[1] * 3].view(last - first, image.shape[1], 3)


class Preprocessor():
    """models.py:169-203: raw scans -> ``processed/samples/<wood>/<name>.png`` (4x cubic resize + dark-band trim)."""

    def __init__(self, target_size=1024, device='cuda:0', io_threads=8):
        self.target_size = target_size
        self.device = torch.device(device)
        self.io_threads = io_threads

    def _load_raw(self, path):
        bmp = read_bmp_pixels(path) if path.lower().endswith('.bmp') else None
        if bmp is not None:
            return bmp
        img = pil_loader(path)
        return np.ascontiguousarray(img).reshape(-1), img.shape[0], img.shape[1], img.shape[1] * 3, False, False

    def preprocess_array(self, buf, H, W, pitch, bgr, bottom_up):
        """One raw pixel array -> processed u8 CUDA tensor [H', W', 3] (models.py:191-203 minus the PNG save)."""
        t = torch.from_numpy(buf)
        raw = t.pin_memory().to(self.device, non_blocking=True) if t.numel() > (1 << 20) else t.to(self.device)
        if max(H, W) > self.target_size:
            if H != 4 * self.target_size or W != 4 * self.target_size:
                # any other size: the general-ratio kernel (f64 restatement of skimage's order-3 resize, models.py:194-198);
                # the result is target x target, i.e. square, so trim_black applies (models.py:200)
                out, fl = ops.preprocess_general(raw, H, W, self.target_size, pitch, bgr=bgr, bottom_up=bottom_up)
                first, last = fl.tolist()
                T = self.target_size
                return out[:(last - first) * T * 3].view(last - first, T, 3)
            out, fl = ops.preprocess_4x(raw, H, W, pitch, bgr=bgr, bottom_up=bottom_up)
            first, last = fl.tolist()
            Wo = W // 4
            return out[:(last - first) * Wo * 3].view(last - first, Wo, 3)
        img = raw.view(H, pitch)[:, :W * 3].reshape(H, W, 3)
        if bottom_up:
            img = img.flip(0)
        if bgr:
            img = img.flip(2)
        img = img.contiguous()
        if H == W:
            return trim_black(img)
        return img

    def preprocess_images(self, root_path):
        output_path = join(root_path, 'processed')
        items = make_dataset(root_path)
        if len(items) == 0:
            raise RuntimeError("Found 0 files in subfolders of: " + root_path)
        processed = {}
        with ThreadPoolExecutor(self.io_threads) as pool, warnings.catch_warnings():
            warnings.simplefilter('ignore')
            loads = [pool.submit(self._load_raw, path) for path, _, _, _ in items]
            saves = []
            for (path, _, fname, wood_type), fut in zip(items, loads):
                out = self.preprocess_array(*fut.result())
                fname = str.replace(fname, '.bmp', '.png')
                dst = join(output_path, 'samples', wood_type, fname)
                host = out.cpu().numpy()
                processed[dst] = host
                saves.append(pool.submit(lambda a, d: Image.fromarray(a).save(d), host, dst))
            for s in saves:
                s.result()
        return processed


class NeuralBarkCalculator():
    """models.py:206-364: loads the checkpoint and writes ``results/outputs/<wood>/*.png`` and
    ``results/final_stats.csv`` for every processed image, plus ``results/combined_images/<wood>/*.png`` as NBC_COMBINED says
    (figure.py: the native two-panel stand-in by default, the reference's matplotlib figure of models.py:280-347 with
    NBC_COMBINED=figure when matplotlib is installed, nothing with NBC_COMBINED=0) -- the same files the streaming
    FolderPipeline writes.

    tta: flip test-time augmentation, 'none' (default), 'h' or 'hv' (``ops.tta_views``): the network runs on each mirrored
    view of the image and the mask is the argmax of the views' mean logits, each flipped back after the bicubic upsample."""

    DEFAULT_MEAN = [0.7399, 0.6139, 0.4401]
    DEFAULT_STD = [0.1068, 0.1272, 0.1271]
    DEFAULT_MM_PER_PIXEL = 3.6 * 3.6

    def __init__(self, model_path, device, mean=DEFAULT_MEAN, std=DEFAULT_STD, target_size=1024,
                 mm_per_pix=DEFAULT_MM_PER_PIXEL, state_dict=None, precision=DEFAULT_PRECISION, load_weights=True, tta='none'):
        self.tta_flags = ops.tta_views(tta)[1]
        self.tta = tta
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError("device '%s': this build runs on CUDA (B200) only -- no CPU path" % device)
        with torch.device('meta'):      # no random init: every parameter is replaced by the checkpoint's tensor below
            self.model = fcn_resnet50(pretrained=False)
        if load_weights:      # --only_preprocess never touches the network (predict.py:55-58)
            if state_dict is None:
                state_dict = torch.load(model_path, map_location=self.device)
            self.model.load_state_dict(state_dict, strict=True, assign=True)
            self.model.to(self.device)
        self.model.eval()  # the reference forgets this (SURVEY.md D5); eval is the reproducible behaviour
        self.model.set_normalisation(mean, std)
        self.model.set_precision(precision)
        self.mean = mean
        self.std = std
        self.target_size = target_size
        self.mm_per_pix = mm_per_pix

    # models.py:323-332 in the reference's float32 arithmetic, from integer pixel counts
    def _stats_strings(self, counts, n_pixels):
        out = []
        for class_idx in (1, 2):
            n = np.float32(counts[class_idx])
            pct = n / np.float32(n_pixels)
            out.append('{:.5f}'.format(pct * np.float32(100)))
            out.append('{:.5f}'.format(float(np.float32(n * np.float32(self.mm_per_pix)))))
        return out

    def predict_array(self, image_u8, excludes_nodes=False):
        """u8 CUDA [H,W,3] processed image -> (u8 mask [H,W] CUDA, counts int32[3] CUDA)."""
        if self.tta == 'none':
            mask = self.model.predict_mask_u8(image_u8.unsqueeze(0))
        else:
            mask = self.tta_mask(image_u8)
        mask, counts = ops.remove_small_zones_u8(mask, 150, exclude_nodes=excludes_nodes)
        return mask[0], counts[0]

    def tta_mask(self, image_u8):
        """The mask of ``self.tta``'s view set for one processed image (u8 CUDA [H,W,3]) -> u8 [1,H,W]: the views run as
        a ragged batch of one image -- flip, network, then the multi-view K3 over all views.  The canvas has at least the
        16 rows the network takes; rows below the image are zero and take no part."""
        H, W = image_u8.shape[0], image_u8.shape[1]
        Hc = max(H, 16)
        canvas = torch.zeros((1, Hc, W, 3), dtype=torch.uint8, device=image_u8.device)
        canvas[0, :H] = image_u8
        heights = torch.tensor([H], dtype=torch.int32, device=image_u8.device)
        self.model._check_eval()
        plan = self.model.native_plan()
        lows = [plan.forward_ragged(canvas if f == 0 else ops.flip_ragged(canvas, heights, f), heights=heights)
                for f in self.tta_flags]
        mask = ops.upsample_argmax_views_ragged(lows, self.tta_flags, heights, (Hc, W))
        return mask[:, :H].contiguous()

    def predict(self, root_path, excludes_nodes, processed=None, io_threads=8):
        output_path = join(root_path, 'results')
        processed_path = join(root_path, 'processed')
        dataset = RegressionDatasetFolder(processed_path, include_fname=True, loader=lambda p, grayscale=False: p)
        results_csv = [['Name', 'Type', 'Image Size', 'Output Bark %', 'Bark area (mm^2)', 'Output Node %',
                        'Node area (mm^2)']]
        processed = processed or {}

        def load(path):
            return processed[path] if path in processed else pil_loader(path)

        with ThreadPoolExecutor(io_threads) as pool:
            loads = [pool.submit(load, dataset.samples[i][0]) for i in range(len(dataset))]
            saves = []
            for i, fut in enumerate(loads):
                _, _, fname, wood_type = dataset.samples[i]
                img = torch.from_numpy(np.ascontiguousarray(fut.result())).to(self.device)
                mask, counts = self.predict_array(img, excludes_nodes)
                mask_h = mask.cpu().numpy()
                dual = _DUAL_LUT[mask_h]                      # models.py:349-353: classes 0 / 1 / 2 -> 0 / 127 / 255
                stats = self._stats_strings(counts.tolist(), mask.numel())
                results_csv.append([fname, wood_type] + stats)
                saves.append(pool.submit(lambda a, d: Image.fromarray(a, mode='L').save(d), dual,
                                         join(output_path, 'outputs', wood_type, fname)))
                from . import pipeline               # (imports models lazily: no cycle at module load)
                saves.append(pool.submit(pipeline.write_combined, join(output_path, 'combined_images', wood_type, fname),
                                         img.cpu().numpy(), mask_h, stats, fname, self.mean, self.std))
            for s in saves:
                s.result()
        with open(join(output_path, 'final_stats.csv'), 'w') as f:   # as models.py:360-364 (tab-delimited)
            csv.writer(f, delimiter='\t').writerows(results_csv)
        return results_csv
