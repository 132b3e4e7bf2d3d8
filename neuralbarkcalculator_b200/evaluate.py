"""Whole-image validation of a network on a ``DeviceDataset`` (the reference selects its checkpoint on validation
metrics and drives ``ReduceLROnPlateau`` / ``EarlyStopping`` from them, ``__main__.py:240-257``).

The reference's validation loader is not available, so the definition here is stated: every image is seen whole, as
``predict.py`` sees it -- batch-1 semantics, eval-mode network (BatchNorm on its running statistics, no dropout) in
predict's storage precision (``models.DEFAULT_PRECISION``), logits upsampled bicubically to the image's own size -- and
each figure is a mean over images of the per-image value:

* ``loss``: the training loss on the full-resolution logits (``weighted_ce``, ``lovasz`` or ``mixed`` = ce / 4 + lovasz);
* ``miou``: ``lovasz_losses.iou`` of the argmax (EMPTY = 1, in %), averaged over the three classes;
* ``f1``: ``PixelWiseF1`` per class: argmax, ``remove_small_zones`` (150 pixels), F1 with the absent-class rule.

Each image costs existing kernels only: a ragged network pass per chunk of equally wide images
(``Plan.forward_ragged``, bit-identical per image to a forward of that image alone), the bicubic upsample, the loss
forward, argmax, two confusion matrices and the region removal; everything is read back once at the end."""
import numpy as np
import torch

from . import ops
from .lovasz_losses import iou_from_confusion
from .models import DEFAULT_PRECISION, NeuralBarkCalculator, fcn_resnet50
from .utils import f1_from_confusion, get_pos_weight

LOSSES = ('weighted_ce', 'lovasz', 'mixed')


def make_plan(state_dict, device, precision=DEFAULT_PRECISION):
    """The inference plan of a 326-key ``fcn_resnet50`` state_dict, with predict's normalisation."""
    with torch.device('meta'):
        keys = list(fcn_resnet50(pretrained=False).state_dict().keys())
    if set(keys) != set(state_dict.keys()):
        raise RuntimeError('evaluate: the state_dict does not have the 326 keys of fcn_resnet50')
    tensors = [state_dict[k].detach().to(device) if state_dict[k].dtype == torch.int64
               else state_dict[k].detach().to(device=device, dtype=torch.float32) for k in keys]
    return ops.Plan(tensors, NeuralBarkCalculator.DEFAULT_MEAN, NeuralBarkCalculator.DEFAULT_STD, device, precision)


def image_logits(plan, ds, indices, chunk=8):
    """Yields (dataset index, full-resolution logits f32 [1,3,h,w], classes u8 [1,h,w]) for every index, in chunks of
    up to ``chunk`` images of one width (one ragged network pass each)."""
    indices = [int(i) for i in indices]
    widths = sorted({int(ds.sizes[i, 1]) for i in indices})
    for w in widths:
        same = [i for i in indices if ds.sizes[i, 1] == w]
        for start in range(0, len(same), chunk):
            part = same[start:start + chunk]
            hs = [int(ds.sizes[i, 0]) for i in part]
            sel = torch.tensor(part, dtype=torch.int64, device=ds.device)
            canvas = ds.images.index_select(0, sel)[:, :max(hs), :w].contiguous()
            heights = torch.tensor(hs, dtype=torch.int32, device=ds.device)
            low = plan.forward_ragged(canvas, heights=heights)
            for j, (i, h) in enumerate(zip(part, hs)):
                full = ops.upsample_bicubic(low[j:j + 1, :, :(h + 7) // 8].contiguous(), (h, w))
                yield i, full, ds.classes[i:i + 1, :h, :w].contiguous()


def evaluate(state_dict, ds, indices, loss='lovasz', class_weights=None, precision=DEFAULT_PRECISION, chunk=8):
    """Validation of ``state_dict`` on the items ``indices`` of ``ds`` (see the module docstring for the definition).
    Returns {'loss', 'miou', 'f1' (3 values): means over the images, 'rows': one dict per image with the same keys and
    'index'}."""
    if loss not in LOSSES:
        raise ValueError("loss must be 'weighted_ce', 'lovasz' or 'mixed'")
    if len(indices) == 0:
        raise RuntimeError('evaluate: no images')
    dev = ds.device
    with torch.cuda.device(dev):
        plan = make_plan(state_dict, dev, precision)
        w = (get_pos_weight() if class_weights is None else class_weights).to(device=dev, dtype=torch.float32).contiguous()
        order, losses, cms = [], [], []
        for i, full, lab in image_logits(plan, ds, indices, chunk):
            zero = torch.zeros((), dtype=torch.float32, device=dev)
            ce = ops.wce_fwd_bwd(full, lab, w, need_grad=False)[0] if loss != 'lovasz' else zero
            lov = ops.lovasz_softmax_fwd_bwd(full, lab, need_grad=False)[0] if loss != 'weighted_ce' else zero
            pred = ops.argmax3_u8(full)
            cm_iou = ops.confusion_matrix(pred, lab)
            ops.remove_small_zones_u8(pred, 150)
            order.append(i)
            losses.append(torch.stack([ce, lov]))
            cms.append(torch.stack([cm_iou, ops.confusion_matrix(pred, lab)]))
        losses = torch.stack(losses).cpu().numpy()
        cms = torch.stack(cms).cpu().numpy()
    rows = []
    for i, (ce, lov), (cm_iou, cm_f1) in zip(order, losses, cms):
        value = {'weighted_ce': ce, 'lovasz': lov, 'mixed': ce / np.float32(4) + lov}[loss]      # f32, as MixedLoss
        rows.append({'index': i, 'loss': float(value), 'miou': float(np.mean(iou_from_confusion(cm_iou))),
                     'f1': f1_from_confusion(cm_f1)})
    return {'loss': float(np.mean([r['loss'] for r in rows])), 'miou': float(np.mean([r['miou'] for r in rows])),
            'f1': np.mean([r['f1'] for r in rows], axis=0), 'rows': rows}
