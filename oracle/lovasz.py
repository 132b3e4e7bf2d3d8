"""Oracle for the Lovasz-Softmax loss and the validation metrics (reference ``lovasz_losses.py:19-31`` lovasz_grad,
``54-77`` iou / miou, ``162-218`` LovaszSoftmax / lovasz_softmax / lovasz_softmax_flat; ``utils.py:185-192`` MixedLoss,
``201-235`` PixelWiseF1).  Test infrastructure only.

Plain torch / numpy restatement; ``oracle/make_golden.py`` pins it against the reference's own ``lovasz_losses``
module (which imports unmodified) and stores the agreed values in ``tests/golden/lovasz_small.npz``."""
import numpy as np
import torch
import torch.nn.functional as F

from . import losses, postprocess


def lovasz_grad(gt_sorted):
    """lovasz_losses.py:19-31."""
    p = len(gt_sorted)
    gts = gt_sorted.sum()
    intersection = gts - gt_sorted.float().cumsum(0)
    union = gts + (1 - gt_sorted).float().cumsum(0)
    jaccard = 1. - intersection / union
    if p > 1:
        jaccard[1:p] = jaccard[1:p] - jaccard[0:-1]
    return jaccard


def lovasz_softmax(logits, labels):
    """LovaszSoftmax.forward (lovasz_losses.py:162-166) -> lovasz_softmax(classes='present', per_image=False) ->
    lovasz_softmax_flat (197-218).  logits [B,C,H,W] f32, labels [B,H,W] int64."""
    probas = F.softmax(logits, dim=1)
    B, C, H, W = probas.shape
    probas = probas.permute(0, 2, 3, 1).contiguous().view(-1, C)
    labels = labels.view(-1)
    if probas.numel() == 0:
        return probas * 0.
    per_class = []
    for c in range(C):
        fg = (labels == c).float()
        if fg.sum() == 0:          # classes='present'
            continue
        errors = (fg - probas[:, c]).abs()
        errors_sorted, perm = torch.sort(errors, 0, descending=True)
        fg_sorted = fg[perm]
        per_class.append(torch.dot(errors_sorted, lovasz_grad(fg_sorted)))
    if not per_class:
        return torch.zeros((), dtype=logits.dtype)   # mean() of an empty generator -> 0
    acc = per_class[0]
    for v in per_class[1:]:
        acc = acc + v
    return acc if len(per_class) == 1 else acc / len(per_class)


def lovasz_softmax_with_grad(logits, labels):
    p = logits.detach().clone().requires_grad_(True)
    loss = lovasz_softmax(p, labels)
    loss.backward()
    return loss.detach(), p.grad


def lovasz_softmax_f64(logits, labels):
    """``lovasz_softmax`` in float64 throughout (softmax, Jaccard), on the device of the operands, with the errors
    sorted STABLY in descending order.  The value does not depend on how tied errors are ordered (a group of equal
    errors adds e * the Jaccard step over the whole group), so this is the reference's value without its rounding.
    Returns (loss, A) with A the same mean of sums over magnitudes, for error bars."""
    probas = F.softmax(logits.double(), dim=1)
    C = probas.shape[1]
    probas = probas.permute(0, 2, 3, 1).reshape(-1, C)
    labels = labels.reshape(-1)
    per_class, mag = [], []
    for c in range(C):
        fg = (labels == c).double()
        gts = fg.sum()
        if gts == 0:
            continue
        errors, perm = torch.sort((fg - probas[:, c]).abs(), dim=0, descending=True, stable=True)
        fg_sorted = fg[perm]
        jaccard = 1. - (gts - fg_sorted.cumsum(0)) / (gts + (1 - fg_sorted).cumsum(0))
        grad = torch.diff(jaccard, prepend=jaccard.new_zeros(1))
        per_class.append(torch.dot(errors, grad))
        mag.append(torch.dot(errors, grad.abs()))
    if not per_class:
        return torch.zeros((), dtype=torch.float64), torch.zeros((), dtype=torch.float64)
    return sum(per_class) / len(per_class), sum(mag) / len(mag)


def mixed_loss(logits, labels, weights):
    """utils.py:185-192: CustomWeightedCrossEntropy / 4 + LovaszSoftmax."""
    return losses.custom_weighted_cross_entropy(logits, labels, weights) / 4 + lovasz_softmax(logits, labels)


def confusion_matrix(pred, labels, C=3):
    """cm[t, p] = number of pixels with label t and prediction p."""
    pred = np.asarray(pred).reshape(-1).astype(np.int64)
    labels = np.asarray(labels).reshape(-1).astype(np.int64)
    return np.bincount(labels * C + pred, minlength=C * C).reshape(C, C)


def iou(logits, labels, C=3, EMPTY=1.):
    """lovasz_losses.py:54-73: per-class IoU (in %) of argmax(logits) over the WHOLE batch."""
    pred = torch.argmax(logits, dim=1)
    out = []
    for i in range(C):
        inter = int(((labels == i) & (pred == i)).sum())
        union = int(((labels == i) | (pred == i)).sum())
        out.append(EMPTY if not union else float(inter) / float(union))
    return 100 * np.array(out)


def miou(logits, labels):
    """lovasz_losses.py:76-77."""
    return np.mean(iou(logits, labels))


def f1_from_confusion(cm):
    """sklearn f1_score(labels=[0,1,2], average=None) from a confusion matrix (0 where a class has no support and no
    prediction, sklearn's zero_division default), then utils.py:224-226: a class absent from both targets and outputs
    takes the mean of the others."""
    cm = np.asarray(cm, dtype=np.float64)
    tp = np.diag(cm)
    denom = cm.sum(0) + cm.sum(1)
    scores = np.where(denom > 0, 2 * tp / np.maximum(denom, 1), 0.0)
    targets_count, outputs_count = cm.sum(1), cm.sum(0)
    for i in range(len(scores)):
        if targets_count[i] == 0 and outputs_count[i] == 0:
            scores[i] = np.delete(scores, i).mean()
    return scores


def pixelwise_f1(logits, labels, class_to_watch=None):
    """utils.py:201-235 with per-image region removal (the reference's 3-D structuring element also links neighbouring
    batch entries; per-image labelling is the documented deviation, SURVEY.md 3.3)."""
    pred = torch.argmax(logits, 1).numpy()
    pred = np.stack([postprocess.remove_small_zones_2d(m) for m in pred])
    scores = f1_from_confusion(confusion_matrix(pred, labels.numpy()))
    if class_to_watch is None:
        return scores.mean()
    if class_to_watch == 'loss':
        return 1 - scores.mean()
    if isinstance(class_to_watch, int):
        return scores[class_to_watch]
    return scores
