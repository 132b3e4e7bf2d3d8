"""Host-side mirror of the hot-path pieces of the reference's ``utils.py``: ``remove_small_zones`` (utils.py:135-148),
``CustomWeightedCrossEntropy`` (utils.py:151-165), ``get_pos_weight`` (utils.py:72-73), the metrics, and the training
loader's index bookkeeping (``get_splits``, utils.py:76-132; the weighted epoch sampler of ``__main__.py:165-172``).  Same
names, arguments and in-place behaviour; the pixel work is done by the CUDA kernels behind ``libnbc.so``."""
import torch
from torch import nn

import numpy as np

from . import ops
from .lovasz_losses import LovaszSoftmax


def get_pos_weight():
    """utils.py:72-73."""
    return torch.FloatTensor([0.4004, 2.0334, 93.1921])


_WOOD_TYPE_TO_IDX = {'epinette_gelee': 0, 'epinette_non_gelee': 1, 'sapin': 2}     # utils.py:83-87


def get_splits(dataset, label_pixels=None):
    """utils.py:76-132: per-wood-type 80 / 10 / 10 split (``ceil`` / ``floor``, each type shuffled with numpy's global
    generator in the fixed type order) and the sampling weights of the training items,
    ``exp(wood_type_weight * labelled_pixels / sum(labelled_pixels))`` normalised over the training split, in the
    reference's float32 arithmetic.  Returns (train_split, valid_split, test_split, train_weights) as numpy arrays.

    ``dataset`` yields ``(_, target, _, wood_type)`` like ``RegressionDatasetFolder(include_fname=True)``; targets may be
    class maps (torch / numpy).  ``label_pixels`` (optional, one number per item: how many pixels are not class 0) skips
    the scan of the targets -- the native loader counts them on the GPU."""
    from math import ceil, floor
    total_items = len(dataset)
    idxs_by_type = [[] for _ in range(3)]
    sample_weight = []
    wood_types = []
    for i, item in enumerate(dataset):
        target, wood_type = item[1], item[3]
        wood_types.append(wood_type)
        idxs_by_type[_WOOD_TYPE_TO_IDX[wood_type]].append(i)
        if label_pixels is not None:
            sample_weight.append(float(label_pixels[i]))
        else:
            t = torch.as_tensor(np.asarray(target) if not isinstance(target, torch.Tensor) else target)
            sample_weight.append(float(t.numel() - int((t == 0).sum())))
    sample_weight = torch.tensor(sample_weight)                    # float32, as the reference's tensor of python floats
    sample_weight = sample_weight / sample_weight.sum()
    train_split, valid_split, test_split = [], [], []
    wood_type_weights = []
    for k in range(3):
        idxs = np.asarray(idxs_by_type[k])
        np.random.shuffle(idxs)
        n_data = len(idxs)
        wood_type_weights.append(total_items / (3 * n_data))
        n_train = int(ceil(0.8 * n_data))
        n_valid = int(floor(0.1 * n_data))
        train_split.extend(idxs[:n_train])
        valid_split.extend(idxs[n_train:n_train + n_valid])
        test_split.extend(idxs[n_train + n_valid:])
    wood_type_weights = np.asarray(wood_type_weights)
    wood_type_weights /= wood_type_weights.sum()
    train_weights = torch.zeros(total_items).float()
    for i, wood_type in enumerate(wood_types):                     # float64 scalar x float32 tensor element, stored as float32
        train_weights[i] = wood_type_weights[_WOOD_TYPE_TO_IDX[wood_type]] * sample_weight[i]
    train_split, valid_split, test_split = np.asarray(train_split), np.asarray(valid_split), np.asarray(test_split)
    train_weights = np.exp(np.asarray(train_weights))
    train_weights = train_weights[train_split]
    train_weights /= train_weights.sum()
    return train_split, valid_split, test_split, train_weights


def weighted_epoch_batches(train_split, train_weights, batch_size, samples_per_item=12, generator=None):
    """The batches of one training epoch as dataset indices, as ``__main__.py:165-172`` draws them:
    ``BatchSampler(WeightedRandomSampler(train_weights, len(train_weights) * 12, replacement=True), batch_size,
    drop_last=True)`` over ``Subset(dataset, train_split)`` -- one ``torch.multinomial`` draw, cut into full batches.
    Returns int64 [n_batches, batch_size]; feed a row to ``augment.augment_batch`` (the native loader)."""
    w = torch.as_tensor(np.asarray(train_weights), dtype=torch.double)
    draws = torch.multinomial(w, len(w) * samples_per_item, True, generator=generator)
    n_batches = len(draws) // batch_size
    idx = torch.as_tensor(np.asarray(train_split), dtype=torch.int64)[draws[:n_batches * batch_size]]
    return idx.view(n_batches, batch_size)


def remove_small_zones(img, threshold=150):
    """In place on ``img`` (integer class tensor [B,H,W] or [H,W], CUDA) and returns it, like utils.py:135-148.

    Regions smaller than ``threshold`` pixels (8-connected) are flipped: small foreground blobs -> 0, then small
    background islands -> 1.  Labelling is per image (the reference's 3-D structuring element also links
    neighbouring batch entries, a bug that predict -- batch 1 -- never exercises; SURVEY.md 3.3)."""
    if not isinstance(img, torch.Tensor) or not img.is_cuda:
        raise RuntimeError('remove_small_zones: CUDA tensor required (no CPU path in neuralbarkcalculator_b200)')
    view = img if img.dim() == 3 else img.unsqueeze(0)
    if view.dtype == torch.uint8 and view.is_contiguous():
        ops.remove_small_zones_u8(view, threshold)
        return img
    m = view.to(torch.uint8).contiguous()
    ops.remove_small_zones_u8(m, threshold)
    view.copy_(m)
    return img


class _WCEFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, predict, true, weights):
        loss, grad = ops.wce_fwd_bwd(predict, true, weights, need_grad=True)
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (grad,) = ctx.saved_tensors
        return grad * grad_out, None, None


class CustomWeightedCrossEntropy(nn.Module):
    """utils.py:151-165: per-pixel CE weighted by ``weights[max(argmax(predict), true)]``, mean over all pixels.
    Forward and backward are one fused kernel (the gradient is produced in the forward pass)."""

    def __init__(self, weights):
        super().__init__()
        self.__name__ = "CustomWeightedCrossEntropy"
        self.weights = weights

    def forward(self, predict, true):
        w = self.weights.to(device=predict.device, dtype=torch.float32)
        return _WCEFunction.apply(predict.float(), true, w)


class MixedLoss(nn.Module):
    """utils.py:185-192: CustomWeightedCrossEntropy / 4 + LovaszSoftmax."""

    def __init__(self, cwe_weights):
        super(MixedLoss, self).__init__()
        self.ce = CustomWeightedCrossEntropy(cwe_weights)
        self.lovasz = LovaszSoftmax()

    def forward(self, predict, true):
        return self.ce(predict, true) / 4 + self.lovasz(predict, true)


class PixelWiseF1(nn.Module):
    """utils.py:201-235: per-class F1 of argmax(outputs) after remove_small_zones.  The argmax, the region removal and the
    3x3 confusion matrix run on the GPU (nbc_argmax3_u8, nbc_remove_small_zones, nbc_confusion_matrix); the F1 formula
    (sklearn f1_score(labels=[0,1,2], average=None) in the reference) is evaluated from the 9 counts on the host."""

    def __init__(self, class_to_watch):
        super().__init__()
        self.class_to_watch = class_to_watch
        if self.class_to_watch is None:
            self.__name__ = "PixelWiseF1"
        else:
            self.__name__ = "PixelWiseF1_class_{}".format(self.class_to_watch)

    def forward(self, outputs, labels):
        if not outputs.is_cuda:
            raise RuntimeError('PixelWiseF1: CUDA tensors required (no CPU path in neuralbarkcalculator_b200)')
        pred = ops.argmax3_u8(outputs.float())
        ops.remove_small_zones_u8(pred, 150)
        scores = f1_from_confusion(ops.confusion_matrix(pred, labels.to(outputs.device)).cpu().numpy())
        if self.class_to_watch is None:
            return scores.mean()
        elif self.class_to_watch == 'loss':
            return 1 - scores.mean()
        elif isinstance(self.class_to_watch, int):
            return scores[self.class_to_watch]
        else:
            return scores


def f1_from_confusion(cm):
    """Per-class F1 of ``PixelWiseF1`` from a 3x3 confusion matrix cm[label, prediction]: sklearn's f1_score (0 for a class
    with neither support nor prediction), then a class absent from both targets and outputs takes the mean of the others
    (utils.py:224-226)."""
    cm = np.asarray(cm, dtype=np.float64)
    tp = np.diag(cm)
    denom = cm.sum(0) + cm.sum(1)
    scores = np.where(denom > 0, 2 * tp / np.maximum(denom, 1), 0.0)
    targets_count, outputs_count = cm.sum(1), cm.sum(0)
    for i, count_i in enumerate(targets_count):
        if count_i == 0 and outputs_count[i] == 0:
            scores[i] = np.delete(scores, i).mean()
    return scores
