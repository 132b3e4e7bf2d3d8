"""Host-side mirror of the pieces of the reference's ``lovasz_losses.py`` that its training script uses
(``__main__.py:4``: ``from lovasz_losses import LovaszSoftmax, miou, iou``): same names and arguments, the work is
done by the CUDA kernels behind ``libnbc.so`` (csrc/lovasz.cu).  CUDA tensors only -- there is no CPU path."""
import numpy as np
import torch
from torch import nn

from . import ops


class _LovaszFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, predict, true):
        loss, grad = ops.lovasz_softmax_fwd_bwd(predict, true, need_grad=True)
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (grad,) = ctx.saved_tensors
        return grad * grad_out, None


class LovaszSoftmax(nn.Module):
    """lovasz_losses.py:162-166: softmax over dim 1, then lovasz_softmax(classes='present', per_image=False).
    ``predict``: logits [B,3,H,W]; ``true``: labels [B,H,W] (uint8 or int64).  Forward and backward are produced
    together (fused softmax + errors, radix sort per class, Lovasz gradient, softmax backward)."""

    def forward(self, predict, true):
        return _LovaszFunction.apply(predict.float(), true)


def _confusion(preds, labels):
    if not preds.is_cuda:
        raise RuntimeError('iou / miou: CUDA tensors required (no CPU path in neuralbarkcalculator_b200)')
    pred = ops.argmax3_u8(preds.float())
    return ops.confusion_matrix(pred, labels).cpu().numpy()


def iou(preds, labels, C=3, EMPTY=1.):
    """lovasz_losses.py:54-73: array of per-class IoU (in %) of argmax(preds, 1) against labels, over the whole batch."""
    if C != 3:
        raise RuntimeError('iou: the B200 path is built for the 3 classes of the reference')
    return iou_from_confusion(_confusion(preds, labels), EMPTY)


def iou_from_confusion(cm, EMPTY=1.):
    """The per-class IoU (in %) of ``iou`` from a 3x3 confusion matrix cm[label, prediction]."""
    out = []
    for i in range(len(cm)):
        inter = int(cm[i, i])
        union = int(cm[i, :].sum() + cm[:, i].sum() - cm[i, i])
        out.append(EMPTY if not union else float(inter) / float(union))
    return 100 * np.array(out)


def miou(preds, labels):
    """lovasz_losses.py:76-77."""
    return np.mean(iou(preds, labels))
