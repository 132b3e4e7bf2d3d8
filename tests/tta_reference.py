"""f32 CPU restatement of flip test-time augmentation (``predict --tta``, ``evaluate --tta``), the reference the TTA tests
compare the GPU path against.  For a normalised image x [1,3,H,W] and a view set of flip flags (1 = columns, 2 = rows):

    L_v  = un-flip_v( bicubic_up( net( flip_v(x) ) ) )       f32 [1,3,H,W], upsample_bicubic_restated (K3's arithmetic)
    mean = (((L_0 + L_1) + L_2) + L_3) * (1/|V|)            f32, round-to-nearest, in view order; one view: L_0 unscaled
"""
import numpy as np
import torch

from oracle import model as omodel


def flip_dims(flags, row_axis, col_axis):
    """The axes ``flags`` mirrors: col_axis for bit 0 (columns), row_axis for bit 1 (rows)."""
    return ([col_axis] if flags & 1 else []) + ([row_axis] if flags & 2 else [])


def mean_of_views(lows, flags, size):
    """The views' mean full-resolution logits from their low-resolution logits: lows[v] f32 [N,3,h,w] is the network's
    output for the input mirrored with flags[v]; each is upsampled to ``size`` (upsample_bicubic_restated), flipped back
    and summed in view order, then scaled by 1/|V|."""
    total = None
    for low, f in zip(lows, flags):
        up = omodel.upsample_bicubic_restated(np.asarray(low, dtype=np.float32), size)
        dims = flip_dims(f, 2, 3)
        if dims:
            up = np.ascontiguousarray(np.flip(up, axis=tuple(dims)))
        total = up if total is None else (total + up).astype(np.float32)
    if len(lows) > 1:
        total = (total * np.float32(1.0 / len(lows))).astype(np.float32)
    return total


def view_lowres(model, x, views):
    """The network's f32 low-resolution logits of every view: x f32 [1,3,H,W] normalised, views a sequence of flip flags."""
    out = []
    for f in views:
        dims = flip_dims(f, 2, 3)
        xf = torch.flip(x, dims) if dims else x
        out.append(omodel.lowres_logits(model, xf).numpy())
    return out


def tta_logits(model, x, views):
    """The mean logits of the view set ``views`` (flip flags in summation order) for x f32 [1,3,H,W] -> f32 [1,3,H,W]."""
    return mean_of_views(view_lowres(model, x, views), views, tuple(x.shape[-2:]))
