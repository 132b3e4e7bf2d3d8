"""Float64 restatements of the training backward, one operation at a time (test infrastructure).

Each helper takes the operands a kernel consumed and returns what it should have produced, so a test can check one
backward kernel from the kernel's own stored inputs (teacher forcing).  Tensors are NCHW; everything is computed in
float64, on the device of the operands.  Each helper is checked against torch autograd in tests/test_oracle.py."""
import numpy as np
import torch
import torch.nn.functional as F

from .model import bicubic_weights_f32


def bn_backward(dy, y, z, gamma, relu, eps=1e-5):
    """Backward of y = relu?(BatchNorm(z)) with batch statistics (training mode), from the incoming dy.

    The ReLU mask comes from the stored output y (the gradient passes where y > 0); mean and biased variance are
    recomputed from z.  Returns dz, dgamma, dbeta and, for error bars, dgamma_abs / dbeta_abs: the same reductions
    taken over magnitudes."""
    z, g = z.double(), dy.double()
    if relu:
        g = torch.where(y > 0, g, torch.zeros_like(g))
    dims = (0, 2, 3)
    M = z.numel() // z.shape[1]
    mean = z.mean(dims, keepdim=True)
    invstd = (z.var(dims, unbiased=False, keepdim=True) + eps).rsqrt()
    xhat = (z - mean) * invstd
    s1, s2 = g.sum(dims, keepdim=True), (g * xhat).sum(dims, keepdim=True)
    dz = gamma.double().view(1, -1, 1, 1) * invstd * (g - s1 / M - xhat * s2 / M)
    return dict(dz=dz, dgamma=s2.flatten(), dbeta=s1.flatten(), dgamma_abs=(g.abs() * xhat.abs()).sum(dims),
                dbeta_abs=g.abs().sum(dims))


def running_stats(z, old_mean, old_var, momentum=0.1, unbiased=True):
    """torch BatchNorm2d's running-statistics update from the batch z: (new mean, new var).  ``unbiased=False`` is the
    wrong estimator (a negative control)."""
    z = z.double()
    dims = (0, 2, 3)
    mean, var = z.mean(dims), z.var(dims, unbiased=unbiased)
    return (1 - momentum) * old_mean.double() + momentum * mean, (1 - momentum) * old_var.double() + momentum * var


def conv_dgrad(dz, w, in_shape, stride=1, pad=0, dil=1):
    """Gradient of conv2d(x, w) with respect to x (shape ``in_shape``)."""
    return torch.nn.grad.conv2d_input(tuple(in_shape), w.double(), dz.double(), stride=stride, padding=pad, dilation=dil)


def conv_wgrad(x, dz, w_shape, stride=1, pad=0, dil=1):
    """Gradient of conv2d(x, w) with respect to w (shape ``w_shape``, OIHW)."""
    return torch.nn.grad.conv2d_weight(x.double(), tuple(w_shape), dz.double(), stride=stride, padding=pad, dilation=dil)


def maxpool_backward(dy, x, last=False):
    """Backward of max_pool2d(x, 3, stride 2, padding 1): each output's gradient goes to the FIRST maximum of its window
    in row-major scan order (torch's rule; ties are common after a ReLU).  ``last=True`` routes to the last maximum
    instead (a negative control)."""
    N, C, H, W = x.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    xp = F.pad(x.double(), (1, 1, 1, 1), value=float('-inf'))
    best = torch.full((N, C, Ho, Wo), float('-inf'), dtype=torch.float64, device=x.device)
    pos = torch.zeros((N, C, Ho, Wo), dtype=torch.int64, device=x.device)
    for k in range(9):
        ky, kx = divmod(k, 3)
        v = xp[:, :, ky:ky + 2 * Ho - 1:2, kx:kx + 2 * Wo - 1:2]
        take = (v >= best) if last else (v > best)
        best, pos = torch.where(take, v, best), torch.where(take, k, pos)
    dxp = torch.zeros_like(xp)
    for k in range(9):
        ky, kx = divmod(k, 3)
        dxp[:, :, ky:ky + 2 * Ho - 1:2, kx:kx + 2 * Wo - 1:2] += torch.where(pos == k, dy.double(), 0.0)
    return dxp[:, :, 1:H + 1, 1:W + 1]


def bicubic_matrix(in_size, out_size, clamp=True, device=None):
    """Dense [out, in] interpolation matrix of F.interpolate(mode='bicubic', align_corners=False) along one axis, from
    the float32 tap weights the kernels use, on ``device`` (default: the CPU).  ``clamp=False`` drops the taps outside
    the input instead of clamping them to the edge (a negative control)."""
    idx, w = bicubic_weights_f32(in_size, out_size, clamp=clamp)
    m = np.zeros((out_size, in_size))
    for d in range(out_size):
        for k in range(4):
            if 0 <= idx[d, k] < in_size:
                m[d, idx[d, k]] += float(w[d, k])
    return torch.from_numpy(m).to(device)


def upsample_bicubic(low, size):
    """up = Wy . low . Wx^T per plane: [N,C,h,w] -> [N,C,H,W]."""
    wy = bicubic_matrix(low.shape[-2], size[0], device=low.device)
    wx = bicubic_matrix(low.shape[-1], size[1], device=low.device)
    return torch.einsum('Yi,ncij,Xj->ncYX', wy, low.double(), wx)


def upsample_adjoint(dup, low_size, clamp=True):
    """Adjoint of ``upsample_bicubic``: dlow = Wy^T . dup . Wx per plane, [N,C,H,W] -> [N,C,h,w]."""
    wy = bicubic_matrix(low_size[0], dup.shape[-2], clamp=clamp, device=dup.device)
    wx = bicubic_matrix(low_size[1], dup.shape[-1], clamp=clamp, device=dup.device)
    return torch.einsum('Yi,ncYX,Xj->ncij', wy, dup.double(), wx)


def dropout_keep(seed, n, p):
    """Keep mask of the head's dropout over flat indices 0..n-1: keep(i) = u(seed, i) >= p with u the top 24 bits of
    splitmix64(seed + golden * (i + 1)) over 2^24 -- the hash the forward and the backward both regenerate."""
    u = (splitmix64_bits(seed, n) >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return u >= np.float32(p)


def splitmix64_bits(seed, n):
    """The raw 64-bit hashes behind ``dropout_keep`` (for known-answer checks)."""
    i = np.arange(n, dtype=np.uint64)
    with np.errstate(over='ignore'):
        z = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * (i + np.uint64(1))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))
