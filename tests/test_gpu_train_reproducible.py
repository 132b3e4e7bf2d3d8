"""Bit-reproducible training on the B200: two Trainers from the same state_dict fed the same batches end with the same
bits in every buffer; the split-K weight gradient adds its splits in a fixed order with one writer per element; and
``training_state`` / ``load_training_state`` carry a Trainer over to a fresh one exactly."""
import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu

_BATCHES = {}


def _batch(dev, N, H, W, j):
    key = (N, H, W, j)
    if key not in _BATCHES:
        _BATCHES[key] = (torch.from_numpy(np.stack([synth.texture_u8(H, W, 31 * j + i) for i in range(N)])).to(dev),
                         torch.from_numpy(np.stack([synth.class_mask(H, W, 700 + 31 * j + i) for i in range(N)])).to(dev))
    return _BATCHES[key]


def _bits(t):
    return t.detach().contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _steps(tr, dev, first, steps, accumulate):
    """``steps`` optimizer steps of ``accumulate`` micro-batches each, as fit runs them; returns the losses and the
    gradient buffer of the last step (before Adam)."""
    losses, grads = [], None
    for s in range(first, first + steps):
        for j in range(accumulate):
            x, t = _batch(dev, tr.N, tr.H, tr.W, s * accumulate + j)
            losses.append(tr.forward_backward(x, t, seed=tr.dropout_seed(j), accumulate=j > 0).clone())
        grads = tr.grads.clone()
        tr.optimizer_step()
    torch.cuda.synchronize()
    return losses, grads


CASES = {
    'fit': dict(N=5, H=512, W=512, loss='lovasz', freeze='none', accumulate=2),       # fit's defaults, --accumulate 2
    'bench': dict(N=8, H=1024, W=1024, loss='weighted_ce', freeze='none', accumulate=1),   # bench.py's train size
    'mixed': dict(N=5, H=512, W=512, loss='mixed', freeze='none', accumulate=1),
    'layer2': dict(N=5, H=512, W=512, loss='lovasz', freeze='layer2', accumulate=1),
}


@pytest.mark.parametrize('case', list(CASES))
def test_two_trainers_are_bit_identical(cuda_device, synthetic_sd, case):
    """Same state_dict, same batches and seeds, three optimizer steps: params, Adam moments, running statistics,
    the last gradients and every loss are the same bits (dropout 0.8)."""
    from neuralbarkcalculator_b200.train import Trainer
    c = CASES[case]
    runs = []
    for _ in range(2):
        tr = Trainer(synthetic_sd, c['N'], c['H'], c['W'], device='cuda:0', loss=c['loss'], freeze=c['freeze'], seed=4)
        losses, grads = _steps(tr, cuda_device, 0, 3, c['accumulate'])
        runs.append((tr, losses, grads))
        del tr
    (a, la, ga), (b, lb, gb) = runs
    assert all(torch.isfinite(v) for v in la)
    assert all(_same(x, y) for x, y in zip(la, lb)), [(float(x), float(y)) for x, y in zip(la, lb)]
    assert _same(ga, gb), 'gradients: %d of %d floats differ' % (int((_bits(ga) != _bits(gb)).sum()), ga.numel())
    for name in ('params', 'adam_m', 'adam_v', 'stats'):
        x, y = getattr(a, name), getattr(b, name)
        assert _same(x, y), '%s: %d of %d floats differ' % (name, int((_bits(x) != _bits(y)).sum()), x.numel())
    assert int((ga[a.param_off:] != 0).sum()) > 0.5 * (ga.numel() - a.param_off)


@pytest.mark.parametrize('N,H,W', [(2, 128, 128), (5, 512, 512)])
def test_accumulated_twice_is_exactly_double(cuda_device, synthetic_sd, N, H, W):
    """Every gradient writer adds a fixed-order sum to what the buffer holds (grads = grads + sum): the same
    micro-batch accumulated twice gives exactly twice the gradient of one, in every element -- the stem's split-K
    tcgen05 gradient, the bottlenecks', BatchNorm's and the classifier's."""
    from neuralbarkcalculator_b200.train import Trainer
    tr = Trainer(synthetic_sd, N, H, W, device='cuda:0', loss='lovasz', seed=2)
    x, t = _batch(cuda_device, N, H, W, 0)
    tr.forward_backward(x, t, seed=9)
    one = tr.grads.clone()
    tr.forward_backward(x, t, seed=9, accumulate=True)
    torch.cuda.synchronize()
    assert _same(tr.grads, 2 * one), '%d of %d floats differ' % (int((tr.grads != 2 * one).sum()), one.numel())
    stem = tr.gradients()['backbone.conv1.weight']
    assert int((stem != 0).sum()) > 0.9 * stem.numel()


@pytest.mark.parametrize('N,H,W,Cin,Cout,k,stride,pad', [
    (8, 128, 128, 64, 256, 1, 1, 0),       # 2 weight tiles x 74 splits of 28 pixel tiles, the last one of 4
    (5, 128, 128, 64, 64, 3, 1, 1),        # 9 taps x 16 splits
    (2, 64, 64, 256, 512, 1, 2, 0),        # stride 2, 4 weight tiles x 2 splits
])
def test_split_k_wgrad_is_deterministic(cuda_device, N, H, W, Cin, Cout, k, stride, pad):
    """nbc_conv_wgrad_bf16_ws (split-K, partials reduced in a fixed order): two runs are bit-identical; with dw
    pre-filled the result is exactly dw + the sum of a zeroed run; and the values match torch within the wgrad tolerance
    of tests/test_gpu_kernels.py.  The entry without scratch (one CTA sums all N*Ho*Wo pixels in one tensor-memory
    accumulator, which rounds less finely than f32 adds over that many terms) is bit-reproducible too and agrees with
    the split result to a relative 1e-3."""
    from neuralbarkcalculator_b200 import _lib, ops
    lib = _lib.load()
    import ctypes as C
    d = _lib.ConvDesc(N, H, W, Cin, Cout, k, k, stride, pad, 1, 0, 1, 0)
    assert lib.nbc_conv_wgrad_workspace_bytes(C.byref(d)) > 0       # the shape does split
    g = torch.Generator().manual_seed(N * Cin + Cout)
    Ho = (H + 2 * pad - k) // stride + 1
    Wo = (W + 2 * pad - k) // stride + 1
    x = torch.randn(N, H, W, Cin, generator=g).to(torch.bfloat16)
    dz = torch.randn(N, Ho, Wo, Cout, generator=g).to(torch.bfloat16)
    xd, dzd = x.to(cuda_device), dz.to(cuda_device)
    a = ops.conv_wgrad_bf16(dzd, xd, k, k, stride=stride, pad=pad, split=True)
    b = ops.conv_wgrad_bf16(dzd, xd, k, k, stride=stride, pad=pad, split=True)
    base = torch.randn(Cout, k, k, Cin, generator=g).to(cuda_device)
    c = ops.conv_wgrad_bf16(dzd, xd, k, k, stride=stride, pad=pad, split=True, out=base.clone())
    one = ops.conv_wgrad_bf16(dzd, xd, k, k, stride=stride, pad=pad, impl=1, split=False)
    one2 = ops.conv_wgrad_bf16(dzd, xd, k, k, stride=stride, pad=pad, impl=1, split=False)
    torch.cuda.synchronize()
    assert _same(a, b) and _same(one, one2)
    assert _same(c, base + a)
    ref = torch.nn.grad.conv2d_weight(x.float().permute(0, 3, 1, 2), (Cout, Cin, k, k), dz.float().permute(0, 3, 1, 2),
                                      stride=stride, padding=pad).permute(0, 2, 3, 1)
    tol = 1e-4 * np.sqrt(N * Ho * Wo) + 1e-5 * ref.abs()
    err = (a.cpu() - ref).abs()
    assert not (err > tol).any(), 'split: max err %.4g' % float(err.max())
    rel = float((one - a).double().norm() / a.double().norm())
    assert rel < 1e-3, 'one split vs split: relative %.3g' % rel


@pytest.mark.parametrize('freeze', ['none', 'layer2'])
def test_training_state_round_trip(cuda_device, synthetic_sd, freeze):
    """training_state -> a fresh Trainer -> load_training_state: the buffers are bit-identical, and two more steps on
    both trainers stay so."""
    from neuralbarkcalculator_b200.train import Trainer
    a = Trainer(synthetic_sd, 2, 256, 256, device='cuda:0', loss='lovasz', freeze=freeze, seed=6)
    _steps(a, cuda_device, 0, 2, 1)
    state = a.training_state()
    assert sorted(state['model']) == sorted(a.keys) and state['step_count'] == 2
    a.lr = 1e-4                      # a plateau drop between epochs travels with the state
    state['lr'] = a.lr
    b = Trainer(synthetic_sd if freeze == 'none' else state['model'], 2, 256, 256, device='cuda:0', loss='lovasz',
                freeze=freeze, seed=6)
    b.load_training_state(state)
    for name in ('params', 'adam_m', 'adam_v', 'stats'):
        assert _same(getattr(a, name), getattr(b, name)), name
    assert b.step_count == a.step_count and b.lr == a.lr and b.num_batches_tracked == a.num_batches_tracked
    if freeze != 'none':
        assert not a.adam_m[:a.param_off].any() and not b.adam_v[:b.param_off].any()
    la, ga = _steps(a, cuda_device, 2, 2, 1)
    lb, gb = _steps(b, cuda_device, 2, 2, 1)
    assert all(_same(x, y) for x, y in zip(la, lb)) and _same(ga, gb)
    for name in ('params', 'adam_m', 'adam_v', 'stats'):
        assert _same(getattr(a, name), getattr(b, name)), name
    sa, sb = a.state_dict(), b.state_dict()
    assert all(_same(sa[k], sb[k]) for k in sa)
