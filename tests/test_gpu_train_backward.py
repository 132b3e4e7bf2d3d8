"""Teacher-forced parity of the training BACKWARD, unit by unit (``pytest -m gpu``).

The forward of the training step is pinned unit by unit in test_gpu_train.py; the end-to-end gradient tests there can
only use cosines and norm ratios, which a kernel that drops a border row or misroutes a maxpool tie still passes.  Here
one step runs with capture on (``Trainer.enable_capture``): the dy every BatchNorm backward consumed and the dz it
produced are kept per unit, and every backward operation is recomputed in float64 (oracle/backward.py) from the
kernel's OWN operands -- stored z / y, captured dy / dz, bf16 weights as the kernels round them.  No error is carried
from one layer to the next, so the bars are those of one operation's arithmetic:

  values stored in bf16 (dz, data gradients):  |got - ref| <= 2^-7 S + 2e-3 max|ref|
      S = sum of the magnitudes of the separately rounded parts: |ref| for one conv, |a| + |b| where the kernel rounds
      the skip gradient b before adding it to a conv's a.  2^-7 covers up to four bf16 roundings (2^-9 each) on the way;
      2e-3 max|ref| the f32 summation order of long reductions whose terms cancel.
  f32 reductions (dW, dgamma, dbeta, classifier dW / db, dL/dlow, logits):  |got - ref| <= 2^-14 A + 2^-20 max A
      A = the same reduction over magnitudes; any summation order, split-K atomics or tensor-core accumulation stays
      orders of magnitude below 2^-14 A, while a missing or shifted row is a sizeable fraction of A.
  running statistics:  relative error <= 1e-5 of the magnitudes summed (0.9 |old| + 0.1 mean |z| or mean z^2).

Four negative controls (biased running variance, last-maximum maxpool routing, unflipped 3x3 taps, bicubic adjoint
without edge clamping) must FAIL the same bars on the same captured tensors, which shows the bars are tight enough."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import backward as ob
from oracle import model as omodel
from oracle import synth
from oracle.teacher import Bars, bf16_bar, check_head, f32_bar, plan_units, run_step, stored_inputs

pytestmark = pytest.mark.gpu

GEOMETRIES = {
    # (N, H, W)
    '2x64x96': (2, 64, 96),       # the shape of the other training tests
    # odd: 29x61 -> 15x31 -> 8x16.  layer2's stride-2 convs see an odd input (zero insertion up to the last row and
    # column), maxpool windows are cut by the bottom and right edges, the upsample ratios 58/8 and 122/16 are not
    # integers; an 8x16 map is one 128-pixel tile, so every layer3 / layer4 launch has 3 pixel tiles and the CTA-pair
    # data-gradient launches (1x1 and 3x3 without residual, 256-column tiles) run a phantom tile
    '3x58x122': (3, 58, 122),
    '2x192x256': (2, 192, 256),   # 2 x 96 x 128 stem pixels = 192 tiles > 148 SMs: the persistent loops wrap
}


def _step(cuda_device, sd, N, H, W, impl, dropout_p, seed):
    """One forward_backward with capture on (after the same step with capture off, which must compute the same)."""
    from neuralbarkcalculator_b200.train import Trainer
    x = torch.cat([omodel.normalise_u8(synth.texture_u8(H, W, 11 + i)) for i in range(N)])   # f32 NCHW input
    tgt = np.stack([synth.class_mask(H, W, 111 + i) for i in range(N)])
    tr = Trainer(sd, N, H, W, device='cuda:0', dropout=dropout_p, class_weights=torch.ones(3))
    run_step(tr, x.to(cuda_device), torch.from_numpy(tgt).to(cuda_device), seed, impl)
    return tr, x


def _check_step(tr, sd, x, dropout_p, seed, bars):
    units, blocks, head = plan_units()
    assert len(units) == tr.lib.nbc_train_num_units(C.c_void_p(tr.handle))
    N = x.shape[0]
    dims = (0, 2, 3)
    cache = {}

    def t(what, u):     # bf16 NHWC debug tensor -> f64 NCHW on the CPU (exact)
        if (what, u) not in cache:
            cache[(what, u)] = tr.debug_tensor(what, u).cpu().permute(0, 3, 1, 2).contiguous()
        return cache[(what, u)].double()

    def weight(u):      # the kernels pack the f32 master weights to bf16 (round to nearest even)
        return sd[units[u]['conv'] + '.weight'].to(torch.bfloat16).double()

    # stored input of every unit: the bf16 staging image, the maxpool output (a max of bf16 values is exact) or a y
    src = stored_inputs(blocks, head)

    def x_of(u):
        s = src[u]
        if s == 'image':
            return x.to(torch.bfloat16).double()
        if s == 'pool':
            return F.max_pool2d(t(1, 0), 3, 2, 1)
        return t(1, s)

    def dgrad(u, w=None):
        U = units[u]
        return ob.conv_dgrad(t(7, u), weight(u) if w is None else w, x_of(u).shape, U['s'], U['p'], U['d'])

    grads = {k: v.cpu().double() for k, v in tr.gradients().items()}
    new = {k: v.cpu().double() for k, v in tr.state_dict().items()}

    # ---- per unit: running statistics, BatchNorm backward, weight gradient
    for u, U in enumerate(units):
        bn, conv = U['bn'], U['conv']
        z, y, dy, dz = t(0, u), t(1, u), t(6, u), t(7, u)
        old_m, old_v = sd[bn + '.running_mean'].double(), sd[bn + '.running_var'].double()
        rm, rv = ob.running_stats(z, old_m, old_v)
        tol_m = 1e-5 * (0.9 * old_m.abs() + 0.1 * z.abs().mean(dims))
        tol_v = 1e-5 * (0.9 * old_v + 0.1 * (z * z).mean(dims))
        bars.check('running stats', bn + '.running_mean', new[bn + '.running_mean'], rm, tol_m)
        bars.check('running stats', bn + '.running_var', new[bn + '.running_var'], rv, tol_v)
        bars.control('biased running var', not bars.within(new[bn + '.running_var'],
                                                           ob.running_stats(z, old_m, old_v, unbiased=False)[1], tol_v))

        ref = ob.bn_backward(dy, y, z, sd[bn + '.weight'], U['relu'])
        bars.check('bn dz', bn, dz, ref['dz'], bf16_bar(ref['dz'].abs(), ref['dz']))
        bars.check('bn dgamma dbeta', bn + '.weight', grads[bn + '.weight'], ref['dgamma'], f32_bar(ref['dgamma_abs']))
        bars.check('bn dgamma dbeta', bn + '.bias', grads[bn + '.bias'], ref['dbeta'], f32_bar(ref['dbeta_abs']))

        xu, wshape = x_of(u), sd[conv + '.weight'].shape
        A = torch.nn.grad.conv2d_weight(xu.abs().float(), wshape, dz.abs().float(), stride=U['s'], padding=U['p'],
                                        dilation=U['d'])       # only an error bar: f32 is plenty
        bars.check('wgrad', conv, grads[conv + '.weight'], ob.conv_wgrad(xu, dz, wshape, U['s'], U['p'], U['d']),
                   f32_bar(A.double()))

    # ---- data gradients, each checked through the dy the next unit upstream captured
    for bi, B in enumerate(blocks):
        c1, c2, c3, ds = B['c1'], B['c2'], B['c3'], B['ds']
        ref = dgrad(c3)
        bars.check('dgrad', units[c3]['conv'], t(6, c2), ref, bf16_bar(ref.abs(), ref))
        ref = dgrad(c2)
        bars.check('dgrad', units[c2]['conv'], t(6, c1), ref, bf16_bar(ref.abs(), ref))
        if bi == 0:
            bad = dgrad(c2, weight(c2).flip(2, 3))          # taps not flipped
            bars.control('unflipped 3x3 taps', not bars.within(t(6, c1), bad, bf16_bar(bad.abs(), bad)))
        masked = torch.where(t(1, c3) > 0, t(6, c3), torch.zeros(()).double())     # the skip path's gradient
        a = dgrad(c1)
        if ds is not None:
            bars.exact('ds dy == masked c3 dy', units[ds]['bn'], t(6, ds), masked)
            b = dgrad(ds)
        else:
            b = masked
        ref, S = a + b, a.abs() + b.abs()
        if bi > 0:
            bars.check('dgrad', units[c1]['conv'] + ' + skip', t(6, blocks[bi - 1]['c3']), ref, bf16_bar(S, ref))
        else:
            # block 0's input gradient -> maxpool backward (first maximum of each window of the stored stem y)
            ys = t(1, 0)
            got, refs = t(6, 0), ob.maxpool_backward(ref, ys)
            tol = bf16_bar(ob.maxpool_backward(S, ys), refs)
            bars.check('maxpool dgrad', 'backbone.bn1 dy', got, refs, tol)
            bars.control('maxpool last maximum', not bars.within(got, ob.maxpool_backward(ref, ys, last=True), tol))
    ref = dgrad(head)
    bars.check('dgrad', 'classifier.0', t(6, blocks[-1]['c3']), ref, bf16_bar(ref.abs(), ref))

    # ---- head: bicubic adjoint, classifier backward (through the dropout mask), low-res logits
    check_head(tr, sd, t(1, head), t(6, head), dropout_p, seed, bars)


@pytest.mark.parametrize('impl', [0, 1], ids=['wgrad_tc', 'wgrad_mma'])
@pytest.mark.parametrize('geom', list(GEOMETRIES))
def test_train_backward_teacher_forced(cuda_device, synthetic_sd, geom, impl):
    """Every backward kernel of the step at three geometries, on both weight-gradient paths (0: tcgen05 wgrad_tc and
    stem_wgrad_tc; 1: mma.sync wgrad_mma and the CUDA-core stem_wgrad), dropout 0."""
    N, H, W = GEOMETRIES[geom]
    tr, x = _step(cuda_device, synthetic_sd, N, H, W, impl, 0.0, 1)
    bars = Bars()
    _check_step(tr, synthetic_sd, x, 0.0, 1, bars)
    bars.report('%s %s' % (geom, 'wgrad_tc' if impl == 0 else 'wgrad_mma'))


def test_train_backward_dropout_mask(cuda_device, synthetic_sd):
    """Dropout 0.8 in the head: the restated hash mask reproduces the low-res logits from the stored head y, appears in
    the head's data gradient (exact zeros where dropped) and in the classifier's weight gradient; kept fraction 0.2."""
    N, H, W = GEOMETRIES['2x64x96']
    seed = (5 << 40) + (1 << 28) + 3      # Trainer.dropout_seed's layout: run seed, rank, step
    tr, x = _step(cuda_device, synthetic_sd, N, H, W, 0, 0.8, seed)
    bars = Bars()
    _check_step(tr, synthetic_sd, x, 0.8, seed, bars)
    bars.report('dropout 0.8')
