"""Machinery of the teacher-forced training tests (test infrastructure): the native plan's units in order, the error
bars, the collector of check results, one captured step, and the checks of the loss head.

tests/test_gpu_train_backward.py (small and odd shapes) and tests/test_gpu_train_production.py (the sizes ``fit`` and
the training benchmark run at) both use it.  The bars are those of one operation's arithmetic, because every reference
is recomputed in float64 from the kernel's own operands:

  values stored in bf16:    |got - ref| <= 2^-7 S + 2e-3 max|ref|      (``bf16_bar``; S = sum of the magnitudes of the
                            separately rounded parts)
  f32 reductions:           |got - ref| <= 2^-14 A + 2^-20 max A       (``f32_bar``; A = the reduction over magnitudes)

Nothing here needs a GPU: the helpers work on tensors of any device, and a test picks the one the reference runs on."""
import numpy as np
import torch

from . import backward as ob
from . import losses as olosses
from . import lovasz as olovasz


def plan_units():
    """The native plan's units in its order (state_dict order, 0 = stem, last = head conv) and its bottleneck blocks."""
    units = [dict(conv='backbone.conv1', bn='backbone.bn1', s=2, p=3, d=1, relu=True)]
    blocks, dil = [], 1
    for li, (nb, stride, dilate) in enumerate(((3, 1, False), (4, 2, False), (6, 1, True), (3, 1, True)), start=1):
        for b in range(nb):
            pre = 'backbone.layer%d.%d.' % (li, b)
            s_ = stride if (b == 0 and not dilate) else 1
            prev = dil
            if b == 0 and dilate:
                dil *= 2
            d2 = prev if b == 0 else dil
            B = dict(c1=len(units), c2=len(units) + 1, c3=len(units) + 2, ds=None)
            units += [dict(conv=pre + 'conv1', bn=pre + 'bn1', s=1, p=0, d=1, relu=True),
                      dict(conv=pre + 'conv2', bn=pre + 'bn2', s=s_, p=d2, d=d2, relu=True),
                      dict(conv=pre + 'conv3', bn=pre + 'bn3', s=1, p=0, d=1, relu=True)]   # ReLU after the residual add
            if b == 0:
                B['ds'] = len(units)
                units.append(dict(conv=pre + 'downsample.0', bn=pre + 'downsample.1', s=s_, p=0, d=1, relu=False))
            blocks.append(B)
    units.append(dict(conv='classifier.0', bn='classifier.1', s=1, p=1, d=1, relu=True))
    return units, blocks, len(units) - 1


def stored_inputs(blocks, head):
    """Where each unit's conv reads its input: 'image' (the bf16 staging image of the stem), 'pool' (the maxpool of the
    stem's y) or the index of the unit whose stored y it is."""
    src, cur = {0: 'image'}, 'pool'
    for B in blocks:
        src[B['c1']], src[B['c2']], src[B['c3']] = cur, B['c1'], B['c2']
        if B['ds'] is not None:
            src[B['ds']] = cur
        cur = B['c3']
    src[head] = cur
    return src


def bf16_bar(S, ref):
    return 2.0 ** -7 * S + 2e-3 * ref.abs().max()


def f32_bar(A):
    return 2.0 ** -14 * A + 2.0 ** -20 * A.max()


class Bars:
    """Worst err / tol per check class.  Failures are collected, not raised at the first one, so that one run on the
    GPU reports every check that fails."""

    def __init__(self):
        self.worst, self.failures, self.controls, self.missed = {}, [], {}, []

    def check(self, cls, what, got, ref, tol):
        got, ref = got.double(), ref.double()
        assert got.shape == ref.shape, (what, got.shape, ref.shape)
        err = (got - ref).abs()
        ratio = err / (tol + 1e-300)
        r = float(ratio.max())
        if cls not in self.worst or r > self.worst[cls][0]:
            self.worst[cls] = (r, what)
        if not r <= 1.0:
            i = int(ratio.argmax())
            idx = np.unravel_index(i, ratio.shape)
            self.failures.append('%s / %s: err/tol %.3g at %s (got %.6g ref %.6g tol %.3g), %d of %d elements out' % (
                cls, what, r, tuple(int(v) for v in idx), float(got.flatten()[i]), float(ref.flatten()[i]),
                float(tol.flatten()[i]) if tol.dim() else float(tol), int((ratio > 1).sum()), ratio.numel()))

    def exact(self, cls, what, got, ref):
        bad = int((got != ref).sum())
        self.worst[cls] = (max(self.worst.get(cls, (0, ''))[0], bad), 'elements that differ')
        if bad:
            self.failures.append('%s / %s: %d of %d elements differ' % (cls, what, bad, got.numel()))

    @staticmethod
    def within(got, ref, tol):
        return bool(((got.double() - ref.double()).abs() <= tol).all())

    def control(self, name, rejected):
        """A deliberately wrong reference that the bars must reject somewhere in the step."""
        self.controls[name] = self.controls.get(name, False) or bool(rejected)

    def control_each(self, name, what, rejected):
        """A deliberately wrong reference that the bars must reject at EVERY site it is applied to (``what``)."""
        self.controls[name] = self.controls.get(name, True) and bool(rejected)
        if not rejected:
            self.missed.append('%s: %s' % (name, what))

    def report(self, tag):
        for cls, (r, what) in sorted(self.worst.items()):
            print('[%s] worst err/tol %-26s %.4f  (%s)' % (tag, cls, r, what))
        for name, rej in sorted(self.controls.items()):
            print('[%s] negative control %-28s %s' % (tag, name, 'rejected' if rej else 'NOT REJECTED'))
        for m in self.missed:
            print('[%s] negative control not rejected at %s' % (tag, m))
        for f in self.failures[:40]:
            print('[%s] FAIL %s' % (tag, f))
        assert not self.failures, '%d checks failed; first: %s' % (len(self.failures), self.failures[0])
        assert all(self.controls.values()), self.controls


def run_step(tr, x, tgt, seed, impl):
    """One ``forward_backward`` with capture on, after the same step with capture off, which must compute the same.
    ``tr``: a fresh ``Trainer``; x: f32 NCHW input on its device; tgt: u8 [N,H,W] on its device; impl: the
    weight-gradient path (0: tcgen05 wgrad_tc and stem_wgrad_tc, 1: mma.sync wgrad_mma and the CUDA-core stem_wgrad)."""
    import ctypes as C
    if tr.lib.nbc_train_set_wgrad_impl(C.c_void_p(tr.handle), impl) != 0:
        raise RuntimeError('nbc_train_set_wgrad_impl failed')
    n_units = tr.lib.nbc_train_num_units(C.c_void_p(tr.handle))
    loss_off = float(tr.forward_backward(x, tgt, seed=seed, update_stats=False))
    zy_off = [tr.debug_tensor(k, u).clone() for u in range(n_units) for k in (0, 1)]
    tr.enable_capture()
    loss = float(tr.forward_backward(x, tgt, seed=seed))
    torch.cuda.synchronize()
    assert loss == loss_off, (loss, loss_off)
    assert all(torch.equal(a, tr.debug_tensor(k, u)) for a, (u, k) in zip(zy_off, [(u, k) for u in range(n_units) for k in (0, 1)]))
    del zy_off
    return loss


def check_head(tr, sd, head_y, head_dy, dropout_p, seed, bars, device='cpu'):
    """Backward of the head from the captured d loss / d full logits: the bicubic adjoint (dlow), the classifier's
    forward (low logits) and weight / bias gradients through the restated dropout mask, and the head unit's dy.
    head_y / head_dy: the head unit's stored y and captured dy as float64 NCHW on ``device``."""
    dims = (0, 2, 3)
    dfull = tr.debug_tensor(4).to(device).double()
    dlow = tr.debug_tensor(5).to(device).double()
    low = tr.debug_tensor(2).to(device).double()
    N, h8, w8 = dlow.shape[0], dlow.shape[-2], dlow.shape[-1]
    wy = ob.bicubic_matrix(h8, dfull.shape[-2], device=device).abs()
    wx = ob.bicubic_matrix(w8, dfull.shape[-1], device=device).abs()
    A = torch.einsum('Yi,ncYX,Xj->ncij', wy, dfull.abs(), wx)
    bars.check('dlow (upsample adjoint)', 'dlow', dlow, ob.upsample_adjoint(dfull, (h8, w8)), f32_bar(A))
    bars.control('adjoint without clamping',
                 not bars.within(dlow, ob.upsample_adjoint(dfull, (h8, w8), clamp=False), f32_bar(A)))
    del dfull, A

    Wc = sd['classifier.4.weight'].view(3, -1).double().to(device)
    bc = sd['classifier.4.bias'].double().to(device)
    yh = head_y
    keep = torch.ones_like(yh, dtype=torch.bool)
    xc = yh
    if dropout_p > 0:
        keep = torch.from_numpy(ob.dropout_keep(seed, yh.numel(), dropout_p)).to(device)
        keep = keep.view(N, h8, w8, -1).permute(0, 3, 1, 2)
        scale = torch.tensor(np.float32(1) / (np.float32(1) - np.float32(dropout_p)))
        xc = torch.where(keep, (yh.float() * scale.to(device)).to(torch.bfloat16).float(), 0.0).double()
        kept = float(keep.double().mean())
        print('dropout p=%.2f: kept fraction %.4f' % (dropout_p, kept))
        assert abs(kept - (1 - dropout_p)) < 0.01
    A = torch.einsum('ck,nkhw->nchw', Wc.abs(), xc.abs()) + bc.abs().view(1, 3, 1, 1)
    bars.check('low logits', 'classifier.4 forward', low, torch.einsum('ck,nkhw->nchw', Wc, xc) + bc.view(1, 3, 1, 1), f32_bar(A))
    g = torch.einsum('nchw,ck->nkhw', dlow, Wc)
    dy = head_dy
    if dropout_p > 0:
        g = torch.where(keep, g * float(scale), 0.0)
        bars.exact('dropped dy(head) == 0', 'classifier.1 dy', dy[~keep], torch.zeros(int((~keep).sum()), device=device).double())
    bars.check('head dy', 'classifier.1 dy', dy, g, bf16_bar(g.abs(), g))
    grads = tr.gradients()
    bars.check('classifier dW db', 'classifier.4.weight', grads['classifier.4.weight'].view(3, -1).to(device),
               torch.einsum('nchw,nkhw->ck', dlow, xc), f32_bar(torch.einsum('nchw,nkhw->ck', dlow.abs(), xc.abs())))
    bars.check('classifier dW db', 'classifier.4.bias', grads['classifier.4.bias'].to(device), dlow.sum(dims),
               f32_bar(dlow.abs().sum(dims)))


def check_loss(tr, tgt, loss, loss_kind, class_weights, bars, device):
    """The loss head at full resolution from the kernel's own low-res logits: the bicubic upsample (full logits), the
    loss value, and -- for the weighted cross-entropy -- its gradient per pixel.

    The Lovasz gradient is not checked here: at millions of pixels it depends on how near-tied errors are ordered, which
    the reference leaves to its sort.  Its value does not (a group of tied errors contributes the same whatever their
    order), so it is compared with a float64 restatement on errors sorted stably in descending order."""
    low = tr.debug_tensor(2).to(device).double()
    full = tr.debug_tensor(3).to(device).double()
    H, W = full.shape[-2:]
    wy = ob.bicubic_matrix(low.shape[-2], H, device=device)
    wx = ob.bicubic_matrix(low.shape[-1], W, device=device)
    A = torch.einsum('Yi,ncij,Xj->ncYX', wy.abs(), low.abs(), wx.abs())
    bars.check('full logits (upsample)', 'full logits', full, ob.upsample_bicubic(low, (H, W)), f32_bar(A))
    bars.control('upsample without clamping', not bars.within(full, torch.einsum(
        'Yi,ncij,Xj->ncYX', ob.bicubic_matrix(low.shape[-2], H, clamp=False, device=device), low,
        ob.bicubic_matrix(low.shape[-1], W, clamp=False, device=device)), f32_bar(A)))
    del A
    t = tgt.to(device).long()
    if loss_kind == 'weighted_ce':
        w = class_weights.to(device).double()
        ref_loss, ref_g = olosses.custom_weighted_cross_entropy_with_grad(full, t, w)
        n = t.numel()
        wp = w[torch.max(full.argmax(1), t)].unsqueeze(1)
        onehot = torch.nn.functional.one_hot(t, 3).permute(0, 3, 1, 2).double()
        A = wp * (torch.softmax(full, 1) + onehot) / n           # magnitudes of w (softmax - onehot) / n
        bars.check('dfull (loss gradient)', 'd weighted CE / d full logits', tr.debug_tensor(4).to(device), ref_g, f32_bar(A))
        ent = torch.nn.functional.cross_entropy(full, t, reduction='none')
        bars.check('loss value', 'weighted CE', torch.tensor(loss, dtype=torch.float64), ref_loss.cpu(),
                   f32_bar((ent * wp[:, 0]).abs().mean().cpu()))
    elif loss_kind == 'lovasz':
        ref_loss, A = olovasz.lovasz_softmax_f64(full, t)
        bars.check('loss value', 'Lovasz-Softmax', torch.tensor(loss, dtype=torch.float64), ref_loss.cpu(), f32_bar(A.cpu()))
    else:
        raise ValueError(loss_kind)
