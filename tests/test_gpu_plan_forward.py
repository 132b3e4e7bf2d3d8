"""Teacher-forced parity of the INFERENCE plan, launch by launch (``pytest -m gpu``).

The plan's forward is otherwise checked only end to end (test_gpu_model.py), after 53 launches of error growth, and its
ragged batches only against single-image runs of the same kernels.  Here the plan stops after step k
(``Plan.set_stop``): every launch up to k is made as in production, programmatic dependent launch included, and no
input of step k is the buffer it writes, so step k's operands and its output are both in the workspace afterwards.
Before each run the workspace is filled with 0xFF bytes -- NaN in bf16 and fp16 -- so a kernel that reads a row nobody
wrote produces NaN and fails.  Each step is then recomputed in float64 from the kernel's OWN stored inputs and the
packed weights of ``ops.fold_bn_pack`` (the fold_pack kernel the plan runs, so the operands are bit-identical).

Bars, each from one operation's arithmetic:
  16-bit conv outputs:  |got - ref| <= 2u |ref| + c A,   c = 2^-14
      u = unit roundoff of the output format (bf16 2^-8, fp16 2^-11): the one rounding of the epilogue, with a factor 2
      of slack.  A = the same launch over magnitudes, conv(|x|, |w|) + |bias| + |residual|: products of 16-bit operands
      are exact in f32, so what remains is the f32 accumulation (and the f32 bias / residual adds), far below 2^-14 A
      for the K <= 18432 terms of these layers, while a wrong tap, row or bias term is a sizeable fraction of A.
  head1x1 (f32 logits):  |got - ref| <= 2^-14 A + 2^-20 max A   (the f32-reduction bar of test_gpu_train_backward.py)
  bit-exact: the stem's staging image ((u8/255 - mean)/std in f32, one rounding; zero border and zero 4th channel),
      maxpool (a max of stored values), the ragged level table (the ceil chain of the clamped heights).
  packed weights (checked once per precision): one 16-bit rounding of the float64 fold, u |ref| + 2^-20 |ref|
      (+ 2^-25 for fp16 subnormals); folded biases 2^-20 (|beta| + |mean scale|).
fp16 stores saturate at +-65504 by design (F2FP.SATFINITE), so the fp16 references are clamped to that range.

Ragged batches: for every step and image, the valid output rows must match the reference of that image alone (input
rows at or beyond its valid height are zero padding) and the next min(4, Ho - vh) rows must be exactly zero -- the
padding the next layer reads.  Rows below those are not checked.

Four deliberately wrong references must FAIL the same bars on the same stored tensors: layer2.0's fused downsample read
from the odd lattice, layer4.1 conv2 with dilation 2 instead of 4, the fused bias without the downsample's, layer1.0
conv2 with its 3x3 taps transposed."""
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model as omodel
from oracle import synth

pytestmark = pytest.mark.gpu

C_ACC = 2.0 ** -14
U16 = {'bf16': 2.0 ** -8, 'fp16': 2.0 ** -11}
DT16 = {'bf16': torch.bfloat16, 'fp16': torch.float16}

DENSE = {
    # odd: 58x122 -> 29x61 -> 15x31 -> 8x16.  layer2's stride-2 convs see an odd input; maxpool windows are cut at the
    # bottom and right edges; Wo = 61 takes the per-window stem (64 x 2 tiles); an 8x16 map is one M tile per image, so
    # the CTA-pair launches of layer3 / layer4 / the head run a phantom tile
    'odd': (3, 58, 122),
    # width 900 (an image <= 1024 px is trimmed, not resized): the stem halo kernel with a partial last tile (450 =
    # 3 x 128 + 66), halo3 with a partial tile (225 px), odd heights at every level (83 -> 42 -> 21 -> 11)
    'w900': (1, 83, 900),
    # production width: every persistent conv loop wraps, the 1/8-resolution layers included (150 M tiles > 148 SMs)
    'wrap': (2, 600, 1024),
}
EXPECTED_LAUNCHES = {0: 53, 2: 56}   # one dense forward: tcgen05 plan (staging + stem + 51), mma.sync plan


class Bars:
    """Worst err / tol per check class; failures are collected, not raised at the first one."""

    def __init__(self):
        self.worst, self.failures, self.controls = {}, [], {}

    def check(self, cls, what, got, ref, tol):
        got, ref = got.double(), ref.double()
        assert got.shape == ref.shape, (what, got.shape, ref.shape)
        if got.numel() == 0:
            return
        ratio = (got - ref).abs() / (tol + 1e-300)
        ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float('inf')), ratio)
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
        self.controls[name] = self.controls.get(name, True) and bool(rejected)

    def report(self, tag):
        for cls, (r, what) in sorted(self.worst.items()):
            print('[%s] worst err/tol %-24s %.4f  (%s)' % (tag, cls, r, what))
        for name, rej in sorted(self.controls.items()):
            print('[%s] negative control %-30s %s' % (tag, name, 'rejected' if rej else 'NOT REJECTED'))
        for f in self.failures[:40]:
            print('[%s] FAIL %s' % (tag, f))
        assert not self.failures, '%d checks failed; first: %s' % (len(self.failures), self.failures[0])
        assert all(self.controls.values()), self.controls


# ---- plan, workspace, step list ---------------------------------------------------------------------------------
def _plan(sd, dev, precision, impl=0):
    import neuralbarkcalculator_b200 as nbc
    m = nbc.fcn_resnet50(pretrained=False)
    m.load_state_dict(sd, strict=True)
    m.to(dev).eval()
    m.set_normalisation(omodel.DEFAULT_MEAN, omodel.DEFAULT_STD)
    m.set_precision(precision)
    plan = m.native_plan()
    plan.set_impl(impl)
    return m, plan


def _workspace(plan, N, H, W):
    """The aligned workspace the plan's forwards use, as a u8 tensor (the offsets of steps() are relative to it)."""
    ptr, nbytes = plan._workspace(N, H, W)
    base = ptr - plan._ws.data_ptr()
    return plan._ws[base:base + nbytes]


def _labels(steps):
    """state_dict prefix of each step's layer (in plan order); checks the plan's layer sequence on the way."""
    blocks = ['backbone.layer%d.%d.' % (li, b) for li, nb in ((1, 3), (2, 4), (3, 6), (4, 3)) for b in range(nb)]
    out, bi = [], -1
    for s in steps:
        n = s['name']
        if n == 'conv1':
            bi += 1
        out.append(blocks[bi] + n if n in ('conv1', 'conv2', 'conv3', 'downsample', 'conv3+downsample') else n)
    assert bi == len(blocks) - 1 and out[:2] == ['stem', 'maxpool'] and out[-2:] == ['head3x3', 'head1x1'], out
    return out


def _conv_keys(label):
    if label == 'stem':
        return 'backbone.conv1', 'backbone.bn1'
    if label == 'head3x3':
        return 'classifier.0', 'classifier.1'
    if label.endswith('downsample'):
        return label + '.0', label + '.1'
    return label, label.replace('.conv', '.bn')


class Weights:
    """Packed 16-bit weights and f32 biases from ops.fold_bn_pack (bit-identical to the plan's), as float64 OIHW."""

    def __init__(self, sd, dev, precision, bars):
        self.sd, self.dev, self.dt, self.u, self.bars = sd, dev, DT16[precision], U16[precision], bars
        self.cache = {}

    def get(self, conv):
        if conv not in self.cache:
            from neuralbarkcalculator_b200 import ops
            bn = conv[:-2] + '.1' if conv.endswith('.0') else conv.replace('conv', 'bn')
            bn = {'backbone.conv1': 'backbone.bn1'}.get(conv, bn)
            w = self.sd[conv + '.weight'].to(self.dev)
            g, b, m, v = [self.sd[bn + s].to(self.dev) for s in ('.weight', '.bias', '.running_mean', '.running_var')]
            wp, bias = ops.fold_bn_pack(w, (g, b, m, v), dtype=self.dt)
            w64 = wp.double().permute(0, 3, 1, 2).contiguous()
            # the fold itself, once: one 16-bit rounding of the float64 fold
            scale = g.double() / torch.sqrt(v.double() + 1e-5)
            ref = w.double() * scale.view(-1, 1, 1, 1)
            tol = (self.u + 2.0 ** -20) * ref.abs() + (2.0 ** -25 if self.dt == torch.float16 else 0.0)
            self.bars.check('fold weights', conv, w64, ref, tol)
            bref = b.double() - m.double() * scale
            self.bars.check('fold bias', conv, bias.double(), bref, 2.0 ** -20 * (b.double().abs() + (m.double() * scale).abs()))
            self.cache[conv] = (w64, bias.double(), bias)
        return self.cache[conv]


# ---- per-step references ----------------------------------------------------------------------------------------
def _t16(ws, off, shape, dt):
    n = int(np.prod(shape)) * 2
    return ws[off:off + n].view(dt).view(*shape)


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


def _zero_rows(t, vh, fill=0.0):
    """t [N,C,H,W]: rows >= vh[n] of image n replaced by `fill` (the conv zero padding of a ragged batch)."""
    if vh is None:
        return t
    rows = torch.arange(t.shape[2], device=t.device).view(1, 1, -1, 1)
    return torch.where(rows >= vh.view(-1, 1, 1, 1), torch.full((), fill, dtype=t.dtype, device=t.device), t)


def _conv(x, w, stride=1, pad=0, dil=1):
    return F.conv2d(x, w, stride=stride, padding=pad, dilation=dil)


def _check16(bars, cls, what, got, ref, A, u, dt, vh=None, halo=True):
    """16-bit output [N,C,Ho,Wo] against ref with the conv bar; ragged: valid rows per image, then the zero halo."""
    if dt == torch.float16:
        ref = ref.clamp(-65504.0, 65504.0)
    tol = 2 * u * ref.abs() + C_ACC * A
    if vh is None:
        bars.check(cls, what, got, ref, tol)
        return
    Ho = got.shape[2]
    for n, v in enumerate(vh.tolist()):
        bars.check(cls, '%s img %d' % (what, n), got[n, :, :v], ref[n, :, :v], tol[n, :, :v])
        if halo:
            z = got[n, :, v:v + min(4, Ho - v)]
            bars.exact('ragged zero halo', '%s img %d' % (what, n), z, torch.zeros_like(z))


def _stem_staging(img_u8, vh, dt, Hp, Wp):
    """Expected staging image [N,Hp,Wp,4]: (u8/255 - mean)/std in f32 (the kernel's IEEE div / sub / div), one rounding,
    3-pixel zero border, zero 4th channel; ragged rows >= vh are zero."""
    x = img_u8.cpu().float()
    mean = torch.tensor(omodel.DEFAULT_MEAN, dtype=torch.float32)
    std = torch.tensor(omodel.DEFAULT_STD, dtype=torch.float32)
    x = ((x / 255.0) - mean) / std
    N, H, W, _ = x.shape
    if vh is not None:
        rows = torch.arange(H).view(1, -1, 1, 1)
        x = torch.where(rows >= vh.cpu().view(-1, 1, 1, 1), torch.zeros(()), x)
    out = torch.zeros((N, Hp, Wp, 4), dtype=dt)
    out[:, 3:3 + H, 3:3 + W, :3] = x.to(dt)
    return out


class Levels:
    """Per-step valid rows of a ragged batch (None for a dense one)."""

    def __init__(self, table):
        self.t = table   # [4, N] int32 on the device, or None

    def __call__(self, level):
        return None if self.t is None or level < 0 else self.t[level].long()


def _check_step(bars, ws, st, label, wts, prec, img_u8, logits, lv, sd):
    """Recompute step st from its stored operands and check its output."""
    dt, u = DT16[prec], U16[prec]
    dev = ws.device
    N, H, W = st['N'], st['H'], st['W']
    kind = st['kind']
    vh_out = lv(st['level'])
    if kind in (0, 5):
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        Hp, Wp = 2 * Ho + 5, 2 * Wo + 6
        w64, b64, _ = wts.get('backbone.conv1')
        if kind == 5:
            stg = _t16(ws, st['x'], (N, Hp, Wp, 4), dt)
            exp = _stem_staging(img_u8, lv(0), dt, Hp, Wp).to(dev)
            if lv.t is None:
                bars.exact('stem staging (bits)', 'staging', stg.view(torch.int16), exp.view(torch.int16))
            else:   # ragged: the staging pass writes padded rows up to vh + 8 (+3 border); the stem reads no further
                for n, v in enumerate(lv(0).tolist()):
                    r = min(Hp, v + 11)
                    bars.exact('stem staging (bits)', 'staging img %d' % n, stg[n, :r].view(torch.int16),
                               exp[n, :r].view(torch.int16))
            x = _zero_rows(_nchw(stg[..., :3]), None if lv.t is None else lv(0) + 3)
            ref = _conv(x, w64, stride=2) + b64.view(1, -1, 1, 1)
            A = _conv(x.abs(), w64.abs(), stride=2) + b64.abs().view(1, -1, 1, 1)
        else:   # CUDA-core stem of the mma.sync plan: f32 normalise + f32 BN-folded weights (float64 fold here)
            x = torch.cat([omodel.normalise_u8(im) for im in img_u8.cpu().numpy()]).to(dev).double()
            g, b, m, v = [sd['backbone.bn1' + s].to(dev).double() for s in ('.weight', '.bias', '.running_mean', '.running_var')]
            scale = g / torch.sqrt(v + 1e-5)
            wf = sd['backbone.conv1.weight'].to(dev).double() * scale.view(-1, 1, 1, 1)
            bf = b - m * scale
            ref = _conv(x, wf, stride=2, pad=3) + bf.view(1, -1, 1, 1)
            A = _conv(x.abs(), wf.abs(), stride=2, pad=3) + bf.abs().view(1, -1, 1, 1)
        got = _nchw(_t16(ws, st['y'], (N, Ho, Wo, 64), dt))
        _check16(bars, 'stem', 'stem', got, ref.relu(), A, u, dt, vh_out)
        return
    if kind == 1:
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        x = _nchw(_t16(ws, st['x'], (N, H, W, 64), dt))
        got = _nchw(_t16(ws, st['y'], (N, Ho, Wo, 64), dt))
        # padding -inf; a ragged image's rows >= its valid height are not part of it
        ref = F.max_pool2d(_zero_rows(x, lv(1), float('-inf')), 3, 2, 1)
        if vh_out is None:
            bars.exact('maxpool', 'maxpool', got, ref)
        else:
            for n, v in enumerate(vh_out.tolist()):
                bars.exact('maxpool', 'maxpool img %d' % n, got[n, :, :v], ref[n, :, :v])
                z = got[n, :, v:v + min(4, Ho - v)]
                bars.exact('ragged zero halo', 'maxpool img %d' % n, z, torch.zeros_like(z))
        return
    if kind == 4:
        x = _nchw(_t16(ws, st['x'], (N, H, W, 512), dt))
        Wc = sd['classifier.4.weight'].to(dev).view(3, -1).double()
        bc = sd['classifier.4.bias'].to(dev).double().view(1, 3, 1, 1)
        x = _zero_rows(x, vh_out)
        ref = torch.einsum('ck,nkhw->nchw', Wc, x) + bc
        A = torch.einsum('ck,nkhw->nchw', Wc.abs(), x.abs()) + bc.abs()
        tol = 2.0 ** -14 * A + 2.0 ** -20 * A.max()
        if vh_out is None:
            bars.check('head1x1 (f32)', 'head1x1', logits, ref, tol)
        else:   # valid rows only: head1x1 writes nothing else
            for n, v in enumerate(vh_out.tolist()):
                bars.check('head1x1 (f32)', 'head1x1 img %d' % n, logits[n, :, :v], ref[n, :, :v], tol[n, :, :v])
        return
    # conv (tcgen05 or mma.sync)
    k, s, p, d = st['k'], st['stride'], st['pad'], st['dil']
    Ho = (H + 2 * p - d * (k - 1) - 1) // s + 1
    Wo = (W + 2 * p - d * (k - 1) - 1) // s + 1
    lvl = st['level']
    vh_in = lv(lvl - 1 if s == 2 else lvl)
    x = _zero_rows(_nchw(_t16(ws, st['x'], (N, H, W, st['Cin']), dt)), vh_in)
    got = _nchw(_t16(ws, st['y'], (N, Ho, Wo, st['Cout']), dt))
    bias_of = lambda b: b.view(1, -1, 1, 1)
    if st['dual']:
        pre = label[:-len('conv3+downsample')]
        w3, b3, b3f = wts.get(pre + 'conv3')
        wd, bd, bdf = wts.get(pre + 'downsample.0')
        s2 = st['stride2']
        x2 = _zero_rows(_nchw(_t16(ws, st['x2'], (N, st['H2'], st['W2'], st['Cin2']), dt)), lv(lvl - 1 if s2 == 2 else lvl))
        bias = (b3f + bdf).double()            # the plan's bias_cat: one f32 add
        main, branch = _conv(x, w3), _conv(x2, wd, stride=s2)
        ref = main + branch + bias_of(bias)
        A = _conv(x.abs(), w3.abs()) + _conv(x2.abs(), wd.abs(), stride=s2) + bias_of(bias.abs())
        _check16(bars, 'conv3+downsample', label, got, ref.relu(), A, u, dt, vh_out)
        if vh_out is not None:
            return
        tol = 2 * u * ref.relu().abs() + C_ACC * A
        if pre == 'backbone.layer2.0.':
            odd = x2[:, :, 1::2, 1::2]
            odd = F.pad(odd, (0, Wo - odd.shape[3], 0, Ho - odd.shape[2]))
            bad = (main + _conv(odd, wd) + bias_of(bias)).relu()
            bars.control('downsample from odd lattice', not Bars.within(got, bad, tol))
        bad = (main + branch + bias_of(b3f.double())).relu()
        bars.control('fused bias without bds', not Bars.within(got, bad, tol))
        return
    conv, _ = _conv_keys(label)
    w64, b64, _ = wts.get(conv)
    ref = _conv(x, w64, s, p, d) + bias_of(b64)
    A = _conv(x.abs(), w64.abs(), s, p, d) + bias_of(b64.abs())
    if st['residual'] >= 0:
        r = _zero_rows(_nchw(_t16(ws, st['residual'], (N, Ho, Wo, st['Cout']), dt)), vh_out)
        ref, A = ref + r, A + r.abs()
    if st['relu']:
        ref = ref.relu()
    cls = 'conv' if kind == 2 else 'conv (mma.sync)'
    _check16(bars, cls, label, got, ref, A, u, dt, vh_out)
    if vh_out is not None:
        return
    tol = 2 * u * ref.abs() + C_ACC * A
    if label == 'backbone.layer4.1.conv2':
        assert d == 4
        bad = (_conv(x, w64, s, 2, 2) + bias_of(b64)).relu()
        bars.control('layer4 conv2 at dilation 2', not Bars.within(got, bad, tol))
    if label == 'backbone.layer1.0.conv2':
        bad = (_conv(x, w64.transpose(2, 3), s, p, d) + bias_of(b64)).relu()
        bars.control('3x3 taps transposed' + (' (halo3)' if st['halo3'] else ''),
                     not Bars.within(got, bad, tol))


def _run_all_steps(plan, fwd, ws, img_u8, sd, dev, prec, bars, levels_ref=None):
    """Full forwards (launch count, determinism), then every step k with the workspace poisoned, then stop = last."""
    from neuralbarkcalculator_b200 import _lib
    full = fwd().clone()
    torch.cuda.synchronize()
    c0 = _lib.launch_count()
    full2 = fwd().clone()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - c0
    steps = plan.steps()
    labels = _labels(steps)
    want = sum(2 if s['kind'] == 5 else 1 for s in steps) + (1 if levels_ref is not None else 0)
    assert launches == want, (launches, want)
    assert torch.equal(full, full2)
    wts = Weights(sd, dev, prec, bars)
    for k, (st, label) in enumerate(zip(steps, labels)):
        ws.fill_(0xFF)
        plan.set_stop(k)
        logits = fwd()
        torch.cuda.synchronize()
        lv = Levels(None)
        if levels_ref is not None:
            N = st['N']
            table = ws[st['levels']:st['levels'] + 16 * N].view(torch.int32).view(4, N)
            bars.exact('level table', 'levels step %d' % k, table.cpu(), levels_ref)
            lv = Levels(table.clone())
        _check_step(bars, ws, st, label, wts, prec, img_u8, logits, lv, sd)
    assert k == len(steps) - 1
    last = fwd().clone()        # stop at the last step: the whole forward
    plan.set_stop(-1)
    assert torch.equal(last, full), 'forward stopped at the last step differs from a full forward'
    return steps, launches


def _dense_input(N, H, W, dev):
    return torch.from_numpy(np.stack([synth.texture_u8(H, W, 70 + i) for i in range(N)])).to(dev)


CASES = [('odd', 'fp16', 0), ('odd', 'bf16', 0), ('odd', 'bf16', 2), ('w900', 'fp16', 0), ('w900', 'bf16', 0),
         ('wrap', 'fp16', 0)]


@pytest.mark.parametrize('case,prec,impl', CASES, ids=['%s-%s-impl%d' % c for c in CASES])
def test_plan_forward_every_step_teacher_forced(cuda_device, synthetic_sd, case, prec, impl):
    """Every launch of a dense forward against its own float64 reference (impl 0: the tcgen05 plan; impl 2: the mma.sync
    cross-check plan with its separate downsample, residual conv3 and CUDA-core stem -- bf16 only)."""
    t0 = time.time()
    N, H, W = DENSE[case]
    m, plan = _plan(synthetic_sd, cuda_device, prec, impl)
    img = _dense_input(N, H, W, cuda_device)
    plan.forward(img)
    ws = _workspace(plan, N, H, W)
    bars = Bars()
    steps, launches = _run_all_steps(plan, lambda: plan.forward(img), ws, img, synthetic_sd, cuda_device, prec, bars)
    assert launches == EXPECTED_LAUNCHES[impl], launches
    tag = '%s %s impl%d' % (case, prec, impl)
    print('\n[%s] %d steps, %d launches per forward, %.1f s' % (tag, len(steps), launches, time.time() - t0))
    bars.report(tag)
    if impl == 0:
        for name in ('fused bias without bds', 'downsample from odd lattice', 'layer4 conv2 at dilation 2'):
            assert name in bars.controls, name
        assert any(n.startswith('3x3 taps transposed') for n in bars.controls)
        if case != 'odd':
            assert '3x3 taps transposed (halo3)' in bars.controls


RAGGED = {
    # heights: h = 1, h = 0 and h > Hc (both clamped), 5 images -> the compact tile map
    'ragged': (5, 120, 1024, [120, 1, 57, 0, 300]),
    # 66 > 64 images: the dense tile numbering with dead tiles skipped
    'ragged66': (66, 40, 64, None),
}


def _ragged_input(N, Hc, W, heights, dev):
    rng = np.random.default_rng(5)
    canvas = rng.integers(0, 256, (N, Hc, W, 3), dtype=np.uint8)     # random bytes below every image
    for i, h in enumerate(heights):
        hv = max(1, min(h, Hc))
        canvas[i, :hv] = synth.texture_u8(hv, W, 90 + i)
    return torch.from_numpy(canvas).to(dev)


def _levels_ref(heights, Hc):
    h = np.clip(np.asarray(heights), 1, Hc)
    rows = [h]
    for _ in range(3):
        h = (h - 1) // 2 + 1
        rows.append(h)
    return torch.from_numpy(np.stack(rows).astype(np.int32))


@pytest.mark.parametrize('case', list(RAGGED))
def test_plan_forward_ragged_every_step_teacher_forced(cuda_device, synthetic_sd, case):
    """Every launch of a ragged forward (fp16): per image, the valid rows against the reference of that image alone,
    the next min(4, Ho - vh) rows exactly zero; the level table against the ceil chain of the clamped heights; the same
    batch through first_last gives the same logits."""
    t0 = time.time()
    N, Hc, W, heights = RAGGED[case]
    if heights is None:
        heights = np.random.default_rng(7).integers(1, Hc + 1, N).tolist()
    m, plan = _plan(synthetic_sd, cuda_device, 'fp16')
    canvas = _ragged_input(N, Hc, W, heights, cuda_device)
    hd = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
    plan.forward_ragged(canvas, heights=hd)
    ws = _workspace(plan, N, Hc, W)
    bars = Bars()
    lref = _levels_ref(heights, Hc)
    steps, launches = _run_all_steps(plan, lambda: plan.forward_ragged(canvas, heights=hd), ws, canvas, synthetic_sd,
                                     cuda_device, 'fp16', bars, levels_ref=lref)
    assert launches == EXPECTED_LAUNCHES[0] + 1, launches     # + the level table
    maps = {s['ragged_map'] for s in steps if s['kind'] in (2, 5)}
    assert maps == ({1} if N <= 64 else {0}), maps
    # the same batch described by K1's {first, last} pairs
    low = plan.forward_ragged(canvas, heights=hd).clone()
    fl = torch.tensor([[7, 7 + h] for h in heights], dtype=torch.int32, device=cuda_device)
    low2 = plan.forward_ragged(canvas, first_last=fl)
    torch.cuda.synchronize()
    bars.exact('level table', 'levels from first_last', ws[steps[0]['levels']:steps[0]['levels'] + 16 * N].view(torch.int32)
               .view(4, N).cpu(), lref)
    assert torch.equal(low, low2)
    print('\n[%s] %d images, heights %s..., %d steps, %.1f s' % (case, N, heights[:8], len(steps), time.time() - t0))
    bars.report(case)


def _tags(st):
    k = st['kind']
    if k == 0:
        return {'stem cuda-core'}
    if k == 5:
        return {'stem halo' if st['stem_halo'] else 'stem per-window'}
    if k == 1:
        return {'maxpool'}
    if k == 4:
        return {'head1x1'}
    if k == 3:
        return {'mma.sync'}
    t = set()
    if st['halo3']:
        t.add('halo3')
    elif st['dual']:
        t.add('dual pair' if st['pair'] else 'dual')
    elif st['pair']:
        t.add('pair%d %dx%d' % (st['block_n'], st['k'], st['k']))
    else:
        t |= {'bn%d' % st['block_n'], 'ob%d' % st['out_bufs'], 'bn%d/ob%d' % (st['block_n'], st['out_bufs'])}
    if st['residual'] >= 0:
        t.add('residual')
    if st['ragged_map'] >= 0:
        t.add('compact map' if st['ragged_map'] else 'dense map')
    return t


def test_plan_forward_variant_coverage(cuda_device, synthetic_sd):
    """The geometries above reach every kernel variant the plan selects today.  If a change to the selection rules drops
    one, this fails instead of leaving it untested."""
    dense, ragged = set(), set()
    _, plan = _plan(synthetic_sd, cuda_device, 'fp16')
    for N, H, W in DENSE.values():
        plan.forward(_dense_input(N, H, W, cuda_device))
        for st in plan.steps():
            dense |= _tags(st)
    for N, Hc, W, heights in RAGGED.values():
        heights = heights or np.random.default_rng(7).integers(1, Hc + 1, N).tolist()
        plan.forward_ragged(_ragged_input(N, Hc, W, heights, cuda_device),
                            heights=torch.tensor(heights, dtype=torch.int32, device=cuda_device))
        for st in plan.steps():
            ragged |= _tags(st)
    torch.cuda.synchronize()
    print('\n[coverage] dense: %s\n[coverage] ragged: %s' % (sorted(dense), sorted(ragged)))
    need = {'stem per-window', 'stem halo', 'halo3', 'bn64', 'bn128', 'bn256', 'ob2', 'ob4', 'pair256 1x1', 'pair256 3x3',
            'dual', 'dual pair', 'residual', 'maxpool', 'head1x1'}
    assert need <= dense, sorted(need - dense)
    assert {'compact map', 'dense map'} <= ragged, sorted(ragged)


def test_plan_stop_hook_defaults(cuda_device, synthetic_sd):
    """stop < 0 is the default and runs the whole list; set_stop(k) runs k + 1 steps' launches."""
    from neuralbarkcalculator_b200 import _lib
    _, plan = _plan(synthetic_sd, cuda_device, 'fp16')
    img = _dense_input(1, 64, 96, cuda_device)
    full = plan.forward(img).clone()
    steps = plan.steps()
    for k, want in ((0, 2), (1, 3), (5, 7)):
        plan.set_stop(k)
        torch.cuda.synchronize()
        c0 = _lib.launch_count()
        plan.forward(img)
        torch.cuda.synchronize()
        assert _lib.launch_count() - c0 == want
    plan.set_stop(-1)
    c0 = _lib.launch_count()
    assert torch.equal(plan.forward(img), full)
    torch.cuda.synchronize()
    assert _lib.launch_count() - c0 == EXPECTED_LAUNCHES[0] == len(steps) + 1
