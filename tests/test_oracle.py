"""CPU tests: the oracle against the golden fixtures (tests/golden, produced by oracle/make_golden.py from the
reference's own code) and against independent restatements."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import losses as olosses
from oracle import model as omodel
from oracle import pipeline as opipe
from oracle import postprocess as opost
from oracle import preprocess as opre
from oracle import synth


def test_model_matches_reference_golden(golden_dir, synthetic_sd):
    g = np.load(os.path.join(golden_dir, 'model_small.npz'))
    net = omodel.load_model(synthetic_sd)
    x = omodel.normalise_u8(g['image'])
    with torch.no_grad():
        logits = net(x).numpy()
    # golden logits come from the reference's models.fcn_resnet50; CPU conv kernels may differ by round-off only
    assert np.abs(logits - g['logits']).max() < 2e-4
    agree = (logits.argmax(1) == g['mask']).mean()
    assert agree > 0.9995


def test_state_dict_layout(synthetic_sd):
    keys = list(synthetic_sd.keys())
    assert len(keys) == 326
    assert keys[0] == 'backbone.conv1.weight' and keys[-1] == 'classifier.4.bias'
    assert sum(v.numel() for k, v in synthetic_sd.items() if 'num_batches' not in k and 'running' not in k) == 32947779


def test_upsample_restated_vs_torch(golden_dir):
    g = np.load(os.path.join(golden_dir, 'upsample_argmax.npz'))
    up = omodel.upsample_bicubic_restated(g['lowres'], g['up'].shape[-2:])
    assert np.abs(up - g['up']).max() < 5e-6
    mism = omodel.argmax_lowest(up) != g['mask']
    assert mism.mean() < 1e-4
    # non-integer scale (trimmed image: 77 -> 611) and exact 8x
    rng = np.random.default_rng(0)
    for (h, w, H, W) in [(77, 128, 611, 1024), (16, 16, 128, 128)]:
        low = rng.standard_normal((1, 3, h, w)).astype(np.float32)
        ref = torch.nn.functional.interpolate(torch.from_numpy(low), size=(H, W), mode='bicubic', align_corners=False)
        got = omodel.upsample_bicubic_restated(low, (H, W))
        # torch's vectorised CPU kernel rounds the source index differently at non-integer scales (~1e-5)
        assert np.abs(got - ref.numpy()).max() < (5e-5 if H % h else 2e-6)


def test_wce_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'wce_small.npz'))
    loss, grad = olosses.custom_weighted_cross_entropy_with_grad(torch.from_numpy(g['logits']),
                                                                 torch.from_numpy(g['target']).long(),
                                                                 torch.from_numpy(g['weights']))
    assert abs(float(loss) - float(g['loss'])) < 1e-6
    assert np.abs(grad.numpy() - g['grad']).max() < 1e-8


def test_wce_gradient_formula():
    """SURVEY 3.5: dL/dlogit = w * (softmax - onehot) / n, w constant w.r.t. autograd."""
    g = torch.Generator().manual_seed(1)
    logits = torch.randn(1, 3, 8, 9, generator=g)
    target = torch.randint(0, 3, (1, 8, 9), generator=g)
    w = torch.tensor(olosses.DEFAULT_WEIGHTS)
    _, grad = olosses.custom_weighted_cross_entropy_with_grad(logits, target, w)
    sm = torch.softmax(logits, 1)
    onehot = torch.nn.functional.one_hot(target, 3).permute(0, 3, 1, 2).float()
    cw = w[torch.max(logits.argmax(1), target)].unsqueeze(1)
    assert torch.allclose(grad, cw * (sm - onehot) / target.numel(), atol=1e-7)


def test_preprocess_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'preprocess_small.npz'))
    raw = g['raw']
    S = opre.resize4x_S(raw)
    Sc = np.clip(S, 256 * int(raw.min()), 256 * int(raw.max()))
    out = ((Sc + 128) >> 8).astype(np.uint8)
    first, last = opre.trim_rows_from_counts((Sc.sum(-1) >= 66).sum(1), Sc.shape[1], Sc.shape[0])
    assert (first, last) == (int(g['first']), int(g['last']))
    assert np.array_equal(out[first:last], g['out'])


def test_resize4x_equals_general_cubic():
    """The integer 4x filter is the Catmull-Rom cubic sampled at 4i+1.5 (general float64 restatement)."""
    img = synth.texture_u8(64, 96, seed=2)
    S = opre.resize4x_S(img)
    f = opre.resize_general_f64(img, 16, 24)
    lo, hi = float(img.min()), float(img.max())
    assert np.abs(np.clip(S / 256.0, lo, hi) - f).max() < 1e-9


def test_preprocess_full_4096_trim():
    raw, top, bottom = synth.raw_image_u8(seed=5, size=4096, top=803, bottom=402)
    out, first, last = opre.preprocess_u8(raw)
    assert out.shape[1] == 1024 and out.shape[0] == last - first
    assert abs(first - top / 4) <= 1 and abs(last - (1024 - bottom / 4)) <= 1


def test_trim_all_dark_and_non_square():
    img = np.zeros((64, 64, 3), np.uint8)
    out, first, last = opre.preprocess_u8(img)
    assert (first, last) == (0, 64) and out.shape[0] == 64      # nothing kept -> argmax of all False -> full image
    img = synth.texture_u8(40, 64, 1)
    img[:10] = 0
    out, first, last = opre.preprocess_u8(img)
    assert out.shape[0] == 40                                    # not square -> not trimmed (models.py:200)


def test_ccl_golden_and_bruteforce(golden_dir):
    g = np.load(os.path.join(golden_dir, 'ccl_small.npz'))
    assert np.array_equal(opost.remove_small_zones_2d(g['mask']), g['out'])
    rng = np.random.default_rng(3)
    for _ in range(3):
        m = (rng.random((40, 56)) < 0.45).astype(np.uint8) * rng.integers(1, 3, (40, 56)).astype(np.uint8)
        assert np.array_equal(opost.remove_small_zones_2d(m, 12), opost.remove_small_zones_bruteforce(m, 12))


def test_ccl_threshold_is_strict():
    m = np.zeros((40, 40), np.uint8)
    m[2:12, 2:17] = 1          # 150 px: kept (size < 150 is strict)
    m[20:30, 2:17] = 1
    m[29, 16] = 0              # 149 px: removed
    out = opost.remove_small_zones_2d(m)
    assert out[5, 5] == 1 and out[25, 5] == 0


def test_stats_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'stats_small.npz'))
    assert list(g['strings']) == opost.class_stats_strings(g['mask'])


def test_dataset_order_golden(golden_dir, tmp_path):
    g = json.load(open(os.path.join(golden_dir, 'dataset_order.json')))
    from PIL import Image
    for wood, files in g['names'].items():
        os.makedirs(tmp_path / 'samples' / wood)
        for fn in files:
            p = tmp_path / 'samples' / wood / fn
            if fn.endswith('.txt'):
                p.write_text('x')
            else:
                Image.fromarray(np.zeros((4, 4, 3), np.uint8)).save(p, format='BMP' if fn.lower().endswith('bmp') else 'PNG')
    items = [(os.path.relpath(a, tmp_path), b, c) for a, b, c in opipe.make_dataset_for_dir(str(tmp_path))]
    assert items == [tuple(x) for x in g['items']]
    opipe.generate_folders(str(tmp_path))
    dirs = sorted(os.path.relpath(os.path.join(dp, d), tmp_path) for dp, dn, _ in os.walk(tmp_path) for d in dn)
    assert dirs == g['dirs']


def test_bmp_roundtrip(tmp_path):
    img = synth.texture_u8(12, 10, 0)       # width 10 -> row padding
    p = str(tmp_path / 'a.bmp')
    synth.write_bmp(p, img)
    assert np.array_equal(opipe.load_rgb(p), img)


# ------------------------------------------------------------------------------------------------- N1 / N2 (next rows)
def test_lovasz_oracle_matches_golden(golden_dir):
    """oracle/lovasz.py reproduces the values make_golden.py pinned against the reference's own lovasz_losses module."""
    from oracle import lovasz as olovasz
    g = np.load(os.path.join(golden_dir, 'lovasz_small.npz'))
    logits, target = torch.from_numpy(g['logits']), torch.from_numpy(g['target']).long()
    loss, grad = olovasz.lovasz_softmax_with_grad(logits, target)
    assert float(loss) == float(g['loss']) and np.array_equal(grad.numpy(), g['grad'])
    two = target.clone()
    two[two == 2] = 1
    loss2, grad2 = olovasz.lovasz_softmax_with_grad(logits, two)
    assert float(loss2) == float(g['loss_two_classes']) and np.array_equal(grad2.numpy(), g['grad_two_classes'])
    assert np.array_equal(olovasz.iou(logits, target), g['iou'])
    assert np.array_equal(olovasz.confusion_matrix(torch.argmax(logits, 1).numpy(), target.numpy()), g['confusion'])
    from oracle import losses as olosses
    assert float(olovasz.mixed_loss(logits, target, torch.tensor(olosses.DEFAULT_WEIGHTS))) == float(g['mixed'])


def test_lovasz_oracle_properties():
    from oracle import lovasz as olovasz
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(1, 3, 16, 16, generator=g)
    target = torch.randint(0, 3, (1, 16, 16), generator=g)
    # perfect, confident predictions -> loss ~ 0; the loss is bounded by 1; gradient sums to ~0 over the classes
    perfect = torch.nn.functional.one_hot(target, 3).permute(0, 3, 1, 2).float() * 40.0
    assert float(olovasz.lovasz_softmax(perfect, target)) < 1e-6
    loss, grad = olovasz.lovasz_softmax_with_grad(logits, target)
    assert 0.0 < float(loss) <= 1.0 and float(grad.sum(1).abs().max()) < 1e-6
    # F1 from the confusion matrix == sklearn, including the "absent class takes the mean of the others" rule
    from sklearn.metrics import f1_score
    pred = torch.randint(0, 2, (1, 16, 16), generator=g).numpy()
    lab = torch.randint(0, 2, (1, 16, 16), generator=g).numpy()
    cm = olovasz.confusion_matrix(pred, lab)
    sk = f1_score(lab.reshape(-1), pred.reshape(-1), labels=[0, 1, 2], average=None, zero_division=0)
    sk[2] = np.delete(sk, 2).mean()
    assert np.allclose(olovasz.f1_from_confusion(cm), sk)


# ------------------------------------------------------------------------------------------------- N4 augmentation
def test_augment_oracle_and_pil_arithmetic():
    """(1) The arithmetic csrc/augment.cu implements -- PIL's ImageEnhance blend (f32, truncation, clip outside [0,1]) and
    integer luma -- restated in numpy equals torchvision's adjust_brightness / adjust_saturation on PIL images exactly;
    (2) the oracle chain applies the explicit parameters in the reference's order."""
    from PIL import Image
    from torchvision.transforms import functional as TF
    from oracle import augment as oaug
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (48, 40, 3), dtype=np.uint8)
    i64 = img.astype(np.int64)
    L = ((19595 * i64[..., 0] + 38470 * i64[..., 1] + 7471 * i64[..., 2] + 0x8000) >> 16).astype(np.int32)

    def blend(a, v, f):
        t = (a.astype(np.float32) + np.float32(f) * (v.astype(np.int32) - a.astype(np.int32)).astype(np.float32)).astype(np.float32)
        if 0 <= f <= 1:
            return t.astype(np.int32)
        return np.where(t <= 0, 0, np.where(t >= 255, 255, t.astype(np.int32)))
    for f in (0.9, 0.95, 1.0, 1.05, 1.1, 0.8123, 1.1999):
        assert np.array_equal(np.asarray(TF.adjust_brightness(Image.fromarray(img), f)), blend(np.zeros_like(L)[..., None], img, f))
        assert np.array_equal(np.asarray(TF.adjust_saturation(Image.fromarray(img), f)),
                              np.stack([blend(L, img[..., c], f) for c in range(3)], -1))
    dual = (rng.integers(0, 3, (48, 40)) * 127.5).astype(np.uint8)
    p = dict(src=0, x0=3, y0=5, hflip=1, vflip=0, order=0, brightness=0.0, saturation=0.0)
    oi, oc = oaug.augment([img], [dual], [p], crop=16, target_hw=(48, 40))
    assert np.array_equal(oi[0], img[5:21, 3:19][:, ::-1]) and np.array_equal(oc[0], np.round(dual[5:21, 3:19][:, ::-1] / 255.0 * 2))
    # reflect padding (even difference): 44 rows -> 48, two rows mirrored on each side without repeating the edge
    oi, _ = oaug.augment([img[2:46]], [dual[2:46]], [dict(p, x0=0, y0=0, hflip=0)], crop=40, target_hw=(48, 40))
    assert np.array_equal(oi[0][:3], img[2:46][[2, 1, 0]])


# ------------------------------------------------------------------------------------------------- training backward
# oracle/backward.py restates each backward operation of the native training step; tests/test_gpu_train_backward.py
# compares the kernels with these helpers, so each one is pinned here to torch autograd in float64.
@pytest.mark.parametrize('relu', [True, False])
def test_backward_oracle_batchnorm(relu):
    from oracle import backward as ob
    g = torch.Generator().manual_seed(0)
    z = (torch.randn(3, 8, 5, 7, generator=g, dtype=torch.float64) * 2 + 0.5).requires_grad_(True)
    gamma = (torch.rand(8, generator=g, dtype=torch.float64) + 0.5).requires_grad_(True)
    beta = torch.randn(8, generator=g, dtype=torch.float64).requires_grad_(True)
    y = torch.nn.functional.batch_norm(z, None, None, gamma, beta, training=True, eps=1e-5)
    if relu:
        y = y.relu()
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    y.backward(dy)
    ref = ob.bn_backward(dy, y.detach(), z.detach(), gamma.detach(), relu)
    assert torch.allclose(ref['dz'], z.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(ref['dgamma'], gamma.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(ref['dbeta'], beta.grad, rtol=1e-10, atol=1e-12)
    assert (ref['dgamma_abs'] >= ref['dgamma'].abs() - 1e-12).all() and (ref['dbeta_abs'] >= ref['dbeta'].abs() - 1e-12).all()
    # running statistics: torch's update (momentum 0.1, unbiased variance), and the biased variant really differs
    rm, rv = torch.randn(8, generator=g, dtype=torch.float64), torch.rand(8, generator=g, dtype=torch.float64) + 0.5
    m_t, v_t = rm.clone(), rv.clone()
    torch.nn.functional.batch_norm(z.detach(), m_t, v_t, training=True, momentum=0.1)
    m, v = ob.running_stats(z.detach(), rm, rv)
    assert torch.allclose(m, m_t, rtol=1e-12, atol=1e-14) and torch.allclose(v, v_t, rtol=1e-12)
    assert not torch.allclose(ob.running_stats(z.detach(), rm, rv, unbiased=False)[1], v_t, rtol=1e-3)


@pytest.mark.parametrize('H,W', [(9, 13), (8, 12), (1, 2)])
def test_backward_oracle_maxpool_ties(H, W):
    """First-maximum routing on inputs full of ties (a ReLU output quantised to three levels), odd and even sizes."""
    from oracle import backward as ob
    g = torch.Generator().manual_seed(H * 100 + W)
    x = torch.randint(-2, 3, (2, 4, H, W), generator=g).clamp_min(0).double().requires_grad_(True)
    y = torch.nn.functional.max_pool2d(x, 3, 2, 1)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    y.backward(dy)
    # up to four windows add into one input: torch sums them in another order (last-bit differences only)
    assert torch.allclose(ob.maxpool_backward(dy, x.detach()), x.grad, rtol=1e-12, atol=1e-14)
    if H > 1:
        assert not torch.allclose(ob.maxpool_backward(dy, x.detach(), last=True), x.grad)


@pytest.mark.parametrize('h,w,H,W', [(8, 16, 58, 122), (8, 12, 64, 96), (24, 32, 192, 256), (5, 3, 9, 31)])
def test_backward_oracle_bicubic_adjoint(h, w, H, W):
    """The dense interpolation matrices reproduce F.interpolate(bicubic) and its autograd gradient (integer and
    non-integer ratios), and the adjoint satisfies <up(a), b> = <a, adj(b)>."""
    from oracle import backward as ob
    g = torch.Generator().manual_seed(h * w)
    low = torch.randn(2, 3, h, w, generator=g).requires_grad_(True)
    up = torch.nn.functional.interpolate(low, size=(H, W), mode='bicubic', align_corners=False)
    # float32 taps on both sides; torch rounds the source index differently at non-integer scales (~1e-5)
    tol = 5e-5 if (H % h or W % w) else 2e-6
    assert (ob.upsample_bicubic(low.detach(), (H, W)) - up.detach().double()).abs().max() < tol
    dup = torch.randn(up.shape, generator=g)
    up.backward(dup)
    adj = ob.upsample_adjoint(dup, (h, w))
    assert (adj - low.grad.double()).abs().max() < tol * dup.abs().sum((2, 3)).max() / min(h, w)
    a, b = torch.randn(2, 3, h, w, dtype=torch.float64), torch.randn(2, 3, H, W, dtype=torch.float64)
    lhs, rhs = float((ob.upsample_bicubic(a, (H, W)) * b).sum()), float((a * ob.upsample_adjoint(b, (h, w))).sum())
    assert abs(lhs - rhs) < 1e-10 * (abs(lhs) + 1)
    assert (ob.upsample_adjoint(dup, (h, w), clamp=False) - adj).abs().max() > 1e-2


def test_backward_oracle_conv_grads():
    """conv_dgrad / conv_wgrad = autograd of conv2d at the geometries of the network: stride 2 on an odd input,
    dilation, 7x7 stem."""
    from oracle import backward as ob
    g = torch.Generator().manual_seed(0)
    for (H, W, cin, cout, k, s, p, d) in [(15, 31, 8, 16, 3, 2, 1, 1), (15, 31, 8, 16, 1, 2, 0, 1), (8, 16, 8, 8, 3, 1, 4, 4),
                                          (29, 61, 3, 8, 7, 2, 3, 1)]:
        x = torch.randn(2, cin, H, W, generator=g, dtype=torch.float64).requires_grad_(True)
        w = torch.randn(cout, cin, k, k, generator=g, dtype=torch.float64).requires_grad_(True)
        y = torch.nn.functional.conv2d(x, w, stride=s, padding=p, dilation=d)
        dz = torch.randn(y.shape, generator=g, dtype=torch.float64)
        y.backward(dz)
        assert torch.allclose(ob.conv_dgrad(dz, w.detach(), x.shape, s, p, d), x.grad, rtol=1e-10, atol=1e-10)
        assert torch.allclose(ob.conv_wgrad(x.detach(), dz, w.shape, s, p, d), w.grad, rtol=1e-10, atol=1e-10)


def test_backward_oracle_dropout_hash():
    """The restated hash is splitmix64 (published outputs for state 0); the keep fraction is 1 - p and the mask depends
    on the seed."""
    from oracle import backward as ob
    assert [int(v) for v in ob.splitmix64_bits(0, 4)] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F,
                                                           0xF88BB8A8724C81EC]
    k1, k2 = ob.dropout_keep(7, 200000, 0.8), ob.dropout_keep(8, 200000, 0.8)
    assert abs(k1.mean() - 0.2) < 0.005 and (k1 != k2).mean() > 0.2
