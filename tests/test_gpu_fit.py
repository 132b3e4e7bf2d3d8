"""Training from a labelled folder on the B200: ragged augmentation with the full pad_resize, whole-image validation and
the ``fit`` entry point."""
import itertools
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import augment as oaug
from oracle import losses as olosses
from oracle import lovasz as olovasz
from oracle import model as omodel
from oracle import postprocess as opost
from oracle import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dual(h, w, seed):
    return (synth.class_mask(h, w, seed).astype(np.float32) * 127.5).astype(np.uint8)


def _sources(shapes, seed):
    return ([synth.texture_u8(h, w, seed + i) for i, (h, w) in enumerate(shapes)],
            [_dual(h, w, seed + 50 + i) for i, (h, w) in enumerate(shapes)])


def _all_combinations(n_sources, crop, target):
    """Every flip x order x jitter (on / off, factors below and above 1) combination; the crop offsets cycle through
    the four corners of the padded frame, so every padded edge is touched, and a few interior offsets."""
    from neuralbarkcalculator_b200 import augment as naug
    corners = [(0, 0), (target[1] - crop, 0), (0, target[0] - crop), (target[1] - crop, target[0] - crop), (37, 101)]
    combos = list(itertools.product((0, 1), (0, 1), (0, 1), (0.0, 0.93, 1.07), (0.0, 0.85, 1.18)))
    p = np.zeros(len(combos), dtype=naug.PARAM_DTYPE)
    for k, (hf, vf, order, b, s) in enumerate(combos):
        x0, y0 = corners[k % len(corners)]
        p[k] = (k % n_sources, x0, y0, hf, vf, order, b, s)
    return p


def _as_dicts(params):
    return [{k: (float(q[k]) if k in ('brightness', 'saturation') else int(q[k])) for k in q.dtype.names} for q in params]


@pytest.mark.parametrize('shapes,target,crop', [
    ([(1024, 1021), (1023, 1021), (612, 1021), (611, 1021), (401, 1021), (343, 1021)], (1024, 1024), 512),
    ([(256, 256), (255, 255), (200, 129), (129, 201), (130, 256)], (256, 256), 128),
])
def test_augment_ragged_vs_oracle(cuda_device, shapes, target, crop):
    """augment_ragged == the reference's torchvision-on-PIL chain (reflect pad, Pillow bilinear resize where a
    difference is odd, jitter, crop, flips, label rounding) bit for bit, images and classes."""
    from neuralbarkcalculator_b200 import augment as naug
    images, duals = _sources(shapes, 7)
    ds = naug.DeviceDataset(images, duals, ['sapin'] * len(images), cuda_device)
    params = _all_combinations(len(images), crop, target)
    out, cls = naug.augment_ragged(ds, params, crop, target)
    ref_i, ref_c = oaug.augment(images, duals, _as_dicts(params), crop, target)
    out, cls = out.cpu().numpy(), cls.cpu().numpy()
    for b in range(len(params)):
        assert np.array_equal(out[b], ref_i[b]), ('image', b, shapes[params['src'][b]], params[b])
        assert np.array_equal(cls[b], ref_c[b]), ('classes', b, shapes[params['src'][b]], params[b])


def test_augment_ragged_uniform_and_rejections(cuda_device):
    from neuralbarkcalculator_b200 import _lib, augment as naug
    images, duals = _sources([(1000, 1024)] * 3, 20)
    ds = naug.DeviceDataset(images, duals, ['sapin'] * 3, cuda_device)
    params = naug.draw_params(np.random.default_rng(3), 8, 3, 384, (1024, 1024))
    a_i, a_c = naug.augment_batch(ds.images, ds.duals, params, 384, (1024, 1024))
    b_i, b_c = naug.augment_ragged(ds, params, 384, (1024, 1024))
    assert torch.equal(a_i, b_i) and torch.equal(a_c, b_c)
    # a source larger than the target, and one whose reflect padding (ceil(176 / 2) = 88 rows) is not narrower than it
    for bad_shape, message in (((300, 256), 'source 1 .* larger than'), ((80, 256), 'source 1 .* not narrower')):
        im, du = _sources([(256, 256), bad_shape], 30)
        bad = naug.DeviceDataset(im, du, ['sapin'] * 2, cuda_device)
        torch.cuda.synchronize()
        before = _lib.launch_count()
        with pytest.raises(RuntimeError, match=message):
            naug.augment_ragged(bad, naug.draw_params(np.random.default_rng(0), 2, 2, 128, (256, 256)), 128, (256, 256))
        assert _lib.launch_count() == before


def _oracle_classes(dual):
    return (torch.from_numpy(dual).float() / 255 * 2).round().long()


def _eval_dataset(device, shapes, seed):
    from neuralbarkcalculator_b200 import augment as naug
    images, duals = _sources(shapes, seed)
    return naug.DeviceDataset(images, duals, ['sapin'] * len(shapes), device), images, duals


# A loss is a sum of non-negative f32 terms (weighted -log p, Lovasz errors x non-negative Jaccard steps) over at most
# 2^21 pixels.  Blocked / pairwise summation of n such terms is within ceil(log2 n) = 21 unit roundoffs (2^-24) of the
# exact sum, relative: 1.3e-6 for the GPU reduction and as much for torch's, plus a few ulps per term for exp / log.
# 1e-5 relative leaves a margin of 3x.
LOSS_REL = 1e-5


def test_evaluate_teacher_forced(cuda_device, synthetic_sd):
    """The rows of evaluate == the oracle's loss / IoU / F1 recomputed from the GPU's own full-resolution logits."""
    from neuralbarkcalculator_b200 import evaluate as nev, utils
    ds, _, duals = _eval_dataset(cuda_device, [(611, 512), (333, 512), (512, 512), (257, 384)], 40)
    idx = [3, 0, 2, 1]
    plan = nev.make_plan(synthetic_sd, cuda_device)
    logits = {i: (full.cpu(), lab.cpu()) for i, full, lab in nev.image_logits(plan, ds, idx, chunk=2)}
    w = utils.get_pos_weight()
    results = {kind: nev.evaluate(synthetic_sd, ds, idx, loss=kind, chunk=2) for kind in nev.LOSSES}
    for kind, res in results.items():
        assert sorted(r['index'] for r in res['rows']) == sorted(idx)
        for r in res['rows']:
            full, lab = logits[r['index']]
            assert torch.equal(lab[0].long(), _oracle_classes(duals[r['index']]))
            lab = lab.long()
            ref = {'weighted_ce': lambda: olosses.custom_weighted_cross_entropy(full, lab, w),
                   'lovasz': lambda: olovasz.lovasz_softmax(full, lab),
                   'mixed': lambda: olovasz.mixed_loss(full, lab, w)}[kind]()
            assert abs(r['loss'] - float(ref)) <= LOSS_REL * abs(float(ref)), (kind, r['index'], r['loss'], float(ref))
            assert r['miou'] == olovasz.miou(full, lab), (kind, r['index'])
            assert np.array_equal(r['f1'], olovasz.pixelwise_f1(full, lab, 'all')), (kind, r['index'])
        assert res['miou'] == np.mean([r['miou'] for r in res['rows']])
        assert res['loss'] == np.mean([r['loss'] for r in res['rows']])
    # the three losses see the same logits: mixed = ce / 4 + lovasz in f32, image by image
    by = {k: {r['index']: r['loss'] for r in v['rows']} for k, v in results.items()}
    for i in idx:
        assert by['mixed'][i] == float(np.float32(by['weighted_ce'][i]) / np.float32(4) + np.float32(by['lovasz'][i]))


def test_evaluate_vs_f32_oracle_forward(cuda_device, trained_like_sd):
    """End to end against the reference's f32 eval-mode forward on ragged odd heights.  The bars follow from the measured
    disagreement, not from tuning: k pixels whose argmax differs move a class's intersection and union by at most k
    each, so |IoU_c - IoU_c'| <= 2k / (U_c - k); after the region removal, k' differing pixels move F1_c = 2tp / (R + P)
    by at most 4k' / (R + P - k').  The Lovasz loss is 1-Lipschitz in the max-norm of its errors, and softmax is
    1/2-Lipschitz from max-norm logits to each probability, so |dloss| <= max|dlogits| / 2 (plus the f32 reduction)."""
    from neuralbarkcalculator_b200 import evaluate as nev, ops
    shapes = [(611, 512), (343, 512)]
    ds, images, duals = _eval_dataset(cuda_device, shapes, 60)
    res = nev.evaluate(trained_like_sd, ds, [0, 1])
    plan = nev.make_plan(trained_like_sd, cuda_device)
    model = omodel.load_model(trained_like_sd)
    rows = {r['index']: r for r in res['rows']}
    for i, full, lab in nev.image_logits(plan, ds, [0, 1]):
        with torch.no_grad():
            ref = model(omodel.normalise_u8(images[i]))
        labels = _oracle_classes(duals[i])[None]
        ours_argmax = ops.argmax3_u8(full)
        ref_argmax = torch.argmax(ref, 1)
        k = int((ours_argmax.cpu().long() != ref_argmax).sum())
        agree = 1 - k / ref_argmax.numel()
        assert agree >= 0.999, agree                               # the north-star bar of the predict path
        cm = olovasz.confusion_matrix(ref_argmax.numpy(), labels.numpy())
        union = cm.sum(0) + cm.sum(1) - np.diag(cm)
        iou_bar = np.mean([100.0 if u <= k else 100.0 * 2 * k / (u - k) for u in union])
        assert abs(rows[i]['miou'] - olovasz.miou(ref, labels)) <= iou_bar + 1e-9, (i, k, iou_bar)
        ours_rsz = ops.remove_small_zones_u8(ours_argmax, 150)[0].cpu().numpy()
        ref_rsz = opost.remove_small_zones_2d(ref_argmax[0].numpy().astype(np.uint8))
        k2 = int((ours_rsz[0] != ref_rsz).sum())
        cm2 = olovasz.confusion_matrix(ref_rsz, labels.numpy())
        assert np.all(cm2.sum(1) > 0)                              # every class labelled: no absent-class rule
        denom = cm2.sum(0) + cm2.sum(1)
        f1_bar = np.array([1.0 if d <= k2 else 4.0 * k2 / (d - k2) for d in denom])
        assert np.all(np.abs(rows[i]['f1'] - olovasz.f1_from_confusion(cm2)) <= f1_bar + 1e-12), (i, k2, f1_bar)
        ref_loss = float(olovasz.lovasz_softmax(ref, labels))
        loss_bar = 0.5 * float((full.cpu() - ref).abs().max()) + LOSS_REL * abs(ref_loss)
        assert abs(rows[i]['loss'] - ref_loss) <= loss_bar, (i, rows[i]['loss'], ref_loss, loss_bar)
        print('image %d: argmax agreement %.5f, |dmiou| %.4f (bar %.4f), |dloss| %.2e (bar %.2e)'
              % (i, agree, abs(rows[i]['miou'] - olovasz.miou(ref, labels)), iou_bar, abs(rows[i]['loss'] - ref_loss), loss_bar))


def test_trainer_evaluate_is_evaluate(cuda_device, synthetic_sd):
    from neuralbarkcalculator_b200 import augment as naug, evaluate as nev
    from neuralbarkcalculator_b200.models import fcn_resnet50
    from neuralbarkcalculator_b200.train import Trainer
    ds, _, _ = _eval_dataset(cuda_device, [(255, 256), (256, 256), (131, 256)], 80)
    tr = Trainer(synthetic_sd, 2, 128, 128, device='cuda:0', loss='lovasz')
    x, t = naug.augment_ragged(ds, naug.draw_params(np.random.default_rng(1), 2, 3, 128, (256, 256)), 128, (256, 256))
    tr.step(x, t)
    a = tr.evaluate(ds, [0, 1, 2])
    sd = tr.state_dict()
    b = nev.evaluate(sd, ds, [0, 1, 2], loss='lovasz')
    model = fcn_resnet50(pretrained=False)
    model.load_state_dict({k: v.cpu() for k, v in sd.items()}, strict=True)
    c = nev.evaluate(model.state_dict(), ds, [0, 1, 2], loss='lovasz')
    for other in (b, c):
        assert other['loss'] == a['loss'] and other['miou'] == a['miou'] and np.array_equal(other['f1'], a['f1'])
        for ra, rb in zip(a['rows'], other['rows']):
            assert ra['index'] == rb['index'] and ra['loss'] == rb['loss'] and ra['miou'] == rb['miou']
            assert np.array_equal(ra['f1'], rb['f1'])


def _make_folder(root):
    """12 labelled items: 10 sapin (split 8 / 1 / 1) and one of each spruce, width 256, odd and even heights."""
    rng = np.random.default_rng(9)
    woods = ['sapin'] * 10 + ['epinette_gelee', 'epinette_non_gelee']
    for k, wood in enumerate(woods):
        h = int(rng.integers(150, 257))
        for sub in ('samples', 'duals'):
            os.makedirs(os.path.join(root, sub, wood), exist_ok=True)
        Image.fromarray(synth.texture_u8(h, 256, 100 + k)).save(os.path.join(root, 'samples', wood, 'img%02d.png' % k))
        Image.fromarray(_dual(h, 256, 200 + k), mode='L').save(os.path.join(root, 'duals', wood, 'img%02d.png' % k))


def test_fit_end_to_end(cuda_device, tmp_path):
    from neuralbarkcalculator_b200 import augment as naug, evaluate as nev, utils
    from neuralbarkcalculator_b200.models import NeuralBarkCalculator
    root = str(tmp_path / 'data')
    _make_folder(root)
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, '-m', 'neuralbarkcalculator_b200.fit', root, '--init', 'random', '--epochs', '2', '--crop', '128',
           '--batch', '2', '--target', '256', '--seed', '3']
    done = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    with open(tmp_path / 'log.tsv') as f:
        lines = [ln.rstrip('\n').split('\t') for ln in f]
    assert lines[0][0] == 'epoch' and [r[0] for r in lines[1:]] == ['1', '2', 'test']
    epochs = lines[1:3]
    for r in epochs:
        assert all(math.isfinite(float(v)) for v in r[1:])
    assert all(math.isfinite(float(v)) for v in lines[3][3:])
    sd = torch.load(tmp_path / 'best_model.pt', map_location='cpu')
    assert len(sd) == 326
    NeuralBarkCalculator(str(tmp_path / 'best_model.pt'), 'cuda:0')          # strict=True load
    # the logged val_miou of the saved epoch == a fresh evaluate of the file on the same split
    best = max(epochs, key=lambda r: float(r[4]))
    np.random.seed(3)
    ds = naug.load_dataset(root, cuda_device)
    _, valid, _, _ = utils.get_splits(ds.split_items(), label_pixels=ds.label_pixels)
    assert nev.evaluate(sd, ds, valid, loss='lovasz')['miou'] == float(best[4])
    # predict.py reads ./best_model.pt
    done = subprocess.run([sys.executable, '-m', 'neuralbarkcalculator_b200.predict', root], cwd=str(tmp_path), env=env,
                          capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    with open(os.path.join(root, 'results', 'final_stats.csv')) as f:
        assert len(f.read().strip().split('\n')) == 13
