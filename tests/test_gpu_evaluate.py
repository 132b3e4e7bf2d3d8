"""The batched evaluation on the B200: ``ops.eval_ragged`` output by output against the per-image ops, ``evaluate_plan``
rows against the per-image loop the package used before it, chunk independence, the call's refusals, and the
``python -m neuralbarkcalculator_b200.evaluate`` command end to end (against predict's ``final_stats.csv``, the dual
images and ``fit``'s split, and on two GPUs)."""
import csv
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dual(h, w, seed):
    return (synth.class_mask(h, w, seed).astype(np.float32) * 127.5).astype(np.uint8)


def _low(h):
    return ((((h - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1


def _per_image(low_j, h, w, lab, weights):
    """What the per-image ops give for one image: (wce, lovasz, cm argmax, cm after region removal, counts)."""
    from neuralbarkcalculator_b200 import ops
    full = ops.upsample_bicubic(low_j[:, :, :_low(h)].contiguous(), (h, w))
    ce = ops.wce_fwd_bwd(full, lab, weights, need_grad=False)[0]
    lov = ops.lovasz_softmax_fwd_bwd(full, lab, need_grad=False)[0]
    pred = ops.argmax3_u8(full)
    cm_raw = ops.confusion_matrix(pred, lab).clone()
    pred, counts = ops.remove_small_zones_u8(pred, 150)
    return ce, lov, cm_raw, ops.confusion_matrix(pred, lab), counts[0]


@pytest.mark.parametrize('W,heights', [(384, [5, 611, 1, 96]), (512, [333, 7, 512, 64, 129]), (1024, [343, 1024, 13])])
def test_eval_ragged_matches_per_image_ops(cuda_device, W, heights):
    """Each output equals the per-image ops on that image alone.  Image 0's logits never choose class 2 and its label has
    none (a class absent from label and prediction); image 1's label is one class (the Lovasz present-class rule)."""
    from neuralbarkcalculator_b200 import ops, utils
    g = torch.Generator().manual_seed(W)
    N, Hc = len(heights), max(heights)
    low = torch.randn((N, 3, _low(Hc), _low(W)), generator=g) * 3
    low[0, 2] = -40.0
    labels = torch.zeros((N, Hc, W), dtype=torch.uint8)
    for j, h in enumerate(heights):
        labels[j, :h] = torch.from_numpy(synth.class_mask(h, W, 10 * W + j))
    labels[0] = labels[0].clamp(max=1)
    labels[1, :heights[1]] = 1
    low, labels = low.to(cuda_device), labels.to(cuda_device)
    hs = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
    w = utils.get_pos_weight().to(cuda_device)
    for bits in (1, 2, 3):
        out = ops.eval_ragged(low, hs, labels, w, bits)
        for j, h in enumerate(heights):
            lab = labels[j:j + 1, :h].contiguous()
            ce, lov, cm_raw, cm_rsz, counts = _per_image(low[j:j + 1], h, W, lab, w)
            assert torch.equal(out['cm_raw'][j], cm_raw), (W, h, bits)
            assert torch.equal(out['cm_rsz'][j], cm_rsz), (W, h, bits)
            assert torch.equal(out['counts'][j], counts), (W, h, bits)
            assert float(out['loss_wce'][j]) == (float(ce) if bits & 1 else 0.0), (W, h, bits)
            assert float(out['loss_lovasz'][j]) == (float(lov) if bits & 2 else 0.0), (W, h, bits)
        cm0 = out['cm_raw'][0].cpu().numpy()
        assert cm0[2].sum() == 0 and cm0[:, 2].sum() == 0
        assert out['cm_raw'][1].cpu().numpy()[[0, 2]].sum() == 0


def _net_dataset(device):
    from neuralbarkcalculator_b200 import augment as naug
    shapes = [(5, 384), (611, 512), (13, 512), (257, 384), (100, 1024), (7, 1024), (343, 1024), (1, 512), (64, 512),
              (129, 384), (200, 1024)]
    images = [synth.texture_u8(h, w, 300 + k) for k, (h, w) in enumerate(shapes)]
    duals = [_dual(h, w, 400 + k) for k, (h, w) in enumerate(shapes)]
    duals[3][:] = 127                                       # one label of a single class
    return naug.DeviceDataset(images, duals, ['sapin'] * len(shapes), device)


def _old_rows(plan, ds, idx, loss, chunk):
    """The per-image loop ``evaluate.evaluate`` ran before the batched pass, restated from the per-image ops."""
    from neuralbarkcalculator_b200 import evaluate as nev, ops
    from neuralbarkcalculator_b200.lovasz_losses import iou_from_confusion
    from neuralbarkcalculator_b200.utils import f1_from_confusion, get_pos_weight
    w = get_pos_weight().to(ds.device)
    rows = []
    for i, full, lab in nev.image_logits(plan, ds, idx, chunk):
        zero = torch.zeros((), dtype=torch.float32, device=ds.device)
        ce = ops.wce_fwd_bwd(full, lab, w, need_grad=False)[0] if loss != 'lovasz' else zero
        lov = ops.lovasz_softmax_fwd_bwd(full, lab, need_grad=False)[0] if loss != 'weighted_ce' else zero
        pred = ops.argmax3_u8(full)
        cm_iou = ops.confusion_matrix(pred, lab).cpu().numpy()
        ops.remove_small_zones_u8(pred, 150)
        cm_f1 = ops.confusion_matrix(pred, lab).cpu().numpy()
        ce, lov = ce.cpu().numpy(), lov.cpu().numpy()
        value = {'weighted_ce': ce, 'lovasz': lov, 'mixed': ce / np.float32(4) + lov}[loss]
        rows.append({'index': i, 'loss': float(value), 'miou': float(np.mean(iou_from_confusion(cm_iou))),
                     'f1': f1_from_confusion(cm_f1)})
    return rows


def test_evaluate_plan_rows_equal_the_per_image_loop(cuda_device, synthetic_sd):
    from neuralbarkcalculator_b200 import evaluate as nev
    ds = _net_dataset(cuda_device)
    idx = [4, 0, 9, 1, 3, 7, 2, 5, 10, 6, 8]
    plan = nev.make_plan(synthetic_sd, cuda_device)
    for loss in nev.LOSSES:
        res = nev.evaluate_plan(plan, ds, idx, loss, chunk=3)
        ref = _old_rows(plan, ds, idx, loss, 3)
        assert [r['index'] for r in res['rows']] == [r['index'] for r in ref]
        for a, b in zip(res['rows'], ref):
            assert a['loss'] == b['loss'] and a['miou'] == b['miou'], (loss, a['index'])
            assert np.array_equal(a['f1'], b['f1']), (loss, a['index'])
        assert res['loss'] == float(np.mean([r['loss'] for r in ref]))
        assert res['miou'] == float(np.mean([r['miou'] for r in ref]))
    # the single-class label: Lovasz over the present class only
    row3 = [r for r in nev.evaluate_plan(plan, ds, [3], 'lovasz')['rows']][0]
    assert row3['cm_rsz'][[0, 2]].sum() == 0


def test_evaluate_plan_chunk_independence(cuda_device, synthetic_sd):
    from neuralbarkcalculator_b200 import evaluate as nev
    ds = _net_dataset(cuda_device)
    plan = nev.make_plan(synthetic_sd, cuda_device)
    # the network takes canvases of 16 rows or more: an image below that is scored only in a chunk with a taller one
    tall = [i for i in range(len(ds)) if ds.sizes[i, 0] >= 16]
    for idx, chunks in ((tall, (1, 3, 16)), (list(range(len(ds))), (3, 16))):
        _same_rows([nev.evaluate_plan(plan, ds, idx, 'mixed', chunk=c) for c in chunks])


def _same_rows(runs):
    for other in runs[1:]:
        assert other['loss'] == runs[0]['loss'] and other['miou'] == runs[0]['miou']
        for a, b in zip(runs[0]['rows'], other['rows']):
            assert a['index'] == b['index'] and a['loss'] == b['loss'] and a['miou'] == b['miou']
            for k in ('f1', 'iou', 'cm_rsz', 'counts'):
                assert np.array_equal(a[k], b[k]), (k, a['index'])


def test_eval_ragged_refusals_launch_nothing(cuda_device):
    from neuralbarkcalculator_b200 import _lib
    lib = _lib.load()
    N, Hc, W = 2, 40, 64
    low = torch.zeros((N, 3, _low(Hc), _low(W)), device=cuda_device)
    labels = torch.zeros((N, Hc, W), dtype=torch.uint8, device=cuda_device)
    w = torch.ones(3, device=cuda_device)
    outs = [torch.empty(64, dtype=torch.int64, device=cuda_device) for _ in range(5)]
    need = lib.nbc_eval_workspace_bytes(N, Hc, W)
    ws = torch.empty(need, dtype=torch.uint8, device=cuda_device)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())          # noqa: E731

    def call(n, hc, wd, heights, ws_bytes):
        hs = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
        torch.cuda.synchronize()
        before = _lib.launch_count()
        rc = lib.nbc_eval_ragged(p(low), n, hc, wd, p(hs), p(labels), p(w), 3, *[p(o) for o in outs], p(ws), ws_bytes, stream)
        torch.cuda.synchronize()
        return rc, _lib.launch_count() - before, _lib.last_error()

    rc, launches, _ = call(N, Hc, W, [40, 17], need)
    assert rc == 0 and launches > 0
    for n, hc, wd, heights, ws_bytes, what in [
            (0, Hc, W, [40, 17], need, 'N must be at least 1'),
            (N, Hc, W, [0, 17], need, 'outside'),
            (N, Hc, W, [40, 41], need, 'outside'),
            (N, Hc, W, [-3, 17], need, 'outside'),
            (N, Hc, W, [40, 17], need - 1, 'workspace'),
            (1, 1 << 15, 1 << 15, [1], need, 'below 2^31')]:
        rc, launches, err = call(n, hc, wd, heights, ws_bytes)
        assert rc != 0 and launches == 0 and what in err, (n, hc, wd, heights, ws_bytes, err)
    assert lib.nbc_eval_workspace_bytes(1, 1 << 15, 1 << 15) == 0


def _make_folder(root, woods, seed, widths=(256, 384, 512, 1024)):
    rng = np.random.default_rng(seed)
    for k, wood in enumerate(woods):
        h, w = int(rng.integers(150, 420)), int(widths[k % len(widths)])
        for sub in ('samples', 'duals'):
            os.makedirs(os.path.join(root, sub, wood), exist_ok=True)
        Image.fromarray(synth.texture_u8(h, w, 500 + k)).save(os.path.join(root, 'samples', wood, 'im%02d.png' % k))
        Image.fromarray(_dual(h, w, 600 + k), mode='L').save(os.path.join(root, 'duals', wood, 'im%02d.png' % k))


def _run(args, cwd, timeout=900):
    env = dict(os.environ, PYTHONPATH=ROOT)
    done = subprocess.run(args, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    assert done.returncode == 0, done.stderr[-3000:]
    return done


def _read_tsv(path):
    with open(path) as f:
        return [ln.rstrip('\n').split('\t') for ln in f]


WOODS = ['sapin'] * 10 + ['epinette_gelee'] * 2 + ['epinette_non_gelee'] * 2


@pytest.fixture(scope='module')
def labelled(tmp_path_factory, synthetic_sd):
    base = tmp_path_factory.mktemp('evalcli')
    root = str(base / 'data')
    _make_folder(root, WOODS, 11)
    torch.save(synthetic_sd, str(base / 'best_model.pt'))
    return str(base), root


def test_cli_against_predict_and_labels(cuda_device, labelled):
    from neuralbarkcalculator_b200.augment import label_classes
    from neuralbarkcalculator_b200.dataset import make_dataset, pil_loader
    from neuralbarkcalculator_b200.evaluate import HEADER
    base, root = labelled
    items = make_dataset(root)
    for exclude in (False, True):
        flag = ['--exclude_nodes'] if exclude else []
        _run([sys.executable, '-m', 'neuralbarkcalculator_b200.predict', root] + flag, base)
        for path, _, fname, wood in items:         # predict ran the images untrimmed: the stats are of the same pixels
            proc = np.asarray(Image.open(os.path.join(root, 'processed', 'samples', wood, fname)).convert('RGB'))
            assert np.array_equal(proc, pil_loader(path)), fname
        out = os.path.join(base, 'eval%d.tsv' % exclude)
        _run([sys.executable, '-m', 'neuralbarkcalculator_b200.evaluate', root, '--model', 'best_model.pt', '--chunk', '3',
              '--block', '5', '--out', out] + flag, base)
        rows = _read_tsv(out)
        with open(os.path.join(root, 'results', 'final_stats.csv')) as f:
            stats = list(csv.reader(f, delimiter='\t'))[1:]
        assert rows[0] == HEADER and len(rows) == len(items) + 2 and rows[-1][0] == 'mean'
        body = rows[1:-1]
        assert [(r[0], r[1]) for r in body] == [(f, w) for _, _, f, w in items] == [(s[0], s[1]) for s in stats]
        for r, s, (_, t, _, _) in zip(body, stats, items):
            assert (r[13], r[15]) == (s[2], s[4]), (r[0], exclude)      # data rows: name, type, bark %, area, node %, area
            cls = label_classes(pil_loader(t, grayscale=True))
            n = np.bincount(cls.ravel(), minlength=3).astype(np.int64)
            if exclude:
                n = np.array([n[0], n[1] + n[2], 0])
            assert [int(r[2]), int(r[3])] == list(cls.shape)
            pct = ['{:.5f}'.format(np.float32(n[c]) / np.float32(cls.size) * np.float32(100)) for c in (1, 2)]
            assert (r[12], r[14]) == tuple(pct), (r[0], exclude)
        metrics = np.array([[float(v) for v in r[4:12]] for r in body])
        assert [float(v) for v in rows[-1][4:12]] == list(metrics.mean(0))
        assert float(rows[-1][13]) == pytest.approx(np.mean([abs(float(r[12]) - float(r[13])) for r in body]), abs=1e-5)


def test_cli_split_is_fits_split(cuda_device, labelled, synthetic_sd):
    from neuralbarkcalculator_b200 import augment as naug, evaluate as nev, utils
    base, root = labelled
    out = os.path.join(base, 'valid.tsv')
    _run([sys.executable, '-m', 'neuralbarkcalculator_b200.evaluate', root, '--model', 'best_model.pt', '--split', 'valid',
          '--seed', '5', '--loss', 'mixed', '--out', out], base)
    rows = _read_tsv(out)[1:-1]
    np.random.seed(5)
    ds = naug.load_dataset(root, cuda_device)
    _, valid, _, _ = utils.get_splits(ds.split_items(), label_pixels=ds.label_pixels)
    valid = sorted(int(i) for i in valid)
    assert len(valid) >= 1 and [r[0] for r in rows] == [ds.fnames[i] for i in valid]
    ref = {r['index']: r for r in nev.evaluate(synthetic_sd, ds, valid, loss='mixed')['rows']}
    for r, i in zip(rows, valid):
        assert r[4] == repr(ref[i]['loss']) and r[8] == repr(ref[i]['miou'])
        assert r[9:12] == [repr(float(v)) for v in ref[i]['f1']]


def test_cli_two_gpus_match_one(cuda_device, labelled):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    base, root = labelled
    one, two = os.path.join(base, 'one.tsv'), os.path.join(base, 'two.tsv')
    _run([sys.executable, '-m', 'neuralbarkcalculator_b200.evaluate', root, '--model', 'best_model.pt', '--out', one], base)
    _run([sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', '2', '-m',
          'neuralbarkcalculator_b200.evaluate', root, '--model', 'best_model.pt', '--block', '3', '--out', two], base)
    with open(one, 'rb') as f1, open(two, 'rb') as f2:
        assert f1.read() == f2.read()
