"""CPU tests of the evaluation command's host side: argument refusals, the percentage columns against predict's
``_stats_strings``, the IoU / F1 columns against their definitions, and split + shard + merge order over two gloo ranks."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from PIL import Image

from neuralbarkcalculator_b200 import distributed as nd
from neuralbarkcalculator_b200 import evaluate as nev
from neuralbarkcalculator_b200.augment import label_classes
from neuralbarkcalculator_b200.dataset import make_dataset
from neuralbarkcalculator_b200.lovasz_losses import iou_from_confusion
from neuralbarkcalculator_b200.models import NeuralBarkCalculator, fcn_resnet50
from neuralbarkcalculator_b200.utils import f1_from_confusion, get_splits

WOODS = ['sapin'] * 10 + ['epinette_gelee'] * 3 + ['epinette_non_gelee']


def _folder(root, woods=WOODS, drop_dual=None):
    rng = np.random.default_rng(4)
    for k, wood in enumerate(woods):
        h, w = int(rng.integers(9, 20)), int(rng.integers(9, 20))
        for sub in ('samples', 'duals'):
            os.makedirs(os.path.join(root, sub, wood), exist_ok=True)
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(os.path.join(root, 'samples', wood, 'i%02d.png' % k))
        if k != drop_dual:
            dual = rng.choice(np.array([0, 127, 255], dtype=np.uint8), (h, w), p=[0.5, 0.3, 0.2])
            Image.fromarray(dual, mode='L').save(os.path.join(root, 'duals', wood, 'i%02d.png' % k))


def _keys_only_sd(path, drop=0):
    """A file with fcn_resnet50's state_dict keys (tiny tensors: only the key set is checked before the GPU is used)."""
    with torch.device('meta'):
        keys = list(fcn_resnet50(pretrained=False).state_dict().keys())
    torch.save({k: torch.zeros(1) for k in keys[drop:]}, path)


@pytest.mark.parametrize('argv', [['r', '--device', 'cpu'], ['r', '--chunk', '0'], ['r', '--block', '0'],
                                  ['r', '--split', 'holdout'], ['r', '--loss', 'dice']])
def test_argument_refusals(argv, capsys):
    with pytest.raises(SystemExit) as e:
        nev.parse_args(argv)
    assert e.value.code == 2 and capsys.readouterr().err


def test_folder_and_checkpoint_refusals(tmp_path):
    root = str(tmp_path / 'data')
    _folder(root, drop_dual=3)
    good = str(tmp_path / 'good.pt')
    _keys_only_sd(good)
    with pytest.raises(RuntimeError, match='no dual image'):
        nev.main(nev.parse_args([root, '--model', good]))
    root2 = str(tmp_path / 'data2')
    _folder(root2)
    bad = str(tmp_path / 'bad.pt')
    _keys_only_sd(bad, drop=1)
    with pytest.raises(RuntimeError, match='326 keys'):
        nev.main(nev.parse_args([root2, '--model', bad]))
    with pytest.raises(RuntimeError, match='no such file'):
        nev.main(nev.parse_args([root2, '--model', str(tmp_path / 'none.pt')]))
    root3 = str(tmp_path / 'data3')
    _folder(root3, woods=['sapin'] * 3 + ['epinette_gelee', 'epinette_non_gelee'])    # floor(0.3) = floor(0.1) = 0 validation items
    with pytest.raises(RuntimeError, match='split .* is empty'):
        nev.main(nev.parse_args([root3, '--model', good, '--split', 'valid']))
    with pytest.raises(RuntimeError, match='no images'):
        os.makedirs(str(tmp_path / 'empty' / 'samples'))
        nev.main(nev.parse_args([str(tmp_path / 'empty'), '--model', good]))


def test_percent_rows_match_stats_strings():
    rng = np.random.default_rng(0)
    stub = types.SimpleNamespace(mm_per_pix=0.0123)
    for h, w in [(343, 1024), (1, 7), (600, 384), (1024, 1024)]:
        for _ in range(20):
            n = h * w
            counts = rng.multinomial(n, rng.dirichlet([1, 1, 1]))
            cm = rng.multinomial(n, rng.dirichlet(np.ones(9))).reshape(3, 3)
            pr = nev.percent_rows(cm, counts, h, w)
            ref_out = NeuralBarkCalculator._stats_strings(stub, counts.tolist(), n)
            ref_lab = NeuralBarkCalculator._stats_strings(stub, cm.sum(1).tolist(), n)
            assert pr == [ref_lab[0], ref_out[0], ref_lab[2], ref_out[2]]
            # --exclude_nodes: predict's counts after its node rewrite are (c0, c1 + c2, 0); labels fold the same way
            folded = nev.percent_rows(cm, counts, h, w, exclude_nodes=True)
            ref_out = NeuralBarkCalculator._stats_strings(stub, [counts[0], counts[1] + counts[2], 0], n)
            lab = cm.sum(1)
            ref_lab = NeuralBarkCalculator._stats_strings(stub, [lab[0], lab[1] + lab[2], 0], n)
            assert folded == [ref_lab[0], ref_out[0], ref_lab[2], ref_out[2]]
            assert folded[2] == folded[3] == '0.00000'


def test_metric_columns_and_mean_row():
    cms = [np.array([[5, 1, 0], [2, 7, 0], [0, 0, 0]]),          # class 2 absent from label and prediction
           np.array([[0, 0, 0], [0, 9, 0], [0, 0, 0]]),          # a single class
           np.array([[3, 0, 1], [0, 0, 2], [1, 1, 4]])]
    rows = []
    for k, cm in enumerate(cms):
        cm_rsz = cm[::-1, ::-1].copy()
        r = nev.image_row(k, 'mixed', np.float32(0.5 + k), np.float32(0.25), cm, cm_rsz, cm_rsz.sum(0))
        assert r['loss'] == float(np.float32(0.5 + k) / np.float32(4) + np.float32(0.25))
        assert np.array_equal(r['iou'], iou_from_confusion(cm)) and r['miou'] == float(np.mean(iou_from_confusion(cm)))
        assert np.array_equal(r['f1'], f1_from_confusion(cm_rsz))
        line = nev.table_row('img%d.png' % k, 'sapin', 3, 3 + k, r)
        assert len(line) == len(nev.HEADER)
        assert [float(v) for v in line[5:8]] == list(iou_from_confusion(cm))
        assert [float(v) for v in line[9:12]] == list(f1_from_confusion(cm_rsz))
        assert line[:4] == ['img%d.png' % k, 'sapin', '3', str(3 + k)]
        rows.append(line)
    mean = nev.mean_row(rows)
    assert len(mean) == len(nev.HEADER) and mean[0] == 'mean'
    for c in range(4, 12):
        assert float(mean[c]) == float(np.mean([float(r[c]) for r in rows]))
    assert mean[13] == '{:.5f}'.format(np.mean([abs(float(r[12]) - float(r[13])) for r in rows]))


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _split_worker(rank, world, port, root, out_path):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    nd.init_from_env(device_type='cpu')
    items = make_dataset(root)
    if rank == 1:
        np.random.seed(12345)            # only rank 0's generator decides the split
    selected = nev.select_items(items, 'train', 7)
    start, end = nd.shard_bounds(len(selected), rank, world)
    rows = [[items[i][2], items[i][3], str(i)] for i in selected[start:end]]
    merged = nd.merge_rows(rows, start, len(selected))
    if rank == 0:
        torch.save({'selected': selected, 'merged': merged}, out_path)
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_split_shard_merge_two_ranks(tmp_path):
    root = str(tmp_path / 'data')
    _folder(root)
    out = str(tmp_path / 'out.pt')
    mp.spawn(_split_worker, args=(2, _free_port(), root, out), nprocs=2, join=True)
    got = torch.load(out)
    items = make_dataset(root)
    # fit's split: np.random.seed(seed), then get_splits scanning the class maps of the dual images itself
    np.random.seed(7)
    classes = [torch.from_numpy(label_classes(np.asarray(Image.open(t).convert('L')))) for _, t, _, _ in items]
    train, valid, test, _ = get_splits([(None, c, f, w) for c, (_, _, f, w) in zip(classes, items)])
    assert got['selected'] == sorted(int(i) for i in train)
    assert got['merged'] == [[items[i][2], items[i][3], str(i)] for i in sorted(int(i) for i in train)]
    assert nev.select_items(items, 'all', 0) == list(range(len(items)))
    np.random.seed(99)
    assert nev.select_items(items, 'valid', 7) == sorted(int(i) for i in valid)
    assert nev.select_items(items, 'test', 7) == sorted(int(i) for i in test)
