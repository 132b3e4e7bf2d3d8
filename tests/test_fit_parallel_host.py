"""Host side of data-parallel ``fit`` (no GPU): which rank runs which samples with which augmentation draws and dropout
seeds, and the sharded validation's merge over two gloo ranks."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from neuralbarkcalculator_b200 import augment, fit, utils
from neuralbarkcalculator_b200 import distributed as nd
from neuralbarkcalculator_b200 import evaluate as nev
from neuralbarkcalculator_b200.train import Trainer, dropout_seed

SEED, BATCH, N_SOURCES, CROP, TARGET = 3, 2, 12, 128, (256, 256)
SPLIT = [0, 2, 3, 5, 6, 7, 8, 10, 11]
WEIGHTS = np.linspace(0.5, 1.5, len(SPLIT)) / np.linspace(0.5, 1.5, len(SPLIT)).sum()


def _schedule(world, accumulate, epochs=2):
    """{(step, global micro-batch j): (params of the micro-batch, dropout seed)} over all ranks, as fit runs them."""
    out, steps = {}, []
    for rank in range(world):
        generator, rng, step = torch.Generator().manual_seed(SEED), np.random.default_rng(SEED), 0
        for _ in range(epochs):
            batches = utils.weighted_epoch_batches(SPLIT, WEIGHTS, world * accumulate * BATCH, generator=generator)
            if rank == 0:
                steps.append(len(batches))
            for row, micro in zip(batches, fit.rank_micro_batches(batches, rng, rank, accumulate, BATCH, N_SOURCES, CROP, TARGET)):
                assert [j for j, _ in micro] == list(range(rank * accumulate, (rank + 1) * accumulate))
                for j, params in micro:
                    assert (step, j) not in out
                    assert np.array_equal(params['src'], row[j * BATCH:(j + 1) * BATCH].numpy())
                    out[(step, j)] = (params, dropout_seed(SEED, j, step))
                step += 1
    return out, steps


def test_micro_batches_do_not_depend_on_the_split_between_ranks_and_accumulation():
    """Every (W, K) with the same W * K gives each global micro-batch the same sources, augmentation parameters and
    dropout seed, and runs every drawn sample exactly once per epoch."""
    runs = {wk: _schedule(*wk) for wk in [(1, 4), (2, 2), (4, 1)]}
    ref, ref_steps = runs[(1, 4)]
    n_steps = sum(ref_steps)
    assert ref_steps == [len(SPLIT) * 12 // (4 * BATCH)] * 2
    assert sorted(ref) == [(s, j) for s in range(n_steps) for j in range(4)]
    for wk, (got, steps) in runs.items():
        assert steps == ref_steps, wk
        assert sorted(got) == sorted(ref), wk
        for key, (params, seed) in got.items():
            assert params.tobytes() == ref[key][0].tobytes() and seed == ref[key][1], (wk, key)
    # one global batch is one draw of G samples: the micro-batches of a step are its consecutive slices
    generator, rng = torch.Generator().manual_seed(SEED), np.random.default_rng(SEED)
    batches = utils.weighted_epoch_batches(SPLIT, WEIGHTS, 4 * BATCH, generator=generator)
    for s, row in enumerate(batches):
        whole = augment.draw_params(rng, 4 * BATCH, N_SOURCES, CROP, TARGET, sources=row.numpy())
        assert np.concatenate([ref[(s, j)][0] for j in range(4)]).tobytes() == whole.tobytes()
    assert len({seed for _, seed in ref.values()}) == len(ref)


def test_one_rank_without_accumulation_makes_the_former_draws():
    """W = 1, K = 1: the batches, augmentation draws and dropout seeds of the one-GPU loop (epoch batches of --batch,
    ``draw_params`` per batch, ``Trainer.dropout_seed`` of rank 0)."""
    got, _ = _schedule(1, 1)
    generator, rng, step = torch.Generator().manual_seed(SEED), np.random.default_rng(SEED), 0
    for _ in range(2):
        for row in utils.weighted_epoch_batches(SPLIT, WEIGHTS, BATCH, generator=generator):
            params = augment.draw_params(rng, BATCH, N_SOURCES, CROP, TARGET, sources=row.numpy())
            assert got[(step, 0)][0].tobytes() == params.tobytes()
            assert got[(step, 0)][1] == (SEED << 40) + (0 << 28) + step
            step += 1
    assert len(got) == step


def test_trainer_dropout_seed_is_the_micro_batch_seed():
    fake = SimpleNamespace(base_seed=5, step_count=17)
    assert Trainer.dropout_seed(fake) == (5 << 40) + 17                 # one process: rank 0
    assert Trainer.dropout_seed(fake, 6) == (5 << 40) + (6 << 28) + 17 == dropout_seed(5, 6, 17)


def test_accumulate_argument():
    assert fit.parse_args(['root', '--init', 'random']).accumulate == 1
    assert fit.parse_args(['root', '--init', 'random', '--accumulate', '3']).accumulate == 3
    for bad in ('0', '-2'):
        with pytest.raises(SystemExit):
            fit.parse_args(['root', '--init', 'random', '--accumulate', bad])


# ---- sharded validation ------------------------------------------------------------------------------------------
def _fake_rows(indices):
    """Per-image rows that depend on the index alone, as ``nbc_eval_ragged``'s do."""
    out = []
    for i in indices:
        r = np.random.default_rng(1000 + i)
        out.append({'index': i, 'loss': float(r.random() * 3), 'miou': float(r.random() * 100), 'f1': r.random(3)})
    return out


def _fake_evaluate_plan(plan, ds, indices, loss='lovasz', class_weights=None, chunk=8):
    """``evaluate_plan`` without the GPU: its row order (widths ascending), its means."""
    assert len(indices) > 0
    return nev.summary(_fake_rows(nev.width_order(ds, indices)))


def _fake_dataset(n):
    widths = np.random.default_rng(n).choice([256, 384, 512], n)
    return SimpleNamespace(sizes=np.stack([np.full(n, 100), widths], 1), device='cpu')


def _sharded_worker(rank, world, port, n_items, indices, out_path):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    nd.init_from_env(device_type='cpu')
    calls = []

    def recording(plan, ds, idx, *a, **k):
        calls.append(list(idx))
        return _fake_evaluate_plan(plan, ds, idx, *a, **k)

    nev.evaluate_plan = recording
    res = nev.evaluate_sharded(None, _fake_dataset(n_items), indices, loss='lovasz')
    torch.save({'res': res, 'calls': calls}, out_path % rank)
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


@pytest.mark.parametrize('n_items,indices', [(23, [7, 3, 19, 0, 12, 5, 22, 1, 9, 14, 18, 2, 11]), (5, [4])])
def test_sharded_validation_equals_one_process(tmp_path, n_items, indices):
    """Over two gloo ranks every rank gets the single-process dict bit for bit: the rows in ``evaluate_plan``'s order
    and the means taken in that order.  With one index, rank 1's shard is empty and it still joins the gather."""
    out = str(tmp_path / 'res%d.pt')
    mp.spawn(_sharded_worker, args=(2, _free_port(), n_items, indices, out), nprocs=2, join=True)
    ref = _fake_evaluate_plan(None, _fake_dataset(n_items), indices)
    got = [torch.load(out % r, weights_only=False) for r in range(2)]
    for g in got:
        res = g['res']
        assert [r['index'] for r in res['rows']] == [r['index'] for r in ref['rows']]
        assert res['loss'] == ref['loss'] and res['miou'] == ref['miou'] and np.array_equal(res['f1'], ref['f1'])
    order = nev.width_order(_fake_dataset(n_items), indices)
    start, end = nd.shard_bounds(len(order), 0, 2)
    assert got[0]['calls'] == [order[start:end]]
    assert got[1]['calls'] == ([order[end:]] if end < len(order) else [])
    # one process: evaluate_sharded is evaluate_plan
    saved = nev.evaluate_plan
    try:
        nev.evaluate_plan = _fake_evaluate_plan
        one = nev.evaluate_sharded(None, _fake_dataset(n_items), indices)
    finally:
        nev.evaluate_plan = saved
    assert [r['index'] for r in one['rows']] == [r['index'] for r in ref['rows']] and one['loss'] == ref['loss']


def test_width_order_is_evaluate_plan_row_order():
    ds = SimpleNamespace(sizes=np.array([[5, 384], [5, 256], [5, 384], [5, 128], [5, 256]]))
    assert nev.width_order(ds, [0, 1, 2, 3, 4]) == [3, 1, 4, 0, 2]
    assert nev.width_order(ds, [4, 2, 3, 1]) == [3, 4, 1, 2]
    assert [i for _, part in nev._width_chunks(ds, [4, 2, 3, 1], 1) for i in part] == [3, 4, 1, 2]
