"""Gradient accumulation in the training step and data-parallel ``fit`` on the B200: accumulated micro-batches sum in one
gradient buffer, ``fit --accumulate`` trains end to end, and a two-GPU ``fit`` under torchrun is the one-GPU training
with the same global batch (the two-GPU tests skip on a one-GPU box)."""
import ctypes as C
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth

from test_gpu_fit import _make_folder

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))


def _micro_batch(dev, N, H, W, j):
    return (torch.from_numpy(np.stack([synth.texture_u8(H, W, 10 * j + i) for i in range(N)])).to(dev),
            torch.from_numpy(np.stack([synth.class_mask(H, W, 50 + 10 * j + i) for i in range(N)])).to(dev))


def _segment_errors(tr, got, want):
    from neuralbarkcalculator_b200.train import gradient_segments
    return [((got[o:o + c] - want[o:o + c]).norm() / (want[o:o + c].norm() + 1e-30)).item()
            for o, c in gradient_segments(tr.lib, tr.handle)]


def test_accumulated_micro_batches_sum_in_one_buffer(cuda_device, synthetic_sd):
    """K = 3 accumulated micro-batches: the buffer holds the sum of three separate gradients of the same inputs and seeds
    (within the atomic-order noise of the weight-gradient kernels: relative 1e-3 per segment, as the NCCL worker), the
    losses are bit-identical, the BatchNorm statistics are updated three times, and Adam applies 1/3.  Then
    accumulate=False overwrites the buffer again."""
    from neuralbarkcalculator_b200.train import Trainer, dropout_seed
    N, H, W, K = 2, 64, 96, 3
    tr = Trainer(synthetic_sd, N, H, W, device='cuda:0', loss='lovasz', seed=4)
    data = [_micro_batch(cuda_device, N, H, W, j) for j in range(K)]
    seeds = [dropout_seed(4, j, 0) for j in range(K)]
    stats0 = tr.stats.clone()
    losses, grads, once = [], [], None
    for (x, t), s in zip(data, seeds):
        losses.append(tr.forward_backward(x, t, seed=s).clone())
        grads.append(tr.grads.clone())
        once = tr.stats.clone() if once is None else once
    separate_stats = tr.stats.clone()
    tr.stats.copy_(stats0)
    tracked = dict(tr.num_batches_tracked)
    acc_losses = [tr.forward_backward(x, t, seed=s, accumulate=i > 0).clone() for i, ((x, t), s) in enumerate(zip(data, seeds))]
    torch.cuda.synchronize()
    assert tr.micro_batches == K
    assert all(torch.equal(a, b) for a, b in zip(acc_losses, losses)), [(float(a), float(b)) for a, b in zip(acc_losses, losses)]
    assert torch.equal(tr.stats, separate_stats) and not torch.equal(tr.stats, once)
    assert all(tr.num_batches_tracked[k] == v + K for k, v in tracked.items())
    total = grads[0] + grads[1] + grads[2]
    errs = _segment_errors(tr, tr.grads, total)
    assert max(errs) <= 1e-3, errs
    assert max(_segment_errors(tr, grads[2], total)) > 0.1          # the sum, not the last micro-batch
    # Adam on the mean of the three: grad_scale 1/3 (one process)
    ref_p, m, v = tr.params.clone(), torch.zeros_like(tr.params), torch.zeros_like(tr.params)
    acc = tr.grads.clone()
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    assert tr.lib.nbc_train_adam(ptr(ref_p), ptr(acc), ptr(m), ptr(v), ref_p.numel(), C.c_float(tr.lr), C.c_float(tr.betas[0]),
                                 C.c_float(tr.betas[1]), C.c_float(tr.eps), C.c_float(tr.wd), 1, C.c_float(1.0 / K),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    tr.optimizer_step()
    torch.cuda.synchronize()
    assert torch.equal(tr.params, ref_p) and tr.micro_batches == 0
    # accumulate=False after the accumulated step: a fresh gradient of the new weights, not added to the old sum
    x, t = data[0]
    tr.forward_backward(x, t, seed=seeds[0])
    fresh = Trainer(tr.state_dict(), N, H, W, device='cuda:0', loss='lovasz')
    fresh.forward_backward(x, t, seed=seeds[0])
    torch.cuda.synchronize()
    assert tr.micro_batches == 1
    errs = _segment_errors(tr, tr.grads, fresh.grads)
    assert max(errs) <= 1e-3, errs


def _log_rows(path):
    with open(path) as f:
        return [ln.rstrip('\n').split('\t') for ln in f]


def _split(root, seed, device):
    from neuralbarkcalculator_b200 import augment as naug, utils
    np.random.seed(seed)
    ds = naug.load_dataset(root, device)
    train, valid, test, _ = utils.get_splits(ds.split_items(), label_pixels=ds.label_pixels)
    return ds, train, valid, test


def _check_checkpoint_and_log(tmp_path, root, steps_per_epoch, micro_per_step, epochs=2):
    """One log and one checkpoint; the best epoch's val_* columns equal, bit for bit, a one-GPU evaluate of the saved
    checkpoint, whose BatchNorm counters hold the micro-batches run up to that epoch.  Returns the log rows."""
    from neuralbarkcalculator_b200 import evaluate as nev
    lines = _log_rows(tmp_path / 'log.tsv')
    assert lines[0][0] == 'epoch' and [r[0] for r in lines[1:]] == [str(e) for e in range(1, epochs + 1)] + ['test']
    rows = lines[1:epochs + 1]
    for r in rows:
        assert all(math.isfinite(float(v)) for v in r[1:])
    sd = torch.load(tmp_path / 'best_model.pt', map_location='cpu')
    assert len(sd) == 326
    best = max(rows, key=lambda r: float(r[4]))
    ds, _, valid, test = _split(root, 3, 'cuda:0')
    res = nev.evaluate(sd, ds, valid, loss='lovasz')
    assert [repr(res['loss']), repr(res['miou'])] + [repr(float(v)) for v in res['f1']] == best[3:8]
    assert int(sd['backbone.bn1.num_batches_tracked']) == int(best[0]) * steps_per_epoch * micro_per_step
    test_res = nev.evaluate(sd, ds, test, loss='lovasz')
    assert [repr(test_res['loss']), repr(test_res['miou'])] + [repr(float(v)) for v in test_res['f1']] == lines[-1][3:8]
    return lines


def _fit_cmd(root, *extra):
    return ['-m', 'neuralbarkcalculator_b200.fit', root, '--init', 'random', '--epochs', '2', '--crop', '128', '--target',
            '256', '--seed', '3'] + list(extra)


def _epoch_steps(stdout):
    return [int(ln.split(': ')[2].split()[0]) for ln in stdout.splitlines() if ln.startswith('fit: epoch ')]


def test_fit_accumulate_end_to_end(cuda_device, tmp_path):
    """fit --accumulate 2 --batch 1: trains, logs the figures of its checkpoint, and predict loads that checkpoint."""
    from neuralbarkcalculator_b200.models import NeuralBarkCalculator
    root = str(tmp_path / 'data')
    _make_folder(root)
    env = dict(os.environ, PYTHONPATH=ROOT)
    done = subprocess.run([sys.executable] + _fit_cmd(root, '--batch', '1', '--accumulate', '2'), cwd=str(tmp_path), env=env,
                          capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    _, train, _, _ = _split(root, 3, cuda_device)
    steps = 12 * len(train) // 2
    assert _epoch_steps(done.stdout) == [steps, steps], done.stdout
    _check_checkpoint_and_log(tmp_path, root, steps, 2)
    NeuralBarkCalculator(str(tmp_path / 'best_model.pt'), 'cuda:0')          # strict=True load
    done = subprocess.run([sys.executable, '-m', 'neuralbarkcalculator_b200.predict', root], cwd=str(tmp_path), env=env,
                          capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    with open(os.path.join(root, 'results', 'final_stats.csv')) as f:
        assert len(f.read().strip().split('\n')) == 13


def _torchrun(nproc, args, cwd, timeout=900):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop('NBC_TRAIN_BUCKETS', None)
    return subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(nproc),
                           '--master-addr', '127.0.0.1', '--master-port', str(port)] + args, cwd=cwd, env=env,
                          capture_output=True, text=True, timeout=timeout)


def test_two_rank_step_equals_one_gpu_accumulation(cuda_device):
    """Two ranks, one micro-batch each, single and bucketed exchange == one Trainer accumulating both micro-batches with
    the same seeds; identical weights on both ranks after Adam (tests/fit_parallel_worker.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    r = _torchrun(2, [os.path.join(HERE, 'fit_parallel_worker.py')], HERE, timeout=600)
    print(r.stdout[-2000:], r.stderr[-3000:])
    assert r.returncode == 0 and 'FIT_PARALLEL_OK world=2' in r.stdout


def test_fit_two_gpus(cuda_device, tmp_path):
    """torchrun --nproc_per_node 2 fit on the 12-item folder (its validation split has one image, so rank 1's validation
    shard is empty): one log, one checkpoint, val_* columns equal to a one-GPU evaluate of the checkpoint bit for bit,
    and floor(12 n_train / (2 batch)) optimizer steps per epoch, against floor(12 n_train / batch) for one GPU."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    root = str(tmp_path / 'data')
    _make_folder(root)
    run = tmp_path / 'run2'
    run.mkdir()
    r = _torchrun(2, _fit_cmd(root, '--batch', '2'), str(run))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert sorted(os.listdir(run)) == ['best_model.pt', 'log.tsv']
    _, train, valid, _ = _split(root, 3, cuda_device)
    assert len(valid) == 1
    steps = 12 * len(train) // (2 * 2)
    assert _epoch_steps(r.stdout) == [steps, steps], r.stdout
    assert sum(ln.startswith('fit: rank ') for ln in r.stdout.splitlines()) == 2
    _check_checkpoint_and_log(run, root, steps, 1)
    one = tmp_path / 'run1'
    one.mkdir()
    done = subprocess.run([sys.executable] + _fit_cmd(root, '--batch', '2'), cwd=str(one), env=dict(os.environ, PYTHONPATH=ROOT),
                          capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    assert _epoch_steps(done.stdout) == [12 * len(train) // 2] * 2
