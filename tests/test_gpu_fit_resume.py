"""``fit --state FILE --resume`` on the B200: a run interrupted after epoch 2 and resumed writes exactly the log (but for
the seconds column), checkpoint and final state of the run that was never interrupted; a changed run-defining argument is
refused; and the same holds for two ranks under torchrun (skips on a one-GPU box)."""
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_fit import _make_folder
from test_gpu_fit_parallel import _torchrun

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cmd(root, epochs, state, *extra):
    # plateau patience 0 and a large lr: the learning rate drops on the first epoch without improvement, so drops and
    # mid-window early-stopping counters fall on both sides of the resume point
    return (['-m', 'neuralbarkcalculator_b200.fit', root, '--init', 'random', '--epochs', str(epochs), '--crop', '128',
             '--target', '256', '--batch', '2', '--seed', '5', '--lr', '5e-3', '--plateau-patience', '0',
             '--plateau-factor', '0.5', '--early-stop-patience', '4', '--state', state] + list(extra))


def _run(args, cwd):
    done = subprocess.run([sys.executable] + args, cwd=str(cwd), env=dict(os.environ, PYTHONPATH=ROOT),
                          capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stdout[-2000:] + done.stderr[-3000:]
    return done


def _log(path):
    with open(path) as f:
        return [ln.rstrip('\n').split('\t')[:-1] for ln in f]        # every column but seconds


def _equal(a, b, where='state'):
    """Recursive bit-for-bit comparison of two state files (tensors by their bytes); log rows without seconds."""
    if isinstance(a, torch.Tensor):
        assert isinstance(b, torch.Tensor) and a.dtype == b.dtype and a.shape == b.shape, where
        assert torch.equal(a.reshape(-1).view(torch.uint8) if a.dtype.is_floating_point else a,
                           b.reshape(-1).view(torch.uint8) if b.dtype.is_floating_point else b), where
    elif isinstance(a, dict):
        assert sorted(a) == sorted(b), where
        for k in a:
            _equal(a[k], b[k], '%s.%s' % (where, k))
    elif isinstance(a, (list, tuple)) and where.endswith('.log'):
        assert [r[:-1] for r in a] == [r[:-1] for r in b], where
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            _equal(x, y, '%s[%d]' % (where, i))
    else:
        assert a == b, (where, a, b)


def _check_same(one, two):
    la, lb = _log(one / 'log.tsv'), _log(two / 'log.tsv')
    assert la == lb, (la, lb)
    assert la[-1][0] == 'test'
    sa = torch.load(one / 'best_model.pt', map_location='cpu')
    sb = torch.load(two / 'best_model.pt', map_location='cpu')
    _equal(sa, sb, 'best_model')
    a = torch.load(one / 'run.state', map_location='cpu', weights_only=False)
    b = torch.load(two / 'run.state', map_location='cpu', weights_only=False)
    _equal(a, b)
    return la, a


def test_resume_equals_the_uninterrupted_run(cuda_device, tmp_path):
    root = str(tmp_path / 'data')
    _make_folder(root)
    one, two = tmp_path / 'one', tmp_path / 'two'
    one.mkdir(), two.mkdir()
    done = _run(_cmd(root, 5, 'run.state'), one)
    assert 'fit: state run.state:' in done.stdout
    _run(_cmd(root, 2, 'run.state'), two)
    mid = torch.load(two / 'run.state', map_location='cpu', weights_only=False)
    assert mid['epoch'] == 2 and not mid['stopped']
    # a row a killed run appended after its last state: the resume drops it (as it drops the test row above)
    with open(two / 'log.tsv', 'a') as f:
        f.write('3\tpartial\n')
    resumed = _run(_cmd(root, 5, 'run.state', '--resume'), two)
    assert 'resuming from run.state after epoch 2' in resumed.stdout
    log, state = _check_same(one, two)
    epochs = [r for r in log[1:] if r[0] != 'test']
    print('lr per epoch', [r[1] for r in epochs], 'stopped', state['stopped'], 'plateau', state['plateau'],
          'early stopping', state['early_stopping'])
    assert len(epochs) == state['epoch'] and state['trainer']['step_count'] > 0
    # a second identical command gives the same bits: training is reproducible, not merely resumable
    three = tmp_path / 'three'
    three.mkdir()
    _run(_cmd(root, 5, 'run.state'), three)
    _check_same(one, three)


def test_resume_refuses_a_changed_argument(cuda_device, tmp_path):
    root = str(tmp_path / 'data')
    _make_folder(root)
    _run(_cmd(root, 1, 'run.state'), tmp_path)
    args = _cmd(root, 2, 'run.state', '--resume')
    args[args.index('--batch') + 1] = '1'
    done = subprocess.run([sys.executable] + args, cwd=str(tmp_path), env=dict(os.environ, PYTHONPATH=ROOT),
                          capture_output=True, text=True, timeout=900)
    assert done.returncode != 0 and '--batch (saved 2, now 1)' in done.stderr, done.stderr[-2000:]
    # --epochs, --log and --out may change
    _run(_cmd(root, 2, 'run.state', '--resume', '--log', 'other.tsv', '--out', 'other.pt'), tmp_path)
    assert [r[0] for r in _log(tmp_path / 'other.tsv')] == ['epoch', '1', '2', 'test']


def test_resume_two_gpus(cuda_device, tmp_path):
    """torchrun --nproc_per_node 2: resumed == uninterrupted; fit itself refuses to write a state when the ranks'
    buffers differ (a digest of params, statistics and Adam moments, compared over the ranks before each write)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    root = str(tmp_path / 'data')
    _make_folder(root)
    one, two = tmp_path / 'one', tmp_path / 'two'
    one.mkdir(), two.mkdir()
    for args, cwd in ((_cmd(root, 4, 'run.state'), one), (_cmd(root, 2, 'run.state'), two),
                      (_cmd(root, 4, 'run.state', '--resume'), two)):
        r = _torchrun(2, args, str(cwd))
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    _check_same(one, two)
