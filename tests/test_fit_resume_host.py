"""fit's resumable state on the host: plateau / early-stopping counters, the sampling and augmentation generators, the
run-compatibility check, the log rewrite and the atomic state write (no GPU)."""
import argparse
import os

import numpy as np
import pytest
import torch

from neuralbarkcalculator_b200 import augment, fit, utils


def test_plateau_and_early_stopping_round_trip_mid_patience():
    losses = [1.0, 0.9, 0.95, 0.96, 0.97, 0.91, 0.99, 0.98, 0.97, 0.96, 0.95, 0.94]
    a, sa = fit.Plateau(1e-3, factor=0.5, patience=2, cooldown=1), fit.EarlyStopping(4)
    for v in losses[:4]:            # two bad epochs: both counters are in the middle of their windows
        a.step(v), sa.step(v)
    assert a.num_bad_epochs == 2 and sa.wait == 2
    b, sb = fit.Plateau(1e-3, factor=0.5, patience=2, cooldown=1), fit.EarlyStopping(4)
    b.load_state_dict(a.state_dict())
    sb.load_state_dict(sa.state_dict())
    for v in losses[4:]:
        assert a.step(v) == b.step(v)
        assert sa.step(v) == sb.step(v)
        assert a.state_dict() == b.state_dict() and sa.state_dict() == sb.state_dict()
    assert a.lr < 1e-3              # the learning rate dropped after the round trip


def test_generator_states_reproduce_the_next_draws():
    train_split = np.arange(3, 40)
    weights = np.linspace(1.0, 2.0, len(train_split))
    g = torch.Generator().manual_seed(5)
    rng = np.random.default_rng(5)
    utils.weighted_epoch_batches(train_split, weights, 4, generator=g)
    augment.draw_params(rng, 4, 40, 128, (256, 256))
    g_state, rng_state = g.get_state(), rng.bit_generator.state
    want_b = utils.weighted_epoch_batches(train_split, weights, 4, generator=g)
    want_p = augment.draw_params(rng, 8, 40, 128, (256, 256))
    g2 = torch.Generator().manual_seed(123)
    rng2 = np.random.default_rng(123)
    g2.set_state(g_state)
    rng2.bit_generator.state = rng_state
    assert torch.equal(utils.weighted_epoch_batches(train_split, weights, 4, generator=g2), want_b)
    assert np.array_equal(augment.draw_params(rng2, 8, 40, 128, (256, 256)), want_p)


def _args(**kw):
    a = fit.parse_args(['root', '--init', 'random', '--state', 's.state'])
    for k, v in kw.items():
        setattr(a, k, v)
    return a


ITEMS = [('a.png', 'sapin', 200, 256), ('b.png', 'sapin', 180, 256)]


def test_compatibility_check_names_each_changed_field():
    saved = fit.run_config(_args(), ITEMS, 1)
    # --epochs, --log, --out, --device and --init may change
    fit.check_resume(saved, fit.run_config(_args(epochs=50, log='other.tsv', out='x.pt', device='cuda:1', init='sd.pt'),
                                           ITEMS, 1))
    changed = fit.run_config(_args(batch=3, lr=1e-4, seed=9), ITEMS[:1] + [('b.png', 'sapin', 181, 256)], 2)
    with pytest.raises(RuntimeError) as e:
        fit.check_resume(saved, changed)
    msg = str(e.value)
    for name in ('--batch', '--lr', '--seed', 'the folder', 'the world size'):
        assert name in msg, (name, msg)
    for name in ('--crop', '--dropout', '--freeze', '--accumulate', '--plateau-patience'):
        assert name not in msg
    for field, flag in (('accumulate', '--accumulate'), ('freeze', '--freeze'), ('target', '--target'), ('loss', '--loss'),
                        ('weight_decay', '--weight-decay'), ('dropout', '--dropout'), ('plateau_factor', '--plateau-factor'),
                        ('plateau_patience', '--plateau-patience'), ('early_stop_patience', '--early-stop-patience'),
                        ('crop', '--crop')):
        other = dict(saved)
        other[field] = 'changed'
        with pytest.raises(RuntimeError, match=flag):
            fit.check_resume(saved, other)


def test_resume_needs_state():
    with pytest.raises(SystemExit):
        fit.parse_args(['root', '--init', 'random', '--resume'])


@pytest.mark.parametrize('extra', [['3', '0.1', '0.5', '0.4', '0.3', '0.1', '0.2', '0.3', '1.000'],
                                   ['test', '', '', '0.4', '0.3', '0.1', '0.2', '0.3', '1.000']])
def test_log_rewrite_drops_rows_after_the_saved_epochs(tmp_path, extra):
    path = str(tmp_path / 'log.tsv')
    rows = [[1, '0.001', '0.5', '0.6', '0.2', '0.1', '0.2', '0.3', '2.000'],
            [2, '0.001', '0.4', '0.5', '0.25', '0.1', '0.2', '0.3', '2.100']]
    fit.rewrite_log(path, rows)
    with open(path, 'a') as f:
        f.write('\t'.join(extra) + '\n')
    fit.rewrite_log(path, rows)
    with open(path) as f:
        lines = [ln.rstrip('\n').split('\t') for ln in f]
    assert lines[0] == fit.LOG_HEADER
    assert lines[1:] == [[str(v) for v in r] for r in rows]


def test_state_write_is_atomic(tmp_path, monkeypatch):
    path = str(tmp_path / 'run.state')
    fit.write_state(path, {'epoch': 1, 'x': torch.arange(5)})
    real_replace = os.replace

    def boom(src, dst):
        raise OSError('killed between the write and the rename')
    monkeypatch.setattr(os, 'replace', boom)
    with pytest.raises(OSError):
        fit.write_state(path, {'epoch': 2, 'x': torch.arange(7)})
    monkeypatch.setattr(os, 'replace', real_replace)
    old = fit.read_state(path)
    assert old['epoch'] == 1 and torch.equal(old['x'], torch.arange(5))
    assert sorted(os.listdir(tmp_path)) == ['run.state']      # no temporary file left behind
    fit.write_state(path, {'epoch': 2})
    assert fit.read_state(path)['epoch'] == 2
