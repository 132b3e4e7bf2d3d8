"""Host side of ``fit --freeze`` (no GPU): the argument, its refusal with ``--init random``, the trainable suffix of the
flat buffers against the state_dict keys of each stage, and the epoch-end average of the running statistics over gloo
ranks, which must leave frozen statistics bit-identical."""
import ctypes as C
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from neuralbarkcalculator_b200 import _lib, fit
from neuralbarkcalculator_b200 import distributed as nd
from neuralbarkcalculator_b200.models import fcn_resnet50
from neuralbarkcalculator_b200.train import FREEZE, frozen_prefixes

# state_dict key prefixes that each --freeze level adds to the frozen set
STAGE_KEYS = {'stem': ('backbone.conv1.', 'backbone.bn1.'), 'layer1': ('backbone.layer1.',),
              'layer2': ('backbone.layer2.',), 'layer3': ('backbone.layer3.',), 'layer4': ('backbone.layer4.',)}


def test_freeze_argument():
    assert fit.parse_args(['root', '--init', 'sd.pt']).freeze == 'none'
    assert fit.parse_args(['root', '--init', 'random']).freeze == 'none'
    for level in FREEZE:
        assert fit.parse_args(['root', '--init', 'sd.pt', '--freeze', level]).freeze == level
    for bad in ('layer5', 'conv1', 'all', ''):
        with pytest.raises(SystemExit):
            fit.parse_args(['root', '--init', 'sd.pt', '--freeze', bad])


@pytest.mark.parametrize('level', FREEZE[1:])
def test_freeze_refuses_random_init(level, capsys):
    with pytest.raises(SystemExit):
        fit.parse_args(['root', '--init', 'random', '--freeze', level])
    assert 'needs --init' in capsys.readouterr().err


def test_frozen_prefixes_follow_the_stages():
    acc = ()
    assert frozen_prefixes('none') == ()
    for level in FREEZE[1:]:
        acc += STAGE_KEYS[level]
        assert frozen_prefixes(level) == acc, level


def test_trainable_offsets_match_the_state_dict():
    """nbc_train_trainable_offsets against the element counts of the frozen keys of fcn_resnet50's state_dict: the
    parameters (conv weights, BatchNorm weight / bias) before the first trainable unit, and the running mean / var."""
    sd = fcn_resnet50(pretrained=False).state_dict()
    lib = _lib.load()
    h = C.c_void_p(lib.nbc_train_create(1, 64, 64))           # host-side bookkeeping only: no CUDA call
    try:
        n_params = lib.nbc_train_param_count(h)
        n_stats = lib.nbc_train_stats_count(h)
        frozen = ()
        for stages, level in enumerate(FREEZE):
            if level != 'none':
                frozen += STAGE_KEYS[level]
            keys = [k for k in sd if k.startswith(frozen)]
            want_p = sum(sd[k].numel() for k in keys if k.endswith(('weight', 'bias')))
            want_s = sum(sd[k].numel() for k in keys if k.endswith(('running_mean', 'running_var')))
            _lib.check(lib.nbc_train_set_frozen(h, stages), 'nbc_train_set_frozen')
            p, s = C.c_int64(-1), C.c_int64(-1)
            _lib.check(lib.nbc_train_trainable_offsets(h, C.byref(p), C.byref(s)), 'nbc_train_trainable_offsets')
            assert (p.value, s.value) == (want_p, want_s), level
            assert 0 <= p.value < n_params and 0 <= s.value < n_stats
            # frozen segments are empty and come last; the others tile the trainable suffix
            segs = []
            for i in range(lib.nbc_train_num_segments(h)):
                off, cnt = C.c_int64(0), C.c_int64(0)
                _lib.check(lib.nbc_train_segment(h, i, C.byref(off), C.byref(cnt)), 'nbc_train_segment')
                segs.append((off.value, cnt.value))
            live = [sg for sg in segs if sg[1] > 0]
            assert segs[:len(live)] == live
            assert live[-1][0] == p.value and sum(c for _, c in live) == n_params - p.value
            n_frozen_blocks = sum(1 for k in keys if k.endswith('conv1.weight') and '.layer' in k)
            assert len(segs) - len(live) == n_frozen_blocks + (stages > 0), level
        for bad in (-1, 6, 100):
            assert lib.nbc_train_set_frozen(h, bad) != 0
            assert 'stages' in _lib.last_error()
    finally:
        lib.nbc_train_destroy(h)


def _average_worker(rank, world, port, stats_off, out_path):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    nd.init_from_env(device_type='cpu')
    stats = torch.rand(1000, generator=torch.Generator().manual_seed(7)) * 3 + 0.1   # identical on every rank
    stats[stats_off:] = torch.rand(1000 - stats_off, generator=torch.Generator().manual_seed(100 + rank))
    fit.average_running_stats(stats, stats_off, world)
    torch.save(stats, out_path % rank)
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def test_running_stats_average_covers_only_the_trainable_suffix(tmp_path):
    """Three gloo ranks with the same frozen prefix: the prefix comes back bit for bit, the suffix is the mean over
    the ranks.  Averaging the whole buffer would change some of the identical prefix values ((x + x + x) / 3 != x)."""
    world, stats_off = 3, 600
    out = str(tmp_path / 'stats%d.pt')
    mp.spawn(_average_worker, args=(world, _free_port(), stats_off, out), nprocs=world, join=True)
    prefix = torch.rand(1000, generator=torch.Generator().manual_seed(7)) * 3 + 0.1
    suffix = sum(torch.rand(1000 - stats_off, generator=torch.Generator().manual_seed(100 + r)) for r in range(world)) / world
    got = [torch.load(out % r) for r in range(world)]
    for g in got:
        assert torch.equal(g[:stats_off], prefix[:stats_off])
        assert torch.allclose(g[stats_off:], suffix, rtol=1e-6, atol=0)
        assert torch.equal(g, got[0])
    assert not torch.equal((prefix + prefix + prefix) / 3, prefix)     # the whole-buffer mean would not be exact
