"""Fine-tuning with a frozen backbone on the B200 (``Trainer(freeze=...)``, ``fit --freeze``): ``none`` is the former
step, frozen units are eval-mode BatchNorm folded into one convolution each, the trainable part matches a float64
autograd reference fed the kernel's own stored input, frozen tensors never change, and ``fit --freeze`` trains end to end
(the two-GPU test skips on a one-GPU box)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import backward as ob
from oracle import losses as olosses
from oracle import model as omodel
from oracle import synth
from oracle.teacher import Bars, bf16_bar, plan_units, stored_inputs

from test_gpu_fit import _make_folder

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
FIRST_BLOCK = {'stem': 0, 'layer1': 3, 'layer2': 7, 'layer3': 13, 'layer4': 16}   # first trainable bottleneck


def _u8_batch(dev, N, H, W, j):
    return (torch.from_numpy(np.stack([synth.texture_u8(H, W, 10 * j + i) for i in range(N)])).to(dev),
            torch.from_numpy(np.stack([synth.class_mask(H, W, 50 + 10 * j + i) for i in range(N)])).to(dev))


def _f32_batch(dev, N, H, W):
    x = torch.cat([omodel.normalise_u8(synth.texture_u8(H, W, 11 + i)) for i in range(N)]).to(dev)
    t = torch.from_numpy(np.stack([synth.class_mask(H, W, 111 + i) for i in range(N)])).to(dev)
    return x, t


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def _segment_errors(tr, got, want):
    from neuralbarkcalculator_b200.train import gradient_segments
    return [_rel(got[o:o + c], want[o:o + c]) for o, c in gradient_segments(tr.lib, tr.handle) if c > 0]


def _first_unit(level):
    units, blocks, head = plan_units()
    fb = FIRST_BLOCK[level]
    return blocks[fb]['c1'] if fb < len(blocks) else head


def _stored(tr, x, s):
    """A unit's stored input as float64 NCHW: the bf16 staging image, the maxpool of the stem's y, or a unit's y."""
    def y(u):
        return tr.debug_tensor(1, u).permute(0, 3, 1, 2).double()
    if s == 'image':
        return x.to(torch.bfloat16).double()
    if s == 'pool':
        return F.max_pool2d(y(0), 3, 2, 1)
    return y(s)


def test_none_is_the_former_step(cuda_device, synthetic_sd):
    """freeze='none' against a Trainer built without the argument, 3 optimizer steps of 2 accumulated micro-batches:
    every step starts from the same state, and then every call issues the same launches and gives the same loss and
    running statistics bit for bit; the gradients, weights and Adam moments agree within the atomic-order noise of the
    gradient writers (relative 1e-3 per segment: two runs of the same step differ there, and Adam amplifies it from
    step to step, so b restarts each step from a's state)."""
    from neuralbarkcalculator_b200 import _lib
    from neuralbarkcalculator_b200.train import Trainer, dropout_seed
    N, H, W = 2, 96, 128
    a = Trainer(synthetic_sd, N, H, W, device='cuda:0', loss='lovasz', seed=2)
    b = Trainer(synthetic_sd, N, H, W, device='cuda:0', loss='lovasz', seed=2, freeze='none')
    assert (b.param_off, b.stats_off) == (0, 0)
    data = [_u8_batch(cuda_device, N, H, W, j) for j in range(2)]
    for step in range(3):
        for j, (x, t) in enumerate(data):
            counts, losses = [], []
            for tr in (a, b):
                c0 = _lib.launch_count()
                losses.append(float(tr.forward_backward(x, t, seed=dropout_seed(2, j, step), accumulate=j > 0)))
                counts.append(_lib.launch_count() - c0)
            torch.cuda.synchronize()
            assert counts[0] == counts[1], counts
            assert losses[0] == losses[1] and torch.equal(a.stats, b.stats), (step, j, losses)
        for tr in (a, b):
            tr.optimizer_step()
        torch.cuda.synchronize()
        for name in ('grads', 'params', 'adam_m', 'adam_v'):
            errs = _segment_errors(a, getattr(b, name), getattr(a, name))
            assert max(errs) <= 1e-3, (step, name, errs)
        for name in ('params', 'adam_m', 'adam_v'):
            getattr(b, name).copy_(getattr(a, name))
    assert a.num_batches_tracked == b.num_batches_tracked


def test_frozen_forward_unit_by_unit(cuda_device, synthetic_sd):
    """Everything through layer4 frozen: each unit's y against the oracle's eval-mode unit (conv with the folded weights
    rounded to bf16, folded bias, residual, ReLU; float64) fed the kernel's own stored input, under the bf16 bar.  The
    control folds the batch statistics of the unit's conv output instead of the running ones (train-mode BatchNorm)."""
    from neuralbarkcalculator_b200.train import Trainer
    N, H, W = 2, 120, 184
    tr = Trainer(synthetic_sd, N, H, W, device='cuda:0', freeze='layer4', dropout=0.0)
    x, t = _f32_batch(cuda_device, N, H, W)
    stats0 = tr.stats.clone()
    tr.forward_backward(x, t, seed=1)
    torch.cuda.synchronize()
    assert torch.equal(tr.stats[:tr.stats_off], stats0[:tr.stats_off])
    units, blocks, head = plan_units()
    src = stored_inputs(blocks, head)
    residual = {B['c3']: (B['ds'] if B['ds'] is not None else src[B['c1']]) for B in blocks}
    sd = {k: v.to(cuda_device) for k, v in synthetic_sd.items()}
    bars = Bars()
    for u in range(_first_unit('layer4')):
        U = units[u]
        for what in (0, 6, 7):
            with pytest.raises(RuntimeError):
                tr.debug_tensor(what, u)
        w = sd[U['conv'] + '.weight'].float()
        gamma, beta, mean, var = [sd[U['bn'] + s].float() for s in ('.weight', '.bias', '.running_mean', '.running_var')]
        scale = gamma / torch.sqrt(var + 1e-5)                 # fold_pack's f32 arithmetic
        wq = (w * scale.view(-1, 1, 1, 1)).to(torch.bfloat16).double()
        bias = (beta - mean * scale).double().view(1, -1, 1, 1)
        xs = _stored(tr, x, src[u])
        conv = dict(stride=U['s'], padding=U['p'], dilation=U['d'])
        ref, S = F.conv2d(xs, wq, **conv) + bias, F.conv2d(xs.abs(), wq.abs(), **conv) + bias.abs()
        z = F.conv2d(xs, w.double(), **conv)                   # control: train-mode BatchNorm of the same conv
        bm, bv = z.mean((0, 2, 3), keepdim=True), z.var((0, 2, 3), unbiased=False, keepdim=True)
        bad = (z - bm) * (bv + 1e-5).rsqrt() * gamma.double().view(1, -1, 1, 1) + beta.double().view(1, -1, 1, 1)
        if u in residual:
            res = _stored(tr, x, residual[u])
            ref, S, bad = ref + res, S + res.abs(), bad + res
        if U['relu']:
            ref, bad = ref.clamp_min(0), bad.clamp_min(0)
        y = tr.debug_tensor(1, u).permute(0, 3, 1, 2).double()
        tol = bf16_bar(S, ref)
        bars.check('frozen y', U['conv'], y, ref, tol)
        bars.control('batch statistics instead of running ones', not bars.within(y, bad, tol))
        del xs, ref, S, z, bad, y
    bars.report('frozen forward')


def _teacher_forced(dev, sd, level, N, H, W):
    from neuralbarkcalculator_b200.train import FREEZE, Trainer, frozen_prefixes
    weights = torch.tensor(olosses.DEFAULT_WEIGHTS)
    tr = Trainer(sd, N, H, W, device='cuda:0', freeze=level, dropout=0.0, loss='weighted_ce', class_weights=weights)
    x, tgt = _f32_batch(dev, N, H, W)
    params0, stats0 = tr.params.clone(), tr.stats.clone()
    tr.forward_backward(x, tgt, seed=1)
    torch.cuda.synchronize()
    units, blocks, head = plan_units()
    fb = FIRST_BLOCK[level]
    h = _stored(tr, x, stored_inputs(blocks, head)[_first_unit(level)])

    model = omodel.fcn_resnet50(dropout=0.0)
    model.load_state_dict(sd)
    model = model.double().to(dev).train()
    bb = model.backbone
    for m in [bb.conv1, bb.bn1] + [getattr(bb, 'layer%d' % i) for i in range(1, FREEZE.index(level))]:
        m.requires_grad_(False)
        m.eval()
    for blk in [blk for i in range(1, 5) for blk in getattr(bb, 'layer%d' % i)][fb:]:
        h = blk(h)
    full = ob.upsample_bicubic(model.classifier(h), (H, W))
    olosses.custom_weighted_cross_entropy(full, tgt.long(), weights.double().to(dev)).backward()

    grads, new = tr.gradients(), tr.state_dict()
    worst = {}
    for k, p in model.named_parameters():
        if p.requires_grad:
            worst[k] = _rel(grads[k], p.grad)
            assert grads[k].abs().sum() > 0, k
        else:
            assert torch.equal(grads[k], torch.zeros_like(grads[k])), k
    stat_err = {}
    for k, v in model.state_dict().items():
        if 'running' in k:
            if k.startswith(frozen_prefixes(level)):
                assert torch.equal(new[k], sd[k].to(dev)), k
            else:
                stat_err[k] = _rel(new[k], v)
    top = sorted(worst.items(), key=lambda kv: -kv[1])[:3]
    print('[%s %dx%dx%d] worst gradient errors %s; worst running-stat error %.3g' % (
        level, N, H, W, top, max(stat_err.values())))
    if level == 'layer4':
        # one trainable unit and the classifier, fed the kernel's own input: the float64 reference is teacher-forced
        assert max(worst.values()) <= 0.05, top
        assert max(stat_err.values()) <= 1e-2, max(stat_err.items(), key=lambda kv: kv[1])
    # the frozen prefix of grads / Adam moments stays zero, the frozen weights stay put
    tr.optimizer_step()
    torch.cuda.synchronize()
    o = tr.param_off
    for name in ('grads', 'adam_m', 'adam_v'):
        buf = getattr(tr, name)
        assert torch.equal(buf[:o], torch.zeros_like(buf[:o])), name
        assert buf[o:].abs().sum() > 0, name
    assert torch.equal(tr.params[:o], params0[:o]) and not torch.equal(tr.params[o:], params0[o:])
    assert torch.equal(tr.stats[:tr.stats_off], stats0[:tr.stats_off])


@pytest.mark.parametrize('level', list(FIRST_BLOCK))
@pytest.mark.parametrize('geom', [(5, 512, 512), (2, 200, 264)], ids=['5x512x512', '2x200x264'])
def test_trainable_part_teacher_forced(cuda_device, synthetic_sd, level, geom):
    """Every freeze level, at fit's default size and at an odd one, against a float64 torch model whose frozen stages
    are ``requires_grad_(False)`` and ``.eval()``, fed the kernel's stored input of the first trainable block: exactly
    the trainable tensors get a gradient, the frozen ones none, and the frozen prefix of grads / Adam moments stays zero.
    The values are compared where one unit is trainable (layer4 frozen: relative L2 per tensor 5 % for gradients, 1 %
    for running statistics).  Deeper trainable parts are not compared end to end here: the bf16 rounding of a
    random-init network's batch-statistics forward compounds over the blocks (the errors reach tens of percent at
    the first block), so such a comparison needs the unit-by-unit teacher forcing of test_gpu_train_production.py,
    whose kernels the trainable part runs unchanged.  The errors are printed at every level."""
    _teacher_forced(cuda_device, synthetic_sd, level, *geom)


def test_frozen_stays_frozen(cuda_device, synthetic_sd):
    """K = 3 optimizer steps of 2 accumulated micro-batches with weight decay 2e-3, layer2 frozen: every frozen weight,
    running statistic and num_batches_tracked equals the loaded state_dict bit for bit, every trainable tensor moved.
    The bucketed exchange drops the empty segments of the frozen blocks."""
    from neuralbarkcalculator_b200.train import Trainer, dropout_seed, frozen_prefixes
    N, H, W, K = 2, 128, 160, 3
    tr = Trainer(synthetic_sd, N, H, W, device='cuda:0', weight_decay=2e-3, loss='lovasz', seed=5, freeze='layer2',
                 bucket_mb=4.0)
    buckets = tr.gradient_buckets()
    assert all(c > 0 for _, _, c in buckets) and sum(c for _, _, c in buckets) == tr.params.numel() - tr.param_off
    assert min(off for _, off, _ in buckets) == tr.param_off
    data = [_u8_batch(cuda_device, N, H, W, j) for j in range(2)]
    for step in range(K):
        for j, (x, t) in enumerate(data):
            tr.forward_backward(x, t, seed=dropout_seed(5, j, step), accumulate=j > 0)
        tr.optimizer_step()
    torch.cuda.synchronize()
    new = {k: v.cpu() for k, v in tr.state_dict().items()}
    frozen = frozen_prefixes('layer2')
    n_frozen = 0
    for k, v in synthetic_sd.items():
        if k.startswith(frozen):
            n_frozen += 1
            assert torch.equal(new[k], v), k
        elif k.endswith('num_batches_tracked'):
            assert int(new[k]) == int(v) + 2 * K, k
        else:
            assert not torch.equal(new[k], v.float()), k
    assert n_frozen == 6 + (3 * 18 + 6) + (4 * 18 + 6)       # stem, layer1, layer2: 6 keys per conv + BatchNorm


def test_fit_freeze_end_to_end(cuda_device, tmp_path):
    """fit --init SD.pt --freeze layer3 --epochs 2 --batch 2 on a small labelled folder: the checkpoint's frozen keys
    equal SD.pt's, and evaluate and predict load and run it."""
    from neuralbarkcalculator_b200.train import frozen_prefixes
    g = np.load(os.path.join(HERE, 'golden', 'model_small.npz'))
    sd = omodel.synthetic_state_dict(seed=int(g['state_dict_seed']), head=(g['head_w'], g['head_b']))
    torch.save(sd, tmp_path / 'SD.pt')
    root = str(tmp_path / 'data')
    _make_folder(root)
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, '-m', 'neuralbarkcalculator_b200.fit', root, '--init', str(tmp_path / 'SD.pt'), '--freeze', 'layer3',
           '--epochs', '2', '--batch', '2', '--crop', '128', '--target', '256', '--seed', '3']
    done = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    assert 'parameters trainable' in done.stdout, done.stdout
    ck = torch.load(tmp_path / 'best_model.pt', map_location='cpu')
    assert sorted(ck) == sorted(sd)
    frozen = frozen_prefixes('layer3')
    for k in sd:
        if k.startswith(frozen):
            assert torch.equal(ck[k], sd[k]), k
    assert not torch.equal(ck['classifier.0.weight'], sd['classifier.0.weight'])
    done = subprocess.run([sys.executable, '-m', 'neuralbarkcalculator_b200.evaluate', root, '--model', str(tmp_path / 'best_model.pt')],
                          cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    with open(tmp_path / 'evaluation.tsv') as f:
        assert f.read().strip().split('\n')[-1].startswith('mean')
    done = subprocess.run([sys.executable, '-m', 'neuralbarkcalculator_b200.predict', root],
                          cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert done.returncode == 0, done.stderr[-3000:]
    with open(os.path.join(root, 'results', 'final_stats.csv')) as f:
        assert len(f.read().strip().split('\n')) == 13


def test_two_rank_frozen_step(cuda_device):
    """Two ranks with layer2 frozen == one GPU accumulating both micro-batches, in both exchange modes; frozen running
    statistics bit-identical after the epoch-end average (tests/freeze_parallel_worker.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop('NBC_TRAIN_BUCKETS', None)
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
                        '127.0.0.1', '--master-port', str(port), os.path.join(HERE, 'freeze_parallel_worker.py')],
                       cwd=HERE, env=env, capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:], r.stderr[-3000:])
    assert r.returncode == 0 and 'FREEZE_PARALLEL_OK world=2' in r.stdout
