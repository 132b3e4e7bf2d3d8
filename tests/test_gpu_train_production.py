"""Teacher-forced parity of the training step at the sizes it is trained at (``pytest -m gpu``).

tests/test_gpu_train_backward.py pins every kernel of the step against float64 at small and odd shapes (2x64x96,
3x58x122, 2x192x256).  Several kernels switch regime above a fixed size that those shapes never reach:

  * the BatchNorm reductions (bn_stats_partial / bn_bwd_partial) cap their grid at 1184 blocks, so past M = 37,888 rows a
    block sums more than 32 rows, a thread loops over several rows, a block's rows stop being a multiple of its row
    lanes, and trailing blocks can be empty;
  * the grid-stride kernels (bn_apply, bn_bwd_apply, the maxpool index kernels) cap their grid at 2368 blocks of 256
    threads and only wrap past 606,208 vectors;
  * the weight gradients split the pixel reduction over hundreds of K steps per CTA.

Here one step runs at 3x1024x1024 (the training benchmark's crop; weighted CE with the reference's class weights, on both
weight-gradient paths) and at 5x512x512 (``fit``'s defaults: Lovasz, dropout 0.8, wgrad_tc; with a random-init and a
trained-like network), and every kernel is recomputed in float64 on the GPU from its own operands, with the bars of
oracle/teacher.py.  The regime each geometry reaches is restated from the C++ (``test_regime_restatement_matches_the_
kernels`` fails when the C++ changes) and asserted before the run, so a retuned constant makes this test say it no
longer covers what it claims instead of passing vacuously.

Convolutions are checked on a channel sample (every pixel and the full reduction, a subset S of the output channels
for z and dW and of the input channels for dx): channel 0, the last channel, both channels on every 64- and
128-channel tile boundary and 8 seeded random channels.  BatchNorm and elementwise checks cover every channel.

Besides the four negative controls of the small test, one for the new regime: the running statistics recomputed
WITHOUT the rows of the last non-empty BatchNorm block must fail the running-statistics bar on every unit that is past
the block cap at 3x1024x1024 -- the bar sees 1/1184 of a reduction going missing."""
import ctypes as C
import math
import os
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import backward as ob
from oracle import losses as olosses
from oracle import model as omodel
from oracle import synth
from oracle.teacher import Bars, bf16_bar, check_head, check_loss, f32_bar, plan_units, run_step, stored_inputs

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'neuralbarkcalculator_b200', 'csrc')

# ------------------------------------------------------------------------------------------------ regimes, from the C++
SMS = 148                       # B200; wgrad_tc.cu sizes its splits by sm_count()
BN_THREADS = 256                # train_kernels.cu kBnThreads
BN_MAX_BLOCKS = 148 * 8         # train_kernels.cu kBnMaxBlocks
GRID_MAX = 148 * 16             # train_kernels.cu grid_for, train_kernels2.cu grid_for2

# the lines the restatements below follow; a change to any of them fails test_regime_restatement_matches_the_kernels
KERNEL_LINES = [
    ('train_kernels.cu', 'constexpr int kBnThreads = 256;'),
    ('train_kernels.cu', 'constexpr int kBnMaxBlocks = 148 * 8;'),
    ('train_kernels.cu', 'const int64_t nb = ceil_div64(M, 32);'),
    ('train_kernels.cu', 'return (int)(nb < kBnMaxBlocks ? (nb < 1 ? 1 : nb) : kBnMaxBlocks);'),
    ('train_kernels.cu', 'const int64_t rpb = ceil_div64(M, nb);'),
    ('train_kernels.cu', 'const int VL = vecs < kBnThreads ? vecs : kBnThreads, RL = kBnThreads / VL;'),
    ('train_kernels.cu', 'const int64_t b = ceil_div64(n, 256LL * per_thread);'),
    ('train_kernels.cu', 'return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));'),
    ('train_kernels.cu', 'bn_apply_kernel<<<grid_for(total8), 256, 0, stream>>>'),
    ('train_kernels.cu', 'bn_bwd_apply_kernel<<<grid_for(total8), 256, 0, stream>>>'),
    ('train_kernels2.cu', 'const int64_t b = ceil_div64(n, 256);'),
    ('train_kernels2.cu', 'return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));'),
    ('train_kernels.cu', 'const int base = co_tiles * p.ci_tiles * g.kh * g.kw;'),
    ('train_kernels.cu', 'int split = ceil_div(148 * 4, base);'),
    ('train_kernels.cu', 'const int64_t max_split = ceil_div64(p.M, 2048);'),
    ('train_kernels.cu', 'p.chunk = ceil_div64(ceil_div64(p.M, split), 32) * 32;'),
    ('wgrad_tc.cu', 'const int bn = (g.Cin % 256 == 0) ? 256 : (g.Cin % 128 == 0 ? 128 : 64);'),
    ('wgrad_tc.cu', 'const int base_items = p.co_tiles * p.ci_tiles * p.taps;'),
    ('wgrad_tc.cu', 'int splits = std::max(1, sm_count() / base_items);'),
    ('wgrad_tc.cu', 'const int max_splits = ceil_div(p.num_pix_tiles, 16);'),
    ('wgrad_tc.cu', 'p.tiles_per_split = ceil_div(p.num_pix_tiles, splits);'),
    ('wgrad_tc.cu', 'int splits = ceil_div(sm_count() * 2, 7);'),
]


def cdiv(a, b):
    return -(-a // b)


def bn_regime(M, C):
    """bn_forward_train / bn_backward (train_kernels.cu): grid bn_blocks(M), rows_per_block, and what one block does."""
    nb = max(1, min(cdiv(M, 32), BN_MAX_BLOCKS))
    rpb = cdiv(M, nb)
    VL = min(C // 8, BN_THREADS)
    RL = BN_THREADS // VL
    used = cdiv(M, rpb)                      # blocks with r0 = blockIdx * rpb < M
    return dict(blocks=nb, rpb=rpb, RL=RL, rows_per_thread=cdiv(rpb, RL), empty=nb - used,
                last_block=(used - 1) * rpb, last_rows=M - (used - 1) * rpb)


def grid_wraps(n):
    """grid_for / grid_for2: ceil(n / 256) blocks of 256 threads, at most GRID_MAX; True when the grid-stride loop runs
    a second iteration."""
    return cdiv(n, 256) > GRID_MAX


def wgrad_mma_k(M, Cin, Cout, k):
    """wgrad_mma (train_kernels.cu): output pixels one CTA accumulates (its chunk)."""
    base = cdiv(Cout, 128) * (Cin // 64) * k * k
    split = max(1, min(cdiv(SMS * 4, base), cdiv(M, 2048)))
    return cdiv(cdiv(M, split), 32) * 32


def wgrad_tc_k(N, Ho, Wo, Cin, Cout, k):
    """wgrad_tc / stem_wgrad_tc (wgrad_tc.cu): output pixels one CTA accumulates (tiles_per_split 64-pixel tiles)."""
    tiles = min(cdiv(Wo, tw) * cdiv(Ho, 64 // tw) for tw in (64, 32, 16, 8)) * N
    if Cin == 3:
        splits = cdiv(SMS * 2, 7)
    else:
        bn = 256 if Cin % 256 == 0 else (128 if Cin % 128 == 0 else 64)
        splits = max(1, SMS // (cdiv(Cout, 128) * (Cin // bn) * k * k))
    splits = max(1, min(splits, cdiv(tiles, 16)))
    return cdiv(tiles, splits) * 64


def unit_shapes(sd, N, H, W):
    """Per unit (plan order): Cin, Cout, k, input and output size, as nbc_train_create (train_plan.cu) lays them out."""
    units, blocks, head = plan_units()
    src = stored_inputs(blocks, head)
    out = []
    for u, U in enumerate(units):
        Cout, Cin, k = sd[U['conv'] + '.weight'].shape[:3]
        s = src[u]
        if s == 'image':
            hi, wi = H, W
        elif s == 'pool':
            hi, wi = (out[0]['Ho'] - 1) // 2 + 1, (out[0]['Wo'] - 1) // 2 + 1
        else:
            hi, wi = out[s]['Ho'], out[s]['Wo']
        ho = (hi + 2 * U['p'] - U['d'] * (k - 1) - 1) // U['s'] + 1
        wo = (wi + 2 * U['p'] - U['d'] * (k - 1) - 1) // U['s'] + 1
        out.append(dict(Cin=Cin, Cout=Cout, k=k, Hin=hi, Win=wi, Ho=ho, Wo=wo, M=N * ho * wo))
    return out


def regime_table(sd, N, H, W):
    """One row per unit: BN reduction and apply regime, K per CTA of both weight-gradient paths; and the maxpool's."""
    units, _, _ = plan_units()
    rows = []
    for U, g in zip(units, unit_shapes(sd, N, H, W)):
        r = dict(name=U['bn'], M=g['M'], C=g['Cout'], **bn_regime(g['M'], g['Cout']))
        r['apply_wraps'] = grid_wraps(g['M'] * g['Cout'] // 8)
        r['k_tc'] = wgrad_tc_k(N, g['Ho'], g['Wo'], g['Cin'], g['Cout'], g['k'])
        r['k_mma'] = None if g['Cin'] == 3 else wgrad_mma_k(g['M'], g['Cin'], g['Cout'], g['k'])   # stem: CUDA-core kernel
        rows.append(r)
    s = unit_shapes(sd, N, H, W)[0]
    H4, W4 = (s['Ho'] - 1) // 2 + 1, (s['Wo'] - 1) // 2 + 1
    pool = dict(fwd_wraps=grid_wraps(N * H4 * W4 * 8), bwd_wraps=grid_wraps(N * s['Ho'] * s['Wo'] * 8))
    return rows, pool


def print_regime(tag, rows, pool):
    print('\n[%s] %-30s %8s %5s %6s %4s %3s %6s %6s %5s %8s %8s' % (tag, 'unit (BN)', 'M', 'C', 'blocks', 'rpb', 'RL',
                                                                   'rows/t', 'empty', 'wraps', 'K wg_tc', 'K wg_mma'))
    for r in rows:
        print('[%s] %-30s %8d %5d %6d %4d %3d %6d %6d %5s %8d %8s' % (
            tag, r['name'], r['M'], r['C'], r['blocks'], r['rpb'], r['RL'], r['rows_per_thread'], r['empty'],
            'yes' if r['apply_wraps'] else 'no', r['k_tc'], '-' if r['k_mma'] is None else r['k_mma']))
    print('[%s] maxpool index kernels wrap: forward %s, backward %s' % (tag, pool['fwd_wraps'], pool['bwd_wraps']))


def assert_regime(geom, rows, pool):
    """What each geometry is here to cover; fails if a retuned constant takes it out of that regime."""
    capped = [r['M'] > 32 * BN_MAX_BLOCKS for r in rows]
    assert any(r['rpb'] % r['RL'] for r in rows), 'no unit has rows per block that are not a multiple of RL'
    if geom == '3x1024x1024':
        assert all(r['rpb'] > 32 and r['rows_per_thread'] > 1 for r in rows), 'a unit with <= 32 rows per BN block'
        assert any(r['empty'] > 0 for r in rows), 'no unit with empty trailing BN blocks'
        assert all(r['apply_wraps'] for r in rows), 'a BN apply grid that does not wrap'
        assert pool['fwd_wraps'] and pool['bwd_wraps'], 'a maxpool grid that does not wrap'
    elif geom == '5x512x512':
        # mixed: the stem and layer1 (and layer2.0.bn1, still at layer1's resolution) are past the block cap, the
        # units at 1/8 resolution are not
        big = [c for r, c in zip(rows, capped) if r['name'].startswith(('backbone.bn1', 'backbone.layer1.'))]
        small = [c for r, c in zip(rows, capped) if r['name'].startswith(('backbone.layer3.', 'backbone.layer4.', 'classifier'))]
        assert all(big) and not any(small), 'the 5x512x512 step no longer mixes capped and uncapped BatchNorms'
    else:
        raise ValueError(geom)


GEOMETRIES = {'3x1024x1024': (3, 1024, 1024), '5x512x512': (5, 512, 512)}


def test_regime_restatement_matches_the_kernels():
    """The constants and expressions the regime restatement follows are still those of the kernels."""
    text = {f: open(os.path.join(CSRC, f)).read() for f in {f for f, _ in KERNEL_LINES}}
    missing = [(f, line) for f, line in KERNEL_LINES if line not in text[f]]
    assert not missing, 'the kernels changed; update the regime restatement in this file: %s' % missing


@pytest.mark.parametrize('geom', list(GEOMETRIES))
def test_production_geometries_reach_the_large_regimes(synthetic_sd, geom):
    """The geometries of the GPU tests below reach the regimes they are there for (no GPU needed)."""
    rows, pool = regime_table(synthetic_sd, *GEOMETRIES[geom])
    print_regime(geom, rows, pool)
    assert_regime(geom, rows, pool)


# ------------------------------------------------------------------------------------------------ the checks
def channel_sample(C, seed):
    """Channel 0, the last channel, both channels on every 64- and 128-channel tile boundary, 8 seeded random ones."""
    s = {0, C - 1}
    for tile in (64, 128):
        for b in range(tile, C, tile):
            s |= {b - 1, b}
    s |= set(int(v) for v in np.random.default_rng(seed).choice(C, size=min(8, C), replace=False))
    return sorted(s)


def _check_units(tr, sd, x, shapes, bars, dev, drop_last_block):
    """Every unit of the step, one unit's tensors at a time, in float64 on ``dev``."""
    units, blocks, head = plan_units()
    assert len(units) == tr.lib.nbc_train_num_units(C.c_void_p(tr.handle))
    src = stored_inputs(blocks, head)
    N = x.shape[0]
    dims = (0, 2, 3)
    sdd = {k: v.to(dev) for k, v in sd.items()}
    grads = {k: v.double() for k, v in tr.gradients().items()}
    new = {k: v.double() for k, v in tr.state_dict().items()}
    residual = {}
    for B in blocks:
        residual[B['c3']] = B['ds'] if B['ds'] is not None else src[B['c1']]

    def t(what, u, S=None):     # bf16 NHWC debug tensor (channels S) -> f64 NCHW on dev (exact)
        v = tr.debug_tensor(what, u)
        if S is not None:
            v = v[..., S]
        return v.permute(0, 3, 1, 2).to(torch.float64, memory_format=torch.contiguous_format)

    def weight(u):              # the kernels pack the f32 master weights to bf16 (round to nearest even)
        return sdd[units[u]['conv'] + '.weight'].to(torch.bfloat16).double()

    def stored(s, S=None):      # a unit's stored input: staging image, maxpool of the stem's y, or a y
        if s == 'image':
            return x.to(dev).to(torch.bfloat16).double()
        if s == 'pool':
            return F.max_pool2d(t(1, 0, S), 3, 2, 1)
        return t(1, s, S)

    def dgrad(u, S, w=None):    # data gradient of unit u on its input channels S
        U, g = units[u], shapes[u]
        w = weight(u)[:, S] if w is None else w
        return ob.conv_dgrad(t(7, u), w, (N, len(S), g['Hin'], g['Win']), U['s'], U['p'], U['d'])

    # ---- per unit: forward z and y, running statistics, BatchNorm backward, weight gradient
    for u, U in enumerate(units):
        bn, conv, g = U['bn'], U['conv'], shapes[u]
        assert tuple(tr.debug_tensor(0, u).shape) == (N, g['Ho'], g['Wo'], g['Cout']), (conv, tr.debug_tensor(0, u).shape)
        So = channel_sample(g['Cout'], u)
        xu, z = stored(src[u]), t(0, u)
        ref = F.conv2d(xu, weight(u)[So], stride=U['s'], padding=U['p'], dilation=U['d'])
        bars.check('forward z', conv, z[:, So], ref, bf16_bar(ref.abs(), ref))

        gamma, beta = sdd[bn + '.weight'].double(), sdd[bn + '.bias'].double()
        mean, var = z.mean(dims, keepdim=True), z.var(dims, unbiased=False, keepdim=True)
        zn = (z - mean) * (var + 1e-5).rsqrt() * gamma.view(1, -1, 1, 1) + beta.view(1, -1, 1, 1)
        res = stored(residual[u]) if u in residual else torch.zeros((), dtype=torch.float64, device=dev)
        ref, S = zn + res, zn.abs() + res.abs()
        if U['relu']:
            ref = ref.clamp_min(0)
        y = t(1, u)
        bars.check('forward y', bn, y, ref, bf16_bar(S, ref))
        del zn, res, ref, S

        old_m, old_v = sdd[bn + '.running_mean'].double(), sdd[bn + '.running_var'].double()
        rm, rv = ob.running_stats(z, old_m, old_v)
        tol_m = 1e-5 * (0.9 * old_m.abs() + 0.1 * z.abs().mean(dims))
        tol_v = 1e-5 * (0.9 * old_v + 0.1 * (z * z).mean(dims))
        bars.check('running stats', bn + '.running_mean', new[bn + '.running_mean'], rm, tol_m)
        bars.check('running stats', bn + '.running_var', new[bn + '.running_var'], rv, tol_v)
        bars.control('biased running var', not bars.within(new[bn + '.running_var'],
                                                           ob.running_stats(z, old_m, old_v, unbiased=False)[1], tol_v))
        if drop_last_block and g['M'] > 32 * BN_MAX_BLOCKS:
            # the rows of the last non-empty block of bn_stats_partial left out of the statistics
            r0 = bn_regime(g['M'], g['Cout'])['last_block']
            kept = z.permute(0, 2, 3, 1).reshape(g['M'], g['Cout'])[:r0].t().reshape(1, g['Cout'], r0, 1)
            dm, dv = ob.running_stats(kept, old_m, old_v)
            bars.control_each('last BN block dropped', bn, not (bars.within(new[bn + '.running_mean'], dm, tol_m)
                                                                and bars.within(new[bn + '.running_var'], dv, tol_v)))
            del kept

        dy, dz = t(6, u), t(7, u)
        ref = ob.bn_backward(dy, y, z, gamma, U['relu'])
        bars.check('bn dz', bn, dz, ref['dz'], bf16_bar(ref['dz'].abs(), ref['dz']))
        bars.check('bn dgamma dbeta', bn + '.weight', grads[bn + '.weight'], ref['dgamma'], f32_bar(ref['dgamma_abs']))
        bars.check('bn dgamma dbeta', bn + '.bias', grads[bn + '.bias'], ref['dbeta'], f32_bar(ref['dbeta_abs']))
        del ref, dy, y, z

        wshape = (len(So),) + tuple(sd[conv + '.weight'].shape[1:])
        A = torch.nn.grad.conv2d_weight(xu.abs().float(), wshape, dz[:, So].abs().float(), stride=U['s'], padding=U['p'],
                                        dilation=U['d'])       # only an error bar: f32 is plenty
        bars.check('wgrad', conv, grads[conv + '.weight'][So], ob.conv_wgrad(xu, dz[:, So], wshape, U['s'], U['p'], U['d']),
                   f32_bar(A.double()))
        del A, xu, dz

    # ---- data gradients on input-channel samples, each checked through the dy the next unit upstream captured
    for bi, B in enumerate(blocks):
        c1, c2, c3, ds = B['c1'], B['c2'], B['c3'], B['ds']
        S = channel_sample(shapes[c3]['Cin'], c3)
        ref = dgrad(c3, S)
        bars.check('dgrad', units[c3]['conv'], t(6, c2, S), ref, bf16_bar(ref.abs(), ref))
        S = channel_sample(shapes[c2]['Cin'], c2)
        ref = dgrad(c2, S)
        bars.check('dgrad', units[c2]['conv'], t(6, c1, S), ref, bf16_bar(ref.abs(), ref))
        if bi == 0:
            bad = dgrad(c2, S, weight(c2)[:, S].flip(2, 3))          # taps not flipped
            bars.control('unflipped 3x3 taps', not bars.within(t(6, c1, S), bad, bf16_bar(bad.abs(), bad)))
        S = channel_sample(shapes[c1]['Cin'], c1)
        masked = torch.where(t(1, c3, S) > 0, t(6, c3, S), 0.0)     # the skip path's gradient
        a = dgrad(c1, S)
        if ds is not None:
            bars.exact('ds dy == masked c3 dy', units[ds]['bn'], t(6, ds), torch.where(t(1, c3) > 0, t(6, c3), 0.0))
            b = dgrad(ds, S)
        else:
            b = masked
        ref, Sm = a + b, a.abs() + b.abs()
        if bi > 0:
            bars.check('dgrad', units[c1]['conv'] + ' + skip', t(6, blocks[bi - 1]['c3'], S), ref, bf16_bar(Sm, ref))
        else:
            # block 0's input gradient -> maxpool backward (first maximum of each window of the stored stem y)
            ys = t(1, 0, S)
            got, refs = t(6, 0, S), ob.maxpool_backward(ref, ys)
            tol = bf16_bar(ob.maxpool_backward(Sm, ys), refs)
            bars.check('maxpool dgrad', 'backbone.bn1 dy', got, refs, tol)
            bars.control('maxpool last maximum', not bars.within(got, ob.maxpool_backward(ref, ys, last=True), tol))
        del a, b, ref, Sm, masked
    S = channel_sample(shapes[head]['Cin'], head)
    ref = dgrad(head, S)
    bars.check('dgrad', 'classifier.0', t(6, blocks[-1]['c3'], S), ref, bf16_bar(ref.abs(), ref))
    return head, t


def _run(cuda_device, sd, geom, impl, loss_kind, class_weights, dropout_p, seed):
    from neuralbarkcalculator_b200.train import Trainer
    N, H, W = GEOMETRIES[geom]
    tag = '%s %s %s dropout %.1f' % (geom, 'wgrad_tc' if impl == 0 else 'wgrad_mma', loss_kind, dropout_p)
    rows, pool = regime_table(sd, N, H, W)
    print_regime(tag, rows, pool)
    assert_regime(geom, rows, pool)
    t0 = time.perf_counter()
    x = torch.cat([omodel.normalise_u8(synth.texture_u8(H, W, 11 + i)) for i in range(N)])   # f32 NCHW input
    tgt = torch.from_numpy(np.stack([synth.class_mask(H, W, 111 + i) for i in range(N)])).to(cuda_device)
    tr = Trainer(sd, N, H, W, device='cuda:0', dropout=dropout_p, class_weights=class_weights, loss=loss_kind)
    loss = run_step(tr, x.to(cuda_device), tgt, seed, impl)
    t1 = time.perf_counter()
    bars = Bars()
    head, t = _check_units(tr, sd, x, unit_shapes(sd, N, H, W), bars, cuda_device, geom == '3x1024x1024')
    check_head(tr, sd, t(1, head), t(6, head), dropout_p, seed, bars, device=cuda_device)
    check_loss(tr, tgt, loss, loss_kind, class_weights, bars, cuda_device)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    print('[%s] loss %.6f; wall time: inputs + two steps %.1f s, float64 checks %.1f s' % (tag, loss, t1 - t0, t2 - t1))
    bars.report(tag)


@pytest.mark.gpu
@pytest.mark.parametrize('impl', [0, 1], ids=['wgrad_tc', 'wgrad_mma'])
def test_train_step_teacher_forced_3x1024(cuda_device, synthetic_sd, impl):
    """Batch 3 at 1024x1024, weighted CE with the reference's class weights, dropout 0, on both weight-gradient paths:
    every BatchNorm past its block cap, every apply kernel wrapping."""
    _run(cuda_device, synthetic_sd, '3x1024x1024', impl, 'weighted_ce', torch.tensor(olosses.DEFAULT_WEIGHTS), 0.0, 1)


@pytest.mark.gpu
@pytest.mark.parametrize('sd_name', ['synthetic_sd', 'trained_like_sd'])
def test_train_step_teacher_forced_fit_defaults(cuda_device, request, sd_name):
    """fit's defaults -- batch 5 at 512x512, Lovasz, dropout 0.8, wgrad_tc -- from a random-init network and from a
    trained-like one (what ``fit --init checkpoint.pt`` starts from)."""
    seed = (5 << 40) + (1 << 28) + 3      # Trainer.dropout_seed's layout: run seed, rank, step
    _run(cuda_device, request.getfixturevalue(sd_name), '5x512x512', 0, 'lovasz', torch.ones(3), 0.8, seed)
