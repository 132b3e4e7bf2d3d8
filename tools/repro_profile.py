"""Cost of bit-reproducible training: the training step (``Trainer.step``: forward, loss, backward with the fixed-order
weight-gradient reductions, Adam) and the ``fit --state`` file, at two sizes:

* ``fit``'s defaults: micro-batch 5 at 512 x 512, Lovasz loss, dropout 0.8;
* the training benchmark's size (``bench.py --workload train``): batch 8 at 1024 x 1024, weighted cross-entropy.

Each size builds one Trainer from a synthetic state_dict, warms it up, then times ``--steps`` steps per round with CUDA
events on the step's stream for ``--rounds`` rounds (median and spread over the rounds).  A separate ``torch.profiler``
pass over ``--steps`` steps then sums the device time of the fixed-order reductions (``wgrad_reduce_kernel``,
``cls_finalize_kernel``) and of the weight-gradient kernels per step.  (The committed r04 figures also hold an A/B
against the former atomic epilogue, alternated round by round in the same run; that epilogue was selectable only in the
development build that took them and no longer exists.)  The state
file is the one ``fit --state`` writes (training state, best state_dict, counters), written with ``fit.write_state``
(temporary file, fsync, rename) to a temporary directory and read back with ``fit.read_state``.  The card's name and
power limit are read with ``nvidia-smi`` in the same run and written beside the figures.

    python tools/repro_profile.py [--out profiles/r04_repro_profile.json] [--steps 20] [--rounds 6] [--warmup 5]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.fit_scaling import card  # noqa: E402

SIZES = {'fit 5x512x512': (5, 512, 512, 'lovasz', 0.8), 'bench train 8x1024x1024': (8, 1024, 1024, 'weighted_ce', 0.0)}


def kernel_times(tr, x, t, steps):
    """Device time per step of the reductions and the weight-gradient kernels (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    groups = {'wgrad_reduce_kernel': 'wgrad_reduce', 'cls_finalize_kernel': 'cls_finalize', 'wgrad_tc_kernel': 'wgrad_tc',
              'cls_bwd_kernel': 'cls_bwd'}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            tr.step(x, t)
        torch.cuda.synchronize()
    out = {v: 0.0 for v in groups.values()}
    launches = {v: 0 for v in groups.values()}
    total = 0.0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = e.device_time if hasattr(e, 'device_time') else e.cuda_time
        total += us
        for k, v in groups.items():
            if k in e.name:
                out[v] += us
                launches[v] += 1
    res = {k: v / 1000.0 / steps for k, v in out.items()}
    res['all_kernels'] = total / 1000.0 / steps
    res['launches_per_step'] = {k: v // steps for k, v in launches.items()}
    return res


def main():
    from oracle import model as omodel, synth
    from neuralbarkcalculator_b200 import _lib, fit
    from neuralbarkcalculator_b200.train import Trainer
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r04_repro_profile.json')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=6)
    ap.add_argument('--warmup', type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('repro_profile: needs a CUDA device (timings are GPU measurements)')
    dev = torch.device('cuda:0')
    _lib.load()
    modes = ['deterministic']

    sd = omodel.synthetic_state_dict(seed=0)
    result = dict(card=card(), steps=args.steps, rounds=args.rounds, warmup=args.warmup, modes=modes, sizes={})
    for name, (N, H, W, loss, dropout) in SIZES.items():
        x = torch.from_numpy(np.stack([synth.texture_u8(H, W, 7 + i) for i in range(N)])).to(dev)
        t = torch.from_numpy(np.stack([synth.class_mask(H, W, 70 + i) for i in range(N)])).to(dev)
        tr = Trainer(sd, N, H, W, device='cuda:0', loss=loss, dropout=dropout)
        for _ in range(args.warmup):
            tr.step(x, t)
        torch.cuda.synchronize()
        times = {m: [] for m in modes}
        for r in range(args.rounds):
            for m in modes:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.steps):
                    tr.step(x, t)
                b.record()
                b.synchronize()
                times[m].append(a.elapsed_time(b) / args.steps)
        rows = {m: dict(step_ms=float(np.median(v)), min_ms=float(min(v)), max_ms=float(max(v)), rounds_ms=[float(u) for u in v])
                for m, v in times.items()}
        for m, row in rows.items():
            print('%-24s %-13s step %8.3f ms (rounds %.3f .. %.3f)' % (name, m, row['step_ms'], row['min_ms'], row['max_ms']),
                  flush=True)
        entry = dict(N=N, H=H, W=W, loss=loss, dropout=dropout, workspace_bytes=int(tr.ws.numel()), step=rows)
        entry['kernels_ms_per_step'] = kernel_times(tr, x, t, args.steps)
        print('%-24s device ms per step: %s' % (name, json.dumps(entry['kernels_ms_per_step'])), flush=True)
        # the fit --state file of this trainer (a few epochs' worth of writes)
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, 'run.state')
            writes, reads = [], []
            for _ in range(3):
                t0 = time.perf_counter()
                state = {'config': {}, 'epoch': 1, 'trainer': tr.training_state(), 'best_model': tr.state_dict(),
                         'plateau': {}, 'early_stopping': {}, 'log': [], 'stopped': False}
                state['best_model'] = {k: v.cpu() for k, v in state['best_model'].items()}
                t1 = time.perf_counter()
                fit.write_state(path, state)
                t2 = time.perf_counter()
                fit.read_state(path)
                t3 = time.perf_counter()
                writes.append((t1 - t0, t2 - t1))
                reads.append(t3 - t2)
            entry['state_file'] = dict(bytes=os.path.getsize(path), gather_s=float(np.median([w[0] for w in writes])),
                                       write_s=float(np.median([w[1] for w in writes])), read_s=float(np.median(reads)))
            print('%-24s state file %.1f MB: gather %.3f s, write+fsync %.3f s, read %.3f s' % (
                name, entry['state_file']['bytes'] / 1e6, entry['state_file']['gather_s'], entry['state_file']['write_s'],
                entry['state_file']['read_s']), flush=True)
        result['sizes'][name] = entry
        del tr
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result['card']))


if __name__ == '__main__':
    main()
