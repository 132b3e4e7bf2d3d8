"""Training step time per ``--freeze`` level (``Trainer(freeze=...)``: forward, loss, backward to the first trainable
block, Adam on the trainable suffix) at two sizes:

* ``fit``'s defaults: micro-batch 5 at 512 x 512, Lovasz loss, dropout 0.8;
* the training benchmark's size (``bench.py --workload train``): batch 8 at 1024 x 1024, weighted cross-entropy.

Each size builds one Trainer per level from the same synthetic state_dict, warms every one up, then times ``--steps``
steps of each level per round, with CUDA events on the step's stream, for ``--rounds`` rounds in alternating order
(the spread over the rounds is the noise).  The card's name and power limit are read with ``nvidia-smi`` in the same
run and written beside the figures.

    python tools/freeze_profile.py [--out profiles/r03_freeze_profile.json] [--steps 20] [--rounds 5] [--warmup 5]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.fit_scaling import card  # noqa: E402

SIZES = {'fit 5x512x512': (5, 512, 512, 'lovasz', 0.8), 'bench train 8x1024x1024': (8, 1024, 1024, 'weighted_ce', 0.0)}


def main():
    from oracle import model as omodel, synth
    from neuralbarkcalculator_b200.train import FREEZE, Trainer
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_freeze_profile.json')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('freeze_profile: needs a CUDA device (timings are GPU measurements)')
    dev = torch.device('cuda:0')
    sd = omodel.synthetic_state_dict(seed=0)
    result = dict(card=card(), steps=args.steps, rounds=args.rounds, warmup=args.warmup, sizes={})
    for name, (N, H, W, loss, dropout) in SIZES.items():
        x = torch.from_numpy(np.stack([synth.texture_u8(H, W, 7 + i) for i in range(N)])).to(dev)
        t = torch.from_numpy(np.stack([synth.class_mask(H, W, 70 + i) for i in range(N)])).to(dev)
        trainers = {lv: Trainer(sd, N, H, W, device='cuda:0', loss=loss, dropout=dropout, freeze=lv) for lv in FREEZE}
        for tr in trainers.values():
            for _ in range(args.warmup):
                tr.step(x, t)
        torch.cuda.synchronize()
        times = {lv: [] for lv in FREEZE}
        for r in range(args.rounds):
            for lv in (FREEZE if r % 2 == 0 else FREEZE[::-1]):
                tr = trainers[lv]
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.steps):
                    tr.step(x, t)
                b.record()
                b.synchronize()
                times[lv].append(a.elapsed_time(b) / args.steps)
        none = float(np.median(times['none']))
        rows = {}
        for lv in FREEZE:
            tr = trainers[lv]
            med = float(np.median(times[lv]))
            rows[lv] = dict(step_ms=med, min_ms=float(min(times[lv])), max_ms=float(max(times[lv])), speedup=none / med,
                            samples_per_s=N * 1000.0 / med, trainable_params=int(tr.params.numel() - tr.param_off))
            print('%-24s freeze %-6s step %8.3f ms (rounds %.3f .. %.3f)  x%.3f vs none  %8.1f samples/s  %d trainable' % (
                name, lv, med, rows[lv]['min_ms'], rows[lv]['max_ms'], rows[lv]['speedup'], rows[lv]['samples_per_s'],
                rows[lv]['trainable_params']), flush=True)
        result['sizes'][name] = dict(N=N, H=H, W=W, loss=loss, dropout=dropout, levels=rows)
        del trainers
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result['card']))


if __name__ == '__main__':
    main()
