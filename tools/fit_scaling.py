"""Data-parallel scaling of ``python -m neuralbarkcalculator_b200.fit``: a synthetic labelled folder (``--images`` PNG
pairs ``--width`` wide, ragged heights width / 3 + 2 .. width (343..1024), as trimmed scans have them), trained for ``--epochs`` at crop 512 /
batch 5 (the reference's settings) on 1, 2, 4 and 8 GPUs (``torchrun`` above one; counts above the box's GPUs are
skipped).  From what ``fit`` prints per run:

* the training loop's samples/s per epoch: optimizer steps x global batch over the host clock around the epoch's
  batches, which ends in the loss read-back (a device synchronise); epoch 1 includes the first launches of every kernel,
  the last epoch is the steady-state figure, and its share of W x the one-GPU rate is the scaling efficiency;
* validation seconds per epoch (whole images, sharded over the ranks);
* the dataset load seconds of every rank (each rank decodes the whole folder).

    python tools/fit_scaling.py [--out profiles/r03_fit_scaling.json] [--gpus 1,2,4,8] [--images 256] [--epochs 2]

The card's name and power limit are read with ``nvidia-smi --query-gpu`` in the same run and written beside the
figures."""
import argparse
import json
import os
import re
import socket
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def make_folder(root, n, width, seed=0):
    """``n`` labelled items ``width`` wide: 80 % sapin, 10 % of each spruce, so every wood type has a validation and
    a test split."""
    from PIL import Image
    from oracle import synth
    rng = np.random.default_rng(seed)
    for k in range(n):
        wood = 'sapin' if k % 10 < 8 else ('epinette_gelee' if k % 10 == 8 else 'epinette_non_gelee')
        h = int(rng.integers(width // 3 + 2, width + 1))     # reflect padding stays narrower than the image
        for sub in ('samples', 'duals'):
            os.makedirs(os.path.join(root, sub, wood), exist_ok=True)
        Image.fromarray(synth.texture_u8(h, width, 1000 + k)).save(os.path.join(root, 'samples', wood, 'img%04d.png' % k))
        dual = (synth.class_mask(h, width, 2000 + k).astype(np.float32) * 127.5).astype(np.uint8)
        Image.fromarray(dual, mode='L').save(os.path.join(root, 'duals', wood, 'img%04d.png' % k))


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return [ln.strip() for ln in out]


EPOCH = re.compile(r'^fit: epoch (\d+): (\d+) steps of (\d+) samples, training ([\d.]+) s, validation ([\d.]+) s$')
LOAD = re.compile(r'^fit: rank (\d+) loaded (\d+) images in ([\d.]+) s$')


def run_fit(gpus, root, workdir, args):
    cmd = ['-m', 'neuralbarkcalculator_b200.fit', root, '--init', 'random', '--epochs', str(args.epochs), '--crop',
           str(args.crop), '--batch', str(args.batch), '--target', str(args.width), '--seed', '0']
    if gpus > 1:
        with socket.socket() as s:
            s.bind(('127.0.0.1', 0))
            port = s.getsockname()[1]
        cmd = ['-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(gpus), '--master-addr', '127.0.0.1',
               '--master-port', str(port)] + cmd
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop('NBC_TRAIN_BUCKETS', None)
    t0 = time.perf_counter()
    done = subprocess.run([sys.executable] + cmd, cwd=workdir, env=env, capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if done.returncode != 0:
        raise RuntimeError('fit on %d GPUs failed:\n%s' % (gpus, done.stderr[-4000:]))
    epochs, loads = [], {}
    for ln in done.stdout.splitlines():
        m = EPOCH.match(ln.strip())
        if m:
            e, steps, g, tt, tv = int(m[1]), int(m[2]), int(m[3]), float(m[4]), float(m[5])
            epochs.append({'epoch': e, 'steps': steps, 'global_batch': g, 'train_s': tt, 'samples_per_s': steps * g / tt,
                           'validation_s': tv})
        m = LOAD.match(ln.strip())
        if m:
            loads[int(m[1])] = float(m[3])
    with open(os.path.join(workdir, 'log.tsv')) as f:
        log = f.read()
    return {'gpus': gpus, 'epochs': epochs, 'load_s_per_rank': [loads[r] for r in sorted(loads)], 'wall_s': wall, 'log': log}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_fit_scaling.json')
    ap.add_argument('--gpus', default='1,2,4,8')
    ap.add_argument('--images', type=int, default=256)
    ap.add_argument('--width', type=int, default=1024)
    ap.add_argument('--crop', type=int, default=512)
    ap.add_argument('--batch', type=int, default=5)
    ap.add_argument('--epochs', type=int, default=2)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('fit_scaling: no CUDA device (this measures the B200 path; there is nothing to time on the CPU)')
    have = torch.cuda.device_count()
    counts = [g for g in (int(v) for v in args.gpus.split(',')) if g <= have]
    result = {'card': card(), 'gpus_on_box': have, 'images': args.images, 'width': args.width, 'crop': args.crop,
              'batch': args.batch, 'epochs': args.epochs, 'skipped_gpu_counts': [int(v) for v in args.gpus.split(',') if int(v) > have],
              'runs': []}
    with tempfile.TemporaryDirectory() as tmp:
        root = os.path.join(tmp, 'data')
        t0 = time.perf_counter()
        make_folder(root, args.images, args.width)
        result['folder_build_s'] = time.perf_counter() - t0
        for g in counts:
            work = os.path.join(tmp, 'g%d' % g)
            os.makedirs(work)
            r = run_fit(g, root, work, args)
            result['runs'].append(r)
            last = r['epochs'][-1]
            print('%d GPU(s): last epoch %d steps x %d samples in %.3f s = %.1f samples/s; validation %.3f s; load %s s'
                  % (g, last['steps'], last['global_batch'], last['train_s'], last['samples_per_s'], last['validation_s'],
                     ', '.join('%.2f' % v for v in r['load_s_per_rank'])), flush=True)
    one = next((r for r in result['runs'] if r['gpus'] == 1), None)
    if one is not None:
        base = one['epochs'][-1]['samples_per_s']
        for r in result['runs']:
            r['efficiency_vs_linear'] = r['epochs'][-1]['samples_per_s'] / (r['gpus'] * base)
    result['card_after'] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != 'runs'}))
    for r in result['runs']:
        print(json.dumps({k: v for k, v in r.items() if k != 'log'}))


if __name__ == '__main__':
    main()
