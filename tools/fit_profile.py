"""Where the time of a training epoch goes (``python -m neuralbarkcalculator_b200.fit``): the augmentation kernel per
batch, the training step, and whole-image validation per image, at the reference's crop 512 / batch 5 on 1024-wide
ragged sources (heights as trimmed scans have them, odd and even).

    python tools/fit_profile.py [--out profiles/r03_fit_profile.txt] [--steps 30] [--sources 24] [--val 8]

Device times are CUDA-event times; ``loop`` is the host clock over augment + step for all timed batches, ending in a
device synchronise, i.e. what an epoch pays per batch including the augmentation's size check (it reads the dims back
and so waits for the previous step)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _synthetic_sources(n, rng):
    from oracle import synth
    heights = rng.integers(343, 1025, n)
    images = [synth.texture_u8(int(h), 1024, 1000 + k) for k, h in enumerate(heights)]
    duals = [(synth.class_mask(int(h), 1024, 2000 + k).astype(np.float32) * 127.5).astype(np.uint8) for k, h in enumerate(heights)]
    return images, duals, heights


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_fit_profile.txt')
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--sources', type=int, default=24)
    ap.add_argument('--val', type=int, default=8)
    ap.add_argument('--crop', type=int, default=512)
    ap.add_argument('--batch', type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('fit_profile: no CUDA device (this measures the B200 path; there is nothing to time on the CPU)')
    from neuralbarkcalculator_b200 import augment, evaluate as nev
    from neuralbarkcalculator_b200.models import fcn_resnet50
    from neuralbarkcalculator_b200.train import Trainer
    dev = torch.device('cuda:0')
    rng = np.random.default_rng(0)
    images, duals, heights = _synthetic_sources(args.sources, rng)
    ds = augment.DeviceDataset(images, duals, ['sapin'] * len(images), dev)
    torch.manual_seed(0)
    sd = fcn_resnet50(pretrained=False, dropout=0.8).state_dict()
    tr = Trainer(sd, args.batch, args.crop, args.crop, device='cuda:0', loss='lovasz')
    target = (1024, 1024)

    def batch_params():
        return augment.draw_params(rng, args.batch, len(ds), args.crop, target)

    for _ in range(args.warmup):
        x, t = augment.augment_ragged(ds, batch_params(), args.crop, target)
        tr.step(x, t)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t0 = time.perf_counter()
    for k in range(args.steps):
        ev[k][0].record()
        x, t = augment.augment_ragged(ds, batch_params(), args.crop, target)
        ev[k][1].record()
        tr.step(x, t)
        ev[k][2].record()
    torch.cuda.synchronize()
    loop_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    aug_ms = np.array([a.elapsed_time(b) for a, b, _ in ev])
    step_ms = np.array([b.elapsed_time(c) for _, b, c in ev])
    # augmentation kernel alone, back to back (its dims check included)
    reps = 50
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        augment.augment_ragged(ds, batch_params(), args.crop, target)
    e.record()
    torch.cuda.synchronize()
    aug_alone_ms = s.elapsed_time(e) / reps
    idx = list(range(min(args.val, len(ds))))
    tr.evaluate(ds, idx)                 # warm: plan creation, first launches
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    val = tr.evaluate(ds, idx)
    val_ms = (time.perf_counter() - t0) * 1e3 / len(idx)
    try:
        smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().split('\n')[0]
    except (OSError, subprocess.SubprocessError):
        smi = torch.cuda.get_device_name(0)
    res = {
        'gpu': smi, 'crop': args.crop, 'batch': args.batch, 'sources': len(ds), 'source_width': 1024,
        'source_heights_mean': float(heights.mean()), 'odd_height_sources': int((heights % 2).sum()),
        'timed_batches': args.steps,
        'augment_ms_per_batch_median': float(np.median(aug_ms)), 'augment_ms_per_batch_back_to_back': aug_alone_ms,
        'step_ms_median': float(np.median(step_ms)), 'loop_ms_per_batch': loop_ms,
        'augment_share_of_step': float(np.median(aug_ms) / np.median(step_ms)),
        'validation_images': len(idx), 'validation_ms_per_image': val_ms,
        'validation_mean_height': float(np.mean(heights[idx])), 'val_loss': val['loss'], 'val_miou': val['miou'],
    }
    text = json.dumps(res, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text + '\n')


if __name__ == '__main__':
    main()
