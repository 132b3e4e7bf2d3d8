"""What scoring a checkpoint on labelled images costs: plan creation, the per-image loop ``evaluate.evaluate`` ran before
the batched pass (restated here from the per-image ops it called), and ``evaluate.evaluate_plan`` at chunk 8 and 16, on
one B200, in one process; then the wall clock of ``python -m neuralbarkcalculator_b200.evaluate`` on 1, 2 and 8 GPUs
(as many as the box has).

    python tools/eval_profile.py [--out profiles/r03_eval_profile.txt] [--images 256] [--repeats 3]

Input: ``--images`` processed images 1024 wide with heights drawn from 343..1024, and their dual label images.  Times are
host-clock times over a whole arm ending in a device synchronise (the read-back of the rows), per image; the arms
alternate ``--repeats`` times after one warm-up run each, and the rows of the loop and of the batched pass are compared in
the same run.  The CLI times include process start, torch import, decoding the PNG folder and plan creation."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def per_image_loop(plan, ds, idx, loss='lovasz', chunk=8):
    """The loop ``evaluate.evaluate`` ran before the batched pass: per image, the bicubic upsample, the loss, argmax, two
    confusion matrices and the region removal."""
    from neuralbarkcalculator_b200 import evaluate as nev, ops
    from neuralbarkcalculator_b200.lovasz_losses import iou_from_confusion
    from neuralbarkcalculator_b200.utils import f1_from_confusion, get_pos_weight
    dev = ds.device
    w = get_pos_weight().to(device=dev, dtype=torch.float32).contiguous()
    order, losses, cms = [], [], []
    for i, full, lab in nev.image_logits(plan, ds, idx, chunk):
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        ce = ops.wce_fwd_bwd(full, lab, w, need_grad=False)[0] if loss != 'lovasz' else zero
        lov = ops.lovasz_softmax_fwd_bwd(full, lab, need_grad=False)[0] if loss != 'weighted_ce' else zero
        pred = ops.argmax3_u8(full)
        cm_iou = ops.confusion_matrix(pred, lab)
        ops.remove_small_zones_u8(pred, 150)
        order.append(i)
        losses.append(torch.stack([ce, lov]))
        cms.append(torch.stack([cm_iou, ops.confusion_matrix(pred, lab)]))
    losses = torch.stack(losses).cpu().numpy()
    cms = torch.stack(cms).cpu().numpy()
    rows = []
    for i, (ce, lov), (cm_iou, cm_f1) in zip(order, losses, cms):
        value = {'weighted_ce': ce, 'lovasz': lov, 'mixed': ce / np.float32(4) + lov}[loss]
        rows.append({'index': i, 'loss': float(value), 'miou': float(np.mean(iou_from_confusion(cm_iou))),
                     'f1': f1_from_confusion(cm_f1)})
    return rows


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_eval_profile.txt')
    ap.add_argument('--images', type=int, default=256)
    ap.add_argument('--repeats', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('eval_profile: no CUDA device (this measures the B200 path; there is nothing to time on the CPU)')
    from neuralbarkcalculator_b200 import augment, evaluate as nev
    from oracle import model as omodel
    from oracle import synth
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True, timeout=60).stdout.strip().split('\n')
    dev = torch.device('cuda:0')
    rng = np.random.default_rng(0)
    heights = rng.integers(343, 1025, args.images)
    images = [synth.texture_u8(int(h), 1024, 1000 + k) for k, h in enumerate(heights)]
    duals = [(synth.class_mask(int(h), 1024, 2000 + k).astype(np.float32) * 127.5).astype(np.uint8) for k, h in enumerate(heights)]
    ds = augment.DeviceDataset(images, duals, ['sapin'] * len(images), dev)
    sd = omodel.synthetic_state_dict(seed=3, branch_gain=0.1, calibration='features', logit_std=0.6, class_bias=(0.8, 0.1, -1.1))
    idx = list(range(len(ds)))
    plan_s = [_timed(lambda: nev.make_plan(sd, dev))[0] for _ in range(3)]
    plan = nev.make_plan(sd, dev)
    arms = {'per_image_loop': lambda: per_image_loop(plan, ds, idx),
            'batched_chunk8': lambda: nev.evaluate_plan(plan, ds, idx, 'lovasz', chunk=8)['rows'],
            'batched_chunk16': lambda: nev.evaluate_plan(plan, ds, idx, 'lovasz', chunk=16)['rows']}
    rows = {k: fn() for k, fn in arms.items()}                    # warm-up
    times = {k: [] for k in arms}
    for _ in range(args.repeats):
        for k, fn in arms.items():
            t, rows[k] = _timed(fn)
            times[k].append(t * 1e3 / len(idx))
    ref = rows['per_image_loop']
    identical = all(len(rows[k]) == len(ref) and all(
        a['index'] == b['index'] and a['loss'] == b['loss'] and a['miou'] == b['miou'] and np.array_equal(a['f1'], b['f1'])
        for a, b in zip(rows[k], ref)) for k in arms)
    res = {'gpu': smi[0], 'gpus_on_box': torch.cuda.device_count(), 'images': len(idx), 'width': 1024,
           'height_mean': float(heights.mean()), 'height_min': int(heights.min()), 'height_max': int(heights.max()),
           'plan_creation_s': [round(v, 4) for v in plan_s],
           'ms_per_image_median': {k: float(np.median(v)) for k, v in times.items()},
           'ms_per_image_all': {k: [round(x, 3) for x in v] for k, v in times.items()},
           'rows_identical': identical}
    # the command, on a PNG folder of the same images
    with tempfile.TemporaryDirectory() as tmp:
        root = os.path.join(tmp, 'data')
        for sub in ('samples', 'duals'):
            os.makedirs(os.path.join(root, sub, 'sapin'))
        for k, (img, dual) in enumerate(zip(images, duals)):
            Image.fromarray(img).save(os.path.join(root, 'samples', 'sapin', 'im%04d.png' % k), compress_level=1)
            Image.fromarray(dual, mode='L').save(os.path.join(root, 'duals', 'sapin', 'im%04d.png' % k), compress_level=1)
        model = os.path.join(tmp, 'model.pt')
        torch.save(sd, model)
        env = dict(os.environ, PYTHONPATH=ROOT)
        cli, outs = {}, {}
        for g in (1, 2, 8):
            if g > torch.cuda.device_count():
                continue
            out = os.path.join(tmp, 'eval%d.tsv' % g)
            cmd = [sys.executable, '-m', 'neuralbarkcalculator_b200.evaluate', root, '--model', model, '--out', out]
            if g > 1:
                cmd = [sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', str(g)] + cmd[1:]
            t0 = time.perf_counter()
            done = subprocess.run(cmd, cwd=tmp, env=env, capture_output=True, text=True, timeout=1800)
            cli['%d_gpu_s' % g] = round(time.perf_counter() - t0, 3)
            if done.returncode != 0:
                raise SystemExit('eval_profile: the command failed on %d GPUs:\n%s' % (g, done.stderr[-3000:]))
            with open(out, 'rb') as f:
                outs[g] = f.read()
        res['cli_wall'] = cli
        res['cli_files_identical'] = len(set(outs.values())) == 1
    text = json.dumps(res, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text + '\n')


if __name__ == '__main__':
    main()
