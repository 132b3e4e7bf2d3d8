"""Cost of flip test-time augmentation (``predict --tta``, ``evaluate --tta``) on one GPU, in one run:

* engine: ``PredictEngine.run_device`` on 64 device-resident standard scans (4096^2, bottom-up BGR) at chunk 16, for
  --tta none / h / hv: images per second over ``--rounds`` timed calls after a warm-up call;
* kernels: on one chunk of 16 processed images (the trimmed heights of the synthetic scans), CUDA-event times of the
  ragged flip copy (``ops.flip_ragged``), one network pass (``Plan.forward_ragged``), plain K3
  (``ops.upsample_argmax_ragged``) and the multi-view K3 (``ops.upsample_argmax_views_ragged``) for 2 and 4 views, each
  the median over ``--reps`` launches; the share of flips + multi-view K3 in the chunk's V network passes;
* CLI: ``predict.main`` wall clock (model construction included, every output file written) on a folder of 256 synthetic
  4096^2 BMPs on tmpfs (8 unique scans, the rest hard links), none / h / hv alternated over three rounds after a warm-up
  round (median);
* evaluate: ``evaluate.main`` wall clock (PNG loading included) and ``evaluate_plan`` time on a labelled folder of 48
  images 1024 wide, none / hv, each after a warm-up call.

The card's name and power limit are read with ``nvidia-smi`` in the same run and written beside the figures.

    python tools/tta_profile.py [--out profiles/r05_tta_profile.json] [--rounds 5] [--reps 20]"""
import argparse
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.fit_scaling import card  # noqa: E402

MODES = ('none', 'h', 'hv')


def event_ms(fn, reps):
    """Median CUDA-event time of fn() over reps launches (after two warm-up calls)."""
    for _ in range(2):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def engine_rates(calc, raws, rounds):
    from neuralbarkcalculator_b200 import engine
    out = {}
    for mode in MODES:
        eng = engine.PredictEngine(calc.model, 'cuda:0', chunk=16, tta=mode)
        eng.run_device(raws)
        torch.cuda.synchronize()
        times = []
        for _ in range(rounds):
            t0 = time.perf_counter()
            eng.run_device(raws)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        out[mode] = {'images_per_s': len(raws) / statistics.median(times), 'median_s': statistics.median(times),
                     'min_s': min(times), 'max_s': max(times)}
        del eng
    return out


def kernel_costs(calc, raws, reps):
    from neuralbarkcalculator_b200 import ops
    procs, heights = [], []
    for r in raws[:16]:
        out, fl = ops.preprocess_4x(r, 4096, 4096, bgr=True, bottom_up=True)
        first, last = fl.tolist()
        procs.append(out.view(1024, 1024, 3))
        heights.append(last - first)
    canvas = torch.stack(procs).contiguous()
    hs = torch.tensor(heights, dtype=torch.int32, device='cuda:0')
    plan = calc.model.native_plan()
    scratch = torch.empty_like(canvas)
    lows = [plan.forward_ragged(canvas, heights=hs).clone() for _ in range(4)]
    mask = torch.empty((16, 1024, 1024), dtype=torch.uint8, device='cuda:0')
    res = {'chunk': 16, 'heights': heights,
           'flip_ms': event_ms(lambda: ops.flip_ragged(canvas, hs, 3, out=scratch), reps),
           'network_ms': event_ms(lambda: plan.forward_ragged(canvas, heights=hs, out=lows[0]), reps),
           'k3_1view_ms': event_ms(lambda: ops.upsample_argmax_ragged(lows[0], hs, (1024, 1024), out=mask), reps)}
    for mode in ('h', 'hv'):
        flags = ops.tta_views(mode)[1]
        V = len(flags)
        k3 = event_ms(lambda: ops.upsample_argmax_views_ragged(lows[:V], flags, hs, (1024, 1024), out=mask), reps)
        extra = (V - 1) * res['flip_ms'] + k3
        res[mode] = {'views': V, 'k3_views_ms': k3, 'flips_plus_k3_ms': extra,
                     'share_of_network_passes': extra / (V * res['network_ms'])}
    return res


def cli_times(sd, base):
    import argparse as ap
    from oracle import synth
    from neuralbarkcalculator_b200 import predict as npredict
    root = tempfile.mkdtemp(prefix='nbc_tta_cli_', dir=base)
    try:
        synth.make_raw_folder(root, 256, size=4096, pool=8, seed0=500)
        out = {m: [] for m in MODES}
        for rnd in range(4):
            for mode in MODES:
                shutil.rmtree(os.path.join(root, 'processed'), ignore_errors=True)
                shutil.rmtree(os.path.join(root, 'results'), ignore_errors=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                npredict.main(ap.Namespace(root_path=root, device='cuda:0', exclude_nodes=True, only_preprocess=False, tta=mode),
                              state_dict=sd)
                torch.cuda.synchronize()
                if rnd > 0:            # round 0 warms up every mode
                    out[mode].append(time.perf_counter() - t0)
        n_files = sum(len(f) for sub in ('processed', 'results') for _, _, f in os.walk(os.path.join(root, sub)))
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return {m: {'seconds': v, 'images_per_s': 256 / statistics.median(v)} for m, v in out.items()}, n_files


def eval_times(sd, base):
    from PIL import Image
    from oracle import synth
    from neuralbarkcalculator_b200 import augment as naug, evaluate as nev
    root = tempfile.mkdtemp(prefix='nbc_tta_eval_', dir=base)
    try:
        rng = np.random.default_rng(0)
        for k in range(48):
            wood = ('sapin', 'epinette_gelee', 'epinette_non_gelee')[k % 3]
            h = int(rng.integers(500, 1025))
            for sub in ('samples', 'duals'):
                os.makedirs(os.path.join(root, sub, wood), exist_ok=True)
            Image.fromarray(synth.texture_u8(h, 1024, 700 + k)).save(os.path.join(root, 'samples', wood, 'im%02d.png' % k))
            dual = (synth.class_mask(h, 1024, 800 + k).astype(np.float32) * 127.5).astype(np.uint8)
            Image.fromarray(dual, mode='L').save(os.path.join(root, 'duals', wood, 'im%02d.png' % k))
        model = os.path.join(root, 'best_model.pt')
        torch.save(sd, model)
        out = {}
        ds = naug.load_dataset(root, 'cuda:0')
        plan = nev.make_plan(sd, 'cuda:0')
        args = lambda mode: nev.parse_args([root, '--model', model, '--out', os.path.join(root, 'eval_%s.tsv' % mode), '--tta', mode])  # noqa: E731
        for mode in ('none', 'hv'):
            nev.main(args(mode))
            nev.evaluate_plan(plan, ds, range(len(ds)), 'lovasz', tta=mode)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nev.evaluate_plan(plan, ds, range(len(ds)), 'lovasz', tta=mode)
            torch.cuda.synchronize()
            t_plan = time.perf_counter() - t0
            t0 = time.perf_counter()
            nev.main(args(mode))
            torch.cuda.synchronize()
            out[mode] = {'evaluate_main_s': time.perf_counter() - t0, 'evaluate_plan_s': t_plan}
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r05_tta_profile.json'))
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=20)
    args = ap.parse_args()
    import neuralbarkcalculator_b200 as nbc
    from oracle import model as omodel, synth
    sd = omodel.synthetic_state_dict(seed=3, branch_gain=0.1, calibration='features', logit_std=0.6, class_bias=(0.8, 0.1, -1.1))
    calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=sd)
    uniq = []
    for i in range(8):
        img, _, _ = synth.raw_image_u8(900 + i, 4096)
        uniq.append(torch.from_numpy(np.ascontiguousarray(img[::-1, :, ::-1]).reshape(-1)).to('cuda:0'))
    raws = [uniq[i % 8].clone() for i in range(64)]
    res = {'card': card(), 'precision': calc.model._precision}
    res['engine'] = engine_rates(calc, raws, args.rounds)
    res['kernels'] = kernel_costs(calc, raws, args.reps)
    del raws, uniq
    torch.cuda.empty_cache()
    base = '/dev/shm' if os.path.isdir('/dev/shm') else None
    res['cli'], res['cli_files_per_run'] = cli_times(sd, base)
    res['evaluate'] = eval_times(sd, base)
    res['host_cores'] = os.cpu_count()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
