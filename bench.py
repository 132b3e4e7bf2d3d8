"""bench.py -- headline benchmark of the B200 segmentation hot path (see the contract in DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload predict64|batch32|train|cli]
                    [--precision bf16|fp16] [--dump-outputs DIR]

workload predict64 (default, BASELINE.json configs[1]): a "step" is one pass of the predict hot path over a batch
of 64 synthetic raw 4096x4096x3 scans (BMP pixel arrays: BGR, bottom-up, dark bands) with --exclude_nodes:
K1 resize+trim -> FCN-ResNet50 (fp16 storage by default, tcgen05) -> K3 upsample+argmax -> K5 region removal + class counts.
  value : images/s, raw scans resident in HBM when the timed region starts (3.2 GB per rank, >> the 126 MB L2)
  e2e   : images/s through PredictEngine.submit_host / collect (the two halves of run_host): pinned host buffers in
          (inside the timed region; the engine copies only the rows between a scan's all-zero dark bands and counts the
          bytes it copies -> h2d_bytes_per_step), masks + counts copied back to pinned host memory and collected every
          step; step k+1 is submitted before step k is collected, as a folder-sized predict run does
  roofline : the tensor-core conv launches of one network pass, per-launch CUDA events, against the BURST 16-bit peak (they
          are timed alone); roofline.whole_step = algorithmic conv FLOPs of the step / ms_per_step against the SUSTAINED peak
workload batch32 (configs[2]): model-only at 1024^2, u8 [32,1024,1024,3] -> mask + counts (e2e: images from / masks to pinned memory).
workload train (configs[3]): one training step (train-mode forward, weighted CE, backward, NCCL all-reduce, Adam), batch 8
per GPU at 1024^2; roofline = conv FLOPs of the step / whole step time; e2e = images + targets from pinned host memory,
loss read back every step.
workload cli (configs[1] literally): predict.py ROOT --exclude_nodes on a folder of 4096^2 BMP files on tmpfs, every output
file written; wall clock.
--impl reference times the CPU oracle (restated reference path, torch CPU f32 with all host threads) on a bounded
sample: one image per step (predict) / one 512^2 crop (train).  Multi-GPU: one process per GPU (torchrun), images sharded,
no collective on the data path; time = max over ranks."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RAW = 4096
BATCH = 64


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='predict64', choices=['predict64', 'batch32', 'train', 'cli'])
    ap.add_argument('--batch', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--precision', default='fp16', choices=['bf16', 'fp16'],
                    help='16-bit storage format of activations / weights on the predict path (same tcgen05 kind::f16 rate); '
                         'fp16 is the shipped default (meets the parity bar), bf16 is opt-in')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / '
                         'float64, at most 64 MB; rank 0), to compare two builds output for output on the same seeded inputs')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    return args


def peaks():
    """(HBM GB/s, dense 16-bit TFLOP/s burst, sustained, kind): MEASURED_PEAKS.json (driver-written) or the profiling
    recipe's fallback.  Burst is the denominator for a kernel timed alone (per-launch events), sustained for a long step."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        burst = d.get('bf16_tflops', 1590.0)
        return d.get('hbm_gbs', 6650.0), burst, d.get('bf16_tflops_sustained', burst), 'measured'
    return 6650.0, 1590.0, 1590.0, 'fallback'


WORKLOADS = {
    'predict64': 'predict.py --exclude_nodes hot path on %d synthetic 4096x4096 raw scans per GPU (K1 resize+trim, '
                 'FCN-ResNet50 3-class random-init, K3 upsample+argmax, K5 <150px region removal + counts)',
    'batch32': 'model-only batched inference: u8 [%d,1024,1024,3] -> mask + counts (configs[2])'}


def predict_config(kind, n_img, gpus):
    """The `config` object of a predict line -- the SAME keys and values for both arms (--impl ours / reference)."""
    if kind == 'batch32':
        l2 = ('inputs %.0f MB per rank, but every step streams %.1f GB of activations through HBM between reuses; no flush '
              'needed' % (n_img * 1024 * 1024 * 3 / 1e6, n_img * 0.168))
    else:
        l2 = 'inputs (%.1f GB per rank) larger than L2; no flush needed' % (n_img * RAW * RAW * 3 / 1e9)
    return {'workload': WORKLOADS[kind] % n_img, 'images_per_step_per_gpu': n_img,
            'parallelism': 'dp%d (images sharded, no collective)' % gpus, 'l2': l2}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=8)      # a query that started inside the timed region still counts (nvidia-smi takes ~0.1-0.3 s)
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ---------------------------------------------------------------------------------------------------- synthetic data
def synth_raw_gpu(n, dev, seed0):
    """n raw scans as BMP pixel arrays (BGR, bottom-up) in HBM: correlated texture + exact-zero dark bands."""
    g = torch.Generator(device=dev)
    mean = torch.tensor([0.4401, 0.6139, 0.7399], device=dev).view(1, 1, 3)   # BGR order
    std = torch.tensor([0.1271, 0.1272, 0.1068], device=dev).view(1, 1, 3)
    raws, bands = [], []
    for i in range(n):
        g.manual_seed(seed0 + i)
        lo = torch.randn(1, 3, RAW // 64, RAW // 64, generator=g, device=dev)
        f = torch.nn.functional.interpolate(lo, size=(RAW, RAW), mode='bicubic', align_corners=False)[0].permute(1, 2, 0)
        f = f + 0.35 * torch.randn(RAW, RAW, 3, generator=g, device=dev)
        img = ((mean + std * f) * 255.0).clamp_(0, 255).round_().to(torch.uint8)
        rng = np.random.default_rng(seed0 + i)
        top, bottom = int(rng.integers(400, 1201)), int(rng.integers(400, 1201))
        img[:bottom] = 0              # memory is bottom-up: the first rows in memory are the bottom of the picture
        img[RAW - top:] = 0
        raws.append(img.contiguous().view(-1))
        bands.append((top, bottom))
        del f, lo
    return raws, bands


def synth_processed_cpu(seed, rows=None):
    from oracle import synth
    raw, top, bottom = synth.raw_image_u8(seed, RAW)
    return raw


# ---------------------------------------------------------------------------------------------------- output dump
# --dump-outputs keeps fixed, seeded samples where the whole output would not fit in DUMP_LIMIT: masks of 64 images as
# float32 are 256 MB, the weights of a training step 132 MB.  The positions depend on nothing but the seed, so two builds
# are compared at the same pixels and the same weights.
DUMP_LIMIT = 64 << 20
DUMP_PIXELS = 1 << 17       # per mask canvas of 1024 x 1024: one pixel in eight (32 MB for 64 images)
DUMP_WEIGHTS = 1 << 20      # of the 32.9 M weights and BatchNorm statistics


def sample_index(n, k, seed=0):
    """k sorted positions out of n, the same from run to run."""
    return np.sort(np.random.default_rng(seed).choice(n, size=min(k, n), replace=False))


def mask_sample(masks, heights=None):
    """masks: u8 class canvases [n, H, W] (device or host); heights: rows of each canvas that belong to its image (None:
    all of them).  -> float32 [n, DUMP_PIXELS], the class at fixed canvas positions, -1 where a position lies below the
    image (those canvas rows are not part of the result)."""
    n, H, W = masks.shape
    idx = torch.from_numpy(sample_index(H * W, DUMP_PIXELS)).to(masks.device)
    out = masks.reshape(n, H * W)[:, idx].float()
    if heights is not None:
        out[(idx // W).view(1, -1) >= heights.to(out.device).view(-1, 1)] = -1.0
    return out.cpu().numpy()


def weight_sample(trainer):
    """float32 [DUMP_WEIGHTS]: the trainer's weights and BatchNorm statistics (state_dict order) at fixed positions."""
    flat = torch.cat([v.detach().float().flatten().cpu() for v in trainer.state_dict().values() if v.is_floating_point()])
    return flat[torch.from_numpy(sample_index(flat.numel(), DUMP_WEIGHTS))].numpy()


def cli_outputs(root, rows):
    """What predict.py left for its caller: the numbers of final_stats.csv and the dual masks of results/outputs (classes
    stored as 0 / 127 / 255), the masks on 1024-wide canvases like the engine's."""
    from PIL import Image
    stats = np.array([[float(v) for v in r[2:]] for r in rows[1:]], dtype=np.float64)
    masks = torch.zeros((len(rows) - 1, RAW // 4, RAW // 4), dtype=torch.uint8)
    heights = torch.zeros(len(rows) - 1, dtype=torch.int64)
    for i, (name, wood) in enumerate(r[:2] for r in rows[1:]):
        m = torch.from_numpy(np.asarray(Image.open(os.path.join(root, 'results', 'outputs', wood, name))) // 127)
        masks[i, :m.shape[0], :m.shape[1]] = m
        heights[i] = m.shape[0]
    return {'stats': stats, 'heights': heights.numpy().astype(np.float64), 'mask_sample': mask_sample(masks, heights)}


def write_dump(path, arrays):
    """arrays: name -> float32 / float64 numpy array, written as path/<name>.npy."""
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError('--dump-outputs: %s is %s, not float32 / float64' % (name, a.dtype))
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


# ---------------------------------------------------------------------------------------------------- reference arm
def train_config(B, gpus):
    """`config` of a training line, identical for both arms."""
    return {'workload': 'training step: FCN-ResNet50 3-class, max-of-index weighted CE, batch %d per GPU at 1024x1024, Adam '
                        'lr 5e-4 wd 2e-3, dropout 0.8, NCCL all-reduce of the gradients (configs[3])' % B,
            'images_per_step_per_gpu': B, 'parallelism': 'dp%d' % gpus,
            'l2': 'activations of one step (tens of GB) are far larger than L2; no flush needed'}


def time_reference(steps, warmup, sd, kind='predict64'):
    """CPU oracle (restated reference predict path, f32, eval) on one image per step, all host threads: a raw 4096^2 scan
    through the whole path (predict64), or one processed 1024^2 image through model + argmax + region removal (batch32)."""
    from oracle import model as omodel, postprocess as opost, preprocess as opre, synth
    torch.set_num_threads(os.cpu_count())
    net = omodel.load_model(sd)
    times = []
    for s in range(warmup + steps):
        raw = synth.raw_image_u8(1000 + s, RAW)[0] if kind == 'predict64' else synth.texture_u8(1024, 1024, 1000 + s)
        t0 = time.perf_counter()
        proc = opre.preprocess_u8(raw)[0] if kind == 'predict64' else raw
        x = omodel.normalise_u8(proc)
        with torch.no_grad():
            logits = net(x)
        mask = torch.argmax(logits, dim=1)[0].numpy()
        mask = opost.exclude_nodes(opost.remove_small_zones_2d(mask))
        opost.class_stats_strings(mask)
        t1 = time.perf_counter()
        if s >= warmup:
            times.append(t1 - t0)
    return len(times) / sum(times), times


def time_reference_train(sd, hw=512):
    """CPU oracle training step (plain torch f32: train(), forward, weighted CE, backward, Adam -- the reference's
    __main__.py:231-269 step) on a bounded sample: ONE hw x hw crop (the reference trains on 512 crops, __main__.py:159),
    scaled to 1024^2-image units by the pixel ratio."""
    from oracle import synth, train as otrain, model as omodel
    torch.set_num_threads(os.cpu_count())
    x = omodel.normalise_u8(synth.texture_u8(hw, hw, 3))
    t = torch.from_numpy(synth.class_mask(hw, hw, 4)).long().unsqueeze(0)
    otrain.train_step(sd, x, t, dropout=0.8)          # warm-up
    t0 = time.perf_counter()
    otrain.train_step(sd, x, t, dropout=0.8)
    dt = time.perf_counter() - t0
    scale = (hw * hw) / (1024.0 * 1024.0)
    return scale / dt, ('1 timed step (after 1 warm-up) of the CPU oracle on one %dx%d crop, batch 1, all host threads; '
                        'value scaled to 1024^2 images by the pixel ratio %.3f' % (hw, hw, scale))


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    from oracle import model as omodel
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'model_small.npz'))
    sd = omodel.synthetic_state_dict(seed=0, head=(g['head_w'], g['head_b']))
    kind = 'batch32' if args.workload == 'batch32' else 'predict64'

    if args.impl == 'reference':
        if rank != 0:
            return
        if args.workload == 'train':
            v, sample = time_reference_train(sd)
            print(json.dumps({'impl': 'reference', 'metric': 'images/sec (training step)', 'value': v, 'unit': 'images/s',
                              'n_gpus': args.gpus, 'steps': 1, 'warmup': 1, 'ms_per_step': 1000.0 / v, 'higher_is_better': True,
                              'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                              'config': train_config(args.batch or 8, args.gpus),
                              'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': os.cpu_count(), 'kind': 'port', 'sample': sample},
                              'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
            return
        v, times = time_reference(args.steps, args.warmup, sd, kind)
        line = {'impl': 'reference', 'metric': 'images/sec', 'value': v, 'unit': 'images/s', 'n_gpus': args.gpus,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * float(np.mean(times)),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': predict_config(kind, args.batch or (32 if kind == 'batch32' else BATCH), args.gpus),
                'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': os.cpu_count(), 'kind': 'port',
                                 'sample': '%d timed steps of 1 synthetic %s each through the CPU oracle (restated reference '
                                           'predict path without the matplotlib figure / PNG IO), batch 1 as models.py:249-250'
                                           % (args.steps, '4096^2 scan' if kind == 'predict64' else 'processed 1024^2 image')},
                'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line))
        return

    import torch.distributed as dist
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import _lib, engine
    from neuralbarkcalculator_b200 import distributed as ndist
    # one process per GPU: keep this rank's pinned staging buffers on the NUMA node of its GPU (see bind_to_gpu_numa)
    numa = ndist.bind_to_gpu_numa(local_rank) if world > 1 else {'numa_node': ndist.gpu_numa_node(local_rank), 'bound': False}

    calc = nbc.NeuralBarkCalculator(None, str(dev), state_dict=sd, precision=args.precision)
    eng = engine.PredictEngine(calc.model, dev)
    hbm_peak, tf_burst, tf_peak, peak_kind = peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup, drain=None):
        for _ in range(warmup):
            fn()
        if drain is not None:
            drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()        # inside the timed region: every submitted step is complete and its results are on the host
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    def dump(outputs):
        """--dump-outputs: outputs() -> what the last timed step returned; called right after the timed steps, before the
        end-to-end pass reuses the buffers."""
        if args.dump_outputs and rank == 0:
            write_dump(args.dump_outputs, outputs())

    if args.workload == 'train':
        # BASELINE.json configs[3]: one training step (fwd + weighted CE + bwd + all-reduce + Adam), batch 8 per GPU
        from oracle import synth
        from neuralbarkcalculator_b200.train import Trainer
        B = args.batch or 8
        imgs_h = torch.from_numpy(np.stack([synth.texture_u8(1024, 1024, 100 * rank + i) for i in range(2)]))
        imgs_h = imgs_h.repeat((B + 1) // 2, 1, 1, 1)[:B].contiguous().pin_memory()
        tgt_h = torch.from_numpy(np.stack([synth.class_mask(1024, 1024, 200 * rank + i) for i in range(2)]))
        tgt_h = tgt_h.repeat((B + 1) // 2, 1, 1)[:B].contiguous().pin_memory()
        imgs, tgt = imgs_h.to(dev), tgt_h.to(dev)
        tr = Trainer(sd, B, 1024, 1024, device=str(dev), dropout=0.8)
        res = {}

        def step():
            res['loss'] = tr.step(imgs, tgt)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms, launches = timed(step, args.steps, args.warmup)
        clocks = sampler.summary()
        dump(lambda: {'loss': np.array([float(res['loss'])], dtype=np.float64), 'weights_sample': weight_sample(tr)})
        # end to end: this step's images and targets come from pinned host memory, the loss is read back every step
        imgs_d, tgt_d = torch.empty_like(imgs), torch.empty_like(tgt)

        def step_host():
            imgs_d.copy_(imgs_h, non_blocking=True)
            tgt_d.copy_(tgt_h, non_blocking=True)
            res['loss_host'] = float(tr.step(imgs_d, tgt_d).item())
        ms_h, _ = timed(step_host, args.steps, max(1, args.warmup))
        if rank == 0:
            # algorithmic FLOPs of the convolutions of one step: forward + data gradient + weight gradient
            # (2*MAC; 1106.64 GFLOP forward per 1024^2 image, SURVEY.md 8a-2; the stem has no data gradient)
            step_flops = (3 * 1106.64e9 - 4.93e9) * B
            achieved = step_flops * args.steps / (ms / 1000.0) / 1e12
            cpu_base = None
            if not args.no_cpu_baseline and world == 1:
                v, sample = time_reference_train(sd)
                cpu_base = {'value': v, 'unit': 'images/s', 'cores': os.cpu_count(), 'kind': 'port', 'sample': sample}
            line = {'metric': 'images/sec (training step)', 'value': world * B * args.steps / (ms / 1000.0), 'unit': 'images/s',
                    'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps,
                    'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
                    'config': train_config(B, world),
                    'clocks': clocks, 'gpu_launches': launches, 'loss': float(res['loss']),
                    'gradient_exchange': ('%d overlapped buckets' % len(tr.gradient_buckets())) if tr.bucket_mb > 0 else 'one all-reduce after the backward',
                    'e2e': {'value': world * B * args.steps / (ms_h / 1000.0), 'unit': 'images/s',
                            'h2d_bytes_per_step': int(imgs_h.numel() + tgt_h.numel()), 'd2h_bytes_per_step': 4,
                            'ms_per_step': ms_h / args.steps},
                    'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': tf_peak, 'unit': 'TFLOP/s',
                                 'frac': achieved / tf_peak, 'traffic': None, 'peak_kind': peak_kind + ' (sustained bf16)',
                                 'kernel': 'conv_tc_kernel / conv_tc_pair_kernel (forward + data gradient) and wgrad_tc_kernel: algorithmic conv FLOPs of '
                                           'the step / WHOLE step time (BatchNorm, loss, Adam and the all-reduce included), i.e. a '
                                           'lower bound on the kernels\' own rate'},
                    'cpu_baseline': cpu_base}
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    if args.workload == 'cli':
        # BASELINE.json configs[1] literally: `predict.py ROOT --exclude_nodes` on a folder of 64 synthetic 4096^2 BMPs
        # (files on tmpfs), every output file written.  Wall clock: file reads and PNG encoding are host work.
        import argparse as _ap
        import shutil
        import tempfile
        from oracle import synth
        from neuralbarkcalculator_b200 import predict as npredict
        B = args.batch or BATCH
        if os.environ.get('NBC_DEBUG_HANG'):      # all thread stacks after N seconds, then exit (debugging aid)
            import faulthandler
            faulthandler.dump_traceback_later(int(os.environ['NBC_DEBUG_HANG']), exit=True)
        base = '/dev/shm' if os.path.isdir('/dev/shm') else None
        root = tempfile.mkdtemp(prefix='nbc_cli_', dir=base)
        try:
            synth.make_raw_folder(root, B, size=RAW, pool=min(B, 8), seed0=500)
            ns = _ap.Namespace(root_path=root, device=str(dev), exclude_nodes=True, only_preprocess=False)
            times = []
            for it in range(args.warmup + args.steps):
                shutil.rmtree(os.path.join(root, 'processed'), ignore_errors=True)
                shutil.rmtree(os.path.join(root, 'results'), ignore_errors=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rows = npredict.main(ns, state_dict=sd)
                torch.cuda.synchronize()
                if it >= args.warmup:
                    times.append(time.perf_counter() - t0)
            n_files = sum(len(f) for _, _, f in os.walk(os.path.join(root, 'results'))) + sum(len(f) for _, _, f in os.walk(os.path.join(root, 'processed')))
            dump(lambda: cli_outputs(root, rows))
        finally:
            shutil.rmtree(root, ignore_errors=True)
        if rank == 0:
            v = B * len(times) / sum(times)
            print(json.dumps({'metric': 'images/sec (predict.py CLI, files in, files out)', 'value': v, 'unit': 'images/s', 'n_gpus': 1,
                              'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * sum(times) / len(times),
                              'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
                              'config': {'workload': 'predict.py ROOT --exclude_nodes on %d synthetic 4096x4096 24-bit BMPs on tmpfs: '
                                                     'BMP read, K1, FCN-ResNet50, K3, K5, processed + dual PNG encode, CSV (configs[1]); '
                                                     'includes model construction and weight packing each step' % B,
                                         'timing': 'wall clock around predict.main(); %d files written per step' % n_files,
                                         'host_cores': os.cpu_count()},
                              'gpu_launches': _lib.launch_count(), 'e2e': {'value': v, 'unit': 'images/s',
                              'h2d_bytes_per_step': B * RAW * RAW * 3, 'd2h_bytes_per_step': B * 4 * 1024 * 1024},
                              'roofline': None, 'cpu_baseline': None, 'rows': len(rows)}))
        return

    if args.workload == 'batch32':
        B = args.batch or 32
        from oracle import synth
        imgs = torch.from_numpy(np.stack([synth.texture_u8(1024, 1024, 100 * rank + i) for i in range(min(B, 4))])).to(dev)
        imgs = imgs.repeat((B + imgs.shape[0] - 1) // imgs.shape[0], 1, 1, 1)[:B].contiguous()
        from neuralbarkcalculator_b200 import ops
        last = {}

        def step():
            mask = calc.model.predict_mask_u8(imgs)
            last['out'] = ops.remove_small_zones_u8(mask, 150, exclude_nodes=True)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms, launches = timed(step, args.steps, args.warmup)
        clocks = sampler.summary()
        dump(lambda: {'counts': last['out'][1].cpu().numpy().astype(np.float64), 'mask_sample': mask_sample(last['out'][0])})
        n_img = B
        mean_rows, prof_n, prof_h = 1024.0, B, 1024
        # end to end: the processed u8 images come from pinned host memory, masks + counts go back to pinned host memory
        imgs_h = imgs.cpu().pin_memory()
        imgs_d = torch.empty_like(imgs)
        mask_h = torch.empty((B, 1024, 1024), dtype=torch.uint8).pin_memory()
        cnt_h = torch.empty((B, 3), dtype=torch.int32).pin_memory()

        def step_host():
            imgs_d.copy_(imgs_h, non_blocking=True)
            mask = calc.model.predict_mask_u8(imgs_d)
            mask, cnt = ops.remove_small_zones_u8(mask, 150, exclude_nodes=True)
            mask_h.copy_(mask, non_blocking=True)
            cnt_h.copy_(cnt, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e2e = None
        if not args.no_e2e:
            ms_h, _ = timed(step_host, args.steps, max(1, args.warmup))
            e2e = {'value': world * B * args.steps / (ms_h / 1000.0), 'unit': 'images/s', 'h2d_bytes_per_step': int(imgs_h.numel()),
                   'd2h_bytes_per_step': int(mask_h.numel() + cnt_h.numel() * 4), 'ms_per_step': ms_h / args.steps}
    else:
        B = args.batch or BATCH
        raws, _ = synth_raw_gpu(B, dev, 10000 * rank)
        torch.cuda.synchronize()

        last = {}

        def step():
            last['out'] = eng.run_device(raws, bgr=True, bottom_up=True, exclude_nodes=True)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms, launches = timed(step, args.steps, args.warmup)
        clocks = sampler.summary()
        counts, masks, heights = last['out']
        dump(lambda: {'counts': counts.cpu().numpy().astype(np.float64), 'heights': heights.cpu().numpy().astype(np.float64),
                      'mask_sample': mask_sample(masks, heights)})
        n_img = B
        mean_rows = float(last['out'][2].float().mean().item())      # trimmed heights of this rank's scans
        prof_n, prof_h = eng.chunk, 624
        e2e = None
        if not args.no_e2e:
            host = [torch.empty(RAW * RAW * 3, dtype=torch.uint8).pin_memory() for _ in range(B)]
            for h, r in zip(host, raws):
                h.copy_(r)
            # two sets of result buffers: step k+1 is submitted (its H2D copies start) before step k is collected
            masks_sets = [[torch.empty(1024 * 1024, dtype=torch.uint8).pin_memory() for _ in range(B)] for _ in range(2)]
            res, pending, turn = {}, [], [0]

            def step_host():
                pending.append(eng.submit_host(host, masks_sets[turn[0] & 1], bgr=True, bottom_up=True, exclude_nodes=True))
                turn[0] += 1
                if len(pending) == 2:
                    res['rows'], res['counts'], _ = eng.collect(pending.pop(0))

            def drain_host():
                while pending:
                    res['rows'], res['counts'], _ = eng.collect(pending.pop(0))
            h0 = eng.h2d_bytes
            ms_h, _ = timed(step_host, args.steps, max(1, args.warmup), drain_host)
            d2h = int(B * 1024 * 1024 + B * 12 + B * 8)     # mask canvases + counts + {first,last}
            # bytes the engine really copied per step (counted from the tensors it copies): the scans' all-zero dark bands
            # stay on the host (engine.py; NBC_ZERO_SPAN=0 copies everything)
            h2d = int((eng.h2d_bytes - h0) // (args.steps + max(1, args.warmup)))
            e2e = {'value': world * B * args.steps / (ms_h / 1000.0), 'unit': 'images/s',
                   'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': ms_h / args.steps,
                   'raw_bytes_per_step': B * RAW * RAW * 3, 'zero_band_rows_skipped': bool(eng.zero_span)}

    value = world * n_img * args.steps / (ms / 1000.0)

    # roofline of the dominant kernel (conv_tc): per-layer CUDA events over one forward of a representative image
    roof = None
    cpu_base = None
    if rank == 0:
        # The engine launches the network once per ragged chunk of scans (engine.DEFAULT_CHUNK); the trimmed height of the
        # synthetic scans averages 624 rows, so the representative launch is a dense [chunk,624,1024,3] batch.
        from oracle import synth
        chunk = prof_n
        one = torch.from_numpy(synth.texture_u8(prof_h, 1024, 5)).unsqueeze(0).to(dev)
        prof_img = one.repeat(chunk, 1, 1, 1).contiguous()
        plan = calc.model.native_plan()
        plan.profile(prof_img)
        reps = [plan.profile(prof_img) for _ in range(3)]
        layers = [(float(np.median([r[i][0] for r in reps])), reps[0][i][1]) for i in range(len(reps[0]))]
        conv = [(m, f) for (m, f) in layers[2:-1]]
        conv_ms, conv_fl = sum(m for m, _ in conv), sum(f for _, f in conv)
        tot_ms = sum(m for m, _ in layers)
        achieved = conv_fl / (conv_ms * 1e-3) / 1e12
        traffic, tensor_pct, ncu_src = None, None, None
        tp = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')     # dram bytes per launch from the committed ncu capture
        if os.path.exists(tp) and kind == 'predict64':      # the capture is of this workload's representative launch set
            tj = json.load(open(tp))
            traffic = tj.get('conv_tc_dram_bytes_per_launch')
            tensor_pct = tj.get('conv_tc_tensor_pipe_active_pct_time_weighted')
            ncu_src = tj.get('source')
        # whole step: algorithmic conv FLOPs of everything the step processed / the driver-visible step time (K1, K3,
        # K5, maxpool, launch gaps included) -- against the SUSTAINED peak, the step being a long back-to-back run
        step_flops = conv_fl / chunk * (mean_rows / float(prof_h)) * n_img
        step_tf = step_flops * args.steps / (ms / 1000.0) / 1e12
        roof = {'bound': 'tensor', 'achieved': achieved, 'peak': tf_burst, 'unit': 'TFLOP/s', 'frac': achieved / tf_burst,
                'traffic': traffic, 'peak_kind': peak_kind + ' (burst 16-bit dense: the launches are timed alone, per-launch events)',
                'kernel': 'conv_tc_kernel / conv_tc_pair_kernel (CTA pairs, cta_group::2): the %d tensor-core conv launches of one network pass over a chunk of %d scans '
                          '(dense [%d,%d,1024,3] batch; each first bottleneck runs conv3 + downsample '
                          'as one launch), per-launch CUDA events, median of 3; achieved = sum of algorithmic FLOPs / sum of '
                          'launch durations' % (len(conv), chunk, chunk, prof_h),
                'tensor_pipe_active_pct_ncu': tensor_pct,      # time-weighted over the same launches (profiles/ncu_traffic.json)
                'ncu_capture': ncu_src,
                'flops_per_launch_avg': conv_fl / len(conv), 'ms_per_launch_avg': conv_ms / len(conv),
                'conv_share_of_forward': conv_ms / tot_ms, 'forward_ms_per_image': tot_ms / chunk,
                'whole_step': {'achieved': step_tf, 'peak': tf_peak, 'frac': step_tf / tf_peak, 'unit': 'TFLOP/s',
                               'peak_kind': peak_kind + ' (sustained 16-bit dense)',
                               'what': 'algorithmic conv FLOPs of the %d images of a step / ms_per_step (every kernel of the hot '
                                       'path and all launch gaps inside)' % n_img}}
        if not args.no_cpu_baseline and world == 1:
            v, times = time_reference(3, 1, sd, kind)
            cpu_base = {'value': v, 'unit': 'images/s', 'cores': os.cpu_count(), 'kind': 'port',
                        'sample': '3 synthetic %s through the CPU oracle after 1 warm-up (restated reference predict path; no '
                                  'matplotlib figure, no file IO)' % ('4096^2 scans' if kind == 'predict64' else 'processed 1024^2 images')}
    if rank == 0:
        line = {'metric': 'images/sec', 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
                'config': predict_config(kind, n_img, world), 'numa': numa,
                'clocks': clocks, 'gpu_launches': launches, 'e2e': e2e, 'roofline': roof, 'cpu_baseline': cpu_base}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
