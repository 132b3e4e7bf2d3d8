"""predict.py on folders that are not standard scans: the per-image route of models.py (``Preprocessor.preprocess_images``
then ``NeuralBarkCalculator.predict``) against the folder pipeline's mixed route, on two folders on tmpfs:

    (a) ``png``:   64 synthetic 4096^2 scans saved as RGB PNG (the standard scans, converted to save disk);
    (b) ``mixed``: 64 files cycling through 4096^2 BMPs of both row orders, a 4096^2 PNG, 3000x2000 / 2048x4096 /
                   1500x1300 PNGs, a 1200x1001 BMP (padded rows), a 1024^2 grey PNG, and 900x700 RGBA, 640x600 palette and
                   500x700 JPEG files that need no resize.

    python tools/cli_mixed_profile.py [--out profiles/r03_cli_mixed_profile.txt] [--images 64] [--repeats 2]

Both routes write every output file (processed, dual and combined images, final_stats.csv) with --exclude_nodes.  The
figure is images / wall second from the first read to the CSV, model construction excluded, after one untimed run of each
route on the same folder; the two routes alternate ``--repeats`` times.  ``read_s`` / ``save_s`` are summed over the IO
threads: file reads (pixel-array copy or PIL decode) and output encoding.  For the per-image route they are the time spent
in ``Preprocessor._load_raw`` and in PIL's ``Image.save`` plus the combined-image writer."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch
from PIL import Image

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def write_bmp(path, rgb, top_down=False):
    import struct
    h, w, _ = rgb.shape
    pitch = (w * 3 + 3) & ~3
    buf = np.zeros((h, pitch), np.uint8)
    buf[:, :w * 3] = (rgb if top_down else rgb[::-1])[:, :, ::-1].reshape(h, w * 3)
    with open(path, 'wb') as f:
        f.write(b'BM' + struct.pack('<IHHI', 54 + buf.size, 0, 0, 54))
        f.write(struct.pack('<IiiHHIIiiII', 40, w, -h if top_down else h, 1, 24, 0, buf.size, 2835, 2835, 0, 0))
        f.write(buf.tobytes())


def make_folder(root, kind, n):
    """n files over the three wood types; ``unique`` distinct images, the rest hard links (decode cost is per file)."""
    from oracle import synth

    def banded(h, w, seed, top, bottom):
        img = synth.texture_u8(h, w, seed)
        img[:top], img[h - bottom:] = 0, 0
        return img

    scan = lambda s: synth.raw_image_u8(s, 4096)[0]      # noqa: E731
    if kind == 'png':
        makers = [('.png', lambda p, s=s: Image.fromarray(scan(600 + s)).save(p, compress_level=1)) for s in range(8)]
    else:
        makers = [('.bmp', lambda p: write_bmp(p, scan(701))),
                  ('.bmp', lambda p: write_bmp(p, scan(702), top_down=True)),
                  ('.png', lambda p: Image.fromarray(scan(703)).save(p, compress_level=1)),
                  ('.png', lambda p: Image.fromarray(banded(3000, 2000, 704, 300, 200)).save(p, compress_level=1)),
                  ('.png', lambda p: Image.fromarray(banded(2048, 4096, 705, 100, 0)).save(p, compress_level=1)),
                  ('.png', lambda p: Image.fromarray(banded(1500, 1300, 706, 120, 80)).save(p, compress_level=1)),
                  ('.bmp', lambda p: write_bmp(p, banded(1200, 1001, 707, 50, 50))),
                  ('.png', lambda p: Image.fromarray(banded(1024, 1024, 708, 60, 30)[:, :, 1]).save(p)),
                  ('.png', lambda p: Image.fromarray(np.dstack([synth.texture_u8(900, 700, 709), np.full((900, 700, 1), 255, np.uint8)])).save(p)),
                  ('.png', lambda p: Image.fromarray(synth.texture_u8(640, 600, 710)).quantize(64).save(p)),
                  ('.jpg', lambda p: Image.fromarray(synth.texture_u8(500, 700, 711)).save(p, quality=90))]
    made = {}
    for i in range(n):
        wood = synth.WOOD_TYPES[i * 3 // n]
        os.makedirs(os.path.join(root, 'samples', wood), exist_ok=True)
        k = i % len(makers)
        ext, make = makers[k]
        p = os.path.join(root, 'samples', wood, 'img_%04d%s' % (i, ext))
        if k in made:
            os.link(made[k], p)
        else:
            make(p)
            made[k] = p


class _Clock:
    """Thread-summed time spent inside wrapped functions."""

    def __init__(self):
        self.s, self.lock = 0.0, threading.Lock()

    def wrap(self, fn):
        def timed(*a, **k):
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                with self.lock:
                    self.s += time.perf_counter() - t0
        return timed


def per_image_route(root, calc, device):
    """Preprocessor.preprocess_images + NeuralBarkCalculator.predict, with read_s / save_s."""
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import models, pipeline
    read, save = _Clock(), _Clock()
    saved = (models.Preprocessor._load_raw, Image.Image.save, pipeline.write_combined)
    models.Preprocessor._load_raw = read.wrap(saved[0])
    Image.Image.save = save.wrap(saved[1])
    pipeline.write_combined = save.wrap(saved[2])
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        processed = nbc.Preprocessor(device=device).preprocess_images(root)
        rows = calc.predict(root, True, processed=processed)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        models.Preprocessor._load_raw, Image.Image.save, pipeline.write_combined = saved
    return dt, read.s, save.s, rows


def pipeline_route(root, pipe):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rows = pipe.run(root, True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, pipe.last_timing['read_s'], pipe.last_timing['save_s'], rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_cli_mixed_profile.txt')
    ap.add_argument('--images', type=int, default=64)
    ap.add_argument('--repeats', type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('cli_mixed_profile: no CUDA device (this measures the B200 path; there is nothing to time on the CPU)')
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import pipeline, predict as npredict
    from neuralbarkcalculator_b200.dataset import make_dataset
    from oracle import model as omodel
    device = 'cuda:0'
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True).stdout.strip()
    g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'model_small.npz'))
    sd = omodel.synthetic_state_dict(seed=0, head=(g['head_w'], g['head_b']))
    calc = nbc.NeuralBarkCalculator(None, device, state_dict=sd)
    pipe = pipeline.FolderPipeline(calc)
    base = '/dev/shm' if os.path.isdir('/dev/shm') else None
    lines = ['# tools/cli_mixed_profile.py: %d images per folder, %d timed runs per route, GPU %s, %d host cores'
             % (args.images, args.repeats, gpu, os.cpu_count()),
             '# folder  route       images/s   wall_s   read_s   save_s']
    result = {'gpu': gpu, 'images': args.images, 'folders': {}}
    for kind in ('png', 'mixed'):
        root = tempfile.mkdtemp(prefix='nbc_mixed_', dir=base)
        try:
            make_folder(root, kind, args.images)
            assert not pipeline.supported(make_dataset(root))
            runs = {'per_image': [], 'pipeline': []}
            for it in range(args.repeats + 1):
                for route in ('per_image', 'pipeline'):
                    shutil.rmtree(os.path.join(root, 'processed'), ignore_errors=True)
                    shutil.rmtree(os.path.join(root, 'results'), ignore_errors=True)
                    npredict.generate_folders(root, False)
                    r = per_image_route(root, calc, device) if route == 'per_image' else pipeline_route(root, pipe)
                    if it > 0:           # the first run of each route warms the plan, the allocator and the page cache
                        runs[route].append(r[:3])
                    with open(os.path.join(root, 'results', 'final_stats.csv'), 'rb') as f:
                        csv_bytes = f.read()
                    if route == 'per_image':
                        ref_csv = csv_bytes
                    else:
                        assert csv_bytes == ref_csv, 'the two routes wrote different CSVs'
            result['folders'][kind] = {}
            for route, rs in runs.items():
                wall, read_s, save_s = (float(np.mean([r[k] for r in rs])) for k in range(3))
                ips = args.images / wall
                result['folders'][kind][route] = {'images_per_s': ips, 'wall_s': wall, 'read_s': read_s, 'save_s': save_s}
                lines.append('%-8s  %-10s %9.2f %8.3f %8.3f %8.3f' % (kind, route, ips, wall, read_s, save_s))
            f = result['folders'][kind]
            lines.append('%-8s  speed-up of the pipeline: %.2fx' % (kind, f['pipeline']['images_per_s'] / f['per_image']['images_per_s']))
        finally:
            shutil.rmtree(root, ignore_errors=True)
    text = '\n'.join(lines) + '\n' + json.dumps(result) + '\n'
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text)


if __name__ == '__main__':
    main()
