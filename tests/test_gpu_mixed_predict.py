"""The mixed route of the folder pipeline on the GPU: K1 for a chunk of heterogeneous raw images against the per-image
entries, predict.py on a folder of mixed inputs against the per-image route of models.py, sharded runs, and the standard
route left on its uniform 4x path (``pytest -m gpu``)."""
import argparse
import os
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bmp_bytes(rgb, top_down=False):
    """24-bit BMP pixel array (BGR, rows padded to 4 bytes) -> (pixel array bytes, pitch)."""
    h, w, _ = rgb.shape
    pitch = (w * 3 + 3) & ~3
    buf = np.zeros((h, pitch), np.uint8)
    buf[:, :w * 3] = (rgb if top_down else rgb[::-1])[:, :, ::-1].reshape(h, w * 3)
    return buf.reshape(-1), pitch


def write_bmp(path, rgb, top_down=False):
    h, w, _ = rgb.shape
    data, pitch = bmp_bytes(rgb, top_down)
    with open(path, 'wb') as f:
        f.write(b'BM' + struct.pack('<IHHI', 54 + data.size, 0, 0, 54))
        f.write(struct.pack('<IiiHHIIiiII', 40, w, -h if top_down else h, 1, 24, 0, data.size, 2835, 2835, 0, 0))
        f.write(data.tobytes())


def banded(h, w, seed, top, bottom):
    img = synth.texture_u8(h, w, seed)
    img[:top] = 0
    img[h - bottom:] = 0
    return img


def scan(seed, top, bottom):
    return synth.raw_image_u8(seed, 4096, top=top, bottom=bottom)[0]


def test_mixed_chunk_is_bit_identical_to_the_per_image_entries(cuda_device):
    """One nbc_preprocess_mixed_batch_u8 call over every kind of input == the per-image entries, image by image."""
    from neuralbarkcalculator_b200 import Preprocessor, ops
    cases = []      # (pixel array u8 1-D, H, W, pitch, bgr, bottom_up)
    a = scan(1, 800, 1100)
    cases.append(bmp_bytes(a) + (4096, 4096, True, True))                             # 4096^2 BGR bottom-up (BMP)
    b = scan(2, 600, 400)
    cases.append((b.reshape(-1), 3 * 4096, 4096, 4096, False, False))                 # 4096^2 RGB top-down
    cases.append((banded(3000, 2000, 3, 300, 200).reshape(-1), 3 * 2000, 3000, 2000, False, False))
    cases.append((banded(2048, 4096, 4, 100, 0).reshape(-1), 3 * 4096, 2048, 4096, False, False))
    cases.append((banded(1500, 1500, 5, 200, 150).reshape(-1), 3 * 1500, 1500, 1500, False, False))
    cases.append((banded(1024, 1024, 6, 90, 50).reshape(-1), 3 * 1024, 1024, 1024, False, False))    # trim only
    cases.append((synth.texture_u8(900, 700, 7).reshape(-1), 3 * 700, 900, 700, False, False))      # untouched
    cases.append((synth.texture_u8(4096, 4096, 8, coarse=64).reshape(-1), 3 * 4096, 4096, 4096, False, False))  # no bands
    cases.append((np.zeros(4096 * 4096 * 3, np.uint8), 3 * 4096, 4096, 4096, False, False))          # all zero
    c = banded(1300, 1001, 9, 100, 100)
    cases.append(bmp_bytes(c) + (1300, 1001, True, True))                             # padded pitch, general ratio
    d = banded(800, 1001, 10, 40, 0)
    cases.append(bmp_bytes(d, top_down=True) + (800, 1001, True, False))              # padded pitch, untouched
    bufs = [x[0] for x in cases]
    geoms = [(H, W, pitch, bgr, bu) for _, pitch, H, W, bgr, bu in cases]
    raws = [torch.from_numpy(np.ascontiguousarray(x)).to(cuda_device) for x in bufs]
    # the 4x scans hold only the rows between their zero bands, as the folder pipeline stages them
    spans = []
    for x, (H, W, pitch, _, _) in zip(bufs, geoms):
        spans.append(ops.host_zero_row_span(x, H, pitch, W * 3) if H == W == 4096 else (0, H))
    span_raws = [r[s0 * g[2]:(s0 + n) * g[2]] for r, (s0, n), g in zip(raws, spans, geoms)]
    assert spans[-3] == (0, 0) and spans[0][1] < 4096
    out, fl = ops.preprocess_mixed_batch(span_raws, geoms, 1024, spans)
    fl = fl.cpu().tolist()
    pre = Preprocessor(device='cuda:0')
    for i, ((x, pitch, H, W, bgr, bu), r) in enumerate(zip(cases, raws)):
        ref = pre.preprocess_array(x, H, W, pitch, bgr, bu)
        h, w = ref.shape[:2]
        got = out[i, :h * w * 3].view(h, w, 3)
        assert fl[i][1] - fl[i][0] == h, i
        assert torch.equal(got, ref), 'image %d (%dx%d) differs' % (i, H, W)
        if H == W == 4096:
            ref_out, ref_fl = ops.preprocess_4x(r[spans[i][0] * pitch:(spans[i][0] + spans[i][1]) * pitch], H, W, pitch, bgr, bu,
                                                span=spans[i])
            assert fl[i] == ref_fl.tolist()
        elif max(H, W) > 1024:
            assert fl[i] == ops.preprocess_general(r, H, W, 1024, pitch, bgr, bu)[1].tolist()
        elif H == W:
            assert fl[i] == ops.trim_u8(torch.from_numpy(x).to(cuda_device).view(H, W, 3))[1].tolist()
        else:
            assert fl[i] == [0, H]
    # a chunk of the engine's size with every kind twice, and alone: the same bytes whatever the neighbours
    order = [9, 0, 6, 2, 10, 5]
    out2, fl2 = ops.preprocess_mixed_batch([span_raws[i] for i in order], [geoms[i] for i in order], 1024, [spans[i] for i in order])
    for k, i in enumerate(order):
        n = (fl[i][1] - fl[i][0]) * ops.processed_size(*geoms[i][:2])[1] * 3
        assert fl2[k].tolist() == fl[i] and torch.equal(out2[k, :n], out[i, :n])


def make_mixed_folder(root, seed=0):
    """Every input kind over the three wood types; names sort the same before and after the .bmp -> .png rename."""
    rng = np.random.default_rng(seed)
    rgba = np.dstack([synth.texture_u8(900, 700, seed + 6), rng.integers(0, 256, (900, 700, 1), np.uint8)])
    files = [
        ('epinette_gelee', 'a00.bmp', lambda p: write_bmp(p, scan(seed + 1, 700, 900))),
        ('epinette_gelee', 'a01.png', lambda p: Image.fromarray(banded(1500, 1300, seed + 2, 120, 80)).save(p)),
        ('epinette_gelee', 'a02.png', lambda p: Image.fromarray(banded(1024, 1024, seed + 3, 60, 30)[:, :, 1]).save(p)),   # grey
        ('epinette_gelee', 'a03.bmp', lambda p: write_bmp(p, banded(1200, 1001, seed + 4, 50, 50))),          # padded rows
        ('epinette_non_gelee', 'b00.bmp', lambda p: write_bmp(p, scan(seed + 5, 500, 600), top_down=True)),
        ('epinette_non_gelee', 'b01.png', lambda p: Image.fromarray(rgba).save(p)),
        ('epinette_non_gelee', 'b02.png', lambda p: Image.fromarray(synth.texture_u8(640, 600, seed + 7)).quantize(64).save(p)),
        ('epinette_non_gelee', 'b03.jpg', lambda p: Image.fromarray(synth.texture_u8(500, 700, seed + 8)).save(p, quality=90)),
        ('sapin', 'c00.bmp', lambda p: write_bmp(p, synth.texture_u8(800, 700, seed + 9))),                   # second 700-wide
        ('sapin', 'c01.png', lambda p: Image.fromarray(scan(seed + 10, 900, 400)).save(p, compress_level=1)),
        ('sapin', 'c02.bmp', lambda p: write_bmp(p, banded(2048, 3000, seed + 11, 200, 100))),
    ]
    for wood, name, write in files:
        os.makedirs(os.path.join(root, 'samples', wood), exist_ok=True)
        write(os.path.join(root, 'samples', wood, name))
    return len(files)


def per_image_route(root, sd, exclude_nodes, only_preprocess=False):
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import predict as npredict
    npredict.generate_folders(root, only_preprocess)
    processed = nbc.Preprocessor(device='cuda:0').preprocess_images(root)
    if not only_preprocess:
        return nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=sd).predict(root, exclude_nodes, processed=processed)


def assert_same_outputs(root, root_b, only_preprocess=False):
    subs = [('processed', 'samples')] + ([] if only_preprocess else [('results', 'outputs'), ('results', 'combined_images')])
    for sub in subs:
        for wood in synth.WOOD_TYPES:
            d = os.path.join(root, *sub, wood)
            names = sorted(os.listdir(d))
            assert names == sorted(os.listdir(os.path.join(root_b, *sub, wood))) and len(names) > 0
            for fn in names:
                ia, ib = Image.open(os.path.join(d, fn)), Image.open(os.path.join(root_b, *sub, wood, fn))
                assert ia.format == ib.format, fn
                assert np.array_equal(np.asarray(ia), np.asarray(ib)), '/'.join(sub) + '/' + wood + '/' + fn
    if not only_preprocess:
        with open(os.path.join(root, 'results', 'final_stats.csv'), 'rb') as f, \
                open(os.path.join(root_b, 'results', 'final_stats.csv'), 'rb') as fb:
            assert f.read() == fb.read()
    else:
        assert not os.path.exists(os.path.join(root, 'results'))


@pytest.fixture(scope='module')
def mixed_src(tmp_path_factory):
    root = str(tmp_path_factory.mktemp('mixed') / 'src')
    make_mixed_folder(root)
    return root


def _copy(src, dst):
    shutil.copytree(os.path.join(src, 'samples'), os.path.join(dst, 'samples'))
    return dst


@pytest.mark.parametrize('exclude_nodes', [False, True])
def test_predict_on_mixed_inputs_matches_the_per_image_route(cuda_device, synthetic_sd, mixed_src, tmp_path, exclude_nodes):
    """predict.main on a folder of every input kind writes what Preprocessor + NeuralBarkCalculator.predict write:
    same names and formats, same decoded pixels, byte-identical final_stats.csv."""
    from neuralbarkcalculator_b200 import pipeline, predict as npredict
    from neuralbarkcalculator_b200.dataset import make_dataset
    root, root_b = _copy(mixed_src, str(tmp_path / 'pipe')), _copy(mixed_src, str(tmp_path / 'single'))
    assert not pipeline.supported(make_dataset(root))
    rows_b = per_image_route(root_b, synthetic_sd, exclude_nodes)
    rows = npredict.main(argparse.Namespace(root_path=root, device='cuda:0', exclude_nodes=exclude_nodes, only_preprocess=False),
                         state_dict=synthetic_sd)
    assert rows == rows_b
    assert_same_outputs(root, root_b)


def test_mixed_pipeline_small_batches_and_only_preprocess(cuda_device, synthetic_sd, mixed_src, tmp_path):
    """Batches of 3 (several width groups per batch, slot reuse, a ragged last batch) give the same files; so does
    --only_preprocess, which writes processed/ only."""
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import pipeline, predict as npredict
    root, root_b = _copy(mixed_src, str(tmp_path / 'pipe')), _copy(mixed_src, str(tmp_path / 'single'))
    rows_b = per_image_route(root_b, synthetic_sd, True)
    npredict.generate_folders(root, False)
    calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=synthetic_sd)
    pipe = pipeline.FolderPipeline(calc, batch=3, io_threads=4)
    assert pipe.run(root, True) == rows_b
    assert_same_outputs(root, root_b)
    assert pipe.last_timing['images'] == len(rows_b) - 1 and pipe.last_timing['read_s'] > 0
    root_c, root_d = _copy(mixed_src, str(tmp_path / 'pre')), _copy(mixed_src, str(tmp_path / 'pre_single'))
    npredict.main(argparse.Namespace(root_path=root_c, device='cuda:0', exclude_nodes=False, only_preprocess=True))
    per_image_route(root_d, synthetic_sd, False, only_preprocess=True)
    assert_same_outputs(root_c, root_d, only_preprocess=True)


def test_mixed_shards_merge_to_the_full_run(cuda_device, synthetic_sd, mixed_src, tmp_path):
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import distributed as ndist, pipeline, predict as npredict
    root = _copy(mixed_src, str(tmp_path / 'full'))
    npredict.generate_folders(root, False)
    calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=synthetic_sd)
    pipe = pipeline.FolderPipeline(calc, batch=4, io_threads=4)
    full = pipe.run(root, False)
    n, k = len(full) - 1, 5
    part = ndist.merge_rows(pipe.run(root, False, shard=(0, k)), 0, n) + ndist.merge_rows(pipe.run(root, False, shard=(k, n)), k, n)
    assert [pipeline.CSV_HEADER] + part == full


def test_mixed_predict_on_two_gpus_matches_one(cuda_device, synthetic_sd, mixed_src, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    root1, root2 = _copy(mixed_src, str(tmp_path / 'one')), _copy(mixed_src, str(tmp_path / 'two'))
    sd_path = str(tmp_path / 'best_model.pt')
    torch.save(synthetic_sd, sd_path)
    env = dict(os.environ, PYTHONPATH=ROOT)
    for root, cmd in ((root1, [sys.executable, '-m', 'neuralbarkcalculator_b200.predict', root1]),
                      (root2, [sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', '2', '-m',
                               'neuralbarkcalculator_b200.predict', root2])):
        done = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
        assert done.returncode == 0, done.stderr[-3000:]
    with open(os.path.join(root1, 'results', 'final_stats.csv'), 'rb') as f1, open(os.path.join(root2, 'results', 'final_stats.csv'), 'rb') as f2:
        assert f1.read() == f2.read()


def test_standard_folder_keeps_the_uniform_route(cuda_device, synthetic_sd, tmp_path, monkeypatch):
    """A folder of 4096x4096 BMP scans goes through submit_host and the 4x batch kernel, never through the mixed path."""
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import engine, pipeline, predict as npredict
    root = str(tmp_path / 'std')
    synth.make_raw_folder(root, 3, size=4096, pool=2, seed0=5)
    npredict.generate_folders(root, False)
    calls = {'submit_host': 0, 'chunk': 0}
    real_submit, real_chunk = engine.PredictEngine.submit_host, engine.PredictEngine._preprocess_chunk

    def submit_host(self, *a, **k):
        calls['submit_host'] += 1
        return real_submit(self, *a, **k)

    def chunk(self, *a, **k):
        calls['chunk'] += 1
        return real_chunk(self, *a, **k)

    def refuse(*a, **k):
        raise AssertionError('the mixed path was taken for a standard folder')

    monkeypatch.setattr(engine.PredictEngine, 'submit_host', submit_host)
    monkeypatch.setattr(engine.PredictEngine, '_preprocess_chunk', chunk)
    monkeypatch.setattr(engine.PredictEngine, 'submit_mixed', refuse)
    monkeypatch.setattr(pipeline, 'read_raw', refuse)
    calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=synthetic_sd)
    rows = pipeline.FolderPipeline(calc, batch=2, io_threads=2).run(root, False)
    assert len(rows) == 4 and calls['submit_host'] == 2 and calls['chunk'] >= 2
