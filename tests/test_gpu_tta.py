"""Flip test-time augmentation on the B200 (``pytest -m gpu``): the ragged flip copy against torch.flip, the multi-view K3
against the f32 restatement bit for bit, the whole predict path against the f32 CPU oracle under the north-star bar, the
engine / folder pipeline against the per-image path, the batched evaluation against the per-image ops, and two GPUs
against one."""
import argparse
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import model as omodel
from oracle import postprocess as opost
from oracle import synth
from tta_reference import flip_dims, mean_of_views, tta_logits, view_lowres

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORTH_STAR = {'max_abs': 2e-2, 'agree': 0.999, 'pp': 0.1}      # tests/test_gpu_model.py


def _low(n):
    return ((((n - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1


@pytest.mark.parametrize('W', [1024, 1000])
def test_flip_ragged_equals_torch_flip(cuda_device, W):
    from neuralbarkcalculator_b200 import ops
    heights = [1, 7, 611, 1024, 300]
    Hc = 1024
    g = torch.Generator().manual_seed(W)
    canvas = torch.randint(0, 256, (len(heights), Hc, W, 3), generator=g, dtype=torch.uint8).to(cuda_device)  # garbage below
    hs = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
    for flags in (0, 1, 2, 3):
        out = ops.flip_ragged(canvas, hs, flags)
        for n, h in enumerate(heights):
            dims = flip_dims(flags, 0, 1)
            ref = torch.flip(canvas[n, :h], dims) if dims else canvas[n, :h]
            assert torch.equal(out[n, :h], ref), (W, flags, h)
            assert not out[n, h:].any(), (W, flags, h)
    for bad in (-1, 4):
        with pytest.raises(RuntimeError, match='flags'):
            ops.flip_ragged(canvas, hs, bad)


# (W, heights): ragged canvases with the smallest heights, a trimmed one and a full one; a dense canvas (every image Hc rows)
K3_CASES = [(1024, [1, 2, 3, 9, 611, 1024]), (1000, [611, 9, 2]), (384, [200, 200, 200])]


def _random_views(V, N, Hc, W, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn((N, 3, _low(Hc), _low(W)), generator=g) * 3 for _ in range(V)]


@pytest.mark.parametrize('W,heights', K3_CASES)
@pytest.mark.parametrize('mode', ['h', 'hv'])
def test_multi_view_k3_equals_the_restatement(cuda_device, W, heights, mode):
    """upsample_bicubic_views_ragged and upsample_argmax_views_ragged equal the restated f32 formula bit for bit, per image
    of the canvas.  The per-pixel path of K3 (a group of 8 rows reading more than 6 source rows) cannot be reached here:
    with the network's ceil(H/8)-row logits no height up to 1024 gets there, flipped or not
    (tests/test_tta_host.py::test_k3_row_groups_never_need_the_per_pixel_path).  The last image carries planted exact ties
    of classes 0 and 1 in every view, which must resolve to class 0."""
    from neuralbarkcalculator_b200 import ops
    flags = ops.tta_views(mode)[1]
    N, Hc = len(heights), max(heights)
    lows = _random_views(len(flags), N, Hc, W, 7 * W + len(flags))
    for low in lows:
        low[N - 1, 1] = low[N - 1, 0]
        low[N - 1, 2] = low[N - 1, 0] - 5.0
    hs = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
    dev_lows = [t.to(cuda_device) for t in lows]
    mean = ops.upsample_bicubic_views_ragged(dev_lows, flags, hs, (Hc, W)).cpu().numpy()
    mask = ops.upsample_argmax_views_ragged(dev_lows, flags, hs, (Hc, W)).cpu().numpy()
    for n, h in enumerate(heights):
        ref = mean_of_views([t[n:n + 1, :, :_low(h)].numpy() for t in lows], flags, (h, W))
        assert np.array_equal(mean[n:n + 1, :, :h], ref), (W, h, mode)
        assert np.array_equal(mask[n, :h], omodel.argmax_lowest(ref)[0]), (W, h, mode)
    tie = mean[N - 1, :, :heights[-1]]
    assert np.array_equal(tie[0], tie[1]) and (mask[N - 1, :heights[-1]] == 0).all()


def test_multi_view_k3_controls(cuda_device):
    """Two copies of one canvas without flips give plain K3's mask bit for bit ((L + L) / 2 = L); swapping the flip flags
    of two views changes the result."""
    from neuralbarkcalculator_b200 import ops
    W, heights = 1024, [611, 1024, 9]
    N, Hc = len(heights), max(heights)
    a, b = [t.to(cuda_device) for t in _random_views(2, N, Hc, W, 99)]
    hs = torch.tensor(heights, dtype=torch.int32, device=cuda_device)
    plain = ops.upsample_argmax_ragged(a, hs, (Hc, W))
    twice = ops.upsample_argmax_views_ragged([a, a], [0, 0], hs, (Hc, W))
    for n, h in enumerate(heights):
        assert torch.equal(twice[n, :h], plain[n, :h])
    m01 = ops.upsample_bicubic_views_ragged([a, b], [0, 1], hs, (Hc, W))
    m10 = ops.upsample_bicubic_views_ragged([a, b], [1, 0], hs, (Hc, W))
    assert not torch.equal(m01[0, :, :heights[0]], m10[0, :, :heights[0]])
    assert not torch.equal(ops.upsample_argmax_views_ragged([a, b], [0, 1], hs, (Hc, W))[1],
                           ops.upsample_argmax_views_ragged([a, b], [1, 0], hs, (Hc, W))[1])
    for views, fl in (([a, b, a], [0, 1, 2]), ([a, b], [0, 4])):
        with pytest.raises(RuntimeError):
            ops.upsample_argmax_views_ragged(views, fl, hs, (Hc, W))


def _gpu_views(calc, img_u8, flags):
    """(mean logits f32 [1,3,H,W], mask u8 [1,H,W]) of the GPU path for one image: flip, network, multi-view K3."""
    from neuralbarkcalculator_b200 import ops
    H, W = img_u8.shape[:2]
    canvas = img_u8.unsqueeze(0).contiguous()
    hs = torch.tensor([H], dtype=torch.int32, device=img_u8.device)
    plan = calc.model.native_plan()
    lows = [plan.forward_ragged(canvas if f == 0 else ops.flip_ragged(canvas, hs, f), heights=hs) for f in flags]
    return (ops.upsample_bicubic_views_ragged(lows, flags, hs, (H, W)).cpu().numpy(),
            ops.upsample_argmax_views_ragged(lows, flags, hs, (H, W)))


def test_tta_north_star_against_the_f32_oracle(cuda_device, trained_like_sd):
    """--tta hv end to end against the f32 CPU oracle (the network's f32 forward per view, restated upsample, un-flip, mean)
    at the default precision: mean logits max-abs <= 2e-2, argmax agreement >= 99.9 %, bark / node percentages after
    region removal within 0.1 pp, and every disagreement a near-tie of the f32 mean logits.  The single-view figures of
    the same images are printed beside them."""
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import ops
    calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=trained_like_sd, tta='hv')
    flags = ops.tta_views('hv')[1]
    net = omodel.load_model(trained_like_sd)
    for seed, (H, W) in ((31, (1024, 1024)), (32, (611, 1024))):
        img = synth.texture_u8(H, W, seed)
        x = omodel.normalise_u8(img)
        ref_lows = view_lowres(net, x, flags)
        t = torch.from_numpy(img).to(cuda_device)
        for name, fl in (('single view', [0]), ('hv', flags)):
            ref = mean_of_views(ref_lows[:len(fl)], fl, (H, W))
            ref_mask = omodel.argmax_lowest(ref)[0]
            mean, mask = _gpu_views(calc, t, fl)
            err = np.abs(mean - ref)
            mask = mask.cpu().numpy()[0]
            agree = (mask == ref_mask).mean()
            top2 = np.sort(ref[0], axis=0)[::-1][:2]
            margin = top2[0] - top2[1]
            near = float(margin[mask != ref_mask].max()) if (mask != ref_mask).any() else 0.0
            _, counts = ops.remove_small_zones_u8(torch.from_numpy(mask).unsqueeze(0).to(cuda_device))
            ref_clean = opost.remove_small_zones_2d(ref_mask)
            pps = [100.0 * abs(int(counts[0, c]) - int((ref_clean == c).sum())) / ref_mask.size for c in (1, 2)]
            print('\n[tta %s %dx%d] mean logits max-abs %.4g mean-abs %.4g; argmax agreement %.5f; largest f32 margin of a '
                  'disagreement %.4g; bark / node off by %.4f / %.4f pp' % (name, H, W, err.max(), err.mean(), agree, near,
                                                                            pps[0], pps[1]))
            assert err.max() <= NORTH_STAR['max_abs']
            assert agree >= NORTH_STAR['agree']
            assert max(pps) <= NORTH_STAR['pp']
            assert near < 4 * err.max()
        # the calculator's own path: the same mask, then the unchanged region removal
        m, c = calc.predict_array(t, excludes_nodes=False)
        ref_m, ref_c = ops.remove_small_zones_u8(_gpu_views(calc, t, flags)[1], 150)
        assert torch.equal(m, ref_m[0]) and torch.equal(c, ref_c[0])
        np.testing.assert_array_equal(tta_logits(net, x, flags), mean_of_views(ref_lows, flags, (H, W)))


def _same_files(root, root_b, exact):
    """The output files of two runs: byte for byte (exact), or the same format and pixels -- the per-image path saves
    processed/ through PIL and the pipeline through the library's PNG encoder -- and the same CSV bytes."""
    for sub in (('processed', 'samples'), ('results', 'outputs'), ('results', 'combined_images')):
        for wood in synth.WOOD_TYPES:
            d = os.path.join(root, *sub, wood)
            names = sorted(os.listdir(d))
            assert names == sorted(os.listdir(os.path.join(root_b, *sub, wood))) and len(names) > 0
            for fn in names:
                a, b = os.path.join(d, fn), os.path.join(root_b, *sub, wood, fn)
                what = '/'.join(sub) + '/' + wood + '/' + fn
                if exact:
                    with open(a, 'rb') as f, open(b, 'rb') as fb:
                        assert f.read() == fb.read(), what
                else:
                    ia, ib = Image.open(a), Image.open(b)
                    assert ia.format == ib.format and np.array_equal(np.asarray(ia), np.asarray(ib)), what
    with open(os.path.join(root, 'results', 'final_stats.csv'), 'rb') as f, \
            open(os.path.join(root_b, 'results', 'final_stats.csv'), 'rb') as fb:
        assert f.read() == fb.read()


def _per_image_route(root, sd, tta):
    import neuralbarkcalculator_b200 as nbc
    from neuralbarkcalculator_b200 import predict as npredict
    npredict.generate_folders(root, False)
    processed = nbc.Preprocessor(device='cuda:0').preprocess_images(root)
    return nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=sd, tta=tta).predict(root, True, processed=processed)


def _dual_images(root):
    d = os.path.join(root, 'results', 'outputs')
    return {(w, f): np.asarray(Image.open(os.path.join(d, w, f)))
            for w in sorted(os.listdir(d)) for f in sorted(os.listdir(os.path.join(d, w)))}


def test_folder_pipeline_with_tta_matches_the_per_image_path(cuda_device, synthetic_sd, tmp_path):
    """predict --tta hv through the streaming FolderPipeline (engine chunks, two batches in flight) writes the per-image
    path's files -- same pixels, same CSV bytes -- on the uniform route (standard 4096^2 BMP scans) and on the mixed route
    (other formats and sizes, narrower canvases); --tta none writes byte for byte what a run without the argument writes."""
    from neuralbarkcalculator_b200 import pipeline, predict as npredict
    from neuralbarkcalculator_b200.dataset import make_dataset
    from test_gpu_mixed_predict import make_mixed_folder
    src_std, src_mixed = str(tmp_path / 'std'), str(tmp_path / 'mixed')
    synth.make_raw_folder(src_std, 5, size=4096, pool=3, seed0=70)
    make_mixed_folder(src_mixed)
    assert pipeline.supported(make_dataset(src_std)) and not pipeline.supported(make_dataset(src_mixed))
    for name, src in (('std', src_std), ('mixed', src_mixed)):
        roots = {k: str(tmp_path / (name + '_' + k)) for k in ('pipe', 'single', 'none', 'plain')}
        for r in roots.values():
            shutil.copytree(os.path.join(src, 'samples'), os.path.join(r, 'samples'))
        _per_image_route(roots['single'], synthetic_sd, 'hv')
        import neuralbarkcalculator_b200 as nbc
        npredict.generate_folders(roots['pipe'], False)
        calc = nbc.NeuralBarkCalculator(None, 'cuda:0', state_dict=synthetic_sd, tta='hv')
        pipeline.FolderPipeline(calc, batch=2, io_threads=4).run(roots['pipe'], True)
        _same_files(roots['pipe'], roots['single'], exact=False)
        ns = dict(root_path=None, device='cuda:0', exclude_nodes=True, only_preprocess=False)
        npredict.main(argparse.Namespace(**dict(ns, root_path=roots['none'], tta='none')), state_dict=synthetic_sd)
        npredict.main(argparse.Namespace(**dict(ns, root_path=roots['plain'])), state_dict=synthetic_sd)
        _same_files(roots['none'], roots['plain'], exact=True)
        tta, plain = _dual_images(roots['pipe']), _dual_images(roots['plain'])
        assert tta.keys() == plain.keys() and any(not np.array_equal(tta[k], plain[k]) for k in tta), name


def test_evaluate_plan_with_tta_equals_the_per_image_ops(cuda_device, synthetic_sd):
    """evaluate_plan(tta='hv') rows equal, bit for bit, the per-image ops applied to upsample_bicubic_views_ragged's mean
    logits of each image run alone; tta='none' rows equal a call without the argument."""
    from neuralbarkcalculator_b200 import evaluate as nev, ops
    from neuralbarkcalculator_b200.utils import get_pos_weight
    from test_gpu_evaluate import _net_dataset
    from test_gpu_evaluate import _same_rows
    ds = _net_dataset(cuda_device)
    idx = [4, 0, 9, 1, 3, 7, 2, 5, 10, 6, 8]
    plan = nev.make_plan(synthetic_sd, cuda_device)
    flags = ops.tta_views('hv')[1]
    wts = get_pos_weight().to(cuda_device)
    ref = {}
    for i in idx:
        h, w = int(ds.sizes[i, 0]), int(ds.sizes[i, 1])
        Hc = max(h, 16)
        canvas = torch.zeros((1, Hc, w, 3), dtype=torch.uint8, device=cuda_device)
        canvas[0, :h] = ds.images[i, :h, :w]
        hs = torch.tensor([h], dtype=torch.int32, device=cuda_device)
        lows = [plan.forward_ragged(canvas if f == 0 else ops.flip_ragged(canvas, hs, f), heights=hs) for f in flags]
        full = ops.upsample_bicubic_views_ragged(lows, flags, hs, (Hc, w))[:, :, :h].contiguous()
        lab = ds.classes[i:i + 1, :h, :w].contiguous()
        ce = ops.wce_fwd_bwd(full, lab, wts, need_grad=False)[0].cpu().numpy()
        lov = ops.lovasz_softmax_fwd_bwd(full, lab, need_grad=False)[0].cpu().numpy()
        pred = ops.argmax3_u8(full)
        cm_raw = ops.confusion_matrix(pred, lab).cpu().numpy()
        pred, counts = ops.remove_small_zones_u8(pred, 150)
        ref[i] = (ce, lov, cm_raw, ops.confusion_matrix(pred, lab).cpu().numpy(), counts[0].cpu().numpy())
    for loss in nev.LOSSES:
        res = nev.evaluate_plan(plan, ds, idx, loss, chunk=3, tta='hv')
        assert sorted(r['index'] for r in res['rows']) == sorted(idx)
        for r in res['rows']:
            ce, lov, cm_raw, cm_rsz, counts = ref[r['index']]
            exp = nev.image_row(r['index'], loss, ce, lov, cm_raw, cm_rsz, counts)
            assert r['loss'] == exp['loss'] and r['miou'] == exp['miou'], (loss, r['index'])
            for k in ('f1', 'iou', 'cm_rsz', 'counts'):
                assert np.array_equal(r[k], exp[k]), (loss, k, r['index'])
        _same_rows([nev.evaluate_plan(plan, ds, idx, loss, chunk=3), nev.evaluate_plan(plan, ds, idx, loss, chunk=3, tta='none')])
    hv = nev.evaluate_plan(plan, ds, idx, 'mixed', chunk=3, tta='hv')
    assert hv['loss'] != nev.evaluate_plan(plan, ds, idx, 'mixed', chunk=3)['loss']


def test_predict_tta_on_two_gpus_matches_one(cuda_device, synthetic_sd, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    base = str(tmp_path)
    torch.save(synthetic_sd, os.path.join(base, 'best_model.pt'))
    one, two = os.path.join(base, 'one'), os.path.join(base, 'two')
    synth.make_raw_folder(one, 5, size=4096, pool=2, seed0=90)
    shutil.copytree(os.path.join(one, 'samples'), os.path.join(two, 'samples'))
    env = dict(os.environ, PYTHONPATH=ROOT)
    for args in ([sys.executable, '-m', 'neuralbarkcalculator_b200.predict', one, '--tta', 'hv'],
                 [sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', '2', '-m',
                  'neuralbarkcalculator_b200.predict', two, '--tta', 'hv']):
        done = subprocess.run(args, cwd=base, env=env, capture_output=True, text=True, timeout=900)
        assert done.returncode == 0, done.stderr[-3000:]
    with open(os.path.join(one, 'results', 'final_stats.csv'), 'rb') as f1, \
            open(os.path.join(two, 'results', 'final_stats.csv'), 'rb') as f2:
        assert f1.read() == f2.read()
