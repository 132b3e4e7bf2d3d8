"""Host-side pieces of the training entry point (no GPU): the pad_resize coefficient table against Pillow, the plateau
rule against torch, and fit's argument checks."""
from math import ceil

import numpy as np
import pytest
from PIL import Image

from neuralbarkcalculator_b200 import augment


def _pad_resize_restated(img, th, tw):
    """numpy restatement of utils.py:242-247 with the table of augment.py: reflect pad by ceil(d/2) per side, then for an
    odd d Pillow's fixed-point bilinear pass over that axis (horizontal first), the intermediate rounded to u8."""
    h, w = img.shape[:2]
    dh, dw = th - h, tw - w
    pads = [(ceil(dh / 2),) * 2, (ceil(dw / 2),) * 2] + ([(0, 0)] if img.ndim == 3 else [])
    a = np.pad(img, pads, mode='reflect').astype(np.int64)

    def resample(a, table, axis):
        a = np.moveaxis(a, axis, 0)
        acc = np.full((table.shape[0],) + a.shape[1:], 1 << 21, dtype=np.int64)
        for k in range(3):
            wk = table[:, 1 + k].astype(np.int64).reshape((-1,) + (1,) * (a.ndim - 1))
            acc += wk * a[np.minimum(table[:, 0] + k, a.shape[0] - 1)]
        return np.moveaxis(np.clip(acc >> 22, 0, 255), 0, axis)

    if dw % 2:
        a = resample(a, augment.pil_bilinear_table(tw + 1, tw), 1)
    if dh % 2:
        a = resample(a, augment.pil_bilinear_table(th + 1, th), 0)
    return a.astype(np.uint8)


def test_pad_resize_table_matches_pillow():
    """Every source height 343..1024 at target 1024 (even and odd differences), RGB and L, even and odd widths."""
    from oracle import augment as oaug
    rng = np.random.default_rng(0)
    tw = 32
    for h in range(343, 1025):
        w_rgb, w_l = (29, 31, 32)[h % 3], (32, 29, 31)[h % 3]
        rgb = rng.integers(0, 256, (h, w_rgb, 3), dtype=np.uint8)
        grey = rng.integers(0, 256, (h, w_l), dtype=np.uint8)
        assert np.array_equal(_pad_resize_restated(rgb, 1024, tw),
                              np.asarray(oaug.pad_resize(Image.fromarray(rgb), tw, 1024))), (h, w_rgb)
        assert np.array_equal(_pad_resize_restated(grey, 1024, tw),
                              np.asarray(oaug.pad_resize(Image.fromarray(grey, mode='L'), tw, 1024))), (h, w_l)
    # the sizes of the GPU tests: 1024-class targets with a 1021-wide source, and the small target
    for (h, w, t) in ((611, 1021, 1024), (1023, 1021, 1024), (129, 255, 256), (201, 256, 256)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(_pad_resize_restated(img, t, t), np.asarray(oaug.pad_resize(Image.fromarray(img), t, t))), (h, w)


def test_pil_bilinear_table_shape():
    t = augment.pil_bilinear_table(1025, 1024)
    assert t.shape == (1024, 4) and t[0, 0] == 0
    last = t[:, 0] + np.where(t[:, 3] != 0, 2, 1)               # the last padded index a non-zero tap reads
    assert last.max() <= 1024 and np.all(np.diff(t[:, 0]) >= 0)
    assert np.all(np.abs(t[:, 1:].sum(1) - (1 << 22)) <= 2)       # normalised weights, each rounded once
    assert augment.resize_tables((256, 512)).shape == (768, 4)


def test_plateau_rule_matches_torch():
    import torch
    from neuralbarkcalculator_b200.fit import EarlyStopping, Plateau
    losses = [1.0, 0.9, 0.9, 0.95, 0.89995, 0.9, 0.9, 0.8, 0.8, 0.8, 0.8, 0.81, 0.8, 0.79999, 0.8, 0.8, 0.7, 0.7, 0.7,
              0.7, 0.7, 0.7, 0.7, 0.7, 0.7, 0.69, 0.7, 0.7]
    for kw in ({}, {'factor': 0.5, 'patience': 2}, {'factor': 0.1, 'patience': 0, 'cooldown': 1, 'min_lr': 1e-6},
               {'factor': 0.3, 'patience': 1, 'threshold': 0.2}):
        p = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.Adam([p], lr=5e-4)
        ref = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode='min', **kw)
        ours = Plateau(5e-4, **kw)
        for v in losses:
            ref.step(v)
            assert ours.step(v) == opt.param_groups[0]['lr'], kw
    stop = EarlyStopping(patience=3)
    assert [stop.step(v) for v in (1.0, 0.9, 0.9, 0.95, 0.91, 0.8, 0.8)] == [False, False, False, False, True, False, False]


def test_fit_rejects_bad_arguments(capsys):
    from neuralbarkcalculator_b200 import fit
    with pytest.raises(SystemExit):
        fit.parse_args(['root', '--init', 'random', '--device', 'cpu'])
    assert 'only CUDA devices' in capsys.readouterr().err
    with pytest.raises(SystemExit):
        fit.parse_args(['root'])
    assert '--init' in capsys.readouterr().err
    args = fit.parse_args(['root', '--init', 'random'])
    assert (args.epochs, args.crop, args.batch, args.loss, args.lr, args.weight_decay, args.dropout, args.out) == \
        (30, 512, 5, 'lovasz', 5e-4, 2e-3, 0.8, 'best_model.pt')
    with pytest.raises(RuntimeError, match='no such file'):
        fit.initial_state_dict('/nonexistent/sd.pt', 0.8)
