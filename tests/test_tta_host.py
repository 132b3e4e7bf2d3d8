"""CPU tests of flip test-time augmentation: the ``--tta`` arguments of predict and evaluate, the view sets, the f32
restatement of the averaged logits against a direct torch computation, and the row bound of K3's shared x pass under
row flips."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model as omodel
from tta_reference import mean_of_views, tta_logits, view_lowres


def test_predict_tta_argument():
    from neuralbarkcalculator_b200 import predict as npredict
    assert npredict.parse_args(['r']).tta == 'none'
    for mode in ('none', 'h', 'hv'):
        assert npredict.parse_args(['r', '--tta', mode]).tta == mode
    assert npredict.parse_args(['r', '--only_preprocess']).tta == 'none'
    assert npredict.parse_args(['r', '--only_preprocess', '--tta', 'none']).only_preprocess


@pytest.mark.parametrize('argv', [['r', '--tta', 'v'], ['r', '--tta', 'rot90'], ['r', '--tta', 'h', '--only_preprocess'],
                                  ['r', '--only_preprocess', '--tta', 'hv']])
def test_predict_tta_refusals(argv, capsys):
    from neuralbarkcalculator_b200 import predict as npredict
    with pytest.raises(SystemExit):
        npredict.parse_args(argv)
    err = capsys.readouterr().err
    assert ('runs no network' in err) if '--only_preprocess' in argv else ('invalid choice' in err)


def test_evaluate_tta_argument(capsys):
    from neuralbarkcalculator_b200 import evaluate as nev
    assert nev.parse_args(['r']).tta == 'none'
    for mode in ('none', 'h', 'hv'):
        assert nev.parse_args(['r', '--tta', mode]).tta == mode
    with pytest.raises(SystemExit):
        nev.parse_args(['r', '--tta', 'vh'])
    assert 'invalid choice' in capsys.readouterr().err


def test_tta_views_order():
    from neuralbarkcalculator_b200 import ops
    assert ops.TTA_MODES == ('none', 'h', 'hv')
    assert ops.tta_views('none') == (['id'], [0])
    assert ops.tta_views('h') == (['id', 'h'], [0, 1])
    assert ops.tta_views('hv') == (['id', 'h', 'v', 'hv'], [0, 1, 2, 3])
    names, flags = ops.tta_views('hv')
    flags.append(9)                                          # callers get copies
    assert ops.tta_views('hv')[1] == [0, 1, 2, 3]
    for bad in ('v', 'HV', None):
        with pytest.raises(ValueError):
            ops.tta_views(bad)


def test_tta_logits_match_a_direct_torch_computation(synthetic_sd):
    """The restated mean logits equal torch.flip + F.interpolate(bicubic, align_corners=False) + torch.flip, summed in view
    order, within f32 rounding (F.interpolate's own arithmetic differs from the restatement by round-off only)."""
    net = omodel.load_model(synthetic_sd)
    H, W = 45, 77                                            # not multiples of 8: the stride-8 grids of the views differ
    x = omodel.normalise_u8(np.random.default_rng(3).integers(0, 256, (H, W, 3), dtype=np.uint8))
    for views in ([0], [0, 1], [0, 1, 2, 3]):
        got = tta_logits(net, x, views)
        total = None
        for f in views:
            dims = ([3] if f & 1 else []) + ([2] if f & 2 else [])
            with torch.no_grad():
                low = net.features(torch.flip(x, dims) if dims else x)
            up = F.interpolate(low, size=(H, W), mode='bicubic', align_corners=False)
            up = torch.flip(up, dims) if dims else up
            total = up if total is None else total + up
        ref = (total / len(views)).numpy()
        assert got.shape == (1, 3, H, W) and got.dtype == np.float32
        np.testing.assert_allclose(got, ref, rtol=0, atol=2e-5 * max(1.0, float(np.abs(ref).max())))
    # one view is the restated upsample itself, unscaled; the mirrored views change the result
    low0 = view_lowres(net, x, [0])
    assert np.array_equal(tta_logits(net, x, [0]), omodel.upsample_bicubic_restated(low0[0], (H, W)))
    assert not np.array_equal(tta_logits(net, x, [0, 1]), tta_logits(net, x, [0]))
    # two identical unflipped views: (L + L) * 0.5 == L exactly
    assert np.array_equal(mean_of_views([low0[0]] * 2, [0, 0], (H, W)), tta_logits(net, x, [0]))


def test_k3_row_groups_never_need_the_per_pixel_path():
    """K3 shares the x pass of 8 consecutive output rows when they read at most 6 source rows.  With the network's
    ceil(H/8)-row logits (every ragged call) any 8 consecutive rows -- the aligned groups of the identity view and the
    mirrored, unaligned ranges of a row flip -- read at most 6, for every height up to 1024: the per-pixel path is
    reachable only through the dense entry with a caller-chosen logits height."""
    worst = 0
    for H in range(1, 1025):
        h = ((((H - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        iy, _ = omodel.bicubic_weights_f32(h, H)
        for rows in range(1, min(8, H) + 1):
            span = iy[rows - 1:, 3] - iy[:H - rows + 1, 0] + 1
            worst = max(worst, int(span.max()))
    assert worst <= 6, worst
