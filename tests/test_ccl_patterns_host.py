"""The K5 catalogue (tests/ccl_patterns.py) on the CPU: the scipy oracle agrees with the pure-Python flood fill on every
small entry, the entries hit the union events they were written for, and every wrong reference is told apart from the
oracle on the entry written for it."""
import numpy as np
import pytest
from scipy import ndimage as ndi

import ccl_patterns as P
from oracle import postprocess as opost


@pytest.fixture(scope='module')
def cases():
    return P.catalogue()


def test_catalogue_is_seeded_and_well_formed(cases):
    again = P.catalogue()
    assert [c.name for c in cases] == [c.name for c in again]
    assert len({c.name for c in cases}) == len(cases)
    assert all(np.array_equal(a.mask, b.mask) and a.threshold == b.threshold for a, b in zip(cases, again))
    for c in cases:
        assert c.mask.dtype == np.uint8 and c.mask.ndim == 2 and c.mask.max(initial=0) <= 2, c.name
    assert {c.family for c in cases} == set(P.FAMILIES)
    widths = {c.mask.shape[1] for c in cases}
    heights = {c.mask.shape[0] for c in cases}
    assert set(P.WIDTHS + P.PIXEL_WIDTHS) <= widths and {1, 2, 8, 9} <= heights
    thresholds = {(c.mask.shape, c.threshold) for c in cases if c.family == 'threshold'}
    for shape in ((37, 65), (8, 1024)):
        assert {(shape, t) for t in (0, 1, 2, 9, 150, shape[0] * shape[1], shape[0] * shape[1] + 1)} <= thresholds
    assert sum(c.family == 'contention' and c.mask.shape == (1024, 1024) for c in cases) == 16


def test_components_mix_classes(cases):
    """Classes 1 and 2 share components: the kernel must label the foreground, not a class."""
    for family in P.FAMILIES:
        mixed = 0
        for c in cases:
            if c.family != family or not (c.mask == 1).any():
                continue
            lab, _ = ndi.label(c.mask != 0, opost.STRUCT8)
            mixed += len(np.intersect1d(lab[c.mask == 1], lab[c.mask == 2]))
        assert mixed > 0, family


def test_entries_reach_the_lane_events(cases):
    """Computed with rows_merge's word expressions: E2 at bit 0 (target: the run holding bit 31 of the lane below), E3 at
    bit 31 (target: the next lane's bit 0), both on one pixel at bit 0 and at bit 31, and runs whose start lies m full
    words back for every m from 1 to 32."""
    hit = set()
    spans = set()
    for c in cases:
        if c.family != 'lanes':
            continue
        _, e2, e3 = P.lane_events(c.mask)
        x = np.arange(c.mask.shape[1])
        hit |= {('E2', b) for b in (0, 31) if (e2 & (x % 32 == b) & (x > 0)).any()}
        hit |= {('E3', b) for b in (0, 31) if (e3 & (x % 32 == b) & (x < c.mask.shape[1] - 1)).any()}
        hit |= {('E2&E3', b) for b in (0, 31) if (e2 & e3 & (x % 32 == b)).any()}
        for row in c.mask != 0:
            padded = np.concatenate([[False], row, [False]]).astype(np.int8)
            starts, ends = np.nonzero(np.diff(padded) == 1)[0], np.nonzero(np.diff(padded) == -1)[0]
            for s, e in zip(starts, ends):
                spans.add(len([w for w in range(s // 32, (e - 1) // 32 + 1) if s <= 32 * w and 32 * w + 32 <= e]))
    assert hit == {(e, b) for e in ('E2', 'E3', 'E2&E3') for b in (0, 31)}
    assert set(range(1, 33)) <= spans


def test_shapes_are_what_they_claim(cases):
    by = {c.name: c for c in cases}

    def ncomp(m):
        return ndi.label(m != 0, opost.STRUCT8)[1]

    assert ncomp(by['topology/spiral_1024'].mask) == 1 and ncomp(by['topology/spiral_1024'].mask == 0) == 1
    assert ncomp(by['topology/spiral_broken_1024'].mask) == 2
    for c in cases:
        if c.name.startswith('topology/checkerboard_cut'):
            assert ncomp(c.mask) == 2, c.name
        elif c.name.startswith('topology/checkerboard') or c.name.startswith('topology/comb'):
            assert ncomp(c.mask) == 1, c.name
        elif c.name.startswith('topology/stripes'):
            assert ncomp(c.mask) == (c.mask.shape[1] + 1) // 2, c.name
    # the exact-size shapes: every component of the L / diagonal entries has T - 1, T or T + 1 pixels
    for c in cases:
        if c.family == 'threshold' and (c.name.startswith('threshold/L_') or c.name.startswith('threshold/diag_')):
            binary = (c.mask != 0) if '_fg_' in c.name else (c.mask == 0)
            lab, n = ndi.label(binary, opost.STRUCT8)
            assert sorted(np.bincount(lab.ravel())[1:].tolist()) == [c.threshold - 1, c.threshold, c.threshold + 1], c.name


def test_oracle_equals_flood_fill_on_small_entries(cases):
    small = [c for c in cases if c.mask.shape[0] * c.mask.shape[1] <= 64 * 64 and max(c.mask.shape) <= 64]
    assert len(small) > 50
    for c in small:
        assert np.array_equal(opost.remove_small_zones_2d(c.mask, c.threshold),
                              opost.remove_small_zones_bruteforce(c.mask, c.threshold)), c.name


def test_right_reference_is_the_oracle(cases):
    """zones_with with the true labelling, comparison and stage order is the oracle: the wrong references below differ
    from it in the one thing each changes."""
    for c in cases[::7]:
        assert np.array_equal(P.zones_with(c.mask, c.threshold, P.label8), opost.remove_small_zones_2d(c.mask, c.threshold))


@pytest.mark.parametrize('control', sorted(P.CONTROLS))
def test_wrong_reference_is_rejected(cases, control):
    name, how = P.CONTROLS[control]
    case = next(c for c in cases if c.name == name)
    T = case.threshold
    if how == 'image':
        exp = opost.remove_small_zones_2d(case.mask, T)
        assert not np.array_equal(P.wrong_output(control, case, None), exp)
    elif how == 'dense':
        batch = P.dense_batch(P.groups(cases)[case.mask.shape + (T,)])
        exp = opost.remove_small_zones(batch, T)
        assert not np.array_equal(P.wrong_output(control, case, batch), exp)
    else:
        canvas, heights, _ = P.ragged_canvas(P.groups(cases)[case.mask.shape + (T,)], seed=1)
        exp, _ = P.ragged_expected(canvas, heights, T)
        assert not np.array_equal(P.wrong_output(control, case, (canvas, heights)), exp)


def test_guards_sit_just_below_the_threshold():
    for H, W, T in ((64, 64, 1428), (9, 1024, 5), (8, 33, 2), (2, 5, 150)):
        before, after = P.guards(H, W, T)
        assert (before[-1] != 0).all() and (after[0] != 0).all()
        assert np.count_nonzero(before) == np.count_nonzero(after) == min(H * W, max(T - 1, W))
