"""Seeded catalogue of adversarial masks for K5 (small-region removal, ``csrc/ccl.cu``) and the references it is held to.

Each entry is ``Case(name, family, mask u8 [H, W] in {0, 1, 2}, threshold)``.  Components mix classes 1 and 2 pixel by
pixel.  The families aim at the parts of the labelling that blobby masks rarely reach:

- ``lanes``: unions across the 32-pixel words of the run kernels.  Diagonal-only staircases through x = 32k - 1 / 32k; one
  pixel under a gap between two runs at bit 0 and bit 31, so that E2 and E3 fire on the same pixel (E2 at bit 0 targets
  the run holding bit 31 of the lane below, E3 at bit 31 the next lane's bit 0); runs that start at bit 0 or bit 31 and
  span 1 to 32 full words, joined to runs that end at W - 1 (the run start is found through a chain of full words).
- ``widths``: random masks at every width from 1 to 2048 that changes the last partial word or the byte path, heights
  1, 2, 8, 9 and 40.  Widths above 1024 always take the per-pixel kernels.
- ``topology``: checkerboards (one diagonal-only component, and one cut in two), width-1 stripes, combs joined only at
  the bottom or the top row, a 1024 x 1024 spiral with and without a break, the snake at full width.
- ``threshold``: components and holes of exactly T - 1, T and T + 1 pixels (L shapes, diagonals, holes on the border),
  and T in {0, 1, 2, 9, 150, H*W, H*W + 1}.
- ``stage``: a blob smaller than T in a hole smaller than T in large foreground, and the inverse: only a stage B that
  labels the result of stage A gets these right.
- ``wrap``: pixels at (y, W - 1) and (y + 1, 0), adjacent in the flat index but not in the image.
- ``contention``: 16 images of 1024 x 1024 filled at random at densities around the percolation threshold.

``dense_batch`` and ``ragged_canvas`` place entries the way the tests hand them to the kernel; ``WRONG`` holds
references that each get one thing wrong, with the entries that must tell them from the oracle (``CONTROLS``).
"""
from collections import namedtuple

import numpy as np
from scipy import ndimage as ndi
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from oracle import postprocess as opost

Case = namedtuple('Case', 'name family mask threshold')

WIDTHS = (1, 5, 31, 32, 33, 63, 64, 65, 200, 333, 513, 1000, 1023, 1024)   # run kernels (W <= 1024)
PIXEL_WIDTHS = (1025, 1100, 2048)                                        # always the per-pixel kernels
FAMILIES = ('lanes', 'widths', 'topology', 'threshold', 'stage', 'wrap', 'contention')
RAGGED_EXTRA = 9                   # canvas rows below the tallest entry
RAGGED_HEIGHTS = (1, 2, 7, 8, 9)   # plus each entry's own height H and the canvas height H + RAGGED_EXTRA


def _paint(binary, rng):
    """Foreground pixels get class 1 or 2 at random, so both classes share every component."""
    return np.where(binary, rng.integers(1, 3, binary.shape), 0).astype(np.uint8)


def _size(binary):
    return int(np.count_nonzero(binary))


# ------------------------------------------------------------------------------------------------------------ lanes
def _staircases(H, W, down):
    """Diagonals of H pixels, each crossing a word boundary halfway down; 32 columns apart, so they never touch."""
    b = np.zeros((H, W), bool)
    for k in range(1, W // 32 + 1):
        for y in range(H):
            x = 32 * k - H // 2 + y if down else 32 * k - 1 + H // 2 - y
            if 0 <= x < W:
                b[y, x] = True
    return b


def _gap_pixels(W, a, b_len):
    """One motif per 3 rows: runs [x - a, x - 1] and [x + 1, x + b_len] over a single pixel at x, x at bit 0 or bit 31.
    The pixel's up neighbour is clear and both diagonals are set: E2 and E3 on the same pixel.  Every motif has
    a + b_len + 1 pixels."""
    xs = [x for k in range(W // 32 + 1) for x in (32 * k, 32 * k + 31) if x - a >= 0 and x + b_len < W]
    m = np.zeros((3 * len(xs), W), bool)
    for j, x in enumerate(xs):
        m[3 * j, x - a:x] = True
        m[3 * j, x + 1:x + 1 + b_len] = True
        m[3 * j + 1, x] = True
    return m


def _long_run(W, m, bit):
    """Rows 7 and 8 (the two sides of an 8-row block): a run starting at bit ``bit`` of word 1 (or 0) that covers ``m``
    full words; below it a run from its last pixel + 1 to W - 1 (an E2 event at bit 0 whose target run starts m words
    back) and a run ending one pixel before its start (an E3 event)."""
    length = 32 * m + (1 if bit == 31 else 0)
    s = 32 + bit if 32 + bit + length <= W else bit
    if s + length > W:
        return None
    e = s + length - 1
    b = np.zeros((9, W), bool)
    b[7, s:e + 1] = True
    b[8, e + 1:] = True
    b[8, max(0, s - 6):s] = True
    return b


def _lanes(rng):
    out = []
    for W in (64, 65, 200, 1000, 1023, 1024):
        for down in (True, False):
            b = _staircases(20, W, down)
            out.append(('stair_%s_w%d' % ('down' if down else 'up', W), _paint(b, rng), 20))
    for W in (65, 200, 513, 1023, 1024):
        out.append(('gap_pixel_w%d' % W, _paint(_gap_pixels(W, 4, 4), rng), 9))
    for W in (200, 1000, 1024):
        out.append(('gap_pixel_long_w%d' % W, _paint(_gap_pixels(W, 70, 70), rng), 141))
    for W, spans in ((1024, range(1, 33)), (1023, (1, 2, 15, 30, 31)), (1000, (1, 2, 15, 30))):
        for m in spans:
            for bit in (0, 31):
                b = _long_run(W, m, bit)
                if b is not None:
                    out.append(('long_run_w%d_m%d_b%d' % (W, m, bit), _paint(b, rng), _size(b)))
    return out


# ----------------------------------------------------------------------------------------------------------- widths
def _widths(rng):
    out = []
    for W in WIDTHS + PIXEL_WIDTHS:
        for H in (1, 2, 8, 9, 40):
            out.append(('random_%dx%d' % (H, W), _paint(rng.random((H, W)) < 0.45, rng), 5))
    return out


# --------------------------------------------------------------------------------------------------------- topology
def spiral(n):
    """Square spiral of 1-pixel walls 1 pixel apart: one 8-connected component with the longest path a square holds."""
    b = np.zeros((n, n), bool)
    y, x, d = 0, 0, 0
    steps = [(0, 1), (1, 0), (0, -1), (-1, 0)]
    lengths = [n - 1, n - 1, n - 1]
    k = n - 3
    while k > 0:
        lengths += [k, k]
        k -= 2
    b[0, 0] = True
    for ln in lengths:
        dy, dx = steps[d % 4]
        for _ in range(ln):
            y, x = y + dy, x + dx
            b[y, x] = True
        d += 1
    return b


def _path_order(b):
    """Pixels of a one-pixel-wide path in order from (0, 0)."""
    order, seen, cur = [], {(0, 0)}, (0, 0)
    while cur is not None:
        order.append(cur)
        nxt = None
        for dy, dx in ((0, 1), (1, 0), (0, -1), (-1, 0)):
            p = (cur[0] + dy, cur[1] + dx)
            if 0 <= p[0] < b.shape[0] and 0 <= p[1] < b.shape[1] and b[p] and p not in seen:
                nxt = p
                break
        if nxt is not None:
            seen.add(nxt)
        cur = nxt
    return order


def _snake(H, W):
    """Full rows every 4 rows joined at alternating ends (the K5 edge case of test_gpu_kernels.py, at full width)."""
    b = np.zeros((H, W), bool)
    for r in range(0, H, 4):
        b[r, :] = True
        b[r:r + 4, W - 1 if (r // 4) % 2 == 0 else 0] = True
    return b


def _topology(rng):
    out = []
    for H, W in ((64, 64), (9, 1023), (200, 333), (1024, 1024), (8, 2048)):
        yy, xx = np.mgrid[:H, :W]
        board = (yy + xx) % 2 == 0
        out.append(('checkerboard_%dx%d' % (H, W), _paint(board, rng), _size(board)))
        c = 2 * ((H + W) // 4)                        # clearing the diagonal x + y = c (even) cuts the board in two
        cut = board & (yy + xx != c)
        lab, _ = ndi.label(cut, opost.STRUCT8)
        sizes = np.bincount(lab.ravel())[1:]
        out.append(('checkerboard_cut_%dx%d' % (H, W), _paint(cut, rng), int(sizes.min()) + 1))
    for H, W in ((64, 64), (9, 1024), (200, 333), (1024, 1024), (40, 1100)):
        stripes = np.zeros((H, W), bool)
        stripes[:, ::2] = True
        out.append(('stripes_keep_%dx%d' % (H, W), _paint(stripes, rng), H))
        out.append(('stripes_drop_%dx%d' % (H, W), _paint(stripes, rng), H + 1))
    for H, W in ((64, 64), (40, 1024), (200, 333), (1024, 1024), (33, 1100)):
        for where in ('bottom', 'top'):
            comb = np.zeros((H, W), bool)
            comb[:, ::3] = True
            comb[0 if where == 'bottom' else H - 1, :] = False
            comb[H - 1 if where == 'bottom' else 0, :] = True
            out.append(('comb_%s_%dx%d' % (where, H, W), _paint(comb, rng), _size(comb)))
    s = spiral(1024)
    bg = _size(~s)
    out.append(('spiral_1024', _paint(s, rng), min(_size(s), bg)))
    order = _path_order(s)
    broken = s.copy()
    broken[order[len(order) // 2]] = False           # both halves fall below T: only a false union keeps them
    out.append(('spiral_broken_1024', _paint(broken, rng), min(_size(s), bg)))
    snake = _snake(1024, 1024)
    out.append(('snake_1024', _paint(snake, rng), _size(snake)))
    snake[64, 50:60] = False
    out.append(('snake_cut_1024', _paint(snake, rng), 150))
    return out


# -------------------------------------------------------------------------------------------------------- threshold
def _L(b, y0, x0, size, v):
    """L shape of ``size`` pixels: a vertical arm of v rows, then a horizontal arm along its last row."""
    b[y0:y0 + v, x0] = True
    b[y0 + v - 1, x0:x0 + size - v + 1] = True


def _diag(b, y0, x0, size):
    for k in range(size):
        b[y0 + k, x0 + k] = True


def _threshold(rng):
    out = []
    for T, v, W in ((40, 10, 240), (150, 40, 1024)):
        Ls = np.zeros((v + 8, W), bool)
        diags = np.zeros((T + 8, W), bool)
        for j, size in enumerate((T - 1, T, T + 1)):
            _L(Ls, 3, 29 + j * (W // 3), size, v)
            _diag(diags, 3, 29 + j * (W // 3), size)
        for name, b in (('L', Ls), ('diag', diags)):
            out.append(('%s_fg_T%d' % (name, T), _paint(b, rng), T))
            out.append(('%s_hole_T%d' % (name, T), _paint(~b, rng), T))
        border = np.zeros((v + 8, W), bool)          # holes on the top-left, top-right and bottom borders
        _L(border, 0, 0, T - 1, v)
        border[0, W - (T - v):] = True
        border[1:v, W - 1] = True                     # T - 1 pixels along the top-right corner ...
        border[v + 7, W // 2:W // 2 + T] = True       # ... and T along the bottom row
        out.append(('border_holes_T%d' % T, _paint(~border, rng), T))
    for H, W in ((37, 65), (8, 1024), (9, 1100)):
        m = _paint(rng.random((H, W)) < 0.5, rng)
        for T in (0, 1, 2, 9, 150, H * W, H * W + 1):
            out.append(('random_%dx%d_T%d' % (H, W, T), m, T))
    for H, W in ((37, 65), (9, 1024)):
        for T in (H * W, H * W + 1):
            out.append(('all2_%dx%d_T%d' % (H, W, T), np.full((H, W), 2, np.uint8), T))
            out.append(('all0_%dx%d_T%d' % (H, W, T), np.zeros((H, W), np.uint8), T))
    return out


# ------------------------------------------------------------------------------------------------------------ stage
def _nested(H, W, cy, cx, blob_fg):
    """A 3 x 3 blob (9 px) in a 1-pixel ring (16 px) in a large field.  blob_fg: foreground blob in a background ring
    in foreground; otherwise the inverse."""
    fg = np.ones((H, W), bool) if blob_fg else np.zeros((H, W), bool)
    fg[cy - 2:cy + 3, cx - 2:cx + 3] = not blob_fg
    fg[cy - 1:cy + 2, cx - 1:cx + 2] = blob_fg
    return fg


def _stage(rng):
    out = []
    for H, W, cx in ((64, 64, 30), (40, 200, 32), (24, 1024, 1000)):
        for blob_fg in (True, False):
            name = 'blob_in_hole' if blob_fg else 'hole_in_blob'
            out.append(('%s_T40_%dx%d' % (name, H, W), _paint(_nested(H, W, H // 2, cx, blob_fg), rng), 40))
            out.append(('%s_T20_%dx%d' % (name, H, W), _paint(_nested(H, W, H // 2, cx, blob_fg), rng), 20))
    return out


# ------------------------------------------------------------------------------------------------------------- wrap
def _wrap(rng):
    out = []
    for W in (5, 31, 32, 33, 64, 65, 1023, 1024, 1025):
        b = np.zeros((8, W), bool)
        b[1, W - 1] = b[2, 0] = True                  # flat neighbours p, p + 1
        b[5, W - 1] = b[7, 0] = True                  # flat neighbours p, p + W + 1
        out.append(('pairs_w%d' % W, _paint(b, rng), 2))
        if W >= 16:
            r = np.zeros((8, W), bool)
            r[2, W - 3:] = r[3, :3] = True
            out.append(('runs_w%d' % W, _paint(r, rng), 4))
    return out


# ------------------------------------------------------------------------------------------------------- contention
def _contention(rng):
    return [('random_1024_d%02d_%d' % (d * 100, k), _paint(rng.random((1024, 1024)) < d, rng), 150)
            for d in (0.3, 0.5, 0.6, 0.7) for k in range(4)]


def catalogue():
    """Every entry, in a fixed order; the same masks on every call."""
    cases = []
    for i, (family, make) in enumerate((('lanes', _lanes), ('widths', _widths), ('topology', _topology),
                                        ('threshold', _threshold), ('stage', _stage), ('wrap', _wrap),
                                        ('contention', _contention))):
        rng = np.random.default_rng(1000 + i)
        cases += [Case('%s/%s' % (family, name), family, np.ascontiguousarray(m, dtype=np.uint8), int(T))
                  for name, m, T in make(rng)]
    return cases


# ----------------------------------------------------------------------------------------------- how entries run
def groups(cases):
    """Entries of one shape and threshold run together: {(H, W, T): [case, ...]} in catalogue order."""
    g = {}
    for c in cases:
        g.setdefault((c.mask.shape[0], c.mask.shape[1], c.threshold), []).append(c)
    return g


def guards(H, W, T):
    """(before, after) images for a dense batch: the last (first) max(T - 1, W) pixels in flat order are foreground, so
    the row at the shared edge is full.  Alone a guard's foreground has T - 1 pixels (or one full row); merged with
    anything across the image boundary, it or what it merged with reaches T."""
    k = min(H * W, max(T - 1, W))
    before = np.zeros(H * W, np.uint8)
    after = np.zeros(H * W, np.uint8)
    before[H * W - k:] = 2
    after[:k] = 1
    return before.reshape(H, W), after.reshape(H, W)


def dense_batch(entries):
    """[N, H, W] batch: guard, entry, guard, entry, ... guard.  An entry after the first guard meets full foreground rows
    on both sides, one after the second guard meets background; a lone entry is placed twice, once each way."""
    H, W = entries[0].mask.shape
    before, after = guards(H, W, entries[0].threshold)
    items = [e.mask for e in entries] if len(entries) > 1 else [entries[0].mask] * 2
    batch = []
    for j, m in enumerate(items):
        batch += [before if j % 2 == 0 else after, m]
    batch.append(before if len(items) % 2 == 0 else after)
    return np.stack(batch)


def ragged_canvas(entries, seed):
    """(canvas u8 [N, H + RAGGED_EXTRA, W], heights int32 [N], index of each image's entry).  Each entry is extended by
    RAGGED_EXTRA random rows and enters at its own height H and at the canvas height; the first two entries of at most
    256 rows also at the heights in RAGGED_HEIGHTS.  Rows below an image's height hold random bytes, zeros included."""
    rng = np.random.default_rng(seed)
    H, W = entries[0].mask.shape
    Hc = H + RAGGED_EXTRA
    rows = []
    for j, e in enumerate(entries):
        ext = np.concatenate([e.mask, _paint(rng.random((RAGGED_EXTRA, W)) < 0.5, rng)])
        for h in ((H, Hc) + (RAGGED_HEIGHTS if j < 2 and H <= 256 else ())):
            rows.append((ext, h, j))
    canvas = rng.integers(0, 256, (len(rows), Hc, W)).astype(np.uint8)
    canvas[rng.random(canvas.shape) < 0.3] = 0
    for n, (ext, h, _) in enumerate(rows):
        canvas[n, :h] = ext[:h]
    return canvas, np.array([h for _, h, _ in rows], np.int32), [j for _, _, j in rows]


def ragged_expected(canvas, heights, threshold, exclude=False):
    """The canvas after K5: each image's valid rows replaced by the oracle's result, the dead rows as they were."""
    exp = canvas.copy()
    counts = np.zeros((len(heights), 3), np.int64)
    for n, h in enumerate(heights):
        out = opost.remove_small_zones_2d(canvas[n, :h], threshold)
        if exclude:
            out = opost.exclude_nodes(out)
        exp[n, :h] = out
        counts[n] = np.bincount(out.ravel(), minlength=3)[:3]
    return exp, counts


def components(mask):
    """8-connected components of the foreground plus those of the background."""
    return ndi.label(mask != 0, opost.STRUCT8)[1] + ndi.label(mask == 0, opost.STRUCT8)[1]


# ---------------------------------------------------------------------------------------------- wrong references
def zones_with(mask, threshold, label, strict=True, stage_b_on_original=False):
    """The oracle's two stages with the labelling, the comparison or the stage-B input swapped out."""
    img = np.array(mask, copy=True)
    fg0 = img != 0

    def small(binary):
        lab = label(binary)
        sizes = np.bincount(lab.ravel())
        s = sizes < threshold if strict else sizes <= threshold
        s[0] = False
        return s[lab]

    bg = ~fg0 | small(fg0)
    bg = bg & ~small(~fg0 if stage_b_on_original else bg)
    img[~bg & (img == 0)] = 1
    img[bg & (img != 0)] = 0
    return img


def label8(b):
    return ndi.label(b, opost.STRUCT8)[0]


def label4(b):
    return ndi.label(b, ndi.generate_binary_structure(2, 1))[0]


def label_flat(b):
    """Neighbours by flat index, p +- 1, p +- (W - 1), p +- W, p +- (W + 1): joins the end of a row to the next row."""
    H, W = b.shape
    f = b.ravel()
    src, dst = [], []
    for d in (1, W - 1, W, W + 1):
        if 0 < d < f.size:
            p = np.nonzero(f[:-d] & f[d:])[0]
            src.append(p)
            dst.append(p + d)
    src, dst = np.concatenate(src), np.concatenate(dst)
    g = coo_matrix((np.ones(src.size, np.int8), (src, dst)), shape=(f.size, f.size))
    _, lab = connected_components(g, directed=False)
    lab = lab + 1
    lab[~f] = 0
    return np.unique(lab, return_inverse=True)[1].reshape(H, W) if f.any() else np.zeros((H, W), np.int64)


def label_volume(b):
    """The reference's structuring element for a [B, H, W] array (SURVEY.md 3.3): in-plane 8-connectivity that also
    links each pixel to neighbouring batch images."""
    return ndi.label(b, ndi.generate_binary_structure(3, 2))[0]


WRONG = {
    'four_connectivity': lambda m, T: zones_with(m, T, label4),
    'threshold_inclusive': lambda m, T: zones_with(m, T, label8, strict=False),
    'stage_b_on_original': lambda m, T: zones_with(m, T, label8, stage_b_on_original=True),
    'flat_row_wrap': lambda m, T: zones_with(m, T, label_flat),
}
# wrong reference -> (entry it is designed to fail on, how the entry is presented: 'image' | 'dense' | 'ragged')
CONTROLS = {
    'four_connectivity': ('lanes/stair_down_w64', 'image'),
    'threshold_inclusive': ('threshold/L_fg_T40', 'image'),
    'stage_b_on_original': ('stage/blob_in_hole_T40_64x64', 'image'),
    'flat_row_wrap': ('wrap/pairs_w33', 'image'),
    'batch_as_volume': ('topology/comb_bottom_64x64', 'dense'),
    'batch_as_one_image': ('topology/comb_bottom_64x64', 'dense'),
    'dead_rows_included': ('topology/stripes_drop_64x64', 'ragged'),
}


def wrong_output(control, case, presented):
    """The wrong reference's result for ``case`` as presented: one image, a dense batch (array) or a ragged canvas
    (canvas, heights), with the dead rows of the canvas read as part of each image."""
    T = case.threshold
    if control in WRONG:
        return WRONG[control](case.mask, T)
    if control == 'batch_as_volume':
        return zones_with(presented, T, label_volume)
    if control == 'batch_as_one_image':
        N, H, W = presented.shape
        return zones_with(presented.reshape(N * H, W), T, label8).reshape(N, H, W)
    if control == 'dead_rows_included':
        canvas, heights = presented
        out = canvas.copy()
        for n, h in enumerate(heights):
            out[n, :h] = zones_with(canvas[n], T, label8)[:h]
        return out
    raise KeyError(control)


def lane_events(mask):
    """Where the run kernels' union events fire, pixel by pixel (rows_merge's word expressions):
    E1 = C & U & ~(L & UL), E2 = C & ~U & UL & ~L, E3 = C & ~U & UR & ~R; row 0 has none."""
    c = mask != 0
    z = np.zeros_like(c)
    U = np.concatenate([z[:1], c[:-1]])
    L = np.pad(c, ((0, 0), (1, 0)))[:, :-1]
    R = np.pad(c, ((0, 0), (0, 1)))[:, 1:]
    UL = np.pad(U, ((0, 0), (1, 0)))[:, :-1]
    UR = np.pad(U, ((0, 0), (0, 1)))[:, 1:]
    return c & U & ~(L & UL), c & ~U & UL & ~L, c & ~U & UR & ~R
