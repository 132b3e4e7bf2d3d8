"""Folder pipeline behind ``predict.py``: raw scans on disk -> ``processed/`` PNGs, ``results/outputs`` PNGs and
``results/final_stats.csv`` in ONE streaming pass (reference: predict.py:51-58 = Preprocessor.preprocess_images followed by
NeuralBarkCalculator.predict, models.py:173-203 and 230-364).

    reader threads : BMP pixel arrays -> pinned host buffers (file.readinto, no decode)
    main thread    : batches of scans -> PredictEngine.submit_host / collect (K1, network, K3, K5 on the GPU; two batches
                     in flight so the PCIe link stays busy)
    writer threads : PNG encode of the processed image and of the 0/127/255 dual image (zlib releases the GIL)

The files are the reference's: same names, same CSV layout, and the pixels of the oracle's restatement of the reference --
processed images equal to the reference's except, possibly, one LSB on exact rounding ties (the float -> u8 rounding of
scikit-image 0.15's save path is unpinned, see oracle/preprocess.py), class maps within the floating-point bar of
DESIGN.md 5.  Only the PNG compression level is a knob (``png_compress_level``, pixels are unaffected).

Two routes, one streaming pass each.  A folder of standard scans (uncompressed 24-bit 4096x4096 BMPs of one row order,
``supported()``) takes the uniform route: the readers copy BMP pixel arrays, K1 is the 4x kernel for every scan.  Any
other folder takes the mixed route, which accepts every input the per-image route of models.py accepts: the readers copy
the pixel array of any 24-bit BMP and decode everything else with ``dataset.pil_loader`` (the per-image route's decoder),
``PredictEngine.submit_mixed`` routes each image as ``Preprocessor.preprocess_array`` does (4x, general-ratio resize,
trim only, or unchanged) and images narrower than the canvas run in ragged chunks of their own width.  Both routes write
the per-image route's files: same names, formats, pixels and CSV rows (in dataset order)."""
import csv
import mmap
import os
import struct
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from os.path import join

import numpy as np
import torch
from ._png import write_png
from .dataset import make_dataset, pil_loader
from . import figure, ops
from .engine import PredictEngine

RAW = 4096
CSV_HEADER = ['Name', 'Type', 'Image Size', 'Output Bark %', 'Bark area (mm^2)', 'Output Node %', 'Node area (mm^2)']
_DUAL_LUT = np.array([0, 127, 255] + [0] * 253, dtype=np.uint8)     # models.py:349-353
# matplotlib's viridis at 0, 0.5, 1 -- the colours of classes 0 / 1 / 2 in the reference figure (imshow(vmax=2), models.py:300)
_VIRIDIS3 = np.array([[68, 1, 84], [33, 145, 140], [253, 231, 37]] + [[0, 0, 0]] * 253, dtype=np.uint8)


_GLYPHS = {}       # character -> (uint8 [16, advance] grey glyph on white, advance in pixels): rendered by PIL once


def _glyph(ch):
    g = _GLYPHS.get(ch)
    if g is None:
        from PIL import Image, ImageDraw, ImageFont
        font = _GLYPHS.get('font')
        if font is None:
            font = _GLYPHS['font'] = ImageFont.load_default()
        adv = max(1, int(np.ceil(font.getlength(ch)))) if hasattr(font, 'getlength') else 6
        im = Image.new('L', (adv + 2, 16), 255)
        ImageDraw.Draw(im).text((0, 2), ch, fill=0, font=font)
        g = _GLYPHS[ch] = (np.ascontiguousarray(np.asarray(im)), adv)
    return g


def title_strip(title, width, height=16):
    """White RGB strip [height, width, 3] with the title in black.  Glyphs come from PIL's default font, rendered once
    per character and cached -- a full PIL text render per image holds the GIL for 1.5 ms and would cap the writer
    threads at ~600 images/s."""
    strip = np.full((height, width), 255, dtype=np.uint8)
    x = 4
    for ch in title:
        g, adv = _glyph(ch)
        w = min(g.shape[1], width - x)
        if w <= 0:
            break
        np.minimum(strip[:, x:x + w], g[:height, :w], out=strip[:, x:x + w])
        x += adv
    return np.repeat(strip[:, :, None], 3, axis=2)


def combined_image(proc, mask, title):
    """Stand-in for the reference's two-panel matplotlib figure (models.py:280-347; matplotlib is not a dependency here):
    the processed image and the class mask in the figure's colours side by side at half resolution, the figure's
    suptitle (class percentages) drawn in a strip above.  Same information, not the same rendering.  The panels are
    composed by nbc_compose_combined (host code in libnbc.so, GIL released)."""
    import ctypes as C
    from . import _lib
    proc, mask = np.ascontiguousarray(proc), np.ascontiguousarray(mask)
    h, w = mask.shape
    hh, hw = (h + 1) // 2, (w + 1) // 2
    strip = title_strip(title, 2 * hw + 8)
    canvas = np.empty((hh + 16, 2 * hw + 8, 3), dtype=np.uint8)
    lib = _lib.load()
    _lib.check(lib.nbc_compose_combined(C.c_void_p(proc.ctypes.data), C.c_void_p(mask.ctypes.data), h, w,
                                        C.c_void_p(_VIRIDIS3.ctypes.data), C.c_void_p(strip.ctypes.data), 16, 8,
                                        C.c_void_p(canvas.ctypes.data)), 'nbc_compose_combined')
    return canvas


_FIGURE_LOCK = threading.Lock()      # pyplot keeps global state: the optional matplotlib renderer runs one figure at a time


def write_combined(path, proc, mask, stats, fname, mean, std, png_level=1):
    """results/combined_images/<wood>/<fname> for one image, by NBC_COMBINED (figure.py): the reference's matplotlib figure
    ('figure'), the native half-resolution stand-in (default) or nothing ('0').  stats = [bark %, bark mm^2, node %, node
    mm^2] as the CSV strings (models.py:323-332)."""
    kind = figure.mode()
    if kind == 'off':
        return
    if kind == 'figure':
        with _FIGURE_LOCK:
            figure.save_reference_figure(path, proc, mask, (float(stats[0]), float(stats[2])), mean, std)
        return
    title = 'Bark : %.3f;  Node : %.3f   (%s)' % (float(stats[0]), float(stats[2]), fname)     # cf. models.py:334-343
    write_png(path, combined_image(proc, mask, title), png_level)


def bmp_geometry(path):
    """(data offset, bottom_up) of an uncompressed 24-bit RAW x RAW BMP, else None."""
    try:
        with open(path, 'rb') as f:
            head = f.read(54)
    except OSError:
        return None
    if len(head) < 54 or head[:2] != b'BM':
        return None
    off = struct.unpack_from('<I', head, 10)[0]
    hdr_size, w, h, planes, bpp, comp = struct.unpack_from('<IiiHHI', head, 14)
    if hdr_size < 40 or bpp != 24 or comp != 0 or planes != 1 or w != RAW or abs(h) != RAW:
        return None
    return off, h > 0


def supported(items):
    """True when every input is a 4096x4096 24-bit BMP with one row orientation (what the scanner produces)."""
    geo = [bmp_geometry(path) if path.lower().endswith('.bmp') else None for path, _, _, _ in items]
    return len(geo) > 0 and all(g is not None for g in geo) and len({g[1] for g in geo}) == 1


def raw_geometry(path):
    """How a reader gets an input's pixels, for the mixed route: (bmp data offset or None, H, W, pitch, bgr, bottom_up).
    An uncompressed 24-bit BMP (any size, either row order) is read as its pixel array, as ``Preprocessor`` reads it
    (``dataset.read_bmp_pixels``); any other file is decoded by ``dataset.pil_loader`` into RGB top-down rows."""
    if path.lower().endswith('.bmp'):
        try:
            with open(path, 'rb') as f:
                head = f.read(54)
            size = os.path.getsize(path)
        except OSError:
            head, size = b'', 0
        if len(head) == 54 and head[:2] == b'BM':
            off = struct.unpack_from('<I', head, 10)[0]
            hdr_size, w, h, planes, bpp, comp = struct.unpack_from('<IiiHHI', head, 14)
            pitch = (w * 3 + 3) & ~3
            if hdr_size >= 40 and bpp == 24 and comp == 0 and planes == 1 and w > 0 and h != 0 and size >= off + pitch * abs(h):
                return off, abs(h), w, pitch, True, h > 0
    from PIL import Image
    with Image.open(path) as im:
        w, h = im.size
    return None, h, w, w * 3, False, False


def read_raw(path, geo, buf, zero_span, target):
    """Pixels of one input of the mixed route into the pinned buffer ``buf`` -> (row0, rows) to copy to the device.  A
    (4 target)^2 image is reduced to the rows between its all-zero bands when ``zero_span`` (``read_scan`` for the BMP,
    the same host scan after decoding otherwise); any other image is copied whole."""
    off, H, W, pitch, _, _ = geo
    scan = zero_span and H == W == 4 * target
    if off is not None and scan and H == RAW:
        return read_scan(path, off, buf, True)
    view = buf.numpy()
    if off is not None:
        with open(path, 'rb', buffering=0) as f:
            f.seek(off)
            mv, got = memoryview(view), 0
            while got < H * pitch:
                n = f.readinto(mv[got:H * pitch])
                if not n:
                    raise IOError('short read: ' + path)
                got += n
    else:
        img = pil_loader(path)
        if img.shape != (H, W, 3):
            raise IOError('%s decodes to %s, its header says %dx%d' % (path, img.shape, H, W))
        np.copyto(view[:H * pitch].reshape(H, W, 3), img)
    return ops.host_zero_row_span(buf, H, pitch, W * 3) if scan else (0, H)


def save_image(path, arr, png_level, lut=None):
    """One output file as the per-image route writes it: a PNG with the library's encoder, any other extension through
    PIL in the format the extension names (models.py:203, 356)."""
    if path.lower().endswith('.png'):
        write_png(path, arr, png_level, lut=lut)
    else:
        from PIL import Image
        Image.fromarray(arr if lut is None else lut[arr]).save(path)


def read_scan(path, off, buf, zero_span=True):
    """Pixel array of a RAW x RAW 24-bit BMP (file offset ``off``) into the pinned buffer ``buf`` -> (row0, rows), the
    memory rows between the scan's all-zero dark bands (whole groups of 4; engine.py).  With ``zero_span`` the file is
    mapped, the bands are found in the page cache (``nbc_host_zero_row_span``: only the zero rows are touched) and ONLY the
    rows in between are copied into ``buf`` -- the engine never reads the others; otherwise the whole array is read."""
    nbytes, pitch = RAW * RAW * 3, RAW * 3
    view = buf.numpy()
    with open(path, 'rb', buffering=0) as f:
        if zero_span:
            try:
                mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
            except (OSError, ValueError):
                mm = None
            if mm is not None:
                try:
                    if len(mm) < off + nbytes:
                        raise IOError('short file: ' + path)
                    src = np.frombuffer(mm, dtype=np.uint8, count=nbytes, offset=off)
                    row0, rows = ops.host_zero_row_span(src, RAW, pitch)
                    if rows:
                        np.copyto(view[row0 * pitch:(row0 + rows) * pitch], src[row0 * pitch:(row0 + rows) * pitch])
                    del src
                finally:
                    mm.close()
                return row0, rows
        f.seek(off)
        mv = memoryview(view)
        got = 0
        while got < nbytes:
            n = f.readinto(mv[got:nbytes])
            if not n:
                raise IOError('short read: ' + path)
            got += n
    return ops.host_zero_row_span(buf, RAW, pitch) if zero_span else (0, RAW)




class FolderPipeline:
    def __init__(self, calculator, batch=16, io_threads=None, png_compress_level=None):
        if png_compress_level is None:      # 0 = stored (fastest, 1.9 MB per processed image), 1 = fast deflate (default)
            png_compress_level = int(os.environ.get('NBC_PNG_LEVEL', '1'))
        # results/combined_images/<wood>/<name>.png (the reference always writes its figure): NBC_COMBINED=0 skips it,
        # NBC_COMBINED=figure draws the reference's matplotlib figure instead of the native stand-in (figure.py)
        self.combined = figure.mode() != 'off'
        self.calc = calculator
        self.batch = batch
        self.io_threads = io_threads or max(4, min(32, (os.cpu_count() or 8)))
        self.png_level = png_compress_level
        self.engine = PredictEngine(calculator.model, calculator.device, raw_size=RAW)

    def run(self, root_path, excludes_nodes, only_preprocess=False, shard=None):
        """shard=(start, end): process only that slice of the dataset order and return its CSV rows WITHOUT writing
        final_stats.csv (data-parallel runs: one process per GPU, rank 0 merges the rows -- distributed.merge_rows).
        A folder of standard scans (``supported``) takes the uniform route: 4x K1 on every scan, one canvas width.  Any
        other folder takes the mixed route: every input the per-image route accepts, each resized / trimmed as
        ``Preprocessor.preprocess_array`` does, in the same streaming pass."""
        t_start = time.perf_counter()
        timing = {'read_s': 0.0, 'save_s': 0.0}      # summed over the IO threads
        items = make_dataset(root_path)
        if len(items) == 0:
            raise RuntimeError("Found 0 files in subfolders of: " + root_path)
        standard = supported(items)
        if shard is not None:
            items = items[shard[0]:shard[1]]
            if len(items) == 0:
                self.last_timing = {'images': 0}
                return []
        rows_csv = [None] * len(items)
        out_proc = join(root_path, 'processed', 'samples')
        out_dual = join(root_path, 'results', 'outputs')
        out_comb = join(root_path, 'results', 'combined_images')
        engine = self.engine
        Wo = RAW // 4
        if standard:
            geo = [bmp_geometry(p) for p, _, _, _ in items]
            bottom_up = geo[0][1]
            nbytes = RAW * RAW * 3

            def read(i, buf):
                # the reader finds the scan's all-zero dark bands while it reads: they never enter the pinned buffer, let
                # alone cross PCIe (engine.py)
                return read_scan(items[i][0], geo[i][0], buf, engine.zero_span)

            def submit(idx, bufs, spans, masks):
                return engine.submit_host(bufs, masks, bgr=True, bottom_up=bottom_up, exclude_nodes=excludes_nodes,
                                          want_processed=True, only_preprocess=only_preprocess, spans=spans)

            def results(ticket):
                rows, counts, masks = engine.collect(ticket)
                proc_host = ticket.slot.proc_host
                for k, h in enumerate(rows):
                    yield proc_host[k, :h], None if only_preprocess else masks[k][:h * Wo].numpy().reshape(h, Wo), counts[k]

            save_file = write_png
        else:
            geo = [raw_geometry(p) for p, _, _, _ in items]
            nbytes = max(g[1] * g[3] for g in geo)
            engine.reserve_mixed(nbytes)

            def read(i, buf):
                return read_raw(items[i][0], geo[i], buf, engine.zero_span, Wo)

            def submit(idx, bufs, spans, masks):
                return engine.submit_mixed(bufs, [geo[i][1:] for i in idx], masks, exclude_nodes=excludes_nodes,
                                           want_processed=True, only_preprocess=only_preprocess, spans=spans)

            def results(ticket):
                rows, widths, counts, masks = engine.collect_mixed(ticket)
                for k, (h, w) in enumerate(zip(rows, widths)):
                    yield (engine.processed(ticket, k, h), None if only_preprocess else masks[k][:h * w].numpy().reshape(h, w),
                           counts[k])

            save_file = save_image
        timing['setup_s'] = time.perf_counter() - t_start
        self._stream(items, nbytes, read, submit, results, save_file, rows_csv, timing, only_preprocess,
                     (out_proc, out_dual, out_comb))
        timing['total_s'] = time.perf_counter() - t_start
        timing['images'] = len(items)
        self.last_timing = timing
        if only_preprocess:
            return None
        if shard is not None:
            return rows_csv
        results_csv = [CSV_HEADER] + rows_csv
        with open(join(root_path, 'results', 'final_stats.csv'), 'w') as f:   # as models.py:360-364 (tab-delimited)
            csv.writer(f, delimiter='\t').writerows(results_csv)
        return results_csv

    def _stream(self, items, nbytes, read, submit, results, save_file, rows_csv, timing, only_preprocess, out_dirs):
        """The streaming pass: reader threads -> batches of B items submitted to the engine (two in flight) -> writer
        threads.  read(i, buf) -> span; submit(idx, bufs, spans, masks) -> ticket; results(ticket) yields (processed u8
        [h, w, 3], mask u8 [h, w] or None, counts) per item of the batch; save_file(path, arr, level, lut=None)."""
        out_proc, out_dual, out_comb = out_dirs
        B = self.batch
        # Pinned staging buffers: 3 batches' worth (2 in flight + 1 being read).  The MAIN thread hands them out as tokens
        # in item order -- a reader can therefore never hold a buffer that an earlier item is still waiting for (a free-for-
        # all pool deadlocks: later items overtake a parked reader and exhaust it) -- while the page-locking itself (about
        # 1 s per GB) is done by the reader threads on a token's first use, overlapping the reads and the GPU work.
        n_tokens = min(3 * B, len(items))
        tokens = list(range(n_tokens))           # free tokens (main thread only)
        pinned = [None] * n_tokens
        spans = [None] * n_tokens
        mask_sets = [[torch.empty((RAW // 4) * (RAW // 4), dtype=torch.uint8).pin_memory() for _ in range(min(B, len(items)))]
                     for _ in range(2)]

        def load(i, tok):
            if pinned[tok] is None:
                pinned[tok] = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            t0 = time.perf_counter()
            spans[tok] = read(i, pinned[tok])
            timing['read_s'] += time.perf_counter() - t0
            return tok

        def save(i, proc, mask, counts):
            t0 = time.perf_counter()
            _, _, fname, wood = items[i]
            fname = fname.replace('.bmp', '.png')           # models.py:185
            save_file(join(out_proc, wood, fname), proc, self.png_level)
            if mask is not None:
                save_file(join(out_dual, wood, fname), mask, self.png_level, lut=_DUAL_LUT)
                rows_csv[i] = [fname, wood] + self.calc._stats_strings(counts, mask.size)
                if self.combined:
                    write_combined(join(out_comb, wood, fname), proc, mask, rows_csv[i][2:], fname, self.calc.mean, self.calc.std,
                                   self.png_level)
            timing['save_s'] += time.perf_counter() - t0

        readers, writers = ThreadPoolExecutor(self.io_threads), ThreadPoolExecutor(self.io_threads)
        loads, fed = [None] * len(items), [0]

        def feed():
            while fed[0] < len(items) and tokens:
                loads[fed[0]] = readers.submit(load, fed[0], tokens.pop(0))
                fed[0] += 1

        try:
            pending, saves = [], []

            def finish(entry):
                ticket, idx, toks = entry
                for i, (proc, mask, counts) in zip(idx, results(ticket)):
                    saves.append(writers.submit(save, i, proc.numpy().copy(), None if mask is None else mask.copy(),
                                                None if only_preprocess else counts.tolist()))
                tokens.extend(toks)      # the H2D copies of this batch are done: its staging buffers are free again
                feed()

            feed()
            for a in range(0, len(items), B):
                idx = list(range(a, min(a + B, len(items))))
                toks = [loads[i].result() for i in idx]
                ticket = submit(idx, [pinned[t] for t in toks], [spans[t] for t in toks],
                                None if only_preprocess else mask_sets[(a // B) & 1][:len(idx)])
                pending.append((ticket, idx, toks))
                if len(pending) == 2:
                    finish(pending.pop(0))
            while pending:
                finish(pending.pop(0))
            for s in saves:
                s.result()
        finally:
            for f in loads:
                if f is not None:
                    f.cancel()
            readers.shutdown(wait=True)
            writers.shutdown(wait=True)
