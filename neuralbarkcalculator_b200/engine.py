"""Batched predict engine: raw scans -> (class mask, class counts) with the whole hot path on the GPU.

One image goes through  K1 resize+trim -> FCN-ResNet50 plan -> K3 upsample+argmax -> K5 region removal+counts
(models.py:191-203 and 247-332 of the reference).  The engine removes the reference's per-image host round trips
entirely: images are processed in RAGGED batches (a canvas of ``chunk`` images of different trimmed heights; every
kernel reads the per-image heights K1 produced on the device), so nothing is read back until the final counts.

``run_host`` is the public end-to-end entry (pinned host buffers in, host masks out).  ``submit_host`` / ``collect``
are its asynchronous halves: a submitted batch only enqueues work, so the host->device copies of the NEXT batch run
under the network passes of the current one (two buffer slots) and the PCIe link -- the end-to-end bound, 50 MB per
scan -- never idles between batches.

Dark bands stay on the host: the rows of a scan above and below the bark that are EXACTLY zero (what trim_black removes)
resize to exact zeros, so ``submit_host`` finds them with a host scan (``nbc_host_zero_row_span``, a few worker threads,
GIL released), copies only the rows in between -- still one ``cudaMemcpyAsync`` per scan -- and K1 treats the rest as
zeros (``nbc_preprocess_4x_span_u8``).  Bit-identical to copying the whole scan (global min / max clip included);
``NBC_ZERO_SPAN=0`` switches it off.

``submit_mixed`` / ``collect_mixed`` take raw images of any sizes and layouts (the folder pipeline's mixed route): K1 routes
each image as ``Preprocessor.preprocess_array`` does (``nbc_preprocess_mixed_batch_u8``), and a batch runs as chunks of one
canvas width."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import torch

from . import ops


# images per ragged batch.  Two effects, both measured (profiles/r02e_chunk_sweep.txt): the per-launch cost of the ~53 network
# kernels (launch gap, pipeline fill and drain) is amortised over the chunk, and -- the larger one -- the last partial WAVE of
# every conv launch: a chunk of 8 trimmed scans has ~620 M tiles at the 128-wide layers, i.e. 8.4 rounds of the 74 CTA pairs
# (9 are paid), a chunk of 16 has 16.9 (17 are paid).  With K1 issued once per chunk the end-to-end path gains as well:
# chunk 8 -> 16: value 1 395 -> 1 419 img/s, e2e 1 358 -> 1 397.
DEFAULT_CHUNK = 16
# raw-scan staging buffers of the host path (50 MB each), in units of chunks: K1 runs once per chunk (three launches for all
# its scans), so the H2D stream needs a second chunk's worth of buffers to keep copying while K1 waits for its turn
DEFAULT_STAGE_DEPTH = 2


class _Slot:
    """Per-batch buffers; two of them alternate so that batch k+1 can be staged while batch k is in flight."""

    def __init__(self, n, Hc, Wo, dev):
        self.n = n
        self.proc = torch.empty((n, Hc, Wo, 3), dtype=torch.uint8, device=dev)      # canvas: image i in rows [0, h_i)
        self.fl = torch.empty((n, 2), dtype=torch.int32, device=dev)
        self.heights = torch.empty(n, dtype=torch.int32, device=dev)
        self.masks = torch.empty((n, Hc, Wo), dtype=torch.uint8, device=dev)
        self.counts = torch.empty((n, 3), dtype=torch.int32, device=dev)
        self.fl_host = torch.empty((n, 2), dtype=torch.int32).pin_memory()
        self.counts_host = torch.empty((n, 3), dtype=torch.int32).pin_memory()
        self.proc_host = None     # pinned copies of the processed canvases (folder pipeline only)
        self.done = None          # event: every consumer of this slot's buffers has finished
        self.pending = False      # a submitted batch in this slot has not been collected yet


class Ticket:
    def __init__(self, slot, n, masks_host):
        self.slot, self.n, self.masks_host = slot, n, masks_host


class PredictEngine:
    """chunk: images per ragged batch (one network launch sequence per chunk); default DEFAULT_CHUNK, or the
    environment variable NBC_CHUNK."""

    def __init__(self, model, device='cuda:0', threshold=150, raw_size=4096, chunk=None, depth=None):
        if chunk is None:
            chunk = int(os.environ.get('NBC_CHUNK', DEFAULT_CHUNK))
        if depth is None:      # staging buffers (NBC_STAGE_DEPTH counts chunks)
            depth = int(os.environ.get('NBC_STAGE_DEPTH', DEFAULT_STAGE_DEPTH)) * chunk
        self.model = model
        self.device = torch.device(device)
        self.threshold = threshold
        self.raw_size = raw_size
        self.out_w = raw_size // 4
        self.chunk = chunk
        self.depth = max(depth, chunk)      # a chunk's scans are all staged before its K1 runs
        self.zero_span = os.environ.get('NBC_ZERO_SPAN', '1') != '0'
        self._scan_pool = None
        self.h2d_bytes = 0        # raw-scan bytes really copied host -> device so far
        self._slots = [None, None]
        self._calls = 0
        self._chunks = 0          # chunks issued so far (logits double buffer)
        self._issued = 0          # host scans staged so far (staging ring)
        self._copy_stream = None
        self._stage = None
        self._mixed_stage, self._mixed_bytes, self._mixed_issued = None, 0, 0

    # -- buffers ------------------------------------------------------------------------------------------------
    def _slot(self, n):
        S, Wo = self.raw_size, self.out_w
        Hc = S // 4
        k = self._calls & 1
        self._calls += 1
        s = self._slots[k]
        if s is not None and s.pending:
            raise RuntimeError('PredictEngine: at most two submitted batches may be outstanding; collect() the oldest first')
        if s is None or s.n < n:
            if s is not None and s.done is not None:
                s.done.synchronize()
            s = self._slots[k] = _Slot(n, Hc, Wo, self.device)
        return s

    def _streams(self):
        if self._copy_stream is not None:
            return False
        dev = self.device
        S, Wo = self.raw_size, self.out_w
        Hc = S // 4
        self._copy_stream = torch.cuda.Stream(dev)      # H2D of raw scans
        self._pre_stream = torch.cuda.Stream(dev)       # K1 (resize + trim)
        self._out_stream = torch.cuda.Stream(dev)       # D2H of masks and counts
        self._post_stream = torch.cuda.Stream(dev)      # K3 + K5 of a chunk, behind the network pass of the next one
        lib = ops._lib.load()
        self._ccl_ws = torch.empty(lib.nbc_ccl_workspace_bytes(self.chunk, Hc, Wo), dtype=torch.uint8, device=dev)
        hl = (((Hc - 1) // 2 + 1 - 1) // 2 + 1 - 1) // 2 + 1
        wl = (((Wo - 1) // 2 + 1 - 1) // 2 + 1 - 1) // 2 + 1
        self._logits = [torch.empty((self.chunk, 3, hl, wl), dtype=torch.float32, device=dev) for _ in range(2)]
        self._logits_free = [None, None]
        return True

    def _standard_buffers(self):
        """Staging ring (``depth`` raw scans of raw_size^2 x 3 bytes) and K1 workspace of the uniform host path."""
        if self._stage is not None:
            return
        S, dev = self.raw_size, self.device
        self._stage = [torch.empty(S * S * 3, dtype=torch.uint8, device=dev) for _ in range(self.depth)]
        self._staged = [torch.cuda.Event() for _ in range(self.depth)]
        self._freed = [torch.cuda.Event() for _ in range(self.depth)]
        self._pre_ws = torch.empty(self.chunk * ops._lib.load().nbc_preprocess_workspace_bytes(S, S), dtype=torch.uint8, device=dev)

    def _preprocess_into(self, slot, i, raw, bgr, bottom_up, span=None):
        """K1 on the current stream.  span = (row0, rows): ``raw`` holds only those memory rows of the scan, the others are
        all zero (see the module docstring)."""
        lib = ops._lib.load()
        S = self.raw_size
        row0, rows = span if span is not None else (0, S)
        ops._lib.check(lib.nbc_preprocess_4x_span_u8(C.c_void_p(raw.data_ptr()), S, S, S * 3, (1 if bgr else 0) | (2 if bottom_up else 0),
                                                     row0, rows, C.c_void_p(slot.proc[i].data_ptr()), C.c_void_p(slot.fl[i].data_ptr()),
                                                     C.c_void_p(self._pre_ws.data_ptr()), self._pre_ws.numel(),
                                                     C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                       'nbc_preprocess_4x_span_u8')

    def _preprocess_chunk(self, slot, a, b, ptrs, spans, bgr, bottom_up):
        """K1 for images a..b-1 of the slot in three launches (nbc_preprocess_4x_batch_u8) on the current stream.  ptrs: device
        addresses of the (span of the) raw scans; spans: (row0, rows) per scan."""
        lib = ops._lib.load()
        S, n = self.raw_size, b - a
        arr = (C.c_void_p * n)(*ptrs)
        r0 = (C.c_int32 * n)(*[sp[0] for sp in spans])
        rows = (C.c_int32 * n)(*[sp[1] for sp in spans])
        ops._lib.check(lib.nbc_preprocess_4x_batch_u8(arr, r0, rows, n, S, S, S * 3, (1 if bgr else 0) | (2 if bottom_up else 0),
                                                      C.c_void_p(slot.proc[a].data_ptr()), slot.proc.stride(0),
                                                      C.c_void_p(slot.fl[a].data_ptr()), C.c_void_p(self._pre_ws.data_ptr()),
                                                      self._pre_ws.numel(),
                                                      C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                       'nbc_preprocess_4x_batch_u8')

    def _scan(self, raw):
        """(row0, rows) of a host scan: the memory rows between its all-zero bands, in whole groups of 4."""
        S = self.raw_size
        r0, rows = C.c_int32(0), C.c_int32(0)
        ops._lib.check(ops._lib.load().nbc_host_zero_row_span(C.c_void_p(raw.data_ptr()), S, S * 3, S * 3, 4, C.byref(r0), C.byref(rows)),
                       'nbc_host_zero_row_span')
        return r0.value, rows.value

    def _spans(self, n, get_raw, spans):
        """Per-scan (row0, rows) futures for a host batch: given by the caller, scanned by the worker threads, or the whole
        scan when the zero-band path is off."""
        S = self.raw_size
        if spans is not None:
            return [(lambda v=v: v) for v in spans]
        if not self.zero_span:
            return [(lambda: (0, S))] * n
        if self._scan_pool is None:
            self._scan_pool = ThreadPoolExecutor(int(os.environ.get('NBC_SCAN_THREADS', 4)), thread_name_prefix='nbc-scan')
        return [self._scan_pool.submit(self._scan, get_raw(i)).result for i in range(n)]

    def _segment_chunk(self, slot, a, b, exclude_nodes, proc=None, masks=None):
        """Images a..b-1 as ONE ragged batch: network, K3 and K5 read the per-image heights on the device.  The network
        runs on the main stream; K3 (upsample+argmax) and K5 (region removal + counts) follow on the post stream (two
        logits buffers).  proc / masks: the chunk's canvases when they are narrower than the slot's (mixed path).
        Returns the event that marks the chunk's masks and counts as final."""
        proc = slot.proc[a:b] if proc is None else proc
        masks = slot.masks[a:b] if masks is None else masks
        plan = self.model.native_plan()
        main = torch.cuda.current_stream(self.device)
        k = self._chunks & 1
        self._chunks += 1
        if self._logits_free[k] is not None:
            main.wait_event(self._logits_free[k])        # K3 of two chunks ago has consumed this logits buffer
        Hc, W = masks.shape[1], masks.shape[2]
        lg = self._logits[k]
        if W == self.out_w:
            lg = lg[:b - a]
        else:        # a narrower canvas: its logits, ceil(W / 8) wide, in the front of the same buffer
            lg = lg.view(-1)[:(b - a) * 3 * lg.shape[2] * ((W + 7) // 8)].view(b - a, 3, lg.shape[2], (W + 7) // 8)
        logits = plan.forward_ragged(proc, heights=slot.heights[a:b], out=lg)
        net_done = torch.cuda.Event()
        net_done.record(main)
        done = torch.cuda.Event()
        with torch.cuda.stream(self._post_stream):
            self._post_stream.wait_event(net_done)
            ops.upsample_argmax_ragged(logits, slot.heights[a:b], (Hc, W), out=masks)
            free = torch.cuda.Event()
            free.record(self._post_stream)
            self._logits_free[k] = free
            ops.remove_small_zones_ragged(masks, slot.heights[a:b], self.threshold, exclude_nodes,
                                          workspace=self._ccl_ws, counts=slot.counts[a:b])
            done.record(self._post_stream)
        return done

    def _run(self, n, get_raw, masks_host, bgr, bottom_up, exclude_nodes, on_device, want_processed=False, only_preprocess=False,
             spans=None):
        """Software pipeline over chunks of images, with NO host synchronisation inside:
             copy stream : H2D of the raw scans (host path only), ``depth`` staging buffers
             pre stream  : K1 + heights for chunk c+1
             main stream : ragged network for chunk c                post stream: K3 + K5 for chunk c-1
             out stream  : D2H of finished masks, then of the counts and {first,last} rows
        Successive calls are NOT separated by a barrier: the side streams are in order, the two slots protect the
        per-batch buffers, so the copies of batch k+1 overlap the tail of batch k."""
        dev = self.device
        chunk, depth = self.chunk, self.depth
        with torch.cuda.device(dev):
            first = self._streams()
            self._standard_buffers()
            slot = self._slot(n)
            main = torch.cuda.current_stream(dev)
            if first or on_device:
                # inputs made on the caller's stream (device-resident scans) / first use: order the side streams after it
                start = torch.cuda.Event()
                start.record(main)
                for st in (self._copy_stream, self._pre_stream, self._out_stream, self._post_stream):
                    st.wait_event(start)
            if slot.done is not None:
                self._pre_stream.wait_event(slot.done)   # the batch that used this slot two calls ago is fully drained
            chunks = [(a, min(a + chunk, n)) for a in range(0, n, chunk)]
            span_of = None if on_device else self._spans(n, get_raw, spans)
            pitch = self.raw_size * 3
            for (a, b) in chunks:
                ptrs, spans_ab, used = [], [], []
                for i in range(a, b):
                    raw = get_raw(i)
                    if not raw.is_cuda:
                        k = self._issued % depth
                        row0, rows = span_of[i]()
                        with torch.cuda.stream(self._copy_stream):
                            if self._issued >= depth:
                                self._copy_stream.wait_event(self._freed[k])
                            if rows:      # one cudaMemcpyAsync per scan: the rows between the dark bands
                                self._stage[k][:rows * pitch].copy_(raw[row0 * pitch:(row0 + rows) * pitch], non_blocking=True)
                        self.h2d_bytes += rows * pitch
                        ptrs.append(self._stage[k].data_ptr())
                        spans_ab.append((row0, rows))
                        used.append(k)
                        self._issued += 1
                    else:
                        ptrs.append(raw.data_ptr())
                        spans_ab.append((0, self.raw_size))
                if used:
                    self._staged[used[-1]].record(self._copy_stream)      # the copy stream is in order: all of the chunk's copies
                    self._pre_stream.wait_event(self._staged[used[-1]])
                with torch.cuda.stream(self._pre_stream):
                    self._preprocess_chunk(slot, a, b, ptrs, spans_ab, bgr, bottom_up)      # K1 for the whole chunk
                    for k in used:
                        self._freed[k].record(self._pre_stream)
                pre_done = torch.cuda.Event()
                with torch.cuda.stream(self._pre_stream):
                    ops.heights_from_first_last(slot.fl[a:b], out=slot.heights[a:b])
                    pre_done.record(self._pre_stream)
                if want_processed:
                    if slot.proc_host is None:
                        slot.proc_host = torch.empty(slot.proc.shape, dtype=torch.uint8).pin_memory()
                    with torch.cuda.stream(self._out_stream):
                        self._out_stream.wait_event(pre_done)
                        slot.proc_host[a:b].copy_(slot.proc[a:b], non_blocking=True)
                if only_preprocess:
                    continue
                main.wait_event(pre_done)
                ev = self._segment_chunk(slot, a, b, exclude_nodes)
                if masks_host is not None:
                    with torch.cuda.stream(self._out_stream):
                        self._out_stream.wait_event(ev)
                        for i in range(a, b):
                            masks_host[i].copy_(slot.masks[i].view(-1), non_blocking=True)
            with torch.cuda.stream(self._out_stream):
                self._out_stream.wait_stream(self._post_stream)
                self._out_stream.wait_stream(self._pre_stream)
                slot.fl_host[:n].copy_(slot.fl[:n], non_blocking=True)
                slot.counts_host[:n].copy_(slot.counts[:n], non_blocking=True)
                slot.done = torch.cuda.Event()
                slot.done.record(self._out_stream)
            if on_device:
                main.wait_stream(self._post_stream)      # the caller consumes masks / counts on its own stream
            return slot

    # -- device-resident batch ---------------------------------------------------------------------------------------
    def run_device(self, raws, bgr=True, bottom_up=True, exclude_nodes=False):
        """raws: list of u8 CUDA tensors, each a raw_size x raw_size x 3 pixel array already in HBM.  Fully
        asynchronous.  Returns (counts int32 [n,3] CUDA, mask canvas u8 [n, raw/4, raw/4] CUDA, heights int32 [n] CUDA):
        image i's mask is ``masks[i, :heights[i]]``.  The tensors stay valid until the call after next."""
        n = len(raws)
        slot = self._run(n, lambda i: raws[i], None, bgr, bottom_up, exclude_nodes, True)
        return slot.counts[:n], slot.masks[:n], slot.heights[:n]

    # -- end to end from pinned host memory --------------------------------------------------------------------------
    def submit_host(self, raws_host, masks_host=None, bgr=True, bottom_up=True, exclude_nodes=False, want_processed=False,
                    only_preprocess=False, spans=None):
        """Enqueue one batch of pinned u8 CPU tensors (raw pixel arrays) and return a ticket at once; at most two
        tickets may be outstanding.  ``collect`` waits for it.  want_processed: also copy the processed (resized +
        trimmed) images back (``ticket.slot.proc_host[i, :rows[i]]`` after collect); only_preprocess: stop after K1.
        spans: optional list of (row0, rows) per scan from a producer that already knows the zero bands (e.g. the thread
        that read the file); otherwise the engine scans."""
        n = len(raws_host)
        slot = self._run(n, lambda i: raws_host[i], masks_host, bgr, bottom_up, exclude_nodes, False, want_processed,
                         only_preprocess, spans)
        slot.pending = True
        return Ticket(slot, n, masks_host)

    def collect(self, ticket):
        """-> (rows list, counts numpy [n,3], masks_host): waits until the ticket's batch is complete.  When
        ``masks_host`` (pinned u8 tensors of raw/4 * raw/4 bytes) was given every mask canvas has been copied back;
        image i's mask is the first rows[i] * (raw/4) bytes."""
        s, n = ticket.slot, ticket.n
        s.done.synchronize()
        s.pending = False
        fl = s.fl_host[:n]
        return (fl[:, 1] - fl[:, 0]).tolist(), s.counts_host[:n].numpy().copy(), ticket.masks_host

    def run_host(self, raws_host, masks_host=None, bgr=True, bottom_up=True, exclude_nodes=False):
        """Synchronous end-to-end call: submit_host + collect."""
        return self.collect(self.submit_host(raws_host, masks_host, bgr, bottom_up, exclude_nodes))

    # -- heterogeneous raw images from pinned host memory -------------------------------------------------------------
    def reserve_mixed(self, nbytes):
        """Size the staging ring of ``submit_mixed`` for raw images of up to ``nbytes`` bytes (``depth`` buffers).  The
        folder pipeline reserves the largest raw image of its run once, before the first submit; a later, larger image
        reallocates after a device synchronise."""
        if nbytes <= self._mixed_bytes:
            return
        with torch.cuda.device(self.device):
            if self._mixed_stage is not None:
                torch.cuda.synchronize(self.device)
            self._mixed_stage = None
            self._mixed_stage = [torch.empty(nbytes, dtype=torch.uint8, device=self.device) for _ in range(self.depth)]
            self._mixed_staged = [torch.cuda.Event() for _ in range(self.depth)]
            self._mixed_freed = [torch.cuda.Event() for _ in range(self.depth)]
            self._mixed_bytes, self._mixed_issued = nbytes, 0

    def _mixed_chunks(self, widths):
        """Slot order and chunks of a mixed batch: the images processed to the full canvas width first, then the narrower
        ones grouped by width (a ragged pass needs one width).  -> (order: slot position -> caller index, [(a, b, width)])"""
        T = self.out_w
        order = sorted(range(len(widths)), key=lambda i: (widths[i] != T, widths[i]))
        chunks, a = [], 0
        while a < len(order):
            w = widths[order[a]]
            b = a + 1
            while b < len(order) and b - a < self.chunk and widths[order[b]] == w:
                b += 1
            chunks.append((a, b, w))
            a = b
        return order, chunks

    def submit_mixed(self, raws_host, geoms, masks_host=None, exclude_nodes=False, want_processed=False, only_preprocess=False,
                     spans=None):
        """``submit_host`` for raw images of any sizes and layouts.  geoms[i] = (H, W, pitch, bgr, bottom_up) of the pixel
        array in the pinned u8 CPU tensor raws_host[i]; spans[i] = (row0, rows): only those memory rows are copied (a
        (4 * out_w)^2 scan's rows between its all-zero bands, see the module docstring; (0, H) otherwise, the default).
        K1 routes each image as ``Preprocessor.preprocess_array`` does (``nbc_preprocess_mixed_batch_u8``).  Images
        processed to the full width share chunks; narrower ones (images that need no resize) form chunks of one width.
        ``collect_mixed`` waits for the ticket; masks_host[i] (pinned, out_w^2 bytes) receives image i's mask in its
        first rows[i] * widths[i] bytes."""
        n = len(raws_host)
        T = self.out_w
        widths = [ops.processed_size(g[0], g[1], T)[1] for g in geoms]
        spans = [(0, g[0]) for g in geoms] if spans is None else list(spans)
        order, chunks = self._mixed_chunks(widths)
        dev, depth = self.device, self.depth
        Hc = self.raw_size // 4
        lib = ops._lib.load()
        self.reserve_mixed(max(rows * g[2] for g, (_, rows) in zip(geoms, spans)))
        with torch.cuda.device(dev):
            first = self._streams()
            if getattr(self, '_mixed_ws', None) is None:
                self._mixed_ws = torch.empty(lib.nbc_preprocess_mixed_workspace_bytes(None, self.chunk, T), dtype=torch.uint8,
                                             device=dev)
            slot = self._slot(n)
            main = torch.cuda.current_stream(dev)
            if first:
                start = torch.cuda.Event()
                start.record(main)
                for st in (self._copy_stream, self._pre_stream, self._out_stream, self._post_stream):
                    st.wait_event(start)
            if slot.done is not None:
                self._pre_stream.wait_event(slot.done)
            if want_processed and slot.proc_host is None:
                slot.proc_host = torch.empty(slot.proc.shape, dtype=torch.uint8).pin_memory()
            proc_flat, masks_flat = slot.proc.view(-1), slot.masks.view(-1)
            views = []        # per chunk: (proc canvas, mask canvas, flat byte offset of the proc canvas)
            for (a, b, w) in chunks:
                off = a * Hc * T * 3
                proc = proc_flat[off:off + (b - a) * Hc * w * 3].view(b - a, Hc, w, 3)
                masks = masks_flat[a * Hc * T:a * Hc * T + (b - a) * Hc * w].view(b - a, Hc, w)
                views.append((proc, masks, off))
                items, used = [], []
                for p in range(a, b):
                    i = order[p]
                    H, W, pitch, bgr, bottom_up = geoms[i]
                    row0, rows = spans[i]
                    k = self._mixed_issued % depth
                    with torch.cuda.stream(self._copy_stream):
                        if self._mixed_issued >= depth:
                            self._copy_stream.wait_event(self._mixed_freed[k])
                        if rows:      # one cudaMemcpyAsync per image
                            self._mixed_stage[k][:rows * pitch].copy_(raws_host[i][row0 * pitch:(row0 + rows) * pitch],
                                                                      non_blocking=True)
                    self.h2d_bytes += rows * pitch
                    items.append((self._mixed_stage[k].data_ptr() if rows else None, H, W, pitch, bgr, bottom_up, (row0, rows)))
                    used.append(k)
                    self._mixed_issued += 1
                self._mixed_staged[used[-1]].record(self._copy_stream)
                self._pre_stream.wait_event(self._mixed_staged[used[-1]])
                descs = ops.mixed_descs(items)
                pre_done = torch.cuda.Event()
                with torch.cuda.stream(self._pre_stream):
                    ops._lib.check(lib.nbc_preprocess_mixed_batch_u8(descs, b - a, T, C.c_void_p(proc.data_ptr()), Hc * w * 3,
                                                                     C.c_void_p(slot.fl[a].data_ptr()), C.c_void_p(self._mixed_ws.data_ptr()),
                                                                     self._mixed_ws.numel(),
                                                                     C.c_void_p(self._pre_stream.cuda_stream)),
                                   'nbc_preprocess_mixed_batch_u8')
                    for k in used:
                        self._mixed_freed[k].record(self._pre_stream)
                    ops.heights_from_first_last(slot.fl[a:b], out=slot.heights[a:b])
                    pre_done.record(self._pre_stream)
                if want_processed:
                    with torch.cuda.stream(self._out_stream):
                        self._out_stream.wait_event(pre_done)
                        slot.proc_host.view(-1)[off:off + proc.numel()].copy_(proc.view(-1), non_blocking=True)
                if only_preprocess:
                    continue
                main.wait_event(pre_done)
                ev = self._segment_chunk(slot, a, b, exclude_nodes, proc=proc, masks=masks)
                if masks_host is not None:
                    with torch.cuda.stream(self._out_stream):
                        self._out_stream.wait_event(ev)
                        for p in range(a, b):
                            masks_host[order[p]][:Hc * w].copy_(masks[p - a].view(-1), non_blocking=True)
            with torch.cuda.stream(self._out_stream):
                self._out_stream.wait_stream(self._post_stream)
                self._out_stream.wait_stream(self._pre_stream)
                slot.fl_host[:n].copy_(slot.fl[:n], non_blocking=True)
                slot.counts_host[:n].copy_(slot.counts[:n], non_blocking=True)
                slot.done = torch.cuda.Event()
                slot.done.record(self._out_stream)
        slot.pending = True
        ticket = Ticket(slot, n, masks_host)
        ticket.order, ticket.widths = order, widths
        ticket.proc_offsets = [0] * n       # caller index -> flat byte offset of its processed image in slot.proc_host
        for (a, b, w), (_, _, off) in zip(chunks, views):
            for p in range(a, b):
                ticket.proc_offsets[order[p]] = off + (p - a) * Hc * w * 3
        return ticket

    def collect_mixed(self, ticket):
        """-> (rows, widths, counts numpy [n,3], masks_host) in the caller's order; image i's processed image is
        ``processed(ticket, i, rows[i])``."""
        rows, counts, masks_host = self.collect(ticket)
        n = ticket.n
        rows_c, counts_c = [0] * n, counts.copy()
        for p, i in enumerate(ticket.order):
            rows_c[i] = rows[p]
            counts_c[i] = counts[p]
        return rows_c, list(ticket.widths), counts_c, masks_host

    @staticmethod
    def processed(ticket, i, rows):
        """Image i of a collected ``submit_mixed(want_processed=True)`` ticket: a u8 view [rows, width, 3] of pinned memory."""
        w, off = ticket.widths[i], ticket.proc_offsets[i]
        return ticket.slot.proc_host.view(-1)[off:off + rows * w * 3].view(rows, w, 3)
