"""Training step of the reference's ``__main__.py:231-269`` on the B200 path (row a14).

``Trainer`` owns the flat parameter / gradient / Adam buffers (torch tensors = device memory only) and drives the native
step in ``libnbc.so``: train-mode forward (batch-statistics BatchNorm, Dropout(0.8) in the head as
``fcn_resnet50(dropout=0.8)``), ``CustomWeightedCrossEntropy`` (utils.py:151-165), full backward, and Adam
(lr 5e-4, L2 weight decay 2e-3 as ``__main__.py:234``).  Data parallel: one process per GPU, the flat gradient buffer is
all-reduced over NCCL (``torch.distributed``) between backward and the optimiser -- the only collective of the path.
Two modes: ONE all-reduce after the backward (the default: 132 MB over NVLink 5 / NVSwitch takes about half a
millisecond of a 47 ms step), or BUCKETS that start while the backward is still running (``bucket_mb > 0`` /
``NBC_TRAIN_BUCKETS=1``): the native backward records an event each time a segment of the gradient buffer (head, then
the bottleneck blocks last to first, then the stem) is final, consecutive segments are merged into buckets of
>= ``bucket_mb`` and each bucket's all-reduce is enqueued on a side stream behind its event; Adam waits for all of them.
Measured on 8 B200 (profiles/r02c_bench_train_g8*.json): 1 336 img/s with the single all-reduce (97.4 % of 8 x one GPU),
1 318 with 7 overlapped buckets -- an NCCL kernel that starts in the middle of the backward takes SMs away from the
persistent convolution kernels, which need all 148, and that costs more than the exposed half millisecond; hence the
default.  No torch autograd, no torch ops on the data path."""
import ctypes as C
import os

import torch

from . import _lib, ops
from .utils import get_pos_weight


def gradient_segments(lib, handle):
    """[(offset, count)] of the flat gradient buffer in the order the native backward finishes them (head + classifier, the
    bottleneck blocks last to first, the stem); needs no GPU."""
    h = C.c_void_p(handle)
    out = []
    for i in range(lib.nbc_train_num_segments(h)):
        off, cnt = C.c_int64(0), C.c_int64(0)
        _lib.check(lib.nbc_train_segment(h, i, C.byref(off), C.byref(cnt)), 'nbc_train_segment')
        out.append((off.value, cnt.value))
    return out


def merge_segments(segments, min_bytes):
    """Consecutive segments (contiguous in memory, descending) merged until a bucket holds at least ``min_bytes`` of f32
    gradients -> [(index of the bucket's last segment, offset, count)]."""
    out, lo, hi = [], None, None
    for i, (off, cnt) in enumerate(segments):
        a, b = off, off + cnt
        if hi is not None and b != lo:
            raise RuntimeError('gradient segments must be contiguous, last layer first')
        lo, hi = a, (b if hi is None else hi)
        if (hi - lo) * 4 >= min_bytes or i == len(segments) - 1:
            out.append((i, lo, hi - lo))
            hi = None
    return out


class Trainer:
    def __init__(self, state_dict, N, H, W, device='cuda:0', lr=5e-4, weight_decay=2e-3, betas=(0.9, 0.999), eps=1e-8,
                 dropout=0.8, class_weights=None, mean=(0.7399, 0.6139, 0.4401), std=(0.1068, 0.1272, 0.1271),
                 loss='weighted_ce', bucket_mb=0.0, seed=0):
        self.lib = _lib.load()
        self.device = torch.device(device)
        _lib.require_device(self.device.index if self.device.index is not None else torch.cuda.current_device())
        self.N, self.H, self.W = N, H, W
        self.lr, self.wd, self.betas, self.eps, self.dropout = lr, weight_decay, betas, eps, dropout
        self.mean3 = (C.c_float * 3)(*mean)
        self.std3 = (C.c_float * 3)(*std)
        self.step_count = 0
        self.base_seed = int(seed)
        env = os.environ.get('NBC_TRAIN_BUCKETS')
        if env is not None and env != '':      # 0: single all-reduce; 1: 16 MB buckets; any other number: that many MB
            bucket_mb = 0.0 if env == '0' else (16.0 if env == '1' else float(env))
        self.bucket_mb = float(bucket_mb)
        self._buckets = None
        self._comm_stream = None
        self.keys = list(state_dict.keys())
        if len(self.keys) != 326:
            raise RuntimeError('Trainer expects the 326-key fcn_resnet50 state_dict')
        with torch.cuda.device(self.device):
            self.handle = self.lib.nbc_train_create(N, H, W)
            if not self.handle:
                raise RuntimeError('nbc_train_create failed: ' + _lib.last_error())
            h = C.c_void_p(self.handle)
            kinds = {'weighted_ce': 0, 'lovasz': 1, 'mixed': 2}   # utils.py:151-165 / __main__.py:239 / utils.py:185-192
            if loss not in kinds:
                raise ValueError("loss must be 'weighted_ce', 'lovasz' or 'mixed'")
            _lib.check(self.lib.nbc_train_set_loss(h, kinds[loss]), 'nbc_train_set_loss')
            self.loss_kind = loss
            n = self.lib.nbc_train_param_count(h)
            self.params = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.grads = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.adam_m = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.adam_v = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.stats = torch.zeros(self.lib.nbc_train_stats_count(h), dtype=torch.float32, device=self.device)
            self.ws = torch.empty(self.lib.nbc_train_workspace_bytes(h) + 1024, dtype=torch.uint8, device=self.device)
            self.loss = torch.zeros((), dtype=torch.float32, device=self.device)
            w = get_pos_weight() if class_weights is None else class_weights
            self.class_weights = w.to(device=self.device, dtype=torch.float32).contiguous()
            self._exchange(self._device_tensors(state_dict), self.params, self.stats, 0)
        self.num_batches_tracked = {k: int(v) for k, v in state_dict.items() if k.endswith('num_batches_tracked')}
        self.capture = None

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                self.lib.nbc_train_destroy(C.c_void_p(self.handle))
                self.handle = None
        except Exception:
            pass

    # -- state_dict <-> flat buffers ---------------------------------------------------------------------------------
    def _device_tensors(self, sd):
        out = []
        for k in self.keys:
            t = sd[k]
            if t.dtype == torch.int64:
                out.append(t.to(self.device))
            else:
                out.append(t.detach().to(device=self.device, dtype=torch.float32).contiguous())
        return out

    def _exchange(self, tensors, flat, stats, direction):
        arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
        _lib.check(self.lib.nbc_train_exchange(C.c_void_p(self.handle), arr, len(tensors), C.c_void_p(flat.data_ptr()),
                                               C.c_void_p(stats.data_ptr()) if stats is not None else C.c_void_p(0), direction,
                                               C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                   'nbc_train_exchange')
        torch.cuda.current_stream(self.device).synchronize()
        return tensors

    def _template(self):
        import neuralbarkcalculator_b200 as nbc
        sd = nbc.fcn_resnet50(pretrained=False).state_dict()
        return {k: torch.zeros_like(v, device=self.device) for k, v in sd.items()}

    def state_dict(self):
        """Current weights (and BatchNorm running statistics) as a 326-key torchvision-layout state_dict."""
        with torch.cuda.device(self.device):
            sd = self._template()
            self._exchange([sd[k] for k in self.keys], self.params, self.stats, 1)
        for k in sd:
            if k.endswith('num_batches_tracked'):
                sd[k].fill_(self.num_batches_tracked.get(k, 0))
        return sd

    def gradients(self):
        """Gradients of the last forward_backward in state_dict layout (OIHW conv weights; BN weight / bias; classifier)."""
        with torch.cuda.device(self.device):
            sd = self._template()
            self._exchange([sd[k] for k in self.keys], self.grads, None, 1)
        return {k: v for k, v in sd.items() if 'running' not in k and 'num_batches' not in k}

    def enable_capture(self):
        """Make every following step keep the dy and dz of each unit's BatchNorm backward (tests; ``debug_tensor`` 6 / 7)."""
        with torch.cuda.device(self.device):
            h = C.c_void_p(self.handle)
            self.capture = torch.empty(self.lib.nbc_train_capture_bytes(h), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.nbc_train_set_capture(h, C.c_void_p(self.capture.data_ptr()), self.capture.numel()),
                       'nbc_train_set_capture')

    def debug_tensor(self, what, index=0):
        """View of an intermediate of the last step (tests): what 0/1 = z / y of unit ``index`` (bf16 NHWC), 2/3 = low / full
        resolution logits, 4/5 = their gradients (f32 [N,3,h,w]), 6/7 = dy / dz of the unit's BatchNorm backward (bf16 NHWC,
        after ``enable_capture``)."""
        if what in (6, 7) and self.capture is None:
            raise RuntimeError('debug tensors 6 / 7 need enable_capture()')
        dims = (C.c_int32 * 4)()
        off = self.lib.nbc_train_debug_offset(C.c_void_p(self.handle), what, index, dims)
        if off < 0:
            raise RuntimeError('bad debug tensor request')
        buf, base = (self.capture, off) if what in (6, 7) else (self.ws, (-self.ws.data_ptr()) % 1024 + off)
        n, h, w, c = [int(v) for v in dims]
        if what in (0, 1, 6, 7):
            return buf[base:base + n * h * w * c * 2].view(torch.bfloat16).view(n, h, w, c)
        return buf[base:base + n * h * w * c * 4].view(torch.float32).view(n, c, h, w)

    def evaluate(self, ds, indices, loss=None, class_weights=None, precision=None, chunk=8):
        """``evaluate.evaluate`` of the current weights: eval-mode forward of whole images, as predict runs them, with
        this trainer's loss and class weights unless given."""
        from . import evaluate as nev
        from .models import DEFAULT_PRECISION
        return nev.evaluate(self.state_dict(), ds, indices, loss=self.loss_kind if loss is None else loss,
                            class_weights=self.class_weights if class_weights is None else class_weights,
                            precision=DEFAULT_PRECISION if precision is None else precision, chunk=chunk)

    # -- the step ------------------------------------------------------------------------------------------------------
    def forward_backward(self, images, targets, seed=0, dropout=None, update_stats=True):
        """images: u8 NHWC [N,H,W,3] (normalised inside) or f32 NCHW [N,3,H,W]; targets: u8 [N,H,W].
        Returns the loss (0-dim CUDA tensor); gradients are left in ``self.grads``."""
        p = self.dropout if dropout is None else dropout
        if images.dtype == torch.uint8:
            kind, shape = 0, (self.N, self.H, self.W, 3)
        elif images.dtype == torch.float32:
            kind, shape = 1, (self.N, 3, self.H, self.W)
        else:
            raise RuntimeError('images must be u8 NHWC or f32 NCHW')
        if not images.is_cuda or tuple(images.shape) != shape:
            raise RuntimeError('images must be a CUDA tensor of shape %s' % (shape,))
        if not targets.is_cuda or targets.dtype != torch.uint8 or tuple(targets.shape) != (self.N, self.H, self.W):
            raise RuntimeError('targets must be a CUDA u8 tensor [N,H,W]')
        images, targets = images.contiguous(), targets.contiguous()
        with torch.cuda.device(self.device):
            off = (-self.ws.data_ptr()) % 1024
            _lib.check(self.lib.nbc_train_forward_backward(
                C.c_void_p(self.handle), C.c_void_p(self.params.data_ptr()),
                C.c_void_p(self.stats.data_ptr()) if update_stats else C.c_void_p(0), C.c_void_p(self.grads.data_ptr()),
                C.c_void_p(images.data_ptr()), kind, self.mean3, self.std3, C.c_void_p(targets.data_ptr()),
                C.c_void_p(self.class_weights.data_ptr()), C.c_float(p), C.c_uint64(seed), C.c_void_p(self.loss.data_ptr()),
                C.c_void_p(self.ws.data_ptr() + off), C.c_size_t(self.ws.numel() - off),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), 'nbc_train_forward_backward')
        if update_stats:
            for k in self.num_batches_tracked:
                self.num_batches_tracked[k] += 1
        return self.loss

    def gradient_buckets(self):
        """[(last segment of the bucket, offset, count)] in the order the backward completes them: consecutive gradient
        segments (``nbc_train_segment``) merged until a bucket holds at least ``bucket_mb`` MB."""
        if self._buckets is None:
            self._buckets = merge_segments(gradient_segments(self.lib, self.handle), self.bucket_mb * 1e6)
            assert sum(c for _, _, c in self._buckets) == self.grads.numel()
        return self._buckets

    def all_reduce_gradients(self):
        """SUM the gradients over the data-parallel group (Adam applies 1/world).  Bucketed: every bucket's all-reduce is
        enqueued on a side stream behind the event the backward records when that part of the buffer is final, so the
        exchange of the last layers runs under the backward of the first ones.  Returns the number of collectives."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if world == 1:
            return 0
        if self.bucket_mb <= 0:
            dist.all_reduce(self.grads, op=dist.ReduceOp.SUM)
            return 1
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(self.device)
        works = []
        with torch.cuda.device(self.device):
            for seg, off, cnt in self.gradient_buckets():
                _lib.check(self.lib.nbc_train_wait_segment(C.c_void_p(self.handle), seg, C.c_void_p(self._comm_stream.cuda_stream)),
                           'nbc_train_wait_segment')
                with torch.cuda.stream(self._comm_stream):
                    works.append(dist.all_reduce(self.grads[off:off + cnt], op=dist.ReduceOp.SUM, async_op=True))
            for w in works:
                w.wait()          # the current stream (Adam's) waits for the collective; the host does not block
        return len(works)

    def optimizer_step(self):
        """All-reduce the gradients over the data-parallel group (if any), then one fused Adam pass."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.all_reduce_gradients()
        self.step_count += 1
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nbc_train_adam(C.c_void_p(self.params.data_ptr()), C.c_void_p(self.grads.data_ptr()),
                                               C.c_void_p(self.adam_m.data_ptr()), C.c_void_p(self.adam_v.data_ptr()),
                                               self.params.numel(), C.c_float(self.lr), C.c_float(self.betas[0]),
                                               C.c_float(self.betas[1]), C.c_float(self.eps), C.c_float(self.wd), self.step_count,
                                               C.c_float(1.0 / world),
                                               C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), 'nbc_train_adam')

    def dropout_seed(self):
        """A different dropout mask per step, per data-parallel rank and per run seed (every rank drawing the same mask
        would correlate the replicas' gradients)."""
        import torch.distributed as dist
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        return (self.base_seed << 40) + (rank << 28) + self.step_count

    def step(self, images, targets, seed=None):
        loss = self.forward_backward(images, targets, seed=self.dropout_seed() if seed is None else seed)
        self.optimizer_step()
        return loss
