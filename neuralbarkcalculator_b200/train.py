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
default.  Gradient accumulation: ``forward_backward(..., accumulate=True)`` adds a micro-batch's gradients to the
buffer, so a global batch of ``world * k`` micro-batches costs k backward passes per rank and ONE exchange; Adam then
applies 1 / (world * k).  Fine-tuning: ``freeze='stem'|'layer1'|..|'layer4'`` freezes the stem through that stage
(``nbc_train_set_frozen``): those units run as eval-mode BatchNorm folded into their convolutions (torchvision's
FrozenBatchNorm2d), their parameters, running statistics and ``num_batches_tracked`` never change, and the backward,
the gradient exchange and Adam cover only the trainable suffix of the flat buffers.  No torch autograd, no torch ops on
the data path."""
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


FREEZE = ('none', 'stem', 'layer1', 'layer2', 'layer3', 'layer4')    # index = nbc_train_set_frozen's stages


def frozen_prefixes(freeze):
    """state_dict key prefixes of the units ``freeze`` freezes (the stem, then whole layers)."""
    stages = FREEZE.index(freeze)
    return tuple((['backbone.conv1.', 'backbone.bn1.'] if stages else []) + ['backbone.layer%d.' % i for i in range(1, stages)])


def dropout_seed(base_seed, micro_batch, step):
    """Dropout seed of global micro-batch ``micro_batch`` of optimizer step ``step``: micro-batch i of rank r, with k
    micro-batches per rank, is j = r * k + i, so a global micro-batch draws the same mask whatever (world, k) runs it
    (with k = 1, j is the rank)."""
    return (int(base_seed) << 40) + (int(micro_batch) << 28) + int(step)


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
                 loss='weighted_ce', bucket_mb=0.0, seed=0, freeze='none'):
        self.lib = _lib.load()
        self.device = torch.device(device)
        _lib.require_device(self.device.index if self.device.index is not None else torch.cuda.current_device())
        self.N, self.H, self.W = N, H, W
        self.lr, self.wd, self.betas, self.eps, self.dropout = lr, weight_decay, betas, eps, dropout
        self.mean3 = (C.c_float * 3)(*mean)
        self.std3 = (C.c_float * 3)(*std)
        self.step_count = 0
        self.base_seed = int(seed)
        self.micro_batches = 0          # forward_backward calls summed in self.grads since the last optimizer_step
        self._accumulating = False      # the plan's nbc_train_set_accumulate state
        env = os.environ.get('NBC_TRAIN_BUCKETS')
        if env is not None and env != '':      # 0: single all-reduce; 1: 16 MB buckets; any other number: that many MB
            bucket_mb = 0.0 if env == '0' else (16.0 if env == '1' else float(env))
        self.bucket_mb = float(bucket_mb)
        self._buckets = None
        self._comm_stream = None
        self.keys = list(state_dict.keys())
        if len(self.keys) != 326:
            raise RuntimeError('Trainer expects the 326-key fcn_resnet50 state_dict')
        if freeze not in FREEZE:
            raise ValueError('freeze must be one of %s' % ', '.join(FREEZE))
        self.freeze = freeze
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
            _lib.check(self.lib.nbc_train_set_frozen(h, FREEZE.index(freeze)), 'nbc_train_set_frozen')
            poff, soff = C.c_int64(0), C.c_int64(0)
            _lib.check(self.lib.nbc_train_trainable_offsets(h, C.byref(poff), C.byref(soff)), 'nbc_train_trainable_offsets')
            self.param_off, self.stats_off = poff.value, soff.value     # first trainable float of params / stats
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
        frozen = frozen_prefixes(freeze)
        self._counted = [k for k in self.num_batches_tracked if not k.startswith(frozen)]   # frozen BNs do not count
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

    def _moments(self, flat):
        """An Adam moment buffer in state_dict layout (a pure permutation of the flat buffer: bit-exact both ways)."""
        with torch.cuda.device(self.device):
            sd = self._template()
            self._exchange([sd[k] for k in self.keys], flat, None, 1)
        return {k: v for k, v in sd.items() if 'running' not in k and 'num_batches' not in k}

    def training_state(self):
        """Everything the next optimizer steps depend on, in state_dict layout (independent of the plan's internal
        buffer layout): ``model`` (the 326-key state_dict), ``adam_m`` / ``adam_v`` (per parameter key; a frozen unit's
        moments are zero), ``step_count``, ``lr`` and ``num_batches_tracked``.  Tensors are on the CPU."""
        if self.micro_batches:
            raise RuntimeError('training_state: %d micro-batches are accumulated but not applied; take it after '
                               'optimizer_step' % self.micro_batches)
        cpu = lambda d: {k: v.cpu() for k, v in d.items()}
        return {'model': cpu(self.state_dict()), 'adam_m': cpu(self._moments(self.adam_m)),
                'adam_v': cpu(self._moments(self.adam_v)), 'step_count': int(self.step_count), 'lr': float(self.lr),
                'num_batches_tracked': dict(self.num_batches_tracked)}

    def load_training_state(self, state):
        """Restore ``training_state()``: afterwards ``params``, ``stats``, ``adam_m`` and ``adam_v`` are bit-identical to
        the trainer that produced it, and so are the following steps (same inputs, same seeds)."""
        if sorted(state['model']) != sorted(self.keys):
            raise RuntimeError('load_training_state: the model is not the 326-key fcn_resnet50 state_dict')
        moment_keys = [k for k in self.keys if 'running' not in k and 'num_batches' not in k]
        for name in ('adam_m', 'adam_v'):
            if sorted(state[name]) != sorted(moment_keys):
                raise RuntimeError('load_training_state: %s does not hold the %d parameter keys' % (name, len(moment_keys)))
        with torch.cuda.device(self.device):
            self._exchange(self._device_tensors(state['model']), self.params, self.stats, 0)
            for name, flat in (('adam_m', self.adam_m), ('adam_v', self.adam_v)):
                sd = dict(state['model'])
                sd.update(state[name])
                flat.zero_()
                self._exchange(self._device_tensors(sd), flat, None, 0)
                flat[:self.param_off].zero_()      # frozen units carry no moments
        self.step_count = int(state['step_count'])
        self.lr = float(state['lr'])
        self.num_batches_tracked = {k: int(v) for k, v in state['num_batches_tracked'].items()}
        self.micro_batches = 0

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
    def forward_backward(self, images, targets, seed=0, dropout=None, update_stats=True, accumulate=False):
        """images: u8 NHWC [N,H,W,3] (normalised inside) or f32 NCHW [N,3,H,W]; targets: u8 [N,H,W].
        Returns the loss (0-dim CUDA tensor); gradients are left in ``self.grads``: overwritten, or with ``accumulate``
        added to what the buffer holds (the first micro-batch of a step overwrites, the next ones accumulate; the next
        ``optimizer_step`` divides by the number of micro-batches summed).  ``update_stats=False`` leaves the running
        statistics as they are (frozen units still read theirs)."""
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
        accumulate = bool(accumulate)
        with torch.cuda.device(self.device):
            if accumulate != self._accumulating:
                _lib.check(self.lib.nbc_train_set_accumulate(C.c_void_p(self.handle), int(accumulate)), 'nbc_train_set_accumulate')
                self._accumulating = accumulate
            off = (-self.ws.data_ptr()) % 1024
            stats = self.stats if update_stats else (self.stats.clone() if self.stats_off else None)
            _lib.check(self.lib.nbc_train_forward_backward(
                C.c_void_p(self.handle), C.c_void_p(self.params.data_ptr()),
                C.c_void_p(stats.data_ptr() if stats is not None else 0), C.c_void_p(self.grads.data_ptr()),
                C.c_void_p(images.data_ptr()), kind, self.mean3, self.std3, C.c_void_p(targets.data_ptr()),
                C.c_void_p(self.class_weights.data_ptr()), C.c_float(p), C.c_uint64(seed), C.c_void_p(self.loss.data_ptr()),
                C.c_void_p(self.ws.data_ptr() + off), C.c_size_t(self.ws.numel() - off),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), 'nbc_train_forward_backward')
        self.micro_batches = self.micro_batches + 1 if accumulate else 1
        if update_stats:
            for k in self._counted:
                self.num_batches_tracked[k] += 1
        return self.loss

    def gradient_buckets(self):
        """[(last segment of the bucket, offset, count)] in the order the backward completes them: consecutive gradient
        segments (``nbc_train_segment``) merged until a bucket holds at least ``bucket_mb`` MB.  The empty segments of
        frozen units come last, so dropping them keeps every other segment's index."""
        if self._buckets is None:
            segments = gradient_segments(self.lib, self.handle)
            trainable = [s for s in segments if s[1] > 0]
            assert segments[:len(trainable)] == trainable
            self._buckets = merge_segments(trainable, self.bucket_mb * 1e6)
            assert sum(c for _, _, c in self._buckets) == self.grads.numel() - self.param_off
        return self._buckets

    def all_reduce_gradients(self):
        """SUM the gradients over the data-parallel group (Adam applies 1 / (world * micro-batches)).  Bucketed: every bucket's all-reduce is
        enqueued on a side stream behind the event the backward records when that part of the buffer is final, so the
        exchange of the last layers runs under the backward of the first ones.  Returns the number of collectives."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if world == 1:
            return 0
        if self.bucket_mb <= 0:
            dist.all_reduce(self.grads[self.param_off:], op=dist.ReduceOp.SUM)
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
        """All-reduce the gradients over the data-parallel group (if any), then one fused Adam pass on their mean over
        the world's micro-batches since the last step, over the trainable suffix only (weight decay never touches a
        frozen weight)."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        micro = max(self.micro_batches, 1)
        self.all_reduce_gradients()
        self.step_count += 1
        self.micro_batches = 0
        o = self.param_off * 4      # bytes
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nbc_train_adam(C.c_void_p(self.params.data_ptr() + o), C.c_void_p(self.grads.data_ptr() + o),
                                               C.c_void_p(self.adam_m.data_ptr() + o), C.c_void_p(self.adam_v.data_ptr() + o),
                                               self.params.numel() - self.param_off, C.c_float(self.lr), C.c_float(self.betas[0]),
                                               C.c_float(self.betas[1]), C.c_float(self.eps), C.c_float(self.wd), self.step_count,
                                               C.c_float(1.0 / (world * micro)),
                                               C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), 'nbc_train_adam')

    def dropout_seed(self, micro_batch=None):
        """A different dropout mask per step, per global micro-batch and per run seed (every rank drawing the same mask
        would correlate the replicas' gradients).  ``micro_batch`` defaults to the rank (one micro-batch per rank)."""
        if micro_batch is None:
            import torch.distributed as dist
            micro_batch = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        return dropout_seed(self.base_seed, micro_batch, self.step_count)

    def step(self, images, targets, seed=None):
        loss = self.forward_backward(images, targets, seed=self.dropout_seed() if seed is None else seed)
        self.optimizer_step()
        return loss
