"""Tensor-level wrappers over the C-ABI (include/nbc.h).  torch is used for device memory and streams only:
every function checks that its tensors are CUDA tensors on a B200 and raises otherwise -- no CPU fallback."""
import ctypes as C

import torch

from . import _lib


def _stream(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _dev(t, name='tensor'):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError('%s must be a CUDA tensor: neuralbarkcalculator_b200 has no CPU path' % name)
    _lib.require_device(t.device.index if t.device.index is not None else torch.cuda.current_device())
    return t


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _contig(t, dtype, name):
    _dev(t, name)
    if t.dtype != dtype:
        raise RuntimeError('%s must be %s (got %s)' % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


HALF_DTYPES = {'bf16': torch.bfloat16, 'fp16': torch.float16}


def _half(t, name):
    """16-bit activation tensor: bf16 or fp16.  Returns (contiguous tensor, f16 flag)."""
    _dev(t, name)
    if t.dtype not in (torch.bfloat16, torch.float16):
        raise RuntimeError('%s must be bfloat16 or float16 (got %s)' % (name, t.dtype))
    return (t if t.is_contiguous() else t.contiguous()), (1 if t.dtype == torch.float16 else 0)


# ---- K1 -------------------------------------------------------------------------------------------------------
def host_zero_row_span(raw_host, H, pitch, row_bytes=None, group=4):
    """(row0, rows) of a HOST pixel array (u8 CPU tensor or numpy array, H rows of ``pitch`` bytes): the memory rows between
    its all-zero bands, widened outwards to whole groups of ``group`` rows; rows = 0 for an all-zero image.  Host code in
    the library (no GPU); ctypes releases the GIL."""
    lib = _lib.load()
    ptr = raw_host.data_ptr() if hasattr(raw_host, 'data_ptr') else raw_host.ctypes.data
    r0, rows = C.c_int32(0), C.c_int32(0)
    _lib.check(lib.nbc_host_zero_row_span(C.c_void_p(ptr), H, pitch, pitch if row_bytes is None else row_bytes, group,
                                          C.byref(r0), C.byref(rows)), 'nbc_host_zero_row_span')
    return r0.value, rows.value


def preprocess_4x(raw, H, W, pitch=None, bgr=False, bottom_up=False, workspace=None, span=None):
    """raw: u8 CUDA tensor holding an H x W x 3 pixel array (row pitch ``pitch`` bytes).
    Returns (out u8 [(H/4)*(W/4)*3] flat buffer, first_last int32[2] CUDA tensor).
    The trimmed image is ``out[:(last-first)*(W/4)*3].view(last-first, W/4, 3)``.  (models.py:191-203)
    span = (row0, rows): ``raw`` holds only those memory rows (multiples of 4); the other rows of the H x W image are all
    zero and never read (see ``host_zero_row_span``) -- same bytes out as for the full image."""
    lib = _lib.load()
    raw = _contig(raw, torch.uint8, 'raw')
    pitch = W * 3 if pitch is None else pitch
    if span is not None:
        with torch.cuda.device(raw.device):
            need = lib.nbc_preprocess_workspace_bytes(H, W)
            if workspace is None or workspace.numel() < need:
                workspace = torch.empty(need, dtype=torch.uint8, device=raw.device)
            out = torch.empty((H // 4) * (W // 4) * 3, dtype=torch.uint8, device=raw.device)
            fl = torch.empty(2, dtype=torch.int32, device=raw.device)
            if raw.numel() < span[1] * pitch - (pitch - W * 3):
                raise RuntimeError('preprocess_4x: the span buffer holds fewer than %d rows' % span[1])
            _lib.check(lib.nbc_preprocess_4x_span_u8(_ptr(raw) if span[1] else None, H, W, pitch,
                                                     (1 if bgr else 0) | (2 if bottom_up else 0), span[0], span[1], _ptr(out),
                                                     _ptr(fl), _ptr(workspace), workspace.numel(), _stream(raw.device)),
                       'nbc_preprocess_4x_span_u8')
        return out, fl
    with torch.cuda.device(raw.device):
        need = lib.nbc_preprocess_workspace_bytes(H, W)
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=raw.device)
        out = torch.empty((H // 4) * (W // 4) * 3, dtype=torch.uint8, device=raw.device)
        fl = torch.empty(2, dtype=torch.int32, device=raw.device)
        _lib.check(lib.nbc_preprocess_4x_u8(_ptr(raw), H, W, pitch, (1 if bgr else 0) | (2 if bottom_up else 0), _ptr(out),
                                            _ptr(fl), _ptr(workspace), workspace.numel(), _stream(raw.device)),
                   'nbc_preprocess_4x_u8')
    return out, fl


def preprocess_4x_batch(raws, H, W, spans=None, pitch=None, bgr=False, bottom_up=False):
    """K1 for a chunk of scans of one size in three launches (nbc_preprocess_4x_batch_u8).  raws: list of u8 CUDA tensors
    (whole pixel arrays, or only the rows of ``spans[i] = (row0, rows)``).  Returns (canvas u8 [n, H/4, W/4, 3] -- image i in
    rows [0, last_i - first_i) --, first_last int32 [n, 2])."""
    lib = _lib.load()
    n = len(raws)
    raws = [_contig(r, torch.uint8, 'raw') for r in raws]
    dev = raws[0].device
    pitch = W * 3 if pitch is None else pitch
    spans = [(0, H)] * n if spans is None else list(spans)
    with torch.cuda.device(dev):
        ws = torch.empty(n * lib.nbc_preprocess_workspace_bytes(H, W), dtype=torch.uint8, device=dev)
        out = torch.empty((n, H // 4, W // 4, 3), dtype=torch.uint8, device=dev)
        fl = torch.empty((n, 2), dtype=torch.int32, device=dev)
        arr = (C.c_void_p * n)(*[r.data_ptr() if r.numel() else None for r in raws])
        r0 = (C.c_int32 * n)(*[s[0] for s in spans])
        rows = (C.c_int32 * n)(*[s[1] for s in spans])
        _lib.check(lib.nbc_preprocess_4x_batch_u8(arr, r0, rows, n, H, W, pitch, (1 if bgr else 0) | (2 if bottom_up else 0), _ptr(out),
                                                  out.stride(0), _ptr(fl), _ptr(ws), ws.numel(), _stream(dev)),
                   'nbc_preprocess_4x_batch_u8')
    return out, fl


def preprocess_general(raw, H, W, target=1024, pitch=None, bgr=False, bottom_up=False):
    """General-ratio variant of ``preprocess_4x``: any H x W pixel array -> target x target cubic resize + trim
    (models.py:194-203).  Returns (out u8 [target*target*3] flat buffer, first_last int32[2] CUDA tensor); the trimmed
    image is ``out[:(last-first)*target*3].view(last-first, target, 3)``.  Byte-exact against oracle/preprocess.py::resize_general_f64
    on B200 (tests/test_gpu_kernels.py::test_preprocess_general_ratio)."""
    lib = _lib.load()
    raw = _contig(raw, torch.uint8, 'raw')
    pitch = W * 3 if pitch is None else pitch
    with torch.cuda.device(raw.device):
        ws = torch.empty(lib.nbc_preprocess_general_workspace_bytes(H, W, target), dtype=torch.uint8, device=raw.device)
        out = torch.empty(target * target * 3, dtype=torch.uint8, device=raw.device)
        fl = torch.empty(2, dtype=torch.int32, device=raw.device)
        _lib.check(lib.nbc_preprocess_general_u8(_ptr(raw), H, W, pitch, (1 if bgr else 0) | (2 if bottom_up else 0), target,
                                                 _ptr(out), _ptr(fl), _ptr(ws), ws.numel(), _stream(raw.device)),
                   'nbc_preprocess_general_u8')
    return out, fl


def processed_size(H, W, target=1024):
    """(rows, cols) of a raw H x W image after the resize and before the trim, as Preprocessor.preprocess_array routes it
    (models.py:194-201): target x target when the larger side exceeds target, unchanged otherwise."""
    return (target, target) if max(H, W) > target else (H, W)


def mixed_descs(items):
    """ctypes array of nbc_mixed_desc from (device address, H, W, pitch, bgr, bottom_up, (span_row0, span_rows))."""
    arr = (_lib.MixedDesc * len(items))()
    for d, (ptr, H, W, pitch, bgr, bottom_up, span) in zip(arr, items):
        d.raw, d.H, d.W, d.pitch = ptr or None, H, W, pitch
        d.flags = (1 if bgr else 0) | (2 if bottom_up else 0)
        d.span_row0, d.span_rows = span
    return arr


def preprocess_mixed_batch(raws, geoms, target=1024, spans=None):
    """K1 for a chunk of raw images of any sizes in one call (nbc_preprocess_mixed_batch_u8), each routed as
    ``Preprocessor.preprocess_array`` routes it.  raws: u8 CUDA tensors; geoms: (H, W, pitch, bgr, bottom_up) per image;
    spans: optional (row0, rows) per image (only a (4 target)^2 scan may hold a part of its rows).  Returns (canvas u8
    [n, Hmax * Wmax * 3] -- image i is ``canvas[i, :(last-first) * w_i * 3].view(last-first, w_i, 3)`` with w_i its
    processed width --, first_last int32 [n, 2])."""
    lib = _lib.load()
    n = len(raws)
    raws = [_contig(r, torch.uint8, 'raw') for r in raws]
    dev = raws[0].device
    spans = [(0, g[0]) for g in geoms] if spans is None else list(spans)
    descs = mixed_descs([(r.data_ptr() if r.numel() else None,) + tuple(g) + (sp,) for r, g, sp in zip(raws, geoms, spans)])
    stride = max(h * w for h, w in (processed_size(g[0], g[1], target) for g in geoms)) * 3
    with torch.cuda.device(dev):
        ws = torch.empty(lib.nbc_preprocess_mixed_workspace_bytes(descs, n, target), dtype=torch.uint8, device=dev)
        out = torch.empty((n, stride), dtype=torch.uint8, device=dev)
        fl = torch.empty((n, 2), dtype=torch.int32, device=dev)
        _lib.check(lib.nbc_preprocess_mixed_batch_u8(descs, n, target, _ptr(out), stride, _ptr(fl), _ptr(ws), ws.numel(),
                                                     _stream(dev)), 'nbc_preprocess_mixed_batch_u8')
    return out, fl


def trim_u8(img):
    """img: u8 CUDA [H, W, 3] that needs no resize -> (out flat, first_last).  (models.py:157-166, 200-201)"""
    lib = _lib.load()
    img = _contig(img, torch.uint8, 'img')
    H, W = img.shape[0], img.shape[1]
    with torch.cuda.device(img.device):
        ws = torch.empty(lib.nbc_preprocess_workspace_bytes(max(H, 4) * 4, 4), dtype=torch.uint8, device=img.device)
        out = torch.empty(H * W * 3, dtype=torch.uint8, device=img.device)
        fl = torch.empty(2, dtype=torch.int32, device=img.device)
        _lib.check(lib.nbc_trim_u8(_ptr(img), H, W, _ptr(out), _ptr(fl), _ptr(ws), ws.numel(), _stream(img.device)),
                   'nbc_trim_u8')
    return out, fl


# ---- weights / single layers (unit-test surface) --------------------------------------------------------------------
def fold_bn_pack(weight, bn=None, conv_bias=None, eps=1e-5, cin_pad=None, dtype=torch.bfloat16):
    """weight f32 OIHW (+ optional (gamma, beta, mean, var)) -> (bf16|fp16 [Cout,kh,kw,cin_pad], f32 bias[Cout])."""
    lib = _lib.load()
    weight = _contig(weight, torch.float32, 'weight')
    Cout, Cin, kh, kw = weight.shape
    cin_pad = Cin if cin_pad is None else cin_pad
    g = b = m = v = None
    if bn is not None:
        g, b, m, v = [_contig(t, torch.float32, 'bn') for t in bn]
    cb = _contig(conv_bias, torch.float32, 'conv_bias') if conv_bias is not None else None
    with torch.cuda.device(weight.device):
        wp = torch.empty((Cout, kh, kw, cin_pad), dtype=dtype, device=weight.device)
        bias = torch.empty(Cout, dtype=torch.float32, device=weight.device)
        _lib.check(lib.nbc_fold_bn_pack(_ptr(weight), _ptr(g), _ptr(b), _ptr(m), _ptr(v), _ptr(cb), eps, Cout, Cin, kh, kw,
                                        cin_pad, 1 if dtype == torch.float16 else 0, _ptr(wp), _ptr(bias),
                                        _stream(weight.device)), 'nbc_fold_bn_pack')
    return wp, bias


def conv_bf16(x, w_packed, bias, stride=1, pad=0, dil=1, relu=False, residual=None, impl=0):
    """x bf16|fp16 NHWC [N,H,W,Cin]; w_packed same dtype [Cout,kh,kw,Cin]; -> NHWC [N,Ho,Wo,Cout] of that dtype."""
    lib = _lib.load()
    x, f16 = _half(x, 'x')
    w_packed = _contig(w_packed, x.dtype, 'w_packed')
    bias = _contig(bias, torch.float32, 'bias')
    N, H, W, Cin = x.shape
    Cout, kh, kw, cin2 = w_packed.shape
    if cin2 != Cin:
        raise RuntimeError('conv_bf16: channel mismatch %d vs %d' % (Cin, cin2))
    Ho = (H + 2 * pad - dil * (kh - 1) - 1) // stride + 1
    Wo = (W + 2 * pad - dil * (kw - 1) - 1) // stride + 1
    if residual is not None:
        residual = _contig(residual, x.dtype, 'residual')
        if tuple(residual.shape) != (N, Ho, Wo, Cout):
            raise RuntimeError('conv_bf16: residual shape mismatch')
    with torch.cuda.device(x.device):
        y = torch.empty((N, Ho, Wo, Cout), dtype=x.dtype, device=x.device)
        d = _lib.ConvDesc(N, H, W, Cin, Cout, kh, kw, stride, pad, dil, 1 if relu else 0, impl, f16)
        _lib.check(lib.nbc_conv_bf16(C.byref(d), _ptr(x), _ptr(w_packed), _ptr(bias), _ptr(residual), _ptr(y),
                                     _stream(x.device)), 'nbc_conv_bf16')
    return y


def conv_dual_bf16(x, w, x2, w2, bias, stride2=1, relu=True):
    """y = act(conv1x1(x; w) + conv1x1(x2; w2, stride2) + bias) in one launch (a bottleneck's conv3 + downsample branch).
    x [N,H,W,C1], w [Cout,1,1,C1]; x2 [N,H2,W2,C2], w2 [Cout,1,1,C2] (bf16|fp16, BN folded); bias f32 [Cout] = sum of both."""
    lib = _lib.load()
    x, f16 = _half(x, 'x')
    x2 = _contig(x2, x.dtype, 'x2')
    w, w2 = _contig(w, x.dtype, 'w'), _contig(w2, x.dtype, 'w2')
    bias = _contig(bias, torch.float32, 'bias')
    N, H, W, C1 = x.shape
    _, H2, W2, C2 = x2.shape
    Cout = w.shape[0]
    w_cat = torch.cat([w.reshape(Cout, C1), w2.reshape(Cout, C2)], dim=1).contiguous()
    with torch.cuda.device(x.device):
        y = torch.empty((N, H, W, Cout), dtype=x.dtype, device=x.device)
        d = _lib.ConvDesc(N, H, W, C1, Cout, 1, 1, 1, 0, 1, 1 if relu else 0, 1, f16)
        d2 = _lib.ConvDesc(N, H2, W2, C2, Cout, 1, 1, stride2, 0, 1, 0, 1, f16)
        _lib.check(lib.nbc_conv_dual_bf16(C.byref(d), _ptr(x), C.byref(d2), _ptr(x2), _ptr(w_cat), _ptr(bias), _ptr(y),
                                          _stream(x.device)), 'nbc_conv_dual_bf16')
    return y


def conv_wgrad_bf16(dz, x, kh, kw, stride=1, pad=0, dil=1, impl=0, out=None, split=True):
    """Weight gradient of conv_bf16: dz bf16 NHWC [N,Ho,Wo,Cout], x bf16 NHWC [N,H,W,Cin] -> f32 [Cout,kh,kw,Cin]
    (accumulated into ``out`` when given).  impl 0 auto, 1 tcgen05, 2 mma.sync.  The tcgen05 kernel runs as the
    training plan runs it: the pixels split over the SMs, the partials in a scratch buffer allocated here and added in a
    fixed order (``nbc_conv_wgrad_bf16_ws``); ``split=False`` makes one CTA per weight tile sum every pixel
    (``nbc_conv_wgrad_bf16`` without scratch).  Both are bit-reproducible; the mma.sync kernel is not."""
    lib = _lib.load()
    dz = _contig(dz, torch.bfloat16, 'dz')
    x = _contig(x, torch.bfloat16, 'x')
    N, H, W, Cin = x.shape
    Cout = dz.shape[3]
    Ho = (H + 2 * pad - dil * (kh - 1) - 1) // stride + 1
    Wo = (W + 2 * pad - dil * (kw - 1) - 1) // stride + 1
    if tuple(dz.shape) != (N, Ho, Wo, Cout):
        raise RuntimeError('conv_wgrad_bf16: dz shape %s does not match the geometry %s' % (tuple(dz.shape), (N, Ho, Wo, Cout)))
    with torch.cuda.device(x.device):
        if out is None:
            out = torch.zeros((Cout, kh, kw, Cin), dtype=torch.float32, device=x.device)
        else:
            out = _contig(out, torch.float32, 'out')
        d = _lib.ConvDesc(N, H, W, Cin, Cout, kh, kw, stride, pad, dil, 0, impl, 0)
        n = lib.nbc_conv_wgrad_workspace_bytes(C.byref(d)) if split and impl != 2 else 0    # 0: no split (or no tcgen05)
        if n > 0:
            ws = torch.empty(n, dtype=torch.uint8, device=x.device)
            _lib.check(lib.nbc_conv_wgrad_bf16_ws(C.byref(d), _ptr(dz), _ptr(x), _ptr(out), _ptr(ws), n, _stream(x.device)),
                       'nbc_conv_wgrad_bf16_ws')
        else:
            _lib.check(lib.nbc_conv_wgrad_bf16(C.byref(d), _ptr(dz), _ptr(x), _ptr(out), _stream(x.device)), 'nbc_conv_wgrad_bf16')
    return out


def stem_u8(img, mean, std, w_stem, bias):
    lib = _lib.load()
    img = _contig(img, torch.uint8, 'img')
    N, H, W, _ = img.shape
    m3 = (C.c_float * 3)(*mean)
    s3 = (C.c_float * 3)(*std)
    with torch.cuda.device(img.device):
        out = torch.empty((N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, 64), dtype=torch.bfloat16, device=img.device)
        _lib.check(lib.nbc_stem_u8(_ptr(img), N, H, W, m3, s3, _ptr(_contig(w_stem, torch.float32, 'w_stem')),
                                   _ptr(_contig(bias, torch.float32, 'bias')), _ptr(out), _stream(img.device)), 'nbc_stem_u8')
    return out


def stem_f32(x, w_stem, bias):
    lib = _lib.load()
    x = _contig(x, torch.float32, 'x')
    N, _, H, W = x.shape
    with torch.cuda.device(x.device):
        out = torch.empty((N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, 64), dtype=torch.bfloat16, device=x.device)
        _lib.check(lib.nbc_stem_f32(_ptr(x), N, H, W, _ptr(_contig(w_stem, torch.float32, 'w_stem')),
                                    _ptr(_contig(bias, torch.float32, 'bias')), _ptr(out), _stream(x.device)), 'nbc_stem_f32')
    return out


def stem_tc(inp, mean, std, w_stem, bias, dtype=torch.bfloat16):
    """Tensor-core stem: inp u8 NHWC or f32 NCHW; w_stem f32 [64,7,7,3] (BN folded) -> bf16 NHWC [N,H/2,W/2,64]."""
    lib = _lib.load()
    _dev(inp, 'input')
    inp = inp.contiguous()
    if inp.dtype == torch.uint8:
        N, H, W, _ = inp.shape
        kind = 0
    else:
        N, _, H, W = inp.shape
        kind = 1
    m3 = (C.c_float * 3)(*mean)
    s3 = (C.c_float * 3)(*std)
    with torch.cuda.device(inp.device):
        f16 = 1 if dtype == torch.float16 else 0
        w224 = torch.empty(64 * 224, dtype=dtype, device=inp.device)
        _lib.check(lib.nbc_stem_pack_weights(_ptr(_contig(w_stem, torch.float32, 'w_stem')), f16, _ptr(w224), _stream(inp.device)),
                   'nbc_stem_pack_weights')
        ws = torch.empty(lib.nbc_stem_tc_workspace_bytes(N, H, W), dtype=torch.uint8, device=inp.device)
        out = torch.empty((N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, 64), dtype=dtype, device=inp.device)
        _lib.check(lib.nbc_stem_tc(_ptr(inp), kind, N, H, W, m3, s3, _ptr(w224), _ptr(_contig(bias, torch.float32, 'bias')),
                                   f16, _ptr(ws), ws.numel(), _ptr(out), _stream(inp.device)), 'nbc_stem_tc')
    return out


def maxpool3x3s2(x):
    lib = _lib.load()
    x, f16 = _half(x, 'x')
    N, H, W, Cc = x.shape
    with torch.cuda.device(x.device):
        y = torch.empty((N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, Cc), dtype=x.dtype, device=x.device)
        _lib.check(lib.nbc_maxpool3x3s2_bf16(_ptr(x), N, H, W, Cc, f16, _ptr(y), _stream(x.device)), 'nbc_maxpool3x3s2_bf16')
    return y


def head_1x1(x, weight, bias):
    """x bf16|fp16 NHWC [N,h,w,Cin], weight f32 [3,Cin], bias f32[3] -> f32 [N,3,h,w]."""
    lib = _lib.load()
    x, f16 = _half(x, 'x')
    N, h, w, Cin = x.shape
    with torch.cuda.device(x.device):
        out = torch.empty((N, 3, h, w), dtype=torch.float32, device=x.device)
        _lib.check(lib.nbc_head_1x1(_ptr(x), h * w, N, Cin, f16, _ptr(_contig(weight, torch.float32, 'weight')),
                                    _ptr(_contig(bias, torch.float32, 'bias')), _ptr(out), _stream(x.device)), 'nbc_head_1x1')
    return out


# ---- K3 -------------------------------------------------------------------------------------------------------
def upsample_argmax(logits, size, out=None):
    """logits f32 [N,3,h,w] -> u8 mask [N,H,W] = argmax(bicubic upsample)  (models.py:38-41, 270)."""
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    N, Cc, h, w = logits.shape
    if Cc != 3:
        raise RuntimeError('upsample_argmax expects 3 classes')
    H, W = size
    with torch.cuda.device(logits.device):
        if out is None:
            out = torch.empty((N, H, W), dtype=torch.uint8, device=logits.device)
        _lib.check(lib.nbc_upsample_argmax(_ptr(logits), N, h, w, H, W, _ptr(out), _stream(logits.device)),
                   'nbc_upsample_argmax')
    return out


def upsample_bicubic(logits, size):
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    N, Cc, h, w = logits.shape
    H, W = size
    with torch.cuda.device(logits.device):
        out = torch.empty((N, Cc, H, W), dtype=torch.float32, device=logits.device)
        _lib.check(lib.nbc_upsample_bicubic(_ptr(logits), N, Cc, h, w, H, W, _ptr(out), _stream(logits.device)),
                   'nbc_upsample_bicubic')
    return out


def upsample_argmax_ragged(logits, heights, canvas_hw, out=None):
    """Ragged batch: logits f32 [N,3,hc,w] canvas, heights int32 [N] (CUDA) -> u8 mask canvas [N,Hc,W]; image n gets
    rows [0, heights[n]) from its ceil(heights[n]/8) logit rows."""
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    heights = _contig(heights, torch.int32, 'heights')
    N, Cc, hc, w = logits.shape
    Hc, W = canvas_hw
    with torch.cuda.device(logits.device):
        if out is None:
            out = torch.zeros((N, Hc, W), dtype=torch.uint8, device=logits.device)
        _lib.check(lib.nbc_upsample_argmax_ragged(_ptr(logits), N, hc, w, Hc, W, _ptr(heights), _ptr(out),
                                                  _stream(logits.device)), 'nbc_upsample_argmax_ragged')
    return out


# ---- flip test-time augmentation ------------------------------------------------------------------------------------
TTA_MODES = ('none', 'h', 'hv')
_TTA_VIEWS = {'none': (['id'], [0]), 'h': (['id', 'h'], [0, 1]), 'hv': (['id', 'h', 'v', 'hv'], [0, 1, 2, 3])}


def tta_views(mode):
    """The view set of ``--tta mode`` in summation order: (names, flip flags), flag 1 mirrors the columns, 2 the rows of
    each image's own height.  'none' -> (['id'], [0]); 'h' -> (['id', 'h'], [0, 1]); 'hv' -> (['id', 'h', 'v', 'hv'],
    [0, 1, 2, 3])."""
    if mode not in _TTA_VIEWS:
        raise ValueError("tta must be one of %s (got %r)" % (', '.join(TTA_MODES), mode))
    names, flags = _TTA_VIEWS[mode]
    return list(names), list(flags)


def flip_ragged(canvas, heights, flags, out=None):
    """canvas u8 [N,Hc,W,3], heights int32 [N] (CUDA) -> a new canvas with image n mirrored within its rows [0, heights[n])
    (flags & 2) and its columns (flags & 1), rows below zero (nbc_flip_ragged_u8)."""
    lib = _lib.load()
    canvas = _contig(canvas, torch.uint8, 'canvas')
    heights = _contig(heights, torch.int32, 'heights')
    if canvas.dim() != 4 or canvas.shape[3] != 3 or tuple(heights.shape) != (canvas.shape[0],):
        raise RuntimeError('flip_ragged: canvas u8 [N,Hc,W,3] and heights [N] expected')
    N, Hc, W, _ = canvas.shape
    with torch.cuda.device(canvas.device):
        if out is None:
            out = torch.empty_like(canvas)
        elif not (out.dtype == torch.uint8 and out.is_contiguous() and out.shape == canvas.shape):
            raise RuntimeError('flip_ragged: out must be a contiguous u8 tensor of the canvas shape')
        _lib.check(lib.nbc_flip_ragged_u8(_ptr(canvas), _ptr(out), N, Hc, W, _ptr(heights), int(flags), _stream(canvas.device)),
                   'nbc_flip_ragged_u8')
    return out


def _view_set(logits, flips, name):
    """Checked view set: (contiguous f32 canvases, ctypes pointer array, ctypes flag array, (N, hc, w))."""
    logits = [_contig(t, torch.float32, name) for t in logits]
    flips = [int(f) for f in flips]
    if len(logits) != len(flips) or len(logits) not in (1, 2, 4):
        raise RuntimeError('%s: 1, 2 or 4 views, one flip flag each (got %d canvases, %d flags)' % (name, len(logits), len(flips)))
    shape = tuple(logits[0].shape)
    if len(shape) != 4 or shape[1] != 3 or any(tuple(t.shape) != shape for t in logits):
        raise RuntimeError('%s: every view is an f32 [N,3,hc,w] canvas of one shape' % name)
    ptrs = (C.c_void_p * len(logits))(*[t.data_ptr() for t in logits])
    fl = (C.c_int32 * len(flips))(*flips)
    return logits, ptrs, fl, (shape[0], shape[2], shape[3])


def upsample_argmax_views_ragged(logits, flips, heights, canvas_hw, out=None):
    """Multi-view K3: logits = list of f32 [N,3,hc,w] canvases (the network's output for the batch mirrored with
    flips[v]), heights int32 [N] -> u8 mask canvas [N,Hc,W] = argmax of the views' mean bicubic logits, each view un-flipped
    (nbc_upsample_argmax_views_ragged)."""
    lib = _lib.load()
    logits, ptrs, fl, (N, hc, w) = _view_set(logits, flips, 'upsample_argmax_views_ragged')
    heights = _contig(heights, torch.int32, 'heights')
    Hc, W = canvas_hw
    dev = logits[0].device
    with torch.cuda.device(dev):
        if out is None:
            out = torch.zeros((N, Hc, W), dtype=torch.uint8, device=dev)
        _lib.check(lib.nbc_upsample_argmax_views_ragged(ptrs, fl, len(logits), N, hc, w, Hc, W, _ptr(heights), _ptr(out),
                                                        _stream(dev)), 'nbc_upsample_argmax_views_ragged')
    return out


def upsample_bicubic_views_ragged(logits, flips, heights, canvas_hw, out=None):
    """The mean logits of ``upsample_argmax_views_ragged`` at full resolution: f32 [N,3,Hc,W], rows [0, heights[n]) of
    image n written (nbc_upsample_bicubic_views_ragged)."""
    lib = _lib.load()
    logits, ptrs, fl, (N, hc, w) = _view_set(logits, flips, 'upsample_bicubic_views_ragged')
    heights = _contig(heights, torch.int32, 'heights')
    Hc, W = canvas_hw
    dev = logits[0].device
    with torch.cuda.device(dev):
        if out is None:
            out = torch.zeros((N, 3, Hc, W), dtype=torch.float32, device=dev)
        _lib.check(lib.nbc_upsample_bicubic_views_ragged(ptrs, fl, len(logits), N, hc, w, Hc, W, _ptr(heights), _ptr(out),
                                                         _stream(dev)), 'nbc_upsample_bicubic_views_ragged')
    return out


def heights_from_first_last(first_last, out=None):
    lib = _lib.load()
    first_last = _contig(first_last, torch.int32, 'first_last')
    N = first_last.shape[0]
    with torch.cuda.device(first_last.device):
        if out is None:
            out = torch.empty(N, dtype=torch.int32, device=first_last.device)
        _lib.check(lib.nbc_heights_from_first_last(_ptr(first_last), N, _ptr(out), _stream(first_last.device)),
                   'nbc_heights_from_first_last')
    return out


# ---- K5 -------------------------------------------------------------------------------------------------------
def remove_small_zones_u8(mask, threshold=150, exclude_nodes=False, workspace=None):
    """mask u8 CUDA [N,H,W], modified in place.  Returns (mask, counts int32 [N,3]).  (utils.py:135-148)"""
    lib = _lib.load()
    _dev(mask, 'mask')
    if mask.dtype != torch.uint8 or not mask.is_contiguous() or mask.dim() != 3:
        raise RuntimeError('remove_small_zones_u8 expects a contiguous u8 [N,H,W] tensor')
    N, H, W = mask.shape
    with torch.cuda.device(mask.device):
        need = lib.nbc_ccl_workspace_bytes(N, H, W)
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=mask.device)
        counts = torch.empty((N, 3), dtype=torch.int32, device=mask.device)
        _lib.check(lib.nbc_remove_small_zones(_ptr(mask), N, H, W, int(threshold), 1 if exclude_nodes else 0, _ptr(counts),
                                              _ptr(workspace), workspace.numel(), _stream(mask.device)),
                   'nbc_remove_small_zones')
    return mask, counts


def remove_small_zones_ragged(mask, heights, threshold=150, exclude_nodes=False, workspace=None, counts=None):
    """Ragged batch: mask u8 canvas [N,Hc,W] in place, only rows [0, heights[n]) of image n take part."""
    lib = _lib.load()
    _dev(mask, 'mask')
    heights = _contig(heights, torch.int32, 'heights')
    if mask.dtype != torch.uint8 or not mask.is_contiguous() or mask.dim() != 3:
        raise RuntimeError('remove_small_zones_ragged expects a contiguous u8 [N,Hc,W] tensor')
    N, H, W = mask.shape
    with torch.cuda.device(mask.device):
        need = lib.nbc_ccl_workspace_bytes(N, H, W)
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=mask.device)
        if counts is None:
            counts = torch.empty((N, 3), dtype=torch.int32, device=mask.device)
        _lib.check(lib.nbc_remove_small_zones_ragged(_ptr(mask), N, H, W, _ptr(heights), int(threshold),
                                                     1 if exclude_nodes else 0, _ptr(counts), _ptr(workspace),
                                                     workspace.numel(), _stream(mask.device)), 'nbc_remove_small_zones_ragged')
    return mask, counts


# ---- K4 -------------------------------------------------------------------------------------------------------
def wce_fwd_bwd(logits, target, weights, need_grad=True):
    """logits f32 [N,3,H,W], target u8 or int64 [N,H,W], weights f32[3] -> (loss 0-dim f32, grad or None)."""
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    _dev(target, 'target')
    if target.dtype not in (torch.uint8, torch.int64):
        raise RuntimeError('target must be uint8 or int64')
    target = target.contiguous()
    weights = _contig(weights, torch.float32, 'weights')
    N, Cc, H, W = logits.shape
    if Cc != 3 or tuple(target.shape) != (N, H, W):
        raise RuntimeError('wce: expected logits [N,3,H,W] and target [N,H,W]')
    with torch.cuda.device(logits.device):
        ws = torch.empty(lib.nbc_wce_workspace_bytes(N, H, W), dtype=torch.uint8, device=logits.device)
        loss = torch.empty((), dtype=torch.float32, device=logits.device)
        grad = torch.empty_like(logits) if need_grad else None
        _lib.check(lib.nbc_wce_fwd_bwd(_ptr(logits), _ptr(target), 1 if target.dtype == torch.int64 else 0, _ptr(weights), N,
                                       H, W, _ptr(loss), _ptr(grad), _ptr(ws), ws.numel(), _stream(logits.device)),
                   'nbc_wce_fwd_bwd')
    return loss, grad


def lovasz_softmax_fwd_bwd(logits, target, need_grad=True, upstream=1.0):
    """N1: LovaszSoftmax (lovasz_losses.py:162-218) on f32 logits [N,3,H,W] and u8|int64 labels [N,H,W] ->
    (loss 0-dim f32, grad f32 [N,3,H,W] or None)."""
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    _dev(target, 'target')
    if target.dtype not in (torch.uint8, torch.int64):
        raise RuntimeError('lovasz_softmax_fwd_bwd: target must be uint8 or int64')
    target = target.contiguous()
    N, Cc, H, W = logits.shape
    if Cc != 3 or tuple(target.shape) != (N, H, W):
        raise RuntimeError('lovasz_softmax_fwd_bwd: logits [N,3,H,W] and target [N,H,W] expected')
    with torch.cuda.device(logits.device):
        loss = torch.zeros((), dtype=torch.float32, device=logits.device)
        grad = torch.empty_like(logits) if need_grad else None
        ws = torch.empty(lib.nbc_lovasz_workspace_bytes(N, H, W), dtype=torch.uint8, device=logits.device)
        _lib.check(lib.nbc_lovasz_softmax_fwd_bwd(_ptr(logits), _ptr(target), 1 if target.dtype == torch.int64 else 0, N, H, W,
                                                  C.c_float(upstream), _ptr(loss), _ptr(grad), _ptr(ws), ws.numel(),
                                                  _stream(logits.device)), 'nbc_lovasz_softmax_fwd_bwd')
    return loss, grad


def argmax3_u8(logits):
    """torch.argmax(logits, 1) of f32 [N,3,H,W] as u8 [N,H,W]."""
    lib = _lib.load()
    logits = _contig(logits, torch.float32, 'logits')
    N, Cc, H, W = logits.shape
    if Cc != 3:
        raise RuntimeError('argmax3_u8: 3 classes expected')
    with torch.cuda.device(logits.device):
        out = torch.empty((N, H, W), dtype=torch.uint8, device=logits.device)
        _lib.check(lib.nbc_argmax3_u8(_ptr(logits), N, H, W, _ptr(out), _stream(logits.device)), 'nbc_argmax3_u8')
    return out


def confusion_matrix(pred_u8, target):
    """N2: cm[t, p] (int64 CUDA tensor [3,3]) over all pixels of pred u8 [...] and target u8|int64 of the same shape."""
    lib = _lib.load()
    pred_u8 = _contig(pred_u8, torch.uint8, 'pred')
    _dev(target, 'target')
    if target.dtype not in (torch.uint8, torch.int64) or target.numel() != pred_u8.numel():
        raise RuntimeError('confusion_matrix: target must be uint8 or int64 with as many elements as pred')
    target = target.contiguous()
    with torch.cuda.device(pred_u8.device):
        cm = torch.zeros(9, dtype=torch.int64, device=pred_u8.device)
        _lib.check(lib.nbc_confusion_matrix(_ptr(pred_u8), _ptr(target), 1 if target.dtype == torch.int64 else 0,
                                            pred_u8.numel(), _ptr(cm), _stream(pred_u8.device)), 'nbc_confusion_matrix')
    return cm.view(3, 3)


EVAL_WCE, EVAL_LOVASZ = 1, 2


def eval_ragged(logits, heights, labels, weights=None, losses=EVAL_WCE | EVAL_LOVASZ, workspace=None):
    """N3: the per-image evaluation of a ragged chunk in one call.  logits f32 [N,3,ceil(Hc/8),ceil(W/8)] as
    ``Plan.forward_ragged`` leaves them, heights int32 [N], labels u8 classes [N,Hc,W], weights f32[3] (needed with
    ``EVAL_WCE``), ``losses`` a bitmask of EVAL_WCE / EVAL_LOVASZ.  Returns a dict of device tensors: loss_wce f32 [N],
    loss_lovasz f32 [N], cm_raw int64 [N,3,3] (argmax), cm_rsz int64 [N,3,3] (after region removal) and counts int32
    [N,3], each equal to the per-image ops on that image alone (see include/nbc.h)."""
    return _eval([logits], [0], heights, labels, weights, losses, workspace, views=False)


def eval_ragged_views(logits, flips, heights, labels, weights=None, losses=EVAL_WCE | EVAL_LOVASZ, workspace=None):
    """``eval_ragged`` on a view set (nbc_eval_ragged_views): logits is a list of 1, 2 or 4 canvases, view v the network's
    output for the chunk mirrored with flips[v] (``flip_ragged``); every output is computed from the views' mean bicubic
    logits, as ``upsample_bicubic_views_ragged`` gives them."""
    return _eval(logits, flips, heights, labels, weights, losses, workspace, views=True)


def _eval(logits, flips, heights, labels, weights, losses, workspace, views):
    """nbc_eval_ragged (views=False: the one canvas logits[0]) or nbc_eval_ragged_views."""
    lib = _lib.load()
    logits, ptrs, fl, _ = _view_set(logits, flips, 'eval_ragged')
    heights = _contig(heights, torch.int32, 'heights')
    labels = _contig(labels, torch.uint8, 'labels')
    if labels.dim() != 3:
        raise RuntimeError('eval_ragged: labels must be u8 [N,Hc,W]')
    N, Hc, W = labels.shape
    hc = ((((Hc - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
    w = ((((W - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
    if tuple(logits[0].shape) != (N, 3, hc, w) or tuple(heights.shape) != (N,):
        raise RuntimeError('eval_ragged: expected logits [%d,3,%d,%d] and heights [%d] for labels %s'
                           % (N, hc, w, N, tuple(labels.shape)))
    if weights is not None:
        weights = _contig(weights, torch.float32, 'weights')
    dev = logits[0].device
    with torch.cuda.device(dev):
        need = lib.nbc_eval_workspace_bytes(N, Hc, W)
        if workspace is None or workspace.numel() < need:
            workspace = torch.empty(max(need, 1), dtype=torch.uint8, device=dev)
        out = {'loss_wce': torch.empty(N, dtype=torch.float32, device=dev),
               'loss_lovasz': torch.empty(N, dtype=torch.float32, device=dev),
               'cm_raw': torch.empty((N, 3, 3), dtype=torch.int64, device=dev),
               'cm_rsz': torch.empty((N, 3, 3), dtype=torch.int64, device=dev),
               'counts': torch.empty((N, 3), dtype=torch.int32, device=dev)}
        rest = (N, Hc, W, _ptr(heights), _ptr(labels), _ptr(weights), int(losses), _ptr(out['loss_wce']), _ptr(out['loss_lovasz']),
                _ptr(out['cm_raw']), _ptr(out['cm_rsz']), _ptr(out['counts']), _ptr(workspace), workspace.numel(), _stream(dev))
        if not views:
            _lib.check(lib.nbc_eval_ragged(_ptr(logits[0]), *rest), 'nbc_eval_ragged')
        else:
            _lib.check(lib.nbc_eval_ragged_views(ptrs, fl, len(logits), *rest), 'nbc_eval_ragged_views')
    return out


# ---- the network plan ---------------------------------------------------------------------------------------------
class Plan:
    """Owns an nbc_plan (BN-folded bf16 weights on the device) built from the 326 state_dict tensors."""

    def __init__(self, tensors, mean, std, device, precision='fp16'):
        lib = _lib.load()
        if precision not in HALF_DTYPES:
            raise ValueError("precision must be 'bf16' or 'fp16'")
        self.precision = precision
        self.device = torch.device(device)
        _lib.require_device(self.device.index if self.device.index is not None else torch.cuda.current_device())
        keep = []
        for t in tensors:
            _dev(t, 'state_dict tensor')
            keep.append(t.detach().contiguous() if t.dtype != torch.int64 else t.detach())
        arr = (C.c_void_p * len(keep))(*[t.data_ptr() for t in keep])
        m3 = (C.c_float * 3)(*mean)
        s3 = (C.c_float * 3)(*std)
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().synchronize()
            self.handle = lib.nbc_plan_create(arr, len(keep), m3, s3, 1 if precision == 'fp16' else 0)
        if not self.handle:
            raise RuntimeError('nbc_plan_create failed: ' + _lib.last_error())
        self._ws = None
        self._lib = lib

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                self._lib.nbc_plan_destroy(C.c_void_p(self.handle))
                self.handle = None
        except Exception:
            pass

    def set_impl(self, impl):
        _lib.check(self._lib.nbc_plan_set_impl(C.c_void_p(self.handle), int(impl)), 'nbc_plan_set_impl')

    def set_stop(self, k):
        """Debug hook: the forwards that follow run steps 0..k of the launch list only (k < 0: all, the default)."""
        _lib.check(self._lib.nbc_plan_set_stop(C.c_void_p(self.handle), int(k)), 'nbc_plan_set_stop')

    def steps(self):
        """The launch list of the most recent forward: one dict per step (nbc_plan_step fields; workspace byte offsets)."""
        out = []
        for i in range(self._lib.nbc_plan_num_steps(C.c_void_p(self.handle))):
            s = _lib.PlanStep()
            _lib.check(self._lib.nbc_plan_step_info(C.c_void_p(self.handle), i, C.byref(s)), 'nbc_plan_step_info')
            d = {n: getattr(s, n) for n, _ in _lib.PlanStep._fields_}
            d['name'] = s.name.decode()
            out.append(d)
        return out

    def _workspace(self, N, H, W):
        need = self._lib.nbc_plan_workspace_bytes(C.c_void_p(self.handle), N, H, W) + 1024
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        off = (-self._ws.data_ptr()) % 1024
        return self._ws.data_ptr() + off, self._ws.numel() - off

    def forward(self, inp, out=None):
        """inp: u8 NHWC [N,H,W,3] (normalised inside) or f32 NCHW [N,3,H,W] (already normalised).
        Returns f32 low-resolution logits [N,3,h,w]."""
        _dev(inp, 'input')
        if inp.dtype == torch.uint8:
            inp = inp if inp.is_contiguous() else inp.contiguous()
            N, H, W, c = inp.shape
            kind = 0
        elif inp.dtype == torch.float32:
            inp = inp if inp.is_contiguous() else inp.contiguous()
            N, c, H, W = inp.shape
            kind = 1
        else:
            raise RuntimeError('Plan.forward expects u8 NHWC or f32 NCHW input')
        if c != 3:
            raise RuntimeError('Plan.forward expects 3 channels')
        h = ((((H - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        w = ((((W - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty((N, 3, h, w), dtype=torch.float32, device=self.device)
            ws_ptr, ws_bytes = self._workspace(N, H, W)
            _lib.check(self._lib.nbc_plan_forward(C.c_void_p(self.handle), _ptr(inp), kind, N, H, W, _ptr(out),
                                                  C.c_void_p(ws_ptr), ws_bytes, _stream(self.device)), 'nbc_plan_forward')
        return out

    def forward_ragged(self, canvas, heights=None, first_last=None, out=None):
        """canvas u8 [N,Hc,W,3]; image n occupies rows [0, h_n) with h_n = heights[n] or last-first of first_last[n]
        (int32 CUDA tensors, read on the device).  Returns the f32 logits canvas [N,3,ceil(Hc/8),ceil(W/8)]."""
        canvas = _contig(canvas, torch.uint8, 'canvas')
        N, H, W, c = canvas.shape
        if c != 3 or (heights is None) == (first_last is None):
            raise RuntimeError('forward_ragged: u8 [N,Hc,W,3] canvas and exactly one of heights / first_last')
        if heights is not None:
            heights = _contig(heights, torch.int32, 'heights')
        else:
            first_last = _contig(first_last, torch.int32, 'first_last')
        h = ((((H - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        w = ((((W - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.zeros((N, 3, h, w), dtype=torch.float32, device=self.device)
            ws_ptr, ws_bytes = self._workspace(N, H, W)
            _lib.check(self._lib.nbc_plan_forward_ragged(C.c_void_p(self.handle), _ptr(canvas), N, H, W, _ptr(heights),
                                                         _ptr(first_last), _ptr(out), C.c_void_p(ws_ptr), ws_bytes,
                                                         _stream(self.device)), 'nbc_plan_forward_ragged')
        return out

    def profile(self, inp):
        """Per-layer CUDA-event timing of one forward: list of (ms, flops)."""
        _dev(inp, 'input')
        N, H, W, _ = inp.shape
        h = ((((H - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        w = ((((W - 1) // 2 + 1) - 1) // 2 + 1 - 1) // 2 + 1
        with torch.cuda.device(self.device):
            out = torch.empty((N, 3, h, w), dtype=torch.float32, device=self.device)
            ws_ptr, ws_bytes = self._workspace(N, H, W)
            ms = (C.c_float * 128)()
            fl = (C.c_double * 128)()
            n = self._lib.nbc_plan_profile(C.c_void_p(self.handle), _ptr(inp), 0, N, H, W, _ptr(out), C.c_void_p(ws_ptr),
                                           ws_bytes, _stream(self.device), ms, fl, 128)
            if n < 0:
                _lib.check(n, 'nbc_plan_profile')
        return [(ms[i], fl[i]) for i in range(n)]
