"""ctypes binding of libnbc.so (the C-ABI declared in include/nbc.h).  Fails loudly: no library -> ImportError-like
RuntimeError with the build command; no B200 -> RuntimeError from nbc_device_check.  Never falls back to torch ops."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnbc.so')

c_void_p, c_int, c_i64, c_size_t, c_float = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('N', 'H', 'W', 'Cin', 'Cout', 'kh', 'kw', 'stride', 'pad', 'dil', 'relu', 'impl', 'f16')]


class PlanStep(C.Structure):
    """nbc_plan_step: one launch of the plan (see include/nbc.h)."""
    _fields_ = ([('name', C.c_char * 24)]
                + [(n, C.c_int32) for n in ('kind', 'pair', 'halo3', 'stem_halo', 'dual', 'block_n', 'kblk', 'out_bufs',
                                            'ragged_map', 'N', 'H', 'W', 'Cin', 'Cout', 'k', 'stride', 'pad', 'dil', 'relu',
                                            'H2', 'W2', 'Cin2', 'stride2', 'level')]
                + [(n, C.c_int64) for n in ('x', 'x2', 'residual', 'y', 'levels')])


class MixedDesc(C.Structure):
    """nbc_mixed_desc: one raw image of a mixed K1 chunk (see include/nbc.h)."""
    _fields_ = [('raw', C.c_void_p), ('H', C.c_int32), ('W', C.c_int32), ('pitch', C.c_int64), ('flags', C.c_int32),
                ('span_row0', C.c_int32), ('span_rows', C.c_int32), ('reserved', C.c_int32)]


# name -> (restype, argtypes); kept in one table so tests can check it against include/nbc.h
SIGNATURES = {
    'nbc_version': (c_int, []),
    'nbc_last_error': (C.c_char_p, []),
    'nbc_device_check': (c_int, [c_int]),
    'nbc_launch_count': (c_i64, []),
    'nbc_preprocess_workspace_bytes': (c_size_t, [c_int, c_int]),
    'nbc_preprocess_4x_u8': (c_int, [c_void_p, c_int, c_int, c_i64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'nbc_preprocess_4x_span_u8': (c_int, [c_void_p, c_int, c_int, c_i64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                          c_void_p]),
    'nbc_preprocess_4x_batch_u8': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_i64, c_int, c_void_p, c_i64, c_void_p,
                                           c_void_p, c_size_t, c_void_p]),
    'nbc_host_zero_row_span': (c_int, [c_void_p, c_int, c_i64, c_i64, c_int, c_void_p, c_void_p]),
    'nbc_preprocess_general_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'nbc_preprocess_general_u8': (c_int, [c_void_p, c_int, c_int, c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                  c_void_p]),
    'nbc_trim_u8': (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'nbc_preprocess_mixed_workspace_bytes': (c_size_t, [C.POINTER(MixedDesc), c_int, c_int]),
    'nbc_preprocess_mixed_batch_u8': (c_int, [C.POINTER(MixedDesc), c_int, c_int, c_void_p, c_i64, c_void_p, c_void_p, c_size_t,
                                      c_void_p]),
    'nbc_fold_bn_pack': (c_int, [c_void_p] * 6 + [c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'nbc_conv_bf16': (c_int, [C.POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_conv_dual_bf16': (c_int, [C.POINTER(ConvDesc), c_void_p, C.POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_conv_wgrad_bf16': (c_int, [C.POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_stem_u8': (c_int, [c_void_p, c_int, c_int, c_int, C.POINTER(c_float), C.POINTER(c_float), c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_stem_f32': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_stem_tc_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'nbc_stem_pack_weights': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'nbc_stem_tc': (c_int, [c_void_p, c_int, c_int, c_int, c_int, C.POINTER(c_float), C.POINTER(c_float), c_void_p, c_void_p,
                    c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    'nbc_maxpool3x3s2_bf16': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'nbc_head_1x1': (c_int, [c_void_p, c_i64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'nbc_upsample_argmax': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'nbc_upsample_bicubic': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'nbc_upsample_argmax_ragged': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'nbc_heights_from_first_last': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'nbc_ccl_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'nbc_remove_small_zones': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    'nbc_remove_small_zones_ragged': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                      c_void_p]),
    'nbc_wce_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'nbc_wce_fwd_bwd': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'nbc_lovasz_workspace_bytes': (c_size_t, [c_int, c_int, c_int]),
    'nbc_lovasz_softmax_fwd_bwd': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                   c_size_t, c_void_p]),
    'nbc_argmax3_u8': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    'nbc_confusion_matrix': (c_int, [c_void_p, c_void_p, c_int, c_i64, c_void_p, c_void_p]),
    'nbc_augment_batch': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                          c_void_p]),
    'nbc_augment_ragged': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int,
                           c_void_p, c_void_p, c_void_p]),
    'nbc_png_idat_bound': (c_size_t, [c_int, c_int, c_int]),
    'nbc_png_idat': (c_i64, [c_void_p, c_int, c_int, c_int, c_i64, c_void_p, c_void_p, c_size_t]),
    'nbc_compose_combined': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    'nbc_plan_create': (c_void_p, [C.POINTER(c_void_p), c_int, C.POINTER(c_float), C.POINTER(c_float), c_int]),
    'nbc_plan_destroy': (None, [c_void_p]),
    'nbc_plan_workspace_bytes': (c_size_t, [c_void_p, c_int, c_int, c_int]),
    'nbc_plan_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    'nbc_plan_forward_ragged': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                c_void_p]),
    'nbc_plan_profile': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p,
                                 C.POINTER(c_float), C.POINTER(C.c_double), c_int]),
    'nbc_plan_set_impl': (c_int, [c_void_p, c_int]),
    'nbc_plan_set_stop': (c_int, [c_void_p, c_int]),
    'nbc_plan_num_steps': (c_int, [c_void_p]),
    'nbc_plan_step_info': (c_int, [c_void_p, c_int, C.POINTER(PlanStep)]),
    'nbc_train_create': (c_void_p, [c_int, c_int, c_int]),
    'nbc_train_destroy': (None, [c_void_p]),
    'nbc_train_param_count': (c_i64, [c_void_p]),
    'nbc_train_stats_count': (c_i64, [c_void_p]),
    'nbc_train_workspace_bytes': (c_size_t, [c_void_p]),
    'nbc_train_exchange': (c_int, [c_void_p, C.POINTER(c_void_p), c_int, c_void_p, c_void_p, c_int, c_void_p]),
    'nbc_train_forward_backward': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, C.POINTER(c_float),
                                   C.POINTER(c_float), c_void_p, c_void_p, c_float, C.c_uint64, c_void_p, c_void_p, c_size_t,
                                   c_void_p]),
    'nbc_train_num_segments': (c_int, [c_void_p]),
    'nbc_train_segment': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'nbc_train_wait_segment': (c_int, [c_void_p, c_int, c_void_p]),
    'nbc_train_debug_offset': (c_i64, [c_void_p, c_int, c_int, C.POINTER(C.c_int32)]),
    'nbc_train_num_units': (c_int, [c_void_p]),
    'nbc_train_capture_bytes': (c_size_t, [c_void_p]),
    'nbc_train_set_capture': (c_int, [c_void_p, c_void_p, c_size_t]),
    'nbc_train_set_wgrad_impl': (c_int, [c_void_p, c_int]),
    'nbc_train_set_loss': (c_int, [c_void_p, c_int]),
    'nbc_train_adam': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_float, c_float, c_float, c_float, c_float,
                       c_int, c_float, c_void_p]),
}

_lib = None
_checked_devices = set()


def load():
    """Load libnbc.so (once).  Raises if the extension has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libnbc.so is missing (%s). Build it with `python -m neuralbarkcalculator_b200.build`; '
                           'this package has no CPU / PyTorch fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().nbc_last_error().decode('utf-8', 'replace')


def check(rc, what=''):
    if rc != 0:
        raise RuntimeError('libnbc %s failed (status %d): %s' % (what, rc, last_error()))


def require_device(index):
    """nbc_device_check: the device must exist and be sm_100 (B200)."""
    if index in _checked_devices:
        return
    check(load().nbc_device_check(int(index)), 'nbc_device_check')
    _checked_devices.add(index)


def launch_count():
    return int(load().nbc_launch_count())
