"""ctypes binding of libpaacb.so (include/paacb.h).  There is no CPU fallback: if the library is
missing, cannot be loaded, or a call fails, this raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('PAACB_LIB') or os.path.join(HERE, 'libpaacb.so')      # PAACB_LIB: A/B timing of two builds

PAACB_OK = 0
ARCH_NIPS, ARCH_NATURE = 0, 1
MATH_FP32, MATH_TF32X3, MATH_TF32, MATH_BF16X3 = 0, 1, 2, 3
CLIP_IGNORE, CLIP_GLOBAL = 0, 1
BWD_ALL, BWD_TAIL, BWD_HEAD = 0, 1, 2
MAX_ACTIONS = 18

_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); must list every symbol include/paacb.h declares (tests check this).
PROTOTYPES = {
    'paacb_version': (_i, []),
    'paacb_last_error': (C.c_char_p, []),
    'paacb_create': (_i, [C.POINTER(_vp), _i, _i, _i]),
    'paacb_destroy': (_i, [_vp]),
    'paacb_set_math': (_i, [_vp, _i]),
    'paacb_get_math': (_i, [_vp]),
    'paacb_set_sm_reserve': (_i, [_vp, _i]),
    'paacb_set_resize_tables': (_i, [_vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'paacb_param_count': (_i64, [_vp]),
    'paacb_num_tensors': (_i, [_vp]),
    'paacb_tensor_info': (_i, [_vp, _i, C.c_char_p, _i, C.POINTER(_i64), C.POINTER(_i), C.POINTER(_i64 * 4),
                               C.POINTER(_i64)]),
    'paacb_forward_workspace_floats': (_i64, [_vp, _i64]),
    'paacb_backward_workspace_floats': (_i64, [_vp, _i64]),
    'paacb_optimizer_workspace_floats': (_i64, [_vp]),
    'paacb_preprocess_u8': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i64, _vp]),
    'paacb_policy_forward': (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'paacb_params_changed': (_i, [_vp]),
    'paacb_backward_part': (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    'paacb_grad_tail_offset': (_i64, [_vp]),
    'paacb_policy_forward_at': (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    'paacb_returns_loss_grad': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _d, _f,
                                     _vp, _vp, _vp, _vp, _vp, _vp]),
    'paacb_backward': (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    'paacb_clip_rmsprop': (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _f, _f, _i, _vp, _vp, _vp]),
    'paacb_observe_u8': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i, _vp]),
    'paacb_policy_forward_sample': (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, C.c_uint64, _i64, _vp, _vp, _vp]),
    'paacb_rng_advance': (_i, [_vp, _vp, C.c_uint64, _vp]),
    'paacb_clip_rmsprop_dlr': (_i, [_vp, _vp, _vp, _vp, _vp, _f, _vp, _f, _f, _f, _f, _i, _vp, _vp, _vp]),
    'paacb_grad_stats': (_i, [_vp, _vp, _f, _vp, _vp, _vp]),
    'paacb_launch_count': (_i64, [_vp]),
    'paacb_profile_enable': (_i, [_vp, _i]),
    'paacb_profile_reset': (_i, [_vp]),
    'paacb_profile_slots': (_i, []),
    'paacb_profile_read': (_i, [_vp, _i, C.c_char_p, _i, C.POINTER(_d), C.POINTER(_i64)]),
    'paacb_host_register': (_i, [_vp, C.c_size_t, C.POINTER(_vp)]),
    'paacb_host_unregister': (_i, [_vp]),
}

_lib = None


class PaacbError(RuntimeError):
    pass


def load():
    """Load libpaacb.so (once).  Raises PaacbError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PaacbError('%s not found: build it with `python -m paac_b200.build` '
                         '(there is no CPU fallback for this path)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    if lib.paacb_version() < 102:
        raise PaacbError('libpaacb.so is stale (version %d); rebuild' % lib.paacb_version())
    _lib = lib
    return lib


def check(rc, what=''):
    if rc < 0:
        msg = load().paacb_last_error()
        raise PaacbError('%s failed (%d): %s' % (what or 'paacb call', rc, msg.decode() if msg else ''))
    return rc


def ptr(t):
    """Raw address of a torch tensor (or None)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())
