"""ctypes binding of libhorizonnet_b200.so (include/horizonnet_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
RuntimeError is raised (the product path never routes through torch ops or the CPU oracle)."""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libhorizonnet_b200.so')
ABI_VERSION = 2

_lib = None
_lock = threading.Lock()

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
vp = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/horizonnet_b200.h one to one
SIGNATURES = {
    'hn_last_error': (ctypes.c_char_p, []),
    'hn_abi_version': (ctypes.c_int, []),
    'hn_build_digest': (ctypes.c_char_p, []),
    'hn_kernel_launches': (ctypes.c_longlong, []),
    'hn_model_create': (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp)]),
    'hn_model_num_tensors': (ctypes.c_int, [vp]),
    'hn_model_tensor_info': (ctypes.c_int, [vp, ctypes.c_int, ctypes.POINTER(ctypes.c_char_p),
                                            ctypes.POINTER(ctypes.c_longlong)]),
    'hn_model_set_tensor': (ctypes.c_int, [vp, ctypes.c_char_p, vp, ctypes.c_longlong, ctypes.c_int]),
    'hn_model_finalize': (ctypes.c_int, [vp]),
    'hn_model_forward': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    'hn_model_forward_async': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    'hn_model_flush': (ctypes.c_int, [vp, vp]),
    'hn_model_num_bn': (ctypes.c_int, [vp]),
    'hn_model_bn_name': (ctypes.c_char_p, [vp, ctypes.c_int]),
    'hn_model_forward_train': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int,
                                              ctypes.c_ulonglong, ctypes.c_double, ctypes.c_double, vp, vp, vp]),
    'hn_train_forward': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int,
                                        ctypes.c_ulonglong, ctypes.c_double, ctypes.c_double, vp, vp, vp]),
    'hn_train_backward': (ctypes.c_int, [vp, vp, vp, vp]),
    'hn_model_get_grad': (ctypes.c_int, [vp, ctypes.c_char_p, vp, ctypes.c_longlong, vp]),
    'hn_conv2d_backward': (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
                           + [ctypes.c_int] * 7 + [vp, vp, vp]),
    'hn_conv2d_wgrad_tc': (ctypes.c_int, [vp] + [ctypes.c_int] * 4 + [vp] + [ctypes.c_int] * 7 + [vp, vp]),
    'hn_wgrad_tc_plan': (ctypes.c_int, [ctypes.c_int] * 12 + [c_int_p]),
    'hn_wgrad_tc_enabled': (ctypes.c_int, []),
    'hn_bn_forward_backward': (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp,
                                              ctypes.c_double, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                              vp]),
    'hn_lstm_layer_backward': (ctypes.c_int, [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    'hn_train_profile': (ctypes.c_int, [vp, ctypes.POINTER(ctypes.c_double)]),
    'hn_train_profile_units': (ctypes.c_int, [vp, ctypes.POINTER(ctypes.c_double)]),
    'hn_train_debug_unit': (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_longlong, c_int_p, ctypes.c_char_p,
                                           ctypes.c_int, vp]),
    'hn_dropout_mask': (ctypes.c_int, [ctypes.c_ulonglong, ctypes.c_int, ctypes.c_double, vp, ctypes.c_longlong, vp]),
    'hn_model_get_tensor': (ctypes.c_int, [vp, ctypes.c_char_p, vp, ctypes.c_longlong, ctypes.c_int, vp]),
    'hn_model_forward_host': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp]),
    'hn_model_submit_host': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int]),
    'hn_model_collect_host': (ctypes.c_int, [vp, vp, vp]),
    'hn_model_infer_tta': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, c_int_p, ctypes.c_int, vp, vp, vp]),
    'hn_layout_workspace_bytes': (ctypes.c_longlong, [ctypes.c_int]),
    'hn_layout': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int] + [vp] * 8),
    'hn_model_infer_layout': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, c_int_p, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_float, ctypes.c_int] + [vp] * 10),
    'hn_model_stage': (ctypes.c_int, [vp, ctypes.c_char_p, vp, ctypes.c_longlong, c_int_p, vp]),
    'hn_model_set_option': (ctypes.c_int, [vp, ctypes.c_char_p, ctypes.c_int]),
    'hn_model_check': (ctypes.c_int, [vp]),
    'hn_model_profile_read': (ctypes.c_int, [vp, c_double_p, c_double_p, ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]),
    'hn_model_destroy': (None, [vp]),
    'hn_pano_stretch': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       c_double_p, c_double_p, ctypes.c_int, vp]),
    'hn_pano_stretch_host': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            c_double_p, c_double_p, ctypes.c_int]),
    'hn_pano_stretch_f64': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           c_double_p, c_double_p, ctypes.c_int, vp]),
    'hn_pano_stretch_host_f64': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                c_double_p, c_double_p, ctypes.c_int]),
    'hn_augment': (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p, c_double_p, c_int_p, c_int_p,
                                  c_float_p, vp]),
    'hn_rotate_panorama': (ctypes.c_int, [vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          c_double_p, vp]),
    'hn_conv2d': (ctypes.c_int, [vp] + [ctypes.c_int] * 5 + [vp, vp, vp, vp] + [ctypes.c_int] * 8 +
                  [vp, ctypes.c_int, ctypes.c_int, vp]),
    'hn_lstm_layer': (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, vp]),
}


def lib():
    """Loads the library once; raises RuntimeError (never falls back) when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                '(horizonnet_b200 has no CPU / PyTorch fallback)')
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if l.hn_abi_version() != ABI_VERSION:
            raise RuntimeError('libhorizonnet_b200 ABI version mismatch; rebuild')
        # a binary built from other sources than the ones checked out (e.g. a stale .so after `git pull`) must not run
        from . import build as _build
        have, want = l.hn_build_digest().decode(), _build.source_digest()
        if have != want:
            raise RuntimeError(f'libhorizonnet_b200.so was built from different sources (digest {have[:12]} != '
                               f'{want[:12]}); run `python -c "import __graft_entry__ as g; g.build()"`')
        _lib = l
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().hn_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'{what} failed: {msg}')
