"""ctypes binding of librw_b200.so (see include/rewriting_b200.h).

The product path has no CPU fallback: if the shared library is missing or an
entry point fails, the caller gets an exception.  (The CPU oracle lives in
/oracle and is only ever imported by tests, smoke() and the bench baseline.)
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('RW_LIB') or os.path.join(_HERE, 'librw_b200.so')

c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_f = ctypes.c_float
c_p = ctypes.c_void_p
c_sz = ctypes.c_size_t


class RwError(RuntimeError):
    pass


class InsertArgs(ctypes.Structure):
    """Mirror of `rw_insert_args`."""
    _fields_ = [
        ('W', c_p), ('m', c_p), ('v', c_p), ('w_ortho', c_p), ('d', c_p),
        ('key_cl', c_p), ('style', c_p), ('target', c_p), ('noise', c_p),
        ('bias', c_p), ('loss_out', c_p),
        ('noise_w', c_f), ('lr', c_f), ('beta1', c_f), ('beta2', c_f), ('eps', c_f),
        ('rank', c_int), ('B', c_int), ('Cin', c_int), ('Cout', c_int),
        ('h', c_int), ('w', c_int), ('has_noise_act', c_int),
        ('it0', c_int), ('nsteps', c_int), ('niter_total', c_int),
        ('piter', c_int), ('project_gradient', c_int),
        ('plain_conv', c_int), ('one_minus_beta1', c_f), ('one_minus_beta2', c_f),
        ('beta1_exact', ctypes.c_double), ('beta2_exact', ctypes.c_double),
    ]


# name -> (restype, argtypes); every symbol include/rewriting_b200.h declares
SIGNATURES = {
    'rw_version': (c_int, []),
    'rw_last_error': (ctypes.c_char_p, []),
    'rw_set_device': (c_int, [c_int]),
    'rw_device_sm_count': (c_int, []),
    'rw_prep_keys': (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p]),
    'rw_split_rows': (c_int, [c_p, c_ll, c_p, c_p, c_p]),
    'rw_prep_weights': (c_int, [c_p, c_int, c_int, c_f, c_int, c_int, c_p, c_p, c_p, c_p]),
    'rw_demod': (c_int, [c_p, c_p, c_int, c_int, c_int, c_f, c_p, c_p]),
    'rw_modconv_fwd': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_int,
                               c_int, c_int, c_int, c_int, c_int, c_p, c_p]),
    'rw_modconv_up_fwd': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_int,
                                  c_p, c_p]),
    'rw_modconv_fwd_fused': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_int,
                                     c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p,
                                     c_p, c_p, c_p]),
    'rw_modconv_rgb_parts': (c_int, [c_int]),
    'rw_modconv_up_fwd_cl': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_int,
                                     c_p, c_p]),
    'rw_modconv_up_fused': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_p, c_p, c_p,
                                    c_int, c_int, c_int, c_int, c_int, c_p]),
    'rw_modconv_up_fused_y': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_int, c_p,
                                      c_int, c_int, c_int, c_int, c_int, c_p]),
    'rw_debug_upconv_taps': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_p, c_p,
                                     c_int, c_int, c_int, c_int, c_int, c_p, c_p]),
    'rw_rowgemm': (c_int, [c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p]),
    'rw_pixel_norm_nchw': (c_int, [c_p, c_int, c_int, c_int, c_int, c_int, c_p, c_p]),
    'rw_nearest_up2': (c_int, [c_p, c_ll, c_int, c_int, c_p, c_p]),
    'rw_conv3x3_bias_act': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_f, c_int, c_int, c_int, c_int,
                                    c_int, c_p, c_p]),
    'rw_debug_upconv_profile': (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_ll, c_p, c_p, c_p, c_p,
                                        c_p, c_int, c_int, c_int, c_int, c_int, c_p, c_p]),
    'rw_blur_up_fused': (c_int, [c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_ll, c_p, c_p,
                                 c_int, c_p, c_p, c_p, c_p, c_p]),
    'rw_styles': (c_int, [c_p, c_int, c_int, c_int, c_f, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    'rw_equal_linear': (c_int, [c_p, c_int, c_int, c_p, c_p, c_int, c_f, c_f, c_int, c_p, c_p]),
    'rw_pixel_norm': (c_int, [c_p, c_int, c_int, c_p, c_p]),
    'rw_demod_multi': (c_int, [c_int, c_f, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    'rw_rgb_combine': (c_int, [c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p]),
    'rw_rgb_combine_u8': (c_int, [c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    'rw_blur_up_act': (c_int, [c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_ll, c_p, c_p,
                               c_int, c_p, c_p]),
    'rw_add_noise': (c_int, [c_p, c_p, c_ll, c_p, c_int, c_int, c_int, c_p, c_p]),
    'rw_torgb': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_f, c_p, c_p]),
    'rw_fused_bias_act': (c_int, [c_p, c_p, c_p, c_int, c_int, c_f, c_f, c_ll, c_int, c_int,
                                  c_p, c_p]),
    'rw_upfirdn2d': (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                             c_int, c_int, c_int, c_int, c_int, c_p, c_int, c_int, c_p]),
    'rw_gram_workspace_bytes': (c_sz, [c_int, c_int, c_ll, c_int]),
    'rw_second_moment_accum': (c_int, [c_p, c_p, c_ll, c_int, c_p, c_p, c_sz, c_p]),
    'rw_conv_wgrad': (c_int, [c_p, c_p, c_p, c_p, c_ll, c_int, c_int, c_int, c_p, c_p, c_sz,
                              c_p]),
    'rw_prep_phase_keys': (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_p]),
    'rw_modconv_up_dgrad': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_int,
                                    c_p, c_p]),
    'rw_conv_up_wgrad': (c_int, [c_p, c_p, c_p, c_p, c_ll, c_int, c_int, c_int, c_p, c_p, c_sz,
                                 c_p]),
    'rw_act_grad_reduce': (c_int, [c_p, c_p, c_p, c_ll, c_p, c_p, c_int, c_int, c_int, c_int,
                                   c_p, c_p, c_p, c_p, c_p]),
    'rw_blur_adj_phase_keys': (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_p]),
    'rw_dgrad_finish': (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p]),
    'rw_wgrad_finish': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_f, c_p, c_p]),
    'rw_style_grad_finish': (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p]),
    'rw_project_rank': (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_f, c_p, c_p]),
    'rw_insert_loop': (c_int, [ctypes.POINTER(InsertArgs), c_p]),
    'rw_debug_rowgemm': (c_int, [c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p]),
    'rw_debug_colgemm': (c_int, [c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_int, c_p,
                                 c_p, c_sz, c_p]),
}

_lib = None


def load():
    """Load the shared library (once) and attach prototypes.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RwError(
            'librw_b200.so is not built (expected %s). Run `python -m rewriting_b200.build` '
            'or __graft_entry__.build(); there is no CPU fallback.' % LIB_PATH)
    # torch loads libcudart.so.12 first so that the library shares torch's CUDA
    # runtime (current device, primary context, streams).
    import torch  # noqa: F401
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    lib = load()
    msg = lib.rw_last_error()
    return msg.decode('utf-8', 'replace') if msg else ''


def check(rc, what):
    if rc != 0:
        raise RwError('%s failed (status %d): %s' % (what, rc, last_error()))


# kernels launched per entry point (for bench.py's `gpu_launches` claim)
LAUNCHES_PER_CALL = {
    'rw_second_moment_accum': 2, 'rw_conv_wgrad': 2, 'rw_conv_up_wgrad': 2,
    'rw_debug_colgemm': 2,
}
launch_count = 0


_FN = {}


def call(name, *args):
    """Invoke an int-returning entry point and raise RwError on a non-zero status."""
    global launch_count
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(load(), name)
    rc = fn(*args)
    if rc != 0:
        check(rc, name)
    launch_count += LAUNCHES_PER_CALL.get(name, 1)
