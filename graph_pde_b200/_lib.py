"""ctypes binding of libnnconv_b200.so (C ABI declared in include/nnconv_b200.h).

The product path has NO fallback: if the shared library is missing or the device is not sm_100-class,
importing / calling raises.  `build()` compiles the library in-tree with nvcc (sm_100a only).
"""
import ctypes
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnnconv_b200.so')
CSRC = os.path.join(_HERE, 'csrc')

OK = 0
ABI_VERSION = 2        # include/nnconv_b200.h: NNCONV_B200_ABI_VERSION this binding was written against
PREC = {'fp32': 0, 'f16': 1, 'fp16': 1, 'bf16': 2, 'f16x2': 3}
AGGR = {'add': 0, 'mean': 1}
APPLY_RELU_IN, APPLY_RESIDUAL = 1, 2        # include/nnconv_b200.h NNCONV_APPLY_*
FLOW = {'source_to_target': 0, 'target_to_source': 1}

# every symbol include/nnconv_b200.h declares (tests/test_cabi_symbols.py checks the .so exports them)
SYMBOLS = [
    'nnconv_last_error', 'nnconv_abi_version', 'nnconv_init', 'nnconv_plan_sizes', 'nnconv_plan_create',
    'nnconv_plan_destroy', 'nnconv_plan_info', 'nnconv_weights_sizes', 'nnconv_weights_create',
    'nnconv_weights_destroy', 'nnconv_weights_tc_supported', 'nnconv_edge_features_sizes',
    'nnconv_edge_features', 'nnconv_apply_sizes', 'nnconv_apply', 'nnconv_gemm_16b',
    'nnconv_profile_begin', 'nnconv_profile_end', 'nnconv_debug_trace_dump',
    'nnconv_backward_sizes', 'nnconv_backward',
    'nnconv_set_option', 'nnconv_get_option', 'nnconv_edge_features_overflow', 'nnconv_debug_occupy',
    'nnconv_backward_tc_supported', 'nnconv_backward_apply_sizes', 'nnconv_backward_apply',
    'nnconv_backward_mlp_sizes', 'nnconv_backward_mlp', 'nnconv_gemm_tn_16b', 'nnconv_gemm_16b_ex',
    'nnconv_halo_push', 'nnconv_halo_wait', 'nnconv_enable_peer_access', 'nnconv_loss_epilogue',
    'nnconv_ipc_alloc', 'nnconv_ipc_open', 'nnconv_ipc_close', 'nnconv_ipc_free',
    'nnconv_ball_count', 'nnconv_ball_fill',
    'nnconv_edge_kernels_sizes', 'nnconv_edge_kernels', 'nnconv_apply_edge',
    'nnconv_edge_acts_sizes', 'nnconv_edge_features_keep', 'nnconv_apply_ex', 'nnconv_apply_edge_ex',
]


class NNConvLibraryError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libnnconv_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ['make', '-C', CSRC, '-j', str(min(8, os.cpu_count() or 1))]
    if shutil.which('nvcc') is None:      # an account whose PATH lacks the CUDA toolkit's bin directory
        cmd.append('NVCC=' + os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'bin', 'nvcc'))
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise NNConvLibraryError('building libnnconv_b200.so failed (see output above)')
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NNConvLibraryError(
            '%s not found: run `python -c "import __graft_entry__ as g; g.build()"` (or make -C %s). '
            'There is no CPU/PyTorch fallback for the NNConv path.' % (LIB_PATH, CSRC))
    L = ctypes.CDLL(LIB_PATH)
    c_i64, c_sz, c_vp, c_int = ctypes.c_int64, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int
    P = ctypes.POINTER
    L.nnconv_last_error.restype = ctypes.c_char_p
    L.nnconv_last_error.argtypes = []
    L.nnconv_abi_version.restype = c_int
    L.nnconv_init.restype = c_int
    L.nnconv_plan_sizes.argtypes = [c_i64, c_i64, P(c_sz), P(c_sz)]
    L.nnconv_plan_create.argtypes = [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_sz, c_vp, c_sz, c_vp, P(c_vp)]
    L.nnconv_plan_destroy.argtypes = [c_vp]
    L.nnconv_plan_destroy.restype = None
    L.nnconv_plan_info.argtypes = [c_vp, P(c_i64), c_int]
    L.nnconv_weights_sizes.argtypes = [c_int, P(c_int), c_int, c_int, c_int, P(c_sz)]
    L.nnconv_weights_create.argtypes = [c_int, P(c_int), c_int, c_int, c_int, P(c_vp), P(c_vp), c_vp, c_sz, c_vp,
                                        P(c_vp)]
    L.nnconv_weights_destroy.argtypes = [c_vp]
    L.nnconv_weights_destroy.restype = None
    L.nnconv_weights_tc_supported.argtypes = [c_vp]
    L.nnconv_edge_features_sizes.argtypes = [c_vp, c_vp, c_sz, P(c_sz), P(c_sz)]
    L.nnconv_edge_features.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp, P(c_i64)]
    L.nnconv_apply_sizes.argtypes = [c_vp, c_vp, c_sz, P(c_sz)]
    L.nnconv_apply.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_sz, c_vp, P(c_i64)]
    L.nnconv_gemm_16b.argtypes = [c_int, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_vp]
    L.nnconv_profile_end.argtypes = [P(ctypes.c_double), P(c_i64), c_int]
    L.nnconv_backward_sizes.argtypes = [c_vp, c_vp, c_sz, P(c_sz)]
    L.nnconv_backward.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, P(c_vp), P(c_vp), c_vp, c_vp, c_vp,
                                  c_sz, c_vp]
    L.nnconv_debug_trace_dump.argtypes = [P(ctypes.c_ulonglong), ctypes.c_uint, P(ctypes.c_uint)]
    L.nnconv_set_option.argtypes = [ctypes.c_char_p, c_int]
    L.nnconv_get_option.argtypes = [ctypes.c_char_p, P(c_int)]
    L.nnconv_edge_features_overflow.argtypes = [c_vp, c_vp, P(c_i64)]
    L.nnconv_debug_occupy.argtypes = [c_int, c_int, ctypes.c_longlong, c_vp]
    L.nnconv_backward_tc_supported.argtypes = [c_vp]
    L.nnconv_backward_apply_sizes.argtypes = [c_vp, c_vp, c_sz, P(c_sz)]
    L.nnconv_backward_apply.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                        c_sz, c_vp]
    L.nnconv_backward_mlp_sizes.argtypes = [c_vp, c_vp, c_int, c_sz, P(c_sz)]
    L.nnconv_backward_mlp.argtypes = [c_vp, c_vp, c_vp, c_vp, c_int, P(c_vp), P(c_vp), c_int, P(c_vp), P(c_vp), c_vp,
                                      c_sz, c_vp, c_vp]
    L.nnconv_edge_acts_sizes.argtypes = [c_vp, c_vp, P(c_sz)]
    L.nnconv_edge_features_keep.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp, P(c_i64)]
    L.nnconv_halo_push.argtypes = [c_vp, c_int, c_i64, c_int, c_i64, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64,
                                   c_i64, c_i64, c_vp, c_vp, c_int, c_vp]
    L.nnconv_halo_wait.argtypes = [c_vp, c_vp, c_int, c_vp]
    L.nnconv_enable_peer_access.argtypes = [c_int]
    L.nnconv_ipc_alloc.argtypes = [c_sz, P(c_vp), ctypes.c_char_p]
    L.nnconv_ipc_open.argtypes = [ctypes.c_char_p, P(c_vp)]
    L.nnconv_ipc_close.argtypes = [c_vp]
    L.nnconv_ipc_free.argtypes = [c_vp]
    L.nnconv_edge_kernels_sizes.argtypes = [c_vp, c_vp, P(c_sz)]
    L.nnconv_edge_kernels.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp]
    L.nnconv_apply_edge.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]
    L.nnconv_apply_edge_ex.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, ctypes.c_uint, c_vp, c_vp]
    L.nnconv_apply_ex.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, ctypes.c_uint, c_vp, c_vp, c_sz, c_vp, P(c_i64)]
    L.nnconv_ball_count.argtypes = [c_vp, c_i64, c_vp, c_i64, ctypes.c_double, c_vp, c_vp]
    L.nnconv_ball_fill.argtypes = [c_vp, c_i64, c_vp, c_i64, ctypes.c_double, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp]
    L.nnconv_loss_epilogue.argtypes = [c_vp, c_vp, c_vp, c_vp, ctypes.c_float, c_int, c_i64, ctypes.c_float, c_vp, c_vp,
                                       c_vp, c_vp]
    L.nnconv_gemm_tn_16b.argtypes = [c_int, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_i64, ctypes.c_float,
                                     c_vp]
    L.nnconv_gemm_16b_ex.argtypes = [c_int, c_vp, c_i64, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_i64, c_vp, c_i64, c_int,
                                     c_vp]
    for name in SYMBOLS:
        getattr(L, name)
    if L.nnconv_abi_version() != ABI_VERSION:
        raise NNConvLibraryError('%s has ABI version %d, this binding needs %d: rebuild it (make -C %s)'
                                 % (LIB_PATH, L.nnconv_abi_version(), ABI_VERSION, CSRC))
    _lib = L
    return L


def check(status):
    if status != OK:
        msg = lib().nnconv_last_error()
        raise NNConvLibraryError('libnnconv_b200 error %d: %s' % (status, msg.decode() if msg else '?'))


def set_option(name, value):
    """Tuning / debugging knob of the library (csrc/options.h); value=None restores the built-in default."""
    check(lib().nnconv_set_option(name.encode(), -2000000 if value is None else int(value)))


def get_option(name):
    v = ctypes.c_int(0)
    check(lib().nnconv_get_option(name.encode(), ctypes.byref(v)))
    return v.value
