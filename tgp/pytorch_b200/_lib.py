"""ctypes binding of `libtgp_b200.so` (the C-ABI declared in include/tgp_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('TGP_B200_LIB', os.path.join(_HERE, 'libtgp_b200.so'))
LIB_PATH = os.environ.get('TGP_B200_LIB', LIB_PATH)      # A/B builds of the same sources (scripts/, profiling)

TGP_F64, TGP_F32, TGP_F64_I8 = 0, 1, 2
LIK_GAUSS_LINEAR, LIK_GAUSS_NONLINEAR, LIK_BERNOULLI = 0, 1, 2
FLOW_IDENTITY, FLOW_AFFINE, FLOW_TANH_STEP, FLOW_SAL, FLOW_ARCSINH, FLOW_BOXCOX, FLOW_INV_BOXCOX = 0, 1, 2, 3, 4, 5, 6
FLOW_STEP_GROUP = 7
KERNEL_RBF, KERNEL_MATERN12, KERNEL_MATERN32, KERNEL_MATERN52 = 0, 1, 2, 3
QU_WHITENED, QU_UNWHITENED = 0, 1
FLOW_RESTRICT, FLOW_ADD_F0, FLOW_PER_ROW, FLOW_SWITCH = 1, 2, 4, 8
MAX_LAYERS = 64
OPT_ROW_CHUNK = 2
OPT_OVERLAP_KGEN = 3


class TgpFlowLayer(C.Structure):
    _fields_ = [('kind', C.c_int), ('flags', C.c_int), ('n_steps', C.c_int), ('p0', C.c_int)]


class TgpModel(C.Structure):
    _fields_ = [('dtype', C.c_int), ('M', C.c_int), ('D', C.c_int), ('likelihood', C.c_int), ('n_quad', C.c_int),
                ('n_theta', C.c_int), ('n_rowparams', C.c_int), ('n_layers', C.c_int),
                ('layers', TgpFlowLayer * MAX_LAYERS), ('kernel', C.c_int), ('q_u_form', C.c_int)]


class TgpParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw', 'log_var_noise',
                                          'theta')]


class TgpReduceLayout(C.Structure):
    _fields_ = [(n, C.c_long) for n in ('ell_sum', 'dlogvar', 'dos', 'dls', 'dtheta', 'dm', 'dZ', 'Gbar', 'Cbar',
                                        'total', 'packed_total')]


class TgpBatch(C.Structure):
    _fields_ = [('X', C.c_void_p), ('Y', C.c_void_p), ('rowparams', C.c_void_p), ('R', C.c_long), ('scale', C.c_double),
                ('quad_t', C.c_void_p), ('quad_w', C.c_void_p)]


class TgpFwdOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('terms', 'status', 'ell_rows', 'mu', 'v')]


class TgpGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('dZ', 'draw_lengthscale', 'draw_outputscale', 'dm', 'dL_raw', 'dlog_var_noise',
                                          'dtheta', 'drowparams', 'dX')]


class TgpMlp(C.Structure):
    _fields_ = [('n_nets', C.c_int), ('n_in', C.c_int), ('hidden', C.c_int), ('n_hidden_layers', C.c_int),
                ('activation', C.c_int), ('mask_mode', C.c_int), ('p_drop', C.c_double)]


# int (*TgpAllReduceFn)(double* buf, long count, void* user, void* stream)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p)


# name -> (restype, argtypes); the exported-symbol test walks this table against include/tgp_b200.h
_P, _I, _L, _D = C.c_void_p, C.c_int, C.c_long, C.c_double
SIGNATURES = {
    'tgp_last_error': (C.c_char_p, []),
    'tgp_version': (_I, []),
    'tgp_step_workspace_bytes': (C.c_size_t, [C.POINTER(TgpModel)]),
    'tgp_batch_workspace_bytes': (C.c_size_t, [C.POINTER(TgpModel), _L]),
    'tgp_reduce_layout': (_I, [C.POINTER(TgpModel), C.POINTER(TgpReduceLayout)]),
    'tgp_prepare': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _D, _P, _P, _P, _P]),
    'tgp_factor_status': (_I, [C.POINTER(C.c_int)]),
    'tgp_qf_forward': (_I, [C.POINTER(TgpModel), _P, _P, _P, _L, _P, _P, _P]),
    'tgp_qf_cov_workspace_bytes': (C.c_size_t, [C.POINTER(TgpModel), _L]),
    'tgp_qf_cov_forward': (_I, [C.POINTER(TgpModel), _P, _P, _P, _L, _P, _P, _L, _P]),
    'tgp_cov_cholesky_workspace_bytes': (C.c_size_t, [_L]),
    'tgp_cov_cholesky': (_I, [_L, _P, _L, _D, _P, _P, _P, _L, _P, _P]),
    'tgp_cov_sample': (_I, [_L, _I, _P, _P, _L, _P, _P, _P]),
    'tgp_ell_forward': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _P, _P, _L, _D, _P, _P, _I, _P, _P, _P,
                             _P, _P, _P]),
    'tgp_qf_backward': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _P, _L, _P, _P, _P, _P]),
    'tgp_qf_backward_dx': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _P, _L, _P, _P, _P, _P, _P]),
    'tgp_chain_backward': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _D, _D, _P, _P, _P, _P, _P, _P, _P,
                                _P, _P]),
    'tgp_test_rows': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _P, _P, _L, _I, _D, _P, _P, _P, _P, _P,
                           _P, _P]),
    'tgp_coverage_rows': (_I, [C.POINTER(TgpModel), C.POINTER(TgpParams), _P, _P, _P, _P, _L, _I, _I, C.c_ulonglong, _P, _D, _D, _P, _P,
                              _P, _P, _P, _P]),
    'tgp_mc_softmax_rows': (_I, [C.POINTER(TgpModel), _I, _I, _L, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    'tgp_mc_softmax_rows_rowp': (_I, [C.POINTER(TgpModel), _I, _I, _L, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    'tgp_reduce_pack': (_I, [C.POINTER(TgpModel), _P, _P, _P]),
    'tgp_reduce_unpack': (_I, [C.POINTER(TgpModel), _P, _P, _P]),
    'tgp_workspace_bytes': (C.c_size_t, [C.POINTER(TgpModel), _L]),
    'tgp_create': (_I, [C.POINTER(TgpModel), _L, C.POINTER(_P)]),
    'tgp_destroy': (None, [_P]),
    'tgp_bind_workspace': (_I, [_P, _P, C.c_size_t]),
    'tgp_elbo_fwd': (_I, [_P, C.POINTER(TgpParams), C.POINTER(TgpBatch), _D, C.POINTER(TgpFwdOut), _P]),
    'tgp_elbo_bwd': (_I, [_P, C.POINTER(TgpParams), C.POINTER(TgpBatch), _P, C.POINTER(TgpGrads), ALLREDUCE_FN, _P, _P]),
    'tgp_test_nll_fwd': (_I, [_P, C.POINTER(TgpParams), C.POINTER(TgpBatch), _I, _I, _D, _P, _P, _P, _P, _P, _P, _P, _P]),
    'tgp_flow_mlp_net_doubles': (_L, [C.POINTER(TgpMlp)]),
    'tgp_flow_mlp_forward': (_I, [C.POINTER(TgpMlp), _P, _P, _L, _P, _P, C.c_ulonglong, _P, _P, _P]),
    'tgp_flow_mlp_backward': (_I, [C.POINTER(TgpMlp), _P, _P, _L, _P, _P, _P, _P]),
    'tgp_flow_mlp_backward_dx': (_I, [C.POINTER(TgpMlp), _P, _P, _L, _P, _P, _P, _P, _P]),
    'tgp_adam_step': (_I, [_I, _L, _P, _P, _P, _P, _P, _P, _D, _D, _D, _P, _P]),
    'tgp_kmeans_iteration': (_I, [_P, _L, _I, _P, _I, _P, _P, _P, _P, _I, _P]),
    'tgp_set_option': (_I, [_I, _I]),
    'tgp_launch_count': (_L, []),
    'tgp_gemm_timing': (_I, [_I, C.POINTER(C.c_double), C.POINTER(C.c_long)]),
    'tgp_debug_gemm_f64': (_I, [_I, _I, _I, _P, _L, _I, _P, _L, _I, _P, _L, _D, _D, _I, _I, _I, _P]),
    'tgp_debug_gemm_tf32x3': (_I, [_I, _I, _I, _P, _P, _L, _P, _P, _L, _P, _P, _L, _I, _I, _I, _I, _I, _P]),
    'tgp_debug_gemm_crt_bytes': (C.c_size_t, [_L, _L, _L, _I]),
    'tgp_debug_gemm_crt': (_I, [_L, _L, _L, _P, _L, _P, _L, _P, _L, _I, _I, _I, _I, _I, _I, _P, _P]),
    'tgp_debug_export_step': (_I, [C.POINTER(TgpModel), _P, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Loads the shared library once; raises if it has not been built (`python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError('%s not found: build it with __graft_entry__.build(); there is no CPU fallback' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().tgp_last_error().decode()
        if rc == -1 or rc == -2:
            raise ValueError('%s: %s' % (what, msg))
        raise RuntimeError('%s failed (%d): %s' % (what, rc, msg))
