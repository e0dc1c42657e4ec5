"""ctypes binding of libmlbp.so (include/mlbp.h).  Fails loudly: no library or no sm_100 device -> exception."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libmlbp.so')

_P, _I, _L, _F = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float

# name -> argument codes (p pointer, i int, l int64, f float); every function returns int unless noted
_SIGNATURES = {
    'mlbp_pointwise_multiply_f64': 'ppplp',
    'mlbp_normalize_f64': 'pplpp',
    'mlbp_dense_dot_f64': 'pppiiip',
    'mlbp_dense_pointwise_multiply_f64': 'ppplp',
    'mlbp_build_pairwise_tables': 'ppiipiplipi' + 'pp' + 'p',
    'mlbp_build_unary_tables': 'ppiiippp',
    'mlbp_unary_stats': 'ipppppppppppppiipppppp',
    'mlbp_unary_products': 'ippppppppppiippplii' + 'ppp',
    'mlbp_fill_uniform_rows': 'ppiipipp',
    'mlbp_var_to_factor': 'ippppppp' + 'ppii' + 'ppif' + 'p',
    'mlbp_spike_scan': 'ppii' + 'iif' + 'ppppp' + 'p',
    'mlbp_spike_correct': 'ppppp' + 'ii' + 'ppii' + 'plif' + 'ppf' + 'p',
    'mlbp_topk_mask_rows': 'ppiiliip',
    'mlbp_topk_rows': 'piiiipppp',
    'mlbp_format_log_rows': 'piiiplpp',
    'mlbp_parse_float_text': 'plli' + 'lpl' + 'ppip' + 'p',
    'mlbp_factor_to_var_gemm': 'pplii' + 'ppii' + 'plifip',
    'mlbp_factor_to_var_gemm_gated': 'pplii' + 'ppii' + 'plifi' + 'pi' + 'ii' + 'f' + 'p',
    'mlbp_marginals': 'ipppp' + 'ppii' + 'ppppf' + 'iff' + 'ppppp' + 'p',
    'mlbp_rescore_candidates': 'ippp' + 'pppp' + 'ppii' + 'pppl' + 'pii' + 'ppff' + 'f' + 'ppp' + 'p',
    'mlbp_zero_words': 'pip',
    'mlbp_pair_expectations': 'ippppp' + 'pppii' + 'p' + 'ppppp' + 'plf' + 'p',
    'mlbp_gradient_reduce': 'ippppppp' + 'p' + 'ppi' + 'pppp',
    'mlbp_batch_reduce': 'ippipppp',
    'mlbp_const_rows': 'piipp',
    'mlbp_joint_logp': 'ii' + 'ppp' + 'pppp' + 'pppp' + 'ppppii' + 'ppi' + 'pi' + 'pp' + 'p',
    'mlbp_factor_to_var_maxprod': 'ppliii' + 'ppiii' + 'pi' + 'pli' + 'p',
    'mlbp_assignment_score': 'iii' + 'pppppppp' + 'pppppppp' + 'pp' + 'ii' + 'ppp' + 'p',
    'mlbp_gibbs_sample': 'iii' + 'pppppppp' + 'l' + 'iii' + 'p' + 'iii' + 'lf' + 'pp' + 'p',
    'mlbp_gibbs_reduce': 'iiipiip' + 'ppppp' + 'p',
    'mlbp_pseudo_likelihood': 'iii' + 'ppppp' + 'pppppp' + 'ppp' + 'pp' + 'l' + 'iii' + 'p' + 'pppp' + 'i' + 'f' + 'ppppp' + 'p',
    'mlbp_plan_compile': 'ipppppp' + 'iip',
    'mlbp_plan_sizes': 'pp',
    'mlbp_plan_export': 'pp',
}
_CODE = {'p': _P, 'i': _I, 'l': _L, 'f': _F}

_lib = None


class MlbpError(RuntimeError):
    pass


def load():
    """Load libmlbp.so (built by macaronicusermodeling_b200.build / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MlbpError('libmlbp.so is not built (run `python -m macaronicusermodeling_b200.build`); '
                        'this package has no CPU fallback')
    lib = ctypes.CDLL(LIB_PATH)
    for name, codes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = [_CODE[c] for c in codes]
        fn.restype = _I
    lib.mlbp_last_error.restype = ctypes.c_char_p
    lib.mlbp_last_error.argtypes = []
    lib.mlbp_version.restype = _I
    lib.mlbp_device_ok.restype = _I
    lib.mlbp_gemm_barrier_timeout_code.restype = _I
    lib.mlbp_plan_destroy.argtypes = [_P]
    lib.mlbp_plan_destroy.restype = None
    _lib = lib
    return lib


def exported_symbols():
    """Every symbol include/mlbp.h declares (used by the CPU-side ABI test)."""
    return sorted(list(_SIGNATURES) + ['mlbp_last_error', 'mlbp_version', 'mlbp_device_ok', 'mlbp_plan_destroy',
                                       'mlbp_debug_k3_times', 'mlbp_gemm_barrier_timeout_code'])


def require_device():
    lib = load()
    if not lib.mlbp_device_ok():
        raise MlbpError('no sm_100 (B200) CUDA device visible: the LBP hot path runs only on the GPU, there is no CPU fallback')
    return lib


def check(rc):
    if rc != 0:
        raise MlbpError('libmlbp error %d: %s' % (rc, load().mlbp_last_error().decode()))


def call(name, *args):
    check(getattr(load(), name)(*args))
