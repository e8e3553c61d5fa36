"""ctypes binding of ``libjamie_b200.so`` (C ABI in ``include/jamie_b200.h``).

There is no CPU fallback: if the shared library is missing or fails to load, importing the engine raises.  The library
is built in-tree by ``__graft_entry__.build()`` (``nvcc -gencode arch=compute_100a,code=sm_100a``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libjamie_b200.so')


class JbConfig(C.Structure):
    _fields_ = [
        ('dims', C.c_int * 2),
        ('latent', C.c_int),
        ('max_batch', C.c_int),
        ('dropout', C.c_float),
        ('lr', C.c_float),
        ('beta1', C.c_float),
        ('beta2', C.c_float),
        ('adam_eps', C.c_float),
        ('max_grad_norm', C.c_float),
        ('loss_w', C.c_float * 4),
        ('pf_ratio', C.c_float),
        ('seed', C.c_ulonglong),
        ('device', C.c_int),
        ('world_size', C.c_int),
    ]


_P = C.c_void_p
_LL = C.c_longlong
_FP = C.POINTER(C.c_float)

# name -> (restype, argtypes); every symbol declared in include/jamie_b200.h
SIGNATURES = {
    'jb_last_error': (C.c_char_p, []),
    'jb_version': (C.c_int, []),
    'jb_create': (C.c_int, [C.POINTER(JbConfig), C.POINTER(_P)]),
    'jb_destroy': (None, [_P]),
    'jb_num_params': (_LL, [_P]),
    'jb_num_bn_floats': (_LL, [_P]),
    'jb_set_params': (C.c_int, [_P, _P, _LL]),
    'jb_get_params': (C.c_int, [_P, _P, _LL]),
    'jb_set_bn_stats': (C.c_int, [_P, _P, _LL, _P]),
    'jb_get_bn_stats': (C.c_int, [_P, _P, _LL, _P]),
    'jb_get_grads': (C.c_int, [_P, _P, _LL]),
    'jb_get_adam_state': (C.c_int, [_P, _P, _P, _LL, C.POINTER(_LL)]),
    'jb_set_adam_state': (C.c_int, [_P, _P, _P, _LL, _LL]),
    'jb_set_dataset': (C.c_int, [_P, C.c_int, _P, _LL, _LL, C.c_int, _P]),
    'jb_set_prior_diag': (C.c_int, [_P, _P, _LL]),
    'jb_set_prior_dense': (C.c_int, [_P, _P, _LL, _LL]),
    'jb_set_f_dense': (C.c_int, [_P, _P, _LL, _LL]),
    'jb_upload_plan': (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, _P]),
    'jb_inject_randomness': (C.c_int, [_P, _P, _P, C.POINTER(_P), _P]),
    'jb_train_steps': (C.c_int, [_P, C.c_int, _P]),
    'jb_step_backward': (C.c_int, [_P, _P]),
    'jb_step_update': (C.c_int, [_P, _P]),
    'jb_grad_buffer': (C.c_int, [_P, C.POINTER(_P), C.POINTER(_LL)]),
    'jb_set_grad_buffer': (C.c_int, [_P, _P, _LL]),
    'jb_set_exchange': (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P), C.POINTER(_P), _P]),
    'jb_exchange_scratch_bytes': (_LL, []),
    'jb_set_grad_accumulate': (C.c_int, [_P, C.c_int]),
    'jb_set_dist_method': (C.c_int, [_P, C.c_int]),
    'jb_pca_colsum': (C.c_int, [_P, _P, _LL, _LL, _P, C.c_int, _P]),
    'jb_pca_gram': (C.c_int, [_P, _P, _LL, _LL, _P, _P, C.c_int, _P]),
    'jb_metric_foscttm': (C.c_int, [_P, _P, _LL, C.c_int, C.c_int, C.POINTER(C.c_ulonglong)]),
    'jb_metric_knn_vote': (C.c_int, [_P, _LL, _P, _P, _LL, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    'jb_metric_feature_pearson': (C.c_int, [_P, _P, _LL, _LL, C.c_int, _P]),
    'jb_metric_feature_auroc': (C.c_int, [_P, _LL, _LL, _P, _P, _LL, C.c_int, _P, _P]),
    'jb_knn': (C.c_int, [_P, _LL, _P, _LL, C.c_int, C.c_int, _LL, C.c_int, _P, _P]),
    'jb_knn_average': (C.c_int, [_P, _P, _LL, C.c_int, _P, _LL, _LL, _LL, _LL, C.c_int, _P]),
    'jb_silhouette': (C.c_int, [_P, _LL, C.c_int, _P, C.c_int, _LL, C.c_int, _P, _P]),
    'jb_dist_create': (C.c_int, [_LL, C.c_int, C.POINTER(_P)]),
    'jb_dist_destroy': (None, [_P]),
    'jb_dist_accumulate': (C.c_int, [_P, C.c_int, _P, _LL, _LL]),
    'jb_dist_finish': (C.c_int, [_P, C.c_int, _P]),
    'jb_dist_knn': (C.c_int, [_P, C.c_int, _P, _P]),
    'jb_dist_geodesic': (C.c_int, [_P, C.c_int, _P]),
    'jb_pcaop_create_dense': (C.c_int, [_P, _LL, _LL, C.c_int, C.POINTER(_P)]),
    'jb_pcaop_create_sparse': (C.c_int, [_LL, _LL, _LL, _P, _P, _P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    'jb_pcaop_stats': (C.c_int, [_P, _P, _P]),
    'jb_pcaop_apply': (C.c_int, [_P, C.c_int, _P, C.c_int, _P, _P]),
    'jb_pcaop_destroy': (None, [_P]),
    'jb_train_step_hostbatch': (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, _P, _P]),
    'jb_step_backward_hostbatch': (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, _P]),
    'jb_hostbatch_submit': (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, _P]),
    'jb_hostbatch_wait': (C.c_int, [_P, _P]),
    'jb_num_phases': (C.c_int, []),
    'jb_phase_name': (C.c_char_p, [C.c_int]),
    'jb_bench_stage': (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_double), _P]),
    'jb_profile_step': (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(C.c_int), _P]),
    'jb_profile_detail': (C.c_int, [_P, _P, C.c_int]),
    'jb_read_losses': (C.c_int, [_P, _P, C.c_int, _P]),
    'jb_encode': (C.c_int, [_P, C.c_int, _P, _LL, _LL, _P, _LL, C.c_int, _P]),
    'jb_predict': (C.c_int, [_P, C.c_int, C.c_int, _P, _LL, _LL, _P, _LL, C.c_int, _P]),
    'jb_pca_project': (C.c_int, [_P, _P, _LL, _LL, _P, _P, C.c_int, C.c_float, C.c_float, _P, C.c_int, _P]),
    'jb_pca_inverse': (C.c_int, [_P, _P, _LL, C.c_int, _P, _P, _LL, C.c_float, C.c_float, _P, C.c_int, _P]),
    'jb_feature_impact': (C.c_int, [_P, C.c_int, C.c_int, _P, _LL, _LL, _P, _P, _P, C.c_int, _P, _P, C.c_float, C.c_float,
                                    _P, _P, _LL, _P, _P, _P, _P, _LL, _P]),
    'jb_shapley': (C.c_int, [_P, C.c_int, C.c_int, _P, _LL, _P, _LL, _LL, _P, _P, _LL, _P, _P, C.c_int, _P, _P, C.c_float,
                             C.c_float, _P, _P, _P, _LL, _P, _P, _P, _LL, _P]),
    'jb_debug_read': (_LL, [_P, C.c_char_p, _P, _LL]),
    'jb_launch_count': (_LL, [_P]),
}

_lib = None


def load():
    """Loads the shared library (once) and attaches the signatures. Raises if it is missing: no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a). jamie_b200 has no CPU or PyTorch fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().jb_last_error()
        raise RuntimeError('jamie_b200: ' + (msg.decode() if msg else f'error {rc}'))
