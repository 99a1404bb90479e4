"""ctypes binding of libnnb.so -- the C ABI declared in include/nnb.h.

This is exactly the stub a reference maintainer would add to nnest (see INTEGRATION.md).  There is
no fallback: if the shared library is missing or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get('NNB_LIB_DIR', 'lib'), 'libnnb.so')   # see build.py

NNB_ABI_VERSION = 14
NNB_MAX_DIM = 128
NNB_MAX_BLOCKS = 16
NNB_MAX_LIKE_PARAMS = 160
NNB_MAX_DERIVED = 32
NNB_MAX_DATA_ARRAYS = 16
NNB_DTYPE_F64, NNB_DTYPE_F32, NNB_DTYPE_I32 = 0, 1, 2

NNB_OK, NNB_ERR_ARG, NNB_ERR_CUDA, NNB_ERR_STATE, NNB_ERR_UNSUPPORTED, NNB_ERR_START = 0, -1, -2, -3, -4, -5
NNB_FLOW_TRANSLATE_ONLY, NNB_FLOW_CONST_SCALE = 1, 2
(NNB_LIKE_ROSENBROCK, NNB_LIKE_HIMMELBLAU, NNB_LIKE_GAUSSIAN, NNB_LIKE_EGGBOX, NNB_LIKE_GAUSSIAN_MIX,
 NNB_LIKE_GAUSSIAN_SHELL, NNB_LIKE_USER) = range(7)
NNB_PRIOR_NONE, NNB_PRIOR_BOX_U, NNB_PRIOR_BOX_V = 0, 1, 2
NNB_MODE_HARD, NNB_MODE_MH = 0, 1
NNB_IMPL_AUTO, NNB_IMPL_FFMA, NNB_IMPL_TCGEN05, NNB_IMPL_WARP = 0, 1, 2, 3

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int64)


class nnb_target(C.Structure):
    _fields_ = [('like_id', C.c_int), ('n_like_params', C.c_int), ('like_params', _dp), ('compute_f64', C.c_int),
                ('t_scale', _dp), ('t_shift', _dp), ('prior_kind', C.c_int), ('prior_lo', _dp), ('prior_hi', _dp)]


class nnb_mcmc_init_args(C.Structure):
    _fields_ = [('n_chains', C.c_int64), ('z', C.c_void_p), ('x', C.c_void_p), ('logl', C.c_void_p),
                ('logdet', C.c_void_p), ('logp', C.c_void_p), ('init_u', C.c_void_p), ('init_z', C.c_void_p),
                ('init_logl', C.c_void_p), ('seed', C.c_uint64), ('chain_offset', C.c_uint64),
                ('start_try', C.c_uint32), ('n_bad_start', _ip), ('ncall', _ip)]


class nnb_mcmc_args(C.Structure):
    _fields_ = [('n_chains', C.c_int64), ('steps', C.c_int), ('mode', C.c_int), ('loglstar', C.c_double),
                ('step_size', C.c_double), ('dynamic_step_size', C.c_int), ('seed', C.c_uint64),
                ('chain_offset', C.c_uint64), ('step_offset', C.c_uint32),
                ('z', C.c_void_p), ('x', C.c_void_p), ('logl', C.c_void_p), ('logdet', C.c_void_p),
                ('logp', C.c_void_p), ('trace_x', C.c_void_p), ('trace_z', C.c_void_p), ('trace_logl', C.c_void_p),
                ('replay_normals', C.c_void_p), ('replay_uniforms', C.c_void_p), ('dump_normals', C.c_void_p),
                ('dump_uniforms', C.c_void_p), ('scale_out', _dp), ('ncall_out', _ip), ('naccept_out', _ip),
                ('impl', C.c_int), ('launches_out', _ip), ('impl_out', C.POINTER(C.c_int))]


class nnb_train_args(C.Structure):
    _fields_ = [('x_dim', C.c_int), ('hidden_dim', C.c_int), ('num_layers', C.c_int), ('num_blocks', C.c_int),
                ('x_train', C.c_void_p), ('n_train', C.c_int64), ('perm', C.c_void_p), ('batch_size', C.c_int),
                ('x_valid', C.c_void_p), ('n_valid', C.c_int64), ('noise', C.c_void_p), ('jitter', C.c_double),
                ('seed', C.c_uint64), ('epoch', C.c_uint32), ('lr', C.c_double), ('beta1', C.c_double),
                ('beta2', C.c_double), ('eps', C.c_double), ('weight_decay', C.c_double), ('step0', C.c_int64),
                ('params', C.c_void_p), ('adam_m', C.c_void_p), ('adam_v', C.c_void_p), ('n_params', C.c_size_t),
                ('grad_out', C.c_void_p), ('do_train', C.c_int), ('train_loss_sum_out', _dp),
                ('val_nll_sum_out', _dp), ('grid_out', C.POINTER(C.c_int)), ('grad_only', C.c_int),
                ('batch_total', C.c_int)]


# name -> (restype, argtypes); every symbol include/nnb.h declares
SYMBOLS = {
    'nnb_abi_version': (C.c_int, []),
    'nnb_create': (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    'nnb_destroy': (None, [C.c_void_p]),
    'nnb_last_error': (C.c_char_p, [C.c_void_p]),
    'nnb_set_flow': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _fp, C.c_size_t]),
    'nnb_set_flow_spline': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _fp, C.c_size_t]),
    'nnb_flow_empty_halves': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                        C.c_void_p]),
    'nnb_flow_inverse': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                   C.c_void_p, C.c_int64, C.c_void_p]),
    'nnb_flow_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                   C.c_void_p, C.c_int64, C.c_void_p]),
    'nnb_set_target': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(nnb_target)]),
    'nnb_set_user_likelihood': (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int)]),
    'nnb_user_likelihood_check': (C.c_int, [C.c_char_p, C.c_char_p, C.c_size_t]),
    'nnb_set_user_likelihood_derived': (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
    'nnb_user_likelihood_check_derived': (C.c_int, [C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]),
    'nnb_set_user_likelihood_data': (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_char_p),
                                               C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'nnb_user_likelihood_check_data': (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int),
                                                 C.c_char_p, C.c_size_t]),
    'nnb_bind_user_data': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _ip]),
    'nnb_derived': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'nnb_derived_trace': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    'nnb_set_user_transform': (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int)]),
    'nnb_user_transform_check': (C.c_int, [C.c_char_p, C.c_char_p, C.c_size_t]),
    'nnb_set_target_user_transform': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(nnb_target), C.c_void_p, C.c_int]),
    'nnb_transform': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                C.c_void_p]),
    'nnb_transform_trace': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                      C.c_void_p]),
    'nnb_loglike': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                              C.c_int64, C.c_void_p]),
    'nnb_mcmc_init': (C.c_int, [C.c_void_p, C.POINTER(nnb_mcmc_init_args), C.c_void_p]),
    'nnb_mcmc_run': (C.c_int, [C.c_void_p, C.POINTER(nnb_mcmc_args), C.c_void_p]),
    'nnb_mcmc_result': (C.c_int, [C.c_void_p, _dp, _ip, _ip, C.c_void_p]),
    'nnb_consume_scan': (C.c_int64, [_fp, _fp, _dp, C.c_int64, C.c_int, C.c_double, _ip]),
    'nnb_ns_consume': (C.c_int64, [_dp, C.c_int64, _fp, _fp, _dp, C.c_int64, C.c_int, _ip, C.c_int64, _ip, _ip, _ip, _dp,
                                   _dp, C.POINTER(C.c_int)]),
    'nnb_gather_rows_f32': (C.c_int, [_fp, C.c_int64, C.c_int, _ip, C.c_int64, _dp]),
    'nnb_ns_apply': (C.c_int, [_ip, _ip, C.c_int64, C.c_int64, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int64, _dp]),
    'nnb_train_epoch': (C.c_int, [C.c_void_p, C.POINTER(nnb_train_args), C.c_void_p]),
    'nnb_train_epoch_begin': (C.c_int, [C.c_void_p, C.POINTER(nnb_train_args), C.c_void_p]),
    'nnb_train_epoch_end': (C.c_int, [C.c_void_p, _dp, _dp, C.POINTER(C.c_int)]),
    'nnb_train_supported': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    'nnb_mean_nn_distance': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, _dp, C.c_void_p]),
    'nnb_chain_stats': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int64, _dp, _dp, _dp, _dp, _dp, _dp,
                                  C.c_void_p]),
    'nnb_chain_autocorr': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int64, _dp, _dp, _dp, C.c_int,
                                     C.c_int, _dp, C.c_void_p]),
    'nnb_ns_information': (C.c_double, [C.c_double, _dp, _dp, _dp, _dp, C.c_int64]),
    'nnb_write_chain_text': (C.c_int64, [C.c_char_p, C.c_char_p, _dp, C.c_int64, C.c_int, C.c_int]),
    'nnb_write_chain_rows': (C.c_int64, [C.c_char_p, C.c_char_p, _dp, _dp, _dp, C.c_int, _dp, C.c_int, C.c_int64,
                                         C.c_double, C.c_int]),
}

_lib = None


class NNBError(RuntimeError):
    def __init__(self, code, msg):
        super(NNBError, self).__init__('libnnb error %d: %s' % (code, msg))
        self.code = code


def _load_nvrtc():
    """Make libnvrtc.so.12 visible to libnnb.so's dlopen (user likelihoods, nnb_jit.cu), from the first place that has
    it: the loader's search path, torch's NVRTC wheel (12.8, which also targets sm_100a), $CUDA_HOME/lib64,
    /usr/local/cuda/lib64.  Without it libnnb.so still loads; only user likelihoods are unavailable."""
    candidates = ['libnvrtc.so.12']
    try:
        import nvidia.cuda_nvrtc
        candidates.append(os.path.join(list(nvidia.cuda_nvrtc.__path__)[0], 'lib', 'libnvrtc.so.12'))
    except Exception:
        pass
    if os.environ.get('CUDA_HOME'):
        candidates.append(os.path.join(os.environ['CUDA_HOME'], 'lib64', 'libnvrtc.so.12'))
    candidates.append('/usr/local/cuda/lib64/libnvrtc.so.12')
    for path in candidates:
        try:
            return C.CDLL(path, mode=C.RTLD_GLOBAL)
        except OSError:
            continue
    return None


def load():
    """Load libnnb.so and set prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('%s not found: build it with `python -m nnest_b200.build` '
                           '(the CUDA path is the only path; there is no CPU fallback)' % LIB_PATH)
    try:      # a library older than the sources is used as is, but never silently
        from . import build as _build
        if os.path.isdir(_build.CSRC) and not _build.up_to_date():
            import warnings
            warnings.warn('libnnb.so does not match nnest_b200/csrc (content digests differ): rebuild with '
                          '`python -m nnest_b200.build`', RuntimeWarning)
    except Exception:
        pass
    _load_nvrtc()
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.nnb_abi_version() != NNB_ABI_VERSION:
        raise RuntimeError('libnnb.so ABI version mismatch: rebuild with `python -m nnest_b200.build --force`')
    _lib = lib
    return lib


def check(handle, rc):
    if rc != NNB_OK:
        msg = load().nnb_last_error(handle)
        raise NNBError(rc, msg.decode() if msg else '')
