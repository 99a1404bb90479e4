"""User prior transforms written in CUDA C++ (CudaTransform, nnb_user_transform_check): what works without a GPU -- the
NVRTC compile of the library's kernels around the user's transform, its error reporting and the ABI."""
import ctypes as C

import numpy as np
import pytest

import transform_sources as ts
from nnest_b200 import _lib as L


@pytest.fixture(scope='module')
def lib():
    lib = L.load()
    log = C.create_string_buffer(256)
    if lib.nnb_user_transform_check(ts.AFFINE.encode(), log, len(log)) == L.NNB_ERR_UNSUPPORTED:
        pytest.skip('NVRTC (libnvrtc.so.12) is not available')
    return lib


def _check(lib, source):
    log = C.create_string_buffer(1 << 16)
    rc = lib.nnb_user_transform_check(source.encode(), log, len(log))
    return rc, log.value.decode()


def test_abi_unchanged_and_new_symbols():
    lib = L.load()
    assert lib.nnb_abi_version() == L.NNB_ABI_VERSION == 14
    for name in ('nnb_set_user_transform', 'nnb_user_transform_check', 'nnb_set_target_user_transform',
                 'nnb_transform', 'nnb_transform_trace'):
        assert getattr(lib, name).argtypes == L.SYMBOLS[name][1]
    assert L.SYMBOLS['nnb_set_target_user_transform'][1][2] == C.POINTER(L.nnb_target)


@pytest.mark.parametrize('name', ['AFFINE', 'GAUSS', 'LOGUNIFORM', 'CHOLESKY'])
def test_check_accepts_the_test_sources(lib, name):
    rc, log = _check(lib, getattr(ts, name))
    assert rc == L.NNB_OK, log


def test_check_reports_syntax_error_with_line(lib):
    rc, log = _check(lib, ts.SYNTAX_ERROR)
    assert rc == L.NNB_ERR_ARG
    # NVRTC names the user's file and the offending line (line 5: the closing brace after the missing semicolon)
    assert 'user_transform.cu(5)' in log and 'error' in log, log


def test_check_reports_missing_function(lib):
    rc, log = _check(lib, ts.MISSING)
    assert rc == L.NNB_ERR_ARG
    assert 'nnb_user_transform' in log and 'error' in log, log


def test_check_log_truncated_to_capacity(lib):
    log = C.create_string_buffer(16)
    assert lib.nnb_user_transform_check(ts.SYNTAX_ERROR.encode(), log, len(log)) == L.NNB_ERR_ARG
    assert len(log.value) == 15
    assert lib.nnb_user_transform_check(ts.SYNTAX_ERROR.encode(), None, 0) == L.NNB_ERR_ARG
    assert lib.nnb_user_transform_check(None, None, 0) == L.NNB_ERR_ARG


def test_cuda_transform_constructor(lib):
    from nnest_b200.likelihoods import CudaTransform
    t = CudaTransform(3, ts.GAUSS, params=[3.0])
    assert t.x_dim == 3 and t.params == [3.0] and t.source == ts.GAUSS and t.float64
    assert not CudaTransform(3, ts.GAUSS, params=[3.0], float64=False).float64
    with pytest.raises(ValueError, match=r'user_transform\.cu\(5\)'):
        CudaTransform(2, ts.SYNTAX_ERROR)
    with pytest.raises(ValueError, match='nnb_user_transform'):
        CudaTransform(2, ts.MISSING)
    with pytest.raises(ValueError, match='non-empty'):
        CudaTransform(2, '   ')


def test_cuda_transform_refuses_too_many_params():
    from nnest_b200.likelihoods import CudaTransform
    with pytest.raises(ValueError, match='at most 160'):
        CudaTransform(2, ts.AFFINE, params=np.zeros(L.NNB_MAX_LIKE_PARAMS + 1))


def test_python_callable_that_is_not_affine_still_raises():
    from nnest_b200.sampler import probe_affine_transform
    with pytest.raises(NotImplementedError, match='CudaTransform'):
        probe_affine_transform(lambda x: np.sinh(3.0 * x), 3)
    # the affine maps are still recovered
    sc, sh, promotes = probe_affine_transform(lambda x: 5 * x + 1, 2)
    assert np.allclose(sc, 5.0) and np.allclose(sh, 1.0) and not promotes
