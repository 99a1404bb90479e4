"""User likelihoods written in CUDA C++ (CudaLikelihood, nnb_user_likelihood_check): what works without a GPU --
the NVRTC compile of the library's kernels around the user's source, its error reporting and the ABI."""
import ctypes as C

import numpy as np
import pytest

import user_sources as us
from nnest_b200 import _lib as L


@pytest.fixture(scope='module')
def lib():
    lib = L.load()
    log = C.create_string_buffer(256)
    if lib.nnb_user_likelihood_check(us.ROSENBROCK.encode(), log, len(log)) == L.NNB_ERR_UNSUPPORTED:
        pytest.skip('NVRTC (libnvrtc.so.12) is not available')
    return lib


def _check(lib, source):
    log = C.create_string_buffer(1 << 16)
    rc = lib.nnb_user_likelihood_check(source.encode(), log, len(log))
    return rc, log.value.decode()


def test_abi_version_and_symbols():
    lib = L.load()
    assert lib.nnb_abi_version() == L.NNB_ABI_VERSION == 14
    assert L.NNB_LIKE_USER == 6 and L.NNB_MAX_LIKE_PARAMS == 160
    for name in ('nnb_set_user_likelihood', 'nnb_user_likelihood_check'):
        assert getattr(lib, name).argtypes == L.SYMBOLS[name][1]


@pytest.mark.parametrize('name', ['ROSENBROCK', 'HIMMELBLAU', 'EGGBOX', 'SHELL', 'GAUSS30'])
def test_check_accepts_the_test_sources(lib, name):
    src = us.gauss_full_source(np.eye(30)) if name == 'GAUSS30' else getattr(us, name)
    rc, log = _check(lib, src)
    assert rc == L.NNB_OK, log


def test_check_reports_syntax_error_with_line(lib):
    rc, log = _check(lib, us.SYNTAX_ERROR)
    assert rc == L.NNB_ERR_ARG
    # NVRTC names the user's file and the offending line (line 5: the closing brace after the missing semicolon)
    assert 'user_likelihood.cu(5)' in log and 'error' in log, log


def test_check_reports_missing_function(lib):
    rc, log = _check(lib, us.MISSING)
    assert rc == L.NNB_ERR_ARG
    assert 'nnb_user_loglike' in log and 'error' in log, log


def test_check_log_truncated_to_capacity(lib):
    log = C.create_string_buffer(16)
    assert lib.nnb_user_likelihood_check(us.SYNTAX_ERROR.encode(), log, len(log)) == L.NNB_ERR_ARG
    assert len(log.value) == 15
    assert lib.nnb_user_likelihood_check(us.SYNTAX_ERROR.encode(), None, 0) == L.NNB_ERR_ARG
    assert lib.nnb_user_likelihood_check(None, None, 0) == L.NNB_ERR_ARG


def test_cuda_likelihood_constructor(lib):
    from nnest_b200.likelihoods import CudaLikelihood, Likelihood
    like = CudaLikelihood(3, us.ROSENBROCK, params=[1.0, 2.0], max_loglike=0.0)
    assert isinstance(like, Likelihood) and like.like_id == L.NNB_LIKE_USER
    assert like.device_params() == [1.0, 2.0] and like.device_source() == us.ROSENBROCK and like.max_loglike == 0.0
    with pytest.raises(ValueError, match=r'user_likelihood\.cu\(5\)'):
        CudaLikelihood(2, us.SYNTAX_ERROR)
    with pytest.raises(ValueError, match='nnb_user_loglike'):
        CudaLikelihood(2, us.MISSING)


def test_cuda_likelihood_refuses_too_many_params():
    from nnest_b200.likelihoods import CudaLikelihood
    with pytest.raises(ValueError, match='at most 160'):
        CudaLikelihood(2, us.ROSENBROCK, params=np.zeros(L.NNB_MAX_LIKE_PARAMS + 1))


def test_builtin_likelihoods_have_no_source():
    from nnest_b200.likelihoods import Rosenbrock
    assert Rosenbrock(2).device_source() is None
