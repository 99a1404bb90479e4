"""Derived parameters of user likelihoods (CudaLikelihood(num_derived=...), nnb_user_derived): what works without a GPU --
the NVRTC compile of the derived kernels around the user's source, its error reporting, the argument checks of
CudaLikelihood and Sampler, and the ABI."""
import ctypes as C

import pytest

import user_sources as us
from nnest_b200 import _lib as L

# The sources of the derived-parameter tests: user Rosenbrock (the built-in one operation for operation) with three
# derived columns -- the likelihood re-evaluated, the first transformed coordinate, and the float64 sum of the squared
# transformed coordinates in index order.
DERIVED3 = us.ROSENBROCK + r'''
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  derived[0] = nnb_user_loglike(x, d, params);
  derived[1] = (double)x(0);
  double s = 0.0;
  for (int i = 0; i < d; ++i) {
    const double v = (double)x(i);
    s = __dadd_rn(s, __dmul_rn(v, v));
  }
  derived[2] = s;
}
'''

DERIVED_WRONG_SIGNATURE = us.ROSENBROCK + r'''
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, double* derived) {
  derived[0] = (double)x(0);
}
'''

DERIVED_SYNTAX_ERROR = us.ROSENBROCK + r'''
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  derived[0] = (double)x(0)   // missing semicolon
}
'''


@pytest.fixture(scope='module')
def lib():
    lib = L.load()
    log = C.create_string_buffer(256)
    if lib.nnb_user_likelihood_check(us.ROSENBROCK.encode(), log, len(log)) == L.NNB_ERR_UNSUPPORTED:
        pytest.skip('NVRTC (libnvrtc.so.12) is not available')
    return lib


def _check(lib, source, num_derived):
    log = C.create_string_buffer(1 << 16)
    rc = lib.nnb_user_likelihood_check_derived(source.encode(), num_derived, log, len(log))
    return rc, log.value.decode()


def test_abi_version_and_symbols():
    lib = L.load()
    assert lib.nnb_abi_version() == L.NNB_ABI_VERSION == 14
    assert L.NNB_LIKE_USER == 6 and L.NNB_MAX_LIKE_PARAMS == 160 and L.NNB_MAX_DERIVED == 32
    for name in ('nnb_set_user_likelihood', 'nnb_user_likelihood_check', 'nnb_set_user_likelihood_derived',
                 'nnb_user_likelihood_check_derived', 'nnb_derived', 'nnb_derived_trace'):
        assert getattr(lib, name).argtypes == L.SYMBOLS[name][1]


def test_check_accepts_derived_source(lib):
    rc, log = _check(lib, DERIVED3, 3)
    assert rc == L.NNB_OK, log


def test_check_reports_missing_derived_function(lib):
    rc, log = _check(lib, us.ROSENBROCK, 3)
    assert rc == L.NNB_ERR_ARG
    assert 'nnb_user_derived' in log and 'error' in log, log


def test_check_reports_wrong_signature(lib):
    rc, log = _check(lib, DERIVED_WRONG_SIGNATURE, 1)
    assert rc == L.NNB_ERR_ARG
    assert 'nnb_user_derived' in log and 'error' in log, log


def test_check_reports_syntax_error_with_line(lib):
    rc, log = _check(lib, DERIVED_SYNTAX_ERROR, 1)
    assert rc == L.NNB_ERR_ARG
    # NVRTC names the user's file and the offending line: the closing brace after the missing semicolon, the last line
    line = len(DERIVED_SYNTAX_ERROR.rstrip('\n').split('\n'))
    assert 'user_likelihood.cu(%d)' % line in log and 'error' in log, log


def test_check_refuses_num_derived_out_of_range(lib):
    for n in (-1, L.NNB_MAX_DERIVED + 1):
        rc, log = _check(lib, DERIVED3, n)
        assert rc == L.NNB_ERR_ARG and 'num_derived' in log


def test_source_without_derived_function_still_compiles_without_derived(lib):
    # num_derived == 0 is nnb_user_likelihood_check: a source without nnb_user_derived is fine, and so is one with it
    assert _check(lib, us.ROSENBROCK, 0)[0] == L.NNB_OK
    assert _check(lib, DERIVED3, 0)[0] == L.NNB_OK


def test_cuda_likelihood_constructor(lib):
    from nnest_b200.likelihoods import CudaLikelihood
    like = CudaLikelihood(3, DERIVED3, num_derived=3)
    assert like.num_derived == 3 and like.device_source() == DERIVED3
    assert CudaLikelihood(3, us.ROSENBROCK).num_derived == 0
    with pytest.raises(ValueError, match='nnb_user_derived'):
        CudaLikelihood(2, us.ROSENBROCK, num_derived=2)
    with pytest.raises(ValueError, match='nnb_user_derived'):
        CudaLikelihood(2, DERIVED_WRONG_SIGNATURE, num_derived=1)
    with pytest.raises(ValueError, match=r'user_likelihood\.cu\(\d+\)'):
        CudaLikelihood(2, DERIVED_SYNTAX_ERROR, num_derived=1)


@pytest.mark.parametrize('n', [-1, L.NNB_MAX_DERIVED + 1, 1.5])
def test_cuda_likelihood_refuses_num_derived_out_of_range(n):
    from nnest_b200.likelihoods import CudaLikelihood
    with pytest.raises(ValueError, match='num_derived'):
        CudaLikelihood(2, DERIVED3, num_derived=n)


def test_sampler_checks_num_derived_before_any_device_work(lib, tmp_path):
    from nnest_b200 import MCMCSampler, NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood, Rosenbrock
    like = CudaLikelihood(2, DERIVED3, num_derived=3)
    for cls in (NestedSampler, MCMCSampler):
        with pytest.raises(ValueError, match='num_derived'):
            cls(2, like, num_derived=2, log_dir=str(tmp_path))
        with pytest.raises(ValueError, match='num_derived'):
            cls(2, like, log_dir=str(tmp_path))
        with pytest.raises(NotImplementedError, match='CudaLikelihood'):
            cls(2, Rosenbrock(2), num_derived=1, log_dir=str(tmp_path))
