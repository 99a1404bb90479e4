"""Datasets of user likelihoods (CudaLikelihood(data=...), nnb_user_likelihood_check_data): what works without a GPU --
the NVRTC compile of the kernels behind the generated declarations of a layout, its refusals and the ABI."""
import ctypes as C

import numpy as np
import pytest

import data_sources as ds
import transform_sources as ts
import user_sources as us
from nnest_b200 import _lib as L

F64, F32, I32 = L.NNB_DTYPE_F64, L.NNB_DTYPE_F32, L.NNB_DTYPE_I32
LINE_LAYOUT = [('t', F64), ('y', F64), ('w', F32), ('mask', I32)]


@pytest.fixture(scope='module')
def lib():
    lib = L.load()
    log = C.create_string_buffer(256)
    if lib.nnb_user_likelihood_check(us.ROSENBROCK.encode(), log, len(log)) == L.NNB_ERR_UNSUPPORTED:
        pytest.skip('NVRTC (libnvrtc.so.12) is not available')
    return lib


def _check(lib, source, layout, num_derived=0):
    names = (C.c_char_p * max(1, len(layout)))(*[n.encode() if isinstance(n, str) else n for n, _ in layout])
    dtypes = (C.c_int * max(1, len(layout)))(*[dt for _, dt in layout])
    log = C.create_string_buffer(1 << 16)
    rc = lib.nnb_user_likelihood_check_data(source.encode(), num_derived, len(layout), names, dtypes, log, len(log))
    return rc, log.value.decode()


def _reader(expr, derived=False):
    """a likelihood (or, derived=True, derived parameters) returning the double value of `expr`"""
    if derived:
        return us.ROSENBROCK + r'''
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  derived[0] = (double)(%s);
}
''' % expr
    return r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  return (double)(%s);
}
''' % expr


def test_abi_unchanged_and_new_symbols():
    lib = L.load()
    assert lib.nnb_abi_version() == L.NNB_ABI_VERSION == 14
    assert L.NNB_MAX_DATA_ARRAYS == 16 and (F64, F32, I32) == (0, 1, 2)
    for name in ('nnb_set_user_likelihood_data', 'nnb_user_likelihood_check_data', 'nnb_bind_user_data'):
        assert getattr(lib, name).argtypes == L.SYMBOLS[name][1]
    assert L.SYMBOLS['nnb_set_user_likelihood_data'][1][4] == C.POINTER(C.c_char_p)
    assert L.SYMBOLS['nnb_bind_user_data'][1][1:] == [C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]


@pytest.mark.parametrize('num_derived', [0, ds.LINE_DERIVED])
def test_check_accepts_every_dtype(lib, num_derived):
    rc, log = _check(lib, ds.LINE, LINE_LAYOUT, num_derived)
    assert rc == L.NNB_OK, log


@pytest.mark.parametrize('dtype,expr', [(F64, 'nnb_data.a[0]'), (F32, 'nnb_data.a[1] * 2.0f'),
                                        (I32, 'nnb_data.a[2] + nnb_data.a.size()')])
def test_check_each_dtype_from_the_derived_function(lib, dtype, expr):
    rc, log = _check(lib, _reader(expr, derived=True), [('a', dtype)], num_derived=1)
    assert rc == L.NNB_OK, log


def test_zero_arrays_is_the_plain_check(lib):
    assert _check(lib, us.ROSENBROCK, [])[0] == L.NNB_OK
    # without a layout nnb_data is not declared
    rc, log = _check(lib, _reader('nnb_data.a[0]'), [])
    assert rc == L.NNB_ERR_ARG and 'nnb_data' in log


def test_check_refuses_an_undeclared_array(lib):
    rc, log = _check(lib, _reader('nnb_data.t[0] +\n nnb_data.q[0]'), [('t', F64)])
    assert rc == L.NNB_ERR_ARG
    assert 'user_likelihood.cu(5)' in log and 'q' in log and 'error' in log, log


def test_check_refuses_an_array_read_as_the_wrong_type(lib):
    src = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  const nnb_span<int> m = nnb_data.t;
  return (double)m[0];
}
'''
    rc, log = _check(lib, src, [('t', F64)])
    assert rc == L.NNB_ERR_ARG and 'user_likelihood.cu(4)' in log and 'error' in log, log
    rc, log = _check(lib, _reader('nnb_data.t.p[0]'), [('t', F64)])
    assert rc == L.NNB_OK, log        # the pointer, read as its own type, is fine


@pytest.mark.parametrize('stmt', ['nnb_data.y[0] = 1.0;', 'nnb_data.y.p[0] = 1.0;'])
def test_check_refuses_a_write_through_a_span(lib, stmt):
    src = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  %s
  return 0.0;
}
''' % stmt
    rc, log = _check(lib, src, [('y', F64)])
    assert rc == L.NNB_ERR_ARG and 'user_likelihood.cu(4)' in log and 'error' in log, log


@pytest.mark.parametrize('layout,what', [
    ([('1t', F64)], 'not a C identifier'),
    ([('t-y', F64)], 'not a C identifier'),
    ([('', F64)], 'not a C identifier'),
    ([(None, F64)], 'not a C identifier'),
    ([('t', F64), ('t', F32)], 'repeated'),
    ([('t', 3)], 'unknown dtype'),
    ([('t', -1)], 'unknown dtype'),
    ([('a%d' % i, F64) for i in range(L.NNB_MAX_DATA_ARRAYS + 1)], 'n_arrays must be in [0, 16]'),
])
def test_check_refuses_bad_layouts(lib, layout, what):
    rc, log = _check(lib, ds.LINE, layout)
    assert rc == L.NNB_ERR_ARG and what in log, log


def test_check_takes_the_maximum_number_of_arrays(lib):
    layout = [('a%d' % i, (F64, F32, I32)[i % 3]) for i in range(L.NNB_MAX_DATA_ARRAYS)]
    expr = ' + '.join('nnb_data.a%d[0]' % i for i in range(L.NNB_MAX_DATA_ARRAYS))
    rc, log = _check(lib, _reader(expr), layout)
    assert rc == L.NNB_OK, log


def test_transform_that_names_the_dataset_is_refused(lib):
    src = r'''
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  return u(i) * nnb_data.t[0];
}
'''
    log = C.create_string_buffer(1 << 16)
    assert lib.nnb_user_transform_check(src.encode(), log, len(log)) == L.NNB_ERR_ARG
    assert 'user_transform.cu(4)' in log.value.decode() and 'nnb_data' in log.value.decode()
    from nnest_b200.likelihoods import CudaTransform
    with pytest.raises(ValueError, match=r'user_transform\.cu\(4\)'):
        CudaTransform(2, src)
    assert CudaTransform(2, ts.GAUSS, params=[1.0]).x_dim == 2


# ---- CudaLikelihood(data=...) ---------------------------------------------------------------------------------------
def test_constructor_copies_freezes_and_keeps_dtypes(lib):
    from nnest_b200.likelihoods import CudaLikelihood
    data = ds.line_data(50)
    t2 = np.arange(12.0).reshape(3, 4)
    like = CudaLikelihood(2, ds.LINE, data=dict(data, t=t2.T), num_derived=ds.LINE_DERIVED)
    dd = like.device_data()
    assert dd.names == ('t', 'y', 'w', 'mask') and dd.dtypes == (F64, F64, F32, I32)
    assert dd.layout == tuple(LINE_LAYOUT)
    assert np.array_equal(like.data['t'], t2.T.ravel())                      # C order of the array as given
    assert [a.dtype for a in dd.arrays] == [np.float64, np.float64, np.float32, np.int32]
    assert all(a.ndim == 1 and a.flags.c_contiguous and not a.flags.writeable for a in dd.arrays)
    with pytest.raises(ValueError):
        dd.arrays[1][0] = 0.0
    before = like.data['y'].copy()
    data['y'][:] = 0.0                                                        # the caller's array changes nothing
    assert np.array_equal(like.data['y'], before)
    other = CudaLikelihood(2, ds.LINE, data=ds.line_data(50), num_derived=ds.LINE_DERIVED)
    assert other.device_data().token != dd.token and other.device_data().layout == dd.layout


def test_constructor_accepts_empty_arrays_and_lists(lib):
    from nnest_b200.likelihoods import CudaLikelihood
    like = CudaLikelihood(2, ds.LINE, data=dict(t=np.zeros(0), y=[1.0, 2.0], w=np.zeros(0, np.float32),
                                                 mask=np.zeros(0, np.int32)))
    assert like.data['t'].size == 0 and like.data['y'].dtype == np.float64


@pytest.mark.parametrize('dtype', [np.float16, np.int64, np.uint32, np.complex128, bool])
def test_constructor_refuses_other_dtypes(lib, dtype):
    from nnest_b200.likelihoods import CudaLikelihood
    with pytest.raises(ValueError, match='float64, float32 and int32'):
        CudaLikelihood(1, _reader('nnb_data.a[0]'), data={'a': np.zeros(3, dtype=dtype)})


def test_constructor_refuses_bad_names_and_sources(lib):
    from nnest_b200.likelihoods import CudaLikelihood
    with pytest.raises(ValueError, match='C identifiers'):
        CudaLikelihood(1, _reader('0.0'), data={'bad name': np.zeros(3)})
    with pytest.raises(ValueError, match='C identifiers'):
        CudaLikelihood(1, _reader('0.0'), data={3: np.zeros(3)})
    with pytest.raises(ValueError, match='repeated'):
        CudaLikelihood(1, _reader('0.0'), data=[('a', np.zeros(3)), ('a', np.zeros(3))])
    with pytest.raises(ValueError, match='at most 16 data arrays'):
        CudaLikelihood(1, _reader('0.0'), data={'a%d' % i: np.zeros(1) for i in range(17)})
    # the layout is checked against the source: an undeclared array, or a layout the source reads as another type
    with pytest.raises(ValueError, match=r'user_likelihood\.cu\(4\)'):
        CudaLikelihood(1, _reader('nnb_data.q[0]'), data={'a': np.zeros(3)})
    with pytest.raises(ValueError, match='does not compile'):
        CudaLikelihood(1, r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  const nnb_span<float> w = nnb_data.w;
  return (double)w[0];
}
''', data={'w': np.zeros(3)})


def test_without_data_nothing_changes(lib):
    from nnest_b200.likelihoods import CudaLikelihood, Rosenbrock
    like = CudaLikelihood(2, us.ROSENBROCK)
    assert like.device_data() is None and like.data == {}
    assert CudaLikelihood(2, us.ROSENBROCK, data={}).device_data() is None
    assert Rosenbrock(2).device_data() is None
    with pytest.raises(ValueError, match='nnb_data'):
        CudaLikelihood(1, _reader('nnb_data.a[0]'))
