"""Datasets of user likelihoods on the device (CudaLikelihood(data=...), nnb_bind_user_data): values against NumPy, bit
identity with the same data written into the source, rebinding without recompiling, host-side refusals, analytic
evidence and posteriors, and two ranks."""
import ctypes as C
import logging
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import data_sources as ds
import transform_sources as ts
import user_sources as us
from nnest_b200 import _lib as L
from test_gpu_user_likelihood import VARIANTS, _assert_same, _nvp, _spline

pytestmark = pytest.mark.gpu

dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
BOX = dict(prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)


@pytest.fixture(scope='module')
def eng():
    from nnest_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope='module')
def line():
    from nnest_b200.likelihoods import CudaLikelihood
    data = ds.line_data(100000, seed=3)
    assert sum(a.nbytes for a in data.values()) == 2_400_000        # beyond the 64 KB of constant memory
    return CudaLikelihood(2, ds.LINE, data=data, num_derived=ds.LINE_DERIVED), data


def _set(eng, like, d, **kw):
    eng.set_target(d, L.NNB_LIKE_USER, like.device_params(), user_source=like.device_source(),
                   num_derived=like.num_derived, user_data=like.device_data(), **kw)


# ---- 1. values against NumPy ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('f64', [False, True])
@pytest.mark.parametrize('target', ['plain', 'affine', 'affine_box', 'box'])
def test_line_chi2_against_numpy(eng, line, f64, target):
    like, data = line
    kw = {}
    if 'affine' in target:
        kw.update(t_scale=[0.25, 0.5], t_shift=[0.7, -1.3])
    if 'box' in target:
        kw.update(BOX)
    _set(eng, like, 2, **kw)
    rng = np.random.RandomState(1)
    u = rng.uniform(-1.05, 1.05, size=(4096, 2))
    u = dev(u if f64 else u.astype(np.float32))
    logl, logp = eng.loglike(u, want_prior=True)
    der = eng.derived(u).cpu().numpy()
    logl, logp = logl.cpu().numpy(), logp.cpu().numpy()
    # the derived columns 2 and 3 are x(0), x(1) as the likelihood saw them (after the transform, in its arithmetic)
    a, b = der[:, 2], der[:, 3]
    if 'affine' not in target:
        assert np.array_equal(a, u[:, 0].double().cpu().numpy()) and np.array_equal(b, u[:, 1].double().cpu().numpy())
    chi2 = ds.line_chi2_np(a, b, data)
    assert np.allclose(logl, -0.5 * chi2, rtol=1e-12, atol=0)
    assert np.allclose(der, ds.line_derived_np(a, b, data), rtol=1e-12, atol=1e-12)
    if 'box' in target:
        inside = np.all(np.abs(u.double().cpu().numpy()) <= 1.0, axis=1)
        assert np.array_equal(logp == 0, inside) and (logp[~inside] == -np.inf).all() and (~inside).any()
    # near the line the fit is good: chi^2 / N is about the unmasked fraction
    best = ds.line_derived_np([0.7], [-1.3], data)[0, 0]
    assert 0.8 < best < 1.0


# ---- 2. bit identity with the dataset written into the source -------------------------------------------------------
def _gauss(d, seed=5):
    rng = np.random.RandomState(seed)
    a = rng.normal(size=(d, d)) * 0.3
    cov = a @ a.T + np.eye(d)
    prec = np.linalg.inv(cov) * 4.0
    mu = rng.uniform(-0.2, 0.2, size=d)
    return prec, list(mu) + [0.0]


def _gauss_pair(d):
    from nnest_b200.likelihoods import CudaLikelihood
    prec, params = _gauss(d)
    baked = CudaLikelihood(d, us.gauss_full_source(prec), params=params)
    data = CudaLikelihood(d, ds.gauss_data_source(d), params=params, data={'prec': prec})
    return baked, data


def test_gauss_values_bit_identical_to_baked(eng):
    d = 30
    baked, data = _gauss_pair(d)
    rng = np.random.RandomState(2)
    for f64 in (False, True):
        u = rng.uniform(-1.0, 1.0, size=(4096, d))
        u = dev(u if f64 else u.astype(np.float32))
        out = []
        for like in (baked, data):
            _set(eng, like, d, t_scale=1.5, t_shift=0.1, **BOX)
            out.append(eng.loglike(u).cpu().numpy())
        assert np.array_equal(out[0], out[1])
        assert np.isfinite(out[0]).all()


def _chains(eng, like, n, d, mode, dynamic, impl, steps, seed=7):
    _set(eng, like, d, t_scale=np.linspace(1.0, 2.0, d), t_shift=np.linspace(-0.1, 0.1, d), **BOX)
    st, nbad, ncall0 = eng.mcmc_init(n, seed=seed, want_counts=True)
    logl0 = st.logl.clone()
    loglstar = float(torch.quantile(logl0[torch.isfinite(logl0)].cpu(), 0.3)) if mode == L.NNB_MODE_HARD else 0.0
    out = eng.mcmc_run(st, steps, mode=mode, loglstar=loglstar, dynamic_step_size=dynamic, seed=seed, trace=True,
                       impl=impl)
    res = {k: v.cpu().numpy() for k, v in out.items() if torch.is_tensor(v)}
    res.update({k: out[k] for k in ('scale', 'ncall', 'naccept', 'impl')})
    res.update(nbad=nbad, ncall0=ncall0, logl0=logl0.cpu().numpy())
    for k in ('z', 'x', 'logl', 'logdet', 'logp'):
        res['st_' + k] = getattr(st, k).cpu().numpy()
    return res


@pytest.mark.parametrize('variant', list(VARIANTS))
def test_gauss_chains_bit_identical_to_baked(eng, variant):
    flow, d, hid, flags, n, impl, mode, dynamic, impl_ran = VARIANTS[variant]
    if flow == 'spline':
        _spline(eng, d)
    else:
        _nvp(eng, d, hid, flags=flags)
    baked, data = _gauss_pair(d)
    a = _chains(eng, baked, n, d, mode, dynamic, impl, 12)
    b = _chains(eng, data, n, d, mode, dynamic, impl, 12)
    assert a['impl'] == impl_ran
    assert a['naccept'] > 0 and a['naccept'] < n * 12
    _assert_same(a, b)


# ---- 3. rebinding without recompiling -------------------------------------------------------------------------------
def _cubins(path):
    return set(path.glob('*.cubin'))


def test_rebinding_compiles_nothing(tmp_path, monkeypatch):
    from nnest_b200.engine import Engine
    from nnest_b200.likelihoods import CudaLikelihood
    monkeypatch.setenv('NNB_JIT_CACHE', str(tmp_path / 'jit'))
    src = ds.LINE + '\n// cache test %d\n' % np.random.randint(1 << 30)      # a source no cache has seen
    da, db = ds.line_data(5000, seed=1), ds.line_data(777, seed=2, a=-0.3, b=0.4)
    A = CudaLikelihood(2, src, data=da, num_derived=ds.LINE_DERIVED)
    B = CudaLikelihood(2, src, data=db, num_derived=ds.LINE_DERIVED)
    d, n = 2, 700
    u = dev(np.random.RandomState(3).uniform(-1, 1, size=(2000, d)))

    def check(e, like, data):
        _set(e, like, d)
        logl = e.loglike(u).cpu().numpy()
        ref = -0.5 * ds.line_chi2_np(u[:, 0].cpu().numpy(), u[:, 1].cpu().numpy(), data)
        assert np.allclose(logl, ref, rtol=1e-12, atol=0)
        assert np.allclose(e.derived(u).cpu().numpy(), ds.line_derived_np(u[:, 0].cpu().numpy(),
                                                                            u[:, 1].cpu().numpy(), data),
                           rtol=1e-12, atol=1e-12)
        st, _, _ = e.mcmc_init(n, seed=3, want_counts=True)
        out = e.mcmc_run(st, 4, mode=L.NNB_MODE_MH, seed=3, impl=L.NNB_IMPL_FFMA, trace=True)
        assert np.allclose(out['trace_logl'][-1].cpu().numpy(),
                           -0.5 * ds.line_chi2_np(*st.x.double().cpu().numpy(), data), rtol=1e-12, atol=0)
        return out

    e = Engine(0)
    _nvp(e, d)
    check(e, A, da)
    first = _cubins(tmp_path / 'jit')
    assert len(first) == 3                              # likelihood + derived kernels, chain start, one step kernel
    for like, data in ((B, db), (A, da), (B, db)):
        tok = like.device_data().token
        check(e, like, data)
        assert e._data_token == tok
    assert _cubins(tmp_path / 'jit') == first and not list((tmp_path / 'jit').glob('*.tmp*'))
    # the installed source and layout again: nothing to compile
    assert e.set_user_likelihood(src, ds.LINE_DERIVED, A.device_data().layout) == 0
    check(e, A, da)
    # the same dataset bound again uploads nothing
    kept = e._data_tensors
    _set(e, A, d)
    assert e._data_tensors is kept
    # a dtype or a name is part of the layout: compiled again
    C64 = CudaLikelihood(2, src, data=dict(da, w=da['w'].astype(np.float64)), num_derived=ds.LINE_DERIVED)
    assert e.set_user_likelihood(src, ds.LINE_DERIVED, C64.device_data().layout) == 1
    check(e, C64, da)
    named = [CudaLikelihood(2, src, data=dict(da, **{extra: np.zeros(1)}), num_derived=ds.LINE_DERIVED)
             for extra in ('extra', 'other')]
    assert e.set_user_likelihood(src, ds.LINE_DERIVED, named[0].device_data().layout) == 1
    assert e.set_user_likelihood(src, ds.LINE_DERIVED, named[1].device_data().layout) == 1
    # a second engine loads every variant from disk and binds its own copy
    grown = _cubins(tmp_path / 'jit')
    e2 = Engine(0)
    _nvp(e2, d)
    assert e2.set_user_likelihood(src, ds.LINE_DERIVED, A.device_data().layout) == 0
    check(e2, B, db)
    check(e2, A, da)
    _set(e, A, d)
    assert {t.data_ptr() for t in e2._data_tensors}.isdisjoint({t.data_ptr() for t in e._data_tensors})
    assert _cubins(tmp_path / 'jit') == grown


def test_direct_calls_upload_once(line):
    from nnest_b200.likelihoods import _eval_engine
    like, data = line
    x = np.array([[0.7, -1.3], [0.0, 0.0]])
    v1, der1 = like(x)
    eng = _eval_engine()
    kept = eng._data_tensors
    v2, der2 = like(x)
    assert eng._data_tensors is kept and eng._data_token == like.device_data().token
    assert np.array_equal(v1, v2) and np.array_equal(der1, der2)
    assert np.allclose(v1, -0.5 * ds.line_chi2_np(x[:, 0], x[:, 1], data), rtol=1e-12, atol=0)


# ---- 4. refusals are host-side only ---------------------------------------------------------------------------------
def test_refusals(tmp_path):
    from nnest_b200.engine import Engine
    from nnest_b200.likelihoods import CudaLikelihood
    data = ds.line_data(1000)
    like = CudaLikelihood(2, ds.LINE, data=data, num_derived=ds.LINE_DERIVED)
    layout = like.device_data().layout
    e = Engine(0)
    _nvp(e, 2)
    lib = e.lib
    u = dev(np.zeros((16, 2)))
    out = torch.empty(16, dtype=torch.float64, device='cuda')
    loglike = lambda: lib.nnb_loglike(e.h, C.c_void_p(u.data_ptr()), 1, 2, 1, C.c_void_p(out.data_ptr()), None, 16,
                                      None)
    # no source at all
    assert lib.nnb_bind_user_data(e.h, None, None) == L.NNB_ERR_STATE
    # a layout without a binding: every launch that needs the likelihood is refused before it runs
    e.set_user_likelihood(ds.LINE, ds.LINE_DERIVED, layout)
    t = L.nnb_target()
    t.like_id = L.NNB_LIKE_USER
    assert lib.nnb_set_target(e.h, 2, C.byref(t)) == L.NNB_OK
    assert loglike() == L.NNB_ERR_STATE and b'not bound' in lib.nnb_last_error(e.h)
    der = torch.empty((16, ds.LINE_DERIVED), dtype=torch.float64, device='cuda')
    assert lib.nnb_derived(e.h, C.c_void_p(u.data_ptr()), 1, 2, 1, C.c_void_p(der.data_ptr()), 16, None) == \
        L.NNB_ERR_STATE
    with pytest.raises(L.NNBError, match='not bound'):
        e.mcmc_init(64, seed=1, want_counts=True)
    # bound: it runs; a new install of the same source and layout drops the binding again
    _set(e, like, 2)
    assert loglike() == L.NNB_OK
    st, _, _ = e.mcmc_init(64, seed=1, want_counts=True)
    e.set_user_likelihood(ds.LINE, ds.LINE_DERIVED, layout)
    assert lib.nnb_set_target(e.h, 2, C.byref(t)) == L.NNB_OK
    with pytest.raises(L.NNBError) as err:
        e.mcmc_run(st, 2, mode=L.NNB_MODE_MH, seed=1, impl=L.NNB_IMPL_FFMA)
    assert err.value.code == L.NNB_ERR_STATE
    # bad bindings, checked on the host: nothing is launched with them
    good = [torch.from_numpy(np.array(a)).cuda() for a in like.device_data().arrays]

    def bind(ptrs, sizes):
        return lib.nnb_bind_user_data(e.h, (C.c_void_p * 4)(*ptrs), (C.c_int64 * 4)(*sizes))

    ptrs, sizes = [t_.data_ptr() for t_ in good], [t_.numel() for t_ in good]
    host = np.zeros(1000)
    for i, (p, s, what) in enumerate([(host.ctypes.data, 1000, 'device or managed'),
                                      (good[0].data_ptr() + 4, 999, 'aligned'),
                                      (None, 1000, 'NULL'),
                                      (good[0].data_ptr(), -1, 'negative')]):
        pp, ss = list(ptrs), list(sizes)
        pp[i % 2], ss[i % 2] = p, s
        assert bind(pp, ss) == L.NNB_ERR_ARG, what
        assert what.encode() in lib.nnb_last_error(e.h)
    pinned = torch.zeros(1000, dtype=torch.float64).pin_memory()
    pp = list(ptrs)
    pp[1] = pinned.data_ptr()
    assert bind(pp, sizes) == L.NNB_ERR_ARG
    assert lib.nnb_bind_user_data(e.h, None, None) == L.NNB_ERR_ARG
    assert loglike() == L.NNB_ERR_STATE                # still unbound
    if torch.cuda.device_count() >= 2:
        other = torch.from_numpy(np.array(like.device_data().arrays[0])).to('cuda:1')
        pp = list(ptrs)
        pp[0] = other.data_ptr()
        assert bind(pp, sizes) == L.NNB_ERR_ARG and b'device' in lib.nnb_last_error(e.h)
    # empty arrays may be NULL; the good binding then runs
    assert bind(ptrs, sizes) == L.NNB_OK
    assert loglike() == L.NNB_OK
    ref = -0.5 * ds.line_chi2_np(np.zeros(16), np.zeros(16), data)
    assert np.allclose(out.cpu().numpy(), ref, rtol=1e-12, atol=0)
    assert bind([None, None, None, None], [0, 0, 0, 0]) == L.NNB_OK
    assert loglike() == L.NNB_OK and (out.cpu().numpy() == 0).all()


# ---- 5. analytic evidence: polynomial regression --------------------------------------------------------------------
POLY_SIGMA, POLY_BOX, POLY_PRIOR_SIGMA = 3.0, 5.0, 2.0


@pytest.fixture(scope='module')
def poly():
    data = ds.poly_data(20000, sigma=POLY_SIGMA, seed=0)
    return data, ds.poly_params(data, sigma=POLY_SIGMA)


def _moments(x, w=None):
    x = np.asarray(x, dtype=np.float64)
    w = np.full(len(x), 1.0 / len(x)) if w is None else np.asarray(w, dtype=np.float64) / np.sum(w)
    mean = w @ x
    return mean, (x - mean).T @ ((x - mean) * w[:, None])


def _assert_posterior(mean, cov, ref_mean, ref_cov, mean_tol, cov_tol):
    sd = np.sqrt(np.diag(ref_cov))
    assert np.abs((mean - ref_mean) / sd).max() < mean_tol, (mean, ref_mean, sd)
    assert np.abs((cov - ref_cov) / np.outer(sd, sd)).max() < cov_tol, (cov, ref_cov)


@pytest.mark.parametrize('seed', [0, 1])
@pytest.mark.parametrize('prior', ['box', 'gauss'])
def test_evidence_polynomial_regression(tmp_path, poly, prior, seed):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood, CudaTransform
    data, params = poly
    d = 3
    np.random.seed(seed)
    torch.manual_seed(seed)
    like = CudaLikelihood(d, ds.POLY, params=params, data=data)
    if prior == 'box':
        transform = lambda x: POLY_BOX * x
        logz, mean, cov = ds.poly_closed_form(data, params, box=POLY_BOX)
    else:
        transform = CudaTransform(d, ts.GAUSS, params=[POLY_PRIOR_SIGMA])
        logz, mean, cov = ds.poly_closed_form(data, params, prior_cov=np.eye(d) * POLY_PRIOR_SIGMA ** 2)
    s = NestedSampler(d, like, transform=transform, num_live_points=1000, flow='nvp', log_dir=str(tmp_path),
                      log_level=logging.WARNING, seed=seed)
    s.run(mcmc_num_chains=1000, train_iters=200)
    assert abs(s.logz - logz) <= min(0.3, 3 * s.logzerr), (s.logz, s.logzerr, logz)
    _assert_posterior(*_moments(s.samples, s.weights), mean, cov, 0.3, 0.2)


# ---- 6. MCMCSampler -------------------------------------------------------------------------------------------------
def test_mcmc_sampler_posterior_and_derived(tmp_path, poly):
    from nnest_b200 import MCMCSampler
    from nnest_b200.likelihoods import CudaLikelihood
    from nnest_b200.priors import UniformPrior
    data, params = poly
    d = 3
    np.random.seed(1)
    torch.manual_seed(1)
    _, mean, cov = ds.poly_closed_form(data, params, box=POLY_BOX)
    like = CudaLikelihood(d, ds.POLY, params=params, data=data, num_derived=2)
    s = MCMCSampler(d, like, prior=UniformPrior(d, -POLY_BOX, POLY_BOX), flow='nvp', num_derived=2,
                    log_dir=str(tmp_path), log_level=logging.WARNING, seed=2)
    training = np.random.multivariate_normal(mean, cov, size=2000)
    s.run(200, 512, training, stats_interval=None, train_iters=100)
    assert s.samples.shape == (512, 201, d + 2)
    tail = s.samples[:, 50:, :d].reshape(-1, d)
    _assert_posterior(*_moments(tail), mean, cov, 0.15, 0.15)
    der = s.samples[..., d:].reshape(-1, 2)
    ref = ds.poly_derived_np(s.samples[..., :d].reshape(-1, d), data)
    assert np.allclose(der, ref, rtol=1e-11, atol=1e-12)
    # the log-likelihood the sampler kept is that of the returned point
    chi2 = ref[:, 0] * len(data['t'])
    assert np.allclose(s.loglikes.reshape(-1), -0.5 * params[0] * chi2 + params[1], rtol=0, atol=1e-7)


# ---- 7. two ranks ---------------------------------------------------------------------------------------------------
def _free_port():
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    p = sock.getsockname()[1]
    sock.close()
    return p


def test_two_rank_nested_run_with_data(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.abspath(__file__), str(tmp_path)]
    subprocess.run(cmd, check=True, timeout=900)
    res = [np.load(tmp_path / ('rank%d.npz' % r)) for r in range(2)]
    for k in res[0].files:
        assert np.array_equal(res[0][k], res[1][k]), k
    assert res[0]['derived_samples'].shape[1] == 2


def _worker(out_dir):
    """one rank of test_two_rank_nested_run_with_data (launched by torch.distributed.run)"""
    import torch.distributed as tdist
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood, CudaTransform
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    tdist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank = tdist.get_rank()
    np.random.seed(6)
    torch.manual_seed(6)
    data = ds.poly_data(20000, sigma=POLY_SIGMA, seed=0)
    like = CudaLikelihood(3, ds.POLY, params=ds.poly_params(data, sigma=POLY_SIGMA), data=data, num_derived=2)
    s = NestedSampler(3, like, transform=CudaTransform(3, ts.GAUSS, params=[POLY_PRIOR_SIGMA]), num_live_points=400,
                      flow='nvp', num_derived=2, log_dir=os.path.join(out_dir, 'run'), log_level=logging.WARNING,
                      seed=6)
    s.run(mcmc_num_chains=200, train_iters=30, max_iters=900, log_interval=300, strategy=['rejection_prior', 'mcmc'])
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), logz=s.logz, niter=s.niter, samples=s.samples,
             weights=s.weights, loglikes=s.loglikes, derived_samples=s.derived_samples)
    tdist.barrier()
    tdist.destroy_process_group()


if __name__ == '__main__':
    _worker(sys.argv[1])
