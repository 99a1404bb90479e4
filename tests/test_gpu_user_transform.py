"""GPU: prior transforms written in CUDA C++ (CudaTransform / nnb_set_user_transform) run in the library's own kernels.
A user copy of the built-in affine map must reproduce the affine target bit for bit -- values, priors, derived values and
every chain, on every kernel variant, including those with an inline Rosenbrock that the user transform has to bypass;
non-affine priors (erfinv, exp, a Cholesky factor) agree with NumPy and with the MCMC oracle; nested sampling recovers
analytic evidences under Gaussian priors; the run plumbing (chain files, checkpoints, resume, rejection strategies,
derived parameters, two ranks) holds physical coordinates; compiled kernels are cached."""
import logging
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip('torch')

import transform_sources as ts
import user_sources as us
from helpers import load
from nnest_b200 import _lib as L
from oracle import flow as oflow
from oracle import likelihoods as olike
from oracle import mcmc as omcmc
from oracle import spline as ospline

pytestmark = pytest.mark.gpu

dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope='module')
def eng():
    from nnest_b200.engine import Engine
    return Engine(0)


def _affine_coeffs(d):
    return np.linspace(2.0, 5.0, d) + 1e-3, np.linspace(-0.5, 0.25, d)


def _target(eng, d, like_id, like_params=(), user_transform=False, compute_f64=False, prior=L.NNB_PRIOR_BOX_U,
            user_source=None, num_derived=0):
    """the affine target (built-in map) or its twin (the same map as a user transform)"""
    sc, sh = _affine_coeffs(d)
    kw = dict(prior_kind=prior, prior_lo=-1.0 if prior == L.NNB_PRIOR_BOX_U else -3.0,
              prior_hi=1.0 if prior == L.NNB_PRIOR_BOX_U else 3.5, user_source=user_source, num_derived=num_derived)
    if user_transform:
        eng.set_target(d, like_id, like_params, compute_f64=compute_f64, transform_source=ts.AFFINE,
                       transform_params=list(sc) + list(sh), **kw)
    else:
        eng.set_target(d, like_id, like_params, compute_f64=compute_f64, t_scale=sc, t_shift=sh, **kw)


# ---- 1. the affine twin, bit for bit --------------------------------------------------------------------------------
LIKES = {'rosen5': (5, L.NNB_LIKE_ROSENBROCK, None), 'rosen30': (30, L.NNB_LIKE_ROSENBROCK, None),
         'himmel': (2, L.NNB_LIKE_HIMMELBLAU, None), 'eggbox': (10, L.NNB_LIKE_EGGBOX, None),
         'user_rosen': (5, L.NNB_LIKE_USER, us.ROSENBROCK)}


@pytest.mark.parametrize('name', list(LIKES))
@pytest.mark.parametrize('f64_rows', [False, True])
@pytest.mark.parametrize('compute_f64', [False, True])
def test_affine_twin_loglike_and_prior(eng, name, f64_rows, compute_f64):
    d, like_id, src = LIKES[name]
    rng = np.random.RandomState(d)
    u = rng.uniform(-1.05, 1.05, size=(3000, d))
    u[:5] *= 1e80                                  # non-finite results: the clamp
    u = dev(u if f64_rows else u.astype(np.float32))
    out = []
    for user in (False, True):
        _target(eng, d, like_id, (), user_transform=user, compute_f64=compute_f64, prior=L.NNB_PRIOR_BOX_V,
                user_source=src)
        logl, logp = eng.loglike(u, want_prior=True)
        out.append((logl.cpu().numpy(), logp.cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert (out[0][1] == -np.inf).any() and (out[0][1] == 0).any()


DERIVED_X = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  double s = 0.0;
  for (int i = 0; i < d; ++i) { const double v = (double)x(i); s += v * v; }
  return -0.5 * s;
}
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  for (int i = 0; i < d; ++i) derived[i] = (double)x(i);
}
'''


@pytest.mark.parametrize('f64_rows', [False, True])
@pytest.mark.parametrize('compute_f64', [False, True])
def test_affine_twin_derived(eng, f64_rows, compute_f64):
    d = 4
    u = np.random.RandomState(2).uniform(-1, 1, size=(2000, d))
    u = dev(u if f64_rows else u.astype(np.float32))
    out = []
    for user in (False, True):
        _target(eng, d, L.NNB_LIKE_USER, (), user_transform=user, compute_f64=compute_f64, user_source=DERIVED_X,
                num_derived=d)
        out.append((eng.loglike(u).cpu().numpy(), eng.derived(u).cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def _nvp(eng, d, H=16, flags=0, seed=0):
    scale = {0: '', L.NNB_FLOW_TRANSLATE_ONLY: 'translate',
             L.NNB_FLOW_TRANSLATE_ONLY | L.NNB_FLOW_CONST_SCALE: 'constant'}[flags]
    w = oflow.NVPWeights.random(d, H, 1, 3, seed=seed, gain=0.5, scale=scale)
    eng.set_flow(w.flat(), d, H, 1, 3, flags)
    return w


def _spline(eng, d):
    g = load('spline_d5.npz')
    assert int(g['d']) == d
    w = ospline.SplineWeights.from_golden(g)
    eng.set_flow_spline(ospline.pack_for_kernel(w, int(g['hidden'])), d, int(g['hidden']), int(g['blocks']), w.K, w.B)


def _chains(eng, n, d, user, mode, dynamic, impl, steps, start, seed=7):
    _target(eng, d, L.NNB_LIKE_ROSENBROCK, (), user_transform=user)
    rng = np.random.RandomState(11)
    kw = {}
    if start == 'u':
        kw['init_u'] = dev(rng.uniform(-0.3, 0.3, size=(d, n)).astype(np.float32))
    elif start == 'z':
        kw['init_z'] = dev(rng.normal(size=(d, n)).astype(np.float32) * 0.3)
    st, nbad, ncall0 = eng.mcmc_init(n, seed=seed, want_counts=True, **kw)
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


H, M, MH = L.NNB_IMPL_FFMA, L.NNB_MODE_HARD, L.NNB_MODE_MH
TR, CS = L.NNB_FLOW_TRANSLATE_ONLY, L.NNB_FLOW_TRANSLATE_ONLY | L.NNB_FLOW_CONST_SCALE
# (flow, d, hidden, flags, n chains, impl, mode, dynamic step, expected impl that ran): every kernel variant; the
# 16-lane and tcgen05 rows on Rosenbrock run the lane-parallel and inline fast paths with the built-in map
VARIANTS = {
    'ffma_h16': ('nvp', 5, 16, 0, 700, L.NNB_IMPL_FFMA, M, True, L.NNB_IMPL_FFMA),
    'ffma_h32_translate': ('nvp', 5, 32, TR, 700, L.NNB_IMPL_AUTO, M, True, L.NNB_IMPL_FFMA),
    'ffma_h64_constant': ('nvp', 5, 64, CS, 700, L.NNB_IMPL_AUTO, M, True, L.NNB_IMPL_FFMA),
    'ffma_h16_fixed_step': ('nvp', 5, 16, 0, 700, L.NNB_IMPL_FFMA, M, False, L.NNB_IMPL_FFMA),
    'ffma_h16_mh': ('nvp', 5, 16, 0, 700, L.NNB_IMPL_FFMA, MH, False, L.NNB_IMPL_FFMA),
    'warp_generic': ('nvp', 5, 16, 0, 700, L.NNB_IMPL_AUTO, M, True, L.NNB_IMPL_WARP),
    'warp_d10': ('nvp', 10, 16, 0, 700, L.NNB_IMPL_WARP, M, True, L.NNB_IMPL_WARP),
    'tc_generic': ('nvp', 5, 16, 0, 20000, L.NNB_IMPL_AUTO, M, True, L.NNB_IMPL_TCGEN05),
    'tc_d10': ('nvp', 10, 16, 0, 20000, L.NNB_IMPL_TCGEN05, M, True, L.NNB_IMPL_TCGEN05),
    'tc_d30': ('nvp', 30, 16, 0, 20000, L.NNB_IMPL_TCGEN05, M, True, L.NNB_IMPL_TCGEN05),
    'tc_d30_mh': ('nvp', 30, 16, 0, 20000, L.NNB_IMPL_TCGEN05, MH, False, L.NNB_IMPL_TCGEN05),
    'spline': ('spline', 5, None, 0, 700, L.NNB_IMPL_AUTO, M, True, L.NNB_IMPL_FFMA),
    'spline_mh': ('spline', 5, None, 0, 700, L.NNB_IMPL_AUTO, MH, False, L.NNB_IMPL_FFMA),
}


@pytest.mark.parametrize('variant', list(VARIANTS))
def test_affine_twin_chains_bit_identical(eng, variant):
    flow, d, hid, flags, n, impl, mode, dynamic, impl_ran = VARIANTS[variant]
    if flow == 'spline':
        _spline(eng, d)
    else:
        _nvp(eng, d, hid, flags=flags)
    starts = ['u', 'z', 'philox'] if variant in ('ffma_h16', 'ffma_h32_translate', 'ffma_h64_constant', 'spline') \
        else ['philox']
    for start in starts:
        a = _chains(eng, n, d, False, mode, dynamic, impl, 12, start)
        b = _chains(eng, n, d, True, mode, dynamic, impl, 12, start)
        assert a['impl'] == impl_ran and b['impl'] == impl_ran
        assert a['naccept'] > 0 and a['naccept'] < n * 12
        assert a.keys() == b.keys()
        for k in a:
            if isinstance(a[k], np.ndarray):
                assert np.array_equal(a[k], b[k]), k
            else:
                assert a[k] == b[k], (k, a[k], b[k])


# ---- 2. non-affine priors against NumPy -----------------------------------------------------------------------------
def _cases(d):
    return {'gauss': (ts.GAUSS, [3.0], lambda u: ts.gauss_np(u, 3.0)),
            'loguniform': (ts.LOGUNIFORM, [np.log(1e-3), np.log(10.0)],
                           lambda u: ts.loguniform_np(u, np.log(1e-3), np.log(10.0))),
            'cholesky': (ts.CHOLESKY, list(ts.CHOL_P.ravel()), lambda u: ts.cholesky_np(u, ts.CHOL_P))}


@pytest.mark.parametrize('case', ['gauss', 'loguniform', 'cholesky'])
@pytest.mark.parametrize('float64', [True, False])
def test_transform_against_numpy(case, float64):
    from nnest_b200.likelihoods import CudaTransform
    d = 3
    src, params, ref = _cases(d)[case]
    t = CudaTransform(d, src, params=params, float64=float64)
    u = np.random.RandomState(4).uniform(-0.999, 0.999, size=(4000, d))
    want = ref(u)
    v = t(u)                                           # float64 rows: always double
    assert v.dtype == np.float64 and v.shape == u.shape
    assert np.allclose(v, want, rtol=1e-12, atol=1e-12 * np.abs(want).max())
    assert np.array_equal(t(u[7]), v[7])               # one row
    u32 = u.astype(np.float32)
    v32 = t(u32)
    want32 = ref(u32.astype(np.float64))
    if float64:                                        # float32 rows promoted: the double transform of the same values
        assert v32.dtype == np.float64
        assert np.allclose(v32, want32, rtol=1e-12, atol=1e-12 * np.abs(want32).max())
    else:                                              # float arithmetic: a few float32 ulps
        assert v32.dtype == np.float32
        assert np.allclose(v32, want32, rtol=8e-7 * (4 if case == 'cholesky' else 1), atol=1e-6 * np.abs(want32).max())


@pytest.mark.parametrize('impl,d,n', [(L.NNB_IMPL_FFMA, 5, 700), (L.NNB_IMPL_WARP, 5, 700),
                                      (L.NNB_IMPL_TCGEN05, 10, 20000)])
def test_gaussian_prior_chains_against_oracle(eng, impl, d, n):
    from nnest_b200.likelihoods import CudaTransform
    sigma, steps = 3.0, 10
    w = _nvp(eng, d, 16, seed=3)
    t = CudaTransform(d, ts.GAUSS, params=[sigma])
    t.install(eng, d, L.NNB_LIKE_GAUSSIAN, [0.0], prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)
    rng = np.random.RandomState(5)
    u0 = rng.uniform(-0.6, 0.6, size=(n, d)).astype(np.float32)
    st, _, _ = eng.mcmc_init(n, init_u=dev(u0.T), seed=1)
    logl0 = st.logl.cpu().numpy()
    target = omcmc.Target(olike.Gaussian(d, 0.0), transform=lambda x: ts.gauss_np(x, sigma),
                          prior=olike.UniformPrior(d, -1.0, 1.0), transform_prior=False)
    x0 = oflow.flow_inverse(w, oflow.flow_forward(w, u0)[0])[0]
    assert np.allclose(logl0, target.loglike(x0), rtol=1e-5, atol=1e-5)
    loglstar = float(np.quantile(logl0, 0.3))
    out = eng.mcmc_run(st, steps, mode=L.NNB_MODE_HARD, loglstar=loglstar, step_size=0.3, dynamic_step_size=True,
                       seed=1, trace=True, dump_noise=True, impl=impl)
    assert out['impl'] == impl
    ref = omcmc.mcmc_sample(w, target, steps, omcmc.ReplayNoise(out['normals'].cpu().numpy(),
                                                                 out['uniforms'].cpu().numpy()),
                            step_size=0.3, dynamic_step_size=True, init_samples=u0, init_loglikes=logl0,
                            loglstar=loglstar)
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    moved = np.any(samples[:, 1:] != samples[:, :-1], axis=2)
    moved_ref = np.any(ref[0][:, 1:] != ref[0][:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    # near-tie flips of the accept test (float32 flow on the device, float64 oracle), as the other oracle replays allow
    assert (~same).sum() <= max(2, n // 2000) and moved.sum() > n
    assert np.abs(samples[same] - ref[0][same]).max() <= 1e-5 * max(1.0, np.abs(ref[0]).max())
    logl = out['trace_logl'].t().cpu().numpy()
    assert np.allclose(logl[same], ref[3][same], rtol=1e-5, atol=1e-5)
    # and the values the host gets back are those the likelihood saw: physical rows of the trace
    v = eng.transform_trace(out['trace_x']).cpu().numpy()              # (T, d, n)
    assert np.array_equal(v[-1].T, eng.transform(st.x.t()).cpu().numpy())


# ---- 3. host values equal the kernel's ------------------------------------------------------------------------------
@pytest.mark.parametrize('float64', [True, False])
def test_host_transform_equals_what_the_likelihood_saw(eng, float64):
    from nnest_b200.likelihoods import CudaTransform
    d = 3
    t = CudaTransform(d, ts.CHOLESKY, params=list(ts.CHOL_P.ravel()), float64=float64)
    t.install(eng, d, L.NNB_LIKE_USER, (), user_source=DERIVED_X, num_derived=d)
    u = np.random.RandomState(6).uniform(-0.99, 0.99, size=(3000, d))
    for rows in (u, u.astype(np.float32)):
        der = eng.derived(dev(rows)).cpu().numpy()
        assert np.array_equal(der, t.apply(eng, rows).astype(np.float64))
        assert np.array_equal(der, eng.transform(dev(rows)).cpu().numpy())


# ---- 4. analytic evidence -------------------------------------------------------------------------------------------
def _nested(tmp_path, d, transform, seed, **kw):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import Gaussian
    np.random.seed(seed)
    torch.manual_seed(seed)
    s = NestedSampler(d, Gaussian(d, 0.0), transform=transform, num_live_points=1000, flow='nvp',
                      log_dir=str(tmp_path), log_level=logging.WARNING, seed=seed, **kw)
    return s


def _posterior_moments(s):
    w = np.asarray(s.weights, dtype=np.float64)
    w = w / w.sum()
    x = np.asarray(s.samples, dtype=np.float64)
    mean = w @ x
    cov = (x - mean).T @ ((x - mean) * w[:, None])
    return mean, cov


@pytest.mark.parametrize('seed', [0, 1])
def test_evidence_gaussian_prior(tmp_path, seed):
    from nnest_b200.likelihoods import CudaTransform
    d, sigma = 5, 3.0
    s = _nested(tmp_path, d, CudaTransform(d, ts.GAUSS, params=[sigma]), seed)
    s.run(mcmc_num_chains=1000, train_iters=200)
    logz = -(d / 2.0) * np.log(2 * np.pi * (1 + sigma ** 2))          # -10.35
    assert abs(s.logz - logz) <= min(0.3, 3 * s.logzerr), (s.logz, s.logzerr, logz)
    mean, cov = _posterior_moments(s)
    var = sigma ** 2 / (1 + sigma ** 2)                                # 0.9
    assert np.abs(mean).max() < 0.1, mean
    assert np.abs(np.diag(cov) - var).max() < 0.12 and np.abs(cov - np.diag(np.diag(cov))).max() < 0.1, cov


@pytest.mark.parametrize('seed', [0, 1])
def test_evidence_correlated_prior(tmp_path, seed):
    from nnest_b200.likelihoods import CudaTransform
    d, sp = 3, ts.SIGMA_P
    s = _nested(tmp_path, d, CudaTransform(d, ts.CHOLESKY, params=list(ts.CHOL_P.ravel())), seed)
    s.run(mcmc_num_chains=1000, train_iters=200)
    logz = -0.5 * np.linalg.slogdet(2 * np.pi * (np.eye(d) + sp))[1]
    assert abs(s.logz - logz) <= min(0.3, 3 * s.logzerr), (s.logz, s.logzerr, logz)
    mean, cov = _posterior_moments(s)
    post = sp @ np.linalg.inv(np.eye(d) + sp)
    assert np.abs(mean).max() < 0.1, mean
    assert np.abs(cov - post).max() < 0.12, (cov, post)


# ---- 5. run plumbing ------------------------------------------------------------------------------------------------
def _ns_small(log_dir, seed=0, num_derived=0, **run_kw):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood, CudaTransform, Gaussian
    np.random.seed(seed)
    torch.manual_seed(seed)
    d = 3
    like = CudaLikelihood(d, DERIVED_X, num_derived=d) if num_derived else Gaussian(d, 0.0)
    s = NestedSampler(d, like, transform=CudaTransform(d, ts.GAUSS, params=[2.0]), num_live_points=400, flow='nvp',
                      num_derived=num_derived, log_dir=str(log_dir), log_level=logging.WARNING, seed=seed)
    s.run(**run_kw)
    return s


def test_chain_file_and_checkpoint_hold_physical_samples(tmp_path):
    s = _ns_small(tmp_path, seed=2, mcmc_num_chains=200, train_iters=30, max_iters=800, log_interval=300,
                  strategy=['mcmc'])
    rows = np.loadtxt(os.path.join(s.logs['chains'], 'chain.txt'))
    assert rows.shape == (len(s.loglikes), 2 + 3)
    assert np.array_equal(rows[:, 2:], np.array([['%.5E' % v for v in r] for r in s.samples], dtype=float))
    # a Gaussian prior of width 2: physical samples leave the unit box
    assert np.abs(s.samples).max() > 1.5
    ck = s.logs['checkpoint']
    its = sorted(int(f.split('checkpoint_')[1].split('.txt')[0]) for f in os.listdir(ck) if f.startswith('checkpoint_'))
    au = np.load(os.path.join(ck, 'active_u_%d.npy' % its[-1]))
    av = np.load(os.path.join(ck, 'active_v_%d.npy' % its[-1]))
    assert np.array_equal(av, s.transform(au))
    assert np.array_equal(av, ts.gauss_np(au, 2.0)) or np.allclose(av, ts.gauss_np(au, 2.0), rtol=1e-12, atol=1e-12)


def test_resume_restores_physical_points_bit_for_bit(tmp_path):
    kw = dict(mcmc_num_chains=200, train_iters=30, log_interval=300, strategy=['mcmc'])
    s1 = _ns_small(tmp_path, seed=3, max_iters=700, **kw)
    run_dir = s1.logs['run_dir']
    ck = os.path.join(run_dir, 'checkpoint')
    its = sorted(int(f.split('checkpoint_')[1].split('.txt')[0]) for f in os.listdir(ck) if f.startswith('checkpoint_'))
    last = its[-1]
    assert last >= 600
    saved_v = np.load(os.path.join(ck, 'saved_v.npy')).reshape(last, 3)
    active_v = np.load(os.path.join(ck, 'active_v_%d.npy' % last))
    assert np.array_equal(saved_v, s1.samples[:last])
    s2 = _ns_small(run_dir, seed=4, **kw)
    assert not s2.logs['created'] and s2.niter > s1.niter
    # the resumed run carries the checkpoint's dead points as they were, and re-forms the live points' physical
    # coordinates from active_u with the same bits the first run wrote
    assert np.array_equal(s2.samples[:last], saved_v)
    assert np.array_equal(s2.transform(np.load(os.path.join(ck, 'active_u_%d.npy' % last))), active_v)
    logz = -1.5 * np.log(2 * np.pi * 5.0)                              # N(0, I) likelihood under N(0, 4 I)
    assert abs(s2.logz - logz) <= 0.3 + 3 * s2.logzerr, (s2.logz, logz)


def test_rejection_strategies_and_derived(tmp_path):
    s = _ns_small(tmp_path, seed=5, num_derived=3, strategy=['rejection_prior', 'rejection_flow'], volume_switch=0.3,
                  max_iters=900, train_iters=30, log_interval=300)
    # the derived parameters are x(i): the physical live points themselves
    assert np.array_equal(s.active_derived, s.transform(s.active_u))
    assert np.array_equal(s.derived_samples, s.samples)
    d = _ns_small(tmp_path / 'density', seed=6, strategy=['density_flow'], max_iters=500, train_iters=30,
                  log_interval=300)
    assert np.isfinite(d.logz) and np.abs(d.samples).max() > 1.0


def test_mcmc_sample_stats_of_transformed_samples(tmp_path, caplog):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaTransform, Gaussian
    d = 3
    s = NestedSampler(d, Gaussian(d, 0.0), transform=CudaTransform(d, ts.GAUSS, params=[2.0]), num_live_points=100,
                      flow='nvp', log_dir=str(tmp_path), log_level=logging.INFO)
    u = np.random.RandomState(1).uniform(-0.5, 0.5, size=(64, d)).astype(np.float32)
    logl, _ = s.loglike(u)
    with caplog.at_level(logging.INFO):
        out = s._mcmc_sample(8, init_samples=u, init_loglikes=logl, loglstar=None, step_size=0.3, stats_interval=8)
    assert any('Step [8] acceptance' in r.getMessage() for r in caplog.records)
    v = s.engine.transform_trace(s._device_trace).cpu().numpy().transpose(2, 0, 1)
    assert np.array_equal(v, s.transform(out[0].reshape(-1, d)).reshape(v.shape))


# ---- 6. compile counts and caches -----------------------------------------------------------------------------------
def test_compile_only_what_runs_and_caches(tmp_path, monkeypatch):
    from nnest_b200.engine import Engine
    monkeypatch.setenv('NNB_JIT_CACHE', str(tmp_path / 'jit'))
    src = ts.GAUSS + '\n// cache test %d\n' % np.random.randint(1 << 30)      # a source no cache has seen
    d, n = 5, 700
    e = Engine(0)
    _nvp(e, d)
    assert e.set_user_transform(src) == 1                      # the likelihood kernels with the row kernels
    aff = dict(prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)

    def run(eng):
        st, _, _ = eng.mcmc_init(n, seed=3, want_counts=True)
        return eng.mcmc_run(st, 4, mode=L.NNB_MODE_MH, seed=3, impl=L.NNB_IMPL_FFMA, trace=True)

    e.set_target(d, L.NNB_LIKE_GAUSSIAN, [0.0], compute_f64=True, transform_source=src, transform_params=[3.0], **aff)
    a = run(e)
    b = run(e)
    assert np.array_equal(a['trace_x'].cpu().numpy(), b['trace_x'].cpu().numpy())
    cubins = set((tmp_path / 'jit').glob('*.cubin'))
    assert len(cubins) == 3                                     # row kernels, chain start, one step kernel
    e2 = Engine(0)
    _nvp(e2, d)
    assert e2.set_user_transform(src) == 0                      # on-disk cache
    e2.set_target(d, L.NNB_LIKE_GAUSSIAN, [0.0], compute_f64=True, transform_source=src, transform_params=[3.0], **aff)
    c = run(e2)
    assert np.array_equal(a['trace_x'].cpu().numpy(), c['trace_x'].cpu().numpy())
    assert set((tmp_path / 'jit').glob('*.cubin')) == cubins and not list((tmp_path / 'jit').glob('*.tmp*'))
    # a different source recompiles
    assert e2.set_user_transform(src + '\n// changed\n') == 1
    # back to an affine target: the ahead-of-time kernels, no new variant, the same bits as a handle that never saw a
    # user transform
    e.set_target(d, L.NNB_LIKE_GAUSSIAN, [0.0], compute_f64=True, t_scale=3.0, t_shift=0.0, **aff)
    x = run(e)
    e3 = Engine(0)
    _nvp(e3, d)
    e3.set_target(d, L.NNB_LIKE_GAUSSIAN, [0.0], compute_f64=True, t_scale=3.0, t_shift=0.0, **aff)
    y = run(e3)
    assert np.array_equal(x['trace_x'].cpu().numpy(), y['trace_x'].cpu().numpy())
    assert len(set((tmp_path / 'jit').glob('*.cubin'))) == 4
    # state errors: no transform installed on a fresh handle, nnb_transform without a user transform
    import ctypes as C
    t = L.nnb_target()
    t.like_id = L.NNB_LIKE_ROSENBROCK
    assert e3.lib.nnb_set_target_user_transform(e3.h, 2, C.byref(t), None, 0) == L.NNB_ERR_STATE
    with pytest.raises(L.NNBError):
        e3.transform(dev(np.zeros((2, d))))


# ---- 7. two ranks ---------------------------------------------------------------------------------------------------
def _free_port():
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    p = sock.getsockname()[1]
    sock.close()
    return p


def test_two_rank_nested_run_with_transform(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.abspath(__file__), str(tmp_path)]
    subprocess.run(cmd, check=True, timeout=900)
    res = [np.load(tmp_path / ('rank%d.npz' % r)) for r in range(2)]
    for k in res[0].files:
        assert np.array_equal(res[0][k], res[1][k]), k
    assert np.abs(res[0]['samples']).max() > 1.5


def _worker(out_dir):
    """one rank of test_two_rank_nested_run_with_transform (launched by torch.distributed.run)"""
    import torch.distributed as tdist
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    tdist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank = tdist.get_rank()
    s = _ns_small(os.path.join(out_dir, 'run'), seed=6, num_derived=3, mcmc_num_chains=200, train_iters=30,
                  max_iters=900, log_interval=300, strategy=['rejection_prior', 'mcmc'])
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), logz=s.logz, niter=s.niter, samples=s.samples,
             weights=s.weights, loglikes=s.loglikes, derived_samples=s.derived_samples)
    tdist.barrier()
    tdist.destroy_process_group()


if __name__ == '__main__':
    _worker(sys.argv[1])
