"""GPU: user likelihoods written in CUDA C++ (CudaLikelihood / nnb_set_user_likelihood) run in the library's own step
kernels.  A user copy of a built-in likelihood must reproduce it bit for bit -- its values and every chain it drives, on
every kernel variant AUTO or an explicit impl reaches; a likelihood with no built-in twin is replayed through the MCMC
oracle; the samplers run on user likelihoods; compiled kernels are cached."""
import ctypes as C
import logging

import numpy as np
import pytest

torch = pytest.importorskip('torch')

import user_sources as us
from helpers import load
from nnest_b200 import _lib as L
from oracle import flow as oflow
from oracle import mcmc as omcmc
from oracle import spline as ospline

pytestmark = pytest.mark.gpu

dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
BUILTIN = {'rosen': (L.NNB_LIKE_ROSENBROCK, us.ROSENBROCK), 'himmel': (L.NNB_LIKE_HIMMELBLAU, us.HIMMELBLAU),
           'eggbox': (L.NNB_LIKE_EGGBOX, us.EGGBOX)}


@pytest.fixture(scope='module')
def eng():
    from nnest_b200.engine import Engine
    e = Engine(0)
    e.set_user_likelihood(us.ROSENBROCK)
    return e


def _target(eng, d, like_id, source, transform=True, prior=True, compute_f64=False, params=()):
    kw = dict(t_scale=np.linspace(2.0, 5.0, d), t_shift=np.linspace(-0.5, 0.25, d)) if transform else {}
    if prior:
        kw.update(prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)
    eng.set_target(d, like_id, params, compute_f64=compute_f64, user_source=source, **kw)


@pytest.mark.parametrize('name,d', [('rosen', 5), ('rosen', 30), ('himmel', 2), ('eggbox', 2), ('eggbox', 10)])
@pytest.mark.parametrize('f64', [False, True])
@pytest.mark.parametrize('transform', [False, True])
def test_loglike_bit_identical_to_builtin(eng, name, d, f64, transform):
    like_id, src = BUILTIN[name]
    rng = np.random.RandomState(d)
    u = rng.uniform(-1.05, 1.05, size=(3000, d))     # some rows outside the prior box, most inside
    u[:5] *= 1e80                                  # non-finite results: the clamp
    u = dev(u if f64 else u.astype(np.float32))
    out = []
    for lid, s in ((like_id, None), (L.NNB_LIKE_USER, src)):
        _target(eng, d, lid, s, transform=transform, prior=True, compute_f64=False)
        logl, logp = eng.loglike(u, want_prior=True)
        out.append((logl.cpu().numpy(), logp.cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert (out[0][1] == -np.inf).any() and (out[0][1] == 0).any()
    if name == 'rosen':
        assert (~np.isfinite(out[0][0])).any() or (out[0][0] <= -1e100).any()


def _nvp(eng, d, H=16, L_=1, B=3, flags=0, seed=0):
    scale = {0: '', L.NNB_FLOW_TRANSLATE_ONLY: 'translate',
             L.NNB_FLOW_TRANSLATE_ONLY | L.NNB_FLOW_CONST_SCALE: 'constant'}[flags]
    w = oflow.NVPWeights.random(d, H, L_, B, seed=seed, gain=0.5, scale=scale)
    eng.set_flow(w.flat(), d, H, L_, B, flags)


def _spline(eng, d):
    g = load('spline_d5.npz')
    assert int(g['d']) == d
    w = ospline.SplineWeights.from_golden(g)
    eng.set_flow_spline(ospline.pack_for_kernel(w, int(g['hidden'])), d, int(g['hidden']), int(g['blocks']), w.K, w.B)


def _chains(eng, n, d, like_id, source, mode, dynamic, impl, steps, start, seed=7):
    _target(eng, d, like_id, source)
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


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), k
        else:
            assert a[k] == b[k], (k, a[k], b[k])


H, M, MH = L.NNB_IMPL_FFMA, L.NNB_MODE_HARD, L.NNB_MODE_MH
TR, CS = L.NNB_FLOW_TRANSLATE_ONLY, L.NNB_FLOW_TRANSLATE_ONLY | L.NNB_FLOW_CONST_SCALE
# (flow, d, hidden, flags, n chains, impl, mode, dynamic step, expected impl that ran)
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
def test_user_rosenbrock_chains_bit_identical(eng, variant):
    flow, d, hid, flags, n, impl, mode, dynamic, impl_ran = VARIANTS[variant]
    if flow == 'spline':
        _spline(eng, d)
    else:
        _nvp(eng, d, hid, flags=flags)
    starts = ['u', 'z', 'philox'] if variant in ('ffma_h16', 'ffma_h32_translate', 'ffma_h64_constant', 'spline') \
        else ['philox']
    for start in starts:
        a = _chains(eng, n, d, L.NNB_LIKE_ROSENBROCK, None, mode, dynamic, impl, 12, start)
        b = _chains(eng, n, d, L.NNB_LIKE_USER, us.ROSENBROCK, mode, dynamic, impl, 12, start)
        assert a['impl'] == impl_ran
        assert a['naccept'] > 0 and a['naccept'] < n * 12
        _assert_same(a, b)


class _GaussOracle(object):
    """the `batch()` interface oracle.mcmc.Target expects: log N(x; mu, C), float64"""

    def __init__(self, mu, prec, lognorm):
        self.mu, self.prec, self.lognorm = mu, prec, lognorm

    def batch(self, x):
        dx = np.asarray(x, dtype=np.float64) - self.mu
        return -0.5 * np.einsum('ni,ij,nj->n', dx, self.prec, dx) + self.lognorm


def test_user_gaussian30_full_covariance_against_oracle(eng):
    d, n, steps = 30, 1024, 10
    rng = np.random.RandomState(5)
    a = rng.normal(size=(d, d)) * 0.3
    cov = a @ a.T + np.eye(d)
    prec = np.linalg.inv(cov)
    mu = rng.uniform(-0.2, 0.2, size=d)
    lognorm = -0.5 * (np.linalg.slogdet(cov)[1] + d * np.log(2 * np.pi))
    src = us.gauss_full_source(prec)
    w = oflow.NVPWeights.random(d, 16, 1, 3, seed=3, gain=0.5)
    eng.set_flow(w.flat(), d, 16, 1, 3, 0)
    eng.set_target(d, L.NNB_LIKE_USER, list(mu) + [lognorm], user_source=src)
    u0 = rng.normal(size=(n, d)).astype(np.float32) * 0.5
    st, _, _ = eng.mcmc_init(n, init_u=dev(u0.T), seed=1)
    logl0 = st.logl.cpu().numpy()
    target = omcmc.Target(_GaussOracle(mu, prec, lognorm))
    out = eng.mcmc_run(st, steps, mode=L.NNB_MODE_MH, step_size=0.3, seed=1, trace=True, dump_noise=True,
                       impl=L.NNB_IMPL_FFMA)
    x0 = oflow.flow_inverse(w, oflow.flow_forward(w, u0)[0])[0]
    assert np.allclose(logl0, target.loglike(x0), rtol=1e-5, atol=1e-5)
    ref = omcmc.mcmc_sample(w, target, steps, omcmc.ReplayNoise(out['normals'].cpu().numpy(),
                                                                 out['uniforms'].cpu().numpy()),
                            step_size=0.3, init_samples=u0, init_loglikes=logl0)
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    moved = np.any(samples[:, 1:] != samples[:, :-1], axis=2)
    moved_ref = np.any(ref[0][:, 1:] != ref[0][:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    assert (~same).sum() <= 2 and moved.sum() > n
    assert np.abs(samples[same] - ref[0][same]).max() <= 1e-5 * max(1.0, np.abs(ref[0]).max())
    logl = out['trace_logl'].t().cpu().numpy()
    assert np.allclose(logl[same], ref[3][same], rtol=1e-5, atol=1e-5)
    assert out['ncall'] == ref[5]


def _shell_logz(sigma=0.1, rshell=2.0, lim=5.0):
    """analytic evidence of the 2-D Gaussian shell under the uniform prior on [-lim, lim]^2"""
    from scipy import integrate
    val, _ = integrate.quad(lambda r: 2 * np.pi * r * np.exp(-(r - rshell) ** 2 / (2 * sigma ** 2)), 0, 4 * rshell)
    return np.log(val / (2 * lim) ** 2)


@pytest.mark.parametrize('case', ['rosen2', 'shell2'])
def test_nested_sampler_on_user_likelihood(tmp_path, case):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood
    np.random.seed(0)
    torch.manual_seed(0)
    if case == 'rosen2':
        like, logz = CudaLikelihood(2, us.ROSENBROCK), -5.8041     # SURVEY.md section 6
    else:
        like, logz = CudaLikelihood(2, us.SHELL, params=[0.1, 2.0, 0.0, 0.0]), _shell_logz()
    s = NestedSampler(2, like, transform=lambda x: 5 * x, num_live_points=1000, log_dir=str(tmp_path),
                      log_level=logging.WARNING)
    s.run(mcmc_num_chains=1000, train_iters=200)
    assert abs(s.logz - logz) <= 0.2, (s.logz, logz)
    assert s.total_calls > 1000


def test_mcmc_sampler_on_user_likelihood_counts_calls(tmp_path):
    from nnest_b200 import MCMCSampler
    from nnest_b200.likelihoods import CudaLikelihood
    from nnest_b200.priors import UniformPrior
    np.random.seed(1)
    torch.manual_seed(1)
    d = 4
    prec = np.eye(d) * 2.0
    like = CudaLikelihood(d, us.gauss_full_source(prec), params=[0.0] * d + [0.0])
    s = MCMCSampler(d, like, prior=UniformPrior(d, -8, 8), flow='nvp', log_dir=str(tmp_path), log_level=logging.WARNING)
    training = np.random.normal(size=(2000, d)) / np.sqrt(2.0)
    calls0 = s.total_calls
    s.run(200, 512, training, stats_interval=None, train_iters=100)
    assert s.samples.shape == (512, 201, d)
    tail = s.samples[:, 50:, :].reshape(-1, d)
    assert np.abs(tail.mean(0)).max() < 0.1 and np.abs(tail.var(0) - 0.5).max() < 0.1
    assert s.total_calls > calls0
    # the direct call of the likelihood runs the user's kernel too
    assert np.allclose(like(np.zeros((3, d))), 0.0)


def test_cache_and_state_errors(tmp_path, monkeypatch):
    from nnest_b200.engine import Engine
    monkeypatch.setenv('NNB_JIT_CACHE', str(tmp_path / 'jit'))
    e = Engine(0)
    # NNB_LIKE_USER before any source: NNB_ERR_STATE
    t = L.nnb_target()
    t.like_id = L.NNB_LIKE_USER
    assert e.lib.nnb_set_target(e.h, 2, C.byref(t)) == L.NNB_ERR_STATE
    src = us.HIMMELBLAU + '\n// cache test %d\n' % np.random.randint(1 << 30)     # a source no cache has seen
    assert e.set_user_likelihood(src) >= 1
    assert e.set_user_likelihood(src) == 0          # per-handle cache
    e2 = Engine(0)
    assert e2.set_user_likelihood(src) == 0         # on-disk cache
    assert len(list((tmp_path / 'jit').glob('*.cubin'))) >= 1
    assert not list((tmp_path / 'jit').glob('*.tmp*'))
    # a source that does not compile is refused with the log, and the installed one stays
    n = C.c_int(-1)
    assert e.lib.nnb_set_user_likelihood(e.h, us.SYNTAX_ERROR.encode(), C.byref(n)) == L.NNB_ERR_ARG and n.value == 0
    assert b'user_likelihood.cu(5)' in e.lib.nnb_last_error(e.h)
    e.set_target(2, L.NNB_LIKE_USER, ())
    assert np.isfinite(e.loglike(dev(np.zeros((4, 2)))).cpu().numpy()).all()
