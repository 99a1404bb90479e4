"""Pins the CPU oracle (oracle/) against the golden vectors recorded from the real reference
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

from oracle import flow as oflow
from oracle import likelihoods as olike
from oracle import mcmc as omcmc
from oracle import nested as onested
from helpers import load, weights_of, rel_err, LIKE_CASES

FLOW_FILES = ['flow_d2.npz', 'flow_d3.npz', 'flow_d4.npz', 'flow_d5.npz', 'flow_d10_p.npz', 'flow_d30_p.npz',
              'flow_d50_p.npz', 'flow_d7_h32_l2_b5.npz', 'flow_d6_translate.npz', 'flow_d6_constant.npz']
TOL = 1e-5   # north_star: flow forward/inverse and log-det within 1e-5 relative


# the float32 oracle keeps its original ids; the float64 oracle (the reference of the GPU flow sweep) is one more dtype
@pytest.mark.parametrize('name,dtype', [pytest.param(n, np.float32, id=n) for n in FLOW_FILES] +
                         [pytest.param(n, np.float64, id=n + '-float64') for n in FLOW_FILES])
def test_flow_matches_reference(name, dtype):
    g = load(name)
    w = weights_of(g)
    z, ld = oflow.flow_forward(w, g['x'], dtype=dtype)
    assert z.dtype == dtype and ld.dtype == dtype
    assert rel_err(z, g['fwd_z']) < TOL
    assert np.allclose(ld, g['fwd_ld'], rtol=TOL, atol=1e-6)
    x, ldx = oflow.flow_inverse(w, g['zin'], dtype=dtype)
    assert rel_err(x, g['inv_x']) < TOL
    assert np.allclose(ldx, g['inv_ld'], rtol=TOL, atol=1e-6)
    # the properties tests/test_flows.py:56-72 checks on the reference
    xr, ldr = oflow.flow_inverse(w, z, dtype=dtype)
    assert np.abs(xr - g['x']).max() <= 2e-5
    assert np.abs(ldr + ld).max() <= 1e-5


def test_flat_weight_count():
    g = load('flow_d30_p.npz')
    w = weights_of(g)
    d, H, L, B = 30, 16, 1, 3
    assert w.flat().size == 2 * B * (H * (2 * d + L * H) + H * (L + 1) + d)   # SURVEY section 6 formula


@pytest.mark.parametrize('case', sorted(LIKE_CASES))
@pytest.mark.parametrize('dt', ['float32', 'float64'])
def test_likelihood_matches_reference(case, dt):
    g = load('like.npz')
    mk, a = LIKE_CASES[case]
    like = mk()
    u = g['%s/%s/u' % (case, dt)]
    v = g['%s/%s/v' % (case, dt)]
    ref = g['%s/%s/logl' % (case, dt)]
    tv = (u * 5 * np.pi) if a is None else a * u
    assert tv.dtype == v.dtype and np.array_equal(tv, v)
    rows = like.rows(v)
    batch = like.batch(v)
    assert rows.dtype == ref.dtype
    if case.startswith('gaussian'):
        # scipy's eigen-decomposition vs the closed form: identical to ~1e-12 relative
        assert np.allclose(rows, ref, rtol=1e-13, atol=0)
        assert np.allclose(batch, ref, rtol=1e-11, atol=1e-9)
    else:
        assert np.array_equal(rows, ref)
        if case in ('rosenbrock2', 'rosenbrock30', 'himmelblau'):
            assert np.array_equal(batch, ref) and batch.dtype == ref.dtype     # pure +,-,* : bit exact
        else:
            assert np.allclose(batch, ref, rtol=2e-6 if dt == 'float32' else 1e-13)


def test_prior_matches_reference():
    g = load('like.npz')
    pr = olike.UniformPrior(4, -1, 1)
    assert np.array_equal(pr.rows(g['prior/x']), g['prior/logp'])
    assert np.array_equal(pr.batch(g['prior/x']), g['prior/logp'])


HARD = {
    'mcmc_hard_rosen2.npz': (lambda: olike.Rosenbrock(2), lambda x: 5 * x),
    'mcmc_hard_himmel2_fixed.npz': (lambda: olike.Himmelblau(2), lambda x: 5 * x),
    'mcmc_hard_mix10.npz': (lambda: olike.GaussianMix(10), lambda x: 10 * x),
    'mcmc_hard_rosen30.npz': (lambda: olike.Rosenbrock(30), lambda x: 5 * x),
    'mcmc_hard_eggbox2.npz': (lambda: olike.Eggbox(2), lambda x: x * 5 * np.pi),
}


def _check_trace(out, g, tol=1e-5):
    samples, latent, derived, loglikes, scale, ncall = out
    moved_ref = np.any(g['latent'][:, 1:] != g['latent'][:, :-1], axis=2)
    moved = np.any(latent[:, 1:] != latent[:, :-1], axis=2)
    assert np.array_equal(moved, moved_ref), 'accept pattern differs from the reference'
    assert ncall == int(g['ncall'])
    assert scale == float(g['scale'])
    assert rel_err(latent, g['latent']) < tol
    assert rel_err(samples, g['samples']) < tol
    assert np.allclose(loglikes, g['loglikes'], rtol=1e-4, atol=1e-4)
    assert derived.shape == (latent.shape[0], latent.shape[1], 0)


@pytest.mark.parametrize('name', sorted(HARD))
@pytest.mark.parametrize('rowwise', [False, True])
def test_mcmc_hard_replay_matches_reference(name, rowwise):
    g = load(name)
    mk, tr = HARD[name]
    d = int(g['d'])
    target = omcmc.Target(mk(), transform=tr, prior=olike.UniformPrior(d, -1, 1), transform_prior=False,
                          rowwise=rowwise)
    out = omcmc.mcmc_sample(weights_of(g), target, int(g['steps']), omcmc.ReplayNoise(g['normals'], g['uniforms']),
                            step_size=float(g['step_size']), dynamic_step_size=bool(g['dynamic']),
                            init_samples=g['init_samples'], init_loglikes=g['init_loglikes'],
                            loglstar=float(g['loglstar']))
    _check_trace(out, g)
    assert target.total_calls == int(g['ncall'])


@pytest.mark.parametrize('name', ['mcmc_mh_gauss8.npz', 'mcmc_mh_gauss50.npz'])
def test_mcmc_mh_replay_matches_reference(name):
    g = load(name)
    d = int(g['d'])
    mean, std = g['mean'], g['std']
    target = omcmc.Target(olike.Gaussian(d, float(g['corr'])), transform=lambda x: x * std + mean,
                          prior=olike.UniformPrior(d, float(g['prior_min']), float(g['prior_max'])),
                          transform_prior=True)
    out = omcmc.mcmc_sample(weights_of(g), target, int(g['steps']), omcmc.ReplayNoise(g['normals'], g['uniforms']),
                            init_z=g['z0'], loglstar=None)
    _check_trace(out, g)


def test_nested_bookkeeping_matches_reference():
    g = load('nested_rosen2.npz')
    batches = list(zip(g['batches_first'], g['batches_last'], g['batches_logl'], g['loglstar'], g['idx']))
    it = iter(batches)
    tr = lambda x: 5 * x

    state = {}

    def randint(n, size):
        state['cur'] = next(it)
        return state['cur'][4]

    def batch_fn(init_samples, init_loglikes, loglstar):
        first, last, logl, lstar, idx = state['cur']
        assert loglstar == lstar                       # identical constraint sequence
        samples = np.stack([first, last], axis=1)
        loglikes = np.stack([np.zeros_like(logl), logl], axis=1)
        return samples, loglikes

    st, au, av, al, trace = onested.run_mcmc_strategy(g['active_u0'], g['active_logl0'], tr, batch_fn,
                                                      mcmc_num_chains=int(g['chains']), randint=randint)
    logz, h, samples, weights, loglikes, logzerr = onested.finalize(st, av, al)
    niter, ncall, logz_ref, logzerr_ref, h_ref = g['final_row']
    assert st.it + 1 == int(niter)
    assert logz == logz_ref == float(g['logz'])           # bit exact
    assert h == h_ref and logzerr == logzerr_ref
    assert np.array_equal(samples, g['samples'])
    assert np.array_equal(weights, g['weights'])
    assert np.array_equal(loglikes, g['loglikes'])
    with pytest.raises(StopIteration):
        next(it)                                           # every recorded batch was consumed


def _long_case():
    g = load('mcmc_long_rosen30.npz')
    b = load('bench_c4.npz')
    rng = np.random.RandomState(int(g['seed']))
    chains, steps, d = int(g['chains']), int(g['steps']), int(g['d'])
    normals = rng.normal(size=(steps, chains, d)).astype(np.float32)
    uniforms = rng.uniform(size=(steps, chains)).astype(np.float32)
    idx = rng.randint(0, 1024, size=chains)
    assert np.array_equal(idx, g['idx'])
    return g, b, normals, uniforms, idx


def compare_long(g, latent, samples, loglikes, ncall, max_flipped):
    """chains whose whole 150-step move pattern equals the reference's must end within 1e-5 of it; a chain may part ways at
    a near-tie of an accept test (SURVEY appendix D): at most `max_flipped` of 1024"""
    steps = int(g['steps'])
    moved_ref = np.unpackbits(g['moved_bits'], axis=1)[:, :steps].astype(bool)
    moved = np.any(latent[:, 1:] != latent[:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    assert (~same).sum() <= max_flipped, 'accept pattern differs in %d chains' % (~same).sum()
    assert rel_err(latent[same, -1], g['last_latent'][same]) < 1e-5
    assert rel_err(samples[same, -1], g['last_samples'][same]) < 1e-5
    assert rel_err(loglikes[same, -1], g['last_loglikes'][same]) < 1e-5
    if (~same).sum() == 0:
        assert ncall == int(g['ncall'])
    return int((~same).sum())


def test_long_replay_1024x150_d30_matches_reference():
    """VERDICT r1 item 9: one long replay (1024 chains x 150 steps, d = 30) recorded from the reference."""
    g, b, normals, uniforms, idx = _long_case()
    w = oflow.NVPWeights.from_state_dict({k[3:]: b[k] for k in b.files if k.startswith('sd/')}, 30)
    target = omcmc.Target(olike.Rosenbrock(30), transform=lambda x: 5 * x, prior=olike.UniformPrior(30, -1, 1),
                          transform_prior=False)
    au, al = b['active_u'].astype(np.float64), b['active_logl']
    out = omcmc.mcmc_sample(w, target, int(g['steps']), omcmc.ReplayNoise(normals, uniforms), step_size=float(g['step_size']),
                            dynamic_step_size=False, init_samples=au[idx], init_loglikes=al[idx],
                            loglstar=float(g['loglstar']))
    compare_long(g, out[1], out[0], out[3], out[5], max_flipped=2)
