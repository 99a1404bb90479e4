"""GPU parity tests: libnnb.so (through the C ABI, nnest_b200.engine) against the committed golden
vectors of the real reference and against the CPU oracle on the same seeded inputs.

Tolerances: flow forward/inverse/log-det 1e-5 relative (north_star); +,-,* likelihoods bit exact;
transcendental likelihoods 2e-6 (float32) / 1e-12 (float64) relative.
"""
import numpy as np
import pytest

torch = pytest.importorskip('torch')

from oracle import flow as oflow
from oracle import likelihoods as olike
from oracle import mcmc as omcmc
from oracle import philox as ophilox
from helpers import load, weights_of, state_dict_of, rel_err, LIKE_CASES

pytestmark = pytest.mark.gpu

FLOW_FILES = ['flow_d2.npz', 'flow_d3.npz', 'flow_d4.npz', 'flow_d5.npz', 'flow_d10_p.npz', 'flow_d30_p.npz',
              'flow_d50_p.npz', 'flow_d7_h32_l2_b5.npz', 'flow_d6_translate.npz', 'flow_d6_constant.npz']
TOL = 1e-5


@pytest.fixture(scope='module')
def engine():
    from nnest_b200.engine import Engine
    return Engine(0)


def _scale_of(g):
    return str(g['scale']) if g['scale'].dtype.kind in 'US' else ''


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


@pytest.mark.parametrize('name', FLOW_FILES)
def test_flow_matches_reference_golden(engine, name):
    g = load(name)
    engine.set_flow_from_state_dict(state_dict_of(g), scale=_scale_of(g))
    z, ld = engine.flow_forward(dev(g['x']))
    assert rel_err(z.cpu().numpy(), g['fwd_z']) < TOL
    assert np.allclose(ld.cpu().numpy(), g['fwd_ld'], rtol=TOL, atol=1e-6)
    x, ldx = engine.flow_inverse(dev(g['zin']))
    assert rel_err(x.cpu().numpy(), g['inv_x']) < TOL
    assert np.allclose(ldx.cpu().numpy(), g['inv_ld'], rtol=TOL, atol=1e-6)
    # reference's own test properties (tests/test_flows.py:56-72)
    xr, ldr = engine.flow_inverse(z)
    assert np.abs(xr.cpu().numpy() - g['x']).max() <= 2e-5
    assert np.abs((ldr + ld).cpu().numpy()).max() <= 1e-5


def test_flow_strided_views_and_ragged_sizes(engine):
    g = load('flow_d5.npz')
    w = weights_of(g)
    engine.set_flow_from_state_dict(state_dict_of(g))
    rng = np.random.RandomState(0)
    for n in (0, 1, 127, 128, 129, 1000):
        zin = rng.normal(size=(n, 5)).astype(np.float32)
        x, ld = engine.flow_inverse(dev(zin))
        assert x.shape == (n, 5) and ld.shape == (n,)
        if n:
            xo, ldo = oflow.flow_inverse(w, zin)
            assert rel_err(x.cpu().numpy(), xo) < TOL
            # chain-minor (transposed) view must give the same numbers
            zt = dev(zin.T.copy()).t()
            x2, ld2 = engine.flow_inverse(zt)
            assert torch.equal(x2, x) and torch.equal(ld2, ld)


def test_flow_full_size_properties(engine):
    """Config-4 size (65536 x 30): round trip and log-det antisymmetry, no oracle needed."""
    g = load('flow_d30_p.npz')
    engine.set_flow_from_state_dict(state_dict_of(g))
    torch.manual_seed(0)
    x = torch.rand((65536, 30), device='cuda') * 2 - 1
    z, ldz = engine.flow_forward(x)
    xr, ldx = engine.flow_inverse(z)
    assert torch.isfinite(z).all()
    assert (xr - x).abs().max().item() <= 5e-5
    assert (ldz + ldx).abs().max().item() <= 5e-5
    sub = slice(1000, 1256)
    zo, ldo = oflow.flow_forward(weights_of(g), x[sub].cpu().numpy())
    assert rel_err(z[sub].cpu().numpy(), zo) < TOL


@pytest.mark.parametrize('case', sorted(LIKE_CASES))
@pytest.mark.parametrize('dt', ['float32', 'float64'])
def test_likelihood_matches_reference_golden(engine, case, dt):
    g = load('like.npz')
    mk, a = LIKE_CASES[case]
    like = mk()
    u = g['%s/%s/u' % (case, dt)]
    ref = g['%s/%s/logl' % (case, dt)]
    d = u.shape[1]
    if a is None:    # eggbox: run.py:36 rounds twice (x * 5 * pi); feed the transformed points directly
        u, a = g['%s/%s/v' % (case, dt)], 1.0
    engine.set_target(d, like.like_id, like.params(), t_scale=a, t_shift=0.0)
    out = engine.loglike(dev(u)).cpu().numpy()
    if case in ('rosenbrock2', 'rosenbrock30', 'himmelblau'):
        assert np.array_equal(out, ref.astype(np.float64))            # bit exact
    elif case.startswith('gaussian') or case.startswith('shell'):
        assert np.allclose(out, ref, rtol=1e-10, atol=1e-9)
    else:
        assert np.allclose(out, ref, rtol=3e-6 if dt == 'float32' else 1e-12)


def test_prior_box_matches_reference_golden(engine):
    g = load('like.npz')
    engine.set_target(4, 0, [], prior_kind=1, prior_lo=-1.0, prior_hi=1.0)
    logl, logp = engine.loglike(dev(g['prior/x']), want_prior=True)
    assert np.array_equal(logp.cpu().numpy(), g['prior/logp'])


def test_likelihood_nonfinite_clamp(engine):
    # sampler.py:128 : non-finite -> -1e100, which is -inf for a float32 result
    engine.set_target(2, 0, [], t_scale=1.0, t_shift=0.0)
    u = torch.tensor([[3e19, 1.0], [0.5, 0.5]], dtype=torch.float32, device='cuda')
    out = engine.loglike(u).cpu().numpy()
    assert out[0] == -np.inf and np.isfinite(out[1])
    out64 = engine.loglike(torch.tensor([[1e200, 1.0]], dtype=torch.float64, device='cuda')).cpu().numpy()
    assert out64[0] == -1e100


def test_philox_stream_matches_oracle(engine):
    g = load('mcmc_hard_mix10.npz')
    d, n, steps = 10, 300, 4
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, 4, olike.GaussianMix(10).params(), t_scale=10.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0,
                      prior_hi=1.0)
    u0 = dev(np.ascontiguousarray(np.random.RandomState(0).uniform(-1, 1, (d, n)).astype(np.float32)))
    st, nbad, ncall = engine.mcmc_init(n, init_u=u0, seed=99, chain_offset=1000)
    out = engine.mcmc_run(st, steps, mode=0, loglstar=-1e30, step_size=0.3, seed=99, chain_offset=1000, step_offset=7,
                          dump_noise=True)
    for s in range(steps):
        nrm = ophilox.normals(99, 7 + s + 1, 1000 + np.arange(n), d)
        uni = ophilox.uniforms(99, 7 + s + 1, 1000 + np.arange(n))
        assert np.array_equal(out['uniforms'][s].cpu().numpy(), uni)          # integer path: bit exact
        assert np.abs(out['normals'][s].cpu().numpy() - nrm).max() < 1e-5      # __logf/__sincosf: abs err 2^-21.4 x radius


HARD = {
    'mcmc_hard_rosen2.npz': (lambda: olike.Rosenbrock(2), 5.0),
    'mcmc_hard_himmel2_fixed.npz': (lambda: olike.Himmelblau(2), 5.0),
    'mcmc_hard_mix10.npz': (lambda: olike.GaussianMix(10), 10.0),
    'mcmc_hard_rosen30.npz': (lambda: olike.Rosenbrock(30), 5.0),
    'mcmc_hard_eggbox2.npz': (lambda: olike.Eggbox(2), float(np.float32(5) * np.float32(np.pi))),
}


IMPLS = [pytest.param(1, id='ffma'), pytest.param(2, id='tcgen05'), pytest.param(3, id='warp16')]


def _run_replay(engine, g, mode, init_u=None, init_z=None, init_logl=None, loglstar=None, step_size=0.0, dynamic=False,
                impl=0):
    steps, n = int(g['steps']), int(g['chains'])
    st, nbad, ncall0 = engine.mcmc_init(n, init_u=init_u, init_z=init_z, init_logl=init_logl)
    out = engine.mcmc_run(st, steps, mode=mode, loglstar=loglstar, step_size=step_size, dynamic_step_size=dynamic,
                          trace=True, replay=(dev(g['normals']), dev(g['uniforms'])), impl=impl)
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    latent = out['trace_z'].permute(2, 0, 1).cpu().numpy()
    loglikes = out['trace_logl'].permute(1, 0).cpu().numpy()
    return samples, latent, loglikes, out['scale'], out['ncall'] + ncall0, st


def _compare_trace(samples, latent, loglikes, scale, ncall, g, max_flipped_chains=0):
    moved_ref = np.any(g['latent'][:, 1:] != g['latent'][:, :-1], axis=2)
    moved = np.any(latent[:, 1:] != latent[:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    # a chain may legitimately part ways at a near-tie of an accept test; none expected in these fixtures
    assert (~same).sum() <= max_flipped_chains, 'accept pattern differs in %d chains' % (~same).sum()
    assert rel_err(latent[same], g['latent'][same]) < TOL
    assert rel_err(samples[same], g['samples'][same]) < TOL
    assert rel_err(loglikes[same], g['loglikes'][same]) < TOL      # 1e-5 relative (north_star), like x and z
    if (~same).sum() == 0:
        assert ncall == int(g['ncall'])
        assert abs(scale - float(g['scale'])) <= 1e-12 * abs(float(g['scale']))


@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', sorted(HARD))
def test_mcmc_hard_replay_matches_reference_golden(engine, name, impl):
    g = load(name)
    mk, ts = HARD[name]
    d = int(g['d'])
    like = mk()
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, like.like_id, like.params(), t_scale=ts, t_shift=0.0, prior_kind=1, prior_lo=-1.0,
                      prior_hi=1.0)
    init_u = dev(np.ascontiguousarray(g['init_samples'].astype(np.float32).T))
    out = _run_replay(engine, g, 0, init_u=init_u, init_logl=dev(g['init_loglikes']), loglstar=float(g['loglstar']),
                      step_size=float(g['step_size']), dynamic=bool(g['dynamic']), impl=impl)
    _compare_trace(*out[:5], g)


@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', ['mcmc_mh_gauss8.npz', 'mcmc_mh_gauss50.npz'])
def test_mcmc_mh_replay_matches_reference_golden(engine, name, impl):
    g = load(name)
    d = int(g['d'])
    like = olike.Gaussian(d, float(g['corr']))
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, like.like_id, like.params(), t_scale=g['std'], t_shift=g['mean'], compute_f64=True,
                      prior_kind=2, prior_lo=float(g['prior_min']), prior_hi=float(g['prior_max']))
    init_z = dev(np.ascontiguousarray(g['z0'].T))
    out = _run_replay(engine, g, 1, init_z=init_z, loglstar=None, step_size=0.0, dynamic=False, impl=impl)
    _compare_trace(*out[:5], g)


@pytest.mark.parametrize('impl', IMPLS)
def test_mcmc_free_running_matches_oracle_on_dumped_noise(engine, impl):
    """Philox mode at a mid size: the kernel dumps the noise it used; the oracle replays it."""
    g = load('mcmc_hard_rosen30.npz')
    d, n, steps = 30, 1024, 12
    w = weights_of(g)
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, 0, [], t_scale=5.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0, prior_hi=1.0)
    rng = np.random.RandomState(3)
    idx = rng.randint(0, g['active_u'].shape[0], size=n)
    init_samples, init_logl = g['active_u'][idx], g['active_logl'][idx]
    st, _, _ = engine.mcmc_init(n, init_u=dev(np.ascontiguousarray(init_samples.astype(np.float32).T)),
                                init_logl=dev(init_logl), seed=5)
    out = engine.mcmc_run(st, steps, mode=0, loglstar=float(g['loglstar']), step_size=1 / 30 ** 0.5,
                          dynamic_step_size=True, seed=5, trace=True, dump_noise=True, impl=impl)
    target = omcmc.Target(olike.Rosenbrock(30), transform=lambda x: 5 * x, prior=olike.UniformPrior(d, -1, 1),
                          transform_prior=False)
    ref = omcmc.mcmc_sample(w, target, steps, omcmc.ReplayNoise(out['normals'].cpu().numpy(),
                                                                 out['uniforms'].cpu().numpy()),
                            step_size=1 / 30 ** 0.5, dynamic_step_size=True, init_samples=init_samples,
                            init_loglikes=init_logl, loglstar=float(g['loglstar']))
    latent = out['trace_z'].permute(2, 0, 1).cpu().numpy()
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    moved_ref = np.any(ref[1][:, 1:] != ref[1][:, :-1], axis=2)
    moved = np.any(latent[:, 1:] != latent[:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    assert (~same).sum() <= 2                       # near-ties only
    assert rel_err(latent[same], ref[1][same]) < TOL
    assert rel_err(samples[same], ref[0][same]) < TOL
    if (~same).sum() == 0:
        assert out['ncall'] == ref[5]
        assert abs(out['scale'] - ref[4]) <= 1e-12 * ref[4]
    # end state == last trace row
    assert torch.equal(st.z, out['trace_z'][-1]) and torch.equal(st.x, out['trace_x'][-1])
    assert torch.equal(st.logl, out['trace_logl'][-1])


@pytest.mark.parametrize('impl', IMPLS)
def test_mcmc_sharding_invariance(engine, impl):
    """Chains keyed by global id: running [0,n) in one call equals running two halves with chain_offset."""
    g = load('mcmc_hard_mix10.npz')
    d, n, steps = 10, 512, 6
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, 4, olike.GaussianMix(10).params(), t_scale=10.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0,
                      prior_hi=1.0)
    rng = np.random.RandomState(1)
    idx = rng.randint(0, g['active_u'].shape[0], size=n)
    u = np.ascontiguousarray(g['active_u'][idx].astype(np.float32).T)
    logl = g['active_logl'][idx]
    kw = dict(mode=0, loglstar=float(g['loglstar']), step_size=0.3, dynamic_step_size=False, seed=11, impl=impl)
    st, _, _ = engine.mcmc_init(n, init_u=dev(u), init_logl=dev(logl))
    engine.mcmc_run(st, steps, **kw)
    halves = []
    for r in range(2):
        sl = slice(r * n // 2, (r + 1) * n // 2)
        s2, _, _ = engine.mcmc_init(n // 2, init_u=dev(np.ascontiguousarray(u[:, sl])), init_logl=dev(logl[sl]))
        engine.mcmc_run(s2, steps, chain_offset=r * n // 2, **kw)
        halves.append(s2)
    assert torch.equal(torch.cat([h.z for h in halves], dim=1), st.z)
    assert torch.equal(torch.cat([h.logl for h in halves]), st.logl)


@pytest.mark.parametrize('impl', IMPLS)
def test_mcmc_hard_constraint_invariants_full_size(engine, impl):
    """Config-4 shape (65536 chains, d=30): every chain's end point obeys the constraint and the box."""
    g = load('mcmc_hard_rosen30.npz')
    d, n, steps = 30, (65536 if impl != 3 else 8192), 10      # the 16-lane kernel's range: the N = 8 shard of config 4
    engine.set_flow_from_state_dict(state_dict_of(g))
    engine.set_target(d, 0, [], t_scale=5.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0, prior_hi=1.0)
    rng = np.random.RandomState(2)
    idx = rng.randint(0, g['active_u'].shape[0], size=n)
    u = dev(np.ascontiguousarray(g['active_u'][idx].astype(np.float32).T))
    logl0 = dev(g['active_logl'][idx])
    loglstar = float(g['loglstar'])
    st, nbad, _ = engine.mcmc_init(n, init_u=u, init_logl=logl0, seed=1)
    z0 = st.z.clone()
    out = engine.mcmc_run(st, steps, mode=0, loglstar=loglstar, step_size=1 / 30 ** 0.5, dynamic_step_size=True, seed=1,
                          impl=impl)
    moved = (st.z != z0).any(dim=0)
    assert 0 < out['naccept'] <= n * steps and out['ncall'] >= out['naccept']
    assert (st.logl[moved] > loglstar).all()
    assert (st.x.abs() <= 1).all()
    assert torch.equal(st.logl[~moved], logl0[~moved])
    # likelihood of the end points recomputed by the batch kernel agrees bit for bit
    again = engine.loglike(st.x.t())
    assert torch.equal(again[moved], st.logl[moved])
    # flow consistency of the end state
    x2, ld2 = engine.flow_inverse(st.z.t())
    if impl == 1:     # same FFMA arithmetic as the batch flow kernel: bit for bit
        assert torch.equal(x2.t().contiguous(), st.x) and torch.equal(ld2, st.logdet)
    else:             # tensor-core 3xTF32 path / 16-lane summation order: FP32-class agreement
        assert (x2.t() - st.x).abs().max().item() < 1e-5 and (ld2 - st.logdet).abs().max().item() < 1e-5
    assert out['impl'] == (impl if impl else out['impl'])


@pytest.mark.parametrize('d,layers,blocks', [(4, 1, 1), (5, 1, 2), (7, 2, 4), (13, 1, 3), (33, 1, 3), (63, 1, 2)])
@pytest.mark.parametrize('npart', ['1', '2'])
def test_mcmc_generic_tensor_core_path_matches_oracle(engine, d, layers, blocks, npart):
    """The non-specialised instantiation of the tcgen05 kernel (any 2 <= d <= 63, any num_layers / num_blocks, N3 = 32
    when more than 16 dims are transformed per block), both thread layouts: free-running Philox noise dumped by the
    kernel, replayed through the oracle."""
    import os
    from nnest_b200 import _lib as L
    steps, n = 6, 700
    w = oflow.NVPWeights.random(d, hidden=16, num_layers=layers, num_blocks=blocks, seed=d, gain=1.3)
    old = os.environ.get('NNB_TC_NPART')
    os.environ['NNB_TC_NPART'] = npart           # read by the library at every launch
    try:
        _generic_case(engine, L.NNB_IMPL_TCGEN05, w, steps, n)
    finally:
        if old is None:
            del os.environ['NNB_TC_NPART']
        else:
            os.environ['NNB_TC_NPART'] = old


@pytest.mark.parametrize('d,layers,blocks', [(2, 1, 3), (4, 0, 1), (5, 1, 2), (7, 2, 4), (13, 1, 3), (33, 1, 3),
                                             (63, 1, 2), (100, 1, 3)])
def test_mcmc_generic_16_lane_path_matches_oracle(engine, d, layers, blocks):
    """The 16-lanes-per-chain kernel on shapes off the beaten track: odd dims, no / two hidden layers, one block (odd dims
    never transformed), more than 16 outputs per block (two per lane), more than 64 dims (two Philox blocks per lane)."""
    from nnest_b200 import _lib as L
    w = oflow.NVPWeights.random(d, hidden=16, num_layers=layers, num_blocks=blocks, seed=d, gain=1.3)
    _generic_case(engine, L.NNB_IMPL_WARP, w, 6, 700)


def _generic_case(engine, impl, w, steps, n, flags=0, target='rosenbrock', dynamic=True):
    """`steps` free-running steps of `n` chains of the flow `w` (any hidden_dim / scale mode; `flags` = its nnb_set_flow
    flags) on `impl`: Philox noise dumped by the kernel, replayed through the oracle.  target 'rosenbrock': the hard
    constraint at the 25th percentile of the start points, with the dynamic or a fixed step size; 'gaussian': Metropolis-
    Hastings on a float64 correlated Gaussian in transformed coordinates.  Returns (end state, mcmc_run result)."""
    d = w.d
    engine.set_flow(w.flat(), d, w.hidden, w.num_layers, w.num_blocks, flags)
    rng = np.random.RandomState(d)
    u0 = rng.uniform(-0.6, 0.6, size=(n, d))
    if target == 'rosenbrock':
        like = olike.Rosenbrock(d)
        engine.set_target(d, 0, [], t_scale=5.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0, prior_hi=1.0)
        tgt = omcmc.Target(like, transform=lambda x: 5 * x, prior=olike.UniformPrior(d, -1, 1), transform_prior=False)
        logl0 = like.batch(5 * u0)
        # a fixed step stays at its start value: a third of the dynamic run's start keeps chains moving
        mode, loglstar, step_size = 0, float(np.percentile(logl0, 25)), (1.0 if dynamic else 0.3) / d ** 0.5
    else:
        assert target == 'gaussian'
        like = olike.Gaussian(d, 0.5)
        engine.set_target(d, like.like_id, like.params(), t_scale=2.0, t_shift=0.5, compute_f64=True, prior_kind=2,
                          prior_lo=-10.0, prior_hi=10.0)
        tgt = omcmc.Target(like, transform=lambda x: x * 2.0 + 0.5, prior=olike.UniformPrior(d, -10, 10),
                           transform_prior=True)
        logl0 = tgt.loglike(u0)
        mode, loglstar, step_size = 1, None, 0.5 / d ** 0.5
    st, _, _ = engine.mcmc_init(n, init_u=dev(np.ascontiguousarray(u0.astype(np.float32).T)), init_logl=dev(logl0),
                                seed=11)
    out = engine.mcmc_run(st, steps, mode=mode, loglstar=loglstar, step_size=step_size, dynamic_step_size=dynamic,
                          seed=11, trace=True, dump_noise=True, impl=impl)
    if impl != 0:
        assert out['impl'] == impl
    ref = omcmc.mcmc_sample(w, tgt, steps, omcmc.ReplayNoise(out['normals'].cpu().numpy(),
                                                              out['uniforms'].cpu().numpy()),
                            step_size=step_size, dynamic_step_size=dynamic, init_samples=u0, init_loglikes=logl0,
                            loglstar=loglstar)
    latent = out['trace_z'].permute(2, 0, 1).cpu().numpy()
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    loglikes = out['trace_logl'].permute(1, 0).cpu().numpy()
    moved_ref = np.any(ref[1][:, 1:] != ref[1][:, :-1], axis=2)
    moved = np.any(latent[:, 1:] != latent[:, :-1], axis=2)
    same = np.all(moved == moved_ref, axis=1)
    assert (~same).sum() <= 2                       # near-ties only
    assert moved.sum() > 0.1 * moved.size           # the test moves chains
    assert rel_err(latent[same], ref[1][same]) < TOL
    assert rel_err(samples[same], ref[0][same]) < TOL
    assert rel_err(loglikes[same], ref[3][same]) < TOL
    if (~same).sum() == 0:
        assert out['ncall'] == ref[5]
        assert abs(out['scale'] - ref[4]) <= 1e-12 * ref[4]
    assert torch.equal(st.z, out['trace_z'][-1]) and torch.equal(st.x, out['trace_x'][-1])
    assert torch.equal(st.logl, out['trace_logl'][-1])
    return st, out


@pytest.mark.parametrize('impl', IMPLS)
def test_long_replay_1024x150_d30_matches_reference(engine, impl):
    """One long replay recorded from the reference (tests/golden/make_golden_long.py): 1024 chains x 150 steps at the
    config-4 shape, noise regenerated from the stored seed."""
    from test_oracle_golden import _long_case, compare_long
    g, b, normals, uniforms, idx = _long_case()
    engine.set_flow_from_state_dict({k[3:]: b[k] for k in b.files if k.startswith('sd/')})
    engine.set_target(30, 0, [], t_scale=5.0, t_shift=0.0, prior_kind=1, prior_lo=-1.0, prior_hi=1.0)
    au, al = b['active_u'].astype(np.float64), b['active_logl']
    st, _, _ = engine.mcmc_init(1024, init_u=dev(np.ascontiguousarray(au[idx].astype(np.float32).T)), init_logl=dev(al[idx]))
    out = engine.mcmc_run(st, int(g['steps']), mode=0, loglstar=float(g['loglstar']), step_size=float(g['step_size']),
                          dynamic_step_size=False, trace=True, replay=(dev(normals), dev(uniforms)), impl=impl)
    assert out['impl'] == impl
    latent = out['trace_z'].permute(2, 0, 1).cpu().numpy()
    samples = out['trace_x'].permute(2, 0, 1).cpu().numpy()
    loglikes = out['trace_logl'].permute(1, 0).cpu().numpy()
    compare_long(g, latent, samples, loglikes, out['ncall'], max_flipped=8)
