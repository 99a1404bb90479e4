"""GPU: the FP32-FMA flow and MCMC kernels (csrc/nnb_kernels.cuh, instantiated for hidden_dim 16, 32 and 64 in
csrc/nnb_h{16,32,64}.cu) on every flow architecture nnb_set_flow admits, against the float64 flow oracle
(oracle/flow.py with dtype=np.float64).  These kernels run every flow the tensor-core and 16-lane step kernels do not
take: hidden_dim 32 / 64, scale 'translate' / 'constant', x_dim 1 and, at large batches, x_dim > 63.

  flow_kernel<H, INV>        flow_forward / flow_inverse
  mcmc_init_kernel<H>        mcmc_init: from init_u, from init_z, from the Philox stream (tag 2)
  mcmc_kernel<H, MODE>       mcmc_run, hard constraint (dynamic and fixed step size) and Metropolis-Hastings
  coupling_block's translate-only branch and the ScaleLayer of flow_{forward,inverse}_inplace (scale != '')

The edges of the shared-memory layout are found by asking nnb_set_flow, not by restating its size formula.

Weights are NVPWeights.random(..., gain=1.0), the nn.Linear default initialisation.  At that gain the float32 oracle stays
within 8.2e-7 (max-norm relative) of the float64 oracle on every flow map below, the deepest and widest shapes included,
so the 1e-5 criterion leaves a margin of 12 over the oracle's own rounding; each test asserts its share of that
(F32_ORACLE_MAX) before it compares the kernel.

The log-det is held to rtol = 1e-5, atol = 1e-6: a float32 sum of up to 16 x 64 log-scale terms of order one, whose value
can be near zero, so the absolute term binds.  Affine flows without a hidden layer have the largest log-scale terms: at
gain 1.0 the float32 oracle itself misses that criterion (by up to 1.6x at 16 blocks of d = 30, and near it at
d >= 87 with three blocks), so those flows use gain 0.35, and the chain starts of affine flows, whose largest shape
(d = 128, two layers) reaches 0.64 of it at gain 1.0, use gain 0.5.  With these gains the float32 oracle meets the
log-det criterion with a quarter to spare (LD_ORACLE_MAX) on every shape, which each test asserts.

The hidden_dim == 16, scale == '' flows at L = 1 are covered by test_gpu_parity.py (goldens, tcgen05 / 16-lane shapes)
and are not repeated here."""
import logging

import numpy as np
import pytest

torch = pytest.importorskip('torch')

from oracle import flow as oflow
from oracle import likelihoods as olike
from oracle import mcmc as omcmc
from oracle import philox as ophilox
from helpers import rel_err
from test_gpu_parity import _generic_case

pytestmark = pytest.mark.gpu

GAIN = 1.0
TOL = 1e-5
F32_ORACLE_MAX = 2.5e-6   # the float32 oracle's own error must stay 4x below TOL (measured: <= 8.2e-7)
LD_ORACLE_MAX = 0.75      # float32 oracle's log-det error / (1e-6 + 1e-5 |ld|), see above (measured: <= 0.61)
HS = [16, 32, 64]
SCALES = ['', 'translate', 'constant']
LAYERS = [0, 2, 8]
SHAPES = ['d1', 'd7', 'max_blocks_d5', 'max_blocks_d30', 'max_dim_b1', 'max_dim_b3']
N = 1000                  # samples / chains: not a multiple of the 128-thread CTA


@pytest.fixture(scope='module')
def engine():
    from nnest_b200.engine import Engine
    return Engine(0)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def scale_id(s):
    return s or 'affine'


def flags_of(scale):
    from nnest_b200 import _lib as L
    return {'': 0, 'translate': L.NNB_FLOW_TRANSLATE_ONLY,
            'constant': L.NNB_FLOW_TRANSLATE_ONLY | L.NNB_FLOW_CONST_SCALE}[scale]


def weights(d, H, L, B, scale, seed=0, gain=GAIN):
    return oflow.NVPWeights.random(d, H, L, B, seed=seed, gain=gain, scale=scale)


def ld_margin(ld, ld64):
    """largest |ld - ld64| / (atol + rtol |ld64|) of the log-det criterion"""
    ld = np.asarray(ld, dtype=np.float64)
    return float((np.abs(ld - ld64) / (1e-6 + TOL * np.abs(ld64))).max())


def install(engine, w, scale):
    engine.set_flow(w.flat(), w.d, w.hidden, w.num_layers, w.num_blocks, flags_of(scale))


def refusal(engine, d, H, L, B, scale):
    """the NNBError code nnb_set_flow returns for this architecture, or None if it installs it"""
    from nnest_b200 import _lib
    try:
        install(engine, weights(d, H, L, B, scale), scale)
        return None
    except _lib.NNBError as e:
        return e.code


_FITS = {}


def fits(engine, d, H, L, B, scale):
    key = (d, H, L, B, scale)
    if key not in _FITS:
        from nnest_b200 import _lib
        code = refusal(engine, d, H, L, B, scale)
        assert code in (None, _lib.NNB_ERR_UNSUPPORTED)
        _FITS[key] = code is None
    return _FITS[key]


def max_blocks(engine, d, H, L, scale):
    """largest num_blocks nnb_set_flow admits at (d, H, L, scale), capped by NNB_MAX_BLOCKS; 0 if none"""
    from nnest_b200 import _lib
    B = 0
    while B < _lib.NNB_MAX_BLOCKS and fits(engine, d, H, L, B + 1, scale):
        B += 1
    return B


def max_dim(engine, B, H, L, scale):
    """largest x_dim nnb_set_flow admits with B blocks, capped by NNB_MAX_DIM (128); 0 if none"""
    from nnest_b200 import _lib
    d = 0
    while d < _lib.NNB_MAX_DIM and fits(engine, d + 1, H, L, B, scale):
        d += 1
    return d


def resolve(engine, H, L, scale, shape):
    """(d, num_blocks) of a named shape; None (after asserting nnb_set_flow refuses it) where no flow of the
    architecture has that shape"""
    fixed = {'d1': (1, 2), 'd7': (7, 3)}
    if shape in fixed:
        d, B = fixed[shape]
        return (d, B) if fits(engine, d, H, L, B, scale) else None
    if shape.startswith('max_blocks_d'):
        d = int(shape[len('max_blocks_d'):])
        B = max_blocks(engine, d, H, L, scale)
        assert B or not fits(engine, d, H, L, 1, scale)
        return (d, B) if B else None
    B = int(shape[len('max_dim_b'):])
    d = max_dim(engine, B, H, L, scale)
    assert d or not fits(engine, 1, H, L, B, scale)
    return (d, B) if d else None


def resolve_or_skip(engine, H, L, scale, shape):
    dB = resolve(engine, H, L, scale, shape)
    if dB is None:
        pytest.skip('hidden %d, %d layers, scale %r: nnb_set_flow admits no flow of shape %s' % (H, L, scale, shape))
    return dB


def const_logdet(w, inverse):
    """the kernel's log-det of a 'constant' flow: the float32 sum of -+const_scale in the order the blocks run"""
    ld = np.float32(0)
    for k in (range(w.num_blocks - 1, -1, -1) if inverse else range(w.num_blocks)):
        cs = np.float32(w.blocks[k]['const_scale'])
        ld = np.float32(ld - cs) if inverse else np.float32(ld + cs)
    return ld


def check_flow_map(w, scale, kernel_out, kernel_ld, inp, inverse):
    f = oflow.flow_inverse if inverse else oflow.flow_forward
    o64, ld64 = f(w, inp, dtype=np.float64)
    o32, ld32 = f(w, inp)
    assert rel_err(o32, o64) < F32_ORACLE_MAX
    assert ld_margin(ld32, ld64) <= LD_ORACLE_MAX
    out, ld = kernel_out.cpu().numpy(), kernel_ld.cpu().numpy()
    assert rel_err(out, o64) < TOL
    assert np.allclose(ld, ld64, rtol=TOL, atol=1e-6)
    if scale == 'translate':
        assert (ld == 0).all()
    elif scale == 'constant':
        assert (ld == const_logdet(w, inverse)).all()


# ---- a. flow maps: flow_kernel<H, false / true> on every architecture and shape --------------------------------------
@pytest.mark.parametrize('shape', SHAPES)
@pytest.mark.parametrize('L', LAYERS)
@pytest.mark.parametrize('scale', SCALES, ids=scale_id)
@pytest.mark.parametrize('H', HS)
def test_flow_maps_match_float64_oracle(engine, H, scale, L, shape):
    """flow_kernel<H, INV> (translate-only coupling and ScaleLayer branches for scale != ''): 1000 samples forward and
    inverse, and a transposed (column-major) input, against the float64 oracle."""
    d, B = resolve_or_skip(engine, H, L, scale, shape)
    w = weights(d, H, L, B, scale, seed=1000 * d + 10 * B + H + L, gain=0.35 if scale == '' and L == 0 else GAIN)
    install(engine, w, scale)
    rng = np.random.default_rng(d + B + H + L)
    x = rng.normal(size=(N, d)).astype(np.float32)
    zin = rng.normal(size=(N, d)).astype(np.float32)
    z, ldz = engine.flow_forward(dev(x))
    check_flow_map(w, scale, z, ldz, x, inverse=False)
    xo, ldx = engine.flow_inverse(dev(zin))
    check_flow_map(w, scale, xo, ldx, zin, inverse=True)
    xt, ldt = engine.flow_inverse(dev(zin.T.copy()).t())
    assert torch.equal(xt, xo) and torch.equal(ldt, ldx)


# ---- b. one past each edge is refused, and the installed flow survives the refusal ----------------------------------
@pytest.mark.parametrize('L', LAYERS)
@pytest.mark.parametrize('scale', SCALES, ids=scale_id)
@pytest.mark.parametrize('H', HS)
def test_one_past_the_edge_is_refused(engine, H, scale, L):
    """At the largest admitted num_blocks (d = 5, 30) and x_dim (B = 1, 3), one more block or dim is refused:
    NNB_ERR_UNSUPPORTED where shared memory is the limit, NNB_ERR_ARG past NNB_MAX_BLOCKS / NNB_MAX_DIM.  The flow that
    was installed before the refusal is still the one flow_inverse runs, bit for bit."""
    from nnest_b200 import _lib
    edges = []
    for d in (5, 30):
        B = max_blocks(engine, d, H, L, scale)
        if B:
            edges.append(((d, B), (d, B + 1), B == _lib.NNB_MAX_BLOCKS))
    for B in (1, 3):
        d = max_dim(engine, B, H, L, scale)
        if d:
            edges.append(((d, B), (d + 1, B), d == _lib.NNB_MAX_DIM))
    if not edges:
        assert not fits(engine, 5, H, L, 1, scale)
        pytest.skip('hidden %d, %d layers, scale %r: no flow fits' % (H, L, scale))
    zin = np.random.default_rng(H + L).normal(size=(300, 128)).astype(np.float32)
    for (d, B), (d1, B1), capped in edges:
        w = weights(d, H, L, B, scale, seed=d + B)
        install(engine, w, scale)
        z = dev(zin[:, :d])
        x0, ld0 = engine.flow_inverse(z)
        code = refusal(engine, d1, H, L, B1, scale)
        assert code == (_lib.NNB_ERR_ARG if capped else _lib.NNB_ERR_UNSUPPORTED), (d1, B1)
        assert engine.d == d
        x1, ld1 = engine.flow_inverse(z)
        assert torch.equal(x1, x0) and torch.equal(ld1, ld0)
        assert rel_err(x1.cpu().numpy(), oflow.flow_inverse(w, zin[:, :d], dtype=np.float64)[0]) < TOL


# ---- c. chain start: mcmc_init_kernel<H>, three start modes ----------------------------------------------------------
def start_target(engine, d):
    like = olike.Gaussian(d, 0.5)
    engine.set_target(d, like.like_id, like.params(), t_scale=2.0, t_shift=0.5, compute_f64=True, prior_kind=2,
                      prior_lo=-1e3, prior_hi=1e3)
    return omcmc.Target(like, transform=lambda x: x * 2.0 + 0.5, prior=olike.UniformPrior(d, -1e3, 1e3),
                        transform_prior=True)


@pytest.mark.parametrize('start', ['init_u', 'init_z', 'philox'])
@pytest.mark.parametrize('shape', ['d7', 'max_dim_b3'])
@pytest.mark.parametrize('scale', SCALES, ids=scale_id)
@pytest.mark.parametrize('H', HS)
def test_chain_start_matches_oracle(engine, H, scale, shape, start):
    """mcmc_init_kernel<H> at two layers: z, x, log-det, log-likelihood and log-prior of 1000 chains against the float64
    oracle.  init_u runs forward then inverse; init_z only the inverse; the Philox start draws z ~ N(0, I) from
    (j, start_try, chain_offset + c, tag 2).  A start with a coordinate at 3e19 has a log-likelihood below -1e30 (or
    none at all: NaN), which n_bad_start must count exactly; ncall counts every chain."""
    L = 2
    d, B = resolve_or_skip(engine, H, L, scale, shape)
    w = weights(d, H, L, B, scale, seed=7 * d + H, gain=0.5 if scale == '' else GAIN)
    install(engine, w, scale)
    tgt = start_target(engine, d)
    rng = np.random.default_rng(d + H)
    bad = np.zeros(N, dtype=bool)
    seed, offset, start_try = 12345, 777, 3
    if start == 'philox':
        st, nbad, ncall = engine.mcmc_init(N, seed=seed, chain_offset=offset, start_try=start_try)
        z = st.z.t().cpu().numpy()
        want = ophilox.normals(seed, start_try, offset + np.arange(N), d, tag=ophilox.TAG_INIT)
        assert np.abs(z - want).max() < 1e-5
    else:
        a = rng.uniform(-0.9, 0.9, size=(N, d)).astype(np.float32)
        bad[[5, 128, N - 1]] = True
        a[bad, d // 2] = 3e19
        kw = {start: dev(a.T.copy())}
        st, nbad, ncall = engine.mcmc_init(N, want_counts=True, **kw)
        z = st.z.t().cpu().numpy()
        if start == 'init_u':
            z64, _ = oflow.flow_forward(w, a[~bad], dtype=np.float64)
            assert rel_err(oflow.flow_forward(w, a[~bad])[0], z64) < F32_ORACLE_MAX
            assert rel_err(z[~bad], z64) < TOL
        else:
            assert np.array_equal(z, a)
    assert nbad == bad.sum() and ncall == N
    ok = ~bad
    x64, ld64 = oflow.flow_inverse(w, z[ok], dtype=np.float64)
    assert ld_margin(oflow.flow_inverse(w, z[ok])[1], ld64) <= LD_ORACLE_MAX
    assert rel_err(st.x.t().cpu().numpy()[ok], x64) < TOL
    assert np.allclose(st.logdet.cpu().numpy()[ok], ld64, rtol=TOL, atol=1e-6)
    logl = st.logl.cpu().numpy()
    assert rel_err(logl[ok], tgt.loglike(x64)) < TOL
    assert (logl[bad] <= -1e30).all() and (logl[ok] > -1e30).all()
    assert np.array_equal(st.logp.cpu().numpy()[ok], tgt.prior(x64))
    x2, ld2 = engine.flow_inverse(st.z.t())      # flow_inverse_inplace<H> is shared by both kernels: same bits
    assert torch.equal(x2.t()[:, ok], st.x[:, ok]) and torch.equal(ld2[ok], st.logdet[ok])


# ---- d. MCMC step: mcmc_kernel<H, MODE> on a representative subset ---------------------------------------------------
@pytest.mark.parametrize('run', ['hard_dynamic', 'hard_fixed', 'mh_gaussian'])
@pytest.mark.parametrize('shape', ['d7', 'max_dim_b3'])
@pytest.mark.parametrize('L', [0, 2])
@pytest.mark.parametrize('scale', SCALES, ids=scale_id)
@pytest.mark.parametrize('H', HS)
def test_mcmc_step_matches_oracle(engine, H, scale, L, shape, run):
    """mcmc_kernel<H, NNB_MODE_HARD> (one launch per step with the dynamic step size, one launch for all steps with a fixed
    one) and mcmc_kernel<H, NNB_MODE_MH> on a float64 Gaussian: 700 chains x 6 steps, Philox noise dumped by the kernel
    and replayed through the float32 oracle (oracle.mcmc).  hidden_dim 16 with scale '' runs impl=FFMA (AUTO would pick a
    tensor-core kernel), every other flow AUTO, which must pick FFMA and refuse the other two kernels."""
    from nnest_b200 import _lib
    d, B = resolve_or_skip(engine, H, L, scale, shape)
    w = weights(d, H, L, B, scale, seed=11 * d + H + L)
    default = H == 16 and scale == ''
    impl = _lib.NNB_IMPL_FFMA if default else _lib.NNB_IMPL_AUTO
    steps = 6
    st, out = _generic_case(engine, impl, w, steps, 700, flags=flags_of(scale),
                            target='gaussian' if run == 'mh_gaussian' else 'rosenbrock', dynamic=run == 'hard_dynamic')
    assert out['impl'] == _lib.NNB_IMPL_FFMA
    assert out['launches'] == (steps if run == 'hard_dynamic' else 1)
    x2, ld2 = engine.flow_inverse(st.z.t())
    assert torch.equal(x2.t().contiguous(), st.x) and torch.equal(ld2, st.logdet)
    if not default:
        for other in (_lib.NNB_IMPL_TCGEN05, _lib.NNB_IMPL_WARP):
            with pytest.raises(_lib.NNBError) as e:
                engine.mcmc_run(st, 1, mode=0, loglstar=-1e30, impl=other)
            assert e.value.code == _lib.NNB_ERR_UNSUPPORTED


# ---- e. Trainer (autograd fit) -> state_dict -> kernels --------------------------------------------------------------
@pytest.mark.parametrize('scale', SCALES, ids=scale_id)
@pytest.mark.parametrize('L', [0, 2])
@pytest.mark.parametrize('H', [32, 64])
def test_trainer_autograd_fit_runs_on_kernels(engine, H, L, scale):
    """Trainer with an architecture only the autograd path fits (hidden 32 at two layers with scale '' runs the fused
    kernel, see test_gpu_train_sweep.py): after a few epochs trainer.forward / trainer.inverse (flow_kernel<H>) agree
    with a float64 CPU copy of trainer.netG, and installing netG.state_dict() with the scale mode inferred from the
    keys (the path of an injected trainer) gives the same kernel outputs bit for bit."""
    import copy
    from nnest_b200 import Trainer
    if H == 32 and L == 2 and scale == '':
        pytest.skip('fitted by the fused kernel (test_gpu_train_sweep.py)')
    d = 6
    torch.manual_seed(H + L)
    rng = np.random.default_rng(H + L)
    data = rng.multivariate_normal(np.zeros(d), 0.5 * np.eye(d) + 0.5, size=800)
    t = Trainer(d, hidden_dim=H, num_layers=L, num_blocks=3, flow='nvp', scale=scale, log_dir=None,
                log_level=logging.ERROR, learning_rate=1e-3, engine=engine)
    assert not t._fused
    p0 = [p.detach().clone() for p in t.netG.parameters()]
    t.train(data, max_iters=5, jitter=0.0)
    assert any(not torch.equal(p, q) for p, q in zip(t.netG.parameters(), p0))      # the fit moved the weights
    net64 = copy.deepcopy(t.netG.flow).to('cpu', torch.float64)
    x = rng.normal(size=(N, d)).astype(np.float32)
    zin = rng.normal(size=(N, d)).astype(np.float32)
    z, ldz = t.forward(x)
    xo, ldx = t.inverse(zin)
    with torch.no_grad():
        z64, ldz64 = [v.numpy() for v in net64.forward(torch.from_numpy(x).double())]
        x64, ldx64 = [v.numpy() for v in net64.inverse(torch.from_numpy(zin).double())]
    assert rel_err(z.cpu().numpy(), z64) < TOL and np.allclose(ldz.cpu().numpy(), ldz64, rtol=TOL, atol=1e-6)
    assert rel_err(xo.cpu().numpy(), x64) < TOL and np.allclose(ldx.cpu().numpy(), ldx64, rtol=TOL, atol=1e-6)
    engine.set_flow_from_state_dict(t.netG.state_dict(), scale=None)
    assert engine.flow_shape == (d, H, L, 3, flags_of(scale))
    z2, ldz2 = engine.flow_forward(dev(x))
    x2, ldx2 = engine.flow_inverse(dev(zin))
    assert torch.equal(z2, z) and torch.equal(ldz2, ldz) and torch.equal(x2, xo) and torch.equal(ldx2, ldx)
