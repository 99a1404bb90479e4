"""GPU: derived parameters of user likelihoods (CudaLikelihood(num_derived=...), nnb_derived / nnb_derived_trace).

The source of every test here is DERIVED3 (tests/test_user_derived.py): user Rosenbrock with the columns
    derived[0] = the likelihood re-evaluated, derived[1] = (double)x(0), derived[2] = sum_i (double)x(i)^2.
Column 0 must equal the log-likelihood the library reports for the same point bit for bit: that shows the derived kernel
sees the step kernel's x, in its arithmetic type.  Derived parameters must change nothing else: chains, evidence and call
counts are compared with the same seeded run without them."""
import logging
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip('torch')

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
if ROOT not in sys.path:       # run as a script: the two-rank worker below
    sys.path.insert(0, ROOT)

from nnest_b200 import _lib as L
from test_gpu_user_likelihood import VARIANTS, _nvp, _spline
from test_user_derived import DERIVED3

pytestmark = pytest.mark.gpu

dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _oracle_cols(u, scale, shift, f64):
    """columns 1 and 2 of DERIVED3 in NumPy: x = u * scale + shift in float32 (float32 rows, float32 transform) or
    float64, then (double)x(0) and the float64 sum of squares in index order"""
    t = np.float64 if f64 else np.float32
    x = np.asarray(u).astype(t) * np.asarray(scale).astype(t) + np.asarray(shift).astype(t)
    x = x.astype(np.float64)
    s = np.zeros(x.shape[:-1])
    for i in range(x.shape[-1]):
        s = s + x[..., i] * x[..., i]
    return x[..., 0], s


# ---- 1. nnb_derived on rows ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('f64_rows', [False, True])
@pytest.mark.parametrize('transform', [False, True])
@pytest.mark.parametrize('compute_f64', [False, True])
def test_derived_rows(f64_rows, transform, compute_f64):
    from nnest_b200.engine import Engine
    d = 7
    eng = Engine(0)
    kw = dict(t_scale=np.linspace(2.0, 5.0, d), t_shift=np.linspace(-0.5, 0.25, d)) if transform else {}
    eng.set_target(d, L.NNB_LIKE_USER, (), compute_f64=compute_f64, user_source=DERIVED3, num_derived=3, **kw)
    rng = np.random.RandomState(1)
    u = rng.uniform(-1.0, 1.0, size=(5000, d))
    u = u if f64_rows else u.astype(np.float32)
    ud = dev(u)
    der = eng.derived(ud).cpu().numpy()
    assert der.shape == (5000, 3)
    assert np.array_equal(der[:, 0], eng.loglike(ud).cpu().numpy())
    # the same rows through a strided view: column-major layout
    ut = dev(np.asarray(u).T.copy()).t()
    assert np.array_equal(eng.derived(ut).cpu().numpy(), der)
    x0, s = _oracle_cols(u, kw.get('t_scale', 1.0), kw.get('t_shift', 0.0), f64_rows or compute_f64)
    assert np.array_equal(der[:, 1], x0)
    assert np.allclose(der[:, 2], s, rtol=1e-15, atol=0)       # the same sum in the same order: exact in practice


def test_derived_state_errors():
    from nnest_b200.engine import Engine
    eng = Engine(0)
    eng.set_target(2, L.NNB_LIKE_ROSENBROCK, ())
    u = dev(np.zeros((4, 2)))
    out = torch.empty((4, 3), dtype=torch.float64, device='cuda')
    assert eng.lib.nnb_derived(eng.h, u.data_ptr(), 1, 2, 1, out.data_ptr(), 4, None) == L.NNB_ERR_STATE
    eng.set_target(2, L.NNB_LIKE_USER, (), user_source=DERIVED3)            # installed without derived parameters
    assert eng.lib.nnb_derived(eng.h, u.data_ptr(), 1, 2, 1, out.data_ptr(), 4, None) == L.NNB_ERR_STATE
    assert eng.lib.nnb_derived_trace(eng.h, u.data_ptr(), 2, 0, 1, 1, None, out.data_ptr(), None) == L.NNB_ERR_STATE
    eng.set_target(2, L.NNB_LIKE_USER, (), user_source=DERIVED3, num_derived=3)
    assert eng.lib.nnb_derived(eng.h, u.data_ptr(), 1, 2, 1, out.data_ptr(), 4, None) == L.NNB_OK


def test_cuda_likelihood_call_returns_logl_and_derived():
    from nnest_b200.likelihoods import CudaLikelihood
    like = CudaLikelihood(3, DERIVED3, num_derived=3)
    x = np.random.RandomState(2).uniform(-2, 2, size=(10, 3))
    logl, der = like(x)
    assert logl.shape == (10,) and der.shape == (10, 3)
    assert np.array_equal(der[:, 0], logl) and np.array_equal(der[:, 1], x[:, 0])
    l1, d1 = like(x[3])
    assert l1 == logl[3] and np.array_equal(d1, der[3])


# ---- 2. _mcmc_sample on every step-kernel variant -------------------------------------------------------------------
def _sampler(tmp_path, d, num_derived, name):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood
    return NestedSampler(d, CudaLikelihood(d, DERIVED3, num_derived=num_derived), transform=lambda x: 5 * x,
                         flow='nvp', num_live_points=10, num_derived=num_derived, log_dir=str(tmp_path / name),
                         log_level=logging.WARNING, seed=3)


def _sample(s, **kw):
    s._step_counter = s._start_counter = 0            # the same Philox counters for every call
    return s._mcmc_sample(12, **kw)


def _bits_moved(samples):
    """(N, T): row t differs from row 0 in some coordinate, bitwise"""
    b = np.ascontiguousarray(samples).view(np.uint32)
    return np.any(b != b[:, :1], axis=2)


@pytest.mark.parametrize('variant', list(VARIANTS))
def test_mcmc_sample_derived_on_every_variant(tmp_path, variant):
    flow, d, hid, flags, n, impl, mode, dynamic, _ = VARIANTS[variant]
    samplers = [_sampler(tmp_path, d, nd, 'nd%d' % nd) for nd in (3, 0)]
    for s in samplers:
        if flow == 'spline':
            _spline(s.engine, d)
        else:
            _nvp(s.engine, d, hid, flags=flags)
        s.engine.default_impl = impl
    s3, s0 = samplers
    rng = np.random.RandomState(4)
    u = rng.uniform(-0.3, 0.3, size=(n, d)).astype(np.float32)
    logl_u, der_u = s3.loglike(u)
    assert np.array_equal(der_u[:, 0], logl_u)
    loglstar = float(np.quantile(logl_u, 0.3)) if mode == L.NNB_MODE_HARD else None
    kw = dict(init_samples=u, init_loglikes=logl_u.astype(np.float64), loglstar=loglstar, step_size=0.3,
              dynamic_step_size=dynamic)
    init_der = np.full((n, 3), -7.0)                  # a marker: the unmoved rows must carry it
    calls = s3.total_calls
    a = _sample(s3, init_derived=init_der, **kw)
    b = _sample(s0, **kw)
    samples, latent, derived, loglikes, scale, ncall = a
    for i in (0, 1, 3):
        assert np.array_equal(a[i], b[i]), i
    assert scale == b[4] and ncall == b[5] and s3.total_calls - calls == ncall
    assert derived.shape == (n, 13, 3) and b[2].shape == (n, 13, 0)
    moved = _bits_moved(samples)
    assert moved.any() and (~moved[:, 1:]).any()
    assert np.array_equal(derived[..., 0][moved], loglikes[moved])
    assert (derived[~moved] == -7.0).all()
    x0, sq = _oracle_cols(samples, 5.0, 0.0, False)
    assert np.array_equal(derived[..., 1][moved], x0[moved])
    assert np.allclose(derived[..., 2][moved], sq[moved], rtol=1e-15, atol=0)
    # thin=k evaluates the kept rows only, and they are the same rows
    t = _sample(s3, init_derived=init_der, thin=5, **kw)
    assert np.array_equal(t[2], derived[:, ::5]) and np.array_equal(t[0], samples[:, ::5])
    # without init_derived row 0 is g(x_0): column 0 is the trace's log-likelihood on every row
    c = _sample(s3, num_chains=n, loglstar=loglstar, step_size=0.3, dynamic_step_size=dynamic)
    assert np.array_equal(c[2][..., 0], c[3])


def test_mcmc_sample_output_interval_chain_files(tmp_path):
    s = _sampler(tmp_path, 3, 3, 'out')
    s.param_names = ['a', 'b', 'c', 'l', 'x0', 's']
    u = np.random.RandomState(5).uniform(-0.3, 0.3, size=(16, 3)).astype(np.float32)
    logl, der = s.loglike(u)
    out = s._mcmc_sample(6, init_samples=u, init_loglikes=logl, init_derived=der, loglstar=None, step_size=0.3,
                         output_interval=6)
    rows = np.loadtxt(os.path.join(s.logs['chains'], 'chain_1.txt'), skiprows=1)
    assert rows.shape == (7, 2 + 3 + 3)
    assert np.array_equal(rows[:, 2 + 3:], np.array([['%.5E' % v for v in r] for r in out[2][0]], dtype=float))


# ---- 3. MCMCSampler.run ---------------------------------------------------------------------------------------------
def _mcmc_run(tmp_path, num_derived):
    from nnest_b200 import MCMCSampler
    from nnest_b200.likelihoods import CudaLikelihood
    from nnest_b200.priors import UniformPrior
    np.random.seed(1)
    torch.manual_seed(1)
    d = 3
    s = MCMCSampler(d, CudaLikelihood(d, DERIVED3, num_derived=num_derived), prior=UniformPrior(d, -8, 8), flow='nvp',
                    num_derived=num_derived, log_dir=str(tmp_path / ('m%d' % num_derived)), log_level=logging.WARNING,
                    seed=2)
    training = np.random.normal(size=(2000, d)) * 0.5 + 1.0
    s.run(100, 512, training, stats_interval=None, train_iters=50)
    return s


def test_mcmc_sampler_run_with_derived(tmp_path):
    s3, s0 = _mcmc_run(tmp_path, 3), _mcmc_run(tmp_path, 0)
    d = 3
    assert s3.samples.shape == (512, 101, d + 3) and s0.samples.shape == (512, 101, d)
    assert np.array_equal(s3.samples[..., :d], s0.samples)
    assert np.array_equal(s3.loglikes, s0.loglikes) and np.array_equal(s3.latent_samples, s0.latent_samples)
    assert s3.total_calls == s0.total_calls
    der = s3.samples[..., d:]
    # the states are transformed in float64 (samples * std + mean): the likelihood and the derived kernel compute in
    # float64 too, so column 1 is the returned first coordinate itself
    assert np.array_equal(der[..., 0], s3.loglikes)
    assert np.array_equal(der[..., 1], s3.samples[..., 0])
    assert np.allclose(der[..., 2], np.sum(s3.samples[..., :d] ** 2, axis=2), rtol=1e-14, atol=0)


# ---- 4. NestedSampler.run -------------------------------------------------------------------------------------------
NAMES = ['p0', 'p1', 'logl', 'x0', 'sq']


def _ns(log_dir, num_derived, seed=0, **run_kw):
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood
    np.random.seed(seed)
    torch.manual_seed(seed)
    s = NestedSampler(2, CudaLikelihood(2, DERIVED3, num_derived=num_derived), transform=lambda x: 5 * x,
                      num_live_points=400, flow='nvp', num_derived=num_derived,
                      param_names=NAMES if num_derived else NAMES[:2], log_dir=str(log_dir), log_level=logging.WARNING)
    s.run(**run_kw)
    return s


def _chain_invariant(path, d=2):
    """the derived-logl column's text is the minusloglike column's text with the sign flipped; header 2 + d + 3 names"""
    lines = open(path).read().splitlines()
    assert lines[0].split()[1:] == ['minusloglike'] + NAMES and len(lines[0].split()) == 2 + d + 3
    flip = lambda t: t[1:] if t.startswith('-') else '-' + t
    rows = [ln.split() for ln in lines[1:]]
    assert rows and all(len(r) == 2 + d + 3 for r in rows)
    assert all(r[2 + d] == flip(r[1]) for r in rows)
    return len(rows)


def test_nested_sampler_run_with_derived(tmp_path):
    kw = dict(mcmc_num_chains=200, train_iters=30, max_iters=1500, log_interval=400)
    a = _ns(tmp_path / 'a', 3, **kw)
    b = _ns(tmp_path / 'b', 0, **kw)
    assert a.logz == b.logz and a.h == b.h and a.niter == b.niter and a.total_calls == b.total_calls
    assert np.array_equal(a.weights, b.weights) and np.array_equal(a.samples, b.samples)
    assert np.array_equal(a.loglikes, b.loglikes)
    assert a.active_derived.shape == (400, 3) and b.active_derived.shape == (400, 0)
    assert np.array_equal(a.active_derived[:, 0], a.active_logl)
    n = _chain_invariant(os.path.join(a.logs['chains'], 'chain.txt'))
    assert n == len(a.loglikes)
    ck = os.path.join(a.logs['checkpoint'])
    assert os.path.exists(os.path.join(ck, 'saved_derived.npy'))
    assert not os.path.exists(os.path.join(b.logs['checkpoint'], 'saved_derived.npy'))
    assert sorted(os.listdir(b.logs['checkpoint'])) == sorted(f for f in os.listdir(ck) if f != 'saved_derived.npy')


def test_nested_sampler_resume_with_derived(tmp_path):
    kw = dict(mcmc_num_chains=200, train_iters=30, log_interval=300, strategy=['mcmc'])
    s1 = _ns(tmp_path, 3, seed=3, max_iters=700, **kw)
    run_dir = s1.logs['run_dir']
    ck = os.path.join(run_dir, 'checkpoint')
    its = sorted(int(f.split('checkpoint_')[1].split('.txt')[0]) for f in os.listdir(ck) if f.startswith('checkpoint_'))
    last = its[-1]
    assert last >= 600
    ad = np.load(os.path.join(ck, 'active_derived_%d.npy' % last))
    assert ad.shape == (400, 3)
    assert np.array_equal(ad[:, 0], np.load(os.path.join(ck, 'active_logl_%d.npy' % last)))
    sd = np.load(os.path.join(ck, 'saved_derived.npy'))
    assert sd.shape == (last, 3) and np.array_equal(sd[:, 0], np.load(os.path.join(ck, 'saved_logl.npy')))
    s2 = _ns(run_dir, 3, seed=4, **kw)
    assert not s2.logs['created'] and s2.niter > s1.niter
    assert np.array_equal(s2.active_derived[:, 0], s2.active_logl)
    n = _chain_invariant(os.path.join(s2.logs['chains'], 'chain.txt'))
    assert n == len(s2.loglikes)


def test_nested_sampler_rejection_strategies_with_derived(tmp_path):
    s = _ns(tmp_path, 3, seed=5, strategy=['rejection_prior', 'rejection_flow'], volume_switch=0.3, max_iters=900,
            train_iters=30, log_interval=300)
    assert np.array_equal(s.active_derived[:, 0], s.active_logl)
    assert _chain_invariant(os.path.join(s.logs['chains'], 'chain.txt')) == len(s.loglikes)


# ---- 5. two ranks ---------------------------------------------------------------------------------------------------
def _free_port():
    sock = socket.socket()
    sock.bind(('127.0.0.1', 0))
    p = sock.getsockname()[1]
    sock.close()
    return p


def test_two_rank_nested_run_with_derived(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.abspath(__file__), str(tmp_path)]
    subprocess.run(cmd, check=True, timeout=900)
    res = [np.load(tmp_path / ('rank%d.npz' % r)) for r in range(2)]
    # every rank ends with the same live set and the same chain-file content (weights, logl, parameters, derived)
    for k in res[0].files:
        assert np.array_equal(res[0][k], res[1][k]), k
    assert np.array_equal(res[0]['active_derived'][:, 0], res[0]['active_logl'])
    assert np.array_equal(res[0]['derived_samples'][:, 0], res[0]['loglikes'])
    run_dir = open(tmp_path / 'run_dir.txt').read()
    assert _chain_invariant(os.path.join(run_dir, 'chains', 'chain.txt')) == len(res[0]['loglikes'])


def _worker(out_dir):
    """one rank of test_two_rank_nested_run_with_derived (launched by torch.distributed.run)"""
    import torch.distributed as tdist
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    tdist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank = tdist.get_rank()
    s = _ns(os.path.join(out_dir, 'run'), 3, seed=6, mcmc_num_chains=200, train_iters=30, max_iters=900,
            log_interval=300, strategy=['rejection_prior', 'mcmc'])
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), logz=s.logz, niter=s.niter, active_derived=s.active_derived,
             active_logl=s.active_logl, samples=s.samples, loglikes=s.loglikes, weights=s.weights,
             derived_samples=s.derived_samples)
    if rank == 0:
        open(os.path.join(out_dir, 'run_dir.txt'), 'w').write(s.logs['run_dir'])
    tdist.barrier()
    tdist.destroy_process_group()


if __name__ == '__main__':
    _worker(sys.argv[1])
