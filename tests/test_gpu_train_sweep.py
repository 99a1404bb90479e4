"""GPU: the fused flow-fitting kernel (train_epoch_kernel<H, L>, csrc/nnb_train.cuh) on every architecture it accepts, at
the edges of its shared-memory layout and on every kind of grid, against the float64 oracle (oracle/train.py).

Weights are oracle.flow.NVPWeights.random(..., gain=1.0), the nn.Linear default initialisation the reference trains
from.  At that gain even the deepest admitted flows (16 coupling blocks, two hidden layers) are well conditioned: the
float32 restatement of the oracle (nll_and_grad(dtype=np.float32)) stays within 5.6e-7 (max-norm relative) of the
float64 gradient on every shape below, so the 1e-5 criterion of the other training tests leaves a margin of 18.

Tolerances: gradients, Adam moments and losses 1e-5 relative (max-norm; losses relative to the sum of |-log p|); one
Adam step's weight change 1e-4 of its largest component, which leaves room for the float32 rounding of the weights."""
import logging

import numpy as np
import pytest

torch = pytest.importorskip('torch')

from oracle import philox as ophilox
from oracle import train as otrain
from oracle.flow import NVPWeights

pytestmark = pytest.mark.gpu

GAIN = 1.0
F32_ORACLE_MAX = 2.5e-6   # float32 restatement's own error must stay 4x below the 1e-5 bound (measured: <= 5.6e-7)
LR, EPS = 1e-2, 1e-8      # lr large enough that one step moves weights by far more than their float32 rounding
ADAM_CASES = [(s, wd, b) for s in (0, 7, 10 ** 6) for wd in (0.0, 0.05) for b in ((0.9, 0.999), (0.5, 0.9))]
ARCHS = [(16, 1), (16, 2), (32, 1), (32, 2)]
SHAPES = ['small', 'odd', 'wide', 'max_blocks_d5', 'max_blocks_d30', 'max_dim']
C4 = (30, 16, 1, 3)       # the config-4 architecture (d, hidden, num_layers, num_blocks)


@pytest.fixture(scope='module')
def engine():
    from nnest_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope='module')
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def dev(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to('cuda', dtype=dtype).contiguous()


def host(t):
    return t.cpu().numpy().astype(np.float64)


def max_blocks(engine, d, H, L):
    """largest num_blocks nnb_train_supported admits at (d, H, L); 0 if none"""
    B = 0
    while engine.train_supported(d, H, L, B + 1):
        B += 1
    return B


def max_dim(engine, H, L):
    """largest x_dim nnb_train_supported admits with one coupling block"""
    d = 2
    while engine.train_supported(d + 1, H, L, 1):
        d += 1
    return d


def resolve(engine, H, L, shape):
    """(d, num_blocks) of a named shape, or None where the architecture admits no such shape"""
    if shape == 'small':
        return 2, 1
    if shape == 'odd':
        return 7, min(3, max_blocks(engine, 7, H, L))
    if shape == 'wide':     # d > 2H: the staging matrices are sized by (d + 1) / 2 rather than by H
        B = max_blocks(engine, 2 * H + 1, H, L)
        return (2 * H + 1, B) if B else None
    if shape.startswith('max_blocks_d'):
        d = int(shape[len('max_blocks_d'):])
        return d, max_blocks(engine, d, H, L)
    assert shape == 'max_dim'
    return max_dim(engine, H, L), 1


def draw_x(rng, n, w0, arch):
    """n standard-normal samples, none within 1e-4 of a ReLU kink: there the gradient jumps, by ~1e-3 of its size at
    batch 128, and float32 rounding decides on which side a sample falls"""
    x = rng.normal(size=(n, arch[0])).astype(np.float32)
    while True:
        near = otrain.relu_margin(w0, x, *arch) < 1e-4
        if not near.any():
            return x
        x[near] = rng.normal(size=(int(near.sum()), arch[0])).astype(np.float32)


def draw_moments(rng, g):
    """Adam moments at the scale of g and g^2, drawn independently of g: the update then depends smoothly on g, unlike
    from zero moments, where the first step is ~lr * sign(g)"""
    s = np.sqrt(np.mean(g * g))
    return (s * rng.normal(size=g.size)).astype(np.float32), (s * s * rng.uniform(0.5, 2.0, size=g.size)).astype(np.float32)


def adam_reference(w0, g, m0, v0, step0, wd, betas):
    opt = otrain.Adam(w0.size, lr=LR, betas=betas, eps=EPS, weight_decay=wd)
    opt.m, opt.v, opt.step = m0.astype(np.float64), v0.astype(np.float64), step0
    w1 = opt.update(w0.astype(np.float64), g)
    return w1, opt.m, opt.v


def check_adam_step(w1, m1, v1, w0, g, m0, v0, step0, wd, betas):
    w_ref, m_ref, v_ref = adam_reference(w0, g, m0, v0, step0, wd, betas)
    assert rel(host(m1), m_ref) < 1e-5
    assert rel(host(v1), v_ref) < 1e-5
    dw_ref = w_ref - w0
    assert np.abs(host(w1) - w0.astype(np.float64) - dw_ref).max() < 1e-4 * np.abs(dw_ref).max()


def check_minibatch(engine, arch, w0, x, rng, adam_cases):
    """one mini-batch = the whole of x: gradient, loss and one Adam step per case in adam_cases against the oracle;
    returns the grid the kernel ran on"""
    nll, g = otrain.nll_and_grad(w0, x, *arch)
    m0, v0 = draw_moments(rng, g)
    grids = set()
    for step0, wd, betas in adam_cases:
        w, m, v, gout = dev(w0), dev(m0), dev(v0), torch.zeros(w0.size, device='cuda')
        tl, vs, grid = engine.train_epoch(arch, w, m, v, step0, dev(x), None, x.shape[0], grad_out=gout, lr=LR,
                                          betas=betas, eps=EPS, weight_decay=wd)
        grids.add(grid)
        assert rel(host(gout), g) < 1e-5
        assert abs(tl - nll.mean()) <= 1e-5 * np.abs(nll).mean()
        assert vs == 0.0
        check_adam_step(w, m, v, w0, g, m0, v0, step0, wd, betas)
    assert len(grids) == 1
    return grids.pop()


def check_validation(engine, arch, w0, xv):
    w = dev(w0)
    _, vs, grid = engine.train_epoch(arch, w, None, None, 0, None, dev(xv), 100, do_train=False)
    nll, _ = otrain.nll_and_grad(w0, xv, *arch, want_grad=False)
    assert abs(vs - nll.sum()) <= 1e-5 * np.abs(nll).sum()
    assert torch.equal(w, dev(w0))
    return grid


# ---- 1. every architecture, at the edges of the shared-memory layout ---------------------------------------------------
@pytest.mark.parametrize('shape', SHAPES)
@pytest.mark.parametrize('H,L', ARCHS)
def test_architecture_sweep_matches_oracle(engine, H, L, shape):
    """Batch 300: three CTAs, the last with a partial slice of 44 samples."""
    dB = resolve(engine, H, L, shape)
    if dB is None:
        assert not engine.train_supported(2 * H + 1, H, L, 1)
        pytest.skip('hidden %d, %d layers: no x_dim > 2 * hidden fits the shared memory' % (H, L))
    d, B = dB
    assert B >= 1 and engine.train_supported(d, H, L, B)
    arch = (d, H, L, B)
    rng = np.random.default_rng(1000 * d + 10 * B + H + L)
    w0 = NVPWeights.random(d, H, L, B, seed=int(rng.integers(1 << 30)), gain=GAIN).flat()
    x = draw_x(rng, 300, w0, arch)
    xv = rng.normal(size=(300, d)).astype(np.float32)
    g64 = otrain.nll_and_grad(w0, x, *arch)[1]
    assert rel(otrain.nll_and_grad(w0, x, *arch, dtype=np.float32)[1], g64) < F32_ORACLE_MAX
    assert check_minibatch(engine, arch, w0, x, rng, ADAM_CASES) == 3
    assert check_validation(engine, arch, w0, xv) == 3


@pytest.mark.parametrize('H,L', ARCHS)
def test_one_past_the_edge_is_refused(engine, H, L, monkeypatch):
    """At the largest admitted num_blocks (d = 5, 30) and x_dim (one block), one more is refused by nnb_train_epoch with
    NNB_ERR_UNSUPPORTED before anything is launched, and Trainer selects the fused kernel exactly for the admitted shapes."""
    from nnest_b200 import Trainer
    from nnest_b200 import _lib
    monkeypatch.delenv('NNB_TRAIN_AUTOGRAD', raising=False)
    dm = max_dim(engine, H, L)
    admitted = [(d, max_blocks(engine, d, H, L)) for d in (5, 30)] + [(dm, 1)]
    refused = [(d, B + 1) for d, B in admitted] + [(dm + 1, 1)]
    for (d, B), ok in [(s, True) for s in admitted] + [(s, False) for s in refused]:
        assert engine.train_supported(d, H, L, B) == ok
        if B > _lib.NNB_MAX_BLOCKS:     # the sampling kernels refuse such a flow, so Trainer does too
            with pytest.raises(_lib.NNBError):
                Trainer(d, hidden_dim=H, num_layers=L, num_blocks=B, flow='nvp', log_dir=None, engine=engine)
            continue
        t = Trainer(d, hidden_dim=H, num_layers=L, num_blocks=B, flow='nvp', log_dir=None, log_level=logging.ERROR,
                    engine=engine)
        assert t._fused == ok
    for d, B in refused:
        w = torch.zeros(2 * B * otrain.net_floats(d, H, L), device='cuda')
        with pytest.raises(_lib.NNBError) as e:
            engine.train_epoch((d, H, L, B), w, w.clone(), w.clone(), 0, torch.zeros((10, d), device='cuda'), None, 10)
        assert e.value.code == _lib.NNB_ERR_UNSUPPORTED
    # the handle is still usable after the refusals
    w0 = NVPWeights.random(5, H, L, 1, seed=5, gain=GAIN).flat()
    rng = np.random.default_rng(5)
    check_minibatch(engine, (5, H, L, 1), w0, draw_x(rng, 40, w0, (5, H, L, 1)), rng, ADAM_CASES[:1])


# ---- 2. grids: one CTA up to every SM, several 128-sample slices per CTA ------------------------------------------------
def odd_grid(sm_count):
    """A grid that does not divide Psm, the config-4 kernel's parameter count in shared memory (nets padded to 4 floats).
    Slices of Psm // grid would leave out the last Psm % grid entries of the reduce-scatter: at least padding + 2 of them
    reach b3[d - 2] of the last net (block 2's translate net), a weight with a non-zero gradient."""
    d, H, L, B = C4
    net = otrain.net_floats(d, H, L)
    netp = (net + 3) // 4 * 4
    psm = 2 * B * netp
    return next(g for g in range(3, sm_count) if psm % g >= netp - net + 2)


@pytest.mark.parametrize('kind', ['128', '129', 'odd_grid', 'sm_count', 'sm_count_x2.5'])
def test_grids_match_oracle(engine, sm_count, kind):
    batch = {'128': 128, '129': 129, 'odd_grid': 128 * odd_grid(sm_count), 'sm_count': 128 * sm_count,
             'sm_count_x2.5': 320 * sm_count}[kind]
    rng = np.random.default_rng(batch)
    w0 = NVPWeights.random(C4[0], C4[1], C4[2], C4[3], seed=batch, gain=GAIN).flat()
    x = draw_x(rng, batch, w0, C4)
    grid = check_minibatch(engine, C4, w0, x, rng, [(7, 0.05, (0.9, 0.999))])
    assert grid == min((batch + 127) // 128, sm_count)


def test_validation_only_on_many_ctas_matches_oracle(engine, sm_count):
    rng = np.random.default_rng(20000)
    w0 = NVPWeights.random(C4[0], C4[1], C4[2], C4[3], seed=11, gain=GAIN).flat()
    xv = rng.normal(size=(20000, C4[0])).astype(np.float32)
    assert check_validation(engine, C4, w0, xv) == min((20000 + 127) // 128, sm_count)


def test_gradient_only_shares_of_a_full_grid_minibatch(engine, sm_count):
    """grad_only: three shares of a mini-batch of 128 x sm_count samples, each on several CTAs, sum to the gradient of
    the whole mini-batch; each share is its part of the oracle's gradient (scaled by share / batch_total)."""
    total = 128 * sm_count
    cuts = [0, total // 4, total // 4 + (total * 7) // 20, total]
    rng = np.random.default_rng(7)
    w0 = NVPWeights.random(C4[0], C4[1], C4[2], C4[3], seed=12, gain=GAIN).flat()
    x = draw_x(rng, total, w0, C4)
    nll, g = otrain.nll_and_grad(w0, x, *C4)
    full = torch.zeros(w0.size, device='cuda')
    engine.train_epoch(C4, dev(w0), dev(np.zeros_like(w0)), dev(np.zeros_like(w0)), 0, dev(x), None, total,
                       grad_out=full, lr=LR)
    w = dev(w0)
    parts, loss = [], 0.0
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        assert hi - lo > 128
        gp = torch.zeros_like(w)
        tl, _, grid = engine.train_epoch(C4, w, None, None, 0, dev(x[lo:hi]), None, hi - lo, grad_out=gp,
                                         grad_only=True, batch_total=total, lr=LR)
        assert grid == (hi - lo + 127) // 128
        g_share = otrain.nll_and_grad(w0, x[lo:hi], *C4)[1] * ((hi - lo) / total)
        assert rel(host(gp), g_share) < 1e-5
        parts.append(host(gp))
        loss += tl
    assert torch.equal(w, dev(w0))
    assert np.abs(sum(parts) - host(full)).max() < 2e-6 * np.abs(host(full)).max()
    assert rel(sum(parts), g) < 1e-5
    assert abs(loss - nll.mean()) <= 1e-5 * np.abs(nll).mean()


# ---- 3. epoch bookkeeping: one launch == the same mini-batches one call each -------------------------------------------
@pytest.mark.parametrize('tail', [260, 100])
def test_epoch_equals_one_call_per_minibatch(engine, tail):
    """An epoch of four mini-batches of 300 (three CTAs each) and a short tail, in a random order, with replayed jitter
    noise and step0 > 0, against the same mini-batches run one call each (rows gathered through the permutation, the
    noise rows of their positions, step0 + i, moments carried over).  A tail of 260 runs on three CTAs in both, so every
    bit must agree; a tail of 100 runs on one CTA when called alone, so its step agrees to the oracle's tolerances."""
    arch, bs, step0, jit, wd, betas = C4, 300, 11, 0.05, 0.05, (0.9, 0.999)
    n = 4 * bs + tail
    rng = np.random.default_rng(tail)
    w0 = NVPWeights.random(arch[0], arch[1], arch[2], arch[3], seed=13, gain=GAIN).flat()
    x = rng.normal(size=(n, arch[0])).astype(np.float32)
    noise = rng.normal(size=(n, arch[0])).astype(np.float32)
    perm = rng.permutation(n)
    m0, v0 = draw_moments(rng, otrain.nll_and_grad(w0, x[:bs], *arch)[1])
    kw = dict(jitter=jit, lr=LR, betas=betas, eps=EPS, weight_decay=wd)

    w_e, m_e, v_e, g_e = dev(w0), dev(m0), dev(v0), torch.zeros(w0.size, device='cuda')
    tl_e, _, grid_e = engine.train_epoch(arch, w_e, m_e, v_e, step0, dev(x), None, bs, perm=dev(perm, torch.int64),
                                         noise=dev(noise), grad_out=g_e, **kw)
    assert grid_e == 3

    w_c, m_c, v_c = dev(w0), dev(m0), dev(v0)
    tl_c = []
    for i, lo in enumerate(range(0, n, bs)):
        if lo + bs >= n:
            w_tail, m_tail, v_tail = host(w_c), host(m_c), host(v_c)
        g_c = torch.zeros(w0.size, device='cuda')
        rows = perm[lo:lo + bs]
        tl, _, grid = engine.train_epoch(arch, w_c, m_c, v_c, step0 + i, dev(x[rows]), None, bs,
                                         noise=dev(noise[lo:lo + bs]), grad_out=g_c, **kw)
        assert grid == (len(rows) + 127) // 128
        tl_c.append(tl)

    # the tail step against the oracle, from the state the full mini-batches left
    rows = perm[4 * bs:]
    xb = x[rows].astype(np.float64) + np.float32(jit) * noise[4 * bs:].astype(np.float64)
    nll, g = otrain.nll_and_grad(w_tail, xb, *arch)
    assert rel(host(g_e), g) < 1e-5
    check_adam_step(w_e, m_e, v_e, w_tail, g, m_tail, v_tail, step0 + 4, wd, betas)
    # float partial losses summed in double in another order: equal up to double rounding when the grids agree
    if tail == 260:
        assert torch.equal(w_e, w_c) and torch.equal(m_e, m_c) and torch.equal(v_e, v_c) and torch.equal(g_e, g_c)
        assert abs(tl_e - sum(tl_c)) <= 1e-12 * abs(tl_e)
    else:
        assert rel(host(g_e), host(g_c)) < 1e-5
        assert abs(tl_e - sum(tl_c)) <= 1e-5 * np.abs(nll).mean()


# ---- 4. the jitter stream against its specification ----------------------------------------------------------------------
@pytest.mark.parametrize('d', [2, 3, 4, 5, 8, 30])
def test_jitter_stream_matches_philox_oracle(engine, d):
    """With zero weights the flow is the identity, and with x_train = 0, jitter = 1 and batch 1 the gradient of the
    translate net's output bias b3[i] (block i % 2, which transforms coordinate i) is exactly the i-th normal drawn for
    the sample: counter (j, epoch, position, tag 3) under the key (seed & 0xffffffff, seed >> 32).  The permutation is
    reversed, so the position (which keys the stream) differs from the row it reads.  lr = 0: the weights never move."""
    H, L, B = 16, 1, 2
    arch = (d, H, L, B)
    net = otrain.net_floats(d, H, L)
    b3 = H * d + H + L * (H * H + H) + d * H
    idx = [(2 * (i % 2) + 1) * net + b3 + i for i in range(d)]
    seed, epoch = (0x9E3779B9 << 32) | 0x2545F491, (1 << 31) + 12345
    for pos in (0, 1, 127, 128, 4099):
        n = pos + 1
        w = torch.zeros(2 * B * net, device='cuda')
        m, v, gout = torch.zeros_like(w), torch.zeros_like(w), torch.zeros_like(w)
        engine.train_epoch(arch, w, m, v, 0, torch.zeros((n, d), device='cuda'), None, 1,
                           perm=torch.arange(n - 1, -1, -1, device='cuda'), jitter=1.0, lr=0.0, seed=seed, epoch=epoch,
                           grad_out=gout)
        want = ophilox.normals(seed, epoch, [pos], d, tag=ophilox.TAG_TRAIN)[0]
        assert np.abs(host(gout)[idx] - want).max() < 1e-5, pos
        assert float(w.abs().max()) == 0.0
