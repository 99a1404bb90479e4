"""GPU: repeated identical launches agree (race detector for the cooperative kernels: per-step grid barrier of the MCMC
step kernel, gradient exchange + grid barrier of the fused fitting kernel).  tests/dev_stress.py is the long version."""
import numpy as np
import pytest

torch = pytest.importorskip('torch')

pytestmark = pytest.mark.gpu


def test_mcmc_refill_is_bit_reproducible():
    import bench
    from nnest_b200 import _lib as L
    from nnest_b200.engine import Engine
    eng = Engine(0)
    wl = dict(bench.WORKLOADS['c4'])
    d, n, S = wl['d'], wl['chains'], 40
    eng.set_target(d, 0, [], t_scale=5.0, t_shift=0.0, prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)
    prob = bench.make_problem('c4', wl, n)
    eng.set_flow_from_state_dict(prob['sd'])
    u = torch.from_numpy(np.ascontiguousarray(prob['init_u'].astype(np.float32).T)).cuda()
    logl = torch.from_numpy(prob['init_logl']).cuda()
    ref = None
    for _ in range(12):
        st, _, _ = eng.mcmc_init(n, init_u=u, init_logl=logl, seed=5)
        out = eng.mcmc_run(st, S, mode=L.NNB_MODE_HARD, loglstar=prob['loglstar'], step_size=1 / d ** 0.5,
                           dynamic_step_size=True, seed=5)
        cur = (st.x.clone(), st.z.clone(), st.logl.clone(), out['naccept'], out['ncall'], out['scale'])
        if ref is None:
            ref = cur
        else:
            assert torch.equal(cur[0], ref[0]) and torch.equal(cur[1], ref[1]) and torch.equal(cur[2], ref[2])
            assert cur[3:] == ref[3:]
    # queued without intermediate synchronisation (sync=False) == the synchronous result
    for _ in range(3):
        st, _, _ = eng.mcmc_init(n, init_u=u, init_logl=logl, seed=5)
        eng.mcmc_run(st, S, mode=L.NNB_MODE_HARD, loglstar=prob['loglstar'], step_size=1 / d ** 0.5,
                     dynamic_step_size=True, seed=5, sync=False)
    res = eng.mcmc_result()
    assert torch.equal(st.x, ref[0]) and torch.equal(st.logl, ref[2])
    assert (res['naccept'], res['ncall'], res['scale']) == ref[3:]


def test_many_cta_fitting_is_bit_reproducible():
    """Several CTAs per mini-batch: partial gradients and losses are reduced in a fixed CTA order (no floating-point
    atomics), so identical inputs give identical bits -- weights, Adam moments, training loss, validation loss.  Batch 4096
    runs on 32 CTAs; batch 320 x sm_count on every SM, each CTA walking two or three 128-sample slices."""
    import bench
    from nnest_b200.engine import Engine
    eng = Engine(0)
    d = 30
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.RandomState(0)
    w0 = torch.from_numpy(bench.flat_weights(bench.make_weights(d, 0))).cuda()
    for batch, n in ((4096, 20000), (320 * sm, 640 * sm + 777)):
        x = torch.from_numpy(rng.uniform(-1, 1, size=(n, d)).astype(np.float32)).cuda()
        ref = None
        for _ in range(10):
            w, m, v = w0.clone(), torch.zeros_like(w0), torch.zeros_like(w0)
            steps = 0
            for ep in range(2):
                tl, vs, grid = eng.train_epoch((d, 16, 1, 3), w, m, v, steps, x, x[:1000].contiguous(), batch,
                                               jitter=0.01, lr=1e-3, weight_decay=1e-6, seed=3, epoch=ep)
                steps += (n + batch - 1) // batch
            assert grid == min(batch // 128, sm)
            if ref is None:
                ref = (w.clone(), m.clone(), v.clone(), tl, vs)
            else:
                assert torch.equal(w, ref[0]) and torch.equal(m, ref[1]) and torch.equal(v, ref[2])
                assert tl == ref[3] and vs == ref[4]


def test_mean_nn_distance_is_bit_reproducible():
    from nnest_b200.engine import Engine
    eng = Engine(0)
    rng = np.random.RandomState(1)
    x = torch.from_numpy(rng.uniform(-1, 1, size=(20000, 10))).cuda()
    vals = {eng.mean_nn_distance(x) for _ in range(6)}
    assert len(vals) == 1
