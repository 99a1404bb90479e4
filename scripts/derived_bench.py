"""What derived parameters (CudaLikelihood(num_derived=...)) cost, on the shapes of bench.py.

    python scripts/derived_bench.py [--rounds 2] [--out result.json] [--only kernel|refill|mcmc_run ...]

1. kernel: nnb_derived_trace over a c5-shaped trace (32 768 chains x 1 001 rows x d = 50, float32, 6.6 GB: far larger
   than the L2, so every pass reads HBM) with 4 derived columns, in chunks of 100 rows as Sampler._trace_to_host runs it.
   CUDA events around the whole sweep; the bytes it has to move (4 d bytes read and 8 n_der written per point) over that
   time, against the 7.7 TB/s of the data sheet.  Both without and with the "unmoved since row 0" test (init given).
2. MCMCSampler.run on the c5 shape per GPU (d = 50, 32 768 chains, 1 000 Metropolis-Hastings steps, thin = 10, a user
   Gaussian likelihood, flow fitted for 20 epochs), with and without the 4 derived columns, alternating.
3. the per-refill cost on the c4 shape (Rosenbrock d = 30, 65 536 chains x 150 steps, hard constraint): the refill
   (chain start + steps) and Sampler._refill_to_host -- where the derived parameters of the end states are evaluated and
   copied -- with 3 and 0 derived columns, alternating.
The card's name, power limit and maximum SM clock are read in the same process.
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# isotropic Gaussian log-likelihood; derived: the likelihood, x(0), sum of squares, max |x(i)|
GAUSS4 = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  double s = 0.0;
  for (int i = 0; i < d; ++i) s += (double)x(i) * (double)x(i);
  return -0.5 * s;
}
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  double s = 0.0, m = 0.0;
  for (int i = 0; i < d; ++i) {
    const double v = (double)x(i);
    s += v * v;
    m = fmax(m, fabs(v));
  }
  derived[0] = -0.5 * s;
  derived[1] = (double)x(0);
  derived[2] = s;
  derived[3] = m;
}
'''

# Rosenbrock with 3 derived columns (tests/test_user_derived.py)
ROSEN3 = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  typedef decltype(x(0)) T;
  T acc = (T)0;
  T prev = x(0);
  for (int i = 1; i < d; ++i) {
    const T cur = x(i);
    const T t1 = cur - prev * prev;
    const T t2 = (T)1 - prev;
    acc = acc + ((T)100 * (t1 * t1) + t2 * t2);
    prev = cur;
  }
  return -(double)acc;
}
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  derived[0] = nnb_user_loglike(x, d, params);
  derived[1] = (double)x(0);
  double s = 0.0;
  for (int i = 0; i < d; ++i) s += (double)x(i) * (double)x(i);
  derived[2] = s;
}
'''

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:
        return {'error': str(e)}


def kernel_bench(rounds):
    import torch
    from nnest_b200 import _lib as L
    from nnest_b200.engine import Engine
    d, n, T, nd, chunk = 50, 32768, 1001, 4, 100
    eng = Engine(0)
    eng.set_target(d, L.NNB_LIKE_USER, (), t_scale=np.ones(d), t_shift=np.zeros(d), user_source=GAUSS4, num_derived=nd)
    g = torch.Generator(device='cuda').manual_seed(0)
    trace = torch.randn((T, d, n), device='cuda', generator=g) * 0.5
    trace[1::3] = trace[0]          # a third of the rows equal to row 0: exercised by the init variant
    init = torch.zeros((nd, n), dtype=torch.float64, device='cuda')
    buf = torch.empty((chunk, nd, n), dtype=torch.float64, device='cuda')
    res = {}
    for name, ini in (('no_init', None), ('with_init', init)):
        def sweep():
            for r0 in range(0, T, chunk):
                nr = min(chunk, T - r0)
                eng.derived_trace(trace, r0, 1, nr, init=ini, out=buf[:nr])
        sweep()
        torch.cuda.synchronize()
        times = []
        for _ in range(max(3, rounds)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sweep()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) / 1e3)
        t = float(np.median(times))
        moved = float(T) * n * (4 * d + 8 * nd)
        res[name] = {'seconds': times, 'median_s': t, 'bytes_needed': moved, 'GB_per_s': moved / t / 1e9,
                     'share_of_hbm_bound': moved / HBM_BYTES_PER_S / t}
    res['shape'] = {'rows': T, 'd': d, 'chains': n, 'num_derived': nd, 'rows_per_launch': chunk}
    del trace, buf
    torch.cuda.empty_cache()
    return res


def mcmc_run_bench(rounds):
    import torch
    from nnest_b200 import MCMCSampler
    from nnest_b200.likelihoods import CudaLikelihood
    from nnest_b200.priors import UniformPrior
    d, n, S = 50, 32768, 1000
    tmp = tempfile.mkdtemp(prefix='derived_bench_')
    samplers = {}
    for nd in (0, 4):
        samplers[nd] = MCMCSampler(d, CudaLikelihood(d, GAUSS4, num_derived=nd), prior=UniformPrior(d, -10, 10),
                                   flow='nvp', num_derived=nd, log_dir=os.path.join(tmp, 'nd%d' % nd),
                                   log_level=logging.WARNING)
    training = np.random.RandomState(0).normal(size=(4000, d))
    times = {0: [], 4: []}
    for r in range(rounds + 1):                      # round 0 warms up (NVRTC compiles, allocations)
        for nd in (0, 4):
            s = samplers[nd]
            np.random.seed(r)
            torch.manual_seed(r)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s.run(S, n, training, stats_interval=None, train_iters=20, thin=10)
            torch.cuda.synchronize()
            if r:
                times[nd].append(time.perf_counter() - t0)
            assert s.samples.shape == (n, S // 10 + 1, d + nd)
            s.samples = s.latent_samples = s.loglikes = None
    return {'shape': {'d': d, 'chains': n, 'steps': S, 'thin': 10, 'train_epochs': 20},
            'seconds_without': times[0], 'seconds_with_4_derived': times[4]}


def refill_bench(rounds):
    import torch
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import CudaLikelihood
    d, n, S = 30, 65536, 150
    tmp = tempfile.mkdtemp(prefix='derived_bench_ns_')
    rng = np.random.RandomState(0)
    u = rng.uniform(-0.2, 0.2, size=(n, d)).astype(np.float32)
    res = {}
    samplers = {nd: NestedSampler(d, CudaLikelihood(d, ROSEN3, num_derived=nd), transform=lambda x: 5 * x, flow='nvp',
                                  num_derived=nd, num_live_points=1000, log_dir=os.path.join(tmp, 'nd%d' % nd),
                                  log_level=logging.WARNING)
                for nd in (0, 3)}
    logl = samplers[0].loglike(u)[0].astype(np.float64)
    loglstar = float(np.quantile(logl, 0.3))
    out = {0: {'refill_s': [], 'to_host_s': []}, 3: {'refill_s': [], 'to_host_s': []}}
    for r in range(rounds * 3 + 1):
        for nd in (0, 3):
            s = samplers[nd]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            batch = s._mcmc_refill(S, u, logl, loglstar, 1 / d ** 0.5, True)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            s._refill_to_host(batch)
            t2 = time.perf_counter()
            if r:
                out[nd]['refill_s'].append(t1 - t0)
                out[nd]['to_host_s'].append(t2 - t1)
    res['shape'] = {'d': d, 'chains': n, 'steps': S}
    res['without'], res['with_3_derived'] = out[0], out[3]
    res['median_to_host_overhead_s'] = float(np.median(out[3]['to_host_s']) - np.median(out[0]['to_host_s']))
    res['median_refill_s'] = float(np.median(out[0]['refill_s']))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--out', default=None)
    ap.add_argument('--only', choices=['kernel', 'refill', 'mcmc_run'], action='append',
                    help='run only these parts (repeatable; default: all three)')
    args = ap.parse_args()
    os.environ.setdefault('NNB_JIT_CACHE', tempfile.mkdtemp(prefix='nnb_jit_'))
    parts = args.only or ['kernel', 'refill', 'mcmc_run']
    result = {'card': card()}
    for part, key, fn in (('kernel', 'derived_trace_kernel_c5', kernel_bench), ('refill', 'refill_c4', refill_bench),
                          ('mcmc_run', 'mcmc_sampler_run_c5', mcmc_run_bench)):
        if part in parts:
            result[key] = fn(args.rounds)
            print(json.dumps(result[key]), flush=True)
    result['card_after'] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, 'w').write(text)


if __name__ == '__main__':
    main()
