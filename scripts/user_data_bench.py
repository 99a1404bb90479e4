"""Datasets of CUDA C++ likelihoods (CudaLikelihood(data=...)): step-kernel cost against the number of data points, the
same dataset written into the source as __constant__ arrays, and the cost of changing the dataset.

    python scripts/user_data_bench.py [--rounds 3] [--out result.json]

Likelihood: the straight-line chi-square of tests/data_sources.py (LINE: t, y float64, w float32, mask int32; x(0) and
x(1) are the line's intercept and slope, the other coordinates are free) at x_dim = 10, with the flow fitted for the c3
workload of bench.py (x_dim = 10) and its recorded live points as chain starts, at the c4 shape: 65 536 chains x 150
steps, hard constraint (the 30 % quantile of the start log-likelihoods), dynamic scale.  Step-kernel variants: tcgen05,
FP32-FMA (H = 16) and the 16-lanes-per-chain kernel at 4 096 chains.  N = 64, 512, 2 048 and 32 768 points.  For
N <= 2 048 the dataset also runs written into the source as __constant__ arrays ('baked'), alternating with the data
path in every round.  Timed: the step kernel alone (CUDA events around nnb_mcmc_run, L2 overwritten before each refill),
median and spread over `rounds` x 4 refills.  Data elements read per second count N x the proposals of the refill (every
proposal reads each of the N points of t, y and mask, and w where the mask is set); they are served from L1 / L2, not
from HBM.  Also reported: the one-off compile of a layout (likelihood and derived kernels, chain start and one step
kernel, fresh cache) and a data swap through Engine.set_target (upload + bind), both at N = 32 768, and the card's name,
power limit and maximum SM clock.  Compiled kernels go to a temporary directory.
"""
import argparse
import concurrent.futures as cf
import json
import multiprocessing as mp
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

NS = [64, 512, 2048, 32768]
BAKED_MAX = 2048
D, CHAINS, STEPS, T_SCALE = 10, 65536, 150, 2.0


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:      # the numbers stay valid, but without the card they cannot be compared
        return {'error': str(e)}


def variants():
    from nnest_b200 import _lib as L
    return [('tcgen05', L.NNB_IMPL_TCGEN05, CHAINS), ('ffma', L.NNB_IMPL_FFMA, CHAINS), ('warp16', L.NNB_IMPL_WARP, 4096)]


KEYS = [(n, 'data') for n in NS] + [(n, 'baked') for n in NS if n <= BAKED_MAX]


def likelihood(key):
    """the CudaLikelihood of key = (N, 'data' | 'baked')"""
    import data_sources as ds
    from nnest_b200.likelihoods import CudaLikelihood
    n, form = key
    data = ds.line_data(n, seed=n)
    if form == 'data':
        return CudaLikelihood(D, ds.LINE, data=data, num_derived=ds.LINE_DERIVED)
    return CudaLikelihood(D, ds.line_baked_source(data), num_derived=ds.LINE_DERIVED)


class Bench(object):
    def __init__(self):
        import torch
        import bench
        from nnest_b200.engine import flatten_state_dict
        wl = bench.WORKLOADS['c3']
        assert wl['d'] == D
        prob = bench.make_problem('c3', wl, CHAINS, seed=0)
        self.flow = flatten_state_dict(prob['sd'], '')
        self.u = torch.from_numpy(np.ascontiguousarray(prob['init_u'].astype(np.float32))).cuda()
        self.likes = {}
        self.starts = {}

    def engine(self):
        from nnest_b200.engine import Engine
        e = Engine(0)
        flat, fd, fh, fl, fb, fflags = self.flow
        e.set_flow(flat, fd, fh, fl, fb, fflags)
        return e

    def target(self, e, key):
        from nnest_b200 import _lib as L
        if key not in self.likes:
            self.likes[key] = likelihood(key)
        like = self.likes[key]
        e.set_target(D, L.NNB_LIKE_USER, (), t_scale=T_SCALE, t_shift=0.0, prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0,
                     prior_hi=1.0, user_source=like.device_source(), num_derived=like.num_derived,
                     user_data=like.device_data())

    def start(self, e, key):
        if key not in self.starts:
            self.target(e, key)
            logl = e.loglike(self.u)
            lstar = float(np.quantile(logl.cpu().numpy(), 0.3))
            self.starts[key] = {n: (self.u[:n].t().contiguous(), logl[:n].contiguous()) for _, _, n in variants()}, lstar
        return self.starts[key]

    def refill(self, e, key, impl, n, it, ev=None):
        from nnest_b200 import _lib as L
        starts, lstar = self.start(e, key)
        u, l = starts[n]
        st, _, _ = e.mcmc_init(n, init_u=u, init_logl=l, seed=1)
        if ev:
            ev[0].record()
        out = e.mcmc_run(st, STEPS, mode=L.NNB_MODE_HARD, loglstar=lstar, step_size=1 / D ** 0.5,
                         dynamic_step_size=True, seed=1, step_offset=it * STEPS, impl=impl, sync=False)
        if ev:
            ev[1].record()
        return st, out


def _warm(key):
    """compile (into the shared $NNB_JIT_CACHE) every kernel `key` runs: one refill per variant"""
    import torch
    b = Bench()
    e = b.engine()
    b.target(e, key)
    for _, impl, n in variants():
        b.refill(e, key, impl, n, 0)
    torch.cuda.synchronize()
    return key


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    result = {'card': card(), 'shape': {'x_dim': D, 'chains': CHAINS, 'steps': STEPS, 'warp16_chains': 4096,
                                        'flow': 'bench.py c3 fixture (fitted, x_dim 10)', 'points': NS},
              'rounds': args.rounds}
    cache = tempfile.mkdtemp(prefix='nnb_jit_data_bench_')
    fresh = tempfile.mkdtemp(prefix='nnb_jit_data_bench_fresh_')
    os.environ['NNB_JIT_CACHE'] = cache
    try:
        b = Bench()
        # ---- one-off compile of a layout and a data swap, N = 32 768 ---------------------------------------------------
        os.environ['NNB_JIT_CACHE'] = fresh
        e = b.engine()
        key, other = (NS[-1], 'data'), (NS[-2], 'data')   # two datasets of the same layout
        for k in (key, other):
            b.likes[k] = likelihood(k)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        b.target(e, key)
        t1 = time.perf_counter()
        b.refill(e, key, variants()[0][1], CHAINS, 0)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        swap = []
        for k in range(6):
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            b.target(e, other if k % 2 == 0 else key)
            torch.cuda.synchronize()
            swap.append(time.perf_counter() - t3)
        result['layout_compile_s'] = {'likelihood_and_derived_kernels': t1 - t0,
                                      'chain_start_and_tcgen05_step_kernel_with_first_refill': t2 - t1}
        result['data_swap_ms'] = {'median': 1e3 * float(np.median(swap)), 'min': 1e3 * min(swap),
                                  'max': 1e3 * max(swap), 'bytes_32768_points': 24 * NS[-1]}
        del e
        os.environ['NNB_JIT_CACHE'] = cache
        # ---- compile every other kernel in parallel processes (into the shared cache) ---------------------------------
        t0 = time.perf_counter()
        with cf.ProcessPoolExecutor(max_workers=len(KEYS), mp_context=mp.get_context('spawn')) as ex:
            list(ex.map(_warm, KEYS))
        result['parallel_warm_compile_s'] = time.perf_counter() - t0
        # ---- alternating timing ----------------------------------------------------------------------------------------
        e = b.engine()
        flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')   # > 126 MB of L2
        timings = {}
        for name, impl, n in variants():
            for N in NS:
                tkeys = [(N, 'data')] + ([(N, 'baked')] if N <= BAKED_MAX else [])
                rec = {k: [] for k in tkeys}
                ends = {}
                for k in tkeys:                                  # warm-up, and the end states of both forms
                    b.target(e, k)
                    for it in range(2):
                        st, out = b.refill(e, k, impl, n, it)
                    torch.cuda.synchronize()
                    ends[k] = (st.x.cpu().numpy(), st.logl.cpu().numpy(), e.mcmc_result())
                for r in range(args.rounds):
                    for k in (tkeys if r % 2 == 0 else tkeys[::-1]):
                        b.target(e, k)
                        for it in range(4):
                            flush.zero_()
                            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                            st, out = b.refill(e, k, impl, n, it, ev)
                            torch.cuda.synchronize()
                            rec[k].append(ev[0].elapsed_time(ev[1]))
                summary = {'chains': n, 'points': N, 'impl_ran': out['impl']}
                for k in tkeys:
                    v = np.array(rec[k])
                    med = float(np.median(v))
                    ncall = ends[k][2]['ncall']
                    summary[k[1]] = {'step_ms': {'median': med, 'min': float(v.min()), 'max': float(v.max())},
                                     'proposals_per_s': n * STEPS / (med * 1e-3),
                                     'data_elements_per_s': float(N) * ncall / (med * 1e-3)}
                if len(tkeys) == 2:
                    summary['data_over_baked'] = summary['data']['step_ms']['median'] / summary['baked']['step_ms']['median']
                    summary['end_states_identical'] = bool(np.array_equal(ends[tkeys[0]][0], ends[tkeys[1]][0]) and
                                                           np.array_equal(ends[tkeys[0]][1], ends[tkeys[1]][1]))
                timings['%s_N%d' % (name, N)] = summary
        result['timings'] = timings
    finally:
        shutil.rmtree(cache, ignore_errors=True)
        shutil.rmtree(fresh, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
