"""The built-in affine map against prior transforms written in CUDA C++ (CudaTransform), on the c4 shape of bench.py
(Rosenbrock x_dim = 30, the fitted c4 flow, 65 536 chains x 150 steps, hard constraint, dynamic scale).

    python scripts/user_transform_bench.py [--rounds 3] [--out result.json]

Targets: 'builtin' (the affine map u * 5, ahead-of-time kernels), 'affine_copy' (the same map as a user transform, which
must reproduce the built-in end states bit for bit -- checked) and 'erfinv' (a Gaussian prior sigma * sqrt(2) erfinv(u),
float arithmetic like the other two).  For each step-kernel variant (tcgen05, FP32-FMA; the 16-lanes-per-chain kernel at
4 096 chains, the largest batch AUTO gives it) the three targets run alternately, `rounds` times each, in one process:
the step kernel alone (CUDA events around nnb_mcmc_run).  The tcgen05 kernel at x_dim = 30 and the 16-lane kernel inline
Rosenbrock together with the built-in map, so a user transform takes the generic likelihood path there.  Also reported:
the one-off NVRTC compile time of each variant, the time to load it again from the on-disk cache, and the card's name,
power limit and maximum SM clock.
"""
import argparse
import json
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


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(',')]
        return {'name': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:      # the numbers stay valid, but without the card they cannot be compared
        return {'error': str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import bench
    import transform_sources as tsrc
    from nnest_b200 import _lib as L
    from nnest_b200.engine import Engine, flatten_state_dict
    from nnest_b200.likelihoods import CudaTransform

    wl = bench.WORKLOADS['c4']
    d, S, scale = wl['d'], wl['mcmc_steps'], wl['ts']
    prob = bench.make_problem('c4', wl, wl['chains'], seed=0)
    flat, fd, fh, fl, fb, fflags = flatten_state_dict(prob['sd'], '')
    cache = tempfile.mkdtemp(prefix='nnb_jit_bench_')
    os.environ['NNB_JIT_CACHE'] = cache
    result = {'card': card(), 'workload': 'c4: ' + wl['desc'], 'rounds': args.rounds}
    transforms = {'affine_copy': CudaTransform(d, tsrc.AFFINE, params=[scale] * d + [0.0] * d, float64=False),
                  'erfinv': CudaTransform(d, tsrc.GAUSS, params=[2.0], float64=False)}
    box = dict(prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0)

    def engine():
        e = Engine(0)
        e.set_flow(flat, fd, fh, fl, fb, fflags)
        return e

    def target(e, key):
        if key == 'builtin':
            e.set_target(d, L.NNB_LIKE_ROSENBROCK, (), t_scale=scale, t_shift=0.0, **box)
        else:
            transforms[key].install(e, d, L.NNB_LIKE_ROSENBROCK, (), **box)

    variants = [('tcgen05', L.NNB_IMPL_TCGEN05, wl['chains']), ('ffma', L.NNB_IMPL_FFMA, wl['chains']),
                ('warp16', L.NNB_IMPL_WARP, 4096)]
    u_all = torch.from_numpy(np.ascontiguousarray(prob['init_u'].astype(np.float32))).cuda()
    # start log-likelihoods and constraint of each target: the c4 constraint's quantile among the start points
    q = float(np.mean(prob['init_logl'] < prob['loglstar']))
    starts = {}
    e = engine()
    for key in ('builtin', 'affine_copy', 'erfinv'):
        target(e, key)
        logl = e.loglike(u_all)
        lstar = prob['loglstar'] if key != 'erfinv' else float(np.quantile(logl.cpu().numpy(), q))
        starts[key] = {n: (u_all[:n].t().contiguous(), logl[:n].contiguous()) for _, _, n in variants}, lstar
    del e

    def refill(e, key, impl, n, it, ev=None):
        (u, l), lstar = starts[key][0][n], starts[key][1]
        st, _, _ = e.mcmc_init(n, init_u=u, init_logl=l, seed=1)
        if ev:
            ev[0].record()
        out = e.mcmc_run(st, S, mode=L.NNB_MODE_HARD, loglstar=lstar, step_size=1 / d ** 0.5, dynamic_step_size=True,
                         seed=1, step_offset=it * S, impl=impl, sync=False)
        if ev:
            ev[1].record()
        return st, out

    # ---- compile: fresh cache, then the same variants again from the on-disk cache in a new handle ---------------------
    compile_s = {}
    for label in ('nvrtc_compile', 'disk_cache_hit'):
        times = {}
        for key in ('affine_copy', 'erfinv'):
            e = engine()
            t0 = time.perf_counter()
            n_comp = e.set_user_transform(transforms[key].source)
            times[key + '_likelihood_kernels'] = time.perf_counter() - t0
            times[key + '_likelihood_kernels_compiled'] = n_comp
            target(e, key)
            for name, impl, n in variants:
                for k in range(2):       # the first run compiles (or loads) the step kernels, the second only runs
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    refill(e, key, impl, n, 0)
                    torch.cuda.synchronize()
                    times['%s_%s_%s_refill' % (key, name, 'first' if k == 0 else 'second')] = time.perf_counter() - t0
                times['%s_%s_load' % (key, name)] = times['%s_%s_first_refill' % (key, name)] - \
                    times['%s_%s_second_refill' % (key, name)]
            del e
        compile_s[label] = times
    result['seconds'] = compile_s

    # ---- alternating timing ------------------------------------------------------------------------------------------
    e = engine()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')   # > 126 MB of L2
    keys = ['builtin', 'affine_copy', 'erfinv']
    timings = {}
    for name, impl, n in variants:
        rec = {k: [] for k in keys}
        ends = {}
        for key in keys:                                # warm-up of all three, and the bit-for-bit check
            target(e, key)
            for it in range(3):
                st, out = refill(e, key, impl, n, it)
            torch.cuda.synchronize()
            ends[key] = (st.x.cpu().numpy(), st.logl.cpu().numpy(), e.mcmc_result())
        same = bool(np.array_equal(ends['builtin'][0], ends['affine_copy'][0]) and
                    np.array_equal(ends['builtin'][1], ends['affine_copy'][1]) and
                    ends['builtin'][2] == ends['affine_copy'][2])
        for r in range(args.rounds):
            for key in keys[r % 3:] + keys[:r % 3]:    # rotate the order between rounds
                target(e, key)
                for it in range(4):
                    flush.zero_()
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                    st, out = refill(e, key, impl, n, it, ev)
                    torch.cuda.synchronize()
                    rec[key].append(ev[0].elapsed_time(ev[1]))
        summary = {'chains': n, 'impl_ran': out['impl'], 'affine_copy_end_states_identical': same}
        for key in keys:
            v = np.array(rec[key])
            summary[key + '_step_ms'] = {'median': float(np.median(v)), 'min': float(v.min()), 'max': float(v.max())}
            summary[key + '_proposals_per_s'] = n * S / (summary[key + '_step_ms']['median'] * 1e-3)
        for key in ('affine_copy', 'erfinv'):
            summary[key + '_over_builtin'] = summary[key + '_step_ms']['median'] / summary['builtin_step_ms']['median']
        timings[name] = summary
    result['timings'] = timings
    shutil.rmtree(cache, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
