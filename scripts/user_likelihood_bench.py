"""Built-in Rosenbrock against a user copy written in CUDA C++ (CudaLikelihood), on the c4 shape of bench.py
(Rosenbrock x_dim = 30, the fitted c4 flow, 65 536 chains x 150 steps, hard constraint, dynamic scale).

    python scripts/user_likelihood_bench.py [--rounds 5] [--out result.json]

For each step-kernel variant (tcgen05, FP32-FMA; the 16-lanes-per-chain kernel at 4 096 chains, the largest batch AUTO
gives it) the two likelihoods run alternately, `rounds` times each, in one process: the step kernel alone (CUDA events
around nnb_mcmc_run) and the whole refill (chain start + steps).  The user copy does the same arithmetic as the built-in
likelihood, so the end states must be equal bit for bit; that is checked too.  The tcgen05 kernel at x_dim = 30 inlines
packed Rosenbrock arithmetic for the built-in id only, so there the user copy takes the generic likelihood path.
Also reported: the one-off NVRTC compile time of each variant and the time to install it again from the on-disk cache,
and the card's name and power limit.
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
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import bench
    import user_sources as us
    from nnest_b200 import _lib as L
    from nnest_b200.engine import Engine, flatten_state_dict

    wl = bench.WORKLOADS['c4']
    d, S = wl['d'], wl['mcmc_steps']
    prob = bench.make_problem('c4', wl, wl['chains'], seed=0)
    flat, fd, fh, fl, fb, fflags = flatten_state_dict(prob['sd'], '')
    cache = tempfile.mkdtemp(prefix='nnb_jit_bench_')
    os.environ['NNB_JIT_CACHE'] = cache
    result = {'card': card(), 'workload': 'c4: ' + wl['desc'], 'rounds': args.rounds}

    def engine():
        e = Engine(0)
        e.set_flow(flat, fd, fh, fl, fb, fflags)
        return e

    def target(e, user):
        e.set_target(d, L.NNB_LIKE_USER if user else L.NNB_LIKE_ROSENBROCK, (), t_scale=wl['ts'], t_shift=0.0,
                     prior_kind=L.NNB_PRIOR_BOX_U, prior_lo=-1.0, prior_hi=1.0,
                     user_source=us.ROSENBROCK if user else None)

    variants = [('tcgen05', L.NNB_IMPL_TCGEN05, wl['chains']), ('ffma', L.NNB_IMPL_FFMA, wl['chains']),
                ('warp16', L.NNB_IMPL_WARP, 4096)]
    inputs = {n: (torch.from_numpy(np.ascontiguousarray(prob['init_u'][:n].astype(np.float32).T)).cuda(),
                  torch.from_numpy(np.ascontiguousarray(prob['init_logl'][:n])).cuda()) for _, _, n in variants}

    def refill(e, impl, n, it, ev=None):
        u, l = inputs[n]
        if ev:
            ev[0].record()
        st, _, _ = e.mcmc_init(n, init_u=u, init_logl=l, seed=1)
        if ev:
            ev[1].record()
        out = e.mcmc_run(st, S, mode=L.NNB_MODE_HARD, loglstar=prob['loglstar'], step_size=1 / d ** 0.5,
                         dynamic_step_size=True, seed=1, step_offset=it * S, impl=impl, sync=False)
        if ev:
            ev[2].record()
        return st, out

    # ---- compile: fresh cache, then the same variants again from the on-disk cache in a new handle ---------------------
    compile_s = {}
    for label in ('nvrtc_compile', 'disk_cache_hit'):
        e = engine()
        t0 = time.perf_counter()
        n_comp = e.set_user_likelihood(us.ROSENBROCK)
        target(e, True)
        times = {'likelihood_kernel': time.perf_counter() - t0, 'likelihood_kernel_compiled': n_comp}
        for name, impl, n in variants:
            for k in range(2):           # the first run compiles (or loads) the step kernels, the second only runs
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                refill(e, impl, n, 0)
                torch.cuda.synchronize()
                times[name + ('_first_refill' if k == 0 else '_second_refill')] = time.perf_counter() - t0
            times[name + '_load'] = times[name + '_first_refill'] - times[name + '_second_refill']
        compile_s[label] = times
        del e
    result['seconds'] = compile_s
    result['nvrtc'] = 'libnvrtc.so.12 as loaded by nnest_b200._lib'

    # ---- alternating timing ------------------------------------------------------------------------------------------
    e = engine()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')   # > 126 MB of L2
    timings = {}
    for name, impl, n in variants:
        rec = {'builtin': {'step_ms': [], 'refill_ms': []}, 'user': {'step_ms': [], 'refill_ms': []}}
        ends = {}
        for user in (False, True):                     # warm-up of both, and the bit-for-bit check
            target(e, user)
            for it in range(3):
                st, out = refill(e, impl, n, it)
            torch.cuda.synchronize()
            ends[user] = (st.x.cpu().numpy(), st.logl.cpu().numpy(), e.mcmc_result())
        same = bool(np.array_equal(ends[False][0], ends[True][0]) and np.array_equal(ends[False][1], ends[True][1])
                    and ends[False][2] == ends[True][2])
        for r in range(args.rounds):
            for user in ((False, True) if r % 2 == 0 else (True, False)):
                target(e, user)
                key = 'user' if user else 'builtin'
                for it in range(4):
                    flush.zero_()
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                    st, out = refill(e, impl, n, it, ev)
                    torch.cuda.synchronize()
                    rec[key]['step_ms'].append(ev[1].elapsed_time(ev[2]))
                    rec[key]['refill_ms'].append(ev[0].elapsed_time(ev[2]))
        summary = {'chains': n, 'impl_ran': out['impl'], 'end_states_identical': same}
        for key in ('builtin', 'user'):
            for m in ('step_ms', 'refill_ms'):
                v = np.array(rec[key][m])
                summary[key + '_' + m] = {'median': float(np.median(v)), 'min': float(v.min()), 'max': float(v.max())}
            summary[key + '_proposals_per_s'] = n * S / (summary[key + '_step_ms']['median'] * 1e-3)
        summary['user_over_builtin_step_time'] = summary['user_step_ms']['median'] / summary['builtin_step_ms']['median']
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
