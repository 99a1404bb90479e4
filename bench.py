#!/usr/bin/env python
"""bench.py -- proposals/sec of the latent-space MCMC hot path (flow inverse + log-Jacobian + prior + likelihood +
accept/reject), the metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c3|c5|ns_c4] [--scaling strong|weak]
                    [--impl reference] [--dump-outputs DIR]

A "step" is one refill: `mcmc_steps` MCMC steps of every chain of the batch (one call of Sampler._mcmc_sample,
nnest/sampler.py:229) on synthetic inputs of the named shape.  Default workload `c4` = BASELINE.json configs[3], the
configuration the metric "at 1/2/4/8 B200" is quoted on (Rosenbrock x_dim=30, 65536 chains, 150 steps, hard likelihood
constraint, dynamic step size).  Inputs follow SURVEY.md section 8(d): live points = best 10 % of uniform prior draws,
flow = the reference's Trainer(flow='nvp') fitted on them (tests/golden/bench_<workload>.npz, recorded from the real
reference by tests/golden/make_bench_flows.py) and loaded into BOTH arms; chains start at active_u[randint].

Multi-GPU (`--gpus N`, launched under torchrun): the partitioning north_star names.  `--scaling strong` (default): the
workload's chains are SHARDED over the ranks (65536 chains -> 8192 per GPU at N = 8), global chain ids key the Philox
streams, and every step contains the collectives of a refill inside the timed region: the NCCL broadcast of the flow
weights (a retrain precedes every refill at this size: update_interval = nlive / 2) and the all_gather of the end states
(start point, end point, end loglike) in rank order (nnest/nested.py:416-427).  `--scaling weak` keeps the chains per
GPU fixed (N independent shards, same collectives).

`value`  = device-timed (CUDA events, max over ranks) steps with the inputs resident in HBM.
`e2e`    = the same refill through the repo's Python API, HOST arrays in, HOST arrays out: Sampler._mcmc_refill ->
           Sampler._refill_to_host (all_gather + pinned D2H); c5: MCMCSampler._mcmc_sample with a thinned host trace.
`ns_loop`= (extra) the refill as NestedSampler.run drives it, including the host replay of the live-point replacement
           over the whole gathered batch (NSBook.bulk -> nnb_ns_consume, nested.py:429-439), replicated on every rank.
`--impl reference` times the reference's own Sampler._mcmc_sample (UNMODIFIED, installed under oracle/_ref by
oracle/build_ref.py; the oracle port if that is absent) on the host cores, on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step handed its caller -- the gathered start points, end points and end
loglikes of every chain, and the step's scale and counters -- to DIR/<name>.npy, so that two builds can be compared output
for output: the inputs depend only on the arguments.
Prints ONE JSON line.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

WORKLOADS = {
    # name: likelihood, d, chains (total for strong scaling / per GPU for weak), mcmc_steps, mode, transform scale
    'c2': dict(like='himmelblau', d=2, chains=1024, mcmc_steps=10, mode='hard', ts=5.0, dynamic=True,
               desc='configs[1]: Himmelblau x_dim=2, 1024 chains x 10 steps, hard constraint'),
    'c3': dict(like='mixture', d=10, chains=16384, mcmc_steps=50, mode='hard', ts=10.0, dynamic=True,
               desc='configs[2]: GaussianMix x_dim=10, 16384 chains x 50 steps, hard constraint'),
    'c4': dict(like='rosenbrock', d=30, chains=65536, mcmc_steps=150, mode='hard', ts=5.0, dynamic=True,
               desc='configs[3]: Rosenbrock x_dim=30, 65536 chains x 150 steps, hard constraint, dynamic scale'),
    'c5': dict(like='gaussian', d=50, chains=262144, mcmc_steps=1000, mode='mh', ts=1.0, dynamic=False,
               desc='configs[4]: Gaussian(rho=0.99) x_dim=50, 262144 chains x 1000 steps, Metropolis-Hastings'),
}
# largest share of a workload one GPU holds (c5 is specified as 32768 chains per GPU on 8 GPUs)
MAX_PER_GPU = {'c5': 32768}
HIDDEN, LAYERS, BLOCKS = 16, 1, 3      # reference defaults, nnest/sampler.py:37,42,43
METRIC = 'latent-space MCMC proposals/sec (flow+loglike)'


def flow_flops_per_proposal(d):
    """Dense nn.Linear count of ONE flow inverse, 4*B*H*(2d + L*H) (SURVEY.md section 8d)."""
    return 4 * BLOCKS * HIDDEN * (2 * d + LAYERS * HIDDEN)


# ---- shared problem definition (both arms) ---------------------------------------------------------------------
def load_fixture(name):
    g = np.load(os.path.join(GOLDEN, 'bench_%s.npz' % name), allow_pickle=False)
    sd = {k[3:]: g[k] for k in g.files if k.startswith('sd/')}
    return g, sd


def make_problem(name, wl, n_total, seed=0):
    """Fitted flow (state_dict of the reference's netG) + chain starts drawn from the recorded live points
    (nested.py:405-407).  Identical on every rank and in both arms."""
    g, sd = load_fixture(name)
    rng = np.random.RandomState(seed)
    prob = dict(sd=sd)
    if wl['mode'] == 'hard':
        active_u, active_logl = g['active_u'].astype(np.float64), g['active_logl']
        idx = rng.randint(0, active_u.shape[0], size=n_total)
        prob.update(init_u=active_u[idx], init_logl=active_logl[idx], loglstar=float(g['loglstar']))
    else:
        prob.update(init_z=(0.5 * rng.normal(size=(n_total, wl['d']))).astype(np.float32), loglstar=None,
                    mean=g['mean'], std=g['std'])
    return prob


# legacy helpers kept for tests/dev scripts that build random-init flows
def make_weights(d, seed=0):
    rng = np.random.default_rng(seed)
    layers = []
    for _ in range(BLOCKS):
        for _net in ('scale', 'translate'):
            for o, i in [(HIDDEN, d)] + [(HIDDEN, HIDDEN)] * LAYERS + [(d, HIDDEN)]:
                b = 1.0 / np.sqrt(i)
                layers.append((rng.uniform(-b, b, size=(o, i)).astype(np.float32),
                               rng.uniform(-b, b, size=(o,)).astype(np.float32)))
    return layers


def flat_weights(layers):
    return np.concatenate([np.concatenate([w.ravel(), b.ravel()]) for w, b in layers])


LIKE_IDS = {'rosenbrock': (0, lambda d: []), 'himmelblau': (1, lambda d: []), 'gaussian': (2, lambda d: [0.99]),
            'mixture': (4, lambda d: [4.0, 1.0, 4.0, 0.4, 0.3, 0.2, 0.1])}


class ClockSampler(object):
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu, self.first = [], None, gpu_index, 0

    def mark(self, wait_s=3.0):
        """Call right before the timed region: waits until nvidia-smi delivers samples (its start-up -- process creation, NVML
        initialisation under the driver's global lock -- stalls CUDA launches for tens of milliseconds and must not fall
        into a timed region that is itself only ~100 ms long) and discards what was sampled before."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < wait_s:
            time.sleep(0.01)
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = self.rows[self.first:] or self.rows[-1:]
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows if len(r) >= 9 for i in range(4) if r[5 + i] == 'Active'})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ---- CPU arm: the reference itself (oracle/_ref) or, without it, the oracle port ---------------------------------
def reference_runner(name, wl, n_cpu):
    """Returns (run(steps) -> None, kind).  kind == 'reference': the UNMODIFIED adammoss/nnest Sampler._mcmc_sample
    (installed by oracle/build_ref.py), use_gpu=False, log_level=INFO, plot_trace=False, the fitted flow loaded into its
    netG, all host threads torch uses.  kind == 'port': oracle/mcmc.py with the reference's per-row loops."""
    import logging
    import tempfile
    d = wl['d']
    prob = make_problem(name, dict(wl), n_cpu)
    from oracle import refload
    if refload.installed_reference_available() or refload.reference_available():
        import torch
        nnest = refload.load_reference(installed=refload.installed_reference_available())
        from nnest import likelihoods as rl
        from nnest.priors import UniformPrior
        like = {'rosenbrock': lambda: rl.Rosenbrock(d), 'himmelblau': lambda: rl.Himmelblau(2),
                'mixture': lambda: rl.GaussianMix(d), 'gaussian': lambda: rl.Gaussian(d, 0.99)}[wl['like']]()
        log_dir = tempfile.mkdtemp(prefix='nnest_ref_bench_')
        kw = dict(hidden_dim=HIDDEN, num_layers=LAYERS, num_blocks=BLOCKS, flow='nvp', use_gpu=False, log_dir=log_dir,
                  log_level=logging.INFO)
        sd = {k: torch.from_numpy(np.array(v)) for k, v in prob['sd'].items()}
        if wl['mode'] == 'hard':
            ts = wl['ts']
            s = nnest.NestedSampler(d, like, transform=lambda x: ts * x, num_live_points=n_cpu, **kw)
            s.trainer.netG.load_state_dict(sd)
            logging.getLogger('nnest.sampler').setLevel(logging.WARNING)      # INFO computes nothing extra; keep stdout clean

            def run(steps):
                s._mcmc_sample(steps, init_samples=prob['init_u'], init_loglikes=prob['init_logl'],
                               init_derived=np.empty((n_cpu, 0)), loglstar=prob['loglstar'], step_size=1 / d ** 0.5,
                               dynamic_step_size=wl['dynamic'], plot_trace=False)
        else:
            s = nnest.MCMCSampler(d, like, prior=UniformPrior(d, -5, 5), **kw)
            s.trainer.netG.load_state_dict(sd)
            mean, std = prob['mean'], prob['std']
            s.transform = lambda x: x * std + mean                             # mcmc.py:111
            x0, _ = s.trainer.inverse(prob['init_z'], to_numpy=True)

            def run(steps):
                s._mcmc_sample(steps, num_chains=n_cpu, init_samples=x0, plot_trace=False)
        return run, 'reference'
    # ---- port ----
    from oracle import flow as oflow, likelihoods as olike, mcmc as omcmc
    like = {'rosenbrock': lambda: olike.Rosenbrock(d), 'himmelblau': lambda: olike.Himmelblau(2),
            'mixture': lambda: olike.GaussianMix(d), 'gaussian': lambda: olike.Gaussian(d, 0.99)}[wl['like']]()
    w = oflow.NVPWeights.from_state_dict(prob['sd'], d)
    if wl['mode'] == 'hard':
        ts = wl['ts']
        tr, prior = (lambda x: ts * x), olike.UniformPrior(d, -1, 1)
    else:
        mean, std = prob['mean'], prob['std']
        tr, prior = (lambda x: x * std + mean), olike.UniformPrior(d, -5, 5)

    def run(steps):
        target = omcmc.Target(like, transform=tr, prior=prior, transform_prior=wl['mode'] != 'hard', rowwise=True)
        kw = dict(init_samples=prob['init_u'], init_loglikes=prob['init_logl'], loglstar=prob['loglstar'],
                  step_size=1 / d ** 0.5, dynamic_step_size=wl['dynamic']) if wl['mode'] == 'hard' else \
            dict(init_z=prob['init_z'], loglstar=None)
        omcmc.mcmc_sample(w, target, steps, omcmc.TorchNoise(), **kw)
    return run, 'port'


def run_reference(args, name, wl):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    n_cpu = min(1024, wl['chains'])
    steps_cpu = min(wl['mcmc_steps'], 20 if wl['d'] <= 30 else 3)
    run, kind = reference_runner(name, wl, n_cpu)
    for _ in range(args.warmup):
        run(steps_cpu)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run(steps_cpu)
    dt = time.perf_counter() - t0
    value = n_cpu * steps_cpu * args.steps / dt
    cores = torch.get_num_threads()
    sample = '%d chains x %d mcmc steps per step (of %d x %d); %s' % (
        n_cpu, steps_cpu, wl['chains'], wl['mcmc_steps'],
        'adammoss/nnest Sampler._mcmc_sample, unmodified (oracle/_ref)' if kind == 'reference'
        else 'oracle port with per-row prior/likelihood loops')
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'proposals/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True,
        'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': name + ': ' + wl['desc'], 'sample': sample,
                   'flow_weights': 'reference Trainer fit (tests/golden/bench_%s.npz)' % name},
        'cpu_baseline': {'value': value, 'unit': 'proposals/s', 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'proposals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


def cpu_baseline_quick(name, wl, budget_s=15.0):
    """The reference (or the port) on rank 0's host cores for ~budget_s seconds."""
    import torch
    n_cpu = min(1024, wl['chains'])
    run, kind = reference_runner(name, wl, n_cpu)
    steps_cpu = 5 if wl['d'] <= 30 else 2
    done, t0 = 0, time.perf_counter()
    while True:
        run(steps_cpu)
        done += n_cpu * steps_cpu
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {'value': done / dt, 'unit': 'proposals/s', 'cores': torch.get_num_threads(), 'kind': kind,
            'sample': '%d chains, %d proposals in %.1f s (%s)' % (
                n_cpu, done, dt, 'unmodified reference Sampler._mcmc_sample from oracle/_ref' if kind == 'reference'
                else 'oracle port, per-row prior/likelihood loops as in the reference')}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, per_chain, scalars, seed=0):
    """Writes every array to out_dir/<name>.npy (float32 arrays stay float32, all others become float64).  `per_chain`
    arrays have one row per chain; if together they exceed DUMP_LIMIT_BYTES, the same seeded sample of rows is kept of
    each and chain_index.npy names the rows kept."""
    per_chain = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in per_chain.items()}
    scalars = {k: np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in scalars.items()}
    n = len(next(iter(per_chain.values())))
    row_bytes = sum(v.nbytes for v in per_chain.values()) // max(n, 1)
    budget = DUMP_LIMIT_BYTES - sum(v.nbytes for v in scalars.values())
    if n * row_bytes > budget:
        keep = budget // (row_bytes + 8)
        rows = np.sort(np.random.RandomState(seed).choice(n, keep, replace=False))
        per_chain = {k: v[rows] for k, v in per_chain.items()}
        per_chain['chain_index'] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in list(per_chain.items()) + list(scalars.items()):
        np.save(os.path.join(out_dir, k + '.npy'), np.ascontiguousarray(v))


def roofline_traffic(kernel_key, n, S):
    """dram bytes per launch from the tracked profile summary (profiles/roofline_traffic.json, written by
    profiles/ncu_summary.py from an `ncu --set full` capture), scaled to this launch's proposals."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')))[kernel_key]
        return t['dram_bytes_per_launch'] * (n * S) / float(t['chains'] * t['mcmc_steps']), t['source']
    except Exception:
        return None, None


# ---- GPU arm -------------------------------------------------------------------------------------------------------
def run_gpu(args, name, wl):
    import logging
    import tempfile
    import torch
    import torch.distributed as dist
    from nnest_b200 import build as nb_build
    from nnest_b200 import _lib as L

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    nb_build.build()
    from nnest_b200.engine import Engine, flatten_state_dict

    d, S = wl['d'], wl['mcmc_steps']
    cap = MAX_PER_GPU.get(name)
    if args.scaling == 'strong':
        n_total = wl['chains']
        if cap and n_total // world > cap:       # the named size does not fit fewer GPUs: keep the per-GPU share
            n_total = cap * world
        n_total -= n_total % world
    else:
        n_total = (min(wl['chains'], cap) if cap else wl['chains']) * world
    n = n_total // world                         # chains of this rank
    chain_offset = rank * n
    mode = L.NNB_MODE_HARD if wl['mode'] == 'hard' else L.NNB_MODE_MH
    prob = make_problem(name, wl, n_total, seed=args.seed)
    flat, fd, fh, fl, fb, fflags = flatten_state_dict(prob['sd'], '')
    eng = Engine(local)
    like_id, like_params = LIKE_IDS[wl['like']][0], LIKE_IDS[wl['like']][1](d)
    if wl['mode'] == 'hard':
        eng.set_target(d, like_id, like_params, t_scale=wl['ts'], t_shift=0.0, prior_kind=L.NNB_PRIOR_BOX_U,
                       prior_lo=-1.0, prior_hi=1.0)
    else:
        eng.set_target(d, like_id, like_params, t_scale=prob['std'], t_shift=prob['mean'], compute_f64=True,
                       prior_kind=L.NNB_PRIOR_BOX_V, prior_lo=-5.0, prior_hi=5.0)
    eng.set_flow(flat, fd, fh, fl, fb, fflags)
    step_size = 1 / d ** 0.5 if wl['mode'] == 'hard' else 0.0
    sl = slice(chain_offset, chain_offset + n)

    # ---- device-resident arm: inputs already in HBM ------------------------------------------------
    if wl['mode'] == 'hard':
        init_kw = dict(init_u=torch.from_numpy(np.ascontiguousarray(prob['init_u'][sl].astype(np.float32).T)).cuda(),
                       init_logl=torch.from_numpy(np.ascontiguousarray(prob['init_logl'][sl])).cuda())
    else:
        init_kw = dict(init_z=torch.from_numpy(np.ascontiguousarray(prob['init_z'][sl].T)).cuda())
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device='cuda')   # > 126 MB L2
    w_dev = torch.from_numpy(flat).cuda()
    gat_first = torch.empty((n_total, d), dtype=torch.float32, device='cuda')
    gat_last = torch.empty((n_total, d), dtype=torch.float32, device='cuda')
    gat_logl = torch.empty((n_total,), dtype=torch.float64, device='cuda')
    kernel_impl = {'auto': L.NNB_IMPL_AUTO, 'ffma': L.NNB_IMPL_FFMA, 'tcgen05': L.NNB_IMPL_TCGEN05,
                   'warp': L.NNB_IMPL_WARP}[args.kernel]
    run_ev = []
    coll = {'bcast': 0, 'all_gather': 0}

    def collect(first_x, st):
        """all_gather of the end states in rank order (nested.py:416-427)"""
        first, last = first_x.t().contiguous(), st.x.t().contiguous()
        if world > 1:
            dist.all_gather_into_tensor(gat_first, first)
            dist.all_gather_into_tensor(gat_last, last)
            dist.all_gather_into_tensor(gat_logl, st.logl)
            coll['all_gather'] += 3
            return gat_first, gat_last, gat_logl
        return first, last, st.logl

    def one_refill(it, timed=False, fixed_scale=False):
        if world > 1 and not fixed_scale:
            # a retrain precedes the refill: rank 0's weights go to every rank as one flat buffer, then to the kernels
            dist.broadcast(w_dev, src=0)
            coll['bcast'] += 1
            eng.set_flow(w_dev.cpu().numpy(), fd, fh, fl, fb, fflags)
        st, _, _ = eng.mcmc_init(n, seed=args.seed, chain_offset=chain_offset, **init_kw)
        first_x = st.x.clone()
        if timed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        out = eng.mcmc_run(st, S, mode=mode, loglstar=prob['loglstar'], step_size=step_size,
                           dynamic_step_size=wl['dynamic'] and not fixed_scale, seed=args.seed,
                           chain_offset=chain_offset, step_offset=it * S, impl=kernel_impl, sync=False)
        if timed:
            b.record()
            run_ev.append((a, b))
        ends = collect(first_x, st)
        return st, out, ends

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # sharding invariance: with a FIXED step size the gathered end states do not depend on how many GPUs the chains are
    # split over (Philox streams keyed by global chain id) -- the hash below must be the same at every N.  (With the dynamic
    # step size of the timed workload the scale adapts on each rank's own accept counts, as under the reference's MPI.)
    _, _, ends = one_refill(0, fixed_scale=True)
    torch.cuda.synchronize()
    hsh = hashlib.sha1()
    for t in ends:
        hsh.update(t.cpu().numpy().tobytes())
    shard_hash = hsh.hexdigest()[:16]

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()                      # (before the warm-up: see ClockSampler.mark)
    for it in range(args.warmup + 8):       # (+ 8 untimed refills: allocator pools, lazy module loads, clocks)
        # keep the results alive as the timed loop does: the previous refill's tensors are released only after the next one
        # has allocated its own, and the caching allocator must own that second set of blocks BEFORE the timed region (a
        # cudaMalloc inside an event pair drains the queue and showed up as one step of 6 - 190 ms)
        st, out, ends = one_refill(it)
    torch.cuda.synchronize()
    if rank == 0:
        clocks.mark()
    launches0 = eng.gpu_launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for it in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (not inside the event pair)
        ev[it][0].record()
        st, out, ends = one_refill(args.warmup + it, timed=True)
        ev[it][1].record()
    barrier()
    last = eng.mcmc_result()                # counters of the last refill
    naccept, ncall = last['naccept'], last['ncall']
    launches = eng.gpu_launches - launches0
    ms = [a.elapsed_time(b) for a, b in ev]
    step_ms = {'min': float(min(ms)), 'median': float(np.median(ms)), 'max': float(max(ms)),   # of this rank's steps
               'outliers': [(i, round(v, 3)) for i, v in enumerate(ms) if v > 1.5 * float(np.median(ms))][:8]}
    total_ms = float(sum(ms))
    t = torch.tensor([total_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    clk = clocks.stop() if rank == 0 else None
    proposals = n_total * S * args.steps
    value = proposals / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'first_x': ends[0].cpu().numpy(), 'last_x': ends[1].cpu().numpy(),
                                         'last_logl': ends[2].cpu().numpy()},
                     {'scale': last['scale'], 'naccept': naccept, 'ncall': ncall}, seed=args.seed)

    # ---- end-to-end arm: the repo's Python API, host arrays in, host live-point replacement out ----------------------
    from nnest_b200 import NestedSampler, MCMCSampler
    from nnest_b200 import likelihoods as nl
    from nnest_b200.priors import UniformPrior
    from nnest_b200.bookkeeping import NSBook
    log_dir = tempfile.mkdtemp(prefix='nnb_bench_')
    sd_t = {k: torch.from_numpy(np.array(v)) for k, v in prob['sd'].items()}
    like = {'rosenbrock': lambda: nl.Rosenbrock(d), 'himmelblau': lambda: nl.Himmelblau(2),
            'mixture': lambda: nl.GaussianMix(d), 'gaussian': lambda: nl.Gaussian(d, 0.99)}[wl['like']]()
    e2e_parts = {}
    if wl['mode'] == 'hard':
        ts = wl['ts']
        smp = NestedSampler(d, like, transform=lambda x: ts * x, flow='nvp', num_live_points=n_total, log_dir=log_dir,
                            log_level=logging.WARNING, seed=args.seed)
        smp.trainer.load_state_dict(sd_t)
        # this rank's start points in PINNED host memory (float32(active_u[idx]), trainer.py:249) and their loglikes
        my_u = torch.from_numpy(np.ascontiguousarray(prob['init_u'][sl], dtype=np.float32)).pin_memory()
        my_l = torch.from_numpy(np.ascontiguousarray(prob['init_logl'][sl])).pin_memory()
        h2d = my_u.numel() * 4 + my_l.numel() * 8
        d2h = n_total * (2 * d * 4 + 8)

        def one_e2e(it):
            """host start points in -> host end states of ALL ranks' chains out (what nested.py:429-439 consumes)"""
            t0 = time.perf_counter()
            batch = smp._mcmc_refill(S, my_u, my_l, prob['loglstar'], step_size, wl['dynamic'])
            t1 = time.perf_counter()
            smp._refill_to_host(batch)
            t2 = time.perf_counter()
            for k, v in (('mcmc_refill_ms', t1 - t0), ('gather_d2h_ms', t2 - t1)):
                e2e_parts[k] = e2e_parts.get(k, 0.0) + 1e3 * v
            return 0

        # the refill as NestedSampler.run drives it: chain starts by INDEX into the device-resident live set, gather + D2H,
        # then the live-point replacement over the whole gathered batch on the host (every rank replays it,
        # nested.py:429-439; NSBook.bulk -> nnb_ns_consume) and the scatter of the replacements into the device live set
        live_u0, live_l0 = prob['init_u'], np.ascontiguousarray(prob['init_logl'])
        live_dev = (torch.from_numpy(np.ascontiguousarray(live_u0)).cuda(), torch.from_numpy(live_l0).cuda())
        my_idx = np.arange(chain_offset, chain_offset + n, dtype=np.int64)
        ns_parts = {}

        def one_ns_refill(it):
            t0 = time.perf_counter()
            batch = smp._mcmc_refill(S, None, None, prob['loglstar'], step_size, wl['dynamic'],
                                     live=(live_dev[0], live_dev[1], my_idx))
            b_first, b_last, b_logl = smp._refill_to_host(batch)
            t1 = time.perf_counter()
            bk = NSBook(n_total)
            au, al = live_u0.copy(), live_l0.copy()
            av = ts * au
            t2 = time.perf_counter()
            bk.bulk(au, av, al, smp.transform, b_first, b_last, b_logl, 0, n_total, 0.0, 1 << 60)
            t3 = time.perf_counter()
            for k, v in (('refill_gather_d2h_ms', t1 - t0), ('consume_replay_ms', t3 - t2)):
                ns_parts[k] = ns_parts.get(k, 0.0) + 1e3 * v
            return bk.it
    else:
        thin = args.thin
        smp = MCMCSampler(d, like, prior=UniformPrior(d, -5, 5), flow='nvp', log_dir=log_dir,
                          log_level=logging.WARNING, seed=args.seed)
        smp.trainer.load_state_dict(sd_t)
        mean, std = prob['mean'], prob['std']
        smp.transform = lambda x: x * std + mean
        x0, _ = smp.trainer.inverse(prob['init_z'][sl], to_numpy=True)
        h2d = x0.size * 4
        rows = S // thin + 1
        d2h = n * rows * (2 * d * 4 + 8)

        def one_e2e(it):
            t0 = time.perf_counter()
            out = smp._mcmc_sample(S, num_chains=n, init_samples=x0, stats_interval=None, thin=thin)
            e2e_parts['mcmc_sample_ms'] = e2e_parts.get('mcmc_sample_ms', 0.0) + 1e3 * (time.perf_counter() - t0)
            return out[0].shape[1]

    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def time_loop(fn, parts):
        fn(0)
        fn(0)                               # two untimed calls: the first allocates pinned staging buffers
        parts.clear()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for it in range(e2e_steps):
            last_ret = fn(it)
        e1.record()
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        for k in list(parts):
            parts[k] /= e2e_steps
        return n_total * S * e2e_steps / (tt.item() * 1e-3), tt.item() / e2e_steps, last_ret

    e2e_value, e2e_ms, consumed = time_loop(one_e2e, e2e_parts)
    ns_loop = None
    if wl['mode'] == 'hard':
        v, ms_, consumed = time_loop(one_ns_refill, ns_parts)
        ns_loop = {'value': v, 'unit': 'proposals/s', 'ms_per_refill': ms_, 'ms_per_refill_parts': ns_parts,
                   'iterations_consumed_per_refill': int(consumed),
                   'what': 'refill as NestedSampler.run drives it: start indices into the device-resident live set -> '
                           'Sampler._mcmc_refill -> _refill_to_host (all_gather + pinned D2H) -> NSBook.bulk (host replay of '
                           'nested.py:429-439 over the whole gathered batch, replicated on every rank)'}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        # dominant kernel = the fused MCMC step kernel: its launches are timed live with CUDA events around nnb_mcmc_run
        run_ms = float(np.mean([a.elapsed_time(b) for a, b in run_ev]))
        kernel_launches = out['launches']
        flops = flow_flops_per_proposal(d)
        used_tc = out['impl'] == L.NNB_IMPL_TCGEN05
        achieved_tflops = n * S * flops / (run_ms * 1e-3) / 1e12           # algorithmic flops of one refill / its duration
        fp32_peak = 148 * 128 * 2 * ((clk or {}).get('sm_max_mhz') or 1965.0) * 1e6 / 1e12
        if used_tc and peaks.get('bf16_tflops'):
            peak, peak_src = peaks['bf16_tflops'] / 2.0, 'tf32 dense = 1/2 of the measured bf16 burst peak (MEASURED_PEAKS.json)'
        elif used_tc:
            peak, peak_src = 1590.0 / 2.0, 'tf32 dense = 1/2 of the fallback bf16 peak (B200_PROFILING.md)'
        else:
            peak, peak_src = fp32_peak, 'FP32 FMA pipe: 148 SMs x 128 lanes x 2 x max SM clock (not in MEASURED_PEAKS.json)'
        kernel_name = {L.NNB_IMPL_TCGEN05: 'mcmc_tc_kernel', L.NNB_IMPL_FFMA: 'mcmc_kernel'}.get(out['impl'], 'mcmc_warp_kernel')
        traffic, traffic_src = roofline_traffic(kernel_name, n, S)
        roofline = {
            'bound': 'tensor' if used_tc else 'fp32-fma', 'achieved': achieved_tflops, 'peak': peak, 'unit': 'TFLOP/s',
            'frac': achieved_tflops / peak, 'traffic': traffic, 'traffic_source': traffic_src,
            'kernel': kernel_name, 'launches_per_step': kernel_launches, 'launch_ms': run_ms / max(kernel_launches, 1),
            'algorithmic_flop_per_proposal': flops, 'peak_source': peak_src,
            'frac_of_fp32_fma_peak': achieved_tflops / fp32_peak,
            'note': 'algorithmic flops = dense nn.Linear count of one flow inverse per proposal, 4*B*H*(2d+L*H); ncu '
                    'summaries of this command: profiles/ (README.md lists them per round)',
        }
        cpu = cpu_baseline_quick(name, wl) if world == 1 and not args.no_cpu_baseline else None
        print(json.dumps({
            'metric': METRIC, 'value': value, 'unit': 'proposals/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms / args.steps,
            'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': name + ': ' + wl['desc'], 'chains_total': n_total, 'chains_per_gpu': n, 'x_dim': d,
                       'mcmc_steps': S, 'hidden_dim': HIDDEN, 'num_blocks': BLOCKS, 'num_layers': LAYERS,
                       'flow_weights': 'reference Trainer fit (tests/golden/bench_%s.npz)' % name,
                       'l2': 'flushed between timed steps',
                       'kernel': 'tcgen05' if used_tc else ('ffma' if out['impl'] == L.NNB_IMPL_FFMA else 'warp'),
                       'accept_rate': naccept / float(n * S), 'loglike_calls_per_proposal': ncall / float(n * S),
                       'collectives_per_step': {k: v / float(args.steps + args.warmup) for k, v in coll.items()}
                       if world > 1 else None,
                       'shard_check': {'hash': shard_hash, 'what': 'sha1 of the gathered end states (first x, last x, '
                                       'last logl) of one fixed-step-size refill of all %d chains; identical for every '
                                       '--gpus N' % n_total}},
            'e2e': {'value': e2e_value, 'unit': 'proposals/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'steps': e2e_steps, 'ms_per_step': e2e_ms,
                    'api': 'Sampler._mcmc_refill(pinned host float32 start points, pinned host loglikes) + Sampler._refill_to_host '
                           '(all_gather over ranks + pinned D2H of first x, last x, last logl)'
                    if wl['mode'] == 'hard' else 'MCMCSampler._mcmc_sample(thin=%d): host start points -> host trace' % args.thin,
                    'ms_per_step_parts': e2e_parts},
            'ns_loop': ns_loop,
            'gpu_launches': launches, 'step_ms': step_ms,
            'clocks': clk, 'roofline': roofline, 'cpu_baseline': cpu,
        }))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='c4', choices=sorted(WORKLOADS) + ['ns_c4'])
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'])
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--kernel', default='auto', choices=['auto', 'ffma', 'tcgen05', 'warp'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--e2e-steps', type=int, default=20, help='timed steps of the end-to-end arm (<= --steps)')
    ap.add_argument('--thin', type=int, default=10, help='c5 end-to-end arm: keep every thin-th state of the trace')
    ap.add_argument('--chains', type=int, default=0, help='development: override the chains of the workload')
    ap.add_argument('--mcmc-steps', type=int, default=0, help='development: override the MCMC steps per refill')
    ap.add_argument('--fixed-scale', action='store_true', help='development: dynamic_step_size=False')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the end states of the last timed step to DIR/<name>.npy (proposals/s workloads on the GPU)')
    args = ap.parse_args()
    if args.dump_outputs and (args.workload == 'ns_c4' or args.impl == 'reference'):
        ap.error('--dump-outputs is implemented for the proposals/s workloads (c2, c3, c4, c5) with --impl b200')
    if args.workload == 'ns_c4':
        import bench_ns
        return bench_ns.main(args)
    wl = dict(WORKLOADS[args.workload])
    if args.chains or args.mcmc_steps or args.fixed_scale:
        wl.update(chains=args.chains or wl['chains'], mcmc_steps=args.mcmc_steps or wl['mcmc_steps'],
                  dynamic=wl['dynamic'] and not args.fixed_scale)
        wl['desc'] += ' [development override: %d chains x %d steps, dynamic=%s]' % (wl['chains'], wl['mcmc_steps'],
                                                                                      wl['dynamic'])
    if args.impl == 'reference':
        run_reference(args, args.workload, wl)
    else:
        run_gpu(args, args.workload, wl)


if __name__ == '__main__':
    main()
