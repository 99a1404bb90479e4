"""bench.py --workload ns_c4: a fixed number of nested-sampling iterations of BASELINE.json configs[3] THROUGH
NestedSampler.run -- MCMC refills, flow retrains (nearest-neighbour jitter + fused fitting kernel), live-point replacement
and evidence bookkeeping -- i.e. the part of a run that the proposals/s microbenchmark does not see (SURVEY.md section
8(f) rows 1 and 2).  A "step" is one run of `--ns-iters` iterations (default 3 x nlive: at least three refills and six
retrains) from a fresh sampler.  Prints ONE JSON line: NS iterations/s, the split of the wall time, and a roofline entry
for train_epoch_kernel (algorithmic flops = 3 x the dense nn.Linear count of one forward pass per training sample
[forward + backward], 1 x per validation sample; FP32 FMA pipe).
"""
import json
import logging
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


def main(args):
    import torch
    import torch.distributed as dist
    from nnest_b200 import build as nb_build
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    nb_build.build()
    import bench
    from nnest_b200 import NestedSampler
    from nnest_b200.likelihoods import Rosenbrock
    from nnest_b200.bookkeeping import NSBook

    d, nlive = 30, args.chains or 65536
    chains = nlive // world if args.scaling == 'strong' else nlive
    ns_iters = int(os.environ.get('NNB_NS_ITERS', 3 * nlive))
    train_iters, batch_size = 50, 8192
    steps, warmup = args.steps, args.warmup
    parts = {}

    def timed(obj, name, key, sync=True):
        fn = getattr(obj, name)

        def wrap(*a, **k):
            if sync:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn(*a, **k)
            if sync:
                torch.cuda.synchronize()
            parts[key] = parts.get(key, 0.0) + time.perf_counter() - t0
            parts[key + '_calls'] = parts.get(key + '_calls', 0) + 1
            return r
        setattr(obj, name, wrap)

    epoch_ms, epoch_n, epoch_ev = [], [], []

    def one_run(seed):
        np.random.seed(seed)
        torch.manual_seed(seed)
        s = NestedSampler(d, Rosenbrock(d), transform=lambda x: 5 * x, flow='nvp', num_live_points=nlive,
                          batch_size=batch_size, log_dir=tempfile.mkdtemp(prefix='nnb_ns_'), log_level=logging.WARNING,
                          seed=seed)
        timed(s.trainer, 'train', 'flow_fit_s')
        timed(s.trainer, '_mean_two_nearest', 'jitter_nn_s')
        timed(s, '_mcmc_refill', 'mcmc_refill_s')
        timed(s, '_refill_to_host', 'gather_d2h_s')
        timed(s, '_save_samples', 'chain_file_s', sync=False)
        timed(s, '_write_checkpoint', 'checkpoint_s', sync=False)
        eng = s.engine
        orig_begin = eng.train_epoch_begin

        def train_epoch_begin(arch, params, m, v, step0, x_train, x_valid, *a, **k):
            # the fit queues epochs ahead of the host: the event pairs are read after the run
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = orig_begin(arch, params, m, v, step0, x_train, x_valid, *a, **k)
            e1.record()
            epoch_ev.append((e0, e1))
            epoch_n.append((0 if x_train is None else x_train.shape[0], 0 if x_valid is None else x_valid.shape[0]))
            return r
        eng.train_epoch_begin = train_epoch_begin
        orig_bulk = NSBook.bulk

        def bulk(self, *a, **k):
            t0 = time.perf_counter()
            r = orig_bulk(self, *a, **k)
            parts['consume_bookkeeping_s'] = parts.get('consume_bookkeeping_s', 0.0) + time.perf_counter() - t0
            return r
        NSBook.bulk = bulk
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s.run(strategy=['mcmc'], mcmc_num_chains=chains, train_iters=train_iters, max_iters=ns_iters,
                  log_interval=10 ** 9, chain_stats=False)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            epoch_ms.extend(e0.elapsed_time(e1) for e0, e1 in epoch_ev)
            del epoch_ev[:]
        finally:
            NSBook.bulk = orig_bulk
        return dt, s

    for w in range(warmup):
        one_run(100 + w)
    parts.clear()
    del epoch_ms[:], epoch_n[:]
    launches0 = None
    total, iters = 0.0, 0
    for k in range(steps):
        dt, s = one_run(k)
        total += dt
        iters += s.niter - 1
    t = torch.tensor([total], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total = t.item()
    if rank == 0:
        flops_fwd = bench.flow_flops_per_proposal(d)
        ms = float(np.mean(epoch_ms))
        ntr, nva = [float(np.mean(c)) for c in zip(*epoch_n)]
        achieved = (3 * ntr + nva) * flops_fwd / (ms * 1e-3) / 1e12
        fp32_peak = 148 * 128 * 2 * 1965.0e6 / 1e12
        split = {k: (v / steps if not k.endswith('_calls') else v / steps) for k, v in parts.items()}
        split['flow_fit_s'] = split.get('flow_fit_s', 0.0) - split.get('jitter_nn_s', 0.0)   # train() contains the jitter
        split['other_host_s'] = total / steps - sum(v for k, v in split.items() if k.endswith('_s'))
        print(json.dumps({
            'metric': 'nested-sampling iterations/sec through NestedSampler.run (C4: MCMC refills + flow retrains + '
                      'live-point replacement)', 'value': iters / total, 'unit': 'iterations/s', 'n_gpus': world,
            'steps': steps, 'warmup': warmup, 'ms_per_step': 1e3 * total / steps, 'higher_is_better': True,
            'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'ns_c4: Rosenbrock x_dim=30, %d live points, %d chains per rank, %d NS iterations '
                                   'per step, retrain every nlive/2 iterations (train_iters %d, batch %d)'
                                   % (nlive, chains, ns_iters, train_iters, batch_size)},
            'wall_split_s_per_step': split,
            'gpu_launches': int(s.engine.gpu_launches),
            'roofline': {'bound': 'fp32-fma', 'kernel': 'train_epoch_kernel<16,1>', 'achieved': achieved,
                         'peak': fp32_peak, 'unit': 'TFLOP/s', 'frac': achieved / fp32_peak, 'traffic': None,
                         'launch_ms': ms, 'launches_per_step': len(epoch_ms) / float(steps),
                         'peak_source': 'FP32 FMA pipe: 148 SMs x 128 lanes x 2 x 1965 MHz',
                         'algorithmic_flop_per_launch': (3 * ntr + nva) * flops_fwd},
        }))
    if world > 1:
        dist.destroy_process_group()
