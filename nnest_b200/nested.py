"""NestedSampler with the reference's interface (nnest/nested.py:24-510).

The MCMC refill (nested.py:398-427) runs in the fused CUDA kernels (Sampler._mcmc_refill); live-point
replacement (nested.py:429-439) uses the exact host routines exported by the C ABI (nnb_consume_scan for a single
iteration, nnb_ns_consume for a run of iterations: the live set sorted once + a heap of the replacements instead of an
O(nlive) argmin per iteration);
evidence bookkeeping (nested.py:272-293,458-464,487-500) is the reference's float64 arithmetic in the reference's
order (bookkeeping.NSBook: sequential NumPy accumulations between refills / retrains / checkpoints, the scalar code
around them), so that logZ, H and the posterior arrays are bit-identical given identical likelihood values
(tests/test_bookkeeping.py, tests/test_gpu_api.py).  The per-iteration O(it) rebuild of self.samples/weights/loglikes
(nested.py:469-471) is deferred to the points where they are read (checkpoints, end of run).

Multi-GPU: one process per GPU under torchrun; every rank runs its own shard of chains, the end states are
all-gathered over NCCL in rank order (the reference's gather + bcast + concatenate, nested.py:416-427) and
every rank replays the identical bookkeeping.
"""
from __future__ import division, print_function

import csv
import ctypes
import glob
import json
import logging
import os

import numpy as np
import torch

from . import _lib as L
from . import dist
from .bookkeeping import NSBook
from .priors import UniformPrior
from .sampler import Sampler
from .trainer import Trainer


class NestedSampler(Sampler):

    def __init__(self,
                 x_dim,
                 loglike,
                 transform=None,
                 append_run_num=True,
                 hidden_dim=16,
                 num_slow=0,
                 num_derived=0,
                 batch_size=100,
                 flow='spline',
                 num_blocks=3,
                 num_layers=1,
                 learning_rate=0.001,
                 log_dir='logs/test',
                 resume=True,
                 base_dist=None,
                 scale='',
                 use_gpu=True,
                 trainer=None,
                 oversample_rate=-1,
                 log_level=logging.INFO,
                 param_names=None,
                 num_live_points=1000,
                 seed=0):

        prior = UniformPrior(x_dim, -1, 1)      # nested.py:76 : the flow lives on the unit hyper-cube [-1, 1]^d

        super(NestedSampler, self).__init__(x_dim, loglike, transform=transform, append_run_num=append_run_num,
                                            hidden_dim=hidden_dim, num_slow=num_slow, num_derived=num_derived,
                                            batch_size=batch_size, flow=flow, num_blocks=num_blocks,
                                            num_layers=num_layers, learning_rate=learning_rate,
                                            log_dir=log_dir, resume=resume,
                                            use_gpu=use_gpu, base_dist=base_dist, scale=scale, trainer=trainer,
                                            prior=prior, transform_prior=False, log_level=log_level,
                                            param_names=param_names, oversample_rate=oversample_rate, seed=seed)

        self.num_live_points = num_live_points
        self.sampler = 'nested'

        if self.single_or_primary_process:
            self.logger.info('Num live points [%d]' % self.num_live_points)
            with open(os.path.join(self.logs['results'], 'results.csv'), 'w') as f:
                writer = csv.writer(f)
                writer.writerow(['step', 'acceptance', 'min_ess',
                                 'max_ess', 'jump_distance', 'scale', 'loglstar', 'logz', 'fraction_remain', 'ncall'])

    # ---- multi-GPU helpers -----------------------------------------------------------------------
    def _bcast_array(self, a):
        return dist.broadcast_array(a, self.device)

    # ---------------------------------------------------------------------------------------------
    def run(
            self,
            strategy=None,
            mcmc_steps=0,
            mcmc_num_chains=10,
            mcmc_dynamic_step_size=True,
            max_iters=1000000,
            update_interval=None,
            log_interval=None,
            dlogz=0.5,
            train_iters=500,
            volume_switch=-1.0,
            step_size=0.0,
            jitter=-1.0,
            rejection_cache_interval=10,
            rejection_enlargement_factor=1.1,
            rejection_trials=None,
            chain_stats=True,
            diagnostics=False):

        if strategy is None or len(strategy) == 0:
            strategy = ['rejection_prior', 'mcmc']
        for method in strategy:
            if method not in ('rejection_prior', 'rejection_flow', 'density_flow', 'mcmc'):
                raise ValueError("unknown sampling strategy %r" % method)
        expired_strategies = []
        current_method = ''

        if update_interval is None:
            update_interval = max(1, round(0.5 * self.num_live_points))
        else:
            update_interval = round(update_interval)
            if update_interval < 1:
                raise ValueError("update_interval must be >= 1")

        if log_interval is None:
            log_interval = max(1, round(0.2 * self.num_live_points))
        else:
            log_interval = round(log_interval)
            if log_interval < 1:
                raise ValueError("log_interval must be >= 1")

        if mcmc_steps <= 0:
            mcmc_steps = 5 * self.x_dim
        if step_size <= 0.0:
            step_size = 1 / self.x_dim ** 0.5

        primary = self.single_or_primary_process
        if primary:
            self.logger.info('MCMC steps [%d]' % mcmc_steps)
            self.logger.info('Initial scale [%5.4f]' % step_size)
            self.logger.info('Volume switch [%5.4f]' % volume_switch)

        nlive = self.num_live_points
        it = -1
        if self.resume and self.logs is not None and not self.logs['created']:
            for f in glob.glob(os.path.join(self.logs['checkpoint'], 'checkpoint_*.txt')):
                it = max(it, int(f.split('/checkpoint_')[1].split('.txt')[0]))

        bk = NSBook(nlive, self.num_derived)
        if it >= 0:
            if primary:
                self.logger.info('Using checkpoint [%d]' % it)
            with open(os.path.join(self.logs['checkpoint'], 'checkpoint_%s.txt' % it), 'r') as f:
                data = json.load(f)
            bk.logz, bk.h, bk.logvol, bk.it = data['logz'], data['h'], data['logvol'], it
            self.total_calls = int(data['ncall'] / self.mpi_size)
            bk.fraction_remain = data['fraction_remain']
            strategy = data['strategy']
            expired_strategies = data['expired_strategies']
            ckpt = self.logs['checkpoint']
            active_u = np.load(os.path.join(ckpt, 'active_u_%s.npy' % it))
            active_v = self.transform(active_u)
            active_logl = np.load(os.path.join(ckpt, 'active_logl_%s.npy' % it))
            active_derived = np.load(os.path.join(ckpt, 'active_derived_%s.npy' % it))
            if it > 0:     # checkpoint_0 holds empty arrays (the reference loads them as empty lists, nested.py:193-195)
                bk.saved_v = [np.load(os.path.join(ckpt, 'saved_v.npy')).reshape(it, self.x_dim)]
                bk.saved_logl = [np.load(os.path.join(ckpt, 'saved_logl.npy'))]
                bk.saved_logwt = [np.load(os.path.join(ckpt, 'saved_logwt.npy'))]
                if self.num_derived:
                    bk.saved_derived = [np.load(os.path.join(ckpt, 'saved_derived.npy')).reshape(it, self.num_derived)]
            assert it == bk.num_dead()
            total_calls = data['ncall']
        else:
            active_u = self.sample_prior(nlive) if primary else np.empty((nlive, self.x_dim), dtype=np.float64)
            active_u = self._bcast_array(active_u)
            active_v = self.transform(active_u)
            # float64 live points -> float64 likelihood (nested.py:228 with priors.py:46).  Multi-GPU: every rank evaluates
            # its contiguous share and the values are all-gathered in rank order (the reference scatters / gathers,
            # nested.py:212-226), so the call counter sums to nlive over the ranks.
            if self.use_mpi:
                lo, hi = dist.shard_bounds(nlive, self.mpi_rank, self.mpi_size)
                part, _ = self.loglike(active_u[lo:hi])
                active_logl = dist.allgather_ragged(np.asarray(part, dtype=np.float64), nlive, self.device)
                active_derived = self._derived_rows(active_u)      # every rank, all rows: no collective
                total_calls = dist.allreduce_sum_int(self.total_calls, self.device)
            else:
                active_logl, active_derived = self.loglike(active_u)
                total_calls = self.total_calls
            if primary:
                self.logger.info('Step [0] max logl [%5.4e] vol [1.0] ncalls [%d]' % (np.max(active_logl), total_calls))
                self._write_checkpoint(bk, active_u, active_v, active_logl, active_derived, total_calls, strategy,
                                       expired_strategies)
        active_u = np.ascontiguousarray(active_u, dtype=np.float64)
        active_v = np.ascontiguousarray(active_v, dtype=np.float64)
        active_logl = np.ascontiguousarray(active_logl, dtype=np.float64)
        active_derived = np.ascontiguousarray(active_derived, dtype=np.float64).reshape(nlive, self.num_derived)

        lib = L.load()
        # Device-resident live set (float64, like the host arrays): chain starts are gathered from it on the device, and the
        # replacements of a batch are applied to it by a scatter from the gathered end states -- only indices cross PCIe.
        # Built at the first MCMC refill (the rejection phase replaces live points on the host only).
        live_dev = None
        pend_slots, pend_chains = [], []

        def flush_live():
            """apply the pending (slot <- chain of the last gathered batch) replacements to the device live set"""
            if not pend_slots:
                return
            slots = np.concatenate(pend_slots)
            chains_ = np.concatenate(pend_chains)
            # last write to a slot wins: NumPy's indexed assignment keeps the last value of a repeated index
            last = np.full(nlive, -1, dtype=np.int64)
            last[slots] = np.arange(len(slots), dtype=np.int64)
            keep = last[last >= 0]
            sl = torch.from_numpy(np.ascontiguousarray(slots[keep])).to(self.device)
            ch = torch.from_numpy(np.ascontiguousarray(chains_[keep])).to(self.device)
            g = self._gathered_dev
            live_dev[0].index_copy_(0, sl, g['last'].index_select(0, ch).double())
            live_dev[1].index_copy_(0, sl, g['logl_last'].index_select(0, ch))
            del pend_slots[:], pend_chains[:]

        self.refill_log = []
        first_time = True
        get_samples = True
        nb = 0
        ncs = []
        mean_calls = 0
        accept_point = True
        scale = step_size
        batch = None
        samples = loglikes = None
        b_first = b_last = b_logl = b_derived = None
        s_derived = None
        max_logl = np.max(active_logl)

        def next_special(i):
            """first iteration index >= i that needs the single-iteration path (retrain, log line, checkpoint)"""
            up = lambda v, q: ((v + q - 1) // q) * q
            return min(up(i, update_interval), up(i, log_interval), up(i + 1, log_interval) - 1)

        while bk.fraction_remain > dlogz and bk.it <= max_iters:

            # ---- many plain iterations at once (bit-identical to running them one by one) ----------------------
            if current_method == 'mcmc' and accept_point and not get_samples and not first_time \
                    and b_first is not None:
                kmax = min(next_special(bk.it) - bk.it, 1 << 20)
                if kmax > 0:
                    nb, n_done, exhausted, finished = bk.bulk(active_u, active_v, active_logl, self.transform, b_first,
                                                              b_last, b_logl, nb, kmax, dlogz, max_iters,
                                                              active_derived=active_derived, b_derived=b_derived)
                    if n_done:
                        max_logl = np.max(active_logl)
                        pend_slots.append(bk.last_slots)
                        pend_chains.append(bk.last_chains)
                    if exhausted:
                        accept_point = False
                    get_samples = nb == b_first.shape[0]
                    if primary and self.trainer.writer is not None and n_done:
                        self.trainer.writer.add_scalar('logz', bk.logz, bk.it)
                    if finished:
                        break
                    continue

            it = bk.it
            worst = int(np.argmin(active_logl))               # nested.py:272 (first index on ties)
            loglstar = active_logl[worst]
            expected_vol = np.exp(-it / nlive)

            if accept_point:                                   # nested.py:280-293
                bk.evidence_update(active_v, active_logl, worst, active_derived)
                accept_point = False

            old_method = current_method
            for method in strategy:
                if method not in expired_strategies:
                    current_method = method
                    break
            if current_method != old_method:
                get_samples = True

            if not current_method == 'rejection_prior' and (first_time or it % update_interval == 0):   # nested.py:311
                kw = {}
                if live_dev is not None and isinstance(self.trainer, Trainer):
                    flush_live()                                # the device copy of the live set == active_u: no upload
                    kw['device_samples'] = live_dev[0]
                    if os.environ.get('NNB_CHECK_LIVE_DEV'):    # tests: the invariant this relies on
                        assert np.array_equal(live_dev[0].cpu().numpy(), active_u)
                        assert np.array_equal(live_dev[1].cpu().numpy(), active_logl)
                        self._live_dev_checks = getattr(self, '_live_dev_checks', 0) + 1
                self.trainer.train(active_u, max_iters=train_iters, jitter=jitter, **kw)     # nested.py:311-314
                first_time = False

            if current_method in ('rejection_prior', 'rejection_flow', 'density_flow'):

                if get_samples:                                 # nested.py:316-377
                    nb = 0
                    if current_method == 'rejection_prior':
                        samples, loglikes, s_derived, nc = self._rejection_prior_sample(loglstar,
                                                                                        num_trials=rejection_trials)
                        label = 'Rejection prior'
                    elif current_method == 'rejection_flow':
                        samples, loglikes, s_derived, nc = self._rejection_flow_sample(
                            active_u, loglstar, enlargement_factor=rejection_enlargement_factor,
                            cache=it % rejection_cache_interval == 0 or it % update_interval == 0)
                        label = 'Rejection flow'
                    else:
                        samples, loglikes, s_derived, nc = self._density_sample(loglstar)
                        label = 'Density flow'
                    ncs.append(nc)
                    mean_calls = np.mean(ncs[-20:]) if len(ncs) > 20 else 0
                    can_switch = 'mcmc' in strategy and 'mcmc' not in expired_strategies
                    expire = False
                    if current_method == 'rejection_prior':
                        expire = expected_vol < volume_switch >= 0 or \
                            (volume_switch < 0 and mean_calls > mcmc_steps and can_switch)
                    else:
                        expire = mean_calls > mcmc_steps and can_switch
                    if self.use_mpi:
                        # nested.py:295-298,366-377: every rank contributes its draw(s), all ranks consume the rank-ordered
                        # concatenation; a strategy expired on any rank is expired on all of them (every rank reaches
                        # this point in the same iteration, so the union is taken where the flag can change)
                        drawn_dtype = np.asarray(samples).dtype
                        samples = dist.allgather_rows(torch.from_numpy(np.ascontiguousarray(
                            samples, dtype=np.float64)).to(self.device)).cpu().numpy()
                        loglikes = dist.allgather_rows(torch.from_numpy(np.ascontiguousarray(
                            loglikes, dtype=np.float64)).to(self.device)).cpu().numpy()
                        # derived parameters of the gathered draws, on every rank, from the draws in the type they were
                        # evaluated in (float32 flow draws travel as exact float64)
                        s_derived = self._derived_rows(samples.astype(drawn_dtype))
                        expire = bool(dist.allreduce_sum_int(int(expire), self.device))
                        total_calls = dist.allreduce_sum_int(self.total_calls, self.device)
                    if expire:
                        self.logger.info('%s no longer efficient, switching sampling method' % label)
                        expired_strategies.append(current_method)
                        ncs = []

                for ib in range(nb, samples.shape[0]):          # nested.py:379-389
                    nb += 1
                    get_samples = nb == samples.shape[0]
                    if loglikes[ib] > loglstar:
                        active_u[worst] = samples[nb - 1, :]
                        active_v[worst] = self.transform(active_u[worst])
                        active_logl[worst] = loglikes[nb - 1]
                        active_derived[worst] = s_derived[nb - 1]
                        live_dev = None                  # replaced on the host only: the device copy is rebuilt when needed
                        accept_point = True
                        break

                if not self.use_mpi:
                    total_calls = self.total_calls
                if accept_point and it > 0 and (it + 1) % log_interval == 0 and primary:
                    self.logger.info(
                        'Step [%d] loglstar [%5.4e] max logl [%5.4e] logz [%5.4e] vol [%6.5e] ncalls [%d] mean '
                        'calls [%5.4f]' % (it + 1, loglstar, np.max(active_logl), bk.logz, expected_vol, total_calls,
                                           mean_calls))

            elif current_method == 'mcmc':

                if get_samples:                                 # nested.py:402-427
                    nb = 0
                    idx = np.random.randint(low=0, high=nlive, size=mcmc_num_chains)
                    if live_dev is None:
                        live_dev = (torch.from_numpy(active_u).to(self.device), torch.from_numpy(active_logl).to(self.device))
                        del pend_slots[:], pend_chains[:]
                    else:
                        flush_live()
                    batch = self._mcmc_refill(mcmc_steps, None, None, loglstar, step_size, mcmc_dynamic_step_size,
                                              keep_trace=chain_stats, live=(live_dev[0], live_dev[1], idx))
                    b_first, b_last, b_logl = self._refill_to_host(batch)     # all ranks' chains, rank order
                    b_derived = self.refill_derived
                    total_calls = dist.allreduce_sum_int(self.total_calls, self.device) if self.use_mpi \
                        else self.total_calls
                    scale = batch['scale']
                    if diagnostics:
                        # run diagnostics (not in the reference, only on request): one record per refill -- iteration,
                        # constraint, this rank's acceptance, fraction of chains that moved in every coordinate and beat
                        # the constraint, final scale
                        moved = np.all(b_first != b_last, axis=1) & (b_logl > loglstar)
                        self.refill_log.append((it, float(loglstar), float(batch.get('acceptance', np.nan)),
                                                float(moved.mean()), float(scale)))

                c_nb = ctypes.c_int64(nb)                       # nested.py:429-439
                fp = ctypes.POINTER(ctypes.c_float)
                ib = lib.nnb_consume_scan(b_first.ctypes.data_as(fp), b_last.ctypes.data_as(fp),
                                          b_logl.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), b_first.shape[0],
                                          self.x_dim, float(loglstar), ctypes.byref(c_nb))
                nb = c_nb.value
                get_samples = nb == b_first.shape[0]
                if ib >= 0:
                    active_u[worst] = b_last[ib, :]
                    active_v[worst] = self.transform(active_u[worst])
                    active_logl[worst] = b_logl[ib]
                    if self.num_derived:
                        active_derived[worst] = b_derived[ib]
                    accept_point = True
                    pend_slots.append(np.array([worst], dtype=np.int64))
                    pend_chains.append(np.array([ib], dtype=np.int64))

                if accept_point and it > 0 and it % log_interval == 0 and primary:
                    if chain_stats and batch.get('trace_x') is not None:
                        acceptance, ess, jump_distance = self._chain_stats(
                            None, trace=batch['trace_x'], mean=np.mean(active_u, axis=0), std=np.std(active_u, axis=0))
                    else:
                        acceptance, ess, jump_distance = np.nan, np.array([np.nan]), np.nan
                    self.logger.info(
                        'Step [%d] loglstar [%5.4e] maxlogl [%5.4e] logz [%5.4e] vol [%6.5e] ncalls [%d] '
                        'scale [%5.4f]' % (it, loglstar, np.max(active_logl), bk.logz, expected_vol, total_calls, scale))
                    with open(os.path.join(self.logs['results'], 'results.csv'), 'a') as f:
                        writer = csv.writer(f)
                        writer.writerow([it, acceptance, np.min(ess), np.max(ess),
                                         jump_distance, scale, loglstar, bk.logz, bk.fraction_remain, total_calls])

            if accept_point:                                    # nested.py:458-485
                # np.max(active_logl) without the O(nlive) pass: the maximum only changes when the new point
                # beats it (the replaced point is the minimum; if min == max every point was equal)
                new_logl = active_logl[worst]
                if loglstar == max_logl:
                    max_logl = np.max(active_logl)
                elif new_logl > max_logl:
                    max_logl = new_logl
                bk.shrink(max_logl)

                if primary and self.trainer.writer is not None:
                    self.trainer.writer.add_scalar('logz', bk.logz, bk.it)

                if bk.it > 0 and bk.it % log_interval == 0 and primary:
                    self._write_checkpoint(bk, active_u, active_v, active_logl, active_derived, total_calls, strategy,
                                           expired_strategies)
                    self.samples, self.loglikes, logwt = bk.dead_points()
                    self.weights = np.exp(logwt - bk.logz)
                    self._save_samples(self.samples, self.loglikes, weights=self.weights,
                                       derived_samples=bk.dead_derived() if self.num_derived else None)

        saved_logl = np.concatenate(bk.saved_logl) if bk.saved_logl else np.empty((0,))
        saved_logwt = np.concatenate(bk.saved_logwt) if bk.saved_logwt else np.empty((0,))
        logz, h, it = bk.logz, bk.h, bk.it
        # nested.py:487-500: the remaining live points, each with the final volume / nlive -- the reference's scalar loop
        # as sequential NumPy accumulations + the exact host recurrence for H (bit-identical, see bookkeeping.NSBook.bulk)
        logvol = -len(saved_logl) / nlive - np.log(nlive)
        fin_logwt = logvol + active_logl
        lz = np.logaddexp.accumulate(np.concatenate(([logz], fin_logwt)))
        lz_prev, lz_new = np.ascontiguousarray(lz[:-1]), np.ascontiguousarray(lz[1:])
        a_term = np.ascontiguousarray(np.exp(fin_logwt - lz_new) * active_logl)
        b_term = np.ascontiguousarray(np.exp(lz_prev - lz_new))
        dp = lambda arr: arr.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        h = lib.nnb_ns_information(float(h), dp(a_term), dp(b_term), dp(lz_prev), dp(lz_new), nlive)
        logz = lz_new[-1]

        self.logz = logz
        self.h = h
        self.logzerr = np.sqrt(h / nlive)
        self.niter = it + 1
        self.samples = bk.samples_with(active_v)        # dead points followed by the remaining live points
        self.weights = np.exp(np.concatenate((saved_logwt, fin_logwt)) - logz)
        self.loglikes = np.concatenate((saved_logl, active_logl))
        self.active_u, self.active_logl, self.active_derived = active_u, active_logl, active_derived
        # derived parameters of self.samples, row for row (None without them): the chain files carry them for the dead
        # points too, an extension -- the reference saves none for its dead points
        self.derived_samples = np.concatenate((bk.dead_derived(), active_derived)) if self.num_derived else None

        if primary:
            with open(os.path.join(self.logs['results'], 'final.csv'), 'w') as f:
                writer = csv.writer(f)
                writer.writerow(['niter', 'ncall', 'logz', 'logzerr', 'h'])
                writer.writerow([it + 1, total_calls, logz, np.sqrt(h / nlive), h])
            self._save_samples(self.samples, self.loglikes, weights=self.weights, derived_samples=self.derived_samples)
            self.logger.info("niter: {:d}\n ncall: {:d}\n nsamples: {:d}\n logz: {:6.3f} +/- {:6.3f}\n h: {:6.3f}"
                             .format(it + 1, int(total_calls), len(self.loglikes), logz, np.sqrt(h / nlive), h))
        # run diagnostics (NOT part of the reference's layout: only on request): one row per MCMC refill / flow fit
        if primary and diagnostics:
            with open(os.path.join(self.logs['results'], 'refill_log.csv'), 'w') as f:
                writer = csv.writer(f)
                writer.writerow(['iteration', 'loglstar', 'acceptance', 'usable_fraction', 'scale'])
                writer.writerows(self.refill_log)
            with open(os.path.join(self.logs['results'], 'fit_log.csv'), 'w') as f:
                writer = csv.writer(f)
                writer.writerow(['total_epochs', 'samples', 'jitter', 'best_epoch', 'best_validation_loss'])
                writer.writerows(getattr(self.trainer, 'fit_log', []))

    def _write_checkpoint(self, bk, active_u, active_v, active_logl, active_derived, total_calls, strategy,
                          expired_strategies):
        """Checkpoint files of the reference (nested.py:249-260,473-484)."""
        ckpt = self.logs['checkpoint']
        it = bk.it
        saved_v, saved_logl, saved_logwt = bk.dead_points()
        np.save(os.path.join(ckpt, 'active_u_%s.npy' % it), active_u)
        np.save(os.path.join(ckpt, 'active_v_%s.npy' % it), active_v)
        np.save(os.path.join(ckpt, 'active_logl_%s.npy' % it), active_logl)
        np.save(os.path.join(ckpt, 'active_derived_%s.npy' % it), active_derived)
        np.save(os.path.join(ckpt, 'saved_v.npy'), saved_v if len(saved_logl) else [])
        np.save(os.path.join(ckpt, 'saved_logl.npy'), saved_logl)
        np.save(os.path.join(ckpt, 'saved_logwt.npy'), saved_logwt)
        if self.num_derived:     # derived parameters of the dead points (not in the reference, which saves none)
            np.save(os.path.join(ckpt, 'saved_derived.npy'), bk.dead_derived())
        with open(os.path.join(ckpt, 'checkpoint_%s.txt' % it), 'w') as f:
            json.dump({'logz': float(bk.logz), 'h': float(bk.h), 'logvol': float(bk.logvol), 'ncall': int(total_calls),
                       'fraction_remain': float(bk.fraction_remain), 'strategy': strategy,
                       'expired_strategies': expired_strategies}, f)
