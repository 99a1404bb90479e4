"""Sampler base class with the reference's interface (nnest/sampler.py:29-527) whose MCMC loop runs in the
fused CUDA chain-step kernels.

What is kept from the reference's contract (SURVEY.md section 8b):
  * constructor kwargs and their defaults; `loglike`, `transform`, `prior` wrappers with the reference's
    counting semantics (`total_calls`, `total_accepted`, `total_rejected`, `total_fast_calls`);
  * `_mcmc_sample(...)` signature and 6-tuple return (arrays shaped (chain, iteration, dim));
  * run-directory layout, `info/params.txt`, chain files written by `_save_samples` ("%.5E").
What differs, by design (north_star: no CPU fallback):
  * `loglike` must be one of nnest_b200.likelihoods (the batched CUDA likelihood library) and `transform`
    must be a per-dimension affine map (probed numerically: the maps of examples/nested/run.py:25-44 and
    nnest/mcmc.py:111 all are) or a CudaTransform, a prior transform written in CUDA C++ (Gaussian, log-uniform,
    correlated priors ...); anything else raises NotImplementedError;
  * random numbers come from a per-chain Philox stream (seed = `seed` kwarg), not torch's global generator.
"""
from __future__ import division, print_function

import json
import logging
import os

import numpy as np
import torch

from . import _lib as L
from . import dist
from .likelihoods import CudaLikelihood, CudaTransform, Likelihood
from .priors import UniformPrior
from .trainer import Trainer
from .utils.evaluation import acceptance_rate, effective_sample_size, mean_jump_distance
from .utils.logger import create_logger, get_or_create_run_dir


def probe_affine_transform(transform, d):
    """Recover (scale, shift, promotes_to_f64) of a per-dimension affine transform by evaluating it, and
    verify it on random points.  Raises NotImplementedError for anything that is not diagonal-affine."""
    if transform is None:
        return None, None, False
    zero = np.zeros((1, d), dtype=np.float32)
    out0 = np.asarray(transform(zero))
    promotes = out0.dtype == np.float64
    z64 = np.zeros((1, d))
    if out0.shape != (1, d) or np.asarray(transform(z64)).shape != (1, d):
        raise NotImplementedError('transform must map (n, x_dim) arrays to (n, x_dim) arrays (per-dimension affine map)')
    shift = np.asarray(transform(z64), dtype=np.float64).reshape(d)
    scale = np.asarray(transform(np.ones((1, d))), dtype=np.float64).reshape(d) - shift
    rng = np.random.RandomState(12345)
    pts = rng.uniform(-1, 1, size=(16, d))
    want = np.asarray(transform(pts), dtype=np.float64)
    got = pts * scale + shift
    tol = 1e-9 * (1.0 + np.abs(want).max())
    if want.shape != pts.shape or np.abs(want - got).max() > tol:
        raise NotImplementedError('transform is not a per-dimension affine map; arbitrary Python transforms '
                                  'cannot run inside the CUDA step kernel (no CPU fallback): write it in CUDA C++ as a '
                                  'nnest_b200.likelihoods.CudaTransform')
    return scale, shift, promotes


class Sampler(object):

    def __init__(self,
                 x_dim,
                 loglike,
                 transform=None,
                 prior=None,
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
                 use_gpu=True,
                 base_dist=None,
                 scale='',
                 trainer=None,
                 transform_prior=True,
                 oversample_rate=-1,
                 log_level=logging.INFO,
                 param_names=None,
                 seed=0,
                 ):
        self.x_dim = x_dim
        self.num_derived = num_derived
        self.num_params = x_dim + num_derived
        assert x_dim > num_slow
        if num_slow != 0:
            raise NotImplementedError('fast/slow hierarchies (num_slow > 0) are not on the accelerated path')
        # derived parameters come from the likelihood's own CUDA C++ (CudaLikelihood(num_derived=...)); checked before
        # any device work, so a wrong combination fails fast
        if num_derived != 0 and not isinstance(loglike, CudaLikelihood):
            raise NotImplementedError('derived parameters (num_derived > 0) need a CudaLikelihood whose source defines '
                                      'nnb_user_derived; the built-in likelihoods have none')
        if isinstance(loglike, Likelihood) and loglike.num_derived != num_derived:
            raise ValueError('num_derived=%d does not match the likelihood, which has %d derived parameters'
                             % (num_derived, loglike.num_derived))
        self.num_slow = num_slow
        self.num_fast = x_dim - num_slow
        self.param_names = param_names
        if self.param_names is not None:
            assert len(param_names) == self.num_params
        self.oversample_rate = oversample_rate if oversample_rate > 0 else self.num_fast / self.x_dim

        if not isinstance(loglike, Likelihood):
            raise NotImplementedError(
                'loglike must be an instance of nnest_b200.likelihoods.* (Rosenbrock, Himmelblau, Gaussian, Eggbox, '
                'GaussianMix, GaussianShell, or CudaLikelihood for your own likelihood written in CUDA C++): arbitrary '
                'Python callables cannot run in the CUDA kernels and there is no CPU fallback')
        self._like = loglike
        self._user_transform = transform
        self._prior_obj = prior
        self._transform_prior = transform_prior
        if prior is not None and not isinstance(prior, UniformPrior):
            raise NotImplementedError('only UniformPrior (box) priors are implemented on the device')

        sample_prior = getattr(prior, 'sample', None)
        self.sample_prior = sample_prior if callable(sample_prior) else None

        # distributed context: one process per GPU (torch.distributed), replaces the reference's mpi4py probe
        dist.ensure_initialized()
        self.mpi_rank, self.mpi_size = dist.rank_world()
        self.use_mpi = self.mpi_size > 1
        self.single_or_primary_process = self.mpi_rank == 0

        args = locals()
        args.update(vars(self))

        if self.single_or_primary_process or os.path.isdir(os.path.join(log_dir, 'info')):
            self.logs = get_or_create_run_dir(log_dir, append_run_num=append_run_num)
            self.log_dir = self.logs['run_dir']
        else:
            self.logs = None
            self.log_dir = None
        if self.single_or_primary_process:
            self._save_params(args)

        self.resume = resume
        self.logger = create_logger(__name__, level=log_level)

        if trainer is None:
            self.trainer = Trainer(
                x_dim, hidden_dim=hidden_dim, num_slow=num_slow, batch_size=batch_size, flow=flow,
                num_blocks=num_blocks, num_layers=num_layers, learning_rate=learning_rate, log_dir=self.log_dir,
                log=self.single_or_primary_process, use_gpu=use_gpu, base_dist=base_dist, scale=scale,
                log_level=log_level)
        else:
            self.trainer = trainer
        # b1 (SURVEY 8b): an injected trainer only has to honour the reference's contract (netG + forward / inverse / train,
        # nnest/sampler.py:196-212).  A nnest_b200.Trainer brings its own Engine; for any other object (e.g. the
        # reference's own Trainer) the kernels get their own Engine and the weights of trainer.netG.state_dict() are
        # re-exported to it before every batch of chains (_sync_foreign_trainer).
        self.engine = getattr(self.trainer, 'engine', None)
        self._foreign_trainer = self.engine is None
        if self._foreign_trainer:
            from .engine import Engine
            self.engine = Engine()
            self._sync_foreign_trainer()
        self.device = self.engine.device

        if self.single_or_primary_process:
            self.logger.info('Num base params [%d]' % (self.x_dim))
            self.logger.info('Num derived params [%d]' % (self.num_derived))
            self.logger.info('Total params [%d]' % (self.num_params))

        self.total_accepted = 0
        self.total_rejected = 0
        self.total_calls = 0
        self.total_fast_calls = 0
        self.seed = int(seed)
        self._step_counter = 0        # Philox step offset: every MCMC step of the run uses fresh counters
        self._start_counter = 0
        self.transform = transform    # property: (re)installs the device target

    # ---- target plumbing ------------------------------------------------------------------------
    @property
    def transform(self):
        return self._transform_fn

    @transform.setter
    def transform(self, fn):
        """Assigning `sampler.transform = ...` (as MCMCSampler.run does, nnest/mcmc.py:111) re-probes the map and
        re-installs likelihood + transform + prior on the device.  A CudaTransform is installed as it is (not probed);
        `sampler.transform(u)` then evaluates it through the sampler's own engine, so the values are those the
        likelihood saw."""
        self._user_transform = fn
        self._cuda_transform = fn if isinstance(fn, CudaTransform) else None
        if self._cuda_transform is not None:
            if fn.x_dim != self.x_dim:
                raise ValueError('the CudaTransform has x_dim %d, the sampler %d' % (fn.x_dim, self.x_dim))
            self._t_scale, self._t_shift, self._t_f64 = None, None, fn.float64

            def cuda_transform(x):
                if isinstance(x, list):
                    x = np.array(x)
                if len(x.shape) == 1:
                    assert x.shape[0] == self.x_dim
                    x = np.expand_dims(x, 0)
                return fn.apply(self.engine, x)
            self._transform_fn = cuda_transform
            self._install_target()
            return
        scale, shift, promotes = probe_affine_transform(fn, self.x_dim)
        self._t_scale, self._t_shift, self._t_f64 = scale, shift, promotes

        if fn is None:
            self._transform_fn = lambda x: x
        else:
            def safe_transform(x):
                if isinstance(x, list):
                    x = np.array(x)
                if len(x.shape) == 1:
                    assert x.shape[0] == self.x_dim
                    x = np.expand_dims(x, 0)
                return fn(x)
            self._transform_fn = safe_transform
        self._install_target()

    def _affine(self):
        """(scale, shift) of the current transform as float64 vectors (identity when there is none)."""
        d = self.x_dim
        sc = np.ones(d) if self._t_scale is None else np.broadcast_to(np.asarray(self._t_scale, dtype=np.float64), (d,))
        sh = np.zeros(d) if self._t_shift is None else np.broadcast_to(np.asarray(self._t_shift, dtype=np.float64), (d,))
        return sc, sh

    def _install_target(self):
        prior = self._prior_obj
        if prior is None:
            kind, lo, hi = L.NNB_PRIOR_NONE, None, None
        else:
            kind = L.NNB_PRIOR_BOX_V if (self._transform_prior and self._user_transform is not None) \
                else L.NNB_PRIOR_BOX_U
            lo, hi = prior.minimum.astype(np.float64), prior.maximum.astype(np.float64)
        if self._cuda_transform is not None:
            self._cuda_transform.install(self.engine, self.x_dim, self._like.like_id, self._like.device_params(),
                                         prior_kind=kind, prior_lo=lo, prior_hi=hi,
                                         user_source=self._like.device_source(), num_derived=self.num_derived,
                                         user_data=self._like.device_data())
            return
        self.engine.set_target(self.x_dim, self._like.like_id, self._like.device_params(), t_scale=self._t_scale,
                               t_shift=self._t_shift, compute_f64=self._t_f64, prior_kind=kind, prior_lo=lo,
                               prior_hi=hi, user_source=self._like.device_source(), num_derived=self.num_derived,
                               user_data=self._like.device_data())

    def _to_device_rows(self, x):
        if isinstance(x, list):
            x = np.array(x)
        x = np.asarray(x)
        if x.ndim == 1:
            assert x.shape[0] == self.x_dim
            x = x[None, :]
        if x.dtype not in (np.float32, np.float64):
            x = x.astype(np.float64)
        return x, torch.from_numpy(np.ascontiguousarray(x)).to(self.device)

    def loglike(self, x):
        """safe_loglike (nnest/sampler.py:110-133): loglike(transform(x)) for a batch of points in the flow's
        coordinates, non-finite -> -1e100, call counter updated.  Returns (logl, derived (n, num_derived)); derived values
        are not counted as calls."""
        x, xd = self._to_device_rows(x)
        logl = self.engine.loglike(xd).cpu().numpy()
        self.total_calls += x.shape[0]
        if self._like.follows_input_dtype and x.dtype == np.float32 and not self._t_f64:
            logl = logl.astype(np.float32)
        return logl, self._derived_rows(xd)

    def _derived_rows(self, x):
        """Derived parameters (n, num_derived) float64 of rows x (host array or cuda tensor, float32 or float64), evaluated
        in the arithmetic the likelihood uses for rows of that type (nnb_derived); (n, 0) without derived parameters."""
        n = x.shape[0] if x.ndim > 1 else 1
        if not self.num_derived:
            return np.empty((n, 0))
        if not isinstance(x, torch.Tensor):
            _, x = self._to_device_rows(x)
        return self.engine.derived(x).cpu().numpy()

    def prior(self, x):
        """safe_prior (nnest/sampler.py:143-163): 0 inside the box, -inf outside."""
        x, xd = self._to_device_rows(x)
        if self._prior_obj is None:
            return np.array([0 for _ in x])
        _, logp = self.engine.loglike(xd, want_prior=True)
        return logp.cpu().numpy()

    def _save_params(self, my_dict):
        my_dict = {k: str(v) for k, v in my_dict.items()}
        with open(os.path.join(self.logs['info'], 'params.txt'), 'w') as f:
            json.dump(my_dict, f, indent=4)

    def _sync_foreign_trainer(self):
        """Weights of an injected trainer that is not a nnest_b200.Trainer: netG.state_dict() in the reference's key
        layout (nnest/networks.py:262-282,328-347) -> nnb_set_flow.  Cheap (<= 47 KB) and done before every batch
        because such a trainer's train() cannot tell the kernels that the weights changed."""
        self.engine.set_flow_from_state_dict(self.trainer.netG.state_dict(), scale=None)

    # ---- the hot path -----------------------------------------------------------------------------
    def _start_chains(self, num_chains, init_samples, init_loglikes, max_start_tries, live=None):
        """Chain start (nnest/sampler.py:262-284) on the device.  Returns (ChainState, ncall).
        live=(live_u_dev (nlive,d) f64, live_logl_dev (nlive,) f64, idx (n,) int64 host): the start points are gathered from
        the device-resident live set (only the indices cross PCIe); values equal float32(init_samples) bit for bit."""
        offset = self.mpi_rank * num_chains
        if live is not None:
            live_u, live_logl, idx = live
            hi = self._pinned('init_idx', (len(idx),), torch.int64)
            hi.numpy()[...] = idx
            di = hi.to(self.device, non_blocking=True)
            u = live_u.index_select(0, di).float()              # float64 -> float32 (trainer.py:249)
            logl = live_logl.index_select(0, di)
            st, nbad, ncall = self.engine.mcmc_init(u.shape[0], init_u=u.t().contiguous(), init_logl=logl,
                                                    seed=self.seed, chain_offset=offset)
            return st, ncall
        if init_samples is not None:
            def staged(name, arr, dtype, shape):
                # page-locked torch tensors of the right dtype go to the device as they are; anything else (NumPy arrays,
                # float64) is converted into a reusable pinned staging buffer first (trainer.py:249: float32 start points)
                if isinstance(arr, torch.Tensor) and arr.dtype == dtype and arr.is_pinned() and arr.is_contiguous():
                    return arr.to(self.device, non_blocking=True)
                h = self._pinned(name, shape, dtype)
                h.numpy()[...] = arr.numpy() if isinstance(arr, torch.Tensor) else np.asarray(arr)
                return h.to(self.device, non_blocking=True)
            shape = tuple(init_samples.shape)
            u = staged('init_u', init_samples, torch.float32, shape)
            logl = None
            if init_loglikes is not None:
                logl = staged('init_logl', init_loglikes, torch.float64, (shape[0],))
            st, nbad, ncall = self.engine.mcmc_init(u.shape[0], init_u=u.t().contiguous(), init_logl=logl,
                                                    seed=self.seed, chain_offset=offset)
            return st, ncall
        ncall = 0
        for i in range(max_start_tries):
            self._start_counter += 1
            st, nbad, nc = self.engine.mcmc_init(num_chains, seed=self.seed, chain_offset=offset,
                                                 start_try=self._start_counter)
            ncall += nc
            if nbad == 0:
                return st, ncall
        raise Exception('Could not find starting value')

    def _mcmc_device(self, mcmc_steps, step_size, dynamic_step_size, num_chains, init_samples, init_loglikes,
                     loglstar, max_start_tries, trace, live=None):
        """Runs the fused kernels; returns (state, result dict, ncall)."""
        if step_size <= 0.0:
            step_size = 2 / self.x_dim ** 0.5
        if self._foreign_trainer:
            self._sync_foreign_trainer()
        st, ncall = self._start_chains(num_chains, init_samples, init_loglikes, max_start_tries, live=live)
        self.total_calls += ncall
        mode = L.NNB_MODE_MH if loglstar is None else L.NNB_MODE_HARD
        first_x = st.x.clone()
        out = self.engine.mcmc_run(st, mcmc_steps, mode=mode, loglstar=loglstar, step_size=step_size,
                                   dynamic_step_size=dynamic_step_size, seed=self.seed,
                                   chain_offset=self.mpi_rank * st.n, step_offset=self._step_counter, trace=trace)
        self._step_counter += mcmc_steps
        n = st.n
        self.total_calls += out['ncall']
        self.total_accepted += out['naccept']
        self.total_rejected += n * mcmc_steps - out['naccept']
        out['first_x'] = first_x
        return st, out, ncall + out['ncall']

    def _mcmc_sample(
            self,
            mcmc_steps,
            step_size=0.0,
            dynamic_step_size=False,
            num_chains=1,
            init_samples=None,
            init_loglikes=None,
            init_derived=None,
            loglstar=None,
            show_progress=False,
            max_start_tries=100,
            output_interval=None,
            stats_interval=None,
            plot_trace=True,
            prior_volume_steps=1,
            thin=1,
            sample_affine=None):
        """Same contract as the reference (nnest/sampler.py:229-463): returns
        (samples (N,S+1,d) f32, latent_samples (N,S+1,d) f32, derived (N,S+1,0), loglikes (N,S+1) f64, scale, ncall).
        The arrays are host views of the chain-minor device trace (no extra transposition pass).
        Extensions (both default to the reference's behaviour): thin=k returns every k-th state of the trace (rows 0, k,
        2k, ...: arrays shaped (N, S//k+1, .)); sample_affine=(scale, shift) returns samples * scale + shift in float64,
        evaluated on the device (what MCMCSampler.run applies to the whole trace on the host, mcmc.py:117).
        With derived parameters `derived` is (N, S//k+1, num_derived) float64: row t is the derived values of the state
        x_t, evaluated on the device for the returned rows only.  Given init_samples and init_derived (N, num_derived),
        row 0 and every later row whose state is still bit-equal to row 0 hold init_derived, as the reference keeps the
        start's values until the chain first moves."""
        if prior_volume_steps != 1:
            raise NotImplementedError('prior_volume_steps != 1')
        st, out, ncall = self._mcmc_device(mcmc_steps, step_size, dynamic_step_size, num_chains, init_samples,
                                           init_loglikes, loglstar, max_start_tries, trace=True)
        rows = list(range(0, mcmc_steps + 1, max(1, int(thin))))
        samples = self._trace_to_host(out['trace_x'], rows, sample_affine).transpose(2, 0, 1)   # (T,d,N) -> (N,T,d) view
        latent_samples = self._trace_to_host(out['trace_z'], rows, None).transpose(2, 0, 1)
        loglikes = self._trace_to_host(out['trace_logl'], rows, None).transpose(1, 0)
        init_der = None
        if self.num_derived and init_samples is not None and init_derived is not None:
            init_der = torch.from_numpy(np.ascontiguousarray(
                np.asarray(init_derived, dtype=np.float64).reshape(st.n, self.num_derived).T)).to(self.device)
        if self.num_derived:
            derived_samples = self._trace_to_host(out['trace_x'], rows, None, derived_init=(init_der,)).transpose(2, 0, 1)
        else:
            derived_samples = np.empty((st.n, len(rows), 0))
        self._device_trace = out['trace_x']          # (S+1, d, N) on the device, for the chain statistics
        ts, tb = self._affine()
        for it in range(1, mcmc_steps + 1):
            if output_interval is not None and it % output_interval == 0:
                full = out['trace_x'][:it + 1].cpu().numpy().transpose(2, 0, 1)
                der = None
                if self.num_derived:
                    der = self.engine.derived_trace(out['trace_x'], 0, 1, it + 1, init=init_der).cpu().numpy()
                    der = der.transpose(2, 0, 1)
                self._save_samples(self.transform(full.reshape(-1, self.x_dim)).reshape(st.n, it + 1, self.x_dim),
                                   out['trace_logl'][:it + 1].cpu().numpy().transpose(1, 0), derived_samples=der)
            if stats_interval is not None and it % stats_interval == 0:
                if self._cuda_transform is not None:
                    # statistics of the transformed samples (the reference's): the transform on the device, the
                    # statistics on the host (utils/evaluation.py) -- a diagnostic, not the hot path
                    v = self.engine.transform_trace(self._device_trace, 0, 1, it + 1).cpu().numpy()
                    self._chain_stats(v.transpose(2, 0, 1), step=it)
                else:
                    self._chain_stats(None, step=it, trace=self._device_trace, t_scale=ts, t_shift=tb)
        return samples, latent_samples, derived_samples, loglikes, out['scale'], ncall

    _STAGE_BYTES = 128 << 20

    def _trace_to_host(self, trace, rows, affine, derived_init=None):
        """Rows `rows` of a device trace (T, d, N) / (T, N) -> pageable host array (len(rows), ...), through two pinned
        staging buffers: the device->host copy of chunk k+1 runs while chunk k is moved into the result by a few host
        threads (a single pageable .cpu() of a multi-GB trace is bound by first-touch page faults on one core).
        affine=(scale, shift): float64 rows * scale[:, None] + shift[:, None], computed on the device.
        derived_init=(init,): the derived parameters (len(rows), num_derived, N) float64 of the rows of the trace x
        (T, d, N) instead, evaluated chunk by chunk (nnb_derived_trace; init: Engine.derived_trace), so that the full
        derived trace never sits on the device."""
        from concurrent.futures import ThreadPoolExecutor
        inner = tuple(trace.shape[1:])
        if derived_init is not None:
            inner = (self.num_derived, trace.shape[2])
        dtype = torch.float64 if affine is not None or derived_init is not None else trace.dtype
        out = np.empty((len(rows),) + inner, dtype=np.float64 if dtype == torch.float64 else np.float32)
        if not rows:
            return out
        row_bytes = int(np.prod(inner)) * out.itemsize
        per = max(1, min(len(rows), self._STAGE_BYTES // max(1, row_bytes)))
        stage = [self._pinned('stage%d' % i, (per,) + inner, dtype) for i in range(2)]
        events = [torch.cuda.Event(), torch.cuda.Event()]
        if affine is not None:
            sc = torch.as_tensor(np.broadcast_to(affine[0], (inner[0],)).copy(), dtype=torch.float64, device=self.device)
            sh = torch.as_tensor(np.broadcast_to(affine[1], (inner[0],)).copy(), dtype=torch.float64, device=self.device)
        step = rows[1] - rows[0] if len(rows) > 1 else 1
        chunks = [(i, min(i + per, len(rows))) for i in range(0, len(rows), per)]

        def launch(ci):
            a, b = chunks[ci]
            if derived_init is not None:
                src = self.engine.derived_trace(trace, rows[a], step, b - a, init=derived_init[0])
            else:
                src = trace[rows[a]:rows[b - 1] + 1:step]
            if affine is not None:
                src = src.double() * sc[:, None] + sh[:, None]
            stage[ci % 2][:b - a].copy_(src, non_blocking=True)
            events[ci % 2].record()

        nthreads = 8
        with ThreadPoolExecutor(nthreads) as pool:
            launch(0)
            for ci, (a, b) in enumerate(chunks):
                events[ci % 2].synchronize()
                if ci + 1 < len(chunks):
                    launch(ci + 1)
                src = stage[ci % 2].numpy()[:b - a].reshape(b - a, -1)
                dst = out[a:b].reshape(b - a, -1)
                cols = dst.shape[1]
                cuts = [cols * t // nthreads for t in range(nthreads + 1)]
                list(pool.map(lambda t: np.copyto(dst[:, cuts[t]:cuts[t + 1]], src[:, cuts[t]:cuts[t + 1]]),
                              range(nthreads)))
        return out

    def _mcmc_refill(self, mcmc_steps, init_samples, init_loglikes, loglstar, step_size, dynamic_step_size,
                     keep_trace=False, live=None):
        """What NestedSampler.run needs from a batch (nested.py:429-439): start point, end point and end
        loglike of every chain (device tensors, chain-major); the trace stays on the device (optional, for chain
        statistics).  `_refill_to_host` gathers them over the ranks and brings them to the host.
        live=(live_u_dev, live_logl_dev, idx): start from rows `idx` of the device-resident live set instead of the host
        arrays init_samples / init_loglikes (which may then be None)."""
        n = len(live[2]) if live is not None else init_samples.shape[0]
        st, out, ncall = self._mcmc_device(mcmc_steps, step_size, dynamic_step_size, n,
                                           init_samples, init_loglikes, loglstar, 0, trace=keep_trace, live=live)
        first = out['first_x'].t().contiguous()
        last = st.x.t().contiguous()
        return dict(first=first, last=last, logl_last=st.logl, scale=out['scale'], ncall=ncall,
                    trace_x=out.get('trace_x'), acceptance=out['naccept'] / float(max(1, st.n * mcmc_steps)))

    def _pinned(self, name, shape, dtype):
        """Page-locked host staging buffers, allocated once per shape and reused by every refill."""
        cache = self.__dict__.setdefault('_pin_cache', {})
        key = (name, tuple(shape), dtype)
        if key not in cache:
            cache[key] = torch.empty(tuple(shape), dtype=dtype).pin_memory()
        return cache[key]

    def _refill_to_host(self, batch):
        """End states of a refill -> host arrays (first (N,d) f32, last (N,d) f32, logl_last (N,) f64), N = chains of all
        ranks in rank order (one NCCL all_gather per array over NVLink = the reference's gather + bcast + concatenate,
        nested.py:416-427).  Copies go through pinned buffers, asynchronously, with ONE synchronisation."""
        out = {}
        dev = {}
        for key in ('first', 'last', 'logl_last'):
            t = dist.allgather_rows(batch[key]) if self.use_mpi else batch[key]
            dev[key] = t
            host = self._pinned(key, t.shape, t.dtype)
            host.copy_(t, non_blocking=True)
            out[key] = host
        self._gathered_dev = dev          # device copies of the gathered batch: source of the live-set updates
        self.refill_derived = None
        if self.num_derived:
            # every rank evaluates the derived parameters of the gathered end states itself: the kernel is deterministic,
            # so the ranks agree bit for bit without another collective
            host = self._pinned('derived_last', (dev['last'].shape[0], self.num_derived), torch.float64)
            host.copy_(self.engine.derived(dev['last']), non_blocking=True)
            self.refill_derived = host.numpy()
        torch.cuda.current_stream().synchronize()
        return out['first'].numpy(), out['last'].numpy(), out['logl_last'].numpy()

    def _plot_trace(self, samples, latent_samples):
        pass    # plotting is outside the accelerated path

    def _chain_stats(self, samples, mean=None, std=None, step=None, trace=None, t_scale=None, t_shift=None):
        """Acceptance, ESS and jump distance with the reference's definitions (sampler.py:474-492).  With `trace` (the
        device trace float32 [T][d][N] nnb_mcmc_run wrote) the statistics of trace * t_scale + t_shift are computed by
        the CUDA kernels behind nnb_chain_stats / nnb_chain_autocorr and `samples` is ignored; host arrays
        (chains, steps, dim) go through the vectorised NumPy restatement in utils/evaluation.py."""
        if trace is not None:
            acceptance, ess, jump_distance = self.engine.chain_stats(trace, steps=step, t_scale=t_scale,
                                                                     t_shift=t_shift, mean=mean, std=std)
        else:
            acceptance = acceptance_rate(samples)
            flat = samples.reshape(-1, samples.shape[2])
            if mean is None:
                mean = flat.mean(0) if isinstance(flat, np.ndarray) else flat.double().mean(0).cpu().numpy()
            if std is None:
                std = flat.std(0) if isinstance(flat, np.ndarray) else \
                    flat.double().std(0, unbiased=False).cpu().numpy()
            ess = effective_sample_size(samples, mean, std)
            jump_distance = mean_jump_distance(samples)
        if step is None:
            self.logger.info('Acceptance [%5.4f] min ESS [%5.4f] max ESS [%5.4f] average jump [%5.4f]' %
                             (acceptance, np.min(ess), np.max(ess), jump_distance))
        else:
            self.logger.info('Step [%d] acceptance [%5.4f] min ESS [%5.4f] max ESS [%5.4f] average jump [%5.4f]' %
                             (step, acceptance, np.min(ess), np.max(ess), jump_distance))
        return acceptance, ess, jump_distance

    def _save_samples(self, samples, loglikes, weights=None, derived_samples=None, min_weight=1e-30,
                      outfile='chain'):
        """Chain files in the reference's text format (sampler.py:494-527): weight, -loglike, parameters,
        every number '%.5E'."""
        if weights is None:
            weights = np.ones_like(loglikes)

        def write(path, smp, lgl, wts, der):
            # the formatter reads the arrays as they are (nnb_write_chain_rows): a config-4 chain is 8.9 M rows, and the
            # (rows, 2 + d) float64 table np.column_stack would build is another 2.3 GB of freshly faulted pages
            f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
            smp, lgl, wts = f64(smp), f64(lgl), f64(wts)
            n, d = smp.shape
            nder = 0
            if der is not None:
                der = f64(der).reshape(n, -1)
                nder = der.shape[1]
            header = None
            if self.param_names is not None:
                header = ('#weight minusloglike ' + ' '.join(self.param_names)).encode()
            rc = L.load().nnb_write_chain_rows(path.encode(), header, wts.ctypes.data_as(L._dp), lgl.ctypes.data_as(L._dp),
                                               smp.ctypes.data_as(L._dp), d, der.ctypes.data_as(L._dp) if nder else None,
                                               nder, n, float(min_weight), 0)
            if rc < 0:
                raise IOError('could not write %s' % path)

        if len(samples.shape) == 2:
            write(os.path.join(self.logs['chains'], outfile + '.txt'), samples, loglikes, weights, derived_samples)
        elif len(samples.shape) == 3:
            for ib in range(samples.shape[0]):
                write(os.path.join(self.logs['chains'], outfile + '_%s.txt' % (ib + 1)), samples[ib], loglikes[ib],
                      weights[ib], None if derived_samples is None else derived_samples[ib])

    # ---- rejection samplers used before / instead of MCMC (nnest/sampler.py:529-630), batched on the device -----------
    # The reference draws ONE candidate per loop turn.  Here a block of k candidates goes through the kernels in one
    # launch and the first acceptable one (in draw order) is returned -- the sequential algorithm exactly, since the
    # candidates are independent; the ones drawn after it are discarded and only the loop turns the reference would have
    # made are counted (ncall, total_calls).
    def _loglike_rows(self, x):
        """likelihood of host rows WITHOUT touching the call counter (the batched samplers count what they consume)"""
        x, xd = self._to_device_rows(x)
        logl = self.engine.loglike(xd).cpu().numpy()
        if self._like.follows_input_dtype and x.dtype == np.float32 and not self._t_f64:
            logl = logl.astype(np.float32)
        return logl

    def _rejection_prior_sample(self, loglstar, num_trials=None):
        """nnest/sampler.py:529-543.  num_trials=None: k prior draws per launch; np.random is then rewound and advanced
        by exactly the draws the one-at-a-time loop would have consumed, so a seeded run sees the same stream."""
        if num_trials is None:
            ncall = 0
            k = int(min(max(8, 2 * getattr(self, '_rej_prior_mean', 4)), 1 << 16))
            rewindable = isinstance(self._prior_obj, UniformPrior) and self.sample_prior == self._prior_obj.sample
            while True:
                state = np.random.get_state() if rewindable else None
                x = self.sample_prior(k if rewindable else 1)
                logl = self._loglike_rows(x)
                ok = np.nonzero(logl > loglstar)[0]
                if len(ok):
                    j = int(ok[0])
                    if rewindable and j + 1 < k:
                        np.random.set_state(state)
                        self.sample_prior(j + 1)
                    ncall += j + 1
                    self.total_calls += j + 1
                    self._rej_prior_mean = 0.8 * getattr(self, '_rej_prior_mean', 4) + 0.2 * ncall
                    return x[j:j + 1], logl[j:j + 1], self._derived_rows(x[j:j + 1]), ncall
                ncall += x.shape[0]
                self.total_calls += x.shape[0]
                k = min(2 * k, 1 << 16)
        x = self.sample_prior(num_trials)
        logl, derived = self.loglike(x)
        ncall = num_trials / np.sum(logl > loglstar)
        return x, logl, derived, ncall

    def _rejection_flow_sample(self, init_samples, loglstar, enlargement_factor=1.1, constant_efficiency_factor=None,
                               cache=False):
        """nnest/sampler.py:545-607: uniform draws in the latent ball of radius enlargement * max |z(live)|, mapped
        through the flow, thinned by the Jacobian envelope exp(log|J| - max log|J|) and by the likelihood constraint."""
        def get_cache():
            z, log_det_J = self.trainer.forward(np.asarray(init_samples, dtype=np.float32))
            self.max_log_det_J = float(enlargement_factor * torch.max(-log_det_J))
            self.max_r = float(torch.linalg.norm(z, dim=1).max())

        if not cache or not hasattr(self, 'max_log_det_J'):
            get_cache()
        if constant_efficiency_factor is not None:
            enlargement_factor = (1 / constant_efficiency_factor) ** (1 / self.x_dim)
        d, ncall = self.x_dim, 0
        k = int(min(max(64, 4 * getattr(self, '_rej_flow_mean', 16)), 1 << 16))
        while True:
            g = torch.randn((k, d), device=self.device)
            r = torch.rand((k, 1), device=self.device) ** (1. / d)
            z = enlargement_factor * self.max_r * g * r / torch.linalg.norm(g, dim=1, keepdim=True)
            x, log_det_J = self.trainer.inverse(z)
            logl, logp = self.engine.loglike(x, want_prior=True)
            rnd_u = torch.rand((k,), device=self.device)
            ratio = (log_det_J.double() - self.max_log_det_J).exp().clamp(max=1)
            inside = logp > -1e30
            if getattr(self.trainer, 'flow_kind', 'nvp') == 'spline':
                # drawn one at a time, such a candidate makes the reference's inverse raise ValueError -> `continue`
                inside = inside & (self.engine.flow_empty_halves(z) == 0)
            evaluated = inside & ~(rnd_u > ratio)                    # the turns that reach self.loglike
            good = evaluated & ~(torch.isfinite(logl) & (logl < loglstar)) & (rnd_u < ratio)
            idx = torch.nonzero(good)
            if idx.numel():
                j = int(idx[0])
                n_eval = int(evaluated[:j + 1].sum())
                ncall += n_eval
                self.total_calls += n_eval
                self._rej_flow_mean = 0.8 * getattr(self, '_rej_flow_mean', 16) + 0.2 * (j + 1)
                lj = logl[j:j + 1].cpu().numpy()
                if self._like.follows_input_dtype and not self._t_f64:
                    lj = lj.astype(np.float32)
                return x[j:j + 1].cpu().numpy(), lj, self._derived_rows(x[j:j + 1]), ncall
            n_eval = int(evaluated.sum())
            ncall += n_eval
            self.total_calls += n_eval
            k = min(2 * k, 1 << 16)

    def _density_sample(self, loglstar):
        """nnest/sampler.py:609-630: draws from the flow's own density until one beats the constraint."""
        ncall = 0
        k = int(min(max(64, 4 * getattr(self, '_dens_mean', 16)), 1 << 16))
        while True:
            z = self.trainer.get_prior_samples(k)
            x = self.trainer.get_samples(z)
            logl, logp = self.engine.loglike(x, want_prior=True)
            inside = logp > -1e30
            if getattr(self.trainer, 'flow_kind', 'nvp') == 'spline':
                inside = inside & (self.engine.flow_empty_halves(z) == 0)
            idx = torch.nonzero(inside & (logl > loglstar))
            if idx.numel():
                j = int(idx[0])
                n_eval = int(inside[:j + 1].sum())
                ncall += n_eval
                self.total_calls += n_eval
                self._dens_mean = 0.8 * getattr(self, '_dens_mean', 16) + 0.2 * (j + 1)
                lj = logl[j:j + 1].cpu().numpy()
                if self._like.follows_input_dtype and not self._t_f64:
                    lj = lj.astype(np.float32)
                return x[j:j + 1].cpu().numpy(), lj, self._derived_rows(x[j:j + 1]), ncall
            n_eval = int(inside.sum())
            ncall += n_eval
            self.total_calls += n_eval
            k = min(2 * k, 1 << 16)
