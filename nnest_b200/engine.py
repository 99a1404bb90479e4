"""Thin torch-tensor front end of the C ABI (include/nnb.h).

PyTorch is used for device memory and streams only; all arithmetic of the hot path happens in
libnnb.so.  One Engine = one nnb_handle = one CUDA device.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _darr(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


def flatten_state_dict(sd, scale=''):
    """netG.state_dict() of a SingleSpeedNVP -> (flat float32 array in nnb_set_flow order, d, H, L, B, flags).
    Key layout: flow.flows.<i>.{scale_net,translate_net}.<2j>.{weight,bias} (+ flow.flows.<i>.scale for
    ScaleLayer), reference nnest/networks.py:262-282,312-347."""
    get = lambda k: np.asarray(sd[k].detach().cpu().numpy() if hasattr(sd[k], 'detach') else sd[k], dtype=np.float32)
    if scale is None:
        # infer the `scale` kwarg of SingleSpeedNVP from the keys: no scale_net -> translate only; ScaleLayer parameters
        # (flow.flows.<odd>.scale) -> 'constant'
        has_s = any('.scale_net.' in k for k in sd)
        has_c = any(k.startswith('flow.flows.') and k.endswith('.scale') for k in sd)
        scale = '' if has_s else ('constant' if has_c else 'translate')
    translate_only = scale in ('translate', 'constant')
    stride = 2 if scale == 'constant' else 1
    idx = sorted({int(k.split('.')[2]) for k in sd if k.startswith('flow.flows.')})
    if not idx:
        raise ValueError('not a SingleSpeedNVP state_dict')
    num_blocks = (max(idx) + stride) // stride
    parts = []
    nlin = None
    for k in range(num_blocks):
        fi = k * stride
        for net in ('scale_net', 'translate_net'):
            if net == 'scale_net' and translate_only:
                continue
            j = 0
            while 'flow.flows.%d.%s.%d.weight' % (fi, net, 2 * j) in sd:
                w = get('flow.flows.%d.%s.%d.weight' % (fi, net, 2 * j))
                if j == 0:
                    hidden, d = w.shape
                parts.append(w.ravel())
                parts.append(get('flow.flows.%d.%s.%d.bias' % (fi, net, 2 * j)).ravel())
                j += 1
            if j < 2:
                raise ValueError('state_dict is missing %s of block %d' % (net, k))
            nlin = j
    flags = 0
    if translate_only:
        flags |= L.NNB_FLOW_TRANSLATE_ONLY
    if scale == 'constant':
        flags |= L.NNB_FLOW_CONST_SCALE
        parts.append(np.array([get('flow.flows.%d.scale' % (k * stride + 1)) for k in range(num_blocks)],
                              dtype=np.float32).ravel())
    return np.concatenate(parts), int(d), int(hidden), int(nlin - 2), int(num_blocks), flags


class ChainState(object):
    """Per-chain state in chain-minor layout (element (i, c) at [i * n + c])."""

    def __init__(self, n, d, device):
        self.n, self.d = n, d
        self.z = torch.empty((d, n), dtype=torch.float32, device=device)
        self.x = torch.empty((d, n), dtype=torch.float32, device=device)
        self.logl = torch.empty((n,), dtype=torch.float64, device=device)
        self.logdet = torch.empty((n,), dtype=torch.float32, device=device)
        self.logp = torch.empty((n,), dtype=torch.float64, device=device)


class Engine(object):

    def __init__(self, device=None):
        self.lib = L.load()
        if not torch.cuda.is_available():
            raise RuntimeError('nnest_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        h = C.c_void_p()
        rc = self.lib.nnb_create(self.device.index, C.byref(h))
        if rc != 0:
            raise L.NNBError(rc, (self.lib.nnb_last_error(None) or b'').decode())
        self.h = h
        self.d = None
        self.num_derived = 0      # derived parameters of the installed user likelihood
        self.user_layout = ()     # (name, NNB_DTYPE_*) of its dataset's arrays
        self._data_token, self._data_tensors = None, ()   # the bound dataset (UserData.token) and its device copy
        self.gpu_launches = 0     # kernels launched through this engine (bench.py reports it)
        self.default_impl = int(os.environ.get('NNB_IMPL', L.NNB_IMPL_AUTO))   # 0 auto, 1 ffma, 2 tcgen05

    def __del__(self):
        try:
            if getattr(self, 'h', None):
                self.lib.nnb_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _check(self, rc):
        L.check(self.h, rc)

    # ---- flow -------------------------------------------------------------------------------
    def set_flow(self, flat, d, hidden, num_layers, num_blocks, flags=0):
        flat = np.ascontiguousarray(flat, dtype=np.float32)
        self._check(self.lib.nnb_set_flow(self.h, d, hidden, num_layers, num_blocks, flags,
                                          flat.ctypes.data_as(C.POINTER(C.c_float)), flat.size))
        self.d = d
        self.flow_shape = (d, hidden, num_layers, num_blocks, flags)

    def set_flow_from_state_dict(self, sd, scale=''):
        flat, d, hidden, nl, nb, flags = flatten_state_dict(sd, scale)
        self.set_flow(flat, d, hidden, nl, nb, flags)

    def set_flow_spline(self, packed, d, hidden, num_blocks, num_bins=8, tail_bound=3.0):
        """Install a neural-spline flow (flow='spline'); `packed` in the layout of include/nnb.h: nnb_set_flow_spline."""
        packed = np.ascontiguousarray(packed, dtype=np.float32)
        self._check(self.lib.nnb_set_flow_spline(self.h, d, hidden, num_blocks, num_bins, float(tail_bound),
                                                 packed.ctypes.data_as(C.POINTER(C.c_float)), packed.size))
        self.d = d
        self.flow_shape = (d, hidden, 'spline', num_blocks, num_bins)

    def flow_empty_halves(self, z, inverse=True):
        """int32 flags (n,): 1 where the reference's RQS would raise ValueError('No input values') on the one-sample batch
        z[r] (a coupling transform with no coordinate inside the tail bound); always 0 for the affine-coupling flow."""
        assert z.is_cuda and z.dtype == torch.float32 and z.dim() == 2 and z.shape[1] == self.d
        flags = torch.zeros((z.shape[0],), dtype=torch.int32, device=z.device)
        if z.shape[0]:
            self._check(self.lib.nnb_flow_empty_halves(self.h, _ptr(z), z.stride(0), z.stride(1), 1 if inverse else 0,
                                                       _ptr(flags), z.shape[0], _stream()))
            self.gpu_launches += 1
        return flags

    def _flow(self, fn, a):
        assert a.is_cuda and a.dtype == torch.float32 and a.dim() == 2 and a.shape[1] == self.d
        n = a.shape[0]
        out = torch.empty((n, self.d), dtype=torch.float32, device=a.device)
        ld = torch.empty((n,), dtype=torch.float32, device=a.device)
        if n:
            self._check(fn(self.h, _ptr(a), a.stride(0), a.stride(1), _ptr(out), out.stride(0), out.stride(1),
                           _ptr(ld), n, _stream()))
            self.gpu_launches += 1
        return out, ld

    def flow_inverse(self, z):
        """z (n,d) float32 cuda (any strides) -> x (n,d), log|det dx/dz| (n,)"""
        return self._flow(self.lib.nnb_flow_inverse, z)

    def flow_forward(self, x):
        return self._flow(self.lib.nnb_flow_forward, x)

    # ---- flow fitting -----------------------------------------------------------------------
    B200_MAX_SMEM = 232448     # sharedMemPerBlockOptin on sm_100

    def train_supported(self, d, hidden, num_layers, num_blocks):
        return bool(self.lib.nnb_train_supported(d, hidden, num_layers, num_blocks, self.B200_MAX_SMEM))

    def _train_args(self, arch, params, adam_m, adam_v, step0, x_train, x_valid, batch_size, perm=None, jitter=0.0,
                    lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, seed=0, epoch=0, noise=None,
                    grad_out=None, do_train=True, grad_only=False, batch_total=0):
        d, hidden, nl, nb = arch
        a = L.nnb_train_args()
        a.x_dim, a.hidden_dim, a.num_layers, a.num_blocks = d, hidden, nl, nb
        for t in (x_train, x_valid):
            assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape[1] == d)
        for t in (params, adam_m, adam_v, grad_out):
            assert t is None or (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous())
        a.x_train, a.n_train = _ptr(x_train), 0 if x_train is None else x_train.shape[0]
        if perm is not None:
            assert perm.is_cuda and perm.dtype == torch.int64 and perm.is_contiguous() and perm.numel() == a.n_train
        a.perm = _ptr(perm)
        a.batch_size = int(batch_size)
        a.x_valid, a.n_valid = _ptr(x_valid), 0 if x_valid is None else x_valid.shape[0]
        if noise is not None:
            assert noise.is_cuda and noise.dtype == torch.float32 and noise.is_contiguous() \
                and tuple(noise.shape) == (a.n_train, d)
        a.noise = _ptr(noise)
        a.jitter = float(jitter)
        a.seed, a.epoch = int(seed) & (2 ** 64 - 1), int(epoch) & 0xffffffff
        a.lr, a.beta1, a.beta2, a.eps, a.weight_decay = float(lr), float(betas[0]), float(betas[1]), float(eps), \
            float(weight_decay)
        a.step0 = int(step0)
        a.params, a.adam_m, a.adam_v, a.n_params = _ptr(params), _ptr(adam_m), _ptr(adam_v), params.numel()
        a.grad_out = _ptr(grad_out)
        a.do_train = 1 if do_train else 0
        a.grad_only, a.batch_total = (1 if grad_only else 0), int(batch_total)
        return a

    def train_epoch(self, *args, **kwargs):
        """One epoch of Trainer._train + _validate in one kernel launch (include/nnb.h: nnb_train_epoch).
        arch = (d, hidden, num_layers, num_blocks); params / adam_m / adam_v: flat float32 cuda vectors in
        state_dict order, updated in place.  Returns (train_loss_sum, val_nll_sum, grid)."""
        a = self._train_args(*args, **kwargs)
        tl, vl, grid = C.c_double(0.0), C.c_double(0.0), C.c_int(0)
        a.train_loss_sum_out, a.val_nll_sum_out, a.grid_out = C.pointer(tl), C.pointer(vl), C.pointer(grid)
        self._check(self.lib.nnb_train_epoch(self.h, C.byref(a), _stream()))
        self.gpu_launches += 1
        return tl.value, vl.value, grid.value

    def train_epoch_begin(self, *args, **kwargs):
        """Queue the epoch without waiting for it (nnb_train_epoch_begin; same arguments as train_epoch); at most two may
        be in flight.  The tensors involved are only touched by stream-ordered work, so the caller may drop them."""
        a = self._train_args(*args, **kwargs)
        self._check(self.lib.nnb_train_epoch_begin(self.h, C.byref(a), _stream()))
        self.gpu_launches += 1
        self._epochs_in_flight = getattr(self, '_epochs_in_flight', 0) + 1

    def train_epoch_end(self):
        """Losses of the oldest epoch in flight: (train_loss_sum, val_nll_sum, grid)."""
        tl, vl, grid = C.c_double(0.0), C.c_double(0.0), C.c_int(0)
        self._epochs_in_flight = max(0, getattr(self, '_epochs_in_flight', 0) - 1)     # the library gives the slot up too
        self._check(self.lib.nnb_train_epoch_end(self.h, C.byref(tl), C.byref(vl), C.byref(grid)))
        return tl.value, vl.value, grid.value

    def train_epoch_drain(self):
        """Collect (and drop) whatever epochs an interrupted fit left in flight."""
        while getattr(self, '_epochs_in_flight', 0) > 0:
            self.train_epoch_end()

    def mean_nn_distance(self, x):
        """x (n, d) float64 cuda -> mean distance to the nearest other row (nnb_mean_nn_distance)."""
        assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and x.dim() == 2
        out = C.c_double(0.0)
        self._check(self.lib.nnb_mean_nn_distance(self.h, _ptr(x), x.shape[0], x.shape[1], C.byref(out), _stream()))
        self.gpu_launches += 1
        return out.value

    # ---- chain diagnostics on the device trace ----------------------------------------------
    def chain_stats(self, trace_x, steps=None, t_scale=None, t_shift=None, mean=None, std=None):
        """Acceptance, effective sample size per dimension and mean jump distance (nnest/utils/evaluation.py:17-73, as
        Sampler._chain_stats uses them) of a device trace float32 [T][d][N]; `steps` restricts it to the first steps + 1
        points.  mean / std default to those of the (transformed) samples; the ESS divides by `std` as the reference does."""
        assert trace_x.is_cuda and trace_x.dtype == torch.float32 and trace_x.is_contiguous() and trace_x.dim() == 3
        T, d, n = trace_x.shape
        if steps is not None:
            T = min(T, int(steps) + 1)
        ka, ts = _darr(np.broadcast_to(1.0 if t_scale is None else t_scale, (d,)))
        kb, tb = _darr(np.broadcast_to(0.0 if t_shift is None else t_shift, (d,)))
        moved, jump = C.c_double(0.0), C.c_double(0.0)
        s1, s2 = np.zeros(d), np.zeros(d)
        want = mean is None or std is None
        self._check(self.lib.nnb_chain_stats(self.h, _ptr(trace_x), T, d, n, ts, tb, C.byref(moved), C.byref(jump),
                                             s1.ctypes.data_as(L._dp) if want else None,
                                             s2.ctypes.data_as(L._dp) if want else None, _stream()))
        self.gpu_launches += 2 if want else 1
        total = float(n) * (T - 1)
        acceptance = moved.value / total if total else 0.0
        jump_distance = jump.value / total if total else 0.0
        if mean is None:
            mean = s1 / (float(n) * T)
        if std is None:
            std = np.sqrt(np.maximum(s2 / (float(n) * T) - (s1 / (float(n) * T)) ** 2, 0.0))
        km, mu = _darr(np.broadcast_to(mean, (d,)))
        var = np.broadcast_to(np.asarray(std, dtype=np.float64), (d,))
        ess = np.ones(d)
        out = np.zeros((32, d))
        s, done = 1, False
        while s < T and not done:                       # evaluation.py:30-37, 32 lags per launch
            nl = min(32, T - s)
            self._check(self.lib.nnb_chain_autocorr(self.h, _ptr(trace_x), T, d, n, ts, tb, mu, s, nl,
                                                    out.ctypes.data_as(L._dp), _stream()))
            self.gpu_launches += 1
            for l in range(nl):
                p = out[l] / (float(n) * (T - s - l)) / var
                if np.sum(p > 0.05) == 0:
                    done = True
                    break
                ess = ess + np.where(p > 0.05, 2.0 * p * (1.0 - float(s + l) / T), 0.0)
            s += nl
        return acceptance, T / ess, jump_distance

    # ---- target -----------------------------------------------------------------------------
    def set_user_likelihood(self, source, num_derived=0, layout=()):
        """Install a CUDA C++ likelihood (nnb_set_user_likelihood, or nnb_set_user_likelihood_derived with num_derived > 0,
        or nnb_set_user_likelihood_data with a dataset layout: (name, NNB_DTYPE_*) per array): returns the number of
        kernel variants compiled.  Drops the bound dataset."""
        n = C.c_int(0)
        layout = tuple(layout)
        self.user_source = None     # until the call succeeds: the library keeps the previous source on failure, unbound
        self._data_token, self._data_tensors = None, ()
        if layout:
            names = (C.c_char_p * len(layout))(*[name.encode() for name, _ in layout])
            dtypes = (C.c_int * len(layout))(*[dt for _, dt in layout])
            self._check(self.lib.nnb_set_user_likelihood_data(self.h, source.encode(), int(num_derived), len(layout),
                                                               names, dtypes, C.byref(n)))
        elif num_derived:
            self._check(self.lib.nnb_set_user_likelihood_derived(self.h, source.encode(), int(num_derived), C.byref(n)))
        else:
            self._check(self.lib.nnb_set_user_likelihood(self.h, source.encode(), C.byref(n)))
        self.user_source = source
        self.num_derived = int(num_derived)
        self.user_layout = layout
        return n.value

    def bind_user_data(self, user_data):
        """Upload a CudaLikelihood's dataset (likelihoods.UserData) to this engine's device and bind it
        (nnb_bind_user_data).  The tensors stay alive until another dataset is bound; binding the dataset already bound
        does nothing, so a dataset is uploaded once per engine however often the target is set."""
        if user_data.token == self._data_token:
            return
        tensors = [torch.from_numpy(np.array(a)).to(self.device) for a in user_data.arrays]
        n = len(tensors)
        ptrs = (C.c_void_p * n)(*[t.data_ptr() if t.numel() else None for t in tensors])
        sizes = (C.c_int64 * n)(*[t.numel() for t in tensors])
        self._data_token = None
        self._check(self.lib.nnb_bind_user_data(self.h, ptrs, sizes))
        self._data_token, self._data_tensors = user_data.token, tuple(tensors)

    def set_user_transform(self, source):
        """Install a CUDA C++ prior transform (nnb_set_user_transform): returns the number of kernel variants compiled."""
        n = C.c_int(0)
        self._check(self.lib.nnb_set_user_transform(self.h, source.encode(), C.byref(n)))
        self.transform_source = source
        return n.value

    def set_target(self, d, like_id, like_params=(), t_scale=None, t_shift=None, compute_f64=False,
                   prior_kind=L.NNB_PRIOR_NONE, prior_lo=None, prior_hi=None, user_source=None, num_derived=0,
                   transform_source=None, transform_params=(), user_data=None):
        """user_source: CUDA C++ of the likelihood NNB_LIKE_USER selects (with num_derived derived parameters and the
        layout of user_data, a likelihoods.UserData), installed first when it is not the current one; user_data is then
        uploaded and bound unless it already is.  transform_source: CUDA C++ of a prior transform, used with its
        transform_params in place of t_scale / t_shift (nnb_set_target_user_transform), installed first likewise."""
        layout = user_data.layout if user_data is not None else ()
        if user_source is not None and (user_source, num_derived, layout) != (getattr(self, 'user_source', None),
                                                                               getattr(self, 'num_derived', 0),
                                                                               getattr(self, 'user_layout', ())):
            self.set_user_likelihood(user_source, num_derived, layout)
        if user_source is not None and user_data is not None:
            self.bind_user_data(user_data)
        if transform_source is not None:
            if t_scale is not None or t_shift is not None:
                raise ValueError('a user transform replaces t_scale / t_shift')
            if transform_source != getattr(self, 'transform_source', None):
                self.set_user_transform(transform_source)
        t = L.nnb_target()
        keep = []
        t.like_id = like_id
        t.n_like_params = len(like_params)
        a, p = _darr(like_params if len(like_params) else [0.0])
        keep.append(a)
        t.like_params = p
        t.compute_f64 = 1 if compute_f64 else 0
        if t_scale is not None:
            a, t.t_scale = _darr(np.broadcast_to(t_scale, (d,)))
            keep.append(a)
            a, t.t_shift = _darr(np.broadcast_to(0.0 if t_shift is None else t_shift, (d,)))
            keep.append(a)
        t.prior_kind = prior_kind
        if prior_kind != L.NNB_PRIOR_NONE:
            a, t.prior_lo = _darr(np.broadcast_to(prior_lo, (d,)))
            keep.append(a)
            a, t.prior_hi = _darr(np.broadcast_to(prior_hi, (d,)))
            keep.append(a)
        if transform_source is not None:
            a, tp = _darr(transform_params if len(transform_params) else [0.0])
            keep.append(a)
            self._check(self.lib.nnb_set_target_user_transform(self.h, d, C.byref(t), tp, len(transform_params)))
        else:
            self._check(self.lib.nnb_set_target(self.h, d, C.byref(t)))
        self.target_d = d

    def transform(self, u, out=None):
        """u (n,d) float32 or float64 cuda -> v = transform(u) float64 (n, d) of the target's user transform
        (nnb_transform): the values the likelihood sees at these points, bit for bit."""
        assert u.is_cuda and u.dim() == 2 and u.shape[1] == self.target_d
        assert u.dtype in (torch.float32, torch.float64)
        n, d = u.shape
        if out is None:
            out = torch.empty((n, d), dtype=torch.float64, device=u.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (n, d)
        if n:
            self._check(self.lib.nnb_transform(self.h, _ptr(u), 1 if u.dtype == torch.float64 else 0, u.stride(0),
                                               u.stride(1), _ptr(out), n, _stream()))
            self.gpu_launches += 1
        return out

    def transform_trace(self, trace_x, row0=0, row_step=1, n_rows=None, out=None):
        """v = transform(x) of rows row0, row0 + row_step, ... (n_rows of them; default: to the end) of a device trace
        float32 (T, d, n) -> float64 (n_rows, d, n) (nnb_transform_trace)."""
        assert trace_x.is_cuda and trace_x.dtype == torch.float32 and trace_x.is_contiguous() and trace_x.dim() == 3
        T, d, n = trace_x.shape
        assert d == self.target_d
        if n_rows is None:
            n_rows = len(range(row0, T, row_step))
        assert n_rows == 0 or row0 + (n_rows - 1) * row_step < T
        if out is None:
            out = torch.empty((n_rows, d, n), dtype=torch.float64, device=trace_x.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (n_rows, d, n)
        if n and n_rows:
            self._check(self.lib.nnb_transform_trace(self.h, _ptr(trace_x), n, row0, row_step, n_rows, _ptr(out),
                                                     _stream()))
            self.gpu_launches += 1
        return out

    def loglike(self, u, want_prior=False):
        """u (n,d) float32 or float64 cuda -> logl float64 (n,) [, logp float64 (n,)]"""
        assert u.is_cuda and u.dim() == 2 and u.shape[1] == self.target_d
        assert u.dtype in (torch.float32, torch.float64)
        n = u.shape[0]
        logl = torch.empty((n,), dtype=torch.float64, device=u.device)
        logp = torch.empty((n,), dtype=torch.float64, device=u.device) if want_prior else None
        if n:
            self._check(self.lib.nnb_loglike(self.h, _ptr(u), 1 if u.dtype == torch.float64 else 0, u.stride(0),
                                             u.stride(1), _ptr(logl), _ptr(logp), n, _stream()))
            self.gpu_launches += 1
        return (logl, logp) if want_prior else logl

    def derived(self, u, out=None):
        """u (n,d) float32 or float64 cuda -> derived parameters float64 (n, num_derived) (nnb_derived)"""
        assert u.is_cuda and u.dim() == 2 and u.shape[1] == self.target_d
        assert u.dtype in (torch.float32, torch.float64)
        n = u.shape[0]
        if out is None:
            out = torch.empty((n, self.num_derived), dtype=torch.float64, device=u.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (n, self.num_derived)
        if n:
            self._check(self.lib.nnb_derived(self.h, _ptr(u), 1 if u.dtype == torch.float64 else 0, u.stride(0),
                                             u.stride(1), _ptr(out), n, _stream()))
            self.gpu_launches += 1
        return out

    def derived_trace(self, trace_x, row0=0, row_step=1, n_rows=None, init=None, out=None):
        """Derived parameters of rows row0, row0 + row_step, ... (n_rows of them; default: to the end) of a device trace
        float32 (T, d, n) -> float64 (n_rows, num_derived, n) (nnb_derived_trace).  init (num_derived, n) float64 cuda: the
        values of chains that have not moved since row 0."""
        assert trace_x.is_cuda and trace_x.dtype == torch.float32 and trace_x.is_contiguous() and trace_x.dim() == 3
        T, d, n = trace_x.shape
        assert d == self.target_d
        if n_rows is None:
            n_rows = len(range(row0, T, row_step))
        assert n_rows == 0 or row0 + (n_rows - 1) * row_step < T
        if out is None:
            out = torch.empty((n_rows, self.num_derived, n), dtype=torch.float64, device=trace_x.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (n_rows, self.num_derived, n)
        if init is not None:
            assert init.is_cuda and init.dtype == torch.float64 and init.is_contiguous() \
                and tuple(init.shape) == (self.num_derived, n)
        if n and n_rows:
            self._check(self.lib.nnb_derived_trace(self.h, _ptr(trace_x), n, row0, row_step, n_rows, _ptr(init),
                                                   _ptr(out), _stream()))
            self.gpu_launches += 1
        return out

    # ---- MCMC -------------------------------------------------------------------------------
    def mcmc_init(self, n, init_u=None, init_z=None, init_logl=None, seed=0, chain_offset=0, start_try=0,
                  want_counts=None):
        """init_u / init_z: chain-minor (d,n) float32 cuda tensors.  Returns (ChainState, n_bad_start, ncall).
        When the start log-likelihoods are supplied nothing has to be counted and the call stays asynchronous
        (the two counters are then returned as 0)."""
        st = ChainState(n, self.d, self.device)
        a = L.nnb_mcmc_init_args()
        a.n_chains = n
        a.z, a.x, a.logl, a.logdet, a.logp = [t.data_ptr() for t in (st.z, st.x, st.logl, st.logdet, st.logp)]
        for name, t, dt in (('init_u', init_u, torch.float32), ('init_z', init_z, torch.float32),
                            ('init_logl', init_logl, torch.float64)):
            if t is not None:
                assert t.is_cuda and t.dtype == dt and t.is_contiguous()
                setattr(a, name, t.data_ptr())
        a.seed, a.chain_offset, a.start_try = seed, chain_offset, start_try
        nbad, ncall = C.c_int64(0), C.c_int64(0)
        if want_counts is None:
            want_counts = init_logl is None
        if want_counts:
            a.n_bad_start, a.ncall = C.pointer(nbad), C.pointer(ncall)
        self._check(self.lib.nnb_mcmc_init(self.h, C.byref(a), _stream()))
        self.gpu_launches += 2          # control-block reset + chain-start kernel
        return st, nbad.value, ncall.value

    def mcmc_run(self, st, steps, mode=L.NNB_MODE_HARD, loglstar=0.0, step_size=0.0, dynamic_step_size=False,
                 seed=0, chain_offset=0, step_offset=0, trace=False, replay=None, dump_noise=False, impl=None,
                 sync=True):
        """Advances `st` in place by `steps` steps.  Returns a dict with scale, ncall, naccept and, if
        requested, the trace tensors (steps+1, d, n) / (steps+1, n) and the dumped noise.  sync=False only enqueues
        the work (no scale / ncall / naccept in the result; `mcmc_result()` fetches those of the last run)."""
        n, d = st.n, st.d
        a = L.nnb_mcmc_args()
        a.n_chains, a.steps, a.mode = n, steps, mode
        a.loglstar = 0.0 if loglstar is None else float(loglstar)
        a.step_size, a.dynamic_step_size = float(step_size), 1 if dynamic_step_size else 0
        a.seed, a.chain_offset, a.step_offset = seed, chain_offset, step_offset
        a.impl = self.default_impl if impl is None else impl
        a.z, a.x, a.logl, a.logdet, a.logp = [t.data_ptr() for t in (st.z, st.x, st.logl, st.logdet, st.logp)]
        out = {}
        if trace:
            out['trace_x'] = torch.empty((steps + 1, d, n), dtype=torch.float32, device=self.device)
            out['trace_z'] = torch.empty((steps + 1, d, n), dtype=torch.float32, device=self.device)
            out['trace_logl'] = torch.empty((steps + 1, n), dtype=torch.float64, device=self.device)
            a.trace_x, a.trace_z, a.trace_logl = [out[k].data_ptr() for k in ('trace_x', 'trace_z', 'trace_logl')]
        if replay is not None:
            nrm, uni = replay
            assert nrm.is_cuda and nrm.dtype == torch.float32 and nrm.is_contiguous() and tuple(nrm.shape) == (steps, n, d)
            assert uni.is_cuda and uni.dtype == torch.float32 and uni.is_contiguous() and tuple(uni.shape) == (steps, n)
            a.replay_normals, a.replay_uniforms = nrm.data_ptr(), uni.data_ptr()
        if dump_noise:
            out['normals'] = torch.empty((steps, n, d), dtype=torch.float32, device=self.device)
            out['uniforms'] = torch.empty((steps, n), dtype=torch.float32, device=self.device)
            a.dump_normals, a.dump_uniforms = out['normals'].data_ptr(), out['uniforms'].data_ptr()
        scale, ncall, nacc, nl, impl_ran = C.c_double(0), C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int(0)
        if sync:
            a.scale_out, a.ncall_out, a.naccept_out = C.pointer(scale), C.pointer(ncall), C.pointer(nacc)
        a.launches_out, a.impl_out = C.pointer(nl), C.pointer(impl_ran)
        self._check(self.lib.nnb_mcmc_run(self.h, C.byref(a), _stream()))
        self.gpu_launches += nl.value + 1          # + the one-thread control-block reset
        out.update(launches=nl.value, impl=impl_ran.value)
        if sync:
            out.update(scale=scale.value, ncall=ncall.value, naccept=nacc.value)
        return out

    def mcmc_result(self):
        """scale, ncall, naccept of the last mcmc_run (synchronises the stream)."""
        scale, ncall, nacc = C.c_double(0), C.c_int64(0), C.c_int64(0)
        self._check(self.lib.nnb_mcmc_result(self.h, C.byref(scale), C.byref(ncall), C.byref(nacc), _stream()))
        return dict(scale=scale.value, ncall=ncall.value, naccept=nacc.value)
