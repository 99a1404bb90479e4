"""Analytic likelihoods with the reference's class names and constructor signatures
(nnest/likelihoods.py), evaluated by the batched CUDA likelihood kernel (nnb_loglike) instead of a
per-row Python loop.  Each class only carries the id and parameter vector the kernel needs; calling an
instance on host arrays uploads them, runs the kernel and downloads the values -- there is no CPU
implementation in this package.
"""
import itertools
import re

import numpy as np

from . import _lib as L

_engines = {}
_data_tokens = itertools.count(1)
# the element types a dataset array may have, and their codes in the C ABI
DATA_DTYPES = {np.dtype(np.float64): L.NNB_DTYPE_F64, np.dtype(np.float32): L.NNB_DTYPE_F32,
               np.dtype(np.int32): L.NNB_DTYPE_I32}


def _eval_engine():
    """One lazily created Engine per process/device for direct `like(x)` calls."""
    import torch
    from .engine import Engine
    dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if dev not in _engines:
        _engines[dev] = Engine(dev)
    return _engines[dev]


class Likelihood(object):
    num_derived = 0
    num_evaluations = 0
    like_id = None
    # True when NumPy keeps the reference's result in the input dtype (float32 rows -> float32 values)
    follows_input_dtype = False

    def __init__(self, x_dim):
        self.x_dim = x_dim

    def device_params(self):
        return []

    def device_source(self):
        """CUDA C++ of a user likelihood (CudaLikelihood), None for the built-in ones."""
        return None

    def device_data(self):
        """The dataset of a CudaLikelihood (a UserData), None for the built-in likelihoods and without data."""
        return None

    def __call__(self, x):
        """x: (n, x_dim) or (x_dim,) array in the likelihood's own coordinates -> log-likelihood(s)."""
        import torch
        if isinstance(x, list):
            x = np.array(x)
        x = np.asarray(x)
        single = x.ndim == 1
        xx = np.ascontiguousarray(x[None, :] if single else x)
        if xx.dtype not in (np.float32, np.float64):
            xx = xx.astype(np.float64)
        self.num_evaluations += xx.shape[0]
        eng = _eval_engine()
        eng.set_target(self.x_dim, self.like_id, self.device_params(), user_source=self.device_source(),
                       num_derived=self.num_derived, user_data=self.device_data())
        xd = torch.from_numpy(xx).to(eng.device)
        out = eng.loglike(xd).cpu().numpy()
        if self.follows_input_dtype and xx.dtype == np.float32:
            out = out.astype(np.float32)
        if self.num_derived:
            der = eng.derived(xd).cpu().numpy()
            return (out[0], der[0]) if single else (out, der)
        return out[0] if single else out

    def loglike(self, x):
        return self(np.asarray(x))

    def sample(self, prior, num_samples):
        """Rejection sampling from the likelihood under `prior` (likelihoods.py:27-36)."""
        max_loglike = self.max_loglike
        samples = np.empty((0, self.x_dim))
        while samples.shape[0] < num_samples:
            x = prior.sample(num_samples)
            ratio = np.exp(self(x) - max_loglike)
            r = np.random.uniform(low=0, high=1, size=(num_samples,))
            samples = np.vstack((x[np.where(ratio > r)], samples))
        return samples[0:num_samples]

    def uniform_sample(self, prior, num_samples, fraction):
        """Best `num_samples` of num_samples/fraction prior draws and the likelihood of the worst kept
        (likelihoods.py:38-42)."""
        x = prior.sample(int(num_samples / fraction))
        loglike = self(x)
        idx = np.argsort(-loglike)
        return x[idx[0:num_samples]], loglike[idx[num_samples - 1]]


class Rosenbrock(Likelihood):
    like_id = L.NNB_LIKE_ROSENBROCK
    follows_input_dtype = True

    @property
    def max_loglike(self):
        return self(np.ones((self.x_dim,)))

    @property
    def sample_range(self):
        return [-2] * self.x_dim, [12] * self.x_dim


class Himmelblau(Likelihood):
    like_id = L.NNB_LIKE_HIMMELBLAU
    follows_input_dtype = True
    x_dim = 2

    def __init__(self, x_dim):
        assert self.x_dim == x_dim
        super(Himmelblau, self).__init__(x_dim)

    @property
    def max_loglike(self):
        return self([3.0, 2.0])


class Gaussian(Likelihood):
    like_id = L.NNB_LIKE_GAUSSIAN

    def __init__(self, x_dim, corr, lim=5):
        self.corr = corr
        self.lim = lim
        super(Gaussian, self).__init__(x_dim)

    def device_params(self):
        return [float(self.corr)]

    @property
    def max_loglike(self):
        return self([0.0] * self.x_dim)

    @property
    def sample_range(self):
        return [-self.lim] * self.x_dim, [self.lim] * self.x_dim


class Eggbox(Likelihood):
    """(2 + prod_i cos(x_i / 2))^5.  The reference asserts x_dim == 2 (likelihoods.py:97-106); the product
    over all dimensions is the generalisation used for the x_dim=10 configuration and is identical at d=2."""
    like_id = L.NNB_LIKE_EGGBOX
    follows_input_dtype = True

    def __init__(self, x_dim=2):
        super(Eggbox, self).__init__(x_dim)

    @property
    def max_loglike(self):
        return self([0.0] * self.x_dim)


class GaussianShell(Likelihood):
    like_id = L.NNB_LIKE_GAUSSIAN_SHELL

    def __init__(self, x_dim, sigma=0.1, rshell=2, center=0):
        self.sigma = sigma
        self.rshell = rshell
        if not hasattr(center, '__len__'):
            self.center = np.array([center] * x_dim)
        else:
            self.center = np.asarray(center)
        super(GaussianShell, self).__init__(x_dim)

    def device_params(self):
        return [float(self.sigma), float(self.rshell)] + [float(c) for c in self.center]

    @property
    def max_loglike(self):
        return self(self.center - np.array([self.rshell] + [0] * (self.x_dim - 1)))


class GaussianMix(Likelihood):
    like_id = L.NNB_LIKE_GAUSSIAN_MIX

    def __init__(self, x_dim, sep=4, weights=(0.4, 0.3, 0.2, 0.1), sigma=1):
        assert len(weights) in [2, 3, 4], ('Weights must have 2, 3 or 4 components. Weights=' + str(weights))
        assert np.isclose(sum(weights), 1), ('Weights must sum to 1! Weights=' + str(weights))
        self.sep = sep
        self.weights = weights
        self.sigma = sigma
        self.sigmas = [sigma] * len(weights)
        pos = [np.asarray([0, sep]), np.asarray([0, -sep]), np.asarray([sep, 0]), np.asarray([-sep, 0])]
        self.positions = pos[:len(weights)]
        super(GaussianMix, self).__init__(x_dim)

    def device_params(self):
        return [float(self.sep), float(self.sigma), float(len(self.weights))] + [float(w) for w in self.weights]

    @property
    def max_loglike(self):
        p = np.zeros(self.x_dim)
        p[:2] = self.positions[int(np.argmax(self.weights))]
        return self(p)


class CudaLikelihood(Likelihood):
    """A likelihood written in CUDA C++, compiled at run time (NVRTC) into the library's own MCMC step kernels.

    `source` defines

        template <typename X>
        __device__ double nnb_user_loglike(const X& x, int d, const double* params);

    where x(i) is coordinate i of the point after the sampler's affine transform -- a float when the target computes in
    float32 (float32 points, float32 transform), a double otherwise: `decltype(x(0))` names it -- and `params` holds the
    `params` given here (at most NNB_MAX_LIKE_PARAMS doubles).  A non-finite value is clamped as for the built-in
    likelihoods: to -inf when x(i) is a float, to -1e100 otherwise.

    Data -- observations, an inverse covariance, anything larger than `params` -- goes into `data`: an ordered mapping
    from name to array (at most NNB_MAX_DATA_ARRAYS of them).  The source reads array `name` as `nnb_data.name[j]` and
    its length as `nnb_data.name.size()`, from nnb_user_loglike and nnb_user_derived alike.  Names are C identifiers;
    each array keeps its dtype, which must be float64 (read as double), float32 (float) or int32 (int) -- convert other
    types on purpose, e.g. an int64 index array with .astype(np.int32).  Arrays are flattened in C order and copied
    here, so later changes to the caller's arrays change nothing; `data` holds the frozen copies.  Only the names and
    dtypes are compiled in: another CudaLikelihood with the same source and the same names and dtypes, but other values
    and sizes, reuses every compiled kernel, and switching between them costs one upload of the data to each device.
    A __constant__ array in the source still works for a small table of fixed constants, but constant memory holds
    64 KB, and a table written into the source makes every new table a new source to compile.

    num_derived > 0 (at most NNB_MAX_DERIVED): the source also defines

        template <typename X>
        __device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived);

    which writes derived[0 .. num_derived) at the point x -- the same x, in the same arithmetic type, as
    nnb_user_loglike sees there; helper functions can be shared between the two.  Derived values are returned as they are
    (no clamp), and they are not likelihood calls: the samplers evaluate them on the points they return, not on every
    proposal.  Calling the likelihood then returns (logl, derived), as a likelihood with derived parameters does in the
    reference.  Write float arithmetic with the *_rn intrinsics (__fadd_rn, __fmul_rn, ...) where
    the exact rounding matters: the compiler contracts a * b + c into one fused multiply-add otherwise.

    The source is compiled once here, without a device: a source that does not compile raises ValueError with the
    compiler's log.  Compiled kernels are cached on disk under $NNB_JIT_CACHE (default ~/.cache/nnest_b200/jit).
    """
    like_id = L.NNB_LIKE_USER

    def __init__(self, x_dim, source, params=(), data=None, max_loglike=None, num_derived=0):
        import ctypes as C
        params = [float(p) for p in np.asarray(params, dtype=np.float64).ravel()]
        if len(params) > L.NNB_MAX_LIKE_PARAMS:
            raise ValueError('CudaLikelihood takes at most %d params, got %d' % (L.NNB_MAX_LIKE_PARAMS, len(params)))
        if not isinstance(source, str):
            raise ValueError('source must be a string of CUDA C++')
        if int(num_derived) != num_derived or not 0 <= num_derived <= L.NNB_MAX_DERIVED:
            raise ValueError('num_derived must be an integer in [0, %d], got %r' % (L.NNB_MAX_DERIVED, num_derived))
        self._data = UserData(data) if data is not None and len(data) else None
        log = C.create_string_buffer(1 << 16)
        if self._data is None:
            rc = L.load().nnb_user_likelihood_check_derived(source.encode(), int(num_derived), log, len(log))
        else:
            names, dtypes = self._data.c_layout()
            rc = L.load().nnb_user_likelihood_check_data(source.encode(), int(num_derived), len(self._data.names),
                                                         names, dtypes, log, len(log))
        if rc == L.NNB_ERR_UNSUPPORTED:
            raise RuntimeError('CudaLikelihood needs NVRTC (libnvrtc.so.12), which could not be loaded')
        if rc != L.NNB_OK:
            raise ValueError('the likelihood source does not compile:\n' + log.value.decode(errors='replace'))
        self.source = source
        self.num_derived = int(num_derived)
        self.params = params
        self._max_loglike = max_loglike
        super(CudaLikelihood, self).__init__(x_dim)

    def device_params(self):
        return list(self.params)

    def device_source(self):
        return self.source

    def device_data(self):
        return self._data

    @property
    def data(self):
        """name -> the frozen flat copy of each dataset array ({} without data)"""
        return dict(zip(self._data.names, self._data.arrays)) if self._data is not None else {}

    @property
    def max_loglike(self):
        if self._max_loglike is None:
            raise AttributeError('max_loglike was not given to CudaLikelihood')
        return self._max_loglike


class UserData(object):
    """The dataset of a CudaLikelihood, frozen at construction: names, NNB_DTYPE_* codes and read-only flat copies of the
    arrays, with a token no other UserData has, so an engine uploads a given dataset at most once."""

    def __init__(self, data):
        items = list(data.items()) if hasattr(data, 'items') else list(data)
        if len(items) > L.NNB_MAX_DATA_ARRAYS:
            raise ValueError('CudaLikelihood takes at most %d data arrays, got %d' % (L.NNB_MAX_DATA_ARRAYS, len(items)))
        names, arrays = [], []
        for name, a in items:
            if not isinstance(name, str) or not re.match(r'^[A-Za-z_][A-Za-z0-9_]*\Z', name):
                raise ValueError('data array names must be C identifiers, got %r' % (name,))
            if name in names:
                raise ValueError('data array name %r is repeated' % name)
            a = np.asarray(a)
            if a.dtype not in DATA_DTYPES:
                raise ValueError('data array %r has dtype %s; the accepted dtypes are float64, float32 and int32 (convert '
                                 'others on purpose, e.g. .astype(np.int32))' % (name, a.dtype))
            a = np.array(a, order='C', copy=True).ravel()
            a.flags.writeable = False
            names.append(name)
            arrays.append(a)
        self.names, self.arrays = tuple(names), tuple(arrays)
        self.dtypes = tuple(DATA_DTYPES[a.dtype] for a in arrays)
        self.token = next(_data_tokens)

    @property
    def layout(self):
        """(name, NNB_DTYPE_*) per array: what the compiled kernels depend on"""
        return tuple(zip(self.names, self.dtypes))

    def c_layout(self):
        import ctypes as C
        n = len(self.names)
        return (C.c_char_p * n)(*[s.encode() for s in self.names]), (C.c_int * n)(*self.dtypes)


class CudaTransform(object):
    """A prior transform written in CUDA C++ -- the sampler's `transform`, from the unit box [-1, 1]^x_dim to the physical
    parameters -- compiled at run time (NVRTC) into the library's own kernels, next to the likelihood.

    `source` defines

        template <typename U>
        __device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0));

    which returns coordinate i of v = transform(u).  u(j) is coordinate j of the unit-box point, a float or a double
    (`decltype(u(0))` names it); any u(j) may be read, so transforms that mix coordinates (a Cholesky factor) are allowed.
    Nothing stores v: every x(i) a likelihood (built-in or CudaLikelihood), the prior or nnb_user_derived reads evaluates
    the transform once, so x(i) costs one transform evaluation per call -- a likelihood that reads a coordinate several
    times does well to keep it in a local variable.  `params` (at most NNB_MAX_LIKE_PARAMS doubles, and together with
    the likelihood's at most that many) reach the function as `params`; larger constants belong in the source as
    __constant__ arrays.  Write float arithmetic with the *_rn intrinsics where the exact rounding matters.

    float64=True (the default): float32 points are promoted to double before the transform, so the transform, the
    likelihood, the prior and the derived parameters all compute in double.  float64=False: the arithmetic follows the
    input, float for float32 points, as the float32 affine maps do.

    Calling the object maps host rows (n, x_dim) or (x_dim,) on the device: float64 out when float64=True or the input is
    float64, float32 otherwise (NumPy's dtype rules for the callable it replaces).  In a sampler the values are those the
    likelihood saw, bit for bit.  The source is compiled once here, without a device: a source that does not compile
    raises ValueError with the compiler's log.  Compiled kernels are cached as for CudaLikelihood.
    """

    def __init__(self, x_dim, source, params=(), float64=True):
        import ctypes as C
        params = [float(p) for p in np.asarray(params, dtype=np.float64).ravel()]
        if len(params) > L.NNB_MAX_LIKE_PARAMS:
            raise ValueError('CudaTransform takes at most %d params, got %d' % (L.NNB_MAX_LIKE_PARAMS, len(params)))
        if not isinstance(source, str) or not source.strip():
            raise ValueError('source must be a non-empty string of CUDA C++')
        log = C.create_string_buffer(1 << 16)
        rc = L.load().nnb_user_transform_check(source.encode(), log, len(log))
        if rc == L.NNB_ERR_UNSUPPORTED:
            raise RuntimeError('CudaTransform needs NVRTC (libnvrtc.so.12), which could not be loaded')
        if rc != L.NNB_OK:
            raise ValueError('the transform source does not compile:\n' + log.value.decode(errors='replace'))
        self.x_dim = int(x_dim)
        self.source = source
        self.params = params
        self.float64 = bool(float64)

    def install(self, engine, d, like_id, like_params=(), **target):
        """Select this transform on `engine`'s target (Engine.set_target with it in place of t_scale / t_shift)."""
        engine.set_target(d, like_id, like_params, compute_f64=self.float64, transform_source=self.source,
                          transform_params=self.params, **target)

    def apply(self, engine, u):
        """Host rows through `engine`, whose target already holds this transform -> host rows (see the class docs)."""
        import torch
        if isinstance(u, list):
            u = np.array(u)
        u = np.asarray(u)
        single = u.ndim == 1
        uu = np.ascontiguousarray(u[None, :] if single else u)
        if uu.dtype not in (np.float32, np.float64):
            uu = uu.astype(np.float64)
        if uu.ndim != 2 or uu.shape[1] != self.x_dim:
            raise ValueError('CudaTransform maps (n, %d) rows, got shape %s' % (self.x_dim, u.shape))
        v = engine.transform(torch.from_numpy(uu).to(engine.device)).cpu().numpy()
        if not self.float64 and uu.dtype == np.float32:
            v = v.astype(np.float32)
        return v[0] if single else v

    def __call__(self, u):
        eng = _eval_engine()
        self.install(eng, self.x_dim, L.NNB_LIKE_ROSENBROCK)
        return self.apply(eng, u)
