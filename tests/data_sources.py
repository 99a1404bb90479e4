"""CUDA C++ sources of user likelihoods that read a dataset (CudaLikelihood(data=...)), their NumPy restatements and the
closed forms they are checked against; shared by the dataset tests and scripts/user_data_bench.py."""
import re

import numpy as np

import user_sources as us

# chi-square of a straight line y = a + b t over the points whose mask is not 0: t, y float64, w = 1 / sigma^2 float32,
# mask int32; x = (a, b).  Derived: chi^2 / N, the model at t[0], and x(0), x(1) as the likelihood saw them.
LINE_BODY = r'''
__device__ double line_chi2(double a, double b) {
  double chi2 = 0.0;
  const long long n = DATA_N;
  for (long long j = 0; j < n; ++j) {
    if (DATA_MASK(j) != 0) {
      const double r = DATA_Y(j) - (a + b * DATA_T(j));
      chi2 += r * r * (double)DATA_W(j);
    }
  }
  return chi2;
}
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  return -0.5 * line_chi2((double)x(0), (double)x(1));
}
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  const double a = (double)x(0), b = (double)x(1);
  derived[0] = line_chi2(a, b) / (double)DATA_N;
  derived[1] = a + b * DATA_T(0);
  derived[2] = a;
  derived[3] = b;
}
'''
LINE_DERIVED = 4

LINE = r'''
#define DATA_N nnb_data.y.size()
#define DATA_T(j) nnb_data.t[j]
#define DATA_Y(j) nnb_data.y[j]
#define DATA_W(j) nnb_data.w[j]
#define DATA_MASK(j) nnb_data.mask[j]
''' + LINE_BODY


def line_baked_source(data):
    """LINE with the dataset written into the source as __constant__ arrays (at most 64 KB of them)"""
    n = len(data['t'])
    f = lambda a: ',\n'.join(', '.join('%.17g' % v for v in a[i:i + 8]) for i in range(0, n, 8))
    return r'''
__constant__ double kT[%d] = {%s};
__constant__ double kY[%d] = {%s};
__constant__ float kW[%d] = {%s};
__constant__ int kMask[%d] = {%s};
#define DATA_N %dLL
#define DATA_T(j) kT[j]
#define DATA_Y(j) kY[j]
#define DATA_W(j) kW[j]
#define DATA_MASK(j) kMask[j]
''' % (n, f(data['t']), n, f(data['y']), n, f(data['w'].astype(np.float64)), n,
       ',\n'.join(', '.join('%d' % v for v in data['mask'][i:i + 8]) for i in range(0, n, 8)), n) + LINE_BODY


def line_data(n, seed=0, a=0.7, b=-1.3):
    """n points of a noisy straight line: t, y float64, w = 1 / sigma^2 float32, mask int32 (about 10 % masked out)"""
    rng = np.random.RandomState(seed)
    t = np.sort(rng.uniform(-2.0, 2.0, n))
    sigma = rng.uniform(0.05, 0.2, n)
    y = a + b * t + rng.normal(size=n) * sigma
    return dict(t=t, y=y, w=(1.0 / sigma ** 2).astype(np.float32),
                mask=(rng.uniform(size=n) > 0.1).astype(np.int32))


def line_chi2_np(a, b, data, chunk=64):
    """chi^2 of each row (a[k], b[k]) in float64, summed over the points in order, as the kernel sums"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    keep = data['mask'] != 0
    t, y, w = data['t'][keep], data['y'][keep], data['w'][keep].astype(np.float64)
    out = np.zeros(len(a))
    if not len(t):
        return out
    for s in range(0, len(a), chunk):
        r = y[None, :] - (a[s:s + chunk, None] + b[s:s + chunk, None] * t[None, :])
        out[s:s + chunk] = np.cumsum(r * r * w[None, :], axis=1)[:, -1]
    return out


def line_derived_np(a, b, data):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.stack([line_chi2_np(a, b, data) / len(data['t']), a + b * data['t'][0], a, b], axis=1)


def gauss_data_source(d):
    """us.gauss_full_source with the same arithmetic, reading the precision matrix from the dataset array `prec` (float64,
    d * d, row-major) instead of a __constant__ array in the source"""
    src = us.gauss_full_source(np.eye(d))
    src = re.sub(r'__constant__ double kPrec\[\d+\] = \{.*?\};\n', '', src, flags=re.S)
    assert 'kPrec[' in src and '__constant__' not in src
    return src.replace('kPrec[', 'nnb_data.prec[')


# quadratic regression y = c0 + c1 t + c2 t^2 with noise of known variance 1 / params[0]; x = (c0, c1, c2); params[1] is a
# constant added to the log-likelihood (keeps its maximum near 0).  Derived: chi^2 / N and the model at t[0].
POLY = r'''
__device__ double poly_chi2(double c0, double c1, double c2) {
  double chi2 = 0.0;
  for (long long j = 0; j < nnb_data.y.size(); ++j) {
    const double t = nnb_data.t[j];
    const double r = nnb_data.y[j] - (c0 + t * (c1 + t * c2));
    chi2 += r * r;
  }
  return chi2;
}
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  return -0.5 * params[0] * poly_chi2((double)x(0), (double)x(1), (double)x(2)) + params[1];
}
template <typename X>
__device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived) {
  const double c0 = (double)x(0), c1 = (double)x(1), c2 = (double)x(2);
  derived[0] = poly_chi2(c0, c1, c2) / (double)nnb_data.y.size();
  const double t = nnb_data.t[0];
  derived[1] = c0 + t * (c1 + t * c2);
}
'''
POLY_TRUTH = np.array([0.4, -0.8, 1.5])


def poly_data(n=20000, sigma=1.0, seed=0):
    rng = np.random.RandomState(seed)
    t = rng.uniform(-1.0, 1.0, n)
    y = POLY_TRUTH[0] + t * (POLY_TRUTH[1] + t * POLY_TRUTH[2]) + rng.normal(size=n) * sigma
    return dict(t=t, y=y)


def poly_design(t):
    return np.stack([np.ones_like(t), t, t * t], axis=1)


def poly_params(data, sigma=1.0):
    """params of POLY: 1 / sigma^2 and the offset 0.5 chi^2_min / sigma^2"""
    phi = poly_design(data['t'])
    coef = np.linalg.lstsq(phi, data['y'], rcond=None)[0]
    r = data['y'] - phi @ coef
    return [1.0 / sigma ** 2, 0.5 * float(r @ r) / sigma ** 2]


def poly_derived_np(c, data):
    c = np.asarray(c, dtype=np.float64).reshape(-1, 3)
    r = data['y'][None, :] - (c[:, :1] + data['t'][None, :] * (c[:, 1:2] + data['t'][None, :] * c[:, 2:3]))
    t0 = data['t'][0]
    return np.stack([np.sum(r * r, axis=1) / len(data['t']), c[:, 0] + t0 * (c[:, 1] + t0 * c[:, 2])], axis=1)


def poly_closed_form(data, params, prior_cov=None, box=None):
    """log-evidence, posterior mean and covariance of POLY (a linear-Gaussian model) under the Gaussian prior
    N(0, prior_cov) or the uniform prior on the box [-box, box]^3 (wide enough to hold the whole posterior)"""
    w, offset = params
    phi = poly_design(data['t'])
    y = data['y']
    A = w * phi.T @ phi
    bvec = w * phi.T @ y
    c = -0.5 * w * float(y @ y) + offset
    if prior_cov is not None:
        M = A + np.linalg.inv(prior_cov)
        mean = np.linalg.solve(M, bvec)
        logz = c + 0.5 * bvec @ mean - 0.5 * np.linalg.slogdet(prior_cov)[1] - 0.5 * np.linalg.slogdet(M)[1]
        return logz, mean, np.linalg.inv(M)
    mean = np.linalg.solve(A, bvec)
    logz = c + 0.5 * bvec @ mean + 1.5 * np.log(2 * np.pi) - 0.5 * np.linalg.slogdet(A)[1] - 3 * np.log(2.0 * box)
    return logz, mean, np.linalg.inv(A)
