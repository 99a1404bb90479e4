"""CUDA C++ sources of user prior transforms (nnest_b200.likelihoods.CudaTransform) and their NumPy restatements, shared
by the user-transform tests.

AFFINE restates the built-in affine map u * scale + shift operation for operation (float32 rows against the scale and
shift rounded to float32, as the built-in map does), so every value and chain it drives must equal the built-in target
bit for bit.  params = scale[d], shift[d]."""
import numpy as np

AFFINE = r'''
__device__ __forceinline__ float aff(float u, double s, double b) { return __fadd_rn(__fmul_rn(u, (float)s), (float)b); }
__device__ __forceinline__ double aff(double u, double s, double b) { return __dadd_rn(__dmul_rn(u, s), b); }
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  return aff(u(i), params[i], params[d + i]);
}
'''

# N(0, params[0]^2) in every coordinate from u in (-1, 1): the inverse CDF sigma * sqrt(2) * erfinv(u)
GAUSS = r'''
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  return params[0] * 1.4142135623730951 * erfinv(u(i));
}
'''

# log-uniform on [exp(params[0]), exp(params[1])]: v = exp(a + (u + 1) / 2 * (b - a))
LOGUNIFORM = r'''
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  return exp(params[0] + 0.5 * ((double)u(i) + 1.0) * (params[1] - params[0]));
}
'''

# correlated Gaussian N(0, L L^T): v = L z, z_j = sqrt(2) erfinv(u_j), L lower triangular (params: d x d row-major)
CHOLESKY = r'''
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  double v = 0.0;
  for (int j = 0; j <= i; ++j) v += params[i * d + j] * (1.4142135623730951 * erfinv((double)u(j)));
  return v;
}
'''

SYNTAX_ERROR = r'''
template <typename U>
__device__ auto nnb_user_transform(const U& u, int i, int d, const double* params) -> decltype(u(0)) {
  return u(i) * 2   // missing semicolon
}
'''

MISSING = r'''
__device__ double some_other_name(double v) { return 2.0 * v; }
'''


def gauss_np(u, sigma):
    from scipy.special import erfinv
    return sigma * np.sqrt(2.0) * erfinv(np.asarray(u, dtype=np.float64))


def loguniform_np(u, a, b):
    return np.exp(a + 0.5 * (np.asarray(u, dtype=np.float64) + 1.0) * (b - a))


def cholesky_np(u, chol):
    from scipy.special import erfinv
    z = np.sqrt(2.0) * erfinv(np.asarray(u, dtype=np.float64))
    return z @ np.asarray(chol).T


# a 3-d prior covariance and its Cholesky factor
SIGMA_P = np.array([[4.0, 1.2, -0.8], [1.2, 2.25, 0.6], [-0.8, 0.6, 1.0]])
CHOL_P = np.linalg.cholesky(SIGMA_P)
