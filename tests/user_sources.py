"""CUDA C++ sources of user likelihoods (nnest_b200.likelihoods.CudaLikelihood) shared by the user-likelihood tests.

ROSENBROCK, HIMMELBLAU and EGGBOX restate the built-in likelihoods operation for operation (the *_rn intrinsics in the
type of x(i)), so their values and every chain they drive must equal the built-in ones bit for bit."""

# overloads of the rounded arithmetic for float and double coordinates
_RN = r'''
__device__ __forceinline__ float u_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double u_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float u_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double u_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float u_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double u_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float u_cos(float a) { return cosf(a); }
__device__ __forceinline__ double u_cos(double a) { return cos(a); }
'''

ROSENBROCK = _RN + r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  typedef decltype(x(0)) T;
  T acc = (T)0;
  T prev = x(0);
  for (int i = 1; i < d; ++i) {
    const T cur = x(i);
    const T t1 = u_sub(cur, u_mul(prev, prev));
    const T t2 = u_sub((T)1, prev);
    acc = u_add(acc, u_add(u_mul((T)100, u_mul(t1, t1)), u_mul(t2, t2)));
    prev = cur;
  }
  return -(double)acc;
}
'''

HIMMELBLAU = _RN + r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  typedef decltype(x(0)) T;
  const T x0 = x(0), x1 = x(1);
  const T a = u_sub(u_add(u_mul(x0, x0), x1), (T)11);
  const T b = u_sub(u_add(x0, u_mul(x1, x1)), (T)7);
  return (double)u_sub(-u_mul(a, a), u_mul(b, b));
}
'''

EGGBOX = _RN + r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  typedef decltype(x(0)) T;
  T chi = u_cos(x(0) / (T)2);
  for (int i = 1; i < d; ++i) chi = u_mul(chi, u_cos(x(i) / (T)2));
  const T b = u_add((T)2, chi);
  const T b2 = u_mul(b, b);
  return (double)u_mul(u_mul(b2, b2), b);
}
'''

# Gaussian shell (likelihoods.py GaussianShell): params = sigma, rshell, center[d]
SHELL = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  double s = 0.0;
  for (int i = 0; i < d; ++i) {
    const double t = params[2 + i] - (double)x(i);
    s += t * t;
  }
  const double r = sqrt(s) - params[1];
  return -(r * r) / (2.0 * params[0] * params[0]);
}
'''


def gauss_full_source(prec):
    """log N(x; mu, C) with the precision matrix C^-1 (d x d) in __constant__ memory and params = mu[d], log-normaliser."""
    d = prec.shape[0]
    vals = ',\n'.join(', '.join('%.17g' % v for v in row) for row in prec)
    return r'''
__constant__ double kPrec[%d] = {
%s};
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  double dx[%d];
  for (int i = 0; i < %d; ++i) dx[i] = (double)x(i) - params[i];
  double q = 0.0;
  for (int i = 0; i < %d; ++i) {
    double r = 0.0;
    for (int j = 0; j < %d; ++j) r += kPrec[i * %d + j] * dx[j];
    q += dx[i] * r;
  }
  return -0.5 * q + params[%d];
}
''' % (d * d, vals, d, d, d, d, d, d)


SYNTAX_ERROR = r'''
template <typename X>
__device__ double nnb_user_loglike(const X& x, int d, const double* params) {
  return -(double)x(0) * x(0)   // missing semicolon
}
'''

MISSING = r'''
__device__ double some_other_name(double v) { return -v * v; }
'''
