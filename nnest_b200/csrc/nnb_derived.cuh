// nnb_derived.cuh -- derived parameters of a user likelihood (nnb_derived, nnb_derived_trace in include/nnb.h).
//
// The user's source defines, next to nnb_user_loglike,
//     template <typename X> __device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived);
// Only the run-time build compiles these kernels (nnb_jit.cu defines NNB_USER_DERIVED when the likelihood has derived
// parameters): the ahead-of-time library holds none of them.  A derived value is a function of the point alone, so it is
// evaluated on the points the samplers return, never on the proposals: the step kernels are untouched.  x(i) is the same
// Transformed<T, XG> accessor in the same arithmetic type that loglike_any gives nnb_user_loglike, so at a point of a
// trace the function sees the bits the step kernel's likelihood saw.
#pragma once
#include "nnb_kernels.cuh"

#ifdef NNB_USER_DERIVED

// derived[0 .. n_der) of the row xg, in float when the likelihood at this point runs in float32, in double otherwise
template <typename XG>
__device__ __forceinline__ void derived_any(const TargetSmem& tg, const XG& xg, bool in_f64, double* der) {
  if (tg.desc.compute_f64 || in_f64) {
    Transformed<double, XG> v{tg, xg};
    nnb_user_derived(v, tg.desc.d, tg.params, der);
  } else {
    Transformed<float, XG> v{tg, xg};
    nnb_user_derived(v, tg.desc.d, tg.params, der);
  }
}

// rows u[c * rs + i * cs] (float32 or float64) -> out[c * n_der + j], as loglike_kernel reads them
template <typename TIN>
__global__ void __launch_bounds__(kBlockThreads)
derived_kernel(TargetDesc td, const double* __restrict__ tgt_g, const TIN* __restrict__ u, long long rs, long long cs,
               double* __restrict__ out, long long n, int n_der) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, 0, td, tgt_g, td.d, 0);
  __syncthreads();
  const long long ntiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long c = tile * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    double der[NNB_MAX_DERIVED];
    for (int j = 0; j < n_der; ++j) der[j] = __longlong_as_double(0x7ff8000000000000LL);   // unwritten: NaN
    GlobalRow<TIN> row{u + c * rs, cs};
    derived_any(sv.tg, row, sizeof(TIN) == 8, der);
    for (int j = 0; j < n_der; ++j) out[c * n_der + j] = der[j];
  }
}

// Rows t_k = row0 + k * row_step (k < n_rows) of the chain-minor float32 trace (T, d, n) nnb_mcmc_run writes ->
// out (n_rows, n_der, n) float64.  With init (n_der, n) a chain whose point at t_k is bit-equal to its row-0 point in every
// coordinate takes init's values (it has not moved since the start, whose values the caller supplied).  One thread per
// (row, chain): loads and stores are coalesced across the chains of a warp.
__global__ void __launch_bounds__(kBlockThreads)
derived_trace_kernel(TargetDesc td, const double* __restrict__ tgt_g, const float* __restrict__ trace, long long n,
                     long long row0, long long row_step, long long n_rows, const double* __restrict__ init,
                     double* __restrict__ out, int n_der) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, 0, td, tgt_g, td.d, 0);
  __syncthreads();
  const int d = td.d;
  const long long ctiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ctiles * n_rows; tile += gridDim.x) {
    const long long k = tile / ctiles;
    const long long c = (tile - k * ctiles) * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    const float* x = trace + (row0 + k * row_step) * d * n + c;
    double* o = out + k * n_der * n + c;
    bool moved = true;
    if (init) {
      moved = false;
      for (int i = 0; i < d; ++i) moved |= __float_as_uint(x[(long long)i * n]) != __float_as_uint(trace[(long long)i * n + c]);
    }
    if (!moved) {
      for (int j = 0; j < n_der; ++j) o[(long long)j * n] = init[(long long)j * n + c];
      continue;
    }
    double der[NNB_MAX_DERIVED];
    for (int j = 0; j < n_der; ++j) der[j] = __longlong_as_double(0x7ff8000000000000LL);
    GlobalRow<float> row{x, n};
    derived_any(sv.tg, row, false, der);
    for (int j = 0; j < n_der; ++j) o[(long long)j * n] = der[j];
  }
}

#endif  // NNB_USER_DERIVED
