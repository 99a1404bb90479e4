// nnb_transform.cuh -- values of a user transform on the host's rows (nnb_transform, nnb_transform_trace in
// include/nnb.h).
//
// The user's source defines
//     template <typename U> __device__ auto nnb_user_transform(const U& u, int i, int d, const double* params)
//         -> decltype(u(0));
// which returns coordinate i of v = transform(u).  Only the run-time build compiles these kernels (nnb_jit.cu defines
// NNB_USER_TRANSFORM and, for the module that holds them, NNB_TRANSFORM_ROWS): the ahead-of-time library holds none of
// them.  v(i) is the Transformed<T, XG> accessor in the arithmetic type loglike_any picks, so the values written here are
// the bits the likelihood, the prior and the derived parameters see at the same point.
#pragma once
#include "nnb_kernels.cuh"

#if defined(NNB_USER_TRANSFORM) && defined(NNB_TRANSFORM_ROWS)

// v of the row xg -> o[i * os], i < d, in float when the likelihood at this point runs in float32, in double otherwise
template <typename XG>
__device__ __forceinline__ void transform_any(const TargetSmem& tg, const XG& xg, bool in_f64, double* o, long long os) {
  const int d = tg.desc.d;
  if (tg.desc.compute_f64 || in_f64) {
    Transformed<double, XG> v{tg, xg};
    for (int i = 0; i < d; ++i) o[i * os] = v(i);
  } else {
    Transformed<float, XG> v{tg, xg};
    for (int i = 0; i < d; ++i) o[i * os] = (double)v(i);
  }
}

// rows u[c * rs + i * cs] (float32 or float64) -> out[c * d + i], as loglike_kernel reads them
template <typename TIN>
__global__ void __launch_bounds__(kBlockThreads)
transform_kernel(TargetDesc td, const double* __restrict__ tgt_g, const TIN* __restrict__ u, long long rs, long long cs,
                 double* __restrict__ out, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, 0, td, tgt_g, td.d, 0);
  __syncthreads();
  const long long ntiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long c = tile * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    GlobalRow<TIN> row{u + c * rs, cs};
    transform_any(sv.tg, row, sizeof(TIN) == 8, out + c * td.d, 1);
  }
}

// Rows t_k = row0 + k * row_step (k < n_rows) of the chain-minor float32 trace (T, d, n) nnb_mcmc_run writes ->
// out (n_rows, d, n) float64.  One thread per (row, chain): loads and stores are coalesced across the chains of a warp.
__global__ void __launch_bounds__(kBlockThreads)
transform_trace_kernel(TargetDesc td, const double* __restrict__ tgt_g, const float* __restrict__ trace, long long n,
                       long long row0, long long row_step, long long n_rows, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, 0, td, tgt_g, td.d, 0);
  __syncthreads();
  const int d = td.d;
  const long long ctiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ctiles * n_rows; tile += gridDim.x) {
    const long long k = tile / ctiles;
    const long long c = (tile - k * ctiles) * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    GlobalRow<float> row{trace + (row0 + k * row_step) * d * n + c, n};
    transform_any(sv.tg, row, false, out + k * d * n + c, n);
  }
}

#endif  // NNB_USER_TRANSFORM && NNB_TRANSFORM_ROWS
