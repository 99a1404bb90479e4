// nnb_spline.cu -- the reference's DEFAULT flow, flow='spline' (SingleSpeedSpline: [ActNorm, Invertible1x1Conv, NSF_CL] x
// num_blocks, nnest/networks.py:393-705), on the device: batched flow maps, chain start and the fused MCMC step.
//
// Same contracts as flow_kernel / mcmc_init_kernel / mcmc_kernel (nnb_kernels.cuh; reference nnest/trainer.py:247-269,
// nnest/sampler.py:262-444) with the per-sample arithmetic of nnb_spline.cuh (pinned to reference goldens on the CPU).
// One chain per thread, 128 chains per CTA, chain vectors as shared-memory columns.  The parameters (46 k floats at
// d = 30, hidden 16: they do not fit next to the chain vectors) stay in global memory: every lane of a warp reads the
// same weight at the same time, i.e. one L1-resident broadcast line per load.
#include <cuda_runtime.h>

#include <string>

#include "nnb_host.h"
#include "nnb_spline_kernels.cuh"

using namespace nnb;

namespace {

spline::Shape shape_of(const nnb_handle* h) {
  spline::Shape sh;
  sh.d = h->spline_d; sh.H = h->spline_hidden; sh.blocks = h->spline_blocks; sh.K = h->spline_bins;
  sh.bound = h->spline_bound;
  return sh;
}

}  // namespace

extern "C" int nnb_set_flow_spline(nnb_handle* h, int d, int hidden, int num_blocks, int num_bins, double tail_bound,
                                   const float* packed, size_t n_floats) {
  if (!h) return NNB_ERR_ARG;
  if (d < 2 || d > NNB_MAX_DIM) return nnb_fail(h, NNB_ERR_ARG, "x_dim must be in [2, NNB_MAX_DIM]");
  if (hidden < 1 || hidden > spline::kMaxHidden) return nnb_fail(h, NNB_ERR_UNSUPPORTED, "hidden_dim must be <= 64");
  if (num_bins < 2 || num_bins > spline::kMaxBins) return nnb_fail(h, NNB_ERR_UNSUPPORTED, "num_bins must be in [2, 16]");
  if (num_blocks < 1 || num_blocks > NNB_MAX_BLOCKS) return nnb_fail(h, NNB_ERR_ARG, "num_blocks out of range");
  if (!(tail_bound > 0.0)) return nnb_fail(h, NNB_ERR_ARG, "tail_bound must be positive");
  spline::Shape sh;
  sh.d = d; sh.H = hidden; sh.blocks = num_blocks; sh.K = num_bins; sh.bound = (float)tail_bound;
  if (!packed || n_floats != (size_t)num_blocks * sh.block_floats())
    return nnb_fail(h, NNB_ERR_ARG, "parameter buffer size does not match (d, hidden, num_blocks, num_bins)");
  if (spline_smem_bytes(target_doubles(d, NNB_MAX_LIKE_PARAMS), d) > (size_t)h->max_smem)
    return nnb_fail(h, NNB_ERR_UNSUPPORTED, "x_dim too large for one CTA's shared memory");
  NNB_CUDA(h, cudaSetDevice(h->device));
  NNB_CUDA(h, nnb_reserve(&h->d_weights_spline, &h->weights_spline_cap, n_floats));
  NNB_CUDA(h, cudaMemcpy(h->d_weights_spline, packed, n_floats * sizeof(float), cudaMemcpyHostToDevice));
  h->spline_d = d; h->spline_hidden = hidden; h->spline_blocks = num_blocks; h->spline_bins = num_bins;
  h->spline_bound = (float)tail_bound;
  h->flow_is_spline = true;
  h->has_flow = true;
  h->flow.d = d;            // x_dim checks of the MCMC entry points
  h->tc_ok = false;
  h->warp_ok = false;
  return NNB_OK;
}

int nnb_spline_flow(nnb_handle* h, bool inverse, const float* in, int64_t irs, int64_t ics, float* out, int64_t ors,
                    int64_t ocs, float* logdet, int* empty_out, int64_t n, cudaStream_t st) {
  const spline::Shape sh = shape_of(h);
  const size_t sm = spline_smem_bytes(0, sh.d);
  const int grid = nnb_grid_for(h, n, 4);
  if (inverse) {
    NNB_CUDA(h, nnb_set_smem(spline_flow_kernel<true>, sm));
    spline_flow_kernel<true><<<grid, kBlockThreads, sm, st>>>(sh, h->d_weights_spline, in, irs, ics, out, ors, ocs, logdet,
                                                              empty_out, n);
  } else {
    NNB_CUDA(h, nnb_set_smem(spline_flow_kernel<false>, sm));
    spline_flow_kernel<false><<<grid, kBlockThreads, sm, st>>>(sh, h->d_weights_spline, in, irs, ics, out, ors, ocs, logdet,
                                                               empty_out, n);
  }
  NNB_CUDA(h, cudaGetLastError());
  return NNB_OK;
}

int nnb_spline_init(nnb_handle* h, const InitParams& p, cudaStream_t st) {
  const spline::Shape sh = shape_of(h);
  int rc = NNB_OK;
  const void* fn = nnb_kernel(h, (const void*)spline_init_kernel, &rc, "spline_init_kernel");
  if (!fn) return rc;
  const size_t sm = spline_smem_bytes(target_doubles(h->tdesc.d, h->tdesc.n_params), sh.d);
  NNB_CUDA(h, nnb_set_smem(fn, sm));
  const int grid = (int)((p.n + kBlockThreads - 1) / kBlockThreads);
  void* args[] = {(void*)&sh, (void*)&h->d_weights_spline, (void*)&h->tdesc, (void*)&h->d_target, (void*)&p};
  NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(kBlockThreads), args, sm, st));
  return NNB_OK;
}

template <int MODE>
static int spline_mcmc_mode(nnb_handle* h, McmcParams p, int steps, cudaStream_t st) {
  const spline::Shape sh = shape_of(h);
  int rc = NNB_OK;
  const void* fn = nnb_kernel(h, (const void*)spline_mcmc_kernel<MODE>, &rc, "spline_mcmc_kernel<%d>", MODE);
  if (!fn) return rc;
  const size_t sm = spline_smem_bytes(target_doubles(h->tdesc.d, h->tdesc.n_params), sh.d);
  NNB_CUDA(h, nnb_set_smem(fn, sm));
  const int grid = (int)((p.n + kBlockThreads - 1) / kBlockThreads);
  void* args[] = {(void*)&sh, (void*)&h->d_weights_spline, (void*)&h->tdesc, (void*)&h->d_target, (void*)&p};
  if (p.dynamic) {
    for (int s = 0; s < steps; ++s) {
      p.s0 = s; p.nsteps = 1;
      NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(kBlockThreads), args, sm, st));
    }
  } else {
    p.s0 = 0; p.nsteps = steps;
    NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(kBlockThreads), args, sm, st));
  }
  h->last_launches = p.dynamic ? steps : 1;
  return NNB_OK;
}

int nnb_spline_mcmc(nnb_handle* h, McmcParams p, int steps, cudaStream_t st) {
  return p.mode == NNB_MODE_MH ? spline_mcmc_mode<NNB_MODE_MH>(h, p, steps, st)
                               : spline_mcmc_mode<NNB_MODE_HARD>(h, p, steps, st);
}

extern "C" int nnb_flow_empty_halves(nnb_handle* h, const float* z, int64_t z_rs, int64_t z_cs, int inverse, int* flags,
                                     int64_t n, void* stream) {
  if (!h || !flags || (n > 0 && !z) || n < 0) return NNB_ERR_ARG;
  if (!h->has_flow) return nnb_fail(h, NNB_ERR_STATE, "no flow set");
  NNB_CUDA(h, cudaSetDevice(h->device));
  if (!h->flow_is_spline) {   // affine coupling layers are defined everywhere
    NNB_CUDA(h, cudaMemsetAsync(flags, 0, sizeof(int) * n, (cudaStream_t)stream));
    return NNB_OK;
  }
  if (n == 0) return NNB_OK;
  // scratch output: the flags come from a full evaluation of the map
  float* scratch = nullptr;
  NNB_CUDA(h, cudaMallocAsync(&scratch, sizeof(float) * (size_t)n * h->spline_d, (cudaStream_t)stream));
  int rc = nnb_spline_flow(h, inverse != 0, z, z_rs, z_cs, scratch, h->spline_d, 1, nullptr, flags, n, (cudaStream_t)stream);
  cudaFreeAsync(scratch, (cudaStream_t)stream);
  return rc;
}
