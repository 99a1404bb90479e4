// nnb_tc_launch.cuh -- launch logic of the tensor-core MCMC kernel, shared by the generic translation unit (nnb_tc.cu)
// and the per-dimension specialisations (nnb_tc_d*.cu: x_dim fixed at compile time, num_layers = 1, num_blocks = 3).
#pragma once
#include <cstdio>
#include <cstdlib>

#include "nnb_host.h"
#include "nnb_tc_kernels.cuh"

namespace nnb {

template <int MODE, int NPART, int DD>
static int launch_tc_mode(nnb_handle* h, McmcParams p, int steps, cudaStream_t st) {
  const int tdoubles = target_doubles(h->tdesc.d, h->tdesc.n_params);
  // kernel-parameter constants: the flow's biases (filled by nnb_tc_pack) + the target's float32 mirrors.  All parameters
  // together stay below 4 KB: larger parameter blocks take a slow launch path in the driver (measured with a 5 KB
  // block: +1.4 ms per cooperative launch).
  static_assert(sizeof(TcFlowDesc) + sizeof(TargetDesc) + sizeof(McmcParams) + sizeof(TcConsts) + 2 * sizeof(void*) + 32 <= 4096,
                "kernel parameters of mcmc_tc_kernel exceed 4 KB");
  int rc = NNB_OK;
  const void* fn = nnb_kernel(h, (const void*)mcmc_tc_kernel<MODE, NPART, DD>, &rc, "nnb::mcmc_tc_kernel<%d, %d, %d>", MODE,
                              NPART, DD);
  if (!fn) return rc;
  TcConsts cst = h->tc_consts;
  {
    const int d = h->tcflow.d, t0 = tc_cb_off(d, h->tcflow.L, h->tcflow.B);
    if ((int)h->target_f32.size() != 4 * d) return nnb_fail(h, NNB_ERR_STATE, "target float32 mirrors missing");
    for (int i = 0; i < 4 * d; ++i) cst.v[t0 + i] = h->target_f32[i];
  }
  // chains per CTA: spread the batch evenly over all SMs in units of a warp (32 chains), at most 4 tiles of 128
  long long cpc = ((p.n + h->sm_count - 1) / h->sm_count + 31) / 32 * 32;
  if (cpc > 128 * kTcMaxTiles) cpc = 128 * kTcMaxTiles;
  if (cpc < 32) cpc = 32;
  int ntiles = (int)((cpc + 127) / 128);
  while (ntiles > 1 && tc_smem_bytes(h->tcflow, tdoubles, ntiles, NPART) > (size_t)h->max_smem) {
    --ntiles;
    cpc = 128 * ntiles;
  }
  size_t sm = tc_smem_bytes(h->tcflow, tdoubles, ntiles, NPART);
  const size_t one_cta_per_sm = 116 * 1024;   // TMEM is allocated per CTA: keep a single CTA resident per SM
  if (sm < one_cta_per_sm) sm = one_cta_per_sm;
  NNB_CUDA(h, nnb_set_smem(fn, sm));
  const int grid = (int)((p.n + cpc - 1) / cpc);
  const int block = ntiles * 128 * NPART;   // fixed warp slots; a partial last tile leaves some idle
  p.cpc = (int)cpc;
  static const int jc_env = [] { const char* e = getenv("NNB_TC_JC"); return e ? atoi(e) : -1; }();
  p.tc_jc = jc_env;
  // start delays of the four tile slots (cycles): NNB_TC_DELAYS="d0,d1,d2,d3"; default: odd slots half a round trip late
  // (sweep on the B200 at c4: 0,700,0,700 and 0,600,0,600 best; four distinct phases or no delay are 1 - 7 % slower)
  struct Delays { int v[4]; };
  static const Delays delays_env = [] {
    Delays dl{{0, 700, 0, 700}};
    if (const char* e = getenv("NNB_TC_DELAYS")) sscanf(e, "%d,%d,%d,%d", &dl.v[0], &dl.v[1], &dl.v[2], &dl.v[3]);
    return dl;
  }();
  for (int j = 0; j < 4; ++j) p.tc_delay[j] = ntiles > 1 ? delays_env.v[j] : 0;
  // Persistent path: all steps in ONE cooperative launch (every CTA resident, one per SM), the global accept count
  // of each step travels through a grid barrier.  Needs grid <= SM count; otherwise one launch per step.
  void* args[] = {(void*)&h->tcflow, (void*)&h->d_weights_tc, (void*)&h->tdesc, (void*)&h->d_target, (void*)&p, (void*)&cst};
  static const bool no_coop = getenv("NNB_NO_COOP") != nullptr;
  if (!no_coop && p.dynamic && h->coop_supported && grid <= h->sm_count && steps > 1) {
    if (h->step_counts_cap < steps) {
      if (h->d_step_counts) cudaFree(h->d_step_counts);
      h->d_step_counts = nullptr;
      NNB_CUDA(h, cudaMalloc(&h->d_step_counts, sizeof(unsigned long long) * steps));
      h->step_counts_cap = steps;
    }
    NNB_CUDA(h, cudaMemsetAsync(h->d_step_counts, 0, sizeof(unsigned long long) * steps, st));
    p.s0 = 0; p.nsteps = steps; p.coop = 1; p.step_counts = h->d_step_counts;
    long long tiles = 0;   // tiles holding at least one chain
    for (int b = 0; b < grid; ++b) {
      const long long left = p.n - (long long)b * cpc;
      const long long mine = left < cpc ? left : cpc;
      tiles += (mine + 127) / 128;
    }
    p.total_tiles = (int)tiles;
    NNB_CUDA(h, cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(block), args, sm, st));
    h->last_launches = 1;
    return NNB_OK;
  }
  p.coop = 0; p.step_counts = nullptr;
  if (p.dynamic) {
    for (int s = 0; s < steps; ++s) {
      p.s0 = s; p.nsteps = 1;
      NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(block), args, sm, st));
    }
  } else {
    p.s0 = 0; p.nsteps = steps;
    NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(block), args, sm, st));
  }
  h->last_launches = p.dynamic ? steps : 1;
  return NNB_OK;
}


}  // namespace nnb

// x_dim-specialised launchers (one translation unit each so that they compile in parallel)
template <int DD>
int nnb_launch_mcmc_tc_fixed(nnb_handle* h, McmcParams p, int steps, cudaStream_t st, int npart);
