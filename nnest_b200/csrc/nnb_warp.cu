// nnb_warp.cu -- host side of the 16-lanes-per-chain MCMC kernel (nnb_warp.cuh): weight packing and launch.
#include <cstdlib>
#include <vector>

#include "nnb_host.h"
#include "nnb_warp.cuh"

using namespace nnb;

// natural (state_dict) order -> per block { W1 | b1 | L x (W2 b2) | W3 | b3 }, (scale, translate) pairs interleaved
int nnb_warp_pack(nnb_handle* h, const float* weights) {
  const FlowDesc& f = h->flow;
  h->warp_ok = false;
  if (!warp_supported(f)) return NNB_OK;
  const int d = f.d, H = 16, L = f.L, B = f.B;
  WarpFlowDesc w{};
  w.d = d; w.L = L; w.B = B;
  int off = 0;
  for (int k = 0; k < B; ++k) { w.off[k] = off; off += warp_block_floats(d, L, k); }
  w.total_floats = off;
  std::vector<float> buf((size_t)off, 0.f);
  const size_t net_nat = (size_t)H * d + H + (size_t)L * (H * H + H) + (size_t)d * H + d;
  for (int k = 0; k < B; ++k) {
    const int nin = blk_nin(d, k), i0 = blk_i0(k), nout = blk_nout(d, k), o0 = blk_o0(k);
    const int NO = warp_round16(nout);
    const float* net[2] = {weights + (size_t)(2 * k) * net_nat, weights + (size_t)(2 * k + 1) * net_nat};
    float* o = buf.data() + w.off[k];
    for (int s = 0; s < 2; ++s) {
      const float* W1 = net[s];
      const float* b1 = W1 + (size_t)H * d;
      for (int a = 0; a < nin; ++a)
        for (int j = 0; j < H; ++j) o[2 * (a * 16 + j) + s] = W1[(size_t)j * d + (i0 + 2 * a)];
      for (int j = 0; j < H; ++j) o[2 * (nin * 16 + j) + s] = b1[j];
    }
    o += 32 * nin + 32;
    size_t nat = (size_t)H * d + H;
    for (int l = 0; l < L; ++l) {
      for (int s = 0; s < 2; ++s) {
        const float* W2 = net[s] + nat;            // (H, H) [j][k]
        const float* b2 = W2 + (size_t)H * H;
        for (int kk = 0; kk < H; ++kk)
          for (int j = 0; j < H; ++j) o[2 * (kk * 16 + j) + s] = W2[(size_t)j * H + kk];
        for (int j = 0; j < H; ++j) o[2 * (256 + j) + s] = b2[j];
      }
      o += 512 + 32;
      nat += (size_t)H * H + H;
    }
    for (int s = 0; s < 2; ++s) {
      const float* W3 = net[s] + nat;              // (d, H)
      const float* b3 = W3 + (size_t)d * H;
      for (int kk = 0; kk < H; ++kk)
        for (int q = 0; q < nout; ++q) o[2 * (kk * NO + q) + s] = W3[(size_t)(o0 + 2 * q) * H + kk];
      for (int q = 0; q < nout; ++q) o[2 * (16 * NO + q) + s] = b3[o0 + 2 * q];
    }
  }
  if (warp_smem_bytes(w, target_doubles(d, NNB_MAX_LIKE_PARAMS), 2) > (size_t)h->max_smem) return NNB_OK;
  NNB_CUDA(h, nnb_reserve(&h->d_weights_warp, &h->weights_warp_cap, buf.size()));
  NNB_CUDA(h, cudaMemcpy(h->d_weights_warp, buf.data(), buf.size() * sizeof(float), cudaMemcpyHostToDevice));
  h->warpflow = w;
  h->warp_ok = true;
  return NNB_OK;
}

namespace {

// chains per CTA and grid such that every CTA is resident (needed by the per-step grid barrier): spread the batch over
// all SMs, two CTAs per SM at most (launch bounds); returns false when the batch does not fit
bool warp_plan(nnb_handle* h, const void* fn, long long n, int tdoubles, int* cpc_out, int* grid_out, size_t* smem_out) {
  for (int per_sm = 1; per_sm <= 2; ++per_sm) {
    long long cpc = (n + (long long)h->sm_count * per_sm - 1) / ((long long)h->sm_count * per_sm);
    cpc = (cpc + 1) & ~1ll;              // whole warps
    if (cpc < 2) cpc = 2;
    if (cpc > kWarpMaxCpc) continue;
    const size_t sm = warp_smem_bytes(h->warpflow, tdoubles, (int)cpc);
    if (sm * per_sm > (size_t)h->max_smem_per_sm || sm > (size_t)h->max_smem) continue;
    int occ = 0;
    if (nnb_set_smem(fn, sm) != cudaSuccess) continue;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, (int)cpc * kWarpLanes, sm) != cudaSuccess)
      continue;
    const long long grid = (n + cpc - 1) / cpc;
    if (grid > (long long)occ * h->sm_count) continue;
    *cpc_out = (int)cpc; *grid_out = (int)grid; *smem_out = sm;
    return true;
  }
  return false;
}

template <int MODE, int DD>
int launch_warp_mode(nnb_handle* h, McmcParams p, int steps, cudaStream_t st, bool* ran) {
  const int tdoubles = target_doubles(h->tdesc.d, h->tdesc.n_params);
  int cpc = 0, grid = 0;
  size_t sm = 0;
  *ran = false;
  int rc = NNB_OK;
  const void* fn = nnb_kernel(h, (const void*)mcmc_warp_kernel<MODE, DD>, &rc, "nnb::mcmc_warp_kernel<%d, %d>", MODE, DD);
  if (!fn) return rc;
  if (!warp_plan(h, fn, p.n, tdoubles, &cpc, &grid, &sm)) return NNB_OK;
  if (p.dynamic && steps > 1 && !h->coop_supported) return NNB_OK;
  p.cpc = cpc;
  p.s0 = 0; p.nsteps = steps;
  void* args[] = {(void*)&h->warpflow, (void*)&h->d_weights_warp, (void*)&h->tdesc, (void*)&h->d_target, (void*)&p};
  if (p.dynamic && steps > 1) {
    if (h->step_counts_cap < steps) {
      if (h->d_step_counts) cudaFree(h->d_step_counts);
      h->d_step_counts = nullptr;
      NNB_CUDA(h, cudaMalloc(&h->d_step_counts, sizeof(unsigned long long) * steps));
      h->step_counts_cap = steps;
    }
    NNB_CUDA(h, cudaMemsetAsync(h->d_step_counts, 0, sizeof(unsigned long long) * steps, st));
    p.coop = 1; p.step_counts = h->d_step_counts;
    NNB_CUDA(h, cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(cpc * kWarpLanes), args, sm, st));
  } else if (p.dynamic) {
    // a single step: the scale update after it is the only one; run it through the cooperative path too when possible,
    // otherwise leave the batch to the other kernels
    return NNB_OK;
  } else {
    p.coop = 0; p.step_counts = nullptr;
    NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(cpc * kWarpLanes), args, sm, st));
  }
  h->last_launches = 1;
  *ran = true;
  return NNB_OK;
}

}  // namespace

// *ran = false: the batch is outside this kernel's range (too many chains to be co-resident, ...): caller falls back
template <int DD>
static int launch_warp_dim(nnb_handle* h, McmcParams p, int steps, cudaStream_t st, bool* ran) {
  return p.mode == NNB_MODE_MH ? launch_warp_mode<NNB_MODE_MH, DD>(h, p, steps, st, ran)
                               : launch_warp_mode<NNB_MODE_HARD, DD>(h, p, steps, st, ran);
}

int nnb_launch_mcmc_warp(nnb_handle* h, McmcParams p, int steps, cudaStream_t st, bool* ran) {
  // the reference's default architecture at the dimensions of the named workloads: fully unrolled kernels
  static const bool generic_only = getenv("NNB_WARP_GENERIC") != nullptr;
  if (!generic_only && h->warpflow.L == 1 && h->warpflow.B == 3) {
    switch (h->warpflow.d) {
      case 2: return launch_warp_dim<2>(h, p, steps, st, ran);
      case 10: return launch_warp_dim<10>(h, p, steps, st, ran);
      case 30: return launch_warp_dim<30>(h, p, steps, st, ran);
      case 50: return launch_warp_dim<50>(h, p, steps, st, ran);
      default: break;
    }
  }
  return launch_warp_dim<0>(h, p, steps, st, ran);
}

// largest batch the kernel holds co-resident (two CTAs of kWarpMaxCpc chains per SM)
long long nnb_warp_capacity(const nnb_handle* h) { return (long long)h->sm_count * 2 * kWarpMaxCpc; }
