// nnb_kernels.cuh -- kernels of libnnb.so and their launchers (see include/nnb.h for the contract).
//
// Kernels (all one chain per thread, 128 chains per CTA, flow weights + target staged in smem):
//   flow_kernel<H, INVERSE>   batched flow map                 (nnest/networks.py:24-42,289-309)
//   loglike_kernel<TIN>       batched likelihood/prior          (nnest/likelihoods.py, priors.py)
//   mcmc_init_kernel<H>       chain start                       (nnest/sampler.py:262-289)
//   mcmc_kernel<H, MODE>      `steps` fused MCMC steps          (nnest/sampler.py:291-444)
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#endif

#include "nnb_device.cuh"

using namespace nnb;

// ---------------------------------------------------------------------------------------------
// Device-side control block of one nnb_mcmc_run call (scale adaptation + counters).
// ---------------------------------------------------------------------------------------------
struct Ctrl {
  double scale;                   // sampler.py:257
  int accept, reject;             // sampler.py:258-259
  unsigned long long ncall;       // sampler.py:260
  unsigned long long naccept;     // total_accepted sampler.py:419
  unsigned long long nbad;        // start points with logl <= -1e30
  unsigned int step_acc;          // accepted proposals of the step in flight
  unsigned int ticket;            // CTAs that finished the step in flight
};

struct McmcParams {
  long long n;
  int s0, nsteps;   // runs steps s0+1 .. s0+nsteps (1-based step index inside this call)
  int mode, dynamic;
  double loglstar;
  unsigned int seed_lo, seed_hi;
  unsigned long long chain_offset;
  unsigned int step_offset;
  float* z;
  float* x;
  double* logl;
  float* logdet;
  double* logp;
  float* trace_x;
  float* trace_z;
  double* trace_logl;
  const float* replay_normals;
  const float* replay_uniforms;
  float* dump_normals;
  float* dump_uniforms;
  Ctrl* ctrl;
  int cpc;                     // chains per CTA (tensor-core kernel)
  int coop;                    // persistent cooperative launch: grid barrier per step (tensor-core kernel)
  unsigned long long* step_counts;   // [nsteps] per-step grid-barrier words, zeroed by the host (coop mode): CTAs that
                                     // arrived << 32 | accepted proposals -- ONE atomic per CTA carries both
  int total_tiles;             // tensor-core kernel, coop mode: tiles that arrive at the per-step grid barrier
  int tc_jc;                   // tensor-core kernel: Philox blocks of the next step drawn during the accept phase (-1 = default)
  int tc_delay[4];  // tensor-core kernel: start delay of tile slot j of a CTA at every step, cycles (see mcmc_tc_kernel)
};

struct SmemView {
  float* w;
  TargetSmem tg;
  float* y;
  float* zp;
  unsigned int* red;
};

// Shared-memory carve-up: [weights][target doubles][y: d*BS][zp: d*BS (optional)][red: 32]
__host__ __device__ inline size_t smem_bytes(int total_floats, int tdoubles, int d, int nvec) {
  return (size_t)total_floats * 4 + (size_t)tdoubles * 8 + (size_t)nvec * d * kBlockThreads * 4 + 32 * 4;
}

__device__ __forceinline__ SmemView carve(unsigned char* base, int total_floats, const TargetDesc& td,
                                          const double* tgt_g, int d, int nvec) {
  SmemView v;
  v.w = reinterpret_cast<float*>(base);
  double* td_s = reinterpret_cast<double*>(base + (size_t)total_floats * 4);
  const int nd = tgt_g ? target_doubles(td.d, td.n_params) : 0;
  for (int i = threadIdx.x; i < nd; i += blockDim.x) td_s[i] = tgt_g[i];
  target_bind(v.tg, td, td_s);
  v.y = reinterpret_cast<float*>(td_s + nd);
  v.zp = v.y + (size_t)d * kBlockThreads;
  v.red = reinterpret_cast<unsigned int*>(v.y + (size_t)nvec * d * kBlockThreads);
  return v;
}

__device__ __forceinline__ void stage_weights(float* dst, const float* __restrict__ src, int total_floats) {
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (int i = threadIdx.x; i < total_floats / 4; i += blockDim.x) d4[i] = s4[i];
}

// ---------------------------------------------------------------------------------------------
// Batched flow map
// ---------------------------------------------------------------------------------------------
template <int H, bool INVERSE>
__global__ void __launch_bounds__(kBlockThreads)
flow_kernel(FlowDesc f, const float* __restrict__ wg, const float* __restrict__ in, long long in_rs, long long in_cs,
            float* __restrict__ out, long long out_rs, long long out_cs, float* __restrict__ logdet, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TargetDesc td{};
  SmemView sv = carve(smem_raw, f.total_floats, td, nullptr, f.d, 1);
  stage_weights(sv.w, wg, f.total_floats);
  __syncthreads();
  float* y = sv.y + threadIdx.x;
  const long long ntiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long c = tile * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    for (int i = 0; i < f.d; ++i) y[i * kBlockThreads] = in[c * in_rs + i * in_cs];
    float ld = INVERSE ? flow_inverse_inplace<H>(f, sv.w, y, kBlockThreads)
                       : flow_forward_inplace<H>(f, sv.w, y, kBlockThreads);
    for (int i = 0; i < f.d; ++i) out[c * out_rs + i * out_cs] = y[i * kBlockThreads];
    if (logdet) logdet[c] = ld;
  }
}

// ---------------------------------------------------------------------------------------------
// Batched likelihood / prior
// ---------------------------------------------------------------------------------------------
template <typename TIN>
struct GlobalRow {
  const TIN* p;
  long long cs;
  __device__ __forceinline__ TIN operator()(int i) const { return p[i * cs]; }
};

template <typename TIN>
__global__ void __launch_bounds__(kBlockThreads)
loglike_kernel(TargetDesc td, const double* __restrict__ tgt_g, const TIN* __restrict__ u, long long rs, long long cs,
               double* __restrict__ logl, double* __restrict__ logp, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, 0, td, tgt_g, td.d, 0);
  __syncthreads();
  const long long ntiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long c = tile * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    GlobalRow<TIN> row{u + c * rs, cs};
    const bool f64 = sizeof(TIN) == 8;
    if (logl) logl[c] = loglike_any(sv.tg, row, f64);
    if (logp) logp[c] = prior_any(sv.tg, row, f64);
  }
}

// ---------------------------------------------------------------------------------------------
// MCMC
// ---------------------------------------------------------------------------------------------
struct SmemRow {
  const float* p;  // y + tid, stride kBlockThreads
  __device__ __forceinline__ float operator()(int i) const { return p[i * kBlockThreads]; }
};

// normals for dims 4j..4j+3 of (chain, step)
__device__ __forceinline__ void philox_normals4(unsigned int j, unsigned int step, unsigned int chain, unsigned int tag,
                                                unsigned int k0, unsigned int k1, float (&nrm)[4]) {
  box_muller4(philox4x32_10(j, step, chain, tag, k0, k1), nrm);
}

struct InitParams {
  long long n;
  float* z;
  float* x;
  double* logl;
  float* logdet;
  double* logp;
  const float* init_u;
  const float* init_z;
  const double* init_logl;
  unsigned int seed_lo, seed_hi;
  unsigned long long chain_offset;
  unsigned int start_try;
  Ctrl* ctrl;
};

template <int H>
__global__ void __launch_bounds__(kBlockThreads)
mcmc_init_kernel(FlowDesc f, const float* __restrict__ wg, TargetDesc td, const double* __restrict__ tgt_g,
                 InitParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, f.total_floats, td, tgt_g, f.d, 1);
  stage_weights(sv.w, wg, f.total_floats);
  __syncthreads();
  const int d = f.d;
  const long long n = p.n;
  const long long c = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const bool active = c < n;
  float* y = sv.y + threadIdx.x;
  unsigned int ncall = 0, nbad = 0;
  if (active) {
    if (p.init_u) {  // sampler.py:264-266: z = forward(u); x = inverse(z) "due to numerical precision"
      for (int i = 0; i < d; ++i) y[i * kBlockThreads] = p.init_u[(long long)i * n + c];
      flow_forward_inplace<H>(f, sv.w, y, kBlockThreads);
    } else if (p.init_z) {
      for (int i = 0; i < d; ++i) y[i * kBlockThreads] = p.init_z[(long long)i * n + c];
    } else {  // sampler.py:276: z ~ N(0, I)
      const unsigned int chain = (unsigned int)(p.chain_offset + (unsigned long long)c);
      for (int j = 0; j < (d + 3) / 4; ++j) {
        float nrm[4];
        philox_normals4(j, p.start_try, chain, kTagInit, p.seed_lo, p.seed_hi, nrm);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * j + q < d) y[(4 * j + q) * kBlockThreads] = nrm[q];
      }
    }
    for (int i = 0; i < d; ++i) p.z[(long long)i * n + c] = y[i * kBlockThreads];
    float ld = flow_inverse_inplace<H>(f, sv.w, y, kBlockThreads);
    for (int i = 0; i < d; ++i) p.x[(long long)i * n + c] = y[i * kBlockThreads];
    p.logdet[c] = ld;
    SmemRow row{y};
    double l;
    if (p.init_logl) {
      l = p.init_logl[c];
    } else {
      l = loglike_any(sv.tg, row, false);
      ncall = 1;
    }
    p.logl[c] = l;
    p.logp[c] = prior_any(sv.tg, row, false);
    nbad = !(l > -1e30);
  }
  unsigned int tc = block_sum_u32(ncall, sv.red);
  unsigned int tb = block_sum_u32(nbad, sv.red);
  if (threadIdx.x == 0) {
    if (tc) atomicAdd(&p.ctrl->ncall, (unsigned long long)tc);
    if (tb) atomicAdd(&p.ctrl->nbad, (unsigned long long)tb);
  }
}

template <int H, int MODE>
__global__ void __launch_bounds__(kBlockThreads)
mcmc_kernel(FlowDesc f, const float* __restrict__ wg, TargetDesc td, const double* __restrict__ tgt_g, McmcParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemView sv = carve(smem_raw, f.total_floats, td, tgt_g, f.d, 2);
  stage_weights(sv.w, wg, f.total_floats);
  __syncthreads();
  const int d = f.d;
  const long long n = p.n;
  const long long c = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const bool active = c < n;
  float* y = sv.y + threadIdx.x;
  float* zp = sv.zp + threadIdx.x;
  const unsigned int chain = (unsigned int)(p.chain_offset + (unsigned long long)c);
  unsigned int acc_total = 0, ncall_total = 0;

  // per-chain scalars kept in registers across the steps of this launch
  float ld_cur = 0.f;
  double logl_cur = 0.0, logp_cur = 0.0;
  if (active) {
    ld_cur = p.logdet[c];
    logl_cur = p.logl[c];
    logp_cur = p.logp[c];
  }

  for (int s = p.s0 + 1; s <= p.s0 + p.nsteps; ++s) {
    // scale is a Python float in the reference; the float32 tensor is multiplied by it (sampler.py:310)
    const float scale_f = (float)(*reinterpret_cast<volatile double*>(&p.ctrl->scale));
    const unsigned int step_abs = p.step_offset + (unsigned int)s;
    bool accept = false;
    unsigned int ncall = 0;
    if (active) {
      // ---- proposal z' = z + scale * N(0, I) -------------------------------------------- :310-316
      if (p.replay_normals) {
        const float* nr = p.replay_normals + ((long long)(s - 1) * n + c) * d;
        for (int i = 0; i < d; ++i) {
          float v = __fadd_rn(p.z[(long long)i * n + c], __fmul_rn(nr[i], scale_f));
          y[i * kBlockThreads] = v;
          zp[i * kBlockThreads] = v;
        }
      } else {
        for (int j = 0; j < (d + 3) / 4; ++j) {
          float nrm[4];
          philox_normals4(j, step_abs, chain, kTagNormal, p.seed_lo, p.seed_hi, nrm);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = 4 * j + q;
            if (i < d) {
              float v = __fadd_rn(p.z[(long long)i * n + c], __fmul_rn(nrm[q], scale_f));
              y[i * kBlockThreads] = v;
              zp[i * kBlockThreads] = v;
              if (p.dump_normals) p.dump_normals[((long long)(s - 1) * n + c) * d + i] = nrm[q];
            }
          }
        }
      }
      // ---- x', log|det J|' = flow.inverse(z') -------------------------------------------- :321
      const float ld_prop = flow_inverse_inplace<H>(f, sv.w, y, kBlockThreads);
      float u01;
      if (p.replay_uniforms) {
        u01 = p.replay_uniforms[(long long)(s - 1) * n + c];
      } else {
        uint4 r = philox4x32_10(0u, step_abs, chain, kTagUniform, p.seed_lo, p.seed_hi);
        u01 = uniform01(r.x);
        if (p.dump_uniforms) p.dump_uniforms[(long long)(s - 1) * n + c] = u01;
      }
      SmemRow row{y};
      double lp = 0.0, logp_prop = 0.0;
      if (MODE == NNB_MODE_HARD) {
        // stage 1: Jacobian ratio + prior box (sampler.py:326-336); NaN ratio rejects
        float lr = __fsub_rn(ld_prop, ld_cur);
        logp_prop = prior_any(sv.tg, row, false);
        if (logp_prop < -1e30) lr = -INFINITY;
        float ratio = expf(lr);
        if (ratio > 1.0f) ratio = 1.0f;
        const bool m1 = u01 < ratio;
        // stage 2: likelihood only for survivors, hard constraint (sampler.py:358-368)
        if (m1) {
          lp = loglike_any(sv.tg, row, false);
          ncall = 1;
          accept = isfinite(lp) && (lp > p.loglstar);
        }
      } else {
        // Metropolis-Hastings ratio (sampler.py:397-414), float64 like torch's promotion
        lp = loglike_any(sv.tg, row, false);
        ncall = 1;
        logp_prop = prior_any(sv.tg, row, false);
        double lr = (double)__fsub_rn(ld_prop, ld_cur) + (lp - logl_cur) + (logp_prop - logp_cur);
        double ratio = exp(lr);
        if (ratio > 1.0) ratio = 1.0;
        accept = (double)u01 < ratio;
      }
      // ---- state update (sampler.py:433-438; select instead of the arithmetic blend) ------
      if (accept) {
        for (int i = 0; i < d; ++i) {
          p.z[(long long)i * n + c] = zp[i * kBlockThreads];
          p.x[(long long)i * n + c] = y[i * kBlockThreads];
        }
        ld_cur = ld_prop;
        logl_cur = lp;
        logp_cur = logp_prop;
      }
      // ---- trace (sampler.py:441-444) -----------------------------------------------------
      if (p.trace_z) {
        float* tz = p.trace_z + (long long)s * d * n + c;
        float* tx = p.trace_x + (long long)s * d * n + c;
        if (accept) {
          for (int i = 0; i < d; ++i) {
            tz[(long long)i * n] = zp[i * kBlockThreads];
            tx[(long long)i * n] = y[i * kBlockThreads];
          }
        } else {
          for (int i = 0; i < d; ++i) {
            tz[(long long)i * n] = p.z[(long long)i * n + c];
            tx[(long long)i * n] = p.x[(long long)i * n + c];
          }
        }
        p.trace_logl[(long long)s * n + c] = logl_cur;
      }
    }
    acc_total += accept ? 1u : 0u;
    ncall_total += ncall;

    if (p.dynamic) {
      // global accept count of this step -> scale adaptation (sampler.py:418-430).  The host issues one
      // launch per step in this mode, so "the last CTA to finish" owns the update.
      unsigned int blk = block_count(accept);
      if (threadIdx.x == 0) {
        if (blk) atomicAdd(&p.ctrl->step_acc, blk);
        __threadfence();
        unsigned int t = atomicAdd(&p.ctrl->ticket, 1u);
        if (t == gridDim.x - 1) {
          __threadfence();
          unsigned int na = atomicExch(&p.ctrl->step_acc, 0u);
          p.ctrl->ticket = 0u;
          int a = p.ctrl->accept, r = p.ctrl->reject;
          if (2ull * na > (unsigned long long)n) a += 1; else r += 1;
          double sc = p.ctrl->scale;
          if (a > r) sc *= exp(1.0 / (1 + a));
          if (a < r) sc /= exp(1.0 / (1 + r));
          p.ctrl->accept = a;
          p.ctrl->reject = r;
          p.ctrl->scale = sc;
        }
      }
    }
  }
  if (active) {
    p.logdet[c] = ld_cur;
    p.logl[c] = logl_cur;
    p.logp[c] = logp_cur;
  }
  unsigned int ta = block_sum_u32(acc_total, sv.red);
  unsigned int tc = block_sum_u32(ncall_total, sv.red);
  if (threadIdx.x == 0) {
    if (ta) atomicAdd(&p.ctrl->naccept, (unsigned long long)ta);
    if (tc) atomicAdd(&p.ctrl->ncall, (unsigned long long)tc);
  }
}

