// nnb_spline_kernels.cuh -- device side of flow='spline' (nnb_spline.cu): batched flow maps, chain start and the fused
// MCMC step.  A header of its own so that NVRTC can instantiate the step kernels around a user likelihood (nnb_jit.cu).
#pragma once
#include "nnb_kernels.cuh"
#include "nnb_spline.cuh"

namespace {

struct SplineSmem {
  TargetSmem tg;
  float* y;
  float* zp;
  float* tmp;
  unsigned int* red;
};

__host__ __device__ inline size_t spline_smem_bytes(int tdoubles, int d) {
  return (size_t)tdoubles * 8 + (size_t)3 * d * kBlockThreads * 4 + 32 * 4;
}

__device__ __forceinline__ SplineSmem spline_carve(unsigned char* base, const TargetDesc& td, const double* tgt_g, int d) {
  SplineSmem v;
  double* td_s = reinterpret_cast<double*>(base);
  const int nd = tgt_g ? target_doubles(td.d, td.n_params) : 0;
  for (int i = threadIdx.x; i < nd; i += blockDim.x) td_s[i] = tgt_g[i];
  target_bind(v.tg, td, td_s);
  v.y = reinterpret_cast<float*>(td_s + nd);
  v.zp = v.y + (size_t)d * kBlockThreads;
  v.tmp = v.zp + (size_t)d * kBlockThreads;
  v.red = reinterpret_cast<unsigned int*>(v.tmp + (size_t)d * kBlockThreads);
  return v;
}

template <bool INVERSE>
__global__ void __launch_bounds__(kBlockThreads)
spline_flow_kernel(spline::Shape sh, const float* __restrict__ packed, const float* __restrict__ in, long long in_rs,
                   long long in_cs, float* __restrict__ out, long long out_rs, long long out_cs,
                   float* __restrict__ logdet, int* __restrict__ empty_out, long long n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TargetDesc td{};
  SplineSmem sv = spline_carve(smem_raw, td, nullptr, sh.d);
  float* y = sv.y + threadIdx.x;
  float* tmp = sv.tmp + threadIdx.x;
  const long long ntiles = (n + kBlockThreads - 1) / kBlockThreads;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long c = tile * kBlockThreads + threadIdx.x;
    if (c >= n) continue;
    for (int i = 0; i < sh.d; ++i) y[i * kBlockThreads] = in[c * in_rs + i * in_cs];
    int empty = 0;
    const float ld = INVERSE ? spline::flow_inverse(sh, packed, y, tmp, kBlockThreads, &empty)
                             : spline::flow_forward(sh, packed, y, tmp, kBlockThreads, &empty);
    for (int i = 0; i < sh.d; ++i) out[c * out_rs + i * out_cs] = y[i * kBlockThreads];
    if (logdet) logdet[c] = ld;
    if (empty_out) empty_out[c] = empty;
  }
}

__global__ void __launch_bounds__(kBlockThreads)
spline_init_kernel(spline::Shape sh, const float* __restrict__ packed, TargetDesc td, const double* __restrict__ tgt_g,
                   InitParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SplineSmem sv = spline_carve(smem_raw, td, tgt_g, sh.d);
  __syncthreads();
  const int d = sh.d;
  const long long n = p.n;
  const long long c = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const bool active = c < n;
  float* y = sv.y + threadIdx.x;
  float* tmp = sv.tmp + threadIdx.x;
  unsigned int ncall = 0, nbad = 0;
  if (active) {
    if (p.init_u) {  // sampler.py:264-266: z = forward(u); x = inverse(z) "due to numerical precision"
      for (int i = 0; i < d; ++i) y[i * kBlockThreads] = p.init_u[(long long)i * n + c];
      spline::flow_forward(sh, packed, y, tmp, kBlockThreads);
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
    const float ld = spline::flow_inverse(sh, packed, y, tmp, kBlockThreads);
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

template <int MODE>
__global__ void __launch_bounds__(kBlockThreads)
spline_mcmc_kernel(spline::Shape sh, const float* __restrict__ packed, TargetDesc td, const double* __restrict__ tgt_g,
                   McmcParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SplineSmem sv = spline_carve(smem_raw, td, tgt_g, sh.d);
  __syncthreads();
  const int d = sh.d;
  const long long n = p.n;
  const long long c = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
  const bool active = c < n;
  float* y = sv.y + threadIdx.x;
  float* zp = sv.zp + threadIdx.x;
  float* tmp = sv.tmp + threadIdx.x;
  const unsigned int chain = (unsigned int)(p.chain_offset + (unsigned long long)c);
  unsigned int acc_total = 0, ncall_total = 0;
  float ld_cur = 0.f;
  double logl_cur = 0.0, logp_cur = 0.0;
  if (active) {
    ld_cur = p.logdet[c];
    logl_cur = p.logl[c];
    logp_cur = p.logp[c];
  }
  for (int s = p.s0 + 1; s <= p.s0 + p.nsteps; ++s) {
    const float scale_f = (float)(*reinterpret_cast<volatile double*>(&p.ctrl->scale));
    const unsigned int step_abs = p.step_offset + (unsigned int)s;
    bool accept = false;
    unsigned int ncall = 0;
    if (active) {
      // ---- proposal z' = z + scale * N(0, I) -------------------------------------------- sampler.py:310-316
      if (p.replay_normals) {
        const float* nr = p.replay_normals + ((long long)(s - 1) * n + c) * d;
        for (int i = 0; i < d; ++i) {
          const float v = __fadd_rn(p.z[(long long)i * n + c], __fmul_rn(nr[i], scale_f));
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
              const float v = __fadd_rn(p.z[(long long)i * n + c], __fmul_rn(nrm[q], scale_f));
              y[i * kBlockThreads] = v;
              zp[i * kBlockThreads] = v;
              if (p.dump_normals) p.dump_normals[((long long)(s - 1) * n + c) * d + i] = nrm[q];
            }
          }
        }
      }
      // ---- x', log|det J|' = flow.inverse(z') -------------------------------------------- sampler.py:320-324
      int empty = 0;
      const float ld_prop = spline::flow_inverse(sh, packed, y, tmp, kBlockThreads, &empty);
      float u01;
      if (p.replay_uniforms) {
        u01 = p.replay_uniforms[(long long)(s - 1) * n + c];
      } else {
        uint4 r = philox4x32_10(0u, step_abs, chain, kTagUniform, p.seed_lo, p.seed_hi);
        u01 = uniform01(r.x);
        if (p.dump_uniforms) p.dump_uniforms[(long long)(s - 1) * n + c] = u01;
      }
      // a ONE-chain batch whose proposal has a coupling half entirely outside the tail bound: the reference's inverse
      // raises ValueError and the proposal is skipped (sampler.py:320-324).  With more than one chain the reference only
      // raises when no chain at all has a coordinate inside, which does not happen in practice: identity map as coded.
      const bool skip = empty != 0 && n == 1;
      SmemRow row{y};
      double lp = 0.0, logp_prop = 0.0;
      if (skip) {
      } else if (MODE == NNB_MODE_HARD) {
        float lr = __fsub_rn(ld_prop, ld_cur);
        logp_prop = prior_any(sv.tg, row, false);
        if (logp_prop < -1e30) lr = -INFINITY;
        float ratio = expf(lr);
        if (ratio > 1.0f) ratio = 1.0f;
        const bool m1 = u01 < ratio;
        if (m1) {
          lp = loglike_any(sv.tg, row, false);
          ncall = 1;
          accept = isfinite(lp) && (lp > p.loglstar);
        }
      } else {
        lp = loglike_any(sv.tg, row, false);
        ncall = 1;
        logp_prop = prior_any(sv.tg, row, false);
        double lr = (double)__fsub_rn(ld_prop, ld_cur) + (lp - logl_cur) + (logp_prop - logp_cur);
        double ratio = exp(lr);
        if (ratio > 1.0) ratio = 1.0;
        accept = (double)u01 < ratio;
      }
      if (accept) {
        for (int i = 0; i < d; ++i) {
          p.z[(long long)i * n + c] = zp[i * kBlockThreads];
          p.x[(long long)i * n + c] = y[i * kBlockThreads];
        }
        ld_cur = ld_prop;
        logl_cur = lp;
        logp_cur = logp_prop;
      }
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
    if (p.dynamic) {   // one launch per step: the last CTA to finish owns the scale update (sampler.py:418-430)
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

}  // namespace
