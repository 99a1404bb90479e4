// nnb_warp.cuh -- small-batch variant of the fused MCMC step kernel: 16 lanes per chain.
//
// Same contract as mcmc_kernel<16, MODE> / mcmc_tc_kernel (reference nnest/sampler.py:291-444).  The thread-per-chain
// kernels need >= ~65 k chains to fill a B200 (a chain's step is a ~14 us dependent instruction chain on one thread);
// when the batch is sharded over several GPUs (8192 chains per GPU at N = 8) or is small to begin with (1024 chains in
// BASELINE configs[1]), that leaves most of the machine idle.  Here a chain is advanced by HALF A WARP:
//   * lane j of the chain's 16-lane group owns hidden unit j of BOTH coupling MLPs (scale net: tanh, translate net:
//     relu, nnest/networks.py:262-282), so every layer is 16-wide SIMD work: nin / 16 / 16 fused multiply-adds per lane
//     with the (s, t) weight pair fetched as ONE 8-byte shared-memory load; activations are exchanged through a
//     64-float shared-memory slot per chain (`__syncwarp` on the group's lanes);
//   * output o of both nets is produced by lane o % 16, which also applies x = (z - t) exp(-log s) to its coordinate,
//     tests it against the prior box and accumulates its share of log|det J| (group reduction by shuffles);
//   * the Philox blocks of a step (4 normals each) are drawn by lanes 0 .. ceil(d/4)-1 in parallel, the accept uniform
//     by the next lane; with a dynamic step size the next step's noise is drawn between "arrive" and "wait" of the
//     per-step grid barrier (cooperative launch), exactly as in the tensor-core kernel;
//   * the chain's current z, x, the proposal and its image stay in shared memory for all steps of the launch (global
//     memory is touched at entry, at exit and for the optional trace);
//   * Rosenbrock (float32 arithmetic): the d-1 terms are evaluated lane-parallel, then added LEFT TO RIGHT by one lane
//     with the same roundings as loglike_T (bit-identical values); other likelihoods run on the group's first lane.
// A step costs ~450 warp instructions per chain instead of ~150 (4 800 thread instructions / 32) in the tensor-core
// kernel, but its latency is ~1.5 us instead of ~14 us: the right trade below ~10 k chains per GPU.
#pragma once
#include "nnb_kernels.cuh"
#include "nnb_warp_desc.h"

namespace nnb {

constexpr int kWarpLanes = 16;          // lanes per chain
constexpr int kWarpMaxCpc = 28;         // chains per CTA (448 threads: two CTAs per SM at 72 registers per thread)

__host__ __device__ inline int warp_round16(int v) { return (v + 15) & ~15; }
__host__ __device__ inline int warp_block_floats(int d, int L, int k) {
  const int nin = blk_nin(d, k), NO = warp_round16(blk_nout(d, k));
  return 32 * nin + 32 + L * (512 + 32) + 32 * NO + 2 * NO;
}
__host__ __device__ inline bool warp_supported(const FlowDesc& f) {
  return f.H == 16 && f.d >= 2 && !(f.flags & (NNB_FLOW_TRANSLATE_ONLY | NNB_FLOW_CONST_SCALE));
}
// per-chain shared-memory slot (floats): zc[d] xc[d] zp[d] y[d] tv[d] tm[d] h[2][32]
// The stride is an odd multiple of 16 floats: the two chains of a warp then sit 16 banks apart, so neither their
// broadcast reads (same index, two addresses) nor their lane-indexed accesses (16 consecutive words each) collide.
__host__ __device__ inline int warp_chain_floats(int d) {
  const int c = 6 * round4(d) + 64;
  return (c & 31) == 16 ? c : ((c + 31) & ~31) + 16;
}
#ifndef __CUDACC_RTC__
__host__ inline size_t warp_smem_bytes(const WarpFlowDesc& f, int tdoubles, int cpc) {
  return (size_t)f.total_floats * 4 + (size_t)((tdoubles + 1) & ~1) * 8 + (size_t)cpc * warp_chain_floats(f.d) * 4 + 64;
}
#endif

__device__ __forceinline__ float warp_tanh(float x) {   // 1 - 2 / (e^{2x} + 1), MUFU ex2 / rcp (as tc_tanh)
  float e, rc;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(e + 1.0f));
  return fmaf(-2.0f, rc, 1.0f);
}
__device__ __forceinline__ float warp_exp(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.4426950408889634f));
  return e;
}

struct ContigRow {
  const float* p;
  __device__ __forceinline__ float operator()(int i) const { return p[i]; }
};

// one 16-wide layer: acc (s, t) += sum_k W[k][lane] * (hs[k], ht[k]), activations read as float4 broadcasts
__device__ __forceinline__ void warp_layer16(const float2* __restrict__ W, int ldw, const float* __restrict__ h, int col,
                                             float& as, float& at) {
  const float4* hs4 = reinterpret_cast<const float4*>(h);
  const float4* ht4 = reinterpret_cast<const float4*>(h + 16);
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    const float4 a = hs4[k4], b = ht4[k4];
    const float2 w0 = W[(4 * k4 + 0) * ldw + col], w1 = W[(4 * k4 + 1) * ldw + col];
    const float2 w2 = W[(4 * k4 + 2) * ldw + col], w3 = W[(4 * k4 + 3) * ldw + col];
    as = fmaf(w0.x, a.x, as); at = fmaf(w0.y, b.x, at);
    as = fmaf(w1.x, a.y, as); at = fmaf(w1.y, b.y, at);
    as = fmaf(w2.x, a.z, as); at = fmaf(w2.y, b.z, at);
    as = fmaf(w3.x, a.w, as); at = fmaf(w3.y, b.w, at);
  }
}

// one out-of-line copy of the generic likelihood / prior switch (register pressure stays out of the step loop)
static __device__ __noinline__ double warp_loglike(TargetDesc td, const double* td_s, const float* y) {
  TargetSmem tg;
  target_bind(tg, td, td_s);
  ContigRow row{y};
  return loglike_any(tg, row, false);
}
static __device__ __noinline__ double warp_prior(TargetDesc td, const double* td_s, const float* y) {
  TargetSmem tg;
  target_bind(tg, td, td_s);
  ContigRow row{y};
  return prior_any(tg, row, false);
}

// DD > 0: x_dim = DD, num_layers = 1 and num_blocks = 3 (the reference's defaults) are compile-time constants: every
// loop unrolls and every shared-memory offset becomes an immediate (the generic instantiation spends most of its
// instructions on loop control and address arithmetic: profiles/r2_warp1_*)
template <int MODE, int DD>
__global__ void __launch_bounds__(kWarpMaxCpc * kWarpLanes, 2)
mcmc_warp_kernel(WarpFlowDesc f, const float* __restrict__ wglob, TargetDesc td, const double* __restrict__ tgt_g,
                 McmcParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int d = DD > 0 ? DD : f.d, L = DD > 0 ? 1 : f.L, nB = DD > 0 ? 3 : f.B;
  const int cpc = p.cpc;
  float* wsm = reinterpret_cast<float*>(smem_raw);
  double* td_s = reinterpret_cast<double*>(smem_raw + (size_t)f.total_floats * 4);
  const int nd = target_doubles(td.d, td.n_params);
  float* chains_s = reinterpret_cast<float*>(td_s + ((nd + 1) & ~1));   // 16-byte aligned (float4 activation loads)
  const int cf = warp_chain_floats(d), dp = round4(d);
  unsigned int* cta_words = reinterpret_cast<unsigned int*>(chains_s + (size_t)cpc * cf);   // [0] accept count [1] scale (f32)
  {
    const float4* s4 = reinterpret_cast<const float4*>(wglob);
    float4* d4 = reinterpret_cast<float4*>(wsm);
    for (int i = threadIdx.x; i < f.total_floats / 4; i += blockDim.x) d4[i] = s4[i];
    for (int i = threadIdx.x; i < nd; i += blockDim.x) td_s[i] = tgt_g[i];
    if (threadIdx.x == 0) {
      cta_words[0] = 0u;
      reinterpret_cast<float*>(cta_words)[1] = (float)(*reinterpret_cast<volatile double*>(&p.ctrl->scale));
    }
  }
  __syncthreads();
  TargetSmem tg;
  target_bind(tg, td, td_s);

  const int lane = threadIdx.x & (kWarpLanes - 1);
  const int grp = threadIdx.x / kWarpLanes;                       // chain slot in the CTA
  const unsigned int gmask = 0xffffu << ((threadIdx.x & 16));     // this group's lanes within the warp
  const long long n = p.n;
  const long long c = (long long)blockIdx.x * cpc + grp;
  const bool active = grp < cpc && c < n;
  const size_t ns = (size_t)n;
  float* zc = chains_s + (size_t)(grp < cpc ? grp : 0) * cf;
  float* xc = zc + dp;
  float* zp = xc + dp;
  float* y = zp + dp;
  float* tv = y + dp;
  float* tm = tv + dp;
  float* hbuf = tm + dp;                                           // [2][32]
  const unsigned int chain = (unsigned int)(p.chain_offset + (unsigned long long)c);
  const int nj = (d + 3) / 4;
  const bool philox = p.replay_normals == nullptr, philox_u = p.replay_uniforms == nullptr;

  float ld_cur = 0.f;
  double logl_cur = 0.0, logp_cur = 0.0;
  if (active) {
    for (int i = lane; i < d; i += kWarpLanes) {
      zc[i] = p.z[(size_t)c + (size_t)i * ns];
      xc[i] = p.x[(size_t)c + (size_t)i * ns];
    }
    ld_cur = p.logdet[c];
    logl_cur = p.logl[c];
    logp_cur = p.logp[c];
  }
  __syncwarp(gmask);

  unsigned int acc_total = 0, ncall_total = 0;
  double co_scale = *reinterpret_cast<volatile double*>(&p.ctrl->scale);
  int co_accept = p.ctrl->accept, co_reject = p.ctrl->reject;       // thread 0's copy of the adaptation state
  // noise of the coming step: lane j < nj holds Philox block j (dims 4j..4j+3); for d > 64 a second block j + 16
  float nrm[2][4];
  float u_next = 0.f;
  auto draw = [&](unsigned int step_abs, int sidx) {
    if (!active) return;
    if (philox) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int j = lane + 16 * r;
        if (j < nj) {
          philox_normals4(j, step_abs, chain, kTagNormal, p.seed_lo, p.seed_hi, nrm[r]);
          if (p.dump_normals)
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (4 * j + q < d) p.dump_normals[((size_t)sidx * ns + (size_t)c) * d + 4 * j + q] = nrm[r][q];
        }
      }
    } else {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int j = lane + 16 * r;
        if (j < nj)
#pragma unroll
          for (int q = 0; q < 4; ++q)
            nrm[r][q] = 4 * j + q < d ? p.replay_normals[((size_t)sidx * ns + (size_t)c) * d + 4 * j + q] : 0.f;
      }
    }
    if (lane == kWarpLanes - 1) {
      if (philox_u) {
        uint4 r = philox4x32_10(0u, step_abs, chain, kTagUniform, p.seed_lo, p.seed_hi);
        u_next = uniform01(r.x);
        if (p.dump_uniforms) p.dump_uniforms[(size_t)sidx * ns + (size_t)c] = u_next;
      } else {
        u_next = p.replay_uniforms[(size_t)sidx * ns + (size_t)c];
      }
    }
  };
  draw(p.step_offset + (unsigned int)(p.s0 + 1), p.s0);
  const bool fast_rosen = tg.desc.like_id == NNB_LIKE_ROSENBROCK && !tg.desc.compute_f64 && builtin_transform(tg.desc);

  for (int s = p.s0 + 1; s <= p.s0 + p.nsteps; ++s) {
    const unsigned int step_abs = p.step_offset + (unsigned int)s;
    const bool more = s < p.s0 + p.nsteps;
    const float scale_f = p.coop ? reinterpret_cast<volatile float*>(cta_words)[1]
                                 : (float)(*reinterpret_cast<volatile double*>(&p.ctrl->scale));
    bool accept = false;
    unsigned int ncall = 0;
    if (active) {
      // ---- proposal z' = z + scale * N(0, I) (sampler.py:310-316) ---------------------------------------------------
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int j = lane + 16 * r;
        if (j < nj)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = 4 * j + q;
            if (i < d) {
              const float v = __fadd_rn(zc[i], __fmul_rn(nrm[r][q], scale_f));
              zp[i] = v;
              y[i] = v;
            }
          }
      }
      const float u01 = __shfl_sync(gmask, u_next, kWarpLanes - 1, kWarpLanes);
      __syncwarp(gmask);
      // ---- flow inverse (networks.py:24-42, 300-309) -----------------------------------------------------------------
      float ld = 0.f;
      bool bad = false;
      int hb = 0;
#pragma unroll
      for (int k = nB - 1; k >= 0; --k) {
        const int nin = blk_nin(d, k), i0 = blk_i0(k), nout = blk_nout(d, k), o0 = blk_o0(k);
        const int NO = warp_round16(nout);
        const int boff = DD > 0 ? (k > 0 ? warp_block_floats(d, L, 0) : 0) + (k > 1 ? warp_block_floats(d, L, 1) : 0)
                                : f.off[k];
        const float* wb = wsm + boff;
        const float2* W1 = reinterpret_cast<const float2*>(wb);
        const float2* b1 = W1 + nin * 16;
        float2 bb = b1[lane];
        float as = bb.x, at = bb.y;
#pragma unroll
        for (int a = 0; a < nin; ++a) {
          const float v = y[i0 + 2 * a];
          const float2 w = W1[a * 16 + lane];
          as = fmaf(w.x, v, as);
          at = fmaf(w.y, v, at);
        }
        float* h = hbuf + 32 * hb;
        h[lane] = warp_tanh(as);
        h[16 + lane] = fmaxf(at, 0.f);
        __syncwarp(gmask);
        const float2* Wl = b1 + 16;
#pragma unroll
        for (int l = 0; l < L; ++l) {
          bb = Wl[256 + lane];
          as = bb.x; at = bb.y;
          warp_layer16(Wl, 16, h, lane, as, at);
          hb ^= 1;
          h = hbuf + 32 * hb;
          h[lane] = warp_tanh(as);
          h[16 + lane] = fmaxf(at, 0.f);
          __syncwarp(gmask);
          Wl += 256 + 16;
        }
        const float2* W3 = Wl;
        const float2* b3 = W3 + 16 * NO;
#pragma unroll
        for (int o = lane; o < nout; o += kWarpLanes) {
          bb = b3[o];
          as = bb.x; at = bb.y;
          warp_layer16(W3, NO, h, o, as, at);
          const int i = o0 + 2 * o;
          const float xv = (y[i] - at) * warp_exp(-as);
          y[i] = xv;
          ld -= as;
        }
        hb ^= 1;     // the next block's first layer writes the other activation buffer
        __syncwarp(gmask);
      }
      // prior box on the flow's own coordinates (priors.py:39-43), every lane its dims
      if (tg.desc.prior_kind == NNB_PRIOR_BOX_U)
        for (int i = lane; i < d; i += kWarpLanes) bad |= (y[i] < tg.lof[i]) | (y[i] > tg.hif[i]);
      // log|det J| of the chain: sum over the group's lanes (butterfly: every lane ends with the same value)
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) ld += __shfl_xor_sync(gmask, ld, o, kWarpLanes);
      const float ld_prop = ld;
      double lp = 0.0, logp_prop = 0.0;
      // ---- accept / reject ---------------------------------------------------------------------------------------
      auto like_group = [&]() -> double {   // likelihood of the point in y, evaluated by the group; same value in all lanes
        double v = 0.0;
        if (fast_rosen) {
          for (int i = lane; i < d; i += kWarpLanes) {
            float t = y[i];
            if (tg.desc.has_transform) t = __fadd_rn(__fmul_rn(t, tg.tsf[i]), tg.tbf[i]);
            tv[i] = t;
          }
          __syncwarp(gmask);
          for (int i = lane; i < d - 1; i += kWarpLanes) {
            const float prev = tv[i], cur = tv[i + 1];
            const float t1 = __fsub_rn(cur, __fmul_rn(prev, prev));
            const float t2 = __fsub_rn(1.0f, prev);
            tm[i] = __fadd_rn(__fmul_rn(100.0f, __fmul_rn(t1, t1)), __fmul_rn(t2, t2));
          }
          __syncwarp(gmask);
          float acc = 0.f;
          if (lane == 0) {
#pragma unroll
            for (int i = 0; i < d - 1; ++i) acc = __fadd_rn(acc, tm[i]);      // left to right, as likelihoods.py:50-51
          }
          acc = __shfl_sync(gmask, acc, 0, kWarpLanes);
          v = -(double)acc;
          if (!isfinite(v)) v = -INFINITY;
        } else {
          if (lane == 0) v = warp_loglike(td, td_s, y);
          v = __shfl_sync(gmask, v, 0, kWarpLanes);
        }
        return v;
      };
      auto prior_group = [&]() -> double {
        double v = 0.0;
        if (lane == 0) v = warp_prior(td, td_s, y);
        return __shfl_sync(gmask, v, 0, kWarpLanes);
      };
      if (MODE == NNB_MODE_HARD) {
        float lr = __fsub_rn(ld_prop, ld_cur);
        if (tg.desc.prior_kind == NNB_PRIOR_BOX_U) {
          const bool anybad = __any_sync(gmask, bad);
          logp_prop = anybad ? -INFINITY : 0.0;
        } else {
          logp_prop = prior_group();
        }
        if (logp_prop < -1e30) lr = -INFINITY;
        float ratio = expf(lr);
        if (ratio > 1.0f) ratio = 1.0f;
        const bool m1 = u01 < ratio;                     // identical in all lanes of the group
        if (m1) {
          lp = like_group();
          ncall = lane == 0 ? 1u : 0u;
          accept = isfinite(lp) && (lp > p.loglstar);
        }
      } else {
        lp = like_group();
        ncall = lane == 0 ? 1u : 0u;
        logp_prop = prior_group();
        double lr = (double)__fsub_rn(ld_prop, ld_cur) + (lp - logl_cur) + (logp_prop - logp_cur);
        double ratio = exp(lr);
        if (ratio > 1.0) ratio = 1.0;
        accept = (double)u01 < ratio;
      }
      // ---- state / trace update (sampler.py:433-444) ---------------------------------------------------------------
      if (accept) {
        for (int i = lane; i < d; i += kWarpLanes) {
          zc[i] = zp[i];
          xc[i] = y[i];
        }
        ld_cur = ld_prop;
        logl_cur = lp;
        logp_cur = logp_prop;
      }
      if (p.trace_z) {
        for (int i = lane; i < d; i += kWarpLanes) {
          p.trace_z[((size_t)s * d + i) * ns + (size_t)c] = zc[i];
          p.trace_x[((size_t)s * d + i) * ns + (size_t)c] = xc[i];
        }
        if (lane == 0) p.trace_logl[(size_t)s * ns + (size_t)c] = logl_cur;
      }
      __syncwarp(gmask);
    }
    acc_total += (accept && lane == 0) ? 1u : 0u;
    ncall_total += ncall;

    // ---- global accept count of the step -> scale adaptation (sampler.py:418-430) ------------------------------------
    if (p.coop) {
      const int si = s - p.s0 - 1;
      if (accept && lane == 0) atomicAdd(&cta_words[0], 1u);
      __syncthreads();
      if (threadIdx.x == 0) {
        const unsigned int blk = cta_words[0];
        cta_words[0] = 0u;
        grid_arrive(&p.step_counts[si], blk);
      }
      if (more) draw(step_abs + 1u, s);                   // overlaps the grid barrier
      if (threadIdx.x == 0) {
        const unsigned int na = grid_wait(&p.step_counts[si], gridDim.x);
        if (p.dynamic) {
          if (2ull * na > (unsigned long long)n) co_accept += 1; else co_reject += 1;
          if (co_accept > co_reject) co_scale *= exp(1.0 / (1 + co_accept));
          if (co_accept < co_reject) co_scale /= exp(1.0 / (1 + co_reject));
          reinterpret_cast<volatile float*>(cta_words)[1] = (float)co_scale;
        }
      }
      __syncthreads();
    } else if (more) {
      draw(step_abs + 1u, s);
    }
  }
  // ---- write the state back ---------------------------------------------------------------------------------------------
  if (active) {
    for (int i = lane; i < d; i += kWarpLanes) {
      p.z[(size_t)c + (size_t)i * ns] = zc[i];
      p.x[(size_t)c + (size_t)i * ns] = xc[i];
    }
    if (lane == 0) {
      p.logdet[c] = ld_cur;
      p.logl[c] = logl_cur;
      p.logp[c] = logp_cur;
    }
  }
  if (p.coop && blockIdx.x == 0 && threadIdx.x == 0) {
    p.ctrl->scale = co_scale;
    p.ctrl->accept = co_accept;
    p.ctrl->reject = co_reject;
  }
  unsigned int ta = __reduce_add_sync(0xffffffffu, acc_total);
  unsigned int tcall = __reduce_add_sync(0xffffffffu, ncall_total);
  if ((threadIdx.x & 31) == 0) {
    if (ta) atomicAdd(&p.ctrl->naccept, (unsigned long long)ta);
    if (tcall) atomicAdd(&p.ctrl->ncall, (unsigned long long)tcall);
  }
}

}  // namespace nnb
