// nnb_device.cuh -- device-side building blocks of libnnb (sm_100a).
//
//   * Philox4x32-10 counter-based RNG + Box-Muller   (replaces torch.randn_like / torch.rand,
//                                                      nnest/sampler.py:310,334,377,412)
//   * affine-coupling block, inverse and forward      (nnest/networks.py:289-309)
//   * analytic likelihoods, transform, box prior      (nnest/likelihoods.py, nnest/priors.py:39-43,
//                                                      nnest/sampler.py:100-163)
// Layout conventions are described in DESIGN.md ("Data layout").
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#else   // NVRTC (user likelihoods, nnb_jit.cu): no toolkit headers
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef long long int64_t;
#define INFINITY __int_as_float(0x7f800000)
#endif

#include "../../include/nnb.h"

namespace nnb {

constexpr int kBlockThreads = 128;  // chains per CTA (one thread = one chain)

// ---------------------------------------------------------------------------------------------
// Flow description (passed by value to kernels) and packed weight layout.
//
// Block k uses mask[i] = (i + k) % 2.  Inputs of its MLPs are the nin dims with mask == 1
// (i = i0 + 2a, i0 = (k + 1) % 2); outputs are needed only on the nout dims with mask == 0
// (i = o0 + 2o, o0 = k % 2) -- the other half of the reference's dense Linear work multiplies
// zeros or is masked away (networks.py:291-296), so it is not computed.
// Packed net (all offsets multiples of 4 floats so rows can be read as float4 broadcasts):
//   W1T [nin][H]      W1T[a][j] = W1[j][i0 + 2a]
//   b1  [H]
//   L x { W2T [H][H]  W2T[k][j] = W2[j][k] ;  b2 [H] }
//   W3  [nout][H]     W3[o][j]  = W3[o0 + 2o][j]
//   b3  [round4(nout)]
// ---------------------------------------------------------------------------------------------
struct FlowDesc {
  int d, H, L, B, flags;
  int total_floats;                // size of the packed buffer
  int off_s[NNB_MAX_BLOCKS];       // offset of block k's scale net (-1 if translate only)
  int off_t[NNB_MAX_BLOCKS];       // offset of block k's translate net
  float cscale[NNB_MAX_BLOCKS];    // ScaleLayer parameter (networks.py:312-325) when NNB_FLOW_CONST_SCALE
};

// Packed weights of the tensor-core variant (layout: nnb_tc_kernels.cuh)
struct TcFlowDesc {
  int d, L, B;
  int total_floats;
  int off[NNB_MAX_BLOCKS];   // float offset of block k in the packed TC buffer
};

__host__ __device__ inline int round4(int v) { return (v + 3) & ~3; }
__host__ __device__ inline int blk_i0(int k) { return (k + 1) & 1; }
__host__ __device__ inline int blk_o0(int k) { return k & 1; }
__host__ __device__ inline int blk_nin(int d, int k) { return (d - blk_i0(k) + 1) / 2; }
__host__ __device__ inline int blk_nout(int d, int k) { return (d - blk_o0(k) + 1) / 2; }
__host__ __device__ inline int net_floats(int d, int H, int L, int k) {
  return blk_nin(d, k) * H + H + L * (H * H + H) + blk_nout(d, k) * H + round4(blk_nout(d, k));
}

// Target (likelihood o transform, prior) as staged in shared memory.
struct TargetDesc {
  int like_id, n_params, compute_f64, prior_kind, has_transform, d;
};
// has_transform: 0 none, 1 the affine map ts / tb, kTransformUser the handle's user transform (nnb_set_user_transform).
// Only the run-time build (nnb_jit.cu, NNB_USER_TRANSFORM) evaluates a user transform; the launchers never hand such a
// target to an ahead-of-time kernel (nnb_kernel, nnb_host.h).  Its params follow the likelihood's in `params`
// (n_params counts both) and ts[0] holds the likelihood's count, i.e. where the transform's params begin.
constexpr int kTransformUser = 2;

// false when the target's transform is the user's: the fast paths that apply ts / tb themselves test it (always true in
// the ahead-of-time build, which has no user transform)
__device__ __forceinline__ bool builtin_transform(const TargetDesc& td) {
#ifdef NNB_USER_TRANSFORM
  return td.has_transform != kTransformUser;
#else
  return true;
#endif
}
struct TargetSmem {
  TargetDesc desc;
  const double* params;  // [n_params]
  const double* ts;      // [d] transform scale
  const double* tb;      // [d] transform shift
  const double* lo;      // [d]
  const double* hi;      // [d]
  // float32 mirrors (4*d floats stored behind the doubles): transform scale/shift rounded to float32 (what NumPy
  // uses for float32 rows) and box bounds rounded so that (double)u < lo  <=>  u < lo_f and (double)u > hi  <=>  u > hi_f
  const float* tsf;
  const float* tbf;
  const float* lof;
  const float* hif;
};
__host__ __device__ inline int target_doubles(int d, int n_params) { return n_params + 4 * d + 2 * d; }

__device__ __forceinline__ void target_bind(TargetSmem& tg, const TargetDesc& td, const double* td_s) {
  tg.desc = td;
  tg.params = td_s;
  tg.ts = td_s + td.n_params;
  tg.tb = tg.ts + td.d;
  tg.lo = tg.tb + td.d;
  tg.hi = tg.lo + td.d;
  tg.tsf = reinterpret_cast<const float*>(tg.hi + td.d);
  tg.tbf = tg.tsf + td.d;
  tg.lof = tg.tbf + td.d;
  tg.hif = tg.lof + td.d;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  Stream specification: oracle/philox.py.
// ---------------------------------------------------------------------------------------------
enum { kTagNormal = 0, kTagUniform = 1, kTagInit = 2 };

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                uint32_t k1) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  return make_uint4(c0, c1, c2, c3);
}

// Four standard normals from one Philox block: Box-Muller on the word pairs (r.x, r.y) -> nrm[0..1] and (r.z, r.w) ->
// nrm[2..3] (u1 in (0,1], angle in [-pi, pi)).  The two transforms run side by side as packed FP32 pairs (FADD2 / FMUL2,
// sm_100): each lane is rounded exactly like the scalar instruction, so the normals are the bits of two scalar transforms.
// (ptxas may contract u2's product with the `- 0.5` into an FFMA2: that product is exact, so the bits do not change.)
__device__ __forceinline__ void box_muller4(uint4 r, float (&nrm)[4]) {
  const float2 k2m24 = make_float2(1.0f / 16777216.0f, 1.0f / 16777216.0f);
  const float2 u1 = __fmul2_rn(__fadd2_rn(make_float2((float)(r.x >> 8), (float)(r.z >> 8)), make_float2(1.0f, 1.0f)), k2m24);
  const float2 u2 = __fmul2_rn(make_float2((float)(r.y >> 8), (float)(r.w >> 8)), k2m24);
  // -2 ln u1 = lg2(u1) * (-2 fl(ln 2)), the bits of -2.0f * __logf(u1) (= -2 * fl(lg2(u1) * fl(ln 2))): u1 >= 2^-24 is never
  // a denormal, so the ftz lg2 returns what the denormal-guarded one inside __logf does, and -2 fl(ln 2) is exact, so one
  // rounded product by it equals the rounded product by fl(ln 2) times -2 (scaling by a power of two commutes with rounding).
  float2 lg;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.x) : "f"(u1.x));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.y) : "f"(u1.y));
  const float2 m2ln2 = make_float2(-2.0f * 0.693147182464599609375f, -2.0f * 0.693147182464599609375f);
  const float2 rr = __fmul2_rn(lg, m2ln2);
  float rad0, rad1;   // sqrt(-2 ln u1): MUFU-based square root (2 ulp) instead of the ~8-instruction IEEE sequence
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad0) : "f"(rr.x));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad1) : "f"(rr.y));
  const float2 ang = __fmul2_rn(__fadd2_rn(u2, make_float2(-0.5f, -0.5f)), make_float2(6.283185307179586f, 6.283185307179586f));
  float s0, c0, s1, c1;
  __sincosf(ang.x, &s0, &c0);
  __sincosf(ang.y, &s1, &c1);
  const float2 n01 = __fmul2_rn(make_float2(rad0, rad0), make_float2(c0, s0));
  const float2 n23 = __fmul2_rn(make_float2(rad1, rad1), make_float2(c1, s1));
  nrm[0] = n01.x;
  nrm[1] = n01.y;
  nrm[2] = n23.x;
  nrm[3] = n23.y;
}

__device__ __forceinline__ float uniform01(uint32_t r) { return __fmul_rn((float)(r >> 8), 1.0f / 16777216.0f); }

// ---------------------------------------------------------------------------------------------
// Coupling-layer MLPs, one chain per thread.  The chain vector lives in shared memory at
// y[i * ys] (ys = CTA width, conflict free); hidden activations live in registers; weights are
// read from shared memory as warp-wide float4 broadcasts.
// ---------------------------------------------------------------------------------------------
template <int ACT>  // 0 tanh (s-net), 1 relu (t-net)   networks.py:266-282
__device__ __forceinline__ float act_fn(float v) {
  if (ACT == 0) return tanhf(v);
  return fmaxf(v, 0.0f);
}

// Runs Linear(d,H) act [Linear(H,H) act] x L of one net on the masked input; returns the pointer
// to that net's W3.  h[] receives the last hidden activation.
template <int H, int ACT>
__device__ __forceinline__ const float* mlp_hidden(const float* __restrict__ w, int L, int nin, int i0,
                                                   const float* __restrict__ y, int ys, float (&h)[H]) {
  const float* b1 = w + nin * H;
#pragma unroll
  for (int j = 0; j < H; ++j) h[j] = b1[j];
  const float* yp = y + i0 * ys;
  for (int a = 0; a < nin; ++a) {
    float v = yp[0];
    yp += 2 * ys;
    const float4* wr = reinterpret_cast<const float4*>(w + a * H);
#pragma unroll
    for (int j4 = 0; j4 < H / 4; ++j4) {
      float4 q = wr[j4];
      h[4 * j4 + 0] = fmaf(q.x, v, h[4 * j4 + 0]);
      h[4 * j4 + 1] = fmaf(q.y, v, h[4 * j4 + 1]);
      h[4 * j4 + 2] = fmaf(q.z, v, h[4 * j4 + 2]);
      h[4 * j4 + 3] = fmaf(q.w, v, h[4 * j4 + 3]);
    }
  }
#pragma unroll
  for (int j = 0; j < H; ++j) h[j] = act_fn<ACT>(h[j]);
  w = b1 + H;
  for (int l = 0; l < L; ++l) {
    float g[H];
    const float* b2 = w + H * H;
#pragma unroll
    for (int j = 0; j < H; ++j) g[j] = b2[j];
#pragma unroll
    for (int k = 0; k < H; ++k) {
      const float4* wr = reinterpret_cast<const float4*>(w + k * H);
      float v = h[k];
#pragma unroll
      for (int j4 = 0; j4 < H / 4; ++j4) {
        float4 q = wr[j4];
        g[4 * j4 + 0] = fmaf(q.x, v, g[4 * j4 + 0]);
        g[4 * j4 + 1] = fmaf(q.y, v, g[4 * j4 + 1]);
        g[4 * j4 + 2] = fmaf(q.z, v, g[4 * j4 + 2]);
        g[4 * j4 + 3] = fmaf(q.w, v, g[4 * j4 + 3]);
      }
    }
#pragma unroll
    for (int j = 0; j < H; ++j) h[j] = act_fn<ACT>(g[j]);
    w = b2 + H;
  }
  return w;
}

template <int H>
__device__ __forceinline__ float dot_row(const float* __restrict__ row, const float (&h)[H]) {
  const float4* wr = reinterpret_cast<const float4*>(row);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
  for (int j4 = 0; j4 < H / 4; ++j4) {
    float4 q = wr[j4];
    a0 = fmaf(q.x, h[4 * j4 + 0], a0);
    a1 = fmaf(q.y, h[4 * j4 + 1], a1);
    a2 = fmaf(q.z, h[4 * j4 + 2], a2);
    a3 = fmaf(q.w, h[4 * j4 + 3], a3);
  }
  return (a0 + a1) + (a2 + a3);
}

// One coupling block applied in place to y.  Returns this block's log-det contribution.
//   inverse: x = (z - t) * exp(-log_s), ld = -sum(log_s)      networks.py:300-309
//   forward: z = x * exp(log_s) + t,    ld = +sum(log_s)      networks.py:289-298
template <int H, bool INVERSE>
__device__ __forceinline__ float coupling_block(const FlowDesc& f, const float* __restrict__ wsm, int k, float* y,
                                                int ys) {
  const int d = f.d, L = f.L;
  const int nin = blk_nin(d, k), i0 = blk_i0(k), nout = blk_nout(d, k), o0 = blk_o0(k);
  float ld = 0.f;
  float ht[H];
  const float* w3t = mlp_hidden<H, 1>(wsm + f.off_t[k], L, nin, i0, y, ys, ht);
  const float* b3t = w3t + nout * H;
  if (f.off_s[k] >= 0) {
    float hs[H];
    const float* w3s = mlp_hidden<H, 0>(wsm + f.off_s[k], L, nin, i0, y, ys, hs);
    const float* b3s = w3s + nout * H;
    float* yp = y + o0 * ys;
#pragma unroll 2
    for (int o = 0; o < nout; ++o) {
      float ls = dot_row<H>(w3s + o * H, hs) + b3s[o];
      float t = dot_row<H>(w3t + o * H, ht) + b3t[o];
      float v = yp[0];
      if (INVERSE) {
        v = (v - t) * expf(-ls);
        ld -= ls;
      } else {
        v = fmaf(v, expf(ls), t);
        ld += ls;
      }
      yp[0] = v;
      yp += 2 * ys;
    }
  } else {  // translate only (scale in {'translate','constant'})
    float* yp = y + o0 * ys;
#pragma unroll 2
    for (int o = 0; o < nout; ++o) {
      float t = dot_row<H>(w3t + o * H, ht) + b3t[o];
      yp[0] = INVERSE ? (yp[0] - t) : (yp[0] + t);
      yp += 2 * ys;
    }
  }
  return ld;
}

// Full flow, in place on y.  networks.py:24-42 (+ ScaleLayer :312-325 when present).
template <int H>
__device__ __forceinline__ float flow_inverse_inplace(const FlowDesc& f, const float* __restrict__ wsm, float* y,
                                                      int ys) {
  float ld = 0.f;
  for (int k = f.B - 1; k >= 0; --k) {
    if (f.flags & NNB_FLOW_CONST_SCALE) {
      float e = expf(-f.cscale[k]);
      for (int i = 0; i < f.d; ++i) y[i * ys] *= e;
      ld -= f.cscale[k];
    }
    ld += coupling_block<H, true>(f, wsm, k, y, ys);
  }
  return ld;
}

template <int H>
__device__ __forceinline__ float flow_forward_inplace(const FlowDesc& f, const float* __restrict__ wsm, float* y,
                                                      int ys) {
  float ld = 0.f;
  for (int k = 0; k < f.B; ++k) {
    ld += coupling_block<H, false>(f, wsm, k, y, ys);
    if (f.flags & NNB_FLOW_CONST_SCALE) {
      float e = expf(f.cscale[k]);
      for (int i = 0; i < f.d; ++i) y[i * ys] *= e;
      ld += f.cscale[k];
    }
  }
  return ld;
}

// ---------------------------------------------------------------------------------------------
// Likelihoods.  T is the arithmetic type the reference's NumPy code ends up in for the given
// input (float32 rows stay float32 until an np.float64 scalar or array is mixed in).  The
// *_rn intrinsics forbid FMA contraction so that +,-,* sequences are bit-identical to NumPy.
// ---------------------------------------------------------------------------------------------
template <typename T> struct Ar;
template <> struct Ar<float> {
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float cosv(float a) { return cosf(a); }
};
template <> struct Ar<double> {
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double cosv(double a) { return cos(a); }
};

#ifdef NNB_USER_TRANSFORM
// u(j): coordinate j of the unit-box point in T, the argument nnb_user_transform reads
template <typename T, typename XG>
struct UnitRow {
  const XG& xg;
  __device__ __forceinline__ T operator()(int j) const { return (T)xg(j); }
};
#endif

// v_i = transform(u)_i in T  (safe_transform, sampler.py:100-108; affine maps run.py:25-44, mcmc.py:111).  A user
// transform (nnest_b200.likelihoods.CudaTransform) is evaluated afresh on every call: no per-chain buffer holds v.
template <typename T, typename XG>
struct Transformed {
  const TargetSmem& tg;
  const XG& xg;
  __device__ __forceinline__ T operator()(int i) const {
#ifdef NNB_USER_TRANSFORM
    if (tg.desc.has_transform == kTransformUser)
      return nnb_user_transform(UnitRow<T, XG>{xg}, i, tg.desc.d, tg.params + (int)tg.ts[0]);
#endif
    T u = (T)xg(i);
    if (!tg.desc.has_transform) return u;
    if (sizeof(T) == 4) return Ar<T>::add(Ar<T>::mul(u, (T)tg.tsf[i]), (T)tg.tbf[i]);
    return Ar<T>::add(Ar<T>::mul(u, (T)tg.ts[i]), (T)tg.tb[i]);
  }
};

// Visit coordinates i = i_begin .. d-1 in order: f(i, v(i)).  With x_dim known at compile time (DFIX > 0) the values of 16
// coordinates are fetched before the first of them is consumed, so that their shared-memory loads are in flight together
// -- a rolled `for (i) acc = g(acc, v(i))` loop pays one load latency plus the dependent arithmetic PER coordinate
// (measured: 2 100 cycles for the 30-dimensional Rosenbrock sum of one warp).  The order of the arithmetic is unchanged.
template <typename T, int DFIX, typename V, typename F>
__device__ __forceinline__ void for_each_coord(int d, int i_begin, const V& v, F f) {
  if constexpr (DFIX > 0) {
    constexpr int CH = 16;
#pragma unroll
    for (int i0 = i_begin; i0 < DFIX; i0 += CH) {
      T c[CH];
#pragma unroll
      for (int j = 0; j < CH; ++j)
        if (i0 + j < DFIX) c[j] = v(i0 + j);
#pragma unroll
      for (int j = 0; j < CH; ++j)
        if (i0 + j < DFIX) f(i0 + j, c[j]);
    }
  } else {
    for (int i = i_begin; i < d; ++i) f(i, v(i));
  }
}

// numpy's pairwise summation of v(i)^2-style terms for n <= 128 (np.sum of a contiguous 1-D array).
template <typename T, typename F>
__device__ __forceinline__ T np_pairwise_sum(int n, F term) {
  if (n < 8) {
    T r = (T)0;
    for (int i = 0; i < n; ++i) r = Ar<T>::add(r, term(i));
    return r;
  }
  T r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = term(j);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = Ar<T>::add(r[j], term(i + j));
  }
  T res = Ar<T>::add(Ar<T>::add(Ar<T>::add(r[0], r[1]), Ar<T>::add(r[2], r[3])),
                     Ar<T>::add(Ar<T>::add(r[4], r[5]), Ar<T>::add(r[6], r[7])));
  for (; i < n; ++i) res = Ar<T>::add(res, term(i));
  return res;
}

// Returns the likelihood value as double plus whether the reference's result is float32-typed
// (matters only for the -1e100 clamp of safe_loglike, sampler.py:128).
template <typename T, typename XG, int DFIX = 0>   // DFIX > 0: x_dim known at compile time
__device__ __forceinline__ double loglike_T(const TargetSmem& tg, const XG& xg) {
  using A = Ar<T>;
  const int d = DFIX > 0 ? DFIX : tg.desc.d;
  Transformed<T, XG> v{tg, xg};
  double out;
  bool f32_typed = false;
  switch (tg.desc.like_id) {
    case NNB_LIKE_ROSENBROCK: {  // likelihoods.py:50-51, left-to-right sum in T
      T acc = (T)0;
      T prev = v(0);
      for_each_coord<T, DFIX>(d, 1, v, [&](int, T cur) {
        T t1 = A::sub(cur, A::mul(prev, prev));
        T t2 = A::sub((T)1, prev);
        acc = A::add(acc, A::add(A::mul((T)100, A::mul(t1, t1)), A::mul(t2, t2)));
        prev = cur;
      });
      out = -(double)acc;
      f32_typed = sizeof(T) == 4;
      break;
    }
    case NNB_LIKE_HIMMELBLAU: {  // likelihoods.py:69-70
      T x0 = v(0), x1 = v(1);
      T a = A::sub(A::add(A::mul(x0, x0), x1), (T)11);
      T b = A::sub(A::add(x0, A::mul(x1, x1)), (T)7);
      out = (double)A::sub(-A::mul(a, a), A::mul(b, b));
      f32_typed = sizeof(T) == 4;
      break;
    }
    case NNB_LIKE_GAUSSIAN: {  // likelihoods.py:84-86 ; closed form (DESIGN.md), always float64 like scipy
      double rho = tg.params[0];
      double s1 = 0.0, s2 = 0.0;
      for_each_coord<T, DFIX>(d, 0, v, [&](int, T vi) {
        double xi = (double)vi;
        s1 += xi;
        s2 = fma(xi, xi, s2);
      });
      double a = 1.0 - rho, bden = 1.0 - rho + d * rho;
      double logdet = (d - 1) * log(a) + log(bden);
      double quad = (s2 - rho * s1 * s1 / bden) / a;
      out = -0.5 * (quad + logdet + d * 1.8378770664093453);
      break;
    }
    case NNB_LIKE_EGGBOX: {  // likelihoods.py:104-106
      T chi = A::cosv(v(0) / (T)2);
      for (int i = 1; i < d; ++i) chi = A::mul(chi, A::cosv(v(i) / (T)2));
      T b = A::add((T)2, chi);
      T b2 = A::mul(b, b);
      out = (double)A::mul(A::mul(b2, b2), b);
      f32_typed = sizeof(T) == 4;
      break;
    }
    case NNB_LIKE_GAUSSIAN_MIX: {  // likelihoods.py:153-162,182-189
      double sep = tg.params[0], sigma = tg.params[1];
      int nc = (int)tg.params[2];
      T two_s2 = (T)(2.0 * sigma * sigma);
      double cst = log(6.283185307179586 * sigma * sigma) * d / 2.0;
      double a[4];
      double m = -INFINITY;
      for (int k = 0; k < nc; ++k) {
        T p0 = (T)(k == 2 ? sep : (k == 3 ? -sep : 0.0));
        T p1 = (T)(k == 0 ? sep : (k == 1 ? -sep : 0.0));
        T s = np_pairwise_sum<T>(d, [&](int i) {
          T t = v(i);
          if (i == 0) t = A::sub(t, p0);
          if (i == 1) t = A::sub(t, p1);
          return A::mul(t, t);
        });
        a[k] = ((double)(-(s / two_s2)) - cst) + log(tg.params[3 + k]);
        m = fmax(m, a[k]);
      }
      double acc = 0.0;
      for (int k = 0; k < nc; ++k) acc += exp(a[k] - m);
      out = m + log(acc);
      break;
    }
    case NNB_LIKE_GAUSSIAN_SHELL: {  // likelihoods.py:126-128 (center is an int64/float64 array -> float64)
      double sigma = tg.params[0], rshell = tg.params[1];
      double s = np_pairwise_sum<double>(d, [&](int i) {
        double t = tg.params[2 + i] - (double)v(i);
        return t * t;
      });
      double rad = sqrt(s);
      out = -((rad - rshell) * (rad - rshell)) / (2.0 * sigma * sigma);
      break;
    }
#ifdef NNB_USER_LOGLIKE
    case NNB_LIKE_USER: {  // the user's CUDA C++ (nnest_b200.likelihoods.CudaLikelihood), compiled in by nnb_jit.cu
      out = nnb_user_loglike(v, d, tg.params);
      f32_typed = sizeof(T) == 4;
      break;
    }
#endif
    default:
      out = __longlong_as_double(0x7ff8000000000000LL);
  }
  if (!isfinite(out)) out = f32_typed ? -INFINITY : -1e100;  // sampler.py:128
  return out;
}

// safe_prior (sampler.py:143-163) with UniformPrior (priors.py:39-43): 0 or -inf.
template <typename T, typename XG, int DFIX = 0>
__device__ __forceinline__ double prior_T(const TargetSmem& tg, const XG& xg) {
  const int d = DFIX > 0 ? DFIX : tg.desc.d;
  if (tg.desc.prior_kind == NNB_PRIOR_NONE) return 0.0;
  bool bad = false;
  if (tg.desc.prior_kind == NNB_PRIOR_BOX_U) {
    if (sizeof(xg(0)) == 4) {   // float32 point against pre-rounded float32 bounds: same truth value, no FP64
      for_each_coord<float, DFIX>(d, 0, xg, [&](int i, float u) { bad |= (u < tg.lof[i]) | (u > tg.hif[i]); });
    } else {
      for (int i = 0; i < d; ++i) {
        double u = (double)xg(i);
        bad |= (u < tg.lo[i]) | (u > tg.hi[i]);
      }
    }
  } else {
    Transformed<T, XG> v{tg, xg};
    for_each_coord<T, DFIX>(d, 0, v, [&](int i, T vi) {
      double t = (double)vi;
      bad |= (t < tg.lo[i]) | (t > tg.hi[i]);
    });
  }
  return bad ? -INFINITY : 0.0;
}

template <typename XG, int DFIX = 0>
__device__ __forceinline__ double loglike_any(const TargetSmem& tg, const XG& xg, bool in_f64) {
  if (tg.desc.compute_f64 || in_f64) return loglike_T<double, XG, DFIX>(tg, xg);
  return loglike_T<float, XG, DFIX>(tg, xg);
}
template <typename XG, int DFIX = 0>
__device__ __forceinline__ double prior_any(const TargetSmem& tg, const XG& xg, bool in_f64) {
  if (tg.desc.compute_f64 || in_f64) return prior_T<double, XG, DFIX>(tg, xg);
  return prior_T<float, XG, DFIX>(tg, xg);
}

// ---------------------------------------------------------------------------------------------
// Per-step grid barrier of the persistent (cooperative) MCMC kernels.  The only thing the CTAs exchange is the step's
// accept count, so arrival and payload travel in ONE 64-bit reduction (arrivals << 32 | accepted): no fence, no second
// word to read back -- two L2 round trips (the RED and one successful poll) instead of five.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void grid_arrive(unsigned long long* word, unsigned int accepted) {
  atomicAdd(word, (1ull << 32) | (unsigned long long)accepted);
}
__device__ __forceinline__ unsigned int grid_wait(const unsigned long long* word, unsigned int n_ctas) {
  unsigned long long w;
  for (;;) {
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(word) : "memory");
    if ((unsigned int)(w >> 32) >= n_ctas) break;
    __nanosleep(20);
  }
  return (unsigned int)(w & 0xffffffffull);
}

// ---------------------------------------------------------------------------------------------
// CTA-wide helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned int block_count(bool pred) { return (unsigned int)__syncthreads_count(pred); }

__device__ __forceinline__ unsigned int block_sum_u32(unsigned int v, unsigned int* red /* >= 32 words smem */) {
  v = __reduce_add_sync(0xffffffffu, v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  unsigned int t = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
  return t;
}

}  // namespace nnb
