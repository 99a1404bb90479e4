// nnb_spline.cuh -- neural-spline flow of the reference (its default flow='spline'), per-sample arithmetic.
//
// Used by the kernels of nnb_spline.cu (batched flow maps, chain start, fused MCMC step for flow='spline').  The
// functions are __host__ __device__ so that the same arithmetic is also checked on the CPU against goldens recorded
// from the real reference (oracle/spline_host.cpp compiles this header with g++; tests/test_oracle_spline.py).
// Vectors are addressed with a stride (x[i * xs]): 1 on the host, the CTA width in the kernels (column layout, conflict
// free).  `empty` (optional) is set when a coupling call finds NONE of its coordinates inside the tail bound: evaluated
// on a one-sample batch the reference's RQS raises ValueError('No input values') there (networks.py:464-465), which
// Sampler._mcmc_sample turns into a skipped proposal (sampler.py:320-324).
//
// Reference (nnest/networks.py): MLP :401-417, unconstrained_RQS / RQS :425-553, NSF_CL :556-619, Invertible1x1Conv
// :622-653, ActNorm :656-695, SingleSpeedSpline :698-705 = [ActNorm, 1x1 conv, NSF_CL] x num_blocks, 8 bins, tail bound 3.
// Quirks kept: the bin widths / heights are soft-maxed twice (NSF_CL scales the first softmax by 2B, RQS soft-maxes again);
// the derivatives go through softplus twice; the last knot is nudged by 1e-6 for the bin search only; identity outside the
// tail bound; the boundary derivatives are min_derivative + softplus(log(exp(1 - min_derivative) - 1)).
//
// Packed parameters of one flow (floats), block after block (see oracle/spline.py: pack_for_kernel):
//   s[d] t[d]                      ActNorm: y = x exp(s) + t
//   Wc[d*d] Wci[d*d] ldc[1]        1x1 convolution: y = x Wc (row vector times matrix), Wci = Wc^-1, ldc = sum log|S|
//   f1: W0[H*nlow] b0[H] W1[H*H] b1[H] W2[H*H] b2[H] W3[o1*H] b3[o1]     o1 = (3K-1) nup    (conditioner of the upper half)
//   f2: W0[H*nup]  b0[H] W1[H*H] b1[H] W2[H*H] b2[H] W3[o2*H] b3[o2]     o2 = (3K-1) nlow   (conditioner of the lower half)
// with nlow = d/2 (+1 when d is odd), nup = d - nlow; all matrices row-major (out, in) like nn.Linear.
#pragma once
#ifndef __CUDACC_RTC__
#include <math.h>
#endif

#ifdef __CUDACC__
#define NNB_HD __host__ __device__ __forceinline__
#else
#define NNB_HD inline
#endif

namespace nnb {
namespace spline {

constexpr int kMaxBins = 16;
constexpr int kMaxHidden = 64;
constexpr float kMinBin = 1e-3f;
constexpr float kMinDeriv = 1e-3f;

struct Shape {
  int d, H, blocks, K;
  float bound;
  NNB_HD int nlow() const { return d / 2 + (d & 1); }
  NNB_HD int nup() const { return d - nlow(); }
  NNB_HD int mlp_floats(int nin, int nout) const { return H * nin + H + 2 * (H * H + H) + nout * H + nout; }
  NNB_HD int block_floats() const {
    return 2 * d + 2 * d * d + 1 + mlp_floats(nlow(), (3 * K - 1) * nup()) + mlp_floats(nup(), (3 * K - 1) * nlow());
  }
};

NNB_HD float softplus(float a) { return a > 20.f ? a : log1pf(expf(a)); }
NNB_HD float leaky(float a) { return a > 0.f ? a : 0.2f * a; }

// knot positions cum[0..K] on [-bound, bound] from the K raw conditioner outputs (softmax, x 2B, softmax, minimum width)
NNB_HD void knots(const float* raw, int K, float bound, float* cum) {
  float e[kMaxBins], u[kMaxBins];
  float m = raw[0];
  for (int k = 1; k < K; ++k) m = fmaxf(m, raw[k]);
  float s = 0.f;
  for (int k = 0; k < K; ++k) { e[k] = expf(raw[k] - m); s += e[k]; }
  for (int k = 0; k < K; ++k) u[k] = 2.f * bound * (e[k] / s);
  m = u[0];
  for (int k = 1; k < K; ++k) m = fmaxf(m, u[k]);
  s = 0.f;
  for (int k = 0; k < K; ++k) { e[k] = expf(u[k] - m); s += e[k]; }
  float c = 0.f;
  cum[0] = -bound;
  for (int k = 0; k < K; ++k) {
    c += kMinBin + (1.f - kMinBin * K) * (e[k] / s);
    cum[k + 1] = 2.f * bound * c - bound;
  }
  cum[K] = bound;
}

// derivatives at the K + 1 knots from the K - 1 raw conditioner outputs
NNB_HD void knot_derivatives(const float* raw, int K, float* der) {
  const float edge = (float)log(exp(1.0 - (double)kMinDeriv) - 1.0);
  der[0] = der[K] = kMinDeriv + softplus(edge);
  for (int k = 1; k < K; ++k) der[k] = kMinDeriv + softplus(softplus(raw[k - 1]));
}

NNB_HD int find_bin(const float* cum, int K, float v) {
  int idx = -1;
  for (int k = 0; k < K; ++k) idx += v >= cum[k] ? 1 : 0;
  idx += v >= cum[K] + 1e-6f ? 1 : 0;
  return idx < 0 ? 0 : (idx > K - 1 ? K - 1 : idx);
}

// one coordinate through the rational-quadratic spline defined by raw = [K widths | K heights | K - 1 derivatives];
// returns the new value, adds the log-derivative to ld.  Identity outside [-bound, bound].
NNB_HD float rqs(float v, const float* raw, int K, float bound, bool inverse, float& ld) {
  if (!(v >= -bound && v <= bound)) return v;
  float cw[kMaxBins + 1], ch[kMaxBins + 1], der[kMaxBins + 1];
  knots(raw, K, bound, cw);
  knots(raw + K, K, bound, ch);
  knot_derivatives(raw + 2 * K, K, der);
  const int i = find_bin(inverse ? ch : cw, K, v);
  const float w = cw[i + 1] - cw[i], h = ch[i + 1] - ch[i];
  const float delta = h / w, d0 = der[i], d1 = der[i + 1];
  if (inverse) {
    const float y = v - ch[i];
    const float a = y * (d0 + d1 - 2.f * delta) + h * (delta - d0);
    const float b = h * d0 - y * (d0 + d1 - 2.f * delta);
    const float c = -delta * y;
    const float disc = b * b - 4.f * a * c;
    const float root = (2.f * c) / (-b - sqrtf(disc));
    const float tt = root * (1.f - root);
    const float den = delta + (d0 + d1 - 2.f * delta) * tt;
    const float num = delta * delta * (d1 * root * root + 2.f * delta * tt + d0 * (1.f - root) * (1.f - root));
    ld -= logf(num) - 2.f * logf(den);
    return root * w + cw[i];
  }
  const float theta = (v - cw[i]) / w;
  const float tt = theta * (1.f - theta);
  const float num = h * (delta * theta * theta + d0 * tt);
  const float den = delta + (d0 + d1 - 2.f * delta) * tt;
  const float dnum = delta * delta * (d1 * theta * theta + 2.f * delta * tt + d0 * (1.f - theta) * (1.f - theta));
  ld += logf(dnum) - 2.f * logf(den);
  return ch[i] + num / den;
}

// hidden part of the conditioner MLP: Linear(nin, H) LeakyReLU [Linear(H, H) LeakyReLU] x 2 -> h[H]; returns the pointer
// to the output layer's weights W3 (o x H) followed by b3
NNB_HD const float* mlp_hidden(const float* w, int nin, int H, const float* x, int xs, float* h) {
  float g[kMaxHidden];
  const float* b = w + H * nin;
  for (int j = 0; j < H; ++j) {
    float a = b[j];
    for (int i = 0; i < nin; ++i) a += w[j * nin + i] * x[i * xs];
    h[j] = leaky(a);
  }
  w = b + H;
  for (int l = 0; l < 2; ++l) {
    b = w + H * H;
    for (int j = 0; j < H; ++j) {
      float a = b[j];
      for (int i = 0; i < H; ++i) a += w[j * H + i] * h[i];
      g[j] = leaky(a);
    }
    for (int j = 0; j < H; ++j) h[j] = g[j];
    w = b + H;
  }
  return w;
}

// transform the `m` coordinates tgt[] conditioned on cond[] (ncond values) with the MLP at `w`
NNB_HD void couple(const float* w, int ncond, int m, int H, int K, float bound, bool inverse, const float* cond, float* tgt,
                   int xs, float& ld, int* empty) {
  float h[kMaxHidden], raw[3 * kMaxBins];
  const int P = 3 * K - 1;
  const float* w3 = mlp_hidden(w, ncond, H, cond, xs, h);
  const float* b3 = w3 + m * P * H;
  int inside = 0;
  for (int j = 0; j < m; ++j) {
    const float v = tgt[j * xs];
    if (!(v >= -bound && v <= bound)) continue;   // identity: skip the output layer rows as well
    ++inside;
    for (int q = 0; q < P; ++q) {
      const float* row = w3 + (j * P + q) * H;
      float a = b3[j * P + q];
      for (int i = 0; i < H; ++i) a += row[i] * h[i];
      raw[q] = a;
    }
    tgt[j * xs] = rqs(v, raw, K, bound, inverse, ld);
  }
  if (empty && inside == 0) *empty = 1;
}

// whole flow on one sample, in place on x[d]; tmp[d] scratch.  Returns log|det|.
NNB_HD float flow_forward(const Shape& sh, const float* packed, float* x, float* tmp, int xs = 1, int* empty = nullptr) {
  const int d = sh.d, nlow = sh.nlow(), nup = sh.nup();
  float ld = 0.f;
  for (int k = 0; k < sh.blocks; ++k) {
    const float* p = packed + k * sh.block_floats();
    const float *s = p, *t = p + d, *Wc = p + 2 * d, *ldc = Wc + 2 * d * d;
    for (int i = 0; i < d; ++i) { tmp[i * xs] = x[i * xs] * expf(s[i]) + t[i]; ld += s[i]; }   // ActNorm
    for (int j = 0; j < d; ++j) {                                                            // 1x1 convolution
      float a = 0.f;
      for (int i = 0; i < d; ++i) a += tmp[i * xs] * Wc[i * d + j];
      x[j * xs] = a;
    }
    ld += ldc[0];
    const float* f1 = ldc + 1;
    const float* f2 = f1 + sh.mlp_floats(nlow, (3 * sh.K - 1) * nup);
    couple(f1, nlow, nup, sh.H, sh.K, sh.bound, false, x, x + nlow * xs, xs, ld, empty);    // upper | lower
    couple(f2, nup, nlow, sh.H, sh.K, sh.bound, false, x + nlow * xs, x, xs, ld, empty);    // lower | new upper
  }
  return ld;
}

NNB_HD float flow_inverse(const Shape& sh, const float* packed, float* z, float* tmp, int xs = 1, int* empty = nullptr) {
  const int d = sh.d, nlow = sh.nlow(), nup = sh.nup();
  float ld = 0.f;
  for (int k = sh.blocks - 1; k >= 0; --k) {
    const float* p = packed + k * sh.block_floats();
    const float *s = p, *t = p + d, *Wci = p + 2 * d + d * d, *ldc = p + 2 * d + 2 * d * d;
    const float* f1 = ldc + 1;
    const float* f2 = f1 + sh.mlp_floats(nlow, (3 * sh.K - 1) * nup);
    couple(f2, nup, nlow, sh.H, sh.K, sh.bound, true, z + nlow * xs, z, xs, ld, empty);
    couple(f1, nlow, nup, sh.H, sh.K, sh.bound, true, z, z + nlow * xs, xs, ld, empty);
    for (int j = 0; j < d; ++j) {
      float a = 0.f;
      for (int i = 0; i < d; ++i) a += z[i * xs] * Wci[i * d + j];
      tmp[j * xs] = a;
    }
    ld -= ldc[0];
    for (int i = 0; i < d; ++i) { z[i * xs] = (tmp[i * xs] - t[i]) * expf(-s[i]); ld -= s[i]; }
  }
  return ld;
}

}  // namespace spline
}  // namespace nnb
