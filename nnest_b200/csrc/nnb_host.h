// nnb_host.h -- host-side handle and the per-hidden-size launchers of libnnb.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <string>
#include <vector>

#include "nnb_kernels.cuh"
#include "nnb_tc_consts.h"
#include "nnb_warp_desc.h"

struct nnb_handle {
  int device = 0;
  int sm_count = 0;
  int max_smem = 0;
  int max_smem_per_sm = 0;
  bool has_flow = false, has_target = false;
  nnb::FlowDesc flow{};
  float* d_weights = nullptr;
  size_t weights_cap = 0, weights_tc_cap = 0, weights_warp_cap = 0, weights_spline_cap = 0, target_cap = 0;   // floats / doubles allocated
  nnb::TargetDesc tdesc{};
  double* d_target = nullptr;
  // tensor-core (tcgen05) variant of the MCMC kernel: weights pre-split hi/lo in the UMMA layout
  bool tc_ok = false;
  nnb::TcFlowDesc tcflow{};
  float* d_weights_tc = nullptr;
  nnb::TcConsts tc_consts{};               // biases of the flow in the kernel-parameter layout (nnb_tc_kernels.cuh)
  std::vector<float> target_f32;           // tsf | tbf | lof | hif of the current target (host copy, same values as d_target)
  // neural-spline flow (flow='spline', nnb_spline.cu): parameters stay in global memory
  bool flow_is_spline = false;
  int spline_d = 0, spline_hidden = 0, spline_blocks = 0, spline_bins = 0;
  float spline_bound = 0.f;
  float* d_weights_spline = nullptr;
  // 16-lanes-per-chain variant (small batches): (s, t) weight pairs interleaved
  bool warp_ok = false;
  nnb::WarpFlowDesc warpflow{};
  float* d_weights_warp = nullptr;
  unsigned long long* d_step_counts = nullptr;   // workspace of the cooperative kernels (per-step barrier words)
  int step_counts_cap = 0;
  int coop_supported = 0;
  long long last_launches = 0;             // kernels launched by the last nnb_mcmc_run
  Ctrl* d_ctrl = nullptr;
  Ctrl* h_ctrl = nullptr;  // pinned
  // flow fitting (nnb_train.cu)
  void* d_train_ctrl = nullptr;
  void* h_train_ctrl = nullptr;   // pinned: two result slots (an epoch may be queued behind the one whose losses are read)
  cudaEvent_t train_ev[2] = {nullptr, nullptr};   // "slot k holds the losses of its epoch"
  int train_slot_grid[2] = {0, 0};
  unsigned train_begun = 0, train_ended = 0;      // epochs begun / collected (begun - ended <= 2)
  float* d_train_ws = nullptr;    // gradient exchange buffers + per-CTA Adam moments (several CTAs per mini-batch)
  size_t train_ws_floats = 0;
  double* d_nn_part = nullptr;    // per-block partial sums of nnb_mean_nn_distance
  float* d_nn_ws = nullptr;       // float32 copy of the rows for the prefilter of nnb_mean_nn_distance
  size_t nn_ws_floats = 0;
  int nn_part_cap = 0;
  double* d_stats_ws = nullptr;   // chain diagnostics (nnb_stats.cu)
  struct nnb_jit_state* jit = nullptr;   // user likelihood and its compiled kernels (nnb_jit.cu)
  std::string err;
};

int nnb_fail(nnb_handle* h, int code, const std::string& msg);
int nnb_tc_pack(nnb_handle* h, const float* weights_natural);                         // nnb_tc.cu
int nnb_launch_mcmc_tc(nnb_handle* h, McmcParams p, int steps, cudaStream_t st);      // nnb_tc.cu
int nnb_warp_pack(nnb_handle* h, const float* weights_natural);                       // nnb_warp.cu
int nnb_launch_mcmc_warp(nnb_handle* h, McmcParams p, int steps, cudaStream_t st, bool* ran);   // nnb_warp.cu
long long nnb_warp_capacity(const nnb_handle* h);                                     // nnb_warp.cu
void nnb_jit_free(nnb_handle* h);                                                      // nnb_jit.cu
// the kernel `name` (a template instantiation, e.g. "mcmc_kernel<16, 0>") compiled around the handle's user likelihood;
// nullptr with *rc set on failure
const void* nnb_user_kernel(nnb_handle* h, const std::string& name, int* rc);          // nnb_jit.cu
// whether the handle holds a user likelihood (like) / a user transform (!like) source                   nnb_jit.cu
bool nnb_jit_has_source(const nnb_handle* h, bool like);
int nnb_spline_flow(nnb_handle* h, bool inverse, const float* in, int64_t irs, int64_t ics, float* out, int64_t ors,
                    int64_t ocs, float* logdet, int* empty_out, int64_t n, cudaStream_t st);      // nnb_spline.cu
int nnb_spline_init(nnb_handle* h, const InitParams& p, cudaStream_t st);              // nnb_spline.cu
int nnb_spline_mcmc(nnb_handle* h, McmcParams p, int steps, cudaStream_t st);          // nnb_spline.cu

#define NNB_CUDA(h, call)                                                                        \
  do {                                                                                           \
    cudaError_t e__ = (call);                                                                    \
    if (e__ != cudaSuccess)                                                                      \
      return nnb_fail((h), NNB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));   \
  } while (0)

// (Re)allocate a device buffer only when it has to grow: cudaFree synchronises the whole device, and the flow weights
// are re-installed after every retrain (several times per second in a large run).
template <typename T>
static inline cudaError_t nnb_reserve(T** ptr, size_t* cap, size_t need) {
  if (*ptr && *cap >= need) return cudaSuccess;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr;
  *cap = 0;
  cudaError_t e = cudaMalloc(ptr, need * sizeof(T));
  if (e == cudaSuccess) *cap = need;
  return e;
}

template <typename K>
static inline cudaError_t nnb_set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// The kernel a launcher runs: `builtin` (the ahead-of-time instantiation), or with the user likelihood (NNB_LIKE_USER)
// or the user transform (nnb_set_target_user_transform) selected the same instantiation compiled by NVRTC around the
// user's sources.  `fmt`/`args` spell the instantiation, e.g. ("mcmc_kernel<%d, %d>", H, MODE).  nullptr with *rc set on
// failure.
template <typename... A>
static inline const void* nnb_kernel(nnb_handle* h, const void* builtin, int* rc, const char* fmt, A... args) {
  if (h->tdesc.like_id != NNB_LIKE_USER && h->tdesc.has_transform != nnb::kTransformUser) return builtin;
  char name[128];
  snprintf(name, sizeof(name), fmt, args...);
  return nnb_user_kernel(h, name, rc);
}

static inline int nnb_grid_for(nnb_handle* h, long long n, int ctas_per_sm) {
  long long tiles = (n + nnb::kBlockThreads - 1) / nnb::kBlockThreads;
  long long cap = (long long)h->sm_count * ctas_per_sm;
  return (int)(tiles < cap ? tiles : cap);
}

// One translation unit per hidden size (nnb_h16.cu, nnb_h32.cu, nnb_h64.cu) so they compile in parallel.
template <int H>
struct LaunchH {
  static int flow(nnb_handle* h, bool inverse, const float* in, int64_t irs, int64_t ics, float* out, int64_t ors,
                  int64_t ocs, float* logdet, int64_t n, cudaStream_t st);
  static int init(nnb_handle* h, const InitParams& p, cudaStream_t st);
  static int mcmc(nnb_handle* h, McmcParams p, int steps, cudaStream_t st);
};
extern template struct LaunchH<16>;
extern template struct LaunchH<32>;
extern template struct LaunchH<64>;
