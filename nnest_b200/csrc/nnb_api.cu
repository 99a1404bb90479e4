// nnb_api.cu -- C ABI of libnnb.so (contract: include/nnb.h): handle management, weight packing,
// dispatch to the per-hidden-size kernels, the likelihood kernel launch and the host-side
// live-point scan.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <unistd.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <charconv>
#include <string>
#include <thread>
#include <vector>

#include "nnb_host.h"

using namespace nnb;

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
static std::string g_create_err;

int nnb_fail(nnb_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_err = msg;
  return code;
}
static int fail(nnb_handle* h, int code, const std::string& msg) { return nnb_fail(h, code, msg); }

extern "C" int nnb_abi_version(void) { return NNB_ABI_VERSION; }

extern "C" const char* nnb_last_error(nnb_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int nnb_create(int device, nnb_handle** out) {
  if (!out) return fail(nullptr, NNB_ERR_ARG, "out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(nullptr, NNB_ERR_CUDA,
                std::string("no CUDA device available (libnnb has no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(nullptr, NNB_ERR_ARG, "device index out of range");
  nnb_handle* h = new nnb_handle();
  h->device = device;
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    delete h;
    return fail(nullptr, NNB_ERR_CUDA, cudaGetErrorString(e));
  }
  if (prop.major < 10) {
    delete h;
    return fail(nullptr, NNB_ERR_CUDA, "libnnb is built for sm_100a (Blackwell B200) only");
  }
  h->sm_count = prop.multiProcessorCount;
  h->coop_supported = prop.cooperativeLaunch;
  h->max_smem = (int)prop.sharedMemPerBlockOptin;
  h->max_smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  if ((e = cudaMalloc(&h->d_ctrl, sizeof(Ctrl))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_ctrl, sizeof(Ctrl))) != cudaSuccess) {
    delete h;
    return fail(nullptr, NNB_ERR_CUDA, cudaGetErrorString(e));
  }
  *out = h;
  return NNB_OK;
}

extern "C" void nnb_destroy(nnb_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->d_weights) cudaFree(h->d_weights);
  if (h->d_weights_tc) cudaFree(h->d_weights_tc);
  if (h->d_weights_warp) cudaFree(h->d_weights_warp);
  if (h->d_weights_spline) cudaFree(h->d_weights_spline);
  if (h->d_step_counts) cudaFree(h->d_step_counts);
  if (h->d_target) cudaFree(h->d_target);
  if (h->d_ctrl) cudaFree(h->d_ctrl);
  if (h->h_ctrl) cudaFreeHost(h->h_ctrl);
  if (h->d_train_ctrl) cudaFree(h->d_train_ctrl);
  if (h->h_train_ctrl) cudaFreeHost(h->h_train_ctrl);
  for (cudaEvent_t e : h->train_ev)
    if (e) cudaEventDestroy(e);
  if (h->d_train_ws) cudaFree(h->d_train_ws);
  if (h->d_stats_ws) cudaFree(h->d_stats_ws);
  if (h->d_nn_part) cudaFree(h->d_nn_part);
  if (h->d_nn_ws) cudaFree(h->d_nn_ws);
  nnb_jit_free(h);
  delete h;
}

// Natural (state_dict) order -> packed device layout; see FlowDesc in nnb_device.cuh.
static size_t natural_floats(int d, int H, int L, int B, int flags) {
  size_t net = (size_t)H * d + H + (size_t)L * (H * H + H) + (size_t)d * H + d;
  size_t nets = (flags & NNB_FLOW_TRANSLATE_ONLY) ? 1 : 2;
  return B * nets * net + ((flags & NNB_FLOW_CONST_SCALE) ? B : 0);
}

static void pack_net(const float* src, int d, int H, int L, int k, float* dst) {
  const int nin = blk_nin(d, k), i0 = blk_i0(k), nout = blk_nout(d, k), o0 = blk_o0(k);
  const float* W1 = src;            // (H, d)
  const float* b1 = W1 + (size_t)H * d;
  float* o = dst;
  for (int a = 0; a < nin; ++a)
    for (int j = 0; j < H; ++j) *o++ = W1[(size_t)j * d + (i0 + 2 * a)];
  for (int j = 0; j < H; ++j) *o++ = b1[j];
  const float* p = b1 + H;
  for (int l = 0; l < L; ++l) {
    const float* W2 = p;            // (H, H) [j][k]
    const float* b2 = W2 + (size_t)H * H;
    for (int kk = 0; kk < H; ++kk)
      for (int j = 0; j < H; ++j) *o++ = W2[(size_t)j * H + kk];
    for (int j = 0; j < H; ++j) *o++ = b2[j];
    p = b2 + H;
  }
  const float* W3 = p;              // (d, H)
  const float* b3 = W3 + (size_t)d * H;
  for (int q = 0; q < nout; ++q)
    for (int j = 0; j < H; ++j) *o++ = W3[(size_t)(o0 + 2 * q) * H + j];
  for (int q = 0; q < round4(nout); ++q) *o++ = q < nout ? b3[o0 + 2 * q] : 0.f;
}

extern "C" int nnb_set_flow(nnb_handle* h, int d, int hidden, int num_layers, int num_blocks, int flags,
                            const float* weights, size_t n_floats) {
  if (!h) return NNB_ERR_ARG;
  if (d < 1 || d > NNB_MAX_DIM) return fail(h, NNB_ERR_ARG, "x_dim must be in [1, NNB_MAX_DIM]");
  if (hidden != 16 && hidden != 32 && hidden != 64)
    return fail(h, NNB_ERR_UNSUPPORTED, "hidden_dim must be 16, 32 or 64");
  if (num_layers < 0 || num_layers > 8) return fail(h, NNB_ERR_ARG, "num_layers must be in [0, 8]");
  if (num_blocks < 1 || num_blocks > NNB_MAX_BLOCKS) return fail(h, NNB_ERR_ARG, "num_blocks out of range");
  if ((flags & NNB_FLOW_CONST_SCALE) && !(flags & NNB_FLOW_TRANSLATE_ONLY))
    return fail(h, NNB_ERR_ARG, "NNB_FLOW_CONST_SCALE implies NNB_FLOW_TRANSLATE_ONLY (networks.py:331)");
  if (!weights || n_floats != natural_floats(d, hidden, num_layers, num_blocks, flags))
    return fail(h, NNB_ERR_ARG, "weight buffer size does not match (d, hidden, num_layers, num_blocks, flags)");
  NNB_CUDA(h, cudaSetDevice(h->device));
  FlowDesc f{};
  f.d = d; f.H = hidden; f.L = num_layers; f.B = num_blocks; f.flags = flags;
  const bool tonly = flags & NNB_FLOW_TRANSLATE_ONLY;
  const size_t net_nat = (size_t)hidden * d + hidden + (size_t)num_layers * (hidden * hidden + hidden) +
                         (size_t)d * hidden + d;
  int off = 0;
  for (int k = 0; k < num_blocks; ++k) {
    const int nf = net_floats(d, hidden, num_layers, k);
    if (tonly) {
      f.off_s[k] = -1;
    } else {
      f.off_s[k] = off;
      off += nf;
    }
    f.off_t[k] = off;
    off += nf;
  }
  f.total_floats = off;
  std::vector<float> packed((size_t)off, 0.f);
  const float* src = weights;
  for (int k = 0; k < num_blocks; ++k) {
    if (!tonly) {
      pack_net(src, d, hidden, num_layers, k, packed.data() + f.off_s[k]);
      src += net_nat;
    }
    pack_net(src, d, hidden, num_layers, k, packed.data() + f.off_t[k]);
    src += net_nat;
  }
  for (int k = 0; k < num_blocks; ++k) f.cscale[k] = (flags & NNB_FLOW_CONST_SCALE) ? src[k] : 0.f;
  if (smem_bytes(f.total_floats, target_doubles(d, NNB_MAX_LIKE_PARAMS), d, 2) > (size_t)h->max_smem)
    return fail(h, NNB_ERR_UNSUPPORTED, "flow too large for one CTA's shared memory (reduce x_dim / hidden_dim / blocks)");
  NNB_CUDA(h, nnb_reserve(&h->d_weights, &h->weights_cap, packed.size()));
  NNB_CUDA(h, cudaMemcpy(h->d_weights, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
  h->flow = f;
  h->has_flow = true;
  h->flow_is_spline = false;
  int rc = nnb_tc_pack(h, weights);
  if (rc) return rc;
  return nnb_warp_pack(h, weights);
}

// user: the handle's user transform with its n_tp params tp replaces t_scale / t_shift (nnb_set_target_user_transform)
static int set_target(nnb_handle* h, int d, const nnb_target* t, bool user, const double* tp, int n_tp) {
  if (!h || !t) return NNB_ERR_ARG;
  if (d < 1 || d > NNB_MAX_DIM) return fail(h, NNB_ERR_ARG, "x_dim must be in [1, NNB_MAX_DIM]");
  if (t->like_id == NNB_LIKE_USER && !nnb_jit_has_source(h, true))
    return fail(h, NNB_ERR_STATE, "NNB_LIKE_USER: no user likelihood installed (nnb_set_user_likelihood)");
  if (user) {
    if (!nnb_jit_has_source(h, false))
      return fail(h, NNB_ERR_STATE, "no user transform installed (nnb_set_user_transform)");
    if (t->t_scale || t->t_shift) return fail(h, NNB_ERR_ARG, "a user transform replaces t_scale / t_shift");
    if (n_tp < 0 || (n_tp && !tp)) return fail(h, NNB_ERR_ARG, "bad transform parameter array");
    if (t->n_like_params >= 0 && t->n_like_params + n_tp > NNB_MAX_LIKE_PARAMS)
      return fail(h, NNB_ERR_ARG, "the likelihood's and the transform's parameters together exceed NNB_MAX_LIKE_PARAMS");
  }
  if (t->n_like_params < 0 || t->n_like_params > NNB_MAX_LIKE_PARAMS || (t->n_like_params && !t->like_params))
    return fail(h, NNB_ERR_ARG, "bad likelihood parameter array");
  int need = 0;
  switch (t->like_id) {
    case NNB_LIKE_ROSENBROCK: need = 0; break;
    case NNB_LIKE_HIMMELBLAU: need = 0; if (d != 2) return fail(h, NNB_ERR_ARG, "Himmelblau needs x_dim == 2"); break;
    case NNB_LIKE_GAUSSIAN: need = 1; break;
    case NNB_LIKE_EGGBOX: need = 0; break;
    case NNB_LIKE_GAUSSIAN_MIX:
      need = 3;
      if (d < 2) return fail(h, NNB_ERR_ARG, "GaussianMix needs x_dim >= 2");
      if (t->n_like_params >= 3) {
        int nc = (int)t->like_params[2];
        if (nc < 2 || nc > 4) return fail(h, NNB_ERR_ARG, "GaussianMix needs 2, 3 or 4 components");
        need = 3 + nc;
      }
      break;
    case NNB_LIKE_GAUSSIAN_SHELL: need = 2 + d; break;
    case NNB_LIKE_USER: need = t->n_like_params; break;   // the user's source reads what it was given
    default: return fail(h, NNB_ERR_UNSUPPORTED, "unknown likelihood id (Python likelihoods cannot run on the device: write it in CUDA C++, nnb_set_user_likelihood)");
  }
  if (t->n_like_params != need) return fail(h, NNB_ERR_ARG, "wrong number of likelihood parameters");
  if (t->prior_kind != NNB_PRIOR_NONE && (!t->prior_lo || !t->prior_hi))
    return fail(h, NNB_ERR_ARG, "box prior needs prior_lo / prior_hi");
  if ((t->t_scale == nullptr) != (t->t_shift == nullptr)) return fail(h, NNB_ERR_ARG, "t_scale and t_shift go together");
  NNB_CUDA(h, cudaSetDevice(h->device));
  TargetDesc td{};
  td.like_id = t->like_id; td.n_params = t->n_like_params; td.compute_f64 = t->compute_f64 ? 1 : 0;
  td.prior_kind = t->prior_kind; td.has_transform = t->t_scale ? 1 : 0; td.d = d;
  if (user) {   // the transform's params follow the likelihood's; ts[0] says where they begin (TargetDesc)
    td.has_transform = kTransformUser;
    td.n_params += n_tp;
  }
  std::vector<double> buf((size_t)target_doubles(d, td.n_params), 0.0);
  for (int i = 0; i < t->n_like_params; ++i) buf[i] = t->like_params[i];
  for (int i = 0; user && i < n_tp; ++i) buf[t->n_like_params + i] = tp[i];
  double* ts = buf.data() + td.n_params;
  for (int i = 0; i < d; ++i) {
    ts[i] = t->t_scale ? t->t_scale[i] : 1.0;
    ts[d + i] = t->t_shift ? t->t_shift[i] : 0.0;
    ts[2 * d + i] = t->prior_lo ? t->prior_lo[i] : -INFINITY;
    ts[3 * d + i] = t->prior_hi ? t->prior_hi[i] : INFINITY;
  }
  if (user) ts[0] = (double)t->n_like_params;
  {  // float32 mirrors behind the doubles (see TargetSmem)
    float* ff = reinterpret_cast<float*>(ts + 4 * d);
    for (int i = 0; i < d; ++i) {
      ff[i] = (float)ts[i];
      ff[d + i] = (float)ts[d + i];
      float lo = (float)ts[2 * d + i], hi = (float)ts[3 * d + i];
      if ((double)lo < ts[2 * d + i]) lo = std::nextafterf(lo, INFINITY);     // smallest float >= lo
      if ((double)hi > ts[3 * d + i]) hi = std::nextafterf(hi, -INFINITY);    // largest float <= hi
      ff[2 * d + i] = lo;
      ff[3 * d + i] = hi;
    }
    h->target_f32.assign(ff, ff + 4 * d);
  }
  NNB_CUDA(h, nnb_reserve(&h->d_target, &h->target_cap, buf.size()));
  NNB_CUDA(h, cudaMemcpy(h->d_target, buf.data(), buf.size() * sizeof(double), cudaMemcpyHostToDevice));
  h->tdesc = td;
  h->has_target = true;
  return NNB_OK;
}

extern "C" int nnb_set_target(nnb_handle* h, int d, const nnb_target* t) {
  return set_target(h, d, t, false, nullptr, 0);
}

extern "C" int nnb_set_target_user_transform(nnb_handle* h, int d, const nnb_target* t, const double* transform_params,
                                             int n_transform_params) {
  return set_target(h, d, t, true, transform_params, n_transform_params);
}

template <bool INV>
static int flow_dispatch(nnb_handle* h, const float* in, int64_t irs, int64_t ics, float* out, int64_t ors,
                         int64_t ocs, float* logdet, int64_t n, void* stream) {
  if (!h) return NNB_ERR_ARG;
  if (!h->has_flow) return fail(h, NNB_ERR_STATE, "nnb_set_flow has not been called");
  if (n < 0 || (n > 0 && (!in || !out))) return fail(h, NNB_ERR_ARG, "bad buffer");
  if (n == 0) return NNB_OK;
  NNB_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (h->flow_is_spline) return nnb_spline_flow(h, INV, in, irs, ics, out, ors, ocs, logdet, nullptr, n, st);
  switch (h->flow.H) {
    case 16: return LaunchH<16>::flow(h, INV, in, irs, ics, out, ors, ocs, logdet, n, st);
    case 32: return LaunchH<32>::flow(h, INV, in, irs, ics, out, ors, ocs, logdet, n, st);
    case 64: return LaunchH<64>::flow(h, INV, in, irs, ics, out, ors, ocs, logdet, n, st);
  }
  return fail(h, NNB_ERR_UNSUPPORTED, "hidden_dim");
}

extern "C" int nnb_flow_inverse(nnb_handle* h, const float* z, int64_t z_rs, int64_t z_cs, float* x, int64_t x_rs,
                                int64_t x_cs, float* logdet, int64_t n, void* stream) {
  return flow_dispatch<true>(h, z, z_rs, z_cs, x, x_rs, x_cs, logdet, n, stream);
}

extern "C" int nnb_flow_forward(nnb_handle* h, const float* x, int64_t x_rs, int64_t x_cs, float* z, int64_t z_rs,
                                int64_t z_cs, float* logdet, int64_t n, void* stream) {
  return flow_dispatch<false>(h, x, x_rs, x_cs, z, z_rs, z_cs, logdet, n, stream);
}

extern "C" int nnb_loglike(nnb_handle* h, const void* u, int in_f64, int64_t u_rs, int64_t u_cs, double* logl,
                           double* logp, int64_t n, void* stream) {
  if (!h) return NNB_ERR_ARG;
  if (!h->has_target) return fail(h, NNB_ERR_STATE, "nnb_set_target has not been called");
  if (n < 0 || (n > 0 && !u)) return fail(h, NNB_ERR_ARG, "bad buffer");
  if (n == 0) return NNB_OK;
  NNB_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t sm = smem_bytes(0, target_doubles(h->tdesc.d, h->tdesc.n_params), h->tdesc.d, 0);
  int grid = nnb_grid_for(h, n, 8);
  int rc = NNB_OK;
  const void* fn = in_f64 ? nnb_kernel(h, (const void*)loglike_kernel<double>, &rc, "loglike_kernel<double>")
                          : nnb_kernel(h, (const void*)loglike_kernel<float>, &rc, "loglike_kernel<float>");
  if (!fn) return rc;
  long long rs = u_rs, cs = u_cs, nn = n;
  void* args[] = {(void*)&h->tdesc, (void*)&h->d_target, (void*)&u, (void*)&rs, (void*)&cs, (void*)&logl, (void*)&logp,
                  (void*)&nn};
  NNB_CUDA(h, cudaLaunchKernel(fn, dim3(grid), dim3(kBlockThreads), args, sm, st));
  return NNB_OK;
}

static int check_mcmc_ready(nnb_handle* h) {
  if (!h->has_flow) return fail(h, NNB_ERR_STATE, "nnb_set_flow has not been called");
  if (!h->has_target) return fail(h, NNB_ERR_STATE, "nnb_set_target has not been called");
  if (h->tdesc.d != h->flow.d) return fail(h, NNB_ERR_STATE, "flow and target have different x_dim");
  return NNB_OK;
}

// zero the control block, scale = `scale` (one thread; keeps asynchronous calls free of host-side staging buffers)
static __global__ void ctrl_init_kernel(Ctrl* c, double scale) {
  Ctrl z{};
  z.scale = scale;
  *c = z;
}

extern "C" int nnb_mcmc_init(nnb_handle* h, const nnb_mcmc_init_args* a, void* stream) {
  if (!h || !a) return NNB_ERR_ARG;
  int rc = check_mcmc_ready(h);
  if (rc) return rc;
  if (a->n_chains <= 0 || !a->z || !a->x || !a->logl || !a->logdet || !a->logp)
    return fail(h, NNB_ERR_ARG, "state buffers missing");
  if (a->init_u && a->init_z) return fail(h, NNB_ERR_ARG, "give at most one of init_u / init_z");
  NNB_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  ctrl_init_kernel<<<1, 1, 0, st>>>(h->d_ctrl, 0.0);
  InitParams p{};
  p.n = a->n_chains; p.z = a->z; p.x = a->x; p.logl = a->logl; p.logdet = a->logdet; p.logp = a->logp;
  p.init_u = a->init_u; p.init_z = a->init_z; p.init_logl = a->init_logl;
  p.seed_lo = (unsigned int)(a->seed & 0xffffffffu); p.seed_hi = (unsigned int)(a->seed >> 32);
  p.chain_offset = a->chain_offset; p.start_try = a->start_try; p.ctrl = h->d_ctrl;
  if (h->flow_is_spline) {
    rc = nnb_spline_init(h, p, st);
  } else
  switch (h->flow.H) {
    case 16: rc = LaunchH<16>::init(h, p, st); break;
    case 32: rc = LaunchH<32>::init(h, p, st); break;
    case 64: rc = LaunchH<64>::init(h, p, st); break;
    default: rc = fail(h, NNB_ERR_UNSUPPORTED, "hidden_dim");
  }
  if (rc) return rc;
  if (!a->n_bad_start && !a->ncall) return NNB_OK;   // counters not wanted: stay asynchronous
  NNB_CUDA(h, cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
  NNB_CUDA(h, cudaStreamSynchronize(st));
  if (a->n_bad_start) *a->n_bad_start = (int64_t)h->h_ctrl->nbad;
  if (a->ncall) *a->ncall = (int64_t)h->h_ctrl->ncall;
  return NNB_OK;
}

extern "C" int nnb_mcmc_run(nnb_handle* h, const nnb_mcmc_args* a, void* stream) {
  if (!h || !a) return NNB_ERR_ARG;
  int rc = check_mcmc_ready(h);
  if (rc) return rc;
  if (a->n_chains <= 0 || a->steps < 0 || !a->z || !a->x || !a->logl || !a->logdet || !a->logp)
    return fail(h, NNB_ERR_ARG, "state buffers missing");
  if (a->mode != NNB_MODE_HARD && a->mode != NNB_MODE_MH) return fail(h, NNB_ERR_ARG, "mode");
  if ((a->trace_x != nullptr) != (a->trace_z != nullptr) || (a->trace_x != nullptr) != (a->trace_logl != nullptr))
    return fail(h, NNB_ERR_ARG, "trace_x, trace_z and trace_logl go together");
  if ((a->replay_normals != nullptr) != (a->replay_uniforms != nullptr))
    return fail(h, NNB_ERR_ARG, "replay_normals and replay_uniforms go together");
  NNB_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int d = h->flow.d;
  const long long n = a->n_chains;
  // control block: zero counters, scale = step_size (default 2 / sqrt(d), sampler.py:248-249).  Set by a one-thread kernel
  // rather than a copy from the pinned mirror, so that asynchronous calls can be queued back to back
  ctrl_init_kernel<<<1, 1, 0, st>>>(h->d_ctrl, a->step_size > 0.0 ? a->step_size : 2.0 / std::sqrt((double)d));
  if (a->trace_x) {  // row 0 = state at entry (sampler.py:286-289)
    NNB_CUDA(h, cudaMemcpyAsync(a->trace_x, a->x, sizeof(float) * d * n, cudaMemcpyDeviceToDevice, st));
    NNB_CUDA(h, cudaMemcpyAsync(a->trace_z, a->z, sizeof(float) * d * n, cudaMemcpyDeviceToDevice, st));
    NNB_CUDA(h, cudaMemcpyAsync(a->trace_logl, a->logl, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
  }
  McmcParams p{};
  p.n = n; p.mode = a->mode; p.dynamic = a->dynamic_step_size ? 1 : 0; p.loglstar = a->loglstar;
  p.seed_lo = (unsigned int)(a->seed & 0xffffffffu); p.seed_hi = (unsigned int)(a->seed >> 32);
  p.chain_offset = a->chain_offset; p.step_offset = a->step_offset;
  p.z = a->z; p.x = a->x; p.logl = a->logl; p.logdet = a->logdet; p.logp = a->logp;
  p.trace_x = a->trace_x; p.trace_z = a->trace_z; p.trace_logl = a->trace_logl;
  p.replay_normals = a->replay_normals; p.replay_uniforms = a->replay_uniforms;
  p.dump_normals = a->dump_normals; p.dump_uniforms = a->dump_uniforms;
  p.ctrl = h->d_ctrl;
  if (a->impl < NNB_IMPL_AUTO || a->impl > NNB_IMPL_WARP) return fail(h, NNB_ERR_ARG, "impl");
  if (a->impl == NNB_IMPL_TCGEN05 && !h->tc_ok)
    return fail(h, NNB_ERR_UNSUPPORTED, "tcgen05 path needs hidden_dim == 16, 2 <= x_dim <= 63 and scale == ''");
  if (a->impl == NNB_IMPL_WARP && !h->warp_ok)
    return fail(h, NNB_ERR_UNSUPPORTED, "the 16-lanes-per-chain kernel needs hidden_dim == 16 and scale == ''");
  bool use_warp = false;
  if (h->flow_is_spline) {
    if (a->impl != NNB_IMPL_AUTO && a->impl != NNB_IMPL_FFMA)
      return fail(h, NNB_ERR_UNSUPPORTED, "flow='spline' runs the FP32 one-thread-per-chain kernel only");
    if (a->steps > 0) {
      rc = nnb_spline_mcmc(h, p, a->steps, st);
      if (rc) return rc;
    }
    if (a->launches_out) *a->launches_out = a->steps > 0 ? h->last_launches : 0;
    if (a->impl_out) *a->impl_out = NNB_IMPL_FFMA;
    NNB_CUDA(h, cudaGetLastError());
    if (!a->scale_out && !a->ncall_out && !a->naccept_out) return NNB_OK;
    return nnb_mcmc_result(h, a->scale_out, a->ncall_out, a->naccept_out, stream);
  }
  if (a->steps > 0 && h->warp_ok && (a->impl == NNB_IMPL_WARP || (a->impl == NNB_IMPL_AUTO && n <= nnb_warp_capacity(h) * 3 / 4))) {
    rc = nnb_launch_mcmc_warp(h, p, a->steps, st, &use_warp);
    if (rc) return rc;
    if (!use_warp && a->impl == NNB_IMPL_WARP)
      return fail(h, NNB_ERR_UNSUPPORTED,
                  "the 16-lanes-per-chain kernel holds every chain co-resident: too many chains (or a single dynamic step)");
  }
  const bool use_tc = !use_warp && h->tc_ok && a->impl != NNB_IMPL_FFMA;
  if (use_warp) {
  } else if (a->steps > 0 && use_tc) {
    rc = nnb_launch_mcmc_tc(h, p, a->steps, st);
    if (rc) return rc;
  } else if (a->steps > 0) {
    switch (h->flow.H) {
      case 16: rc = LaunchH<16>::mcmc(h, p, a->steps, st); break;
      case 32: rc = LaunchH<32>::mcmc(h, p, a->steps, st); break;
      case 64: rc = LaunchH<64>::mcmc(h, p, a->steps, st); break;
      default: rc = fail(h, NNB_ERR_UNSUPPORTED, "hidden_dim");
    }
    if (rc) return rc;
  }
  if (a->launches_out) *a->launches_out = a->steps > 0 ? h->last_launches : 0;
  if (a->impl_out) *a->impl_out = use_warp ? NNB_IMPL_WARP : (use_tc ? NNB_IMPL_TCGEN05 : NNB_IMPL_FFMA);
  NNB_CUDA(h, cudaGetLastError());
  // no result requested: the call stays asynchronous (results of the last run: nnb_mcmc_result)
  if (!a->scale_out && !a->ncall_out && !a->naccept_out) return NNB_OK;
  return nnb_mcmc_result(h, a->scale_out, a->ncall_out, a->naccept_out, stream);
}

extern "C" int nnb_mcmc_result(nnb_handle* h, double* scale_out, int64_t* ncall_out, int64_t* naccept_out, void* stream) {
  if (!h) return NNB_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  NNB_CUDA(h, cudaSetDevice(h->device));
  NNB_CUDA(h, cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
  NNB_CUDA(h, cudaStreamSynchronize(st));
  if (scale_out) *scale_out = h->h_ctrl->scale;
  if (ncall_out) *ncall_out = (int64_t)h->h_ctrl->ncall;
  if (naccept_out) *naccept_out = (int64_t)h->h_ctrl->naccept;
  return NNB_OK;
}

extern "C" int64_t nnb_consume_scan(const float* first, const float* last, const double* logl_last, int64_t n_chains,
                                    int d, double loglstar, int64_t* nb) {
  if (!first || !last || !logl_last || !nb) return -1;
  for (int64_t ib = *nb; ib < n_chains; ++ib) {
    *nb = ib + 1;
    const float* a = first + ib * d;
    const float* b = last + ib * d;
    bool all_differ = true;
    for (int i = 0; i < d; ++i) all_differ &= (a[i] != b[i]);   // np.all(samples[ib,0,:] != samples[ib,-1,:])
    if (all_differ && logl_last[ib] > loglstar) return ib;
  }
  return -1;
}

// Which point is the worst, iteration after iteration (np.argmin(active_logl): first index among equal minima), without
// an O(nlive) pass -- or a 16-level heap walk -- per iteration.  A replacement always takes the place of the current minimum,
// so the points present at the start leave in sorted order: they are sorted ONCE per call, and the points that came in during the call wait in a small min-heap.  The worst is the smaller of the two fronts under
// the total order (logl, slot).
namespace {
struct LiveNode { double key; int64_t slot; };
inline bool live_less(const LiveNode& a, const LiveNode& b) { return a.key < b.key || (a.key == b.key && a.slot < b.slot); }

// The `need` smallest live points (and every tie of the largest of them) in (logl, slot) order: the points are reduced
// to an order-preserving integer image of the key, the need-th smallest image is found by selection, and only the points at
// or below it go through a stable byte-wise radix sort (slots enter in increasing order, so equal keys stay in slot order;
// passes whose byte is the same for every point are skipped).  A call consumes at most as many points as it has chains left
// and iterations allowed -- on average a third of a 65 536-point live set -- and std::sort with the pair comparator would
// cost ten times the radix passes.
void sort_live(const double* logl, int64_t n, int64_t need, std::vector<LiveNode>& out) {
  struct Img { uint64_t k; int64_t slot; };
  // scratch kept between calls (a run makes hundreds of them; fresh megabyte-sized vectors are page faults every time)
  static thread_local std::vector<Img> a, b;
  static thread_local std::vector<uint64_t> keys;
  keys.resize((size_t)n);
  for (int64_t i = 0; i < n; ++i) {
    const double v = logl[i] + 0.0;               // -0.0 == +0.0 for np.argmin: one image for both
    uint64_t u;
    memcpy(&u, &v, 8);
    keys[(size_t)i] = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
  }
  uint64_t thr = ~0ull;
  if (need < n) {
    static thread_local std::vector<uint64_t> sel;
    sel = keys;
    std::nth_element(sel.begin(), sel.begin() + (need - 1), sel.end());
    thr = sel[(size_t)(need - 1)];
  }
  a.clear();
  a.reserve((size_t)n);
  size_t hist[8][256] = {};
  for (int64_t i = 0; i < n; ++i) {
    const uint64_t u = keys[(size_t)i];
    if (u > thr) continue;
    a.push_back(Img{u, i});
    for (int p = 0; p < 8; ++p) ++hist[p][(u >> (8 * p)) & 255];
  }
  const size_t m = a.size();
  b.resize(m);
  Img* src = a.data();
  Img* dst = b.data();
  for (int p = 0; p < 8; ++p) {
    size_t* h = hist[p];
    bool single = false;
    for (int j = 0; j < 256; ++j) single |= (h[j] == m);
    if (single) continue;
    size_t sum = 0;
    for (int j = 0; j < 256; ++j) { const size_t c = h[j]; h[j] = sum; sum += c; }
    for (size_t i = 0; i < m; ++i) dst[h[(src[i].k >> (8 * p)) & 255]++] = src[i];
    std::swap(src, dst);
  }
  out.resize(m);
  for (size_t i = 0; i < m; ++i) out[i] = LiveNode{logl[src[i].slot], src[i].slot};
}

struct NewHeap {   // binary min-heap of the replacements, key stored with the slot
  std::vector<LiveNode> h;
  bool empty() const { return h.empty(); }
  const LiveNode& top() const { return h[0]; }
  void push(LiveNode x) {
    size_t i = h.size();
    h.push_back(x);
    while (i > 0) {
      const size_t p = (i - 1) / 2;
      if (!live_less(x, h[p])) break;
      h[i] = h[p];
      i = p;
    }
    h[i] = x;
  }
  void pop() {
    const LiveNode x = h.back();
    h.pop_back();
    const size_t n = h.size();
    if (!n) return;
    size_t i = 0;
    for (;;) {
      size_t c = 2 * i + 1;
      if (c >= n) break;
      if (c + 1 < n && live_less(h[c + 1], h[c])) ++c;
      if (!live_less(h[c], x)) break;
      h[i] = h[c];
      i = c;
    }
    h[i] = x;
  }
};
}  // namespace

extern "C" int64_t nnb_ns_consume(const double* active_logl, int64_t nlive, const float* first, const float* last,
                                  const double* logl_last, int64_t n_chains, int d, int64_t* nb, int64_t max_iters,
                                  int64_t* worst_out, int64_t* chain_out, int64_t* prev_out, double* loglstar_out,
                                  double* maxlogl_out, int* exhausted) {
  if (!active_logl || nlive <= 0 || !first || !last || !logl_last || !nb || !worst_out || !chain_out || !prev_out ||
      !loglstar_out || !maxlogl_out || !exhausted || max_iters < 0)
    return NNB_ERR_ARG;
  for (int64_t i = 0; i < nlive; ++i)
    if (active_logl[i] != active_logl[i]) return NNB_ERR_ARG;   // NaN has no place in the ordering
  *exhausted = 0;
  if (max_iters == 0) return 0;
  const int64_t nb0 = *nb < 0 ? 0 : *nb;
  const int64_t left = n_chains > nb0 ? n_chains - nb0 : 0;
  // np.all(first != last, axis=1) of the chains not yet consumed does not depend on the constraint: evaluated once, by a few
  // threads (two 8 MB arrays at config-4 size); the per-iteration scan then reads one byte and one double per chain
  static thread_local std::vector<unsigned char> moved;
  static thread_local std::vector<LiveNode> init;
  static thread_local NewHeap fresh;
  static thread_local std::vector<double> cur;
  static thread_local std::vector<int64_t> writer;
  moved.resize((size_t)left);
  {
    unsigned hw = std::thread::hardware_concurrency();
    const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<unsigned>(hw ? hw : 1u, 8u), left * d / 65536));
    unsigned char* flags = moved.data();          // (the vector itself is thread_local: the workers must not name it)
    auto work = [=](int64_t a, int64_t b) {
      for (int64_t c = a; c < b; ++c) {
        const float* x = first + (nb0 + c) * d;
        const float* y = last + (nb0 + c) * d;
        bool all_differ = true;
        for (int i = 0; i < d; ++i) all_differ &= (x[i] != y[i]);
        flags[c] = all_differ ? 1 : 0;
      }
    };
    if (nt <= 1) {
      work(0, left);
    } else {
      std::vector<std::thread> th;
      const int64_t per = (left + nt - 1) / nt;
      for (int t = 0; t < nt; ++t) th.emplace_back(work, std::min(left, t * per), std::min(left, (t + 1) * per));
      for (auto& x : th) x.join();
    }
  }
  // every iteration consumes at least one chain, the last one started may find none: at most `pops` minima are needed
  const int64_t pops = std::min<int64_t>(std::min(max_iters, left + 1), nlive);
  sort_live(active_logl, nlive, pops, init);      // init.size() >= pops
  const int64_t ninit = (int64_t)init.size();
  int64_t front = 0;   // next of the initial points to leave
  fresh.h.clear();
  fresh.h.reserve((size_t)pops);
  cur.assign(active_logl, active_logl + nlive);   // current value of every slot
  writer.assign((size_t)nlive, -1);
  double maxl = active_logl[0];
  for (int64_t i = 1; i < nlive; ++i) maxl = active_logl[i] > maxl ? active_logl[i] : maxl;
  int64_t k = 0;
  for (; k < max_iters; ++k) {
    // at most one initial point leaves per iteration and at most `pops` iterations take one: front < ninit here unless the
    // whole live set has been replaced (pops == nlive), in which case the heap holds every live point
    const bool from_init = front < ninit && (fresh.empty() || live_less(init[(size_t)front], fresh.top()));
    if (!from_init && fresh.empty()) return NNB_ERR_STATE;   // cannot happen (see above)
    const int64_t worst = from_init ? init[(size_t)front].slot : fresh.top().slot;
    const double loglstar = cur[(size_t)worst];
    worst_out[k] = worst;
    loglstar_out[k] = loglstar;
    prev_out[k] = writer[(size_t)worst];
    int64_t ib = -1;
    for (int64_t c = (*nb < 0 ? 0 : *nb); c < n_chains; ++c) {        // nnb_consume_scan with the precomputed flags
      *nb = c + 1;
      if (moved[(size_t)(c - nb0)] && logl_last[c] > loglstar) { ib = c; break; }
    }
    if (ib < 0) {
      *exhausted = 1;
      return k;
    }
    const double nl = logl_last[ib];
    chain_out[k] = ib;
    writer[(size_t)worst] = k;
    if (from_init) ++front; else fresh.pop();
    fresh.push(LiveNode{nl, worst});
    cur[(size_t)worst] = nl;
    if (loglstar == maxl) {   // every live point was equal: recompute (np.max after the replacement)
      maxl = cur[0];
      for (int64_t i = 1; i < nlive; ++i) maxl = cur[(size_t)i] > maxl ? cur[(size_t)i] : maxl;
    } else if (nl > maxl) {
      maxl = nl;
    }
    maxlogl_out[k] = maxl;
  }
  return k;
}

// ---- row movements of a run of nested-sampling iterations (include/nnb.h) -----------------------------------------------
namespace {
template <typename F>
void parallel_for(int64_t n, int64_t grain, F fn) {   // fn(begin, end, thread index, thread count)
  unsigned hw = std::thread::hardware_concurrency();
  int nt = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<unsigned>(hw ? hw : 1u, 8u), (n + grain - 1) / grain));
  if (nt <= 1) { fn((int64_t)0, n, 0, 1); return; }
  std::vector<std::thread> th;
  const int64_t per = (n + nt - 1) / nt;
  for (int t = 0; t < nt; ++t) th.emplace_back([=] { fn(std::min(n, t * per), std::min(n, (t + 1) * per), t, nt); });
  for (auto& x : th) x.join();
}
}  // namespace

extern "C" int nnb_gather_rows_f32(const float* src, int64_t n_src, int d, const int64_t* idx, int64_t n, double* out) {
  if (!src || !idx || !out || d <= 0 || n < 0) return NNB_ERR_ARG;
  for (int64_t i = 0; i < n; ++i)
    if (idx[i] < 0 || idx[i] >= n_src) return NNB_ERR_ARG;
  parallel_for(n, 4096, [=](int64_t a, int64_t b, int, int) {
    for (int64_t i = a; i < b; ++i) {
      const float* s = src + idx[i] * d;
      double* o = out + i * d;
      for (int j = 0; j < d; ++j) o[j] = (double)s[j];
    }
  });
  return NNB_OK;
}

extern "C" int nnb_ns_apply(const int64_t* worst, const int64_t* prev, int64_t n_ev, int64_t n_done, int d,
                            const double* new_u, const double* new_v, const double* new_logl, double* active_u,
                            double* active_v, double* active_logl, int64_t nlive, double* dead_out) {
  if (!worst || !prev || !active_u || !active_v || !active_logl || !dead_out || d <= 0 || n_ev < 0 || n_done < 0 ||
      n_done > n_ev || (n_done > 0 && (!new_u || !new_v || !new_logl)))
    return NNB_ERR_ARG;
  for (int64_t i = 0; i < n_ev; ++i)
    if (worst[i] < 0 || worst[i] >= nlive || prev[i] >= n_done || prev[i] >= i) return NNB_ERR_ARG;
  const size_t row = sizeof(double) * (size_t)d;
  // dead points first: they read the live set as it was before this call's replacements
  parallel_for(n_ev, 4096, [=](int64_t a, int64_t b, int, int) {
    for (int64_t i = a; i < b; ++i)
      memcpy(dead_out + i * d, prev[i] >= 0 ? new_v + prev[i] * d : active_v + worst[i] * d, row);
  });
  // replacements in iteration order; thread t owns the slots with slot % T == t, so "the last write wins" holds per slot
  parallel_for(n_done >= 8192 ? 8 * 16384 : (n_done > 0 ? 1 : 0), 16384, [=](int64_t, int64_t, int t, int nt) {
    for (int64_t i = 0; i < n_done; ++i) {
      const int64_t s = worst[i];
      if ((int)(s % nt) != t) continue;
      memcpy(active_u + s * d, new_u + i * d, row);
      memcpy(active_v + s * d, new_v + i * d, row);
      active_logl[s] = new_logl[i];
    }
  });
  return NNB_OK;
}

// Chain files of the reference (nnest/sampler.py:494-511): one row per sample, every number '%.5E', single spaces.
// Rows are formatted by several host threads into private buffers, batch by batch, and written in order by the calling
// thread WHILE the next batch is being formatted (two sets of buffers): a config-4 chain is 3.6 GB of text, and the
// page-cache write of a batch takes about as long as formatting it.
namespace {
// 10^k, k in [-kP10, kP10], as an unevaluated sum hi + lo of two doubles (taken from the x87 80-bit value: relative
// error < 2^-63), built once.
constexpr int kP10 = 300;
struct Pow10Table {
  double hi[2 * kP10 + 1], lo[2 * kP10 + 1];
  Pow10Table() {
    for (int k = -kP10; k <= kP10; ++k) {
      const long double p = powl(10.0L, (long double)k);
      hi[k + kP10] = (double)p;
      lo[k + kP10] = (double)(p - (long double)hi[k + kP10]);
    }
  }
};
const Pow10Table g_pow10;

// The slow, always-correct spelling: std::to_chars(scientific, 5) is the correctly rounded form printf("%.5e") prints
// (identical bytes, 3x faster than snprintf); the reference writes an upper-case E.
inline char* format_5e_exact(char* w, double v) {
  if (std::isfinite(v)) {
    auto r = std::to_chars(w, w + 16, v, std::chars_format::scientific, 5);
    for (char* q = w; q < r.ptr; ++q)
      if (*q == 'e') *q = 'E';
    return r.ptr;
  }
  if (v != v) { memcpy(w, "NAN", 3); return w + 3; }     // Python prints NAN whatever the sign bit (printf: "-NAN")
  return w + snprintf(w, 16, "%.5E", v);                  // INF / -INF
}

// One value as printf("%.5E") / Python's '%.5E' % v spell it; returns the end of the text.
// Fast path: the six significant digits are round(|v| * 10^(5 - e)) with the product carried as a double-double
// (error < 1e-12 of a unit in the last digit); whenever the fraction is within 1e-6 of a rounding tie -- or the value is
// zero, non-finite or outside 1e-290 .. 1e290 -- the exact formatter decides.  A config-4 chain file is 285 M numbers.
inline char* format_5e(char* w, double v) {
  const double a = std::fabs(v);
  if (!(a >= 1e-290 && a <= 1e290)) return format_5e_exact(w, v);
  int e2;
  std::frexp(a, &e2);                                         // a = f * 2^e2, f in [0.5, 1)
  int e10 = (int)std::floor((e2 - 1) * 0.30102999566398120);  // floor(log10(2^(e2-1))) <= floor(log10(a)), off by <= 1
  for (int attempt = 0; attempt < 2; ++attempt) {
    const int k = 5 - e10 + kP10;
    const double hi = g_pow10.hi[k], lo = g_pow10.lo[k];
    const double p = a * hi;
    const double err = std::fma(a, hi, -p) + a * lo;
    if (p >= 999999.75) { ++e10; continue; }                  // (also sends p within rounding of 10^6 up a decade)
    if (p < 99999.75) return format_5e_exact(w, v);            // cannot happen for the estimate above; stay safe
    const double fl = std::floor(p);
    const double frac = (p - fl) + err;
    if (std::fabs(frac - 0.5) < 1e-6) return format_5e_exact(w, v);
    long m = (long)fl + (frac > 0.5 ? 1 : 0);
    if (m < 100000) return format_5e_exact(w, v);             // p in [99999.75, 100000): a decade boundary, rare
    if (m >= 1000000) { m = 100000; ++e10; }
    if (std::signbit(v)) *w++ = '-';
    char d[6];
    for (int i = 5; i >= 0; --i) { d[i] = (char)('0' + m % 10); m /= 10; }
    *w++ = d[0];
    *w++ = '.';
    memcpy(w, d + 1, 5);
    w += 5;
    *w++ = 'E';
    int ea = e10;
    if (ea < 0) { *w++ = '-'; ea = -ea; } else { *w++ = '+'; }
    if (ea >= 100) { *w++ = (char)('0' + ea / 100); ea %= 100; }
    *w++ = (char)('0' + ea / 10);
    *w++ = (char)('0' + ea % 10);
    return w;
  }
  return format_5e_exact(w, v);
}

// fill(r, out): the `cols` values of row r.
// Batches of rows are formatted by all host threads into private buffers; while batch k + 1 is being formatted, the buffers
// of batch k go to the file through a few concurrent pwrite()s at their final offsets (the page-cache copy of one writer is
// the bottleneck of a 3.6 GB chain file: 1.8 GB/s with one writer, ~3 GB/s with two to four).
template <typename Fill>
int64_t write_chain(const char* path, const char* header, int64_t rows, int cols, int append, Fill fill) {
  const int fd = open(path, O_WRONLY | O_CREAT | (append ? 0 : O_TRUNC), 0644);
  if (fd < 0) return NNB_ERR_ARG;
  bool ok = true;
  auto write_all = [fd](const char* p, size_t n, int64_t off) {
    while (n > 0) {
      const ssize_t w = pwrite(fd, p, n, (off_t)off);
      if (w <= 0) return false;
      p += w; n -= (size_t)w; off += w;
    }
    return true;
  };
  int64_t pos = append ? (int64_t)lseek(fd, 0, SEEK_END) : 0;
  if (pos < 0) { close(fd); return NNB_ERR_ARG; }
  const int64_t pos0 = pos;
  if (header && header[0]) {
    std::string hline = std::string(header) + "\n";
    ok = write_all(hline.data(), hline.size(), pos);
    pos += (int64_t)hline.size();
  }
  const int64_t chunk = 1 << 14;   // rows per work item
  unsigned hw = std::thread::hardware_concurrency();
  const int nthreads = (int)std::max(1u, std::min(hw ? hw : 1u, 32u));
  const int nwriters = std::min(4, nthreads);
  const size_t per_row = (size_t)cols * 14 + 2;   // "-1.23456E+308 " is 14 characters at most
  std::vector<std::string> bufs[2] = {std::vector<std::string>((size_t)nthreads), std::vector<std::string>((size_t)nthreads)};
  auto format_batch = [&](int64_t r0, std::vector<std::string>& set) {
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t) {
      const int64_t a = r0 + t * chunk, b = std::min(rows, a + chunk);
      set[(size_t)t].clear();
      if (a >= b) continue;
      th.emplace_back([&set, &fill, t, a, b, cols, per_row] {
        std::string& out = set[(size_t)t];
        out.resize((size_t)(b - a) * per_row);
        std::vector<double> rowbuf((size_t)cols);
        char* w = &out[0];
        for (int64_t r = a; r < b; ++r) {
          fill(r, rowbuf.data());
          for (int c = 0; c < cols; ++c) {
            w = format_5e(w, rowbuf[(size_t)c]);
            *w++ = c + 1 < cols ? ' ' : '\n';
          }
        }
        out.resize((size_t)(w - &out[0]));
      });
    }
    for (auto& x : th) x.join();
  };
  const int64_t batch = chunk * nthreads;
  int cur = 0;
  if (rows > 0) format_batch(0, bufs[0]);
  for (int64_t r0 = 0; r0 < rows && ok; r0 += batch) {
    std::thread next;
    if (r0 + batch < rows) next = std::thread([&, r0, cur] { format_batch(r0 + batch, bufs[cur ^ 1]); });
    // final offsets of this batch's buffers, then a few writers take them round robin
    std::vector<int64_t> off((size_t)nthreads);
    for (int t = 0; t < nthreads; ++t) { off[(size_t)t] = pos; pos += (int64_t)bufs[cur][(size_t)t].size(); }
    std::vector<std::thread> wr;
    std::vector<char> good((size_t)nwriters, 1);
    for (int wi = 0; wi < nwriters; ++wi)
      wr.emplace_back([&, wi, cur] {
        for (int t = wi; t < nthreads; t += nwriters) {
          const std::string& o = bufs[cur][(size_t)t];
          if (!o.empty() && !write_all(o.data(), o.size(), off[(size_t)t])) good[(size_t)wi] = 0;
        }
      });
    for (auto& x : wr) x.join();
    for (char g : good) ok = ok && g;
    if (next.joinable()) next.join();
    cur ^= 1;
  }
  if (close(fd) != 0) ok = false;
  return ok ? pos - pos0 : (int64_t)NNB_ERR_ARG;
}
}  // namespace

extern "C" int64_t nnb_write_chain_text(const char* path, const char* header, const double* table, int64_t rows,
                                        int cols, int append) {
  if (!path || (!table && rows > 0) || rows < 0 || cols <= 0) return NNB_ERR_ARG;
  return write_chain(path, header, rows, cols, append, [=](int64_t r, double* out) {
    memcpy(out, table + r * cols, sizeof(double) * (size_t)cols);
  });
}

// The same file straight from the arrays the sampler holds (sampler.py:494-511: np.column_stack of the clipped weights,
// -loglikes, samples, derived), without materialising that table: row r = max(weights[r], min_weight), -loglikes[r],
// samples[r][0..d), derived[r][0..n_derived).  weights == NULL means all ones.
extern "C" int64_t nnb_write_chain_rows(const char* path, const char* header, const double* weights,
                                        const double* loglikes, const double* samples, int d, const double* derived,
                                        int n_derived, int64_t rows, double min_weight, int append) {
  if (!path || rows < 0 || d <= 0 || n_derived < 0 || (rows > 0 && (!loglikes || !samples)) ||
      (n_derived > 0 && rows > 0 && !derived))
    return NNB_ERR_ARG;
  const int cols = 2 + d + n_derived;
  return write_chain(path, header, rows, cols, append, [=](int64_t r, double* out) {
    const double w = weights ? weights[r] : 1.0;
    out[0] = w < min_weight ? min_weight : w;            // max(w, min_weight) of the reference: NaN stays NaN
    out[1] = -loglikes[r];
    memcpy(out + 2, samples + r * d, sizeof(double) * (size_t)d);
    if (n_derived) memcpy(out + 2 + d, derived + r * n_derived, sizeof(double) * (size_t)n_derived);
  });
}

// Information recurrence of nested sampling (nnest/nested.py:283), sequential over the iterations of a run:
//     h <- (a[i] + b[i] * (h + zp[i])) - zn[i]
// with a = exp(logwt - logz_new) * L_worst, b = exp(logz_old - logz_new), zp = logz_old, zn = logz_new prepared by the
// caller in float64.  Plain IEEE double arithmetic, one rounding per operation (no contraction), i.e. the reference's Python
// expression evaluated left to right.
extern "C" double nnb_ns_information(double h, const double* a, const double* b, const double* zp, const double* zn,
                                     int64_t n) {
  volatile double t;   // keeps every intermediate a rounded double (no fused multiply-add, no extended precision)
  for (int64_t i = 0; i < n; ++i) {
    t = h + zp[i];
    t = b[i] * t;
    t = a[i] + t;
    h = t - zn[i];
  }
  return h;
}
