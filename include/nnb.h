/*
 * nnb.h -- C ABI of libnnb.so: the B200-native (sm_100a) hot path of adammoss/nnest.
 *
 * The reference is pure Python and has no FFI; its boundary for this path is Python-level
 * (SURVEY.md section 8b).  Each entry point below names the reference code it replaces.  A
 * reference maintainer binds these with ctypes from nnest/trainer.py and nnest/sampler.py
 * (stub shown in INTEGRATION.md); nnest_b200/_lib.py is exactly that binding.
 *
 * Conventions
 *   - every function returns 0 (NNB_OK) or a negative error code; nnb_last_error() gives text.
 *     Nothing throws across the ABI.  There is no CPU fallback: without a CUDA device
 *     nnb_create fails with NNB_ERR_CUDA.
 *   - pointers marked [dev] are device pointers owned by the caller (e.g. torch tensors);
 *     pointers marked [host] are host memory read during the call.  The library owns only its
 *     handle and a small device workspace.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     stream-ordered and asynchronous unless stated otherwise.  One handle per device; a handle is
 *     not re-entrant.
 *   - matrices of per-chain vectors are addressed as ptr[row * row_stride + col * col_stride]
 *     (strides in elements): row-major (n,d) is (d,1); chain-minor "SoA" (d,n) is (1,n).
 */
#ifndef NNB_H_
#define NNB_H_

#ifndef __CUDACC_RTC__
#include <stddef.h>
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define NNB_ABI_VERSION 14
#define NNB_MAX_DIM 128      /* x_dim */
#define NNB_MAX_BLOCKS 16    /* num_blocks */
#define NNB_MAX_LIKE_PARAMS 160
/* derived parameters of a user likelihood (nnb_set_user_likelihood_derived).  The derived kernels hold them in a
 * per-thread array of this many doubles: 32 doubles = 256 bytes a thread, which stays in registers / L1-resident local
 * memory at 128 threads a CTA; more columns than this are better computed from the returned samples afterwards. */
#define NNB_MAX_DERIVED 32

enum {
  NNB_OK = 0,
  NNB_ERR_ARG = -1,          /* invalid argument / unsupported shape */
  NNB_ERR_CUDA = -2,         /* CUDA runtime error (text in nnb_last_error) */
  NNB_ERR_STATE = -3,        /* flow or target not set */
  NNB_ERR_UNSUPPORTED = -4,  /* valid in the reference but not implemented on the device */
  NNB_ERR_START = -5         /* 'Could not find starting value' (nnest/sampler.py:284) */
};

/* flags for nnb_set_flow (reference: `scale` kwarg of SingleSpeedNVP, nnest/networks.py:330-346) */
enum { NNB_FLOW_TRANSLATE_ONLY = 1, NNB_FLOW_CONST_SCALE = 2 };

/* likelihood ids (reference: nnest/likelihoods.py) */
enum {
  NNB_LIKE_ROSENBROCK = 0,     /* :48-51   params: none */
  NNB_LIKE_HIMMELBLAU = 1,     /* :62-70   params: none, d == 2 */
  NNB_LIKE_GAUSSIAN = 2,       /* :77-86   params: corr */
  NNB_LIKE_EGGBOX = 3,         /* :97-106  params: none (product over all dims; reference has d == 2) */
  NNB_LIKE_GAUSSIAN_MIX = 4,   /* :165-189 params: sep, sigma, ncomp, w[ncomp] */
  NNB_LIKE_GAUSSIAN_SHELL = 5, /* :113-128 params: sigma, rshell, center[d] */
  NNB_LIKE_USER = 6            /* the handle's user likelihood (nnb_set_user_likelihood)   params: any, up to the maximum */
};

enum { NNB_PRIOR_NONE = 0, NNB_PRIOR_BOX_U = 1, NNB_PRIOR_BOX_V = 2 };
enum { NNB_MODE_HARD = 0, NNB_MODE_MH = 1 };
/* kernel variant of nnb_mcmc_run.  AUTO: batches of up to ~6 k chains (3/4 of what the 16-lanes-per-chain kernel holds
 * co-resident: 2 x 28 chains per SM; hidden_dim == 16, scale == '') run there -- a step's latency is 2-3x shorter than with
 * one thread per chain, which is what bounds small / sharded batches; larger batches run the tcgen05 (tensor-core, 3xTF32)
 * kernel when the flow shape allows it (hidden_dim == 16, 2 <= x_dim <= 63, scale == ''), else the FP32-FMA kernel */
enum { NNB_IMPL_AUTO = 0, NNB_IMPL_FFMA = 1, NNB_IMPL_TCGEN05 = 2, NNB_IMPL_WARP = 3 };

typedef struct nnb_handle nnb_handle;

int nnb_abi_version(void);

/* Create / destroy a per-device context. */
int nnb_create(int device, nnb_handle** out);
void nnb_destroy(nnb_handle* h);
/* Text of the last error on this handle (or of the last failed nnb_create when h == NULL). */
const char* nnb_last_error(nnb_handle* h);

/*
 * Install the weights of a SingleSpeedNVP (replaces holding an nn.Module: nnest/networks.py:328-347,
 * built at nnest/trainer.py:90).  weights [host]: netG.state_dict() order -- for each block k,
 * the scale net (omitted if NNB_FLOW_TRANSLATE_ONLY) then the translate net, each as
 * Linear(d,H), [Linear(H,H)] x num_layers, Linear(H,d), every Linear as weight (out*in, row-major)
 * followed by bias (out); then, if NNB_FLOW_CONST_SCALE, one float per block (ScaleLayer.scale).
 * Coupling masks are not parameters: block k uses mask[i] = (i + k) % 2 (networks.py:333-346).
 * Synchronous (small H2D copy).  hidden must be one of 16, 32, 64.
 */
int nnb_set_flow(nnb_handle* h, int d, int hidden, int num_layers, int num_blocks, int flags,
                 const float* weights, size_t n_floats);

/*
 * Install a neural-spline flow, the reference's DEFAULT flow='spline' (SingleSpeedSpline = [ActNorm, Invertible1x1Conv,
 * NSF_CL] x num_blocks with num_bins = 8, tail_bound = 3: nnest/networks.py:393-705, built at nnest/trainer.py:92-98).
 * It replaces whatever flow the handle held; nnb_flow_forward / nnb_flow_inverse / nnb_mcmc_init / nnb_mcmc_run then use
 * it.  packed [host], per block (d = x_dim, H = hidden, nlow = d/2 (+1 if d is odd), nup = d - nlow, P = 3 num_bins - 1):
 *     s[d] t[d]                              ActNorm: y = x exp(s) + t                       (networks.py:656-695)
 *     W[d*d] Winv[d*d] logdet[1]             1x1 convolution y = x W, W = P L (U + diag S) assembled by the caller
 *                                            (row-major), its inverse, sum(log|S|)           (networks.py:622-653)
 *     f1: W0[H*nlow] b0[H] W1[H*H] b1[H] W2[H*H] b2[H] W3[(P*nup)*H] b3[P*nup]               conditioner of the upper half
 *     f2: W0[H*nup]  b0[H] W1[H*H] b1[H] W2[H*H] b2[H] W3[(P*nlow)*H] b3[P*nlow]             conditioner of the lower half
 * (nn.Linear weights row-major (out, in); MLP = Linear, LeakyReLU(0.2) x 3, Linear, networks.py:401-417).  Synchronous.
 */
int nnb_set_flow_spline(nnb_handle* h, int d, int hidden, int num_blocks, int num_bins, double tail_bound,
                        const float* packed, size_t n_floats);
/*
 * flags[r] = 1 when, for sample r, some coupling transform of the map (inverse != 0: the inverse map) finds NONE of its
 * coordinates inside the tail bound: evaluated on a one-sample batch the reference's RQS raises ValueError('No input
 * values') there (networks.py:464-465; caught as "skip this proposal" at nnest/sampler.py:320-324).  Always 0 for the
 * affine-coupling flow.  z [dev] n x d with strides, flags [dev] int32 n.
 */
int nnb_flow_empty_halves(nnb_handle* h, const float* z, int64_t z_rs, int64_t z_cs, int inverse, int* flags, int64_t n,
                          void* stream);

/*
 * Flow maps (replace Trainer.inverse / Trainer.forward, nnest/trainer.py:247-269 ->
 * NormalizingFlow.inverse / forward nnest/networks.py:24-42 -> CouplingLayer nnest/networks.py:289-309).
 * in/out [dev] float32 n x d with the given strides, logdet [dev] float32 n (may be NULL).
 * in and out may alias when their strides are equal.
 */
int nnb_flow_inverse(nnb_handle* h, const float* z, int64_t z_rs, int64_t z_cs, float* x, int64_t x_rs,
                     int64_t x_cs, float* logdet, int64_t n, void* stream);
int nnb_flow_forward(nnb_handle* h, const float* x, int64_t x_rs, int64_t x_cs, float* z, int64_t z_rs,
                     int64_t z_cs, float* logdet, int64_t n, void* stream);

/*
 * Likelihood o transform, and prior (replace safe_loglike / safe_prior / safe_transform,
 * nnest/sampler.py:100-163, and the per-row loops of nnest/likelihoods.py:14-22, nnest/priors.py:39-43).
 *   transform: v[i] = u[i] * t_scale[i] + t_shift[i]  (the affine maps of examples/nested/run.py:25-44
 *              and nnest/mcmc.py:111); NULL arrays = identity.
 *   compute_f64: 0 = arithmetic follows the float32 input as NumPy does in the reference;
 *                1 = inputs are promoted to float64 before the transform (float64 live points,
 *                    nnest/priors.py:46, or a float64 transform, nnest/mcmc.py:111).
 *   prior_kind: NNB_PRIOR_BOX_U tests lo <= u <= hi (NestedSampler: transform_prior=False,
 *               nnest/nested.py:76,84); NNB_PRIOR_BOX_V tests transform(u) (nnest/sampler.py:158-159).
 * All arrays [host], d entries each (like_params: n_like_params entries).  Synchronous.
 */
typedef struct {
  int like_id;
  int n_like_params;
  const double* like_params;
  int compute_f64;
  const double* t_scale;
  const double* t_shift;
  int prior_kind;
  const double* prior_lo;
  const double* prior_hi;
} nnb_target;

int nnb_set_target(nnb_handle* h, int d, const nnb_target* t);

/*
 * A likelihood written by the user in CUDA C++ (no counterpart in the reference, whose likelihoods are Python callables
 * that cannot run inside the kernels).  `source` defines
 *     template <typename X> __device__ double nnb_user_loglike(const X& x, int d, const double* params);
 * x(i) is coordinate i after the target's transform, in the arithmetic type the built-in likelihoods see at the same place
 * (float when compute_f64 == 0 and the input is float32, double otherwise); params are the target's like_params (up to
 * NNB_MAX_LIKE_PARAMS).  Data of any size -- observations, a covariance -- goes into device arrays the source reads as
 * nnb_data.<name>[j] (nnb_set_user_likelihood_data below); a small table of fixed constants may also be written into the
 * source as a __constant__ array (64 KB per module, and a new table is a new source to compile).  A non-finite result becomes -inf
 * when x(i) is float and -1e100 otherwise, as for the built-in likelihoods.
 * nnb_set_user_likelihood installs the source on the handle; nnb_set_target with like_id NNB_LIKE_USER then selects it
 * (NNB_ERR_STATE before a source is installed).  NVRTC compiles the library's own kernel templates around the source:
 * the likelihood kernel during this call (NNB_ERR_ARG with NVRTC's log in nnb_last_error when the source does not
 * compile), every other kernel variant the first time a call runs it.  Compiled variants are kept per handle and on
 * disk under $NNB_JIT_CACHE (default ~/.cache/nnest_b200/jit), which the ranks of a run may share.  n_compiled_out (may
 * be NULL) receives the number of variants this call compiled (0 when they came from either cache).  Needs a device of
 * compute capability 10.0 and libnvrtc.so.12 (else NNB_ERR_UNSUPPORTED).  Synchronous.
 */
int nnb_set_user_likelihood(nnb_handle* h, const char* source, int* n_compiled_out);
/*
 * Compiles `source` as nnb_set_user_likelihood would, without a handle or a device: NNB_OK, or NNB_ERR_ARG when it does
 * not compile (NNB_ERR_UNSUPPORTED without NVRTC).  log [host] (may be NULL) receives up to cap - 1 characters of NVRTC's
 * log, NUL-terminated.
 */
int nnb_user_likelihood_check(const char* source, char* log, size_t cap);

/*
 * Derived parameters of a user likelihood (the reference's `num_derived`: a likelihood returning (logl, derived)).
 * With num_derived > 0 the source also defines
 *     template <typename X> __device__ void nnb_user_derived(const X& x, int d, const double* params, double* derived);
 * which writes derived[0 .. num_derived).  x and params mean what they mean for nnb_user_loglike, in the same arithmetic
 * type; non-finite values are returned as they are (only the log-likelihood is clamped).
 * nnb_set_user_likelihood_derived is nnb_set_user_likelihood that also compiles the derived kernels during the call, so a
 * missing or wrong nnb_user_derived is refused here with NVRTC's log (NNB_ERR_ARG).  num_derived == 0 is exactly
 * nnb_set_user_likelihood.  0 <= num_derived <= NNB_MAX_DERIVED, else NNB_ERR_ARG.
 * nnb_user_likelihood_check_derived checks the same without a handle or a device, as nnb_user_likelihood_check does.
 */
int nnb_set_user_likelihood_derived(nnb_handle* h, const char* source, int num_derived, int* n_compiled_out);
int nnb_user_likelihood_check_derived(const char* source, int num_derived, char* log, size_t cap);

/*
 * A dataset of a user likelihood: up to NNB_MAX_DATA_ARRAYS named, typed, read-only device arrays.  With n_arrays > 0
 * the source is compiled behind generated declarations (the file user_data.cuh):
 *     template <typename T> struct nnb_span {        // T: double, float or int (NNB_DTYPE_F64 / _F32 / _I32)
 *       const T* p; long long n;
 *       __device__ T operator[](long long j) const;  // p[j] through the read-only data path
 *       __device__ long long size() const;           // n
 *     };
 *     struct nnb_user_data_t { nnb_span<T0> <name0>; nnb_span<T1> <name1>; ... };   // in the order given
 *     __constant__ nnb_user_data_t nnb_data;
 * so nnb_user_loglike and nnb_user_derived read array k as nnb_data.<name k>[j] and its length as .size().  A user
 * transform does not see nnb_data.  names [host] are C identifiers, none repeated; dtypes [host] NNB_DTYPE_*.  The layout
 * (names and dtypes) is compiled in, and the cache keys name it; the values, sizes and pointers are not, so a new
 * dataset of the same layout needs no compile.
 * nnb_set_user_likelihood_data is nnb_set_user_likelihood_derived with that layout; n_arrays == 0 is exactly
 * nnb_set_user_likelihood_derived.  A bad layout (a name that is not an identifier or repeats, an unknown dtype, more
 * than NNB_MAX_DATA_ARRAYS arrays) is NNB_ERR_ARG.  Installing a source or layout drops the dataset's binding.
 * nnb_user_likelihood_check_data checks the same without a handle or a device, as nnb_user_likelihood_check does: a
 * source that reads an undeclared array, or an array as the wrong type, is refused with NVRTC's log.
 * nnb_bind_user_data binds the dataset: ptrs [host] n_arrays pointers to device (or managed) memory of the handle's
 * device, each aligned to its element size (NULL only for an empty array); sizes [host] n_arrays element counts >= 0.
 * Anything else is NNB_ERR_ARG, checked on the host.  The table is written into every loaded kernel module that holds
 * the likelihood, and into later ones as they load.  Synchronous, and ordered as nnb_set_target.  The caller owns the
 * arrays and keeps them alive and unchanged while launches that read them are in flight.  A launch that needs the
 * likelihood of a layout with arrays before nnb_bind_user_data is NNB_ERR_STATE, refused before anything runs.
 */
#define NNB_MAX_DATA_ARRAYS 16
enum { NNB_DTYPE_F64 = 0, NNB_DTYPE_F32 = 1, NNB_DTYPE_I32 = 2 };
int nnb_set_user_likelihood_data(nnb_handle* h, const char* source, int num_derived, int n_arrays,
                                 const char* const* names, const int* dtypes, int* n_compiled_out);
int nnb_user_likelihood_check_data(const char* source, int num_derived, int n_arrays, const char* const* names,
                                   const int* dtypes, char* log, size_t cap);
int nnb_bind_user_data(nnb_handle* h, const void* const* ptrs, const int64_t* sizes);

/*
 * derived values of the target selected by nnb_set_target (like_id NNB_LIKE_USER with num_derived > 0, else
 * NNB_ERR_STATE).  x(i) is formed from each row exactly as nnb_loglike and the step kernels form it, so derived values
 * belong to the very point whose log-likelihood those report.
 *   nnb_derived:       u [dev] n rows, float32 or float64 (in_f64), strides as nnb_loglike; out [dev] float64 (n, num_derived)
 *                      row-major.
 *   nnb_derived_trace: trace_x [dev] float32 (T, d, n) as nnb_mcmc_run writes it; evaluates the rows
 *                      t_k = row0 + k * row_step, k < n_rows, into out [dev] float64 (n_rows, num_derived, n) chain-minor
 *                      (element (k, j, c) at [(k * num_derived + j) * n + c]).  init [dev] float64 (num_derived, n) or
 *                      NULL: when given, a chain whose point at t_k equals its row-0 point bit for bit in every
 *                      coordinate gets init's values (the start's derived values the caller already has).
 * Stream-ordered and asynchronous.
 */
int nnb_derived(nnb_handle* h, const void* u, int in_f64, int64_t u_rs, int64_t u_cs, double* out, int64_t n,
                void* stream);
int nnb_derived_trace(nnb_handle* h, const float* trace_x, int64_t n, int64_t row0, int64_t row_step, int64_t n_rows,
                      const double* init, double* out, void* stream);

/*
 * A prior transform written by the user in CUDA C++ (the reference's `transform` callable, nnest/sampler.py:100-108,
 * when it is not the affine map of t_scale / t_shift).  `source` defines
 *     template <typename U> __device__ auto nnb_user_transform(const U& u, int i, int d, const double* params)
 *         -> decltype(u(0));
 * which returns coordinate i of v = transform(u).  u(j) is coordinate j of the unit-box point in the arithmetic type of
 * the target (float when compute_f64 == 0 and the input is float32, double otherwise); any u(j) may be read, so
 * transforms that mix coordinates are allowed.  v is not stored: every x(i) the likelihood, the BOX_V prior or the derived
 * parameters read evaluates the transform once.  params are the transform_params given to nnb_set_target_user_transform.
 * nnb_set_user_transform installs the source on the handle and compiles the likelihood kernels around it during the call
 * (NNB_ERR_ARG with NVRTC's log in nnb_last_error when it does not compile); it compiles, caches and needs what
 * nnb_set_user_likelihood does, and the two sources may be installed together.  n_compiled_out as there.  Synchronous.
 * nnb_user_transform_check compiles `source` without a handle or a device, as nnb_user_likelihood_check does.
 */
int nnb_set_user_transform(nnb_handle* h, const char* source, int* n_compiled_out);
int nnb_user_transform_check(const char* source, char* log, size_t cap);

/*
 * nnb_set_target with the installed user transform in place of the affine map: t->t_scale / t->t_shift must be NULL.
 * transform_params [host] n_transform_params doubles; together with the likelihood's at most NNB_MAX_LIKE_PARAMS (else
 * NNB_ERR_ARG).  NNB_ERR_STATE before nnb_set_user_transform.  Every kernel then runs the NVRTC-compiled variant.
 */
int nnb_set_target_user_transform(nnb_handle* h, int d, const nnb_target* t, const double* transform_params,
                                  int n_transform_params);

/*
 * v = transform(u) of the target selected by nnb_set_target_user_transform (else NNB_ERR_STATE), formed exactly as the
 * likelihood sees it, so the values equal the likelihood's x(i) bit for bit.
 *   nnb_transform:       u [dev] n rows, float32 or float64 (in_f64), strides as nnb_loglike; out [dev] float64 (n, d)
 *                        row-major.
 *   nnb_transform_trace: trace_x [dev] float32 (T, d, n) as nnb_mcmc_run writes it; rows t_k = row0 + k * row_step,
 *                        k < n_rows, into out [dev] float64 (n_rows, d, n) chain-minor.
 * Stream-ordered and asynchronous.
 */
int nnb_transform(nnb_handle* h, const void* u, int in_f64, int64_t u_rs, int64_t u_cs, double* out, int64_t n,
                  void* stream);
int nnb_transform_trace(nnb_handle* h, const float* trace_x, int64_t n, int64_t row0, int64_t row_step, int64_t n_rows,
                        double* out, void* stream);

/*
 * logl[r] = safe_loglike(u[r]) for n rows (nnest/sampler.py:110-133): non-finite values become
 * -1e100 (-inf when the reference's result would be float32).  u [dev] n x d, float32 or float64
 * (in_f64); logl [dev] float64 n.  logp (may be NULL) [dev] float64 n receives safe_prior: 0 or -inf.
 */
int nnb_loglike(nnb_handle* h, const void* u, int in_f64, int64_t u_rs, int64_t u_cs, double* logl,
                double* logp, int64_t n, void* stream);

/*
 * The batched latent-space MCMC step (replaces Sampler._mcmc_sample, nnest/sampler.py:229-463):
 * `steps` Metropolis steps of n_chains independent chains entirely on the device.
 *
 * Per-chain state lives in caller-owned chain-minor buffers (element (i, c) at [i * n_chains + c]):
 *   z, x [dev] float32 d x n; logl [dev] float64 n; logdet [dev] float32 n; logp [dev] float64 n.
 * nnb_mcmc_init fills them from start points; nnb_mcmc_run advances them in place.
 */
typedef struct {
  int64_t n_chains;
  /* state (in/out) */
  float* z;
  float* x;
  double* logl;
  float* logdet;
  double* logp;
  /* start: exactly one of init_u / init_z may be non-NULL, both NULL = draw z ~ N(0,I) from Philox
   * (nnest/sampler.py:262-284).  Chain-minor d x n [dev] float32. */
  const float* init_u;
  const float* init_z;
  const double* init_logl; /* [dev] n, NULL = evaluate the likelihood of the start points */
  uint64_t seed;
  uint64_t chain_offset; /* global id of chain 0 (multi-GPU sharding: results independent of the split) */
  uint32_t start_try;    /* retry counter for Philox starts */
  /* out [host] */
  int64_t* n_bad_start;  /* chains whose start logl <= -1e30 (nnest/sampler.py:281) */
  int64_t* ncall;        /* likelihood evaluations performed */
} nnb_mcmc_init_args;

/* synchronous when n_bad_start or ncall is requested, otherwise stream-ordered and asynchronous */
int nnb_mcmc_init(nnb_handle* h, const nnb_mcmc_init_args* a, void* stream);

typedef struct {
  int64_t n_chains;
  int steps;
  int mode;              /* NNB_MODE_HARD: accept iff Jacobian/prior test passes and logl > loglstar
                            (sampler.py:299-370); NNB_MODE_MH: Metropolis ratio (sampler.py:372-416) */
  double loglstar;
  double step_size;      /* initial scale; <= 0 -> 2/sqrt(d) (sampler.py:248-249) */
  int dynamic_step_size; /* sampler.py:422-430, one scale per call (= per rank, as under MPI) */
  uint64_t seed;
  uint64_t chain_offset;
  uint32_t step_offset;  /* Philox step counter of the first step is step_offset + 1 */
  /* state (in/out), as nnb_mcmc_init */
  float* z;
  float* x;
  double* logl;
  float* logdet;
  double* logp;
  /* optional full trace [dev]: row t (0..steps) of trace_x/trace_z is d x n chain-minor, i.e. element
   * (t, i, c) at [(t * d + i) * n + c]; trace_logl (t, c) at [t * n + c].  Row 0 = the state at entry
   * (samples.append before the loop, sampler.py:286-289).  NULL = not recorded. */
  float* trace_x;
  float* trace_z;
  double* trace_logl;
  /* optional replay noise [dev] (parity tests): normals (steps, n, d) row-major float32 in the
   * reference's draw order torch.randn_like(z) (sampler.py:310/:377); uniforms (steps, n)
   * (sampler.py:334/:412).  NULL = Philox4x32-10 keyed (seed; chain, step). */
  const float* replay_normals;
  const float* replay_uniforms;
  /* optional dump of the noise actually used, same layouts [dev] */
  float* dump_normals;
  float* dump_uniforms;
  /* out [host] */
  double* scale_out;     /* final scale (sampler.py:463) */
  int64_t* ncall_out;    /* likelihood calls (sampler.py:363,397) */
  int64_t* naccept_out;  /* accepted proposals (total_accepted, sampler.py:418-420) */
  int impl;              /* NNB_IMPL_* */
  int64_t* launches_out; /* [host] kernels launched by this call (1 when the persistent cooperative kernel ran) */
  int* impl_out;         /* [host] NNB_IMPL_FFMA, NNB_IMPL_TCGEN05 or NNB_IMPL_WARP: the variant that ran */
} nnb_mcmc_args;

int nnb_mcmc_run(nnb_handle* h, const nnb_mcmc_args* a, void* stream);
/*
 * nnb_mcmc_run synchronises the stream before returning when any of scale_out / ncall_out / naccept_out is given; with
 * all three NULL it only enqueues the work (several refills can be queued back to back) and the figures of the LAST
 * run are fetched with nnb_mcmc_result, which synchronises.
 */
int nnb_mcmc_result(nnb_handle* h, double* scale_out, int64_t* ncall_out, int64_t* naccept_out, void* stream);

/*
 * Live-point replacement (replaces the consume loop of NestedSampler.run, nnest/nested.py:429-439,
 * together with the selection of the worst point nnest/nested.py:272-276).  Host-side, exact:
 * scans chains ib = *nb .. n_chains-1 (incrementing *nb for each inspected chain) for the first whose
 * end point differs from its start point in EVERY coordinate and whose end loglike > loglstar.
 * first/last [host] float32 row-major (n_chains, d); logl_last [host] float64 n_chains.
 * Returns the chain index used, or -1 if the rest of the batch was exhausted without a usable chain.
 */
int64_t nnb_consume_scan(const float* first, const float* last, const double* logl_last, int64_t n_chains,
                         int d, double loglstar, int64_t* nb);

/*
 * Many nested-sampling iterations at once (replaces a run of iterations of the loop nnest/nested.py:269-471 in
 * strategy 'mcmc' between two refills / retrains / checkpoints).  Host-side and exact.  Starting from the live
 * likelihoods active_logl [host] (nlive, NOT modified) and the consume pointer *nb into the current batch, it
 * repeats up to max_iters times:
 *     worst = first index of min(active_logl)               (np.argmin, nested.py:272)
 *     scan the batch from *nb as nnb_consume_scan does      (nested.py:429-439)
 *     on success the live point `worst` takes the end loglike of the chain found
 * and records for every successful iteration k: worst_out[k], chain_out[k], loglstar_out[k] (the likelihood of the
 * worst point = the constraint of that iteration), maxlogl_out[k] (np.max(active_logl) after the replacement,
 * nested.py:462) and prev_out[k] (the earlier iteration of this call that wrote the slot `worst`, or -1: tells which
 * physical point is saved as dead point, nested.py:288-290).  It stops early when the batch is exhausted without a
 * usable chain: then *exhausted = 1 and worst_out[K] / loglstar_out[K] describe that unfinished iteration (its evidence
 * update is due, nested.py:280-293).  Output arrays need max_iters + 1 entries.  Returns K, or a negative error code.
 */
int64_t nnb_ns_consume(const double* active_logl, int64_t nlive, const float* first, const float* last,
                       const double* logl_last, int64_t n_chains, int d, int64_t* nb, int64_t max_iters,
                       int64_t* worst_out, int64_t* chain_out, int64_t* prev_out, double* loglstar_out,
                       double* maxlogl_out, int* exhausted);

/*
 * Information H of nested sampling over a run of n iterations (nnest/nested.py:283), sequentially and in the reference's
 * operation order:  h <- (a[i] + b[i] * (h + zp[i])) - zn[i]  with a = exp(logwt - logz_new) * L_worst,
 * b = exp(logz_old - logz_new), zp = logz_old, zn = logz_new (float64, host).  Returns the final h.  Host-side, exact.
 */
double nnb_ns_information(double h, const double* a, const double* b, const double* zp, const double* zn, int64_t n);

/*
 * Row movements of a run of nested-sampling iterations (the array side of nnest/nested.py:288-290,432-437 for the iterations
 * nnb_ns_consume selected), host-side, multi-threaded, exact:
 *   nnb_gather_rows_f32: out[i][:] = (double) src[idx[i]][:]  for i < n   (new_u = float32 end points of the chains used);
 *   nnb_ns_apply:        dead_out[i] = prev[i] >= 0 ? new_v[prev[i]] : active_v[worst[i]]   for i < n_ev   (the physical point
 *                        that sat in slot worst[i] when iteration i started), then for i = 0 .. n_done-1 IN ORDER
 *                        active_u[worst[i]] = new_u[i], active_v[worst[i]] = new_v[i], active_logl[worst[i]] = new_logl[i]
 *                        (a later iteration overwrites an earlier one: the last write to a slot wins).
 * All matrices row-major with d columns.  Return 0 or NNB_ERR_ARG.
 */
int nnb_gather_rows_f32(const float* src, int64_t n_src, int d, const int64_t* idx, int64_t n, double* out);
int nnb_ns_apply(const int64_t* worst, const int64_t* prev, int64_t n_ev, int64_t n_done, int d, const double* new_u,
                 const double* new_v, const double* new_logl, double* active_u, double* active_v, double* active_logl,
                 int64_t nlive, double* dead_out);

/*
 * Flow fitting: ONE EPOCH of the reference's Trainer._train + Trainer._validate (nnest/trainer.py:384-418) in one
 * kernel launch.  For every mini-batch (visiting order `perm`, the short tail batch is kept like DataLoader does)
 *     data = x_train[perm[..]] + jitter * N(0, I);  loss = -mean(log p(data));  backward;  Adam step
 * with torch.optim.Adam semantics (L2 weight decay added to the gradient, bias corrections from the step count),
 * then the validation negative log-likelihood with the final weights.  log p is the flow's forward map + log-det under
 * a N(0, I) base density (nnest/networks.py:71-76, 289-298).
 *   params / adam_m / adam_v [device] float32, n_params = netG.state_dict() order as for nnb_set_flow (scale == '' only),
 *       updated in place; step0 = optimizer steps taken so far (the call takes ceil(n_train / batch_size) more).
 *   x_train (n_train, x_dim), x_valid (n_valid, x_dim) [device] float32 row-major; perm [device] int64 or NULL.
 *   noise [device] optional (n_train, x_dim) N(0,1) draws in visiting order (replays torch.randn_like); NULL = the
 *       library's Philox stream keyed by (seed, epoch, position).
 *   grad_out [device] optional: data gradient (without weight decay) of the last mini-batch.
 *   do_train == 0: validation only (params untouched).
 *   train_loss_sum_out [host] = sum over mini-batches of the mini-batch mean loss (trainer.py:396; the reference then
 *       divides by the dataset size); val_nll_sum_out [host] = sum of -log p over x_valid.
 * Synchronises the stream before returning (the losses drive early stopping on the host).
 */
typedef struct nnb_train_args {
  int x_dim, hidden_dim, num_layers, num_blocks;
  const float* x_train;
  int64_t n_train;
  const int64_t* perm;
  int batch_size;
  const float* x_valid;
  int64_t n_valid;
  const float* noise;
  double jitter;
  uint64_t seed;
  uint32_t epoch;
  double lr, beta1, beta2, eps, weight_decay;
  int64_t step0;
  float* params;
  float* adam_m;
  float* adam_v;
  size_t n_params;
  float* grad_out;
  int do_train;
  double* train_loss_sum_out;
  double* val_nll_sum_out;
  int* grid_out;               /* [host] optional: CTAs the epoch kernel ran on */
  /* Data-parallel fitting over several GPUs (north_star: all-reduce of gradients): with grad_only != 0 the call treats
   * x_train (n_train rows, batch_size ignored) as THIS rank's share of ONE mini-batch of batch_total samples: it writes
   * the share's gradient of the mini-batch mean loss to grad_out (required) and adds the share's part of that mean to
   * train_loss_sum_out; no Adam step, no validation.  The caller all-reduces grad_out over the ranks and applies the
   * update.  epoch / seed key the jitter noise: give every (rank, step) its own. */
  int grad_only;
  int batch_total;
} nnb_train_args;

int nnb_train_epoch(nnb_handle* h, const nnb_train_args* args, void* stream);
/*
 * The same epoch in two halves, so that the device does not idle while the host looks at the losses (the reference's loop,
 * trainer.py:170-207, decides after EVERY epoch whether the validation loss improved and whether patience ran out):
 *   nnb_train_epoch_begin queues the epoch on `stream` (the *_out members of args are ignored) and returns;
 *   nnb_train_epoch_end   waits for the OLDEST epoch in flight and returns its losses.
 * At most two epochs may be in flight.  A caller that knows epoch e cannot end the fit (patience cannot run out at e, e is
 * not the last one) begins epoch e + 1 before it ends epoch e; weights it may still need (the best-so-far copy) have to
 * be snapshotted by stream-ordered copies between the two begins.  nnb_train_epoch == begin + end.
 */
int nnb_train_epoch_begin(nnb_handle* h, const nnb_train_args* args, void* stream);
int nnb_train_epoch_end(nnb_handle* h, double* train_loss_sum, double* val_nll_sum, int* grid);
/* 1 when nnb_train_epoch handles this architecture with max_smem_bytes of shared memory per CTA (B200: 232448) */
int nnb_train_supported(int x_dim, int hidden_dim, int num_layers, int num_blocks, int max_smem_bytes);

/*
 * Mean over the n rows of x [device] float64 row-major (n, d) of the distance to the nearest OTHER row: the quantity
 * behind the reference's training jitter, 0.2 * np.mean(cKDTree(x).query(x, 2)[0]) = 0.1 * this (trainer.py:147-150).
 */
int nnb_mean_nn_distance(nnb_handle* h, const double* x, int64_t n, int d, double* out, void* stream);

/*
 * Chain diagnostics on the device trace (reference nnest/utils/evaluation.py:6-73 as used by Sampler._chain_stats,
 * nnest/sampler.py:474-492).  trace_x [device] float32 [T][d][n] as written by nnb_mcmc_run (a prefix T' <= T of a longer
 * trace is a valid input); statistics are taken on v = x * t_scale + t_shift in float64 (t_scale / t_shift [host] d
 * doubles or NULL = identity).
 *   nnb_chain_stats:    *moved_out = number of (chain, step >= 1) whose point differs from the previous one in any
 *                       coordinate, *jump_sum_out = sum of the Euclidean step lengths, sum_out / sumsq_out [host, d,
 *                       optional] = sum of v and of v^2 per dimension over all chains and steps.
 *   nnb_chain_autocorr: out [host] (nlags, d): sum over chains and t of (v[t] - mean)(v[t - s] - mean) for the lags
 *                       s = lag0 .. lag0 + nlags - 1, nlags <= 32; divide by n (T - s) and the variance to obtain
 *                       evaluation.py:6-14.
 */
int nnb_chain_stats(nnb_handle* h, const float* trace_x, int64_t T, int d, int64_t n, const double* t_scale,
                    const double* t_shift, double* moved_out, double* jump_sum_out, double* sum_out, double* sumsq_out,
                    void* stream);
int nnb_chain_autocorr(nnb_handle* h, const float* trace_x, int64_t T, int d, int64_t n, const double* t_scale,
                       const double* t_shift, const double* mean, int lag0, int nlags, double* out, void* stream);

/*
 * Chain / posterior text files in the reference's layout (nnest/sampler.py:494-511, `_save_samples`): `rows` lines of
 * `cols` numbers, each formatted '%.5E' and separated by single spaces (weight, -loglike, parameters, derived).
 * table [host] float64 row-major (rows, cols); header (may be NULL/empty) is written first, followed by '\n';
 * append != 0 appends to an existing file.  Host-side (multi-threaded formatting).  Returns the number of bytes
 * written, or a negative error code.
 */
int64_t nnb_write_chain_text(const char* path, const char* header, const double* table, int64_t rows, int cols,
                             int append);
/*
 * The same file written straight from the arrays `_save_samples` receives (no (rows, cols) table in between): row r is
 * max(weights[r], min_weight), -loglikes[r], samples[r][0..d), derived[r][0..n_derived).  All arrays [host] float64,
 * row-major; weights may be NULL (all ones, sampler.py:495-496), derived may be NULL when n_derived == 0.  NaN is spelled
 * "NAN" whatever its sign bit, as Python's '%.5E' does.
 */
int64_t nnb_write_chain_rows(const char* path, const char* header, const double* weights, const double* loglikes,
                             const double* samples, int d, const double* derived, int n_derived, int64_t rows,
                             double min_weight, int append);

#ifdef __cplusplus
}
#endif
#endif /* NNB_H_ */
