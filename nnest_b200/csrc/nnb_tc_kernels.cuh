// nnb_tc_kernels.cuh -- tensor-core (tcgen05 / TMEM, 3xTF32) variant of the fused MCMC step kernel.
//
// Same contract as mcmc_kernel<16, MODE> (nnb_kernels.cuh; reference nnest/sampler.py:291-444); the six
// small GEMMs of every coupling block -- s/t MLPs Linear(d,16) -> [Linear(16,16)] x L -> Linear(16,d),
// nnest/networks.py:262-282 -- run on the 5th-generation tensor cores:
//   * a tile of 128 chains = the M dimension of one tcgen05.mma is owned by NPART warpgroups (128 threads each);
//     thread (part, t) works on chain t = TMEM lane t (warps w and w+4 address the same lane quarter), so
//     activations never leave the chain's own threads: D row -> registers (tcgen05.ld) -> bias + tanh/relu ->
//     hi/lo split -> A row of the next layer (tcgen05.st).  NPART = 1 (default): one thread per chain, 128 registers,
//     the chain's current latent point resident in shared memory.  NPART = 2 (NNB_TC_NPART=2): the two threads of a
//     chain split the 8-column chunks of every phase (noise, A operands, epilogues, state update) between them;
//   * weights (B operands) are pre-split into tf32 hi/lo halves on the host and staged once per CTA in shared
//     memory in the canonical K-major core-matrix layout (nnb_tc.cuh);
//   * layer 1 of both nets shares its input, so it is ONE N=32 MMA group; the hidden and output layers are
//     block diagonal and issued as two N=16 (N=round16(nout)) groups.
// Everything else of the step (Philox noise, box test, likelihood, accept/reject, state/trace update) is the
// same per-thread code as the FFMA kernel.
#pragma once
#include "nnb_kernels.cuh"
#include "nnb_tc.cuh"
#include "nnb_tc_consts.h"

namespace nnb {

constexpr int kTcMaxTiles = 4;          // warpgroups per CTA
constexpr int kTcColsPerTile = 128;     // TMEM columns per tile: A hi [0,32) lo [32,64); D [64,128)

__host__ __device__ inline int round8(int v) { return (v + 7) & ~7; }
__host__ __device__ inline int round16(int v) { return (v + 15) & ~15; }
// per-block packed layout (floats):
//   B1_hi [K1*32] B1_lo [K1*32] bias1 [32]
//   L x { B2s_hi [256] B2s_lo [256] B2t_hi [256] B2t_lo [256] bias2 [32] }
//   B3s_hi [16*N3] B3s_lo B3t_hi B3t_lo   bias3s [N3] bias3t [N3]
__host__ __device__ inline int tc_block_floats(int d, int L, int k) {
  const int K1 = round8(blk_nin(d, k)), N3 = round16(blk_nout(d, k));
  return 64 * K1 + 32 + L * 1056 + 64 * N3 + 2 * N3;
}
// Warp-uniform constants of a step -- the biases of every layer, the prior box and the affine transform in float32 --
// travel as a KERNEL PARAMETER: parameters live in constant bank 0, and with x_dim fixed at compile time every index
// below is an immediate, so an `x + bias` reads its second operand straight from c[0x0][imm] -- no load instruction, no
// shared-memory bandwidth.  (As shared-memory broadcasts these were 258 of the ~630 shared-memory instructions of a
// proposal at d = 30, on a pipe that moves 128 B per cycle per SM and bounds the proposal / likelihood / update phases.)
//   per block k at tc_cb_off(d, L, k):  bias1 [32]  L x bias2 [32]  bias3s [N3]  bias3t [N3]
//   then  tsf [d]  tbf [d]  lof [d]  hif [d]   (TargetSmem's float32 mirrors)
// (struct TcConsts: nnb_tc_consts.h)
__host__ __device__ inline int tc_cb_block_floats(int d, int L, int k) { return 32 + 32 * L + 2 * round16(blk_nout(d, k)); }
__host__ __device__ inline int tc_cb_off(int d, int L, int k) {
  int off = 0;
  for (int j = 0; j < k; ++j) off += tc_cb_block_floats(d, L, j);
  return off;
}
__host__ __device__ inline int tc_cb_floats(int d, int L, int B) { return tc_cb_off(d, L, B) + 4 * d; }
__host__ __device__ inline bool tc_supported(const FlowDesc& f) {
  return f.H == 16 && f.d >= 2 && blk_nin(f.d, 0) <= 32 && blk_nin(f.d, 1) <= 32 && blk_nout(f.d, 0) <= 32 &&
         blk_nout(f.d, 1) <= 32 && !(f.flags & (NNB_FLOW_TRANSLATE_ONLY | NNB_FLOW_CONST_SCALE)) &&
         tc_cb_floats(f.d, f.L, f.B) <= kTcConstFloats;
}

// The scale net's constants are folded into its weights by the host (nnb_tc_pack): the layers that feed a tanh are packed
// times 2 log2(e), the output layer times -log2(e), so that the tensor core delivers x' = 2 log2(e) x and l' = -log2(e) log_s
// and the epilogues need no multiply in front of MUFU.EX2:
//   tanh(x) = 1 - 2 / (2^{x'} + 1)   (e -> inf gives 1, e -> 0 gives -1; near 0 the ABSOLUTE error stays ~2e-7, which is what
//   matters for the sums the activations feed),   exp(-log_s) = 2^{l'},   log-det = ln 2 * sum l'.
constexpr float kTcTanhScale = 2.885390081777927f;    // 2 log2(e)
constexpr float kTcExpScale = -1.4426950408889634f;   // -log2(e)
__device__ __forceinline__ float tc_exp2(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
  return e;
}
__device__ __forceinline__ float tc_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// two tanh side by side: the add and the FMA as packed FP32 pairs (each lane rounded like FADD / FFMA)
__device__ __forceinline__ float2 tc_tanh_scaled2(float2 xs) {
  const float2 e1 = __fadd2_rn(make_float2(tc_exp2(xs.x), tc_exp2(xs.y)), make_float2(1.0f, 1.0f));
  return __ffma2_rn(make_float2(-2.0f, -2.0f), make_float2(tc_rcp(e1.x), tc_rcp(e1.y)), make_float2(1.0f, 1.0f));
}
// z' = z + scale * n of two dims, the bits of __fadd_rn(z, __fmul_rn(n, scale)) in each lane: the products as one packed
// pair, the adds scalar.  (ptxas of CUDA 12.9 contracts a packed multiply that feeds a packed add into one FFMA2 even for
// the .rn forms -- one rounding instead of two, other bits -- so no packed product here goes straight into a packed add.)
__device__ __forceinline__ float2 tc_propose2(float2 z, float2 n, float scale) {
  const float2 ns = __fmul2_rn(n, make_float2(scale, scale));
  return make_float2(__fadd_rn(z.x, ns.x), __fadd_rn(z.y, ns.y));
}

// Philox blocks drawn side by side (c4, B200, with the packed epilogues: 2 and 8 within 0.3 % of 4)
#ifndef NNB_TC_PHILOX_ILP
#define NNB_TC_PHILOX_ILP 4
#endif
constexpr int kTcPhiloxIlp = NNB_TC_PHILOX_ILP;

#ifdef NNB_TC_TIMING
// development probe (NNB_EXTRA_NVCC_FLAGS=-DNNB_TC_TIMING, scripts/dev/tc_timing.py): clock64 stamps of every tile leader at
// points of every step -- [0] step start (scale read) [1] flow inverse done [2] accept + state update done [3] next step's
// noise drawn [4] grid barrier released -- plus [5] globaltimer at step start, [6] proposal written, [7] likelihood done,
// [8] tile's accept count known.  Each translation unit has its own copy.
constexpr int kTimeSteps = 160, kTimeSlots = 10;
static __device__ unsigned long long g_tc_time[160 * kTcMaxTiles * kTimeSteps * kTimeSlots];
#define NNB_TSTAMP(slot)                                                                                              \
  do {                                                                                                               \
    if (tit == 0 && si_t < kTimeSteps)                                                                               \
      g_tc_time[(((size_t)blockIdx.x * kTcMaxTiles + tile) * kTimeSteps + si_t) * kTimeSlots + (slot)] = clock64();  \
  } while (0)
#else
#define NNB_TSTAMP(slot) do {} while (0)
#endif

// Shared-memory read-modify-write loops over a chain's coordinates: the pointers involved (y, zp, nz, the global state)
// may alias as far as the compiler can tell, so a loop of the form `dst[i] = f(src[i])` keeps every load behind the
// previous iteration's store -- one shared-memory latency (~30 cycles) per coordinate, 30 coordinates, several loops per
// step, all of it on the step's critical path.  batched<CH>() evaluates `ld` for CH coordinates first (all loads in
// flight together) and only then runs the stores.
template <int CH, typename LD, typename ST>
__device__ __forceinline__ void batched(int d, LD ld, ST st) {
#pragma unroll
  for (int i0 = 0; i0 < d; i0 += CH) {
    float v[CH];
#pragma unroll
    for (int j = 0; j < CH; ++j)
      if (i0 + j < d) v[j] = ld(i0 + j);
#pragma unroll
    for (int j = 0; j < CH; ++j)
      if (i0 + j < d) st(i0 + j, v[j]);
  }
}

struct TcTile {
  uint32_t tmem;        // TMEM address of the tile's column 0 (lane 0)
  uint32_t lane_tmem;   // + this warp's lane quarter
  uint64_t* mbar;       // two mbarriers: [0] scale-net group, [1] translate-net group
  uint32_t phase;
  uint32_t bar_id;
  uint32_t bar_threads; // 128 * NPART
  int part;             // which of the chain's NPART threads this is
  bool single;          // only one issuing warp exists (32-chain tile): it issues both MMA groups
  int issuer;           // 0 / 1: this warp issues MMA group 0 / 1 (warps 0 and 1 of the tile); -1: none
};

__device__ __forceinline__ void tile_sync(const TcTile& t) { tc::named_bar_sync(t.bar_id, t.bar_threads); }

// Hand the freshly written A operands to the tensor core and wait for completion.  The MMAs of a round trip are split
// into two independent groups (different D columns) issued concurrently by the elected lane of the tile's warps 0 and 1
// (elect.sync: the operands stay in uniform registers, ~23 cycles per tcgen05.mma, csrc/dev/tc_latency.cu), each
// committing to its own mbarrier.  Only those two warps poll; the other warps sleep on the hardware barrier (letting
// every warp poll measured slower: the polling costs issue slots).
// MEASURED alternatives (round 2, B200, c4; all correct, all slower, removed): every warp of the tile sleeping on the two
// mbarriers (try_wait with a suspend-time hint) instead of the second tile barrier: +3 %; one Philox block of the next
// step's noise between the MMA issue and the wait ("slack" work, parked in spare TMEM columns), by every warp: +6 %, by
// the two non-issuing warps only (which otherwise sleep at the tile barrier): +1.5 % -- the noise phase shrinks by what
// the flow phase grows; four tanh sharing one MUFU.RCP (5 MUFU + 9 FMUL instead of 8 MUFU): +2 %.
template <typename F0, typename F1>
__device__ __forceinline__ void tc_round_trip(TcTile& t, F0 issue0, F1 issue1) {
  tc::wait_st();
  tc::fence_before_sync();
  tile_sync(t);
  if (t.issuer >= 0) {   // warp-uniform: the whole warp takes the branch so that no lane spins next to the issuing lane
    tc::fence_after_sync();
    if (tc::elect_one()) {
      if (t.issuer == 0) issue0(); else issue1();
      tc::mma_commit(t.mbar + t.issuer);
    }
    __syncwarp();
  }
  if (t.issuer >= 0) {
    tc::mbar_wait(t.mbar + t.issuer, t.phase);
    __syncwarp();
  }
  t.phase ^= 1u;
  tile_sync(t);
  tc::fence_after_sync();
}

// bias + activation + hi/lo split of the 32 hidden pre-activations (s-net 16 tanh | t-net 16 relu):
// D cols [64,96) -> A hi cols [0,32), lo cols [32,64), in 8-column chunks dealt round-robin to the chain's threads
// (NPART = 2: each gets one tanh chunk and one relu chunk).  A rolled loop keeps the code small.
template <int NPART>
__device__ __forceinline__ void tc_hidden_epilogue(const TcTile& t, const float* __restrict__ bias) {
  if (NPART == 1) {
    // one thread per chain: all 32 pre-activations arrive with ONE tcgen05.ld (one TMEM latency instead of four); the two
    // nets' halves are then independent work for the scheduler, each leaving with one tcgen05.st per hi / lo half
    uint32_t r[32];
    tc::tmem_ld32(t.lane_tmem + 64, r);
    tc::wait_ld();
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t hi[16], lo[16];
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[16 * c + j]) + bias[16 * c + j];
      if (c == 0) {
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const float2 th = tc_tanh_scaled2(make_float2(v[j], v[j + 1]));
          v[j] = th.x;
          v[j + 1] = th.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
      }
      tc::split_tf32<16>(v, hi, lo);
      tc::tmem_st16(t.lane_tmem + 16 * c, hi);
      tc::tmem_st16(t.lane_tmem + 32 + 16 * c, lo);
    }
    return;
  }
  // two threads per chain: a rolled loop keeps the code (and the 64-register budget) small
#pragma unroll 1
  for (int c = t.part; c < 4; c += NPART) {
    uint32_t r[8], hi[8], lo[8];
    tc::tmem_ld8(t.lane_tmem + 64 + 8 * c, r);
    tc::wait_ld();
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[j]) + bias[8 * c + j];
    if (c < 2) {
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        const float2 th = tc_tanh_scaled2(make_float2(v[j], v[j + 1]));
        v[j] = th.x;
        v[j + 1] = th.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    tc::split_tf32<8>(v, hi, lo);
    tc::tmem_st8(t.lane_tmem + 8 * c, hi);
    tc::tmem_st8(t.lane_tmem + 32 + 8 * c, lo);
  }
}

// Output epilogue of a coupling block, columns o = ob + j (j < W) of the dims it transforms (dim o0 + 2 o).
// yv <- the dims' current values (src 0: y; 1: nz; 2: the proposal z + scale * n, also written back to nz).  Loads first,
// then the stores (see batched<>).
template <int W>
__device__ __forceinline__ void tc_out_y(float* yv, int ob, int nout, int o0, int ys, int src, const float* y,
                                         const float* zc, float* nz, float scale) {
#pragma unroll
  for (int j = 0; j < W; j += 2) {
    const int o = ob + j, i = o0 + 2 * o;
    if (src == 2 && o + 1 < nout) {
      const float2 zz = tc_propose2(make_float2(zc[i * ys], zc[(i + 2) * ys]), make_float2(nz[i * ys], nz[(i + 2) * ys]), scale);
      yv[j] = zz.x;
      yv[j + 1] = zz.y;
    } else {
#pragma unroll
      for (int q = 0; q < 2; ++q)
        if (o + q < nout) {
          const int iq = i + 2 * q;
          yv[j + q] = src == 2 ? __fadd_rn(zc[iq * ys], __fmul_rn(nz[iq * ys], scale)) : (src == 1 ? nz[iq * ys] : y[iq * ys]);
        }
    }
  }
  if (src == 2) {
#pragma unroll
    for (int j = 0; j < W; ++j)
      if (ob + j < nout) nz[(o0 + 2 * (ob + j)) * ys] = yv[j];
  }
}
// x = (y - t) * 2^{l'} of the same columns (0 past nout), ld += l' in column order (l' = -log2(e) log_s).  The bias adds
// stay scalar (constant-bank operands); the subtract and the multiply run as packed FP32 pairs.
template <int W>
__device__ __forceinline__ void tc_out_x(const uint32_t* rs, const uint32_t* rt, const float* yv,
                                         const float* __restrict__ b3s, const float* __restrict__ b3t, int ob, int nout,
                                         float* xv, float& ld) {
#pragma unroll
  for (int j = 0; j < W; j += 2) {
    const int o = ob + j;
    xv[j] = xv[j + 1] = 0.f;
    if (o + 1 < nout) {
      const float ls0 = __uint_as_float(rs[j]) + b3s[o], ls1 = __uint_as_float(rs[j + 1]) + b3s[o + 1];
      const float tt0 = __uint_as_float(rt[j]) + b3t[o], tt1 = __uint_as_float(rt[j + 1]) + b3t[o + 1];
      const float2 x2 = __fmul2_rn(__fadd2_rn(make_float2(yv[j], yv[j + 1]), make_float2(-tt0, -tt1)),
                                   make_float2(tc_exp2(ls0), tc_exp2(ls1)));
      xv[j] = x2.x;
      xv[j + 1] = x2.y;
      ld += ls0;
      ld += ls1;
    } else if (o < nout) {
      const float ls = __uint_as_float(rs[j]) + b3s[o], tt = __uint_as_float(rt[j]) + b3t[o];
      xv[j] = (yv[j] - tt) * tc_exp2(ls);
      ld += ls;
    }
  }
}

// Flow inverse of one tile, in place on y (shared memory, stride ys).  Returns this thread's share of
// log|det dx/dz| of the chain (the sum over the chain's NPART threads is the log-det).  Ends with a tile barrier:
// afterwards every thread of the tile sees the complete x.
// fused == false: the caller has written the flow's input z' to y.  fused == true (needs at least two blocks): y holds NO
// input -- the proposal z'_i = zc[i] + scale * nz[i] (sampler.py:310-316) is formed where the flow first consumes dim i
// (the first block's inputs and the dims it transforms) and is written back over the noise, nz[i] = z'_i: the second
// block reads the dims it transforms from there, and after an accepted step the caller just swaps its zc / nz pointers
// instead of copying.  Every dim is transformed by one of the first two blocks, so y is complete at the end.
// t_col: TMEM column of the translate net's output (96; 80 when every block transforms at most 16 dims, which leaves
// columns [96,128) to the kernel).
template <int NPART, int DD>
__device__ __forceinline__ float tc_flow_inverse(const TcFlowDesc& f, const float* __restrict__ wsm, uint32_t wsm_u32,
                                                 TcTile& t, float* y, int ys, float* ld_slot, int* bad_slot,
                                                 const float* __restrict__ cb, const float* __restrict__ lof,
                                                 const float* __restrict__ hif, bool box_check, bool& bad, uint32_t t_col,
                                                 bool fused, const float* zc, float* nz, float scale) {
  // DD > 0: x_dim, num_layers = 1 and num_blocks = 3 (the reference's defaults) are compile-time constants: every loop
  // below unrolls and every shared-memory / TMEM offset becomes an immediate
  const int d = DD > 0 ? DD : f.d, L = DD > 0 ? 1 : f.L, nB = DD > 0 ? 3 : f.B;
  float ld = 0.f;
  bad = false;
#pragma unroll
  for (int k = nB - 1; k >= 0; --k) {
    const int nin = blk_nin(d, k), i0 = blk_i0(k), nout = blk_nout(d, k), o0 = blk_o0(k);
    const int K1 = round8(nin), N3 = round16(nout);
    const int base = DD > 0 ? (k > 0 ? tc_block_floats(d, L, 0) : 0) + (k > 1 ? tc_block_floats(d, L, 1) : 0) : f.off[k];
    // ---- layer 1: A = masked inputs (dims with mask == 1), zero padded to K1.  Only the first block reads them from
    // y: the inputs of every later block are exactly the dims the previous block's output epilogue has just produced
    // (masks alternate, input a of block k-1 == output o of block k), and that epilogue stores them straight into the
    // A columns -- same thread, same column chunk, no shared-memory round trip and no tile barrier in between.
    if (k == nB - 1) {
      for (int c0 = (NPART == 1 ? 0 : 8 * t.part); c0 < K1; c0 += 8 * NPART) {
        uint32_t hi[8], lo[8];
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          const int a = c0 + j, i = i0 + 2 * a;   // inputs a, a + 1 = dims i, i + 2
          if (fused && a + 1 < nin) {
            const float2 zz = tc_propose2(make_float2(zc[i * ys], zc[(i + 2) * ys]),
                                          make_float2(nz[i * ys], nz[(i + 2) * ys]), scale);
            v[j] = zz.x;
            v[j + 1] = zz.y;
          } else {
            v[j] = a < nin ? (fused ? __fadd_rn(zc[i * ys], __fmul_rn(nz[i * ys], scale)) : y[i * ys]) : 0.f;
            v[j + 1] = a + 1 < nin ? y[(i + 2) * ys] : 0.f;   // (fused: a + 1 >= nin here)
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {   // (stores after all loads of the chunk: see batched<>)
          const int a = c0 + j, i = i0 + 2 * a;
          if (fused && a < nin) nz[i * ys] = v[j];
        }
        tc::split_tf32<8>(v, hi, lo);
        tc::tmem_st8(t.lane_tmem + c0, hi);
        tc::tmem_st8(t.lane_tmem + 32 + c0, lo);
      }
    }
    {
      const uint32_t b_hi = wsm_u32 + 4u * base, b_lo = b_hi + 4u * 32u * K1;
      // B1 is packed for N = 32 (nN = 4 n-blocks per K chunk); the two issuers take n-blocks {0,1} / {2,3}:
      // same LBO (4 * 128 B), start address + 2 * 128 B, N = 16
      tc_round_trip(t,
                    [&] {
                      if (t.single) tc::mma_3xtf32(t.tmem + 64, t.tmem, t.tmem + 32, b_hi, b_lo, K1 / 8, 32, false);
                      else tc::mma_3xtf32_n(t.tmem + 64, t.tmem, t.tmem + 32, b_hi, b_lo, K1 / 8, 16, 4, false);
                    },
                    [&] { tc::mma_3xtf32_n(t.tmem + 80, t.tmem, t.tmem + 32, b_hi + 256u, b_lo + 256u, K1 / 8, 16, 4, false); });
    }
    int off = base + 64 * K1 + 32;   // past B1 and (the shared-memory copy of) bias1
    // biases: constant bank (cb), see TcConsts
    const int cbk = DD > 0 ? tc_cb_off(DD, 1, k) : tc_cb_off(d, L, k);
    tc_hidden_epilogue<NPART>(t, cb + cbk);
    // ---- hidden layers: block diagonal, s-net cols [0,16), t-net cols [16,32) --------------------------------
    for (int l = 0; l < L; ++l) {
      const uint32_t bs_hi = wsm_u32 + 4u * off, bs_lo = bs_hi + 1024u, bt_hi = bs_hi + 2048u, bt_lo = bs_hi + 3072u;
      tc_round_trip(t,
                    [&] {
                      tc::mma_3xtf32(t.tmem + 64, t.tmem, t.tmem + 32, bs_hi, bs_lo, 2, 16, false);
                      if (t.single) tc::mma_3xtf32(t.tmem + 80, t.tmem + 16, t.tmem + 48, bt_hi, bt_lo, 2, 16, false);
                    },
                    [&] { tc::mma_3xtf32(t.tmem + 80, t.tmem + 16, t.tmem + 48, bt_hi, bt_lo, 2, 16, false); });
      tc_hidden_epilogue<NPART>(t, cb + cbk + 32 + 32 * l);
      off += 1056;
    }
    // ---- output layer: log_s -> D cols [64, 64+N3), t -> D cols [96, 96+N3) ------------------------------------
    {
      const uint32_t sz = 4u * 16u * N3;
      const uint32_t bs_hi = wsm_u32 + 4u * off, bs_lo = bs_hi + sz, bt_hi = bs_hi + 2 * sz, bt_lo = bs_hi + 3 * sz;
      tc_round_trip(t,
                    [&] {
                      tc::mma_3xtf32(t.tmem + 64, t.tmem, t.tmem + 32, bs_hi, bs_lo, 2, N3, false);
                      if (t.single) tc::mma_3xtf32(t.tmem + t_col, t.tmem + 16, t.tmem + 48, bt_hi, bt_lo, 2, N3, false);
                    },
                    [&] { tc::mma_3xtf32(t.tmem + t_col, t.tmem + 16, t.tmem + 48, bt_hi, bt_lo, 2, N3, false); });
    }
    const float* b3s = cb + cbk + 32 + 32 * L;
    const float* b3t = b3s + N3;
    // x = (z - t) * exp(-log_s), ld -= log_s on the dims with mask == 0   (networks.py:300-309).  The values a dim keeps
    // (its last update: blocks 1 and 0) are tested against the prior box right here (priors.py:39-43).
    const bool chk = box_check && k <= 1;
    // where y of a transformed dim comes from: the proposal z + scale * n formed here (first block of a fused flow), the
    // first block's output left in nz (second block of a fused flow), or y
    const int ysrc = fused && k == nB - 1 ? 2 : (fused && k == nB - 2 ? 1 : 0);
    if (NPART == 1 && N3 == 16) {
      // one thread per chain, at most 16 transformed dims: both output rows arrive before a single wait, and the A operand
      // of the next block leaves with one tcgen05.st per half (columns past nout: zeros, never read by layer 1)
      uint32_t rs[16], rt[16], hi[16], lo[16];
      tc::tmem_ld16(t.lane_tmem + 64, rs);
      tc::tmem_ld16(t.lane_tmem + t_col, rt);
      float yv[16];   // the dims this block transforms, read before any of them is written back (see batched<>)
      tc_out_y<16>(yv, 0, nout, o0, ys, ysrc, y, zc, nz, scale);
      tc::wait_ld();
#pragma unroll
      for (int c0 = 0; c0 < 16; c0 += 8) {
        float xv[8];
        tc_out_x<8>(rs + c0, rt + c0, yv + c0, b3s, b3t, c0, nout, xv, ld);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int o = c0 + j;
          if (o < nout) {
            y[(o0 + 2 * o) * ys] = xv[j];
            if (chk) bad |= (xv[j] < lof[o0 + 2 * o]) | (xv[j] > hif[o0 + 2 * o]);
          }
        }
        tc::split_tf32<8>(xv, hi + c0, lo + c0);
      }
      if (k > 0) {   // A operand of block k-1's first layer
        tc::tmem_st16(t.lane_tmem, hi);
        tc::tmem_st16(t.lane_tmem + 32, lo);
      }
    } else {
    for (int c0 = (NPART == 1 ? 0 : 8 * t.part); c0 < nout; c0 += 8 * NPART) {
      uint32_t rs[8], rt[8], hi[8], lo[8];
      tc::tmem_ld8(t.lane_tmem + 64 + c0, rs);
      tc::tmem_ld8(t.lane_tmem + t_col + c0, rt);
      float yv[8], xv[8];
      tc_out_y<8>(yv, c0, nout, o0, ys, ysrc, y, zc, nz, scale);
      tc::wait_ld();
      tc_out_x<8>(rs, rt, yv, b3s, b3t, c0, nout, xv, ld);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int o = c0 + j;
        if (o < nout) {
          y[(o0 + 2 * o) * ys] = xv[j];
          if (chk) bad |= (xv[j] < lof[o0 + 2 * o]) | (xv[j] > hif[o0 + 2 * o]);
        }
      }
      if (k > 0) {   // A operand of block k-1's first layer
        tc::split_tf32<8>(xv, hi, lo);
        tc::tmem_st8(t.lane_tmem + c0, hi);
        tc::tmem_st8(t.lane_tmem + 32 + c0, lo);
      }
    }
    }
    if (k == 0) ld *= 0.6931471805599453f;   // sum of -log2(e) log_s  ->  -sum log_s
    if (NPART > 1 && k == 0) {
      ld_slot[0] = ld;                          // the chain's threads exchange their log-det shares and box flags through
      if (t.part == 1) *bad_slot = bad;         // shared memory (the flag slot carries the accept decision later on)
      tile_sync(t);                             // every thread of the tile now sees the complete x
    }
  }
  return ld;
}

// one out-of-line copy of the likelihood / prior switch per kernel (code size)
// (the target is re-bound from its descriptor inside the call: passing the bound struct by reference would park its
// pointers in local memory and reload them for every coordinate)
template <int DD>
static __device__ __noinline__ double tc_loglike(TargetDesc td, const double* td_s, const float* y) {
  TargetSmem tg;
  target_bind(tg, td, td_s);
  SmemRow row{y};
  return loglike_any<SmemRow, DD>(tg, row, false);
}
template <int DD>
static __device__ __noinline__ double tc_prior(TargetDesc td, const double* td_s, const float* y) {
  TargetSmem tg;
  target_bind(tg, td, td_s);
  SmemRow row{y};
  return prior_any<SmemRow, DD>(tg, row, false);
}

// shared-memory carve-up (bytes): [tc weights][target doubles][y: ntiles*d*128 f][zp: ntiles*d*128 f]
//   [nz: ntiles*d*128 f][ldp: ntiles*(NPART + 1)*128 f][flag: ntiles*128 i][mbar: 8 x 8][tmem base 8][red 32 x 4]
//   [weight mbarriers: NNB_MAX_BLOCKS x 8]
template <int MODE, int NPART, int DD>
__global__ void __launch_bounds__(kTcMaxTiles * 128 * NPART, 1)
mcmc_tc_kernel(TcFlowDesc f, const float* __restrict__ wglob, TargetDesc td, const double* __restrict__ tgt_g,
               McmcParams p, const __grid_constant__ TcConsts cst) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // A CTA owns p.cpc chains (a multiple of 32): full tiles of 128 plus, possibly, a partial last tile, so that
  // the batch can be spread evenly over all SMs (65 536 chains = 148 x 448 - a few).  Threads are laid out
  // tile-major, then part-major; a partial tile simply has fewer warps per part (lane quarters).
  const int d = DD > 0 ? DD : f.d;
  const float* cst_t = cst.v + (DD > 0 ? tc_cb_off(DD, 1, 3) : tc_cb_off(f.d, f.L, f.B));   // tsf | tbf | lof | hif
  const int cpc = p.cpc;
  const int ntiles = (cpc + 127) >> 7;
  float* wsm = reinterpret_cast<float*>(smem_raw);
  double* td_s = reinterpret_cast<double*>(smem_raw + (size_t)f.total_floats * 4);
  const int nd = target_doubles(td.d, td.n_params);
  float* y_all = reinterpret_cast<float*>(td_s + nd);
  float* zp_all = y_all + (size_t)ntiles * d * 128;
  float* nz_all = zp_all + (size_t)ntiles * d * 128;
  float* ldp_all = nz_all + (size_t)ntiles * d * 128;
  int* flag_all = reinterpret_cast<int*>(ldp_all + (size_t)ntiles * (NPART + 1) * 128);
  uint64_t* mbars = reinterpret_cast<uint64_t*>(flag_all + (size_t)ntiles * 128);
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(mbars + 2 * kTcMaxTiles);
  uint64_t* wbars = reinterpret_cast<uint64_t*>(tmem_base_s + 2 + 32);   // one mbarrier per coupling block's weights
  uint64_t* sbar = wbars + NNB_MAX_BLOCKS;   // per-step hand-off of the new scale from the CTA's poller to the tile leaders

  // Weights: TMA bulk copies (cp.async.bulk -> UBLKCP), one per coupling block in the order the flow inverse needs them
  // (last block first), each completing on its own mbarrier.  They land while the CTA allocates TMEM, loads the chains'
  // state and draws the first step's noise; the wait sits in front of the step loop.
  const int nblk_w = DD > 0 ? 3 : f.B;
  if (threadIdx.x == 0) {
    for (int k = 0; k < nblk_w; ++k) tc::mbar_init(&wbars[k], 1);
    tc::mbar_init(sbar, 1);
    tc::mbar_fence_init();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int k = nblk_w - 1; k >= 0; --k) {
      const int off = f.off[k];
      const uint32_t bytes = 4u * (uint32_t)((k + 1 < nblk_w ? f.off[k + 1] : f.total_floats) - off);
      tc::mbar_expect_tx(&wbars[k], bytes);
      tc::tma_bulk_g2s(wsm + off, wglob + off, bytes, &wbars[k]);
    }
  }
  for (int i = threadIdx.x; i < nd; i += blockDim.x) td_s[i] = tgt_g[i];
  TargetSmem tg;
  target_bind(tg, td, td_s);

  const int warp = threadIdx.x >> 5;
  // warp slots: tile j owns warps [4*NPART*j, 4*NPART*(j+1)); part p, lane quarter q -> warp 4*NPART*j + 4p + q.  The
  // hardware lets a warp touch only the TMEM lane quarter (warp id % 4), so a partial tile keeps this layout and
  // leaves the warps of its unused quarters idle.
  const int tile = threadIdx.x / (128 * NPART);
  const int rows = tile == ntiles - 1 ? cpc - 128 * (ntiles - 1) : 128;   // chains of this tile
  const int tit = threadIdx.x % (128 * NPART);                             // thread slot in tile
  const int m = tit & 127;                                                 // chain in tile = TMEM lane
  const uint32_t tmem_cols = ntiles <= 1 ? 128u : (ntiles == 2 ? 256u : 512u);
  if (warp == 0) tc::tmem_alloc(tmem_base_s, tmem_cols);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2 * kTcMaxTiles; ++i) tc::mbar_init(&mbars[i], 1);
    tc::mbar_fence_init();
  }
  // (the TMA writes the weights through the async proxy, which is also how the tensor core reads them)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();

  TcTile t;
  t.tmem = *tmem_base_s + (uint32_t)tile * kTcColsPerTile;
  t.lane_tmem = t.tmem + (((uint32_t)(m >> 5) * 32u) << 16);   // == (warp id % 4) * 32
  t.mbar = &mbars[2 * tile];
  t.phase = 0;
  t.bar_id = 1 + tile;
  t.bar_threads = rows * NPART;
  t.part = tit >> 7;
  // the two MMA-issuing warps of a tile: tiles 1 and 2 use their warps 2 and 3 (schedulers 2 and 3), tiles 0 and 3 their
  // warps 0 and 1 -- every tcgen05.mma keeps its warp's scheduler busy for ~23 cycles, and with all issuers on
  // schedulers 0 and 1 those two carried half as much work again as the others
  {
    const int wq = tit >> 5, first = (rows == 128 && (tile == 1 || tile == 2)) ? 2 : 0;
    t.issuer = wq == first ? 0 : (wq == first + 1 && rows > 32 ? 1 : -1);
  }
  t.single = rows <= 32;   // a 32-chain tile has only one warp per part
  const int part = NPART == 1 ? 0 : t.part;
  const uint32_t wsm_u32 = tc::smem_u32(wsm);

  const long long n = p.n;
  const long long tile_base = (long long)blockIdx.x * cpc + tile * 128;
  const bool tile_active = tile_base < n && m < rows;   // uniform over a warp; idle quarter warps of a partial tile skip
  const long long c = tile_base + m;
  const bool active = c < n && m < rows;   // idle quarter warps of a partial tile own no chain
  float* y = y_all + (size_t)tile * d * 128 + m;
  float* zp = zp_all + (size_t)tile * d * 128 + m;
  float* ldp = ldp_all + (size_t)tile * (NPART + 1) * 128 + m;   // [ld: NPART x 128][u: 128]
  float* u_slot = ldp + NPART * 128;
  int* flag = flag_all + (size_t)tile * 128 + m;
  const unsigned int chain = (unsigned int)(p.chain_offset + (unsigned long long)c);
  unsigned int acc_total = 0, ncall_total = 0;
  float ld_cur = 0.f;
  double logl_cur = 0.0, logp_cur = 0.0;
  if (active && part == 0) {
    ld_cur = p.logdet[c];
    logl_cur = p.logl[c];
    logp_cur = p.logp[c];
  }
  const int nj = (d + 3) / 4;
  const size_t ns = (size_t)n;
  float* nz = nz_all + (size_t)tile * d * 128 + m;
  // cooperative (persistent) mode: every tile leader keeps its own copy of (scale, accept, reject); they stay identical
  // because each is updated from the same grid-wide accept count after the per-step grid barrier
  double co_scale = 0.0;
  // CTA-level rendezvous words of the cooperative mode (red region, 32 words):
  //   [0] scale (float) of the step about to start   [1] tiles arrived   [2] accepted proposals of the arrived tiles
  //   [3] epoch = steps whose grid-wide count has been consumed          [4] accept  [5] reject  [6..7] scale (double)
  unsigned int* co_words = tmem_base_s + 2;
  float* co_scale_s = reinterpret_cast<float*>(co_words);
  const int my_tiles = (int)(((n - (long long)blockIdx.x * cpc < cpc ? n - (long long)blockIdx.x * cpc : cpc) + 127) >> 7);
  if (p.coop) {
    if (threadIdx.x == 0) {
      co_scale = *reinterpret_cast<volatile double*>(&p.ctrl->scale);
      *co_scale_s = (float)co_scale;
      co_words[1] = co_words[2] = co_words[3] = 0u;
      co_words[4] = (unsigned int)p.ctrl->accept;
      co_words[5] = (unsigned int)p.ctrl->reject;
      *reinterpret_cast<double*>(co_words + 6) = co_scale;
    }
    __syncthreads();
  }

  // one thread per chain: the current latent point stays in shared memory for all steps of the launch
  constexpr bool kZcur = NPART == 1;
  constexpr int kCh = DD > 0 ? 16 : 8;   // coordinates per batch of the shared-memory loops (batched<>)
  if (kZcur && tile_active)   // (idle lanes of a live warp: zeros, so that their rows of the MMAs stay finite)
    for (int i = 0; i < d; ++i) {
      zp[i * 128] = active ? p.z[(size_t)c + (size_t)i * ns] : 0.f;
      if (!active) nz[i * 128] = 0.f;
    }

  // raw N(0,1) draws of Philox blocks j = j0, j0 + jstep, ... < j1 of step `step_abs` into nz (and the dump buffer)
  auto gen_normals = [&](int j0, int j1, int jstep, unsigned int step_abs, int sidx) {
    if (DD > 0 && NPART == 1) {
      // one thread per chain, x_dim fixed: all blocks 0 .. nj-1, kTcPhiloxIlp of them at a time -- the Philox rounds and the
      // Box-Muller transforms of a group are straight-line code (one basic block) that the scheduler interleaves; the
      // stores and the optional dump follow the group.  (A block is a serial chain: ten dependent rounds, then
      // lg2 -> sqrt and sin / cos; one at a time it runs at ~330 cycles per block.)
      constexpr int NJ = DD > 0 ? (DD + 3) / 4 : 1;
#pragma unroll
      for (int jb = 0; jb < NJ; jb += kTcPhiloxIlp) {
        float nrm[kTcPhiloxIlp][4];
#pragma unroll
        for (int u = 0; u < kTcPhiloxIlp; ++u)
          if (jb + u < NJ) philox_normals4(jb + u, step_abs, chain, kTagNormal, p.seed_lo, p.seed_hi, nrm[u]);
#pragma unroll
        for (int u = 0; u < kTcPhiloxIlp; ++u)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = 4 * (jb + u) + q;
            if (jb + u < NJ && i < DD) nz[i * 128] = nrm[u][q];
          }
        if (p.dump_normals) {
#pragma unroll
          for (int u = 0; u < kTcPhiloxIlp; ++u)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int i = 4 * (jb + u) + q;
              if (jb + u < NJ && i < DD) p.dump_normals[((size_t)sidx * ns + (size_t)c) * d + i] = nrm[u][q];
            }
        }
      }
      return;
    }
#pragma unroll(DD > 0 ? 2 : 1)
    for (int j = j0; j < j1; j += jstep) {
      float nrm[4];
      philox_normals4(j, step_abs, chain, kTagNormal, p.seed_lo, p.seed_hi, nrm);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = 4 * j + q;
        if (i < d) {
          nz[i * 128] = nrm[q];
          if (p.dump_normals) p.dump_normals[((size_t)sidx * ns + (size_t)c) * d + i] = nrm[q];
        }
      }
    }
  };
  // The noise of step s+1 does not depend on the adapted scale, so it is produced while step s finishes: jc blocks
  // by the chain's second thread during the accept phase of the first, the rest by both after the CTA has arrived
  // at the grid barrier (overlapping its latency).
  const int jc = NPART > 1 ? (p.tc_jc >= 0 ? (p.tc_jc < nj ? p.tc_jc : nj) : (3 * nj + 4) / 8) : 0;
  const bool philox = p.replay_normals == nullptr;
  // the accept test's uniform of step `step_abs` (sampler.py:334), drawn ahead of time by the chain's last thread
  auto gen_uniform = [&](unsigned int step_abs, int sidx) {
    uint4 r = philox4x32_10(0u, step_abs, chain, kTagUniform, p.seed_lo, p.seed_hi);
    const float u = uniform01(r.x);
    *u_slot = u;
    if (p.dump_uniforms) p.dump_uniforms[(size_t)sidx * ns + (size_t)c] = u;
  };
  const bool philox_u = p.replay_uniforms == nullptr;
  if (tile_active && active && philox) gen_normals(part, nj, NPART, p.step_offset + (unsigned int)(p.s0 + 1), p.s0);
  if (tile_active && active && philox_u && part == NPART - 1) gen_uniform(p.step_offset + (unsigned int)(p.s0 + 1), p.s0);
  // weights have landed (each thread observes every block's mbarrier: phase 0 completes when its bytes are in)
  for (int k = nblk_w - 1; k >= 0; --k) tc::mbar_wait(&wbars[k], 0u);
  // TMEM column of the translate net's output: 80 when every block transforms at most 16 dims, else 96
  const bool small_d = DD > 0 ? DD <= 32 : d <= 32;
  const uint32_t t_col = small_d ? 80u : 96u;
  // One thread per chain and at least two coupling blocks: the proposal is formed inside the flow (tc_flow_inverse: zsrc)
  const bool fused = NPART == 1 && (DD > 0 || f.B >= 2);
  // prior box on the flow's own coordinates (nested sampling): tested inside the output epilogues of the flow
  const bool fast_box = MODE == NNB_MODE_HARD && tg.desc.prior_kind == NNB_PRIOR_BOX_U && (DD > 0 || f.B >= 2);

  // x = flow^-1(z) of a chain is needed only when the launch ends (or for a trace): with all steps in one launch, an
  // accepted proposal just marks the chain as moved, and ONE extra pass of the flow after the last step -- the step loop's
  // own code with scale = 0, i.e. z' = z exactly -- recomputes x of the moved chains from their final z.  Same thread, same
  // tile slot, same instruction sequence on the same z bits as the step that accepted it: the same x bits, without 30
  // shared-memory loads + 30 global stores per accepted step.
  const bool defer_x = fused && p.nsteps > 1 && p.trace_z == nullptr;
  bool moved = false;
  const int s_end = p.s0 + p.nsteps + (defer_x ? 1 : 0);
  for (int s = p.s0 + 1; s <= s_end; ++s) {
    const unsigned int step_abs = p.step_offset + (unsigned int)s;
    const bool more = s < p.s0 + p.nsteps;
    const bool x_pass = s > p.s0 + p.nsteps;   // the extra pass (defer_x)
    bool accept = false;
    unsigned int ncall = 0, tile_cnt = 0;
    bool acc_chain = false;
#ifdef NNB_TC_TIMING
    const int si_t = s - p.s0 - 1;
#endif
    if (tile_active) {
      if (NPART > 1 || p.coop) tile_sync(t);   // nz complete (written by both threads of the chain); scale published
      NNB_TSTAMP(0);
      // The tiles of an SM leave the grid barrier together and would then all run their epilogues at the same moments and
      // all wait for their MMAs at the same moments; odd tiles therefore start the step about half a round trip late
      // (p.tc_delay, NNB_TC_DELAYS; measured on the B200 at c4: 2.23 ms -> 2.14 ms per refill at 700 cycles; re-swept with the
      // packed epilogues (1.82 ms): 500 / 900 cycles within 0.3 % of 700, no delay +1.2 %)
      if (p.tc_delay[tile & 3] > 0) {
        const long long t0 = clock64();
        while (clock64() - t0 < (long long)p.tc_delay[tile & 3]) {}
      }
#ifdef NNB_TC_TIMING
      if (tit == 0 && si_t < kTimeSteps) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        g_tc_time[(((size_t)blockIdx.x * kTcMaxTiles + tile) * kTimeSteps + si_t) * kTimeSlots + 5] = gt;
      }
#endif
      const float scale_f = x_pass ? 0.f
                                   : (p.coop ? *reinterpret_cast<volatile float*>(co_scale_s)
                                             : (float)(*reinterpret_cast<volatile double*>(&p.ctrl->scale)));
      // this step's accept uniform: read now, the slot is refilled for the next step while the flow runs
      const float u01_cur = (active && philox_u && part == NPART - 1) ? *u_slot : 0.f;
      // ---- proposal z' = z + scale * N(0, I) (sampler.py:310-316) ---------------------------------------------------
      if (kZcur) {
        // one thread per chain: the current z (zp) and the step's noise (nz) live in shared memory; replayed noise is
        // copied into nz first so that the flow and the accept update have a single source
        if (!philox && active && !x_pass) {
          const float* nr = p.replay_normals + ((size_t)(s - 1) * ns + (size_t)c) * d;
          batched<kCh>(d, [&](int i) { return nr[i]; }, [&](int i, float v) { nz[i * 128] = v; });
        }
        if (!fused)   // (single-block flows: z' goes through y; idle lanes hold zeros in zp and nz)
          batched<kCh>(d, [&](int i) { return __fadd_rn(zp[i * 128], __fmul_rn(nz[i * 128], scale_f)); },
                       [&](int i, float v) { y[i * 128] = v; });
      } else if (active) {   // dims dealt to the chain's threads
        const float* pz = p.z + (size_t)c + (size_t)part * ns;
        if (philox) {
          for (int i = part; i < d; i += NPART, pz += NPART * ns) {
            float v = __fadd_rn(*pz, __fmul_rn(nz[i * 128], scale_f));
            y[i * 128] = v;
            zp[i * 128] = v;
          }
        } else {
          const float* nr = p.replay_normals + ((size_t)(s - 1) * ns + (size_t)c) * d;
          for (int i = part; i < d; i += NPART, pz += NPART * ns) {
            float v = __fadd_rn(*pz, __fmul_rn(nr[i], scale_f));
            y[i * 128] = v;
            zp[i * 128] = v;
          }
        }
      } else {
        for (int i = part; i < d; i += NPART) y[i * 128] = 0.f;
      }
      __syncwarp();
      NNB_TSTAMP(6);
      if (NPART > 1) tile_sync(t);   // layer 1 reads dims written by the partner thread
      // ---- flow inverse on the tensor cores (all threads of the tile, converged) ----------------------------------
      bool bad_part;
      const float ld_part = tc_flow_inverse<NPART, DD>(
          f, wsm, wsm_u32, t, y, 128, ldp + part * 128, flag, cst.v, cst_t + 2 * d, cst_t + 3 * d, fast_box, bad_part, t_col,
          fused, zp, nz, scale_f);
      NNB_TSTAMP(1);
      if (x_pass) {   // (uniform over the grid)
        if (active && moved) {
          float* px = p.x + (size_t)c;
          batched<kCh>(d, [&](int i) { return y[i * 128]; }, [&](int i, float v) { px[(size_t)i * ns] = v; });
        }
        break;
      }
      // ---- accept / reject: thread 0 of the chain; thread 1 starts on the next step's noise -------------------------
      if (active && part == 0) {
        float ld_prop = ld_part;
        if (NPART > 1) ld_prop = ld_part + ldp[128];
        const float u01 = philox_u ? (NPART == 1 ? u01_cur : *u_slot) : p.replay_uniforms[(size_t)(s - 1) * ns + (size_t)c];
        double lp = 0.0, logp_prop = 0.0;
        if (MODE == NNB_MODE_HARD) {
          float lr = __fsub_rn(ld_prop, ld_cur);
          if (fast_box) {
            bool bad = bad_part;
            if (NPART > 1) bad |= *flag != 0;
            logp_prop = bad ? -INFINITY : 0.0;
          } else {
            logp_prop = tc_prior<DD>(td, td_s, y);
          }
          if (logp_prop < -1e30) lr = -INFINITY;
          float ratio = expf(lr);
          if (ratio > 1.0f) ratio = 1.0f;
          const bool m1 = u01 < ratio;
          if (m1) {
            if (DD > 0 && td.like_id == NNB_LIKE_ROSENBROCK && !td.compute_f64 && td.has_transform &&
                builtin_transform(td)) {
              // the config-4 target inline (same arithmetic as loglike_T<float>: likelihoods.py:50-51 after the float32
              // affine transform), transform coefficients as constant-bank operands
              // The terms i = 1 .. N run as packed FP32 pairs (i, i + h), h = ceil(N / 2): with V_m = (x_m, x_{m+h}) a pair's
              // current and previous values are V_i and V_{i-1}.  acc still adds the terms in the order i = 1 .. N: the first
              // lanes as they come, then the second lanes (terms h+1 .. N).
              constexpr int D1 = DD > 0 ? DD : 1, N = D1 - 1, h = (N + 1) / 2;
              auto xt = [&](int i) { return i < D1 ? __fadd_rn(__fmul_rn(y[i * 128], cst_t[i]), cst_t[D1 + i]) : 0.f; };
              float acc = 0.f, late[h > 0 ? h : 1];
              float2 prev = make_float2(xt(0), xt(h));
#pragma unroll
              for (int i = 1; i <= h; ++i) {
                const float2 cur = make_float2(xt(i), xt(i + h));
                // (the adds that take a product are scalar: see tc_propose2)
                const float2 sq = __fmul2_rn(prev, prev);
                const float2 t1 = make_float2(__fsub_rn(cur.x, sq.x), __fsub_rn(cur.y, sq.y));
                const float2 t2 = __fadd2_rn(make_float2(1.f, 1.f), make_float2(-prev.x, -prev.y));
                const float2 a = __fmul2_rn(make_float2(100.f, 100.f), __fmul2_rn(t1, t1)), b = __fmul2_rn(t2, t2);
                acc = __fadd_rn(acc, __fadd_rn(a.x, b.x));
                late[i - 1] = __fadd_rn(a.y, b.y);   // term i + h (i + h > N: the padding lane, unused)
                prev = cur;
              }
#pragma unroll
              for (int i = h + 1; i <= N; ++i) acc = __fadd_rn(acc, late[i - h - 1]);
              const double out = -(double)acc;
              lp = isfinite(out) ? out : (double)-INFINITY;   // float32-typed result: sampler.py:128 leaves -inf
            } else {
              lp = tc_loglike<DD>(td, td_s, y);
            }
            ncall = 1;
            accept = isfinite(lp) && (lp > p.loglstar);
          }
        } else {
          lp = tc_loglike<DD>(td, td_s, y);
          ncall = 1;
          logp_prop = tc_prior<DD>(td, td_s, y);
          double lr = (double)__fsub_rn(ld_prop, ld_cur) + (lp - logl_cur) + (logp_prop - logp_cur);
          double ratio = exp(lr);
          if (ratio > 1.0) ratio = 1.0;
          accept = (double)u01 < ratio;
        }
        if (accept) {
          ld_cur = ld_prop;
          logl_cur = lp;
          logp_cur = logp_prop;
        }
        if (NPART > 1) *flag = accept ? 1 : 0;
        if (p.trace_z) p.trace_logl[(size_t)s * ns + (size_t)c] = logl_cur;
      } else if (NPART > 1 && active && more && philox) {
        gen_normals(0, jc, 1, step_abs + 1u, s);
      }
      __syncwarp();
      NNB_TSTAMP(7);
      acc_chain = accept;
      if (p.coop) {   // the tile barrier doubles as the count of the tile's accepted proposals
        tile_cnt = tc::named_bar_popc(t.bar_id, t.bar_threads, accept);
        if (NPART > 1) acc_chain = active && (*flag != 0);
      } else if (NPART > 1) {
        tile_sync(t);
        acc_chain = active && (*flag != 0);
      }
      NNB_TSTAMP(8);
      // ---- state / trace update, dims dealt to the chain's threads (sampler.py:433-444) -------------------------------
      if (active && kZcur) {
        // z' is recomputed from the same operands as the proposal (bit-identical); this step's noise is still intact
        // because the next step's is drawn after this point
        float* px = p.x + (size_t)c;
        if (acc_chain) {
          if (fused) {   // the flow left z' in nz: the accepted point becomes the current one by a swap of the two pointers
            float* tmp = zp;
            zp = nz;
            nz = tmp;
          } else {
            batched<kCh>(d, [&](int i) { return __fadd_rn(zp[i * 128], __fmul_rn(nz[i * 128], scale_f)); },
                         [&](int i, float v) { zp[i * 128] = v; });
          }
          if (defer_x) moved = true;
          else batched<kCh>(d, [&](int i) { return y[i * 128]; }, [&](int i, float v) { px[(size_t)i * ns] = v; });
        }
        if (p.trace_z) {
          float* tz = p.trace_z + (size_t)s * d * ns + (size_t)c;
          float* tx = p.trace_x + (size_t)s * d * ns + (size_t)c;
          batched<kCh>(d, [&](int i) { return zp[i * 128]; }, [&](int i, float v) { tz[(size_t)i * ns] = v; });
          batched<kCh>(d, [&](int i) { return acc_chain ? y[i * 128] : px[(size_t)i * ns]; },
                      [&](int i, float v) { tx[(size_t)i * ns] = v; });
        }
      } else if (active) {
        float* pz = p.z + (size_t)c + (size_t)part * ns;
        float* px = p.x + (size_t)c + (size_t)part * ns;
        if (acc_chain) {
          for (int i = part; i < d; i += NPART, pz += NPART * ns, px += NPART * ns) {
            *pz = zp[i * 128];
            *px = y[i * 128];
          }
        }
        if (p.trace_z) {
          float* tz = p.trace_z + (size_t)s * d * ns + (size_t)c + (size_t)part * ns;
          float* tx = p.trace_x + (size_t)s * d * ns + (size_t)c + (size_t)part * ns;
          if (acc_chain) {
            for (int i = part; i < d; i += NPART, tz += NPART * ns, tx += NPART * ns) {
              *tz = zp[i * 128];
              *tx = y[i * 128];
            }
          } else {
            pz = p.z + (size_t)c + (size_t)part * ns;
            px = p.x + (size_t)c + (size_t)part * ns;
            for (int i = part; i < d; i += NPART, tz += NPART * ns, tx += NPART * ns, pz += NPART * ns, px += NPART * ns) {
              *tz = *pz;
              *tx = *px;
            }
          }
        }
      }
    }
    if (x_pass) break;
    acc_total += accept ? 1u : 0u;
    ncall_total += ncall;
    NNB_TSTAMP(2);

    // ---- global accept count of the step -> scale adaptation (sampler.py:418-430) ------------------------------------
    const int si = s - p.s0 - 1;
    bool cta_poller = false;
    if (p.coop) {
      // Tiles rendezvous inside the CTA through shared-memory atomics (no CTA-wide barrier: the tiles of an SM drift apart
      // freely inside a step); the LAST tile of the CTA to finish the step carries the CTA's count to the grid barrier
      // (all CTAs are co-resident: cooperative launch) and becomes the CTA's poller for this step.  step_counts[si] was
      // zeroed by the host: CTA arrivals and the accept count travel in one 64-bit reduction (grid_arrive / grid_wait).
      if (tile_active && tit == 0) {
        if (tile_cnt) atomicAdd(&co_words[2], tile_cnt);
        __threadfence_block();
        if (atomicAdd(&co_words[1], 1u) == (unsigned int)(my_tiles - 1)) {
          co_words[1] = 0u;
          const unsigned int blk = atomicExch(&co_words[2], 0u);
          grid_arrive(&p.step_counts[si], blk);
          cta_poller = true;
        }
      }
    } else if (p.dynamic) {
      unsigned int blk = block_count(accept);
      if (threadIdx.x == 0) {
        if (blk) atomicAdd(&p.ctrl->step_acc, blk);
        __threadfence();
        unsigned int tk = atomicAdd(&p.ctrl->ticket, 1u);
        if (tk == gridDim.x - 1) {
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
    // ---- rest of the next step's noise (overlaps the grid barrier) --------------------------------------------------------
    if (tile_active && active && more && philox) gen_normals(jc + part, nj, NPART, step_abs + 1u, s);
    if (tile_active && active && more && philox_u && part == NPART - 1) gen_uniform(step_abs + 1u, s);
    NNB_TSTAMP(3);
    if (p.coop && tile_active && tit == 0) {
      // The CTA's poller waits for the grid-wide count and updates the CTA's copy of (scale, accept, reject) -- identical
      // in every CTA; the other tile leaders wait for the epoch word in shared memory.  The tile barrier at the top of the
      // next step publishes the new scale to the tile's threads.
      volatile unsigned int* vw = co_words;
      if (cta_poller) {
        const unsigned int na = grid_wait(&p.step_counts[si], gridDim.x);
        if (p.dynamic) {
          int a = (int)vw[4], r = (int)vw[5];
          double sc = *reinterpret_cast<volatile double*>(co_words + 6);
          if (2ull * na > (unsigned long long)n) a += 1; else r += 1;
          if (a > r) sc *= exp(1.0 / (1 + a));
          if (a < r) sc /= exp(1.0 / (1 + r));
          vw[4] = (unsigned int)a;
          vw[5] = (unsigned int)r;
          *reinterpret_cast<volatile double*>(co_words + 6) = sc;
          *reinterpret_cast<volatile float*>(co_scale_s) = (float)sc;
        }
        __threadfence_block();
        vw[3] = (unsigned int)(si + 1);
        tc::mbar_arrive(sbar);                          // completes phase si of the hand-off barrier
      } else {
        // the other tile leaders sleep on the mbarrier (hardware-suspended try_wait) instead of spinning on the epoch
        // word: the spin loop was 6.7 % of all issued instructions (profiles/r2_tc1_*)
#ifdef NNB_TC_WAIT_HINT
        tc::mbar_wait_long(sbar, (uint32_t)(si & 1));
#else
        tc::mbar_wait(sbar, (uint32_t)(si & 1));
#endif
      }
      NNB_TSTAMP(4);
    }
  }
  if (kZcur && active)
    for (int i = 0; i < d; ++i) p.z[(size_t)c + (size_t)i * ns] = zp[i * 128];
  if (active && part == 0) {
    p.logdet[c] = ld_cur;
    p.logl[c] = logl_cur;
    p.logp[c] = logp_cur;
  }
  __syncthreads();
  if (p.coop && blockIdx.x == 0 && threadIdx.x == 0) {   // publish the final scale bookkeeping
    p.ctrl->scale = *reinterpret_cast<volatile double*>(co_words + 6);
    p.ctrl->accept = (int)co_words[4];
    p.ctrl->reject = (int)co_words[5];
  }
  // totals: one atomic per warp (the counts of non-zero lanes only)
  unsigned int ta = __reduce_add_sync(0xffffffffu, acc_total);
  unsigned int tcall = __reduce_add_sync(0xffffffffu, ncall_total);
  if ((threadIdx.x & 31) == 0) {
    if (ta) atomicAdd(&p.ctrl->naccept, (unsigned long long)ta);
    if (tcall) atomicAdd(&p.ctrl->ncall, (unsigned long long)tcall);
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(*tmem_base_s, tmem_cols);
}

#ifndef __CUDACC_RTC__
__host__ inline size_t tc_smem_bytes(const TcFlowDesc& f, int tdoubles, int ntiles, int npart) {
  return (size_t)f.total_floats * 4 + (size_t)tdoubles * 8 + 3 * (size_t)ntiles * f.d * 128 * 4 +
         (size_t)ntiles * (npart + 1) * 128 * 4 + (size_t)ntiles * 128 * 4 + 2 * kTcMaxTiles * 8 + 8 + 32 * 4 +
         NNB_MAX_BLOCKS * 8 + 8;
}
#endif

}  // namespace nnb
