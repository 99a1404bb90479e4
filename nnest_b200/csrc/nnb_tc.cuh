// nnb_tc.cuh -- tcgen05 / TMEM primitives (sm_100a inline PTX) used by the tensor-core MLP path.
//
// Conventions used throughout (cta_group::1, M = 128, kind::tf32, FP32 accumulate in TMEM):
//   * one warpgroup (4 warps, 128 threads) owns one tile of 128 chains; thread t of the warpgroup owns
//     TMEM lane t, so a chain's row of A / D is read and written by the chain's own thread with the
//     32x32b tcgen05.ld / tcgen05.st shapes (warp w of the warpgroup addresses lanes 32w..32w+31);
//   * A operands (activations) live in TMEM: A[m][k] = lane m, column a_col + k (32-bit per tf32);
//   * B operands (weights, nn.Linear (out,in) = N x K, "K-major") live in shared memory in the canonical
//     no-swizzle core-matrix layout: element (n, k) of one K=8 step at byte
//         (kb * nN + nb) * 128 + r * 16 + e * 4,   n = 8 nb + r, k = 4 kb + e, nN = N / 8
//     i.e. LBO (K direction) = nN * 128 B, SBO (N direction) = 128 B; successive K steps are 2*nN*128 B apart;
//   * FP32 parity: every product is evaluated as 3xTF32 (a_hi*b_hi + a_lo*b_hi + a_hi*b_lo).
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#endif

namespace nnb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- TMEM allocation (one warp, power-of-two columns >= 32) --------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- mbarrier ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "NNB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra NNB_DONE;\n"
      "bra NNB_WAIT;\n"
      "NNB_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// Long waits (the per-step hand-off of the scale): try_wait with a suspend-time hint.  Without the hint the instruction
// returns after a few cycles and the loop is a busy spin -- 2.7 % of ALL executed instructions were this TRYWAIT and
// another 5.4 % its branch / yield (profiles/r2_final_mcmc_tc_kernel: SASS page), issued by the tile leaders, which all
// sit on scheduler 0.  With the hint the warp is suspended until the phase completes (or the time runs out).
__device__ __forceinline__ void mbar_wait_long(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "NNB_WAITL:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra NNB_DONEL;\n"
      "bra NNB_WAITL;\n"
      "NNB_DONEL:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(0x989680u)
      : "memory");
}
// ---- TMA bulk copy global -> shared (cp.async.bulk, SASS: UBLKCP), completion counted in bytes on an mbarrier -------
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bytes: multiple of 16; dst / src 16-byte aligned.  Issued by ONE thread.
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_global, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(__cvta_generic_to_global(src_global)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// arrive on `bar` when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// named barrier + population count of `pred` over the participating threads (every participant gets the count)
__device__ __forceinline__ uint32_t named_bar_popc(uint32_t id, uint32_t nthreads, bool pred) {
  uint32_t r;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.u32 p, %3, 0;\n"
      "bar.red.popc.u32 %0, %1, %2, p;\n"
      "}\n"
      : "=r"(r)
      : "r"(id), "r"(nthreads), "r"((uint32_t)pred)
      : "memory");
  return r;
}

// exactly one lane of the (converged) warp gets true.  ptxas knows that the guarded region runs on a single thread, so
// register operands of the tcgen05 instructions inside move to uniform registers without a per-operand waterfall loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- descriptors ------------------------------------------------------------------------------------------
// instruction descriptor: D f32, A/B tf32, both K-major, M = 128, N = n (cute::UMMA::InstrDescriptor bit layout)
__host__ __device__ inline uint32_t idesc_tf32_m128(uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
// shared-memory matrix descriptor, no swizzle, K-major (cute::UMMA::SmemDescriptor bit layout, version 1)
__device__ __forceinline__ uint64_t smem_desc_kmajor(uint32_t smem_byte_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_byte_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// D[tmem] (+)= A[tmem] * B[smem]^T for one K = 8 step.  Issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 3xTF32 product over `ksteps` K=8 steps: D (+)= A_hi*B_hi + A_lo*B_hi + A_hi*B_lo.
//   a_hi / a_lo: TMEM addresses of the hi / lo activations (column of k = 0)
//   b_hi / b_lo: shared-memory byte addresses of the packed weights (k step 0); nN = N / 8
// n: N of the instruction; nN_packed: n-blocks per K chunk in the packed buffer (== n / 8 unless a wider packed
// matrix is issued in column slices)
__device__ __forceinline__ void mma_3xtf32_n(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                             int ksteps, uint32_t n, uint32_t nN_packed, bool accumulate_first) {
  const uint32_t idesc = idesc_tf32_m128(n);
  // descriptor = hi word (SBO = 128 B, version 1) : lo word (start address >> 4 | LBO >> 4 << 16); a K step moves
  // the start address by 2 * nN * 128 B
  const uint64_t desc_hi = ((uint64_t)((128u >> 4) | (1u << 14))) << 32;
  const uint32_t lbo_field = ((nN_packed * 128u) >> 4) << 16;
  uint32_t lo_h = ((b_hi & 0x3FFFFu) >> 4) | lbo_field;
  uint32_t lo_l = ((b_lo & 0x3FFFFu) >> 4) | lbo_field;
  const uint32_t kstep = (2u * nN_packed * 128u) >> 4;
  uint32_t acc = accumulate_first ? 1u : 0u;
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint64_t dh = desc_hi | lo_h, dl = desc_hi | lo_l;
    mma_tf32_ts(d_tmem, a_lo, dh, idesc, acc);   // small terms first
    mma_tf32_ts(d_tmem, a_hi, dl, idesc, 1u);
    mma_tf32_ts(d_tmem, a_hi, dh, idesc, 1u);
    acc = 1u;
    lo_h += kstep; lo_l += kstep; a_hi += 8u; a_lo += 8u;
  }
}
__device__ __forceinline__ void mma_3xtf32(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                           int ksteps, uint32_t n, bool accumulate_first) {
  mma_3xtf32_n(d_tmem, a_hi, a_lo, b_hi, b_lo, ksteps, n, n >> 3, accumulate_first);
}

// ---- TMEM <-> registers, 32x32b (thread = lane), 8 columns at a time -------------------------------------------
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]),
        "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]),
        "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
          taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}

// hi = x truncated to tf32 (low 13 mantissa bits cleared), lo = x - hi (exact in fp32; |lo| < 2^-10 |x|, and the
// tensor core reads its top 19 bits: a relative error below 2^-20 of x).  2 ALU instructions per element.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
// the same split of N values, the subtractions as packed FP32 pairs (FADD2 rounds each lane like FADD: the same bits)
template <int N>
__device__ __forceinline__ void split_tf32(const float* x, uint32_t* hi, uint32_t* lo) {
#pragma unroll
  for (int j = 0; j + 1 < N; j += 2) {
    hi[j] = __float_as_uint(x[j]) & 0xffffe000u;
    hi[j + 1] = __float_as_uint(x[j + 1]) & 0xffffe000u;
    const float2 l = __fadd2_rn(make_float2(x[j], x[j + 1]), make_float2(-__uint_as_float(hi[j]), -__uint_as_float(hi[j + 1])));
    lo[j] = __float_as_uint(l.x);
    lo[j + 1] = __float_as_uint(l.y);
  }
  if (N & 1) split_tf32(x[N - 1], hi[N - 1], lo[N - 1]);
}

// host mirror of cvt.rna.tf32.f32 (round half away from zero on the magnitude), used to pre-split weights
inline float host_rna_tf32(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return x;
  u = (u + 0x1000u) & 0xffffe000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

// host: pack W (N x K row-major, nn.Linear (out, in)) into the canonical K-major no-swizzle layout for
// ksteps = Kpad/8 steps, zero padded to (Npad, Kpad).  dst has Npad*Kpad floats.
inline void host_pack_b(const float* W, int N, int K, int ldw, int Npad, int Kpad, float* dst_hi, float* dst_lo) {
  const int nN = Npad / 8;
  for (int n = 0; n < Npad; ++n)
    for (int k = 0; k < Kpad; ++k) {
      float w = (n < N && k < K) ? W[(size_t)n * ldw + k] : 0.f;
      float hi = host_rna_tf32(w);
      float lo = host_rna_tf32(w - hi);
      int ks = k / 8, kb = (k % 8) / 4, e = k % 4, nb = n / 8, r = n % 8;
      size_t off = (size_t)ks * (2 * nN * 32) + (size_t)(kb * nN + nb) * 32 + r * 4 + e;
      dst_hi[off] = hi;
      dst_lo[off] = lo;
    }
}

}  // namespace tc
}  // namespace nnb
