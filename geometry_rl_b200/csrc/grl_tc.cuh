// tcgen05 / TMEM / mbarrier building blocks (sm_100a inline PTX) for the bf16 tensor-core path.
//
// Operand staging convention used by every tensor-core kernel in this library (no TMA, no swizzle: the A
// operands are PRODUCED by threads — gathered rows, LayerNorm / GELU outputs — so they are written straight
// into the layout the MMA reads):
//   a K-major operand tile [R rows][K elements] of bf16 lives in shared memory as [K/8 chunks][R rows][8 bf16]
//   i.e. 16-byte "core rows", 8 consecutive rows = one 128-byte core matrix,
//        SBO (stride between 8-row groups)        = 128 B
//        LBO (stride between the 16-byte K chunks) = R * 16 B
//   One tcgen05.mma (kind::f16) consumes K = 16 (two chunks); the k-th step starts at base + k * 2 * LBO.
// Accumulators: M = 128 rows <-> the 128 TMEM lanes, one fp32 column per output column.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace grl {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}

// ---- 1-D bulk async copies (TMA engine, no tensor map): global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// dst, src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- tensor-map TMA (cp.async.bulk.tensor, SASS UTMALDG): one box global -> shared, bytes counted on an mbarrier -------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

// ---- proxy / tcgen05 fences ---------------------------------------------------------------------
// generic-proxy st.shared -> visible to the async proxy (the tensor core reads operands through it)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM allocation (one full warp executes these) -----------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- descriptors ------------------------------------------------------------------------------------
// shared-memory matrix descriptor, no swizzle, K-major (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (Blackwell)
  return d;                // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// instruction descriptor: D fp32, A/B bf16, both K-major, dense (cute::UMMA::InstrDescriptor bit layout)
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kind::f16 takes fp16 or bf16 per operand (format bits 7-9 for A, 10-12 for B: 0 = fp16, 1 = bf16)
__host__ __device__ constexpr uint32_t idesc_f16_ex(int M, int N, int a_mn, int b_mn, int a_bf16, int b_bf16) {
  return (1u << 4) | ((uint32_t)a_bf16 << 7) | ((uint32_t)b_bf16 << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMA issue (ONE thread) ----------------------------------------------------------------------------
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread -> one arrival on `bar` when they have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// D[128 x N] (+)= A[128 x K] * B[N x K]^T, operands in the chunked layout described at the top.
// a_rows / b_rows = number of rows of the staged A / B tiles (LBO = rows * 16 B).
template <int N, int K>
__device__ __forceinline__ void issue_gemm(uint32_t tmem_d, uint32_t a_saddr, int a_rows, uint32_t b_saddr, int b_rows,
                                           bool accumulate_first) {
  constexpr uint32_t idesc = idesc_bf16(128, N);
#pragma unroll
  for (int k = 0; k < K / 16; ++k) {
    const uint64_t da = smem_desc(a_saddr + k * 2 * a_rows * 16, a_rows * 16, 128);
    const uint64_t db = smem_desc(b_saddr + k * 2 * b_rows * 16, b_rows * 16, 128);
    mma_bf16(tmem_d, da, db, idesc, (k > 0 || accumulate_first) ? 1u : 0u);
  }
}

// Operand view for the generic issue loop: start address + (LBO, SBO, byte advance per K = 16 step).
//   K-major  view of a [rows][cols] image (M/N = rows, K = cols): lbo = rows*16, sbo = 128,     adv = 2*rows*16
//   MN-major view of the same image       (K = rows, M/N = cols): lbo = 128,     sbo = rows*16, adv = 256
struct OpView {
  uint32_t addr, lbo, sbo, adv;
};
__device__ __forceinline__ OpView view_k(uint32_t addr, int rows) { return OpView{addr, (uint32_t)rows * 16u, 128u, (uint32_t)rows * 32u}; }
__device__ __forceinline__ OpView view_mn(uint32_t addr, int rows) { return OpView{addr, 128u, (uint32_t)rows * 16u, 256u}; }
__host__ __device__ constexpr uint32_t idesc_bf16_ex(int M, int N, int a_mn, int b_mn) {
  return idesc_bf16(M, N) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16);
}
// ---- cheap MMA issue: descriptor halves precomputed once, K steps fully unrolled -----------------------------------
// The generic loop above rebuilds both 64-bit descriptors for every K = 16 step (~30 uniform-datapath instructions per
// UTCHMMA, all dependent): at 80+ MMAs per 128-row tile the ISSUING THREAD, not the tensor pipe, bounds the kernel.
// Only the 14-bit start-address field changes between the K steps of one operand view, so a view is kept as the two
// descriptor words of its first step plus the per-step increment (in 16-byte units) and each further step costs one add.
struct Op {
  uint32_t lo, hi, step;
};
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
__device__ __forceinline__ Op op_k(uint32_t addr, int rows) { return Op{desc_lo(addr, (uint32_t)rows * 16u), desc_hi(128u), (uint32_t)rows * 2u}; }
__device__ __forceinline__ Op op_mn(uint32_t addr, int rows) { return Op{desc_lo(addr, 128u), desc_hi((uint32_t)rows * 16u), 16u}; }
__device__ __forceinline__ void mma_f16_words(uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
template <int KSTEPS>
__device__ __forceinline__ void issue_mma_fast(uint32_t tmem_d, const Op& a, const Op& b, uint32_t idesc, bool accumulate_first) {
  mma_f16_words(tmem_d, a.lo, a.hi, b.lo, b.hi, idesc, accumulate_first ? 1u : 0u);
#pragma unroll
  for (int k = 1; k < KSTEPS; ++k) mma_f16_words(tmem_d, a.lo + k * a.step, a.hi, b.lo + k * b.step, b.hi, idesc, 1u);
}
// A operand from TENSOR MEMORY (TS mode): row m of A sits in TMEM lane m, its K elements packed two 16-bit values per
// 32-bit column (element 2 j in the low half of column j); one MMA consumes K = 16 = 8 columns.  An epilogue thread
// that owns row m therefore feeds the next GEMM with tcgen05.st of the packed pairs it already holds - no shared-memory
// image, no fence.proxy.async, and the MMA does not re-read a 4 KB A tile from shared memory per K step.
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t blo, uint32_t bhi, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D (+)= A_tmem[128 x 16 ksteps] * B^T: A at columns tmem_a, tmem_a + 8, ...; B as an operand view in shared memory
__device__ __forceinline__ void issue_mma_ts(uint32_t tmem_d, uint32_t tmem_a, const OpView& b, uint32_t idesc, int ksteps,
                                             bool accumulate_first) {
  const uint32_t blo = desc_lo(b.addr, b.lbo), bhi = desc_hi(b.sbo), bs = b.adv >> 4;
#pragma unroll
  for (int k = 0; k < ksteps; ++k)
    mma_f16_ts(tmem_d, tmem_a + 8u * k, blo + k * bs, bhi, idesc, (k > 0 || accumulate_first) ? 1u : 0u);
}

// generic entry used by every kernel: the operand views' descriptor words are formed once, each K step adds a constant;
// ksteps is a compile-time constant at every call site, so the loop unrolls into back-to-back UTCHMMA.
__device__ __forceinline__ void issue_mma(uint32_t tmem_d, const OpView& a, const OpView& b, uint32_t idesc, int ksteps,
                                          bool accumulate_first) {
  const uint32_t alo = desc_lo(a.addr, a.lbo), ahi = desc_hi(a.sbo), blo = desc_lo(b.addr, b.lbo), bhi = desc_hi(b.sbo);
  const uint32_t as = a.adv >> 4, bs = b.adv >> 4;
#pragma unroll
  for (int k = 0; k < ksteps; ++k)
    mma_f16_words(tmem_d, alo + k * as, ahi, blo + k * bs, bhi, idesc, (k > 0 || accumulate_first) ? 1u : 0u);
}
// the same with the K loop kept rolled (two adds + one UTCHMMA per step): for kernels whose issuing thread is short of registers
__device__ __forceinline__ void issue_mma_rolled(uint32_t tmem_d, const OpView& a, const OpView& b, uint32_t idesc, int ksteps,
                                                 bool accumulate_first) {
  uint32_t alo = desc_lo(a.addr, a.lbo), blo = desc_lo(b.addr, b.lbo);
  const uint32_t ahi = desc_hi(a.sbo), bhi = desc_hi(b.sbo), as = a.adv >> 4, bs = b.adv >> 4;
  mma_f16_words(tmem_d, alo, ahi, blo, bhi, idesc, accumulate_first ? 1u : 0u);
#pragma unroll 1
  for (int k = 1; k < ksteps; ++k) {
    alo += as;
    blo += bs;
    mma_f16_words(tmem_d, alo, ahi, blo, bhi, idesc, 1u);
  }
}
// one elected lane of a converged warp (the MMA-issue warp runs its loop warp-uniformly and issues under this predicate)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// Sum over the 32 lanes of a warp of NV per-lane values by recursive halving: NV - 2 + ... shuffles instead of
// 5 * NV.  On return lane l holds in v[0 .. NV/32) the totals of the ORIGINAL indices  i = l * (NV/32) + j
// (NV must be a multiple of 32).  Fixed exchange pattern -> deterministic summation order.
template <int NV>
__device__ __forceinline__ void warp_colsum(float (&v)[NV], int lane) {
  static_assert(NV % 32 == 0, "NV must be a multiple of 32");
#pragma unroll
  for (int step = 0; step < 5; ++step) {
    const int half = NV >> (step + 1);       // values kept after this step
    const int bit = 16 >> step;              // partner = lane ^ bit
    const bool upper = (lane & bit) != 0;    // upper lanes keep the upper half of the current range
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = upper ? v[i + half] : v[i];
      const float send = upper ? v[i] : v[i + half];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
  }
}

// ---- TMEM -> registers: 32 lanes x 32b, 16 consecutive columns per thread ---------------------------------
// taddr = (lane_base << 16) | column; lane_base must be 32 * (warp_id % 4).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- registers -> TMEM: 32 lanes x 32b, 16 consecutive columns per thread (SASS STTM); same addressing as tmem_ld16 ------
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16_raw(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// one arrival (release) on an mbarrier of this CTA
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- L2 prefetch of a contiguous global range (bytes: multiple of 16) issued by ONE thread -----------------------
// Pulls a tile that will be read a few microseconds later (by LDG or cp.async) into L2, so that the later access pays
// an L2 hit instead of a DRAM round trip; no shared memory or registers are tied up while the data is in flight.
__device__ __forceinline__ void prefetch_l2(const void* gptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}

// ---- named barrier for a sub-group of the CTA (id 1..15, `count` threads, multiple of 32) -----------------------
__device__ __forceinline__ void group_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// ---- packed fp16 GELU (tanh form) for the activation epilogues ------------------------------------------------
// The epilogues are issue-bound on the activation; HFMA2 / MUFU.TANH.F16 evaluate two elements per instruction and
// the result is an fp16 MMA operand anyway (11-bit mantissa: finer than the bf16 operands of the other contractions).
__device__ __forceinline__ __half2 tanh_h2(__half2 x) {
  uint32_t r;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(r) : "r"(*reinterpret_cast<uint32_t*>(&x)));
  return *reinterpret_cast<__half2*>(&r);
}
__device__ __forceinline__ __half2 gelu_h2(__half2 x) {
  const __half2 k = __floats2half2_rn(0.7978845608028654f, 0.7978845608028654f);
  const __half2 kc = __floats2half2_rn(0.7978845608028654f * 0.044715f, 0.7978845608028654f * 0.044715f);
  const __half2 half = __floats2half2_rn(0.5f, 0.5f);
  const __half2 t = tanh_h2(__hmul2(x, __hfma2(__hmul2(x, x), kc, k)));
  const __half2 hx = __hmul2(x, half);
  return __hfma2(hx, t, hx);
}
// value and derivative with e = 0.5 (1 + t):  y = x e,  dy = e + x (1 - t^2) (k / 2 + 3 kc / 2 x^2)   (10 fma-pipe ops + 1 MUFU)
// x^2 overflows fp16 for |x| > 256; there t = +-1 and the first factor of the derivative term is 0, so its second factor
// takes min(x^2, 1024) (the exact x^2 below |x| = 32, where t is not yet +-1): 0 * inf would make dy NaN instead of e.
__device__ __forceinline__ void gelu_h2(__half2 x, __half2& y, __half2& dy) {
  const __half2 k = __floats2half2_rn(0.7978845608028654f, 0.7978845608028654f);
  const __half2 kc = __floats2half2_rn(0.7978845608028654f * 0.044715f, 0.7978845608028654f * 0.044715f);
  const __half2 kh = __floats2half2_rn(0.5f * 0.7978845608028654f, 0.5f * 0.7978845608028654f);
  const __half2 k3h = __floats2half2_rn(1.5f * 0.7978845608028654f * 0.044715f, 1.5f * 0.7978845608028654f * 0.044715f);
  const __half2 half = __floats2half2_rn(0.5f, 0.5f), one = __floats2half2_rn(1.0f, 1.0f);
  const __half2 x2max = __floats2half2_rn(1024.0f, 1024.0f);
  const __half2 x2 = __hmul2(x, x);
  const __half2 t = tanh_h2(__hmul2(x, __hfma2(x2, kc, k)));
  const __half2 e = __hfma2(t, half, half);
  y = __hmul2(x, e);
  dy = __hfma2(__hmul2(x, __hfma2(__hneg2(t), t, one)), __hfma2(__hmin2(x2, x2max), k3h, kh), e);
}
__device__ __forceinline__ uint4 pack_h8(const __half2 (&h)[4]) {
  uint4 o;
  o.x = *reinterpret_cast<const uint32_t*>(&h[0]);
  o.y = *reinterpret_cast<const uint32_t*>(&h[1]);
  o.z = *reinterpret_cast<const uint32_t*>(&h[2]);
  o.w = *reinterpret_cast<const uint32_t*>(&h[3]);
  return o;
}

// ---- operand staging helpers -----------------------------------------------------------------------------
// address (in bf16 elements) of element (row, k) of a tile with `rows` rows in the chunked layout
__device__ __forceinline__ int op_index(int rows, int row, int k) { return ((k >> 3) * rows + row) * 8 + (k & 7); }

// pack 8 floats into 8 bf16 (16 bytes)
__device__ __forceinline__ uint4 pack8(const float* v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]);
  __nv_bfloat162 d = __floats2bfloat162_rn(v[6], v[7]);
  uint4 o;
  o.x = *reinterpret_cast<uint32_t*>(&a);
  o.y = *reinterpret_cast<uint32_t*>(&b);
  o.z = *reinterpret_cast<uint32_t*>(&c);
  o.w = *reinterpret_cast<uint32_t*>(&d);
  return o;
}

// pack 8 floats into 8 fp16 (16 bytes)
__device__ __forceinline__ uint4 pack8_h(const float* v) {
  const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
  const __half2 c = __floats2half2_rn(v[4], v[5]), d = __floats2half2_rn(v[6], v[7]);
  uint4 o;
  o.x = *reinterpret_cast<const uint32_t*>(&a);
  o.y = *reinterpret_cast<const uint32_t*>(&b);
  o.z = *reinterpret_cast<const uint32_t*>(&c);
  o.w = *reinterpret_cast<const uint32_t*>(&d);
  return o;
}

// Gradient scale for fp16 gradient operands: gradients are multiplied by a power of two chosen from the tensor's
// absolute maximum (grl_absmax) so that max |g * scale| lies in [32, 64): every element within 2^-20 of the maximum
// keeps fp16's 11-bit mantissa (bf16 keeps 8), products stay far below 65504, and the power of two is removed
// exactly in the epilogues.  amax_bits = bit pattern of the (non-negative) maximum; 0 / inf / nan -> scale 1.
__device__ __forceinline__ float grad_scale_from_amax(uint32_t amax_bits) {
  const int e = (int)((amax_bits >> 23) & 0xFFu);      // biased exponent: amax in [2^(e-127), 2^(e-126))
  if (e == 0 || e == 255) return 1.0f;
  int k = 127 + 5 - (e - 127);                         // scale = 2^(5 - (e - 127))  ->  amax * scale in [32, 64)
  k = k < 1 ? 1 : (k > 254 ? 254 : k);
  return __uint_as_float((uint32_t)k << 23);
}

// Stage a [rows][K] fp32 row-major GLOBAL matrix (weights) as a bf16 operand tile. Whole CTA cooperates.
__device__ __forceinline__ void stage_weight_bf16(__nv_bfloat16* dst, const float* __restrict__ src, int rows, int K, int ld) {
  const int n_chunks = rows * (K >> 3);
  for (int i = threadIdx.x; i < n_chunks; i += blockDim.x) {
    const int row = i % rows, kc = i / rows;
    const float4 lo = __ldg(reinterpret_cast<const float4*>(src + (size_t)row * ld + kc * 8));
    const float4 hi = __ldg(reinterpret_cast<const float4*>(src + (size_t)row * ld + kc * 8 + 4));
    const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    *reinterpret_cast<uint4*>(dst + ((size_t)kc * rows + row) * 8) = pack8(v);
  }
}

// fp16 variant of stage_weight_bf16 (same [K/8][rows][8] image)
__device__ __forceinline__ void stage_weight_f16(__half* dst, const float* __restrict__ src, int rows, int K, int ld) {
  const int n_chunks = rows * (K >> 3);
  for (int i = threadIdx.x; i < n_chunks; i += blockDim.x) {
    const int row = i % rows, kc = i / rows;
    const float4 lo = __ldg(reinterpret_cast<const float4*>(src + (size_t)row * ld + kc * 8));
    const float4 hi = __ldg(reinterpret_cast<const float4*>(src + (size_t)row * ld + kc * 8 + 4));
    const __half2 h[4] = {__floats2half2_rn(lo.x, lo.y), __floats2half2_rn(lo.z, lo.w), __floats2half2_rn(hi.x, hi.y),
                          __floats2half2_rn(hi.z, hi.w)};
    *reinterpret_cast<uint4*>(dst + ((size_t)kc * rows + row) * 8) = pack_h8(h);
  }
}

}  // namespace tc
}  // namespace grl
