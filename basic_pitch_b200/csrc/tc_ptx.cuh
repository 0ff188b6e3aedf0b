// Inline-PTX helpers shared by the tcgen05 kernels (tc_conv.cu, cqt_tc.cu): mbarriers, bulk async copies (UBLKCP),
// UMMA shared-memory / instruction descriptors, tcgen05.mma / commit / fences, TMEM loads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace bp {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// raise the expected transaction count without arriving (the caller arrives later, after its own writes)
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// mbar_wait with a watchdog: after ~2 s of spinning it reports who waits on what and traps, so that a protocol error
// shows up as a launch failure with a message instead of a hung GPU.  `tag` identifies the wait site.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
static __device__ __noinline__ void mbar_deadlock(int tag, uint32_t parity) {
  if ((threadIdx.x & 31) == 0)
    printf("libbp_b200: mbarrier wait timed out: block %d warp %d site %d parity %u\n", (int)blockIdx.x, (int)(threadIdx.x >> 5),
           tag, parity);
  __trap();
}
#ifdef BP_MBAR_DEBUG
__device__ __forceinline__ void mbar_wait_wd(uint64_t* bar, uint32_t parity, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ffu) == 0 && clock64() - t0 > 4000000000ll) mbar_deadlock(tag, parity);
  }
}
#else
// Production form: the whole spin loop is one asm block (a C++ loop on the returned predicate makes the compiler treat the
// issuing warps' loop state as divergent, which takes the MMA loops off the uniform datapath: R2UR before every UTCHMMA),
// bounded by a spin count (each try_wait suspends for a hardware-defined time first) and ending in a trap.
// Build with -DBP_MBAR_DEBUG to get the message with the wait site instead.
__device__ __forceinline__ void mbar_wait_wd(uint64_t* bar, uint32_t parity, int /*tag*/) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      ".reg .u32 spins;\n\t"
      "mov.u32 spins, 0;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "add.u32 spins, spins, 1;\n\t"
      "setp.lt.u32 q, spins, 0x4000000;\n\t"
      "@q bra WAIT_LOOP;\n\t"
      "trap;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
#endif
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// expect_tx + bulk copy by the elected lane only (PTX predication): with warp-uniform operands the producer loop stays on
// the uniform datapath (no per-step R2UR / elect loop around UBLKCP)
__device__ __forceinline__ void bulk_g2s_expect_pred(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                                     uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %4, 0;\n\t"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%3], %2;\n\t"
      "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t"
      "}\n" ::"r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "r"(leader)
      : "memory");
}
// K-major, no-swizzle shared-memory matrix descriptor (SM100 "version 1"):
//   [0,14) start >> 4, [16,30) leading-dimension byte offset >> 4 (between the two 8-element k-chunks),
//   [32,46) stride byte offset >> 4 (between 8-row groups), [46,48) = 1, layout type [61,64) = 0.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}
// instruction descriptor, kind::f16: D = f32 (bit 4), A = B = bf16 (bits 7, 10), both K-major, N>>3 @17, M>>4 @24
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The three split-precision products of one program use, issued by the elected lane only (PTX predication, no
// branch): D (+)= Ahi*Bhi ; D += Ahi*Blo ; D += Alo*Bhi.  Descriptors are passed as (low word, shared high word).
__device__ __forceinline__ void umma_bf16_x3(uint32_t tmem_d, uint32_t a_hi_lo32, uint32_t a_lo_lo32, uint32_t b_hi_lo32,
                                             uint32_t b_lo_lo32, uint32_t desc_hi32, uint32_t idesc, uint32_t accumulate,
                                             uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q, t;\n\t"
      ".reg .b64 dah, dal, dbh, dbl;\n\t"
      "setp.ne.b32 p, %7, 0;\n\t"
      "setp.ne.b32 q, %8, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 dah, {%1, %5};\n\t"
      "mov.b64 dal, {%2, %5};\n\t"
      "mov.b64 dbh, {%3, %5};\n\t"
      "mov.b64 dbl, {%4, %5};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], dah, dbh, %6, p;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], dah, dbl, %6, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], dal, dbh, %6, t;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(a_hi_lo32), "r"(a_lo_lo32), "r"(b_hi_lo32), "r"(b_lo_lo32), "r"(desc_hi32), "r"(idesc), "r"(accumulate),
      "r"(leader)
      : "memory");
}
// Six products of a three-way split with the A operand in tensor memory (TS form): a_* are tensor-memory addresses (K = 16 ->
// 8 columns each), b_* descriptor low words.  D (+)= Ah*Bh ; += Ah*Bm ; += Am*Bh ; += Ah*Bl ; += Al*Bh ; += Am*Bm.
__device__ __forceinline__ void umma_ts_bf16_x6(uint32_t tmem_d, uint32_t a_h, uint32_t a_m, uint32_t a_l, uint32_t b_h,
                                                uint32_t b_m, uint32_t b_l, uint32_t desc_hi32, uint32_t idesc,
                                                uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q, t;\n\t"
      ".reg .b64 dbh, dbm, dbl;\n\t"
      "setp.ne.b32 p, %9, 0;\n\t"
      "setp.ne.b32 q, %10, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 dbh, {%4, %7};\n\t"
      "mov.b64 dbm, {%5, %7};\n\t"
      "mov.b64 dbl, {%6, %7};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], dbh, %8, p;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], dbm, %8, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%2], dbh, %8, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], dbl, %8, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%3], dbh, %8, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%2], dbm, %8, t;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(a_h), "r"(a_m), "r"(a_l), "r"(b_h), "r"(b_m), "r"(b_l), "r"(desc_hi32), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void umma_commit_pred(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Packed FP32 FMA (FFMA2): d.{x,y} += o * w.{x,y}.  One issue slot for two FMAs; with the scalar broadcast in a register and
// the weight pair in a uniform register (constant memory, static offset) the epilogue FMA streams need half the issue
// slots of scalar FFMAs — what the fused epilogues compete for with the MMA-issuing warps.
__device__ __forceinline__ void ffma2(float2& d, float o, float2 w) {
  unsigned long long dd, oo, ww;
  asm("mov.b64 %0, {%1, %2};" : "=l"(dd) : "f"(d.x), "f"(d.y));
  asm("mov.b64 %0, {%1, %1};" : "=l"(oo) : "f"(o));
  asm("mov.b64 %0, {%1, %2};" : "=l"(ww) : "f"(w.x), "f"(w.y));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(dd) : "l"(oo), "l"(ww));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(dd));
}

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}

// ---- A operand in tensor memory (tcgen05.mma "TS" form) -------------------------------------------------------------
// kind::f16, M = 128: row = TMEM lane, two 16-bit elements per 32-bit column (element 2c in the low half), so a K = 16 step
// reads 8 columns starting at the given column (measured with tools/ubench/umma_ts.cu, which also shows that the D
// operand of a small-N MMA may start at ANY column).  The three split-precision products, all accumulating:
//   D += Ahi*Bhi ; D += Ahi*Blo ; D += Alo*Bhi        (issued by the elected lane only)
__device__ __forceinline__ void umma_ts_bf16_x3(uint32_t tmem_d, uint32_t tmem_a_hi, uint32_t tmem_a_lo, uint32_t b_hi_lo32,
                                                uint32_t b_lo_lo32, uint32_t desc_hi32, uint32_t idesc, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q, t;\n\t"
      ".reg .b64 dbh, dbl;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 dbh, {%3, %5};\n\t"
      "mov.b64 dbl, {%4, %5};\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], dbh, %6, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], dbl, %6, t;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%2], dbh, %6, t;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a_hi), "r"(tmem_a_lo), "r"(b_hi_lo32), "r"(b_lo_lo32), "r"(desc_hi32), "r"(idesc), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tmem_ld2_nowait(uint32_t taddr, uint32_t (&v)[2]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
// zero `N` consecutive columns of the calling warp's 32 lanes (N = 8, 16 or 32)
template <int N>
__device__ __forceinline__ void tmem_zero(uint32_t taddr) {
  static_assert(N == 8 || N == 16 || N == 32, "tmem_zero");
  const uint32_t z = 0u;
  if constexpr (N == 8) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z) : "memory");
  } else if constexpr (N == 16) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr),
        "r"(z)
        : "memory");
  } else {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
        "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr),
        "r"(z)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

}  // namespace bp
