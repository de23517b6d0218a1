// Blackwell tensor-core plumbing shared by the tcgen05 kernels of this library (hamming_mma.cu: int8 Hamming and bf16 L2
// matchers; score_mma.cuh: bf16-split RANSAC scoring): mbarriers, bulk copies (TMA engine), tcgen05.mma / commit / ld, and the
// shared-memory matrix descriptor of the canonical K-major no-swizzle layout (8-row x 16-byte core matrices).
#pragma once
#include <stdint.h>

namespace sos_tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait suspends the thread in hardware; the spin bound only turns a lost arrival (a bug) into a trap instead of a hang
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done && spin > (1u << 20)) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// One lane of a CONVERGED warp (elect.sync).  Code that issues tcgen05.mma / cp.async.bulk from `if (lane == 0)` is compiled
// as divergent code: every instruction with uniform-register operands (UTCHMMA, UBLKCP, UTCBAR) gets wrapped in an
// elect + broadcast loop of ~13 instructions, which made the issuing thread — not the tensor pipe — the bound (83 cycles per
// 64-cycle MMA, measured with clock64 stamps).  With the whole warp running the loop and only the instruction itself
// predicated on the elected lane the operands are warp-uniform by construction.
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{ .reg .pred p; elect.sync _|p, 0xFFFFFFFF; selp.u32 %0, 1, 0, p; }" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], M128 N128, 32 bytes of K per instruction:
//   KIND_HAMMING: int8 x int8 -> int32 (K32);   KIND_L2, KIND_L2F: bf16 x bf16 -> float32 (K16)
constexpr int KIND_HAMMING = 0, KIND_L2 = 1, KIND_L2F = 2;
template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if (KIND == KIND_HAMMING)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// shared-memory matrix descriptor: K-major, no swizzle; core matrices 128 bytes apart along K (LBO) and `sbo_bytes` apart
// along M/N (SBO); bits [46,48) = 1 (Blackwell descriptor version)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t sbo_bytes) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         ((uint64_t)1 << 46);
}
// 32 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, int (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// tcgen05.wait::ld with the destination registers as in/out operands: ties every later use of v[] to the wait, so neither
// the compiler nor ptxas can schedule a consumer above it (the load itself returns before the registers are written)
__device__ __forceinline__ void tmem_ld_wait(int (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                 "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]),
                 "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]),
                 "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :
               : "memory");
}


}  // namespace sos_tc
