// Device helpers shared by the tensor-core kernels (sl_rx_ssb_tc.cu, sl_tx_ssb_tc.cu): mbarriers, bulk asynchronous copies,
// tcgen05 descriptors / MMA issue / TMEM loads. Included inside each translation unit's anonymous namespace.
#pragma once
__device__ __forceinline__ uint32_t smem_u32 (const void *p) { return (uint32_t) __cvta_generic_to_shared (p); }
__device__ __forceinline__ void mbar_init (uint64_t *bar, unsigned count)
{
  asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32 (bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx (uint64_t *bar, unsigned bytes)
{
  asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32 (bar)), "r"(bytes) : "memory");
}
#include "sl_stress.cuh"
__device__ __forceinline__ void mbar_arrive (uint64_t *bar)
{
  sl_jitter ();
  asm volatile ("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32 (bar)) : "memory");
}
// A plain try_wait loop polls every ~20 clocks, and every poll is a shared-memory wavefront on the L1 data pipe the tensor core
// fetches its operands through (ncu, round 2: 411 polls per supertile). Still, a suspend-time hint or a nanosleep back-off
// measured slower (profiles/r02_summary.md): plain polling 416 Gsamples/s, hint 2000 ns 412, sleep 64 ns 410, both 409 — the
// polls do not cost what their count suggests and the wake-up latency does.
__device__ __forceinline__ void mbar_wait (uint64_t *bar, unsigned parity)
{
  sl_jitter ();
  asm volatile ("{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n"
                ::"r"(smem_u32 (bar)), "r"(parity) : "memory");
}
// Watchdog. Every wait in these kernels is bounded by one pipeline step (microseconds); a wait that fails 2^26 polls in a row
// (seconds) is a broken hand-over protocol. The two single-lane roles every supertile passes through — the producer (waits for a
// free raw stage) and the MMA issuer (waits for operands and a free accumulator) — count their failed polls and trap, so a
// deadlock anywhere in the pipeline ends the launch with an error the host reports instead of hanging the GPU. The other roles
// poll without the counter: with it in every wait the kernels lost 2 .. 4 % (s30_*: TX 431 vs 450, RX 408 vs 415 Gsamples/s).
#ifndef SL_TC_WAIT_LIMIT
#define SL_TC_WAIT_LIMIT 67108864
#endif
__device__ __forceinline__ void mbar_wait_guarded (uint64_t *bar, unsigned parity)
{
#if SL_TC_WAIT_LIMIT > 0
  sl_jitter ();
  asm volatile ("{\n .reg .pred p;\n .reg .u32 n;\n mov.u32 n, 0;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n"
                " add.u32 n, n, 1;\n setp.lt.u32 p, n, %2;\n @p bra WAIT_%=;\n trap;\n DONE_%=:\n}\n"
                ::"r"(smem_u32 (bar)), "r"(parity), "n"(SL_TC_WAIT_LIMIT) : "memory");
#else
  mbar_wait (bar, parity);
#endif
}
__device__ __forceinline__ void bulk_g2s (void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
  asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                ::"r"(smem_u32 (dst)), "l"(src), "r"(bytes), "r"(smem_u32 (bar)) : "memory");
}
__device__ __forceinline__ void named_bar (int id, int threads) { sl_jitter (); asm volatile ("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// ---- tcgen05 ----
// shared-memory matrix descriptor, K-major, no swizzle: core matrix = 8 rows x 16 bytes (128 contiguous bytes);
// LBO = distance between the two 16-byte K-chunks of one instruction, SBO = distance between 8-row groups
// (verified on B200 by tools/microbench/umma_i8_probe.cu, including the aliased SBO used for A)
__device__ __forceinline__ uint64_t umma_desc (uint32_t addr, uint32_t lbo, uint32_t sbo)
{
  return (uint64_t) ((addr & 0x3FFFFu) >> 4) | ((uint64_t) (lbo >> 4) << 16) | ((uint64_t) (sbo >> 4) << 32) | (1ull << 46);
}
// instruction descriptor, kind::i8: D = s32, A / B signedness, both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t umma_idesc (int N, int a_signed, int b_signed)
{
  return (2u << 4) | ((uint32_t) a_signed << 7) | ((uint32_t) b_signed << 10) | ((uint32_t) (N >> 3) << 17) | ((uint32_t) (128 >> 4) << 24);
}
__device__ __forceinline__ void umma_i8 (uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
  asm volatile ("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ bool elect_one ()
{
  uint32_t pred;
  asm volatile ("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit (uint64_t *bar)
{
  asm volatile ("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32 (bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before () { asm volatile ("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after () { asm volatile ("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16 (uint32_t addr, uint32_t *v)
{
  asm volatile ("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                  "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(addr));
}
__device__ __forceinline__ void tmem_ld8 (uint32_t addr, uint32_t *v)
{
  asm volatile ("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(addr));
}
__device__ __forceinline__ void tmem_ld4 (uint32_t addr, uint32_t *v)
{
  asm volatile ("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr));
}
// zero `cols` (a multiple of 4) accumulator columns of the calling thread's TMEM lane
template <int cols> __device__ __forceinline__ void tmem_zero (uint32_t addr)
{
  const uint32_t z = 0u;
#pragma unroll
  for (int c = 0; c + 16 <= cols; c += 16)
    asm volatile ("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(addr + c), "r"(z) : "memory");
  if (cols % 16 >= 8)
    asm volatile ("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(addr + cols / 16 * 16), "r"(z) : "memory");
  if (cols % 8 >= 4)
    asm volatile ("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%1,%1,%1};" ::"r"(addr + cols / 8 * 8), "r"(z) : "memory");
  asm volatile ("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld_wait () { asm volatile ("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

