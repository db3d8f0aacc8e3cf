// PTX wrappers shared by the tcgen05 kernels (conv_tc.cu, wgrad_tc.cu): mbarriers with bounded waits, warp-uniform
// leader election, proxy / tcgen05 fences, asynchronous copies, tcgen05.mma / commit / ld.  sm_100a only.
#pragma once
#include "common.cuh"

namespace tcptx {

constexpr uint32_t SPIN_LIMIT = 1u << 20;   // try_wait blocks for a while per call: this is seconds

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint (ns): the thread sleeps in hardware until the phase completes or the hint runs out.
// Without a hint the default limit is a few tens of cycles on sm_100a: the issuing / epilogue / loader warps then
// spin through try_wait ~20 times per stage, and those loops were 28% of all instructions the kernel issued (ncu,
// profiles/r02d_conv_tc_ncu_*): issue slots taken from the gathering warps of an issue-bound kernel.
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity, uint32_t hint_ns = 1000u) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(hint_ns)
      : "memory");
  return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a while; test_wait never does)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (launch failure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try(bar, parity)) {
    if (++spins > SPIN_LIMIT) __trap();
  }
}
// Two forms of a long wait.  mbar_wait_long: try_wait with a long suspend hint; on sm_100a it compiles to TRYWAIT +
// NANOSLEEP.SYNCS, which wakes on the CTA's mbarrier traffic (a phase completes every ~50 cycles in these kernels), so
// the epilogue warps still retry ~2600 times per launch and the retry loops are 28% of the instructions issued (ncu,
// profiles/r02f_conv_tc_*).  mbar_wait_sleep: probe + a real nanosleep -- almost no instructions, but the waiter
// notices completion up to `ns` late.  Measured A/B on the six level shapes: the spinning form is 1-3% FASTER wherever a
// CTA walks several groups (the kernel is bound by latencies, not by issue slots: the spare slots are free), the
// sleeping form wins 5% on single-tile CTAs (K-split), where the epilogue wait sits on the critical path next to two
// issuing warps.  Each is used where it won.
__device__ __forceinline__ void mbar_wait_long(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try(bar, parity, 4000u)) {
    if (++spins > SPIN_LIMIT) __trap();
  }
}
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t spins = 0;
  while (!mbar_test(bar, parity)) {
    __nanosleep(ns);
    if (++spins > SPIN_LIMIT) __trap();
  }
}
// Warp-uniform leader election.  The issuing warps keep their whole control flow warp-uniform and only predicate
// the tcgen05 / bulk-copy instruction itself on the elected lane: operands then live in uniform registers.  (With an
// `if (lane == 0)` around the loop the compiler cannot prove uniformity and wraps every UTCHMMA / UTCBAR / UBLKCP in
// an R2UR + ELECT + BRA.U.ANY waterfall: ~80 cycles each, which made the single MMA thread the bottleneck.)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// Stage-ready flags: a monotonically increasing sequence number per A slot (release store / acquire poll).  A parity
// mbarrier cannot be used here: the issuing warps run up to SA stages apart, and a warp waiting for phase k of a slot
// would be released by phase k-2 when the warp that must consume phase k-1 lags behind.
__device__ __forceinline__ void st_release_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ uint4 ldg_nc128(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ int ldg_nc32(const int* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
// 16-byte asynchronous global->shared copy (LDGSTS, L2 only); src_bytes == 0 writes zeros without reading
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// this thread's arrival on `bar` fires when all its cp.async issued so far have landed (the count is pre-charged at init)
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// tcgen05.mma with a disable-output-lane mask: bit r of {m0..m3} set => TMEM lane (= output row) r is NOT updated, so the
// A-tile row r may hold anything (stale shared memory): rows without a neighbour at this offset are never gathered.
// TF32: the kind::tf32 form (fp32 bits in shared memory, 10-bit mantissa operands, K = 8 per instruction).
template <bool TF32 = false>
__device__ __forceinline__ void umma_masked(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate,
                                            uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
  if constexpr (TF32)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
        : "memory");
}
// fp32 -> TF32 bits, rounded to nearest (ties away from zero); the low 13 bits of the result are zero
__device__ __forceinline__ float to_tf32_rna(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// two 16-column loads in flight, one wait (the K-split epilogue adds two accumulators)
__device__ __forceinline__ void tmem_ld16x2(uint32_t taddr_a, uint32_t taddr_b, uint32_t* a, uint32_t* b) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]),
        "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15])
      : "r"(taddr_a));
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]), "=r"(b[8]),
        "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15])
      : "r"(taddr_b));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

}  // namespace tcptx
