// Thin inline-PTX wrappers for the sm_100a features the batched kernels use:
// mbarrier, 1-D bulk async copy (TMA engine, SASS UBLKCP), tcgen05 (alloc / mma / commit / ld / st
// / fences).  Descriptor bit layouts follow the PTX ISA "tcgen05" chapter (same fields as
// cute/arch/mma_sm100_desc.hpp in the CUTLASS headers shipped with this image).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace go2p {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One lane of a fully converged warp (elect.sync).  Unlike `lane == 0`, the compiler knows that exactly one
// thread runs the guarded region, so warp-uniform instructions inside it (UTCHMMA, UBLKCP, ...) are emitted
// straight instead of inside a per-active-thread "waterfall" loop (measured: ~150 -> ~64 cycles per MMA).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// fire-and-forget: bring the line holding p into L2
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ------------------------------------------------------------------ programmatic dependent launch
// wait: the grids this launch depends on (the previous kernel of the stream) have completed and their memory is visible
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// the dependent launch (the next kernel of the stream, if it opted in) may begin once every CTA has said so or exited
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// non-blocking probe (try_wait may suspend the thread for a system-dependent time before answering "not yet":
// measured ~1000+ cycles, which serialises a poller that watches several barriers)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// A protocol bug must surface as a launch failure, never as a hung GPU: the wait traps after 2^25 failed polls.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // the whole wait as one PTX loop: two instructions when the phase is already complete, no convergence bookkeeping;
  // the watchdog is a poll counter (a failed try_wait parks the warp for a bounded time, so 2^25 polls is seconds)
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .pred q;\n\t.reg .u32 n;\n\t"
      "mov.u32 n, 0;\n"
      "GO2P_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra GO2P_DONE;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 q, n, 0x2000000;\n\t"
      "@q bra GO2P_WAIT;\n\t"
      "trap;\n"
      "GO2P_DONE:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// suspend-time hint of a blocking wait: a waiting warp sleeps in the barrier unit until the phase completes (it is woken
// by the completing arrival) or this many nanoseconds pass, instead of re-polling every few hundred cycles -- the
// re-polls of the warps that run ahead took issue slots from the warps they were waiting for
constexpr uint32_t kMbarSuspendNs = 4000;

// the same operations on 32-bit shared-window addresses (no generic -> shared conversion per call)
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .pred q;\n\t.reg .u32 n;\n\t"
      "mov.u32 n, 0;\n"
      "GO2P_WAITU:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra GO2P_DONEU;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 q, n, 0x2000000;\n\t"
      "@q bra GO2P_WAITU;\n\t"
      "trap;\n"
      "GO2P_DONEU:\n\t}"
      ::"r"(bar), "r"(parity), "r"(kMbarSuspendNs) : "memory");
}

// generic-proxy smem writes -> visible to the async proxy (tensor core / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------ bulk async copy (global -> shared)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// shared -> global bulk async copy (the generic-proxy writes to the source must be fenced with fence.proxy.async and
// ordered before the issuing thread by a barrier); completion is tracked per issuing thread in bulk groups
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // sources may be overwritten
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }          // writes are complete

// ------------------------------------------------------------------ tcgen05: TMEM management
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(kCols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {        // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ tcgen05: descriptors
// Shared-memory matrix descriptor, K-major operand, SWIZZLE_NONE ("interleaved" 8x16B core matrices):
//   bits [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (between the two core matrices
//   along K) | [32,46) stride byte offset >> 4 (between 8-row groups) | [46,48) version = 1 | [61,64) layout = 0
__device__ __forceinline__ uint64_t make_smem_desc_nosw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46);
}
// Instruction descriptor for kind::f16 / kind::tf32 with fp32 accumulation, K-major A and B:
//   [4,6) D format (1 = F32) | [7,10) A format | [10,13) B format (0 = F16, 1 = BF16, 2 = TF32)
//   [17,23) N >> 3 | [24,29) M >> 4
enum : uint32_t { FMT_F16 = 0, FMT_BF16 = 1, FMT_TF32 = 2 };
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, uint32_t M, uint32_t N) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[tmem] * B[smem]^T   (one thread issues for the CTA)
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// all previously issued MMAs of this thread -> one arrival on the mbarrier when they complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------ tcgen05: TMEM <-> registers
// 32x32b: lane i of the warp accesses TMEM lane (32*(warp%4) + i); .xN = N consecutive 32-bit columns.
#define GO2P_R4(v, o) "=r"(v[o]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3])
#define GO2P_W4(v, o) "r"(v[o]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3])

__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : GO2P_R4(v, 0), GO2P_R4(v, 4), GO2P_R4(v, 8), GO2P_R4(v, 12), GO2P_R4(v, 16), GO2P_R4(v, 20), GO2P_R4(v, 24), GO2P_R4(v, 28)
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : GO2P_R4(v, 0), GO2P_R4(v, 4), GO2P_R4(v, 8), GO2P_R4(v, 12)
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : GO2P_R4(v, 0) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), GO2P_W4(v, 0), GO2P_W4(v, 4), GO2P_W4(v, 8), GO2P_W4(v, 12) : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), GO2P_W4(v, 0), GO2P_W4(v, 4) : "memory");
}

// ------------------------------------------------------------------ conversions / math
// packs {lo -> bits[0,16), hi -> bits[16,32)}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// per 16-bit half: neg where z < 0 (ONNX Elu: -0.0 and NaN take the pass-through side), else z
__device__ __forceinline__ uint32_t select_neg_f16x2(uint32_t z, uint32_t neg) {
  uint32_t m;
  asm("set.lt.u32.f16x2 %0, %1, %2;" : "=r"(m) : "r"(z), "r"(0u));
  return (neg & m) | (z & ~m);
}
__device__ __forceinline__ uint32_t select_neg_bf16x2(uint32_t z, uint32_t neg) {
  uint32_t m;
  asm("set.lt.u32.bf16x2 %0, %1, %2;" : "=r"(m) : "r"(z), "r"(0u));
  return (neg & m) | (z & ~m);
}
// packed fp16 pair: 2^x (two MUFU.EX2.F16 operations) and a*b+c (one HFMA2)
__device__ __forceinline__ uint32_t ex2_f16x2(uint32_t x) {
  uint32_t r;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(r) : "r"(x));
  return r;
}
__device__ __forceinline__ uint32_t fma_f16x2(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
__device__ __forceinline__ uint32_t add_f16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t sub_f16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// per half: the larger operand; a NaN operand yields the other one
__device__ __forceinline__ uint32_t max_f16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// per half: the larger operand; NaN if either operand is NaN (one HMNMX2.NAN)
__device__ __forceinline__ uint32_t max_nan_f16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.NaN.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t max_nan_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.NaN.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// a*b + c (mod 2^32) as one IMAD: the compiler splits a multiplication by a power of two into a shift and an add
__device__ __forceinline__ uint32_t mad_lo_u32(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
// per half: -|x|.  Two separate PTX operations so that ptxas folds them into the consumer's source operand as the -|.|
// modifier (MUFU.EX2.F16 R, -|R0|; HMNMX2 R, -|R0|, ...): no instruction of its own
__device__ __forceinline__ uint32_t negabs_f16x2(uint32_t x) {
  uint32_t a, r;
  asm("abs.f16x2 %0, %1;" : "=r"(a) : "r"(x));
  asm("neg.f16x2 %0, %1;" : "=r"(r) : "r"(a));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

}  // namespace ptx
}  // namespace go2p
