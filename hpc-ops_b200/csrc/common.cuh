// Shared sm_100a device helpers: mbarrier, TMA, tcgen05/TMEM, UMMA descriptors, vector ld/st.
// Everything here is hand-written inline PTX for Blackwell (no CuTe / CUTLASS).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace b200 {

// ---------------------------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

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

__device__ __forceinline__ float exp2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float log2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// warp-wide float max in one instruction (sm_100a REDUX.f32)
__device__ __forceinline__ float warp_max_f32(float v) {
  float m;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));
  return m;
}
__device__ __forceinline__ float warp_sum_f32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// two fp32 -> packed e4m3x2 (lo = a, hi = b), round-nearest, saturate-to-finite (448)
__device__ __forceinline__ uint16_t cvt_e4m3x2(float a, float b) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t cvt_e4m3x4(float a, float b, float c, float d) {
  return static_cast<uint32_t>(cvt_e4m3x2(a, b)) | (static_cast<uint32_t>(cvt_e4m3x2(c, d)) << 16);
}

// two fp32 -> packed bf16x2 (lo = a, hi = b), round-nearest-even
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Programmatic dependent launch (PDL). A kernel launched with the programmatic-stream-serialization
// attribute may begin while its predecessor in the stream is still running: everything before
// pdl_wait() (barrier init, TMEM allocation, descriptor prefetch) overlaps the predecessor's tail;
// pdl_wait() returns once the predecessor has completed and its writes are visible. Every kernel of
// this library waits before its first access to global memory, so chains stay correct with or
// without the attribute. pdl_launch_dependents() lets the successor's CTAs be scheduled early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// 16-byte streaming global accesses
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_nc_f4(const void* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_v4(void* p, uint4 v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
               : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// generic-proxy writes (st.shared) -> visible to the async proxy (UMMA / TMA reads of smem)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
// suspend-time hint: a waiting thread sleeps in hardware (woken by the phase completion) instead of
// re-issuing try_wait; polling instructions otherwise steal issue slots from the working warps
// B200_MBAR_SUSPEND_NS > 0 adds the suspend-time hint (the waiting thread may be parked by the
// hardware until the phase completes or the hint expires). Measured on B200: parking costs ~6 % on
// the decode-attention and grouped-GEMM kernels (slower wake-up on short waits), so the default is
// a plain try_wait spin.
#ifndef B200_MBAR_SUSPEND_NS
#define B200_MBAR_SUSPEND_NS 0
#endif
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
#if B200_MBAR_SUSPEND_NS > 0
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(static_cast<uint32_t>(B200_MBAR_SUSPEND_NS))
      : "memory");
#else
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
#endif
  return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a launch failure) instead of hanging the GPU.
#ifndef B200_MBAR_SPIN_LIMIT
#if B200_MBAR_SUSPEND_NS > 0
#define B200_MBAR_SPIN_LIMIT (1u << 22)
#else
#define B200_MBAR_SPIN_LIMIT (1u << 26)
#endif
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > B200_MBAR_SPIN_LIMIT) {
      printf("mbar_wait timeout: block %d thread %d bar@%u parity %u\n", blockIdx.x, threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

// Whole-warp roles (warp-uniform producer / issuer loops) poll with ALL lanes. Polling with one lane
// and parking the others at __syncwarp() was measured 1.6x slower on the grouped GEMM and the
// prefill (on-box A/B, profiles/r2_ab_polling.txt): the divergent spin loop costs the uniformity the
// whole-warp structure exists for.

// ---------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) — tile mode loads, completion on an mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ uint64_t make_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t make_policy_evict_normal() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t make_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(void* dst, const CUtensorMap* map, uint64_t* bar,
                                                 int c0, int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* map, uint64_t* bar,
                                                 int c0, int c1, int c2, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_hint(void* dst, const CUtensorMap* map, uint64_t* bar,
                                                 int c0, int c1, int c2, int c3, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy)
      : "memory");
}
// TMA prefetch of a tile into L2 only (no shared-memory destination, no completion to wait for)
__device__ __forceinline__ void tma_prefetch_l2_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(map),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// Bulk prefetch of a contiguous global range into L2 (16-B aligned, size a multiple of 16 B)
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// 1-D bulk copy global -> shared (size multiple of 16 B, 16-B aligned), completes on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// smem -> global tile store (bulk group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0,
                                             int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::
                   "l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read0() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait0() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], fp8 (e4m3/e5m2) inputs, fp32 accumulate
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// bf16/fp16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}
// commit that arrives on the mbarrier at the same CTA-relative offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// ---- cta_group::2: one UMMA spans the two CTAs of a cluster pair -----------------------------
// Each CTA stages its own 128 rows of A and its own half of B's N rows at the SAME smem offsets;
// the leader CTA (even cluster rank) issues the MMA, D lands at the same TMEM address in both CTAs
// (each holds its 128 rows x all N columns). Per SM the B-operand smem reads are halved.
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void umma_f8_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once the issuing thread's earlier MMAs are complete) on the mbarrier at this
// CTA-relative offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// TMA tile loads of a CTA pair: data lands in the executing CTA's smem, the transaction bytes are
// counted on the mbarrier at `bar_cluster_addr` (a shared::cluster address, normally the leader's)
__device__ __forceinline__ void tma_load_2d_2cta(void* dst, const CUtensorMap* map,
                                                 uint32_t bar_cluster_addr, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2cta(void* dst, const CUtensorMap* map,
                                                 uint32_t bar_cluster_addr, int c0, int c1, int c2,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// 32 lanes x 32-bit, N consecutive columns; thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]),
                 "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

// registers -> TMEM, 32 lanes x 16 consecutive 32-bit columns (mirror of tmem_ld_x16)
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// Compiler-level anchor: values produced by an (asynchronous) tcgen05.ld may only be consumed after
// tcgen05.wait::ld. Passing the registers through an empty volatile asm placed after the wait
// keeps the compiler from scheduling their consumers above it (zero instructions emitted).
__device__ __forceinline__ void tmem_anchor16(uint32_t* r) {
  asm volatile(""
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]),
                 "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]),
                 "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// ---------------------------------------------------------------------------------------------
// Thread-block clusters: rank, barrier, distributed shared memory loads
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// all threads of all CTAs of the cluster; release/acquire so smem writes before are visible after
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;\n"
               "barrier.cluster.wait.acquire;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t cluster_addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(cluster_addr)
               : "memory");
  return v;
}
__device__ __forceinline__ void st_dsmem_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
// arrive on an mbarrier of another CTA of the cluster (release at cluster scope: stores to that
// CTA's shared memory issued before it are visible to a waiter that acquires at cluster scope)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr)
               : "memory");
}
// same, without ordering of surrounding memory accesses (pure "slot is free" notifications)
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_bar_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr)
               : "memory");
}
// local wait that acquires at cluster scope (pairs with mbar_arrive_cluster / multicast commits)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (true) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) return;
    if (++spins > B200_MBAR_SPIN_LIMIT) {
      printf("mbar_wait_cluster timeout: block %d thread %d bar@%u parity %u\n", blockIdx.x,
             threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}
// TMA tile load multicast to the CTAs of `cta_mask`: the box lands at the same CTA-relative smem
// offset in every destination CTA and completes tx bytes on the mbarrier at the same offset there
__device__ __forceinline__ void tma_load_2d_mcast(void* dst, const CUtensorMap* map, uint64_t* bar,
                                                  int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_mcast(void* dst, const CUtensorMap* map, uint64_t* bar,
                                                  int c0, int c1, int c2, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      ".multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
      : "memory");
}

// ---------------------------------------------------------------------------------------------
// Packed fp32 pairs (sm_100 FMUL2 / FFMA2 / FADD2: one issue slot for two lanes of work)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pack_f2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

// ---------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts: PTX ISA "tcgen05 matrix / instruction descriptor")
// ---------------------------------------------------------------------------------------------
enum : uint32_t { kLayoutNone = 0, kLayoutSW128 = 2, kLayoutSW64 = 4, kLayoutSW32 = 6 };

// 64-bit shared-memory matrix descriptor. addr/lbo/sbo in BYTES (multiples of 16).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);          // [0,14)  start address
  d |= static_cast<uint64_t>((lbo_bytes & 0x3FFFFu) >> 4) << 16;    // [16,30) leading byte offset
  d |= static_cast<uint64_t>((sbo_bytes & 0x3FFFFu) >> 4) << 32;    // [32,46) stride byte offset
  d |= static_cast<uint64_t>(1) << 46;                              // [46,48) version = 1 (sm_100)
  d |= static_cast<uint64_t>(layout & 7u) << 61;                    // [61,64) swizzle mode
  return d;
}

// 32-bit instruction descriptor for kind::f8f6f4 (a/b fmt 0 = e4m3) and kind::f16 (fmt 1 = bf16).
// major: 0 = K-major, 1 = MN-major.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t M, uint32_t N, uint32_t a_fmt,
                                                  uint32_t b_fmt, uint32_t a_major,
                                                  uint32_t b_major) {
  return (1u << 4)                 // c_format = F32
         | (a_fmt << 7)            // a_format
         | (b_fmt << 10)           // b_format
         | (a_major << 15)         // a_major
         | (b_major << 16)         // b_major
         | ((N >> 3) << 17)        // n_dim
         | ((M >> 4) << 24);       // m_dim
}
constexpr uint32_t kFmtE4M3 = 0;
constexpr uint32_t kFmtBF16 = 1;

// byte offset of (row r, 16-byte chunk c) inside a 128B-swizzled tile whose rows are 128 B wide
// and whose base is 1024-B aligned (this is what TMA SWIZZLE_128B writes and UMMA SW128 reads).
__host__ __device__ constexpr uint32_t sw128_offset(uint32_t r, uint32_t c) {
  return r * 128u + ((c ^ (r & 7u)) << 4);
}

}  // namespace b200
