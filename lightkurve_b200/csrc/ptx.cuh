// Inline-PTX wrappers for sm_100a: mbarrier, named barriers, cp.async, TMA bulk copies, tcgen05 / TMEM.
// Under the CPU emulator (LKB_CUDA_EMU, tests/native/cuda_emu.h) the few that ls_nufft.cu uses have host versions at
// the end of this file.
#pragma once
#if !defined(LKB_CUDA_EMU)
#include <stdint.h>
#include <cuda.h>

namespace lkb {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier -------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes or ~hint_ns pass
// (no polling instructions in between - the nanosleep loops were measured to re-poll every ~36 ns)
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t hint_ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_park(uint64_t* bar, uint32_t parity, uint32_t hint_ns) {
  while (!mbar_try_wait_hint(bar, parity, hint_ns)) {
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// Same, but backs off with nanosleep between polls: for warps that wait long (TMA producer,
// epilogue) so that their polling does not steal issue slots from the compute warps.
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, uint32_t ns) {
  while (!mbar_try_wait(bar, parity)) {
    if (ns) __nanosleep(ns);
  }
}

// %tid.x read afresh at each call (volatile: not hoisted out of a loop).  In a persistent kernel the compiler would
// otherwise keep every per-thread offset derived from it live across the whole loop body - at a register cap, in local
// memory.
__device__ __forceinline__ int tid_x() {
  int t;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
  return t;
}

// ---- named barriers / cp.async ---------------------------------------------------
// barrier `id` (1 .. 15) over `nthreads` threads (a multiple of 32) of the CTA
__device__ __forceinline__ void bar_sync_named(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// 8-byte copy global -> shared (SASS: LDGSTS); src_bytes = 0 zero-fills the destination and reads nothing
__device__ __forceinline__ void cp_async_8(void* dst_smem, const void* src_gmem, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(src_bytes)
               : "memory");
}
// one arrival on `bar` once every cp.async this thread has issued so far has landed; the arrival is one of the count
// the barrier was initialised with (.noinc)
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// wait until every cp.async this thread has issued has landed
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- async-proxy fences / TMA ---------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk copy global -> shared (TMA engine; SASS: UBLKCP).  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// 2-D tiled TMA load (SASS: UTMALDG).
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const CUtensorMap* map, int32_t c0, int32_t c1,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(smem_u32(dst_smem)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (fp16/bf16 in, fp32 accumulate).
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued MMAs of this thread arrive on `bar` when complete
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: 32 lanes x 32 columns of 32-bit (one warp reads its own 32-lane quadrant).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// ---- thread-block clusters / CTA pairs (cta_group::2) -----------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in the pair's LEADER CTA (rank 0): the CTA rank
// sits in bit 24 of a shared-window address (CUTLASS: Sm100MmaPeerBitMask)
__device__ __forceinline__ uint32_t leader_addr(const void* p) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(0));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster_sleep(uint64_t* bar, uint32_t parity, uint32_t ns) {
  while (!mbar_try_wait_cluster(bar, parity)) __nanosleep(ns);
}
// 2-D tiled TMA load into THIS CTA's shared memory whose transaction bytes are counted on an mbarrier of
// the pair's leader CTA (SASS: UTMALDG with cta_group::2).
__device__ __forceinline__ void tma_load_2d_2sm(void* dst_smem, const CUtensorMap* map, int32_t c0, int32_t c1,
                                                uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst_smem)),
      "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs, M = 256] (+)= A[128 rows in each CTA] * B[N/2 rows in each CTA]; leader CTA only.
__device__ __forceinline__ void umma_f16_ss_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this shared-memory offset in BOTH CTAs of the pair once all MMAs issued so far retire
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                   "r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

}  // namespace ptx
}  // namespace lkb

#else  // LKB_CUDA_EMU
// Host versions for the CPU emulator, which runs every thread of a block as a host thread and one block at a time, so
// state shared by all blocks is the state of the running block.  The kernels run the same ring logic - buffer indices,
// parities, group handoff - as on the device.
// mbarrier word: bits 0-31 the arrival count it was initialised with, 32-62 arrivals still pending in the current
// phase, 63 the current phase's parity.  A parity wait returns once the phase of that parity has completed, i.e. while
// the current phase's parity differs - so, as on the device, a wait two phases ahead passes on the phase before.
// cp.async is a synchronous copy, so the arrive that tracks it is a plain arrive.
#include <stdint.h>
#include <string.h>
#include <condition_variable>
#include <mutex>

namespace lkb {
namespace ptx {
struct EmuSync {
  std::mutex m;
  std::condition_variable cv;
  int arrived[16] = {};
  long generation[16] = {};
};
inline EmuSync& emu_sync() {
  static EmuSync s;
  return s;
}
inline int tid_x() { return (int)threadIdx.x; }
inline void bar_sync_named(int id, int nthreads) {
  EmuSync& e = emu_sync();
  std::unique_lock<std::mutex> lk(e.m);
  const long gen = e.generation[id];
  if (++e.arrived[id] == nthreads) {
    e.arrived[id] = 0;
    ++e.generation[id];
    e.cv.notify_all();
    return;
  }
  e.cv.wait(lk, [&] { return gen != e.generation[id]; });
}
inline void mbar_init(uint64_t* bar, uint32_t count) {
  std::lock_guard<std::mutex> lk(emu_sync().m);
  *bar = (uint64_t)count | ((uint64_t)count << 32);
}
inline void mbar_arrive(uint64_t* bar) {
  EmuSync& e = emu_sync();
  std::lock_guard<std::mutex> lk(e.m);
  const uint64_t count = *bar & 0xffffffffull, phase = *bar >> 63, pending = ((*bar >> 32) & 0x7fffffffull) - 1;
  if (pending == 0) {
    *bar = count | (count << 32) | ((phase ^ 1ull) << 63);
    e.cv.notify_all();
  } else {
    *bar = count | (pending << 32) | (phase << 63);
  }
}
inline void mbar_wait(uint64_t* bar, uint32_t parity) {
  EmuSync& e = emu_sync();
  std::unique_lock<std::mutex> lk(e.m);
  e.cv.wait(lk, [&] { return (uint32_t)(*bar >> 63) != (parity & 1u); });
}
inline void cp_async_8(void* dst_smem, const void* src_gmem, uint32_t src_bytes) {
  memset(dst_smem, 0, 8);
  if (src_bytes) memcpy(dst_smem, src_gmem, src_bytes);
}
inline void cp_async_mbar_arrive_noinc(uint64_t* bar) { mbar_arrive(bar); }
inline void cp_async_wait_all() {}
}  // namespace ptx
}  // namespace lkb
#endif  // LKB_CUDA_EMU
