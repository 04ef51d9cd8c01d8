// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Everything here is a one-instruction wrapper; protocols live in the kernels that use them.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace b200 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// One lane of a fully converged warp. Single-thread instructions (tcgen05.mma / commit, TMA) are issued as
// `if (elect_one()) {...}` from warp-uniform control flow: their descriptor operands then stay in uniform registers,
// whereas code under `if (lane == 0)` makes the compiler wrap every such instruction in a vote/elect loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Probe that may stay suspended in hardware for up to `hint_ns` nanoseconds before it reports "not yet".
__device__ __forceinline__ bool mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
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
// Bounded wait. A protocol slip (or a fault in another role) must not hang the GPU: a wait that has lasted
// B200_WAIT_LIMIT_NS raises the library's abort word (mapped host memory, see host_util.cu) and returns; once the word
// is set, every wait that has lasted B200_WAIT_WATCH_NS (far longer than any wait of a healthy kernel, which are
// microseconds) sees it and falls through, so the kernel drains in bounded time with garbage results and the next
// C-ABI call returns an error instead of enqueueing more work.
// mbarrier.try_wait comes back "not yet" long before any useful time limit (a wait of a few hundred clocks already
// takes several probes), so the probe loop is hot: it is 16 back-to-back probes — exactly the instructions of a plain
// spin — and only every 16th failed probe pays for a counter, every 1024th for a timer read. Round-2 A/B on the
// attention kernel: a counter or a memory read per probe costs 5-7 %; this form measures the same as the plain spin.
#ifndef B200_WAIT_LIMIT_NS
#define B200_WAIT_LIMIT_NS 4000000000ull
#endif
#ifndef B200_WAIT_WATCH_NS
#define B200_WAIT_WATCH_NS 2000000ull
#endif
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Plain spin, for the one role whose register budget is too tight for the bounded form (the attention kernel's MMA
// issuer, 88 registers after setmaxnreg): everything it waits on is produced by roles that ARE bounded and that keep
// walking the protocol after giving up, so its waits still complete.
__device__ __forceinline__ void mbar_wait_plain(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization attribute may
// become resident while its predecessor on the stream is still draining; `griddep_wait` blocks until the predecessor
// has completed and its memory is visible, and must come before the first global access. `griddep_launch_dependents`
// lets the successor's CTAs be scheduled as soon as resources free up.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Wait that parks the warp in hardware: mbarrier.try_wait with an explicit suspend-time hint stays suspended until the
// phase completes (or the hint runs out) instead of coming back after a few dozen clocks, so a waiting warp issues
// almost nothing and leaves its sub-partition's issue slots to the warps that compute.
#ifndef B200_WAIT_HINT_NS
#define B200_WAIT_HINT_NS 100000u
#endif
__device__ __forceinline__ void mbar_wait_parked(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait_hint(bar, parity, B200_WAIT_HINT_NS)) {
  }
}
struct WaitCtx {
  unsigned int* abort_word;  // may be nullptr (stand-alone tools): then a wait never gives up
};
__device__ __forceinline__ WaitCtx make_wait_ctx(unsigned int* abort_word) { return WaitCtx{abort_word}; }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, const WaitCtx& w) {
  uint32_t rounds = 0;
  uint64_t t0 = 0;
  for (;;) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (mbar_try_wait(bar, parity)) return;
    if ((++rounds & 63u) == 0u && w.abort_word != nullptr) {  // every 1024 failed probes
      const uint64_t now = global_timer_ns();
      if (t0 == 0) {
        t0 = now;
      } else if (now - t0 > B200_WAIT_WATCH_NS) {
        volatile unsigned int* aw = reinterpret_cast<volatile unsigned int*>(w.abort_word);
        if (*aw != 0u) return;
        if (now - t0 > B200_WAIT_LIMIT_NS) {
          *aw = 0xB200DEADu;
          __threadfence_system();
          return;
        }
      }
    }
  }
}

__device__ __forceinline__ uint32_t lds_u32_volatile(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32_volatile(uint32_t addr, uint32_t v) {
  asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// ---------------------------------------------------------------- clusters (CTA pairs)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// Relaxed: the callers only order tcgen05 (TMEM) accesses, which tcgen05.fence::before_thread_sync covers; a
// release at cluster scope would add MEMBAR + ERRBAR (measured: ~20% of the GEMM epilogue's stall samples).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint32_t bar, uint32_t dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// cta_group::2 variants: data lands in this CTA's smem, the transaction bytes are signalled on `bar_cluster`
// (a shared::cluster address — the leader CTA's barrier).
__device__ __forceinline__ void tma_load_2d_2cta(const CUtensorMap* m, uint32_t bar_cluster, uint32_t dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2cta(const CUtensorMap* m, uint32_t bar_cluster, uint32_t dst, int c0, int c1,
                                                 int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------- register re-allocation between warpgroups
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ---------------------------------------------------------------- TMEM alloc
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(NCOLS)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// CTA-pair versions: executed by the same warp of BOTH CTAs of the pair.
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(NCOLS)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

// ---------------------------------------------------------------- tcgen05.mma
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (bf16/fp16 in, fp32 accumulate).
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand read from TMEM (16-bit elements packed two per 32-bit column).
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// CTA-pair MMA (issued by the leader CTA only): M = 256 spans both CTAs' TMEM, each CTA supplies half of B.
__device__ __forceinline__ void umma_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ... and its completion signal, multicast to the barrier at the same smem offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   bar),
               "h"(cta_mask)
               : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// kind::f8f6f4 (here: e4m3 x e4m3 -> fp32, K = 32 per instruction): the optional FP8 variant of the linears
__device__ __forceinline__ void umma_ss_f8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ss_f8_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Instruction descriptor for kind::f8f6f4 with both operands e4m3 (format code 0), fp32 accumulate, K-major.
__host__ __device__ constexpr uint32_t make_idesc_e4m3(int M, int N) {
  return (1u << 4)                       // c_format = F32
         | (0u << 7) | (0u << 10)        // a_format = b_format = E4M3
         | (uint32_t(N >> 3) << 17)      // n_dim
         | (uint32_t(M >> 4) << 24);     // m_dim
}

// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32 (bit layout: cute/arch/mma_sm100_desc.hpp InstrDescriptor).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                           // c_format = F32
         | (1u << 7)                         // a_format = BF16
         | (1u << 10)                        // b_format = BF16
         | (uint32_t(a_mn_major) << 15)      // a_major (0 = K-major)
         | (uint32_t(b_mn_major) << 16)      // b_major
         | (uint32_t(N >> 3) << 17)          // n_dim
         | (uint32_t(M >> 4) << 24);         // m_dim
}

// Shared-memory matrix descriptor (SmemDescriptor in the same header): 128-byte swizzle, version 1.
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1     bits [61,64) layout (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFFu) >> 4);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(2) << 61;
  return d;
}

// 32-byte swizzle (layout 6): K-major rows of 32 bytes, 8-row atoms of 256 bytes; one K step of a bf16 MMA (16
// elements) is exactly one atom wide, so only sbo (the distance between 8-row groups) matters.
__device__ __forceinline__ uint64_t make_smem_desc_sw32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFFu) >> 4);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(6) << 61;
  return d;
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint32_t bar, uint32_t dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---------------------------------------------------------------- TMEM <-> registers
// 32 lanes x 32 columns of 32-bit: thread t of the warp gets lane (base_lane + t), columns [col, col+32).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return r;
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- small math helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace b200
