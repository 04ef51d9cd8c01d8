// What the two attention kernels (attention_stream.cuh, attention_short.cuh) share: the tile geometry, the register
// split between the control and softmax warpgroups, the exponential helpers and the event trace of the -DATT_TRACE
// build.
//
// Both kernels run 384 threads as one persistent CTA per SM with the same roles: warp 0 TMA producer, warp 1
// tcgen05.mma issuer, warp 2 watchdog, warp 3 idle (warps 2..3 complete warpgroup 0 so that it can hand registers to
// the softmax warpgroups), warps 4..11 softmax / output of the two 128-row query tiles. Q/K/V are read straight out of
// the fused QKV activation [rows, 3d] through strided 3-D tensor maps (no head transpose is materialised); the output
// is written head-interleaved as [rows, d] for out_proj.
//
// Watchdog: the working warps wait on their mbarriers without a time limit (a bounded loop costs the streaming kernel
// 3-7 %, round-2 A/B). The watchdog warp sleeps on a DONE barrier and, if the MMA issuer's progress counter has not
// moved for B200_WAIT_LIMIT_NS, raises the library's abort word and keeps arriving on every protocol barrier, so that
// every stuck waiter falls through, the roles run out of work and the kernel exits (garbage results, reported by the
// next C-ABI call) instead of hanging the GPU. The loop is written out in each kernel: as a shared function it
// changed the kernels' instruction schedules.
#pragma once
#include "ptx.cuh"

namespace b200 {

constexpr int ATT_BQ = 128;
constexpr int ATT_BKV = 128;
constexpr int ATT_HD = 64;
constexpr int ATT_THREADS = 384;  // warpgroup 0: producer, MMA issuer, watchdog, 1 idle warp; warpgroups 1, 2: softmax
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KB: 128 rows x 64 bf16, 128B-swizzled
constexpr int ATT_STG_BYTES = 32 * 128;       // one softmax warp's output rows: 32 x 64 bf16
constexpr int ATT_SOFTMAX_REGS = 208;  // setmaxnreg: the increase blocks until the control warpgroup has released enough
constexpr int ATT_CONTROL_REGS = 88;   //   (the kernel starts with 168 x 384 = 64512 registers: 4 x 32 x 88 + 8 x 32 x 208 uses exactly that)

// Every ATT_POLY_EVERY-th pair of scores takes its exponentials from exp2_poly2 instead of MUFU.EX2 (0 = never).
// Same-box A/B at 25 %: L=1500 0.176 -> 0.169 ms, L=576 0.110 -> 0.106 ms, L=197 0.0555 -> 0.0545 ms; 50 % is slower
// than none (the FMA pipe and the issue slots become the limit), 12-33 % are within noise of each other.
#ifndef ATT_POLY_EVERY
#define ATT_POLY_EVERY 4
#endif
// 2^x for x <= ~8 on the FMA pipe (Cody-Waite split + degree-3 minimax of 2^f on [-0.5, 0.5], max relative error
// 7.7e-5, far below the bf16 rounding of P): takes a share of the exponentials off the MUFU pipe.
__device__ __forceinline__ float2 exp2_poly2(float2 x) {
  x = make_float2(fmaxf(x.x, -126.0f), fmaxf(x.y, -126.0f));
  const float2 magic = make_float2(12582912.0f, 12582912.0f);  // 1.5 * 2^23: the sum's low mantissa bits hold round(x)
  const float2 t = __fadd2_rn(x, magic);
  const float2 n = __fadd2_rn(t, make_float2(-12582912.0f, -12582912.0f));
  const float2 f = __ffma2_rn(n, make_float2(-1.0f, -1.0f), x);
  float2 q = __ffma2_rn(f, make_float2(0.05508868396282196f, 0.05508868396282196f),
                        make_float2(0.24260404706001282f, 0.24260404706001282f));
  q = __ffma2_rn(q, f, make_float2(0.6932762265205383f, 0.6932762265205383f));
  q = __ffma2_rn(q, f, make_float2(0.9999289512634277f, 0.9999289512634277f));
  return make_float2(__int_as_float(__float_as_int(q.x) + (__float_as_int(t.x) << 23)),
                     __int_as_float(__float_as_int(q.y) + (__float_as_int(t.y) << 23)));
}

// three-input maximum (FMNMX3): two scores per instruction in the row-maximum chains
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// Offset-causal mode (the kOffset instantiation of the streaming kernels; b200enc_attention_extend): K/V are the rows
// [0, capacity) of a KV cache, the Lq query rows of sequence b sit at absolute positions off_b + i, and query i sees
// key j iff j <= off_b + i (bottom-right aligned causal). Sequence b has kv_len = off_b + Lq keys; blocks past it are
// never visited. The rows [kv_len, capacity) of the cache are not ours: they may hold anything, NaN included, and
// 0 * NaN = NaN in the P.V product. K there only feeds masked scores, but V rows [kv_len, ceil16(kv_len)) are inside
// the last P.V K-step, so the MMA issuer zeroes them in shared memory (att_zero_rows) before it issues that P.V.
// An offset outside [0, capacity - Lq] is computed as offset 0 and the sequence's outputs are set to NaN.
struct AttOffset {
  int off;   // query offset of the sequence (0 if out of range)
  bool bad;  // the device offset was out of range
};
__device__ __forceinline__ AttOffset att_seq_offset(const int* off, int stride, int b, int Lq, int capacity) {
  const int o = off[b * stride];
  const bool bad = o < 0 || o > capacity - Lq;
  return AttOffset{bad ? 0 : o, bad};
}

// Zero rows [r0, r1) of a 128-row x 128-byte shared-memory box (whole rows: the 128B swizzle only permutes the 16-byte
// chunks inside a row), then make the generic-proxy stores visible to the tensor core. Called by one full warp.
__device__ __forceinline__ void att_zero_rows(uint32_t box, int r0, int r1) {
  const int lane = threadIdx.x & 31;
  for (int i = r0 * 8 + lane; i < r1 * 8; i += 32) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(box + 16u * i), "r"(0u) : "memory");
  }
  fence_proxy_async_smem();
  __syncwarp();
}

// Event trace of the -DATT_TRACE build (make ../b200enc_trace): (event, clock) records of CTA 0 in per-role private
// slots (no atomics: a store and a clock read per event). ATT_EV expects `p.trace`, `tr_n` and `tr_role` in scope;
// AttTrace carries the same handle into a helper function (one designated lane per softmax warpgroup).
#ifdef ATT_TRACE
#define ATT_EV(ev)                                                              \
  do {                                                                          \
    if (p.trace != nullptr && blockIdx.x == 0 && tr_n < 1000) {                 \
      p.trace[2 * (tr_role * 1000 + tr_n)] = (ev);                              \
      p.trace[2 * (tr_role * 1000 + tr_n) + 1] = clock64();                     \
      ++tr_n;                                                                   \
    }                                                                           \
  } while (0)
struct AttTrace {
  long long* buf;
  int role;
  int* n;
  bool on;
  __device__ __forceinline__ void ev(int e) const {
    if (on && buf != nullptr && blockIdx.x == 0 && *n < 1000) {
      buf[2 * (role * 1000 + *n)] = e;
      buf[2 * (role * 1000 + *n) + 1] = clock64();
      ++*n;
    }
  }
};
#define ATT_TR(tr, e) (tr).ev(e)
#else
#define ATT_EV(ev) do {} while (0)
struct AttTrace {};
#define ATT_TR(tr, e) do {} while (0)
#endif

}  // namespace b200
