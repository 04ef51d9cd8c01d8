// Flash-style attention (optionally causal) for head_dim 64 on sm_100a (reference: F.scaled_dot_product_attention at
// pytorch_models/transformer.py:52 with attn_mask=None, dropout_p=0, is_causal = MHA.forward's `causal`).
//
// One work item = (batch, head, pair of 128-row query tiles). One persistent CTA per SM loops over items; key/value
// rows stream through a 4-stage TMA ring in blocks of 128 with an online softmax. 384 threads:
//   warp 0      : TMA producer (Q pair, double-buffered across items; K/V blocks)
//   warp 1      : tcgen05.mma issuer, one stream across items in the order  PV0(n) PV1(n) QK0(n+2) QK1(n+2)
//                   S_t = Q_t K_j^T          -> TMEM, fp32, 128 columns per tile
//                   O_t (+)= P_t V_j         -> TMEM, 64 columns, accumulated in place; P_t is the TMEM A operand
//   warp 2      : watchdog (see attention_common.cuh), warp 3 : idle
//   warps 4..7  : softmax warpgroup of tile 0, warps 8..11 : tile 1. One thread per query row (= TMEM lane): the
//                 whole 128-column S row is read ONCE into registers (setmaxnreg gives these warps 208 registers),
//                 row max, exp2 with the softmax scale folded in, P written as packed bf16.
//                 The maximum is updated lazily (only when a row outgrows 2^8 of head-room), so the accumulator
//                 in TMEM is rescaled rarely; the normalised output leaves through one TMA store per warp.
// TMEM per tile (256 columns, two tiles fill the SM's 512): S [0,128) | P [128,192) | O [192,256). P has its own
// columns instead of aliasing S (round 1), so a tile's S buffer is free again as soon as its softmax warps hold the
// row in registers: they arrive on S_EMPTY right after the TMEM loads, and the issuer puts the NEXT block's
// S = Q K^T into the buffer while the exponentials of the current block are still being computed. The softmax warps
// therefore never wait for the P.V -> Q.K round trip of the tensor core (round 1: ~1400 of ~3800 clocks per block).
// See DESIGN.md section 3.2 for the measurements behind this layout.
#pragma once
#include "attention_common.cuh"

namespace b200 {

// Every role spins on its barriers with the tightest loop, mbar_wait_plain (a bounded loop in the softmax warps costs
// 3-5 % here, same box A/B); the watchdog warp bounds them from outside.
#ifndef ATT_KV_STAGES
#define ATT_KV_STAGES 4  // blocks n .. n+2 are live in the issuer's stream (P.V of n, Q.K of n+2) + one being fetched
#endif
constexpr int ATT_TM_TILE = 256;  // TMEM columns per query tile
constexpr int ATT_TM_P = 128;     //   P (bf16 pairs) at [128, 192)
constexpr int ATT_TM_O = 192;     //   O accumulator at [192, 256)
constexpr int ATT_SMEM_Q = 0;                                   // 2 buffers x 2 tiles
constexpr int ATT_SMEM_K = 4 * ATT_TILE_BYTES;                  // ATT_KV_STAGES tiles
constexpr int ATT_SMEM_V = ATT_SMEM_K + ATT_KV_STAGES * ATT_TILE_BYTES;
constexpr int ATT_SMEM_STG = ATT_SMEM_V + ATT_KV_STAGES * ATT_TILE_BYTES;  // 8 warps, 1024-aligned
constexpr int ATT_SMEM_BAR = ATT_SMEM_STG + 8 * ATT_STG_BYTES;
constexpr float ATT_RESCALE_LOG2 = 8.0f;  // head-room of the lazily updated softmax maximum: P <= 2^8
constexpr int ATT_SMEM_BYTES = ATT_SMEM_BAR + 256;

struct AttnParams {
  int B, H, Lq, Lkv;
  int n_qp;           // ceil(Lq / 256): query-tile pairs per (batch, head)
  int n_items;        // B * H * n_qp
  float scale_log2e;  // softmax scale * log2(e)
  int causal;         // 1: key j attends only to queries i >= j (top-left aligned, as F.scaled_dot_product_attention)
  __nv_bfloat16* out; // [B, Lq, ldo] with head h at columns [64h, 64h+64)
  long long out_batch_stride;
  int ldo;
  // additive attention bias (attn_bias / attn_mask of SDPA), fp32, element strides; nullptr = none. Strides of 0
  // broadcast over batch / head; the innermost (key) stride is 1.
  const float* bias;
  long long bias_b_stride, bias_h_stride, bias_row_stride;
  long long* trace;   // debug only: (event, clock) records of CTA 0 (nullptr in production)
  unsigned int* abort_word;  // raised by the watchdog warp when the CTA stops making progress; may be nullptr
  // kOffset instantiation only (offset-causal mode, attention_common.cuh): query offsets off[b * off_stride]
  const int* off;
  int off_stride;
};

// One 128-column block of the online softmax for one query row (= one thread = one TMEM lane).
// The whole S row is pulled into registers with back-to-back tcgen05.ld (one wait), so S is read once; P goes back
// as packed bf16 for the TS MMA. n_chunks (warp-uniform) = 32-column chunks that hold valid columns; `masked`
// (warp-uniform): the block has a partial last chunk or holds the causal diagonal — columns >= lim are set to -inf
// before the maximum, after which the exponential pass needs no predicates.
// (One copy of this code on purpose: two inlined specialisations made ptxas spill the 128-register row.)
// kBias: x = s * c + bias * log2(e) is formed right after the load (bias_row points at this row's bias for the
// block's first column, n_cols = valid columns of the block) and the rest runs with c = 1.
// The row arrives in two halves (two tcgen05.ld each, one wait each) so that the maximum of the first 64 columns is
// formed while the second half is still on its way; as soon as the whole row is in registers the warp arrives on
// `bar_s_empty`: the issuer may overwrite S with the next block's scores. P is written to its own columns `tP`, which
// the previous block's P.V may still be reading: `o_parity` >= 0 names the phase of `bar_o_full` that marks its
// completion (also what a rescale of O needs), < 0 = nothing to wait for (first block of a tile).
struct SoftmaxSync {
  uint32_t bar_s_empty, bar_o_full;
  int o_parity;
  AttTrace tr;
};

// The two softmax warps of an SM sub-partition (same TMEM lane quarter, one per query tile) share one MUFU pipe.
// Left alone they fall into lockstep — both in their exponential phase, then both in their MUFU-free phases (TMEM
// load, row maximum, TMEM store, barrier round trips: ~1700 of ~3650 clocks per block in the round-2 event trace),
// during which the pipe idles. Tile 1's softmax warps therefore start ATT_SKEW_CLKS late, which keeps the two in
// anti-phase: nothing in the pipeline re-synchronises them afterwards.
#ifndef ATT_SKEW_CLKS
#define ATT_SKEW_CLKS 1500  // one-time phase offset of tile 1's softmax warps (same box: -1.5 % at L = 1370 / 1500)
#endif

template <bool kBias>
__device__ __forceinline__ void softmax_block(uint32_t tS, uint32_t tP, const SoftmaxSync sy, int n_chunks, bool masked,
                                              int lim, float c, float& m, float& l, float& alpha, bool& rescale,
                                              const float* bias_row = nullptr, int n_cols = 0) {
  uint32_t v[4][32];
  float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
  const float c_in = c;
  auto prep_max = [&](int ch) {  // bias, mask and running maximum of one 32-column chunk (ch is a literal after unrolling)
    if (kBias) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int col = ch * 32 + i;
        const float bv = col < n_cols ? __ldg(bias_row + col) : 0.0f;
        v[ch][i] = __float_as_uint(fmaf(__uint_as_float(v[ch][i]), c_in, bv * 1.4426950408889634f));
      }
    }
    if (masked) {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (ch * 32 + i >= lim) v[ch][i] = 0xff800000u;
    }
    // four chains of three-input maxima (FMNMX3: two scores per instruction): two chains of FMNMX are bound by the
    // latency of 64 dependent FMNMX (~450 clocks per block in the trace — on the critical path now that the softmax
    // warps no longer wait for the tensor core)
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
      mx0 = fmax3(mx0, __uint_as_float(v[ch][i]), __uint_as_float(v[ch][i + 1]));
      mx1 = fmax3(mx1, __uint_as_float(v[ch][i + 2]), __uint_as_float(v[ch][i + 3]));
      mx2 = fmax3(mx2, __uint_as_float(v[ch][i + 4]), __uint_as_float(v[ch][i + 5]));
      mx3 = fmax3(mx3, __uint_as_float(v[ch][i + 6]), __uint_as_float(v[ch][i + 7]));
    }
  };
  tmem_ld32(tS, v[0]);
  if (1 < n_chunks) tmem_ld32(tS + 32, v[1]);
  tmem_wait_ld();
  if (2 < n_chunks) tmem_ld32(tS + 64, v[2]);
  if (3 < n_chunks) tmem_ld32(tS + 96, v[3]);
  prep_max(0);
  if (1 < n_chunks) prep_max(1);
  tmem_wait_ld();
  tc_fence_before();
  __syncwarp();
  if (lane_id() == 0) mbar_arrive(sy.bar_s_empty);
  ATT_TR(sy.tr, 201);
  if (2 < n_chunks) prep_max(2);
  if (3 < n_chunks) prep_max(3);
  if (kBias) c = 1.0f;
  const float m_new = fmax3(m, fmaxf(mx0, mx1), fmaxf(mx2, mx3));
  // lazy rescale: only when some row of this warp gained more than ATT_RESCALE_LOG2 of head-room (always true for
  // the first block with a visible key, where m = -inf)
  rescale = __any_sync(0xffffffffu, (m_new - m) * c > ATT_RESCALE_LOG2);
  if (rescale) {
    // m = -inf, m_new finite: 0 (nothing accumulated yet). m_new = -inf (no visible key so far, additive bias only):
    // nothing to rescale — exp2(-inf - -inf) would be NaN and poison l
    alpha = m_new == -INFINITY ? 1.0f : fast_exp2((m - m_new) * c);
    m = m_new;
    l *= alpha;
  }
  // a row whose keys so far are all masked (-inf; additive bias only) keeps m = -inf: exponentials are taken against 0
  // so that P = exp2(-inf) = 0 instead of exp2(-inf + inf) = NaN
  const float m_off = m == -INFINITY ? 0.0f : m;
  const float2 c2 = make_float2(c, c);
  const float2 nmc2 = make_float2(-m_off * c, -m_off * c);
  ATT_TR(sy.tr, 202);
  float2 sum0 = make_float2(0.f, 0.f), sum1 = make_float2(0.f, 0.f);
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    if (ch < n_chunks) {
      uint32_t pk[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float2 e = __ffma2_rn(make_float2(__uint_as_float(v[ch][2 * i]), __uint_as_float(v[ch][2 * i + 1])), c2,
                                    nmc2);
#if ATT_POLY_EVERY > 0
        const float2 pr = (i % ATT_POLY_EVERY) == ATT_POLY_EVERY - 1 ? exp2_poly2(e)
                                                                     : make_float2(fast_exp2(e.x), fast_exp2(e.y));
#else
        const float2 pr = make_float2(fast_exp2(e.x), fast_exp2(e.y));
#endif
        if (i & 1) sum1 = __fadd2_rn(sum1, pr); else sum0 = __fadd2_rn(sum0, pr);
        pk[i] = pack_bf16x2(pr.x, pr.y);
      }
      if (ch == 0 && sy.o_parity >= 0) {
        // P.V of the previous block has finished: P's columns are free and O is complete. It was issued a whole
        // block ago; the wait sits here, after the first chunk's exponentials, so that its latency is covered.
        mbar_wait_plain(sy.bar_o_full, uint32_t(sy.o_parity));
        tc_fence_after();
      }
      tmem_st16(tP + ch * 16, pk);
    }
  }
  const float2 sum = __fadd2_rn(sum0, sum1);
  l += sum.x + sum.y;
  ATT_TR(sy.tr, 203);
}

// kOffset: offset-causal mode (attention_common.cuh); p.Lkv is then the cache capacity and p.causal is 1.
template <bool kBias, bool kOffset = false>
__global__ void __launch_bounds__(ATT_THREADS, 1)
attention_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                 const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + ATT_SMEM_BAR;
  // barrier slots: q_full[2], q_empty[2], s_full[2], s_empty[2], p_full[2], o_full[2], kv_full[stages], kv_empty[stages]
  auto bar = [&](int i) { return bars + 8u * i; };
  constexpr int Q_FULL = 0, Q_EMPTY = 2, S_FULL = 4, S_EMPTY = 6, P_FULL = 8, O_FULL = 10, KV_FULL = 12,
                KV_EMPTY = 12 + ATT_KV_STAGES, DONE = 12 + 2 * ATT_KV_STAGES;
  constexpr int kProtocolBarriers = DONE;  // every barrier below DONE takes part in the data-flow protocol
  static_assert(kProtocolBarriers <= 32, "the watchdog flips one protocol barrier per lane");
  static_assert(8 * (DONE + 1) + 8 <= ATT_SMEM_BYTES - ATT_SMEM_BAR, "barrier block overflows its shared memory");
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + ATT_SMEM_BAR + 8 * (DONE + 1));
  const uint32_t progress_addr = sbase + ATT_SMEM_BAR + 8 * (DONE + 1) + 4;  // blocks issued by the MMA warp (watchdog input)
  unsigned int* const abw = p.abort_word;

  // Role index, not the hardware warp id: the SM sub-partition's arbiter serves the HIGHEST warp id first (measured),
  // so the control roles (TMA producer, MMA issuer, watchdog) sit in the LAST warpgroup (hardware warps 8..11 ->
  // roles 0..3) where a handful of instructions per block are issued at once instead of queueing behind the softmax
  // warps' exponential loops; hardware warps 0..7 are the softmax warpgroups (roles 4..11). The TMEM lane quarter
  // (warp % 4) is the same in both numberings.
  const int warp = ((threadIdx.x >> 5) + 4) % 12;
  const int lane = threadIdx.x & 31;
#ifdef ATT_TRACE
  int tr_n = 0;
  const int tr_role = warp == 0 ? 0 : warp == 1 ? 1 : warp < 8 ? 2 : 3;
#endif

  if (sbase & 1023u) {  // the 128B swizzle needs 1024-aligned tiles: report through the status word, never trap
    if (threadIdx.x == 0 && abw != nullptr) *reinterpret_cast<volatile unsigned int*>(abw) = 0xB200A117u;
    return;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(Q_FULL + i), 1);
      mbar_init(bar(Q_EMPTY + i), 1);
      mbar_init(bar(S_FULL + i), 1);
      mbar_init(bar(S_EMPTY + i), 4);
      mbar_init(bar(P_FULL + i), 4);
      mbar_init(bar(O_FULL + i), 1);
    }
    for (int s = 0; s < ATT_KV_STAGES; ++s) {
      mbar_init(bar(KV_FULL + s), 1);
      mbar_init(bar(KV_EMPTY + s), 1);
    }
    mbar_init(bar(DONE), 10);  // producer, MMA issuer and the eight softmax warps arrive when they run out of work
    sts_u32_volatile(progress_addr, 0u);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmO);
  }
  if (warp == 1) {
    tmem_alloc<512>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch_dependents();  // (ptx.cuh: programmatic dependent launch; nothing above touched global memory)
  griddep_wait();
  const int n_kvb = (p.Lkv + ATT_BKV - 1) / ATT_BKV;
  // K/V blocks a query tile has to visit: all of them, or with a causal mask only those up to its last row's diagonal
  auto tile_blocks = [&](int item, int t) {
    const int row0 = (item % p.n_qp) * 256 + t * ATT_BQ;
    if (row0 >= p.Lq) return 0;
    if (kOffset) {
      const int o = att_seq_offset(p.off, p.off_stride, item / p.n_qp / p.H, p.Lq, p.Lkv).off;
      return min(o + p.Lq - 1, o + row0 + ATT_BQ - 1) / ATT_BKV + 1;
    }
    if (!p.causal) return n_kvb;
    return min(p.Lkv - 1, row0 + ATT_BQ - 1) / ATT_BKV + 1;
  };
  auto item_blocks = [&](int item) { return max(tile_blocks(item, 0), tile_blocks(item, 1)); };

  if (warp < 4) setmaxnreg_dec<ATT_CONTROL_REGS>();  // whole warpgroup 0 (the two idle warps included)
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (whole warp converged, one lane issues)
    uint32_t it = 0, stage = 0, phase = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
      const int qp = item % p.n_qp;
      const int bh = item / p.n_qp;
      const int h = bh % p.H;
      const int b = bh / p.H;
      const bool two = qp * 256 + ATT_BQ < p.Lq;  // second query tile has at least one valid row
      const uint32_t qb = it & 1u;
      mbar_wait_plain(bar(Q_EMPTY + qb), ((it >> 1) & 1u) ^ 1u);
      if (elect_one()) {
        mbar_expect_tx(bar(Q_FULL + qb), (two ? 2 : 1) * ATT_TILE_BYTES);
        const uint32_t sq = sbase + ATT_SMEM_Q + qb * 2 * ATT_TILE_BYTES;
        tma_load_3d(&tmQ, bar(Q_FULL + qb), sq, h * ATT_HD, qp * 256, b);
        if (two) tma_load_3d(&tmQ, bar(Q_FULL + qb), sq + ATT_TILE_BYTES, h * ATT_HD, qp * 256 + ATT_BQ, b);
      }
      __syncwarp();
      const int nb = item_blocks(item);
      for (int j = 0; j < nb; ++j) {
        mbar_wait_plain(bar(KV_EMPTY + stage), phase ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(bar(KV_FULL + stage), 2 * ATT_TILE_BYTES);
          tma_load_3d(&tmK, bar(KV_FULL + stage), sbase + ATT_SMEM_K + stage * ATT_TILE_BYTES, h * ATT_HD, j * ATT_BKV, b);
          tma_load_3d(&tmV, bar(KV_FULL + stage), sbase + ATT_SMEM_V + stage * ATT_TILE_BYTES, h * ATT_HD, j * ATT_BKV, b);
        }
        __syncwarp();
        if (++stage == ATT_KV_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
    if (lane == 0) mbar_arrive(bar(DONE));
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp converged, one lane issues)
    {
      // The (item, kv-block) sequence of this CTA is walked as ONE stream of blocks n = 0, 1, 2, ...: while block n is
      // being finished (P.V of both tiles) the scores of block n+2 — possibly of the next item — are issued into the
      // S buffers that the softmax warps released when they pulled block n+1 into registers. Per tile the order is
      // QK(n+1) PV(n) QK(n+2) PV(n+1) ..., each waiting on an event of that tile's softmax warps in the order in which
      // they occur (S_EMPTY(n+1) before P_FULL(n+1)), so the stream never waits on something that needs a later MMA.
      uint32_t blocks_done = 0;
      uint32_t nqk[2] = {0, 0};  // score MMAs issued so far per tile (S_EMPTY parity)
      uint32_t npv[2] = {0, 0};  // P.V MMAs issued so far per tile (P_FULL parity)
      const uint32_t idesc_o = make_idesc_bf16(ATT_BQ, ATT_HD, 0, 1);
      struct Blk {
        int item, j;
        uint32_t it, stage, phase;
        int nb0, nb1;  // blocks visited by query tile 0 / 1 of this item (0 = tile absent)
        int kv;        // kOffset: keys of the item's sequence (offset + Lq)
      };
      auto active = [&](const Blk& bl, int t) { return bl.j < (t == 0 ? bl.nb0 : bl.nb1); };
      auto set_item = [&](Blk& bl) {
        bl.nb0 = bl.item < p.n_items ? tile_blocks(bl.item, 0) : 0;
        bl.nb1 = bl.item < p.n_items ? tile_blocks(bl.item, 1) : 0;
        if (kOffset && bl.item < p.n_items)
          bl.kv = att_seq_offset(p.off, p.off_stride, bl.item / p.n_qp / p.H, p.Lq, p.Lkv).off + p.Lq;
      };
      auto n_mma_of = [&](const Blk& bl) { return (min(ATT_BKV, (kOffset ? bl.kv : p.Lkv) - bl.j * ATT_BKV) + 15) & ~15; };
      auto issue_qk = [&](const Blk& bl, int t) {
        if (nqk[t] > 0) {  // the softmax warps of this tile hold the previous scores in registers
          mbar_wait_plain(bar(S_EMPTY + t), (nqk[t] - 1) & 1u);
          tc_fence_after();
        }
        const uint32_t sq = sbase + ATT_SMEM_Q + (bl.it & 1u) * 2 * ATT_TILE_BYTES + t * ATT_TILE_BYTES;
        const uint64_t dq = make_smem_desc_sw128(sq, 16, 1024);
        const uint64_t dk = make_smem_desc_sw128(sbase + ATT_SMEM_K + bl.stage * ATT_TILE_BYTES, 16, 1024);
        const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, n_mma_of(bl), 0, 0);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < ATT_HD / 16; ++k)
            umma_ss(tmem_base + t * ATT_TM_TILE, dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          umma_commit(bar(S_FULL + t));
        }
        __syncwarp();
        ++nqk[t];
        if (lane == 0) ATT_EV(100 + t);
      };
      // wait for the operands of a block (and, for the first block of an item, its Q tiles), then issue its scores
      auto start_block = [&](const Blk& bl) {
        if (bl.j == 0) mbar_wait_plain(bar(Q_FULL + (bl.it & 1u)), (bl.it >> 1) & 1u);
        mbar_wait_plain(bar(KV_FULL + bl.stage), bl.phase);
        if (lane == 0) ATT_EV(130);
        tc_fence_after();
        for (int t = 0; t <= 1; ++t)
          if (active(bl, t)) issue_qk(bl, t);
        // after the last score MMA that reads this item's Q tiles has been issued, hand the Q buffer back
        if (bl.j == max(bl.nb0, bl.nb1) - 1) {
          if (elect_one()) umma_commit(bar(Q_EMPTY + (bl.it & 1u)));
          __syncwarp();
        }
      };
      auto advance = [&](Blk bl) {
        if (++bl.stage == ATT_KV_STAGES) {
          bl.stage = 0;
          bl.phase ^= 1u;
        }
        if (++bl.j == max(bl.nb0, bl.nb1)) {
          bl.j = 0;
          bl.item += gridDim.x;
          ++bl.it;
          set_item(bl);
        }
        return bl;
      };

      Blk cur{int(blockIdx.x), 0, 0u, 0u, 0u, 0, 0, p.Lkv};
      // Lean issue loop (round 2, second session). The event trace showed that this warp, not the softmax warps, set
      // the period: ~1000 clocks of its own serial work per (tile, block) around ~600 clocks of tcgen05.mma issue.
      // Here everything that does not depend on the softmax warps (operand barriers of block n+2, descriptors) happens
      // BEFORE the P_FULL wait; per block there are three elected regions: P.V(n) of tile 0, P.V(n) of tile 1, and the
      // score MMAs of block n+2 for both tiles together with every commit of the block.
      // P.V of both tiles first: a tile that has published its probabilities (in particular its last ones: the item's
      // epilogue waits for this P.V) is never queued behind the other tile's S_EMPTY, which at an item boundary only
      // comes after that tile's epilogue. The scores of block n+2 are not needed before the softmax warps finish block
      // n+1, a whole block from now.
      if (cur.item < p.n_items) {
        set_item(cur);
        start_block(cur);
        Blk nx1 = advance(cur);
        bool have1 = nx1.item < p.n_items;
        if (have1) start_block(nx1);
        while (true) {
          Blk nx2 = nx1;
          bool have2 = false;
          if (have1) {
            nx2 = advance(nx1);
            have2 = nx2.item < p.n_items;
          }
          if (have2) {  // loaded long ago (4-stage ring): off the critical path
            if (nx2.j == 0) mbar_wait_plain(bar(Q_FULL + (nx2.it & 1u)), (nx2.it >> 1) & 1u);
            mbar_wait_plain(bar(KV_FULL + nx2.stage), nx2.phase);
          }
          // per K step only immediates change: V is MN-major (head_dim contiguous), 16 kv rows = 2048 bytes (+128 in
          // the descriptor); P: 8 TMEM columns
          const uint64_t dv0 = make_smem_desc_sw128(sbase + ATT_SMEM_V + cur.stage * ATT_TILE_BYTES, 16, 1024);
          const uint64_t dk0 = make_smem_desc_sw128(sbase + ATT_SMEM_K + nx2.stage * ATT_TILE_BYTES, 16, 1024);
          const uint32_t sq_n = sbase + ATT_SMEM_Q + (nx2.it & 1u) * 2 * ATT_TILE_BYTES;
          const uint64_t dq0 = make_smem_desc_sw128(sq_n, 16, 1024);
          const uint64_t dq1 = make_smem_desc_sw128(sq_n + ATT_TILE_BYTES, 16, 1024);
          const int ksteps = n_mma_of(cur) / 16;
          const uint32_t acc0 = cur.j > 0 ? 1u : 0u;
          const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, have2 ? n_mma_of(nx2) : ATT_BKV, 0, 0);
          if (kOffset) {  // V rows past the sequence's keys inside the last P.V K-step (see att_zero_rows)
            const int keys = cur.kv - cur.j * ATT_BKV;
            if (keys < ATT_BKV && (keys & 15) != 0)
              att_zero_rows(sbase + ATT_SMEM_V + cur.stage * ATT_TILE_BYTES, keys, (keys + 15) & ~15);
          }
          const bool q_done = have2 && nx2.j == max(nx2.nb0, nx2.nb1) - 1;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            if (!active(cur, t)) continue;
            const uint32_t tT = tmem_base + t * ATT_TM_TILE;
            mbar_wait_plain(bar(P_FULL + t), npv[t] & 1u);
            if (lane == 0) ATT_EV(110 + t);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < ATT_BKV / 16; ++k)
                if (k < ksteps) umma_ts(tT + ATT_TM_O, tT + ATT_TM_P + 8u * k, dv0 + 128u * k, idesc_o, k != 0 ? 1u : acc0);
              umma_commit(bar(O_FULL + t));
            }
            __syncwarp();
            if (lane == 0) ATT_EV(120 + t);
            ++npv[t];
          }
          const bool qk0 = have2 && active(nx2, 0), qk1 = have2 && active(nx2, 1);
          if (qk0 && nqk[0] > 0) mbar_wait_plain(bar(S_EMPTY + 0), (nqk[0] - 1) & 1u);
          if (qk1 && nqk[1] > 0) mbar_wait_plain(bar(S_EMPTY + 1), (nqk[1] - 1) & 1u);
          tc_fence_after();
          if (elect_one()) {
            if (qk0) {
#pragma unroll
              for (int k = 0; k < ATT_HD / 16; ++k) umma_ss(tmem_base, dq0 + 2u * k, dk0 + 2u * k, idesc_s, k != 0 ? 1u : 0u);
              umma_commit(bar(S_FULL + 0));
            }
            if (qk1) {
#pragma unroll
              for (int k = 0; k < ATT_HD / 16; ++k)
                umma_ss(tmem_base + ATT_TM_TILE, dq1 + 2u * k, dk0 + 2u * k, idesc_s, k != 0 ? 1u : 0u);
              umma_commit(bar(S_FULL + 1));
            }
            if (q_done) umma_commit(bar(Q_EMPTY + (nx2.it & 1u)));
            umma_commit(bar(KV_EMPTY + cur.stage));  // free once everything issued so far completes
          }
          __syncwarp();
          if (lane == 0) ATT_EV(100);
          if (qk0) ++nqk[0];
          if (qk1) ++nqk[1];
          if (lane == 0) sts_u32_volatile(progress_addr, ++blocks_done);  // the watchdog's sign of life
          if (!have1) break;
          cur = nx1;
          nx1 = nx2;
          have1 = have2;
        }
      }
      if (lane == 0) mbar_arrive(bar(DONE));
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------ watchdog (input: the issuer's block counter)
    if (abw != nullptr) {
      uint32_t last = 0xFFFFFFFFu;
      uint64_t t_last = 0;
      bool raised = false;
      while (!mbar_try_wait_hint(bar(DONE), 0u, 20000u)) {
        const uint64_t now = global_timer_ns();
        const uint32_t pr = lds_u32_volatile(progress_addr);
        if (pr != last || t_last == 0) {
          last = pr;
          t_last = now;
        } else if (now - t_last > B200_WAIT_LIMIT_NS) {
          if (!raised && lane == 0) {
            *reinterpret_cast<volatile unsigned int*>(abw) = 0xB200DEADu;
            __threadfence_system();
          }
          raised = true;
          if (lane < kProtocolBarriers) {
#pragma unroll 1
            for (int k = 0; k < 4; ++k) mbar_arrive(bar(lane));
          }
          __nanosleep(2000);
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ softmax / output warpgroups
    setmaxnreg_inc<ATT_SOFTMAX_REGS>();  // a whole S row (128 fp32) lives in registers
    const int t = (warp - 4) >> 2;  // query tile of this warpgroup
    const int qd = warp & 3;        // TMEM lane quarter
    const int r = qd * 32 + lane;   // row inside the tile == TMEM lane
    const uint32_t lane_off = uint32_t(qd * 32) << 16;
    const uint32_t tS = tmem_base + t * ATT_TM_TILE + lane_off;
    const uint32_t tP = tS + ATT_TM_P;
    const uint32_t tO = tS + ATT_TM_O;
    const float c = p.scale_log2e;
    const uint32_t stg = sbase + ATT_SMEM_STG + uint32_t(warp - 4) * ATT_STG_BYTES;  // this warp's 32 x 128 B staging
    uint32_t g = 0;  // blocks processed so far by this tile
#if ATT_SKEW_CLKS > 0
    // One-time phase offset between the two tiles' softmax warps: left alone they run in lockstep (both in the
    // exponential phase, then both in the ALU-bound maximum / TMEM phases), so the MUFU pipe idles ~1/3 of the time.
    // Nothing in the pipeline re-synchronises them afterwards (S is produced a block ahead).
    if (t == 1) {
      const long long t0 = clock64();
      while (clock64() - t0 < ATT_SKEW_CLKS) {
      }
    }
#endif
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const int qp = item % p.n_qp;
      const int bh = item / p.n_qp;
      const int h = bh % p.H;
      const int b = bh / p.H;
      const int row0 = qp * 256 + t * ATT_BQ;
      const int nb = tile_blocks(item, t);
      if (nb == 0) continue;                              // tile not scheduled at all (same rule as the MMA warp)
      const bool warp_live = row0 + qd * 32 < p.Lq;       // any valid row in this warp?
      const int qrow = row0 + r;
      // kOffset: query row i is at position q_off + i, the sequence has kv_len keys
      const AttOffset so = kOffset ? att_seq_offset(p.off, p.off_stride, b, p.Lq, p.Lkv) : AttOffset{0, false};
      const int q_off = so.off;
      const int kv_len = kOffset ? q_off + p.Lq : p.Lkv;
      // m: the maximum the exponentials are taken against. It trails the true running maximum by at most
      // ATT_RESCALE_LOG2 (in the log2 domain), so P <= 2^ATT_RESCALE_LOG2 and the accumulator in TMEM is rescaled
      // only when some row of the warp outgrows that head-room (rare after the first block).
      float m = -INFINITY, l = 0.0f;

      for (int j = 0; j < nb; ++j, ++g) {
        const int nvalid = min(ATT_BKV, kv_len - j * ATT_BKV);
        // columns of this block this row may attend to: all valid ones, or up to the diagonal with a causal mask
        const bool diag = p.causal && j * ATT_BKV + ATT_BKV - 1 > row0 + q_off;  // warp-uniform
        const int lim = diag ? min(nvalid, qrow + q_off - j * ATT_BKV + 1) : nvalid;
        mbar_wait_plain(bar(S_FULL + t), g & 1u);
        if (lane == 0 && qd == 2) ATT_EV(200 + t);
        tc_fence_after();
        float alpha = 1.0f;
        bool rescale = false;
        // P.V(j-1) of this tile must have completed before P(j) is written over P(j-1) (and before O is rescaled).
        // O_FULL cannot be lapped: its next flip needs this warp's P_FULL arrive below.
#ifdef ATT_TRACE
        const SoftmaxSync sy{bar(S_EMPTY + t), bar(O_FULL + t), j > 0 ? int((g - 1) & 1u) : -1,
                             AttTrace{p.trace, tr_role, &tr_n, lane == 0 && qd == 2}};
#else
        const SoftmaxSync sy{bar(S_EMPTY + t), bar(O_FULL + t), j > 0 ? int((g - 1) & 1u) : -1, AttTrace{}};
#endif
        if (warp_live) {
          const bool masked = diag || (nvalid & 31) != 0;
          if (kBias) {
            const float* brow = p.bias + (long long)b * p.bias_b_stride + (long long)h * p.bias_h_stride +
                                (long long)min(qrow, p.Lq - 1) * p.bias_row_stride + j * ATT_BKV;
            softmax_block<true>(tS, tP, sy, (nvalid + 31) >> 5, masked, lim, c, m, l, alpha, rescale, brow, nvalid);
          } else {
            softmax_block<false>(tS, tP, sy, (nvalid + 31) >> 5, masked, lim, c, m, l, alpha, rescale);
          }
          if (j > 0 && rescale) {  // warp-uniform; P.V(j-1) has landed (softmax_block waited for it)
            uint32_t o0[32], o1[32];
            tmem_ld32(tO, o0);
            tmem_ld32(tO + 32, o1);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              o0[i] = __float_as_uint(__uint_as_float(o0[i]) * alpha);
              o1[i] = __float_as_uint(__uint_as_float(o1[i]) * alpha);
            }
            tmem_st32(tO, o0);
            tmem_st32(tO + 32, o1);
          }
        } else {
          // rows past Lq: nothing to compute, but the protocol is the same (release S, then publish an unused P)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(sy.bar_s_empty);
          if (sy.o_parity >= 0) mbar_wait_plain(sy.bar_o_full, uint32_t(sy.o_parity));
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(P_FULL + t));
        if (lane == 0 && qd == 2) ATT_EV(210 + t);
      }
      mbar_wait_plain(bar(O_FULL + t), (g - 1) & 1u);  // cannot be lapped: the next flip needs this warp's next P_FULL arrive
      tc_fence_after();
      if (lane == 0 && qd == 2) ATT_EV(220 + t);
      // normalise the 64 output columns of this head and hand the warp's 32 rows to one TMA store (rows >= Lq are
      // clipped by the tensor map)
      if (warp_live) {
        uint32_t o0[32], o1[32];
        tmem_ld32(tO, o0);
        tmem_ld32(tO + 32, o1);
        if (elect_one()) tma_store_wait_read<0>();  // the previous item's store has finished reading the staging
        __syncwarp();
        tmem_wait_ld();
        const float inv = kOffset && so.bad ? __int_as_float(0x7fc00000) : 1.0f / l;
        uint8_t* dst = smem + ATT_SMEM_STG + (warp - 4) * ATT_STG_BYTES + lane * 128;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          uint4 w;
          if (i < 4) {
            w.x = pack_bf16x2(__uint_as_float(o0[8 * i + 0]) * inv, __uint_as_float(o0[8 * i + 1]) * inv);
            w.y = pack_bf16x2(__uint_as_float(o0[8 * i + 2]) * inv, __uint_as_float(o0[8 * i + 3]) * inv);
            w.z = pack_bf16x2(__uint_as_float(o0[8 * i + 4]) * inv, __uint_as_float(o0[8 * i + 5]) * inv);
            w.w = pack_bf16x2(__uint_as_float(o0[8 * i + 6]) * inv, __uint_as_float(o0[8 * i + 7]) * inv);
          } else {
            w.x = pack_bf16x2(__uint_as_float(o1[8 * i - 32]) * inv, __uint_as_float(o1[8 * i - 31]) * inv);
            w.y = pack_bf16x2(__uint_as_float(o1[8 * i - 30]) * inv, __uint_as_float(o1[8 * i - 29]) * inv);
            w.z = pack_bf16x2(__uint_as_float(o1[8 * i - 28]) * inv, __uint_as_float(o1[8 * i - 27]) * inv);
            w.w = pack_bf16x2(__uint_as_float(o1[8 * i - 26]) * inv, __uint_as_float(o1[8 * i - 25]) * inv);
          }
          *reinterpret_cast<uint4*>(dst + ((i ^ (lane & 7)) << 4)) = w;  // 128B swizzle of the store's tensor map
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (elect_one()) {  // bulk groups are per thread: elect.sync picks the same lane of a full warp every time
          tma_store_3d(&tmO, stg, h * ATT_HD, row0 + qd * 32, b);
          tma_store_commit();
        }
        __syncwarp();
      }
      tc_fence_before();  // the TMEM reads above are ordered before this warp's next P_FULL arrive
      if (lane == 0 && qd == 2) ATT_EV(230 + t);
    }
    if (elect_one()) tma_store_wait_all<0>();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(DONE));
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace b200
