// Flash-style attention for head_dim 80, 96, 112 and 128 on sm_100a (every multiple of 16 above 64 up to 128), with
// every mode of the head_dim-64 kernels: self / cross attention, any Lq and Lkv, causal, additive bias, causal + bias.
// Reference: F.scaled_dot_product_attention at pytorch_models/transformer.py:52.
//
// Derived from the round-1 streaming kernel (DESIGN.md section 3.2.0), whose TMEM layout writes P back over S: a
// query tile needs S 128 | O head_dim columns, at most 256, so the two tiles of a work item still fit in the SM's
// 512 columns. The layout of the head_dim-64 streaming kernel (S 128 | P 64 | O 64) has no room for a wider O.
//
// One work item = (batch, head, pair of 128-row query tiles). One persistent CTA per SM loops over items; key/value
// rows stream through a 2-stage TMA ring in blocks of 128 with an online softmax. 384 threads, roles as in
// attention_common.cuh:
//   warp 0      : TMA producer (Q pair, single-buffered; K/V blocks)
//   warp 1      : tcgen05.mma issuer, one stream across items in the order  PV0(j) QK0(j+1) PV1(j) QK1(j+1)
//                   S_t = Q_t K_j^T          -> TMEM, fp32, 128 columns per tile, head_dim/16 K steps
//                   O_t (+)= P_t V_j         -> TMEM, head_dim columns (N = head_dim), P_t (over S_t) the A operand
//   warp 2      : watchdog (see attention_common.cuh), warp 3 : idle
//   warps 4..7  : softmax warpgroup of tile 0, warps 8..11 : tile 1. One thread per query row (= TMEM lane): the
//                 whole 128-column S row is read once into registers, row max, exp2 with the softmax scale folded in,
//                 P written back over S as packed bf16. The maximum is updated lazily (only when a row outgrows 2^8 of
//                 head-room), so O is rescaled rarely; the normalised output leaves through two TMA stores per warp.
//
// Operands: Q, K, V and O are 4-D tensor maps (head_dim columns, H heads, L rows, B). A 128-row tile is two
// 64-column boxes with 128B swizzle, 16 KB each; the columns >= head_dim of the second box lie outside dimension 0,
// so TMA fills them with zeros on load (no HBM traffic) and clips them on store.
// Shared memory (the same for every head_dim): Q pair 64 KB | 2 K/V stages 128 KB | output staging 8 x 4 KB.
#pragma once
#include "attention_common.cuh"

namespace b200 {

constexpr int ATW_MAX_HD = 128;
constexpr int ATW_BOX_BYTES = ATT_TILE_BYTES;        // 16 KB: 128 rows x 64 bf16 columns, 128B-swizzled
constexpr int ATW_TILE_BYTES = 2 * ATW_BOX_BYTES;    // one 128-row tile of up to 128 columns: two boxes
constexpr int ATW_KV_STAGES = 2;
constexpr int ATW_SMEM_Q = 0;                                             // 2 tiles (single-buffered)
constexpr int ATW_SMEM_K = 2 * ATW_TILE_BYTES;                            // ATW_KV_STAGES tiles
constexpr int ATW_SMEM_V = ATW_SMEM_K + ATW_KV_STAGES * ATW_TILE_BYTES;
constexpr int ATW_SMEM_STG = ATW_SMEM_V + ATW_KV_STAGES * ATW_TILE_BYTES;  // 8 warps x 32 rows x 64 columns
constexpr int ATW_SMEM_BAR = ATW_SMEM_STG + 8 * ATT_STG_BYTES;
constexpr int ATW_SMEM_BYTES = ATW_SMEM_BAR + 256;
static_assert(ATW_SMEM_BYTES <= 227 * 1024, "wide attention kernel exceeds the shared memory of a CTA");
constexpr int ATW_TM_O = 128;             // per tile: S (P over its first 64 columns) [0, 128), O [128, 128 + head_dim)
constexpr float ATW_RESCALE_LOG2 = 8.0f;  // head-room of the lazily updated softmax maximum: P <= 2^8

struct AttnWideParams {
  int B, H, Lq, Lkv;
  int head_dim;       // 80, 96, 112 or 128
  int n_qp;           // ceil(Lq / 256): query-tile pairs per (batch, head)
  int n_items;        // B * H * n_qp
  float scale_log2e;  // softmax scale * log2(e)
  int causal;         // 1: key j attends only to queries i >= j (top-left aligned, as F.scaled_dot_product_attention)
  // additive attention bias (attn_bias / attn_mask of SDPA), fp32, element strides; nullptr = none. Strides of 0
  // broadcast over batch / head; the innermost (key) stride is 1.
  const float* bias;
  long long bias_b_stride, bias_h_stride, bias_row_stride;
  unsigned int* abort_word;  // raised by the watchdog warp when the CTA stops making progress; may be nullptr
  // kOffset instantiation only (offset-causal mode, attention_common.cuh): query offsets off[b * off_stride]
  const int* off;
  int off_stride;
};

// One 128-column block of the online softmax for one query row (= one thread = one TMEM lane). The whole S row is
// pulled into registers with back-to-back tcgen05.ld (one wait); P goes back over the same TMEM columns as packed
// bf16 for the TS MMA. n_chunks (warp-uniform) = 32-column chunks that hold valid columns; `masked` (warp-uniform):
// the block has a partial last chunk or holds the causal diagonal — columns >= lim are set to -inf before the
// maximum, after which the exponential pass needs no predicates.
// kBias: x = s * c + bias * log2(e) is formed right after the load (bias_row points at this row's bias for the
// block's first column, n_cols = valid columns of the block) and the rest runs with c = 1.
template <bool kBias>
__device__ __forceinline__ void softmax_block_wide(uint32_t tS, int n_chunks, bool masked, int lim, float c, float& m,
                                                   float& l, float& alpha, bool& rescale,
                                                   const float* bias_row = nullptr, int n_cols = 0) {
  uint32_t v[4][32];
#pragma unroll
  for (int ch = 0; ch < 4; ++ch)
    if (ch < n_chunks) tmem_ld32(tS + ch * 32, v[ch]);
  tmem_wait_ld();
  if (kBias) {
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      if (ch < n_chunks) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int col = ch * 32 + i;
          const float bv = col < n_cols ? __ldg(bias_row + col) : 0.0f;
          v[ch][i] = __float_as_uint(fmaf(__uint_as_float(v[ch][i]), c, bv * 1.4426950408889634f));
        }
      }
    }
    c = 1.0f;
  }
  if (masked) {
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (ch * 32 + i >= lim) v[ch][i] = 0xff800000u;
  }
  // four chains of three-input maxima (FMNMX3: two scores per instruction)
  float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    if (ch < n_chunks) {
#pragma unroll
      for (int i = 0; i < 32; i += 8) {
        mx0 = fmax3(mx0, __uint_as_float(v[ch][i]), __uint_as_float(v[ch][i + 1]));
        mx1 = fmax3(mx1, __uint_as_float(v[ch][i + 2]), __uint_as_float(v[ch][i + 3]));
        mx2 = fmax3(mx2, __uint_as_float(v[ch][i + 4]), __uint_as_float(v[ch][i + 5]));
        mx3 = fmax3(mx3, __uint_as_float(v[ch][i + 6]), __uint_as_float(v[ch][i + 7]));
      }
    }
  }
  const float m_new = fmax3(m, fmaxf(mx0, mx1), fmaxf(mx2, mx3));
  // lazy rescale: only when some row of this warp gained more than ATW_RESCALE_LOG2 of head-room (always true for
  // the first block with a visible key, where m = -inf)
  rescale = __any_sync(0xffffffffu, (m_new - m) * c > ATW_RESCALE_LOG2);
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
      tmem_st16(tS + ch * 16, pk);
    }
  }
  const float2 sum = __fadd2_rn(sum0, sum1);
  l += sum.x + sum.y;
}

// kOffset: offset-causal mode (attention_common.cuh); p.Lkv is then the cache capacity and p.causal is 1.
template <bool kBias, bool kOffset = false>
__global__ void __launch_bounds__(ATT_THREADS, 1)
attention_wide_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                      const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                      const AttnWideParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + ATW_SMEM_BAR;
  // barrier slots: q_full, q_empty, kv_full[stages], kv_empty[stages], s_full[2], p_full[2], o_full[2], done
  auto bar = [&](int i) { return bars + 8u * i; };
  constexpr int Q_FULL = 0, Q_EMPTY = 1, KV_FULL = 2, KV_EMPTY = 2 + ATW_KV_STAGES, S_FULL = 2 + 2 * ATW_KV_STAGES,
                P_FULL = S_FULL + 2, O_FULL = S_FULL + 4, DONE = S_FULL + 6;
  constexpr int kProtocolBarriers = DONE;  // every barrier below DONE takes part in the data-flow protocol
  static_assert(kProtocolBarriers <= 32, "the watchdog flips one protocol barrier per lane");
  static_assert(8 * (DONE + 1) + 8 <= ATW_SMEM_BYTES - ATW_SMEM_BAR, "barrier block overflows its shared memory");
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + ATW_SMEM_BAR + 8 * (DONE + 1));
  const uint32_t progress_addr = sbase + ATW_SMEM_BAR + 8 * (DONE + 1) + 4;  // blocks issued by the MMA warp
  unsigned int* const abw = p.abort_word;

  // role index: the control roles sit in the last hardware warpgroup (see attention_stream.cuh)
  const int warp = ((threadIdx.x >> 5) + 4) % 12;
  const int lane = threadIdx.x & 31;
  const int hd = p.head_dim;

  if (sbase & 1023u) {  // the 128B swizzle needs 1024-aligned tiles: report through the status word, never trap
    if (threadIdx.x == 0 && abw != nullptr) *reinterpret_cast<volatile unsigned int*>(abw) = 0xB200A117u;
    return;
  }
  if (threadIdx.x == 0) {
    mbar_init(bar(Q_FULL), 1);
    mbar_init(bar(Q_EMPTY), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(S_FULL + i), 1);
      mbar_init(bar(P_FULL + i), 4);
      mbar_init(bar(O_FULL + i), 1);
    }
    for (int s = 0; s < ATW_KV_STAGES; ++s) {
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
      mbar_wait_plain(bar(Q_EMPTY), (it & 1u) ^ 1u);
      if (elect_one()) {
        mbar_expect_tx(bar(Q_FULL), (two ? 2 : 1) * ATW_TILE_BYTES);
        for (int t = 0; t < (two ? 2 : 1); ++t)
          for (int x = 0; x < 2; ++x)
            tma_load_4d(&tmQ, bar(Q_FULL), sbase + ATW_SMEM_Q + t * ATW_TILE_BYTES + x * ATW_BOX_BYTES, x * 64, h,
                        qp * 256 + t * ATT_BQ, b);
      }
      __syncwarp();
      const int nb = item_blocks(item);
      for (int j = 0; j < nb; ++j) {
        mbar_wait_plain(bar(KV_EMPTY + stage), phase ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(bar(KV_FULL + stage), 2 * ATW_TILE_BYTES);
          for (int x = 0; x < 2; ++x) {
            tma_load_4d(&tmK, bar(KV_FULL + stage), sbase + ATW_SMEM_K + stage * ATW_TILE_BYTES + x * ATW_BOX_BYTES,
                        x * 64, h, j * ATT_BKV, b);
            tma_load_4d(&tmV, bar(KV_FULL + stage), sbase + ATW_SMEM_V + stage * ATW_TILE_BYTES + x * ATW_BOX_BYTES,
                        x * 64, h, j * ATT_BKV, b);
          }
        }
        __syncwarp();
        if (++stage == ATW_KV_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
    if (lane == 0) mbar_arrive(bar(DONE));
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp converged, one lane issues)
    // The (item, kv-block) sequence of this CTA is walked as ONE stream: while block `cur` is being finished (P.V of
    // both tiles) the score MMAs of the following block `nxt` — possibly the first block of the next item — go out
    // right behind the same tile's P.V (they overwrite the S columns that P.V reads; the tensor core runs a thread's
    // MMAs in issue order). Everything that does not depend on P is done before the P_FULL wait.
    uint32_t g[2] = {0, 0};  // blocks issued so far per tile (P_FULL parity)
    uint32_t blocks_done = 0;
    // P.V: N = head_dim spans both 64-column boxes of V; V is MN-major, so the descriptor's leading byte offset is the
    // distance between the boxes (16 KB) and a K step of 16 kv rows is 2048 bytes (+128 in the descriptor)
    const uint32_t idesc_o = make_idesc_bf16(ATT_BQ, hd, 0, 1);
    const int qk_steps = hd / 16;
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
    auto advance = [&](Blk bl) {
      if (++bl.stage == ATW_KV_STAGES) {
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
    // Q.K of one tile: K step k reads columns [16k, 16k+16) of Q and K, from the second box (+16 KB = +1024 in the
    // descriptor) from k = 4 on
    auto issue_qk = [&](uint32_t d_tmem, uint64_t dq, uint64_t dk, uint32_t idesc_s) {
#pragma unroll
      for (int k = 0; k < ATW_MAX_HD / 16; ++k) {
        const uint32_t off = 2u * (k & 3) + (k >= 4 ? uint32_t(ATW_BOX_BYTES >> 4) : 0u);
        if (k < qk_steps) umma_ss(d_tmem, dq + off, dk + off, idesc_s, k != 0 ? 1u : 0u);
      }
    };

    Blk cur{int(blockIdx.x), 0, 0u, 0u, 0u, 0, 0, p.Lkv};
    if (cur.item < p.n_items) {
      set_item(cur);
      // scores of the first block
      mbar_wait_plain(bar(Q_FULL), 0u);
      mbar_wait_plain(bar(KV_FULL), 0u);
      tc_fence_after();
      {
        const uint64_t dk0 = make_smem_desc_sw128(sbase + ATW_SMEM_K, 16, 1024);
        const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, n_mma_of(cur), 0, 0);
        if (elect_one()) {
          for (int t = 0; t < 2; ++t) {
            if (!active(cur, t)) continue;
            issue_qk(tmem_base + t * 256, make_smem_desc_sw128(sbase + ATW_SMEM_Q + t * ATW_TILE_BYTES, 16, 1024), dk0,
                     idesc_s);
            umma_commit(bar(S_FULL + t));
          }
          if (max(cur.nb0, cur.nb1) == 1) umma_commit(bar(Q_EMPTY));
        }
        __syncwarp();
      }
      while (true) {
        const Blk nxt = advance(cur);
        const bool more = nxt.item < p.n_items;
        if (more) {  // operands of the next block; its Q only after the previous item's last scores released the buffer
          if (nxt.j == 0) mbar_wait_plain(bar(Q_FULL), nxt.it & 1u);
          mbar_wait_plain(bar(KV_FULL + nxt.stage), nxt.phase);
        }
        const uint64_t dv0 = make_smem_desc_sw128(sbase + ATW_SMEM_V + cur.stage * ATW_TILE_BYTES, ATW_BOX_BYTES, 1024);
        const uint64_t dk0 = make_smem_desc_sw128(sbase + ATW_SMEM_K + nxt.stage * ATW_TILE_BYTES, 16, 1024);
        const int ksteps = n_mma_of(cur) / 16;
        const uint32_t acc0 = cur.j > 0 ? 1u : 0u;
        const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, more ? n_mma_of(nxt) : ATT_BKV, 0, 0);
        if (kOffset) {  // V rows past the sequence's keys inside the last P.V K-step (see att_zero_rows), both boxes
          const int keys = cur.kv - cur.j * ATT_BKV;
          if (keys < ATT_BKV && (keys & 15) != 0)
            for (int x = 0; x < 2; ++x)
              att_zero_rows(sbase + ATW_SMEM_V + cur.stage * ATW_TILE_BYTES + x * ATW_BOX_BYTES, keys, (keys + 15) & ~15);
        }
        const bool q_done = more && nxt.j == max(nxt.nb0, nxt.nb1) - 1;  // last block that reads nxt's Q tiles
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const bool pv = active(cur, t);
          const bool qk = more && active(nxt, t);
          const uint64_t dq = make_smem_desc_sw128(sbase + ATW_SMEM_Q + t * ATW_TILE_BYTES, 16, 1024);
          const uint32_t tS = tmem_base + t * 256;
          if (pv) mbar_wait_plain(bar(P_FULL + t), g[t] & 1u);
          tc_fence_after();
          if (elect_one()) {
            if (pv) {
#pragma unroll
              for (int k = 0; k < ATT_BKV / 16; ++k)
                if (k < ksteps) umma_ts(tS + ATW_TM_O, tS + 8u * k, dv0 + 128u * k, idesc_o, k != 0 ? 1u : acc0);
              umma_commit(bar(O_FULL + t));
            }
            if (qk) {
              issue_qk(tS, dq, dk0, idesc_s);
              umma_commit(bar(S_FULL + t));
            }
            if (t == 1) {
              if (q_done) umma_commit(bar(Q_EMPTY));
              umma_commit(bar(KV_EMPTY + cur.stage));  // free once everything issued so far completes
            }
          }
          __syncwarp();
          if (pv) ++g[t];
        }
        if (lane == 0) sts_u32_volatile(progress_addr, ++blocks_done);  // the watchdog's sign of life
        if (!more) break;
        cur = nxt;
      }
    }
    if (lane == 0) mbar_arrive(bar(DONE));
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
    const uint32_t tS = tmem_base + t * 256 + lane_off;
    const uint32_t tO = tS + ATW_TM_O;
    const float c = p.scale_log2e;
    const uint32_t stg = sbase + ATW_SMEM_STG + uint32_t(warp - 4) * ATT_STG_BYTES;  // this warp's 32 x 128 B staging
    uint8_t* const stg_row = smem + ATW_SMEM_STG + (warp - 4) * ATT_STG_BYTES + lane * 128;
    uint32_t g = 0;  // blocks processed so far by this tile
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
      // ATW_RESCALE_LOG2 (in the log2 domain), so P <= 2^ATW_RESCALE_LOG2 and O is rescaled only when some row of
      // the warp outgrows that head-room (rare after the first block).
      float m = -INFINITY, l = 0.0f;

      for (int j = 0; j < nb; ++j, ++g) {
        const int nvalid = min(ATT_BKV, kv_len - j * ATT_BKV);
        // columns of this block this row may attend to: all valid ones, or up to the diagonal with a causal mask
        const bool diag = p.causal && j * ATT_BKV + ATT_BKV - 1 > row0 + q_off;  // warp-uniform
        const int lim = diag ? min(nvalid, qrow + q_off - j * ATT_BKV + 1) : nvalid;
        mbar_wait_plain(bar(S_FULL + t), g & 1u);
        tc_fence_after();
        float alpha = 1.0f;
        bool rescale = false;
        if (warp_live) {
          const bool masked = diag || (nvalid & 31) != 0;
          if (kBias) {
            const float* brow = p.bias + (long long)b * p.bias_b_stride + (long long)h * p.bias_h_stride +
                                (long long)min(qrow, p.Lq - 1) * p.bias_row_stride + j * ATT_BKV;
            softmax_block_wide<true>(tS, (nvalid + 31) >> 5, masked, lim, c, m, l, alpha, rescale, brow, nvalid);
          } else {
            softmax_block_wide<false>(tS, (nvalid + 31) >> 5, masked, lim, c, m, l, alpha, rescale);
          }
        }
        if (j > 0 && rescale) {  // warp-uniform
          // P.V(j-1) must have landed before O is rescaled. O_FULL has completed either g-1 or g phases here (P.V(j)
          // cannot be issued before this warp publishes P(j) below), and the two cases differ in parity. Without a
          // rescale no wait is needed: the tensor core accumulates P.V(j) onto O in issue order.
          mbar_wait_plain(bar(O_FULL + t), (g - 1) & 1u);
          tc_fence_after();
          // 32-column chunks up to head_dim (for 80 / 112 the last chunk also scales 16 unused columns)
#pragma unroll 1
          for (int c0 = 0; c0 < hd; c0 += 32) {
            uint32_t o[32];
            tmem_ld32(tO + c0, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st32(tO + c0, o);
          }
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(P_FULL + t));
      }
      mbar_wait_plain(bar(O_FULL + t), (g - 1) & 1u);  // cannot be lapped: the next flip needs this warp's next P_FULL arrive
      tc_fence_after();
      // normalise the head_dim output columns and hand the warp's 32 rows to two TMA stores of 64 columns (columns
      // >= head_dim and rows >= Lq are clipped by the tensor map); the halves share one staging buffer
      if (warp_live) {
        const float inv = kOffset && so.bad ? __int_as_float(0x7fc00000) : 1.0f / l;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const int col0 = half * 64;
          uint32_t o0[32], o1[32];
          tmem_ld32(tO + col0, o0);
          if (col0 + 32 < hd) tmem_ld32(tO + col0 + 32, o1);
          if (elect_one()) tma_store_wait_read<0>();  // the previous store has finished reading the staging
          __syncwarp();
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (col0 + 8 * i >= hd) break;
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
            *reinterpret_cast<uint4*>(stg_row + ((i ^ (lane & 7)) << 4)) = w;  // 128B swizzle of the store's map
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {  // bulk groups are per thread: elect.sync picks the same lane of a full warp every time
            tma_store_4d(&tmO, stg, col0, h, row0 + qd * 32, b);
            tma_store_commit();
          }
          __syncwarp();
        }
      }
      tc_fence_before();  // the TMEM reads above are ordered before this warp's next P_FULL arrive
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
