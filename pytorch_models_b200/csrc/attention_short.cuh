// Attention for SHORT key/value sequences (Lkv <= 256, head_dim 64, no mask) on sm_100a: the whole score row of a
// query fits in tensor memory, so the softmax is exact and single-pass (reference: F.scaled_dot_product_attention at
// pytorch_models/transformer.py:52 with attn_mask=None, is_causal=False — ViT-B/16 at 224 px has 197 tokens, the
// configuration the headline metric is quoted on; longer, causal or biased calls use attention_stream.cuh).
//
// Why a second kernel: with two 128-key blocks per item the general kernel pays its per-block fixed costs (barrier
// round trips S_FULL -> P_FULL -> O_FULL, the rescale bookkeeping of the online softmax, an item boundary every
// second block) on almost every block: 10.8 k clocks per (batch, head) at L=197 against ~3 k of exponentials. Here:
//   work item = (batch, head, pair of 128-row query tiles); one persistent CTA per SM, 384 threads
//   warp 0      : TMA producer. One stage = both Q tiles + ALL of K and V of the item (box of nk16 = ceil16(Lkv)
//                 rows, one load each); two stages, so the next item's operands arrive while this one is computed
//   warp 1      : tcgen05.mma issuer:  S_t = Q_t K^T  as ONE group of 4 MMAs with N = nk16 (up to 256 columns of
//                 TMEM), O_t = P_t V as nk16/16 MMAs with P as the TMEM A operand. Order per item:
//                 PV0(n) QK0(n+1) PV1(n) QK1(n+1)
//   warp 2      : watchdog (attention_common.cuh: no unbounded wait can hang the GPU)
//   warps 4..7  : softmax of tile 0, warps 8..11 of tile 1; one thread per query row. Pass 1 streams the row out of
//                 TMEM in 32-column chunks for the exact maximum (FMNMX3), pass 2 streams it again, takes the
//                 exponentials and writes P back over S as packed bf16 (chunk c of P lands on columns of S that
//                 pass 2 has already consumed). No running maximum, no rescale, one barrier round trip per item.
//                 Both passes are rolled loops over chunks: the softmax code is ~1/4 of the general kernel's.
// TMEM (512 columns): S_t takes nk16 columns, O_t 64. For nk16 <= 192 everything has its own columns. For
// 192 < nk16 <= 224 (L = 197!) tile 0 keeps a private O (S0 [0,224) | S1 [224,448) | O0 [448,512)) so that
// QK0(n+1) can be issued right behind PV0(n); O1 lies over the upper columns of S1, which are dead once P1 is
// complete, and QK1(n+1) waits (T_FREE) until the epilogue has pulled O1(n) into registers. Above 224 both tiles
// alias. The host picks the layout (api_attention.cu).
// The normalised output leaves through one TMA store per warp, Q/K/V are read straight out of the fused QKV
// activation through strided tensor maps (attention_common.cuh). Every role waits with mbar_wait_parked: a waiting
// warp issues almost nothing and leaves its sub-partition's issue slots to the warps that compute.
#pragma once
#include "attention_common.cuh"

namespace b200 {

constexpr int ATS_MAX_KV = 256;
constexpr int ATS_KV_BYTES = ATS_MAX_KV * 128;                         // 32 KB: up to 256 rows x 64 bf16
constexpr int ATS_STAGE_BYTES = 2 * ATT_TILE_BYTES + 2 * ATS_KV_BYTES;  // Q0 | Q1 | K | V = 96 KB
constexpr int ATS_OFF_K = 2 * ATT_TILE_BYTES;
constexpr int ATS_OFF_V = ATS_OFF_K + ATS_KV_BYTES;
constexpr int ATS_SMEM_STG = 2 * ATS_STAGE_BYTES;                       // 8 warps x 4 KB output staging
constexpr int ATS_SMEM_ONES = ATS_SMEM_STG + 8 * ATT_STG_BYTES;  // 16 rows x 128 B of bf16 1.0: B operand of the row-sum MMA
constexpr int ATS_SMEM_BAR = ATS_SMEM_ONES + 2048;
constexpr int ATS_SMEM_BYTES = ATS_SMEM_BAR + 256;
static_assert(ATS_SMEM_BYTES <= 232448, "short attention kernel: shared memory budget");

struct AttnShortParams {
  int B, H, Lq, Lkv;
  int nk16;           // Lkv rounded up to 16: N of the score MMA, rows of the K/V boxes
  int n_qp, n_items;  // as AttnParams
  float scale_log2e;
  int tm_s0, tm_s1, tm_o0, tm_o1;  // TMEM columns of S_t (P_t in place) and O_t
  int tm_l0, tm_l1;                // 16 TMEM columns per tile that receive the row sums l = P . 1 (all 16 equal)
  int alias0, alias1;              // 1: O_t overlaps S_t, the next score MMA of the tile waits for the epilogue's read of O_t
  unsigned int* abort_word;
  long long* trace;
};

// kNH: number of 16-column halves of the score row (nk16 / 16) as a compile-time constant, 0 = read it from the
// parameters. With a constant every chunk guard folds away: no taken branches over skipped code (ncu: `no_inst`
// stalls on the instruction after each skipped masking block), and ptxas schedules across chunks.
template <int kNH>
__global__ void __launch_bounds__(ATT_THREADS, 1)
attention_short_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                       const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                       const AttnShortParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bars = sbase + ATS_SMEM_BAR;
  auto bar = [&](int i) { return bars + 8u * i; };
  constexpr int FULL = 0, EMPTY = 2, S_FULL = 4, P_FULL = 6, O_FULL = 8, T_FREE = 10, DONE = 12;
  constexpr int kProtocolBarriers = 12;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + ATS_SMEM_BAR + 8 * 13);
  const uint32_t progress_addr = sbase + ATS_SMEM_BAR + 8 * 13 + 4;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
#ifdef ATT_TRACE
  int tr_n = 0;
  const int tr_role = warp == 0 ? 0 : warp == 1 ? 1 : warp < 8 ? 2 : 3;
#endif
  unsigned int* const abw = p.abort_word;
  if (sbase & 1023u) {
    if (threadIdx.x == 0 && abw != nullptr) *reinterpret_cast<volatile unsigned int*>(abw) = 0xB200A117u;
    return;
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(FULL + i), 1);
      mbar_init(bar(EMPTY + i), 1);
      mbar_init(bar(S_FULL + i), 1);
      mbar_init(bar(P_FULL + i), 4);
      mbar_init(bar(O_FULL + i), 1);
      mbar_init(bar(T_FREE + i), 4);
    }
    mbar_init(bar(DONE), 10);
    *reinterpret_cast<volatile uint32_t*>(smem + ATS_SMEM_BAR + 8 * 13 + 4) = 0u;
    fence_mbar_init();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmO);
  }
  for (int i = threadIdx.x; i < 2048 / 4; i += ATT_THREADS) reinterpret_cast<uint32_t*>(smem + ATS_SMEM_ONES)[i] = 0x3f803f80u;
  fence_proxy_async_smem();  // the tensor core reads the tile through the async proxy
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
  const int n_my = p.n_items > int(blockIdx.x) ? (p.n_items - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x) : 0;
  auto item_of = [&](int n) { return int(blockIdx.x) + n * int(gridDim.x); };
  auto two_of = [&](int item) { return (item % p.n_qp) * 256 + ATT_BQ < p.Lq; };  // second query tile has a valid row

  if (warp < 4) setmaxnreg_dec<ATT_CONTROL_REGS>();
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    for (int n = 0; n < n_my; ++n) {
      const int item = item_of(n);
      const int qp = item % p.n_qp;
      const int bh = item / p.n_qp;
      const int h = bh % p.H;
      const int b = bh / p.H;
      const bool two = two_of(item);
      const uint32_t s = uint32_t(n) & 1u;
      mbar_wait_parked(bar(EMPTY + s), ((uint32_t(n) >> 1) & 1u) ^ 1u);
      if (elect_one()) {
        const uint32_t st = sbase + s * ATS_STAGE_BYTES;
        mbar_expect_tx(bar(FULL + s), (two ? 2 : 1) * ATT_TILE_BYTES + 2 * p.nk16 * 128);
        tma_load_3d(&tmQ, bar(FULL + s), st, h * ATT_HD, qp * 256, b);
        if (two) tma_load_3d(&tmQ, bar(FULL + s), st + ATT_TILE_BYTES, h * ATT_HD, qp * 256 + ATT_BQ, b);
        tma_load_3d(&tmK, bar(FULL + s), st + ATS_OFF_K, h * ATT_HD, 0, b);
        tma_load_3d(&tmV, bar(FULL + s), st + ATS_OFF_V, h * ATT_HD, 0, b);
      }
      __syncwarp();
    }
    if (lane == 0) mbar_arrive(bar(DONE));
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp converged, one lane issues)
    uint32_t nq[2] = {0, 0};   // score MMAs issued per tile (T_FREE parity)
    uint32_t npv[2] = {0, 0};  // P.V MMAs issued per tile (P_FULL parity)
    uint32_t done = 0;
    const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, p.nk16, 0, 0);
    const uint32_t idesc_o = make_idesc_bf16(ATT_BQ, ATT_HD, 0, 1);
    const uint32_t idesc_l = make_idesc_bf16(ATT_BQ, 16, 0, 0);
    const uint64_t d_ones = make_smem_desc_sw128(sbase + ATS_SMEM_ONES, 16, 1024);
    const int ksteps = p.nk16 >> 4;
    auto issue_qk = [&](int n, int t) {
      const uint32_t st = sbase + (uint32_t(n) & 1u) * ATS_STAGE_BYTES;
      if ((t == 0 ? p.alias0 : p.alias1) && nq[t] > 0) {  // the epilogue has pulled the previous O_t out of the columns S_t covers
        mbar_wait_parked(bar(T_FREE + t), (nq[t] - 1) & 1u);
        tc_fence_after();
      }
      const uint64_t dq = make_smem_desc_sw128(st + t * ATT_TILE_BYTES, 16, 1024);
      const uint64_t dk = make_smem_desc_sw128(st + ATS_OFF_K, 16, 1024);
      if (elect_one()) {
        {
#pragma unroll
          for (int k = 0; k < ATT_HD / 16; ++k)
            umma_ss(tmem_base + (t == 0 ? p.tm_s0 : p.tm_s1), dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
        }
        umma_commit(bar(S_FULL + t));
      }
      __syncwarp();
      ++nq[t];
      if (lane == 0) ATT_EV(100 + t);
    };
    auto issue_pv = [&](int n, int t) {
      const uint32_t st = sbase + (uint32_t(n) & 1u) * ATS_STAGE_BYTES;
      mbar_wait_parked(bar(P_FULL + t), npv[t] & 1u);
      if (lane == 0) ATT_EV(110 + t);
      tc_fence_after();
      const uint64_t dv0 = make_smem_desc_sw128(st + ATS_OFF_V, 16, 1024);
      const uint32_t pa0 = tmem_base + (t == 0 ? p.tm_s0 : p.tm_s1);
      const uint32_t d_o = tmem_base + (t == 0 ? p.tm_o0 : p.tm_o1);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < ATS_MAX_KV / 16; ++k)
          if (k < ksteps) umma_ts(d_o, pa0 + 8u * k, dv0 + 128u * k, idesc_o, k != 0 ? 1u : 0u);
        // l_t = P_t . 1: the row sums of the bf16 probabilities the tensor core actually multiplies with, for the price
        // of nk16/16 MMAs of N = 16 (8 clocks each) instead of 128 FADD2 per softmax thread
#pragma unroll
        for (int k = 0; k < ATS_MAX_KV / 16; ++k)
          if (k < ksteps) umma_ts(tmem_base + (t == 0 ? p.tm_l0 : p.tm_l1), pa0 + 8u * k, d_ones + 2u * (k & 3), idesc_l, k != 0 ? 1u : 0u);
        umma_commit(bar(O_FULL + t));
      }
      __syncwarp();
      ++npv[t];
      if (lane == 0) ATT_EV(120 + t);
    };
    if (n_my > 0) {
      mbar_wait_parked(bar(FULL + 0), 0u);
      tc_fence_after();
      issue_qk(0, 0);
      if (two_of(item_of(0))) issue_qk(0, 1);
      for (int n = 0; n < n_my; ++n) {
        const bool two = two_of(item_of(n));
        const bool more = n + 1 < n_my;
        issue_pv(n, 0);
        if (more) {
          mbar_wait_parked(bar(FULL + ((uint32_t(n) + 1u) & 1u)), ((uint32_t(n) + 1u) >> 1) & 1u);
          if (lane == 0) ATT_EV(130);
          tc_fence_after();
          issue_qk(n + 1, 0);
        }
        if (two) issue_pv(n, 1);
        if (elect_one()) umma_commit(bar(EMPTY + (uint32_t(n) & 1u)));  // every MMA reading this stage has been issued
        __syncwarp();
        if (more && two_of(item_of(n + 1))) issue_qk(n + 1, 1);
        if (lane == 0) sts_u32_volatile(progress_addr, ++done);
      }
    }
    if (lane == 0) mbar_arrive(bar(DONE));
  } else if (warp == 2) {
    // ------------------------------------------------------------ watchdog (input: the issuer's item counter)
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
    setmaxnreg_inc<ATT_SOFTMAX_REGS>();
    const int t = (warp - 4) >> 2;
    const int qd = warp & 3;
    const uint32_t lane_off = uint32_t(qd * 32) << 16;
    const uint32_t tS = tmem_base + uint32_t(t == 0 ? p.tm_s0 : p.tm_s1) + lane_off;
    const uint32_t tO = tmem_base + uint32_t(t == 0 ? p.tm_o0 : p.tm_o1) + lane_off;
    const uint32_t tL = tmem_base + uint32_t(t == 0 ? p.tm_l0 : p.tm_l1) + lane_off;
    const float c = p.scale_log2e;
    const int nkv = p.Lkv;
    const int nh = kNH > 0 ? kNH : (p.nk16 >> 4);  // 16-column halves of the score row (compile-time for kNH > 0)
    const int n_ch = (nh + 1) >> 1;                // 32-column chunks
    const uint32_t stg = sbase + ATS_SMEM_STG + uint32_t(warp - 4) * ATT_STG_BYTES;
    const bool alias = (t == 0 ? p.alias0 : p.alias1) != 0;
    uint32_t g = 0;  // units processed by this tile
    for (int n = 0; n < n_my; ++n) {
      const int item = item_of(n);
      const int qp = item % p.n_qp;
      const int bh = item / p.n_qp;
      const int h = bh % p.H;
      const int b = bh / p.H;
      const int row0 = qp * 256 + t * ATT_BQ;
      if (row0 >= p.Lq) continue;  // tile absent (same rule as the issuer)
      const bool warp_live = row0 + qd * 32 < p.Lq;
      mbar_wait_parked(bar(S_FULL + t), g & 1u);
      if (lane == 0 && qd == 0) ATT_EV(200 + t);
      tc_fence_after();
      if (warp_live) {
        uint32_t v0[32], v1[32], v2[32], v3[32];
        // ---- pass 1: exact row maximum. Chunks 4..7 first, then chunks 0..3 — which stay in registers for pass 2.
        // Each group is four back-to-back tcgen05.ld with one wait (a chunk-by-chunk loop is bound by the TMEM load
        // latency: 160 clocks per chunk in the event trace). Only the last 16-column half of the row can hold
        // columns >= Lkv (zero scores of the zero-filled K rows): those are set to -inf. The half above it, when nh
        // is odd, holds stale TMEM and is never looked at.
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
        auto mask_half = [&](uint32_t(&v)[32], int ch, int hf) {
          if (kNH > 0) {  // compile-time position of the row's last half
            if (2 * ch + hf == kNH - 1) {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (ch * 32 + hf * 16 + i >= nkv) v[hf * 16 + i] = 0xff800000u;
            }
          } else if (ch * 32 + hf * 16 + 16 > nkv) {  // warp-uniform; written per element so that the arrays stay in registers
#pragma unroll
            for (int i = 0; i < 16; ++i) v[hf * 16 + i] = ch * 32 + hf * 16 + i >= nkv ? 0xff800000u : v[hf * 16 + i];
          }
        };
        auto max_chunk = [&](uint32_t(&v)[32], int ch) {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            if (2 * ch + hf < nh) {
              mask_half(v, ch, hf);
              mx0 = fmax3(mx0, __uint_as_float(v[hf * 16 + 0]), __uint_as_float(v[hf * 16 + 1]));
              mx1 = fmax3(mx1, __uint_as_float(v[hf * 16 + 2]), __uint_as_float(v[hf * 16 + 3]));
              mx2 = fmax3(mx2, __uint_as_float(v[hf * 16 + 4]), __uint_as_float(v[hf * 16 + 5]));
              mx3 = fmax3(mx3, __uint_as_float(v[hf * 16 + 6]), __uint_as_float(v[hf * 16 + 7]));
              mx0 = fmax3(mx0, __uint_as_float(v[hf * 16 + 8]), __uint_as_float(v[hf * 16 + 9]));
              mx1 = fmax3(mx1, __uint_as_float(v[hf * 16 + 10]), __uint_as_float(v[hf * 16 + 11]));
              mx2 = fmax3(mx2, __uint_as_float(v[hf * 16 + 12]), __uint_as_float(v[hf * 16 + 13]));
              mx3 = fmax3(mx3, __uint_as_float(v[hf * 16 + 14]), __uint_as_float(v[hf * 16 + 15]));
            }
          }
        };
        if (4 < n_ch) {
          tmem_ld32(tS + 4 * 32, v0);
          if (5 < n_ch) tmem_ld32(tS + 5 * 32, v1);
          if (6 < n_ch) tmem_ld32(tS + 6 * 32, v2);
          if (7 < n_ch) tmem_ld32(tS + 7 * 32, v3);
          tmem_wait_ld();
          max_chunk(v0, 4);
          if (5 < n_ch) max_chunk(v1, 5);
          if (6 < n_ch) max_chunk(v2, 6);
          if (7 < n_ch) max_chunk(v3, 7);
        }
        tmem_ld32(tS, v0);
        if (1 < n_ch) tmem_ld32(tS + 1 * 32, v1);
        if (2 < n_ch) tmem_ld32(tS + 2 * 32, v2);
        if (3 < n_ch) tmem_ld32(tS + 3 * 32, v3);
        tmem_wait_ld();
        max_chunk(v0, 0);
        if (1 < n_ch) max_chunk(v1, 1);
        if (2 < n_ch) max_chunk(v2, 2);
        if (3 < n_ch) max_chunk(v3, 3);
        const float m = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        const float m_off = m == -INFINITY ? 0.0f : m;
        const float2 c2 = make_float2(c, c);
        const float2 nmc2 = make_float2(-m_off * c, -m_off * c);
        if (lane == 0 && qd == 0) ATT_EV(202 + t);
        // ---- pass 2: exponentials, row sum, P over S. Chunks 0..3 come out of the registers of pass 1 (already
        // masked); each array is refilled with chunk 4..7 as soon as its chunk is done, so those loads hide behind
        // the exponentials.
        auto exp_chunk = [&](uint32_t(&v)[32], int ch, bool remask) {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            if (2 * ch + hf < nh) {
              if (remask) mask_half(v, ch, hf);
              uint32_t pk[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float2 e = __ffma2_rn(make_float2(__uint_as_float(v[hf * 16 + 2 * i]),
                                                        __uint_as_float(v[hf * 16 + 2 * i + 1])), c2, nmc2);
#if ATT_POLY_EVERY > 0
                const float2 pr = (i % ATT_POLY_EVERY) == ATT_POLY_EVERY - 1 ? exp2_poly2(e)
                                                                             : make_float2(fast_exp2(e.x), fast_exp2(e.y));
#else
                const float2 pr = make_float2(fast_exp2(e.x), fast_exp2(e.y));
#endif
                pk[i] = pack_bf16x2(pr.x, pr.y);
              }
              tmem_st8(tS + ch * 16 + hf * 8, pk);
            }
          }
        };
        exp_chunk(v0, 0, false);
        if (4 < n_ch) tmem_ld32(tS + 4 * 32, v0);
        if (1 < n_ch) exp_chunk(v1, 1, false);
        if (5 < n_ch) tmem_ld32(tS + 5 * 32, v1);
        if (2 < n_ch) exp_chunk(v2, 2, false);
        if (6 < n_ch) tmem_ld32(tS + 6 * 32, v2);
        if (3 < n_ch) exp_chunk(v3, 3, false);
        if (7 < n_ch) tmem_ld32(tS + 7 * 32, v3);
        if (4 < n_ch) {
          tmem_wait_ld();
          exp_chunk(v0, 4, true);
          if (5 < n_ch) exp_chunk(v1, 5, true);
          if (6 < n_ch) exp_chunk(v2, 6, true);
          if (7 < n_ch) exp_chunk(v3, 7, true);
        }
        tmem_wait_st();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(P_FULL + t));
      if (lane == 0 && qd == 0) ATT_EV(210 + t);
      mbar_wait_parked(bar(O_FULL + t), g & 1u);
      tc_fence_after();
      if (lane == 0 && qd == 0) ATT_EV(220 + t);
      if (warp_live) {
        uint32_t o0[32], o1[32];
        tmem_ld32(tO, o0);
        tmem_ld32(tO + 32, o1);
        const uint32_t lsum = tmem_ld1(tL);
        if (elect_one()) tma_store_wait_read<0>();  // the previous item's store has finished reading the staging
        __syncwarp();
        tmem_wait_ld();
        if (alias) {  // O_t is in registers: the tile's next scores may overwrite its columns
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(T_FREE + t));
        }
        const float inv = 1.0f / __uint_as_float(lsum);
        uint8_t* dst = smem + ATS_SMEM_STG + (warp - 4) * ATT_STG_BYTES + lane * 128;
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
        if (elect_one()) {
          tma_store_3d(&tmO, stg, h * ATT_HD, row0 + qd * 32, b);
          tma_store_commit();
        }
        __syncwarp();
      } else if (alias) {
        if (lane == 0) mbar_arrive(bar(T_FREE + t));
      }
      tc_fence_before();  // the TMEM reads above are ordered before this warp's next P_FULL arrive
      if (lane == 0 && qd == 0) ATT_EV(230 + t);
      ++g;
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
