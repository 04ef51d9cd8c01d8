// Persistent warp-specialised bf16 GEMM for sm_100a:  out[b][m][n] = epilogue( sum_k A[b][m][k] * W[n][k] )
//
//   warp 0      : TMA producer (A/W tiles -> 128B-swizzled smem ring, mbarrier complete_tx)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (128 x 256 x 16 per instruction)
//   warps 2..9  : epilogue (tcgen05.ld -> registers -> bias / LayerNorm-fold / activation / residual -> bf16 ->
//                 swizzled smem -> TMA store), overlapped with the next tile's main loop through two
//                 256-column TMEM accumulators. Two warps per TMEM lane quarter, each owning 128 of the 256
//                 columns, so every SM sub-partition has two epilogue warps to hide latencies with.
//
// kCtas == 2 runs the same roles on a CTA pair (cluster of 2, tcgen05 cta_group::2): one 256 x 256 x 16 MMA spans both
// SMs, each CTA stages only its 128 rows of A and its 128 rows of W, so the L2 -> SM operand traffic per FLOP drops by a
// third (the 1-CTA tile needs 96 B/clk/SM at full tensor rate, more than the ~64 B/clk an SM can pull from L2) and the
// same smem holds 5 instead of 3 pipeline stages.
//
// This one kernel serves every linear on the encoder path (reference call sites: transformer.py:47-49 fused QKV,
// transformer.py:53 out_proj, transformer.py:59-67 MLP, vit.py:78 patch embedding as a GEMM over patch rows).
#pragma once
#include "ptx.cuh"

namespace b200 {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BN = 256;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 320;
constexpr int GEMM_EPI_WARPS = 8;
#ifndef GEMM_STAGES_2CTA
#define GEMM_STAGES_2CTA 5
#endif
constexpr int GEMM_STAT_SLICE = 128;  // columns per partial LayerNorm statistic
constexpr int GEMM_A_BYTES = GEMM_BM * GEMM_BK * 2;  // 16 KB
constexpr int GEMM_B_BYTES = GEMM_BN * GEMM_BK * 2;  // 32 KB
constexpr int GEMM_STAGE_BYTES = GEMM_A_BYTES + GEMM_B_BYTES;
constexpr int GEMM_STG_BYTES = 32 * 128;  // one staging buffer: 32 rows x 64 bf16
constexpr int GEMM_SMEM_COLVEC = GEMM_EPI_WARPS * 2 * 128 * 4;  // per warp: bias|c and colsum of its 128 columns
// smem plan: kCtas == 1: 3 stages x 48 KB + 1 staging buffer per epilogue warp (only used for problems of <= 128 rows)
//            kCtas == 2: 5 stages x 32 KB + 1 staging buffer per epilogue warp, or — residual epilogues — 4 stages +
//            2 buffers (one per 64-column chunk): there the buffer is claimed BEFORE the chunk's math (the residual is
//            transposed through it), so with a single buffer the previous chunk's TMA store would have to drain first.
//            (Round 1 measured 5 + 1 and 4 + 2 equal for the main loop.)
template <int kCtas, bool kRes = false>
struct GemmSmem {
  static constexpr int kStages = kCtas == 2 ? (kRes ? 4 : GEMM_STAGES_2CTA) : 3;
  static constexpr int kBRows = GEMM_BN / kCtas;
  static constexpr int kStageBytes = GEMM_A_BYTES + kBRows * GEMM_BK * 2;
  static constexpr int kRing = kStages * kStageBytes;
  static constexpr int kStgBufs = (kCtas == 2 && kStages <= 4) ? 2 : 1;
  static constexpr int kStg = GEMM_EPI_WARPS * kStgBufs * GEMM_STG_BYTES;
  static constexpr int kBytes = kRing + kStg + GEMM_SMEM_COLVEC + 256;
  static_assert(kBytes <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
};

struct GemmParams {
  int M;  // rows per batch
  int N;
  int K;
  int batches;
  int tiles_m;  // per batch
  int tiles_n;
  const float* bias;         // [N]  bias, or the folded constant vector c when ln_fold
  const float* colsum;       // [N]  s_n = sum_k W'[n][k] (ln_fold only)
  const float2* rowstats;    // ln_fold only: [batches*M] (mean, rstd) when stat_parts == 0, else
                             // [batches*M][stat_parts] partial (mean_t, M2_t) over 128-column slices of the row
  int stat_parts;
  float ln_eps;
  float2* stats_out;         // kStats: partial (mean_t, M2_t) of the OUTPUT rows, row (b, m) at
                             // [b * stats_rows + stats_off + m][ceil(N/128)]  (stats_rows = M, stats_off = 0 by default)
  int stats_rows, stats_off;
  const __nv_bfloat16* res;  // residual / positional table, nullptr if unused
  long long res_batch_stride;  // elements; 0 => same table for every batch (positional embedding)
  int ldr;                     // residual row stride (elements)
  __nv_bfloat16* out;          // kPatch only (per-thread store of the token rows)
  long long out_batch_stride;
  int ldo;
  const float* acc_scale;  // kF8 only: device scalar, dequantisation scale of the accumulator
  // kPatch only (im2col-free patch embedding, p = 16): patch grid of one image and the tiling of its rows. An M tile is
  // 8 patch rows x 16 patch columns: tile row r <-> patch (ph0 + r % 8, pw0 + r / 8), tiles_m = pt_nph8 * pt_nw16.
  int pt_hp, pt_wp, pt_nw16;
  unsigned int* abort_word;  // raised by a bounded barrier wait that ran out (ptx.cuh: mbar_wait); may be nullptr
};

// erf-GELU: x*Phi(x) = relu(x) - |x| * 2^Q(|x|), Q = degree-6 minimax fit of log2(0.5*erfc(t/sqrt2)) on [0,6]
// (max abs error 2.8e-7 vs the exact erf form, measured in fp32; reference op: nn.GELU(), transformer.py:61).
// Evaluated on two columns at once with the packed fp32 pipe (FFMA2): s = -min(|x|, 6), Horner in s (odd
// coefficients negated), one MUFU.EX2 per element, result = s * 2^Q + relu(x)  (for |x| > 6 the factor is < 1e-9).
__device__ __forceinline__ float2 gelu_erf_fast2(float2 x) {
  const float2 s = make_float2(fmaxf(-fabsf(x.x), -6.0f), fmaxf(-fabsf(x.y), -6.0f));
  float2 q = make_float2(3.310347528895363e-05f, 3.310347528895363e-05f);
  q = __ffma2_rn(q, s, make_float2(0.0007693132502026856f, 0.0007693132502026856f));
  q = __ffma2_rn(q, s, make_float2(0.008081023581326008f, 0.008081023581326008f));
  q = __ffma2_rn(q, s, make_float2(0.053412578999996185f, 0.053412578999996185f));
  q = __ffma2_rn(q, s, make_float2(-0.45877063274383545f, -0.45877063274383545f));
  q = __ffma2_rn(q, s, make_float2(1.151201844215393f, 1.151201844215393f));
  q = __ffma2_rn(q, s, make_float2(-0.9999930262565613f, -0.9999930262565613f));
  const float2 e = make_float2(fast_exp2(q.x), fast_exp2(q.y));
  return __ffma2_rn(s, e, make_float2(fmaxf(x.x, 0.0f), fmaxf(x.y, 0.0f)));
}

// tanh-GELU (nn.GELU(approximate="tanh"), transformer.py:62; GPT / GPT-2): 0.5x(1 + tanh(u)) = x / (1 + e^(-2u)),
// u = sqrt(2/pi)(x + 0.044715 x^3); the exponent is evaluated in base 2: w = x(c1 + c3 x^2), c1 = -2 sqrt(2/pi) log2 e.
// One MUFU.EX2 and one MUFU.RCP per element; x -> -inf gives x * 0 = -0, x -> +inf gives x * 1.
__device__ __forceinline__ float2 gelu_tanh_fast2(float2 x) {
  const float2 t = __fmul2_rn(x, x);
  const float2 g = __ffma2_rn(t, make_float2(-0.10294324f, -0.10294324f), make_float2(-2.3022082f, -2.3022082f));
  const float2 w = __fmul2_rn(x, g);
  const float2 den = __fadd2_rn(make_float2(fast_exp2(w.x), fast_exp2(w.y)), make_float2(1.0f, 1.0f));
  return make_float2(x.x * __frcp_rn(den.x), x.y * __frcp_rn(den.y));
}

// SiLU (nn.SiLU, transformer.py:64): x * sigmoid(x) = x / (1 + 2^(-x log2 e)); one MUFU.EX2 and one MUFU.RCP per element.
__device__ __forceinline__ float2 silu_fast2(float2 x) {
  const float2 w = __fmul2_rn(x, make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 den = __fadd2_rn(make_float2(fast_exp2(w.x), fast_exp2(w.y)), make_float2(1.0f, 1.0f));
  return make_float2(x.x * __frcp_rn(den.x), x.y * __frcp_rn(den.y));
}

// kAct: 0 = none, 1 = erf-GELU, 2 = tanh-GELU, 3 = ReLU, 4 = SiLU
// kF8: operands are e4m3 bytes (the optional FP8 variant, b200enc.h B200ENC_LINEAR_FP8): a stage still holds 128-byte
// rows, i.e. 128 instead of 64 K elements, each tcgen05.mma (kind::f8f6f4) consumes K = 32, and the accumulator is
// multiplied by *p.acc_scale (the product of the two per-tensor dequantisation scales) before the bias is added.
// kPatch: the A operand is the NCHW bf16 image itself (nn.Conv2d(3, d, 16, 16) as a GEMM without an im2col buffer,
// image/vit.py:64,78). tmA is a 4-D view (16 pixels, plane*Hp + ph, pixel row, pw) with byte strides (2, 16W*2, 2W, 32)
// and the 32-byte swizzle: ONE box (16, 8, 4, 16) per K block (one channel, four pixel rows: K index c*256 + i*16 + j,
// the order of conv.weight.view(d, 768)) lands in shared memory as [pw][i][ph % 8][16 pixels] — for every (pw, i) an
// 8-row x 32-byte atom of a K-major SWIZZLE_32B operand, one MMA K step wide (256 B between K steps, 1024 B between
// 8-row groups). The 128-byte swizzle of the other GEMMs cannot be produced from NCHW: a 32-byte inner box is padded to
// 128-byte rows there (csrc/probe_im2col_tma.cu). Rows of a tile are patches in (pw, ph % 8) order, so the epilogue maps
// tile row -> token row and stores per thread instead of through tmC; patches outside the grid are zero-filled / skipped.
template <int kCtas, bool kFold, int kAct, bool kRes, bool kStats, bool kF8 = false, bool kPatch = false>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  using SM = GemmSmem<kCtas, kRes>;
  const uint32_t ring = smem_base;
  float* colvec = reinterpret_cast<float*>(smem + SM::kRing + SM::kStg);
  const uint32_t bars = smem_base + SM::kRing + SM::kStg + GEMM_SMEM_COLVEC;
  // Per-CTA geometry: with kCtas == 2 this CTA stages 128 rows of A and 128 (of the tile's 256) rows of W per stage.
  constexpr int kStages = SM::kStages;
  constexpr int kBRows = SM::kBRows;
  constexpr int kStageBytes = SM::kStageBytes;
  constexpr int kTileM = GEMM_BM * kCtas;
  constexpr bool kTmaOut = !kPatch;  // output tiles leave through tmC (TMA store); kPatch stores per thread
  // barrier slots (8 bytes each): full[kStages] empty[kStages] tfull[2] tempty[2]; then the TMEM base address word.
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * kStages + 2 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(
      smem + SM::kRing + SM::kStg + GEMM_SMEM_COLVEC + 8 * (2 * kStages + 4));

  // Role index, not the hardware warp id: the sub-partition's arbiter serves the HIGHEST warp id first (measured,
  // B300_MICROARCH.md; attention_stream.cuh too), so the two control roles (TMA producer, MMA issuer: a handful of
  // instructions per K block, but every one of them on the tensor core's critical path) sit in hardware warps 8 and 9,
  // above the epilogue warps whose GELU / LayerNorm-fold arithmetic keeps the issue slots ~45 % busy; the epilogue
  // roles 2..9 are hardware warps 0..7. TMEM lane quarters follow the hardware warp id.
  const int hw_warp = threadIdx.x >> 5;
  const int warp = (hw_warp + 2) % (GEMM_THREADS / 32);
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = kCtas == 2 ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs)

  if (smem_base & 1023u) {  // the 128B swizzle needs a 1024-aligned ring: report through the status word, never trap
    if (threadIdx.x == 0 && p.abort_word != nullptr) *reinterpret_cast<volatile unsigned int*>(p.abort_word) = 0xB200A116u;
    return;  // uniform over the CTA (and over a CTA pair: both CTAs see the same shared-memory layout)
  }
  WaitCtx wctx = make_wait_ctx(p.abort_word);
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);   // the leader's producer arrives (expect_tx covers both CTAs' bytes)
      mbar_init(empty_bar(s), 1);  // tcgen05.commit (multicast to both CTAs when kCtas == 2)
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), GEMM_EPI_WARPS * kCtas);  // both CTAs' epilogue warps release the leader's MMA warp
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (kTmaOut) tma_prefetch_desc(&tmC);
  }
  if (warp == 1) {
    if (kCtas == 2) {
      tmem_alloc_2cta<512>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
      tmem_relinquish_2cta();
    } else {
      tmem_alloc<512>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (kCtas == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only this CTA's shared / tensor memory: it may overlap the previous kernel's tail
  griddep_launch_dependents();
  griddep_wait();

  constexpr int kBKe = kF8 ? 2 * GEMM_BK : GEMM_BK;  // K elements per 128-byte stage row
  const int num_kb = (p.K + kBKe - 1) / kBKe;
  const int tiles_per_batch = p.tiles_m * p.tiles_n;
  const int total_tiles = tiles_per_batch * p.batches;
  const int first_tile = blockIdx.x / kCtas;  // both CTAs of a pair walk the same tile sequence
  const int tile_step = gridDim.x / kCtas;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (one warp per CTA, converged;
    // a single elected lane issues, so tensor-map / barrier operands stay in uniform registers)
    uint32_t stage = 0, phase = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
      const int b = tile / tiles_per_batch;
      const int r = tile - b * tiles_per_batch;
      const int m0 = (r / p.tiles_n) * kTileM + int(cta_rank) * GEMM_BM;
      const int n0 = (r % p.tiles_n) * GEMM_BN + int(cta_rank) * kBRows;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, wctx);
        const uint32_t sa = ring + stage * kStageBytes;
        if (elect_one()) {
          if (kCtas == 2) {
            // both CTAs' bytes are accounted on the leader's barrier; only the leader arms it
            const uint32_t leader_full = map_to_cta(full_bar(stage), 0);
            if (cta_rank == 0) mbar_expect_tx(full_bar(stage), 2 * kStageBytes);
            tma_load_3d_2cta(&tmA, leader_full, sa, kb * kBKe, m0, b);
            tma_load_2d_2cta(&tmB, leader_full, sa + GEMM_A_BYTES, kb * kBKe, n0);
          } else if (kPatch) {
            const int tm = r / p.tiles_n;
            mbar_expect_tx(full_bar(stage), kStageBytes);
            tma_load_4d(&tmA, full_bar(stage), sa, 0, (b * 3 + (kb >> 2)) * p.pt_hp + 8 * (tm / p.pt_nw16), (kb & 3) * 4,
                        16 * (tm % p.pt_nw16));
            tma_load_2d(&tmB, full_bar(stage), sa + GEMM_A_BYTES, kb * kBKe, n0);
          } else {
            mbar_expect_tx(full_bar(stage), kStageBytes);
            tma_load_3d(&tmA, full_bar(stage), sa, kb * kBKe, m0, b);
            tma_load_2d(&tmB, full_bar(stage), sa + GEMM_A_BYTES, kb * kBKe, n0);
          }
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only; converged warp)
    if (cta_rank == 0) {
      constexpr uint32_t idesc = kF8 ? make_idesc_e4m3(kTileM, GEMM_BN) : make_idesc_bf16(kTileM, GEMM_BN, 0, 0);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u, wctx);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * GEMM_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase, wctx);
          tc_fence_after();
          const uint32_t sa = ring + stage * kStageBytes;
          const uint64_t da = kPatch ? make_smem_desc_sw32(sa, 256, 1024) : make_smem_desc_sw128(sa, 16, 1024);
          constexpr uint32_t kAStep = kPatch ? 16u : 2u;  // 16 K elements further: two 128-byte core matrices / 32 bytes in the swizzle atom
          const uint64_t db = make_smem_desc_sw128(sa + GEMM_A_BYTES, 16, 1024);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < GEMM_BK / 16; ++k) {
              // advancing K by 16 bf16 (32 e4m3) = 32 bytes inside the 128B swizzle atom: +2 in the (addr >> 4) field
              if (kF8) {
                if (kCtas == 2)
                  umma_ss_f8_2cta(d_tmem, da + kAStep * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
                else
                  umma_ss_f8(d_tmem, da + kAStep * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
              } else if (kCtas == 2)
                umma_ss_2cta(d_tmem, da + kAStep * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else
                umma_ss(d_tmem, da + kAStep * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            if (kCtas == 2) umma_commit_2cta(empty_bar(stage), 3); else umma_commit(empty_bar(stage));
            if (kb == num_kb - 1) {
              if (kCtas == 2) umma_commit_2cta(tfull_bar(acc), 3); else umma_commit(tfull_bar(acc));
            }
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        acc ^= 1u;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps
    const int q = hw_warp & 3;             // TMEM lane quarter this warp may access
    const int hf = (warp - 2) >> 2;        // which 128-column half of the tile this warp owns
    const uint32_t stg = smem_base + SM::kRing + (warp - 2) * (SM::kStgBufs * GEMM_STG_BYTES);
    uint8_t* stg_ptr = smem + SM::kRing + (warp - 2) * (SM::kStgBufs * GEMM_STG_BYTES);
    float* cv_b = colvec + (warp - 2) * 256;  // this warp's private copy of bias|c for its 128 columns ...
    float* cv_s = cv_b + 128;                 // ... and of the LayerNorm-fold column sums
    const int n_slices = (p.N + GEMM_STAT_SLICE - 1) / GEMM_STAT_SLICE;
    uint32_t acc = 0, acc_phase = 0;
    const uint32_t tempty_leader0 = kCtas == 2 ? map_to_cta(tempty_bar(0), 0) : tempty_bar(0);
    for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
      const int b = tile / tiles_per_batch;
      const int r = tile - b * tiles_per_batch;
      const int m0 = (r / p.tiles_n) * kTileM + int(cta_rank) * GEMM_BM;  // first row owned by this CTA
      const int n0 = (r % p.tiles_n) * GEMM_BN;
      // row of the batch this lane owns. kPatch: tile row -> patch index (see the kernel comment)
      const int pt_ph0 = kPatch ? 8 * ((r / p.tiles_n) / p.pt_nw16) : 0;
      const int pt_pw0 = kPatch ? 16 * ((r / p.tiles_n) % p.pt_nw16) : 0;
      auto tile_row = [&](int rt, bool& ok) {  // rt = row inside this CTA's 128-row tile
        if (kPatch) {
          const int ph = pt_ph0 + (rt & 7), pw = pt_pw0 + (rt >> 3);
          ok = ph < p.pt_hp && pw < p.pt_wp;
          return ph * p.pt_wp + pw;
        }
        ok = m0 + rt < p.M;
        return m0 + rt;
      };
      bool row_ok;
      const int row = tile_row(q * 32 + lane, row_ok);
      const int nh = n0 + hf * 128;  // first column owned by this warp

      // ---- issue every global load of this tile up front: they complete while the tile's main loop still runs
      float4 my_b = make_float4(0.f, 0.f, 0.f, 0.f), my_s = make_float4(0.f, 0.f, 0.f, 0.f);
      if (nh + 4 * lane < p.N) {  // N is a multiple of 8: the 4 columns of a lane are all valid or all out of range
        if (p.bias != nullptr) my_b = __ldg(reinterpret_cast<const float4*>(p.bias + nh) + lane);
        if (kFold) my_s = __ldg(reinterpret_cast<const float4*>(p.colsum + nh) + lane);
      }
      float2 st_full = make_float2(0.0f, 1.0f);
      constexpr int kMaxParts = 12;
      float2 st_part[kMaxParts];
      if (kFold && row_ok) {
        const long long grow = (long long)b * p.M + row;
        if (p.stat_parts == 0) {
          st_full = __ldg(p.rowstats + grow);
        } else {
#pragma unroll
          for (int t = 0; t < kMaxParts; ++t)
            if (t < p.stat_parts) st_part[t] = __ldg(p.rowstats + grow * p.stat_parts + t);
        }
      }
      // Residual tile of this warp (32 rows x 128 columns), fetched COALESCED: per 64-column chunk, load j of lane l
      // reads the 16 bytes at (row 4j + l/8, piece l%8), so one warp instruction covers 4 rows x 128 contiguous bytes
      // (whole 32-byte sectors; the round-1 form — every lane its own row — used half of each sector it pulled over
      // the L2 -> SM path, the tightest resource of the N = K = 768 GEMM). The lanes swap to row ownership through
      // the warp's staging buffer just before the values are needed (see below).
      uint4 rres[2][8];
      if (kRes) {
        const __nv_bfloat16* res_base = p.res + (long long)b * p.res_batch_stride + nh;
#pragma unroll
        for (int cc = 0; cc < 2; ++cc)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            bool rr_ok;
            const int rr = tile_row(q * 32 + 4 * j + (lane >> 3), rr_ok);
            const int col = cc * 64 + (lane & 7) * 8;
            rres[cc][j] = make_uint4(0, 0, 0, 0);
            if (rr_ok && nh + col < p.N)
              rres[cc][j] = __ldg(reinterpret_cast<const uint4*>(res_base + (long long)rr * p.ldr + col));
          }
      }

      __syncwarp();  // every lane finished reading the previous tile's column vectors
      reinterpret_cast<float4*>(cv_b)[lane] = my_b;
      if (kFold) reinterpret_cast<float4*>(cv_s)[lane] = my_s;
      __syncwarp();

      float rstd = 1.0f, nmr = 0.0f;  // nmr = -mean * rstd
      if (kFold) {
        if (p.stat_parts == 0) {
          rstd = st_full.y;
          nmr = -st_full.x * st_full.y;
        } else if (row_ok) {
          // combine the per-slice (mean, M2) written by the producing GEMM's epilogue (Chan et al.), fixed order
          float mean = 0.0f;
#pragma unroll
          for (int t = 0; t < kMaxParts; ++t)
            if (t < p.stat_parts) mean += float(min(GEMM_STAT_SLICE, p.K - t * GEMM_STAT_SLICE)) * st_part[t].x;
          mean /= float(p.K);
          float m2 = 0.0f;
#pragma unroll
          for (int t = 0; t < kMaxParts; ++t)
            if (t < p.stat_parts) {
              const float dm = st_part[t].x - mean;
              m2 += st_part[t].y + float(min(GEMM_STAT_SLICE, p.K - t * GEMM_STAT_SLICE)) * dm * dm;
            }
          rstd = rsqrtf(m2 / float(p.K) + p.ln_eps);
          nmr = -mean * rstd;
        }
      }
      const float f8_scale = kF8 ? __ldg(p.acc_scale) : 1.0f;
      float st_shift = 0.0f;
      float2 st_s1 = make_float2(0.f, 0.f), st_s2 = make_float2(0.f, 0.f);
      bool released = false;

      mbar_wait(tfull_bar(acc), acc_phase, wctx);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * GEMM_BN + hf * 128 + (uint32_t(q * 32) << 16);

#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int nc = nh + cc * 64;
        if (nc >= p.N) break;
        uint32_t v0[32], v1[32];
        tmem_ld32(taddr + cc * 64, v0);
        tmem_ld32(taddr + cc * 64 + 32, v1);
        tmem_wait_ld();
        if (cc == 1 || nc + 64 >= p.N) {
          // last TMEM read of this accumulator by this warp: hand it back to the MMA warp before doing the math
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (kCtas == 2) mbar_arrive_cluster(tempty_leader0 + 8u * acc); else mbar_arrive(tempty_bar(acc));
          }
          released = true;
        }

        uint4 own[8];  // this lane's row of the residual chunk (kRes only)
        if (kRes) {
          constexpr int kBufOffR = SM::kStgBufs == 2 ? GEMM_STG_BYTES : 0;
          if (kTmaOut) {  // the TMA store that last used this staging buffer has finished reading it
            if (elect_one()) tma_store_wait_read<SM::kStgBufs - 1>();
            __syncwarp();
          }
          uint8_t* tb = stg_ptr + cc * kBufOffR;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rw = 4 * j + (lane >> 3);
            *reinterpret_cast<uint4*>(tb + rw * 128 + (((lane & 7) ^ (rw & 7)) << 4)) = rres[cc][j];
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) own[j] = *reinterpret_cast<const uint4*>(tb + lane * 128 + ((j ^ (lane & 7)) << 4));
          // no second barrier: from here on every lane touches only the 128 bytes of its own row
        }
        uint32_t packed[32];
        const float2 rstd2 = make_float2(rstd, rstd), nmr2 = make_float2(nmr, nmr);
        const float2 f8_scale2 = make_float2(f8_scale, f8_scale);
#pragma unroll
        for (int j4 = 0; j4 < 16; ++j4) {
          // 4 columns per step as two fp32 pairs (packed FFMA2 pipe); column vectors are broadcast 16-byte smem loads
          const float4 cb = *reinterpret_cast<const float4*>(cv_b + cc * 64 + 4 * j4);
          float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
          if (kFold) cs = *reinterpret_cast<const float4*>(cv_s + cc * 64 + 4 * j4);
          float2 x[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int idx = 4 * j4 + 2 * u;
            const float2 a = make_float2(__uint_as_float(idx < 32 ? v0[idx] : v1[idx - 32]),
                                         __uint_as_float(idx < 32 ? v0[idx + 1] : v1[idx + 1 - 32]));
            const float2 cb2 = u == 0 ? make_float2(cb.x, cb.y) : make_float2(cb.z, cb.w);
            const float2 cs2 = u == 0 ? make_float2(cs.x, cs.y) : make_float2(cs.z, cs.w);
            x[u] = kFold ? __ffma2_rn(rstd2, a, __ffma2_rn(nmr2, cs2, cb2))
                         : (kF8 ? __ffma2_rn(a, f8_scale2, cb2) : __fadd2_rn(a, cb2));
            if (kAct == 1) x[u] = gelu_erf_fast2(x[u]);
            if (kAct == 2) x[u] = gelu_tanh_fast2(x[u]);
            if (kAct == 3) x[u] = make_float2(fmaxf(x[u].x, 0.0f), fmaxf(x[u].y, 0.0f));
            if (kAct == 4) x[u] = silu_fast2(x[u]);
            if (kRes) {
              const uint32_t rr = reinterpret_cast<const uint32_t*>(own)[2 * j4 + u];
              x[u] = __fadd2_rn(x[u], make_float2(bf16_lo(rr), bf16_hi(rr)));
            }
            packed[2 * j4 + u] = pack_bf16x2(x[u].x, x[u].y);
          }
          if (kStats) {
            // statistics of the values as stored (bf16-rounded), shifted by the row's first value in this slice
            if (cc == 0 && j4 == 0) st_shift = bf16_lo(packed[0]);
            const float2 sh2 = make_float2(-st_shift, -st_shift);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              float2 dlt = __fadd2_rn(make_float2(bf16_lo(packed[2 * j4 + u]), bf16_hi(packed[2 * j4 + u])), sh2);
              if (nc + 4 * j4 + 2 * u + 1 >= p.N) {  // only possible in the last, partial chunk of the matrix
                if (nc + 4 * j4 + 2 * u >= p.N) dlt.x = 0.0f;
                dlt.y = 0.0f;
              }
              st_s1 = __fadd2_rn(st_s1, dlt);
              st_s2 = __ffma2_rn(dlt, dlt, st_s2);
            }
          }
        }

        // A warp whose 32 rows all lie past M has nothing to store (the TMA store would clip every row). The branch
        // also gives the chunk loop a join point before the store: without it ptxas duplicates the chunk's math for
        // the one-chunk and two-chunk paths (+640 instructions in the residual + statistics epilogue).
        if (kTmaOut && m0 + q * 32 >= p.M) continue;
        if (kTmaOut) {
          // with two buffers the store that last used this one was issued a whole tile ago: no drain on the critical path
          constexpr int kBufOff = SM::kStgBufs == 2 ? GEMM_STG_BYTES : 0;
          if (!kRes) {  // (with a residual the buffer was already claimed for the transposition above)
            if (elect_one()) tma_store_wait_read<SM::kStgBufs - 1>();
            __syncwarp();
          }
          uint8_t* dst = stg_ptr + cc * kBufOff + lane * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            *reinterpret_cast<uint4*>(dst + ((j ^ (lane & 7)) << 4)) =
                make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {  // bulk groups are per thread: elect.sync picks the same lane of a full warp every time
            tma_store_3d(&tmC, stg + cc * kBufOff, nc, m0 + q * 32, b);
            tma_store_commit();
          }
        } else {
          if (row_ok) {
            __nv_bfloat16* orow = p.out + (long long)b * p.out_batch_stride + (long long)row * p.ldo + nc;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (nc + j * 8 < p.N)
                *(reinterpret_cast<uint4*>(orow) + j) =
                    make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
            }
          }
        }
      }
      if (kStats && row_ok && nh < p.N) {
        const float nt = float(min(GEMM_STAT_SLICE, p.N - nh));
        const float s1 = st_s1.x + st_s1.y, s2 = st_s2.x + st_s2.y;
        const float mean_t = st_shift + s1 / nt;
        const float m2_t = fmaxf(s2 - s1 * s1 / nt, 0.0f);
        p.stats_out[((long long)b * p.stats_rows + p.stats_off + row) * n_slices + nh / GEMM_STAT_SLICE] =
            make_float2(mean_t, m2_t);
      }
      if (!released) {  // warp owned no valid columns in this tile (N tail)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCtas == 2) mbar_arrive_cluster(tempty_leader0 + 8u * acc); else mbar_arrive(tempty_bar(acc));
        }
      }
      acc ^= 1u;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (kTmaOut && elect_one()) tma_store_wait_all<0>();
  }

  tc_fence_before();
  if (kCtas == 2) cluster_sync_all(); else __syncthreads();  // the peer may still arrive on / read from this CTA's smem
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    if (kCtas == 2) tmem_dealloc_2cta<512>(tmem_base); else tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace b200
