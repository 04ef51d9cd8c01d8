// C-ABI entry point for the linear layers of the encoder block (see include/b200enc.h).
#include "../../include/b200enc.h"
#include "gemm.cuh"
#include "host_util.h"

using namespace b200;

namespace {

template <int kCtas, bool kFold, int kAct, bool kRes, bool kStats, bool kF8 = false, bool kPatch = false>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p, int grid,
                cudaStream_t stream) {
  auto kern = gemm_bf16_kernel<kCtas, kFold, kAct, kRes, kStats, kF8, kPatch>;
  constexpr int kSmem = GemmSmem<kCtas, kRes>::kBytes;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), kSmem)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = kSmem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCtas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  B200_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, p));
  return 0;
}

template <int kCtas, bool kFold, int kAct, bool kRes>
int dispatch_store(bool stats, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                   int grid, cudaStream_t s) {
  if constexpr (kRes && !kFold) {
    if (stats) return launch_gemm<kCtas, kFold, kAct, kRes, true>(ta, tb, tc, p, grid, s);
  }
  if (stats) return set_error(-1, "b200enc_linear: stats_out needs a residual, non-folded epilogue");
  return launch_gemm<kCtas, kFold, kAct, kRes, false>(ta, tb, tc, p, grid, s);
}

// The FP8 variant: bias [+ erf-GELU] [+ residual], TMA store
template <int kCtas>
int dispatch_fp8(bool gelu, bool res, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                 int grid, cudaStream_t s) {
  if (gelu && res) return set_error(-1, "b200enc_linear: FP8 variant: GELU and residual cannot be combined");
  if (gelu) return launch_gemm<kCtas, false, 1, false, false, true>(ta, tb, tc, p, grid, s);
  if (res) return launch_gemm<kCtas, false, 0, true, false, true>(ta, tb, tc, p, grid, s);
  return launch_gemm<kCtas, false, 0, false, false, true>(ta, tb, tc, p, grid, s);
}

template <int kCtas>
int dispatch_epilogue(int sel, bool stats, const CUtensorMap& ta, const CUtensorMap& tb,
                      const CUtensorMap& tc, const GemmParams& p, int grid, cudaStream_t s) {
  switch (sel) {
    case 0: return dispatch_store<kCtas, false, 0, false>(stats, ta, tb, tc, p, grid, s);
    case 1: return dispatch_store<kCtas, false, 0, true>(stats, ta, tb, tc, p, grid, s);
    case 2: return dispatch_store<kCtas, false, 1, false>(stats, ta, tb, tc, p, grid, s);
    case 3: return dispatch_store<kCtas, false, 1, true>(stats, ta, tb, tc, p, grid, s);
    case 4: return dispatch_store<kCtas, true, 0, false>(stats, ta, tb, tc, p, grid, s);
    case 5: return dispatch_store<kCtas, true, 0, true>(stats, ta, tb, tc, p, grid, s);
    case 6: return dispatch_store<kCtas, true, 1, false>(stats, ta, tb, tc, p, grid, s);
    case 7: return dispatch_store<kCtas, true, 1, true>(stats, ta, tb, tc, p, grid, s);
    case 8: return dispatch_store<kCtas, false, 2, false>(stats, ta, tb, tc, p, grid, s);   // tanh-GELU
    case 12: return dispatch_store<kCtas, true, 2, false>(stats, ta, tb, tc, p, grid, s);   // LN fold + tanh-GELU
    case 16: return dispatch_store<kCtas, false, 3, false>(stats, ta, tb, tc, p, grid, s);  // ReLU
    case 20: return dispatch_store<kCtas, true, 3, false>(stats, ta, tb, tc, p, grid, s);
    case 32: return dispatch_store<kCtas, false, 4, false>(stats, ta, tb, tc, p, grid, s);  // SiLU
    case 36: return dispatch_store<kCtas, true, 4, false>(stats, ta, tb, tc, p, grid, s);
    default: return set_error(-1, "b200enc_linear: tanh-GELU / ReLU / SiLU cannot be combined with a residual");
  }
}

}  // namespace

// ---------------------------------------------------------------- im2col-free patch embedding (p = 16)
extern "C" int b200enc_patch_embed16(const b200enc_linear_args* a, int img_h, int img_w, void* stream) {
  if (int rc0 = check_abort("b200enc_patch_embed16")) return rc0;
  B200_CHECK_ARG(a != nullptr && a->x && a->w && a->out && a->residual, "b200enc_patch_embed16: null image / weight / output / residual");
  B200_CHECK_ARG(img_h >= 16 && img_w >= 16 && img_h % 16 == 0 && img_w % 16 == 0,
                 "b200enc_patch_embed16: image %d x %d is not a multiple of the 16-pixel patch", img_h, img_w);
  const int hp = img_h / 16, wp = img_w / 16, P = hp * wp, n = a->batches, N = a->N;
  B200_CHECK_ARG(n >= 1 && a->M == P && a->K == 768 && N >= 8 && N % 8 == 0,
                 "b200enc_patch_embed16: expects M = %d patches, K = 768, got M=%d K=%d N=%d", P, a->M, a->K, N);
  B200_CHECK_ARG(a->colsum == nullptr && a->flags == 0 && a->ldw >= 768 && a->ldo >= N && a->ldr >= N,
                 "b200enc_patch_embed16: bias + positional rows (+ statistics) only");
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(a->out) & 15u) == 0 && a->ldo % 8 == 0 && a->out_batch_stride % 8 == 0 &&
                     (reinterpret_cast<uintptr_t>(a->residual) & 15u) == 0 && a->ldr % 8 == 0,
                 "b200enc_patch_embed16: output and residual rows must be 16-byte aligned");
  B200_CHECK_ARG((long long)n * 3 * hp < (1ll << 31), "b200enc_patch_embed16: too many image planes");
  CUtensorMap ta, tb;
  int rc;
  // see the kPatch comment in gemm.cuh
  const uint64_t dims[4] = {16, uint64_t(n) * 3 * hp, 16, uint64_t(wp)};
  const uint64_t strides[3] = {uint64_t(16) * img_w * 2, uint64_t(img_w) * 2, 32};
  const uint32_t box[4] = {16, 8, 4, 16};
  if ((rc = make_tmap_bf16_nd(&ta, a->x, 4, dims, strides, box, 32))) return rc;
  if ((rc = make_tmap_bf16(&tb, a->w, 768, N, 0, a->ldw, 0, GEMM_BK, GEMM_BN, 128))) return rc;
  GemmParams p = {};
  p.M = P;
  p.N = N;
  p.K = 768;
  p.batches = n;
  p.pt_hp = hp;
  p.pt_wp = wp;
  p.pt_nw16 = (wp + 15) / 16;
  p.tiles_m = ((hp + 7) / 8) * p.pt_nw16;
  p.tiles_n = (N + GEMM_BN - 1) / GEMM_BN;
  p.bias = a->bias;
  p.stats_out = reinterpret_cast<float2*>(a->stats_out);
  p.stats_rows = a->stats_rows_per_batch > 0 ? a->stats_rows_per_batch : P;
  p.stats_off = a->stats_row_offset;
  B200_CHECK_ARG(a->stats_row_offset >= 0 && p.stats_rows >= P + a->stats_row_offset,
                 "b200enc_patch_embed16: stats_rows_per_batch=%d cannot hold %d rows at offset %d", p.stats_rows, P,
                 a->stats_row_offset);
  p.res = reinterpret_cast<const __nv_bfloat16*>(a->residual);
  p.res_batch_stride = a->res_batch_stride;
  p.ldr = a->ldr;
  p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
  p.out_batch_stride = a->out_batch_stride;
  p.ldo = a->ldo;
  p.abort_word = abort_word();
  const long long total = (long long)p.tiles_m * p.tiles_n * n;
  const int grid = int(total < sm_count() ? total : sm_count());
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (a->stats_out != nullptr) return launch_gemm<1, false, 0, true, true, false, true>(ta, tb, tb, p, grid, s);
  return launch_gemm<1, false, 0, true, false, false, true>(ta, tb, tb, p, grid, s);
}

extern "C" int b200enc_linear(const b200enc_linear_args* a, void* stream) {
  B200_CHECK_ARG(a != nullptr, "b200enc_linear: null argument struct");
  if (int rc = check_abort("b200enc_linear")) return rc;
  const int batches = a->batches, M = a->M, N = a->N, K = a->K;
  B200_CHECK_ARG(a->x && a->w && a->out, "b200enc_linear: null tensor pointer");
  B200_CHECK_ARG(batches >= 1 && M >= 1 && N >= 1 && K >= 1, "b200enc_linear: bad shape batches=%d M=%d N=%d K=%d",
                 batches, M, N, K);
  B200_CHECK_ARG(K % 8 == 0 && N % 8 == 0, "b200enc_linear: K=%d and N=%d must be multiples of 8", K, N);
  const bool fp8 = (a->flags & B200ENC_LINEAR_FP8) != 0;
  if (fp8) {
    B200_CHECK_ARG(K % 16 == 0 && a->ldx % 16 == 0 && a->ldw % 16 == 0 && a->x_batch_stride % 16 == 0,
                   "b200enc_linear: FP8 variant needs K, ldx, ldw and the batch stride to be multiples of 16 bytes");
    B200_CHECK_ARG(a->acc_scale != nullptr && a->colsum == nullptr && a->stats_out == nullptr,
                   "b200enc_linear: FP8 variant needs acc_scale and supports neither the LayerNorm fold nor stats_out");
    B200_CHECK_ARG((a->flags & (B200ENC_LINEAR_GELU_TANH | B200ENC_LINEAR_RELU | B200ENC_LINEAR_SILU)) == 0,
                   "b200enc_linear: FP8 variant supports bias, erf-GELU and residual epilogues only");
  }
  // ldx < K is allowed on purpose: overlapping rows express a strided 1-D convolution as a GEMM (whisper stem).
  B200_CHECK_ARG(a->ldx >= 8 && a->ldw >= K && a->ldo >= N,
                 "b200enc_linear: leading dimension smaller than the row length");
  B200_CHECK_ARG((a->colsum == nullptr) == (a->rowstats == nullptr),
                 "b200enc_linear: colsum and rowstats must be given together (LayerNorm fold)");
  if (a->colsum) {
    const int want = (K + GEMM_STAT_SLICE - 1) / GEMM_STAT_SLICE;
    B200_CHECK_ARG(a->rowstats_parts == 0 || (a->rowstats_parts == want && want <= 12),
                   "b200enc_linear: rowstats_parts=%d must be 0 or ceil(K/128)=%d (<= 12)", a->rowstats_parts, want);
  }
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(a->bias) & 15u) == 0 && (reinterpret_cast<uintptr_t>(a->colsum) & 15u) == 0,
                 "b200enc_linear: bias / colsum must be 16-byte aligned");
  if (a->residual) {
    B200_CHECK_ARG(a->ldr >= N && a->ldr % 8 == 0 && a->res_batch_stride % 8 == 0 &&
                       (reinterpret_cast<uintptr_t>(a->residual) & 15u) == 0,
                   "b200enc_linear: residual must be 16-byte aligned with strides that are multiples of 8");
  }
  const bool fold = a->colsum != nullptr;
  const bool gelu = (a->flags & B200ENC_LINEAR_GELU) != 0;
  const bool gelu_tanh = (a->flags & B200ENC_LINEAR_GELU_TANH) != 0;
  const bool relu = (a->flags & B200ENC_LINEAR_RELU) != 0;
  const bool silu = (a->flags & B200ENC_LINEAR_SILU) != 0;
  B200_CHECK_ARG(int(gelu) + int(gelu_tanh) + int(relu) + int(silu) <= 1,
                 "b200enc_linear: at most one activation flag may be set");
  constexpr int kLinearFlags =
      B200ENC_LINEAR_GELU | B200ENC_LINEAR_GELU_TANH | B200ENC_LINEAR_RELU | B200ENC_LINEAR_SILU | B200ENC_LINEAR_FP8;
  B200_CHECK_ARG((a->flags & ~kLinearFlags) == 0, "b200enc_linear: flags=%d has bits outside the documented set (0x%x)",
                 a->flags, kLinearFlags);
  const bool res = a->residual != nullptr;
  const bool stats = a->stats_out != nullptr;

  // CTA pairs (256-row tiles) unless the problem has at most one 128-row tile per batch — or unless wave quantisation
  // says otherwise (SURVEY §7 hard part 3): the kernel is persistent, so its time is ceil(tiles / slots) tile-times.
  // At the strong-scaled ViT-B/16 shard (M = 25 216 = 98.5 x 256) the N = 768 GEMMs have 99 x 3 = 297 pair-tiles on
  // 74 pairs = 4.01 -> 5 waves, the last one a single tile (20 % lost), while 128-row tiles give 197 x 3 = 591 tiles
  // on 148 CTAs = 3.99 -> 4 waves. A 128-row tile costs about 1.15x half a pair-tile (3-stage ring, no operand
  // sharing: round-1 A/B), which the model below charges.
  int ctas = M > GEMM_BM ? 2 : 1;
  // (Measured at M = 25 216, round 2: out_proj 0.036 vs 0.037 ms in favour of 128-row tiles, FC2 (K = 3072) 0.101 vs
  // 0.099 ms in favour of pairs — the longer main loop amortises the lone tile of the last wave — so the switch is
  // limited to K <= 1024.)
  if (ctas == 2 && K <= 1024) {
    const long long tn = (N + GEMM_BN - 1) / GEMM_BN;
    const long long t2 = (long long)((M + 2 * GEMM_BM - 1) / (2 * GEMM_BM)) * tn * batches;
    const long long t1 = (long long)((M + GEMM_BM - 1) / GEMM_BM) * tn * batches;
    const long long s2 = sm_count() / 2, s1 = sm_count();
    const double cost2 = double((t2 + s2 - 1) / s2);            // in pair-tile times
    const double cost1 = double((t1 + s1 - 1) / s1) * 1.15;     // a wave of 128-row tiles covers the same area
    if (cost1 < cost2 * 0.97) ctas = 1;
  }
  CUtensorMap ta, tb, tc;
  int rc;
  if (fp8) {  // 1-byte elements: the 128-byte swizzled stage row holds 128 of them
    if ((rc = make_tmap_u8(&ta, a->x, K, M, batches, a->ldx, batches > 1 ? a->x_batch_stride : (long long)M * a->ldx,
                           2 * GEMM_BK, GEMM_BM, 128)))
      return rc;
    if ((rc = make_tmap_u8(&tb, a->w, K, N, 0, a->ldw, 0, 2 * GEMM_BK, GEMM_BN / ctas, 128))) return rc;
  } else {
    if ((rc = make_tmap_bf16(&ta, a->x, K, M, batches, a->ldx, batches > 1 ? a->x_batch_stride : (long long)M * a->ldx,
                             GEMM_BK, GEMM_BM, 128)))
      return rc;
    if ((rc = make_tmap_bf16(&tb, a->w, K, N, 0, a->ldw, 0, GEMM_BK, GEMM_BN / ctas, 128))) return rc;
  }
  if ((rc = make_tmap_bf16(&tc, a->out, N, M, batches, a->ldo,
                           batches > 1 ? a->out_batch_stride : (long long)M * a->ldo, 64, 32, 128)))
    return rc;

  GemmParams p = {};
  p.M = M;
  p.N = N;
  p.K = K;
  p.batches = batches;
  p.tiles_m = (M + GEMM_BM * ctas - 1) / (GEMM_BM * ctas);
  p.tiles_n = (N + GEMM_BN - 1) / GEMM_BN;
  p.bias = a->bias;
  p.colsum = a->colsum;
  p.rowstats = reinterpret_cast<const float2*>(a->rowstats);
  p.stat_parts = a->rowstats_parts;
  p.ln_eps = a->ln_eps;
  p.stats_out = reinterpret_cast<float2*>(a->stats_out);
  p.stats_rows = a->stats_rows_per_batch > 0 ? a->stats_rows_per_batch : M;
  p.stats_off = a->stats_row_offset;
  B200_CHECK_ARG(a->stats_row_offset >= 0 && p.stats_rows >= M + a->stats_row_offset,
                 "b200enc_linear: stats_rows_per_batch=%d cannot hold M=%d rows at offset %d", p.stats_rows, M,
                 a->stats_row_offset);
  p.res = reinterpret_cast<const __nv_bfloat16*>(a->residual);
  p.res_batch_stride = a->res_batch_stride;
  p.ldr = a->ldr;
  p.acc_scale = a->acc_scale;
  p.abort_word = abort_word();

  const long long total = (long long)p.tiles_m * p.tiles_n * batches;
  const int slots = sm_count() / ctas;  // CTAs (or CTA pairs) resident at once: the kernel is persistent
  const int grid = int(total < slots ? total : slots) * ctas;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (fp8) {
    if (ctas == 2) return dispatch_fp8<2>(gelu, res, ta, tb, tc, p, grid, s);
    return dispatch_fp8<1>(gelu, res, ta, tb, tc, p, grid, s);
  }
  const int sel = (silu ? 32 : 0) | (relu ? 16 : 0) | (gelu_tanh ? 8 : 0) | (fold ? 4 : 0) | (gelu ? 2 : 0) | (res ? 1 : 0);
  if (ctas == 2) return dispatch_epilogue<2>(sel, stats, ta, tb, tc, p, grid, s);
  return dispatch_epilogue<1>(sel, stats, ta, tb, tc, p, grid, s);
}
