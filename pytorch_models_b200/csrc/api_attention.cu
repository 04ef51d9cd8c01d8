// C-ABI entry point for the attention core (see include/b200enc.h).
#include "../../include/b200enc.h"
#include "attention_short.cuh"
#include "attention_stream.cuh"
#include "attention_wide.cuh"
#include "host_util.h"

using namespace b200;

#ifdef ATT_TRACE
// debug builds only (make ../b200enc_trace): event trace buffer of CTA 0, see ATT_EV in attention_common.cuh
static long long* g_attention_trace = nullptr;
extern "C" void b200enc_debug_attention_trace(long long* buf) { g_attention_trace = buf; }
#endif

namespace {
// one launch path for every attention kernel: programmatic dependent launch unless disabled (host_util.h)
template <typename Kern, typename Params>
int launch_pdl(Kern kern, int grid, int threads, int smem, cudaStream_t s, const CUtensorMap& tq, const CUtensorMap& tk,
               const CUtensorMap& tv, const CUtensorMap& to, const Params& p) {
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), smem)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  B200_CUDA(cudaLaunchKernelEx(&cfg, kern, tq, tk, tv, to, p));
  return 0;
}
}  // namespace

// head_dim 64 has two kernels: Lkv <= 256 without a mask runs the single-pass kernel of attention_short.cuh, everything
// else (longer rows, causal, biased, or B200ENC_ATTN_GENERAL) the streaming kernel of attention_stream.cuh.
// head_dim 80, 96, 112 and 128 run the kernel of attention_wide.cuh for every Lkv, mask and bias.
static int attention_wide(const void* q, long long qbs, int ldq, const void* k, const void* v, long long kbs, int ldkv,
                          void* out, long long obs, int ldo, int B, int H, int Lq, int Lkv, int head_dim,
                          float scale_log2e, int flags, const float* bias, long long bias_b_stride,
                          long long bias_h_stride, long long bias_row_stride, const int* off, int off_stride,
                          cudaStream_t s) {
  // 4-D maps (head_dim columns, H heads, L rows, B): a tile is two 64-column boxes; the columns >= head_dim of the
  // second box are zero-filled on load and clipped on store. Output: 32 rows x 64 columns per softmax warp and store.
  auto map = [&](CUtensorMap* m, const void* base, int L, int ld, long long bs, uint32_t box_rows) {
    const uint64_t dims[4] = {uint64_t(head_dim), uint64_t(H), uint64_t(L), uint64_t(B)};
    const uint64_t strides[3] = {uint64_t(head_dim) * 2, uint64_t(ld) * 2, uint64_t(bs) * 2};
    const uint32_t box[4] = {64, 1, box_rows, 1};
    return make_tmap_bf16_nd(m, base, 4, dims, strides, box, 128);
  };
  CUtensorMap tq, tk, tv, to;
  int rc;
  if ((rc = map(&tq, q, Lq, ldq, qbs, ATT_BQ))) return rc;
  if ((rc = map(&tk, k, Lkv, ldkv, kbs, ATT_BKV))) return rc;
  if ((rc = map(&tv, v, Lkv, ldkv, kbs, ATT_BKV))) return rc;
  if ((rc = map(&to, out, Lq, ldo, obs, 32))) return rc;
  AttnWideParams p;
  p.B = B;
  p.H = H;
  p.Lq = Lq;
  p.Lkv = Lkv;
  p.head_dim = head_dim;
  p.n_qp = (Lq + 2 * ATT_BQ - 1) / (2 * ATT_BQ);
  p.n_items = B * H * p.n_qp;
  p.scale_log2e = scale_log2e;
  p.causal = (flags & B200ENC_ATTN_CAUSAL) ? 1 : 0;
  p.bias = bias;
  p.bias_b_stride = bias_b_stride;
  p.bias_h_stride = bias_h_stride;
  p.bias_row_stride = bias_row_stride;
  p.abort_word = abort_word();
  p.off = off;
  p.off_stride = off_stride;
  const int grid = p.n_items < sm_count() ? p.n_items : sm_count();
  const auto kern = off != nullptr    ? attention_wide_kernel<false, true>
                    : bias != nullptr ? attention_wide_kernel<true>
                                      : attention_wide_kernel<false>;
  return launch_pdl(kern, grid, ATT_THREADS, ATW_SMEM_BYTES, s, tq, tk, tv, to, p);
}

// off != nullptr: offset-causal mode (b200enc_attention_extend): Lkv is the cache capacity, the query rows of sequence b
// start at position off[b * off_stride]; always the streaming kernels, flags = B200ENC_ATTN_CAUSAL, no bias.
static int attention_impl(const char* who, const void* q, long long q_batch_stride, int ldq, const void* k,
                          const void* v, long long kv_batch_stride, int ldkv, void* out, long long out_batch_stride,
                          int ldo, int B, int H, int Lq, int Lkv, int head_dim, float scale, int flags,
                          const float* bias, long long bias_b_stride, long long bias_h_stride,
                          long long bias_row_stride, const int* off, int off_stride, void* stream) {
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(q && k && v && out, "%s: null tensor pointer", who);
  B200_CHECK_ARG(head_dim == ATT_HD || (head_dim > ATT_HD && head_dim <= ATW_MAX_HD && head_dim % 16 == 0),
                 "%s: head_dim=%d is not supported (64, 80, 96, 112 or 128)", who, head_dim);
  B200_CHECK_ARG(B >= 1 && H >= 1 && Lq >= 1 && Lkv >= 1, "%s: bad shape B=%d H=%d Lq=%d Lkv=%d", who, B, H, Lq, Lkv);
  B200_CHECK_ARG(ldq >= H * head_dim && ldkv >= H * head_dim && ldo >= H * head_dim,
                 "%s: leading dimension smaller than H*head_dim", who);
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 15u) == 0 && ldo % 8 == 0 && out_batch_stride % 8 == 0,
                 "%s: output rows must be 16-byte aligned", who);
  constexpr int kAttnFlags = B200ENC_ATTN_CAUSAL | B200ENC_ATTN_GENERAL;
  B200_CHECK_ARG((flags & ~kAttnFlags) == 0, "%s: flags=%d has bits outside the documented set (0x%x)", who, flags,
                 kAttnFlags);
  const long long qbs = B > 1 ? q_batch_stride : (long long)Lq * ldq;
  const long long kbs = B > 1 ? kv_batch_stride : (long long)Lkv * ldkv;
  const long long obs = B > 1 ? out_batch_stride : (long long)Lq * ldo;
  const float scale_log2e = scale * 1.4426950408889634f;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (head_dim != ATT_HD)
    return attention_wide(q, qbs, ldq, k, v, kbs, ldkv, out, obs, ldo, B, H, Lq, Lkv, head_dim, scale_log2e, flags,
                          bias, bias_b_stride, bias_h_stride, bias_row_stride, off, off_stride, s);
  const bool short_kv = Lkv <= ATS_MAX_KV && bias == nullptr && off == nullptr &&
                        !(flags & (B200ENC_ATTN_CAUSAL | B200ENC_ATTN_GENERAL));
  // K/V boxes: the whole row rounded up to 16 for the short kernel (N of its score MMA), 128-row blocks otherwise
  const int nk16 = (Lkv + 15) & ~15;
  const int kv_box = short_kv ? nk16 : ATT_BKV;
  CUtensorMap tq, tk, tv, to;
  int rc;
  if ((rc = make_tmap_bf16(&tq, q, uint64_t(H) * ATT_HD, Lq, B, ldq, qbs, ATT_HD, ATT_BQ, 128))) return rc;
  if ((rc = make_tmap_bf16(&tk, k, uint64_t(H) * ATT_HD, Lkv, B, ldkv, kbs, ATT_HD, kv_box, 128))) return rc;
  if ((rc = make_tmap_bf16(&tv, v, uint64_t(H) * ATT_HD, Lkv, B, ldkv, kbs, ATT_HD, kv_box, 128))) return rc;
  // output: one TMA store of 32 rows x 64 columns per softmax warp; rows >= Lq of a batch are clipped by the map
  if ((rc = make_tmap_bf16(&to, out, uint64_t(H) * ATT_HD, Lq, B, ldo, obs, ATT_HD, 32, 128))) return rc;
  const int n_qp = (Lq + 2 * ATT_BQ - 1) / (2 * ATT_BQ);
  const int n_items = B * H * n_qp;
  const int grid = n_items < sm_count() ? n_items : sm_count();
#ifdef ATT_TRACE
  long long* const trace = g_attention_trace;
#else
  long long* const trace = nullptr;
#endif

  if (short_kv) {
    AttnShortParams p;
    p.B = B;
    p.H = H;
    p.Lq = Lq;
    p.Lkv = Lkv;
    p.nk16 = nk16;
    p.n_qp = n_qp;
    p.n_items = n_items;
    p.scale_log2e = scale_log2e;
    // TMEM layout (see attention_short.cuh): private columns for S and O where 512 columns allow it, otherwise O_t
    // over the upper columns of S_t
    if (nk16 <= 176) {  // everything has its own columns: S_t 176 | O_t 64 | l_t 16
      p.tm_s0 = 0, p.tm_o0 = 176, p.tm_l0 = 240, p.tm_s1 = 256, p.tm_o1 = 432, p.tm_l1 = 496, p.alias0 = p.alias1 = 0;
    } else if (nk16 <= 208) {  // S0 208 | l0 16 | S1 208 | l1 16 | O0 64; O1 over the upper columns of S1
      p.tm_s0 = 0, p.tm_l0 = 208, p.tm_s1 = 224, p.tm_l1 = 432, p.tm_o0 = 448, p.tm_o1 = 224 + 128, p.alias0 = 0, p.alias1 = 1;
    } else if (nk16 <= 240) {  // both O_t over S_t; l_t behind the scores
      p.tm_s0 = 0, p.tm_o0 = 128, p.tm_l0 = 240, p.tm_s1 = 256, p.tm_o1 = 256 + 128, p.tm_l1 = 496, p.alias0 = p.alias1 = 1;
    } else {  // the scores fill all 256 columns of a tile: O_t and l_t both lie over them
      p.tm_s0 = 0, p.tm_o0 = 128, p.tm_l0 = 192, p.tm_s1 = 256, p.tm_o1 = 256 + 128, p.tm_l1 = 256 + 192, p.alias0 = p.alias1 = 1;
    }
    p.abort_word = abort_word();
    p.trace = trace;
    // the row length of ViT at 224 px (197 tokens -> 13 halves of 16 columns) has its own instantiation
    const auto kern = nk16 == 208 ? attention_short_kernel<13> : attention_short_kernel<0>;
    return launch_pdl(kern, grid, ATT_THREADS, ATS_SMEM_BYTES, s, tq, tk, tv, to, p);
  }

  AttnParams p;
  p.B = B;
  p.H = H;
  p.Lq = Lq;
  p.Lkv = Lkv;
  p.n_qp = n_qp;
  p.n_items = n_items;
  p.scale_log2e = scale_log2e;
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.out_batch_stride = out_batch_stride;
  p.ldo = ldo;
  p.causal = (flags & B200ENC_ATTN_CAUSAL) ? 1 : 0;
  p.bias = bias;
  p.bias_b_stride = bias_b_stride;
  p.bias_h_stride = bias_h_stride;
  p.bias_row_stride = bias_row_stride;
  p.abort_word = abort_word();
  p.trace = trace;
  p.off = off;
  p.off_stride = off_stride;
  const auto kern = off != nullptr    ? attention_kernel<false, true>
                    : bias != nullptr ? attention_kernel<true>
                                      : attention_kernel<false>;
  return launch_pdl(kern, grid, ATT_THREADS, ATT_SMEM_BYTES, s, tq, tk, tv, to, p);
}

extern "C" int b200enc_attention(const void* q, long long q_batch_stride, int ldq, const void* k, const void* v,
                                 long long kv_batch_stride, int ldkv, void* out, long long out_batch_stride, int ldo,
                                 int B, int H, int Lq, int Lkv, int head_dim, float scale, int flags, void* stream) {
  return attention_impl("b200enc_attention", q, q_batch_stride, ldq, k, v, kv_batch_stride, ldkv, out,
                        out_batch_stride, ldo, B, H, Lq, Lkv, head_dim, scale, flags, nullptr, 0, 0, 0, nullptr, 0,
                        stream);
}

extern "C" int b200enc_attention_bias(const void* q, long long q_batch_stride, int ldq, const void* k, const void* v,
                                      long long kv_batch_stride, int ldkv, void* out, long long out_batch_stride,
                                      int ldo, int B, int H, int Lq, int Lkv, int head_dim, float scale, int flags,
                                      const float* bias, long long bias_b_stride, long long bias_h_stride,
                                      long long bias_row_stride, void* stream) {
  B200_CHECK_ARG(bias != nullptr, "b200enc_attention_bias: null bias");
  B200_CHECK_ARG(bias_b_stride >= 0 && bias_h_stride >= 0 && bias_row_stride >= 0,
                 "b200enc_attention_bias: negative bias stride");
  return attention_impl("b200enc_attention", q, q_batch_stride, ldq, k, v, kv_batch_stride, ldkv, out,
                        out_batch_stride, ldo, B, H, Lq, Lkv, head_dim, scale, flags, bias, bias_b_stride,
                        bias_h_stride, bias_row_stride, nullptr, 0, stream);
}

extern "C" int b200enc_attention_extend(const void* q, long long q_batch_stride, int ldq, const void* k_cache,
                                        const void* v_cache, long long cache_batch_stride, int ld_cache, int capacity,
                                        const int* lens, int len_stride, void* out, long long out_batch_stride,
                                        int ldo, int B, int H, int P, int head_dim, float scale, void* stream) {
  const char* who = "b200enc_attention_extend";
  B200_CHECK_ARG(lens != nullptr, "%s: lens=(nil): the query offsets are the device cache lengths", who);
  B200_CHECK_ARG(len_stride == 0 || len_stride == 1, "%s: len_stride=%d must be 0 (one length) or 1 (one per sequence)",
                 who, len_stride);
  B200_CHECK_ARG(capacity >= 1 && P >= 1 && P <= capacity, "%s: P=%d new rows do not fit a cache of capacity=%d", who,
                 P, capacity);
  B200_CHECK_ARG(cache_batch_stride >= (long long)capacity * ld_cache || B == 1,
                 "%s: cache_batch_stride=%lld is smaller than capacity*ld_cache=%lld", who, cache_batch_stride,
                 (long long)capacity * ld_cache);
  const bool aligned = ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k_cache) |
                         reinterpret_cast<uintptr_t>(v_cache)) & 15u) == 0;
  B200_CHECK_ARG(aligned && ldq % 8 == 0 && ld_cache % 8 == 0 && (B == 1 || (q_batch_stride % 8 == 0 &&
                                                                            cache_batch_stride % 8 == 0)),
                 "%s: q and cache rows must be 16-byte aligned (q=%p k_cache=%p v_cache=%p ldq=%d ld_cache=%d)", who, q,
                 k_cache, v_cache, ldq, ld_cache);
  return attention_impl(who, q, q_batch_stride, ldq, k_cache, v_cache, cache_batch_stride, ld_cache, out,
                        out_batch_stride, ldo, B, H, P, capacity, head_dim, scale, B200ENC_ATTN_CAUSAL, nullptr, 0, 0,
                        0, lens, len_stride, stream);
}
