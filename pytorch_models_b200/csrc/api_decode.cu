// C-ABI entry points of incremental decoding (see include/b200enc.h): single-query attention over a KV cache, the
// token + position embedding at the device-side cache length, the length update that ends a decode step, and the row
// writer of an extend (its attention is b200enc_attention_extend in api_attention.cu), and the argmax, acceptance and
// n-gram draft kernels of a speculative-decoding round. Every entry point that reads the device lengths takes them as
// (lens, len_stride): sequence b reads lens[b * len_stride], so one function serves a shared length (stride 0) and
// per-sequence lengths (stride 1).
#include "../../include/b200enc.h"
#include "attention_decode.cuh"
#include "host_util.h"
#include "speculative.cuh"

using namespace b200;

namespace {
// Keys per work item. It depends on (B, H, keys) only, never on the device or the current length: the same shapes
// give the same chunking (and so bit-identical results) on every GPU and at every step. About 4096 work items fill
// 148 SMs x 8 CTAs several times over, so the tail of the persistent grid stays short.
int decode_chunk(int B, int H, int keys) {
  constexpr long long kTargetItems = 4096;
  const long long bh = (long long)B * H;
  const long long nch = bh >= kTargetItems ? 1 : (kTargetItems + bh - 1) / bh;
  long long kc = (keys + nch - 1) / nch;
  kc = (kc + DEC_MIN_CHUNK - 1) / DEC_MIN_CHUNK * DEC_MIN_CHUNK;
  return int(kc < DEC_MIN_CHUNK ? DEC_MIN_CHUNK : (kc > DEC_MAX_CHUNK ? DEC_MAX_CHUNK : kc));
}

long long decode_ws_bytes(int B, int H, int head_dim, int keys) {
  const int kc = decode_chunk(B, H, keys);
  return (long long)B * H * ((keys + kc - 1) / kc) * (head_dim + 2) * (long long)sizeof(float);
}

template <typename Kern, typename... Args>
int launch_pdl(Kern kern, int grid, int threads, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  B200_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
}  // namespace

extern "C" long long b200enc_attention_decode_workspace_bytes(int B, int H, int head_dim, int keys) {
  if (B < 1 || H < 1 || head_dim < 1 || keys < 1) return 0;
  return decode_ws_bytes(B, H, head_dim, keys);
}

extern "C" int b200enc_attention_decode(const void* q, long long q_batch_stride, const void* k_new, const void* v_new,
                                        long long new_batch_stride, void* k_cache, void* v_cache,
                                        long long cache_batch_stride, int ld_cache, int capacity, const int* lens,
                                        int len_stride, int Lkv, void* out, long long out_batch_stride, int B, int H,
                                        int head_dim, float scale, float* workspace, long long workspace_bytes,
                                        void* stream) {
  const char* who = "b200enc_attention_decode";
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(q && k_cache && v_cache && out && workspace, "%s: null pointer (q=%p k_cache=%p v_cache=%p out=%p "
                 "workspace=%p)", who, q, k_cache, v_cache, out, static_cast<void*>(workspace));
  B200_CHECK_ARG(len_stride == 0 || len_stride == 1, "%s: len_stride=%d must be 0 (one length) or 1 (one per sequence)",
                 who, len_stride);
  const bool append = lens != nullptr;
  B200_CHECK_ARG(append || len_stride == 0, "%s: lens=(nil) with len_stride=%d: per-sequence lengths are append mode "
                 "only", who, len_stride);
  B200_CHECK_ARG(!append || (k_new && v_new), "%s: append mode (lens != NULL) needs k_new and v_new", who);
  B200_CHECK_ARG(append || (!k_new && !v_new), "%s: cross mode (lens == NULL) takes no k_new / v_new", who);
  B200_CHECK_ARG(head_dim >= 64 && head_dim <= 128 && head_dim % 16 == 0,
                 "%s: head_dim=%d is not supported (64, 80, 96, 112 or 128)", who, head_dim);
  B200_CHECK_ARG(B >= 1 && H >= 1, "%s: bad shape B=%d H=%d", who, B, H);
  B200_CHECK_ARG(capacity >= 1, "%s: capacity=%d must be >= 1", who, capacity);
  B200_CHECK_ARG(append || (Lkv >= 1 && Lkv <= capacity), "%s: Lkv=%d must be in [1, capacity=%d] in cross mode", who,
                 Lkv, capacity);
  const long long width = (long long)H * head_dim;
  B200_CHECK_ARG(ld_cache >= width, "%s: ld_cache=%d is smaller than H*head_dim=%lld", who, ld_cache, width);
  B200_CHECK_ARG(cache_batch_stride >= (long long)capacity * ld_cache || B == 1,
                 "%s: cache_batch_stride=%lld is smaller than capacity*ld_cache=%lld", who, cache_batch_stride,
                 (long long)capacity * ld_cache);
  B200_CHECK_ARG(q_batch_stride >= width || B == 1, "%s: q_batch_stride=%lld is smaller than H*head_dim=%lld", who,
                 q_batch_stride, width);
  B200_CHECK_ARG(out_batch_stride >= width || B == 1, "%s: out_batch_stride=%lld is smaller than H*head_dim=%lld", who,
                 out_batch_stride, width);
  B200_CHECK_ARG(!append || new_batch_stride >= width || B == 1,
                 "%s: new_batch_stride=%lld is smaller than H*head_dim=%lld", who, new_batch_stride, width);
  B200_CHECK_ARG(aligned16(q) && aligned16(k_cache) && aligned16(v_cache) && aligned16(out) &&
                     (!append || (aligned16(k_new) && aligned16(v_new))) && aligned16(workspace),
                 "%s: every tensor must be 16-byte aligned (q=%p k_cache=%p v_cache=%p out=%p)", who, q, k_cache,
                 v_cache, out);
  B200_CHECK_ARG(q_batch_stride % 8 == 0 && out_batch_stride % 8 == 0 && ld_cache % 8 == 0 &&
                     cache_batch_stride % 8 == 0 && (!append || new_batch_stride % 8 == 0),
                 "%s: strides must be multiples of 8 elements (16 bytes): q %lld, out %lld, ld_cache %d, cache batch "
                 "%lld, new rows %lld", who, q_batch_stride, out_batch_stride, ld_cache, cache_batch_stride,
                 new_batch_stride);
  const int keys = append ? capacity : Lkv;
  const long long need = decode_ws_bytes(B, H, head_dim, keys);
  B200_CHECK_ARG(workspace_bytes >= need, "%s: workspace_bytes=%lld, this shape needs %lld "
                 "(b200enc_attention_decode_workspace_bytes)", who, workspace_bytes, need);

  DecodeParams p;
  p.q = static_cast<const __nv_bfloat16*>(q);
  p.q_bs = q_batch_stride;
  p.k_new = static_cast<const __nv_bfloat16*>(k_new);
  p.v_new = static_cast<const __nv_bfloat16*>(v_new);
  p.new_bs = new_batch_stride;
  p.k_cache = static_cast<__nv_bfloat16*>(k_cache);
  p.v_cache = static_cast<__nv_bfloat16*>(v_cache);
  p.cache_bs = cache_batch_stride;
  p.ld_cache = ld_cache;
  p.capacity = capacity;
  p.len = lens;
  p.len_stride = len_stride;
  p.Lkv = append ? 0 : Lkv;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.out_bs = out_batch_stride;
  p.B = B;
  p.H = H;
  p.head_dim = head_dim;
  p.scale_log2e = scale * 1.4426950408889634f;
  p.kc = decode_chunk(B, H, keys);
  p.max_chunks = (keys + p.kc - 1) / p.kc;
  p.ws = workspace;
  const long long items = (long long)B * H * p.max_chunks;
  const long long slots = (long long)sm_count() * DEC_CTAS_PER_SM;
  const int grid = int(items < slots ? items : slots);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const auto partial = len_stride != 0
                           ? (head_dim == 64 ? decode_partial_kernel<8, true> : decode_partial_kernel<16, true>)
                           : (head_dim == 64 ? decode_partial_kernel<8, false> : decode_partial_kernel<16, false>);
  if (int rc = launch_pdl(partial, grid, DEC_THREADS, s, p)) return rc;
  return launch_pdl(decode_combine_kernel, B * H, 128, s, p);
}

extern "C" int b200enc_embed_rows_at(const long long* ids, long long rows, int L, const void* tok, const void* pos,
                                     int n_pos, const int* pos0, int pos0_stride, int dtype, int vocab, int d,
                                     void* out, void* stream) {
  const char* who = "b200enc_embed_rows_at";
  B200_CHECK_ARG(ids && tok && pos && pos0 && out, "%s: null pointer", who);
  B200_CHECK_ARG(pos0_stride == 0 || pos0_stride == 1,
                 "%s: pos0_stride=%d must be 0 (one length) or 1 (one per sequence)", who, pos0_stride);
  B200_CHECK_ARG(rows >= 1 && L >= 1 && rows % L == 0, "%s: rows=%lld must be a positive multiple of L=%d", who, rows,
                 L);
  B200_CHECK_ARG(vocab >= 1 && n_pos >= 1, "%s: vocab=%d and n_pos=%d must be >= 1", who, vocab, n_pos);
  B200_CHECK_ARG(d >= 8 && d % 8 == 0, "%s: d=%d must be a multiple of 8", who, d);
  B200_CHECK_ARG(aligned16(out), "%s: out must be 16-byte aligned", who);
  const long long total = rows * (d / 8);
  const unsigned grid = unsigned((total + 255) / 256);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* dst = static_cast<__nv_bfloat16*>(out);
  if (dtype == B200ENC_DTYPE_BF16)
    embed_rows_at_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(ids, rows, L, static_cast<const __nv_bfloat16*>(tok),
                                                             static_cast<const __nv_bfloat16*>(pos), n_pos, pos0,
                                                             pos0_stride, vocab, d, dst);
  else if (dtype == B200ENC_DTYPE_F32)
    embed_rows_at_kernel<float><<<grid, 256, 0, s>>>(ids, rows, L, static_cast<const float*>(tok),
                                                     static_cast<const float*>(pos), n_pos, pos0, pos0_stride, vocab,
                                                     d, dst);
  else
    return set_error(-1, "%s: unsupported dtype %d", who, dtype);
  B200_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int b200enc_kv_append(const void* src, long long src_batch_stride, int ld_src, void* cache,
                                 long long cache_batch_stride, int ld_cache, int capacity, const int* lens,
                                 int len_stride, int B, int P, int width, void* stream) {
  const char* who = "b200enc_kv_append";
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(src && cache && lens, "%s: null pointer (src=%p cache=%p lens=%p)", who, src, cache,
                 static_cast<const void*>(lens));
  B200_CHECK_ARG(len_stride == 0 || len_stride == 1, "%s: len_stride=%d must be 0 (one length) or 1 (one per sequence)",
                 who, len_stride);
  B200_CHECK_ARG(B >= 1 && P >= 1 && width >= 8 && width % 8 == 0, "%s: bad shape B=%d P=%d width=%d (a multiple of 8)",
                 who, B, P, width);
  B200_CHECK_ARG(capacity >= 1 && P <= capacity, "%s: P=%d new rows do not fit a cache of capacity=%d", who, P,
                 capacity);
  B200_CHECK_ARG(ld_src >= width && ld_cache >= width, "%s: ld_src=%d / ld_cache=%d smaller than width=%d", who, ld_src,
                 ld_cache, width);
  B200_CHECK_ARG(cache_batch_stride >= (long long)capacity * ld_cache || B == 1,
                 "%s: cache_batch_stride=%lld is smaller than capacity*ld_cache=%lld", who, cache_batch_stride,
                 (long long)capacity * ld_cache);
  B200_CHECK_ARG(aligned16(src) && aligned16(cache) && ld_src % 8 == 0 && ld_cache % 8 == 0 &&
                     (B == 1 || (src_batch_stride % 8 == 0 && cache_batch_stride % 8 == 0)),
                 "%s: rows must be 16-byte aligned (src=%p cache=%p ld_src=%d ld_cache=%d)", who, src, cache, ld_src,
                 ld_cache);
  const long long total = (long long)B * P * (width / 8);
  return launch_pdl(kv_append_kernel, int((total + 255) / 256), 256, static_cast<cudaStream_t>(stream),
                    static_cast<const __nv_bfloat16*>(src), src_batch_stride, ld_src,
                    static_cast<__nv_bfloat16*>(cache), cache_batch_stride, ld_cache, capacity, lens, len_stride, B, P,
                    width);
}

extern "C" int b200enc_decode_advance(int* lens, int n, int delta, void* stream) {
  const char* who = "b200enc_decode_advance";
  B200_CHECK_ARG(lens != nullptr, "%s: null lens", who);
  B200_CHECK_ARG(n >= 1, "%s: n=%d must be >= 1", who, n);
  const int threads = n < 256 ? n : 256;
  return launch_pdl(decode_advance_kernel, 1, threads, static_cast<cudaStream_t>(stream), lens, n, delta);
}

extern "C" int b200enc_argmax_rows(const void* logits, long long ld, int rows, int V, long long* out,
                                   long long out_stride, void* stream) {
  const char* who = "b200enc_argmax_rows";
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(logits && out, "%s: null pointer (logits=%p out=%p)", who, logits, static_cast<void*>(out));
  B200_CHECK_ARG(rows >= 1 && V >= 1, "%s: bad shape rows=%d V=%d", who, rows, V);
  B200_CHECK_ARG(ld >= V, "%s: ld=%lld is smaller than V=%d", who, ld, V);
  B200_CHECK_ARG(aligned16(logits) && ld % 8 == 0, "%s: logits rows must be 16-byte aligned (logits=%p ld=%lld)", who,
                 logits, ld);
  B200_CHECK_ARG(out_stride >= 1 || rows == 1, "%s: out_stride=%lld must be >= 1", who, out_stride);
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 7u) == 0, "%s: out=%p must be 8-byte aligned", who,
                 static_cast<void*>(out));
  return launch_pdl(argmax_rows_kernel, rows, ARGMAX_THREADS, static_cast<cudaStream_t>(stream),
                    static_cast<const __nv_bfloat16*>(logits), ld, V, out, out_stride);
}

extern "C" int b200enc_speculative_accept(const long long* picks, long long* ids, int* budget, long long eos,
                                          int* len_target, int target_len_stride, int* len_draft,
                                          int draft_len_stride, long long* emitted, long long* n_emitted,
                                          long long out_stride, int B, int k, void* stream) {
  const char* who = "b200enc_speculative_accept";
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(picks && ids && budget && len_target && len_draft && emitted && n_emitted,
                 "%s: null pointer (picks=%p ids=%p budget=%p len_target=%p len_draft=%p emitted=%p n_emitted=%p)",
                 who, static_cast<const void*>(picks), static_cast<void*>(ids), static_cast<void*>(budget),
                 static_cast<void*>(len_target), static_cast<void*>(len_draft), static_cast<void*>(emitted),
                 static_cast<void*>(n_emitted));
  B200_CHECK_ARG(B >= 1, "%s: B=%d must be >= 1", who, B);
  B200_CHECK_ARG(k >= 1 && k <= 15, "%s: k=%d draft tokens, must be in [1, 15]", who, k);
  B200_CHECK_ARG(target_len_stride == 1 || (target_len_stride == 0 && B == 1),
                 "%s: target_len_stride=%d must be 1 (one length per sequence), or 0 (one length) with B=1 (B=%d)",
                 who, target_len_stride, B);
  B200_CHECK_ARG(draft_len_stride == 1 || (draft_len_stride == 0 && B == 1),
                 "%s: draft_len_stride=%d must be 1 (one length per sequence), or 0 (one length) with B=1 (B=%d)", who,
                 draft_len_stride, B);
  B200_CHECK_ARG(out_stride >= k + 1 || B == 1, "%s: out_stride=%lld is smaller than k+1=%d", who, out_stride, k + 1);
  B200_CHECK_ARG(eos >= -1, "%s: eos=%lld must be a token id or -1 (none)", who, eos);
  return launch_pdl(speculative_accept_kernel, (B + 127) / 128, 128, static_cast<cudaStream_t>(stream), picks, ids,
                    budget, eos, len_target, target_len_stride, len_draft, draft_len_stride, emitted, n_emitted,
                    out_stride, B, k);
}

extern "C" int b200enc_ngram_draft(long long* hist, long long hist_stride, int capacity, int* len, int len_stride,
                                   long long* ids, int B, int k, int max_ngram, int min_ngram, void* stream) {
  const char* who = "b200enc_ngram_draft";
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(hist && len && ids, "%s: null pointer (hist=%p len=%p ids=%p)", who, static_cast<void*>(hist),
                 static_cast<void*>(len), static_cast<void*>(ids));
  B200_CHECK_ARG(B >= 1, "%s: B=%d must be >= 1", who, B);
  B200_CHECK_ARG(k >= 1 && k <= 15, "%s: k=%d draft tokens, must be in [1, 15]", who, k);
  B200_CHECK_ARG(min_ngram >= 1 && min_ngram <= max_ngram && max_ngram <= NGRAM_MAX,
                 "%s: min_ngram=%d and max_ngram=%d must satisfy 1 <= min_ngram <= max_ngram <= %d", who, min_ngram,
                 max_ngram, NGRAM_MAX);
  B200_CHECK_ARG(len_stride == 1 || (len_stride == 0 && B == 1),
                 "%s: len_stride=%d must be 1 (one length per sequence), or 0 (one length) with B=1 (B=%d)", who,
                 len_stride, B);
  B200_CHECK_ARG(capacity >= k + 1, "%s: capacity=%d cannot hold the k+1=%d rows of a round", who, capacity, k + 1);
  B200_CHECK_ARG(hist_stride >= capacity || B == 1, "%s: hist_stride=%lld is smaller than capacity=%d", who,
                 hist_stride, capacity);
  B200_CHECK_ARG(((reinterpret_cast<uintptr_t>(hist) | reinterpret_cast<uintptr_t>(ids)) & 7u) == 0,
                 "%s: hist=%p and ids=%p must be 8-byte aligned", who, static_cast<void*>(hist),
                 static_cast<void*>(ids));
  return launch_pdl(ngram_draft_kernel, B, NGRAM_THREADS, static_cast<cudaStream_t>(stream), hist, hist_stride,
                    capacity, len, len_stride, ids, k, max_ngram, min_ngram);
}
