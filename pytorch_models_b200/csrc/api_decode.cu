// C-ABI entry points of incremental decoding (see include/b200enc.h): single-query attention over a KV cache, the
// token + position embedding at the device-side cache length, the length update that ends a decode step, and the row
// writer of an extend (its attention is b200enc_attention_extend in api_attention.cu).
#include "../../include/b200enc.h"
#include "attention_decode.cuh"
#include "host_util.h"

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

// b200enc_attention_decode (len_stride 0) and b200enc_attention_decode_ragged (len_stride 1, append mode only)
int attention_decode(const char* who, const void* q, long long q_batch_stride, const void* k_new, const void* v_new,
                     long long new_batch_stride, void* k_cache, void* v_cache, long long cache_batch_stride,
                     int ld_cache, int capacity, const int* len, int len_stride, int Lkv, void* out,
                     long long out_batch_stride, int B, int H, int head_dim, float scale, float* workspace,
                     long long workspace_bytes, void* stream) {
  if (int rc0 = check_abort(who)) return rc0;
  B200_CHECK_ARG(q && k_cache && v_cache && out && workspace, "%s: null pointer (q=%p k_cache=%p v_cache=%p out=%p "
                 "workspace=%p)", who, q, k_cache, v_cache, out, static_cast<void*>(workspace));
  const bool append = len != nullptr;
  B200_CHECK_ARG(!append || (k_new && v_new), "%s: append mode (len != NULL) needs k_new and v_new", who);
  B200_CHECK_ARG(append || (!k_new && !v_new), "%s: cross mode (len == NULL) takes no k_new / v_new", who);
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
  p.len = len;
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

int embed_rows_at(const char* who, const long long* ids, long long rows, int L, const void* tok, const void* pos,
                  int n_pos, const int* pos0, int pos0_stride, int dtype, int vocab, int d, void* out, void* stream) {
  B200_CHECK_ARG(ids && tok && pos && pos0 && out, "%s: null pointer", who);
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

int decode_advance(const char* who, int* len, int n, int delta, void* stream) {
  B200_CHECK_ARG(len != nullptr, "%s: null len", who);
  B200_CHECK_ARG(n >= 1, "%s: n=%d must be >= 1", who, n);
  const int threads = n < 256 ? n : 256;
  return launch_pdl(decode_advance_kernel, 1, threads, static_cast<cudaStream_t>(stream), len, n, delta);
}
}  // namespace

extern "C" long long b200enc_attention_decode_workspace_bytes(int B, int H, int head_dim, int keys) {
  if (B < 1 || H < 1 || head_dim < 1 || keys < 1) return 0;
  return decode_ws_bytes(B, H, head_dim, keys);
}

extern "C" int b200enc_attention_decode(const void* q, long long q_batch_stride, const void* k_new, const void* v_new,
                                        long long new_batch_stride, void* k_cache, void* v_cache,
                                        long long cache_batch_stride, int ld_cache, int capacity, const int* len,
                                        int Lkv, void* out, long long out_batch_stride, int B, int H, int head_dim,
                                        float scale, float* workspace, long long workspace_bytes, void* stream) {
  return attention_decode("b200enc_attention_decode", q, q_batch_stride, k_new, v_new, new_batch_stride, k_cache,
                          v_cache, cache_batch_stride, ld_cache, capacity, len, 0, Lkv, out, out_batch_stride, B, H,
                          head_dim, scale, workspace, workspace_bytes, stream);
}

extern "C" int b200enc_attention_decode_ragged(const void* q, long long q_batch_stride, const void* k_new,
                                               const void* v_new, long long new_batch_stride, void* k_cache,
                                               void* v_cache, long long cache_batch_stride, int ld_cache, int capacity,
                                               const int* lens, void* out, long long out_batch_stride, int B, int H,
                                               int head_dim, float scale, float* workspace, long long workspace_bytes,
                                               void* stream) {
  const char* who = "b200enc_attention_decode_ragged";
  B200_CHECK_ARG(lens != nullptr, "%s: lens=(nil): per-sequence lengths are append mode only", who);
  return attention_decode(who, q, q_batch_stride, k_new, v_new, new_batch_stride, k_cache, v_cache,
                          cache_batch_stride, ld_cache, capacity, lens, 1, 0, out, out_batch_stride, B, H, head_dim,
                          scale, workspace, workspace_bytes, stream);
}

extern "C" int b200enc_embed_rows_at(const long long* ids, long long rows, int L, const void* tok, const void* pos,
                                     int n_pos, const int* pos0, int dtype, int vocab, int d, void* out, void* stream) {
  return embed_rows_at("b200enc_embed_rows_at", ids, rows, L, tok, pos, n_pos, pos0, 0, dtype, vocab, d, out, stream);
}

extern "C" int b200enc_embed_rows_at_ragged(const long long* ids, long long rows, int L, const void* tok,
                                            const void* pos, int n_pos, const int* pos0, int dtype, int vocab, int d,
                                            void* out, void* stream) {
  return embed_rows_at("b200enc_embed_rows_at_ragged", ids, rows, L, tok, pos, n_pos, pos0, 1, dtype, vocab, d, out,
                       stream);
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

extern "C" int b200enc_decode_advance(int* len, int delta, void* stream) {
  return decode_advance("b200enc_decode_advance", len, 1, delta, stream);
}

extern "C" int b200enc_decode_advance_ragged(int* lens, int n, int delta, void* stream) {
  return decode_advance("b200enc_decode_advance_ragged", lens, n, delta, stream);
}
