/*
 * b200enc — C-ABI of the B200-native encoder-block hot path (libb200enc.so).
 *
 * The reference (gau-nernst/pytorch-models) has no FFI: its boundary for this path is the nn.Module protocol of
 * pytorch_models/transformer.py. Each entry point below replaces the ATen ops that one reference call site
 * dispatches (cited per function). All tensors are device pointers owned by the caller (PyTorch); activations and
 * weights are bf16 row-major, vectors and statistics fp32. Every call enqueues on `stream` (a cudaStream_t) and
 * returns without synchronising; nothing is allocated or freed by the library.
 *
 * Return value: 0 = ok; < 0 = argument / shape / alignment error (-3: an earlier kernel gave up on a barrier wait, see
 * b200enc_async_status); > 0 = cudaError_t or CUresult.
 * b200enc_last_error() returns a thread-local description of the last non-zero return.
 */
#ifndef B200ENC_H_
#define B200ENC_H_

#ifdef __cplusplus
extern "C" {
#endif

#define B200ENC_VERSION 100

int b200enc_version(void);
const char* b200enc_last_error(void);

/*
 * Device-side health. The tcgen05 kernels synchronise their warps through on-chip barriers; every such wait is
 * bounded (4 s). A wait that runs out stores a non-zero code into a process-wide status word (mapped host memory),
 * after which the kernel drains without hanging the GPU and every later entry point returns -3 instead of enqueueing
 * work whose inputs are invalid. Kernels never printf, trap or abort (reference convention: Python exceptions only).
 * Returns the status word (0 = healthy); clear != 0 also resets it.
 */
unsigned int b200enc_async_status(int clear);

/* Tensor maps (CUtensorMap) are encoded once per distinct (pointer, shape, strides, box) and cached; counters for tests. */
void b200enc_tensor_map_cache_stats(unsigned long long* hits, unsigned long long* misses);

/* flags for b200enc_linear */
#define B200ENC_LINEAR_GELU 1          /* exact (erf) GELU after bias: nn.GELU(), transformer.py:61 */
#define B200ENC_LINEAR_GELU_TANH 2     /* tanh GELU after bias: nn.GELU(approximate="tanh"), transformer.py:62 (no residual) */
#define B200ENC_LINEAR_RELU 4          /* nn.ReLU, transformer.py:63 (no residual) */
#define B200ENC_LINEAR_SILU 8          /* nn.SiLU, transformer.py:64 (no residual) */
#define B200ENC_LINEAR_FP8 16           /* OPTIONAL variant, never the default: x and w are e4m3 bytes, see acc_scale below */
/* any other flag bit is refused (-1) */

/*
 * out[b][m][n] = epi( sum_k x[b][m][k] * w[n][k] )   for b < batches, m < M, n < N      (tcgen05 GEMM)
 *
 * Replaces nn.Linear at transformer.py:47-49 (q/k/v projections, fused as one [3d,d] weight), :53 (out_proj),
 * :59 (linear1 + nn.GELU :61), :66 (linear2), the residual adds at :125-126, and — with x = patch rows —
 * the patch-embedding Conv2d at image/vit.py:78 plus the positional add at :79.
 *
 *   epi(acc) = acc + bias[n]                                        (colsum == NULL)
 *            = rstd[m]*(acc - mean[m]*colsum[n]) + bias[n]           (LayerNorm folded into the GEMM: w must be
 *              gamma-scaled, colsum[n] = sum_k w[n][k], bias[n] = W.beta + b)
 *   then GELU if flags & B200ENC_LINEAR_GELU (or its tanh form with B200ENC_LINEAR_GELU_TANH), then + residual[b][m][n] if residual != NULL
 *   (res_batch_stride == 0 broadcasts one [M, N] table over the batch: the positional embedding).
 *
 * Row statistics of the folded LayerNorm come in one of two forms:
 *   rowstats_parts == 0 : rowstats[b*M + m] = (mean, rstd)                  (written by b200enc_row_stats)
 *   rowstats_parts  > 0 : rowstats[(b*M + m)*parts + t] = (mean_t, M2_t) of columns [128t, 128t+128) of row m of x,
 *                         as written through `stats_out` by the b200enc_linear call that produced x; they are
 *                         combined in a fixed order (Chan's parallel variance) with ln_eps. parts = ceil(K/128) <= 12.
 * stats_out (optional, needs a residual epilogue): per-128-column (mean, M2) of the bf16-rounded OUTPUT rows, laid
 * out [(b*M + m)][ceil(N/128)] — the fused replacement of the row pass of the next LayerNorm.
 *
 * Strides are in elements. K and N must be multiples of 8; rows 16-byte aligned. x rows may overlap (ldx < K).
 */
typedef struct b200enc_linear_args {
  const void* x;               /* bf16 [batches][M][K], row stride ldx, batch stride x_batch_stride */
  long long x_batch_stride;
  int ldx;
  const void* w;               /* bf16 [N][K], row stride ldw */
  int ldw;
  const float* bias;           /* fp32 [N] or NULL */
  const float* colsum;         /* fp32 [N] or NULL (LayerNorm fold) */
  const float* rowstats;       /* fp32 pairs, see above; required iff colsum != NULL */
  int rowstats_parts;
  float ln_eps;
  const void* residual;        /* bf16 [batches or 1][M][N] or NULL */
  long long res_batch_stride;
  int ldr;
  void* out;                   /* bf16 [batches][M][N] */
  long long out_batch_stride;
  int ldo;
  float* stats_out;            /* fp32 pairs [(batches*M)][ceil(N/128)] or NULL */
  int batches, M, N, K;
  int flags;
  int stats_rows_per_batch;    /* 0 = M. Otherwise row (b, m) of stats_out lives at b*stats_rows_per_batch +            */
  int stats_row_offset;        /* stats_row_offset + m: lets the patch-embedding GEMM, which writes tokens 1.. of every */
                               /* image, put its statistics where the first encoder layer looks for them               */
  const float* acc_scale;      /* B200ENC_LINEAR_FP8 only: DEVICE pointer to one fp32, the product of the per-tensor   */
                               /* dequantisation scales of x and w: out = epi(acc_scale * sum_k x8*w8 + bias ...).     */
                               /* The FP8 variant (SURVEY §8 f rank 4) has no counterpart in the reference (its linears */
                               /* are nn.Linear in the module's dtype, transformer.py:28-31,59,66); it exists as an    */
                               /* opt-in with its own tolerance: K % 16 == 0, no LayerNorm fold, no statistics output. */
} b200enc_linear_args;

int b200enc_linear(const b200enc_linear_args* args, void* stream);

/*
 * tokens[b][patch][:] = conv(img[b])[:, ph, pw] + bias + residual[patch][:]   (patch = ph * (W/16) + pw)
 *
 * nn.Conv2d(3, d, 16, 16) + flatten + transpose + positional embedding (image/vit.py:64,78-79) as ONE GEMM whose A
 * operand is the NCHW bf16 image itself: no im2col / patch-row buffer (b200enc_patch_rows + b200enc_linear remain
 * for other patch sizes and fp32 images). Uses the fields of b200enc_linear_args as follows: x = image
 * [batches][3][img_h][img_w] bf16 contiguous (ldx, x_batch_stride ignored), w = conv.weight viewed as [N][768],
 * M = (img_h/16)*(img_w/16), K = 768, bias, residual (required: the positional rows, res_batch_stride 0 broadcasts
 * them), out / out_batch_stride / ldo (point `out` at token 1 of image 0 to leave room for a class token),
 * stats_out / stats_rows_per_batch / stats_row_offset as in b200enc_linear; colsum, rowstats, flags must be 0.
 */
int b200enc_patch_embed16(const b200enc_linear_args* args, int img_h, int img_w, void* stream);

/* flags for b200enc_attention */
#define B200ENC_ATTN_CAUSAL 1 /* key j only visible to queries i >= j (is_causal=True of SDPA: DecoderLayer, transformer.py:97) */
#define B200ENC_ATTN_GENERAL 131072 /* use the streaming (online-softmax) kernel even where the short-sequence kernel
                                       applies: the reference the tests check the short kernel against */
/* any other flag bit is refused (-1) */

/*
 * out[b][i][hd*h + :] = softmax_j( q[b][i][hd*h + :] . k[b][j][hd*h + :] * scale ) v[b][j][hd*h + :],  hd = head_dim
 *
 * Replaces F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0, is_causal=False) at
 * transformer.py:52 together with the head split/merge views at :47-49 and :53: q, k, v are column slices of the
 * projection output (row strides ldq / ldkv, head h at columns [hd*h, hd*h + hd)), the result is head-interleaved
 * [B, Lq, H*hd] ready for out_proj. head_dim is 64 (every BASELINE config) or 80, 96, 112, 128 (ViT-H/14: 80); any
 * other value is refused. Lq != Lkv is allowed (the 1-query MAP pooling head, image/vit.py:41). K/V stream in blocks
 * of 128 rows with an online softmax. With B200ENC_ATTN_CAUSAL the K/V blocks above the diagonal are skipped entirely.
 * head_dim 64: unmasked calls with Lkv <= 256 (ViT-B/16 at 224 px: 197 tokens) take a single-pass kernel instead: the
 * whole score row of a query lives in tensor memory, exact maximum, no rescaling (csrc/attention_short.cuh).
 * head_dim 80-128 run one streaming kernel for every shape, mask and bias (csrc/attention_wide.cuh).
 */
int b200enc_attention(const void* q, long long q_batch_stride, int ldq, const void* k, const void* v,
                      long long kv_batch_stride, int ldkv, void* out, long long out_batch_stride, int ldo, int B,
                      int H, int Lq, int Lkv, int head_dim, float scale, int flags, void* stream);

/*
 * out[r][:] = (x[r][:] - mean_r) * rsqrt(var_r + eps) * gamma + beta, biased variance (nn.LayerNorm:
 * transformer.py:87,93; vit.py:69,83; whisper.py:27,33; bert.py:31,37). Row r of x starts at x + r*ldx elements, so a
 * strided view (e.g. only the class-token rows, vit.py:20-22) can be normalised without a gather.
 * stats (optional) receives (mean, rstd) pairs.
 */
int b200enc_layernorm(const void* x, long long ldx, const float* gamma, const float* beta, float eps, int rows, int d,
                      void* out, long long ldo, float* stats, void* stream);

/* stats[r] = (mean_r, rsqrt(var_r + eps)) only: the per-row half of a LayerNorm folded into the next GEMM. */
int b200enc_row_stats(const void* x, long long ldx, float eps, int rows, int d, float* stats, void* stream);

/* out[b][:] = mean over the L token rows of x[b] (GlobalAveragePooling, image/vit.py:25-27). */
int b200enc_mean_tokens(const void* x, long long batch_stride, long long ldx, int B, int L, int d, void* out,
                        long long ldo, void* stream);

#define B200ENC_DTYPE_BF16 0
#define B200ENC_DTYPE_F32 1

/*
 * rows[b*P + ph*(W/p) + pw][c*p*p + i*p + j] = img[b][c][ph*p + i][pw*p + j]  (NCHW image, 3 channels), bf16, row
 * stride Kpad with zero padding: the A operand that turns nn.Conv2d(3, d, p, p) (image/vit.py:64,78) into
 * b200enc_linear with w = conv.weight.view(d, 3*p*p).
 */
int b200enc_patch_rows(const void* img, int img_dtype, int B, int H, int W, int p, int Kpad, void* rows, void* stream);

/* tokens[b][0][:] = cls[:] for every image (torch.cat([cls_token, out], -2) at image/vit.py:80-81). */
int b200enc_cls_rows(const void* cls, int B, int d, void* tokens, long long batch_stride, void* stream);

/*
 * b200enc_attention with an additive bias: softmax_j(scale * q_i . k_j + bias[b][h][i][j]) — the `attn_bias` argument
 * of MHA.forward (transformer.py:41,52: SDPA's attn_mask; T5's relative position bias). bias is fp32 with element
 * strides (batch, head, query row); a stride of 0 broadcasts over that dimension, consecutive keys are contiguous.
 * -inf entries mask a key. May be combined with B200ENC_ATTN_CAUSAL. The bias is read straight from global memory
 * by the softmax threads (one row each): correct for any shape, but slower than the unbiased kernel.
 */
int b200enc_attention_bias(const void* q, long long q_batch_stride, int ldq, const void* k, const void* v,
                           long long kv_batch_stride, int ldkv, void* out, long long out_batch_stride, int ldo, int B,
                           int H, int Lq, int Lkv, int head_dim, float scale, int flags, const float* bias,
                           long long bias_b_stride, long long bias_h_stride, long long bias_row_stride, void* stream);

/*
 * Token + position embedding: out[r][:] = bf16(tok[ids[r]][:] + pos[r % L][:]) for r < rows (= batch * L).
 * Replaces `self.token_embs(x) + self.pos_embs[:L]` (text/bert.py:35-36, text/gpt2.py:22-23, text/gpt.py:25-26,
 * audio2text/whisper.py:47-48). ids: int64 device pointer; tok [vocab, d] and pos [>= L, d] contiguous, both `dtype`
 * (B200ENC_DTYPE_*); d % 8 == 0; out [rows, d] bf16 contiguous. A row whose id is outside [0, vocab) is set to NaN.
 */
int b200enc_embed_rows(const long long* ids, long long rows, int L, const void* tok, const void* pos, int dtype,
                       int vocab, int d, void* out, void* stream);

/*
 * rows[n][t + 1][c] = x[n][c][t], rows[n][0] = rows[n][T + 1] = 0   (x: (N, C, T) fp32/bf16 -> (N, T+2, C) bf16).
 * Time-major, zero-padded input of the Whisper conv stem (nn.Conv1d(k=3, pad=1) at audio2text/whisper.py:16-21): output
 * step t of a stride-s convolution reads the 3*C contiguous values starting at row s*t, so each convolution is a
 * b200enc_linear call over an overlapping strided view with w[n][k*C + c] = conv.weight[n][c][k].
 */
int b200enc_time_rows(const void* x, int dtype, int N, int C, int T, void* rows, void* stream);

/*
 * Whisper audio front end: out[n][m][t] = (max(log10(mel[n][m][t]), max_n - 8) + 4) / 4 with
 * mel = filters @ |STFT(audio, n_fft 400, hop 160, periodic Hann, centred, reflect padded)|^2, t < T = L / 160 and
 * max_n the maximum of the log-mel values of sample n. Replaces WhisperPreprocessor.forward
 * (audio2text/whisper.py:143-148) = MelSpectrogram / Spectrogram (audio/spectrogram.py:15-16,44-45). fp32 throughout.
 * audio [N][audio_stride] (L valid samples each, L > 200); filters_t [201][n_mels] = the mel filter bank transposed;
 * out [N][n_mels][T] contiguous; sample_max: N ints of scratch.
 */
int b200enc_whisper_logmel(const float* audio, long long audio_stride, int N, int L, const float* filters_t, int n_mels,
                           float* out, int* sample_max, void* stream);

/*
 * Incremental decoding.
 *
 * Device cache lengths: the lengths of a KV cache live in device int32 memory, so a step's arguments are the same at
 * every position (CUDA-graph capture) and the host never reads them back. Every entry point below that reads them
 * takes a pointer `lens` and a stride `len_stride`: sequence b reads lens[b * len_stride]. len_stride 0 gives the
 * batch one shared length (lens holds 1 int), 1 gives each sequence its own (lens holds B ints: a ragged batch, the
 * prompts of text/generator.py:11-39 run several at a time). Any other stride is refused (-1).
 */

/*
 * Single-query attention over a KV cache (csrc/attention_decode.cuh).
 *
 *   out[b][hd*h + :] = softmax_j( q[b][hd*h + :] . k[b][j][hd*h + :] * scale ) v[b][j][hd*h + :]
 *
 * Replaces F.scaled_dot_product_attention at transformer.py:52 for ONE query row per sequence, where the keys and
 * values of the earlier positions come from a cache instead of being recomputed: the causal self-attention of
 * DecoderLayer (transformer.py:97) one token at a time, and its cross-attention (:98) against a memory whose k|v
 * projection was computed once. head_dim is 64, 80, 96, 112 or 128. q, out: one row per sequence (batch strides in
 * elements). k_cache / v_cache: [B][capacity] rows of row stride ld_cache and batch stride cache_batch_stride (the K
 * and V halves of one k|v buffer are two pointers with the same strides).
 *
 *   append mode (lens != NULL): with n_b = lens[b * len_stride] (the device cache lengths above), the keys of sequence
 *     b are cache rows [0, n_b) plus the new row k_new / v_new (the step's output of the fused q|k|v projection, batch
 *     stride new_batch_stride). The new row is also written to cache row n_b; the caller advances the lengths
 *     (b200enc_decode_advance). An n_b outside [0, capacity) gives NaN outputs and writes no cache row for sequence b
 *     only. Lkv is ignored. With per-sequence lengths, work items past a sequence's own length are skipped, so the K/V
 *     bytes read follow the sum of the lengths; with equal lengths the outputs are bit-identical to len_stride 0.
 *   cross mode (lens == NULL, k_new = v_new = NULL, len_stride 0): the keys are cache rows [0, Lkv), Lkv <= capacity;
 *     read-only. Per-sequence lengths are append mode only.
 *
 * workspace: fp32 device scratch of at least b200enc_attention_decode_workspace_bytes(B, H, head_dim, keys) bytes with
 * keys = capacity (append mode) or Lkv (cross mode): per (sequence, head, chunk of keys) the partial softmax state.
 * Two launches: the chunk partials, then their combination in a fixed order (repeats are bit-identical).
 */
int b200enc_attention_decode(const void* q, long long q_batch_stride, const void* k_new, const void* v_new,
                             long long new_batch_stride, void* k_cache, void* v_cache, long long cache_batch_stride,
                             int ld_cache, int capacity, const int* lens, int len_stride, int Lkv, void* out,
                             long long out_batch_stride, int B, int H, int head_dim, float scale, float* workspace,
                             long long workspace_bytes, void* stream);

/* Workspace size in bytes of b200enc_attention_decode (0 for non-positive arguments). Host-only, no device needed. */
long long b200enc_attention_decode_workspace_bytes(int B, int H, int head_dim, int keys);

/*
 * b200enc_embed_rows at positions held on the device: out[r][:] = bf16(tok[ids[r]][:] + pos[p_s + r % L][:]) for
 * r < rows, with s = r / L the sequence of row r and p_s = pos0[s * pos0_stride] (the device cache lengths above). The
 * embedding of a decode step (text/gpt2.py:22-23 at position L - 1 of each growing sequence). pos has n_pos rows; a
 * position outside [0, n_pos) or an id outside [0, vocab) gives a NaN row.
 */
int b200enc_embed_rows_at(const long long* ids, long long rows, int L, const void* tok, const void* pos, int n_pos,
                          const int* pos0, int pos0_stride, int dtype, int vocab, int d, void* out, void* stream);

/*
 * Extending a filled KV cache by P rows per sequence (multi-turn continuation, chunked prefill): causal attention whose
 * queries start at each sequence's cache length ("bottom-right aligned").
 *
 *   out[b][i][hd*h + :] = softmax_{j <= n_b + i}( q[b][i][hd*h + :] . k[b][j][hd*h + :] * scale ) v[b][j][hd*h + :]
 *
 * with n_b = lens[b * len_stride] the device cache length of sequence b (the device cache lengths above) and i < P.
 * Replaces F.scaled_dot_product_attention at transformer.py:52 for the causal self-attention of DecoderLayer
 * (transformer.py:97) when the keys and values of the first n_b positions come from a cache: the P query rows see the
 * cached keys and the new ones up to their own position. The new rows' k|v must already be in cache rows [n_b, n_b + P)
 * (b200enc_kv_append), so every key is read from the cache. q, out: P rows per sequence as in b200enc_attention;
 * k_cache / v_cache: [B][capacity] rows of row stride ld_cache and batch stride cache_batch_stride (the K and V halves
 * of one k|v buffer). head_dim 64 or 80-128 (the streaming kernels of b200enc_attention with the causal diagonal
 * shifted by n_b). Only the K/V blocks below row n_b + P are read, so a ragged batch costs what its own lengths cost.
 * The lengths are read on the device; P <= capacity is checked here and n_b + P <= capacity is the caller's (a sequence
 * whose n_b is outside [0, capacity - P] gets NaN outputs).
 * With n_b = 0 the result is bit-identical to b200enc_attention with B200ENC_ATTN_CAUSAL on the same rows.
 */
int b200enc_attention_extend(const void* q, long long q_batch_stride, int ldq, const void* k_cache, const void* v_cache,
                             long long cache_batch_stride, int ld_cache, int capacity, const int* lens, int len_stride,
                             void* out, long long out_batch_stride, int ldo, int B, int H, int P, int head_dim,
                             float scale, void* stream);

/*
 * cache[b][n_b + r][:width] = src[b][r][:width] for r < P, n_b = lens[b * len_stride] (the device cache lengths
 * above): writes the k|v rows of the fused q|k|v projection (transformer.py:47-49) into a KV cache at each sequence's
 * length, ahead of b200enc_attention_extend. bf16, strides in elements, rows 16-byte aligned, width % 8 == 0. A row
 * that would land outside [0, capacity) is not written; the lengths are not changed.
 */
int b200enc_kv_append(const void* src, long long src_batch_stride, int ld_src, void* cache, long long cache_batch_stride,
                      int ld_cache, int capacity, const int* lens, int len_stride, int B, int P, int width,
                      void* stream);

/*
 * lens[i] += delta for i < n on the device cache lengths above (n = 1: the shared length, n = B: one per sequence):
 * the last launch of a decode step, so that the captured step can be replayed.
 */
int b200enc_decode_advance(int* lens, int n, int delta, void* stream);

/*
 * Greedy speculative decoding: the picks and the acceptance of one round (draft steps, one verify extend of the last
 * token and k draft tokens, the argmax of its k + 1 logits rows per sequence, then the acceptance below), all on the
 * device, so that a round can be captured as one CUDA graph.
 *
 * out[r * out_stride] = argmax_j logits[r * ld + j] over j < V for r < rows: bf16 logits rows of row stride ld (the
 * tied-logits GEMM writes rows of ceil8(V) columns; the columns past V are never picked), int64 indices. The order is
 * torch.argmax's: NaN is greater than any number and of equal values the lowest index wins. One kernel.
 */
int b200enc_argmax_rows(const void* logits, long long ld, int rows, int V, long long* out, long long out_stride,
                        void* stream);

/*
 * The acceptance of a round with k in [1, 15] draft tokens, one thread per sequence b. ids (B, k+1) int64 holds the
 * verify extend's input [last, d_1 .. d_k] per sequence, picks (B, k+1) int64 the target's argmax of each verify row
 * [t_0 .. t_k]. With a the number of leading i < k where t_i == d_{i+1}, the candidates are d_1 .. d_a, t_a; they are
 * cut after the first token equal to eos (-1: none) and at budget[b] tokens (a budget <= 0 keeps none), leaving m.
 * Writes emitted[b * out_stride + i] = the kept tokens for i < m and -1 up to i = k, n_emitted[b * out_stride] = m,
 * budget[b] -= m (0 after an EOS), len[b * len_stride] -= k + 1 - m in both caches (the target's extend and the
 * draft's k + 1 steps each added k + 1 rows; the kept ones are last and the accepted drafts), and ids[b][0] = the last
 * kept token when m > 0, the next round's input. The lengths are the device cache lengths above, with a shared length
 * (stride 0) accepted only when B = 1.
 */
int b200enc_speculative_accept(const long long* picks, long long* ids, int* budget, long long eos, int* len_target,
                               int target_len_stride, int* len_draft, int draft_len_stride, long long* emitted,
                               long long* n_emitted, long long out_stride, int B, int k, void* stream);

/*
 * Draft-free proposals: the k in [1, 15] drafts of a round by n-gram lookup in each sequence's own token history, in
 * place of the draft model's steps. hist (B, capacity) int64 with row stride hist_stride holds n = len[b * len_stride]
 * tokens of sequence b (len_stride as in b200enc_speculative_accept); ids (B, k+1) int64 holds last in column 0. With s = hist[b][0, n)
 * followed by last: for g = max_ngram down to min_ngram (1 <= min_ngram <= max_ngram <= 8, g <= n), the suffix
 * s[n-g+1 .. n] is looked up at its latest earlier end e < n; the first g that occurs gives d_i = s'[e + i] for
 * i = 1..k, s' being s followed by the drafts themselves (so a periodic history keeps its period), and no match gives
 * d_i = last. Writes ids[b][1..k] = d, hist[b][n] = last, hist[b][n+1 .. n+k] = d and len += k + 1: the history then
 * holds the rows the verify appends to the target cache, and b200enc_speculative_accept rolls both back alike. A
 * length outside [0, capacity - k - 1] gets d_i = last and no history write, and still advances by k + 1. Rows at or
 * past len are never read. One CTA per sequence.
 */
int b200enc_ngram_draft(long long* hist, long long hist_stride, int capacity, int* len, int len_stride, long long* ids,
                        int B, int k, int max_ngram, int min_ngram, void* stream);

/*
 * Launch plan: a recorded sequence of the entry points above, enqueued by ONE call.
 *
 * The reference's forward is a Python loop over modules (nn.Sequential at transformer.py:133-149, the layer body at
 * :122-130); the drop-in modules of this package used to make one ctypes call per kernel from the same kind of loop,
 * which costs ~29 us of interpreter time per launch (1.9 ms for the 65 launches of a ViT-B/16 forward). A model
 * records its launches once per (input shape, weights) — every argument of every call, workspaces included — and
 * replays the array; only the input / output pointers are patched by the host between replays. Each element names
 * an entry point (`kind`) and carries its arguments in declaration order: the struct for the two GEMM entry points,
 * pointer arguments in p[], integer arguments (int / long long) in i[], float arguments in f[]. The calls are
 * made in order on `stream`, with the same validation and error behaviour as the individual entry points; on a
 * non-zero return *failed_op (if not NULL) is the index of the element that failed and nothing after it was enqueued.
 */
#define B200ENC_OP_LINEAR 1
#define B200ENC_OP_PATCH_EMBED16 2   /* i[0] = img_h, i[1] = img_w */
#define B200ENC_OP_ATTENTION 3
#define B200ENC_OP_ATTENTION_BIAS 4
#define B200ENC_OP_LAYERNORM 5
#define B200ENC_OP_ROW_STATS 6
#define B200ENC_OP_MEAN_TOKENS 7
#define B200ENC_OP_PATCH_ROWS 8
#define B200ENC_OP_CLS_ROWS 9
#define B200ENC_OP_EMBED_ROWS 10
#define B200ENC_OP_TIME_ROWS 11

typedef struct b200enc_op {
  int kind;                    /* B200ENC_OP_* */
  int reserved;
  b200enc_linear_args linear;  /* B200ENC_OP_LINEAR, B200ENC_OP_PATCH_EMBED16 */
  const void* p[8];
  long long i[16];
  float f[2];
} b200enc_op;

int b200enc_run_ops(const b200enc_op* ops, int n_ops, int* failed_op, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ENC_H_ */
