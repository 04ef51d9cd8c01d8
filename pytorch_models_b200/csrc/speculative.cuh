// The device half of a greedy speculative-decoding round (see DESIGN §3.2.5): the argmax of logits rows, the
// acceptance of draft tokens against the target's picks, which also rolls both KV caches back past the rejected rows,
// and the draft-free proposal of §3.2.6 by n-gram lookup in each sequence's own token history. None needs the host, so
// a whole round (drafts, verify extend, picks, accept) replays as one CUDA graph.
#pragma once

#include <cuda_bf16.h>
#include <stdint.h>

#include "ptx.cuh"

namespace b200 {

constexpr int ARGMAX_THREADS = 512;
constexpr int ARGMAX_UNROLL = 4;  // 16-byte loads in flight per thread before it compares

// (value, index) order of torch.argmax: NaN is greater than any number (so the first NaN wins), and of two equal
// values the lower index wins.
__device__ __forceinline__ bool argmax_better(float a, int ia, float b, int ib) {
  const bool na = a != a, nb = b != b;
  if (na || nb) return na && (!nb || ia < ib);
  return a > b || (a == b && ia < ib);
}

// out[r * out_stride] = argmax_j logits[r * ld + j] over j < V. One CTA per row; thread t reads the 16-byte vectors
// t, t + 512, ... of the row, so its own indices increase and a strict comparison keeps the first of equal values.
// Columns in [V, ld) (the GEMM's padding to a multiple of 8) are never candidates.
__global__ void __launch_bounds__(ARGMAX_THREADS)
argmax_rows_kernel(const __nv_bfloat16* __restrict__ logits, long long ld, int V, long long* __restrict__ out,
                   long long out_stride) {
  griddep_wait();  // the logits GEMM wrote the row
  const __nv_bfloat16* row = logits + blockIdx.x * ld;
  const int nvec = (V + 7) >> 3;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int v0 = threadIdx.x; v0 < nvec; v0 += ARGMAX_THREADS * ARGMAX_UNROLL) {
    uint4 raw[ARGMAX_UNROLL];
#pragma unroll
    for (int u = 0; u < ARGMAX_UNROLL; ++u) {
      const int v = v0 + u * ARGMAX_THREADS;
      raw[u] = v < nvec ? __ldg(reinterpret_cast<const uint4*>(row) + v) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < ARGMAX_UNROLL; ++u) {
      const int c0 = (v0 + u * ARGMAX_THREADS) * 8;
      const __nv_bfloat16* h = reinterpret_cast<const __nv_bfloat16*>(&raw[u]);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = __bfloat162float(h[e]);
        const int c = c0 + e;
        // within a thread the indices increase: a NaN replaces a number, a larger number replaces a smaller one
        if (c < V && (x > best || (x != x && best == best) || bi == 0x7fffffff)) {
          best = x;
          bi = c;
        }
      }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
    if (argmax_better(ob, oi, best, bi)) {
      best = ob;
      bi = oi;
    }
  }
  __shared__ float sb[ARGMAX_THREADS / 32];
  __shared__ int si[ARGMAX_THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sb[warp] = best;
    si[warp] = bi;
  }
  __syncthreads();
  if (warp == 0) {
    best = lane < ARGMAX_THREADS / 32 ? sb[lane] : -INFINITY;
    bi = lane < ARGMAX_THREADS / 32 ? si[lane] : 0x7fffffff;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (argmax_better(ob, oi, best, bi)) {
        best = ob;
        bi = oi;
      }
    }
    if (lane == 0) out[blockIdx.x * out_stride] = bi;
  }
}

// Step 4 of a round, one thread per sequence b, with k draft tokens:
//   ids[b]    = [last, d_1 .. d_k], the verify extend's input; picks[b] = [t_0 .. t_k], the target's argmax per row.
//   a         = the number of leading i < k with t_i == d_{i+1}; the candidates are d_1 .. d_a, t_a.
//   m         = the candidates up to and including the first EOS, at most budget[b] of them (0 once budget[b] <= 0).
//   emitted[b][0, m) = the kept candidates, emitted[b][m, k] = -1, n_emitted[b] = m.
//   budget[b] -= m, or 0 after an EOS.
//   both caches' lengths -= k + 1 - m: the rows kept are `last` and the accepted drafts, so the newest token is in
//   neither cache, as before the round.
//   ids[b][0] = emitted[b][m - 1] when m > 0: the next round's `last`.
// len_t / len_d use the len_stride convention of DecodeParams (0: one length, only with B = 1; 1: len[b]).
__global__ void speculative_accept_kernel(const long long* __restrict__ picks, long long* __restrict__ ids,
                                          int* __restrict__ budget, long long eos, int* __restrict__ len_t,
                                          int stride_t, int* __restrict__ len_d, int stride_d,
                                          long long* __restrict__ emitted, long long* __restrict__ n_emitted,
                                          long long out_stride, int B, int k) {
  griddep_wait();  // the argmax of the verify rows wrote the picks
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const long long* t = picks + (long long)b * (k + 1);
  long long* row = ids + (long long)b * (k + 1);
  long long* em = emitted + b * out_stride;
  int a = 0;
  while (a < k && t[a] == row[a + 1]) ++a;
  const int left = budget[b];
  int m = 0;
  bool stop = false;
  for (int i = 0; i <= a && m < left && !stop; ++i) {
    const long long tok = i < a ? row[i + 1] : t[a];
    em[m++] = tok;
    stop = tok == eos;
  }
  for (int i = m; i <= k; ++i) em[i] = -1;
  n_emitted[b * out_stride] = m;
  budget[b] = stop ? 0 : (left > m ? left - m : 0);
  len_t[b * stride_t] -= k + 1 - m;
  len_d[b * stride_d] -= k + 1 - m;
  if (m > 0) row[0] = em[m - 1];
}

constexpr int NGRAM_THREADS = 256;
constexpr int NGRAM_MAX = 8;  // the longest n-gram matched

// Step 1 of a draft-free round (DESIGN §3.2.6), one CTA per sequence b with n = len[b * len_stride] tokens in its
// history row h = hist + b * ld and ids[b] = [last, ..]. With s = h[0, n) followed by last (T = n + 1 tokens):
//   L(e)  = the number of leading j < max_ngram with j <= e and s[e - j] == s[n - j], for each end e < n;
//   g*    = the largest min(L(e), max_ngram) over e, e* the largest e reaching it; no match when g* < min_ngram.
//   This is "the longest g in [min_ngram, max_ngram] whose suffix occurs earlier, at its latest occurrence".
//   d_i   = s'[e* + i] for i = 1..k, s' being s followed by the drafts (an overlapping copy keeps a period), or last
//           for every i without a match.
// Writes ids[b][1..k] = d, h[n] = last, h[n + 1 .. n + k] = d and len += k + 1, so that the history holds the rows
// the verify appends to the target cache and speculative_accept rolls both back alike. A length outside
// [0, capacity - k - 1] drafts last, writes no history row and still advances. Only rows below n are read.
__global__ void __launch_bounds__(NGRAM_THREADS)
ngram_draft_kernel(long long* __restrict__ hist, long long ld, int capacity, int* __restrict__ len, int len_stride,
                   long long* __restrict__ ids, int k, int max_ngram, int min_ngram) {
  griddep_wait();  // the previous round's accept wrote len and ids[b][0]
  const int b = blockIdx.x;
  long long* h = hist + b * ld;
  long long* row = ids + (long long)b * (k + 1);
  const int n = len[b * len_stride];
  const long long last = row[0];
  const bool ok = n >= 0 && n <= capacity - k - 1;
  __shared__ long long suf[NGRAM_MAX];  // suf[j] = s[n - j]
  __shared__ long long red[NGRAM_THREADS / 32];
  if (ok && threadIdx.x < max_ngram && threadIdx.x <= n)
    suf[threadIdx.x] = threadIdx.x == 0 ? last : h[n - threadIdx.x];
  __syncthreads();
  // key = (min(L(e), max_ngram) << 32) | e for the matches of at least min_ngram tokens, else -1; the largest wins
  long long key = -1;
  if (ok) {
    for (int e = threadIdx.x; e < n; e += NGRAM_THREADS) {
      int l = 0;
      while (l < max_ngram && l <= e && h[e - l] == suf[l]) ++l;
      if (l >= min_ngram) key = max(key, ((long long)l << 32) | e);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, off));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = key;
  __syncthreads();  // also: every thread has read len[b] before thread 0 advances it
  if (threadIdx.x != 0) return;
  for (int w = 1; w < NGRAM_THREADS / 32; ++w) key = max(key, red[w]);
  const int e = key < 0 ? -1 : int(key & 0xffffffffLL);
  // s'[p] = s'[p - q] for p > n with q = n - e, so d_i = s[e + 1 + (i - 1) % q], a row below n or last
  const int q = e < 0 ? 1 : n - e;
  for (int i = 1; i <= k; ++i) {
    const int p = e + 1 + (i - 1) % q;
    const long long d = e < 0 || p == n ? last : h[p];
    row[i] = d;
    if (ok) h[n + i] = d;
  }
  if (ok) h[n] = last;
  len[b * len_stride] = n + k + 1;
}

}  // namespace b200
