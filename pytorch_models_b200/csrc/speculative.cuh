// The device half of a greedy speculative-decoding round (see DESIGN §3.2.5): the argmax of logits rows, and the
// acceptance of draft tokens against the target's picks, which also rolls both KV caches back past the rejected rows.
// Neither needs the host, so a whole round (draft steps, verify extend, picks, accept) replays as one CUDA graph.
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

}  // namespace b200
