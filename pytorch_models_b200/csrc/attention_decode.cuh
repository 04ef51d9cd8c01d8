// Single-query attention over a KV cache: one decode step of a causal decoder, or its cross-attention against a
// cached encoder memory (reference: F.scaled_dot_product_attention at transformer.py:52 with Lq = 1).
//
//   out[b, h] = softmax_j(scale · q[b, h] · k[b, j, h]) · v[b, j, h]
//
// Per key the kernel does 4·head_dim FLOPs and reads 4·head_dim bytes, so it is bound by HBM: there is no tensor-core
// work and the design is about keeping enough loads in flight.
//
//   decode_partial_kernel  persistent grid over work items (b·H + h, chunk of kc keys). A CTA of 4 warps walks its
//                          chunk; a group of kLanes lanes owns one key at a time (lane c holds columns [8c, 8c+8) of
//                          q, k and v), each lane has kUnroll keys' 16-byte K and V loads in flight before it reduces.
//                          Scores, the online softmax and the P·V sum are fp32 on the CUDA cores. The CTA merges its
//                          warps and writes (max, sum, o[head_dim]) of the chunk, unnormalised, to the workspace.
//   decode_combine_kernel  one CTA per (b, h): merges the chunk partials in chunk order (fixed order: bit-identical
//                          repeats) and writes bf16 out.
//
// Append mode (len != nullptr): the keys of sequence b are cache rows [0, len_b) plus the new row, which is read from
// the QKV GEMM's output (k_new / v_new) instead of the cache; the one CTA whose chunk holds key `len_b` also copies the
// new row into cache row `len_b`. No CTA reads a row that another CTA of the launch writes. The lengths are read on the
// device, and the grid and the chunk size depend only on (B, H, head_dim, capacity), so a decode step's launch
// arguments do not change from one step to the next (CUDA-graph replay). A sequence whose length is outside
// [0, capacity) gets NaN outputs and touches no cache row; the other sequences of the launch are unaffected.
//   len_stride 0: one length `len[0]` shared by the batch.
//   len_stride 1: per-sequence lengths `len[b]` (a ragged batch). Sequence b has nch_b = ceil(keys_b / kc) chunks;
//     the items are numbered densely in (b, h, chunk) order, H·nch_b per sequence, and every CTA reduces the lengths
//     to the item count H·Σ nch_b. A CTA's items increase, so it finds each item's sequence by advancing a cursor over
//     the sequences (B length reads per CTA in all). Only real items are enumerated, so the grid stride spreads them as
//     evenly over the CTAs as the shared-length launch does, and the K/V bytes read follow the sum of the lengths, not
//     B times the longest. With equal lengths the numbering is the shared-length one: every item does the same
//     arithmetic (bit-identical outputs). The ragged enumeration is its own instantiation (kRagged), so the
//     shared-length one keeps its direct item -> (b, h, chunk) division.
// Cross mode (len == nullptr): keys [0, Lkv) of a read-only cache.
#pragma once
#include "ptx.cuh"

namespace b200 {

constexpr int DEC_WARPS = 4;
constexpr int DEC_THREADS = DEC_WARPS * 32;
constexpr int DEC_UNROLL = 4;          // keys per lane group whose K/V loads are issued before the first is used
constexpr int DEC_MIN_CHUNK = 64;      // keys per work item: a multiple of 64 (one CTA iteration is 32 or 64 keys)
constexpr int DEC_MAX_CHUNK = 4096;
constexpr int DEC_CTAS_PER_SM = 6;

struct DecodeParams {
  const __nv_bfloat16* q;      // [B] rows, head h at columns [hd*h, hd*h + hd)
  long long q_bs;
  const __nv_bfloat16* k_new;  // append mode: the step's k / v rows (batch stride new_bs), else nullptr
  const __nv_bfloat16* v_new;
  long long new_bs;
  __nv_bfloat16* k_cache;      // [B][capacity] rows of row stride ld_cache, batch stride cache_bs
  __nv_bfloat16* v_cache;
  long long cache_bs;
  long long ld_cache;
  int capacity;
  const int* len;              // device length(s) (append mode) or nullptr (cross mode: Lkv keys)
  int len_stride;              // 0: len[0] for every sequence, 1: len[b] for sequence b
  int Lkv;
  __nv_bfloat16* out;          // [B] rows, batch stride out_bs
  long long out_bs;
  int B, H, head_dim;
  float scale_log2e;
  int kc;                      // keys per chunk
  int max_chunks;              // ceil(capacity + 1, kc) in append mode, ceil(Lkv, kc) in cross mode
  float* ws;                   // [B*H][max_chunks][head_dim + 2] fp32
};

// number of keys of sequence b, or -1 if its device length is out of range
__device__ __forceinline__ int decode_keys(const DecodeParams& p, int b) {
  if (p.len == nullptr) return p.Lkv;
  const int n = p.len[b * p.len_stride];
  return (n >= 0 && n < p.capacity) ? n + 1 : -1;
}

__device__ __forceinline__ float dec_scale(float m, float mx) { return m == -INFINITY ? 0.0f : exp2f(m - mx); }

__device__ __forceinline__ void dec_unpack(uint4 w, float (&f)[8]) {
  const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(u[i] << 16);
    f[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
  }
}

// kLanes = lanes per key (8: head_dim 64, 16: head_dim 80-128); lanes c >= head_dim / 8 of a group idle.
// kRagged: per-sequence lengths (len_stride 1), else one length or Lkv for the whole batch.
template <int kLanes, bool kRagged>
__global__ void __launch_bounds__(DEC_THREADS, DEC_CTAS_PER_SM) decode_partial_kernel(const DecodeParams p) {
  constexpr int kGroups = 32 / kLanes;
  __shared__ float sm_ml[DEC_WARPS][2];
  __shared__ float sm_o[DEC_WARPS][128];
  __shared__ int sm_chunks[DEC_WARPS];
  griddep_wait();  // the previous kernel (the QKV GEMM) wrote q and the new k / v row
  int n_keys = decode_keys(p, 0);
  if (!kRagged && n_keys < 0) return;  // the combine kernel writes NaN
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // chunks of a sequence: 0 when its length is out of range (the combine kernel writes its NaN)
  auto chunks = [&](int keys) { return keys < 0 ? 0 : (keys + p.kc - 1) / p.kc; };
  int nch = chunks(n_keys), total = p.B * nch;
  if constexpr (kRagged) {
    total = 0;
    for (int b = threadIdx.x; b < p.B; b += DEC_THREADS) total += chunks(decode_keys(p, b));
    total = __reduce_add_sync(0xffffffffu, total);
    if (lane == 0) sm_chunks[warp] = total;
    __syncthreads();
    total = 0;
#pragma unroll
    for (int w = 0; w < DEC_WARPS; ++w) total += sm_chunks[w];
  }
  const int grp = lane / kLanes, c = lane % kLanes;
  const int hd = p.head_dim;
  const bool col_ok = c < (hd >> 3);
  const int n_items = p.H * total;
  int b = 0, first = 0;                 // ragged: the items of sequence b start at `first`
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    int bh, h, chunk;
    if constexpr (kRagged) {
      while (item >= first + p.H * nch) {  // a later sequence (CTA-uniform; skips sequences without items)
        first += p.H * nch;
        n_keys = decode_keys(p, ++b);
        nch = chunks(n_keys);
      }
      const int local = item - first;
      h = local / nch;
      chunk = local - h * nch;
      bh = b * p.H + h;
    } else {
      bh = item / nch;
      chunk = item - bh * nch;
      b = bh / p.H;
      h = bh - b * p.H;
    }
    const int new_row = p.len != nullptr ? n_keys - 1 : -1;
    const long long col = (long long)h * hd + 8 * c;
    float qf[8];
    {
      uint4 qw = make_uint4(0, 0, 0, 0);
      if (col_ok) qw = __ldg(reinterpret_cast<const uint4*>(p.q + b * p.q_bs + col));
      dec_unpack(qw, qf);
#pragma unroll
      for (int i = 0; i < 8; ++i) qf[i] *= p.scale_log2e;
    }
    const __nv_bfloat16* kc_base = p.k_cache + b * p.cache_bs + col;
    const __nv_bfloat16* vc_base = p.v_cache + b * p.cache_bs + col;
    const int j0 = chunk * p.kc, j1 = min(j0 + p.kc, n_keys);
    float m = -INFINITY, l = 0.0f, o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = 0.0f;
    constexpr int kStep = DEC_WARPS * kGroups * DEC_UNROLL;
    for (int jb = j0 + warp * kGroups * DEC_UNROLL; jb < j1; jb += kStep) {
      uint4 kw[DEC_UNROLL], vw[DEC_UNROLL];
#pragma unroll
      for (int u = 0; u < DEC_UNROLL; ++u) {
        const int j = jb + u * kGroups + grp;
        kw[u] = vw[u] = make_uint4(0, 0, 0, 0);
        if (col_ok && j < j1) {
          const __nv_bfloat16 *kr, *vr;
          if (j == new_row) {
            kr = p.k_new + b * p.new_bs + col;
            vr = p.v_new + b * p.new_bs + col;
          } else {
            kr = kc_base + j * p.ld_cache;
            vr = vc_base + j * p.ld_cache;
          }
          kw[u] = __ldg(reinterpret_cast<const uint4*>(kr));
          vw[u] = __ldg(reinterpret_cast<const uint4*>(vr));
        }
      }
      float s[DEC_UNROLL];
      float mx = m;
#pragma unroll
      for (int u = 0; u < DEC_UNROLL; ++u) {
        float kf[8];
        dec_unpack(kw[u], kf);
        float d = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) d = fmaf(qf[i], kf[i], d);
#pragma unroll
        for (int off = kLanes / 2; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
        s[u] = (jb + u * kGroups + grp < j1) ? d : -INFINITY;
        mx = fmaxf(mx, s[u]);
      }
      if (mx == -INFINITY) continue;  // no key of this group in range (group-uniform)
      const float alpha = dec_scale(m, mx);
      l *= alpha;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] *= alpha;
#pragma unroll
      for (int u = 0; u < DEC_UNROLL; ++u) {
        const float pu = exp2f(s[u] - mx);  // 0 for keys out of range
        float vf[8];
        dec_unpack(vw[u], vf);
        l += pu;
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = fmaf(pu, vf[i], o[i]);
      }
      m = mx;
    }
    // merge the lane groups of the warp (lanes c, c + kLanes, ... hold the same columns)
#pragma unroll
    for (int off = kLanes; off < 32; off <<= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, off);
      const float l2 = __shfl_xor_sync(0xffffffffu, l, off);
      const float mx = fmaxf(m, m2);
      const float a = dec_scale(m, mx), a2 = dec_scale(m2, mx);
      l = l * a + l2 * a2;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = o[i] * a + __shfl_xor_sync(0xffffffffu, o[i], off) * a2;
      m = mx;
    }
    if (lane == 0) sm_ml[warp][0] = m, sm_ml[warp][1] = l;
    if (lane < kLanes && col_ok) {
#pragma unroll
      for (int i = 0; i < 8; ++i) sm_o[warp][8 * c + i] = o[i];
    }
    // the chunk that holds the new key copies it into the cache (nobody in this launch reads that cache row)
    if (new_row >= j0 && new_row < j1 && warp == 0 && lane < kLanes && col_ok) {
      const long long src = b * p.new_bs + col, dst = b * p.cache_bs + col + new_row * p.ld_cache;
      *reinterpret_cast<uint4*>(p.k_cache + dst) = __ldg(reinterpret_cast<const uint4*>(p.k_new + src));
      *reinterpret_cast<uint4*>(p.v_cache + dst) = __ldg(reinterpret_cast<const uint4*>(p.v_new + src));
    }
    __syncthreads();
    float* rec = p.ws + ((long long)bh * p.max_chunks + chunk) * (hd + 2);
    float mx = sm_ml[0][0];
#pragma unroll
    for (int w = 1; w < DEC_WARPS; ++w) mx = fmaxf(mx, sm_ml[w][0]);
    for (int t = threadIdx.x; t < hd + 2; t += DEC_THREADS) {
      float acc = 0.0f;
#pragma unroll
      for (int w = 0; w < DEC_WARPS; ++w) {
        const float a = dec_scale(sm_ml[w][0], mx);
        acc += a * (t == 0 ? 0.0f : (t == 1 ? sm_ml[w][1] : sm_o[w][t - 2]));
      }
      rec[t] = t == 0 ? mx : acc;
    }
    __syncthreads();
  }
  griddep_launch_dependents();
}

// One CTA per (b, h); thread t < head_dim owns output column t.
__global__ void __launch_bounds__(128) decode_combine_kernel(const DecodeParams p) {
  griddep_wait();
  const int bh = blockIdx.x, t = threadIdx.x, hd = p.head_dim;
  if (t >= hd) return;
  const int b = bh / p.H, h = bh - b * p.H;
  __nv_bfloat16* dst = p.out + b * p.out_bs + (long long)h * hd + t;
  const int n_keys = decode_keys(p, b);
  if (n_keys < 0) {
    *dst = __float2bfloat16_rn(__int_as_float(0x7fc00000));
    return;
  }
  const int nch = (n_keys + p.kc - 1) / p.kc;
  const float* rec = p.ws + (long long)bh * p.max_chunks * (hd + 2);
  float mx = -INFINITY;
  for (int c = 0; c < nch; ++c) mx = fmaxf(mx, rec[c * (hd + 2)]);
  float l = 0.0f, o = 0.0f;
  for (int c = 0; c < nch; ++c) {
    const float* r = rec + c * (hd + 2);
    const float a = dec_scale(r[0], mx);
    l += a * r[1];
    o += a * r[2 + t];
  }
  *dst = __float2bfloat16_rn(o / l);
}

// out[r] = bf16(tok[ids[r]] + pos[pos0[(r / L) * pos0_stride] + r % L]): the embedding of a decode step, whose
// position is the cache length on the device (pos0_stride 0: one length for all rows, 1: one per sequence of L rows).
// An id outside [0, vocab) or a position outside [0, n_pos) gives a NaN row.
template <typename TIn>
__global__ void __launch_bounds__(256)
embed_rows_at_kernel(const long long* __restrict__ ids, long long rows, int L, const TIn* __restrict__ tok,
                     const TIn* __restrict__ pos, int n_pos, const int* __restrict__ pos0, int pos0_stride, int vocab,
                     int d, __nv_bfloat16* __restrict__ out) {
  const int vec_per_row = d >> 3;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * vec_per_row) return;
  const long long r = t / vec_per_row;
  const int c = int(t % vec_per_row) * 8;
  const long long id = ids[r];
  const long long pr = (long long)pos0[(r / L) * pos0_stride] + r % L;
  const bool ok = id >= 0 && id < vocab && pr >= 0 && pr < n_pos;
  const TIn* trow = tok + (ok ? id : 0) * (long long)d + c;
  const TIn* prow = pos + (ok ? pr : 0) * (long long)d + c;
  uint32_t packed[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = ok ? float(trow[2 * i]) + float(prow[2 * i]) : __int_as_float(0x7fc00000);
    const float b = ok ? float(trow[2 * i + 1]) + float(prow[2 * i + 1]) : __int_as_float(0x7fc00000);
    packed[i] = pack_bf16x2(a, b);
  }
  *reinterpret_cast<uint4*>(out + r * d + c) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
}

// cache[b][len_b + r][:width] = src[b][r][:width] for r < P (len_b = len[b * len_stride]): the k|v rows of an extend,
// written before its attention reads every key from the cache. One thread per 16-byte vector. A row that would land
// outside [0, capacity) is not written.
__global__ void kv_append_kernel(const __nv_bfloat16* __restrict__ src, long long src_bs, int ld_src,
                                 __nv_bfloat16* __restrict__ cache, long long cache_bs, int ld_cache, int capacity,
                                 const int* __restrict__ len, int len_stride, int B, int P, int width) {
  griddep_wait();  // the previous kernel (the QKV GEMM) wrote the rows
  const int vec_per_row = width >> 3;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * P * vec_per_row) return;
  const long long row = t / vec_per_row;
  const int c = int(t % vec_per_row) * 8;
  const int b = int(row / P), r = int(row % P);
  const int n = len[b * len_stride];
  if (n < 0 || n >= capacity - r) return;
  const uint4 v = *reinterpret_cast<const uint4*>(src + b * src_bs + (long long)r * ld_src + c);
  *reinterpret_cast<uint4*>(cache + b * cache_bs + (long long)(n + r) * ld_cache + c) = v;
}

// len[i] += delta for i < n: the last launch of a decode step (n = 1 shared length, or one per sequence)
__global__ void decode_advance_kernel(int* len, int n, int delta) {
  griddep_wait();
  for (int i = threadIdx.x; i < n; i += blockDim.x) len[i] += delta;
}

}  // namespace b200
