// Stand-alone GPU self-test / micro-benchmark for libb200enc (no PyTorch): each case checks a kernel against a
// straightforward fp64 CPU computation on the same inputs. Test infrastructure only; run on the B200 box:
//   ./b200enc_selftest <case> [args]      (exit code 0 = pass)
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/b200enc.h"

#define CK(x)                                                                         \
  do {                                                                                \
    cudaError_t e = (x);                                                              \
    if (e != cudaSuccess) {                                                           \
      printf("CUDA error %s at %s:%d: %s\n", #x, __FILE__, __LINE__, cudaGetErrorString(e)); \
      exit(3);                                                                        \
    }                                                                                 \
  } while (0)

static uint64_t g_seed = 0x9E3779B97F4A7C15ull;
static inline uint32_t rnd() {
  g_seed = g_seed * 6364136223846793005ull + 1442695040888963407ull;
  return uint32_t(g_seed >> 33);
}
static inline float urand() { return (rnd() & 0xFFFFFF) / float(0x1000000) * 2.0f - 1.0f; }  // [-1, 1)

static inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return uint16_t(u >> 16);
}
static inline float bf2f(uint16_t h) {
  uint32_t u = uint32_t(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  explicit DevBuf(size_t b) : bytes(b) { CK(cudaMalloc(&p, b ? b : 16)); }
  ~DevBuf() { cudaFree(p); }
};

// Device buffer with 4 KB guard bands on both sides (compute-sanitizer is closed on this pool: out-of-bounds writes
// of the st.global paths are caught by checking that the bands still hold their fill pattern).
struct GuardedBuf {
  static constexpr size_t kGuard = 4096;
  DevBuf raw;
  size_t bytes;
  explicit GuardedBuf(size_t b) : raw(b + 2 * kGuard), bytes(b) { CK(cudaMemset(raw.p, 0x5a, raw.bytes)); }
  void* p() const { return static_cast<char*>(raw.p) + kGuard; }
  bool intact(const char* what) const {
    std::vector<unsigned char> h(raw.bytes);
    CK(cudaMemcpy(h.data(), raw.p, raw.bytes, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < kGuard; ++i)
      if (h[i] != 0x5a || h[kGuard + bytes + i] != 0x5a) {
        printf("  [FAIL] %s: guard band overwritten at %s%zu\n", what, h[i] != 0x5a ? "-" : "+", i);
        return false;
      }
    return true;
  }
};

static std::vector<uint16_t> rand_bf16(size_t n, float scale, bool ints) {
  std::vector<uint16_t> v(n);
  for (size_t i = 0; i < n; ++i) v[i] = f2bf(ints ? float(int(rnd() % 5) - 2) : urand() * scale);
  return v;
}
static std::vector<float> rand_f32(size_t n, float scale) {
  std::vector<float> v(n);
  for (size_t i = 0; i < n; ++i) v[i] = urand() * scale;
  return v;
}

static double gelu_ref(double x) { return 0.5 * x * (1.0 + erf(x / sqrt(2.0))); }
static double gelu_tanh_ref(double x) { return 0.5 * x * (1.0 + tanh(0.7978845608028654 * (x + 0.044715 * x * x * x))); }

struct CmpStat {
  double max_abs = 0, max_rel = 0;
  long long bad = 0, n = 0;
  int shown = 0;
  long long bad_rowmod8[8] = {0}, bad_colblk[8] = {0};
};
static void cmp_one(CmpStat& st, double want, float got, double atol, double rtol, int r, int c, const char* tag) {
  double d = fabs(double(got) - want);
  st.n++;
  if (!(d <= st.max_abs)) st.max_abs = (d != d) ? INFINITY : (d > st.max_abs ? d : st.max_abs);
  double rel = d / (fabs(want) + 1e-6);
  if (rel > st.max_rel && fabs(want) > 1e-2) st.max_rel = rel;
  if (!(d <= atol + rtol * fabs(want))) {
    st.bad++;
    st.bad_rowmod8[r & 7]++;
    st.bad_colblk[(c >> 3) & 7]++;
    if (st.shown < 12) {
      printf("    MISMATCH %s row=%d col=%d got=%.6g want=%.6g\n", tag, r, c, got, want);
      st.shown++;
    }
  }
}
static bool report(const char* name, const CmpStat& st) {
  printf("  [%s] %s: checked=%lld bad=%lld max_abs=%.4g max_rel=%.4g\n", st.bad ? "FAIL" : "ok", name, st.n, st.bad,
         st.max_abs, st.max_rel);
  if (st.bad) {
    printf("    bad by row%%8:");
    for (int i = 0; i < 8; ++i) printf(" %lld", st.bad_rowmod8[i]);
    printf("   by (col/8)%%8:");
    for (int i = 0; i < 8; ++i) printf(" %lld", st.bad_colblk[i]);
    printf("\n");
  }
  fflush(stdout);
  return st.bad == 0;
}

// ------------------------------------------------------------------------------------------ linear
struct LinearCase {
  const char* name;
  int batches, M, N, K;
  bool fold;
  int gelu;  // activation: 0 none, 1 erf-GELU, 2 tanh-GELU, 3 ReLU, 4 SiLU
  bool res, res_bcast, ints;
  int out_row_off;  // output rows shifted by this inside a (M + off)-row batch (patch-embed layout)
  int check_rows;   // rows per batch checked on the CPU (0 = all)
  int time_iters;
};

static bool run_linear(const LinearCase& c) {
  printf("linear %s: batches=%d M=%d N=%d K=%d fold=%d gelu=%d res=%d bcast=%d\n", c.name, c.batches, c.M, c.N, c.K,
         c.fold, c.gelu, c.res, c.res_bcast);
  fflush(stdout);
  const int B = c.batches, M = c.M, N = c.N, K = c.K;
  const int Mo = M + c.out_row_off;
  const float xs = c.ints ? 1.f : 1.0f, ws = c.ints ? 1.f : 0.05f;
  auto hx = rand_bf16(size_t(B) * M * K, xs, c.ints);
  auto hw = rand_bf16(size_t(N) * K, ws, c.ints);
  auto hb = rand_f32(N, c.ints ? 0.f : 0.5f);
  std::vector<float> hs(N, 0.f), hstats(size_t(B) * M * 2, 0.f);
  if (c.fold) {
    for (int n = 0; n < N; ++n) {
      double s = 0;
      for (int k = 0; k < K; ++k) s += bf2f(hw[size_t(n) * K + k]);
      hs[n] = float(s);
    }
    for (size_t i = 0; i < size_t(B) * M; ++i) {
      hstats[2 * i] = urand() * 0.3f;
      hstats[2 * i + 1] = 0.5f + fabsf(urand());
    }
  }
  const size_t res_rows = c.res_bcast ? size_t(M) : size_t(B) * M;
  auto hr = rand_bf16(c.res ? res_rows * N : 1, 1.0f, c.ints);

  DevBuf dx(hx.size() * 2), dw(hw.size() * 2), db(N * 4), ds(N * 4), dst(hstats.size() * 4), dr(hr.size() * 2),
      dout(size_t(B) * Mo * N * 2);
  CK(cudaMemcpy(dx.p, hx.data(), hx.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw.p, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(db.p, hb.data(), N * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ds.p, hs.data(), N * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dst.p, hstats.data(), hstats.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dr.p, hr.data(), hr.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemset(dout.p, 0x7f, dout.bytes));  // sentinel 0x7f7f = 3.39e38 in bf16

  const int flags = c.gelu == 1 ? B200ENC_LINEAR_GELU : c.gelu == 2 ? B200ENC_LINEAR_GELU_TANH : c.gelu == 3 ? B200ENC_LINEAR_RELU : c.gelu == 4 ? B200ENC_LINEAR_SILU : 0;
  const int n_slices = (N + 127) / 128;
  const bool want_stats = c.res && !c.fold;
  GuardedBuf gso(size_t(B) * M * n_slices * 8);
  struct { void* p; } dso = {gso.p()};
  auto call = [&]() {
    b200enc_linear_args a;
    memset(&a, 0, sizeof(a));
    a.x = dx.p; a.x_batch_stride = (long long)M * K; a.ldx = K;
    a.w = dw.p; a.ldw = K;
    a.bias = (const float*)db.p;
    a.colsum = c.fold ? (const float*)ds.p : nullptr;
    a.rowstats = c.fold ? (const float*)dst.p : nullptr;
    a.rowstats_parts = 0; a.ln_eps = 0.f;
    a.residual = c.res ? dr.p : nullptr; a.res_batch_stride = c.res_bcast ? 0 : (long long)M * N; a.ldr = N;
    a.out = (uint16_t*)dout.p + size_t(c.out_row_off) * N; a.out_batch_stride = (long long)Mo * N; a.ldo = N;
    a.stats_out = want_stats ? (float*)dso.p : nullptr;
    a.batches = B; a.M = M; a.N = N; a.K = K; a.flags = flags;
    return b200enc_linear(&a, nullptr);
  };
  int rc = call();
  if (rc) {
    printf("  [FAIL] b200enc_linear rc=%d: %s\n", rc, b200enc_last_error());
    return false;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("  [FAIL] kernel error: %s\n", cudaGetErrorString(e));
    return false;
  }
  std::vector<uint16_t> ho(size_t(B) * Mo * N);
  CK(cudaMemcpy(ho.data(), dout.p, ho.size() * 2, cudaMemcpyDeviceToHost));

  CmpStat st;
  const int step = (c.check_rows > 0 && c.check_rows < M) ? M / c.check_rows : 1;
  for (int b = 0; b < B; ++b) {
    for (int m = 0; m < M; m += 1) {
      // always check the first and last 130 rows (tile edges), sample the middle
      if (!(m < 130 || m >= M - 130 || (m % step) == 0)) continue;
      const uint16_t* xr = &hx[(size_t(b) * M + m) * K];
      for (int n = 0; n < N; ++n) {
        const uint16_t* wr = &hw[size_t(n) * K];
        double acc = 0;
        for (int k = 0; k < K; ++k) acc += double(bf2f(xr[k])) * double(bf2f(wr[k]));
        double v;
        if (c.fold) {
          const double mean = hstats[2 * (size_t(b) * M + m)], rstd = hstats[2 * (size_t(b) * M + m) + 1];
          v = rstd * (acc - mean * hs[n]) + hb[n];
        } else {
          v = acc + hb[n];
        }
        if (c.gelu == 1) v = gelu_ref(v);
        if (c.gelu == 2) v = gelu_tanh_ref(v);
        if (c.gelu == 3) v = v > 0 ? v : 0;
        if (c.gelu == 4) v = v / (1.0 + exp(-v));
        if (c.res) v += bf2f(hr[(c.res_bcast ? size_t(m) : size_t(b) * M + m) * N + n]);
        const float got = bf2f(ho[(size_t(b) * Mo + c.out_row_off + m) * N + n]);
        cmp_one(st, v, got, c.ints ? 1e-6 : 0.02, c.ints ? 0.0 : 0.01, b * M + m, n, c.name);
      }
    }
    // rows before out_row_off must keep the sentinel
    for (int m = 0; m < c.out_row_off; ++m)
      for (int n = 0; n < N; ++n)
        if (ho[(size_t(b) * Mo + m) * N + n] != 0x7f7f) {
          st.bad++;
          if (st.shown++ < 12) printf("    CLOBBERED guard row b=%d m=%d n=%d\n", b, m, n);
        }
  }
  bool ok = report(c.name, st);
  if (want_stats) {
    // fused partial LayerNorm statistics: (mean, M2) of every 128-column slice of the stored (bf16) output rows
    std::vector<float> hso(size_t(B) * M * n_slices * 2);
    CK(cudaMemcpy(hso.data(), dso.p, hso.size() * 4, cudaMemcpyDeviceToHost));
    CmpStat ss;
    for (int b = 0; b < B; ++b)
      for (int m = 0; m < M; m += (M > 400 ? 7 : 1))
        for (int t = 0; t < n_slices; ++t) {
          const int w = std::min(128, N - t * 128);
          double mu = 0, m2 = 0;
          for (int k = 0; k < w; ++k) mu += bf2f(ho[(size_t(b) * Mo + c.out_row_off + m) * N + t * 128 + k]);
          mu /= w;
          for (int k = 0; k < w; ++k) {
            const double dlt = bf2f(ho[(size_t(b) * Mo + c.out_row_off + m) * N + t * 128 + k]) - mu;
            m2 += dlt * dlt;
          }
          const float* g = &hso[((size_t(b) * M + m) * n_slices + t) * 2];
          cmp_one(ss, mu, g[0], 1e-4, 1e-4, b * M + m, t, "slice_mean");
          cmp_one(ss, m2, g[1], 1e-2, 1e-3, b * M + m, t, "slice_m2");
        }
    ok = report("fused_stats", ss) && ok;
  }
  ok = gso.intact("stats_out") && ok;

  if (ok && c.time_iters > 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int iters = getenv("B200_ITERS") ? atoi(getenv("B200_ITERS")) : c.time_iters;
    for (int i = 0; i < 3; ++i) call();
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) call();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= iters;
    const double fl = 2.0 * B * double(M) * N * K;
    printf("  time %s: %.3f ms  %.1f TFLOP/s\n", c.name, ms, fl / ms * 1e-9);
    fflush(stdout);
  }
  return ok;
}

static const LinearCase kLinearCases[] = {
    //  name            B   M      N     K    fold   gelu   res    bcast  ints  off rows iters
    {"min_tma", 1, 128, 256, 64, false, false, false, false, true, 0, 0, 0},
    {"k256_tma", 1, 128, 256, 256, false, false, false, false, true, 0, 0, 0},
    {"multi_tile", 1, 512, 768, 768, false, false, false, false, false, 0, 0, 0},
    {"tails_tma", 1, 300, 576, 192, false, false, false, false, false, 0, 0, 0},
    {"many_tiles", 1, 19000, 768, 768, false, false, false, false, false, 0, 40, 0},
    {"embed_like", 3, 196, 768, 768, false, false, true, true, false, 1, 0, 0},
    {"fold_gelu", 1, 1000, 3072, 768, true, true, false, false, false, 0, 60, 0},
    {"fold_gelu_tanh", 1, 1000, 3072, 768, true, 2, false, false, false, 0, 60, 0},
    {"gelu_tanh", 2, 300, 512, 256, false, 2, false, false, false, 0, 60, 0},
    {"relu", 2, 300, 512, 256, false, 3, false, false, false, 0, 60, 0},
    {"fold_silu", 1, 1000, 1024, 512, true, 4, false, false, false, 0, 60, 0},
    {"residual", 1, 1000, 768, 3072, false, false, true, false, false, 0, 60, 0},
    {"fold_qkv", 1, 1000, 2304, 768, true, false, false, false, false, 0, 60, 0},
    {"perf_qkv", 1, 25216, 2304, 768, true, false, false, false, false, 0, 16, 20},
    {"perf_out", 1, 25216, 768, 768, false, false, true, false, false, 0, 16, 20},
    {"perf_fc1", 1, 25216, 3072, 768, true, true, false, false, false, 0, 16, 20},
    {"perf_fc2", 1, 25216, 768, 3072, false, false, true, false, false, 0, 16, 20},
    {"perf_qkv_l2fit", 1, 8192, 2304, 768, true, false, false, false, false, 0, 16, 60},
    {"perf_qkv_big", 1, 201728, 2304, 768, true, false, false, false, false, 0, 8, 10},
    {"perf_out_big", 1, 201728, 768, 768, false, false, true, false, false, 0, 8, 10},
    {"perf_fc2_big", 1, 201728, 768, 3072, false, false, true, false, false, 0, 8, 10},
    {"perf_fc1_big", 1, 201728, 3072, 768, true, true, false, false, false, 0, 8, 10},
    {"perf_k4096", 1, 25216, 2304, 4096, false, false, false, false, false, 0, 8, 10},
};


// ------------------------------------------------------------------------------------------ attention
struct AttnCase {
  const char* name;
  int B, H, Lq, Lkv;
  bool self_qkv;  // q/k/v are slices of one fused [B, L, 3*H*64] buffer
  bool causal;
  float mag;
  int check_bh;  // number of (b,h) pairs checked (0 = all)
  int time_iters;
};

static bool run_attn(const AttnCase& c) {
  printf("attention %s: B=%d H=%d Lq=%d Lkv=%d self=%d causal=%d\n", c.name, c.B, c.H, c.Lq, c.Lkv, c.self_qkv,
         c.causal);
  fflush(stdout);
  const int B = c.B, H = c.H, Lq = c.Lq, Lkv = c.Lkv, D = H * 64;
  std::vector<uint16_t> hq, hkv;
  int ldq, ldkv;
  size_t koff, voff;
  if (c.self_qkv) {
    hq = rand_bf16(size_t(B) * Lq * 3 * D, c.mag, false);
    ldq = ldkv = 3 * D;
    koff = D;
    voff = 2 * D;
  } else {
    hq = rand_bf16(size_t(B) * Lq * D, c.mag, false);
    hkv = rand_bf16(size_t(B) * Lkv * 2 * D, c.mag, false);
    ldq = D;
    ldkv = 2 * D;
    koff = 0;
    voff = D;
  }
  DevBuf dq(hq.size() * 2), dkv(hkv.size() * 2 + 16);
  GuardedBuf gout(size_t(B) * Lq * D * 2);
  struct { void* p; size_t bytes; } dout = {gout.p(), gout.bytes};
  CK(cudaMemcpy(dq.p, hq.data(), hq.size() * 2, cudaMemcpyHostToDevice));
  if (!c.self_qkv) CK(cudaMemcpy(dkv.p, hkv.data(), hkv.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemset(dout.p, 0x7f, dout.bytes));
  const uint16_t* kvbase_h = c.self_qkv ? hq.data() : hkv.data();
  uint16_t* kvbase_d = (uint16_t*)(c.self_qkv ? dq.p : dkv.p);
  const float scale = 0.125f;
  auto call = [&]() {
    return b200enc_attention(dq.p, (long long)Lq * ldq, ldq, kvbase_d + koff, kvbase_d + voff, (long long)Lkv * ldkv,
                             ldkv, dout.p, (long long)Lq * D, D, B, H, Lq, Lkv, 64, scale,
                             c.causal ? B200ENC_ATTN_CAUSAL : 0, nullptr);
  };
  int rc = call();
  if (rc) {
    printf("  [FAIL] b200enc_attention rc=%d: %s\n", rc, b200enc_last_error());
    return false;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("  [FAIL] kernel error: %s\n", cudaGetErrorString(e));
    return false;
  }
  std::vector<uint16_t> ho(size_t(B) * Lq * D);
  CK(cudaMemcpy(ho.data(), dout.p, ho.size() * 2, cudaMemcpyDeviceToHost));
  CmpStat st;
  const int nbh = B * H;
  const int stepbh = (c.check_bh > 0 && c.check_bh < nbh) ? nbh / c.check_bh : 1;
  std::vector<double> sc(Lkv);
  for (int bh = 0; bh < nbh; bh += stepbh) {
    const int b = bh / H, h = bh % H;
    for (int i = 0; i < Lq; ++i) {
      const uint16_t* qr = &hq[(size_t(b) * Lq + i) * ldq + h * 64];
      double mx = -1e300;
      const int jmax = c.causal ? std::min(Lkv, i + 1) : Lkv;
      for (int j = 0; j < jmax; ++j) {
        const uint16_t* kr = kvbase_h + (size_t(b) * Lkv + j) * ldkv + koff + h * 64;
        double a = 0;
        for (int t = 0; t < 64; ++t) a += double(bf2f(qr[t])) * double(bf2f(kr[t]));
        sc[j] = a * scale;
        mx = sc[j] > mx ? sc[j] : mx;
      }
      double den = 0;
      for (int j = 0; j < Lkv; ++j) {
        sc[j] = j < jmax ? exp(sc[j] - mx) : 0.0;
        den += sc[j];
      }
      for (int t = 0; t < 64; ++t) {
        double o = 0;
        for (int j = 0; j < Lkv; ++j)
          o += sc[j] * double(bf2f(kvbase_h[(size_t(b) * Lkv + j) * ldkv + voff + h * 64 + t]));
        o /= den;
        cmp_one(st, o, bf2f(ho[(size_t(b) * Lq + i) * D + h * 64 + t]), 0.01 * c.mag, 0.02, i, h * 64 + t, c.name);
      }
    }
  }
  bool ok = report(c.name, st);
  ok = gout.intact(c.name) && ok;
  if (ok && c.time_iters > 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) call();
    CK(cudaEventRecord(e0));
    for (int i = 0; i < c.time_iters; ++i) call();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= c.time_iters;
    const double fl = 4.0 * B * H * double(Lq) * Lkv * 64;
    const double bytes = 2.0 * B * D * (2.0 * Lq + 2.0 * Lkv);
    printf("  time %s: %.3f ms  %.1f TFLOP/s  %.1f GB/s (algorithmic)\n", c.name, ms, fl / ms * 1e-9,
           bytes / ms * 1e-6);
    fflush(stdout);
  }
  return ok;
}

static const AttnCase kAttnCases[] = {
    // name        B   H   Lq    Lkv   self  causal mag  bh iters
    {"causal_l64", 1, 1, 64, 64, true, true, 1.0f, 0, 0},
    {"l64_tmem", 1, 1, 64, 64, true, false, 1.0f, 0, 0},
    {"causal_l128", 2, 2, 128, 128, true, true, 1.0f, 0, 0},
    {"l128_tmem", 2, 2, 128, 128, true, false, 1.0f, 0, 0},
    {"l197_tmem", 2, 3, 197, 197, true, false, 2.0f, 0, 0},
    {"l576_tmem", 1, 2, 576, 576, true, false, 2.0f, 0, 0},
    {"l1370_tmem", 1, 2, 1370, 1370, true, false, 3.0f, 1, 0},
    {"cross_q1", 3, 2, 1, 576, false, false, 2.0f, 0, 0},
    {"l16", 3, 2, 16, 16, true, false, 2.0f, 0, 0},
    {"causal_l16", 3, 2, 16, 16, true, true, 2.0f, 0, 0},
    {"causal_l197", 2, 3, 197, 197, true, true, 2.0f, 0, 0},
    {"causal_l448", 2, 2, 448, 448, true, true, 2.0f, 0, 0},
    {"causal_l700", 1, 2, 700, 700, true, true, 2.0f, 0, 0},
    {"causal_many", 30, 6, 300, 300, true, true, 2.0f, 8, 0},
    {"perf_causal_1500", 8, 20, 1500, 1500, true, true, 1.0f, 1, 10},
    {"l130", 2, 2, 130, 130, true, false, 2.0f, 0, 0},
    {"l256", 2, 2, 256, 256, true, false, 2.0f, 0, 0},
    {"cross_q300_kv200", 2, 2, 300, 200, false, false, 2.0f, 0, 0},
    {"cross_q1_kv200", 5, 3, 1, 200, false, false, 2.0f, 0, 0},
    {"many_short", 150, 4, 197, 197, true, false, 2.0f, 10, 0},
    {"many_items", 40, 12, 197, 197, true, false, 2.0f, 6, 0},
    {"perf_vitb", 128, 12, 197, 197, true, false, 1.0f, 2, 20},
    {"perf_vitb_causal", 128, 12, 197, 197, true, true, 1.0f, 2, 20},
    {"perf_whisper", 8, 20, 1500, 1500, true, false, 1.0f, 1, 10},
    {"perf_siglip", 32, 16, 576, 576, true, false, 1.0f, 1, 10},
    // full-batch shapes of BASELINE configs C2..C5 (one GPU): what one attention launch of the bench processes
    {"perf_vitb_b1024", 1024, 12, 197, 197, true, false, 1.0f, 2, 10},
    {"perf_siglip_b256", 256, 16, 576, 576, true, false, 1.0f, 1, 5},
    {"perf_dinov2_b128", 128, 16, 1370, 1370, true, false, 1.0f, 1, 5},
    {"perf_whisper_b64", 64, 20, 1500, 1500, true, false, 1.0f, 1, 5},
    {"l1500_wide", 1, 3, 1500, 1500, true, false, 4.0f, 0, 0},
    // short-sequence kernel (attention_short.cuh): every TMEM layout (nk16 <= 192, <= 224, <= 256), ragged tails
    {"l192", 2, 2, 192, 192, true, false, 2.0f, 0, 0},
    {"l193", 2, 2, 193, 193, true, false, 2.0f, 0, 0},
    {"l208", 2, 2, 208, 208, true, false, 2.0f, 0, 0},
    {"l224", 2, 2, 224, 224, true, false, 2.0f, 0, 0},
    {"l225", 2, 2, 225, 225, true, false, 2.0f, 0, 0},
    {"l250", 3, 2, 250, 250, true, false, 2.0f, 0, 0},
    {"l1", 3, 2, 1, 1, true, false, 2.0f, 0, 0},
    {"l33", 3, 2, 33, 33, true, false, 2.0f, 0, 0},
    {"cross_q600_kv250", 2, 2, 600, 250, false, false, 2.0f, 0, 0},
    {"cross_q700_kv100", 2, 2, 700, 100, false, false, 2.0f, 0, 0},
    {"many_short_items", 300, 6, 197, 197, true, false, 3.0f, 30, 0},
    {"many_short_q300", 200, 2, 300, 200, false, false, 2.0f, 20, 0},
    {"causal_l1100", 2, 2, 1100, 1100, true, true, 3.0f, 0, 0},
};

#ifdef ATT_TRACE
extern "C" void b200enc_debug_attention_trace(long long* buf);
static void run_attn_trace(int B, int H, int L) {
  const int D = H * 64;
  auto hq = rand_bf16(size_t(B) * L * 3 * D, 1.0f, false);
  DevBuf dq(hq.size() * 2), dout(size_t(B) * L * D * 2), dtr(8 * 10000);  // 5 roles x 1000 events x (id, clock)
  CK(cudaMemcpy(dq.p, hq.data(), hq.size() * 2, cudaMemcpyHostToDevice));
  uint16_t* base = (uint16_t*)dq.p;
  auto call = [&]() {
    return b200enc_attention(dq.p, (long long)L * 3 * D, 3 * D, base + D, base + 2 * D, (long long)L * 3 * D, 3 * D,
                             dout.p, (long long)L * D, D, B, H, L, L, 64, 0.125f, 0, nullptr);
  };
  for (int i = 0; i < 3; ++i) call();
  CK(cudaDeviceSynchronize());
  CK(cudaMemset(dtr.p, 0, dtr.bytes));
  b200enc_debug_attention_trace((long long*)dtr.p);
  call();
  CK(cudaDeviceSynchronize());
  std::vector<long long> h(10000);
  CK(cudaMemcpy(h.data(), dtr.p, h.size() * 8, cudaMemcpyDeviceToHost));
  long long t0 = 1LL << 62;
  for (int i = 0; i < 5000; ++i)
    if (h[2 * i + 1] > 0) t0 = std::min(t0, h[2 * i + 1]);
  for (int i = 0; i < 5000; ++i)
    if (h[2 * i + 1] > 0) printf("EV %lld %lld\n", h[2 * i], h[2 * i + 1] - t0);
}
#endif

// ------------------------------------------------------------------------------------------ layernorm / stats
static bool run_layernorm(int rows, int d, float eps, int row_mult, int iters) {
  printf("layernorm rows=%d d=%d eps=%g row_mult=%d\n", rows, d, eps, row_mult);
  const long long ldx = (long long)d * row_mult;
  auto hx = rand_bf16(size_t(rows) * ldx, 2.0f, false);
  for (size_t i = 0; i < hx.size(); ++i) hx[i] = f2bf(bf2f(hx[i]) + 0.7f);  // non-zero mean
  auto hg = rand_f32(d, 1.0f), hb = rand_f32(d, 0.5f);
  DevBuf dx(hx.size() * 2), dg(d * 4), db(d * 4), dst2(size_t(rows) * 8);
  GuardedBuf gout(size_t(rows) * d * 2), gst(size_t(rows) * 8);
  struct { void* p; } dout = {gout.p()}, dst = {gst.p()};
  CK(cudaMemcpy(dx.p, hx.data(), hx.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dg.p, hg.data(), d * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(db.p, hb.data(), d * 4, cudaMemcpyHostToDevice));
  int rc = b200enc_layernorm(dx.p, ldx, (float*)dg.p, (float*)db.p, eps, rows, d, dout.p, d, (float*)dst.p, nullptr);
  if (!rc) rc = b200enc_row_stats(dx.p, ldx, eps, rows, d, (float*)dst2.p, nullptr);
  if (rc) {
    printf("  [FAIL] rc=%d: %s\n", rc, b200enc_last_error());
    return false;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("  [FAIL] kernel error: %s\n", cudaGetErrorString(e));
    return false;
  }
  std::vector<uint16_t> ho(size_t(rows) * d);
  std::vector<float> hs(size_t(rows) * 2), hs2(size_t(rows) * 2);
  CK(cudaMemcpy(ho.data(), dout.p, ho.size() * 2, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hs.data(), dst.p, hs.size() * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hs2.data(), dst2.p, hs2.size() * 4, cudaMemcpyDeviceToHost));
  CmpStat st, ss;
  const int step = rows > 512 ? rows / 512 : 1;
  for (int r = 0; r < rows; r += step) {
    const uint16_t* xr = &hx[size_t(r) * ldx];
    double m = 0, v = 0;
    for (int k = 0; k < d; ++k) m += bf2f(xr[k]);
    m /= d;
    for (int k = 0; k < d; ++k) v += (bf2f(xr[k]) - m) * (bf2f(xr[k]) - m);
    v /= d;
    const double rstd = 1.0 / sqrt(v + eps);
    cmp_one(ss, m, hs[2 * r], 1e-5, 1e-5, r, 0, "mean");
    cmp_one(ss, rstd, hs[2 * r + 1], 1e-5, 1e-4, r, 1, "rstd");
    cmp_one(ss, m, hs2[2 * r], 1e-5, 1e-5, r, 2, "mean2");
    cmp_one(ss, rstd, hs2[2 * r + 1], 1e-5, 1e-4, r, 3, "rstd2");
    for (int k = 0; k < d; ++k)
      cmp_one(st, (bf2f(xr[k]) - m) * rstd * hg[k] + hb[k], bf2f(ho[size_t(r) * d + k]), 0.01, 0.008, r, k, "ln");
  }
  bool ok = report("layernorm", st);
  ok = report("row_stats", ss) && ok;
  ok = gout.intact("layernorm out") && gst.intact("layernorm stats") && ok;
  if (ok && iters > 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i)
      b200enc_layernorm(dx.p, ldx, (float*)dg.p, (float*)db.p, eps, rows, d, dout.p, d, nullptr, nullptr);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= iters;
    printf("  time layernorm: %.3f ms  %.1f GB/s\n", ms, 4.0 * rows * d / ms * 1e-6);
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) b200enc_row_stats(dx.p, ldx, eps, rows, d, (float*)dst2.p, nullptr);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= iters;
    printf("  time row_stats: %.3f ms  %.1f GB/s\n", ms, 2.0 * rows * d / ms * 1e-6);
  }
  return ok;
}

// ------------------------------------------------------------------------------------------ patch rows
static bool run_patch(int B, int HW, int p, bool f32) {
  const int Kp = (3 * p * p + 7) / 8 * 8, P = (HW / p) * (HW / p);
  printf("patch_rows B=%d HW=%d p=%d f32=%d Kpad=%d\n", B, HW, p, f32, Kp);
  const size_t n = size_t(B) * 3 * HW * HW;
  std::vector<float> hf(n);
  std::vector<uint16_t> hb(n);
  for (size_t i = 0; i < n; ++i) {
    hf[i] = urand() * 2;
    hb[i] = f2bf(hf[i]);
  }
  DevBuf dimg(n * 4), drows(size_t(B) * P * Kp * 2);
  if (f32)
    CK(cudaMemcpy(dimg.p, hf.data(), n * 4, cudaMemcpyHostToDevice));
  else
    CK(cudaMemcpy(dimg.p, hb.data(), n * 2, cudaMemcpyHostToDevice));
  CK(cudaMemset(drows.p, 0x7f, drows.bytes));
  int rc = b200enc_patch_rows(dimg.p, f32 ? B200ENC_DTYPE_F32 : B200ENC_DTYPE_BF16, B, HW, HW, p, Kp, drows.p, nullptr);
  if (rc) {
    printf("  [FAIL] rc=%d: %s\n", rc, b200enc_last_error());
    return false;
  }
  CK(cudaDeviceSynchronize());
  std::vector<uint16_t> hr(size_t(B) * P * Kp);
  CK(cudaMemcpy(hr.data(), drows.p, hr.size() * 2, cudaMemcpyDeviceToHost));
  CmpStat st;
  const int Wp = HW / p;
  for (int b = 0; b < B; ++b)
    for (int t = 0; t < P; ++t)
      for (int k = 0; k < Kp; ++k) {
        double want = 0;
        if (k < 3 * p * p) {
          const int c = k / (p * p), i = (k / p) % p, j = k % p, ph = t / Wp, pw = t % Wp;
          want = bf2f(hb[((size_t(b) * 3 + c) * HW + ph * p + i) * HW + pw * p + j]);
        }
        cmp_one(st, want, bf2f(hr[(size_t(b) * P + t) * Kp + k]), 0, 0, b * P + t, k, "patch");
      }
  return report("patch_rows", st);
}

// im2col-free patch embedding (b200enc_patch_embed16): tokens[b][off + patch] = conv(img)[patch] + bias + pe[patch],
// optional LayerNorm partial statistics of the stored rows; fp64 CPU check of every output, guard bands around the
// token buffer (the class-token rows and the tail must stay untouched).
static bool run_patch_embed(int n, int H, int W, int N, int tok_off, bool stats, int iters) {
  const int hp = H / 16, wp = W / 16, P = hp * wp, L = P + tok_off, K = 768;
  printf("patch_embed16 n=%d %dx%d N=%d token offset %d stats=%d\n", n, H, W, N, tok_off, int(stats));
  fflush(stdout);
  std::vector<uint16_t> himg = rand_bf16(size_t(n) * 3 * H * W, 1.0f, false);
  std::vector<uint16_t> hw = rand_bf16(size_t(N) * K, 0.06f, false);
  std::vector<uint16_t> hpe = rand_bf16(size_t(P) * N, 1.0f, false);
  std::vector<float> hbias(N);
  for (auto& v : hbias) v = urand();
  const int n_sl = (N + 127) / 128;
  DevBuf dimg(himg.size() * 2), dw(hw.size() * 2), dpe(hpe.size() * 2), dbias(N * 4);
  GuardedBuf gtok(size_t(n) * L * N * 2), gst(size_t(n) * L * n_sl * 8);
  CK(cudaMemcpy(dimg.p, himg.data(), himg.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw.p, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dpe.p, hpe.data(), hpe.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dbias.p, hbias.data(), N * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(gtok.p(), 0x7f, gtok.bytes));
  CK(cudaMemset(gst.p(), 0x7f, gst.bytes));
  b200enc_linear_args a;
  memset(&a, 0, sizeof(a));
  a.x = dimg.p;
  a.w = dw.p;
  a.ldw = K;
  a.bias = (const float*)dbias.p;
  a.residual = dpe.p;
  a.res_batch_stride = 0;
  a.ldr = N;
  a.out = (uint16_t*)gtok.p() + size_t(tok_off) * N;
  a.out_batch_stride = (long long)L * N;
  a.ldo = N;
  a.stats_out = stats ? (float*)gst.p() : nullptr;
  a.stats_rows_per_batch = L;
  a.stats_row_offset = tok_off;
  a.batches = n;
  a.M = P;
  a.N = N;
  a.K = K;
  auto call = [&]() { return b200enc_patch_embed16(&a, H, W, nullptr); };
  int rc = call();
  if (rc) {
    printf("  [FAIL] rc=%d: %s\n", rc, b200enc_last_error());
    return false;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("  [FAIL] kernel error: %s\n", cudaGetErrorString(e));
    return false;
  }
  std::vector<uint16_t> ho(size_t(n) * L * N);
  std::vector<float> hs(size_t(n) * L * n_sl * 2);
  CK(cudaMemcpy(ho.data(), gtok.p(), ho.size() * 2, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hs.data(), gst.p(), hs.size() * 4, cudaMemcpyDeviceToHost));
  CmpStat st, sst;
  long untouched_bad = 0;
  std::vector<float> arow(K);
  const int bstep = n > 4 ? n / 4 : 1;
  for (int b = 0; b < n; b += bstep) {
    for (int t = 0; t < tok_off; ++t)
      for (int c = 0; c < N; ++c) untouched_bad += ho[(size_t(b) * L + t) * N + c] != 0x7f7f;
    for (int pt = 0; pt < P; ++pt) {
      const int ph = pt / wp, pw = pt % wp;
      for (int k = 0; k < K; ++k) {
        const int c = k / 256, i = (k / 16) % 16, j = k % 16;
        arow[k] = bf2f(himg[((size_t(b) * 3 + c) * H + ph * 16 + i) * W + pw * 16 + j]);
      }
      std::vector<double> orow(N);
      for (int c = 0; c < N; ++c) {
        double acc = 0;
        const uint16_t* wr = &hw[size_t(c) * K];
        for (int k = 0; k < K; ++k) acc += double(arow[k]) * double(bf2f(wr[k]));
        acc += hbias[c] + bf2f(hpe[size_t(pt) * N + c]);
        const float got = bf2f(ho[(size_t(b) * L + tok_off + pt) * N + c]);
        cmp_one(st, acc, got, 0.02, 0.01, b * P + pt, c, "patch_embed16");
        orow[c] = got;  // statistics are those of the stored values
      }
      if (stats)
        for (int sl = 0; sl < n_sl; ++sl) {
          const int c0 = sl * 128, c1 = std::min(N, c0 + 128);
          double mean = 0, m2 = 0;
          for (int c = c0; c < c1; ++c) mean += orow[c];
          mean /= (c1 - c0);
          for (int c = c0; c < c1; ++c) m2 += (orow[c] - mean) * (orow[c] - mean);
          const float* g = &hs[((size_t(b) * L + tok_off + pt) * n_sl + sl) * 2];
          cmp_one(sst, mean, g[0], 1e-3, 1e-3, b * P + pt, sl, "patch_embed16 mean");
          cmp_one(sst, m2, g[1], 1e-2, 1e-3, b * P + pt, sl, "patch_embed16 M2");
        }
    }
  }
  bool ok = report("patch_embed16", st);
  if (stats) ok = report("patch_embed16 statistics", sst) && ok;
  if (untouched_bad) {
    printf("  [FAIL] %ld class-token elements were overwritten\n", untouched_bad);
    ok = false;
  }
  ok = gtok.intact("patch_embed16 tokens") && ok;
  ok = gst.intact("patch_embed16 statistics") && ok;
  if (ok && iters > 0) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) call();
    CK(cudaEventRecord(e0));
    for (int i = 0; i < iters; ++i) call();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= iters;
    printf("  time patch_embed16: %.3f ms  %.1f TFLOP/s  %.1f GB/s (image in, tokens out, pe)\n", ms,
           2.0 * n * P * N * K / ms * 1e-9, (2.0 * n * 3 * H * W + 2.0 * n * P * N) / ms * 1e-6);
  }
  return ok;
}

int main(int argc, char** argv) {
  if (argc < 2) {
    printf("usage: %s <case>|list\n", argv[0]);
    return 2;
  }
  std::string which = argv[1];
  if (which == "list") {
    for (auto& c : kLinearCases) printf("linear:%s\n", c.name);
    for (auto& c : kAttnCases) printf("attn:%s\n", c.name);
    printf("rows:all\n");
    return 0;
  }
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("device: %s sm_%d%d, %d SMs\n", prop.name, prop.major, prop.minor, prop.multiProcessorCount);
  bool ok = true, found = false;
  for (auto& c : kLinearCases) {
    if (which == std::string("linear:") + c.name || which == "linear:all") {
      found = true;
      ok = run_linear(c) && ok;
    }
  }
  for (auto& c : kAttnCases) {
    if (which == std::string("attn:") + c.name || which == "attn:all") {
      found = true;
      ok = run_attn(c) && ok;
    }
  }
#ifdef ATT_TRACE
  if (which == "attn:trace") {
    found = true;
    run_attn_trace(argc > 2 ? atoi(argv[2]) : 128, argc > 3 ? atoi(argv[3]) : 12, argc > 4 ? atoi(argv[4]) : 197);
  }
#endif
  if (which == "patch:all" || which == "patch:perf") {
    found = true;
    if (which == "patch:all") {
      ok = run_patch_embed(2, 224, 224, 768, 1, true, 0) && ok;
      ok = run_patch_embed(1, 384, 384, 1024, 0, false, 0) && ok;   // 24 x 24 patches: 3 x 2 tiles per image
      ok = run_patch_embed(3, 64, 48, 256, 1, true, 0) && ok;        // 4 x 3 patches: one sparse tile
      ok = run_patch_embed(5, 16, 16, 64, 0, true, 0) && ok;         // a single patch per image
      ok = run_patch_embed(2, 272, 400, 384, 1, true, 0) && ok;      // 17 x 25 patches: ragged in both directions
      ok = run_patch_embed(300, 32, 32, 128, 1, false, 0) && ok;     // more tiles than SMs
    } else {
      ok = run_patch_embed(1024, 224, 224, 768, 1, true, 10) && ok;
    }
  }
  if (which == "rows:all") {
    found = true;
    ok = run_layernorm(1000, 768, 1e-6f, 1, 0) && ok;
    ok = run_layernorm(333, 192, 1e-5f, 1, 0) && ok;
    ok = run_layernorm(77, 1280, 1e-5f, 1, 0) && ok;
    ok = run_layernorm(64, 1024, 1e-6f, 5, 0) && ok;  // strided rows (class-token gather)
    ok = run_layernorm(201728, 768, 1e-6f, 1, 20) && ok;
    ok = run_patch(2, 224, 16, false) && ok;
    ok = run_patch(2, 224, 16, true) && ok;
    ok = run_patch(1, 518, 14, false) && ok;
    ok = run_patch(1, 518, 14, true) && ok;
    ok = run_patch(2, 64, 8, false) && ok;
  }
  if (!found) {
    printf("unknown case %s\n", which.c_str());
    return 2;
  }
  printf("%s\n", ok ? "SELFTEST PASS" : "SELFTEST FAIL");
  return ok ? 0 : 1;
}
