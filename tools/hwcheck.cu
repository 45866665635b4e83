// Stand-alone hardware check of the pieces that were written after the round's GPU budget was (almost) spent:
// no Python, no PyTorch -- the process starts in a fraction of a second, so it fits into a few seconds of GPU time.
// Calls the C ABI of libcrf_sm100.so directly and compares with plain C++ references evaluated in double precision
// on the same bf16-rounded inputs:
//   1. window-attention core forward / backward: head_dim 32 (the verified kernels: validates THIS harness), then
//      head_dim 64 and 128 (csrc/crf_attn_wide.cu)
//   2. the stand-alone LayerNorm forward (crf_layernorm_fwd)
//   3. the multi-tensor Adam step (crf_adam_step)
// Every result line goes to stdout and to gpurun_out/hwcheck.txt as soon as it is known.
//   make -C monocular_depth_estimation_b200/csrc hwcheck
//   tools/hwcheck            (on a B200)          tools/hwcheck --dry DIR   (no GPU: dumps inputs + references to DIR)
//   tools/hwcheck --bench    (on a B200: CUDA-event timings of these kernels at config-2 sizes, a few seconds)
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <string>
#include <vector>

#include "crf_adam_math.h"
#include "crf_sm100.h"
#include "crf_window.cuh"

static FILE* g_log = nullptr;
static double now_s() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}
static double g_t0 = 0;
static void say(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  printf("[%6.2fs] %s\n", now_s() - g_t0, buf);
  fflush(stdout);
  if (g_log) {
    fprintf(g_log, "[%6.2fs] %s\n", now_s() - g_t0, buf);
    fflush(g_log);
  }
}

// ---- bf16 helpers (round to nearest even) and a small deterministic generator ----
static uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}
static float bf2f(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed * 2862933555777941757ull + 3037000493ull) {}
  float uni() {  // (-1, 1)
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    return static_cast<float>((s >> 40) & 0xFFFFFF) / 8388608.0f - 1.0f;
  }
  float gauss() { return (uni() + uni() + uni() + uni()) * 0.8660254f; }  // ~N(0,1)
};

static double rel_l2(const std::vector<double>& a, const std::vector<double>& b) {
  double num = 0, den = 0;
  for (size_t i = 0; i < a.size(); ++i) {
    num += (a[i] - b[i]) * (a[i] - b[i]);
    den += b[i] * b[i];
  }
  return sqrt(num / (den > 1e-300 ? den : 1e-300));
}

// rel_l2 per 32-wide slice of a head (aggregated over heads and tokens): tells which slice of a wide head went wrong
static std::string slice_errs(const std::vector<double>& got, const std::vector<double>& ref, int T, int C, int hd) {
  std::string out;
  for (int s = 0; s < hd / 32; ++s) {
    double num = 0, den = 0;
    for (int t = 0; t < T; ++t)
      for (int c = 0; c < C; ++c)
        if ((c % hd) / 32 == s) {
          const double a = got[static_cast<size_t>(t) * C + c], b = ref[static_cast<size_t>(t) * C + c];
          num += (a - b) * (a - b);
          den += b * b;
        }
    char buf[32];
    snprintf(buf, sizeof(buf), "%s%.1e", s ? " " : "", sqrt(num / (den > 1e-300 ? den : 1e-300)));
    out += buf;
  }
  return out;
}

#define CK(call)                                                                     \
  do {                                                                               \
    cudaError_t e_ = (call);                                                         \
    if (e_ != cudaSuccess) {                                                         \
      say("CUDA error %s at %s:%d", cudaGetErrorString(e_), __FILE__, __LINE__);     \
      return 1;                                                                      \
    }                                                                                \
  } while (0)

template <typename T>
static T* dev_copy(const std::vector<T>& h) {
  T* d = nullptr;
  if (cudaMalloc(&d, h.size() * sizeof(T) + 64) != cudaSuccess) return nullptr;
  cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  return d;
}
template <typename T>
static std::vector<T> host_copy(const T* d, size_t n) {
  std::vector<T> h(n);
  cudaMemcpy(h.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost);
  return h;
}
static void dump(const std::string& dir, const char* name, const void* p, size_t bytes) {
  FILE* f = fopen((dir + "/" + name).c_str(), "wb");
  if (f) {
    fwrite(p, 1, bytes, f);
    fclose(f);
  }
}

// =====================================================================================================
// attention core
// =====================================================================================================
struct AttnCase {
  int B, H, W, C, nH, shift;
};
struct AttnRef {
  std::vector<double> o, lse, dq, dk, dv, dtable, dbias;  // o (T,C); lse (B*nW,nH,64); dq,dk,dv (T,C); dtable (169,nH); dbias (2C)
  std::vector<char> lse_valid;
};

static void attn_reference(const AttnCase& c, const std::vector<uint16_t>& qk, const std::vector<uint16_t>& vb,
                           const std::vector<float>& bias, const std::vector<float>& table,
                           const std::vector<uint16_t>& dout, float scale, AttnRef& R) {
  const int C = c.C, nH = c.nH, hd = C / nH, T = c.B * c.H * c.W;
  crf::WindowGeom gm(c.H, c.W, 7, c.shift);
  const int nWin = c.B * gm.nW;
  R.o.assign(static_cast<size_t>(T) * C, 0.0);
  R.dq.assign(static_cast<size_t>(T) * C, 0.0);
  R.dk.assign(static_cast<size_t>(T) * C, 0.0);
  R.dv.assign(static_cast<size_t>(T) * C, 0.0);
  R.lse.assign(static_cast<size_t>(nWin) * nH * 64, 0.0);
  R.lse_valid.assign(static_cast<size_t>(nWin) * nH * 64, 0);
  R.dtable.assign(169 * nH, 0.0);
  R.dbias.assign(2 * C, 0.0);
  std::vector<double> q(49 * hd), k(49 * hd), v(49 * hd), g(49 * hd), S(49 * 49), P(49 * 49), dP(49 * 49), dS(49 * 49);
  for (int wg = 0; wg < nWin; ++wg) {
    const int b = wg / gm.nW, win = wg % gm.nW;
    int tok[49], reg[49];
    for (int p = 0; p < 49; ++p) {
      const int s = gm.source(win, p);
      tok[p] = s < 0 ? -1 : b * c.H * c.W + s;
      reg[p] = c.shift > 0 ? gm.region(win, p) : 0;
    }
    for (int h = 0; h < nH; ++h) {
      for (int p = 0; p < 49; ++p)
        for (int d = 0; d < hd; ++d) {
          const int col = h * hd + d;
          if (tok[p] >= 0) {
            q[p * hd + d] = bf2f(qk[static_cast<size_t>(tok[p]) * 2 * C + col]);
            k[p * hd + d] = bf2f(qk[static_cast<size_t>(tok[p]) * 2 * C + C + col]);
            v[p * hd + d] = bf2f(vb[static_cast<size_t>(tok[p]) * C + col]);
            g[p * hd + d] = bf2f(dout[static_cast<size_t>(tok[p]) * C + col]);
          } else {  // zero-padded token: q row unused (cropped), k = bf16(bias), v = 0, no incoming gradient
            q[p * hd + d] = 0.0;
            k[p * hd + d] = bf2f(f2bf(bias[C + col]));
            v[p * hd + d] = 0.0;
            g[p * hd + d] = 0.0;
          }
        }
      for (int i = 0; i < 49; ++i) {
        double mx = -1e300;
        for (int j = 0; j < 49; ++j) {
          double s = 0;
          for (int d = 0; d < hd; ++d) s += q[i * hd + d] * k[j * hd + d];
          const int idx = (i / 7 - j / 7 + 6) * 13 + (i % 7 - j % 7 + 6);
          s += table[idx * nH + h];
          if (c.shift > 0 && reg[i] != reg[j]) s += -100.0;
          S[i * 49 + j] = s;
          mx = s > mx ? s : mx;
        }
        double sum = 0;
        for (int j = 0; j < 49; ++j) sum += exp(S[i * 49 + j] - mx);
        const double lse = mx + log(sum);
        for (int j = 0; j < 49; ++j) P[i * 49 + j] = exp(S[i * 49 + j] - lse);
        R.lse[(static_cast<size_t>(wg) * nH + h) * 64 + i] = lse;
        R.lse_valid[(static_cast<size_t>(wg) * nH + h) * 64 + i] = tok[i] >= 0;
        if (tok[i] >= 0)
          for (int d = 0; d < hd; ++d) {
            double o = 0;
            for (int j = 0; j < 49; ++j) o += P[i * 49 + j] * v[j * hd + d];
            R.o[static_cast<size_t>(tok[i]) * C + h * hd + d] = o;
          }
      }
      // backward
      for (int i = 0; i < 49; ++i) {
        double dot = 0;
        for (int j = 0; j < 49; ++j) {
          double s = 0;
          for (int d = 0; d < hd; ++d) s += g[i * hd + d] * v[j * hd + d];
          dP[i * 49 + j] = s;
          dot += P[i * 49 + j] * s;
        }
        for (int j = 0; j < 49; ++j) {
          dS[i * 49 + j] = tok[i] >= 0 ? P[i * 49 + j] * (dP[i * 49 + j] - dot) : 0.0;
          const int idx = (i / 7 - j / 7 + 6) * 13 + (i % 7 - j % 7 + 6);
          R.dtable[idx * nH + h] += dS[i * 49 + j];
        }
      }
      for (int j = 0; j < 49; ++j)
        for (int d = 0; d < hd; ++d) {
          double dv = 0, dk = 0;
          for (int i = 0; i < 49; ++i) {
            if (tok[i] < 0) continue;
            dv += P[i * 49 + j] * g[i * hd + d];
            dk += dS[i * 49 + j] * q[i * hd + d];
          }
          if (tok[j] >= 0) {
            R.dv[static_cast<size_t>(tok[j]) * C + h * hd + d] = dv;
            R.dk[static_cast<size_t>(tok[j]) * C + h * hd + d] = dk;
          } else {
            R.dbias[C + h * hd + d] += dk;
          }
        }
      for (int i = 0; i < 49; ++i)
        if (tok[i] >= 0)
          for (int d = 0; d < hd; ++d) {
            double dq = 0;
            for (int j = 0; j < 49; ++j) dq += dS[i * 49 + j] * k[j * hd + d];
            R.dq[static_cast<size_t>(tok[i]) * C + h * hd + d] = dq * scale;  // the kernel returns d(pre-scale q)
          }
    }
  }
}

static int run_attn_case(const AttnCase& c, const char* tag, const std::string& dry_dir) {
  const int C = c.C, nH = c.nH, T = c.B * c.H * c.W, hd = C / nH;
  const float scale = 1.0f / sqrtf(static_cast<float>(hd));
  crf::WindowGeom gm(c.H, c.W, 7, c.shift);
  const int nWin = c.B * gm.nW;
  Rng rng(1000 + C * 7 + nH * 3 + c.shift + c.H);
  std::vector<uint16_t> qk(static_cast<size_t>(T) * 2 * C), vb(static_cast<size_t>(T) * C), dout(static_cast<size_t>(T) * C);
  for (auto& x : qk) x = f2bf(0.7f * rng.gauss());
  for (size_t t = 0; t < static_cast<size_t>(T); ++t)   // q is stored pre-multiplied by scale (GEMM epilogue)
    for (int cc = 0; cc < C; ++cc) qk[t * 2 * C + cc] = f2bf(bf2f(qk[t * 2 * C + cc]) * scale * 2.0f);
  for (auto& x : vb) x = f2bf(rng.gauss());
  for (auto& x : dout) x = f2bf(rng.gauss());
  std::vector<float> bias(2 * C), table(169 * nH);
  for (auto& x : bias) x = bf2f(f2bf(0.5f * rng.gauss()));
  for (auto& x : table) x = 0.5f * rng.gauss();
  AttnRef R;
  attn_reference(c, qk, vb, bias, table, dout, scale, R);
  if (!dry_dir.empty()) {
    const std::string d = dry_dir + "/" + tag;
    std::string cmd = "mkdir -p " + d;
    if (system(cmd.c_str()) != 0) return 1;
    const int meta[8] = {c.B, c.H, c.W, c.C, c.nH, c.shift, nWin, 0};
    dump(d, "meta.i32", meta, sizeof(meta));
    dump(d, "qk.bf16", qk.data(), qk.size() * 2);
    dump(d, "vb.bf16", vb.data(), vb.size() * 2);
    dump(d, "dout.bf16", dout.data(), dout.size() * 2);
    dump(d, "bias.f32", bias.data(), bias.size() * 4);
    dump(d, "table.f32", table.data(), table.size() * 4);
    dump(d, "o.f64", R.o.data(), R.o.size() * 8);
    dump(d, "lse.f64", R.lse.data(), R.lse.size() * 8);
    dump(d, "dq.f64", R.dq.data(), R.dq.size() * 8);
    dump(d, "dk.f64", R.dk.data(), R.dk.size() * 8);
    dump(d, "dv.f64", R.dv.data(), R.dv.size() * 8);
    dump(d, "dtable.f64", R.dtable.data(), R.dtable.size() * 8);
    dump(d, "dbias.f64", R.dbias.data(), R.dbias.size() * 8);
    say("%s: dry run, reference dumped to %s", tag, d.c_str());
    return 0;
  }

  crf_block_desc d;
  memset(&d, 0, sizeof(d));
  d.B = c.B; d.H = c.H; d.W = c.W; d.C = C; d.num_heads = nH; d.window = 7; d.shift = c.shift; d.training = 1;
  d.device = 0; d.x_dtype = CRF_DT_F32; d.v_dtype = CRF_DT_BF16; d.v_preconverted = 1;
  d.x_stride_b = static_cast<int64_t>(c.H) * c.W * C; d.x_stride_t = C; d.x_stride_c = 1;
  d.v_stride_b = d.x_stride_b; d.v_stride_h = static_cast<int64_t>(c.W) * C; d.v_stride_w = C; d.v_stride_c = 1;

  uint16_t *d_qk = dev_copy(qk), *d_vb = dev_copy(vb), *d_dout = dev_copy(dout);
  float *d_bias = dev_copy(bias), *d_table = dev_copy(table);
  uint16_t *d_o = nullptr, *d_dqk = nullptr;
  float *d_lse = nullptr, *d_dv = nullptr, *d_dtable = nullptr, *d_dbias = nullptr;
  CK(cudaMalloc(&d_o, static_cast<size_t>(T) * C * 2));
  CK(cudaMalloc(&d_dqk, static_cast<size_t>(T) * 2 * C * 2));
  CK(cudaMalloc(&d_lse, static_cast<size_t>(nWin) * nH * 64 * 4));
  CK(cudaMalloc(&d_dv, static_cast<size_t>(T) * C * 4));
  CK(cudaMalloc(&d_dtable, 169 * nH * 4));
  CK(cudaMalloc(&d_dbias, 2 * C * 4));
  CK(cudaMemset(d_o, 0, static_cast<size_t>(T) * C * 2));
  CK(cudaMemset(d_dqk, 0, static_cast<size_t>(T) * 2 * C * 2));
  CK(cudaMemset(d_lse, 0, static_cast<size_t>(nWin) * nH * 64 * 4));
  CK(cudaMemset(d_dv, 0, static_cast<size_t>(T) * C * 4));
  CK(cudaMemset(d_dtable, 0, 169 * nH * 4));
  CK(cudaMemset(d_dbias, 0, 2 * C * 4));

  if (crf_attn_fwd(&d, d_qk, d_vb, d_bias, scale, d_table, nullptr, 0, d_o, d_lse, nullptr)) {
    say("%s: FAIL crf_attn_fwd: %s", tag, crf_last_error());
    return 1;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    say("%s: FAIL forward kernel: %s", tag, cudaGetErrorString(e));
    return 2;
  }
  {
    const auto o = host_copy(d_o, static_cast<size_t>(T) * C);
    const auto lse = host_copy(d_lse, static_cast<size_t>(nWin) * nH * 64);
    std::vector<double> og(o.size());
    for (size_t i = 0; i < o.size(); ++i) og[i] = bf2f(o[i]);
    double lse_err = 0;
    for (size_t i = 0; i < lse.size(); ++i)
      if (R.lse_valid[i]) lse_err = fmax(lse_err, fabs(lse[i] - R.lse[i]));
    const double eo = rel_l2(og, R.o);
    say("%s fwd: rel_l2(o) %.2e (tol 1e-2; per 32-col slice: %s)  max|lse err| %.2e (tol 2e-3)  -> %s", tag, eo,
        slice_errs(og, R.o, T, C, hd).c_str(), lse_err, (eo < 1e-2 && lse_err < 2e-3) ? "PASS" : "FAIL");
  }
  if (crf_attn_bwd(&d, d_qk, d_vb, d_bias, scale, d_table, nullptr, 0, d_lse, d_dout, d_dqk, d_dv, 0, d_dtable, d_dbias,
                   nullptr)) {
    say("%s: FAIL crf_attn_bwd: %s", tag, crf_last_error());
    return 1;
  }
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    say("%s: FAIL backward kernel: %s", tag, cudaGetErrorString(e));
    return 2;
  }
  {
    const auto dqk = host_copy(d_dqk, static_cast<size_t>(T) * 2 * C);
    const auto dv = host_copy(d_dv, static_cast<size_t>(T) * C);
    const auto dt = host_copy(d_dtable, static_cast<size_t>(169) * nH);
    const auto db = host_copy(d_dbias, static_cast<size_t>(2) * C);
    std::vector<double> gq(static_cast<size_t>(T) * C), gk(gq.size()), gv(gq.size()), gt(dt.begin(), dt.end()), gb(db.begin(), db.end());
    for (size_t t = 0; t < static_cast<size_t>(T); ++t)
      for (int cc = 0; cc < C; ++cc) {
        gq[t * C + cc] = bf2f(dqk[t * 2 * C + cc]);
        gk[t * C + cc] = bf2f(dqk[t * 2 * C + C + cc]);
        gv[t * C + cc] = dv[t * C + cc];
      }
    const double eq = rel_l2(gq, R.dq), ek = rel_l2(gk, R.dk), ev = rel_l2(gv, R.dv), et = rel_l2(gt, R.dtable);
    double nb = 0;
    for (double x : R.dbias) nb += x * x;
    const double eb = nb > 0 ? rel_l2(gb, R.dbias) : 0.0;
    const bool ok = eq < 1.5e-2 && ek < 1.5e-2 && ev < 1e-2 && et < 1.5e-2 && eb < 1.5e-2;
    say("%s bwd: rel_l2 dq %.2e [%s] dk %.2e [%s] dv %.2e [%s] d_table %.2e d_bias_k %.2e (tol 1.5e-2, dv 1e-2) -> %s", tag,
        eq, slice_errs(gq, R.dq, T, C, hd).c_str(), ek, slice_errs(gk, R.dk, T, C, hd).c_str(), ev,
        slice_errs(gv, R.dv, T, C, hd).c_str(), et, eb, ok ? "PASS" : "FAIL");
  }
  cudaFree(d_qk); cudaFree(d_vb); cudaFree(d_dout); cudaFree(d_bias); cudaFree(d_table); cudaFree(d_o); cudaFree(d_dqk);
  cudaFree(d_lse); cudaFree(d_dv); cudaFree(d_dtable); cudaFree(d_dbias);
  return 0;
}

// =====================================================================================================
// LayerNorm forward
// =====================================================================================================
static int run_ln_case(int T, int C) {
  Rng rng(77 + C);
  std::vector<float> x(static_cast<size_t>(T) * C), gamma(C), beta(C);
  for (auto& v : x) v = 1.7f * rng.gauss() + 0.3f;
  for (auto& v : gamma) v = 1.0f + 0.2f * rng.gauss();
  for (auto& v : beta) v = 0.1f * rng.gauss();
  float *dx = dev_copy(x), *dg = dev_copy(gamma), *db = dev_copy(beta), *dy = nullptr, *ds = nullptr;
  CK(cudaMalloc(&dy, x.size() * 4));
  CK(cudaMalloc(&ds, static_cast<size_t>(T) * 2 * 4));
  CK(cudaMemset(dy, 0xFF, x.size() * 4));
  if (crf_layernorm_fwd(dx, dg, db, 1e-5f, dy, CRF_DT_F32, ds, T, C, 0, nullptr)) {
    say("layernorm T%d C%d: FAIL %s", T, C, crf_last_error());
    return 1;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    say("layernorm T%d C%d: FAIL kernel: %s", T, C, cudaGetErrorString(e));
    return 2;
  }
  const auto y = host_copy(dy, x.size());
  const auto st = host_copy(ds, static_cast<size_t>(T) * 2);
  std::vector<double> got(y.begin(), y.end()), ref(y.size());
  double se = 0;
  for (int t = 0; t < T; ++t) {
    double m = 0, q = 0;
    for (int c = 0; c < C; ++c) m += x[static_cast<size_t>(t) * C + c];
    m /= C;
    for (int c = 0; c < C; ++c) q += (x[static_cast<size_t>(t) * C + c] - m) * (x[static_cast<size_t>(t) * C + c] - m);
    const double rstd = 1.0 / sqrt(q / C + 1e-5);
    se = fmax(se, fmax(fabs(st[2 * t] - m), fabs(st[2 * t + 1] - rstd) / rstd));
    for (int c = 0; c < C; ++c) ref[static_cast<size_t>(t) * C + c] = (x[static_cast<size_t>(t) * C + c] - m) * rstd * gamma[c] + beta[c];
  }
  const double ey = rel_l2(got, ref);
  say("layernorm_fwd T%d C%d: rel_l2(y) %.2e  stats err %.2e (tol 1e-5) -> %s", T, C, ey, se,
      (ey < 1e-5 && se < 1e-5) ? "PASS" : "FAIL");
  cudaFree(dx); cudaFree(dg); cudaFree(db); cudaFree(dy); cudaFree(ds);
  return 0;
}

// =====================================================================================================
// Adam
// =====================================================================================================
static int run_adam() {
  const int sizes[4] = {5, 16385, 4096 * 33, 1031};
  const float lr = 1e-3f, b1 = 0.9f, b2 = 0.999f, eps = 1e-8f;
  Rng rng(5);
  std::vector<std::vector<float>> p(4), m(4), v(4);
  std::vector<float*> dp(4), dm(4), dv(4), dgbase(4);
  for (int i = 0; i < 4; ++i) {
    p[i].resize(sizes[i]);
    for (auto& x : p[i]) x = rng.gauss();
    m[i].assign(sizes[i], 0.f);
    v[i].assign(sizes[i], 0.f);
    dp[i] = dev_copy(p[i]);
    dm[i] = dev_copy(m[i]);
    dv[i] = dev_copy(v[i]);
    CK(cudaMalloc(&dgbase[i], (sizes[i] + 8) * 4));
  }
  float* dstep = nullptr;
  CK(cudaMalloc(&dstep, 4));
  CK(cudaMemset(dstep, 0, 4));
  for (int step = 1; step <= 3; ++step) {
    crf_adam_tensor rec[4];
    for (int i = 0; i < 4; ++i) {
      std::vector<float> g(sizes[i]);
      for (auto& x : g) x = rng.gauss() * powf(10.f, static_cast<float>(step - 2));
      float* dg = dgbase[i] + (i == 3 ? 1 : 0);   // tensor 3: 4-byte-aligned gradient view
      CK(cudaMemcpy(dg, g.data(), g.size() * 4, cudaMemcpyHostToDevice));
      rec[i] = {dp[i], dg, dm[i], dv[i], sizes[i]};
      const crf::AdamCoef c = crf::adam_coef(lr, b1, b2, eps, 0.0, static_cast<double>(step));
      for (int k = 0; k < sizes[i]; ++k) crf::adam_update(c, p[i][k], g[k], m[i][k], v[i][k]);
    }
    if (crf_adam_step(rec, 4, 16384, lr, b1, b2, eps, 0.f, dstep, 0, nullptr)) {
      say("adam: FAIL %s", crf_last_error());
      return 1;
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      say("adam: FAIL kernel: %s", cudaGetErrorString(e));
      return 2;
    }
  }
  double worst = 0;
  for (int i = 0; i < 4; ++i) {
    const auto gp = host_copy(dp[i], sizes[i]);
    const auto gm = host_copy(dm[i], sizes[i]);
    const auto gv = host_copy(dv[i], sizes[i]);
    for (int k = 0; k < sizes[i]; ++k) {
      worst = fmax(worst, fabs(gp[k] - p[i][k]) / fmax(1.0, fabs(p[i][k])));
      worst = fmax(worst, fabs(gm[k] - m[i][k]) / fmax(1e-3, fabs(m[i][k])));
      worst = fmax(worst, fabs(gv[k] - v[i][k]) / fmax(1e-6, fabs(v[i][k])));
    }
  }
  const auto st = host_copy(dstep, 1);
  say("adam_step (4 tensors incl. an unaligned gradient view, 3 steps): worst rel err vs host update %.2e (tol 1e-5), "
      "device step counter %.0f -> %s", worst, st[0], (worst < 1e-5 && st[0] == 3.0f) ? "PASS" : "FAIL");
  return 0;
}

static int init_device_quiet();
// =====================================================================================================
// --bench: CUDA-event timings at config-2 sizes (seconds of GPU time; one child process per job)
// =====================================================================================================
static float time_ms(cudaEvent_t e0, cudaEvent_t e1) {
  float ms = 0;
  cudaEventSynchronize(e1);
  cudaEventElapsedTime(&ms, e0, e1);
  return ms;
}
static int bench_ln(int T, int C) {
  if (init_device_quiet()) return 1;
  float *x = nullptr, *y = nullptr, *g = nullptr, *b = nullptr, *st = nullptr;
  CK(cudaMalloc(&x, static_cast<size_t>(T) * C * 4));
  CK(cudaMalloc(&y, static_cast<size_t>(T) * C * 4));
  CK(cudaMalloc(&g, C * 4));
  CK(cudaMalloc(&b, C * 4));
  CK(cudaMalloc(&st, static_cast<size_t>(T) * 8));
  CK(cudaMemset(x, 0, static_cast<size_t>(T) * C * 4));
  CK(cudaMemset(g, 0, C * 4));
  CK(cudaMemset(b, 0, C * 4));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  for (int dt = 0; dt < 2; ++dt) {  // output bf16 (the in-block LayerNorms) and fp32
    for (int i = 0; i < 3; ++i) crf_layernorm_fwd(x, g, b, 1e-5f, y, dt == 0 ? CRF_DT_BF16 : CRF_DT_F32, st, T, C, 0, nullptr);
    cudaEventRecord(e0);
    const int it = 20;
    for (int i = 0; i < it; ++i) crf_layernorm_fwd(x, g, b, 1e-5f, y, dt == 0 ? CRF_DT_BF16 : CRF_DT_F32, st, T, C, 0, nullptr);
    cudaEventRecord(e1);
    const float ms = time_ms(e0, e1) / it;
    const double bytes = static_cast<double>(T) * C * (4 + (dt == 0 ? 2 : 4));
    say("bench layernorm_fwd T%d C%d out=%s: %.2f us, %.0f GB/s", T, C, dt == 0 ? "bf16" : "f32", ms * 1e3,
        bytes / ms / 1e6);
  }
  return 0;
}
static int bench_adam(long long n_total, int n_tensors) {
  if (init_device_quiet()) return 1;
  const long long n = n_total / n_tensors;
  std::vector<crf_adam_tensor> rec(n_tensors);
  for (int i = 0; i < n_tensors; ++i) {
    float* buf[4];
    for (auto& p : buf) {
      CK(cudaMalloc(&p, n * 4));
      CK(cudaMemset(p, 0, n * 4));
    }
    rec[i] = {buf[0], buf[1], buf[2], buf[3], n};
  }
  float* step = nullptr;
  CK(cudaMalloc(&step, 4));
  CK(cudaMemset(step, 0, 4));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  for (int i = 0; i < 2; ++i) crf_adam_step(rec.data(), n_tensors, 16384, 1e-4f, 0.9f, 0.999f, 1e-8f, 0.f, step, 0, nullptr);
  cudaEventRecord(e0);
  const int it = 10;
  for (int i = 0; i < it; ++i) crf_adam_step(rec.data(), n_tensors, 16384, 1e-4f, 0.9f, 0.999f, 1e-8f, 0.f, step, 0, nullptr);
  cudaEventRecord(e1);
  const float ms = time_ms(e0, e1) / it;
  say("bench adam_step %lld parameters in %d tensors: %.1f us, %.0f GB/s (28 B per parameter)", n * n_tensors, n_tensors,
      ms * 1e3, 28.0 * n * n_tensors / ms / 1e6);
  return 0;
}
static int bench_attn(const AttnCase& c) {
  if (init_device_quiet()) return 1;
  const int C = c.C, T = c.B * c.H * c.W;
  crf::WindowGeom gm(c.H, c.W, 7, c.shift);
  const int nWin = c.B * gm.nW;
  crf_block_desc d;
  memset(&d, 0, sizeof(d));
  d.B = c.B; d.H = c.H; d.W = c.W; d.C = C; d.num_heads = c.nH; d.window = 7; d.shift = c.shift; d.training = 1;
  d.x_dtype = CRF_DT_F32; d.v_dtype = CRF_DT_BF16; d.v_preconverted = 1;
  d.x_stride_b = static_cast<int64_t>(c.H) * c.W * C; d.x_stride_t = C; d.x_stride_c = 1;
  d.v_stride_b = d.x_stride_b; d.v_stride_h = static_cast<int64_t>(c.W) * C; d.v_stride_w = C; d.v_stride_c = 1;
  uint16_t *qk, *vb, *o, *dout, *dqk;
  float *bias, *table, *lse, *dv, *dt, *db;
  CK(cudaMalloc(&qk, static_cast<size_t>(T) * 2 * C * 2)); CK(cudaMemset(qk, 0, static_cast<size_t>(T) * 2 * C * 2));
  CK(cudaMalloc(&vb, static_cast<size_t>(T) * C * 2));     CK(cudaMemset(vb, 0, static_cast<size_t>(T) * C * 2));
  CK(cudaMalloc(&o, static_cast<size_t>(T) * C * 2));
  CK(cudaMalloc(&dout, static_cast<size_t>(T) * C * 2));   CK(cudaMemset(dout, 0, static_cast<size_t>(T) * C * 2));
  CK(cudaMalloc(&dqk, static_cast<size_t>(T) * 2 * C * 2));
  CK(cudaMalloc(&bias, 2 * C * 4));                         CK(cudaMemset(bias, 0, 2 * C * 4));
  CK(cudaMalloc(&table, 169 * c.nH * 4));                   CK(cudaMemset(table, 0, 169 * c.nH * 4));
  CK(cudaMalloc(&lse, static_cast<size_t>(nWin) * c.nH * 64 * 4));
  CK(cudaMalloc(&dv, static_cast<size_t>(T) * C * 4));
  CK(cudaMalloc(&dt, 169 * c.nH * 4));                      CK(cudaMemset(dt, 0, 169 * c.nH * 4));
  CK(cudaMalloc(&db, 2 * C * 4));                           CK(cudaMemset(db, 0, 2 * C * 4));
  const float scale = 1.0f / sqrtf(static_cast<float>(C / c.nH));
  cudaEvent_t e0, e1, e2;
  cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
  for (int i = 0; i < 2; ++i) {
    if (crf_attn_fwd(&d, qk, vb, bias, scale, table, nullptr, 0, o, lse, nullptr)) { say("bench attn: %s", crf_last_error()); return 1; }
    crf_attn_bwd(&d, qk, vb, bias, scale, table, nullptr, 0, lse, dout, dqk, dv, 0, dt, db, nullptr);
  }
  const int it = 5;
  cudaEventRecord(e0);
  for (int i = 0; i < it; ++i) crf_attn_fwd(&d, qk, vb, bias, scale, table, nullptr, 0, o, lse, nullptr);
  cudaEventRecord(e1);
  for (int i = 0; i < it; ++i) crf_attn_bwd(&d, qk, vb, bias, scale, table, nullptr, 0, lse, dout, dqk, dv, 0, dt, db, nullptr);
  cudaEventRecord(e2);
  const float f = time_ms(e0, e1) / it, b = time_ms(e1, e2) / it;
  const double tc = static_cast<double>(T) * C;
  say("bench attn B%d %dx%d C%d heads %d (head_dim %d) shift %d: fwd %.1f us (%.0f GB/s algorithmic), bwd %.1f us (%.0f GB/s)",
      c.B, c.H, c.W, C, c.nH, C / c.nH, c.shift, f * 1e3, 8.0 * tc / f / 1e6, b * 1e3, 16.0 * tc / b / 1e6);
  return 0;
}

static int init_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    say("no CUDA device");
    return 1;
  }
  cudaSetDevice(0);
  cudaFree(0);
  return 0;
}

static int init_device_quiet() { return init_device(); }

static const AttnCase kCases[] = {
    {2, 9, 10, 64, 2, 3},     // head_dim 32: the verified kernels -- validates this harness
    {2, 9, 10, 64, 1, 3},     // head_dim 64, padded + shifted
    {1, 14, 14, 128, 2, 0},   // head_dim 64, two heads, no padding, unshifted
    {1, 15, 20, 128, 1, 3},   // head_dim 128, padded + shifted
    {3, 16, 23, 256, 2, 3},   // head_dim 128, two heads, several CTAs per head
};
static const char* kTags[] = {"attn_hd32_verified", "attn_hd64_9x10_s3", "attn_hd64x2_14x14_s0", "attn_hd128_15x20_s3",
                              "attn_hd128x2_16x23_s3"};

// One group per child process: a device-side fault of an unverified kernel kills only its own CUDA context.
static int run_group(int grp) {
  if (init_device()) return 1;
  if (grp == 0) {
    cudaDeviceProp pr;
    cudaGetDeviceProperties(&pr, 0);
    say("device: %s, sm_%d%d, %d SMs; crf_abi_version %d", pr.name, pr.major, pr.minor, pr.multiProcessorCount, crf_abi_version());
  }
  int bad = 0;
  if (grp == 0 || grp == 1) {
    const int lo = grp == 0 ? 0 : 3, hi = grp == 0 ? 3 : 5;
    for (int i = lo; i < hi; ++i) {
      const int rc = run_attn_case(kCases[i], kTags[i], "");
      if (rc == 2) {
        say("group %d stops: its CUDA context is unusable after a kernel fault", grp);
        return 3;
      }
      bad += rc != 0;
    }
  } else if (grp == 2) {
    bad += run_ln_case(777, 128) != 0;
    bad += run_ln_case(331, 256) != 0;
  } else {
    bad += run_adam() != 0;
  }
  return bad;
}

#include <sys/wait.h>
#include <unistd.h>

int main(int argc, char** argv) {
  g_t0 = now_s();
  if (argc >= 3 && strcmp(argv[1], "--dry") == 0) {
    for (int i = 0; i < 5; ++i) run_attn_case(kCases[i], kTags[i], argv[2]);
    return 0;
  }
  if (system("mkdir -p gpurun_out") != 0) return 1;
  g_log = fopen("gpurun_out/hwcheck.txt", "a");
  if (argc >= 3 && strcmp(argv[1], "--group") == 0) return run_group(atoi(argv[2]));
  if (argc >= 2 && strcmp(argv[1], "--bench") == 0) {
    // config-2 sizes; every job in its own child, one after the other
    struct Job { int kind; AttnCase c; };
    const Job jobs[] = {
        {0, {}},                                              // LayerNorm forward, 1/4 and 1/8 scale
        {1, {}},                                              // Adam over 45 M parameters
        {2, {8, 120, 160, 128, 4, 3}},                        // attention, head_dim 32 (tuned kernels)
        {2, {8, 120, 160, 128, 2, 3}}, {2, {8, 120, 160, 128, 1, 3}},   // head_dim 64, 128 at the 1/4 scale
        {2, {8, 30, 40, 512, 8, 3}}, {2, {8, 30, 40, 512, 4, 3}},       // head_dim 64, 128 at the 1/16 scale
    };
    for (const Job& j : jobs) {
      const pid_t pid = fork();
      if (pid == 0) {
        int rc = 0;
        if (j.kind == 0) rc = bench_ln(153600, 128) | bench_ln(38400, 256);
        else if (j.kind == 1) rc = bench_adam(45000000LL, 300);
        else rc = bench_attn(j.c);
        _exit(rc);
      }
      int st = 0;
      waitpid(pid, &st, 0);
    }
    say("hwcheck --bench finished");
    return 0;
  }
  // all groups at once, each in its own process (no CUDA call has been made in the parent)
  pid_t pids[4];
  for (int grp = 0; grp < 4; ++grp) {
    pids[grp] = fork();
    if (pids[grp] == 0) _exit(run_group(grp));
  }
  for (int grp = 0; grp < 4; ++grp) {
    int st = 0;
    waitpid(pids[grp], &st, 0);
    say("group %d (%s): exit %d%s", grp, grp == 0 ? "hd32 + hd64" : grp == 1 ? "hd128" : grp == 2 ? "layernorm" : "adam",
        WIFEXITED(st) ? WEXITSTATUS(st) : -1, WIFSIGNALED(st) ? " (killed by a signal)" : "");
  }
  say("hwcheck finished (PASS / FAIL per line above)");
  return 0;
}
