// Plan = per-geometry twiddle tables (computed on the host in fp64, rounded once to fp32) and the
// kept-row -> (corner, local index) maps.  Mirrors oracle/closed_form.py::SpecGeom one to one.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "common.cuh"

static int g_sm_count[64];
long long g_b2no_launches = 0;
extern "C" int64_t b2no_kernel_launches(void) { return (int64_t)g_b2no_launches; }

int b2no_sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (g_sm_count[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_sm_count[dev] = n;
  }
  return g_sm_count[dev];
}

extern "C" int b2no_version(void) { return B2NO_ABI_VERSION; }

extern "C" const char* b2no_error_string(int code) {
  if (code == 0) return "ok";
  if (code == B2NO_E_ARG) return "b2no: bad argument";
  if (code == B2NO_E_UNSUPPORTED) return "b2no: unsupported shape or option";
  if (code == B2NO_E_NODEVICE) return "b2no: no CUDA device";
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "b2no: unknown error";
}

extern "C" int b2no_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes) {
  int dev = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  B2NO_CHECK_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (l2_bytes) *l2_bytes = (int64_t)p.l2CacheSize;
  return 0;
}

namespace {

struct Row { int f, corner, local; };

// kept rows of a two-sided dim: [0,h) U [N-h,N); on overlap (2h > N) the high corner wins
// (assignment order spectral_convolution.py:412-416, rno.py:71-74, basics.py:127-139).
std::vector<Row> kept_rows(int N, int h, bool last) {
  std::vector<Row> r;
  if (last) {
    for (int k = 0; k < h; k++) r.push_back({k, 0, k});
    return r;
  }
  for (int f = 0; f < N; f++) {
    bool lo = f < h, hi = f >= N - h;
    if (hi) r.push_back({f, 1, f - (N - h)});
    else if (lo) r.push_back({f, 0, f});
  }
  return r;
}

inline void unit(long num, long den, double* c, double* s) {
  // exp(2 pi i num/den) with exact integer argument reduction
  long m = ((num % den) + den) % den;
  double a = 2.0 * M_PI * (double)m / (double)den;
  *c = cos(a);
  *s = sin(a);
}

template <typename T>
int upload(T** dst, const std::vector<T>& v) {
  size_t bytes = v.size() * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  B2NO_CHECK_CUDA(cudaMalloc((void**)dst, bytes));
  if (!v.empty()) B2NO_CHECK_CUDA(cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return 0;
}

// round-to-nearest (ties away) fp32 -> tf32, like cvt.rna.tf32.f32
float tf32_round_host(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return x;
  u += 0x1000u;
  u &= 0xFFFFE000u;
  memcpy(&x, &u, 4);
  return x;
}

void choose_chunks(int q2, int* qc, int* nchunk) {
  if (q2 <= 4) { *qc = 4; *nchunk = 1; return; }
  if (q2 <= 8) { *qc = 8; *nchunk = 1; return; }
  if (q2 <= 12) { *qc = 12; *nchunk = 1; return; }
  // chunks of 8 or 12 table rows: k_r2c_last keeps 8 * QC accumulators per thread, and the QC = 16 instantiation
  // spilled all 128 of them to local memory (ptxas: 512 B stack) -- 1.2 ms for the 306 MB last-dim pass of the PINO layer
  int n8 = (q2 + 7) / 8, n12 = (q2 + 11) / 12;
  if (n12 * 12 <= n8 * 8) { *qc = 12; *nchunk = n12; }
  else { *qc = 8; *nchunk = n8; }
}

}  // namespace

extern "C" int b2no_plan_create(const b2no_geom* g, b2no_plan** out) {
  if (!g || !out) return B2NO_E_ARG;
  if (g->ndim < 1 || g->ndim > B2NO_MAX_DIM) return B2NO_E_UNSUPPORTED;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return B2NO_E_NODEVICE;
  const int d = g->ndim;
  for (int j = 0; j < d; j++) {
    if (g->nin[j] < 1 || g->nfft[j] < 1 || g->nout[j] < 1 || g->half[j] < 1) return B2NO_E_ARG;
    if (j < d - 1 && g->half[j] > g->nfft[j]) return B2NO_E_ARG;
  }
  if (g->norm < 0 || g->norm > 2) return B2NO_E_ARG;
  if (g->spec_layout != 0 && g->spec_layout != 1) return B2NO_E_ARG;
  if (g->spec_layout == 1 && d != 2) return B2NO_E_UNSUPPORTED;

  b2no_plan* p = (b2no_plan*)calloc(1, sizeof(b2no_plan));
  if (!p) return B2NO_E_ARG;
  p->g = *g;
  B2NO_CHECK_CUDA(cudaGetDevice(&p->device));

  double nprod = 1.0, noutprod = 1.0;
  for (int j = 0; j < d; j++) { nprod *= g->nfft[j]; noutprod *= g->nout[j]; }
  double sf = 1.0, si = 1.0;
  if (g->norm == B2NO_NORM_FORWARD) { sf = 1.0 / nprod; si = 1.0; }
  else if (g->norm == B2NO_NORM_BACKWARD) { sf = 1.0; si = 1.0 / noutprod; }
  else { sf = 1.0 / sqrt(nprod); si = 1.0 / sqrt(noutprod); }

  // ---- last dim (real tables) ---------------------------------------------------------------
  {
    const int j = d - 1;
    const int N = g->nfft[j], Np = g->nout[j], nin = g->nin[j];
    std::vector<Row> rows = kept_rows(N, g->half[j], true);
    const int K = (int)rows.size();
    p->K[j] = K;
    p->q2 = 2 * K;
    choose_chunks(p->q2, &p->qc, &p->nchunk);
    p->qpad = p->qc * p->nchunk;
    p->npad_in = b2no_round_up(nin, 128);
    p->npad_out = b2no_round_up(Np, 128);
    std::vector<float> tin((size_t)p->qpad * p->npad_in, 0.f), tout((size_t)p->qpad * p->npad_out, 0.f);
    for (int k = 0; k < K; k++) {
      const int f = rows[k].f;
      // T_in: s_f * exp(-2 pi i f n / N), n < min(nin, N); modes beyond the rfft length read as zero
      if (f < N / 2 + 1) {
        for (int n = 0; n < nin && n < N; n++) {
          double c, s;
          unit((long)f * n, N, &c, &s);
          tin[(size_t)(2 * k) * p->npad_in + n] = (float)(sf * c);
          tin[(size_t)(2 * k + 1) * p->npad_in + n] = (float)(-sf * s);
        }
      }
      // T_out: s_i * c(k) * exp(+2 pi i f n / N') as (cos, -sin) rows
      double ck = 2.0;
      if (f == 0) ck = 1.0;
      if (Np % 2 == 0 && f == Np / 2) ck = 1.0;
      if (f >= Np / 2 + 1) ck = 0.0;
      if (f >= N / 2 + 1) ck = 0.0;
      for (int n = 0; n < Np; n++) {
        double c, s;
        unit((long)f * n, Np, &c, &s);
        tout[(size_t)(2 * k) * p->npad_out + n] = (float)(si * ck * c);
        tout[(size_t)(2 * k + 1) * p->npad_out + n] = (float)(-si * ck * s);
      }
    }
    int rc;
    if ((rc = upload(&p->t_in, tin))) return rc;
    if ((rc = upload(&p->t_out, tout))) return rc;
    // tensor-core operand images (2-D and up, last dim dividing the 128-pixel tile)
    for (int which = 0; which < 2; which++) {
      const int Wd = which == 0 ? Np : nin;
      const std::vector<float>& tab = which == 0 ? tout : tin;
      const int npad = which == 0 ? p->npad_out : p->npad_in;
      b2no_tc_tables& tt = p->tc[which];
      tt.timg = nullptr;
      if (d < 2 || Wd > 128 || 128 % Wd != 0) continue;
      tt.R = 128 / Wd;
      tt.Qp = b2no_round_up(2 * K, 8);
      tt.Ks = tt.R * tt.Qp;
      if (tt.Ks > 128) continue;
      std::vector<float> img((size_t)2 * 128 * tt.Ks, 0.f);
      for (int m = 0; m < 128; m++)
        for (int k = 0; k < tt.Ks; k++) {
          const int r = k / tt.Qp, q = k % tt.Qp;
          float v = 0.f;
          if (r == m / Wd && q < 2 * K) v = tab[(size_t)q * npad + (m % Wd)];
          const float hi = tf32_round_host(v);
          const size_t off = (size_t)m * tt.Ks + k;   // row-major: thread m of the converter loads row m into TMEM
          img[off] = hi;
          img[(size_t)128 * tt.Ks + off] = tf32_round_host(v - hi);
        }
      if ((rc = upload(&tt.timg, img))) return rc;
    }
  }

  // ---- middle dims (complex matrices) -------------------------------------------------------
  for (int j = 0; j < d - 1; j++) {
    const int N = g->nfft[j], Np = g->nout[j], nin = g->nin[j];
    std::vector<Row> rows = kept_rows(N, g->half[j], false);
    const int K = (int)rows.size();
    p->K[j] = K;
    std::vector<float2> mf((size_t)nin * K), mi((size_t)K * Np), mai((size_t)Np * K), maf((size_t)K * nin);
    std::vector<int> rcorner(K), rlocal(K);
    for (int k = 0; k < K; k++) {
      const int f = rows[k].f;
      rcorner[k] = rows[k].corner;
      rlocal[k] = rows[k].local;
      for (int n = 0; n < nin; n++) {
        double c = 0.0, s = 0.0;
        if (n < N) unit((long)f * n, N, &c, &s);
        else { c = 0.0; s = 0.0; }
        mf[(size_t)n * K + k] = make_float2((float)c, (float)(-s));     // exp(-i)
        maf[(size_t)k * nin + n] = make_float2((float)c, (float)(s));   // conj(m_fwd)^T = exp(+i)
      }
      for (int n = 0; n < Np; n++) {
        double c = 0.0, s = 0.0;
        if (f < Np) unit((long)f * n, Np, &c, &s);
        else { c = 0.0; s = 0.0; }
        mi[(size_t)k * Np + n] = make_float2((float)c, (float)(s));      // exp(+i)
        mai[(size_t)n * K + k] = make_float2((float)c, (float)(-s));     // conj(m_inv)^T
      }
    }
    int rc;
    if ((rc = upload(&p->m_fwd[j], mf))) return rc;
    if ((rc = upload(&p->m_inv[j], mi))) return rc;
    if ((rc = upload(&p->m_adjinv[j], mai))) return rc;
    if ((rc = upload(&p->m_adjfwd[j], maf))) return rc;
    if ((rc = upload(&p->row_corner[j], rcorner))) return rc;
    if ((rc = upload(&p->row_local[j], rlocal))) return rc;
  }
  // ---- per-mode table of the spectral normalisation (spec_norm.cu) ----------------------------
  {
    std::vector<Row> rows[B2NO_MAX_DIM];
    std::vector<int> pos[B2NO_MAX_DIM];     // frequency -> kept row, -1 when not kept (two-sided dims)
    for (int j = 0; j < d; j++) {
      rows[j] = kept_rows(g->nfft[j], g->half[j], j == d - 1);
      if (j == d - 1) continue;
      pos[j].assign(g->nfft[j], -1);
      for (int r = 0; r < (int)rows[j].size(); r++) pos[j][rows[j][r].f] = r;
    }
    int kt = 1;
    for (int j = 0; j < d; j++) kt *= p->K[j];
    std::vector<int2> tab(kt);
    const int N = g->nfft[d - 1], Np = g->nout[d - 1];
    for (int k = 0; k < kt; k++) {
      int idx[B2NO_MAX_DIM], rem = k;
      for (int j = d - 1; j >= 0; j--) { idx[j] = rem % p->K[j]; rem /= p->K[j]; }
      const int f = idx[d - 1];
      int c = 2;                                            // c(k_d) exactly as the last-dim table T_out above
      if (f == 0 || (Np % 2 == 0 && f == Np / 2)) c = 1;
      if (f >= Np / 2 + 1 || f >= N / 2 + 1) c = 0;
      int mirror = -1;
      if (c == 1) {
        mirror = 0;
        for (int j = 0; j < d - 1 && mirror >= 0; j++) {
          const int Nj = g->nfft[j], r = pos[j][(Nj - rows[j][idx[j]].f) % Nj];
          mirror = r < 0 ? -1 : mirror * p->K[j] + r;
        }
        if (mirror >= 0) mirror = mirror * p->K[d - 1] + f;
      }
      tab[k] = make_int2(mirror, c);
    }
    int rc;
    if ((rc = upload(&p->norm_tab, tab))) return rc;
  }
  // ---- tensor-core forward-DFT operand images (2-D; tc_dft.cu) --------------------------------
  for (int which = 0; which < 2; which++) {
    b2no_tc_fwd_tables& tf = p->tcf[which];
    tf.tb = nullptr; tf.mimg = nullptr;
    if (d != 2) continue;
    const int Wd = which == 0 ? g->nin[1] : g->nout[1];
    const int Hd = which == 0 ? g->nin[0] : g->nout[0];
    if (which == 0 && (g->nin[0] != g->nfft[0] || g->nin[1] != g->nfft[1])) continue;   // crop / zero-pad (rno.py:66-67)
    const int Kx = p->K[0], Ky = p->K[1];
    if (Hd < 8 || Hd > 128 || 128 % Hd != 0 || Wd % 32 != 0 || Wd > 256 || Kx > 32 || 2 * Ky > 32) continue;
    const int N1 = b2no_round_up(2 * Ky, 8);
    tf.W = Wd; tf.H = Hd; tf.N1 = N1; tf.Kx = Kx; tf.Ky = Ky;
    // stage 1: T[q][w] (q = 2 ky -> re, 2 ky + 1 -> im) = the last-dim real table of this direction
    std::vector<float> tab_host((size_t)p->qpad * (which == 0 ? p->npad_in : p->npad_out));
    B2NO_CHECK_CUDA(cudaMemcpy(tab_host.data(), which == 0 ? p->t_in : p->t_out, tab_host.size() * sizeof(float),
                               cudaMemcpyDeviceToHost));
    const int npad = which == 0 ? p->npad_in : p->npad_out;
    std::vector<float> tb((size_t)2 * N1 * Wd, 0.f);
    for (int q = 0; q < 2 * Ky; q++)
      for (int w = 0; w < Wd; w++) {
        const float v = tab_host[(size_t)q * npad + w];
        const float hi = tf32_round_host(v);
        // K-major, no swizzle: 8-row groups, 16-byte K chunks (tc.cuh::kmajor_off), in floats
        const size_t off = (size_t)(q >> 3) * (Wd >> 2) * 32 + (size_t)(w >> 2) * 32 + (q & 7) * 4 + (w & 3);
        tb[off] = hi;
        tb[(size_t)N1 * Wd + off] = tf32_round_host(v - hi);
      }
    // stage 2: M[h][kx] complex (exp(-i) for both directions: m_fwd / m_adjinv), scale already in stage 1
    std::vector<float2> m_host((size_t)Hd * Kx);
    B2NO_CHECK_CUDA(cudaMemcpy(m_host.data(), which == 0 ? p->m_fwd[0] : p->m_adjinv[0], m_host.size() * sizeof(float2),
                               cudaMemcpyDeviceToHost));
    std::vector<float> mi((size_t)2 * 128 * Hd, 0.f);
    for (int kx = 0; kx < Kx; kx++)
      for (int h = 0; h < Hd; h++) {
        const float2 m = m_host[(size_t)h * Kx + kx];
        const float rh = tf32_round_host(m.x), ih = tf32_round_host(m.y);
        mi[(size_t)kx * Hd + h] = rh;
        mi[(size_t)(32 + kx) * Hd + h] = ih;
        mi[(size_t)128 * Hd + (size_t)kx * Hd + h] = tf32_round_host(m.x - rh);
        mi[(size_t)128 * Hd + (size_t)(32 + kx) * Hd + h] = tf32_round_host(m.y - ih);
      }
    // compact staging image of the same table for one bulk copy: [hi | lo][Re rows 0..Kx-1, Im rows 0..Kx-1][H + 4]
    std::vector<float> ms((size_t)2 * 2 * Kx * (Hd + 4), 0.f);
    for (int pass = 0; pass < 2; pass++)
      for (int r = 0; r < 2 * Kx; r++)
        for (int h = 0; h < Hd; h++) {
          const int srow = r < Kx ? r : 32 + (r - Kx);
          ms[((size_t)pass * 2 * Kx + r) * (Hd + 4) + h] = mi[(size_t)pass * 128 * Hd + (size_t)srow * Hd + h];
        }
    int rc;
    if ((rc = upload(&tf.tb, tb))) return rc;
    if ((rc = upload(&tf.mimg, ms))) return rc;
  }
  *out = p;
  return 0;
}

extern "C" int b2no_plan_destroy(b2no_plan* p) {
  if (!p) return 0;
  cudaFree(p->t_in);
  cudaFree(p->t_out);
  cudaFree(p->tc[0].timg);
  cudaFree(p->tc[1].timg);
  cudaFree(p->norm_tab);
  for (int w = 0; w < 2; w++) { cudaFree(p->tcf[w].tb); cudaFree(p->tcf[w].mimg); }
  for (int j = 0; j < 2; j++) {
    cudaFree(p->m_fwd[j]); cudaFree(p->m_inv[j]); cudaFree(p->m_adjinv[j]); cudaFree(p->m_adjfwd[j]);
    cudaFree(p->row_corner[j]); cudaFree(p->row_local[j]);
  }
  free(p);
  return 0;
}

extern "C" int b2no_plan_kept(const b2no_plan* p, int32_t kept[B2NO_MAX_DIM]) {
  if (!p || !kept) return B2NO_E_ARG;
  for (int j = 0; j < B2NO_MAX_DIM; j++) kept[j] = j < p->g.ndim ? p->K[j] : 1;
  return 0;
}

extern "C" int64_t b2no_plan_workspace_floats(const b2no_plan* p, int64_t batch, int64_t channels) {
  if (!p || batch < 0 || channels < 0) return B2NO_E_ARG;
  const int64_t bc = batch * channels;
  const int d = p->g.ndim;
  if (d == 1) return 0;
  // stage buffers (complex): A = [bc * n_0..n_{d-2}][K_last];  B (3-D only) = [bc * n_0][K_1][K_2]
  int64_t best = 0;
  for (int which = 0; which < 2; which++) {
    const int32_t* n = which == 0 ? p->g.nin : p->g.nout;
    int64_t a = bc, b = 0;
    for (int j = 0; j < d - 1; j++) a *= n[j];
    a *= p->K[d - 1];
    if (d == 3) b = bc * n[0] * p->K[1] * p->K[2];
    int64_t tot = 2 * (a + b);
    if (d == 3) {
      tot += bc * n[0] * n[1] * n[2];       // T: the transform's result handed to the pointwise tile kernel (split path)
      // row image of the fused path: [batch][n0 * n1 rows][Qp][Np] + the rows the last tiles read past the end
      const int64_t qp = (2 * p->K[2] + 7) / 8 * 8, np = (channels + 15) / 16 * 16, r = 127 / n[2] + 3;
      tot += (batch * n[0] * n[1] + r) * qp * np;
    }
    if (tot > best) best = tot;
    // tensor-core path: A' rows (hi + lo), [batch][rows][Qp][channels rounded up to 16]
    if (d == 2 && p->tc[which].timg) {
      const int64_t np = (channels + 15) / 16 * 16;
      const int64_t t = 2 * batch * n[0] * p->tc[which].Qp * np;
      if (t > best) best = t;
    }
  }
  return best;
}
