// Group / instance normalisation of a spectral convolution's output, applied to its kept-mode spectrum
// (fno_block.py:94-105,142-150: Norm(SpectralConv(x) + bias) before the skip is added).
//
// The conv output s = s_i Re IDFT_trunc(c Yh) + bias is band-limited, so its mean and variance over the output grid are
// exact quadratic forms of the kept modes (DESIGN.md section 4, "Normalisation in the spectrum").  With the per-mode table
// of the plan (plan.cu: the kept mirror of mode k, -1 when there is none or c(k_d) = 2, and c(k_d)):
//   S_k  = 1/2 s_i c(k_d) (Yh_k + conj(Yh_mirror(k)))        the coefficient of frequency k on the full grid
//   mean = bias + s_i Re Yh_0,   var = sum_{k != 0} w_k |S_k|^2,   w_k = 1 when the mirror is kept, else 2
//   d var / d Yh_k = 2 s_i c(k_d) S_k                          (PyTorch's complex-gradient convention)
// Normalising s is then a real per-(sample, channel) scale of every non-DC mode plus a new real DC value; the inverse
// transform's fused epilogue runs unchanged on the result, without the bias.
//
// One warp per (sample, channel) spectrum row.  A group's statistics need every row of the group, so each direction is a
// per-row pass followed by a pass that combines the group (a few floats per row, from L2) and writes the rows:
//   forward : k_spec_norm_stats (mu_c, var_c) -> k_spec_norm_fwd (group mean / rstd, Yh')
//   backward: k_spec_norm_dots (P_c, q_c)     -> k_spec_norm_bwd (gYh, per-row parameter terms) -> k_spec_norm_reduce
// The parameter gradients are summed over the batch in a fixed order by k_spec_norm_reduce (no float atomics).
#include "common.cuh"

namespace {

constexpr int kWarps = 8;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// S_k of the header comment (k != 0); c = 0 rows give 0
__device__ __forceinline__ float2 coef_S(const float2* __restrict__ y, int2 t, int k, float half_si) {
  float2 a = y[k];
  if (t.x >= 0) {
    const float2 m = y[t.x];
    a.x += m.x;
    a.y -= m.y;
  }
  const float f = half_si * (float)t.y;
  return make_float2(f * a.x, f * a.y);
}

__global__ void __launch_bounds__(kWarps * 32)
k_spec_norm_stats(const float2* __restrict__ spec, const int2* __restrict__ tab, const float* __restrict__ bias,
                  float* __restrict__ stats, int rows, int C, int K, float s_i) {
  const int row = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float2* y = spec + (size_t)row * K;
  const float half_si = 0.5f * s_i;
  float v = 0.f;
  for (int k = 1 + lane; k < K; k += 32) {
    const int2 t = __ldg(tab + k);
    if (t.y == 0) continue;
    const float2 S = coef_S(y, t, k, half_si);
    v += (t.x >= 0 ? 1.f : 2.f) * (S.x * S.x + S.y * S.y);
  }
  v = warp_sum(v);
  if (lane == 0) {
    stats[2 * row] = s_i * y[0].x + (bias ? __ldg(bias + row % C) : 0.f);
    stats[2 * row + 1] = v;
  }
}

// group mean and variance of the rows [c0, c0 + cg) of sample b, from their (mu_c, var_c): every lane gets both
__device__ __forceinline__ void group_moments(const float* __restrict__ st, int cg, int lane, float* mu_g, float* var_g) {
  float s = 0.f;
  for (int i = lane; i < cg; i += 32) s += st[2 * i];
  const float mu = warp_sum(s) / (float)cg;
  float v = 0.f;
  for (int i = lane; i < cg; i += 32) {
    const float d = st[2 * i] - mu;
    v += st[2 * i + 1] + d * d;
  }
  *mu_g = mu;
  *var_g = warp_sum(v) / (float)cg;
}

// stats = [ (mu_c, var_c) per row | (mu_g, rstd_g) per (sample, group) ]
__global__ void __launch_bounds__(kWarps * 32)
k_spec_norm_fwd(const float2* __restrict__ spec, const float* __restrict__ gamma, const float* __restrict__ beta,
                float* __restrict__ stats, float2* __restrict__ out, int rows, int C, int G, int K, float s_i, float eps) {
  const int row = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int b = row / C, c = row % C, cg = C / G, g = c / cg, c0 = g * cg;
  float mu_g, var_g;
  group_moments(stats + 2 * ((size_t)b * C + c0), cg, lane, &mu_g, &var_g);
  const float r = 1.0f / sqrtf(var_g + eps);
  const float gam = gamma ? __ldg(gamma + c) : 1.f, bet = beta ? __ldg(beta + c) : 0.f;
  const float a = gam * r;
  const float2* y = spec + (size_t)row * K;
  float2* o = out + (size_t)row * K;
  for (int k = 1 + lane; k < K; k += 32) {
    const float2 v = y[k];
    o[k] = make_float2(a * v.x, a * v.y);
  }
  if (lane == 0) {
    const float mu_c = stats[2 * row];
    o[0] = make_float2((gam * (mu_c - mu_g) * r + bet) / s_i, 0.f);
    if (c == c0) {
      float* gs = stats + 2 * (size_t)rows + 2 * ((size_t)b * G + g);
      gs[0] = mu_g;
      gs[1] = r;
    }
  }
}

// dots[row] = (P_c, q_c): P_c = sum_{k != 0} Re(conj(G_k) Yh_k) = dL / d(scale), q_c = Re G_0 / s_i = dL / d(output mean)
__global__ void __launch_bounds__(kWarps * 32)
k_spec_norm_dots(const float2* __restrict__ spec, const float2* __restrict__ gspec, float* __restrict__ dots, int rows,
                 int K, float s_i) {
  const int row = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float2* y = spec + (size_t)row * K;
  const float2* gy = gspec + (size_t)row * K;
  float p = 0.f;
  for (int k = 1 + lane; k < K; k += 32) {
    const float2 a = y[k], g = gy[k];
    p = fmaf(g.x, a.x, fmaf(g.y, a.y, p));
  }
  p = warp_sum(p);
  if (lane == 0) {
    dots[2 * row] = p;
    dots[2 * row + 1] = gy[0].x / s_i;
  }
}

// With r = rstd_g, cg = channels per group and, over the channels of the group,
//   A = sum_c gamma_c (P_c + q_c (mu_c - mu_g)) = dL / dr,   Q = sum_c gamma_c q_c
//   dL/dvar_g = -1/2 r^3 A;  dL/dmu_c = gamma_c r q_c - r Q / cg + dL/dvar_g 2 (mu_c - mu_g) / cg;  dL/dvar_c = dL/dvar_g / cg
//   gYh_k = gamma_c r G_k + dL/dvar_c 2 s_i c(k_d) S_k  (k != 0),   gYh_0 = s_i dL/dmu_c
// part[row] = (dgamma, dbeta, dbias) terms of this row: (r (P_c + q_c (mu_c - mu_g)), q_c, dL/dmu_c)
__global__ void __launch_bounds__(kWarps * 32)
k_spec_norm_bwd(const float2* __restrict__ spec, const float2* __restrict__ gspec, const int2* __restrict__ tab,
                const float* __restrict__ stats, const float* __restrict__ gamma, const float* __restrict__ dots,
                float2* __restrict__ gout, float* __restrict__ part, int rows, int C, int G, int K, float s_i) {
  const int row = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int b = row / C, c = row % C, cg = C / G, g = c / cg, c0 = g * cg;
  const float* gs = stats + 2 * (size_t)rows + 2 * ((size_t)b * G + g);
  const float mu_g = gs[0], r = gs[1];
  const size_t base = (size_t)b * C + c0;
  float A = 0.f, Q = 0.f;
  for (int i = lane; i < cg; i += 32) {
    const float gi = gamma ? __ldg(gamma + c0 + i) : 1.f;
    const float q = dots[2 * (base + i) + 1];
    A += gi * (dots[2 * (base + i)] + q * (stats[2 * (base + i)] - mu_g));
    Q = __fadd_rn(Q, __fmul_rn(gi, q));
  }
  A = warp_sum(A);
  Q = warp_sum(Q);
  const float inv_cg = 1.0f / (float)cg;
  const float dvar_g = -0.5f * r * r * r * A;
  const float gam = gamma ? __ldg(gamma + c) : 1.f;
  const float P = dots[2 * row], q = dots[2 * row + 1], dmu = stats[2 * row] - mu_g;
  // with one channel per group (instance norm) Q = gamma_c q_c and dmu = 0: the explicitly rounded products (no FMA
  // contraction) make dmu_c exactly 0, as the conv bias cancels in the instance statistics
  const float dmu_c = r * (__fmul_rn(gam, q) - __fmul_rn(Q, inv_cg)) + 2.f * dvar_g * dmu * inv_cg;
  const float a = gam * r, e = dvar_g * inv_cg * 2.f * s_i, half_si = 0.5f * s_i;
  const float2* y = spec + (size_t)row * K;
  const float2* gy = gspec + (size_t)row * K;
  float2* o = gout + (size_t)row * K;
  for (int k = 1 + lane; k < K; k += 32) {
    const int2 t = __ldg(tab + k);
    const float2 G_ = gy[k];
    float2 v = make_float2(a * G_.x, a * G_.y);
    if (t.y != 0) {
      const float2 S = coef_S(y, t, k, half_si);
      const float f = e * (float)t.y;
      v.x = fmaf(f, S.x, v.x);
      v.y = fmaf(f, S.y, v.y);
    }
    o[k] = v;
  }
  if (lane == 0) {
    o[0] = make_float2(s_i * dmu_c, 0.f);
    part[3 * row] = r * (P + q * dmu);
    part[3 * row + 1] = q;
    part[3 * row + 2] = dmu_c;
  }
}

// d{gamma, beta, bias}[c] = sum over the batch, in order, of the per-row terms
__global__ void __launch_bounds__(256)
k_spec_norm_reduce(const float* __restrict__ part, float* __restrict__ dgamma, float* __restrict__ dbeta,
                   float* __restrict__ dbias, int B, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float sg = 0.f, sb = 0.f, sd = 0.f;
  for (int b = 0; b < B; b++) {
    const float* p = part + 3 * ((size_t)b * C + c);
    sg += p[0];
    sb += p[1];
    sd += p[2];
  }
  if (dgamma) dgamma[c] = sg;
  if (dbeta) dbeta[c] = sb;
  if (dbias) dbias[c] = sd;
}

float inverse_scale(const b2no_plan* p) {
  double n = 1.0;
  for (int j = 0; j < p->g.ndim; j++) n *= p->g.nout[j];
  if (p->g.norm == B2NO_NORM_FORWARD) return 1.0f;
  if (p->g.norm == B2NO_NORM_BACKWARD) return (float)(1.0 / n);
  return (float)(1.0 / sqrt(n));
}

int check_shape(const b2no_plan* p, int batch, int channels, int groups) {
  if (!p || batch < 1 || channels < 1 || groups < 1 || channels % groups != 0) return B2NO_E_ARG;
  if (p->g.spec_layout != 0) return B2NO_E_UNSUPPORTED;
  for (int j = 0; j < p->g.ndim; j++)
    if (p->g.nout[j] != p->g.nfft[j]) return B2NO_E_UNSUPPORTED;
  if ((long)batch * channels > 0x7fffffffL / 2) return B2NO_E_UNSUPPORTED;
  return 0;
}

}  // namespace

extern "C" int b2no_spec_norm_fwd(const b2no_plan* plan, const float* spec, const float* bias, const float* gamma,
                                  const float* beta, float eps, float* out, float* stats, int batch, int channels, int groups,
                                  void* stream) {
  int rc = check_shape(plan, batch, channels, groups);
  if (rc) return rc;
  if (!spec || !out || !stats || (gamma == nullptr) != (beta == nullptr) || !(eps > 0.f)) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = batch * channels, K = total_modes(plan), grid = b2no_ceil_div(rows, kWarps);
  const float s_i = inverse_scale(plan);
  k_spec_norm_stats<<<grid, kWarps * 32, 0, st>>>((const float2*)spec, plan->norm_tab, bias, stats, rows, channels, K, s_i);
  B2NO_LAUNCH_CHECK();
  k_spec_norm_fwd<<<grid, kWarps * 32, 0, st>>>((const float2*)spec, gamma, beta, stats, (float2*)out, rows, channels, groups,
                                                K, s_i, eps);
  B2NO_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t b2no_spec_norm_bwd_scratch_floats(int batch, int channels) {
  if (batch < 1 || channels < 1) return B2NO_E_ARG;
  return (int64_t)5 * batch * channels;
}

extern "C" int b2no_spec_norm_bwd(const b2no_plan* plan, const float* spec, const float* gspec, const float* stats,
                                  const float* gamma, float* gout, float* dbias, float* dgamma, float* dbeta, float* scratch,
                                  int batch, int channels, int groups, void* stream) {
  int rc = check_shape(plan, batch, channels, groups);
  if (rc) return rc;
  if (!spec || !gspec || !stats || !gout || !scratch || (gamma == nullptr && (dgamma || dbeta))) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = batch * channels, K = total_modes(plan), grid = b2no_ceil_div(rows, kWarps);
  const float s_i = inverse_scale(plan);
  float* dots = scratch;
  float* part = scratch + 2 * (size_t)rows;
  k_spec_norm_dots<<<grid, kWarps * 32, 0, st>>>((const float2*)spec, (const float2*)gspec, dots, rows, K, s_i);
  B2NO_LAUNCH_CHECK();
  k_spec_norm_bwd<<<grid, kWarps * 32, 0, st>>>((const float2*)spec, (const float2*)gspec, plan->norm_tab, stats, gamma, dots,
                                                (float2*)gout, part, rows, channels, groups, K, s_i);
  B2NO_LAUNCH_CHECK();
  if (dbias || dgamma || dbeta) {
    k_spec_norm_reduce<<<b2no_ceil_div(channels, 256), 256, 0, st>>>(part, dgamma, dbeta, dbias, batch, channels);
    B2NO_LAUNCH_CHECK();
  }
  return 0;
}
