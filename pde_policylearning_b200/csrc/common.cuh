// Shared helpers for the b2no kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/b2no.h"

#define B2NO_CHECK_CUDA(expr)                      \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

// every kernel launch of the library is followed by this check; it also counts the launch (b2no_kernel_launches)
extern long long g_b2no_launches;
#define B2NO_LAUNCH_CHECK()                        \
  do {                                             \
    cudaError_t _e = cudaGetLastError();           \
    if (_e != cudaSuccess) return (int)_e;         \
    g_b2no_launches++;                             \
  } while (0)

static inline int b2no_ceil_div(long a, long b) { return (int)((a + b - 1) / b); }
static inline int b2no_round_up(int a, int b) { return ((a + b - 1) / b) * b; }

int b2no_sm_count();   // cached, current device
// tensor-core products per fp32 product: 3 = 3xTF32 (hi*hi + lo*hi + hi*lo, fp32 parity <= 1e-5), 1 = single-pass TF32
// (hi*hi only: the reduced-precision tensor-core mode, tolerance 2e-2 class)  -- b2no_set_precision()
int b2no_tc_passes();
bool b2no_tc_available();
int b2no_tc_mlp_fwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* out, int batch,
                    int ci, int hidden, int co2, long pixels, int b1_per_sample, int act, cudaStream_t st);
int b2no_tc_wgrad(const float* g, const float* x, float* partial, int max_blocks, int batch, int ci, int co, long pixels,
                  int* nblk, cudaStream_t st);
// weight-gradient variant of the 2-D dx pass (b2no_dft_inverse_wgrad): dW[o, i] = sum pw_x[b, o, p] x[b, i, p] and
// db[o] = sum pw_x[b, o, p] into per-CTA partials [Co*Ci | Co] (*nblk of them, summed by k_pw_wgrad_reduce)
struct b2no_tc_wg {
  const float* x;
  int ci;
  float* partial;
  int* nblk;
};
int b2no_tc_pointwise(const b2no_plan* plan, int which, const float* spec, float* y, float* work, int batch, int channels,
                      long pixels, const b2no_epilogue* e, cudaStream_t st, const b2no_tc_wg* wg = nullptr);

// operand images for the tensor-core tile kernel (tc_pointwise.cu): the last-dim inverse table as a
// block-diagonal row-major [128 x Ks] matrix, hi then lo (3xTF32); it becomes a TMEM-resident A operand
struct b2no_tc_tables {
  float* timg;     // 2 * 128 * Ks floats, or nullptr when the geometry is not eligible
  int Ks, Qp, R;   // Ks = R * Qp, R = rows per 128-pixel tile, Qp = 2*K_last rounded up to 8
};

// operand images for the tensor-core forward-DFT kernel (tc_dft.cu), one per direction
struct b2no_tc_fwd_tables {
  float* tb;     // stage-1 B operand: [2 (hi, lo)][N1 x W] floats in the K-major core-matrix order, or nullptr (not eligible)
  float* mimg;   // stage-2 A operand, compact staging image: [2 (hi, lo)][2 Kx rows: Re M[., kx] then Im M[., kx]][H + 4]
  int W, H, N1, Kx, Ky;
};
int b2no_tc_dft_forward(const b2no_plan* plan, int which, const float* x, float* spec, long planes, cudaStream_t st);

struct b2no_plan {
  b2no_geom g;
  b2no_tc_tables tc[2];  // [0]: inverse on the nout grid, [1]: adjoint of the forward on the nin grid
  b2no_tc_fwd_tables tcf[2];  // [0]: forward DFT on the nin grid, [1]: adjoint of the inverse on the nout grid
  int K[B2NO_MAX_DIM];   // kept modes per dim
  int device;
  // last-dim real tables, layout [qpad][npad] (q = 2k -> re, 2k+1 -> im), zero padded
  float* t_in;   // over the nin grid, scale s_f            (forward DFT / adjoint of forward)
  float* t_out;  // over the nout grid, scale s_i * c(k)    (inverse DFT / adjoint of inverse)
  int npad_in, npad_out, q2, qc, nchunk, qpad;
  // middle dims j < ndim-1: complex matrices, row-major
  float2* m_fwd[2];     // [nin_j][K_j]    exp(-i)
  float2* m_inv[2];     // [K_j][nout_j]   exp(+i)
  float2* m_adjinv[2];  // [nout_j][K_j]   conj(m_inv)^T
  float2* m_adjfwd[2];  // [K_j][nin_j]    conj(m_fwd)^T
  int* row_corner[2];   // [K_j] 0 = low corner, 1 = high corner
  int* row_local[2];    // [K_j] index inside the corner's weight
};

// ---- kept-mode bookkeeping shared by the mixing kernels (spectral.cu, tc_mix.cu) -----------------------------------
// A flattened kept-mode index k (over K_0 x .. x K_{d-1}, last fastest) -> the corner weight tensor that holds it and
// the offset inside that tensor (complex elements), following the corner convention of b2no_weights.
struct ModeMap {
  const int* corner[2];
  const int* local[2];
  int K[3];
  int ndim;
};

__device__ __forceinline__ void decode_mode(const ModeMap& mm, const b2no_weights& w, int k, int* corner,
                                            long* woff) {
  int c = 0;
  long off = 0;
  const int d = mm.ndim;
  int rem = k;
  int idx[3] = {0, 0, 0};
  for (int j = d - 1; j >= 0; j--) {
    idx[j] = rem % mm.K[j];
    rem /= mm.K[j];
  }
  for (int j = 0; j < d - 1; j++) {
    c = c * 2 + mm.corner[j][idx[j]];
    off += (long)mm.local[j][idx[j]] * w.stride_k[j];
  }
  off += (long)idx[d - 1] * w.stride_k[d - 1];
  *corner = c;
  *woff = off;
}

static inline ModeMap make_mode_map(const b2no_plan* p) {
  ModeMap mm;
  mm.ndim = p->g.ndim;
  for (int j = 0; j < 3; j++) mm.K[j] = j < p->g.ndim ? p->K[j] : 1;
  for (int j = 0; j < 2; j++) { mm.corner[j] = p->row_corner[j]; mm.local[j] = p->row_local[j]; }
  return mm;
}

static inline int total_modes(const b2no_plan* p) {
  int kt = 1;
  for (int j = 0; j < p->g.ndim; j++) kt *= p->K[j];
  return kt;
}

// tensor-core per-mode mixing (tc_mix.cu): return 0 = ran, 1 = shape not eligible (caller uses the CUDA-core kernel)
int b2no_tc_mix_feasible(int batch, int ci, int co, int mode);
int b2no_tc_mix_dw_feasible(int batch, int ci, int co);
int b2no_tc_mix(const b2no_plan* p, int mode, const float* in, const b2no_weights* w, float* out, int batch, int ci, int co,
                int accumulate, cudaStream_t st);
int b2no_tc_mix_dw(const b2no_plan* p, const float* xh, const float* gyh, const b2no_weights* dw, int batch, int ci, int co,
                   int accumulate, cudaStream_t st);

// ---- activations (exact forms: F.gelu default is the erf form) ---------------------------------
// erf(x) as a rational minimax x * P(x^2) / Q(x^2) on [-4, 4] (clamped; erf(4) = 1 - 1.5e-8): max abs error
// 4.5e-7 against float64 erf, 13 FMA-pipe instructions + one reciprocal instead of the ~40 of erff().  The GELU
// built on it differs from F.gelu by 7e-8 relative L2 (tests/test_host_cpu.py pins the coefficients on the CPU).
__device__ __forceinline__ float b2no_erf(float x) {
  x = fminf(fmaxf(x, -4.0f), 4.0f);
  const float x2 = x * x;
  float p = -2.72614225801306e-10f;
  p = fmaf(p, x2, 2.77068142495902e-08f);
  p = fmaf(p, x2, -2.10102402082508e-06f);
  p = fmaf(p, x2, -5.69250639462346e-05f);
  p = fmaf(p, x2, -7.34990630326855e-04f);
  p = fmaf(p, x2, -2.95459980854025e-03f);
  p = fmaf(p, x2, -1.60960333262415e-02f);
  float q = -1.45660718464996e-05f;
  q = fmaf(q, x2, -2.13374055278905e-04f);
  q = fmaf(q, x2, -1.68282697438203e-03f);
  q = fmaf(q, x2, -7.37332916720468e-03f);
  q = fmaf(q, x2, -1.42647390514189e-02f);
  return __fdividef(x * p, q);
}

// ---- packed fp32x2 forms (FFMA2 / FMUL2 / FADD2, sm_100): one FMA-pipe instruction per TWO elements, no branches.
// Same rational erf as above; the quotient uses MUFU.RCP (1 ulp), the Gaussian of the derivative MUFU.EX2.
__device__ __forceinline__ float2 b2no_f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float b2no_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float b2no_ex2(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float2 b2no_erf2(float2 x) {
  x.x = fminf(fmaxf(x.x, -4.0f), 4.0f);
  x.y = fminf(fmaxf(x.y, -4.0f), 4.0f);
  const float2 x2 = __fmul2_rn(x, x);
  float2 p = b2no_f2(-2.72614225801306e-10f);
  p = __ffma2_rn(p, x2, b2no_f2(2.77068142495902e-08f));
  p = __ffma2_rn(p, x2, b2no_f2(-2.10102402082508e-06f));
  p = __ffma2_rn(p, x2, b2no_f2(-5.69250639462346e-05f));
  p = __ffma2_rn(p, x2, b2no_f2(-7.34990630326855e-04f));
  p = __ffma2_rn(p, x2, b2no_f2(-2.95459980854025e-03f));
  p = __ffma2_rn(p, x2, b2no_f2(-1.60960333262415e-02f));
  float2 q = b2no_f2(-1.45660718464996e-05f);
  q = __ffma2_rn(q, x2, b2no_f2(-2.13374055278905e-04f));
  q = __ffma2_rn(q, x2, b2no_f2(-1.68282697438203e-03f));
  q = __ffma2_rn(q, x2, b2no_f2(-7.37332916720468e-03f));
  q = __ffma2_rn(q, x2, b2no_f2(-1.42647390514189e-02f));
  const float2 r = make_float2(b2no_rcp(q.x), b2no_rcp(q.y));
  return __fmul2_rn(__fmul2_rn(x, p), r);
}
// gelu(x) = 0.5 x (1 + erf(x / sqrt 2))
__device__ __forceinline__ float2 b2no_gelu2(float2 x) {
  const float2 e = b2no_erf2(__fmul2_rn(x, b2no_f2(0.70710678118654752440f)));
  const float2 h = __fmul2_rn(x, b2no_f2(0.5f));
  return __ffma2_rn(h, e, h);
}
// gelu(x) and gelu'(x) = Phi(x) + x phi(x) together.  The derivative needs the Gaussian g = exp(-x^2 / 2) anyway, and with g in
// hand the normal CDF comes cheaper through Abramowitz-Stegun 7.1.26 than through the rational erf above:
//     erfc(u) = (a1 t + .. + a5 t^5) exp(-u^2),  t = 1 / (1 + p u),  |error| <= 1.5e-7,   u = |x| / sqrt 2  =>  exp(-u^2) = g
//     Phi(x) = 1/2 + copysign(1/2 - 1/2 poly(t) g, x)
// 14 FMA-pipe instructions per PAIR instead of 22 (the backward epilogues are FMA-pipe bound), the same 4 MUFU (2 rcp, 2 ex2).
// Against float64: gelu 8e-8, gelu' 9e-8 relative L2 on N(0, 1.5) inputs (tests/test_host_cpu.py restates it in float32).
__device__ __forceinline__ void b2no_gelu2_both(float2 x, float2* val, float2* grad) {
  const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 den = __ffma2_rn(ax, b2no_f2(0.23164189f), b2no_f2(1.0f));                 // p / sqrt 2
  const float2 t = make_float2(b2no_rcp(den.x), b2no_rcp(den.y));
  float2 q = __ffma2_rn(b2no_f2(1.061405429f), t, b2no_f2(-1.453152027f));
  q = __ffma2_rn(q, t, b2no_f2(1.421413741f));
  q = __ffma2_rn(q, t, b2no_f2(-0.284496736f));
  q = __ffma2_rn(q, t, b2no_f2(0.254829592f));
  q = __fmul2_rn(q, t);
  const float2 a = __fmul2_rn(__fmul2_rn(x, x), b2no_f2(-0.72134752044448170368f));       // -0.5 x^2 log2(e)
  const float2 g = make_float2(b2no_ex2(a.x), b2no_ex2(a.y));
  const float2 h = __ffma2_rn(__fmul2_rn(q, g), b2no_f2(-0.5f), b2no_f2(0.5f));           // 1/2 erf(|x| / sqrt 2)
  const float2 cdf = __fadd2_rn(b2no_f2(0.5f), make_float2(copysignf(h.x, x.x), copysignf(h.y, x.y)));
  *val = __fmul2_rn(x, cdf);
  *grad = __ffma2_rn(__fmul2_rn(x, b2no_f2(0.39894228040143267794f)), g, cdf);
}
__device__ __forceinline__ float2 b2no_gelu2_grad(float2 x) {
  float2 v, g;
  b2no_gelu2_both(x, &v, &g);
  return g;
}

__device__ __forceinline__ float b2no_act(float x, int act) {
  switch (act) {
    case B2NO_ACT_GELU: return 0.5f * x * (1.0f + b2no_erf(x * 0.70710678118654752440f));
    case B2NO_ACT_RELU: return x > 0.f ? x : 0.f;
    case B2NO_ACT_SIGMOID: return 1.0f / (1.0f + expf(-x));
    case B2NO_ACT_SELU: {
      const float scale = 1.0507009873554804934193349852946f, alpha = 1.6732632423543772848170429916717f;
      return x > 0.f ? scale * x : scale * alpha * expm1f(x);
    }
    case B2NO_ACT_TANH: return tanhf(x);
    default: return x;
  }
}

__device__ __forceinline__ float b2no_act_grad(float x, int act) {
  switch (act) {
    case B2NO_ACT_GELU: {
      const float cdf = 0.5f * (1.0f + b2no_erf(x * 0.70710678118654752440f));
      const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
      return cdf + x * pdf;
    }
    case B2NO_ACT_RELU: return x > 0.f ? 1.f : 0.f;
    case B2NO_ACT_SIGMOID: {
      const float s = 1.0f / (1.0f + expf(-x));
      return s * (1.0f - s);
    }
    case B2NO_ACT_SELU: {
      const float scale = 1.0507009873554804934193349852946f, alpha = 1.6732632423543772848170429916717f;
      return x > 0.f ? scale : scale * alpha * expf(x);
    }
    case B2NO_ACT_TANH: {
      const float t = tanhf(x);
      return 1.0f - t * t;
    }
    default: return 1.f;
  }
}
