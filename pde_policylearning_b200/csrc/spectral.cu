// Mode-restricted DFT stages, per-mode channel mixing and the fused inverse epilogue (fp32 CUDA-core
// path).  Only the kept low modes are ever materialised: no full-size spectrum, no zero-filled out_fft.
//
//   k_r2c_last   x[R, N]  -> A[R, K_d]          real -> complex along the contiguous (rfft) axis
//   k_cmat       [outer, J, inner] -> [outer, M, inner]   complex matrix along a middle axis (both directions)
//   k_mix        Yh[b,o,k] = sum_i Xh[b,i,k] W[i,o,k]     (and the conj/transposed adjoint)
//   k_dw         dW[i,o,k] = sum_b conj(Xh) gYh
//   k_c2r_fused  y = act(irfft_last(Bq) + bias + W1x1 x (+ W' x') + add) * mul
#include <string.h>
#include "common.cuh"

// =============================================================================================
// k_r2c_last
//   One warp transforms 8 rows at a time.  Lane l owns samples n = l + 32 j; the twiddle table sits in
//   shared memory as [q][n] (conflict-free, one LDS feeds 8 FMAs); the 32 partial sums of every
//   (row, q) are combined with a transposing butterfly: after 5 shuffle stages lane l holds the QC/4
//   finished values with linear index [l*QC/4, (l+1)*QC/4) of the 8 x QC block -> coalesced store.
// =============================================================================================
template <int QC>
__global__ void __launch_bounds__(256)
k_r2c_last(const float* __restrict__ x, float* __restrict__ out, const float* __restrict__ tab,
           long R, int N, int npad, int q2, int nchunk) {
  extern __shared__ float s_tab[];  // [QC*nchunk][npad]
  const int qpad = QC * nchunk;
  for (int i = threadIdx.x; i < qpad * npad; i += blockDim.x) s_tab[i] = tab[i];
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int npl = (N + 31) >> 5;
  const long ngroups = (R + 7) >> 3;
  for (long g = (long)blockIdx.x * 8 + warp; g < ngroups; g += (long)gridDim.x * 8) {
    const long r0 = g << 3;
    for (int c = 0; c < nchunk; c++) {
      float v[8 * QC];
#pragma unroll
      for (int i = 0; i < 8 * QC; i++) v[i] = 0.f;
      for (int j = 0; j < npl; j++) {
        const int n = lane + (j << 5);
        float xv[8];
#pragma unroll
        for (int r = 0; r < 8; r++) xv[r] = (n < N && r0 + r < R) ? __ldg(x + (r0 + r) * N + n) : 0.f;
        const float* tq = s_tab + (size_t)(c * QC) * npad + n;
#pragma unroll
        for (int q = 0; q < QC; q++) {
          const float t = tq[(size_t)q * npad];
#pragma unroll
          for (int r = 0; r < 8; r++) v[r * QC + q] = fmaf(xv[r], t, v[r * QC + q]);
        }
      }
      // transposing butterfly over the 32 lanes
#pragma unroll
      for (int s = 0; s < 5; s++) {
        const int off = 16 >> s;
        const int half = (8 * QC) >> (s + 1);
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < half; i++) {
          const float a = v[i], b = v[i + half];
          const float send = upper ? a : b;
          const float keep = upper ? b : a;
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      constexpr int PER = QC / 4;
#pragma unroll
      for (int i = 0; i < PER; i++) {
        const int idx = lane * PER + i;
        const int r = idx / QC, q = c * QC + idx % QC;
        if (r0 + r < R && q < q2) out[(r0 + r) * q2 + q] = v[i];
      }
    }
  }
}

template <int QC>
static int launch_r2c(const float* x, float* out, const float* tab, long R, int N, int npad, int q2,
                      int nchunk, cudaStream_t st) {
  const size_t smem = (size_t)QC * nchunk * npad * sizeof(float);
  if (smem > 200 * 1024) return B2NO_E_UNSUPPORTED;
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_r2c_last<QC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long ngroups = (R + 7) / 8;
  long blocks = (ngroups + 7) / 8;
  const long cap = (long)b2no_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_r2c_last<QC><<<(unsigned)blocks, 256, smem, st>>>(x, out, tab, R, N, npad, q2, nchunk);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// =============================================================================================
// k_r2c_rows: the same stage for few kept modes (q2 <= 16, e.g. the PINO layer: 73 samples -> 8 modes).  A warp stages 8
// consecutive rows (8 N contiguous floats, 128-bit loads) in shared memory; lane l then owns row l / 4 and QL of its q2
// outputs: per sample one broadcast LDS of x, one vector LDS of the transposed table row and QL FMAs -- no cross-lane
// reduction at all.  (k_r2c_last spends as many instructions on its transposing butterfly as on FMAs: ncu showed it
// issue-bound at 70 % with FSEL + SHFL + FADD = 32 % of the instructions, profiles/r02_d_ncu_pino_r2c.txt.)
// =============================================================================================
template <int QL>
__global__ void __launch_bounds__(256)
k_r2c_rows(const float* __restrict__ x, float* __restrict__ out, const float* __restrict__ tab, long R, int N, int npad, int q2) {
  extern __shared__ float s_dyn[];
  constexpr int Q2P = 4 * QL;
  float* s_tabT = s_dyn;                              // [N][Q2P]
  float* s_rows = s_dyn + (size_t)N * Q2P;            // [8 warps][8 N]
  for (int i = threadIdx.x; i < N * Q2P; i += 256) {
    const int n = i / Q2P, q = i - n * Q2P;
    s_tabT[i] = q < q2 ? tab[(size_t)q * npad + n] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* rows = s_rows + (size_t)warp * 8 * N;
  const int r = lane >> 2, q0 = (lane & 3) * QL;
  const long ngroups = R >> 3;                        // R % 8 == 0 (checked by the launcher)
  for (long g = (long)blockIdx.x * 8 + warp; g < ngroups; g += (long)gridDim.x * 8) {
    const float4* src = reinterpret_cast<const float4*>(x + (g << 3) * N);
    for (int i = lane; i < 2 * N; i += 32) reinterpret_cast<float4*>(rows)[i] = __ldg(src + i);
    __syncwarp();
    float acc[QL];
#pragma unroll
    for (int i = 0; i < QL; i++) acc[i] = 0.f;
    const float* xr = rows + r * N;
#pragma unroll 4
    for (int n = 0; n < N; n++) {
      const float xv = xr[n];
      const float* t = s_tabT + n * Q2P + q0;
#pragma unroll
      for (int i = 0; i < QL; i++) acc[i] = fmaf(xv, t[i], acc[i]);
    }
    float* dst = out + ((g << 3) + r) * q2 + q0;
#pragma unroll
    for (int i = 0; i < QL; i++)
      if (q0 + i < q2) dst[i] = acc[i];
    __syncwarp();
  }
}

// 32 rows per warp, lane = row: the table row of a sample is read with warp-UNIFORM vector loads (one shared-memory
// wavefront each, whatever the number of lanes), so a sample costs Q2P / 4 + 1 wavefronts for 32 x Q2P FMAs -- the 8-row
// variant above pays 5 wavefronts for 8 x 16 and was LSU-bound (214 us for the 306 MB PINO pass).
template <int Q2P>
__global__ void __launch_bounds__(256)
k_r2c_rows32(const float* __restrict__ x, float* __restrict__ out, const float* __restrict__ tab, long R, int N, int npad, int q2) {
  extern __shared__ float s_dyn[];
  const int NS = N | 1;                               // odd row stride: lane-strided reads are conflict-free
  float* s_tabT = s_dyn;                              // [N][Q2P]
  float* s_rows = s_dyn + (size_t)N * Q2P;            // [8 warps][32 NS]
  for (int i = threadIdx.x; i < N * Q2P; i += 256) {
    const int n = i / Q2P, q = i - n * Q2P;
    s_tabT[i] = q < q2 ? tab[(size_t)q * npad + n] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* rows = s_rows + (size_t)warp * 32 * NS;
  const long ngroups = R >> 5;                        // R % 32 == 0 (checked by the launcher)
  for (long g = (long)blockIdx.x * 8 + warp; g < ngroups; g += (long)gridDim.x * 8) {
    const float* src = x + (g << 5) * N;
    if (NS == N) {
      const float4* s4 = reinterpret_cast<const float4*>(src);
      for (int i = lane; i < 8 * N; i += 32) reinterpret_cast<float4*>(rows)[i] = __ldg(s4 + i);
    } else {
      for (int i = lane; i < 32 * N; i += 32) {
        const int rr = i / N, n = i - rr * N;
        rows[rr * NS + n] = __ldg(src + i);
      }
    }
    __syncwarp();
    float acc[Q2P];
#pragma unroll
    for (int i = 0; i < Q2P; i++) acc[i] = 0.f;
    const float* xr = rows + lane * NS;
#pragma unroll 2
    for (int n = 0; n < N; n++) {
      const float xv = xr[n];
      const float4* t4 = reinterpret_cast<const float4*>(s_tabT + n * Q2P);
#pragma unroll
      for (int i = 0; i < Q2P / 4; i++) {
        const float4 t = t4[i];
        acc[4 * i] = fmaf(xv, t.x, acc[4 * i]);
        acc[4 * i + 1] = fmaf(xv, t.y, acc[4 * i + 1]);
        acc[4 * i + 2] = fmaf(xv, t.z, acc[4 * i + 2]);
        acc[4 * i + 3] = fmaf(xv, t.w, acc[4 * i + 3]);
      }
    }
    float* dst = out + ((g << 5) + lane) * q2;
    if (q2 == Q2P) {
#pragma unroll
      for (int i = 0; i < Q2P / 4; i++)
        reinterpret_cast<float4*>(dst)[i] = make_float4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < Q2P; i++)
        if (i < q2) dst[i] = acc[i];
    }
    __syncwarp();
  }
}

template <int Q2P>
static int launch_r2c_rows32(const float* x, float* out, const float* tab, long R, int N, int npad, int q2, cudaStream_t st) {
  const size_t smem = ((size_t)N * Q2P + (size_t)8 * 32 * (N | 1)) * sizeof(float);
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_r2c_rows32<Q2P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long ngroups = R / 32;
  long blocks = (ngroups + 7) / 8;
  const long cap = (long)b2no_sm_count() * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_r2c_rows32<Q2P><<<(unsigned)blocks, 256, smem, st>>>(x, out, tab, R, N, npad, q2);
  B2NO_LAUNCH_CHECK();
  return 0;
}

template <int QL>
static int launch_r2c_rows(const float* x, float* out, const float* tab, long R, int N, int npad, int q2, cudaStream_t st) {
  const size_t smem = ((size_t)N * 4 * QL + (size_t)8 * 8 * N) * sizeof(float);
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_r2c_rows<QL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long ngroups = R / 8;
  long blocks = (ngroups + 7) / 8;
  const long cap = (long)b2no_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_r2c_rows<QL><<<(unsigned)blocks, 256, smem, st>>>(x, out, tab, R, N, npad, q2);
  B2NO_LAUNCH_CHECK();
  return 0;
}

static int run_r2c(const b2no_plan* p, int which, const float* x, float* out, long R, cudaStream_t st) {
  const int d = p->g.ndim;
  const int N = which == 0 ? p->g.nin[d - 1] : p->g.nout[d - 1];
  const int npad = which == 0 ? p->npad_in : p->npad_out;
  const float* tab = which == 0 ? p->t_in : p->t_out;
  if (R % 32 == 0 && R >= 32 * 8 * 64 && p->q2 <= 16 && p->q2 % 4 == 0 && N >= 8 && N <= 160 && (((uintptr_t)x) & 15) == 0 &&
      (((uintptr_t)out) & 15) == 0) {
    // many rows: lane = row (warp-uniform table reads)
    if (p->q2 <= 8) return launch_r2c_rows32<8>(x, out, tab, R, N, npad, p->q2, st);
    return launch_r2c_rows32<16>(x, out, tab, R, N, npad, p->q2, st);
  }
  if (R % 8 == 0 && p->q2 <= 16 && N >= 8 && N <= 512 && (((uintptr_t)x) & 15) == 0) {
    if (p->q2 <= 4) return launch_r2c_rows<1>(x, out, tab, R, N, npad, p->q2, st);
    if (p->q2 <= 8) return launch_r2c_rows<2>(x, out, tab, R, N, npad, p->q2, st);
    return launch_r2c_rows<4>(x, out, tab, R, N, npad, p->q2, st);
  }
  switch (p->qc) {
    case 4: return launch_r2c<4>(x, out, tab, R, N, npad, p->q2, p->nchunk, st);
    case 8: return launch_r2c<8>(x, out, tab, R, N, npad, p->q2, p->nchunk, st);
    case 12: return launch_r2c<12>(x, out, tab, R, N, npad, p->q2, p->nchunk, st);
    case 16: return launch_r2c<16>(x, out, tab, R, N, npad, p->q2, p->nchunk, st);
  }
  return B2NO_E_UNSUPPORTED;
}

// =============================================================================================
// k_cmat: out[o, m, i] = sum_j in[o, j, i] * T[j, m]   (complex), one thread per (o, i) column and
// an MT-wide tile of m in registers; T tile in shared memory (broadcast reads).
// =============================================================================================
template <int MT>
__global__ void __launch_bounds__(128)
k_cmat(const float2* __restrict__ in, float2* __restrict__ out, const float2* __restrict__ T,
       long outer, int J, int M, int inner) {
  extern __shared__ float2 s_T[];  // [J][MT]
  const int m0 = blockIdx.y * MT;
  for (int idx = threadIdx.x; idx < J * MT; idx += blockDim.x) {
    const int j = idx / MT, mm = idx - j * MT;
    s_T[idx] = (m0 + mm < M) ? T[(size_t)j * M + m0 + mm] : make_float2(0.f, 0.f);
  }
  __syncthreads();
  const long total = outer * inner;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const long o = t / inner;
    const int i = (int)(t - o * inner);
    float2 acc[MT];
#pragma unroll
    for (int mm = 0; mm < MT; mm++) acc[mm] = make_float2(0.f, 0.f);
    const float2* src = in + (o * J) * inner + i;
#pragma unroll 4
    for (int j = 0; j < J; j++) {
      const float2 v = __ldg(src + (size_t)j * inner);
      const float2* trow = s_T + j * MT;
#pragma unroll
      for (int mm = 0; mm < MT; mm++) {
        const float2 w = trow[mm];
        acc[mm].x = fmaf(v.x, w.x, fmaf(-v.y, w.y, acc[mm].x));
        acc[mm].y = fmaf(v.x, w.y, fmaf(v.y, w.x, acc[mm].y));
      }
    }
#pragma unroll
    for (int mm = 0; mm < MT; mm++)
      if (m0 + mm < M) out[(o * M + m0 + mm) * inner + i] = acc[mm];
  }
}

template <int MT>
static int launch_cmat(const float2* in, float2* out, const float2* T, long outer, int J, int M, int inner,
                       cudaStream_t st) {
  const size_t smem = (size_t)J * MT * sizeof(float2);
  if (smem > 200 * 1024) return B2NO_E_UNSUPPORTED;
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_cmat<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long total = outer * inner;
  long bx = (total + 127) / 128;
  const long cap = (long)b2no_sm_count() * 16;
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  dim3 grid((unsigned)bx, (unsigned)((M + MT - 1) / MT));
  k_cmat<MT><<<grid, 128, smem, st>>>(in, out, T, outer, J, M, inner);
  B2NO_LAUNCH_CHECK();
  return 0;
}

static int run_cmat(const float2* in, float2* out, const float2* T, long outer, int J, int M, int inner,
                    cudaStream_t st) {
  if (M <= 4) return launch_cmat<4>(in, out, T, outer, J, M, inner, st);
  if (M <= 8) return launch_cmat<8>(in, out, T, outer, J, M, inner, st);
  if (M <= 12 || M == 24) return launch_cmat<12>(in, out, T, outer, J, M, inner, st);
  return launch_cmat<16>(in, out, T, outer, J, M, inner, st);
}

// =============================================================================================
// k_fwd_plane32: both stages of the 2-D forward transform for SMALL planes (H, W <= 32: the RNO 32 x 32 grid), one WARP per
// plane, nothing but the plane read and the kept modes written.
//   stage 1 (lane = row h, the row of x in 32 registers):  A[h, ky] = sum_w x[h, w] (T[2ky, w] + i T[2ky+1, w])
//   stage 2 (lane = kept row kx):                          Xh[kx, ky] = sum_h M[h, kx] A[h, ky]
// Packed fp32x2 arithmetic (exact fp32, no tensor cores): stage 1 one FFMA2 per (w, ky), stage 2 two per (h, ky) with
// separate accumulators for the Re M and Im M products (no operand swaps).  Why not k_fwd_tc here: on 32 x 32 planes its
// 128-row tile is four planes = 16 KB per ~60 MMAs and two hand-overs; measured 58 us for 35.7 MB (0.6 TB/s) at the cfg3 shape.
// Measured at the cfg3 shape (8704 planes): 64 us against 58 - 82 us of k_fwd_tc -- latency-bound (issue slots 33 % busy, one
// plane per warp at a time), not the FMA-pipe bound of (384 + 768) FFMA2 per plane; cfg3 gains 2.7 %.  Forcing four blocks
// per SM (64 registers, spills) changed nothing.
// Tables in shared memory: sT[w][ky] (pairs), sM[h][kx]; A goes through shared memory ([h][KL + 2] pairs per warp: the
// lane changes from "row" to "kept row").
// =============================================================================================
template <int KL>
__global__ void __launch_bounds__(256)
k_fwd_plane32(const float* __restrict__ x, float2* __restrict__ spec, const float* __restrict__ tab, int npad,
              const float2* __restrict__ M, long planes, int H, int W, int K0, int Kl, int layout) {
  extern __shared__ float2 sm2[];
  float2* sT = sm2;                                  // [32][KL]
  float2* sM = sT + 32 * KL;                         // [32][32]
  float2* sA = sM + 32 * 32;                         // [8 warps][32][KL + 2]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 32 * KL; i += 256) {
    const int w = i / KL, ky = i - w * KL;
    sT[i] = (w < W && ky < Kl) ? make_float2(__ldg(tab + (size_t)(2 * ky) * npad + w), __ldg(tab + (size_t)(2 * ky + 1) * npad + w))
                               : make_float2(0.f, 0.f);
  }
  for (int i = threadIdx.x; i < 32 * 32; i += 256) {
    const int h = i >> 5, kx = i & 31;
    sM[i] = (h < H && kx < K0) ? __ldg(M + (size_t)h * K0 + kx) : make_float2(0.f, 0.f);
  }
  __syncthreads();
  float2* myA = sA + (size_t)warp * 32 * (KL + 2);
  for (long p0 = (long)blockIdx.x * 8; p0 < planes; p0 += (long)gridDim.x * 8) {
    const long plane = p0 + warp;
    const bool live = plane < planes;
    // ---- stage 1 ----
    float xr[32];
#pragma unroll
    for (int w = 0; w < 32; w++) xr[w] = 0.f;
    if (live && lane < H) {
      const float4* row = reinterpret_cast<const float4*>(x + ((size_t)plane * H + lane) * W);
#pragma unroll
      for (int w4 = 0; w4 < 8; w4++)
        if (w4 * 4 < W) {
          const float4 v = __ldg(row + w4);
          xr[4 * w4] = v.x; xr[4 * w4 + 1] = v.y; xr[4 * w4 + 2] = v.z; xr[4 * w4 + 3] = v.w;
        }
    }
    float2 acc[KL];
#pragma unroll
    for (int k = 0; k < KL; k++) acc[k] = make_float2(0.f, 0.f);
#pragma unroll
    for (int w = 0; w < 32; w++) {
      if (w < W) {
        const float2 xx = make_float2(xr[w], xr[w]);
#pragma unroll
        for (int k = 0; k < KL; k += 2) {
          const float4 t = *reinterpret_cast<const float4*>(sT + w * KL + k);
          acc[k] = __ffma2_rn(xx, make_float2(t.x, t.y), acc[k]);
          acc[k + 1] = __ffma2_rn(xx, make_float2(t.z, t.w), acc[k + 1]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < KL; k++) myA[lane * (KL + 2) + k] = acc[k];
    __syncwarp();
    // ---- stage 2 ----
    float2 pr[KL], pi[KL];
#pragma unroll
    for (int k = 0; k < KL; k++) { pr[k] = make_float2(0.f, 0.f); pi[k] = make_float2(0.f, 0.f); }
    for (int h = 0; h < H; h++) {
      const float2 m = sM[h * 32 + lane];
      const float2 mr = make_float2(m.x, m.x), mi = make_float2(m.y, m.y);
#pragma unroll
      for (int k = 0; k < KL; k += 2) {
        const float4 a = *reinterpret_cast<const float4*>(myA + h * (KL + 2) + k);
        pr[k] = __ffma2_rn(mr, make_float2(a.x, a.y), pr[k]);
        pi[k] = __ffma2_rn(mi, make_float2(a.x, a.y), pi[k]);
        pr[k + 1] = __ffma2_rn(mr, make_float2(a.z, a.w), pr[k + 1]);
        pi[k + 1] = __ffma2_rn(mi, make_float2(a.z, a.w), pi[k + 1]);
      }
    }
    // (m.re + i m.im)(a.re + i a.im) = (m.re a.re - m.im a.im) + i (m.re a.im + m.im a.re)
    if (layout == 0) {
      if (live && lane < K0) {
        float2* dst = spec + ((size_t)plane * K0 + lane) * Kl;
#pragma unroll
        for (int k = 0; k < KL; k++)
          if (k < Kl) dst[k] = make_float2(pr[k].x - pi[k].y, pr[k].y + pi[k].x);
      }
      __syncwarp();
    } else {
      // mode-major: the 8 planes of a block are consecutive, so the eight 8-byte stores of a mode (one per warp) fall into
      // two 32-byte sectors and merge in L2
      if (live && lane < K0) {
        float2* dst = spec + (size_t)lane * Kl * planes + plane;
#pragma unroll
        for (int k = 0; k < KL; k++)
          if (k < Kl) dst[(size_t)k * planes] = make_float2(pr[k].x - pi[k].y, pr[k].y + pi[k].x);
      }
      __syncwarp();
    }
  }
}

static int launch_fwd_plane32(const b2no_plan* p, int which, const float* x, float* spec, long planes, cudaStream_t st) {
  const int32_t* n = which == 0 ? p->g.nin : p->g.nout;
  const int H = n[0], W = n[1], K0 = p->K[0], Kl = p->K[1];
  const float* tab = which == 0 ? p->t_in : p->t_out;
  const int npad = which == 0 ? p->npad_in : p->npad_out;
  const float2* M = which == 0 ? p->m_fwd[0] : p->m_adjinv[0];
  const int KL = Kl <= 8 ? 8 : (Kl <= 12 ? 12 : 16);
  const size_t smem = sizeof(float2) * ((size_t)32 * KL + 32 * 32 + (size_t)8 * 32 * (KL + 2));
  long blocks = (planes + 7) / 8;
  const long cap = (long)b2no_sm_count() * 8;
  if (blocks > cap) blocks = cap;
#define FP32_LAUNCH(K)                                                                                                      \
  do {                                                                                                                      \
    if (smem > 48 * 1024) B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_fwd_plane32<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_fwd_plane32<K><<<(unsigned)blocks, 256, smem, st>>>(x, (float2*)spec, tab, npad, M, planes, H, W, K0, Kl, p->g.spec_layout); \
  } while (0)
  if (KL == 8) FP32_LAUNCH(8); else if (KL == 12) FP32_LAUNCH(12); else FP32_LAUNCH(16);
#undef FP32_LAUNCH
  B2NO_LAUNCH_CHECK();
  return 0;
}

// =============================================================================================
// forward pipeline
// =============================================================================================
extern "C" int b2no_dft_forward(const b2no_plan* p, int which, const float* x, float* spec, float* work,
                                int64_t bc, void* stream) {
  if (!p || !x || !spec || bc < 1 || (which != 0 && which != 1)) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int d = p->g.ndim;
  const int32_t* n = which == 0 ? p->g.nin : p->g.nout;
  const int Kl = p->K[d - 1];
  if (d == 1) return run_r2c(p, which, x, spec, bc, st);
  if (d == 2) {
    // small planes (RNO 32 x 32): one warp per plane on the FMA pipe -- the 128-row tensor-core tile is four planes there
    if (n[0] <= 32 && n[1] <= 32 && n[1] % 4 == 0 && p->K[0] <= 32 && Kl <= 16 && (((uintptr_t)x) & 15) == 0 &&
        (p->g.spec_layout == 0 || p->g.spec_layout == 1))
      return launch_fwd_plane32(p, which, x, spec, (long)bc, st);
    // tensor-core path (tc_dft.cu): one kernel, no intermediate, when the plane shape fits the 128-row tile
    const int rc = b2no_tc_dft_forward(p, which, x, spec, (long)bc, st);
    if (rc != 1) return rc;
  }
  if (p->g.spec_layout != 0) return B2NO_E_UNSUPPORTED;     // mode-major spectra exist on the tensor-core kernels only
  if (!work) return B2NO_E_ARG;
  float2* A = (float2*)work;
  if (d == 2) {
    int rc = run_r2c(p, which, x, (float*)A, bc * n[0], st);
    if (rc) return rc;
    const float2* T = which == 0 ? p->m_fwd[0] : p->m_adjinv[0];
    return run_cmat(A, (float2*)spec, T, bc, n[0], p->K[0], Kl, st);
  }
  // d == 3
  float2* Bb = A + (size_t)bc * n[0] * n[1] * Kl;
  int rc = run_r2c(p, which, x, (float*)A, bc * n[0] * n[1], st);
  if (rc) return rc;
  const float2* T1 = which == 0 ? p->m_fwd[1] : p->m_adjinv[1];
  rc = run_cmat(A, Bb, T1, bc * n[0], n[1], p->K[1], Kl, st);
  if (rc) return rc;
  const float2* T0 = which == 0 ? p->m_fwd[0] : p->m_adjinv[0];
  return run_cmat(Bb, (float2*)spec, T0, bc, n[0], p->K[0], p->K[1] * Kl, st);
}

// =============================================================================================
// k_mix / k_dw
// =============================================================================================
// out[b,p,k] (+)= sum_q in[b,q,k] * Wq    with  Wq = W[q,p,k] (CONJT=false)  or  conj(W[p,q,k]) (CONJT=true)
template <int BT, int PT, bool CONJT>
__global__ void __launch_bounds__(128)
k_mix(const float2* __restrict__ in, float2* __restrict__ out, b2no_weights w, ModeMap mm, int B, int Cq,
      int Cp, int Kt, int accumulate) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= Kt) return;
  const int b0 = blockIdx.y * BT, p0 = blockIdx.z * PT;
  int corner;
  long woff;
  decode_mode(mm, w, k, &corner, &woff);
  const float2* wbase = (const float2*)w.corner[corner] + woff;
  float2 acc[BT][PT];
#pragma unroll
  for (int bb = 0; bb < BT; bb++)
#pragma unroll
    for (int pp = 0; pp < PT; pp++) acc[bb][pp] = make_float2(0.f, 0.f);
  for (int q = 0; q < Cq; q++) {
    float2 xin[BT], wv[PT];
#pragma unroll
    for (int bb = 0; bb < BT; bb++)
      xin[bb] = (b0 + bb < B) ? __ldg(in + ((size_t)(b0 + bb) * Cq + q) * Kt + k) : make_float2(0.f, 0.f);
#pragma unroll
    for (int pp = 0; pp < PT; pp++) {
      float2 t = make_float2(0.f, 0.f);
      if (p0 + pp < Cp) {
        const long off = CONJT ? ((long)(p0 + pp) * w.stride_i + (long)q * w.stride_o)
                               : ((long)q * w.stride_i + (long)(p0 + pp) * w.stride_o);
        t = __ldg(wbase + off);
        if (CONJT) t.y = -t.y;
      }
      wv[pp] = t;
    }
#pragma unroll
    for (int bb = 0; bb < BT; bb++)
#pragma unroll
      for (int pp = 0; pp < PT; pp++) {
        acc[bb][pp].x = fmaf(xin[bb].x, wv[pp].x, fmaf(-xin[bb].y, wv[pp].y, acc[bb][pp].x));
        acc[bb][pp].y = fmaf(xin[bb].x, wv[pp].y, fmaf(xin[bb].y, wv[pp].x, acc[bb][pp].y));
      }
  }
#pragma unroll
  for (int bb = 0; bb < BT; bb++)
#pragma unroll
    for (int pp = 0; pp < PT; pp++)
      if (b0 + bb < B && p0 + pp < Cp) {
        float2* dst = out + ((size_t)(b0 + bb) * Cp + p0 + pp) * Kt + k;
        float2 r = acc[bb][pp];
        if (accumulate) { const float2 old = *dst; r.x += old.x; r.y += old.y; }
        *dst = r;
      }
}

// One thread per output (b, p, k), k fastest: a warp reads contiguous runs of the spectrum and of the weights; the
// Cq-long sum is unrolled so that 8 independent load pairs are in flight.  Grid = B*Cp*Kt / 256 blocks (576 at cfg2)
// instead of the 256 two-warp blocks of k_mix, which was latency-bound at 22-34 us for 1.2 MB of data.
template <bool CONJT>
__global__ void __launch_bounds__(256)
k_mix2(const float2* __restrict__ in, float2* __restrict__ out, b2no_weights w, ModeMap mm, int B, int Cq, int Cp,
       int Kt, int accumulate) {
  const long idx = (long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (long)B * Cp * Kt) return;
  const int k = (int)(idx % Kt);
  const long t = idx / Kt;
  const int pp = (int)(t % Cp), b = (int)(t / Cp);
  int corner;
  long woff;
  decode_mode(mm, w, k, &corner, &woff);
  const float2* wp = (const float2*)w.corner[corner] + woff + (CONJT ? (long)pp * w.stride_i : (long)pp * w.stride_o);
  const long wq = CONJT ? w.stride_o : w.stride_i;
  const float2* xp = in + (size_t)b * Cq * Kt + k;
  float2 acc = make_float2(0.f, 0.f);
  int q = 0;
  for (; q + 8 <= Cq; q += 8) {
    float2 xv[8], wv[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      xv[u] = __ldg(xp + (size_t)(q + u) * Kt);
      wv[u] = __ldg(wp + (long)(q + u) * wq);
    }
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const float wy = CONJT ? -wv[u].y : wv[u].y;
      acc.x = fmaf(xv[u].x, wv[u].x, fmaf(-xv[u].y, wy, acc.x));
      acc.y = fmaf(xv[u].x, wy, fmaf(xv[u].y, wv[u].x, acc.y));
    }
  }
  for (; q < Cq; q++) {
    const float2 xv = __ldg(xp + (size_t)q * Kt), wv = __ldg(wp + (long)q * wq);
    const float wy = CONJT ? -wv.y : wv.y;
    acc.x = fmaf(xv.x, wv.x, fmaf(-xv.y, wy, acc.x));
    acc.y = fmaf(xv.x, wy, fmaf(xv.y, wv.x, acc.y));
  }
  float2* dst = out + ((size_t)b * Cp + pp) * Kt + k;
  if (accumulate) { const float2 old = *dst; acc.x += old.x; acc.y += old.y; }
  *dst = acc;
}

// dW[i,o,k] = sum_b conj(Xh[b,i,k]) gYh[b,o,k]: one thread per output, k fastest, the batch sum unrolled by 8
__global__ void __launch_bounds__(256)
k_dw2(const float2* __restrict__ xh, const float2* __restrict__ gyh, b2no_weights w, ModeMap mm, int B, int Ci, int Co,
      int Kt, int accumulate) {
  const long idx = (long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (long)Ci * Co * Kt) return;
  const int k = (int)(idx % Kt);
  const long t = idx / Kt;
  const int o = (int)(t % Co), i = (int)(t / Co);
  const float2* xp = xh + (size_t)i * Kt + k;
  const float2* gp = gyh + (size_t)o * Kt + k;
  const size_t xs = (size_t)Ci * Kt, gs = (size_t)Co * Kt;
  float2 acc = make_float2(0.f, 0.f);
  int b = 0;
  for (; b + 8 <= B; b += 8) {
    float2 xv[8], gv[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      xv[u] = __ldg(xp + (size_t)(b + u) * xs);
      gv[u] = __ldg(gp + (size_t)(b + u) * gs);
    }
#pragma unroll
    for (int u = 0; u < 8; u++) {
      acc.x = fmaf(xv[u].x, gv[u].x, fmaf(xv[u].y, gv[u].y, acc.x));
      acc.y = fmaf(xv[u].x, gv[u].y, fmaf(-xv[u].y, gv[u].x, acc.y));
    }
  }
  for (; b < B; b++) {
    const float2 xv = __ldg(xp + (size_t)b * xs), gv = __ldg(gp + (size_t)b * gs);
    acc.x = fmaf(xv.x, gv.x, fmaf(xv.y, gv.y, acc.x));
    acc.y = fmaf(xv.x, gv.y, fmaf(-xv.y, gv.x, acc.y));
  }
  int corner;
  long woff;
  decode_mode(mm, w, k, &corner, &woff);
  float2* dst = (float2*)w.corner[corner] + woff + (long)i * w.stride_i + (long)o * w.stride_o;
  if (accumulate) { const float2 old = *dst; acc.x += old.x; acc.y += old.y; }
  *dst = acc;
}

extern "C" int b2no_mix(const b2no_plan* p, int mode, const float* in, const b2no_weights* w, float* out,
                        int batch, int ci, int co, int accumulate, void* stream) {
  if (!p || !in || !w || !out || batch < 1 || ci < 1 || co < 1 || (mode != 0 && mode != 1)) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int Kt = total_modes(p);
  const ModeMap mm = make_mode_map(p);
  {
    // large batches: per-mode [batch x 2Cq] x [2Cq x 2Cp] real-block products on the tensor cores (tc_mix.cu)
    const int rc = b2no_tc_mix(p, mode, in, w, out, batch, ci, co, accumulate, st);
    if (rc != 1) return rc;
  }
  if (p->g.spec_layout != 0) return B2NO_E_UNSUPPORTED;
  const int Cq = mode == 0 ? ci : co, Cp = mode == 0 ? co : ci;
  const long total = (long)batch * Cp * Kt;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (mode == 0)
    k_mix2<false><<<blocks, 256, 0, st>>>((const float2*)in, (float2*)out, *w, mm, batch, Cq, Cp, Kt, accumulate);
  else
    k_mix2<true><<<blocks, 256, 0, st>>>((const float2*)in, (float2*)out, *w, mm, batch, Cq, Cp, Kt, accumulate);
  B2NO_LAUNCH_CHECK();
  return 0;
}

template <int IT, int OT>
__global__ void __launch_bounds__(128)
k_dw(const float2* __restrict__ xh, const float2* __restrict__ gyh, b2no_weights w, ModeMap mm, int B, int Ci,
     int Co, int Kt, int accumulate) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= Kt) return;
  const int i0 = blockIdx.y * IT, o0 = blockIdx.z * OT;
  int corner;
  long woff;
  decode_mode(mm, w, k, &corner, &woff);
  float2 acc[IT][OT];
#pragma unroll
  for (int ii = 0; ii < IT; ii++)
#pragma unroll
    for (int oo = 0; oo < OT; oo++) acc[ii][oo] = make_float2(0.f, 0.f);
  for (int b = 0; b < B; b++) {
    float2 xi[IT], go[OT];
#pragma unroll
    for (int ii = 0; ii < IT; ii++)
      xi[ii] = (i0 + ii < Ci) ? __ldg(xh + ((size_t)b * Ci + i0 + ii) * Kt + k) : make_float2(0.f, 0.f);
#pragma unroll
    for (int oo = 0; oo < OT; oo++)
      go[oo] = (o0 + oo < Co) ? __ldg(gyh + ((size_t)b * Co + o0 + oo) * Kt + k) : make_float2(0.f, 0.f);
#pragma unroll
    for (int ii = 0; ii < IT; ii++)
#pragma unroll
      for (int oo = 0; oo < OT; oo++) {
        // conj(xi) * go
        acc[ii][oo].x = fmaf(xi[ii].x, go[oo].x, fmaf(xi[ii].y, go[oo].y, acc[ii][oo].x));
        acc[ii][oo].y = fmaf(xi[ii].x, go[oo].y, fmaf(-xi[ii].y, go[oo].x, acc[ii][oo].y));
      }
  }
  float2* wbase = (float2*)w.corner[corner] + woff;
#pragma unroll
  for (int ii = 0; ii < IT; ii++)
#pragma unroll
    for (int oo = 0; oo < OT; oo++)
      if (i0 + ii < Ci && o0 + oo < Co) {
        float2* dst = wbase + (long)(i0 + ii) * w.stride_i + (long)(o0 + oo) * w.stride_o;
        float2 r = acc[ii][oo];
        if (accumulate) { const float2 old = *dst; r.x += old.x; r.y += old.y; }
        *dst = r;
      }
}

// Small batches (PINO: B = 4, 2048 modes, 64 x 64 channels -> 67 MB of dW per layer): the output is the traffic.  One block
// per (256 modes, input channel i); a thread decodes its mode ONCE, keeps conj(Xh[b, i, k]) in registers and walks the
// output channels, so every dW element costs BT loads (L2-resident gYh) + one coalesced store instead of a mode decode
// (eight integer divisions) per element as in k_dw2.
template <int BT>
__global__ void __launch_bounds__(256)
k_dw_small(const float2* __restrict__ xh, const float2* __restrict__ gyh, b2no_weights w, ModeMap mm, int B, int Ci, int Co,
           int Kt, int accumulate) {
  const int k = blockIdx.x * 256 + threadIdx.x;
  const int i = blockIdx.y;
  if (k >= Kt) return;
  int corner;
  long woff;
  decode_mode(mm, w, k, &corner, &woff);
  float2 xv[BT];
#pragma unroll
  for (int b = 0; b < BT; b++) xv[b] = b < B ? __ldg(xh + ((size_t)b * Ci + i) * Kt + k) : make_float2(0.f, 0.f);
  float2* dst = (float2*)w.corner[corner] + woff + (long)i * w.stride_i;
  const float2* gp = gyh + k;
  for (int o = 0; o < Co; o++) {
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int b = 0; b < BT; b++) {
      if (b < B) {
        const float2 gv = __ldg(gp + ((size_t)b * Co + o) * Kt);
        acc.x = fmaf(xv[b].x, gv.x, fmaf(xv[b].y, gv.y, acc.x));
        acc.y = fmaf(xv[b].x, gv.y, fmaf(-xv[b].y, gv.x, acc.y));
      }
    }
    float2* d = dst + (long)o * w.stride_o;
    if (accumulate) { const float2 old = *d; acc.x += old.x; acc.y += old.y; }
    *d = acc;
  }
}

extern "C" int b2no_mix_dw(const b2no_plan* p, const float* xh, const float* gyh, const b2no_weights* dw,
                           int batch, int ci, int co, int accumulate, void* stream) {
  if (!p || !xh || !gyh || !dw || batch < 1 || ci < 1 || co < 1) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int Kt = total_modes(p);
  const ModeMap mm = make_mode_map(p);
  {
    const int rc = b2no_tc_mix_dw(p, xh, gyh, dw, batch, ci, co, accumulate, st);
    if (rc != 1) return rc;
  }
  if (p->g.spec_layout != 0) return B2NO_E_UNSUPPORTED;
  if (batch <= 8 && Kt >= 256) {
    dim3 grid((unsigned)((Kt + 255) / 256), (unsigned)ci);
    if (batch <= 4)
      k_dw_small<4><<<grid, 256, 0, st>>>((const float2*)xh, (const float2*)gyh, *dw, mm, batch, ci, co, Kt, accumulate);
    else
      k_dw_small<8><<<grid, 256, 0, st>>>((const float2*)xh, (const float2*)gyh, *dw, mm, batch, ci, co, Kt, accumulate);
    B2NO_LAUNCH_CHECK();
    return 0;
  }
  const long total = (long)ci * co * Kt;
  k_dw2<<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const float2*)xh, (const float2*)gyh, *dw, mm, batch, ci, co, Kt, accumulate);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// =============================================================================================
// k_c2r_fused: last inverse stage + epilogue.  One warp per (batch, row, n-chunk, o-tile) item; lane l
// owns n = nbase + l + 32 j.  The inverse table [q][n] and the (transposed, zero-padded) 1x1 weights sit
// in shared memory; Bq values are warp-uniform loads.
// =============================================================================================
struct EpiDev {
  const float* bias;
  const float* pw_w; const float* pw_x; int pw_ci; int pw_t;
  const float* pw2_w; const float* pw2_x; int pw2_ci; int pw2_t;
  const float* add;
  const float* mul;
  float* preact;
  int act;
  const float* dz;
  int dact;
  const float* gate_z; const float* gate_h;
  long mul_bs, gate_bs;     // floats between consecutive samples of mul / gate_z (channel slices of a wider tensor)
};

template <int NPT, int OT>
__global__ void __launch_bounds__(256)
k_c2r_fused(const float2* __restrict__ spec, float* __restrict__ y, const float* __restrict__ tab, EpiDev e,
            int B, int Co, long RPI, int N, long P, int Kd, int npad) {
  extern __shared__ float smem[];
  const int n_ot = (Co + OT - 1) / OT;
  const int copad = n_ot * OT;
  const int q2 = spec ? 2 * Kd : 0;
  float* s_tab = smem;                            // [q2][npad]
  float* s_w1 = s_tab + (size_t)q2 * npad;        // [ci1][copad]
  float* s_w2 = s_w1 + (size_t)e.pw_ci * copad;   // [ci2][copad]
  for (int i = threadIdx.x; i < q2 * npad; i += blockDim.x) s_tab[i] = tab[i];
  for (int i = threadIdx.x; i < e.pw_ci * copad; i += blockDim.x) {
    const int ci = i / copad, o = i - ci * copad;
    float v = 0.f;
    if (o < Co) v = e.pw_t ? e.pw_w[(size_t)ci * Co + o] : e.pw_w[(size_t)o * e.pw_ci + ci];
    s_w1[i] = v;
  }
  for (int i = threadIdx.x; i < e.pw2_ci * copad; i += blockDim.x) {
    const int ci = i / copad, o = i - ci * copad;
    float v = 0.f;
    if (o < Co) v = e.pw2_t ? e.pw2_w[(size_t)ci * Co + o] : e.pw2_w[(size_t)o * e.pw2_ci + ci];
    s_w2[i] = v;
  }
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_nc = (N + 32 * NPT - 1) / (32 * NPT);
  const long n_items = (long)B * RPI * n_nc * n_ot;
  const bool plain = !e.add && !e.preact && !e.mul && !e.dz && !e.gate_z && e.act == B2NO_ACT_NONE;
  for (long item = (long)blockIdx.x * 8 + warp; item < n_items; item += (long)gridDim.x * 8) {
    const int ot = (int)(item % n_ot);
    long t = item / n_ot;
    const int nc = (int)(t % n_nc);
    t /= n_nc;
    const long r = t % RPI;
    const int b = (int)(t / RPI);
    const int o0 = ot * OT;
    const int nbase = nc * 32 * NPT;

    float acc[OT][NPT];
#pragma unroll
    for (int oo = 0; oo < OT; oo++)
#pragma unroll
      for (int j = 0; j < NPT; j++) acc[oo][j] = 0.f;

    if (spec) {
      const float2* sp = spec + (((size_t)b * Co + o0) * RPI + r) * Kd;
      const size_t ostride = (size_t)RPI * Kd;
      for (int k = 0; k < Kd; k++) {
        float tr[NPT], ti[NPT];
#pragma unroll
        for (int j = 0; j < NPT; j++) {
          const int n = nbase + lane + 32 * j;  // < npad by construction (npad multiple of 128)
          tr[j] = s_tab[(size_t)(2 * k) * npad + n];
          ti[j] = s_tab[(size_t)(2 * k + 1) * npad + n];
        }
#pragma unroll
        for (int oo = 0; oo < OT; oo++) {
          if (o0 + oo < Co) {
            const float2 v = __ldg(sp + oo * ostride + k);
#pragma unroll
            for (int j = 0; j < NPT; j++) acc[oo][j] = fmaf(v.x, tr[j], fmaf(v.y, ti[j], acc[oo][j]));
          }
        }
      }
    }
    bool valid[NPT];
    long pix[NPT];
#pragma unroll
    for (int j = 0; j < NPT; j++) {
      const int n = nbase + lane + 32 * j;
      pix[j] = r * N + n;
      valid[j] = (n < N) && (pix[j] < P);
    }
    if (e.pw_ci > 0) {
      const float* xb = e.pw_x + (size_t)b * e.pw_ci * P;
      for (int i = 0; i < e.pw_ci; i++) {
        float xv[NPT];
#pragma unroll
        for (int j = 0; j < NPT; j++) xv[j] = valid[j] ? __ldg(xb + (size_t)i * P + pix[j]) : 0.f;
        const float* wr = s_w1 + (size_t)i * copad + o0;
#pragma unroll
        for (int oo = 0; oo < OT; oo++) {
          const float wv = wr[oo];
#pragma unroll
          for (int j = 0; j < NPT; j++) acc[oo][j] = fmaf(wv, xv[j], acc[oo][j]);
        }
      }
    }
    if (e.pw2_ci > 0) {
      const float* xb = e.pw2_x + (size_t)b * e.pw2_ci * P;
      for (int i = 0; i < e.pw2_ci; i++) {
        float xv[NPT];
#pragma unroll
        for (int j = 0; j < NPT; j++) xv[j] = valid[j] ? __ldg(xb + (size_t)i * P + pix[j]) : 0.f;
        const float* wr = s_w2 + (size_t)i * copad + o0;
#pragma unroll
        for (int oo = 0; oo < OT; oo++) {
          const float wv = wr[oo];
#pragma unroll
          for (int j = 0; j < NPT; j++) acc[oo][j] = fmaf(wv, xv[j], acc[oo][j]);
        }
      }
    }
#pragma unroll
    for (int oo = 0; oo < OT; oo++) {
      const int o = o0 + oo;
      if (o < Co) {
        const float bv = e.bias ? __ldg(e.bias + o) : 0.f;
        if (plain) {
          // transform (+ bias) only: one add and one store per output.  (The generic epilogue below costs ~120 instructions
          // per output -- pointer tests, 64-bit index arithmetic, the activation switch -- and made the 3-D last stage
          // instruction-bound: 1.13 ms for 306 MB, ncu profiles/r02_d_ncu_pino_c2r.txt.)
          float* yr = y + ((size_t)b * Co + o) * P + (size_t)r * N + nbase + lane;
#pragma unroll
          for (int j = 0; j < NPT; j++)
            if (valid[j]) yr[32 * j] = acc[oo][j] + bv;
          continue;
        }
#pragma unroll
        for (int j = 0; j < NPT; j++) {
          if (valid[j]) {
            const size_t idx = ((size_t)b * Co + o) * P + pix[j];
            float z = acc[oo][j] + bv;
            if (e.add) z += __ldg(e.add + idx);
            if (e.preact) e.preact[idx] = z;
            float v = b2no_act(z, e.act);
            const size_t inner = (size_t)o * P + pix[j];
            if (e.mul) v *= __ldg(e.mul + (size_t)b * e.mul_bs + inner);
            if (e.dz) v *= b2no_act_grad(__ldg(e.dz + idx), e.dact);
            if (e.gate_z) v = fmaf(1.0f - __ldg(e.gate_z + (size_t)b * e.gate_bs + inner), __ldg(e.gate_h + idx), v);
            y[idx] = v;
          }
        }
      }
    }
  }
}

template <int NPT, int OT>
static int launch_c2r(const float2* spec, float* y, const float* tab, const EpiDev& e, int B, int Co, long RPI,
                      int N, long P, int Kd, int npad, cudaStream_t st) {
  const int n_ot = (Co + OT - 1) / OT;
  const int copad = n_ot * OT;
  const size_t smem = ((size_t)(spec ? 2 * Kd : 0) * npad + (size_t)(e.pw_ci + e.pw2_ci) * copad) * sizeof(float);
  if (smem > 200 * 1024) return B2NO_E_UNSUPPORTED;
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_c2r_fused<NPT, OT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_nc = (N + 32 * NPT - 1) / (32 * NPT);
  const long n_items = (long)B * RPI * n_nc * n_ot;
  long blocks = (n_items + 7) / 8;
  const long cap = (long)b2no_sm_count() * 4;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_c2r_fused<NPT, OT><<<(unsigned)blocks, 256, smem, st>>>(spec, y, tab, e, B, Co, RPI, N, P, Kd, npad);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// =============================================================================================
// k_c2r_plain: the last inverse stage alone (+ bias) for K_last = 8 kept modes -- the PINO layer, whose 1x1 conv and
// activation run on the tensor-core tile kernel.  Same item decomposition as k_c2r_fused (warp = one row x 16 channels),
// but the item's 16 x 8 spectrum values are fetched with FOUR coalesced loads per lane (each value once per warp, the
// next item's loads issued before this item's arithmetic) and handed round by shuffles, instead of 128 warp-uniform
// loads in eight dependent rounds: ncu showed the fused kernel latency-bound at 30 % issue utilisation, 0.8 TB/s.
// =============================================================================================
template <int NPT>
__global__ void __launch_bounds__(256)
k_c2r_plain8(const float2* __restrict__ spec, float* __restrict__ y, const float* __restrict__ tab,
             const float* __restrict__ bias, int B, int Co, long RPI, int N, long P, int npad) {
  constexpr int OT = 16, KD = 8;
  extern __shared__ float s_tab8[];                   // [2 KD][npad]
  for (int i = threadIdx.x; i < 2 * KD * npad; i += blockDim.x) s_tab8[i] = tab[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_ot = (Co + OT - 1) / OT;
  const int n_nc = (N + 32 * NPT - 1) / (32 * NPT);
  const long n_items = (long)B * RPI * n_nc * n_ot;
  const size_t ostride = (size_t)RPI * KD;
  auto fetch = [&](long item, float2 (&v)[4]) {
    const int ot = (int)(item % n_ot);
    long t = item / n_ot / n_nc;
    const long r = t % RPI;
    const int b = (int)(t / RPI);
    const float2* sp = spec + (((size_t)b * Co + ot * OT) * RPI + r) * KD;
#pragma unroll
    for (int m = 0; m < 4; m++) {
      const int idx = lane + 32 * m, oo = idx >> 3, k = idx & 7;
      v[m] = (ot * OT + oo < Co) ? __ldg(sp + oo * ostride + k) : make_float2(0.f, 0.f);
    }
  };
  long item = (long)blockIdx.x * 8 + warp;
  const long step = (long)gridDim.x * 8;
  float2 cur[4], nxt[4];
  if (item < n_items) fetch(item, cur);
  for (; item < n_items; item += step) {
    if (item + step < n_items) fetch(item + step, nxt);
    const int ot = (int)(item % n_ot);
    long t = item / n_ot;
    const int nc = (int)(t % n_nc);
    t /= n_nc;
    const long r = t % RPI;
    const int b = (int)(t / RPI);
    const int o0 = ot * OT, nbase = nc * 32 * NPT;
    float acc[OT][NPT];
#pragma unroll
    for (int oo = 0; oo < OT; oo++)
#pragma unroll
      for (int j = 0; j < NPT; j++) acc[oo][j] = 0.f;
#pragma unroll
    for (int k = 0; k < KD; k++) {
      float tr[NPT], ti[NPT];
#pragma unroll
      for (int j = 0; j < NPT; j++) {
        const int n = nbase + lane + 32 * j;            // < npad by construction
        tr[j] = s_tab8[(size_t)(2 * k) * npad + n];
        ti[j] = s_tab8[(size_t)(2 * k + 1) * npad + n];
      }
#pragma unroll
      for (int oo = 0; oo < OT; oo++) {
        const int idx = oo * KD + k;
        const float vx = __shfl_sync(0xffffffffu, cur[idx >> 5].x, idx & 31);
        const float vy = __shfl_sync(0xffffffffu, cur[idx >> 5].y, idx & 31);
#pragma unroll
        for (int j = 0; j < NPT; j++) acc[oo][j] = fmaf(vx, tr[j], fmaf(vy, ti[j], acc[oo][j]));
      }
    }
#pragma unroll
    for (int oo = 0; oo < OT; oo++) {
      const int o = o0 + oo;
      if (o < Co) {
        const float bv = bias ? __ldg(bias + o) : 0.f;
        float* yr = y + ((size_t)b * Co + o) * P + (size_t)r * N + nbase + lane;
#pragma unroll
        for (int j = 0; j < NPT; j++) {
          const int n = nbase + lane + 32 * j;
          if (n < N) yr[32 * j] = acc[oo][j] + bv;
        }
      }
    }
#pragma unroll
    for (int m = 0; m < 4; m++) cur[m] = nxt[m];
  }
}

template <int NPT>
static int launch_c2r_plain8(const float2* spec, float* y, const float* tab, const float* bias, int B, int Co, long RPI,
                             int N, long P, int npad, cudaStream_t st) {
  const size_t smem = (size_t)16 * npad * sizeof(float);
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_c2r_plain8<NPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_ot = (Co + 15) / 16, n_nc = (N + 32 * NPT - 1) / (32 * NPT);
  const long n_items = (long)B * RPI * n_nc * n_ot;
  long blocks = (n_items + 7) / 8;
  const long cap = (long)b2no_sm_count() * 6;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  k_c2r_plain8<NPT><<<(unsigned)blocks, 256, smem, st>>>(spec, y, tab, bias, B, Co, RPI, N, P, npad);
  B2NO_LAUNCH_CHECK();
  return 0;
}

static int run_c2r(const float2* spec, float* y, const float* tab, const EpiDev& e, int B, int Co, long RPI, int N,
                   long P, int Kd, int npad, cudaStream_t st) {
  constexpr int OT = 16;
  const bool plain = !e.add && !e.preact && !e.mul && !e.dz && !e.gate_z && e.act == B2NO_ACT_NONE;
  if (spec && plain && e.pw_ci == 0 && e.pw2_ci == 0 && Kd == 8 && npad * 16 * 4 <= 160 * 1024) {
    if (N <= 32) return launch_c2r_plain8<1>(spec, y, tab, e.bias, B, Co, RPI, N, P, npad, st);
    if (N <= 64) return launch_c2r_plain8<2>(spec, y, tab, e.bias, B, Co, RPI, N, P, npad, st);
    if (N <= 96) return launch_c2r_plain8<3>(spec, y, tab, e.bias, B, Co, RPI, N, P, npad, st);
    if (N <= 128) return launch_c2r_plain8<4>(spec, y, tab, e.bias, B, Co, RPI, N, P, npad, st);
  }
  if (N <= 32) return launch_c2r<1, OT>(spec, y, tab, e, B, Co, RPI, N, P, Kd, npad, st);
  if (N <= 64) return launch_c2r<2, OT>(spec, y, tab, e, B, Co, RPI, N, P, Kd, npad, st);
  if (N <= 96) return launch_c2r<3, OT>(spec, y, tab, e, B, Co, RPI, N, P, Kd, npad, st);
  return launch_c2r<4, OT>(spec, y, tab, e, B, Co, RPI, N, P, Kd, npad, st);
}

// Mode-major spectra (b2no_geom.spec_layout = 1) live on the tensor-core kernels only: every call the RNO layer makes with
// base width `channels` (mixing C -> C, C -> 2C, 2C -> C and their weight gradients, transforms of C and 2C channel tensors)
// must be eligible, otherwise the caller keeps the default layout.
extern "C" int b2no_plan_layout_supported(const b2no_plan* p, int64_t batch, int64_t channels) {
  if (!p || batch < 1 || channels < 1) return 0;
  if (p->g.spec_layout == 0) return 1;
  if (!b2no_tc_available() || p->g.ndim != 2) return 0;
  if (!p->tcf[0].tb || !p->tcf[1].tb || !p->tc[0].timg || !p->tc[1].timg) return 0;
  if (((long)p->g.nin[0] * p->g.nin[1]) % 128 != 0 || ((long)p->g.nout[0] * p->g.nout[1]) % 128 != 0) return 0;
  if (p->K[0] > 32) return 0;
  if (((size_t)2 * channels * ((size_t)p->K[0] * p->K[1] + 1) + (size_t)p->K[0] * 32) * 8 > 200 * 1024) return 0;   // k_inv_h staging
  const int c = (int)channels, b = (int)(batch > 1 << 30 ? 1 << 30 : batch);
  return b2no_tc_mix_feasible(b, c, c, 0) && b2no_tc_mix_feasible(b, c, 2 * c, 0) && b2no_tc_mix_feasible(b, c, 2 * c, 1) &&
         b2no_tc_mix_dw_feasible(b, c, c) && b2no_tc_mix_dw_feasible(b, c, 2 * c);
}

// n x n identity matrices on the device, one per (device, n), created on first use (never inside a graph capture: the
// first call of every shape is an eager warm-up, as for the plans) and kept for the life of the process
__global__ void k_fill_identity(float* m, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n * n) m[i] = (i / n == i % n) ? 1.0f : 0.0f;
}
static const float* identity_matrix(int n, cudaStream_t st) {
  static float* cache[8][129] = {};
  int dev = 0;
  if (n < 1 || n > 128 || cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 8) return nullptr;
  if (!cache[dev][n]) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return nullptr;
    float* m = nullptr;
    if (cudaMalloc(&m, (size_t)n * n * sizeof(float)) != cudaSuccess) return nullptr;
    k_fill_identity<<<(n * n + 255) / 256, 256, 0, st>>>(m, n);
    if (cudaGetLastError() != cudaSuccess) { cudaFree(m); return nullptr; }
    cache[dev][n] = m;
  }
  return cache[dev][n];
}

extern "C" int b2no_dft_inverse(const b2no_plan* p, int which, const float* spec, float* y, float* work,
                                int batch, int channels, int64_t pixels, const b2no_epilogue* epi, void* stream) {
  if (!y || batch < 1 || channels < 1 || (which != 0 && which != 1)) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  EpiDev e;
  memset(&e, 0, sizeof(e));
  if (epi) {
    e.bias = epi->bias;
    e.pw_w = epi->pw_w; e.pw_x = epi->pw_x; e.pw_ci = (epi->pw_w && epi->pw_x) ? epi->pw_ci : 0; e.pw_t = epi->pw_transposed;
    e.pw2_w = epi->pw2_w; e.pw2_x = epi->pw2_x; e.pw2_ci = (epi->pw2_w && epi->pw2_x) ? epi->pw2_ci : 0; e.pw2_t = epi->pw2_transposed;
    e.add = epi->add; e.mul = epi->mul; e.preact = epi->preact; e.act = epi->act;
    e.dz = epi->dact_z; e.dact = epi->dact_z ? epi->dact : 0;
    e.gate_z = (epi->gate_z && epi->gate_h) ? epi->gate_z : nullptr; e.gate_h = e.gate_z ? epi->gate_h : nullptr;
    if (e.pw_ci < 0 || e.pw2_ci < 0 || epi->mul_bstride < 0 || epi->gate_bstride < 0) return B2NO_E_ARG;
  }
  // tensor-core tile kernel when the shape is eligible (tc_pointwise.cu); otherwise the CUDA-core kernels below
  if (epi && (spec == nullptr || (p && p->g.ndim == 2))) {
    long px = pixels;
    if (spec && p) {
      const int32_t* nn = which == 0 ? p->g.nout : p->g.nin;
      px = (long)nn[0] * nn[1];
      if (pixels > 0 && pixels != px) return B2NO_E_ARG;
    }
    const int rc = b2no_tc_pointwise(p, which, spec, y, work, batch, channels, px, epi, st);
    if (rc != 1) return rc;
  }
  if (spec && p && p->g.spec_layout != 0) return B2NO_E_UNSUPPORTED;
  auto set_strides = [&](long P_) {
    e.mul_bs = (epi && epi->mul_bstride) ? (long)epi->mul_bstride : (long)channels * P_;
    e.gate_bs = (epi && epi->gate_bstride) ? (long)epi->gate_bstride : (long)channels * P_;
  };
  if (!spec) {
    // pure pointwise op on a flattened grid
    if (pixels < 1) return B2NO_E_ARG;
    set_strides(pixels);
    const int N = 128;
    const long RPI = (pixels + N - 1) / N;
    return run_c2r(nullptr, y, nullptr, e, batch, channels, RPI, N, pixels, 0, 128, st);
  }
  if (!p) return B2NO_E_ARG;
  const int d = p->g.ndim;
  const int32_t* n = which == 0 ? p->g.nout : p->g.nin;
  const int Kl = p->K[d - 1];
  const float* tab = which == 0 ? p->t_out : p->t_in;
  const int npad = which == 0 ? p->npad_out : p->npad_in;
  const long bc = (long)batch * channels;
  long P = 1;
  for (int j = 0; j < d; j++) P *= n[j];
  if (pixels > 0 && pixels != P) return B2NO_E_ARG;
  set_strides(P);
  if (d == 1) return run_c2r((const float2*)spec, y, tab, e, batch, channels, 1, n[0], P, Kl, npad, st);
  if (!work) return B2NO_E_ARG;
  float2* A = (float2*)work;
  if (d == 2) {
    const float2* T = which == 0 ? p->m_inv[0] : p->m_adjfwd[0];
    int rc = run_cmat((const float2*)spec, A, T, bc, p->K[0], n[0], Kl, st);
    if (rc) return rc;
    return run_c2r(A, y, tab, e, batch, channels, n[0], n[1], P, Kl, npad, st);
  }
  float2* Bb = A + (size_t)bc * n[0] * n[1] * Kl;
  const float2* T0 = which == 0 ? p->m_inv[0] : p->m_adjfwd[0];
  int rc = run_cmat((const float2*)spec, Bb, T0, bc, p->K[0], n[0], p->K[1] * Kl, st);
  if (rc) return rc;
  // 3-D, fused: the middle-dim stage writes the row image (k_inv_h) and the tile kernel does the last dim itself, with a
  // per-tile T operand built by its converter warps -- the transform's result never exists in HBM (this replaced the
  // k_c2r_plain8 pass + the T round trip below: 1.5 ms + 0.4 ms of the 9.6 ms PINO step).
  if (epi && e.pw_ci > 0 && b2no_tc_available() && P % 128 == 0) {
    float* img = work + 2 * ((size_t)bc * n[0] * n[1] * Kl + (size_t)bc * n[0] * p->K[1] * Kl) + (size_t)bc * P;
    const int rc3 = b2no_tc_pointwise(p, which, (const float*)Bb, y, img, batch, channels, P, epi, st);
    if (rc3 != 1) return rc3;
  }
  const float2* T1 = which == 0 ? p->m_inv[1] : p->m_adjfwd[1];
  rc = run_cmat(Bb, A, T1, bc * n[0], p->K[1], n[1], Kl, st);
  if (rc) return rc;
  // 3-D (PINO, basics.py:114-143 + pinobserver.py:222-226): the last transform stage is 2 K_last FMAs per output, the 1x1
  // convolution next to it Ci of them -- the convolution (+ bias, activation, saved pre-activation) goes to the tensor-core
  // tile kernel as a pure pointwise op, with the transform's result T entering through `add`:
  //     T = irfft_last(stage) (CUDA cores, no epilogue)      y = epilogue(W x + bias + T) (tcgen05, k_pw_tc)
  // (the tile kernel's own last-stage operand needs pixel tiles that are whole rows; 73-point rows are not)
  if (epi && e.pw_ci > 0 && !e.add && b2no_tc_available() && P % 128 == 0) {
    float* T = (float*)(Bb + (size_t)bc * n[0] * p->K[1] * Kl);
    EpiDev e0;
    memset(&e0, 0, sizeof(e0));
    rc = run_c2r(A, T, tab, e0, batch, channels, (long)n[0] * n[1], n[2], P, Kl, npad, st);
    if (rc) return rc;
    b2no_epilogue epi2 = *epi;
    // T enters the tile kernel as a SECOND 1x1 operand with identity weights when that slot is free: it then arrives
    // through the TMA ring like x and is added by the tensor core, and the specialised epilogues (bias / GELU + saved
    // pre-activation) stay eligible.  Through `add` it would take the generic epilogue, whose per-thread loads held the
    // PINO layer at 2.4 TB/s (499 us per pass, profiles/r02_c_pino_step_breakdown.txt).
    const float* ident = (!epi->pw2_w && channels <= 128) ? identity_matrix(channels, st) : nullptr;
    if (ident) {
      epi2.pw2_w = ident; epi2.pw2_x = T; epi2.pw2_ci = channels; epi2.pw2_transposed = 0;
    } else {
      epi2.add = T;
    }
    rc = b2no_tc_pointwise(nullptr, which, nullptr, y, nullptr, batch, channels, P, &epi2, st);
    if (rc == 1 && ident) {                    // shape without the two-operand tile kernel: T through `add` instead
      epi2 = *epi;
      epi2.add = T;
      rc = b2no_tc_pointwise(nullptr, which, nullptr, y, nullptr, batch, channels, P, &epi2, st);
    }
    if (rc != 1) return rc;
    EpiDev e2 = e;
    e2.add = T;
    return run_c2r(nullptr, y, nullptr, e2, batch, channels, (P + 127) / 128, 128, P, 0, 128, st);
  }
  return run_c2r(A, y, tab, e, batch, channels, (long)n[0] * n[1], n[2], P, Kl, npad, st);
}
