// Pointwise / reduction kernels around the spectral convolution: activation backward, 1x1-conv weight
// gradient, fused projection head, RNO gate, relative-L2 loss.  All HBM-bound except the head.
#include "common.cuh"

static inline long grid_for(long n, int threads, int per_sm) {
  long blocks = (n + threads - 1) / threads;
  const long cap = (long)b2no_sm_count() * per_sm;
  if (blocks > cap) blocks = cap;
  return blocks < 1 ? 1 : blocks;
}

// ---------------------------------------------------------------------------------------------
// gz = gy * act'(z)     128-bit vectorised, grid-stride
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_act_bwd(const float* __restrict__ gy, const float* __restrict__ z, float* __restrict__ gz, long n, int act) {
  const long n4 = n >> 2;
  const long stride = (long)gridDim.x * blockDim.x;
  const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const float4* g4 = reinterpret_cast<const float4*>(gy);
  const float4* z4 = reinterpret_cast<const float4*>(z);
  float4* o4 = reinterpret_cast<float4*>(gz);
  for (long i = tid; i < n4; i += stride) {
    const float4 g = __ldg(g4 + i), zz = __ldg(z4 + i);
    float4 o;
    o.x = g.x * b2no_act_grad(zz.x, act);
    o.y = g.y * b2no_act_grad(zz.y, act);
    o.z = g.z * b2no_act_grad(zz.z, act);
    o.w = g.w * b2no_act_grad(zz.w, act);
    o4[i] = o;
  }
  for (long i = (n4 << 2) + tid; i < n; i += stride) gz[i] = gy[i] * b2no_act_grad(z[i], act);
}

extern "C" int b2no_act_bwd(const float* gy, const float* z, float* gz, int64_t n, int act, void* stream) {
  if (!gy || !z || !gz || n < 0) return B2NO_E_ARG;
  if (n == 0) return 0;
  if (((uintptr_t)gy | (uintptr_t)z | (uintptr_t)gz) & 15) return B2NO_E_ARG;
  k_act_bwd<<<(unsigned)grid_for((n + 3) / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(gy, z, gz, n, act);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// 1x1-conv weight gradient: dW[o,i] = sum_{b,p} g[b,o,p] x[b,i,p],  db[o] = sum g.
// Block = 256 threads.  Tiles of TP pixels are staged as [channel][TP+4] in shared memory; thread
// (to, ti) owns outputs o = to + a*T_O, i = ti + c*T_I (a,c < 4) and reads float4 over 4 pixels.
// Threads are split into pixel groups; per-block partials go to `partial`, a second kernel sums them
// (deterministic, no atomics).
// ---------------------------------------------------------------------------------------------
#define WG_TP 64
#define WG_TPP (WG_TP + 4)

__global__ void __launch_bounds__(256)
k_pw_wgrad(const float* __restrict__ g, const float* __restrict__ x, float* __restrict__ partial, int B, int Ci,
           int Co, long P, int o_per_block, int tiles_o, int tiles_i, int has_db) {
  extern __shared__ float smem[];
  float* gs = smem;                               // [o_per_block][WG_TPP]
  float* xs = gs + (size_t)o_per_block * WG_TPP;  // [Ci][WG_TPP]
  const int ob0 = blockIdx.y * o_per_block;
  const int nt = tiles_o * tiles_i;               // thread tiles (<= 256)
  const int groups = 256 / nt;                    // pixel groups
  const int tid = threadIdx.x;
  const int grp = tid / nt, tile = tid - grp * nt;
  const int to = tile / tiles_i, ti = tile - to * tiles_i;
  const bool active = grp < groups;
  const int px_per_grp = WG_TP / 4 / groups;      // float4 columns per group (may be 0 -> handled below)

  float acc[4][4];
  float accb[4];
#pragma unroll
  for (int a = 0; a < 4; a++) {
    accb[a] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; c++) acc[a][c] = 0.f;
  }

  const long chunks_per_img = (P + WG_TP - 1) / WG_TP;
  const long n_chunks = (long)B * chunks_per_img;
  for (long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    const int b = (int)(ch / chunks_per_img);
    const long p0 = (ch - (long)b * chunks_per_img) * WG_TP;
    __syncthreads();
    for (int idx = tid; idx < o_per_block * WG_TP; idx += 256) {
      const int c = idx / WG_TP, pp = idx - c * WG_TP;
      const int o = ob0 + c;
      gs[c * WG_TPP + pp] = (o < Co && p0 + pp < P) ? __ldg(g + ((size_t)b * Co + o) * P + p0 + pp) : 0.f;
    }
    for (int idx = tid; idx < Ci * WG_TP; idx += 256) {
      const int c = idx / WG_TP, pp = idx - c * WG_TP;
      xs[c * WG_TPP + pp] = (p0 + pp < P) ? __ldg(x + ((size_t)b * Ci + c) * P + p0 + pp) : 0.f;
    }
    __syncthreads();
    if (active) {
      // this group's float4 columns: q = grp, grp + groups, ...
      for (int q = grp; q < WG_TP / 4; q += groups) {
        float4 gv[4], xv[4];
#pragma unroll
        for (int a = 0; a < 4; a++) {
          const int o = to + a * tiles_o;
          gv[a] = (o < o_per_block) ? *reinterpret_cast<const float4*>(gs + o * WG_TPP + 4 * q)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int c = 0; c < 4; c++) {
          const int i = ti + c * tiles_i;
          xv[c] = (i < Ci) ? *reinterpret_cast<const float4*>(xs + i * WG_TPP + 4 * q)
                           : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int a = 0; a < 4; a++) {
#pragma unroll
          for (int c = 0; c < 4; c++) {
            acc[a][c] = fmaf(gv[a].x, xv[c].x, acc[a][c]);
            acc[a][c] = fmaf(gv[a].y, xv[c].y, acc[a][c]);
            acc[a][c] = fmaf(gv[a].z, xv[c].z, acc[a][c]);
            acc[a][c] = fmaf(gv[a].w, xv[c].w, acc[a][c]);
          }
          if (ti == 0) accb[a] += (gv[a].x + gv[a].y) + (gv[a].z + gv[a].w);
        }
      }
    }
  }
  (void)px_per_grp;
  // reduce the pixel groups through shared memory, then write this block's partial
  __syncthreads();
  float* red = smem;  // reuse: [groups][nt][20]
  if (active) {
    float* dst = red + ((size_t)grp * nt + tile) * 20;
#pragma unroll
    for (int a = 0; a < 4; a++) {
#pragma unroll
      for (int c = 0; c < 4; c++) dst[a * 4 + c] = acc[a][c];
      dst[16 + a] = accb[a];
    }
  }
  __syncthreads();
  const size_t pstride = (size_t)Co * Ci + Co;
  float* pout = partial + (size_t)blockIdx.x * pstride;
  if (grp == 0) {
    float s[20];
#pragma unroll
    for (int v = 0; v < 20; v++) s[v] = 0.f;
    for (int gq = 0; gq < groups; gq++) {
      const float* src = red + ((size_t)gq * nt + tile) * 20;
#pragma unroll
      for (int v = 0; v < 20; v++) s[v] += src[v];
    }
#pragma unroll
    for (int a = 0; a < 4; a++) {
      const int ol = to + a * tiles_o;
      const int o = ob0 + ol;
      if (ol < o_per_block && o < Co) {
#pragma unroll
        for (int c = 0; c < 4; c++) {
          const int i = ti + c * tiles_i;
          if (i < Ci) pout[(size_t)o * Ci + i] = s[a * 4 + c];
        }
        if (has_db && ti == 0) pout[(size_t)Co * Ci + o] = s[16 + a];
      }
    }
  }
}

// Deterministic sum of the per-CTA partials: a block owns 32 consecutive outputs; its 8 warps split the partials
// (each warp reads 128 contiguous bytes per partial, 4 independent loads in flight), then combine through shared memory
// in a fixed order.  (The one-thread-per-output loop it replaces was a 148-deep dependent load chain: 13 us.)
__global__ void __launch_bounds__(256)
k_pw_wgrad_reduce(const float* __restrict__ partial, float* __restrict__ dw, float* __restrict__ db, int nblk, int Ci, int Co) {
  __shared__ float red[8][33];
  const int n = Co * Ci + Co;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + lane;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (idx < n) {
    int b = warp;
    for (; b + 24 < nblk; b += 32) {
      s0 += __ldg(partial + (size_t)b * n + idx);
      s1 += __ldg(partial + (size_t)(b + 8) * n + idx);
      s2 += __ldg(partial + (size_t)(b + 16) * n + idx);
      s3 += __ldg(partial + (size_t)(b + 24) * n + idx);
    }
    for (; b < nblk; b += 8) s0 += __ldg(partial + (size_t)b * n + idx);
  }
  red[warp][lane] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (warp == 0 && idx < n) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; w8++) s += red[w8][lane];
    if (idx < Co * Ci) dw[idx] = s;
    else if (db) db[idx - Co * Ci] = s;
  }
}

static void wgrad_cfg(int ci, int co, int* tiles_i, int* tiles_o, int* o_per_block, int* gy) {
  *tiles_i = (ci + 3) / 4;
  int to_all = (co + 3) / 4;
  int max_to = 256 / *tiles_i;
  if (max_to < 1) max_to = 1;
  *tiles_o = to_all < max_to ? to_all : max_to;
  *o_per_block = *tiles_o * 4;
  *gy = (co + *o_per_block - 1) / *o_per_block;
}

static int wgrad_blocks_x() { return b2no_sm_count() * 2; }

extern "C" int64_t b2no_pw_wgrad_scratch_floats(int ci, int co) {
  if (ci < 1 || co < 1) return B2NO_E_ARG;
  return (int64_t)wgrad_blocks_x() * ((int64_t)co * ci + co);
}

extern "C" int b2no_pw_wgrad(const float* g, const float* x, float* dw, float* db, float* partial, int batch,
                             int ci, int co, int64_t pixels, void* stream) {
  if (!g || !x || !dw || !partial || batch < 1 || ci < 1 || co < 1 || pixels < 1) return B2NO_E_ARG;
  if (ci > 1024) return B2NO_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  {
    // tensor-core path (tc_wgrad.cu) when eligible: per-CTA partials, same deterministic reduction
    int nblk = 0;
    const int rc = b2no_tc_wgrad(g, x, partial, wgrad_blocks_x(), batch, ci, co, pixels, &nblk, st);
    if (rc == 0) {
      const int n = co * ci + co;
      k_pw_wgrad_reduce<<<(n + 31) / 32, 256, 0, st>>>(partial, dw, db, nblk, ci, co);
      B2NO_LAUNCH_CHECK();
      return 0;
    }
    if (rc != 1) return rc;
  }
  int tiles_i, tiles_o, opb, gy;
  wgrad_cfg(ci, co, &tiles_i, &tiles_o, &opb, &gy);
  const int nt = tiles_o * tiles_i;
  const int groups = 256 / nt;
  size_t smem = ((size_t)opb + ci) * WG_TPP * sizeof(float);
  const size_t red = (size_t)groups * nt * 20 * sizeof(float);
  if (red > smem) smem = red;
  if (smem > 200 * 1024) return B2NO_E_UNSUPPORTED;
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_pw_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long chunks = (long)batch * ((pixels + WG_TP - 1) / WG_TP);
  long bx = wgrad_blocks_x();
  if (bx > chunks) bx = chunks;
  // every block (x) writes a full partial for its o-range; blocks with different y write disjoint o's.
  B2NO_CHECK_CUDA(cudaMemsetAsync(partial, 0, (size_t)bx * ((size_t)co * ci + co) * sizeof(float), st));
  dim3 grid((unsigned)bx, (unsigned)gy);
  k_pw_wgrad<<<grid, 256, smem, st>>>(g, x, partial, batch, ci, co, pixels, opb, tiles_o, tiles_i, db ? 1 : 0);
  B2NO_LAUNCH_CHECK();
  const int n = co * ci + co;
  k_pw_wgrad_reduce<<<(n + 31) / 32, 256, 0, st>>>(partial, dw, db, (int)bx, ci, co);
  B2NO_LAUNCH_CHECK();
  return 0;
}

extern "C" int b2no_dft_inverse_wgrad(const b2no_plan* plan, int which, const float* spec, float* y, float* work, int batch,
                                     int channels, int64_t pixels, const b2no_epilogue* epi, const float* wg_x, int wg_ci,
                                     float* dw, float* db, float* partial, void* stream) {
  if (!plan || !spec || !y || !work || !epi || !wg_x || !dw || !partial || batch < 1 || channels < 1 || wg_ci < 1 ||
      (which != 0 && which != 1))
    return B2NO_E_ARG;
  if (!epi->pw_w || !epi->pw_x || epi->pw_ci < 1) return B2NO_E_ARG;
  if (plan->g.ndim != 2) return B2NO_E_UNSUPPORTED;
  const int32_t* n = which == 0 ? plan->g.nout : plan->g.nin;
  const long px = (long)n[0] * n[1];
  if (pixels > 0 && pixels != px) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int nblk = 0;
  const b2no_tc_wg wg = {wg_x, wg_ci, partial, &nblk};
  const int rc = b2no_tc_pointwise(plan, which, spec, y, work, batch, channels, px, epi, st, &wg);
  if (rc == 1) return B2NO_E_UNSUPPORTED;
  if (rc) return rc;
  const int co = epi->pw_ci, nw = co * wg_ci + co;
  k_pw_wgrad_reduce<<<(nw + 31) / 32, 256, 0, st>>>(partial, dw, db, nblk, wg_ci, co);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// fused projection head, out_channels == 1: two pixels per thread, W1 in shared memory
// ---------------------------------------------------------------------------------------------
template <int CI>
__global__ void __launch_bounds__(128)
k_mlp_head_fwd(const float* __restrict__ x, const float* __restrict__ w1, const float* __restrict__ b1,
               const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ out, int B,
               int hidden, long P, int b1_per_sample, int act) {
  extern __shared__ float smem[];
  float* w1s = smem;                          // [hidden][CI]
  float* w2s = w1s + (size_t)hidden * CI;     // [hidden]
  float* b1s = w2s + hidden;                  // [hidden]
  for (int i = threadIdx.x; i < hidden * CI; i += blockDim.x) w1s[i] = w1[i];
  for (int i = threadIdx.x; i < hidden; i += blockDim.x) w2s[i] = w2[i];
  const long chunks_per_img = (P + 255) / 256;
  const long n_chunks = (long)B * chunks_per_img;
  const float bias2 = b2 ? __ldg(b2) : 0.f;
  int cur_b = -1;
  for (long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    const int b = (int)(ch / chunks_per_img);
    const long p0 = (ch - (long)b * chunks_per_img) * 256;
    if (b != cur_b) {
      __syncthreads();
      for (int i = threadIdx.x; i < hidden; i += blockDim.x)
        b1s[i] = b1 ? (b1_per_sample ? b1[(size_t)b * hidden + i] : b1[i]) : 0.f;
      cur_b = b;
    }
    __syncthreads();
    const long pa = p0 + threadIdx.x, pb = pa + 128;
    const bool va = pa < P, vb = pb < P;
    float xa[CI], xb[CI];
    const float* xbase = x + (size_t)b * CI * P;
#pragma unroll
    for (int i = 0; i < CI; i++) {
      xa[i] = va ? __ldg(xbase + (size_t)i * P + pa) : 0.f;
      xb[i] = vb ? __ldg(xbase + (size_t)i * P + pb) : 0.f;
    }
    float oa = bias2, ob = bias2;
    for (int j = 0; j < hidden; j++) {
      const float4* wr = reinterpret_cast<const float4*>(w1s + (size_t)j * CI);
      float ha = b1s[j], hb = ha;
#pragma unroll
      for (int i4 = 0; i4 < CI / 4; i4++) {
        const float4 w = wr[i4];
        ha = fmaf(w.x, xa[4 * i4], ha); hb = fmaf(w.x, xb[4 * i4], hb);
        ha = fmaf(w.y, xa[4 * i4 + 1], ha); hb = fmaf(w.y, xb[4 * i4 + 1], hb);
        ha = fmaf(w.z, xa[4 * i4 + 2], ha); hb = fmaf(w.z, xb[4 * i4 + 2], hb);
        ha = fmaf(w.w, xa[4 * i4 + 3], ha); hb = fmaf(w.w, xb[4 * i4 + 3], hb);
      }
      const float w2v = w2s[j];
      oa = fmaf(w2v, b2no_act(ha, act), oa);
      ob = fmaf(w2v, b2no_act(hb, act), ob);
    }
    if (va) out[(size_t)b * P + pa] = oa;
    if (vb) out[(size_t)b * P + pb] = ob;
  }
}

template <int CI>
static int launch_head(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                       float* out, int B, int hidden, long P, int per_sample, int act, cudaStream_t st) {
  const size_t smem = ((size_t)hidden * CI + 2 * (size_t)hidden) * sizeof(float);
  if (smem > 200 * 1024) return B2NO_E_UNSUPPORTED;
  if (smem > 48 * 1024)
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_mlp_head_fwd<CI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long chunks = (long)B * ((P + 255) / 256);
  long blocks = chunks;
  const long cap = (long)b2no_sm_count() * 4;
  if (blocks > cap) blocks = cap;
  k_mlp_head_fwd<CI><<<(unsigned)blocks, 128, smem, st>>>(x, w1, b1, w2, b2, out, B, hidden, P, per_sample, act);
  B2NO_LAUNCH_CHECK();
  return 0;
}

extern "C" int b2no_mlp_head_fwd(const float* x, const float* w1, const float* b1, const float* w2,
                                 const float* b2, float* out, int batch, int ci, int hidden, int64_t pixels,
                                 int b1_per_sample, int act, void* stream) {
  if (!x || !w1 || !w2 || !out || batch < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  {
    // tensor-core fused MLP (tc_mlp.cu) when eligible
    const int rc = b2no_tc_mlp_fwd(x, w1, b1, w2, b2, out, batch, ci, hidden, 1, pixels, b1_per_sample, act, st);
    if (rc != 1) return rc;
  }
  switch (ci) {
    case 8: return launch_head<8>(x, w1, b1, w2, b2, out, batch, hidden, pixels, b1_per_sample, act, st);
    case 16: return launch_head<16>(x, w1, b1, w2, b2, out, batch, hidden, pixels, b1_per_sample, act, st);
    case 32: return launch_head<32>(x, w1, b1, w2, b2, out, batch, hidden, pixels, b1_per_sample, act, st);
    case 64: return launch_head<64>(x, w1, b1, w2, b2, out, batch, hidden, pixels, b1_per_sample, act, st);
  }
  return B2NO_E_UNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------
// RNO gate (rno.py:259)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_rno_gate_fwd(const float* __restrict__ z, const float* __restrict__ z2, const float* __restrict__ hh,
               const float* __restrict__ h, float* __restrict__ out, long n) {
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (1.0f - z[i]) * h[i] + z2[i] * hh[i];
}

__global__ void __launch_bounds__(256)
k_rno_gate_bwd(const float* __restrict__ g, const float* __restrict__ z, const float* __restrict__ z2,
               const float* __restrict__ hh, const float* __restrict__ h, float* __restrict__ gz,
               float* __restrict__ gz2, float* __restrict__ ghh, float* __restrict__ gh, long n) {
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gg = g[i];
    gz[i] = -gg * h[i];
    gz2[i] = gg * hh[i];
    ghh[i] = gg * z2[i];
    gh[i] = gg * (1.0f - z[i]);
  }
}

extern "C" int b2no_rno_gate_fwd(const float* z, const float* z2, const float* hhat, const float* h, float* out,
                                 int64_t n, void* stream) {
  if (!z || !z2 || !hhat || !h || !out || n < 0) return B2NO_E_ARG;
  if (n == 0) return 0;
  k_rno_gate_fwd<<<(unsigned)grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(z, z2, hhat, h, out, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}

extern "C" int b2no_rno_gate_bwd(const float* g, const float* z, const float* z2, const float* hhat,
                                 const float* h, float* gz, float* gz2, float* ghhat, float* gh, int64_t n,
                                 void* stream) {
  if (!g || !z || !z2 || !hhat || !h || !gz || !gz2 || !ghhat || !gh || n < 0) return B2NO_E_ARG;
  if (n == 0) return 0;
  k_rno_gate_bwd<<<(unsigned)grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(g, z, z2, hhat, h, gz, gz2, ghhat, gh, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Backward of the fused RNO cell update (the forward is the gate term of the inverse-transform epilogue): one pass
// reads g, h, z, z2, ah and writes the pre-activation gradients of the three branches plus the direct dh term,
// 128-bit vectorised (7 x 4 B per element: HBM-bound).  zz2 / g_zz2 are (batch, 2C, p): z in channels [0, C), z2 in [C, 2C).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_rno_cell_bwd(const float* __restrict__ g, const float* __restrict__ h, const float* __restrict__ zz2,
               const float* __restrict__ ah, float* __restrict__ g_zz2, float* __restrict__ g_ah, float* __restrict__ g_h,
               int B, long cp4) {
  // cp4 = C * p / 4 float4 per sample; element (b, i) of the C-channel tensors sits at b * cp4 + i, of the 2C-channel ones
  // at b * 2 cp4 + i (z) and b * 2 cp4 + cp4 + i (z2)
  const long total = (long)B * cp4;
  const long stride = (long)gridDim.x * blockDim.x;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  const float4* h4 = reinterpret_cast<const float4*>(h);
  const float4* z4 = reinterpret_cast<const float4*>(zz2);
  const float4* a4 = reinterpret_cast<const float4*>(ah);
  float4* oz4 = reinterpret_cast<float4*>(g_zz2);
  float4* oa4 = reinterpret_cast<float4*>(g_ah);
  float4* oh4 = reinterpret_cast<float4*>(g_h);
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const long b = t / cp4, i = t - b * cp4;
    const long iz = b * 2 * cp4 + i;
    const float4 gv = __ldg(g4 + t), hv = __ldg(h4 + t), zv = __ldg(z4 + iz), z2v = __ldg(z4 + iz + cp4), av = __ldg(a4 + t);
    float4 oz, oz2, oa, oh;
#define B2NO_CELL(c)                                                          \
    {                                                                         \
      const float hh = b2no_act(av.c, B2NO_ACT_SELU);                         \
      oz.c = -gv.c * hv.c * zv.c * (1.0f - zv.c);                             \
      oz2.c = gv.c * hh * z2v.c * (1.0f - z2v.c);                             \
      oa.c = gv.c * z2v.c * b2no_act_grad(av.c, B2NO_ACT_SELU);               \
      oh.c = gv.c * (1.0f - zv.c);                                            \
    }
    B2NO_CELL(x) B2NO_CELL(y) B2NO_CELL(z) B2NO_CELL(w)
#undef B2NO_CELL
    oz4[iz] = oz;
    oz4[iz + cp4] = oz2;
    oa4[t] = oa;
    oh4[t] = oh;
  }
}

// reset gate inside f6(r * h):  g_ar = g_rh h r (1 - r),  g_h += g_rh r,  r = sigmoid(ar)
__global__ void __launch_bounds__(256)
k_rno_reset_bwd(const float* __restrict__ g_rh, const float* __restrict__ h, const float* __restrict__ ar,
                float* __restrict__ g_ar, float* __restrict__ g_h, long n4) {
  const long stride = (long)gridDim.x * blockDim.x;
  const float4* g4 = reinterpret_cast<const float4*>(g_rh);
  const float4* h4 = reinterpret_cast<const float4*>(h);
  const float4* a4 = reinterpret_cast<const float4*>(ar);
  float4* o4 = reinterpret_cast<float4*>(g_ar);
  float4* gh4 = reinterpret_cast<float4*>(g_h);
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < n4; t += stride) {
    const float4 gv = __ldg(g4 + t), hv = __ldg(h4 + t), av = __ldg(a4 + t);
    float4 o, acc = gh4[t];
#define B2NO_RST(c)                                                           \
    {                                                                         \
      const float r = b2no_act(av.c, B2NO_ACT_SIGMOID);                       \
      o.c = gv.c * hv.c * r * (1.0f - r);                                     \
      acc.c = fmaf(gv.c, r, acc.c);                                           \
    }
    B2NO_RST(x) B2NO_RST(y) B2NO_RST(z) B2NO_RST(w)
#undef B2NO_RST
    o4[t] = o;
    gh4[t] = acc;
  }
}

extern "C" int b2no_rno_cell_bwd(const float* g, const float* h, const float* zz2, const float* ah, float* g_zz2, float* g_ah,
                                 float* g_h, int batch, int c, int64_t p, void* stream) {
  if (!g || !h || !zz2 || !ah || !g_zz2 || !g_ah || !g_h || batch < 1 || c < 1 || p < 1) return B2NO_E_ARG;
  const long cp = (long)c * p;
  if (cp % 4) return B2NO_E_UNSUPPORTED;
  if (((uintptr_t)g | (uintptr_t)h | (uintptr_t)zz2 | (uintptr_t)ah | (uintptr_t)g_zz2 | (uintptr_t)g_ah | (uintptr_t)g_h) & 15)
    return B2NO_E_ARG;
  k_rno_cell_bwd<<<(unsigned)grid_for((long)batch * (cp / 4), 256, 8), 256, 0, (cudaStream_t)stream>>>(g, h, zz2, ah, g_zz2, g_ah, g_h, batch, cp / 4);
  B2NO_LAUNCH_CHECK();
  return 0;
}

extern "C" int b2no_rno_reset_bwd(const float* g_rh, const float* h, const float* ar, float* g_ar, float* g_h, int64_t n,
                                  void* stream) {
  if (!g_rh || !h || !ar || !g_ar || !g_h || n < 1) return B2NO_E_ARG;
  if (n % 4) return B2NO_E_UNSUPPORTED;
  if (((uintptr_t)g_rh | (uintptr_t)h | (uintptr_t)ar | (uintptr_t)g_ar | (uintptr_t)g_h) & 15) return B2NO_E_ARG;
  k_rno_reset_bwd<<<(unsigned)grid_for(n / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(g_rh, h, ar, g_ar, g_h, n / 4);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// relative L2: per-sample sums with warp-shuffle + block reduction, one atomicAdd pair per block
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

__global__ void __launch_bounds__(256)
k_rel_l2_sums(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ sums, long n) {
  const int b = blockIdx.y;
  const float* xb = x + (size_t)b * n;
  const float* yb = y + (size_t)b * n;
  float d = 0.f, s = 0.f;
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float yv = __ldg(yb + i), dv = __ldg(xb + i) - yv;
    d = fmaf(dv, dv, d);
    s = fmaf(yv, yv, s);
  }
  __shared__ float sd[8], ss[8];
  d = warp_sum(d);
  s = warp_sum(s);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sd[warp] = d; ss[warp] = s; }
  __syncthreads();
  if (warp == 0) {
    d = lane < 8 ? sd[lane] : 0.f;
    s = lane < 8 ? ss[lane] : 0.f;
    d = warp_sum(d);
    s = warp_sum(s);
    if (lane == 0) {
      atomicAdd(sums + 2 * b, d);
      atomicAdd(sums + 2 * b + 1, s);
    }
  }
}

extern "C" int b2no_rel_l2_sums(const float* x, const float* y, float* sums, int batch, int64_t n, void* stream) {
  if (!x || !y || !sums || batch < 1 || n < 1) return B2NO_E_ARG;
  if (batch > 65535) return B2NO_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  B2NO_CHECK_CUDA(cudaMemsetAsync(sums, 0, (size_t)batch * 2 * sizeof(float), st));
  long bx = (n + 256 * 8 - 1) / (256 * 8);
  if (bx < 1) bx = 1;
  if (bx > 64) bx = 64;
  dim3 grid((unsigned)bx, (unsigned)batch);
  k_rel_l2_sums<<<grid, 256, 0, st>>>(x, y, sums, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}

__global__ void __launch_bounds__(256)
k_rel_l2_bwd(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ coef,
             float* __restrict__ dx, long n) {
  const int b = blockIdx.y;
  const float c = __ldg(coef + b);
  const size_t base = (size_t)b * n;
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dx[base + i] = c * (x[base + i] - y[base + i]);
}

extern "C" int b2no_rel_l2_bwd(const float* x, const float* y, const float* coef, float* dx, int batch,
                               int64_t n, void* stream) {
  if (!x || !y || !coef || !dx || batch < 1 || n < 1) return B2NO_E_ARG;
  if (batch > 65535) return B2NO_E_UNSUPPORTED;
  long bx = (n + 256 * 4 - 1) / (256 * 4);
  if (bx < 1) bx = 1;
  if (bx > 128) bx = 128;
  dim3 grid((unsigned)bx, (unsigned)batch);
  k_rel_l2_bwd<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, coef, dx, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// loss = sum_b (or mean_b) sqrt(sums[b][0]) / sqrt(sums[b][1]);  coef[b] = scale / (||x_b - y_b|| * ||y_b||) is what the
// backward multiplies (x - y) with (scale = 1/B for the mean).  One block; fixed summation order (deterministic).
__global__ void __launch_bounds__(256)
k_rel_l2_finish(const float* __restrict__ sums, float* __restrict__ loss, float* __restrict__ coef, int batch, float scale) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int b = threadIdx.x; b < batch; b += 256) {
    const float d = sqrtf(sums[2 * b]), n = sqrtf(sums[2 * b + 1]);
    acc += d / n;
    if (coef) coef[b] = scale / (d * n);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) s += red[w];
    *loss = s * scale;
  }
}

extern "C" int b2no_rel_l2_finish(const float* sums, float* loss, float* coef, int batch, int size_average, void* stream) {
  if (!sums || !loss || batch < 1) return B2NO_E_ARG;
  k_rel_l2_finish<<<1, 256, 0, (cudaStream_t)stream>>>(sums, loss, coef, batch, size_average ? 1.0f / (float)batch : 1.0f);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// dx = g * coef[b] * (x - y), g = the upstream scalar gradient read on the device
__global__ void __launch_bounds__(256)
k_rel_l2_bwd_g(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ coef,
               const float* __restrict__ g, float* __restrict__ dx, long n) {
  const int b = blockIdx.y;
  const float c = __ldg(coef + b) * __ldg(g);
  const size_t base = (size_t)b * n;
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dx[base + i] = c * (x[base + i] - y[base + i]);
}

extern "C" int b2no_rel_l2_bwd_g(const float* x, const float* y, const float* coef, const float* g, float* dx, int batch,
                                 int64_t n, void* stream) {
  if (!x || !y || !coef || !g || !dx || batch < 1 || n < 1) return B2NO_E_ARG;
  if (batch > 65535) return B2NO_E_UNSUPPORTED;
  long bx = (n + 256 * 4 - 1) / (256 * 4);
  if (bx < 1) bx = 1;
  if (bx > 128) bx = 128;
  dim3 grid((unsigned)bx, (unsigned)batch);
  k_rel_l2_bwd_g<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, coef, g, dx, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}
