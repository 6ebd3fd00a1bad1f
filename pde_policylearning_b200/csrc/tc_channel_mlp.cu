// Channel MLP of an FNO block with its soft-gating skip (neuralop fno_block.py:123-170, mlp.py:10-54,
// skip_connections.py:5-74) on tcgen05, per pixel, without writing the hidden tensor in the forward:
//   forward :  a1 = W1 u + b1,  h = gelu(a1),  a2 = W2 h + b2,  s = gelu(a2) + g x,  y = act(s)      (pre = s when asked)
//   backward:  dy = gy act'(pre) (gy without a block activation),  d2 = dy gelu'(a2),  d1 = (W2^T d2) gelu'(a1),
//              du = W1^T d1,  dx = g dy,  dg[c] = sum_{b,p} dy x  (per-warp partials, summed in a fixed order);
//              h, d1 and d2 are written once for the weight-gradient kernel (dW1 = sum d1 u^T, dW2 = sum d2 h^T)
// One 128-pixel tile per step, TMEM lane = pixel, every warp of the CTA on every phase (no warp roles): load the tile into
// TMEM as the A operand (hi / lo), one elected thread issues the product (3xTF32, or single-pass TF32), all threads read
// the accumulator, apply the element-wise stage and store the next A operand over the previous one.  C and H are compile-time
// (padded to 16), so every MMA-issue and epilogue loop is unrolled.  The CTA needs 3 max(C, H) (+ H in the backward) TMEM
// columns; the shared-memory request caps the CTAs per SM at what the 512 columns hold, and the co-resident CTAs overlap
// each other's loads, products and stores.
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

struct ChMlp {
  int C, H, tiles_per_img, npass, act;
  long P, tiles;
  const float* u; const float* x; const float* w1; const float* b1; const float* w2; const float* b2; const float* g;
  const float* gy; const float* pre_in;   // backward
  float* y; float* pre;                   // forward
  float* du; float* dx; float* h; float* d1; float* d2; float* dg_partial;   // backward
};

// sum over the warp's 32 lanes of each of 16 columns (transposing butterfly): lane l returns the sum of column l >> 1
__device__ __forceinline__ float col_sum16(float (&v)[16], int lane) {
#pragma unroll
  for (int s = 0; s < 4; s++) {
    const int off = 16 >> s, hw = 8 >> s;
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      if (i < hw) {
        const float a0 = v[i], a1 = v[i + hw];
        v[i] = (upper ? a1 : a0) + __shfl_xor_sync(0xffffffffu, upper ? a0 : a1, off);
      }
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// D[128 x N] = A[128 x K] (TMEM, hi at a_hi, lo at a_lo) * B[N x K]^T (shared memory, K-major core layout, hi / lo)
template <int K, int N>
__device__ __forceinline__ void issue_mma(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, int npass) {
  constexpr uint32_t id = idesc_tf32(128, N, 0, 0);
  const uint64_t dh = smem_desc(b_hi, 128, (K / 4) * 128, LAYOUT_NONE), dl = smem_desc(b_lo, 128, (K / 4) * 128, LAYOUT_NONE);
#pragma unroll
  for (int pass = 0; pass < 3; pass++) {
    if (pass >= npass) break;
    const uint32_t a = pass == 1 ? a_lo : a_hi;
    const uint64_t b = pass == 2 ? dl : dh;
#pragma unroll
    for (int k = 0; k < K / 8; k++) mma_tf32_ts(d, a + 8 * k, b + (uint64_t)(k * 16), id, (pass > 0 || k > 0) ? 1u : 0u);
  }
}

template <int K_, int N_>
struct KN { static constexpr int K = K_, N = N_; };

template <int CP, int HP, bool BWD>
struct ChLayout {
  static constexpr int MX = CP > HP ? CP : HP;
  static constexpr uint32_t IMG = (uint32_t)CP * HP * 4;        // one [HP x CP] or [CP x HP] image
  static constexpr int NIMG = BWD ? 8 : 4;                      // (W1, W2[, W2^T, W1^T]) x (hi, lo)
  static constexpr uint32_t VEC = NIMG * IMG;                   // b1 [HP] | b2 [CP] | g [CP] | dg [4 warps x CP]
  static constexpr uint32_t BAR = VEC + (uint32_t)(HP + 6 * CP) * 4;
  static constexpr uint32_t BYTES = BAR + 16 + 128;             // + alignment slack
  static constexpr uint32_t COLS_USED = 3 * MX + (BWD ? HP : 0);
  static constexpr uint32_t COLS = COLS_USED <= 32 ? 32 : COLS_USED <= 64 ? 64 : COLS_USED <= 128 ? 128 : COLS_USED <= 256 ? 256 : 512;
};

template <int CP, int HP, bool BWD>
__global__ void __launch_bounds__(128, BWD ? 1 : 4) k_channel_mlp(const ChMlp p) {
  using L = ChLayout<CP, HP, BWD>;
  constexpr int MX = L::MX;
  constexpr bool PF = !BWD && CP <= 32;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  float* sb1 = (float*)(smem + L::VEC);
  float* sb2 = sb1 + HP;
  float* sg = sb2 + CP;
  uint64_t* bar = (uint64_t*)(smem + L::BAR);
  uint32_t* tslot = (uint32_t*)(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* sdg = sg + CP + warp * CP;   // this warp's dg sums: column c belongs to one lane, added in tile order
  const int C = p.C, H = p.H;
  auto put = [&](int img, uint32_t off, float w) {
    const float hi = tf32_rna(w);
    *(float*)(smem + (2 * img) * L::IMG + off) = hi;
    *(float*)(smem + (2 * img + 1) * L::IMG + off) = tf32_rna(w - hi);
  };
  // images 0: W1 [HP x CP], 1: W2 [CP x HP]; backward 2: W2^T [HP x CP], 3: W1^T [CP x HP]; zero padded
  for (int i = tid; i < HP * CP; i += 128) {
    const int n = i / CP, k = i - n * CP;
    const bool in = n < H && k < C;
    put(0, kmajor_off(n, k, CP), in ? p.w1[n * C + k] : 0.f);
    if (BWD) put(2, kmajor_off(n, k, CP), in ? p.w2[k * H + n] : 0.f);
  }
  for (int i = tid; i < CP * HP; i += 128) {
    const int n = i / HP, k = i - n * HP;
    const bool in = n < C && k < H;
    put(1, kmajor_off(n, k, HP), in ? p.w2[n * H + k] : 0.f);
    if (BWD) put(3, kmajor_off(n, k, HP), in ? p.w1[k * C + n] : 0.f);
  }
  for (int i = tid; i < HP; i += 128) sb1[i] = (i < H && p.b1) ? p.b1[i] : 0.f;
  for (int i = tid; i < CP; i += 128) {
    sb2[i] = (i < C && p.b2) ? p.b2[i] : 0.f;
    sg[i] = i < C ? p.g[i] : 0.f;
  }
  for (int i = tid; i < 4 * CP; i += 128) sg[CP + i] = 0.f;
  if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  fence_proxy_async();
  if (warp == 0) tmem_alloc(tslot, L::COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  // TMEM: [A hi (MX) | A lo (MX)] [accumulator (MX)] [gelu'(a1) (HP), backward]
  const uint32_t lb = (uint32_t)(warp * 32) << 16;
  const uint32_t t_a = tbase + lb, t_alo = t_a + MX, t_acc = t_a + 2 * MX, t_gp = t_a + 3 * MX;
  const uint32_t s0 = smem_u32(smem);
  uint32_t phase = 0;
  // A operand written by every thread -> one product -> accumulator readable
  auto product = [&](auto kn, int img) {
    constexpr int K = decltype(kn)::K, N = decltype(kn)::N;
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      issue_mma<K, N>(tbase + 2 * MX, tbase, tbase + MX, s0 + 2 * img * L::IMG, s0 + (2 * img + 1) * L::IMG, p.npass);
      mma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1u;
    __syncwarp();
    tc_fence_after();
  };
  // hi / lo of 16 values into A columns c0..c0+15
  auto store_a = [&](int c0, float (&v)[16]) {
    float lo[16];
#pragma unroll
    for (int j = 0; j < 16; j++) lo[j] = tf32_lo(v[j]);
    tmem_st16(t_a + c0, v);
    tmem_st16(t_alo + c0, lo);
  };
  for (long tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
    const int b = (int)(tile / p.tiles_per_img);
    const size_t px = (size_t)(tile - (long)b * p.tiles_per_img) * 128 + tid;
    const size_t cbase = (size_t)b * C * p.P + px, hbase = (size_t)b * H * p.P + px;
    // ---- u -> A; up to 32 channels, the epilogue's inputs are loaded here too, so that their latency overlaps the products
    // instead of following them (one memory round trip per tile) ----
    float xv_pf[PF ? CP : 1], gy_pf[PF && BWD ? CP : 1], pre_pf[PF && BWD ? CP : 1];
#pragma unroll(BWD ? 1 : CP / 16)
    for (int c0 = 0; c0 < CP; c0 += 16) {
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; j++) {
        const bool in = c0 + j < C;
        const size_t o = cbase + (size_t)(c0 + j) * p.P;
        v[j] = in ? __ldg(p.u + o) : 0.f;
        if constexpr (PF) {
          xv_pf[c0 + j] = in ? __ldg(p.x + o) : 0.f;
          if constexpr (BWD) {
            gy_pf[c0 + j] = in ? __ldg(p.gy + o) : 0.f;
            pre_pf[c0 + j] = (in && p.act) ? __ldg(p.pre_in + o) : 0.f;
          }
        }
      }
      store_a(c0, v);
    }
    product(KN<CP, HP>{}, 0);
    // ---- a1 -> h = gelu(a1) -> A  (gelu'(a1) kept in TMEM for the backward) ----
#pragma unroll 1
    for (int j0 = 0; j0 < HP; j0 += 16) {
      float v[16], gp[16];
      tmem_ld16(t_acc + j0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        float2 val, grad;
        b2no_gelu2_both(make_float2(v[j] + sb1[j0 + j], v[j + 1] + sb1[j0 + j + 1]), &val, &grad);
        v[j] = val.x; v[j + 1] = val.y; gp[j] = grad.x; gp[j + 1] = grad.y;
      }
      if (BWD) {
        tmem_st16(t_gp + j0, gp);
#pragma unroll
        for (int j = 0; j < 16; j++)
          if (j0 + j < H) p.h[hbase + (size_t)(j0 + j) * p.P] = v[j];
      }
      store_a(j0, v);
    }
    product(KN<HP, CP>{}, 1);
    if constexpr (!BWD) {
      // ---- a2 -> y = act(gelu(a2 + b2) + g x) ----
#pragma unroll
      for (int c0 = 0; c0 < CP; c0 += 16) {
        float v[16], xv[16];
#pragma unroll
        for (int j = 0; j < 16; j++) {
          if constexpr (PF) xv[j] = xv_pf[c0 + j];
          else xv[j] = c0 + j < C ? __ldg(p.x + cbase + (size_t)(c0 + j) * p.P) : 0.f;
        }
        tmem_ld16(t_acc + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const float2 m = b2no_gelu2(make_float2(v[j] + sb2[c0 + j], v[j + 1] + sb2[c0 + j + 1]));
          v[j] = fmaf(sg[c0 + j], xv[j], m.x);
          v[j + 1] = fmaf(sg[c0 + j + 1], xv[j + 1], m.y);
        }
#pragma unroll
        for (int j = 0; j < 16; j++) {
          if (c0 + j < C) {
            const size_t o = cbase + (size_t)(c0 + j) * p.P;
            if (p.pre) p.pre[o] = v[j];
            p.y[o] = p.act ? b2no_act(v[j], p.act) : v[j];
          }
        }
      }
    } else {
    // ---- backward: a2 -> dy, d2 = dy gelu'(a2) -> A;  dx = g dy;  dg += dy x ----
#pragma unroll 1
    for (int c0 = 0; c0 < CP; c0 += 16) {
      float v[16], dy[16], xv[16];
#pragma unroll
      for (int j = 0; j < 16; j++) {
        const bool in = c0 + j < C;
        const size_t o = cbase + (size_t)(c0 + j) * p.P;
        if constexpr (PF) {
          dy[j] = gy_pf[c0 + j];
          xv[j] = xv_pf[c0 + j];
          if (p.act && in) dy[j] *= b2no_act_grad(pre_pf[c0 + j], p.act);
        } else {
          dy[j] = in ? __ldg(p.gy + o) : 0.f;
          xv[j] = in ? __ldg(p.x + o) : 0.f;
          if (p.act && in) dy[j] *= b2no_act_grad(__ldg(p.pre_in + o), p.act);
        }
      }
      tmem_ld16(t_acc + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; j += 2) {
        const float2 gr = b2no_gelu2_grad(make_float2(v[j] + sb2[c0 + j], v[j + 1] + sb2[c0 + j + 1]));
        v[j] = dy[j] * gr.x;
        v[j + 1] = dy[j + 1] * gr.y;
      }
#pragma unroll
      for (int j = 0; j < 16; j++) {
        if (c0 + j < C) {
          const size_t o = cbase + (size_t)(c0 + j) * p.P;
          p.dx[o] = sg[c0 + j] * dy[j];
          p.d2[o] = v[j];
        }
        xv[j] *= dy[j];
      }
      const float s = col_sum16(xv, lane);
      if ((lane & 1) == 0) sdg[c0 + (lane >> 1)] += s;
      store_a(c0, v);
    }
    product(KN<CP, HP>{}, 2);
    // ---- W2^T d2 -> d1 = (.) gelu'(a1) -> A ----
#pragma unroll 1
    for (int j0 = 0; j0 < HP; j0 += 16) {
      float v[16], gp[16];
      tmem_ld16(t_acc + j0, v);
      tmem_ld16(t_gp + j0, gp);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; j++) {
        v[j] *= gp[j];
        if (j0 + j < H) p.d1[hbase + (size_t)(j0 + j) * p.P] = v[j];
      }
      store_a(j0, v);
    }
    product(KN<HP, CP>{}, 3);
    // ---- du = W1^T d1 ----
#pragma unroll 1
    for (int c0 = 0; c0 < CP; c0 += 16) {
      float v[16];
      tmem_ld16(t_acc + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; j++)
        if (c0 + j < C) p.du[cbase + (size_t)(c0 + j) * p.P] = v[j];
    }
    }
  }
  if (BWD) {
    __syncwarp();
    for (int c = lane; c < CP; c += 32) p.dg_partial[((size_t)blockIdx.x * 4 + warp) * CP + c] = sdg[c];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, L::COLS);
}

// dg[c] = sum over the rows of partial[rows x stride] of column c, in a fixed order (8 warps x strided rows, then the 8 sums)
__global__ void __launch_bounds__(256) k_channel_mlp_dg(const float* __restrict__ partial, float* __restrict__ dg, int rows,
                                                         int stride, int n) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < n)
    for (int r = warp; r < rows; r += 8) s += __ldg(partial + (size_t)r * stride + c);
  red[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && c < n) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) t += red[w][lane];
    dg[c] = t;
  }
}

constexpr uint32_t kSmemPerSm = 233472;   // 228 KB of shared memory per SM (sm_100)

int channel_mlp_shape_ok(int C, int H, int64_t pixels) {
  return b2no_tc_available() && C >= 1 && C <= 64 && H >= 1 && H <= 64 && pixels >= 128 && pixels % 128 == 0;
}

template <int CP, int HP, bool BWD>
int channel_mlp_run(ChMlp& p, cudaStream_t st, int* grid_out) {
  using L = ChLayout<CP, HP, BWD>;
  // at most 512 / COLS CTAs may share an SM's tensor memory: ask for enough shared memory that no more fit
  const int by_tmem = (int)(512 / L::COLS);
  uint32_t smem = kSmemPerSm / (uint32_t)(by_tmem + 1) + 16;
  if (smem < L::BYTES) smem = L::BYTES;
  int dev = 0, max_smem = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  B2NO_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if ((int)smem > max_smem) return 1;
  B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_channel_mlp<CP, HP, BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the full carveout, so that the by_tmem CTAs the shared-memory request allows do fit
  B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_channel_mlp<CP, HP, BWD>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
  // CTAs per SM from the TMEM budget, the registers and the shared memory.  Not from
  // cudaOccupancyMaxActiveBlocksPerMultiprocessor: it reports 1 for these kernels with any shared-memory size (B200), while 4
  // CTAs of the cfg2 shapes run side by side there: forward 551 -> 259 us, backward 1646 -> 507 us, bit-identical results.
  cudaFuncAttributes fa;
  B2NO_CHECK_CUDA(cudaFuncGetAttributes(&fa, k_channel_mlp<CP, HP, BWD>));
  int per_sm = 65536 / (128 * (fa.numRegs > 0 ? fa.numRegs : 255));
  const int by_smem = (int)(kSmemPerSm / (smem + 1024));
  if (by_smem < per_sm) per_sm = by_smem;
  if (by_tmem < per_sm) per_sm = by_tmem;
  if (per_sm < 1) per_sm = 1;
  long grid = (long)b2no_sm_count() * per_sm;
  if (grid > p.tiles) grid = p.tiles;
  k_channel_mlp<CP, HP, BWD><<<(unsigned)grid, 128, smem, st>>>(p);
  B2NO_LAUNCH_CHECK();
  *grid_out = (int)grid;
  return 0;
}

template <bool BWD>
int channel_mlp_dispatch(ChMlp& p, cudaStream_t st, int* grid) {
  const int cp = b2no_round_up(p.C, 16), hp = b2no_round_up(p.H, 16);
#define CH_CASE(A, B) \
  if (cp == A && hp == B) return channel_mlp_run<A, B, BWD>(p, st, grid);
#define CH_ROW(A) CH_CASE(A, 16) CH_CASE(A, 32) CH_CASE(A, 48) CH_CASE(A, 64)
  CH_ROW(16) CH_ROW(32) CH_ROW(48) CH_ROW(64)
#undef CH_ROW
#undef CH_CASE
  return 1;
}

}  // namespace

void b2no_tc_count_launch();

extern "C" int b2no_channel_mlp_supported(int channels, int hidden, int64_t pixels) {
  return channel_mlp_shape_ok(channels, hidden, pixels);
}

extern "C" int64_t b2no_channel_mlp_scratch_floats(int channels) {
  if (channels < 1) return B2NO_E_ARG;
  // one row per warp of every CTA: at most 8 CTAs per SM (the backward needs >= 64 TMEM columns), 4 warps each
  return (int64_t)b2no_sm_count() * 8 * 4 * b2no_round_up(channels, 16);
}

extern "C" int b2no_channel_mlp_fwd(const float* u, const float* x, const float* w1, const float* b1, const float* w2,
                                    const float* b2, const float* g, float* y, float* pre, int batch, int channels, int hidden,
                                    int64_t pixels, int act, void* stream) {
  if (!u || !x || !w1 || !w2 || !g || !y || batch < 1 || channels < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  if (!channel_mlp_shape_ok(channels, hidden, pixels)) return B2NO_E_UNSUPPORTED;
  ChMlp p;
  memset(&p, 0, sizeof(p));
  p.C = channels; p.H = hidden; p.P = pixels; p.tiles_per_img = (int)(pixels / 128); p.tiles = (long)batch * p.tiles_per_img;
  p.npass = b2no_tc_passes(); p.act = act;
  p.u = u; p.x = x; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.g = g; p.y = y; p.pre = act ? pre : nullptr;
  int grid = 0;
  const int rc = channel_mlp_dispatch<false>(p, (cudaStream_t)stream, &grid);
  if (rc == 1) return B2NO_E_UNSUPPORTED;
  if (rc) return rc;
  b2no_tc_count_launch();
  return 0;
}

extern "C" int b2no_channel_mlp_bwd(const float* u, const float* x, const float* pre, const float* gy, const float* w1,
                                    const float* b1, const float* w2, const float* b2, const float* g, float* du, float* dx,
                                    float* h, float* d1, float* d2, float* dg, float* scratch, int batch, int channels,
                                    int hidden, int64_t pixels, int act, void* stream) {
  if (!u || !x || !gy || !w1 || !w2 || !g || !du || !dx || !h || !d1 || !d2 || !dg || !scratch || (act && !pre) || batch < 1 ||
      channels < 1 || hidden < 1 || pixels < 1)
    return B2NO_E_ARG;
  if (!channel_mlp_shape_ok(channels, hidden, pixels)) return B2NO_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  ChMlp p;
  memset(&p, 0, sizeof(p));
  p.C = channels; p.H = hidden; p.P = pixels; p.tiles_per_img = (int)(pixels / 128); p.tiles = (long)batch * p.tiles_per_img;
  p.npass = b2no_tc_passes(); p.act = act;
  p.u = u; p.x = x; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.g = g; p.gy = gy; p.pre_in = act ? pre : nullptr;
  p.du = du; p.dx = dx; p.h = h; p.d1 = d1; p.d2 = d2; p.dg_partial = scratch;
  int grid = 0;
  const int rc = channel_mlp_dispatch<true>(p, st, &grid);
  if (rc == 1) return B2NO_E_UNSUPPORTED;
  if (rc) return rc;
  b2no_tc_count_launch();
  k_channel_mlp_dg<<<(channels + 31) / 32, 256, 0, st>>>(scratch, dg, grid * 4, b2no_round_up(channels, 16), channels);
  B2NO_LAUNCH_CHECK();
  return 0;
}
