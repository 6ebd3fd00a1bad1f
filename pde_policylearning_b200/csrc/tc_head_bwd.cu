// Whole backward of the projection head in ONE kernel (tfno.py:34-38: Conv(C->H) -> GELU -> Conv(H->1); rno.py:170-174):
//
//   z1[j,p] = b1[j] + sum_c W1[j,c] x[c,p]                      (recomputed, never stored)
//   f[j,p]  = g[p] w2[j] act'(z1[j,p])
//   gx[c,p] = sum_j W1[j,c] f[j,p]   (* dact'(dz[c,p]) when given)
//   dW1[j,c] = sum_p f[j,p] x[c,p],   db1[j] = sum_p f[j,p],   dw2[j] = sum_p g[p] act(z1[j,p]),   db2 = sum_p g[p]
//
// Round 1 wrote f ("gz", batch x H x pixels fp32 = 1.07 GB at BASELINE config 2) to HBM for a separate weight-gradient
// kernel.  Here f never leaves the SM.  Orientation: TMEM lane = hidden unit j (blocks of 128), column = pixel, so
//   * b1[j], w2[j] are per-thread constants and dw2[j], db1[j] per-thread register sums (no cross-lane reduction);
//   * dW1 is a TS-form product straight from the F tile the thread just wrote to TMEM (contraction over pixels = columns);
//   * only gx contracts over lanes: F goes through shared memory once more, as the A operand [pixel x hidden] (K-major, K
//     chunks padded to 144 B so the per-thread scalar stores are conflict-free).
// Per 128-pixel tile, 2 pixel chunks (64) x NB hidden blocks (128) = "steps":
//   G1 (TS): D1[128 j x 64 px]  = W1 block (TMEM resident, hi | lo) x XT chunk [64 px x C] (smem, hi / lo)       3xTF32
//   epilogue: D1 -> f (packed fp32x2 GELU math) -> F hi | lo to TMEM and to smem, dw2 / db1 register sums
//   G3 (TS): D3[b][128 j x 2C] += F (TMEM) x XK chunk [(x hi ; x lo) x 64 px]   (cols [0,C): f x_hi, [C,2C): f_hi x_lo)
//   G2 (SS, M = 64): D2[64 px x 2C] += Fs (smem) x WT block [(W1^T hi ; W1^T lo) x 128 j]; after the last block: gx epilogue
// Everything is single buffered (TMEM: W1 4 NB C + D1 64 + F 128 + D3 2 NB C + D2 2C = 512 columns at C = 32, H = 256;
// shared memory 226 KB of 227): the steps are a hand-over chain  F(n) visible -> G3 / G2(n) -> F(n + 1) may be written.
// Measured (B200, cfg2 shape, 429 us; DESIGN.md section 4, profiles/r02_l ... r02_p): step period ~4000 cycles = FMA-pipe math
// ~1800 + TMEM read / F write ~1000 + barrier round trips; the tensor pipe is ~40 % busy.  F has two hand-overs: the TMEM copy is
// released by G3 (ft_*), the shared-memory copy by G2 (fs_*).
// Warp roles: 0 TMA producer (x tile + g tile), 1 MMA issuer, 2-5 X converter (thread = pixel: raw tile -> XT, XK images, hi / lo)
// which also drain the gx accumulator (D2 -> 4 KB staging -> TMA store, off the chain), 6-21 epilogue (4 lane quadrants x 4
// column parts of 16 pixels).
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

constexpr int kHbEpiThreads = 512;
constexpr int kHbThreads = 192 + kHbEpiThreads;
constexpr uint32_t kHbLbo = 144;                 // bytes between K-adjacent core matrices of the padded operands
constexpr uint32_t kHbSbo = 32 * kHbLbo;         // 128 K elements per 8-row group

struct HeadBwd {
  int B, Ci, Cq, H, Hp, NB, act, dact, npass;
  int tiles_per_img;
  int tiles, tiles_per_cta;                       // 128-pixel tiles (checked < 2^30 on the host: no 64-bit divisions in the kernel)
  long P;
  const float* w1; const float* b1; const float* w2; const float* g; const float* dz;
  float* gx; float* partial;
  int nsum;                                      // floats per partial row: H*Ci + 2H + 1
};

// act'(z) of the layer below, out of line: the switch over the activations would otherwise be unrolled 32 times
__device__ __noinline__ float hb_act_grad(float z, int act) { return b2no_act_grad(z, act); }

// one arrival per warp: every lane has fenced its own writes before the call
__device__ __forceinline__ void warp_arrive(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void warp_arrive2(uint64_t* bar_a, uint64_t* bar_b) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) { mbar_arrive(bar_a); mbar_arrive(bar_b); }
}

struct HbLayout { uint32_t fs, fs_img, wt, xt, xt_img, xk, raw, g, gxb, bars, total; };

__host__ __device__ inline HbLayout hb_layout(int Cq, int Hp) {
  HbLayout L;
  uint32_t o = 0;
  L.fs = o; L.fs_img = 8 * kHbSbo; o += 2 * L.fs_img;              // [64 px (8 row groups)][128 j] hi, lo
  L.wt = o; o += (uint32_t)(2 * Cq) * Hp * 4;
  L.xt = o; L.xt_img = 128u * Cq * 4; o += 2 * L.xt_img;
  L.xk = o; o += (uint32_t)(2 * Cq / 8) * kHbSbo;
  L.raw = o; o += (uint32_t)Cq * 512;
  L.g = o; o += 3 * 512;
  L.gxb = o; o += 64 * 16 * 4;                                     // gx epilogue: [16 channels][64 px] staging of the TMA store
  L.bars = o; o += 8 * 13 + 16;
  L.total = o + 1024;
  return L;
}

__host__ __device__ inline uint32_t hb_tmem_cols(int Cq, int NB) { return (uint32_t)(4 * NB * Cq + 192 + 2 * Cq); }

template <bool GELU, int CQ>
__global__ void __launch_bounds__(kHbThreads, 1)
k_head_bwd(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmg, const HeadBwd p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int Cq = CQ;                     // channels rounded up to 16 (compile time: the MMA issue loops unroll)
  const int NB = p.NB, NS = 2 * p.NB, Hp = p.Hp;
  const HbLayout L = hb_layout(Cq, Hp);
  uint64_t* bars = (uint64_t*)(smem + L.bars);
  uint64_t* raw_full = bars + 0;  uint64_t* raw_empty = bars + 1;
  uint64_t* xt_full = bars + 2;   uint64_t* xt_empty = bars + 3;
  uint64_t* xk_full = bars + 4;   uint64_t* xk_empty = bars + 5;
  uint64_t* d1_full = bars + 6;   uint64_t* d1_empty = bars + 7;
  uint64_t* f_full = bars + 8;    uint64_t* f_empty = bars + 9;
  uint64_t* d2_full = bars + 10;  uint64_t* d2_empty = bars + 11;
  uint64_t* done = bars + 12;
  uint32_t* tslot = (uint32_t*)(bars + 13);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t ncols = 32;
  while (ncols < hb_tmem_cols(Cq, NB)) ncols <<= 1;

  // ---- setup: WT = (W1^T hi ; W1^T lo), the B operand of G2: [2 Cq rows (channel)][Hp (hidden)], K-major core layout ----
  for (int i = tid; i < Cq * Hp; i += kHbThreads) {
    const int j = i / Cq, c = i - j * Cq;
    const float w = (j < p.H && c < p.Ci) ? p.w1[(size_t)j * p.Ci + c] : 0.f;
    const float hi = tf32_rna(w);
    *(float*)(smem + L.wt + kmajor_off(c, j, Hp)) = hi;
    *(float*)(smem + L.wt + kmajor_off(Cq + c, j, Hp)) = tf32_rna(w - hi);
  }
  if (tid == 0) {
    // consumer-side barriers count WARPS: every lane fences its own writes, the warp converges (__syncwarp), one lane
    // arrives -- 512 per-thread arrivals on one mbarrier word serialise in the shared-memory atomic unit
    mbar_init(raw_full, 1);  mbar_init(raw_empty, 4);
    mbar_init(xt_full, 4);   mbar_init(xt_empty, 1);
    mbar_init(xk_full, 4);   mbar_init(xk_empty, 1);
    mbar_init(d1_full, 1);   mbar_init(d1_empty, kHbEpiThreads / 32);
    mbar_init(f_full, kHbEpiThreads / 32); mbar_init(f_empty, 1);
    mbar_init(d2_full, 1);   mbar_init(d2_empty, 4);
    mbar_init(done, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 1) tmem_alloc(tslot, ncols);
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmx); tma_prefetch_desc(&tmg); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  // TMEM map: [W1 block b: hi Cq | lo Cq] x NB, D1 64, F hi 64 | lo 64, [D3 block b: 2 Cq] x NB, D2 2 Cq
  const uint32_t t_w = tbase, t_d1 = t_w + (uint32_t)(2 * NB * Cq), t_f = t_d1 + 64u, t_d3 = t_f + 128u,
                 t_d2 = t_d3 + (uint32_t)(2 * NB * Cq);
  // W1 -> TMEM (the A operand of G1): lane = hidden unit of the block, column = channel
  if (warp >= 6 && warp < 10) {
    const int quad = warp & 3;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    for (int b = 0; b < NB; b++) {
      const int j = b * 128 + quad * 32 + lane;
      for (int c0 = 0; c0 < Cq; c0 += 8) {
        float hi[8], lo[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const float w = (j < p.H && c0 + u < p.Ci) ? p.w1[(size_t)j * p.Ci + c0 + u] : 0.f;
          hi[u] = tf32_rna(w);
          lo[u] = tf32_rna(w - hi[u]);
        }
        tmem_st8(t_w + lane_base + (uint32_t)(b * 2 * Cq + c0), hi);
        tmem_st8(t_w + lane_base + (uint32_t)(b * 2 * Cq + Cq + c0), lo);
      }
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const int t_first = (int)blockIdx.x * p.tiles_per_cta;
  const int t_end = t_first + p.tiles_per_cta < p.tiles ? t_first + p.tiles_per_cta : p.tiles;
  const uint32_t sbo_xt = (uint32_t)(Cq / 4) * 128;

  if (warp == 0) {
    // ===================== TMA producer: x tile [Cq x 128 px] and the g tile (512 B) =====================
    if (lane == 0) {
      int it = 0;
      for (int tile = t_first; tile < t_end; tile++, it++) {
        mbar_wait(raw_empty, ((uint32_t)it & 1u) ^ 1u);
        mbar_arrive_expect_tx(raw_full, (uint32_t)Cq * 512u + 512u);
        const int b = tile / p.tiles_per_img;
        const int px0 = (tile - b * p.tiles_per_img) * 128;
        tma_load_3d(smem + L.raw, &tmx, raw_full, px0, 0, b);
        bulk_load(smem + L.g + (uint32_t)(it % 3) * 512u, p.g + (size_t)b * p.P + px0, 512u, raw_full);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t id_g1 = idesc_tf32(128, 64, 0, 0), id_n2 = idesc_tf32(128, 2 * Cq, 0, 0), id_n1 = idesc_tf32(128, Cq, 0, 0),
                   id_g2h = idesc_tf32(64, 2 * Cq, 0, 0), id_g2l = idesc_tf32(64, Cq, 0, 0);
    const uint32_t sbase = smem_u32(smem);
    const uint64_t d_xth = smem_desc(sbase + L.xt, 128, sbo_xt, LAYOUT_NONE);
    const uint64_t d_xtl = smem_desc(sbase + L.xt + L.xt_img, 128, sbo_xt, LAYOUT_NONE);
    const uint64_t d_xk = smem_desc(sbase + L.xk, kHbLbo, kHbSbo, LAYOUT_NONE);
    const uint64_t d_fsh = smem_desc(sbase + L.fs, kHbLbo, kHbSbo, LAYOUT_NONE);
    const uint64_t d_fsl = smem_desc(sbase + L.fs + L.fs_img, kHbLbo, kHbSbo, LAYOUT_NONE);
    const uint64_t d_wt = smem_desc(sbase + L.wt, 128, (uint32_t)(Hp / 4) * 128, LAYOUT_NONE);
    constexpr int k1 = Cq / 8;
    const bool lo_pass = p.npass >= 3;
    // G3 + G2 of step pn (tile index pit of this CTA, step ps inside the tile)
    auto g3g2 = [&](long pn, int pit, int ps) {
      const int q = ps / NB, b = ps - q * NB;
      mbar_wait(f_full, (uint32_t)pn & 1u);
      if (ps == 0) mbar_wait(xk_full, (uint32_t)pit & 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d3 = t_d3 + (uint32_t)(b * 2 * Cq);
        const uint64_t dxk = d_xk + (uint64_t)(q * 16 * (kHbLbo / 16));        // 64 px = 16 K-chunks of 4
        const uint32_t first = (pit == 0 && q == 0) ? 0u : 1u;
#pragma unroll
        for (int k = 0; k < 8; k++) mma_tf32_ts(d3, t_f + 8 * k, dxk + (uint64_t)(k * (2 * kHbLbo / 16)), id_n2, (k > 0) ? 1u : first);
        if (lo_pass) {
#pragma unroll
          for (int k = 0; k < 8; k++) mma_tf32_ts(d3, t_f + 64 + 8 * k, dxk + (uint64_t)(k * (2 * kHbLbo / 16)), id_n1, 1u);
        }
      }
      __syncwarp();
      if (b == 0) {
        const long qc = (long)pit * 2 + q;
        mbar_wait(d2_empty, ((uint32_t)qc & 1u) ^ 1u);
        tc_fence_after();
      }
      if (elect_one()) {
        const uint64_t dw = d_wt + (uint64_t)(b * 32 * (128 / 16));             // 128 j = 32 K-chunks of 4
#pragma unroll
        for (int k = 0; k < 16; k++)
          mma_tf32_ss(t_d2, d_fsh + (uint64_t)(k * (2 * kHbLbo / 16)), dw + (uint64_t)(k * 16), id_g2h, (b > 0 || k > 0) ? 1u : 0u);
        if (lo_pass) {
#pragma unroll
          for (int k = 0; k < 16; k++)
            mma_tf32_ss(t_d2, d_fsl + (uint64_t)(k * (2 * kHbLbo / 16)), dw + (uint64_t)(k * 16), id_g2l, 1u);
        }
        mma_commit(f_empty);
        if (b == NB - 1) mma_commit(d2_full);
        if (ps == NS - 1) mma_commit(xk_empty);
      }
      __syncwarp();
    };
    // software pipeline over the steps of this CTA: G1 of step n is issued before G3 / G2 of step n - 1 (one call site each)
    const long nsteps = (long)(t_end - t_first) * NS;
    int it = 0, s = 0;
    for (long n = 0; n <= nsteps; n++) {
      if (n < nsteps) {
        const int q = s / NB, b = s - q * NB;
        if (s == 0) { mbar_wait(xt_full, (uint32_t)it & 1u); tc_fence_after(); }
        mbar_wait(d1_empty, ((uint32_t)n & 1u) ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t qoff = (uint64_t)(q * 8 * (sbo_xt / 16));               // 64 px rows = 8 row groups
          uint32_t acc = 0;
          _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;
            const uint32_t a = t_w + (uint32_t)(b * 2 * Cq) + (pass == 1 ? (uint32_t)Cq : 0u);
            const uint64_t dx = (pass == 2 ? d_xtl : d_xth) + qoff;
            _Pragma("unroll") for (int k = 0; k < k1; k++) { mma_tf32_ts(t_d1, a + 8 * k, dx + (uint64_t)(k * 16), id_g1, acc); acc = 1; }
          }
          mma_commit(d1_full);
          if (s == NS - 1) mma_commit(xt_empty);
        }
        __syncwarp();
      }
      if (n > 0) {
        const int ps = s > 0 ? s - 1 : NS - 1;
        g3g2(n - 1, s > 0 ? it : it - 1, ps);
      }
      if (++s == NS) { s = 0; it++; }
    }
    if (elect_one()) mma_commit(done);
    __syncwarp();
  } else if (warp < 6) {
    // ===================== converter: raw x tile -> XT (B operand of G1) and XK (B operand of G3), hi / lo =====================
    const int m = (warp - 2) * 32 + lane;                                       // pixel of the tile
    const uint32_t sb = smem_u32(smem);
    const uint32_t sx = sb + L.raw + (uint32_t)m * 4;
    const uint32_t xt_row = sb + L.xt + (uint32_t)(m >> 3) * sbo_xt + (uint32_t)(m & 7) * 16;
    const uint32_t xk_col = sb + L.xk + (uint32_t)(m >> 2) * kHbLbo + (uint32_t)(m & 3) * 4;
    // gx epilogue of a finished pixel chunk (these warps have the slack; the stores stay off the F hand-over chain).  D2 comes
    // from M = 64 MMAs: pixel m of the chunk lives in TMEM lane 32 (m / 16) + m % 16 (lanes 0..15 of every quadrant);
    // columns [0,Cq) + [Cq,2Cq) = channels
    const int quad = warp & 3;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    // The chunk leaves as TMA stores of [16 channels x 64 px] boxes from a 4 KB staging buffer (issued by one thread, asynchronous):
    // 32 per-channel 64-byte global stores per warp kept these warps busy for ~1500 cycles per chunk and delayed the X images
    // of the next tile (60 us of the kernel).
    const uint32_t gxb = sb + L.gxb;
    auto gx_epilogue = [&](long qc, int tile_of, int q) {
      mbar_wait(d2_full, (uint32_t)qc & 1u);
      tc_fence_after();
      float r[Cq];
#pragma unroll
      for (int c0 = 0; c0 < Cq; c0 += 16) {
        float a[16], l[16];
        tmem_ld16(t_d2 + lane_base + (uint32_t)c0, a);
        tmem_ld16(t_d2 + lane_base + (uint32_t)(Cq + c0), l);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; i++) r[c0 + i] = a[i] + l[i];
      }
      tc_fence_before();
      warp_arrive(d2_empty);
      const int bimg = tile_of / p.tiles_per_img;
      const int pxc = (tile_of - bimg * p.tiles_per_img) * 128 + q * 64;        // first pixel of the chunk inside its image
      const int pl = quad * 16 + lane;                                          // pixel of the chunk (lanes 0..15 hold rows)
      if (p.dz && lane < 16) {
        const float* zp = p.dz + (size_t)bimg * p.Ci * p.P + (size_t)(pxc + pl);
#pragma unroll
        for (int c = 0; c < Cq; c++)
          if (c < p.Ci) r[c] *= hb_act_grad(__ldg(zp + (size_t)c * p.P), p.dact);
      }
#pragma unroll
      for (int c0 = 0; c0 < Cq; c0 += 16) {
        if (warp == 2 && lane == 0) tma_store_wait_read();                      // the staging buffer is free again
        asm volatile("bar.sync 2, 128;" ::: "memory");
        if (lane < 16) {
#pragma unroll
          for (int i = 0; i < 16; i++) sts_f32(gxb + (uint32_t)(i * 64 + pl) * 4u, r[c0 + i]);
        }
        fence_proxy_async();
        asm volatile("bar.sync 2, 128;" ::: "memory");
        if (warp == 2 && lane == 0) {
          tma_store_3d(&tmg, smem + L.gxb, pxc, c0, bimg);                      // channels >= Ci are clipped by the tensor map
          tma_store_commit();
        }
      }
    };
    const int cpt = NS / NB;                                                    // pixel chunks per tile (2)
    int it = 0;
    for (int tile = t_first; tile < t_end; tile++, it++) {
      mbar_wait(raw_full, (uint32_t)it & 1u);
      mbar_wait(xt_empty, ((uint32_t)it & 1u) ^ 1u);
      // the raw tile is read twice (8 channels at a time) instead of being held in 32 registers across the two waits
      for (int c0 = 0; c0 < Cq; c0 += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = lds_f32(sx + (uint32_t)(c0 + u) * 512u);
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const float4 hi = make_float4(v[4 * h], v[4 * h + 1], v[4 * h + 2], v[4 * h + 3]);
          const float4 lo = make_float4(tf32_lo(hi.x), tf32_lo(hi.y), tf32_lo(hi.z), tf32_lo(hi.w));
          sts_v4(xt_row + (uint32_t)(c0 / 4 + h) * 128u, hi);
          sts_v4(xt_row + L.xt_img + (uint32_t)(c0 / 4 + h) * 128u, lo);
        }
      }
      fence_proxy_async();
      warp_arrive(xt_full);
      mbar_wait(xk_empty, ((uint32_t)it & 1u) ^ 1u);
      for (int c0 = 0; c0 < Cq; c0 += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = lds_f32(sx + (uint32_t)(c0 + u) * 512u);
        const uint32_t gh = xk_col + (uint32_t)(c0 >> 3) * kHbSbo, gl = xk_col + (uint32_t)((Cq + c0) >> 3) * kHbSbo;
#pragma unroll
        for (int u = 0; u < 8; u++) {
          sts_f32(gh + (uint32_t)u * 16u, v[u]);
          sts_f32(gl + (uint32_t)u * 16u, tf32_lo(v[u]));
        }
      }
      fence_proxy_async();
      warp_arrive2(raw_empty, xk_full);
      if (it > 0) gx_epilogue((long)it * cpt - 1, tile - 1, cpt - 1);           // closed by the last step of the previous tile
      gx_epilogue((long)it * cpt, tile, 0);
    }
    if (it > 0) gx_epilogue((long)it * cpt - 1, t_end - 1, cpt - 1);
    if (warp == 2 && lane == 0) tma_store_wait_all();
  } else {
    // ===================== epilogue: 4 lane quadrants (hidden units) x 4 column parts (16 pixels of the chunk) =====================
    const int part = (warp - 6) >> 2;
    const int quad = warp & 3;
    const int jl = quad * 32 + lane;                                            // hidden unit inside the block
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float b1r[2], w2r[2];
    float2 dw2a[2], dsa[2];
#pragma unroll
    for (int b = 0; b < 2; b++) {
      const int j = b * 128 + jl;
      b1r[b] = (b < NB && j < p.H && p.b1) ? __ldg(p.b1 + j) : 0.f;
      w2r[b] = (b < NB && j < p.H) ? __ldg(p.w2 + j) : 0.f;
      dw2a[b] = make_float2(0.f, 0.f);
      dsa[b] = make_float2(0.f, 0.f);
    }
    float2 gsum = make_float2(0.f, 0.f);          // sum of this thread's 16 g columns over the steps of hidden block 0 (-> db2)
    const uint32_t fs_base = smem_u32(smem) + L.fs + (uint32_t)(2 * part) * kHbSbo + (uint32_t)(jl >> 2) * kHbLbo + (uint32_t)(jl & 3) * 4;
    int it = 0;
    long n = 0;
    for (int tile = t_first; tile < t_end; tile++, it++) {
      const uint32_t gs = smem_u32(smem) + L.g + (uint32_t)(it % 3) * 512u;
      for (int s = 0; s < NS; s++, n++) {
        const int q = NB == 2 ? (s >> 1) : s, b = NB == 2 ? (s & 1) : 0;
        mbar_wait(d1_full, (uint32_t)n & 1u);
        tc_fence_after();
        float v[16], gv[16];
        tmem_ld16(t_d1 + lane_base + (uint32_t)(16 * part), v);
#pragma unroll
        for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(gv + i) = lds_v4(gs + (uint32_t)(q * 64 + part * 16 + i) * 4u);
        tmem_ld_wait();
        tc_fence_before();
        warp_arrive(d1_empty);
        if (b == 0) {
#pragma unroll
          for (int i = 0; i < 16; i += 2) gsum = __fadd2_rn(gsum, make_float2(gv[i], gv[i + 1]));
        }
        const float b1j = b == 0 ? b1r[0] : b1r[1], w2j = b == 0 ? w2r[0] : w2r[1];
        float2 dw2v = b == 0 ? dw2a[0] : dw2a[1], dsv = b == 0 ? dsa[0] : dsa[1];
        if (GELU) {
          float2* v2 = reinterpret_cast<float2*>(v);
          const float2* g2 = reinterpret_cast<const float2*>(gv);
          const float2 bb = b2no_f2(b1j), ww = b2no_f2(w2j);
#pragma unroll
          for (int i = 0; i < 8; i++) {
            float2 val, grad;
            b2no_gelu2_both(__fadd2_rn(v2[i], bb), &val, &grad);
            dw2v = __ffma2_rn(g2[i], val, dw2v);
            const float2 t = __fmul2_rn(g2[i], grad);
            dsv = __fadd2_rn(dsv, t);
            v2[i] = __fmul2_rn(t, ww);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; i++) {
            const float z = v[i] + b1j;
            const float t = gv[i] * b2no_act_grad(z, p.act);
            if (i & 1) { dw2v.y = fmaf(gv[i], b2no_act(z, p.act), dw2v.y); dsv.y += t; }
            else { dw2v.x = fmaf(gv[i], b2no_act(z, p.act), dw2v.x); dsv.x += t; }
            v[i] = t * w2j;
          }
        }
        if (b == 0) { dw2a[0] = dw2v; dsa[0] = dsv; } else { dw2a[1] = dw2v; dsa[1] = dsv; }
        // F of the previous step must have been consumed by its G3 / G2
        mbar_wait(f_empty, ((uint32_t)n & 1u) ^ 1u);
        tc_fence_after();
        tmem_st16(t_f + lane_base + (uint32_t)(16 * part), v);
#pragma unroll
        for (int h = 0; h < 2; h++) {
          float fl[8];
#pragma unroll
          for (int i = 0; i < 8; i++) fl[i] = v[8 * h + i] - tf32_trunc(v[8 * h + i]);     // exact; the tensor core reads its top 19 bits
          tmem_st8(t_f + lane_base + 64u + (uint32_t)(16 * part + 8 * h), fl);
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const uint32_t off = (uint32_t)h * kHbSbo + (uint32_t)i * 16;
            sts_f32(fs_base + off, v[8 * h + i]);
            sts_f32(fs_base + L.fs_img + off, fl[i]);
          }
        }
        tmem_st_wait();
        fence_proxy_async();
        tc_fence_before();
        warp_arrive(f_full);
      }
    }
    // ---- read-out: dW1 from D3, dw2 / db1 from the register sums (column parts combined through shared memory) ----
    mbar_wait(done, 0);
    tc_fence_after();
    float* row = p.partial + (size_t)blockIdx.x * p.nsum;
    for (int b = 0; b < NB; b++) {
      const int j = b * 128 + jl;
      if (8 * part < Cq) {
        float a[8], l[8];
        tmem_ld8(t_d3 + lane_base + (uint32_t)(b * 2 * Cq + 8 * part), a);
        tmem_ld8(t_d3 + lane_base + (uint32_t)(b * 2 * Cq + Cq + 8 * part), l);
        tmem_ld_wait();
        if (j < p.H) {
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const int c = 8 * part + i;
            if (c < p.Ci) row[(size_t)j * p.Ci + c] = a[i] + l[i];
          }
        }
      }
    }
    // every MMA has completed (done): the F staging area is free.  The last F stores of the other epilogue threads are ordered
    // before this point through fs_full -> G2 -> done; the named barrier states the same thing in a form compute-sanitizer's
    // racecheck understands (it does not follow mbarrier / tcgen05.commit chains)
    asm volatile("bar.sync 1, %0;" ::"n"(kHbEpiThreads) : "memory");
    float* red = (float*)(smem + L.fs);                                        // [part][NB * 128][2]
#pragma unroll
    for (int b = 0; b < 2; b++) {
      if (b < NB) {
        const int j = b * 128 + jl;
        red[((size_t)part * NB * 128 + j) * 2 + 0] = dw2a[b].x + dw2a[b].y;
        red[((size_t)part * NB * 128 + j) * 2 + 1] = (dsa[b].x + dsa[b].y) * w2r[b];
      }
    }
    float* redg = red + (size_t)4 * NB * 128 * 2;                               // [part]: sum of g over this CTA's pixels
    if (jl == 0) redg[part] = gsum.x + gsum.y;
    asm volatile("bar.sync 1, %0;" ::"n"(kHbEpiThreads) : "memory");
    if (part == 0 && jl == 0) row[(size_t)p.H * p.Ci + 2 * p.H] = (redg[0] + redg[1]) + (redg[2] + redg[3]);   // db2
    if (part == 0) {
      for (int b = 0; b < NB; b++) {
        const int j = b * 128 + jl;
        if (j < p.H) {
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int q = 0; q < 4; q++) {
            s0 += red[((size_t)q * NB * 128 + j) * 2 + 0];
            s1 += red[((size_t)q * NB * 128 + j) * 2 + 1];
          }
          row[(size_t)p.H * p.Ci + j] = s1;              // db1
          row[(size_t)p.H * p.Ci + p.H + j] = s0;        // dw2
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tbase, ncols);
}

// deterministic sum of per-CTA partial rows (same scheme as tc_mlp.cu's k_sum_partials)
__global__ void __launch_bounds__(256)
k_hb_sum(const float* __restrict__ partial, float* __restrict__ out, int nblk, int n) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + lane;
  float s0 = 0.f, s1 = 0.f;
  if (idx < n) {
    int b = warp;
    for (; b + 8 < nblk; b += 16) {
      s0 += __ldg(partial + (size_t)b * n + idx);
      s1 += __ldg(partial + (size_t)(b + 8) * n + idx);
    }
    for (; b < nblk; b += 8) s0 += __ldg(partial + (size_t)b * n + idx);
  }
  red[warp][lane] = s0 + s1;
  __syncthreads();
  if (warp == 0 && idx < n) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; w8++) s += red[w8][lane];
    out[idx] = s;
  }
}

bool hb_shape_ok(int ci, int hidden, long pixels) {
  if (!b2no_tc_available()) return false;
  if (pixels < 128 || pixels % 128 != 0 || ci < 1 || ci > 32 || hidden < 1 || hidden > 256) return false;
  const int Cq = b2no_round_up(ci, 16), Hp = b2no_round_up(hidden, 128);
  if (hb_tmem_cols(Cq, Hp / 128) > 512) return false;
  int dev = 0, max_smem = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return false;
  return (int)hb_layout(Cq, Hp).total <= max_smem;
}

}  // namespace

void b2no_tc_count_launch();

extern "C" int b2no_mlp_head_bwd_fused_supported(int ci, int hidden, int64_t pixels) {
  return hb_shape_ok(ci, hidden, (long)pixels) ? 1 : 0;
}

extern "C" int64_t b2no_mlp_head_bwd_fused_scratch_floats(int ci, int hidden) {
  if (ci < 1 || hidden < 1) return B2NO_E_ARG;
  return (int64_t)b2no_sm_count() * ((int64_t)hidden * ci + 2 * hidden + 1);
}

extern "C" int b2no_mlp_head_bwd_fused(const float* x, const float* w1, const float* b1, const float* w2, const float* g,
                                       float* gx, float* grads, float* partial, int batch, int ci, int hidden,
                                       int64_t pixels, int act, const float* dact_z, int dact, void* stream) {
  if (!x || !w1 || !w2 || !g || !gx || !grads || !partial || batch < 1 || ci < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  if (!hb_shape_ok(ci, hidden, (long)pixels) || ((uintptr_t)x & 15) || ((uintptr_t)g & 15)) return B2NO_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  HeadBwd p;
  memset(&p, 0, sizeof(p));
  p.npass = b2no_tc_passes();
  p.B = batch; p.Ci = ci; p.Cq = b2no_round_up(ci, 16); p.H = hidden; p.Hp = b2no_round_up(hidden, 128); p.NB = p.Hp / 128;
  p.act = act; p.dz = dact_z; p.dact = dact_z ? dact : 0;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.g = g; p.gx = gx; p.partial = partial;
  p.P = (long)pixels;
  p.tiles_per_img = (int)(pixels / 128);
  const long tiles = (long)batch * p.tiles_per_img;
  if (tiles >= (1L << 30)) return B2NO_E_UNSUPPORTED;
  p.tiles = (int)tiles;
  p.nsum = hidden * ci + 2 * hidden + 1;
  int grid = p.tiles < b2no_sm_count() ? p.tiles : b2no_sm_count();
  p.tiles_per_cta = (p.tiles + grid - 1) / grid;
  grid = (p.tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  const HbLayout L = hb_layout(p.Cq, p.Hp);
  CUtensorMap tmx;
  uint64_t dims[3] = {(uint64_t)pixels, (uint64_t)ci, (uint64_t)batch};
  uint64_t str[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * ci};
  uint32_t box[3] = {128, (uint32_t)p.Cq, 1};
  if (make_tmap_f32(&tmx, x, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return B2NO_E_UNSUPPORTED;
  CUtensorMap tmg;
  uint32_t gbox[3] = {64, 16, 1};
  if (((uintptr_t)gx & 15) || make_tmap_f32(&tmg, gx, 3, dims, str, gbox, CU_TENSOR_MAP_SWIZZLE_NONE)) return B2NO_E_UNSUPPORTED;
#define HB_LAUNCH(G, C)                                                                                                   \
  do {                                                                                                                   \
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_head_bwd<G, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total)); \
    k_head_bwd<G, C><<<(unsigned)grid, kHbThreads, L.total, st>>>(tmx, tmg, p);                                              \
  } while (0)
  const bool gelu = act == B2NO_ACT_GELU;
  if (p.Cq == 32) { if (gelu) HB_LAUNCH(true, 32); else HB_LAUNCH(false, 32); }
  else { if (gelu) HB_LAUNCH(true, 16); else HB_LAUNCH(false, 16); }
#undef HB_LAUNCH
  B2NO_LAUNCH_CHECK();
  b2no_tc_count_launch();
  k_hb_sum<<<(p.nsum + 31) / 32, 256, 0, st>>>(partial, grads, (int)grid, p.nsum);
  B2NO_LAUNCH_CHECK();
  return 0;
}
