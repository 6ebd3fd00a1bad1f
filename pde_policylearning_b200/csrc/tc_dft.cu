// Truncated forward DFT of 2-D planes on the 5th-gen tensor cores (tcgen05 / TMEM), fed by TMA: replaces the
// rfftn + corner slicing of spectral_convolution.py:324-337, rno.py:67-74 (and, as the adjoint of the inverse, the
// backward of irfftn) for the planes that fit the tile shape.  Only the kept modes are ever produced.
//
//   stage 1 (W axis, real -> complex):   A[h, q]    = sum_w x[h, w] T[q, w]                q = (2 ky | 2 ky + 1) = (re | im)
//   stage 2 (H axis, complex):           Xh[kx, ky] = sum_h M[h, kx] (A[h, 2ky] + i A[h, 2ky+1])
//
// One tile = 128 consecutive rows of the [planes * H, W] matrix (R = 128 / H planes), exactly as it lies in HBM:
//   stage 1:  D1[128 rows, N1]     = X[128 x W] (A operand, TMEM, K-major as stored)  x  T[N1 x W]^T (smem, constant)
//             the X tile arrives as W/32 TMA boxes [32 floats x 128 rows] (128B swizzle); converter warps (thread = row)
//             move it to TMEM as hi (raw fp32, the tensor core reads the top 19 bits) and lo = rna_tf32(x - trunc x)
//   hand-over: epilogue warps (thread = row h) read D1 from TMEM, split hi/lo, and store it as the K-major B operand
//             of stage 2 ([q][h], conflict-free: K chunks padded to 144 B)
//   stage 2:  D2[128, N1] (per plane) = Mt[128 x H] (A operand, TMEM, constant: lane kx = Re M[., kx], lane 32 + kx = Im)
//                                         x  A[N1 x H]^T (smem)
//             Xh[kx, ky] = (D2[kx, 2ky] - D2[32+kx, 2ky+1]) + i (D2[kx, 2ky+1] + D2[32+kx, 2ky])
// All products 3xTF32 (hi*hi + lo*hi + hi*lo).  512 threads, persistent CTAs over contiguous tile ranges; warp roles are
// listed at the kernel (two converter groups alternate K chunks; stage 1 of tile t+1 is issued before stage 2 of tile t;
// hand-over and spectrum write-out run in different warps).  The constant Mt operand arrives by ONE bulk copy issued
// ahead of the x stream.  HBM-bound by design: per plane the tensor pipe needs ~800 cycles, shared memory ~1100,
// HBM ~2900 (64 KB at 44 GB/s/SM).  Measured (B200, cfg2, 134 MB): 37.6 us = 3.6 TB/s; 4.2 TB/s at 4x the batch.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

constexpr int kThreadsFd = 512;
constexpr uint32_t kB2Lbo = 144;            // bytes between K-adjacent core matrices of the stage-2 B operand (padded: no bank conflicts)
constexpr uint32_t kB2Sbo = 32 * kB2Lbo;    // bytes between 8-row groups (128 lanes = 32 K chunks)

struct FdTc {
  int W, H, R, nk, N1, Kx, Ky, S;
  int MG;      // 1: the hi*hi and hi*lo products of a K step run as ONE MMA against the stacked [hi; lo] B operand (N = 2 N1)
  long tiles, tiles_per_cta, planes;
  const float* tb; const float* mimg;
  float* spec;
  int npass;   // 3: 3xTF32, 1: single-pass TF32 (never merged)
  int layout;  // 0: spectrum (plane, kx, ky); 1: mode-major (kx, ky, plane)
};

struct FdLayout { uint32_t tbh, tbl, b2, b2_bytes, xch, mts, mts_stride, stages, bars, total; };

__host__ __device__ inline FdLayout fd_layout(const FdTc& p) {
  FdLayout L;
  uint32_t o = 0;
  const uint32_t tbb = (uint32_t)p.N1 * p.W * 4;
  L.tbh = o; o += tbb; L.tbl = o; o += tbb;
  L.b2_bytes = (uint32_t)(p.N1 / 8) * kB2Sbo;          // one (hi or lo) image
  o = (o + 127u) & ~127u;
  L.b2 = o; o += 4 * L.b2_bytes;                        // [buf 0/1][hi, lo]
  L.xch = o; o += 2u * p.R * 32 * p.N1 * 4;             // [buf 0/1][plane][kx][N1]: Im-row partial sums
  L.mts_stride = (uint32_t)(p.H + 4) * 4;               // staging rows of the constant Mt operand, padded (no bank conflicts)
  o = (o + 127u) & ~127u;
  L.mts = o; o += 4u * p.Kx * L.mts_stride;             // [hi | lo][Re rows | Im rows], one bulk copy
  o = (o + 1023u) & ~1023u;
  L.stages = o; o += (uint32_t)p.S * 16384;
  L.bars = o; o += 8 * (2 * p.S + 20) + 16;
  L.total = o + 1024;
  return L;
}

// warp roles (16 warps; a warp may only touch TMEM lanes 32 * (warp % 4) .. + 31)
//   0-3   converter A (even K chunks)      4-7  converter B (odd K chunks)      8-9  spectrum write-out (lanes 0-63)
//   10    TMA producer                     11   MMA issuer                      12-15 hand-over D1 -> stage-2 B operand
__global__ void __launch_bounds__(kThreadsFd, 1)
k_fwd_tc(const __grid_constant__ CUtensorMap tmx, const FdTc p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const FdLayout L = fd_layout(p);
  uint64_t* full = (uint64_t*)(smem + L.bars);
  uint64_t* empty = full + p.S;
  uint64_t* xa_full = empty + p.S;
  uint64_t* xa_empty = xa_full + 2;
  uint64_t* d1_full = xa_empty + 2;
  uint64_t* d1_empty = d1_full + 2;
  uint64_t* b2_full = d1_empty + 2;
  uint64_t* b2_empty = b2_full + 2;
  uint64_t* d2_full = b2_empty + 2;
  uint64_t* d2_empty = d2_full + 2;
  uint64_t* mt_ready = d2_empty + 2;
  uint64_t* mt_staged = mt_ready + 1;
  uint32_t* tslot = (uint32_t*)(mt_staged + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N1 = p.N1, H = p.H, R = p.R, nk = p.nk;

  // ---- one-time setup ----
  {
    const float4* src = (const float4*)p.tb;
    float4* dst = (float4*)(smem + L.tbh);
    for (int i = tid; i < 2 * N1 * p.W / 4; i += kThreadsFd) dst[i] = __ldg(src + i);
  }
  if (tid == 0) {
    for (int s = 0; s < p.S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 128); }
    for (int a = 0; a < 2; a++) {
      mbar_init(&xa_full[a], 128); mbar_init(&xa_empty[a], 1);
      mbar_init(&d1_full[a], 1); mbar_init(&d1_empty[a], 128);
      mbar_init(&b2_full[a], 128); mbar_init(&b2_empty[a], 1);
      mbar_init(&d2_full[a], 1); mbar_init(&d2_empty[a], 64);
    }
    mbar_init(mt_ready, 128);
    mbar_init(mt_staged, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 11) tmem_alloc(tslot, 512);
  if (warp == 10 && lane == 0) tma_prefetch_desc(&tmx);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  // TMEM columns: [xa: 2 x (32 hi | 32 lo)] [d1: 2 x ND] [mt: H hi | H lo] [d2: 2 x R*ND], ND = N1 or (merged) 2 N1.
  // A tcgen05.mma of this shape costs ~40 cycles whatever its N (TMEM A-operand fetch), and this kernel's steady state was
  // exactly its 96 MMAs per tile; the B operands already hold their hi and lo images back to back with one row-group
  // stride, so A_hi x [B_hi; B_lo] is one instruction with N = 2 N1 and the two accumulator halves are added by the
  // threads that read them anyway: 64 MMAs per tile.
  const int ND = p.MG ? 2 * N1 : N1;
  const uint32_t t_xa = tbase, t_d1 = tbase + 128u, t_mt = t_d1 + 2u * ND, t_d2 = t_mt + 2u * H;
  const long t_first = (long)blockIdx.x * p.tiles_per_cta;
  const long t_end = t_first + p.tiles_per_cta < p.tiles ? t_first + p.tiles_per_cta : p.tiles;
  const int ntiles = (int)(t_end > t_first ? t_end - t_first : 0);
  const int quad = warp & 3;
  const int m = quad * 32 + lane;                          // TMEM lane = tile row handled by this thread
  const uint32_t lane_base = (uint32_t)(quad * 32) << 16;

  if (warp == 10) {
    // ===================== TMA producer: W/32 boxes [32 floats x 128 rows] per tile =====================
    if (lane == 0) {
      // the constant stage-2 operand first (ahead of the x stream in the memory queues), one bulk copy
      mbar_arrive_expect_tx(mt_staged, 4u * p.Kx * L.mts_stride);
      bulk_load(smem + L.mts, p.mimg, 4u * p.Kx * L.mts_stride, mt_staged);
      long g = 0;
      for (int it = 0; it < ntiles; it++) {
        const long tile = t_first + it;
        for (int c = 0; c < nk; c++, g++) {
          const int s = (int)(g % p.S);
          mbar_wait(&empty[s], ((uint32_t)(g / p.S) & 1u) ^ 1u);
          mbar_arrive_expect_tx(&full[s], 16384);
          tma_load_2d(smem + L.stages + (size_t)s * 16384, &tmx, &full[s], c * 32, (int)(tile * 128));
        }
      }
    }
  } else if (warp == 11) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = idesc_tf32(128, N1, 0, 0), idesc2 = idesc_tf32(128, 2 * N1, 0, 0);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t sbo1 = (uint32_t)(p.W / 4) * 128;
    const uint64_t d_th = smem_desc(sbase + L.tbh, 128, sbo1, LAYOUT_NONE), d_tl = smem_desc(sbase + L.tbl, 128, sbo1, LAYOUT_NONE);
    long g = 0;
    auto stage1 = [&](int it) {
      const int db = it & 1;
      for (int c = 0; c < nk; c++, g++) {
        const int xb = (int)(g & 1);
        mbar_wait(&xa_full[xb], (uint32_t)(g >> 1) & 1u);
        if (c == 0) mbar_wait(&d1_empty[db], ((uint32_t)(it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d = t_d1 + (uint32_t)(db * ND);
          const uint32_t xa = t_xa + 64u * xb;
          if (p.MG) {
            // x_hi * [T_hi; T_lo] (N = 2 N1), then x_lo * T_hi into the first half
            const uint64_t dt = d_th + (uint64_t)(c * 64);
#pragma unroll
            for (int j = 0; j < 4; j++) mma_tf32_ts(d, xa + 8 * j, dt + (uint64_t)(j * 16), idesc2, (c > 0 || j > 0) ? 1u : 0u);
#pragma unroll
            for (int j = 0; j < 4; j++) mma_tf32_ts(d, xa + 32 + 8 * j, dt + (uint64_t)(j * 16), idesc, 1u);
          } else {
            _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
              if (pass >= p.npass) break;
              const uint32_t ac = pass == 1 ? xa + 32 : xa;
              const uint64_t dt = (pass == 2 ? d_tl : d_th) + (uint64_t)(c * 64);     // 32 K elements = 8 chunks of 128 B
#pragma unroll
              for (int j = 0; j < 4; j++)
                mma_tf32_ts(d, ac + 8 * j, dt + (uint64_t)(j * 16), idesc, (c > 0 || pass > 0 || j > 0) ? 1u : 0u);
            }
          }
          mma_commit(&xa_empty[xb]);
          if (c == nk - 1) mma_commit(&d1_full[db]);
        }
        __syncwarp();
      }
    };
    auto stage2 = [&](int it) {
      const int db = it & 1;
      mbar_wait(&b2_full[db], (uint32_t)(it >> 1) & 1u);
      mbar_wait(&d2_empty[db], ((uint32_t)(it >> 1) & 1u) ^ 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t bh = sbase + L.b2 + (uint32_t)db * 2 * L.b2_bytes, bl = bh + L.b2_bytes;
        for (int r = 0; r < R; r++) {
          const uint32_t d = t_d2 + (uint32_t)((db * R + r) * ND);
          if (p.MG) {
            // Mt_hi * [A_hi; A_lo] (the lo image follows the hi image at the row-group stride), then Mt_lo * A_hi
            const uint64_t db2 = smem_desc(bh + (uint32_t)(r * H / 4) * kB2Lbo, kB2Lbo, kB2Sbo, LAYOUT_NONE);
            for (int j = 0; j < H / 8; j++)
              mma_tf32_ts(d, t_mt + 8 * j, db2 + (uint64_t)(j * (2 * kB2Lbo / 16)), idesc2, j > 0 ? 1u : 0u);
            for (int j = 0; j < H / 8; j++)
              mma_tf32_ts(d, t_mt + H + 8 * j, db2 + (uint64_t)(j * (2 * kB2Lbo / 16)), idesc, 1u);
          } else {
            _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
              const uint32_t am = pass == 1 ? t_mt + H : t_mt;
              const uint32_t bb = (pass == 2 ? bl : bh) + (uint32_t)(r * H / 4) * kB2Lbo;
              const uint64_t db2 = smem_desc(bb, kB2Lbo, kB2Sbo, LAYOUT_NONE);
              for (int j = 0; j < H / 8; j++)
                mma_tf32_ts(d, am + 8 * j, db2 + (uint64_t)(j * (2 * kB2Lbo / 16)), idesc, (pass > 0 || j > 0) ? 1u : 0u);
            }
          }
        }
        mma_commit(&b2_empty[db]);
        mma_commit(&d2_full[db]);
      }
      __syncwarp();
    };
    for (int it = 0; it < ntiles; it++) {
      stage1(it);
      if (it == 1) { mbar_wait(mt_ready, 0); tc_fence_after(); }
      if (it > 0) stage2(it - 1);
    }
    if (ntiles == 1) { mbar_wait(mt_ready, 0); tc_fence_after(); }
    if (ntiles > 0) stage2(ntiles - 1);
  } else if (warp < 8) {
    // ===================== converters: thread = row; shared memory (swizzled box) -> TMEM A operand =====================
    // group A (warps 0-3) takes the even chunks / TMEM buffer 0, group B (warps 4-7) the odd chunks / buffer 1
    const int grp = warp >> 2;
    const long total = (long)ntiles * nk;
    for (long g = grp; g < total; g += 2) {
      const int s = (int)(g % p.S);
      mbar_wait(&full[s], (uint32_t)(g / p.S) & 1u);
      const uint8_t* row = smem + L.stages + (size_t)s * 16384 + (size_t)m * 128;
      float hi[32], lo[32];
#pragma unroll
      for (int i = 0; i < 8; i++)
        *reinterpret_cast<float4*>(hi + 4 * i) = *reinterpret_cast<const float4*>(row + ((i ^ (m & 7)) << 4));
      mbar_arrive(&empty[s]);
#pragma unroll
      for (int i = 0; i < 32; i++) lo[i] = tf32_lo(hi[i]);
      mbar_wait(&xa_empty[grp], ((uint32_t)(g >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t xa = t_xa + lane_base + 64u * grp;
      tmem_st16(xa, hi); tmem_st16(xa + 16, hi + 16);
      tmem_st16(xa + 32, lo); tmem_st16(xa + 48, lo + 16);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&xa_full[grp]);
    }
  } else if (warp >= 12) {
    // ===================== hand-over: D1 (TMEM) -> hi/lo K-major B operand of stage 2 (shared memory) =====================
    // first, once: the constant stage-2 A operand Mt.  Rows kx (Re) and 32 + kx (Im) are staged through shared memory
    // with coalesced loads (one L2 round trip per pass), then every thread moves ITS lane's row into TMEM.
    {
      const int Kx = p.Kx;
      float* mts = (float*)(smem + L.mts);
      const int rs = (int)(L.mts_stride / 4);
      mbar_wait(mt_staged, 0);
      const int r = m < Kx ? m : ((m >= 32 && m < 32 + Kx) ? Kx + (m - 32) : -1);
      for (int pass = 0; pass < 2; pass++) {
        const float* src = mts + (size_t)pass * 2 * Kx * rs;
        for (int c0 = 0; c0 < H; c0 += 8) {
          float v[8];
          if (r >= 0) {
            *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(src + (size_t)r * rs + c0);
            *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(src + (size_t)r * rs + c0 + 4);
          } else {
#pragma unroll
            for (int j = 0; j < 8; j++) v[j] = 0.f;
          }
          tmem_st8(t_mt + lane_base + (uint32_t)(pass * H + c0), v);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(mt_ready);
    }
    for (int it = 0; it < ntiles; it++) {
      const int db = it & 1;
      mbar_wait(&d1_full[db], (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      float v[32];
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 8)
        if (c0 < N1) tmem_ld8(t_d1 + lane_base + (uint32_t)(db * ND + c0), v + c0);
      if (p.MG) {
        tmem_ld_wait();
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 8) {
          if (c0 < N1) {
            float u[8];
            tmem_ld8(t_d1 + lane_base + (uint32_t)(db * ND + N1 + c0), u);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 8; q++) v[c0 + q] += u[q];
          }
        }
      }
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&d1_empty[db]);
      mbar_wait(&b2_empty[db], ((uint32_t)(it >> 1) & 1u) ^ 1u);
      uint8_t* bh = smem + L.b2 + (size_t)db * 2 * L.b2_bytes;
      uint8_t* bl = bh + L.b2_bytes;
      const uint32_t koff = (uint32_t)(m >> 2) * kB2Lbo + (uint32_t)(m & 3) * 4;
#pragma unroll
      for (int q = 0; q < 32; q++) {
        if (q < N1) {
          const uint32_t off = (uint32_t)(q >> 3) * kB2Sbo + (uint32_t)(q & 7) * 16 + koff;
          *(float*)(bh + off) = v[q];
          *(float*)(bl + off) = tf32_lo(v[q]);
        }
      }
      fence_proxy_async();
      mbar_arrive(&b2_full[db]);
    }
  } else {
    // ===================== spectrum write-out (warps 8, 9 = TMEM lanes 0-31 Re rows, 32-63 Im rows) =====================
    const int Ky = p.Ky, Kx = p.Kx;
    for (int it = 0; it < ntiles; it++) {
      const int db = it & 1;
      const long tile = t_first + it;
      float* xch = (float*)(smem + L.xch) + (size_t)db * R * 32 * N1;
      mbar_wait(&d2_full[db], (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      if (quad == 1) {
        // Im rows: lane kx holds sum_h Im M[h, kx] * (A re | A im)
        for (int r = 0; r < R; r++) {
          float v[32];
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 8)
            if (c0 < N1) tmem_ld8(t_d2 + lane_base + (uint32_t)((db * R + r) * ND + c0), v + c0);
          if (p.MG) {
            tmem_ld_wait();
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 8) {
              if (c0 < N1) {
                float u[8];
                tmem_ld8(t_d2 + lane_base + (uint32_t)((db * R + r) * ND + N1 + c0), u);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 8; q++) v[c0 + q] += u[q];
              }
            }
          }
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 32; q++)
            if (q < N1) xch[((size_t)r * 32 + lane) * N1 + q] = v[q];
        }
        tc_fence_before();
        mbar_arrive(&d2_empty[db]);
        asm volatile("bar.sync 2, 64;" ::: "memory");
      } else {
        asm volatile("bar.sync 2, 64;" ::: "memory");
        for (int r = 0; r < R; r++) {
          float v[32];
#pragma unroll
          for (int c0 = 0; c0 < 32; c0 += 8)
            if (c0 < N1) tmem_ld8(t_d2 + lane_base + (uint32_t)((db * R + r) * ND + c0), v + c0);
          if (p.MG) {
            tmem_ld_wait();
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 8) {
              if (c0 < N1) {
                float u[8];
                tmem_ld8(t_d2 + lane_base + (uint32_t)((db * R + r) * ND + N1 + c0), u);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 8; q++) v[c0 + q] += u[q];
              }
            }
          }
          tmem_ld_wait();
          const long plane = tile * R + r;
          if (lane < Kx && plane < p.planes) {
            const float* im = xch + ((size_t)r * 32 + lane) * N1;
            if (p.layout == 0) {
              float2* dst = (float2*)p.spec + ((size_t)plane * Kx + lane) * Ky;
#pragma unroll
              for (int ky = 0; ky < 16; ky++)
                if (ky < Ky) dst[ky] = make_float2(v[2 * ky] - im[2 * ky + 1], v[2 * ky + 1] + im[2 * ky]);
            } else {
              // mode-major: the R planes of a tile are consecutive channels of one sample, so the R stores of a mode fall
              // into one or two 32-byte sectors (merged in L2); same number of store instructions as the default layout
              float2* dst = (float2*)p.spec + (size_t)lane * Ky * p.planes + plane;
#pragma unroll
              for (int ky = 0; ky < 16; ky++)
                if (ky < Ky) dst[(size_t)ky * p.planes] = make_float2(v[2 * ky] - im[2 * ky + 1], v[2 * ky + 1] + im[2 * ky]);
            }
          }
        }
        tc_fence_before();
        mbar_arrive(&d2_empty[db]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 11) tmem_dealloc(tbase, 512);
}

}  // namespace

void b2no_tc_count_launch();

// Returns 0 when the kernel ran, 1 when the shape is not eligible (caller uses the CUDA-core stages), else an error.
int b2no_tc_dft_forward(const b2no_plan* plan, int which, const float* x, float* spec, long planes, cudaStream_t st) {
  if (!b2no_tc_available() || !plan || plan->g.ndim != 2) return 1;
  const b2no_tc_fwd_tables& tf = plan->tcf[which];
  if (!tf.tb || !tf.mimg) return 1;
  if ((uintptr_t)x & 15) return 1;
  FdTc p;
  memset(&p, 0, sizeof(p));
  p.W = tf.W; p.H = tf.H; p.R = 128 / tf.H; p.nk = tf.W / 32; p.N1 = tf.N1; p.Kx = tf.Kx; p.Ky = tf.Ky;
  p.planes = planes;
  const long rows = planes * tf.H;
  p.tiles = (rows + 127) / 128;
  p.tb = tf.tb; p.mimg = tf.mimg; p.spec = spec; p.layout = plan->g.spec_layout;
  p.npass = b2no_tc_passes();
  p.MG = (128u + 4u * p.N1 + 2u * p.H + 4u * p.R * p.N1 <= 512u && p.npass == 3) ? 1 : 0;
  if (!p.MG && 128u + 2u * p.N1 + 2u * p.H + 2u * p.R * p.N1 > 512u) return 1;
  int dev = 0, max_smem = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  B2NO_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  FdLayout L;
  for (p.S = 10; p.S >= 3; p.S--) {
    L = fd_layout(p);
    if ((int)L.total <= max_smem) break;
  }
  if (p.S < 3) return 1;
  CUtensorMap tmx;
  {
    uint64_t dims[2] = {(uint64_t)p.W, (uint64_t)rows};
    uint64_t str[2] = {4, (uint64_t)p.W * 4};
    uint32_t box[2] = {32, 128};
    if (make_tmap_f32(&tmx, x, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  long grid = p.tiles < b2no_sm_count() ? p.tiles : b2no_sm_count();
  p.tiles_per_cta = (p.tiles + grid - 1) / grid;
  grid = (p.tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  k_fwd_tc<<<(unsigned)grid, kThreadsFd, L.total, st>>>(tmx, p);
  B2NO_LAUNCH_CHECK();
  b2no_tc_count_launch();
  return 0;
}
