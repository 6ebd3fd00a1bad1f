// Fused pixel-tile kernel on the 5th-gen tensor cores (tcgen05 / TMEM), fed by TMA.
//
//   out[b, o, p] = act( sum_i W1[o,i] X1[b,i,p] + sum_i W2[o,i] X2[b,i,p]            1x1 convolutions
//                       + sum_q T[p, q] A'[b, row(p), q, o]                            last inverse-DFT stage
//                       + bias[o] + add[b,o,p] ) * mul[b,o,p] * dact'(dz[b,o,p])
//
// One tile = 128 consecutive pixels of one sample = the M dimension of every MMA (TMEM lane = pixel), the
// output channels are N (TMEM columns), the input channels / spectral index q are K.  All three sums
// accumulate into the SAME TMEM tile, so the FNO layer (spectral_convolution.py:342-345 + fno_block.py:131-150),
// the RNO FourierLayer2d (rno.py:224-228) and their dx adjoints are one pass over HBM: read x once, write y once.
//
// Operand placement (measured on B200, see DESIGN.md): feeding the pixel tile to the tensor core from shared
// memory costs one 4 KB A-read per MMA and made the MMAs the bottleneck, so the A operands live in TMEM:
//   - X tile: TMA box [C x 128 px] -> shared memory -> converter warps (thread = pixel) -> tcgen05.st as
//     K-major A [128 lanes x C columns], hi (raw fp32; the tensor core reads only the upper 19 bits) and
//     lo = rna_tf32(x - trunc(x));
//   - T (block-diagonal last-dim inverse table, constant): loaded into TMEM once per CTA, hi and lo;
//   - B operands (1x1 weights, A' rows) stay in shared memory, K-major no-swizzle core-matrix layout.
// fp32 parity: every product is issued three times (3xTF32: hi*hi + lo*hi + hi*lo), error 4e-7 (tools/tc_probe.cu).
//
// Warp roles (704 threads, persistent CTAs, each CTA owns a contiguous run of tiles):
//   warp 0      TMA producer (X boxes, cp.async.bulk for the A' rows), S-deep mbarrier ring
//   warp 1      MMA issuer (one lane): tcgen05.mma.kind::tf32 TS form, tcgen05.commit -> mbarriers
//   warps 2-5   converter: shared memory -> TMEM A operand (double buffered)
//   warps 6-21  epilogue: two groups of eight warps on alternate tiles (r2; round 1: all sixteen on each tile, 4 lane quadrants x 4 column parts of 8 channels: the
//               epilogue is a latency chain -- tcgen05.ld, GELU, 128-byte stores per channel row -- and eight warps
//               left the issue slots half empty), tcgen05.ld -> bias/act -> coalesced global stores;
//               two TMEM accumulators so the MMAs of tile i+1 overlap the epilogue of tile i.  MODE 3 fetches the
//               saved pre-activations of the NEXT tile before it waits for the current accumulator.
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

constexpr int kParts = 2;                       // column parts of one epilogue group (kParts x 4 warps); two groups take alternate tiles
constexpr int kGroups = 2;
constexpr int kCW = 8;                          // output channels per epilogue thread per pass
constexpr int kEpiThreadsPw = 128 * kParts * kGroups;
constexpr int kGroupThreadsPw = 128 * kParts;   // the threads that work on one tile (= arrivals on its barriers)
constexpr int kThreads = 192 + kEpiThreadsPw;

struct PwTc {
  int B, Co, Np, C1, C1p, C2, C2p, Ks, Qp, R, S;
  int NA;             // TMEM A-operand buffers: 2 (conversion of tile i+1 overlaps the MMAs of tile i), or 1 when two do not fit
  int Cz;             // > 0: MODE 3 streams the saved pre-activations dz through the TMA ring, [Cz x 128 px] per stage
  int tiles_per_img;
  long tiles, tiles_per_cta, P;
  const float* w1; int w1_t;
  const float* w2; int w2_t;
  const float* ahi; const float* alo; const float* timg;
  const float* bias; const float* add; const float* mul; const float* dz;
  const float* gate_z; const float* gate_h;
  long mul_bs, gate_bs;   // floats between consecutive samples of mul / gate_z
  float* preact; float* y;
  int act, dact;
  int npass;          // 3: 3xTF32, 1: single-pass TF32 (hi * hi only)
  // 3-D mode (zlen > 0): rows of the last dim have zlen points, a 128-pixel tile touches up to R = 127 / zlen + 2 of them.
  // The last-stage operand T[pixel, (row slot, q)] then depends on where the tile starts, so the converter warps build it
  // per tile from the plan's [q][z] table (staged hi / lo in shared memory) instead of loading one constant image.
  int zlen, q2, tz_npad;
  long RPI;           // rows per sample (n0 * n1)
  const float* tz;
  // Weight-gradient variant (k_pw_tc<MODE, true>, 2-D dx passes): dWp[o, i] = sum_p X1[o, p] XW[i, p], db[o] = sum_p X1[o, p]
  // over the tiles of the CTA, written as per-CTA partials.  MW = M of those MMAs (64 or 128 >= the 2 C1p rows [X1 hi ; X1 lo];
  // the rows past them read whatever follows in the stage and land in accumulator rows nobody reads), NW = their N
  // ([XW hi ; XW lo ; ones], Cxp = XW channels rounded up to 8; the ones block makes db an accumulator column); 0 in the
  // plain kernel.
  int MW, NW, Cx, Cxp;
  float* wpart;
};

struct PwLayout {
  uint32_t w1h, w1l, w2h, w2l, bias, tzh, tzl, stages, stage_bytes, x2, xw, ah, al, dz, bars, total;
};

// WG (compile-time, so that the plain kernels' code does not depend on the variant): the weight-gradient variant, where X1
// arrives as four SW128 boxes [32 px x C1p], each followed by its lo copy (2 C1p rows per box), then four XW boxes of NW rows
template <bool WG>
__host__ __device__ inline PwLayout pw_layout(const PwTc& p) {
  PwLayout L;
  const uint32_t wb1 = (uint32_t)p.Np * p.C1p * 4, wb2 = (uint32_t)p.Np * p.C2p * 4;
  const uint32_t xb1 = (uint32_t)p.C1p * (WG ? 1024 : 512), xb2 = (uint32_t)p.C2p * 512;
  const uint32_t xwb = WG ? (uint32_t)p.NW * 512 : 0u, ab = (uint32_t)p.Ks * p.Np * 4;
  uint32_t o = 0;
  L.w1h = o; o += wb1; L.w1l = o; o += wb1;
  L.w2h = o; o += wb2; L.w2l = o; o += wb2;
  L.bias = o; o += (uint32_t)p.Np * 4;
  L.tzh = o; o += (uint32_t)p.Qp * p.zlen * 4;       // 3-D mode: last-dim table [q][z], hi then lo
  L.tzl = o; o += (uint32_t)p.Qp * p.zlen * 4;
  o = (o + 1023u) & ~1023u;
  L.stages = o;
  L.x2 = xb1; L.xw = xb1 + xb2; L.ah = L.xw + xwb; L.al = L.ah + ab;
  L.dz = (L.al + ab + 127u) & ~127u;
  L.stage_bytes = (L.dz + (uint32_t)p.Cz * 512 + 1023u) & ~1023u;
  o += L.stage_bytes * p.S;
  L.bars = o;
  o += 8 * (2 * p.S + 8 + (WG ? 1 : 0)) + 16;
  L.total = o + 1024;  // slack for the manual 1024-byte alignment of the dynamic window
  return L;
}

__host__ __device__ inline uint32_t pw_tmem_cols_dx(const PwTc& p) {
  if (p.zlen) return 2u * p.Np + (uint32_t)p.NA * (2u * (p.C1p + p.C2p) + 2u * p.Ks);   // T lives in the per-tile operand buffer
  return 2u * p.Np + 2u * p.Ks + 2u * (uint32_t)p.NA * (p.C1p + p.C2p);
}
// weight-gradient variant: its [MW x NW] accumulator follows, 32-column aligned
__host__ __device__ inline uint32_t pw_tmem_wcol(const PwTc& p) { return (pw_tmem_cols_dx(p) + 31u) & ~31u; }
template <bool WG>
__host__ __device__ inline uint32_t pw_tmem_cols(const PwTc& p) { return WG ? pw_tmem_wcol(p) + p.NW : pw_tmem_cols_dx(p); }

// MODE 1: no activation;  2: GELU;  3: multiply by GELU'(dz);  0: generic (runtime act / dact, add, mul)
template <int MODE>
__device__ __forceinline__ float epi_value(float z, float mulv, float dzv, int act, int dact) {
  if (MODE == 1) return z;
  if (MODE == 2) return b2no_act(z, B2NO_ACT_GELU);
  if (MODE == 3) return z * dzv;   // dzv already holds GELU'(dz) (packed evaluation in the epilogue)
  float v = b2no_act(z, act) * mulv;
  if (dact) v *= b2no_act_grad(dzv, dact);
  return v;
}

// WG: also the 1x1 weight gradient of the dx pass (MODE 1 only; see PwTc::MW; tm2 is then the XW map, there is no second
// 1x1 operand)
template <int MODE, bool WG>
__global__ void __launch_bounds__(kThreads, 1)
k_pw_tc(const __grid_constant__ CUtensorMap tm1, const __grid_constant__ CUtensorMap tm2, const __grid_constant__ CUtensorMap tm3,
        const PwTc p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const PwLayout L = pw_layout<WG>(p);
  uint64_t* full = (uint64_t*)(smem + L.bars);
  uint64_t* empty = full + p.S;
  uint64_t* a_full = empty + p.S;
  uint64_t* a_empty = a_full + 2;
  uint64_t* acc_full = a_empty + 2;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* wdone = acc_empty + 2;                       // WG only
  uint32_t* tslot = (uint32_t*)(acc_empty + 2 + (WG ? 1 : 0));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t ncols = 32;
  while (ncols < pw_tmem_cols<WG>(p)) ncols <<= 1;

  // ---- one-time setup: weights (hi/lo, K-major core-matrix layout), bias, barriers, TMEM ----
  for (int i = tid; i < p.Np * p.C1p; i += kThreads) {
    const int n = i / p.C1p, k = i - n * p.C1p;
    float w = 0.f;
    if (n < p.Co && k < p.C1) w = p.w1_t ? p.w1[(size_t)k * p.Co + n] : p.w1[(size_t)n * p.C1 + k];
    const float hi = tf32_rna(w);
    *(float*)(smem + L.w1h + kmajor_off(n, k, p.C1p)) = hi;
    *(float*)(smem + L.w1l + kmajor_off(n, k, p.C1p)) = tf32_rna(w - hi);
  }
  for (int i = tid; i < p.Np * p.C2p; i += kThreads) {
    const int n = i / p.C2p, k = i - n * p.C2p;
    float w = 0.f;
    if (n < p.Co && k < p.C2) w = p.w2_t ? p.w2[(size_t)k * p.Co + n] : p.w2[(size_t)n * p.C2 + k];
    const float hi = tf32_rna(w);
    *(float*)(smem + L.w2h + kmajor_off(n, k, p.C2p)) = hi;
    *(float*)(smem + L.w2l + kmajor_off(n, k, p.C2p)) = tf32_rna(w - hi);
  }
  for (int i = tid; i < p.Np; i += kThreads) ((float*)(smem + L.bias))[i] = (p.bias && i < p.Co) ? p.bias[i] : 0.f;
  for (int i = tid; i < p.Qp * p.zlen; i += kThreads) {
    const int q = i / p.zlen, z = i - q * p.zlen;
    const float v = q < p.q2 ? p.tz[(size_t)q * p.tz_npad + z] : 0.f;
    const float hi = tf32_rna(v);
    ((float*)(smem + L.tzh))[i] = hi;
    ((float*)(smem + L.tzl))[i] = tf32_rna(v - hi);
  }
  if (WG) {
    // the rows no TMA box writes: the lo copies start (and in single-pass mode stay) zero, the ones block of every XW box
    // stays 1
    for (uint32_t i = tid; i < (uint32_t)p.S * L.stage_bytes / 16u; i += kThreads)
      *(float4*)(smem + L.stages + i * 16u) = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    const uint32_t ones = (uint32_t)(p.NW - 2 * p.Cxp) * 8u;   // float4 per box
    for (uint32_t i = tid; i < (uint32_t)p.S * 4u * ones; i += kThreads) {
      const uint32_t s = i / (4u * ones), r = i - s * 4u * ones, j = r / ones;
      *(float4*)(smem + L.stages + s * L.stage_bytes + L.xw + j * (uint32_t)p.NW * 128u + (uint32_t)p.Cxp * 256u + (r - j * ones) * 16u) =
          make_float4(1.f, 1.f, 1.f, 1.f);
    }
  }
  if (tid == 0) {
    // a stage is free when its MMAs have completed and (dz ring) every epilogue thread has taken its dz values
    for (int s = 0; s < p.S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1 + ((MODE == 3 && p.Cz) ? kGroupThreadsPw : 0)); }
    for (int a = 0; a < 2; a++) {
      mbar_init(&a_full[a], 128); mbar_init(&a_empty[a], 1);
      mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], kGroupThreadsPw);
    }
    if (WG) mbar_init(wdone, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 1) tmem_alloc(tslot, ncols);
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm1); if (p.C2p || WG) tma_prefetch_desc(&tm2); if (MODE == 3 && p.Cz) tma_prefetch_desc(&tm3); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  const uint32_t t_hi = tbase + 2u * p.Np, t_lo = t_hi + p.Ks;                       // 2-D: the constant T operand
  const uint32_t x_width = 2u * (p.C1p + p.C2p);
  const uint32_t a_base = p.zlen ? tbase + 2u * p.Np : t_lo + p.Ks;
  const uint32_t a_width = p.zlen ? x_width + 2u * p.Ks : x_width;                    // 3-D: [X hi | lo ...][T hi | T lo] per buffer
  const uint32_t t_w = tbase + pw_tmem_wcol(p);                                        // WG: the weight-gradient accumulator

  const uint32_t xb1 = (uint32_t)p.C1p * 512, xb2 = (uint32_t)p.C2p * 512, ab = (uint32_t)p.Ks * p.Np * 4;
  // each CTA owns a contiguous run of tiles (sequential DRAM pages per channel row, same sample for A')
  const long t_first = (long)blockIdx.x * p.tiles_per_cta;
  const long t_end = t_first + p.tiles_per_cta < p.tiles ? t_first + p.tiles_per_cta : p.tiles;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const uint32_t bytes = xb1 + xb2 + ab + ((MODE == 3) ? (uint32_t)p.Cz * 512 : 0u) + (WG ? (uint32_t)p.Cxp * 512 : 0u);
      int it = 0;
      for (long tile = t_first; tile < t_end; tile++, it++) {
        const int s = it % p.S;
        const uint32_t ph = (uint32_t)(it / p.S) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full[s], bytes);
        uint8_t* st = smem + L.stages + (size_t)s * L.stage_bytes;
        const int b = (int)(tile / p.tiles_per_img);
        const int t_in_img = (int)(tile - (long)b * p.tiles_per_img);
        if (WG) {
          for (int j = 0; j < 4; j++) {
            tma_load_3d(st + (uint32_t)j * p.C1p * 256u, &tm1, &full[s], t_in_img * 128 + 32 * j, 0, b);
            tma_load_3d(st + L.xw + (uint32_t)j * p.NW * 128u, &tm2, &full[s], t_in_img * 128 + 32 * j, 0, b);
          }
        } else {
          tma_load_3d(st, &tm1, &full[s], t_in_img * 128, 0, b);
        }
        if (p.C2p) tma_load_3d(st + L.x2, &tm2, &full[s], t_in_img * 128, 0, b);
        if (MODE == 3 && p.Cz) tma_load_3d(st + L.dz, &tm3, &full[s], t_in_img * 128, 0, b);
        if (p.Ks) {
          // 2-D: the tile's R whole rows; 3-D: the R rows the tile touches, from the row of its first pixel on
          const size_t off = p.zlen ? ((size_t)b * p.RPI + (size_t)(t_in_img * 128) / p.zlen) * p.Qp * p.Np
                                    : (size_t)tile * p.R * p.Qp * p.Np;
          bulk_load(st + L.ah, p.ahi + off, ab, &full[s]);     // fp32 image; the converter warps split it into hi | lo
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs the loop with warp-uniform values (descriptors stay in uniform registers); one
    // elected lane issues the tcgen05 instructions.
    {
      const uint32_t idesc = idesc_tf32(128, p.Np, 0, 0);
      const uint32_t sbase = smem_u32(smem);
      const uint64_t d_w1h = smem_desc(sbase + L.w1h, 128, (p.C1p / 4) * 128, LAYOUT_NONE);
      const uint64_t d_w1l = smem_desc(sbase + L.w1l, 128, (p.C1p / 4) * 128, LAYOUT_NONE);
      const uint64_t d_w2h = smem_desc(sbase + L.w2h, 128, (p.C2p / 4) * 128, LAYOUT_NONE);
      const uint64_t d_w2l = smem_desc(sbase + L.w2l, 128, (p.C2p / 4) * 128, LAYOUT_NONE);
      const uint32_t lbo_a = (uint32_t)(p.Np / 8) * 128;
      int it = 0;
      for (long tile = t_first; tile < t_end; tile++, it++) {
        const int s = it % p.S;
        const uint32_t ph = (uint32_t)(it / p.S) & 1u;
        const int a = it & 1;
        const uint32_t aph = (uint32_t)(it >> 1) & 1u;
        const int xi = p.NA == 2 ? a : 0;                                  // A-operand buffer and its phase
        const uint32_t xph = p.NA == 2 ? aph : ((uint32_t)it & 1u);
        mbar_wait(&full[s], ph);         // A' rows landed (and X, consumed by the converter)
        mbar_wait(&a_full[xi], xph);     // converter filled TMEM A buffer xi
        mbar_wait(&acc_empty[a], aph ^ 1u);
        tc_fence_after();
        const uint32_t st = sbase + L.stages + (uint32_t)s * L.stage_bytes;
        const uint32_t d = tbase + (uint32_t)a * p.Np;
        const uint32_t xa = a_base + (uint32_t)xi * a_width;
        uint32_t acc = 0;
        if (elect_one()) {
          _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
            const uint32_t ac = pass == 1 ? xa + p.C1p : xa;
            const uint64_t dw = pass == 2 ? d_w1l : d_w1h;
            for (int k = 0; k < p.C1p / 8; k++) {
              mma_tf32_ts(d, ac + 8 * k, dw + (uint64_t)(k * 16), idesc, acc);
              acc = 1;
            }
          }
          if (p.C2p) {
            const uint32_t x2 = xa + 2 * p.C1p;
            _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
              const uint32_t ac = pass == 1 ? x2 + p.C2p : x2;
              const uint64_t dw = pass == 2 ? d_w2l : d_w2h;
              for (int k = 0; k < p.C2p / 8; k++) mma_tf32_ts(d, ac + 8 * k, dw + (uint64_t)(k * 16), idesc, 1);
            }
          }
          if (p.Ks) {
            // B operand A'[n = channel][k = (row, q)]: K-chunks outermost (LBO = Np/8 * 128), channel groups 128 B apart
            const uint64_t d_ah = smem_desc(st + L.ah, lbo_a, 128, LAYOUT_NONE);
            const uint64_t d_al = smem_desc(st + L.al, lbo_a, 128, LAYOUT_NONE);
            _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
              const uint32_t tcn = p.zlen ? (pass == 1 ? xa + x_width + p.Ks : xa + x_width) : (pass == 1 ? t_lo : t_hi);
              const uint64_t da = pass == 2 ? d_al : d_ah;
              for (int k = 0; k < p.Ks / 8; k++)
                mma_tf32_ts(d, tcn + 8 * k, da + (uint64_t)(k * (2 * lbo_a / 16)), idesc, 1);
            }
          }
        }
        if (elect_one()) {
          if (!WG) mma_commit(&empty[s]);
          mma_commit(&a_empty[xi]);
          mma_commit(&acc_full[a]);
        }
        __syncwarp();
        if (WG) {
          // dWp += [X1 hi ; X1 lo] x [XW hi ; XW lo ; ones]^T over the tile's 128 px (K), both operands K-major SW128 boxes in
          // the stage (the lo rows were written by the converter before it arrived on a_full); issued after the commits of
          // the dx accumulator so that its epilogue does not wait for them
          if (elect_one()) {
            const uint32_t idesc_w = idesc_tf32(p.MW, p.NW, 0, 0);
#pragma unroll 1
            for (int j = 0; j < 4; j++) {
              const uint64_t dg = smem_desc(st + (uint32_t)j * p.C1p * 256u, 16, 1024, LAYOUT_SW128);
              const uint64_t dxw = smem_desc(st + L.xw + (uint32_t)j * p.NW * 128u, 16, 1024, LAYOUT_SW128);
#pragma unroll
              for (int ks = 0; ks < 4; ks++)
                mma_tf32_ss(t_w, dg + (uint64_t)(ks * 2), dxw + (uint64_t)(ks * 2), idesc_w, (it > 0 || j > 0 || ks > 0) ? 1u : 0u);
            }
            mma_commit(&empty[s]);
          }
          __syncwarp();
        }
      }
      if (WG) {
        if (elect_one()) mma_commit(wdone);
        __syncwarp();
      }
    }
  } else if (warp < 6) {
    // ===================== converter: shared memory -> TMEM A operand (thread = pixel = TMEM lane) =====================
    const int quad = warp & 3;
    const int m = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    // constant T operand, once (2-D)
    for (int c0 = 0; c0 < (p.zlen ? 0 : p.Ks); c0 += 8) {
      float hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        hi[j] = __ldg(p.timg + (size_t)m * p.Ks + c0 + j);
        lo[j] = __ldg(p.timg + (size_t)128 * p.Ks + (size_t)m * p.Ks + c0 + j);
      }
      tmem_st8(t_hi + lane_base + c0, hi);
      tmem_st8(t_lo + lane_base + c0, lo);
    }
    int it = 0;
    for (long tile = t_first; tile < t_end; tile++, it++) {
      const int s = it % p.S;
      const uint32_t ph = (uint32_t)(it / p.S) & 1u;
      const int a = p.NA == 2 ? (it & 1) : 0;
      const uint32_t aph = p.NA == 2 ? ((uint32_t)(it >> 1) & 1u) : ((uint32_t)it & 1u);
      mbar_wait(&full[s], ph);
      if (p.Ks) {
        // A' rows arrive as ONE fp32 image (half the bytes k_inv_h writes and this kernel reads); split it in place into
        // the tf32 hi image and the lo image next to it, then make the generic-proxy writes visible to the MMAs
        // (explicit shared-space accesses: a generic pointer into the dynamic window compiles to LD.E / ST.E)
        const uint32_t ah = smem_u32(smem) + L.stages + (uint32_t)s * L.stage_bytes + L.ah;
        const uint32_t al = smem_u32(smem) + L.stages + (uint32_t)s * L.stage_bytes + L.al;
        for (int i = m * 4; i < p.Ks * p.Np; i += 512) {
          const float4 v = lds_v4(ah + (uint32_t)i * 4u);
          const float4 h = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
          sts_v4(ah + (uint32_t)i * 4u, h);
          sts_v4(al + (uint32_t)i * 4u, make_float4(tf32_rna(v.x - h.x), tf32_rna(v.y - h.y), tf32_rna(v.z - h.z), tf32_rna(v.w - h.w)));
        }
        fence_proxy_async();
      }
      mbar_wait(&a_empty[a], aph ^ 1u);
      tc_fence_after();
      const uint32_t sx = smem_u32(smem) + L.stages + (uint32_t)s * L.stage_bytes + (uint32_t)m * 4u;
      const uint32_t xa = a_base + (uint32_t)a * a_width + lane_base;
      if (WG) {
        // X1 from its SW128 box (pixel m: box m / 32, 16-byte chunk (m / 4) % 8 of row c swizzled by c % 8 -- a warp reads one
        // 128-byte row per channel); the lo values also go to the rows after the box, the weight-gradient A operand
        const uint32_t stg = smem_u32(smem) + L.stages + (uint32_t)s * L.stage_bytes;
        const uint32_t gb = stg + (uint32_t)(m >> 5) * (uint32_t)p.C1p * 256u + (uint32_t)(m & 3) * 4u;
        const uint32_t sw = (uint32_t)(m >> 2) & 7u;
        const bool lo_rows = p.npass == 3;
        for (int c0 = 0; c0 < p.C1p; c0 += 8) {
          float hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; j++) hi[j] = lds_f32(gb + (uint32_t)(c0 + j) * 128u + ((sw ^ (uint32_t)j) << 4));
#pragma unroll
          for (int j = 0; j < 8; j++) lo[j] = tf32_lo(hi[j]);
          tmem_st8(xa + c0, hi);
          tmem_st8(xa + p.C1p + c0, lo);
          if (lo_rows) {
#pragma unroll
            for (int j = 0; j < 8; j++) sts_f32(gb + (uint32_t)(p.C1p + c0 + j) * 128u + ((sw ^ (uint32_t)j) << 4), lo[j]);
          }
        }
        if (lo_rows) {
          // XW lo rows: elementwise copy of each box (same swizzle phase: Cxp is a multiple of 8 rows)
          const uint32_t per_box = (uint32_t)p.Cxp * 8u;   // float4 per box
          for (int j = 0; j < 4; j++) {
            const uint32_t xb = stg + L.xw + (uint32_t)j * (uint32_t)p.NW * 128u;
            for (uint32_t i = (uint32_t)m; i < per_box; i += 128u) {
              const float4 v = lds_v4(xb + i * 16u);
              sts_v4(xb + (uint32_t)p.Cxp * 128u + i * 16u, make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)));
            }
          }
        }
      } else {
        for (int c0 = 0; c0 < p.C1p; c0 += 8) {
          float hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; j++) hi[j] = lds_f32(sx + (uint32_t)(c0 + j) * 512u);
#pragma unroll
          for (int j = 0; j < 8; j++) lo[j] = tf32_lo(hi[j]);
          tmem_st8(xa + c0, hi);
          tmem_st8(xa + p.C1p + c0, lo);
        }
      }
      if (p.C2p) {
        const uint32_t sx2 = sx + L.x2;
        for (int c0 = 0; c0 < p.C2p; c0 += 8) {
          float hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; j++) hi[j] = lds_f32(sx2 + (uint32_t)(c0 + j) * 512u);
#pragma unroll
          for (int j = 0; j < 8; j++) lo[j] = tf32_lo(hi[j]);
          tmem_st8(xa + 2 * p.C1p + c0, hi);
          tmem_st8(xa + 2 * p.C1p + p.C2p + c0, lo);
        }
      }
      if (p.zlen) {
        // 3-D: T[m, (slot, q)] = table[q][z(m)] in the slot of pixel m's row, zero elsewhere
        const long tin = tile % p.tiles_per_img;
        const long pix = tin * 128 + m;
        const int r0 = (int)((tin * 128) / p.zlen);
        const int slot = (int)(pix / p.zlen) - r0, z = (int)(pix % p.zlen);
        const float* th = (const float*)(smem + L.tzh);
        const float* tl = (const float*)(smem + L.tzl);
        const uint32_t ta = xa + x_width;
        for (int c0 = 0; c0 < p.Ks; c0 += 8) {
          float hi[8], lo[8];
          const int sl = c0 / p.Qp, q0 = c0 - sl * p.Qp;      // Qp is a multiple of 8: a chunk never straddles slots
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const bool on = sl == slot;
            hi[j] = on ? th[(q0 + j) * p.zlen + z] : 0.f;
            lo[j] = on ? tl[(q0 + j) * p.zlen + z] : 0.f;
          }
          tmem_st8(ta + c0, hi);
          tmem_st8(ta + p.Ks + c0, lo);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      if (WG) fence_proxy_async();
      mbar_arrive(&a_full[a]);
    }
    if (WG) {
      // read-out of the weight gradient: accumulator row r = X1 hi row r (r < C1p) or lo row r - C1p; columns [0, Cxp) +
      // [Cxp, 2 Cxp) are the XW hi and lo products, column 2 Cxp the ones (db).  The hi rows write the CTA's partial in the
      // first gridDim.x slots, the lo rows theirs in the next gridDim.x; the reduction adds both in a fixed order.
      // (M = 64: row r lives in TMEM lane 32 (r / 16) + r % 16.)
      mbar_wait(wdone, 0);
      tc_fence_after();
      const int r = p.MW == 64 ? quad * 16 + (lane & 15) : m;
      const int half = r >= p.C1p ? 1 : 0, o = r - half * p.C1p;
      const bool own = (p.MW != 64 || lane < 16) && o < p.C1;
      const bool any = t_end > t_first;
      float* pout = p.wpart + ((size_t)half * gridDim.x + blockIdx.x) * ((size_t)p.C1 * p.Cx + p.C1);
      const uint32_t tw = t_w + lane_base;
      for (int c0 = 0; c0 < p.Cxp; c0 += 8) {
        float v[8], u[8];
        tmem_ld8(tw + (uint32_t)c0, v);
        tmem_ld8(tw + (uint32_t)(p.Cxp + c0), u);
        tmem_ld_wait();
        if (own) {
#pragma unroll
          for (int j = 0; j < 8; j++)
            if (c0 + j < p.Cx) pout[(size_t)o * p.Cx + c0 + j] = any ? v[j] + u[j] : 0.f;
        }
      }
      float v[8];
      tmem_ld8(tw + 2u * (uint32_t)p.Cxp, v);
      tmem_ld_wait();
      if (own) pout[(size_t)p.C1 * p.Cx + o] = any ? v[0] : 0.f;
    }
  } else {
    // ===================== epilogue: 8 warps per tile = 4 lane quadrants x 2 column parts, two groups =====================
    // sixteen warps = two groups of eight (4 lane quadrants x 2 column parts); group g owns the tiles with it % 2 == g, i.e. the
    // accumulator a = g: while one group is in its stores, the other reads its accumulator and computes (every SMSP holds two
    // warps of each group).  Round 1 had all sixteen warps on every tile, in the same phase at the same time.
    const int sub = (warp - 6) >> 2, grp = sub & 1;
    const int part = sub >> 1;
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int t = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t sbias = smem_u32(smem) + L.bias;
    // MODE 3: the saved pre-activations of the layer below arrive through the TMA ring (dz tile [Cz x 128 px] in the
    // stage, S tiles ahead of their use); with one pass per tile (Co <= 32) the thread takes its 8 values and releases the
    // stage right away, otherwise it reads them pass by pass and releases the stage at the end of the tile.  (Fetching
    // them with plain loads left only one tile of dz in flight per SM: 133 us, 3.0 TB/s.)
    const bool dz_ring = MODE == 3 && p.Cz > 0;
    const bool dz_single = p.Co <= kCW * kParts;
    int it = grp;
    for (long tile = t_first + grp; tile < t_end; tile += kGroups, it += kGroups) {
      const int a = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const int b = (int)(tile / p.tiles_per_img);
      const long px = (tile - (long)b * p.tiles_per_img) * 128 + t;
      const size_t base = (size_t)b * p.Co * p.P + px;
      const int s = it % p.S;
      const uint32_t sdz = smem_u32(smem) + L.stages + (uint32_t)s * L.stage_bytes + L.dz + (uint32_t)t * 4u;
      float dcur[kCW];
      if (dz_ring) {
        mbar_wait(&full[s], (uint32_t)(it / p.S) & 1u);
        if (dz_single) {
#pragma unroll
          for (int j = 0; j < kCW; j++) dcur[j] = (part * kCW + j < p.Cz) ? lds_f32(sdz + (uint32_t)(part * kCW + j) * 512u) : 0.f;
          mbar_arrive(&empty[s]);
        }
      }
      mbar_wait(&acc_full[a], aph);
      tc_fence_after();
      for (int c0 = part * kCW; c0 < p.Co; c0 += kCW * kParts) {
        float v[kCW];
        tmem_ld8(tbase + lane_base + (uint32_t)(a * p.Np + c0), v);
        if (MODE == 0) {
          float av[kCW], mv[kCW], dv[kCW], gzv[kCW], ghv[kCW];
#pragma unroll
          for (int j = 0; j < kCW; j++) {
            const bool ok = c0 + j < p.Co;
            const size_t idx = base + (size_t)(c0 + j) * p.P;
            const size_t inner = (size_t)(c0 + j) * p.P + px;
            av[j] = (p.add && ok) ? __ldg(p.add + idx) : 0.f;
            mv[j] = (p.mul && ok) ? __ldg(p.mul + (size_t)b * p.mul_bs + inner) : 1.f;
            dv[j] = (p.dz && ok) ? __ldg(p.dz + idx) : 0.f;
            gzv[j] = (p.gate_z && ok) ? __ldg(p.gate_z + (size_t)b * p.gate_bs + inner) : 1.f;
            ghv[j] = (p.gate_z && ok) ? __ldg(p.gate_h + idx) : 0.f;
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < kCW; j++) {
            if (c0 + j < p.Co) {
              const size_t idx = base + (size_t)(c0 + j) * p.P;
              const float z = v[j] + lds_f32(sbias + (uint32_t)(c0 + j) * 4u) + av[j];
              if (p.preact) p.preact[idx] = z;
              const float r = fmaf(1.0f - gzv[j], ghv[j], epi_value<0>(z, mv[j], dv[j], p.act, p.dact));
              p.y[idx] = r;
            }
          }
        } else {
          float dv[kCW];
          if (MODE == 3) {
            if (dz_ring && dz_single) {
#pragma unroll
              for (int j = 0; j < kCW; j++) dv[j] = dcur[j];
            } else if (dz_ring) {
#pragma unroll
              for (int j = 0; j < kCW; j++) dv[j] = (c0 + j < p.Cz) ? lds_f32(sdz + (uint32_t)(c0 + j) * 512u) : 0.f;
            } else {
#pragma unroll
              for (int j = 0; j < kCW; j++) dv[j] = (c0 + j < p.Co) ? __ldg(p.dz + base + (size_t)(c0 + j) * p.P) : 0.f;
            }
            // packed GELU' (two channels per FMA-pipe instruction)
#pragma unroll
            for (int j = 0; j < kCW; j += 2) {
              const float2 gg = b2no_gelu2_grad(make_float2(dv[j], dv[j + 1]));
              dv[j] = gg.x; dv[j + 1] = gg.y;
            }
          }
          float bv[kCW];
#pragma unroll
          for (int j = 0; j < kCW; j += 4) *reinterpret_cast<float4*>(bv + j) = lds_v4_ro(sbias + (uint32_t)(c0 + j) * 4u);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < kCW; j++) v[j] += bv[j];
          float* yp = p.y + base + (size_t)c0 * p.P;
          if (MODE == 2) {
            if (p.preact) {
              float* zp = p.preact + base + (size_t)c0 * p.P;
#pragma unroll
              for (int j = 0; j < kCW; j++)
                if (c0 + j < p.Co) zp[(size_t)j * p.P] = v[j];
            }
            // packed GELU (two channels per FMA-pipe instruction)
#pragma unroll
            for (int j = 0; j < kCW; j += 2) {
              const float2 gg = b2no_gelu2(make_float2(v[j], v[j + 1]));
              v[j] = gg.x; v[j + 1] = gg.y;
            }
          } else if (MODE == 3) {
#pragma unroll
            for (int j = 0; j < kCW; j++) v[j] *= dv[j];
          }
#pragma unroll
          for (int j = 0; j < kCW; j++)
            if (c0 + j < p.Co) yp[(size_t)j * p.P] = v[j];
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[a]);
      if (dz_ring && !dz_single) mbar_arrive(&empty[s]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tbase, ncols);
}

// A'[b][row][q/4][n/8][n%8][q%4] (one fp32 image) from the kept spectrum: the second-to-last inverse stage.
//   S[b,o,h,ky] = sum_kx M[kx][h] * spec[b][o][kx][ky];   q = 2 ky -> Re S, 2 ky + 1 -> Im S
// One block per (sample, group of HB rows): the sample's spectrum is staged in shared memory once.
constexpr int kInvHB = 32;
template <int KXM, bool PAIR>   // KXM: compile-time bound on the kept rows Kx (register array size); PAIR: two modes per thread
__global__ void __launch_bounds__(256)
k_inv_h(const float2* __restrict__ spec, const float2* __restrict__ M, float* __restrict__ ahi, float* __restrict__ alo,
        int Co, int Np, int Kx, int H, int Ky, int Qp, int layout, int n0) {
  extern __shared__ float2 s_spec[];  // [Co][Kx*Ky + 1] then the M rows of this block [Kx][kInvHB]
  const int b = blockIdx.y, h0 = blockIdx.x * kInvHB;
  const int kk = Kx * Ky, stride = kk + 1;
  float2* s_m = s_spec + (size_t)Co * stride;
  const float2* sp = spec + (size_t)b * Co * kk;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (layout == 0) {
    for (int o = warp; o < Co; o += 8)
      for (int r = lane; r < kk; r += 32) s_spec[o * stride + r] = __ldg(sp + (size_t)o * kk + r);
  } else if (layout == 2) {
    // 3-D: "sample" = (b, x); the x-stage output is [(b, channel, x)][K1][K2] -- the middle-dim inverse of the PINO layer
    const int b3 = b / n0, x = b - b3 * n0;
    for (int o = warp; o < Co; o += 8) {
      const float2* so = spec + (((size_t)b3 * Co + o) * n0 + x) * kk;
      for (int r = lane; r < kk; r += 32) s_spec[o * stride + r] = __ldg(so + r);
    }
  } else {
    // mode-major spectrum (mode, batch, channel): a mode's Co values of this sample are contiguous
    const size_t nb = gridDim.y;
    for (int idx = threadIdx.x; idx < Co * kk; idx += 256) {
      const int r = idx / Co, o = idx - r * Co;
      s_spec[o * stride + r] = __ldg(spec + ((size_t)r * nb + b) * Co + o);
    }
  }
  for (int i = threadIdx.x; i < Kx * kInvHB; i += 256) {
    const int kx = i / kInvHB, hl = i - kx * kInvHB;
    s_m[i] = (h0 + hl < H) ? __ldg(M + (size_t)kx * H + h0 + hl) : make_float2(0.f, 0.f);
  }
  __syncthreads();
  const int ng = Np >> 3, nq = Qp >> 2;
  const int rows = H - h0 < kInvHB ? H - h0 : kInvHB;
  // A thread owns one output slot; its Kx spectrum values do not depend on the row, so they are read once into registers and
  // every row then costs Kx x (one broadcast LDS.64 of M + packed FFMA2s):
  //   acc_a += Re M * v,  acc_b += Im M * v   ->   S = (acc_a.x - acc_b.y) + i (acc_a.y + acc_b.x)
  // PAIR: the slot is (kq, og, o8) = TWO modes ky = 2 kq, 2 kq + 1 of one channel, stored as one 16-byte word (half the
  // instructions per complex MAC; used when there are enough slots to keep all 256 threads busy, e.g. the RNO shape -- one
  // output per thread with scalar FMAs made this kernel issue-bound there: 60 us).
  if (PAIR) {
    const int per_row = nq * ng * 8;
    for (int e = threadIdx.x; e < per_row; e += 256) {
      const int o8 = e & 7;
      const int r = e >> 3;
      const int og = r % ng, kq = r / ng;
      const int ky0 = kq * 2, o = og * 8 + o8;
      const bool valid0 = o < Co && ky0 < Ky, valid1 = o < Co && ky0 + 1 < Ky;
      float2 v0[KXM], v1[KXM];
#pragma unroll
      for (int kx = 0; kx < KXM; kx++) {
        v0[kx] = (valid0 && kx < Kx) ? s_spec[o * stride + kx * Ky + ky0] : make_float2(0.f, 0.f);
        v1[kx] = (valid1 && kx < Kx) ? s_spec[o * stride + kx * Ky + ky0 + 1] : make_float2(0.f, 0.f);
      }
      const size_t off0 = ((size_t)b * H + h0) * Qp * Np + (size_t)kq * ng * 32 + og * 32 + o8 * 4;
      for (int hl = 0; hl < rows; hl++) {
        float2 a0 = make_float2(0.f, 0.f), b0 = a0, a1 = a0, b1 = a0;
#pragma unroll
        for (int kx = 0; kx < KXM; kx++) {
          if (kx < Kx) {
            const float2 m = s_m[kx * kInvHB + hl];
            const float2 mr = make_float2(m.x, m.x), mi = make_float2(m.y, m.y);
            a0 = __ffma2_rn(mr, v0[kx], a0);
            b0 = __ffma2_rn(mi, v0[kx], b0);
            a1 = __ffma2_rn(mr, v1[kx], a1);
            b1 = __ffma2_rn(mi, v1[kx], b1);
          }
        }
        const size_t off = off0 + (size_t)hl * Qp * Np;
        // fp32; k_pw_tc's converter warps make the hi / lo split
        *reinterpret_cast<float4*>(ahi + off) = make_float4(a0.x - b0.y, a0.y + b0.x, a1.x - b1.y, a1.y + b1.x);
      }
    }
  } else {
    const int per_row = nq * ng * 16;                    // (kq, og, o8, l0): one complex output each
    for (int e = threadIdx.x; e < per_row; e += 256) {
      const int l0 = e & 1, o8 = (e >> 1) & 7;
      const int r = e >> 4;
      const int og = r % ng, kq = r / ng;
      const int ky = kq * 2 + l0, o = og * 8 + o8;
      const bool valid = o < Co && ky < Ky;
      float2 v[KXM];
#pragma unroll
      for (int kx = 0; kx < KXM; kx++)
        v[kx] = (valid && kx < Kx) ? s_spec[o * stride + kx * Ky + ky] : make_float2(0.f, 0.f);
      const size_t off0 = ((size_t)b * H + h0) * Qp * Np + (size_t)kq * ng * 32 + og * 32 + o8 * 4 + l0 * 2;
      for (int hl = 0; hl < rows; hl++) {
        float2 a0 = make_float2(0.f, 0.f), b0 = a0;
#pragma unroll
        for (int kx = 0; kx < KXM; kx++) {
          if (kx < Kx) {
            const float2 m = s_m[kx * kInvHB + hl];
            a0 = __ffma2_rn(make_float2(m.x, m.x), v[kx], a0);
            b0 = __ffma2_rn(make_float2(m.y, m.y), v[kx], b0);
          }
        }
        const size_t off = off0 + (size_t)hl * Qp * Np;
        *reinterpret_cast<float2*>(ahi + off) = make_float2(a0.x - b0.y, a0.y + b0.x);
      }
    }
  }
}

int g_tc_state = -1;  // -1 unknown, 0 off, 1 on
long g_tc_launches = 0;
int g_tc_npass = 3;

}  // namespace

bool b2no_tc_available() {
  if (g_tc_state < 0) {
    int on = 1;
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
        major != 10)
      on = 0;
    if (on && !encode_fn()) on = 0;
    g_tc_state = on;
  }
  return g_tc_state == 1;
}

extern "C" int64_t b2no_tensor_core_launches(void) { return g_tc_launches; }
int b2no_tc_passes() { return g_tc_npass; }
// 0 = fp32-accurate (3xTF32, default), 1 = single-pass TF32.  Returns the mode now in force.
extern "C" int b2no_set_precision(int mode) {
  g_tc_npass = mode == 1 ? 1 : 3;
  return g_tc_npass == 1 ? 1 : 0;
}
void b2no_tc_count_launch() { g_tc_launches++; }

extern "C" int b2no_set_tensor_core_mode(int on) {
  g_tc_state = -1;
  if (!on) { g_tc_state = 0; return 0; }
  return b2no_tc_available() ? 1 : 0;
}

// Returns 0 when the tile kernel ran, 1 when the shape is not eligible (caller falls back to the CUDA-core
// kernel), otherwise an error code.  With `wg` only the weight-gradient variant is eligible, and nothing is launched when it
// is not.
int b2no_tc_pointwise(const b2no_plan* plan, int which, const float* spec, float* y, float* work, int batch, int channels,
                      long pixels, const b2no_epilogue* e, cudaStream_t st, const b2no_tc_wg* wg) {
  if (!b2no_tc_available()) return 1;
  if (!e || !e->pw_w || !e->pw_x || e->pw_ci < 1) return 1;          // needs at least one 1x1 operand (the TMA-fed A tile)
  if (pixels % 128 != 0 || channels > 256 || e->pw_ci > 128 || e->pw2_ci > 128) return 1;
  if (((uintptr_t)e->pw_x | (uintptr_t)y) & 15) return 1;
  const bool has2 = e->pw2_w && e->pw2_x && e->pw2_ci > 0;
  if (has2 && ((uintptr_t)e->pw2_x & 15)) return 1;
  PwTc p;
  memset(&p, 0, sizeof(p));
  p.B = batch; p.Co = channels; p.Np = b2no_round_up(channels, 16); p.P = pixels;
  p.C1 = e->pw_ci; p.C1p = b2no_round_up(e->pw_ci, 8);
  p.C2 = has2 ? e->pw2_ci : 0; p.C2p = has2 ? b2no_round_up(e->pw2_ci, 8) : 0;
  p.tiles_per_img = (int)(pixels / 128);
  p.tiles = (long)batch * p.tiles_per_img;
  p.w1 = e->pw_w; p.w1_t = e->pw_transposed; p.w2 = has2 ? e->pw2_w : nullptr; p.w2_t = e->pw2_transposed;
  p.bias = e->bias; p.add = e->add; p.mul = e->mul; p.dz = e->dact_z; p.preact = e->preact; p.y = y;
  p.act = e->act; p.dact = e->dact_z ? e->dact : 0;
  p.gate_z = (e->gate_z && e->gate_h) ? e->gate_z : nullptr; p.gate_h = p.gate_z ? e->gate_h : nullptr;
  p.mul_bs = e->mul_bstride ? (long)e->mul_bstride : (long)channels * pixels;
  p.gate_bs = e->gate_bstride ? (long)e->gate_bstride : (long)channels * pixels;
  const bool three_d = spec && plan && plan->g.ndim == 3;
  if (spec && !three_d) {
    if (!plan || plan->g.ndim != 2 || !work) return 1;
    const b2no_tc_tables& tt = plan->tc[which];
    if (!tt.timg) return 1;
    p.Ks = tt.Ks; p.Qp = tt.Qp; p.R = tt.R; p.timg = tt.timg;
    const int32_t* n = which == 0 ? plan->g.nout : plan->g.nin;
    if ((long)n[0] * n[1] != pixels) return B2NO_E_ARG;
    const size_t afl = (size_t)batch * n[0] * p.Qp * p.Np;
    p.ahi = work;
    p.alo = work + afl;
  }
  if (three_d) {
    // 3-D: `spec` is the x-stage output [(b, channel, x)][K1][K2]; k_inv_h does the middle-dim stage into the row image,
    // the tile kernel the last dim with a per-tile T operand (rows of n2 points do not align with 128-pixel tiles)
    if (!work) return 1;
    const int32_t* n = which == 0 ? plan->g.nout : plan->g.nin;
    if ((long)n[0] * n[1] * n[2] != pixels) return B2NO_E_ARG;
    p.zlen = n[2]; p.q2 = 2 * plan->K[2]; p.Qp = b2no_round_up(p.q2, 8);
    p.R = 127 / p.zlen + 2; p.Ks = p.R * p.Qp;
    p.RPI = (long)n[0] * n[1];
    p.tz = which == 0 ? plan->t_out : plan->t_in;
    p.tz_npad = which == 0 ? plan->npad_out : plan->npad_in;
    if (p.zlen < 8 || p.Ks > 192 || plan->K[1] > 32 || p.Qp > 64) return 1;
    p.ahi = work;
    p.alo = work;
  }
  if (wg) {
    // 2-D plans, one 1x1 operand of <= 64 channels ([hi ; lo] rows fill at most M = 128), XW of <= 112 channels (N <= 256)
    if (!spec || three_d || has2 || p.C1p > 64 || wg->ci < 1 || wg->ci > 112 || ((uintptr_t)wg->x & 15)) return 1;
    p.Cx = wg->ci; p.Cxp = b2no_round_up(wg->ci, 8);
    p.MW = 2 * p.C1p <= 64 ? 64 : 128;
    p.NW = b2no_round_up(2 * p.Cxp + 1, p.MW == 64 ? 8 : 16);   // the ones block: 8 or 16 rows
    p.wpart = wg->partial;
  }
  p.NA = 2;
  auto tmem_cols = [&]() { return wg ? pw_tmem_cols<true>(p) : pw_tmem_cols<false>(p); };
  auto layout = [&]() { return wg ? pw_layout<true>(p) : pw_layout<false>(p); };
  if (tmem_cols() > 512) p.NA = 1;              // wide operands: one A buffer (the converter then waits for the tile's MMAs)
  if (tmem_cols() > 512) return 1;
  const bool extras = p.add || p.mul || p.gate_z;
  int mode = 0;
  if (!extras && !p.dact && p.act == B2NO_ACT_NONE && !p.preact) mode = 1;
  else if (!extras && !p.dact && p.act == B2NO_ACT_GELU) mode = 2;
  else if (!extras && p.dact == B2NO_ACT_GELU && p.act == B2NO_ACT_NONE && !p.preact) mode = 3;
  // The dx pass without activation only.  Measured on a B200 (1000 W) at the cfg2 layer shape (B 64, 32 ch, 128^2, modes 12,
  // inputs larger than L2, scripts/fused_wgrad_timing.py): this variant 172 us against 179 us for k_pw_tc<1> + k_wgrad_tc +
  // reduce; with GELU'(dz) (MODE 3) 203 us against 193 us -- the dz tile makes a stage 90 KB, two fit next to the weights
  // (102 KB of payload in flight against six stages of k_pw_tc<3> alone), so MODE 3 keeps the two launches.
  if (wg && mode != 1) return 1;
  // dz through the TMA ring: enabled for the single-pass case (Co <= 32: every epilogue thread takes its 8 values and
  // releases the stage at once), which is what the parity tests and the bench exercise; wider layers keep the per-thread
  // loads until the multi-pass variant of the ring has its own GPU test
  if (mode == 3 && (((uintptr_t)p.dz & 15) == 0) && channels <= kCW * kParts * kGroups) p.Cz = b2no_round_up(channels, 8);
  // shared-memory budget -> number of stages
  int dev = 0, max_smem = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  B2NO_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  PwLayout L;
  for (p.S = 6; p.S >= 2; p.S--) {
    L = layout();
    if ((int)L.total <= max_smem) break;
  }
  if (p.S < 3 && p.Cz) {          // not enough room for a useful ring with the dz tile: plain loads instead
    p.Cz = 0;
    for (p.S = 6; p.S >= 2; p.S--) {
      L = layout();
      if ((int)L.total <= max_smem) break;
    }
  }
  if (p.S < 2) return 1;

  CUtensorMap tm1, tm2, tm3;
  {
    uint64_t dims[3] = {(uint64_t)pixels, (uint64_t)p.C1, (uint64_t)batch};
    uint64_t str[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * p.C1};
    uint32_t box[3] = {128, (uint32_t)p.C1p, 1};
    if (wg) box[0] = 32;                         // [32 px x C1p] boxes with the 128-byte swizzle: K-major operands
    if (make_tmap_f32(&tm1, e->pw_x, 3, dims, str, box, wg ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE)) return 1;
    tm2 = tm1;
    if (wg) {
      uint64_t dimsw[3] = {(uint64_t)pixels, (uint64_t)p.Cx, (uint64_t)batch};
      uint64_t strw[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * p.Cx};
      uint32_t boxw[3] = {32, (uint32_t)p.Cxp, 1};
      if (make_tmap_f32(&tm2, wg->x, 3, dimsw, strw, boxw, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    }
    if (has2) {
      uint64_t dims2[3] = {(uint64_t)pixels, (uint64_t)p.C2, (uint64_t)batch};
      uint64_t str2[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * p.C2};
      uint32_t box2[3] = {128, (uint32_t)p.C2p, 1};
      if (make_tmap_f32(&tm2, e->pw2_x, 3, dims2, str2, box2, CU_TENSOR_MAP_SWIZZLE_NONE)) return 1;
    }
    tm3 = tm1;
    if (p.Cz) {
      uint64_t dims3[3] = {(uint64_t)pixels, (uint64_t)channels, (uint64_t)batch};
      uint64_t str3[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * channels};
      uint32_t box3[3] = {128, (uint32_t)p.Cz, 1};
      if (make_tmap_f32(&tm3, p.dz, 3, dims3, str3, box3, CU_TENSOR_MAP_SWIZZLE_NONE)) return 1;
    }
  }
  if (spec) {
    const int32_t* n = which == 0 ? plan->g.nout : plan->g.nin;
    // the stage k_inv_h contracts: dim 0 of a 2-D plan, dim 1 of a 3-D one (its "samples" are then the (b, x) pairs)
    const int jd = three_d ? 1 : 0;
    const float2* M = which == 0 ? plan->m_inv[jd] : plan->m_adjfwd[jd];
    const int ikx = plan->K[jd], iky = plan->K[jd + 1], ih = n[jd];
    const int ilayout = three_d ? 2 : plan->g.spec_layout, in0 = three_d ? n[0] : 1;
    const size_t smem = ((size_t)channels * (ikx * iky + 1) + (size_t)ikx * kInvHB) * sizeof(float2);
    if (smem > 200 * 1024) return 1;
    if ((long)batch * in0 > 65535) return 1;
    dim3 grid((unsigned)((ih + kInvHB - 1) / kInvHB), (unsigned)(batch * in0));
    if (three_d) {
      // the tiles at the end of the image read up to R rows past it: keep those finite (they meet zero T entries)
      B2NO_CHECK_CUDA(cudaMemsetAsync(work + (size_t)batch * p.RPI * p.Qp * p.Np, 0, (size_t)(p.R + 1) * p.Qp * p.Np * sizeof(float), st));
    }
    const bool pair = (p.Qp / 4) * (p.Np / 8) * 8 >= 256;      // enough two-mode slots for every thread of the block
#define INVH_LAUNCH1(KXM, PAIR)                                                                                         \
  do {                                                                                                                  \
    if (smem > 48 * 1024) B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_inv_h<KXM, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_inv_h<KXM, PAIR><<<grid, 256, smem, st>>>((const float2*)spec, M, (float*)p.ahi, (float*)p.alo, channels, p.Np, ikx, ih, \
                                                iky, p.Qp, ilayout, in0);                                               \
  } while (0)
#define INVH_LAUNCH(KXM)                                                                                                \
  do {                                                                                                                  \
    if (pair) INVH_LAUNCH1(KXM, true); else INVH_LAUNCH1(KXM, false);                                                   \
  } while (0)
    const int kx = ikx;
    if (kx <= 8) INVH_LAUNCH(8);
    else if (kx <= 12) INVH_LAUNCH(12);
    else if (kx <= 16) INVH_LAUNCH(16);
    else if (kx <= 24) INVH_LAUNCH(24);
    else if (kx <= 32) INVH_LAUNCH(32);
    else return 1;
#undef INVH_LAUNCH1
#undef INVH_LAUNCH
    B2NO_LAUNCH_CHECK();
  }
  long grid = p.tiles < b2no_sm_count() ? p.tiles : b2no_sm_count();
  p.tiles_per_cta = (p.tiles + grid - 1) / grid;
  grid = (p.tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  p.npass = b2no_tc_passes();
#define LAUNCH(M, W)                                                                                                  \
  do {                                                                                                                \
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_pw_tc<M, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));  \
    k_pw_tc<M, W><<<(unsigned)grid, kThreads, L.total, st>>>(tm1, tm2, tm3, p);                                           \
  } while (0)
  if (wg) {
    LAUNCH(1, true);
    *wg->nblk = 2 * (int)grid;                    // the hi-row and lo-row partials of every CTA
  } else {
    switch (mode) {
      case 1: LAUNCH(1, false); break;
      case 2: LAUNCH(2, false); break;
      case 3: LAUNCH(3, false); break;
      default: LAUNCH(0, false); break;
    }
  }
#undef LAUNCH
  B2NO_LAUNCH_CHECK();
  g_tc_launches++;
  return 0;
}
