// Fused two-layer pointwise MLP on tcgen05: the projection head of the FNO (tfno.py:34-38: Conv(C->H) -> GELU ->
// Conv(H->1)), the PINO tail (pinobserver.py:230-232) and the RNO regressor (rno.py:170-174), forward AND the
// input-gradient half of the backward, without ever writing the H-channel hidden tensor for the forward
// (64 x 256 x 128^2 fp32 = 1.07 GB at BASELINE config 2).
//
//   forward :  out[b,n,p] = b2[n] + sum_j W2[n,j] act(z1[j]),     z1[j] = b1[j] + sum_i W1[j,i] x[b,i,p]
//   backward:  f[j] = g[b,p] w2[j] act'(z1[j])  (z1 recomputed),   gx[b,i,p] = sum_j W1[j,i] f[j]
//              optional: gz[b,j,p] = f[j] written once for the weight-gradient kernel (tc_wgrad.cu),
//              dw2[j] = sum_{b,p} g act(z1[j])  (warp butterfly + shared-memory atomics, per-CTA partials)
//
// Structure per 128-pixel tile (TMEM lane = pixel), hidden dimension processed in chunks of 64:
//   MMA1 (TS):  acc1[128 x 64]  = X[128 x C] (TMEM, hi/lo)  *  W1 chunk[64 x C]^T (smem)         3xTF32
//   epilogue-f: tcgen05.ld acc1 -> f -> tcgen05.st F[128 x 64] hi/lo (the A operand of MMA2 never leaves the SM)
//   MMA2 (TS):  acc2[128 x N2] += F[128 x 64] * W2' chunk[N2 x 64]^T (smem)                        3xTF32
//   epilogue-2: tcgen05.ld acc2 -> bias / dact -> coalesced stores
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 X converter (smem -> TMEM), warps 6-13 epilogue
// (4 lane quadrants x 2 column halves).  acc1, F and acc2 are double buffered in TMEM.
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

constexpr int kEW = 16;                        // hidden columns per epilogue thread per 64-column chunk
constexpr int kNP = 64 / kEW;                  // column parts -> kNP x 4 epilogue warps (latency hiding for the GELU math)
constexpr int kEpiThreads = 128 * kNP;
constexpr int kThreadsMlp = 192 + kEpiThreads;

// generic activation out of line (the switch would otherwise be unrolled 32 times in the two-group forward)
__device__ __noinline__ float mlp_act_ool(float z, int act) { return b2no_act(z, act); }

struct MlpTc {
  int B, Ci, Cip, H, Hp, NC, N2, Co2, S, fbufs, mode, act, b1_per_sample, dact, direct;
  int npass;   // 3: 3xTF32, 1: single-pass TF32
  int tiles_per_img;
  long tiles, tiles_per_cta, P;
  const float* w1; const float* b1; const float* w2; const float* b2; const float* g; const float* dz;
  float* out; float* gz; float* dw2_partial;
};

struct MlpLayout { uint32_t w1h, w1l, w2h, w2l, b1, w2v, dw2, part, stages, stage_bytes, bars, total; };

// no: output channels of a backward launch (the w2 rows and dw2 accumulators kept in shared memory); 1 otherwise
__host__ __device__ inline MlpLayout mlp_layout(const MlpTc& p, int no = 1) {
  MlpLayout L;
  uint32_t o = 0;
  const uint32_t wb1 = (uint32_t)p.Hp * p.Cip * 4, wb2 = (uint32_t)p.N2 * p.Hp * 4;
  L.w1h = o; o += wb1; L.w1l = o; o += wb1;
  L.w2h = o; o += wb2; L.w2l = o; o += wb2;
  L.b1 = o; o += (uint32_t)p.Hp * 4;
  L.w2v = o; o += (uint32_t)no * p.Hp * 4;
  L.dw2 = o; o += (uint32_t)no * p.Hp * 4;
  L.part = o; o += 2 * 4 * 128 * 4;
  o = (o + 1023u) & ~1023u;
  L.stages = o;
  L.stage_bytes = (uint32_t)p.Cip * 512;
  o += L.stage_bytes * p.S;
  L.bars = o;
  o += 8 * (2 * p.S + 20) + 16;
  L.total = o + 1024;
  return L;
}

__host__ __device__ inline uint32_t mlp_tmem_cols(const MlpTc& p) {
  if (p.direct) return 2u * p.Cip + 256u;
  return 2u * p.Cip + 128u + 128u * p.fbufs + 2u * p.N2;
}

// dw2[col] += sum over the warp's 32 pixels of ga[col] (kEW columns per lane): transposing butterfly; while a lane still
// holds more than one column the halves are exchanged, afterwards plain xor-sums.  Returns the sum of column
// lane >> (5 - log2 kEW), identical in the 32 / kEW lanes of each group.
__device__ __forceinline__ float warp_column_sum(float (&ga)[kEW], int lane) {
  int cnt = kEW;
#pragma unroll
  for (int s = 0; s < 5; s++) {
    const int off = 16 >> s;
    if (cnt > 1) {
      const int hw = cnt >> 1;
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < kEW / 2; i++) {
        if (i < hw) {
          const float a0 = ga[i], a1 = ga[i + hw];
          const float send = upper ? a0 : a1;
          const float keep = upper ? a1 : a0;
          ga[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      cnt = hw;
    } else {
      ga[0] += __shfl_xor_sync(0xffffffffu, ga[0], off);
    }
  }
  return ga[0];
}

// NO: output channels of the head (backward only; the forward takes p.Co2 at run time).  With NO > 1 the backward reads NO
// upstream gradients per pixel, forms f[j] = act'(z1[j]) sum_o g[o] w2[o,j] and keeps NO dw2 rows.
template <bool GELU, bool BWD, bool DIRECT, int NO = 1>
__global__ void __launch_bounds__(kThreadsMlp, 1)
k_mlp_tc(const __grid_constant__ CUtensorMap tmx, const MlpTc p) {
  static_assert(NO >= 1 && (NO == 1 || (BWD && !DIRECT)), "several outputs: backward kernel only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const MlpLayout L = mlp_layout(p, NO);
  uint64_t* full = (uint64_t*)(smem + L.bars);
  uint64_t* empty = full + p.S;
  uint64_t* x_full = empty + p.S;
  uint64_t* x_empty = x_full + 1;
  uint64_t* acc1_full = x_empty + 1;
  uint64_t* acc1_empty = acc1_full + 4;
  uint64_t* f_full = acc1_empty + 4;
  uint64_t* f_empty = f_full + 2;
  uint64_t* acc2_full = f_empty + 2;
  uint64_t* acc2_empty = acc2_full + 2;
  uint32_t* tslot = (uint32_t*)(acc2_empty + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t ncols = 32;
  while (ncols < mlp_tmem_cols(p)) ncols <<= 1;
  constexpr bool bwd = BWD;
  // DIRECT (forward, one output channel): out = b2 + sum_j w2[j] act(z1[j]) is accumulated by the epilogue threads in fp32
  // registers (FFMA2) -- no F operand, no second MMA; exact fp32 accumulation for the cancelling sum over the hidden units
  constexpr bool direct = DIRECT;

  // ---- setup: W1 (B operand of MMA1, [Hp x Cip]) and W2' (B operand of MMA2, [N2 x Hp]), hi/lo, K-major core layout ----
  for (int i = tid; i < p.Hp * p.Cip; i += kThreadsMlp) {
    const int n = i / p.Cip, k = i - n * p.Cip;
    const float w = (n < p.H && k < p.Ci) ? p.w1[(size_t)n * p.Ci + k] : 0.f;
    const float hi = tf32_rna(w);
    *(float*)(smem + L.w1h + kmajor_off(n, k, p.Cip)) = hi;
    *(float*)(smem + L.w1l + kmajor_off(n, k, p.Cip)) = tf32_rna(w - hi);
  }
  for (int i = tid; i < p.N2 * p.Hp; i += kThreadsMlp) {
    const int n = i / p.Hp, k = i - n * p.Hp;
    float w = 0.f;
    if (k < p.H) {
      if (bwd) { if (n < p.Ci) w = p.w1[(size_t)k * p.Ci + n]; }       // W1^T : gx[i] = sum_j W1[j,i] f[j]
      else if (n < p.Co2) w = p.w2[(size_t)n * p.H + k];
    }
    const float hi = tf32_rna(w);
    *(float*)(smem + L.w2h + kmajor_off(n, k, p.Hp)) = hi;
    *(float*)(smem + L.w2l + kmajor_off(n, k, p.Hp)) = tf32_rna(w - hi);
  }
  for (int i = tid; i < p.Hp; i += kThreadsMlp) {
    ((float*)(smem + L.b1))[i] = (!p.b1_per_sample && p.b1 && i < p.H) ? p.b1[i] : 0.f;
#pragma unroll
    for (int o = 0; o < NO; o++) {
      ((float*)(smem + L.w2v))[o * p.Hp + i] = ((bwd || direct) && i < p.H) ? p.w2[(size_t)o * p.H + i] : 0.f;
      ((float*)(smem + L.dw2))[o * p.Hp + i] = 0.f;
    }
  }
  if (tid == 0) {
    for (int s = 0; s < p.S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 128); }
    mbar_init(x_full, 128); mbar_init(x_empty, 1);
    // two-group DIRECT forward: a 64-column chunk belongs to one group of 8 epilogue warps (one arrival per warp); the
    // f_full / f_empty slots serve as "partials of tile parity a written" (16 warps) / "... consumed" (4 converter warps)
    const bool two_groups = DIRECT && (p.NC & 1) == 0;
    for (int a = 0; a < 4; a++) { mbar_init(&acc1_full[a], 1); mbar_init(&acc1_empty[a], two_groups ? 8 : kEpiThreads); }
    for (int a = 0; a < 2; a++) {
      mbar_init(&f_full[a], two_groups ? 16 : kEpiThreads); mbar_init(&f_empty[a], two_groups ? 4 : 1);
      mbar_init(&acc2_full[a], 1); mbar_init(&acc2_empty[a], kEpiThreads);
    }
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 1) tmem_alloc(tslot, ncols);
  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmx);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  // TMEM map: [X hi | X lo] [acc1 x2] [F (hi 64 | lo 64) x fbufs] [acc2 x2]
  constexpr int NA = DIRECT ? 4 : 2;   // acc1 ring depth (DIRECT has no F / acc2, so the TMEM goes to a deeper ring)
  const uint32_t t_x = tbase, t_acc1 = t_x + 2u * p.Cip, t_f = t_acc1 + 64u * NA, t_acc2 = t_f + 128u * p.fbufs;
  const long t_first = (long)blockIdx.x * p.tiles_per_cta;
  const long t_end = t_first + p.tiles_per_cta < p.tiles ? t_first + p.tiles_per_cta : p.tiles;
  const int NC = p.NC;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int it = 0;
      for (long tile = t_first; tile < t_end; tile++, it++) {
        const int s = it % p.S;
        const uint32_t ph = (uint32_t)(it / p.S) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full[s], L.stage_bytes);
        const int b = (int)(tile / p.tiles_per_img);
        tma_load_3d(smem + L.stages + (size_t)s * L.stage_bytes, &tmx, &full[s], (int)(tile - (long)b * p.tiles_per_img) * 128, 0, b);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-uniform loop, one elected lane issues) =====================
    const uint32_t id1 = idesc_tf32(128, 64, 0, 0), id2 = idesc_tf32(128, p.N2, 0, 0);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t sbo1 = (uint32_t)(p.Cip / 4) * 128, sbo2 = (uint32_t)(p.Hp / 4) * 128;
    const uint64_t d_w1h = smem_desc(sbase + L.w1h, 128, sbo1, LAYOUT_NONE), d_w1l = smem_desc(sbase + L.w1l, 128, sbo1, LAYOUT_NONE);
    const uint64_t d_w2h = smem_desc(sbase + L.w2h, 128, sbo2, LAYOUT_NONE), d_w2l = smem_desc(sbase + L.w2l, 128, sbo2, LAYOUT_NONE);
    const int k1 = p.Cip / 8;
    int it = 0;
    long n1 = 0;  // chunk counter of this CTA (acc1 / F ring position)
    auto mma1 = [&](long n, int c) {
      const int ab = (int)(n % NA);
      mbar_wait(&acc1_empty[ab], ((uint32_t)(n / NA) & 1u) ^ 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d = t_acc1 + 64u * ab;
        const uint64_t woff = (uint64_t)((uint32_t)c * 8u * sbo1 / 16u);   // 64 rows = 8 row groups
        uint32_t acc = 0;
        _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
          const uint32_t ac = pass == 1 ? t_x + p.Cip : t_x;
          const uint64_t dw = (pass == 2 ? d_w1l : d_w1h) + woff;
          for (int k = 0; k < k1; k++) { mma_tf32_ts(d, ac + 8 * k, dw + (uint64_t)(k * 16), id1, acc); acc = 1; }
        }
        mma_commit(&acc1_full[ab]);
      }
      __syncwarp();
    };
    for (long tile = t_first; tile < t_end; tile++, it++) {
      mbar_wait(x_full, (uint32_t)it & 1u);
      tc_fence_after();
      if (direct) {
        for (int c = 0; c < NC; c++) mma1(n1 + c, c);
        if (elect_one()) mma_commit(x_empty);
        __syncwarp();
        n1 += NC;
        continue;
      }
      mma1(n1, 0);
      if (NC > 1) mma1(n1 + 1, 1);
      if (NC <= 2) { if (elect_one()) mma_commit(x_empty); __syncwarp(); }
      for (int c = 0; c < NC; c++) {
        const long nf = n1 + c;
        const int fb = (int)(nf % p.fbufs);
        mbar_wait(&f_full[fb], (uint32_t)(nf / p.fbufs) & 1u);
        if (c == 0) mbar_wait(&acc2_empty[it & 1], ((uint32_t)(it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d = t_acc2 + (uint32_t)(it & 1) * p.N2;
          const uint32_t fa = t_f + 128u * fb;
          const uint64_t koff = (uint64_t)(c * 16 * 8);   // 64 k = 16 chunks of 4, 128 B each -> /16
          _Pragma("unroll") for (int pass = 0; pass < 3; pass++) {
            if (pass >= p.npass) break;   // compile-time trip count (descriptors stay folded); 1-pass mode leaves early
            const uint32_t ac = pass == 1 ? fa + 64 : fa;
            const uint64_t dw = (pass == 2 ? d_w2l : d_w2h) + koff;
            for (int k = 0; k < 8; k++) mma_tf32_ts(d, ac + 8 * k, dw + (uint64_t)(k * 16), id2, (c > 0 || pass > 0 || k > 0) ? 1u : 0u);
          }
          mma_commit(&f_empty[fb]);
        }
        __syncwarp();
        if (c + 2 < NC) {
          mma1(n1 + c + 2, c + 2);
          if (c + 2 == NC - 1) { if (elect_one()) mma_commit(x_empty); __syncwarp(); }
        }
      }
      if (elect_one()) mma_commit(&acc2_full[it & 1]);
      __syncwarp();
      n1 += NC;
    }
  } else if (warp < 6) {
    // ===================== converter: X tile -> TMEM A operand (single buffer per tile) =====================
    const int quad = warp & 3;
    const int m = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    // two-group DIRECT forward: out[pixel m] of a finished tile = b2 + the four partial sums (2 groups x 2 column halves) the
    // epilogue warps left in shared memory, added in a fixed order; the store and the wait stay off the epilogue's chain
    auto direct_combine = [&](int jt, long jtile) {
      const int a = jt & 1;
      mbar_wait(&f_full[a], (uint32_t)(jt >> 1) & 1u);
      const uint32_t pp = smem_u32(smem) + L.part + (uint32_t)(a * 4 * 128 + m) * 4u;
      float o = p.b2 ? __ldg(p.b2) : 0.f;
#pragma unroll
      for (int q = 0; q < 4; q++) o += lds_f32(pp + (uint32_t)q * 512u);
      __syncwarp();
      if (lane == 0) mbar_arrive(&f_empty[a]);
      const int b = (int)(jtile / p.tiles_per_img);
      p.out[(size_t)b * p.P + (jtile - (long)b * p.tiles_per_img) * 128 + m] = o;
    };
    int it = 0;
    for (long tile = t_first; tile < t_end; tile++, it++) {
      const int s = it % p.S;
      const uint32_t ph = (uint32_t)(it / p.S) & 1u;
      mbar_wait(&full[s], ph);
      mbar_wait(x_empty, ((uint32_t)it & 1u) ^ 1u);
      tc_fence_after();
      const float* sx = (const float*)(smem + L.stages + (size_t)s * L.stage_bytes);
      for (int c0 = 0; c0 < p.Cip; c0 += 8) {
        float hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
          hi[j] = sx[(c0 + j) * 128 + m];
          lo[j] = tf32_lo(hi[j]);
        }
        tmem_st8(t_x + lane_base + c0, hi);
        tmem_st8(t_x + lane_base + p.Cip + c0, lo);
      }
      mbar_arrive(&empty[s]);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(x_full);
      if (DIRECT && (NC & 1) == 0 && it > 0) direct_combine(it - 1, tile - 1);
    }
    if (DIRECT && (NC & 1) == 0 && it > 0) direct_combine(it - 1, t_end - 1);
  } else {
    // ===================== epilogue: 4 lane quadrants x kNP column parts =====================
    const int part_id = (warp - 6) >> 2;
    const int quad = warp & 3;
    const int t = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const float* sb1 = (const float*)(smem + L.b1);
    const float* sw2 = (const float*)(smem + L.w2v);
    float* sdw2 = (float*)(smem + L.dw2);
    if (DIRECT && (NC & 1) == 0) {
      // ---- forward, one output channel, two groups of 8 warps on alternating 64-column chunks: while one group waits for
      // its accumulator and reads it, the other one keeps the FMA pipe busy with the GELU math (every SMSP holds two warps of
      // each group).  Each thread owns 32 columns of its group's chunks and sums w2[j] gelu(z1[j]) in fp32 registers.
      const int sub = (warp - 6) >> 2, grp = sub & 1, half = sub >> 1;
      const uint32_t s_b1 = smem_u32(smem) + L.b1, s_w2 = smem_u32(smem) + L.w2v;
      const uint32_t s_part = smem_u32(smem) + L.part + (uint32_t)(sub * 128 + t) * 4u;
      const long ntot = (t_end - t_first) * (long)NC;
      int it = 0, c = grp;
      long tile = t_first;
      float2 oacc = make_float2(0.f, 0.f);
      for (long n = grp; n < ntot; n += 2) {
        const int ab = (int)(n % NA);
        const int col0 = c * 64 + half * 32;
        mbar_wait(&acc1_full[ab], (uint32_t)(n / NA) & 1u);
        tc_fence_after();
        float v[32];
        tmem_ld32(t_acc1 + lane_base + 64u * ab + half * 32, v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc1_empty[ab]);
        if (GELU && !p.b1_per_sample) {
          const float2* v2 = reinterpret_cast<const float2*>(v);
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const float4 bq = lds_v4_ro(s_b1 + (uint32_t)(col0 + 4 * j) * 4u), wq = lds_v4_ro(s_w2 + (uint32_t)(col0 + 4 * j) * 4u);
            oacc = __ffma2_rn(b2no_gelu2(__fadd2_rn(v2[2 * j], make_float2(bq.x, bq.y))), make_float2(wq.x, wq.y), oacc);
            oacc = __ffma2_rn(b2no_gelu2(__fadd2_rn(v2[2 * j + 1], make_float2(bq.z, bq.w))), make_float2(wq.z, wq.w), oacc);
          }
        } else {
          const int b = (int)(tile / p.tiles_per_img);
          const float* b1g = p.b1_per_sample ? p.b1 + (size_t)b * p.H : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const float bj = b1g ? __ldg(b1g + min(col0 + j, p.H - 1)) : lds_f32(s_b1 + (uint32_t)(col0 + j) * 4u);
            oacc.x = fmaf(mlp_act_ool(v[j] + bj, p.act), lds_f32(s_w2 + (uint32_t)(col0 + j) * 4u), oacc.x);
          }
        }
        c += 2;
        if (c >= NC) {
          // this group's part of the tile is done: leave the partial sum for the converter warps (buffer of the tile's parity,
          // free again once they have consumed the tile two back)
          const int a = it & 1;
          mbar_wait(&f_empty[a], ((uint32_t)(it >> 1) & 1u) ^ 1u);
          sts_f32(s_part + (uint32_t)a * 2048u, oacc.x + oacc.y);
          __syncwarp();
          if (lane == 0) mbar_arrive(&f_full[a]);
          oacc = make_float2(0.f, 0.f);
          c = grp; tile++; it++;
        }
      }
    } else {
    int it = 0;
    long n1 = 0;
    for (long tile = t_first; tile < t_end; tile++, it++) {
      const int b = (int)(tile / p.tiles_per_img);
      const long px = (tile - (long)b * p.tiles_per_img) * 128 + t;
      float gvo[NO];
#pragma unroll
      for (int o = 0; o < NO; o++) gvo[o] = bwd ? __ldg(p.g + ((size_t)b * NO + o) * p.P + px) : 0.f;
      const float gv = gvo[0];
      const float* b1g = p.b1_per_sample ? p.b1 + (size_t)b * p.H : nullptr;
      float2 oacc = make_float2(0.f, 0.f);
      for (int c = 0; c < NC; c++) {
        const long n = n1 + c;
        const int ab = (int)(n % NA);
        const int col0 = c * 64 + part_id * kEW;   // first hidden index of this thread's kEW columns
        mbar_wait(&acc1_full[ab], (uint32_t)(n / NA) & 1u);
        tc_fence_after();
        float v[kEW];
        tmem_ld16(t_acc1 + lane_base + 64u * ab + part_id * kEW, v);
        // hidden bias for this thread's 32 columns (loads overlap the TMEM read); pad columns (>= H) carry zero
        // W1 rows, zero w2 and a finite bias, so they contribute exactly 0 and need no branches
        float bj[kEW];
        if (b1g) {
#pragma unroll
          for (int j = 0; j < kEW; j++) bj[j] = __ldg(b1g + min(col0 + j, p.H - 1));
        } else {
#pragma unroll
          for (int j = 0; j < kEW; j += 4) *reinterpret_cast<float4*>(bj + j) = *reinterpret_cast<const float4*>(sb1 + col0 + j);
        }
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&acc1_empty[ab]);
        float ga[kEW];
        if (GELU) {
          // packed fp32x2 math: one FMA-pipe instruction per two hidden units
          float2* v2 = reinterpret_cast<float2*>(v);
          const float2* b2 = reinterpret_cast<const float2*>(bj);
          if (bwd && NO > 1) {
            // ga = gelu(z) (scaled by each g[o] in the dw2 reduction below), f = gelu'(z) sum_o g[o] w2[o,j]
            float2* ga2 = reinterpret_cast<float2*>(ga);
#pragma unroll
            for (int j = 0; j < kEW / 2; j++) {
              float2 val, grad;
              b2no_gelu2_both(__fadd2_rn(v2[j], b2[j]), &val, &grad);
              float2 s = __fmul2_rn(b2no_f2(gvo[0]), *reinterpret_cast<const float2*>(sw2 + col0 + 2 * j));
#pragma unroll
              for (int o = 1; o < NO; o++)
                s = __ffma2_rn(b2no_f2(gvo[o]), *reinterpret_cast<const float2*>(sw2 + o * p.Hp + col0 + 2 * j), s);
              ga2[j] = val;
              v2[j] = __fmul2_rn(s, grad);
            }
          } else if (bwd) {
            float2* ga2 = reinterpret_cast<float2*>(ga);
            const float2 gv2 = b2no_f2(gv);
#pragma unroll
            for (int j = 0; j < kEW / 2; j++) {
              const float2 w2p = *reinterpret_cast<const float2*>(sw2 + col0 + 2 * j);
              float2 val, grad;
              b2no_gelu2_both(__fadd2_rn(v2[j], b2[j]), &val, &grad);
              ga2[j] = __fmul2_rn(gv2, val);
              v2[j] = __fmul2_rn(__fmul2_rn(gv2, w2p), grad);
            }
          } else if (direct) {
#pragma unroll
            for (int j = 0; j < kEW / 2; j++) {
              const float2 w2p = *reinterpret_cast<const float2*>(sw2 + col0 + 2 * j);
              oacc = __ffma2_rn(b2no_gelu2(__fadd2_rn(v2[j], b2[j])), w2p, oacc);
            }
          } else {
#pragma unroll
            for (int j = 0; j < kEW / 2; j++) v2[j] = b2no_gelu2(__fadd2_rn(v2[j], b2[j]));
          }
        } else {
#pragma unroll
          for (int j = 0; j < kEW; j++) {
            const float z = v[j] + bj[j];
            if (bwd && NO > 1) {
              float s = gvo[0] * sw2[col0 + j];
#pragma unroll
              for (int o = 1; o < NO; o++) s = fmaf(gvo[o], sw2[o * p.Hp + col0 + j], s);
              ga[j] = b2no_act(z, p.act);
              v[j] = s * b2no_act_grad(z, p.act);
            } else if (bwd) {
              ga[j] = gv * b2no_act(z, p.act);
              v[j] = gv * sw2[col0 + j] * b2no_act_grad(z, p.act);
            } else if (direct) {
              oacc.x = fmaf(b2no_act(z, p.act), sw2[col0 + j], oacc.x);
            } else {
              v[j] = b2no_act(z, p.act);
            }
          }
        }
        if (direct) continue;
        if (bwd) {
          if (p.gz) {
            float* gp = p.gz + ((size_t)b * p.H + col0) * p.P + px;
#pragma unroll
            for (int j = 0; j < kEW; j++)
              if (col0 + j < p.H) gp[(size_t)j * p.P] = v[j];
          }
          // dw2[o,col] += sum over the warp's 32 pixels of g[o] * act(z) (warp_column_sum); one lane of each group of
          // 32 / kEW adds it to the shared-memory total
          constexpr int kDup = 32 / kEW;
          if (NO == 1) {
            const float s = warp_column_sum(ga, lane);
            if ((lane & (kDup - 1)) == 0) atomicAdd(&sdw2[col0 + lane / kDup], s);
          } else {
#pragma unroll
            for (int o = 0; o < NO; o++) {
              float go[kEW];
#pragma unroll
              for (int j = 0; j < kEW; j++) go[j] = gvo[o] * ga[j];
              const float s = warp_column_sum(go, lane);
              if ((lane & (kDup - 1)) == 0) atomicAdd(&sdw2[o * p.Hp + col0 + lane / kDup], s);
            }
          }
        }
        const int fb = (int)(n % p.fbufs);
        mbar_wait(&f_empty[fb], ((uint32_t)(n / p.fbufs) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t fa = t_f + lane_base + 128u * fb + part_id * kEW;
#pragma unroll
        for (int j0 = 0; j0 < kEW; j0 += 8) {
          float lo[8];
#pragma unroll
          for (int j = 0; j < 8; j++) lo[j] = tf32_lo(v[j0 + j]);
          tmem_st8(fa + j0, v + j0);
          tmem_st8(fa + 64 + j0, lo);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&f_full[fb]);
      }
      n1 += NC;
      if (direct) {
        // the column parts of a pixel live in different warps: combine through shared memory (double buffered, one
        // named barrier over the epilogue threads per tile)
        float* part = (float*)(smem + L.part) + (size_t)(it & 1) * (kNP - 1) * 128;
        if (part_id > 0) part[(part_id - 1) * 128 + t] = oacc.x + oacc.y;
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        if (part_id == 0) {
          float o = (oacc.x + oacc.y) + (p.b2 ? __ldg(p.b2) : 0.f);
#pragma unroll
          for (int q = 0; q < kNP - 1; q++) o += part[q * 128 + t];
          p.out[(size_t)b * p.P + px] = o;
        }
        continue;
      }
      // ---- epilogue-2 ----
      const int a2 = it & 1;
      mbar_wait(&acc2_full[a2], (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      for (int cb = part_id; cb * 16 < p.N2; cb += kNP) {
        float o[16];
        tmem_ld16(t_acc2 + lane_base + (uint32_t)(a2 * p.N2 + cb * 16), o);
        tmem_ld_wait();
        const int nout = bwd ? p.Ci : p.Co2;
        float* op = p.out + ((size_t)b * nout + cb * 16) * p.P + px;
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const int ch = cb * 16 + j;
          if (ch < nout) {
            float r = o[j];
            if (!bwd) r += p.b2 ? __ldg(p.b2 + ch) : 0.f;
            else if (p.dz) r *= b2no_act_grad(__ldg(p.dz + ((size_t)b * nout + ch) * p.P + px), p.dact);
            op[(size_t)j * p.P] = r;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&acc2_empty[a2]);
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (bwd && p.dw2_partial)
    for (int i = tid; i < p.H; i += kThreadsMlp)
#pragma unroll
      for (int o = 0; o < NO; o++)
        p.dw2_partial[((size_t)blockIdx.x * NO + o) * p.H + i] = ((float*)(smem + L.dw2))[o * p.Hp + i];
  if (warp == 1) tmem_dealloc(tbase, ncols);
}

// deterministic sum of per-CTA partials: block = 32 outputs x 8 warps over the partials, fixed combine order
__global__ void __launch_bounds__(256)
k_sum_partials(const float* __restrict__ partial, float* __restrict__ out, int nblk, int n) {
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

int mlp_launch(MlpTc& p, const float* x, int batch, long pixels, cudaStream_t st, int* grid_out) {
  if (!b2no_tc_available()) return 1;
  if (pixels % 128 != 0 || p.Ci < 1 || p.Ci > 64 || p.H < 1 || p.H > 512) return 1;
  if (p.mode == 1 && (p.Co2 < 1 || p.Co2 > 4)) return 1;
  const int no = p.mode == 1 ? p.Co2 : 1;   // dw2 rows of the backward
  if ((uintptr_t)x & 15) return 1;
  p.Cip = b2no_round_up(p.Ci, 8);
  p.Hp = b2no_round_up(p.H, 64);
  p.NC = p.Hp / 64;
  p.N2 = p.mode == 1 ? b2no_round_up(p.Ci, 16) : b2no_round_up(p.Co2, 16);
  if (p.N2 > 32) { if (p.mode == 0) return 1; }
  if (p.N2 > 64) return 1;
  p.P = pixels;
  p.tiles_per_img = (int)(pixels / 128);
  p.tiles = (long)batch * p.tiles_per_img;
  p.direct = (p.mode == 0 && p.Co2 == 1) ? 1 : 0;
  p.fbufs = 2;
  if (mlp_tmem_cols(p) > 512) p.fbufs = 1;
  if (mlp_tmem_cols(p) > 512) return 1;
  int dev = 0, max_smem = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  // cuTensorMapEncodeTiled (driver API) needs a current context; a thread whose first CUDA call is this one (autograd's
  // backward thread, when every tensor it allocated came from the caching allocator's pool) has none yet
  B2NO_CHECK_CUDA(cudaSetDevice(dev));
  B2NO_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  MlpLayout L;
  for (p.S = 4; p.S >= 2; p.S--) {
    L = mlp_layout(p, no);
    if ((int)L.total <= max_smem) break;
  }
  if (p.S < 2) return 1;
  long grid = p.tiles < b2no_sm_count() ? p.tiles : b2no_sm_count();
  p.tiles_per_cta = (p.tiles + grid - 1) / grid;
  grid = (p.tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  CUtensorMap tmx;
  uint64_t dims[3] = {(uint64_t)pixels, (uint64_t)p.Ci, (uint64_t)batch};
  uint64_t str[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * p.Ci};
  uint32_t box[3] = {128, (uint32_t)p.Cip, 1};
  if (make_tmap_f32(&tmx, x, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return 1;
#define MLP_LAUNCH(G, W, D, ...)                                                                                        \
  do {                                                                                                                    \
    B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_mlp_tc<G, W, D, ##__VA_ARGS__>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                         (int)L.total));                                                                  \
    k_mlp_tc<G, W, D, ##__VA_ARGS__><<<(unsigned)grid, kThreadsMlp, L.total, st>>>(tmx, p);                             \
  } while (0)
  const bool gelu = p.act == B2NO_ACT_GELU;
  if (p.mode == 1 && no == 2) { if (gelu) MLP_LAUNCH(true, true, false, 2); else MLP_LAUNCH(false, true, false, 2); }
  else if (p.mode == 1 && no == 3) { if (gelu) MLP_LAUNCH(true, true, false, 3); else MLP_LAUNCH(false, true, false, 3); }
  else if (p.mode == 1 && no == 4) { if (gelu) MLP_LAUNCH(true, true, false, 4); else MLP_LAUNCH(false, true, false, 4); }
  else if (p.mode == 1) { if (gelu) MLP_LAUNCH(true, true, false); else MLP_LAUNCH(false, true, false); }
  else if (p.direct) { if (gelu) MLP_LAUNCH(true, false, true); else MLP_LAUNCH(false, false, true); }
  else { if (gelu) MLP_LAUNCH(true, false, false); else MLP_LAUNCH(false, false, false); }
#undef MLP_LAUNCH
  B2NO_LAUNCH_CHECK();
  *grid_out = (int)grid;
  return 0;
}

}  // namespace

void b2no_tc_count_launch();

// forward; returns 0 ok, 1 not eligible
int b2no_tc_mlp_fwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* out, int batch,
                    int ci, int hidden, int co2, long pixels, int b1_per_sample, int act, cudaStream_t st) {
  MlpTc p;
  memset(&p, 0, sizeof(p));
  p.npass = b2no_tc_passes();
  p.B = batch; p.Ci = ci; p.H = hidden; p.Co2 = co2; p.mode = 0; p.act = act; p.b1_per_sample = b1_per_sample;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.out = out;
  int grid = 0;
  const int rc = mlp_launch(p, x, batch, pixels, st, &grid);
  if (rc == 0) b2no_tc_count_launch();
  return rc;
}

// 1 when the backward has a kernel for this shape and `no` outputs (mirrors the checks of mlp_launch)
static int mlp_bwd_supported(int ci, int hidden, int no, int64_t pixels) {
  if (!b2no_tc_available()) return 0;
  if (pixels < 128 || pixels % 128 != 0 || ci < 1 || ci > 64 || hidden < 1 || hidden > 512) return 0;
  MlpTc p;
  memset(&p, 0, sizeof(p));
  p.npass = b2no_tc_passes();
  p.Cip = b2no_round_up(ci, 8); p.Hp = b2no_round_up(hidden, 64); p.N2 = b2no_round_up(ci, 16); p.fbufs = 1; p.S = 2;
  if (mlp_tmem_cols(p) > 512) return 0;
  int dev = 0, max_smem = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 0;
  return (int)mlp_layout(p, no).total <= max_smem ? 1 : 0;
}

extern "C" int b2no_mlp_head_bwd_supported(int ci, int hidden, int64_t pixels) { return mlp_bwd_supported(ci, hidden, 1, pixels); }

extern "C" int64_t b2no_mlp_head_bwd_scratch_floats(int hidden) {
  if (hidden < 1) return B2NO_E_ARG;
  return (int64_t)b2no_sm_count() * hidden;
}

extern "C" int b2no_mlp_head_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* g, float* gx,
                                 float* gz, float* dw2, float* partial, int batch, int ci, int hidden, int64_t pixels,
                                 int b1_per_sample, int act, const float* dact_z, int dact, void* stream) {
  if (!x || !w1 || !w2 || !g || !gx || !dw2 || !partial || batch < 1 || ci < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  MlpTc p;
  memset(&p, 0, sizeof(p));
  p.npass = b2no_tc_passes();
  p.B = batch; p.Ci = ci; p.H = hidden; p.Co2 = 1; p.mode = 1; p.act = act; p.b1_per_sample = b1_per_sample;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.g = g; p.out = gx; p.gz = gz; p.dw2_partial = partial;
  p.dz = dact_z; p.dact = dact_z ? dact : 0;
  int grid = 0;
  const int rc = mlp_launch(p, x, batch, (long)pixels, st, &grid);
  if (rc == 1) return B2NO_E_UNSUPPORTED;
  if (rc) return rc;
  b2no_tc_count_launch();
  k_sum_partials<<<(hidden + 31) / 32, 256, 0, st>>>(partial, dw2, grid, hidden);
  B2NO_LAUNCH_CHECK();
  return 0;
}

// ---- heads with 2..4 output channels (PINObserverFullField's plane_num * out_dim tail, pinobserver.py:230-232 / :257-273;
// neuralop Projection with out_channels > 1, tfno.py:34-38) ----

extern "C" int b2no_mlp_head_fwd_multi(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* out,
                                       int batch, int ci, int hidden, int out_channels, int64_t pixels, int b1_per_sample, int act,
                                       void* stream) {
  if (!x || !w1 || !w2 || !out || batch < 1 || ci < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  if (out_channels < 2 || out_channels > 4) return B2NO_E_UNSUPPORTED;
  const int rc = b2no_tc_mlp_fwd(x, w1, b1, w2, b2, out, batch, ci, hidden, out_channels, (long)pixels, b1_per_sample, act,
                                 (cudaStream_t)stream);
  return rc == 1 ? B2NO_E_UNSUPPORTED : rc;
}

extern "C" int b2no_mlp_head_bwd_multi_supported(int ci, int hidden, int out_channels, int64_t pixels) {
  if (out_channels < 2 || out_channels > 4) return 0;
  return mlp_bwd_supported(ci, hidden, out_channels, pixels);
}

extern "C" int64_t b2no_mlp_head_bwd_multi_scratch_floats(int hidden, int out_channels) {
  if (hidden < 1 || out_channels < 1) return B2NO_E_ARG;
  return (int64_t)b2no_sm_count() * hidden * out_channels;
}

extern "C" int b2no_mlp_head_bwd_multi(const float* x, const float* w1, const float* b1, const float* w2, const float* g, float* gx,
                                       float* gz, float* dw2, float* partial, int batch, int ci, int hidden, int out_channels,
                                       int64_t pixels, int b1_per_sample, int act, const float* dact_z, int dact, void* stream) {
  if (!x || !w1 || !w2 || !g || !gx || !dw2 || !partial || batch < 1 || ci < 1 || hidden < 1 || pixels < 1) return B2NO_E_ARG;
  if (out_channels < 2 || out_channels > 4) return B2NO_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  MlpTc p;
  memset(&p, 0, sizeof(p));
  p.npass = b2no_tc_passes();
  p.B = batch; p.Ci = ci; p.H = hidden; p.Co2 = out_channels; p.mode = 1; p.act = act; p.b1_per_sample = b1_per_sample;
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.g = g; p.out = gx; p.gz = gz; p.dw2_partial = partial;
  p.dz = dact_z; p.dact = dact_z ? dact : 0;
  int grid = 0;
  const int rc = mlp_launch(p, x, batch, (long)pixels, st, &grid);
  if (rc == 1) return B2NO_E_UNSUPPORTED;
  if (rc) return rc;
  b2no_tc_count_launch();
  const int n = out_channels * hidden;   // partial rows: (o, j) of every CTA
  k_sum_partials<<<(n + 31) / 32, 256, 0, st>>>(partial, dw2, grid, n);
  B2NO_LAUNCH_CHECK();
  return 0;
}
