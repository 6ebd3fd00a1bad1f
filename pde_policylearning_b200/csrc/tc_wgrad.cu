// 1x1-convolution weight gradient on tcgen05:  dW[o,i] = sum_{b,p} G[b,o,p] X[b,i,p],  db[o] = sum_{b,p} G[b,o,p]
// (backward of fno_block.py:131 skips, tfno.py:11-38 lifting/projection, rno.py:224-228 / pinobserver.py:223 convs).
//
// The contraction runs over pixels and both tensors are pixel-contiguous, so both operands are K-major exactly as they
// sit in HBM: TMA boxes of [32 px x channels] with the 128-byte swizzle.
//   A = G tile (M = output channels).  Few channels (32) would waste 3/4 of a 128-row shared-memory A read per MMA
//       (measured: the SS form was shared-memory bound, 1.8 TB/s), so the converter warps (thread = channel row) move
//       the G tile into TMEM as hi (raw fp32) | lo = rna_tf32(g - trunc g) and the MMAs run in the TS form;
//   B = X tile straight from the TMA box, each box followed by its elementwise lo copy (written by the converter warps
//       that own no G row), so [X_hi; X_lo] is one B operand of 2 Ci rows;
//   D = [Co x 2 Ci] fp32 in TMEM (the two halves are added at read-out), accumulated over every tile a CTA owns and written once at the end as a per-CTA
//       partial; k_pw_wgrad_reduce (pointwise.cu) sums the partials deterministically;
//   db[o] = sum G[o, .] is summed in registers by the converter thread that owns row o (it reads every G element anyway).
// 3xTF32: hi*hi + lo*hi + hi*lo.
// HBM-bound: what matters is bytes in flight per SM.  With the lo copy and a ones block inside every stage only 3 stages
// (96 KB of payload) fitted and the bare TMA ring topped out at 4.6 TB/s; payload-only stages give 6 x 32 KB.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tc.cuh"

using namespace tc;

namespace {

constexpr int kThreadsWg = 320;  // warps 0-3 converter group A (+ final read-out), 4-7 converter group B, 8 TMA, 9 MMA
constexpr int kWgSlots = 2;      // A-ring slots (TMEM operand + lo copy), one per converter group

struct WgTc {
  int Co, Cop, Ci, Cip, TP, SUB, nb, S, mblocks;   // TP = pixels per TMA stage, SUB = pixels per MMA chunk (A ring slot)
  int tiles_per_img;
  long tiles, tiles_per_cta;
  float* partial;
  int npass;    // 3: 3xTF32, 1: single-pass TF32 (G_hi x X_hi only, accumulator columns [0, Cip))
};

struct WgLayout { uint32_t gbytes, xbytes, x, stage_bytes, dbs, bars, total; };

// A TMA stage = the G boxes [nb][Cop rows x 128 B] and, per X box, 2 Cip rows: the box itself (hi: the tensor core reads the
// top 19 bits of the raw fp32) followed by its elementwise lo copy, so that [X_hi; X_lo] is ONE B operand of 2 Cip rows.
__host__ __device__ inline WgLayout wg_layout(const WgTc& p) {
  WgLayout L;
  L.gbytes = (uint32_t)p.Cop * p.TP * 4;
  L.xbytes = 2u * (uint32_t)p.Cip * p.TP * 4;
  L.x = L.gbytes;
  L.stage_bytes = (L.gbytes + L.xbytes + 1023u) & ~1023u;
  L.dbs = L.stage_bytes * p.S;
  L.bars = L.dbs + 2u * p.mblocks * 128 * 4;
  L.total = L.bars + 8 * (2 * p.S + 2 * kWgSlots + 1) + 16 + 1024;
  return L;
}

// TMEM columns: A operand ring [slot][M-block][hi SUB | lo SUB], then the accumulators [M-block][2 Cip]
// (columns [0, Cip): G_hi X_hi + G_lo X_hi, columns [Cip, 2 Cip): G_hi X_lo; added at read-out)
__host__ __device__ inline uint32_t wg_tmem_cols(const WgTc& p) { return 2u * kWgSlots * p.SUB * p.mblocks + 2u * p.mblocks * p.Cip; }

__global__ void __launch_bounds__(kThreadsWg, 1)
k_wgrad_tc(const __grid_constant__ CUtensorMap tmg, const __grid_constant__ CUtensorMap tmx, const WgTc p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const WgLayout L = wg_layout(p);
  uint64_t* full = (uint64_t*)(smem + L.bars);
  uint64_t* empty = full + p.S;
  uint64_t* a_full = empty + p.S;
  uint64_t* a_empty = a_full + kWgSlots;
  uint64_t* done = a_empty + kWgSlots;
  uint32_t* tslot = (uint32_t*)(done + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NW = p.Cip, TP = p.TP;
  uint32_t ncols = 32;
  while (ncols < wg_tmem_cols(p)) ncols <<= 1;

  if (tid == 0) {
    for (int s = 0; s < p.S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < kWgSlots; a++) { mbar_init(&a_full[a], 128); mbar_init(&a_empty[a], 1); }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 9) tmem_alloc(tslot, ncols);
  if (warp == 8 && lane == 0) { tma_prefetch_desc(&tmg); tma_prefetch_desc(&tmx); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tslot;
  const int SUB = p.SUB, nsub = TP / SUB, nbs = SUB / 32;
  const uint32_t t_acc = tbase + 2u * kWgSlots * SUB * p.mblocks;
  const long t_first = (long)blockIdx.x * p.tiles_per_cta;
  const long t_end = t_first + p.tiles_per_cta < p.tiles ? t_first + p.tiles_per_cta : p.tiles;

  if (warp == 8) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const uint32_t bytes = (uint32_t)(p.Cop + p.Cip) * TP * 4;
      int it = 0;
      for (long tile = t_first; tile < t_end; tile++, it++) {
        const int s = it % p.S;
        const uint32_t ph = (uint32_t)(it / p.S) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full[s], bytes);
        uint8_t* st = smem + (size_t)s * L.stage_bytes;
        const int b = (int)(tile / p.tiles_per_img);
        const int p0 = (int)(tile - (long)b * p.tiles_per_img) * TP;
        for (int j = 0; j < p.nb; j++) {
          tma_load_3d(st + (size_t)j * p.Cop * 128, &tmg, &full[s], p0 + 32 * j, 0, b);
          tma_load_3d(st + L.x + (size_t)j * 2 * NW * 128, &tmx, &full[s], p0 + 32 * j, 0, b);
        }
      }
    }
  } else if (warp == 9) {
    // ===================== MMA issuer (TS form: A = G from TMEM, B = X from shared memory) =====================
    // Per K step of 8 px: G_hi x [X_hi; X_lo] as ONE MMA with N = 2 Cip, then G_lo x X_hi (N = Cip) -- an MMA of this shape
    // costs ~40 cycles whatever its N, and the issue of a chunk's MMAs was the longest item of the hand-over period
    const uint32_t idesc = idesc_tf32(128, NW, 0, 0), idesc2 = idesc_tf32(128, 2 * NW, 0, 0);
    const uint32_t sbase = smem_u32(smem);
    int it = 0;
    long n = 0;                      // A-ring position (sub-chunk counter)
    uint32_t acc = 0;
    for (long tile = t_first; tile < t_end; tile++, it++) {
      const int s = it % p.S;
      const uint32_t ph = (uint32_t)(it / p.S) & 1u;
      mbar_wait(&full[s], ph);
      for (int sub = 0; sub < nsub; sub++, n++) {
        const uint32_t un = (uint32_t)n, uq = un / kWgSlots;   // 32-bit: a 64-bit division here cost 15 us per launch
        const int ab = (int)(un % kWgSlots);
        mbar_wait(&a_full[ab], uq & 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t st = sbase + (uint32_t)s * L.stage_bytes;
          for (int mb = 0; mb < p.mblocks; mb++) {
            const uint32_t d = t_acc + (uint32_t)(mb * 2 * NW);
            const uint32_t a0 = tbase + (uint32_t)((ab * p.mblocks + mb) * 2 * SUB);
            uint32_t a2 = acc;
            for (int j = 0; j < nbs; j++) {
              const uint64_t dx = smem_desc(st + L.x + (uint32_t)(sub * nbs + j) * 2 * NW * 128, 16, 1024, LAYOUT_SW128);
#pragma unroll
              for (int ks = 0; ks < 4; ks++) {
                mma_tf32_ts(d, a0 + (uint32_t)(j * 32 + ks * 8), dx + (uint64_t)(ks * 2), p.npass == 3 ? idesc2 : idesc, a2);
                a2 = 1;
              }
              if (p.npass == 3) {
#pragma unroll
                for (int ks = 0; ks < 4; ks++)
                  mma_tf32_ts(d, a0 + (uint32_t)(SUB + j * 32 + ks * 8), dx + (uint64_t)(ks * 2), idesc, 1u);
              }
            }
          }
          if (sub == nsub - 1) mma_commit(&empty[s]);
          mma_commit(&a_empty[ab]);
        }
        acc = 1;
        __syncwarp();
      }
    }
    if (elect_one()) mma_commit(done);
    __syncwarp();
  } else {
    // ===================== converter: X lo in shared memory; G rows -> TMEM A operand (thread = channel row) =====================
    // two groups of four warps alternate over the sub-chunks (chunk n -> group n % 2 and ring slot n % 2), so conversion of
    // chunk n+1 overlaps the MMAs of chunk n
    const int grp = warp >> 2;
    const int ct = tid & 127;
    const int quad = warp & 3;
    const int m = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float dbsum[3] = {0.f, 0.f, 0.f};          // db partial of rows m, 128 + m, 256 + m over this group's chunks
    int it = 0;
    long n = 0;
    for (long tile = t_first; tile < t_end; tile++, it++) {
      const int s = it % p.S;
      const uint32_t ph = (uint32_t)(it / p.S) & 1u;
      mbar_wait(&full[s], ph);
      uint8_t* st = smem + (size_t)s * L.stage_bytes;
      for (int sub = 0; sub < nsub; sub++, n++) {
        // (measured and rejected: BOTH groups converting every chunk, one box each: 96 vs 80 us -- every chunk then
        // synchronises all eight warps; G rows loaded into registers ahead of the slot wait: 90 vs 80 us)
        if ((int)(n & 1) != grp) continue;
        {
          // lo copy of this chunk's X boxes, elementwise (layout-agnostic), into the rows right after each box; it needs
          // no ring slot, so it runs before the slot wait -- and on the warps that own no real G row when there are such
          // (Co <= 96: the quad-0 warp converts while the other three copy)
          const int first_idle = (p.mblocks == 1) ? ((p.Cop + 31) >> 5) : 4;      // quads >= first_idle hold only pad rows
          const int nidle = 4 - first_idle;
          const bool copier = nidle == 0 || quad >= first_idle;
          if (copier) {
            const int cthreads = nidle == 0 ? 128 : nidle * 32;
            const int cid = nidle == 0 ? ct : (quad - first_idle) * 32 + lane;
            const uint32_t per_box = (uint32_t)NW * 128 / 16;
            for (int j = 0; j < nbs; j++) {
              const float4* src = (const float4*)(st + L.x + (size_t)(sub * nbs + j) * 2 * NW * 128);
              float4* dst = (float4*)((uint8_t*)src + (size_t)NW * 128);
              for (uint32_t i = cid; i < per_box; i += cthreads) {
                const float4 x = src[i];
                dst[i] = make_float4(x.x - tf32_trunc(x.x), x.y - tf32_trunc(x.y), x.z - tf32_trunc(x.z), x.w - tf32_trunc(x.w));
              }
            }
          }
        }
        const uint32_t un = (uint32_t)n, uq = un / kWgSlots;
        const int ab = (int)(un % kWgSlots);
        mbar_wait(&a_empty[ab], (uq & 1u) ^ 1u);                     // MMAs of this slot's previous chunk are complete
        tc_fence_after();
#pragma unroll
        for (int mb = 0; mb < 3; mb++) {
          if (mb >= p.mblocks) break;
          const int row = mb * 128 + m;
          const uint32_t a0 = tbase + lane_base + (uint32_t)((ab * p.mblocks + mb) * 2 * SUB);
          // tcgen05.st is warp-collective (.sync.aligned): the branch must be warp-uniform, so a warp that owns at least
          // one real row converts all 32 of its rows (pad rows as zeros); warps of pure pad rows zero their lanes once
          if (mb * 128 + quad * 32 < p.Cop) {
            const bool real = row < p.Cop;
            for (int j = 0; j < nbs; j++) {
              float hi[32], lo[32];
              const uint8_t* rp = st + (size_t)(sub * nbs + j) * p.Cop * 128 + (size_t)(real ? row : 0) * 128;
#pragma unroll
              for (int i = 0; i < 8; i++)
                *reinterpret_cast<float4*>(hi + 4 * i) = *reinterpret_cast<const float4*>(rp + ((i ^ (row & 7)) << 4));
              if (!real) {
#pragma unroll
                for (int i = 0; i < 32; i++) hi[i] = 0.f;
              }
              float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                s0 += hi[i]; s1 += hi[i + 1]; s2 += hi[i + 2]; s3 += hi[i + 3];
              }
              dbsum[mb] += (s0 + s1) + (s2 + s3);
#pragma unroll
              for (int i = 0; i < 32; i++) lo[i] = hi[i] - tf32_trunc(hi[i]);   // exact; the tensor core truncates it to tf32
              tmem_st16(a0 + (uint32_t)(j * 32), hi); tmem_st16(a0 + (uint32_t)(j * 32 + 16), hi + 16);
              tmem_st16(a0 + (uint32_t)(SUB + j * 32), lo); tmem_st16(a0 + (uint32_t)(SUB + j * 32 + 16), lo + 16);
            }
          } else if (n < kWgSlots) {
            // pad rows (>= Cop) of an M block: zeroed once per ring slot, never written again
            float z[16];
#pragma unroll
            for (int i = 0; i < 16; i++) z[i] = 0.f;
            for (int c = 0; c < 2 * SUB; c += 16) tmem_st16(a0 + (uint32_t)c, z);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        fence_proxy_async();
        mbar_arrive(&a_full[ab]);
      }
    }
    // db: both groups publish their row sums, group A combines them (fixed order)
    float* dbs = (float*)(smem + L.dbs);
#pragma unroll
    for (int mb = 0; mb < 3; mb++)
      if (mb < p.mblocks) dbs[(grp * p.mblocks + mb) * 128 + m] = dbsum[mb];
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // read-out (group A): thread = accumulator row
    if (grp == 0) {
      mbar_wait(done, 0);
      tc_fence_after();
      float* pout = p.partial + (size_t)blockIdx.x * ((size_t)p.Co * p.Ci + p.Co);
      const bool any = t_end > t_first;
      for (int mb = 0; mb < p.mblocks; mb++) {
        const int o = mb * 128 + m;
        for (int c0 = 0; c0 < NW; c0 += 16) {
          float v[16], u[16];
          tmem_ld16(t_acc + lane_base + (uint32_t)(mb * 2 * NW + c0), v);
          tmem_ld16(t_acc + lane_base + (uint32_t)(mb * 2 * NW + NW + c0), u);
          tmem_ld_wait();
          if (p.npass == 3) {
#pragma unroll
            for (int j = 0; j < 16; j++) v[j] += u[j];
          }
          if (o < p.Co) {
#pragma unroll
            for (int j = 0; j < 16; j++) {
              const int c = c0 + j;
              if (c < p.Ci) pout[(size_t)o * p.Ci + c] = any ? v[j] : 0.f;
            }
          }
        }
        if (o < p.Co) pout[(size_t)p.Co * p.Ci + o] = dbs[mb * 128 + m] + dbs[(p.mblocks + mb) * 128 + m];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc(tbase, ncols);
}

}  // namespace

void b2no_tc_count_launch();

// Fills `partial` with *nblk per-CTA partials laid out [Co*Ci | Co]; returns 0 on success, 1 if not eligible.
int b2no_tc_wgrad(const float* g, const float* x, float* partial, int max_blocks, int batch, int ci, int co, long pixels,
                  int* nblk, cudaStream_t st) {
  if (!b2no_tc_available()) return 1;
  if (pixels % 128 != 0 || ci > 240 || co > 384 || ci < 1 || co < 1) return 1;
  if (((uintptr_t)g | (uintptr_t)x) & 15) return 1;
  WgTc p;
  memset(&p, 0, sizeof(p));
  p.Co = co; p.Cop = b2no_round_up(co, 8); p.Ci = ci; p.Cip = b2no_round_up(ci, 16);
  p.mblocks = (p.Cop + 127) / 128;
  int dev = 0, max_smem = 0;
  B2NO_CHECK_CUDA(cudaGetDevice(&dev));
  B2NO_CHECK_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  WgLayout L;
  bool ok = false;
  // two ring slots of 64 px (one M block) / 32 px.  Measured on B200 (cfg2, Co = Ci = 32): four slots of 32 px are SLOWER
  // (155 us vs 87 us) -- the cost is per chunk hand-over (~0.7 us), not per pixel, so chunks are as large as TMEM allows;
  // a third 64-px slot changes nothing (93.6 vs 93.4 us): the converters do not wait for free slots
  p.SUB = p.mblocks == 1 ? 64 : 32;
  if (p.mblocks > 3 || wg_tmem_cols(p) > 512) return 1;
  // bytes in flight decide an HBM-bound kernel: take the largest tile that still leaves >= 4 stages, else the deepest ring
  for (int pass = 0; pass < 2 && !ok; pass++)
    for (p.TP = 256; p.TP >= p.SUB && !ok; p.TP >>= 1) {
      if (pixels % p.TP != 0) continue;
      for (p.S = 8; p.S >= (pass == 0 ? 4 : 2); p.S--) {
        L = wg_layout(p);
        if ((int)L.total <= max_smem) { ok = true; break; }
      }
      if (ok) break;
    }
  if (!ok) return 1;
  p.nb = p.TP / 32;
  p.tiles_per_img = (int)(pixels / p.TP);
  p.tiles = (long)batch * p.tiles_per_img;
  long grid = b2no_sm_count();
  if (grid > max_blocks) grid = max_blocks;
  if (grid > p.tiles) grid = p.tiles;
  p.tiles_per_cta = (p.tiles + grid - 1) / grid;
  grid = (p.tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
  p.partial = partial;
  p.npass = b2no_tc_passes();
  CUtensorMap tmg, tmx;
  {
    uint64_t dims[3] = {(uint64_t)pixels, (uint64_t)co, (uint64_t)batch};
    uint64_t str[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * co};
    uint32_t box[3] = {32, (uint32_t)p.Cop, 1};
    if (make_tmap_f32(&tmg, g, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    uint64_t dims2[3] = {(uint64_t)pixels, (uint64_t)ci, (uint64_t)batch};
    uint64_t str2[3] = {4, (uint64_t)pixels * 4, (uint64_t)pixels * 4 * ci};
    uint32_t box2[3] = {32, (uint32_t)p.Cip, 1};
    if (make_tmap_f32(&tmx, x, 3, dims2, str2, box2, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  B2NO_CHECK_CUDA(cudaFuncSetAttribute(k_wgrad_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  k_wgrad_tc<<<(unsigned)grid, kThreadsWg, L.total, st>>>(tmg, tmx, p);
  B2NO_LAUNCH_CHECK();
  b2no_tc_count_launch();
  *nblk = (int)grid;
  return 0;
}
