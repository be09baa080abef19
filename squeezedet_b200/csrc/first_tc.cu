// First layer on tcgen05 (SQDET_MATH_TF32X3_TC): conv over the 3-channel image (KxK, stride 2) +
// bias [+ frozen BN] + ReLU + stride-2 max-pool, ONE kernel, the conv tensor never exists.
//
// Replaces _conv_layer('conv1') + _pooling_layer('pool1') of the reference
// (src/nets/squeezeDet.py:40-44, src/nn_skeleton.py:471-586; SqueezeDet 1242x375: 3x3/2 SAME,
// 64 filters, 3x3/2 SAME pool) - until now the largest kernel of the step, on FFMA lanes.
//
// Formulation ("the pool is a max over accumulators"): the GEMM's M rows are POOLED pixels.
//   item      = an 8 x 16 tile of pooled pixels of one image (TMEM lane = pooled pixel)
//   stage j   = one of the PK*PK pooling-window offsets (a, b): the conv evaluated at conv pixel
//               (2*Y - pad + a, 2*X - pad + b) for every pooled pixel (Y, X) of the tile:
//               D_j[128 pooled pixels, Cout] = A_j[128, K] * Wt[K, Cout],  K = 3*KS*KS padded to 32s
//   drain     = acc = max(acc, D_j) over the valid window cells (cells outside the conv image are
//               skipped = tf.nn.max_pool's "ignore padding"), then +bias [*scale+shift], ReLU
//               (max commutes with the monotone per-channel epilogue, so the result is the
//               reference's max-pool of the activated conv), TMA store of the pooled tile.
// A conv pixel is shared by up to 2.25 windows and is recomputed for each (the tensor pipe has the
// room: 12 MMAs of N/2 clocks per stage), in exchange for an epilogue with no cross-lane traffic
// at all - the pooled-epilogue variant of conv_tc.cu lost to the FFMA kernel because of its ~1300
// dependent instructions of smem pooling per item.
// Operands: the input patch of an item (35 rows x 67 pixels for 3x3/2 + 3x3/2) is fetched ONCE, row
//   by row, with 1-D TMA loads (double-buffered).  Rows of a 3-channel fp32 image are only 4-byte
//   aligned and TMA wants 16-byte aligned global starts, so each row is fetched from its start
//   rounded down to 4 floats; out-of-range coordinates are zero-filled by the TMA unit.  (A first
//   version copied the patch with 4-byte cp.async from three warps: 217 clocks per element issued,
//   the loader was 96 % of the kernel.)  Four splitter warps build each stage's im2col rows from
//   the patch with aligned 128-bit reads - the 9 floats of a tap row start at 12*px + 6*b floats
//   plus the row's alignment shift, which is warp-uniform, so the 0..3 float offset is resolved by a
//   uniform 4-way branch - mask the taps that fall outside the image (SAME padding; only on edge
//   tiles), split a = a_hi + a_lo (3xTF32, see conv_tc.cu) and write [a_hi | a_lo] into tensor
//   memory (tcgen05.st); the MMAs take A from TMEM and the packed hi/lo weights from shared
//   memory, where they stay RESIDENT for the whole launch (one TMA load per CTA).
// Roles (640 threads): warpgroup 4 = two MMA issuers (one per accumulator buffer; warp 17 owns
//   TMEM) and two repack warps, one of which also issues the TMA row fetches;
//   warpgroups 2,3 splitters
//   (alternate stages: one warp per scheduler could not hide its own lds -> tcgen05.st latency,
//   ~1080 clocks per stage measured); warpgroups 0,1 drain + epilogue, each owning alternate
//   32-channel groups of EVERY stage (alternating items left one group idle while the other
//   paced the MMAs through the two accumulator buffers).
#include <cuda.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"
#include "first_tc.cuh"
#include "tc_ptx.cuh"

namespace sqdet {
namespace {

constexpr int FT_THREADS = 640;   // 5 warpgroups: {TMA, MMA, 2 spare} | splitter x2 | drain x2
constexpr int FT_MAX_N = 64;       // output channels (the drain keeps one running max per channel)
constexpr int FT_SA = 4;                      // A slots ([a_hi | a_lo] = 64 columns each) in TMEM
constexpr int FT_PT_H = 8, FT_PT_W = 16;      // pooled tile
constexpr int FT_STAGING = 8 * 2 * 4096;      // per drain warp: ring of two 32-pixel x 32-channel tiles
constexpr int FT_PARAMS = 2 * 3 * FT_MAX_N * 4;   // per drain group: bias, scale, shift
constexpr int FT_XCHG = 2 * 2 * 32 * 128 * 4;     // [item parity][group][32 channels][128 pixels]

struct FirstParams {
  CUtensorMap tmW;     // packed weights [kblock][hi N rows | lo N rows][32], box {32, N}
  CUtensorMap tmY;     // pooled output [B, Hp, Wp, Cout], box {32 ch, 16 w, 2 h, 1}
  CUtensorMap tmX;     // the whole input as a 1-D array of floats, box = `box` floats
  const float* x;
  const float* bias;
  const float* scale;  // null unless frozen BN
  const float* shift;
  int B, H, W;
  int Hc, Wc, cpad_t, cpad_l;       // conv output grid and pad_before
  int pk, ppad_t, ppad_l, Hp, Wp;   // pool window (2 or 3, stride 2), pad_before, pooled grid
  int N, cout, relu;
  int tiles_h, tiles_w, ntiles;
  int prows, box, pitch;            // patch: rows, floats fetched per row, floats between rows
  int patch_bytes;
  int tmem_cols;
  float bias_comp;
  long long* dbg;      // optional per-CTA cycle counters (SQDET_TC_DEBUG=1)
};

#define FT_WAIT(counter, bar, parity)                       \
  do {                                                      \
    if (p.dbg) {                                            \
      const long long _t0 = clock64();                      \
      mbar_wait(bar, parity);                               \
      counter += clock64() - _t0;                           \
    } else {                                                \
      mbar_wait(bar, parity);                               \
    }                                                       \
  } while (0)

// One 32-wide K block of the im2col row of a conv pixel, read straight from the TMA-fetched patch.
// k = (dy, dx, c) in HWIO order; the 3*KS floats of tap row dy are contiguous.  Patch row R holds
// the input row from its global start rounded down to 4 floats, i.e. shifted right by
// (M0 + DSH*R) & 3 floats (M0 = the item's origin & 3, DSH = floats per image row & 3; R = row0 + dy
// with row0 even, so for DSH in {0, 2} the shift of tap row dy is (M0 + DSH*dy) & 3, warp-uniform).
// `rowaddr` = shared address of float (row0, f0 & ~3); FSH = f0 & 3 (f0 = 6 * conv column: 0 or 2).
// All alignment cases are compile-time: 8 variants, selected by one warp-uniform branch per stage.
template <int KS, int KB, int M0, int FSH, int DSH>
__device__ __forceinline__ void gather_kblock(uint32_t rowaddr, uint32_t pitch_b, float (&v)[32]) {
  constexpr int RUN = 3 * KS, KTOT = KS * KS * 3;
  constexpr int K0 = KB * 32, K1 = (K0 + 32 < KTOT) ? K0 + 32 : KTOT;
  constexpr int DY0 = K0 / RUN, DY1 = (K1 - 1) / RUN;
#pragma unroll
  for (int e = 0; e < 32; ++e) v[e] = 0.f;
#pragma unroll
  for (int dy = DY0; dy <= DY1; ++dy) {
    const int r_lo = (K0 > dy * RUN) ? K0 - dy * RUN : 0;
    const int r_hi = (K1 - 1 < dy * RUN + RUN - 1) ? K1 - 1 - dy * RUN : RUN - 1;
    const int tot = FSH + ((M0 + DSH * dy) & 3);
    const uint32_t ra = rowaddr + (uint32_t)dy * pitch_b;
#pragma unroll
    for (int c = (r_lo + tot) >> 2; c <= ((r_hi + tot) >> 2); ++c) {
      const float4 q = lds128(ra + (uint32_t)(c * 16));
      const float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = 4 * c + i - tot;
        if (r >= r_lo && r <= r_hi) v[dy * RUN + r - K0] = qq[i];
      }
    }
  }
}

// zero the taps outside the image (SAME padding; columns outside hold a neighbour row's data):
// bit dy of rmask / bit dx of cmask = tap row / column inside.  Tiles on the image border only.
template <int KS, int KB>
__device__ __forceinline__ void mask_kblock(uint32_t rmask, uint32_t cmask, float (&v)[32]) {
  constexpr int RUN = 3 * KS, KTOT = KS * KS * 3;
#pragma unroll
  for (int e = 0; e < 32; ++e) {
    const int k = KB * 32 + e;
    if (k < KTOT) {
      const int dy = k / RUN, dx = (k % RUN) / 3;
      if (!(((rmask >> dy) & 1u) && ((cmask >> dx) & 1u))) v[e] = 0.f;
    }
  }
}

template <int KS, int KB, int M0, int FSH, int DSH>
__device__ __forceinline__ void split_kblock(uint32_t rowaddr, uint32_t pitch_b, bool edge,
                                             uint32_t rmask, uint32_t cmask, uint32_t a_slot) {
  float v[32];
  gather_kblock<KS, KB, M0, FSH, DSH>(rowaddr, pitch_b, v);
  if (edge) mask_kblock<KS, KB>(rmask, cmask, v);
#pragma unroll
  for (int hblk = 0; hblk < 2; ++hblk) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const float h = rn_tf32(v[hblk * 16 + e]);
      hi[e] = __float_as_uint(h);
      lo[e] = __float_as_uint(v[hblk * 16 + e] - h);
    }
    tmem_st16(a_slot + (uint32_t)(hblk * 16), hi);
    tmem_st16(a_slot + (uint32_t)(32 + hblk * 16), lo);
  }
}

template <int KS, int M0, int FSH, int DSH>
__device__ __forceinline__ void split_kblock_n(int kb, uint32_t rowaddr, uint32_t pitch_b, bool edge,
                                               uint32_t rmask, uint32_t cmask, uint32_t a_slot) {
  constexpr int NKB = (KS * KS * 3 + 31) / 32;
  if (kb == 0) split_kblock<KS, 0, M0, FSH, DSH>(rowaddr, pitch_b, edge, rmask, cmask, a_slot);
  if (NKB > 1 && kb == 1)
    split_kblock<KS, (NKB > 1 ? 1 : 0), M0, FSH, DSH>(rowaddr, pitch_b, edge, rmask, cmask, a_slot);
  if (NKB > 2 && kb == 2)
    split_kblock<KS, (NKB > 2 ? 2 : 0), M0, FSH, DSH>(rowaddr, pitch_b, edge, rmask, cmask, a_slot);
  if (NKB > 3 && kb == 3)
    split_kblock<KS, (NKB > 3 ? 3 : 0), M0, FSH, DSH>(rowaddr, pitch_b, edge, rmask, cmask, a_slot);
  if (NKB > 4 && kb == 4)
    split_kblock<KS, (NKB > 4 ? 4 : 0), M0, FSH, DSH>(rowaddr, pitch_b, edge, rmask, cmask, a_slot);
}

// End of an item in drain group DG: write the partial maxima of the channels the OTHER group stores
// to the exchange buffer, meet at a named barrier, combine ours with the other group's, apply the
// epilogue and stage the 32-pixel x 32-channel tile for the TMA store.  TWO = 64 output channels
// (both groups store), else 32 (group 0 stores).  Returns whether a tile was staged.
template <int DG, bool TWO>
__device__ __forceinline__ bool drain_tail(float (&acc)[FT_MAX_N], uint32_t xb, int tt, uint32_t par,
                                           uint32_t tile_w, int lane, float gain, bool affine,
                                           float lo_clip) {
  constexpr int OWN = TWO ? DG * 32 : 0, GIVE = TWO ? (1 - DG) * 32 : 0;
  if (TWO || DG == 1) {
#pragma unroll
    for (int e = 0; e < 32; ++e)
      sts32(xb + 4u * (uint32_t)((DG * 32 + e) * 128 + tt), acc[GIVE + e]);
  }
  asm volatile("bar.sync 3, 256;" ::: "memory");
  if (!TWO && DG == 1) return false;
  if (lane == 0) tma_store_wait_read_le1();               // the tile used two stores ago is free
  __syncwarp();
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    const int c = OWN + kk * 4;
    const float4 b0 = lds128(par + 4u * (uint32_t)c);
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float other = lds32(xb + 4u * (uint32_t)(((1 - DG) * 32 + kk * 4 + i) * 128 + tt));
      o[i] = fmaxf(acc[OWN + kk * 4 + i], other) * gain;
    }
    o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w;
    if (affine) {
      const float4 s0 = lds128(par + 4u * (uint32_t)(FT_MAX_N + c));
      const float4 h0 = lds128(par + 4u * (uint32_t)(2 * FT_MAX_N + c));
      o[0] = o[0] * s0.x + h0.x; o[1] = o[1] * s0.y + h0.y;
      o[2] = o[2] * s0.z + h0.z; o[3] = o[3] * s0.w + h0.w;
    }
    float4 v;
    v.x = fmaxf(o[0], lo_clip); v.y = fmaxf(o[1], lo_clip);
    v.z = fmaxf(o[2], lo_clip); v.w = fmaxf(o[3], lo_clip);
    sts128(tile_w + (uint32_t)(lane * 128 + ((kk ^ (lane & 7)) << 4)), v);
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
template <int KS, int DSH>
__global__ void __launch_bounds__(FT_THREADS, 1)
first_tc_kernel(const __grid_constant__ FirstParams p) {
  constexpr int CS = 2;                                  // conv stride
  constexpr int NKB = (KS * KS * 3 + 31) / 32;           // 32-wide K blocks per window offset
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                             ~uintptr_t(1023));
  const int N = p.N;
  const uint32_t WB = (uint32_t)N * 128u;                // one [N][32] fp32 tile
  const uint32_t smem_b = smem_u32(smem);
  const uint32_t w_b = smem_b;                           // [NKB][hi | lo]
  const uint32_t out_b = w_b + (uint32_t)NKB * 2u * WB;  // 1024-aligned (N % 8 == 0)
  const uint32_t par_b = out_b + FT_STAGING;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)NKB * 2 * WB + FT_STAGING + FT_PARAMS);
  uint64_t* wfull = bars;               // weights landed
  uint64_t* pfull = bars + 1;           // [2] TMA -> splitters (patch rows landed)
  uint64_t* pempty = bars + 3;          // [2] splitters -> TMA producer
  uint64_t* split = bars + 5;           // [SA] splitter -> MMA
  uint64_t* aempty = bars + 5 + FT_SA;  // [SA] MMA (commit) -> splitter
  uint64_t* tfull = bars + 5 + 2 * FT_SA;   // [2 pipelines][2] MMA -> drain
  uint64_t* tempty = tfull + 4;         // [2 pipelines][2] drain -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 4);
  const uint32_t xchg_b = smem_b + (uint32_t)((size_t)NKB * 2 * WB + FT_STAGING + FT_PARAMS + 256);
  const uint32_t patch_b = xchg_b + FT_XCHG;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Role of each warpgroup.  The issue arbiter of an SM sub-partition favours the highest warp id
  // among its eligible warps (B300 microarchitecture notes), and every sub-partition here holds one
  // warp of every role: the short critical roles (TMA producer, MMA issuer, repack) get the highest
  // ids, then the splitters, the drains run in what is left.
  const int wg = warp >> 2;   // 0,1 drains, 2,3 splitters, 4 TMA + MMA
  const int wq = warp & 3;                                 // warp within its warpgroup
  const int PK = p.pk, NOFF = PK * PK;

  if (threadIdx.x == 0) {
    mbar_init(wfull, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&pfull[b], 1);
      mbar_init(&pempty[b], 256);
    }
    for (int s = 0; s < FT_SA; ++s) {
      mbar_init(&split[s], 128);
      mbar_init(&aempty[s], 1);
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (wg == 4 && wq == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (wg == 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (wq == 1 || wq == 2) {
      // ============================ MMA issuers (warps 17, 18) ================================
      // One issuer per accumulator buffer: warp 17 + mw takes the window offsets g with g % 2 == mw
      // (D buffer mw, A slots mw and mw + 2, fed by splitter group mw).  Measured: with ONE
      // issuer its serial path per stage (two barrier waits, fence, 12 MMAs, two commits: ~650
      // clocks) paced the whole kernel although the 12 MMAs are only 384 clocks of tensor pipe.
      const int mw = wq - 1;
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) |
                             ((uint32_t)(128 >> 4) << 24);
      const uint32_t w_u = __shfl_sync(0xffffffffu, w_b, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint64_t desc_hi = make_desc<32>(0) & 0xFFFFFFFF00000000ull;
      const uint32_t desc_lo0 = (uint32_t)(make_desc<32>(0) & 0xFFFFFFFFull);
      mbar_wait(wfull, 0u);
      int c = 0, g = 0, n = 0;
      long long w_split = 0, w_tempty = 0;
      const long long t_begin = clock64();
      for (int item = blockIdx.x; item < p.ntiles; item += gridDim.x) {
        for (int j = 0; j < NOFF; ++j, ++g) {
          if ((g & 1) != mw) continue;
          const int buf = mw * 2 + (n & 1);                 // this pipeline's two accumulator buffers
          FT_WAIT(w_tempty, &tempty[buf], (((uint32_t)n >> 1) & 1u) ^ 1u);
          ++n;
          const uint32_t d_tmem = tmem_u + (uint32_t)(buf * N);
#pragma unroll 1
          for (int kb = 0; kb < NKB; ++kb, ++c) {
            const int slot = mw + 2 * (c & 1);
            FT_WAIT(w_split, &split[slot], ((uint32_t)c >> 1) & 1u);
            tc_fence_after();
            const uint32_t b_hi = desc_lo0 | ((w_u + (uint32_t)kb * 2u * WB) >> 4);
            const uint32_t b_lo = b_hi + (WB >> 4);
            const uint32_t a_hi = tmem_u + (uint32_t)(4 * N + slot * 64);
            const uint32_t a_lo = a_hi + 32u;
            if (elect_one()) {
              // not unrolled: hoisting all 12 descriptors makes the 32-register issuer warps spill
#pragma unroll 1
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t dbh = desc_hi | (uint64_t)(b_hi + 2 * ks);
                const uint64_t dbl = desc_hi | (uint64_t)(b_lo + 2 * ks);
                umma_tf32_ts(d_tmem, a_lo + 8 * ks, dbh, idesc, (kb != 0 || ks != 0) ? 1u : 0u);
                umma_tf32_ts(d_tmem, a_hi + 8 * ks, dbl, idesc, 1u);
                umma_tf32_ts(d_tmem, a_hi + 8 * ks, dbh, idesc, 1u);
              }
              umma_commit(&aempty[slot]);                 // the A slot may be rewritten
              if (kb == NKB - 1) umma_commit(&tfull[buf]);
            }
            __syncwarp();
          }
        }
      }
      if (p.dbg && lane == 0 && mw == 0) {
        p.dbg[blockIdx.x * 12 + 0] = clock64() - t_begin;
        p.dbg[blockIdx.x * 12 + 1] = w_split;
        p.dbg[blockIdx.x * 12 + 2] = w_tempty;
        p.dbg[blockIdx.x * 12 + 3] = g;
      }
    } else {
      // ================================ TMA producer (warp 16) ================================
      // one 1-D row fetch per lane; rows above / below the image fetch a neighbour's data or zero
      // fill, columns left / right of it the neighbouring row's - the splitters mask those taps
      if (wq == 0) {
        if (lane == 0) {
          mbar_expect_tx(wfull, (uint32_t)NKB * 2u * WB);
          for (int i = 0; i < NKB * 2; ++i)
            tma_load_2d(smem + (size_t)i * WB, &p.tmW, wfull, 0, i * N);
        }
        const int row_f = p.W * 3;
        long long w_pempty = 0;
        int k = 0;
        for (int item = blockIdx.x; item < p.ntiles; item += gridDim.x, ++k) {
          const int pb = k & 1;
          int tile = item;
          const int tw = tile % p.tiles_w;
          tile /= p.tiles_w;
          const int th = tile % p.tiles_h;
          const int img = tile / p.tiles_h;
          const int iy0 = (th * FT_PT_H * 2 - p.ppad_t) * CS - p.cpad_t;
          const int if0 = ((tw * FT_PT_W * 2 - p.ppad_l) * CS - p.cpad_l) * 3;
          const int e0 = (img * p.H + iy0) * row_f + if0;     // flat float index of the patch origin
          uint8_t* dst0 = smem + (size_t)(patch_b - smem_b) + (size_t)pb * p.patch_bytes;
          if (lane == 0) {
            FT_WAIT(w_pempty, &pempty[pb], (((uint32_t)k >> 1) & 1u) ^ 1u);
            mbar_expect_tx(&pfull[pb], (uint32_t)(p.prows * p.box * 4));
          }
          __syncwarp();
          for (int r = lane; r < p.prows; r += 32)
            tma_load_1d(dst0 + (size_t)r * p.pitch * 4, &p.tmX, &pfull[pb], (e0 + r * row_f) & ~3);
        }
        if (p.dbg && lane == 0) p.dbg[blockIdx.x * 12 + 4] = w_pempty;
      }
    }
  } else if (wg >= 2) {
    // ================================ operand splitters =====================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    const int sgroup = wg - 2;                          // feeds MMA issuer `sgroup`: window offsets g % 2 == sgroup
    const int t = threadIdx.x & 127;
    const int py = t >> 4, px = t & 15;
    const uint32_t pitch_b = (uint32_t)p.pitch * 4u;
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    int k = 0, c = 0, g = 0;
    long long w_pfull = 0, w_aempty = 0;
    const int row_f = p.W * 3;
    const int pcols = ((FT_PT_W - 1) * 2 + PK - 1) * CS + KS;
    for (int item = blockIdx.x; item < p.ntiles; item += gridDim.x, ++k) {
      const int pb = k & 1;
      int tile = item;
      const int tw = tile % p.tiles_w;
      tile /= p.tiles_w;
      const int th = tile % p.tiles_h;
      const int img = tile / p.tiles_h;
      const int iy0 = (th * FT_PT_H * 2 - p.ppad_t) * CS - p.cpad_t;
      const int ix0 = (tw * FT_PT_W * 2 - p.ppad_l) * CS - p.cpad_l;
      const int m0 = ((img * p.H + iy0) * row_f + ix0 * 3) & 3;     // shift of the even patch rows
      const bool edge = iy0 < 0 || iy0 + p.prows > p.H || ix0 < 0 || ix0 + pcols > p.W;   // uniform
      FT_WAIT(w_pfull, &pfull[pb], ((uint32_t)k >> 1) & 1u);
      const uint32_t patch = patch_b + (uint32_t)(pb * p.patch_bytes);
      int a = 0, b = 0;
      for (int j = 0; j < NOFF; ++j, ++g) {
        if ((g & 1) == sgroup) {                            // this group's window offsets
          const int row0 = (2 * py + a) * CS;
          const int f0 = (2 * px + b) * CS * 3;             // 6 * conv column: 0 or 2 mod 4
          const uint32_t rowaddr = patch + (uint32_t)row0 * pitch_b + 4u * (uint32_t)(f0 & ~3);
          uint32_t rmask = 0u, cmask = 0u;
          if (edge) {
#pragma unroll
            for (int d = 0; d < KS; ++d) {
              const int gy = iy0 + row0 + d, gx = ix0 + (2 * px + b) * CS + d;
              rmask |= (gy >= 0 && gy < p.H) ? (1u << d) : 0u;
              cmask |= (gx >= 0 && gx < p.W) ? (1u << d) : 0u;
            }
          }
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb, ++c) {
            const int slot = sgroup + 2 * (c & 1);
            FT_WAIT(w_aempty, &aempty[slot], (((uint32_t)c >> 1) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t a_slot = tmem_base + lane_sel + (uint32_t)(4 * N + slot * 64);
            switch (m0 * 2 + (b & 1)) {                     // warp-uniform
              case 0: split_kblock_n<KS, 0, 0, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 1: split_kblock_n<KS, 0, 2, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 2: split_kblock_n<KS, 1, 0, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 3: split_kblock_n<KS, 1, 2, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 4: split_kblock_n<KS, 2, 0, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 5: split_kblock_n<KS, 2, 2, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              case 6: split_kblock_n<KS, 3, 0, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
              default: split_kblock_n<KS, 3, 2, DSH>(kb, rowaddr, pitch_b, edge, rmask, cmask, a_slot); break;
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(&split[slot]);
          }
        }
        if (++b == PK) { b = 0; ++a; }
      }
      mbar_arrive(&pempty[pb]);       // every read of this patch has been consumed
    }
    if (p.dbg && t == 0 && sgroup == 0) {
      p.dbg[blockIdx.x * 12 + 6] = w_pfull;
      p.dbg[blockIdx.x * 12 + 7] = w_aempty;
    }
  } else {
    // ============================ max-drain + epilogue ========================================
    // register pool of the CTA: 640 x 96 at launch; warpgroup 4 gives back 128 x 64, the splitters
    // 256 x 16 -> the drain warpgroups can grow by 12288 / 256 = 48 (asking for more than the CTA's
    // own pool holds blocks forever)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 144;");
    // Drain group dg serves pipeline dg: the window offsets g with g % 2 == dg, ALL channels; the
    // two partial maxima of an item meet through shared memory and group dg stores the channel
    // group jg = dg.
    const int dg = wg;
    const int q = warp & 3;
    const int r = q * 32 + lane;                 // accumulator row = pooled pixel of the tile
    const int py = r >> 4, px = r & 15;
    const int tt = threadIdx.x & 127;
    // epilogue parameters: the same for every item of the launch
    const uint32_t par = par_b + (uint32_t)(dg * 3 * FT_MAX_N * 4);
    {
      const bool in = tt < p.cout;
      sts32(par + 4u * (uint32_t)tt, (in && p.bias) ? __ldg(p.bias + tt) : 0.f);
      sts32(par + 4u * (uint32_t)(FT_MAX_N + tt), (in && p.scale) ? __ldg(p.scale + tt) : 1.f);
      sts32(par + 4u * (uint32_t)(2 * FT_MAX_N + tt), (in && p.scale) ? __ldg(p.shift + tt) : 0.f);
      asm volatile("bar.sync %0, 128;" ::"r"(1 + dg) : "memory");
    }
    const bool affine = p.scale != nullptr;
    const float lo_clip = p.relu ? 0.f : -CUDART_INF_F;
    // every accumulator is a chain of 12*NKB MMAs from zero (see conv_tc.cu: truncation bias)
    const float gain = 1.f + p.bias_comp * (float)(12 * NKB);
    const bool two = N > 32;
    float acc[FT_MAX_N];
    int g = 0, n = 0, k = 0, n_store = 0;
    long long w_tfull = 0, c_epi = 0;
    for (int item = blockIdx.x; item < p.ntiles; item += gridDim.x, ++k) {
      int tile = item;
      const int tw = tile % p.tiles_w;
      tile /= p.tiles_w;
      const int th = tile % p.tiles_h;
      const int img = tile / p.tiles_h;
      const int cy0 = (th * FT_PT_H + py) * 2 - p.ppad_t;      // conv row of window offset a = 0
      const int cx0 = (tw * FT_PT_W + px) * 2 - p.ppad_l;
      int a = 0, b = 0;
      bool first = true;
      for (int j = 0; j < NOFF; ++j, ++g) {
        if ((g & 1) == dg) {
          const int buf = dg * 2 + (n & 1);
          FT_WAIT(w_tfull, &tfull[buf], ((uint32_t)n >> 1) & 1u);
          ++n;
          tc_fence_after();
          const bool valid = (cy0 + a) >= 0 && (cy0 + a) < p.Hc && (cx0 + b) >= 0 && (cx0 + b) < p.Wc;
          const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * N);
          // all of the accumulator's columns in ONE tcgen05.ld round trip (~250 clocks each:
          // two rounds per stage made the drain the pacing role)
          uint32_t v[4][16];
          tmem_ld16_nowait(trow, v[0]);
          tmem_ld16_nowait(trow + 16u, v[1]);
          if (two) {                             // warp-uniform
            tmem_ld16_nowait(trow + 32u, v[2]);
            tmem_ld16_nowait(trow + 48u, v[3]);
          }
          tmem_wait_ld();
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            if (h < 2 || two) {
              if (first) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  acc[h * 16 + e] = valid ? __uint_as_float(v[h][e]) : -CUDART_INF_F;
              } else if (valid) {
#pragma unroll
                for (int e = 0; e < 16; ++e)
                  acc[h * 16 + e] = fmaxf(acc[h * 16 + e], __uint_as_float(v[h][e]));
              }
            }
          }
          first = false;
          // Free the buffer only once the loaded values have been consumed: an arrive issued
          // right after tcgen05.wait::ld let the next window's MMAs overwrite columns the last
          // tcgen05.ld had not read yet (intermittently wrong pool1 channels 32-63).
          tc_fence_before();
          mbar_arrive(&tempty[buf]);
        }
        if (++b == PK) { b = 0; ++a; }
      }
      // ---- the two pipelines' partial maxima meet: hand the other group its channels, take ours;
      // then each warp stores pooled rows 2q, 2q+1 of the tile (its 32 TMEM lanes), channel group dg
      const long long te0 = p.dbg ? clock64() : 0;
      const uint32_t xb = xchg_b + (uint32_t)((k & 1) * 2 * 32 * 128 * 4);
      const uint32_t tile_w = out_b + (uint32_t)((dg * 4 + q) * 8192 + (n_store & 1) * 4096);
      bool stored;
      if (dg == 0) {
        stored = two ? drain_tail<0, true>(acc, xb, tt, par, tile_w, lane, gain, affine, lo_clip)
                     : drain_tail<0, false>(acc, xb, tt, par, tile_w, lane, gain, affine, lo_clip);
      } else {
        stored = two ? drain_tail<1, true>(acc, xb, tt, par, tile_w, lane, gain, affine, lo_clip)
                     : drain_tail<1, false>(acc, xb, tt, par, tile_w, lane, gain, affine, lo_clip);
      }
      if (stored) {                              // warp-uniform
        fence_async_proxy();
        __syncwarp();
        if (lane == 0)
          tma_store_4d(tile_w, &p.tmY, dg * 32, tw * FT_PT_W, th * FT_PT_H + q * 2, img);
        ++n_store;
      }
      if (p.dbg) c_epi += clock64() - te0;
    }
    if (lane == 0) tma_store_wait_all();
    if (p.dbg && dg == 0 && tt == 0) {
      p.dbg[blockIdx.x * 12 + 8] = w_tfull;
      p.dbg[blockIdx.x * 12 + 9] = c_epi;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (wg == 4 && wq == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
struct FirstImpl {
  FirstParams prm;
  int ksize = 3, nkb = 1;
  size_t smem_bytes = 0;
  dim3 grid;
  float* d_w = nullptr;
  float* d_bias = nullptr;
  float* d_scale = nullptr;
  float* d_shift = nullptr;
  // the input address is baked into the 1-D tensor map; the engine feeds the first layer from
  // several buffers (pipelined inputs), so maps are cached per address
  long long x_floats = 0;
  mutable std::vector<std::pair<const float*, CUtensorMap>> xmaps;
};

inline float ft_rn_tf32(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

void release_first(void** impl) {
  if (!*impl) return;
  FirstImpl* im = static_cast<FirstImpl*>(*impl);
  cudaFree(im->d_w);
  cudaFree(im->d_bias);
  cudaFree(im->d_scale);
  cudaFree(im->d_shift);
  delete im;
  *impl = nullptr;
}

}  // namespace

int first_tc_plan(FirstTcPlan* plan, int B, int H, int W, int Cout, int ksize, int stride,
                  int conv_padding, int relu, bool has_affine, int pool_size, int pool_stride,
                  int pool_padding, float* y_dev) {
  plan->enabled = false;
  if (ksize != 3 || stride != 2 || pool_stride != 2 || (pool_size != 2 && pool_size != 3)) return 0;
  if (Cout % 32 != 0 || Cout < 32 || Cout > FT_MAX_N) return 0;
  const Geom ch = tf_geometry(H, ksize, stride, conv_padding), cw = tf_geometry(W, ksize, stride, conv_padding);
  if (ch.out <= 0 || cw.out <= 0) return 0;
  const Geom ph = tf_geometry(ch.out, pool_size, 2, pool_padding), pw = tf_geometry(cw.out, pool_size, 2, pool_padding);
  if (ph.out <= 0 || pw.out <= 0) return 0;
  if ((long long)B * H * W * 3 >= (1LL << 31)) return 0;
  if (W % 2 != 0) return 0;      // floats per image row must be 0 or 2 mod 4 (see gather_kblock)
  FirstImpl* im = new FirstImpl();
  FirstParams& P = im->prm;
  memset(&P, 0, sizeof P);
  im->ksize = ksize;
  im->nkb = (ksize * ksize * 3 + 31) / 32;
  P.B = B; P.H = H; P.W = W;
  im->x_floats = (long long)B * H * W * 3;
  P.Hc = ch.out; P.Wc = cw.out; P.cpad_t = ch.pad_before; P.cpad_l = cw.pad_before;
  P.pk = pool_size; P.ppad_t = ph.pad_before; P.ppad_l = pw.pad_before; P.Hp = ph.out; P.Wp = pw.out;
  P.N = Cout; P.cout = Cout; P.relu = relu;
  P.tiles_h = (P.Hp + FT_PT_H - 1) / FT_PT_H;
  P.tiles_w = (P.Wp + FT_PT_W - 1) / FT_PT_W;
  P.ntiles = B * P.tiles_h * P.tiles_w;
  P.prows = ((FT_PT_H - 1) * 2 + pool_size - 1) * stride + ksize;
  // floats per patch row + up to 3 floats of alignment shift, rounded to 16 bytes; TMA wants
  // 128-byte aligned shared destinations, so rows sit at a pitch that is a multiple of 32 floats
  P.box = ((((FT_PT_W - 1) * 2 + pool_size - 1) * stride + ksize) * 3 + 3 + 3) / 4 * 4;
  if (P.box > 256) { delete im; return 0; }
  P.pitch = (P.box + 31) / 32 * 32;
  P.patch_bytes = P.prows * P.pitch * 4;
  {
    int cols = 32;
    while (cols < 4 * P.N + FT_SA * 64) cols <<= 1;
    if (cols > 512) { delete im; return 0; }
    P.tmem_cols = cols;
  }
  static const float env_comp = env_float("SQDET_TC_BIAS_COMP", 1.4e-8f);
  P.bias_comp = env_comp;
  im->smem_bytes = 1024 + (size_t)im->nkb * 2 * P.N * 128 + FT_STAGING + FT_PARAMS + 256 + FT_XCHG +
                   2 * (size_t)P.patch_bytes;
  if (im->smem_bytes > 232448) { delete im; return 0; }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  im->grid = dim3((unsigned)(P.ntiles < sms ? P.ntiles : sms));
  void* pim = im;
  const size_t wfloats = (size_t)im->nkb * 2 * P.N * 32;
  if (cudaMalloc(&im->d_w, sizeof(float) * wfloats) != cudaSuccess ||
      cudaMalloc(&im->d_bias, sizeof(float) * Cout) != cudaSuccess) {
    release_first(&pim);
    return fail(SQDET_ERR_CUDA, "first_tc_plan: cudaMalloc failed");
  }
  cudaMemset(im->d_w, 0, sizeof(float) * wfloats);
  cudaMemset(im->d_bias, 0, sizeof(float) * Cout);
  P.bias = im->d_bias;
  if (has_affine) {
    if (cudaMalloc(&im->d_scale, sizeof(float) * Cout) != cudaSuccess ||
        cudaMalloc(&im->d_shift, sizeof(float) * Cout) != cudaSuccess) {
      release_first(&pim);
      return fail(SQDET_ERR_CUDA, "first_tc_plan: cudaMalloc failed");
    }
    P.scale = im->d_scale;
    P.shift = im->d_shift;
  }
  int rc = tc_encode_w_map(&P.tmW, im->d_w, im->nkb * 2 * P.N, 32, P.N);
  if (!rc) rc = tc_encode_act_map(&P.tmY, y_dev, B, P.Hp, P.Wp, Cout, 32, FT_PT_W, 2);
  if (rc) {
    release_first(&pim);
    return rc;
  }
  cudaError_t ce = cudaFuncSetAttribute(first_tc_kernel<3, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        232448);
  if (ce == cudaSuccess)
    ce = cudaFuncSetAttribute(first_tc_kernel<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  if (ce != cudaSuccess) {
    release_first(&pim);
    return cuda_fail(ce, "cudaFuncSetAttribute(first_tc_kernel)");
  }
  plan->enabled = true;
  plan->B = B; plan->H = H; plan->W = W; plan->Cout = Cout; plan->ksize = ksize;
  plan->impl = im;
  return 1;
}

int first_tc_pack_weights(FirstTcPlan* plan, const float* w_hwio, const float* bias) {
  FirstImpl* im = static_cast<FirstImpl*>(plan->impl);
  const int N = im->prm.N, ktot = im->ksize * im->ksize * 3;
  // HWIO flattened is [k = (dy, dx, c)][Cout]; packed rows: [kblock][hi rows 0..N) | lo rows][32]
  std::vector<float> packed((size_t)im->nkb * 2 * N * 32, 0.f);
  for (int kb = 0; kb < im->nkb; ++kb)
    for (int n = 0; n < plan->Cout; ++n)
      for (int e = 0; e < 32; ++e) {
        const int k = kb * 32 + e;
        if (k >= ktot) continue;
        const float v = w_hwio[(size_t)k * plan->Cout + n];
        const float hi = ft_rn_tf32(v);
        packed[((size_t)(kb * 2) * N + n) * 32 + e] = hi;
        packed[((size_t)(kb * 2 + 1) * N + n) * 32 + e] = ft_rn_tf32(v - hi);
      }
  SQ_CUDA(cudaMemcpy(im->d_w, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (bias) SQ_CUDA(cudaMemcpy(im->d_bias, bias, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int first_tc_set_affine(FirstTcPlan* plan, const float* scale, const float* shift) {
  FirstImpl* im = static_cast<FirstImpl*>(plan->impl);
  if (!im->d_scale) return fail(SQDET_ERR_STATE, "first layer planned without an affine epilogue");
  SQ_CUDA(cudaMemcpy(im->d_scale, scale, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_shift, shift, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int launch_first_tc(const FirstTcPlan& plan, const float* x_dev, cudaStream_t stream) {
  const FirstImpl* im = static_cast<const FirstImpl*>(plan.impl);
  FirstParams prm = im->prm;
  prm.x = x_dev;
  {
    bool found = false;
    for (auto& m : im->xmaps)
      if (m.first == x_dev) { prm.tmX = m.second; found = true; break; }
    if (!found) {
      CUtensorMap m;
      int rc = tc_encode_flat_map(&m, x_dev, im->x_floats, prm.box);
      if (rc) return rc;
      if (im->xmaps.size() >= 8) im->xmaps.erase(im->xmaps.begin());
      im->xmaps.emplace_back(x_dev, m);
      prm.tmX = m;
    }
  }
  static const int debug = env_int("SQDET_TC_DEBUG", 0);
  long long* dbg = nullptr;
  const int nb = (int)im->grid.x;
  if (debug) {
    SQ_CUDA(cudaMalloc(&dbg, sizeof(long long) * 12 * nb));
    SQ_CUDA(cudaMemsetAsync(dbg, 0, sizeof(long long) * 12 * nb, stream));
    prm.dbg = dbg;
  }
  if ((prm.W * 3) & 3)
    SQ_CUDA(launch_kernel(first_tc_kernel<3, 2>, im->grid, dim3(FT_THREADS), im->smem_bytes, stream, prm));
  else
    SQ_CUDA(launch_kernel(first_tc_kernel<3, 0>, im->grid, dim3(FT_THREADS), im->smem_bytes, stream, prm));
  SQ_CHECK_LAUNCH("first_tc_kernel");
  if (debug) {
    std::vector<long long> h((size_t)12 * nb);
    SQ_CUDA(cudaStreamSynchronize(stream));
    SQ_CUDA(cudaMemcpy(h.data(), dbg, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    cudaFree(dbg);
    double a[12] = {0};
    for (int b = 0; b < nb; ++b)
      for (int k = 0; k < 12; ++k) a[k] += (double)h[(size_t)b * 12 + k] / nb;
    fprintf(stderr,
            "[first_tc] grid %d tiles %d N %d offsets %d | per-CTA avg cycles: total %.0f (%.0f stages) | "
            "mma waits: split %.0f tempty %.0f | producer: wait-empty %.0f (%.0f) | splitter waits: "
            "patch %.0f a-slot %.0f | drain(group 0): wait-tfull %.0f epilogue %.0f\n",
            nb, prm.ntiles, prm.N, prm.pk * prm.pk, a[0], a[3], a[1], a[2], a[4], a[5], a[6], a[7], a[8],
            a[9]);
  }
  return SQDET_OK;
}

void first_tc_release(FirstTcPlan* plan) {
  release_first(&plan->impl);
  plan->enabled = false;
}

}  // namespace sqdet
