// tcgen05 implicit-GEMM convolution with the 3xTF32 split (SQDET_MATH_TF32X3_TC).
//
// Replaces tf.nn.conv2d + bias_add [+ batch_normalization] + relu of the reference
// (src/nn_skeleton.py:539-547, :441-449) for every stride-1 conv whose Cin is a multiple
// of 16 (all fire squeeze/expand convs, the ConvDet head, the VGG/ResNet body) and for 3x3
// convs over 3-channel images ("gather mode"), and fuses a fire module's expand1x1 ||
// expand3x3 + channel concat (src/nets/squeezeDet.py:96-106) into one launch.
//
// GEMM view per CTA:  D[128 pixels, N] += A[128 pixels, K] * W[K, N]
//   M tile  = an 8 x 16 patch of output pixels of one image (TMEM lane = pixel); 128 consecutive
//             pixels of the flattened B*H*W list when the launch holds only 1x1 convs
//   N       = one chunk of output channels (multiple of 16, <= 128; TMEM column = channel)
//   K       = taps x Cin, walked as (tap, 32- or 16-channel chunk)
//   A       : TMA tiled load of the NHWC activation tensor, box {KC ch, 16 w, 8 h, 1 n} at
//             the tap-shifted coordinate; out-of-image coordinates are zero-filled by the
//             TMA unit = TF "SAME" zero padding; lands K-major with the 128B/64B swizzle.
//   W       : host-packed [chunk][tap][kchunk][N][KC] fp32 (hi and lo halves), 2-D TMA.
// Precision: fp32 operands are split a = a_hi + a_lo with a_hi = rn_tf32(a), a_lo = a - a_hi
//   (exact; the tensor core reads its top 19 bits); D += a_lo*b_hi + a_hi*b_lo + a_hi*b_hi with
//   fp32 accumulation in TMEM (kind::tf32).  Dropped terms ~ 2^-21: fp32-grade results, which the
//   1e-4 parity bar against the fp32 reference needs through ~25 stacked convs (plain TF32
//   or BF16 miss it by 1-2 orders of magnitude).  Weights are pre-split on the host.  The
//   activation split is done by 4 warps between the TMA landing and the MMA issue: each thread
//   reads its pixel's row of the raw tile from smem and writes a_hi / a_lo into TENSOR MEMORY
//   (tcgen05.st); the MMAs take A from TMEM (.ts form) and only B from smem.  (With A in smem
//   the kernel was shared-memory-bandwidth bound; measured, see DESIGN.md.)
// Accumulation: the tensor core adds into its fp32 accumulator with truncation (measured
//   on B200: a systematic shrink, linear in the number of chained MMAs, 3.6e-5 of max at
//   K=6912 vs 2e-6 for fp32 FFMA).  So a tile's K loop is cut into SEGMENTS of 36 MMAs, each
//   accumulated from zero in one of two TMEM buffers; the drain warps add finished segments
//   into fp32 registers (round-to-nearest) scaled by 1 + 1.4e-8 * (MMAs in the segment), the
//   measured first-order size of the remaining bias; the drain of segment g overlaps the MMAs of
//   segment g+1.
// Persistent CTAs (one per SM, 512 threads = 4 warpgroups) over (chunk, tile) items, round-robin
//   or a host-computed longest-processing-time-first schedule:  warpgroup 0: warp 0 = TMA
//   producer, warp 1 = TMEM owner + MMA issuer (one elected lane), warps 2-3 idle;  warpgroup 1 =
//   operand splitter;  warpgroups 2 and 3 = segment drain + epilogue (tcgen05.ld -> fp32 FFMA ->
//   +bias [*scale+shift] -> relu -> TMA store), alternating items (measured: one drain group was
//   the bottleneck of the small-K layers - the MMA warp spent 30-45 % of its time waiting for
//   TMEM buffers).  setmaxnreg moves registers from warpgroups 0/1 to the drain warpgroups, whose
//   running sums (up to 128 per thread) must stay out of local memory.
// Pipelines: full[s] (TMA -> splitter), split[s] (splitter -> MMA), empty[s]
//   (tcgen05.commit -> TMA), tfull[group][b] (tcgen05.commit -> drain), tempty[b] (drain -> MMA).
// Variants measured and removed (weight multicast over CTA clusters, CTA-pair MMA, a second
//   splitter warpgroup, a fused max-pool epilogue): DESIGN.md 4.1.
// Roofline: SqueezeDet fire2-9 are HBM-bound even fused (AI 24-95 FLOP/B fp32 I/O),
//   fire10/11 ~ridge, ConvDet tensor-bound (SURVEY.md §8d); 3xTF32 costs 3 MMAs at the
//   TF32 rate per algorithmic MAC.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <math_constants.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <queue>
#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace sqdet {
namespace {

constexpr int TILE_H = 8, TILE_W = 16, TILE_M = TILE_H * TILE_W;   // 128 pixels
constexpr int NUM_THREADS = 512;       // 4 warpgroups: {TMA, MMA, 2 spare} | splitter | drain A | drain B
constexpr int MAX_CHUNKS = 16;
constexpr int MAX_N = 128;          // output channels per item (register-resident running sums)
constexpr int MAX_STAGES = 8;
constexpr int GATHER_PITCH = 128;   // floats between patch rows in the stage (gather mode)

struct TcChunk {
  int ksize;        // 1 or 3 (square)
  int pad;          // SAME: (ksize-1)/2
  int w_row_base;   // first row of this chunk in the packed weight matrix (hi half)
  int ch_base;      // output channel (within this conv group) of TMEM column 0
  int ch_count;     // valid output channels in this chunk
  int y_coff;       // channel offset of ch_base..ch_base+ch_count in the output tensor
  int bias_base;    // index of ch_base in the bias/scale/shift arrays
  int tap_begin;    // first filter tap of this chunk (split-K partials cover tap sub-ranges)
  int tap_count;    // number of taps (ksize*ksize unless split)
  int kc_begin;     // first K chunk (of KC input channels) of this chunk; split-K partials cover ranges
  int kc_count;     // number of K chunks (Cin / KC unless split)
};

struct TcParams {
  CUtensorMap tmA;
  CUtensorMap tmW;
  CUtensorMap tmY;      // output tensor, box {32 ch, 16 w, 8 h, 1}, SWIZZLE_128B (TMA-store epilogue)
  const float* bias;    // may be null
  const float* scale;   // may be null (frozen BN)
  const float* shift;
  float* y;
  int B, Ho, Wo, tiles_h, tiles_w;
  int kch;              // Cin / KC
  int N;                // UMMA N (uniform over chunks)
  int tmem_cols;        // power of two >= 2*N (two accumulator buffers) + stages*2*KC (A slots)
  int seg_stages;       // pipeline stages (K blocks) per accumulation segment
  float bias_comp;      // first-order compensation of the accumulator's truncation bias, per chained MMA
  int ntiles;           // B * tiles_h * tiles_w
  int tma_store;        // 1: epilogue stages 32-channel groups in smem and issues TMA stores
  // conv tile (rows of the M=128 MMA tile): ct_h x ct_w output pixels, tile t starts at t * ct
  int ct_h, ct_w;
  int sq_w, sq_h;       // TMA-store epilogue: offset of drain warp q's 32-pixel slab in the tile
  // gather mode (first layer: 3x3 conv over a 3-channel image): the A tile is the im2col
  // of an input patch; the producer fetches the patch row by row with 1-D TMA loads (rows of a
  // 3-channel fp32 image are only 4-byte aligned, which rules out the tiled 4-D map), K = 27
  // padded to one 32-wide K block
  CUtensorMap tmX;      // the whole input as a 1-D array of floats, box = g_box floats
  int gather;           // 1 = gather mode
  int g_H, g_W, g_stride, g_pad_t, g_pad_l;
  int g_ph, g_box;      // patch rows; floats fetched per patch row (patch columns * 3, padded to 4)
  int store_ring;       // per-warp TMA-store staging tiles (2, or 1 to buy one more pipeline stage)
  // static schedule (launches whose chunks differ in cost): sched[0 .. nbins] = first entry of each
  // CTA's item list, followed by the lists (longest-processing-time-first assignment);
  // null = round-robin `item = CTA id + k * CTAs`
  const int* sched;
  long long* dbg;       // optional per-CTA cycle counters (SQDET_TC_DEBUG=1), else null
  int y_cstride, relu;
  int lo_row_offset;    // rows between the hi and the lo copy of the packed weights
  int stages;
  int nchunks;
  TcChunk chunk[MAX_CHUNKS];
};

// Debug-only stall accounting: cycles spent inside a barrier wait, per role.
#define SQ_TIMED_WAIT(counter, bar, parity)                 \
  do {                                                      \
    if (p.dbg) {                                            \
      const long long _t0 = clock64();                      \
      mbar_wait(bar, parity);                               \
      counter += clock64() - _t0;                           \
    } else {                                                \
      mbar_wait(bar, parity);                               \
    }                                                       \
  } while (0)

// ---------------------------------------------------------------------------------------------
template <int KC, bool GATHER>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_tc_kernel(const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                             ~uintptr_t(1023));
  constexpr int A_BYTES = TILE_M * KC * 4;
  const int B_BYTES = p.N * KC * 4;
  const int STAGE_BYTES = A_BYTES + 2 * B_BYTES;   // [A raw][B hi][B lo]
  const int S = p.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)S * STAGE_BYTES);
  uint64_t* full = bars;                    // [S]  TMA -> splitter
  uint64_t* split = bars + MAX_STAGES;      // [S]  splitter -> MMA
  uint64_t* empty = bars + 2 * MAX_STAGES;  // [S]  MMA -> TMA
  // tfull is per (drain group, TMEM buffer): an mbarrier waiter must observe every phase in
  // order, so each group gets barriers only it waits on; tempty's only waiter is the MMA warp.
  uint64_t* tfull = bars + 3 * MAX_STAGES;  // [2 groups][2]  MMA -> drain (segment accumulated)
  uint64_t* tempty = tfull + 4;             // [2]  drain -> MMA (buffer read out)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  // per-item epilogue parameters (bias, scale, shift), double-buffered by item parity
  float* s_par = reinterpret_cast<float*>(tempty + 4);   // [2 groups][2][3][MAX_N]
  // two 16 KB output staging tiles (128 pixels x 32 channels, 128B-swizzled) for TMA stores
  uint8_t* s_out = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(s_par + 4 * 3 * MAX_N) + 1023) & ~uintptr_t(1023));

  // 32-bit shared-window addresses of the regions above (see lds128 / sts128)
  const uint32_t smem_b = smem_u32(smem);
  const uint32_t par_b = smem_b + (uint32_t)(reinterpret_cast<uint8_t*>(s_par) - smem);
  const uint32_t out_b = smem_b + (uint32_t)(s_out - smem);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Work decomposition: items are (chunk, tile) pairs, item = chunk * ntiles + tile.
  const int cta = (int)blockIdx.x, n_ctas = (int)gridDim.x;
  const int total_items = p.ntiles * p.nchunks;
  const int G = p.seg_stages;
  // this CTA's items: entries [k_begin, k_end) of the static schedule, or round-robin
  const int k_begin = p.sched ? __ldg(p.sched + cta) : 0;
  const int k_end = p.sched ? __ldg(p.sched + cta + 1) : (total_items - cta + n_ctas - 1) / n_ctas;
#define SQ_FOR_ITEMS(...)                                                                \
  for (int k_ = k_begin, nxt_ = (p.sched && k_begin < k_end) ? __ldg(p.sched + k_begin) : 0, \
           item = p.sched ? nxt_ : cta;                                                  \
       k_ < k_end;                                                                       \
       ++k_, item = p.sched ? nxt_ : cta + k_ * n_ctas __VA_ARGS__)                      \
    if (p.sched && k_ + 1 < k_end ? (nxt_ = __ldg(p.sched + k_ + 1), true) : true)

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&split[s], 128);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 4; ++b) mbar_init(&tfull[b], 1);
    for (int b = 0; b < 2; ++b) mbar_init(&tempty[b], 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Register re-balancing between the warpgroups (launch bound: 168/thread) happens at the top
  // of every role branch, so that ptxas sees one register budget per branch.
  // Items are ordered chunk-major (all tiles of chunk 0, then chunk 1, ...) so that the static
  // round-robin gives every CTA the same mix of cheap (1x1) and expensive (3x3) items.
  if (warp < 4) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");   // one instruction for the whole warpgroup
   if (warp == 0) {
    // ================================ TMA producer =====================================
    if (lane == 0) {
      int it = 0, st_i = 0;
      uint32_t st_ph = 0;
      long long w_empty = 0;
      const long long t_begin = clock64();
      SQ_FOR_ITEMS() {
        const TcChunk ck = p.chunk[item / p.ntiles];
        int tile = item % p.ntiles;
        const int tw = tile % p.tiles_w;
        tile /= p.tiles_w;
        const int h0 = (tile % p.tiles_h) * p.ct_h, w0 = tw * p.ct_w;
        const int img = tile / p.tiles_h;
        const int iters = ck.tap_count * ck.kc_count;
        const uint32_t a_bytes = (uint32_t)(p.ct_h * p.ct_w * KC * 4);   // the TMA box
        for (int i = 0; i < iters; ++i, ++it) {
          const int s = st_i;
          const uint32_t ph = st_ph;
          if (++st_i == S) { st_i = 0; st_ph ^= 1u; }
          SQ_TIMED_WAIT(w_empty, &empty[s], ph ^ 1u);
          uint8_t* st = smem + (size_t)s * STAGE_BYTES;
          mbar_expect_tx(&full[s], (GATHER ? (uint32_t)(p.g_ph * p.g_box * 4) : a_bytes) +
                                       (uint32_t)(2 * B_BYTES));
          const int tl = i / ck.kc_count, kc = ck.kc_begin + (i - tl * ck.kc_count);
          const int tap = ck.tap_begin + tl;
          const int dy = tap / ck.ksize, dx = tap - dy * ck.ksize;
          if (GATHER) {
            // patch rows at a 512-byte pitch in the stage's A region.  TMA needs a 16-byte aligned global start: every row is fetched from its start
            // rounded down to 4 floats (the splitter adds the 0..3 float offset back); rows
            // above / below the image fetch a neighbour's data or zero fill, which the splitter
            // masks (padding) or which only feed conv pixels the epilogue masks
            const int e0 = ((img * p.g_H + h0 * p.g_stride - p.g_pad_t) * p.g_W +
                            (w0 * p.g_stride - p.g_pad_l)) * 3;
            for (int r = 0; r < p.g_ph; ++r)
              tma_load_1d(st + r * (GATHER_PITCH * 4), &p.tmX, &full[s],
                          (e0 + r * p.g_W * 3) & ~3);
          } else {
            tma_load_4d(st, &p.tmA, &full[s], kc * KC, w0 + dx - ck.pad, h0 + dy - ck.pad, img);
          }
          const int row = ck.w_row_base + i * p.N;
          tma_load_2d(st + A_BYTES, &p.tmW, &full[s], 0, row);
          tma_load_2d(st + A_BYTES + B_BYTES, &p.tmW, &full[s], 0, row + p.lo_row_offset);
        }
      }
      if (p.dbg) {
        p.dbg[blockIdx.x * 12 + 0] = w_empty;
        p.dbg[blockIdx.x * 12 + 5] = clock64() - t_begin;
        p.dbg[blockIdx.x * 12 + 6] = it;
      }
    }
   } else if (warp == 1) {
    // ================================ MMA issuer =========================================
    // The whole warp walks the loop (warp-uniform addresses/descriptors live in uniform
    // registers); only lane 0 issues tcgen05.mma / tcgen05.commit.
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.N >> 3) << 17) |
                           ((uint32_t)(TILE_M >> 4) << 24);
    const uint32_t smem_base = __shfl_sync(0xffffffffu, smem_u32(smem), 0);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);   // provably warp-uniform
    const uint64_t desc_hi = make_desc<KC>(0) & 0xFFFFFFFF00000000ull;   // layout/SBO/version
    const uint32_t desc_lo0 = (uint32_t)(make_desc<KC>(0) & 0xFFFFFFFFull);  // LBO field
    int it = 0, g = 0, st_i = 0, n_item = 0;
    uint32_t st_ph = 0;
    long long w_split = 0, w_tempty = 0;
    SQ_FOR_ITEMS(, ++n_item) {
      const TcChunk ck = p.chunk[item / p.ntiles];
      const int iters = ck.tap_count * ck.kc_count;
      const int owner = n_item & 1;             // drain group of this item
      for (int i0 = 0; i0 < iters; i0 += G, ++g) {
        const int buf = g & 1;
        SQ_TIMED_WAIT(w_tempty, &tempty[buf], (((uint32_t)g >> 1) & 1u) ^ 1u);   // buffer drained
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + (uint32_t)(buf * p.N);
        const int i1 = (i0 + G < iters) ? (i0 + G) : iters;
        for (int i = i0; i < i1; ++i, ++it) {
          const int s = st_i;
          const uint32_t ph = st_ph;
          if (++st_i == S) { st_i = 0; st_ph ^= 1u; }
          SQ_TIMED_WAIT(w_split, &split[s], ph);
          tc_fence_after();
          // B descriptor low words (start address >> 4 | LBO), +2 per 32-byte K step;
          // A operand: TMEM slot s = 2*KC columns [hi | lo], 8 columns per K step
          const uint32_t b_hi =
              desc_lo0 | ((smem_base + (uint32_t)(s * STAGE_BYTES) + (uint32_t)A_BYTES) >> 4);
          const uint32_t b_lo = b_hi + (uint32_t)(B_BYTES >> 4);
          const uint32_t a_hi = tmem_u + (uint32_t)(2 * p.N + s * 2 * KC);
          const uint32_t a_lo = a_hi + KC;
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < KC / 8; ++j) {
              const uint64_t dbh = desc_hi | (uint64_t)(b_hi + 2 * j);
              const uint64_t dbl = desc_hi | (uint64_t)(b_lo + 2 * j);
              umma_tf32_ts(d_tmem, a_lo + 8 * j, dbh, idesc, (i != i0 || j != 0) ? 1u : 0u);
              umma_tf32_ts(d_tmem, a_hi + 8 * j, dbl, idesc, 1u);
              umma_tf32_ts(d_tmem, a_hi + 8 * j, dbh, idesc, 1u);
            }
            umma_commit(&empty[s]);               // frees the smem stage once the MMAs read it
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(&tfull[owner * 2 + buf]);   // segment complete -> its drain group
        __syncwarp();
      }
    }
    if (p.dbg && lane == 0) {
      p.dbg[blockIdx.x * 12 + 1] = w_split;
      p.dbg[blockIdx.x * 12 + 2] = w_tempty;
    }
   }   // warps 2-3 of warpgroup 0 are spare: straight to the teardown barrier
  } else if (warp < 8) {
    // ================================ operand splitter ====================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    const int t = threadIdx.x & 127;   // 0..127
    int it = 0, st_i = 0;
    uint32_t st_ph = 0;
    long long w_full = 0;
    SQ_FOR_ITEMS() {
      const TcChunk ck = p.chunk[item / p.ntiles];
      const int iters = ck.tap_count * ck.kc_count;
      for (int i = 0; i < iters; ++i, ++it) {
        const int s = st_i;
        const uint32_t ph = st_ph;
        if (++st_i == S) { st_i = 0; st_ph ^= 1u; }
        SQ_TIMED_WAIT(w_full, &full[s], ph);
        // row t of the raw tile (KC*4 bytes, swizzled 16-byte chunks) -> registers ->
        // a_hi / a_lo -> TMEM slot s, lane t (this warp owns lanes 32*(warp%4)..+31)
        if (KC == 32 && GATHER) {
          // gather mode: row t of A = the 27 taps (dy, dx, c) of conv pixel t, read from the
          // patch rows; taps outside the image (SAME padding), taps 27..31 and rows past the
          // tile are zero
          const uint32_t patch = smem_b + (uint32_t)(s * STAGE_BYTES);
          int tile = item % p.ntiles;
          const int tw = tile % p.tiles_w;
          tile /= p.tiles_w;
          const int h0 = (tile % p.tiles_h) * p.ct_h, w0 = tw * p.ct_w;
          const int img = tile / p.tiles_h;
          const int r_h = t / p.ct_w, r_w = t - r_h * p.ct_w;
          const bool live = r_h < p.ct_h;
          const int iy0 = (h0 + r_h) * p.g_stride - p.g_pad_t;      // input row of tap dy = 0
          const int ix0 = (w0 + r_w) * p.g_stride - p.g_pad_l;      // input column of tap dx = 0
          // global element index of (row iy0, tile's first patch column): its low 2 bits are the
          // offset the producer's 16-byte alignment shifted this patch row by
          const int g0 = ((img * p.g_H + iy0) * p.g_W + (w0 * p.g_stride - p.g_pad_l)) * 3;
          uint32_t prow[3];
          bool rok[3], cok[3];
#pragma unroll
          for (int d = 0; d < 3; ++d) {
            const int g = g0 + d * p.g_W * 3;
            prow[d] = patch + 4u * (uint32_t)(live ? (r_h * p.g_stride + d) * GATHER_PITCH + (g & 3) +
                                                        r_w * p.g_stride * 3
                                                  : 0);
            rok[d] = live && (iy0 + d) >= 0 && (iy0 + d) < p.g_H;
            cok[d] = (ix0 + d) >= 0 && (ix0 + d) < p.g_W;
          }
          const uint32_t a_slot = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) +
                                  (uint32_t)(2 * p.N + s * 2 * KC);
#pragma unroll
          for (int hblk = 0; hblk < 2; ++hblk) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const int k = hblk * 16 + e;
              float v = 0.f;
              if (k < 27) {
                v = lds32(prow[k / 9] + 4u * (uint32_t)(k % 9));
                if (!(rok[k / 9] && cok[(k % 9) / 3])) v = 0.f;
              }
              const float h = rn_tf32(v);
              hi[e] = __float_as_uint(h);
              lo[e] = __float_as_uint(v - h);
            }
            tmem_st16(a_slot + (uint32_t)(hblk * 16), hi);
            tmem_st16(a_slot + (uint32_t)(KC + hblk * 16), lo);
          }
          tmem_wait_st();
          tc_fence_before();
          mbar_arrive(&split[s]);
          continue;
        }
        const uint32_t arow = smem_b + (uint32_t)(s * STAGE_BYTES + t * (KC * 4));
        const int sw = (KC == 32) ? (t & 7) : ((t >> 1) & 3);
        const uint32_t a_slot = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) +
                                (uint32_t)(2 * p.N + s * 2 * KC);
#pragma unroll
        for (int hblk = 0; hblk < KC / 16; ++hblk) {       // 16 columns at a time
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int chunk = hblk * 4 + k;
            const float4 v = lds128(arow + (uint32_t)((chunk ^ sw) << 4));
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              // a = h + l exactly (h: 11-bit RN of a, l = a - h fits fp32); the tensor core
              // reads the top 19 bits of l, i.e. |l| * 2^-10 <= 2^-21 |a| is dropped
              const float h = rn_tf32(vv[e]);
              hi[k * 4 + e] = __float_as_uint(h);
              lo[k * 4 + e] = __float_as_uint(vv[e] - h);
            }
          }
          tmem_st16(a_slot + (uint32_t)(hblk * 16), hi);
          tmem_st16(a_slot + (uint32_t)(KC + hblk * 16), lo);
        }
        tmem_wait_st();
        tc_fence_before();             // order the TMEM writes before the barrier hand-off
        mbar_arrive(&split[s]);
      }
    }
    if (p.dbg && t == 0) p.dbg[blockIdx.x * 12 + 3] = w_full;
  } else {
    // ============================ segment drain + epilogue ================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 192;");
    // two drain groups (warps 8-11 and 12-15) take alternate items
    const int dgroup = (warp >= 12) ? 1 : 0;
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;                 // accumulator row = pixel within the tile
    const int tt = threadIdx.x - 256 - 128 * dgroup;   // 0..127 within the drain group
    float acc[MAX_N];
    int g = 0;
    long long w_tfull = 0, c_epi = 0, c_stw = 0, c_par = 0;
    int n_item = 0, n_own = 0, n_store = 0;
    uint32_t use0 = 0u, use1 = 0u;               // own segments seen per TMEM buffer
    SQ_FOR_ITEMS(, ++n_item) {
      const TcChunk ck = p.chunk[item / p.ntiles];
      const int iters = ck.tap_count * ck.kc_count;
      if ((n_item & 1) != dgroup) {
        g += (iters + G - 1) / G;                // segments of an item the other group drains
        continue;
      }
      int tile = item % p.ntiles;
      const int tw = tile % p.tiles_w;
      tile /= p.tiles_w;
      const int h0 = (tile % p.tiles_h) * p.ct_h, w0 = tw * p.ct_w;
      const int img = tile / p.tiles_h;
      const int ncols = (ck.ch_count + 15) & ~15;
      // stage this item's bias / scale / shift in smem (one element per drain thread); the
      // named barrier also orders it against the previous item's epilogue reads.
      const uint32_t par = par_b + 4u * (uint32_t)((dgroup * 2 + (n_own & 1)) * 3 * MAX_N);
      const long long tpar0 = p.dbg ? clock64() : 0;
      {
        const bool in = tt < ck.ch_count;
        sts32(par + 4u * (uint32_t)tt, (in && p.bias) ? __ldg(p.bias + ck.bias_base + tt) : 0.f);
        sts32(par + 4u * (uint32_t)(MAX_N + tt),
              (in && p.scale) ? __ldg(p.scale + ck.bias_base + tt) : 1.f);
        sts32(par + 4u * (uint32_t)(2 * MAX_N + tt),
              (in && p.scale) ? __ldg(p.shift + ck.bias_base + tt) : 0.f);
        asm volatile("bar.sync %0, 128;" ::"r"(1 + dgroup) : "memory");
      }
      if (p.dbg) c_par += clock64() - tpar0;
      ++n_own;
      for (int i0 = 0; i0 < iters; i0 += G, ++g) {
        const int buf = g & 1;
        SQ_TIMED_WAIT(w_tfull, &tfull[dgroup * 2 + buf], (buf ? use1 : use0) & 1u);
        if (buf) ++use1; else ++use0;
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.N);
        // The tensor core truncates when it adds into its fp32 accumulator: a segment of m chained
        // MMAs comes out short by ~bias_comp * m relative (measured, tests/debug_accuracy.py);
        // scale the segment sum back while adding it (one FFMA instead of the FADD).
        const int seg_st = (iters - i0) < G ? (iters - i0) : G;
        const float seg_gain = 1.f + p.bias_comp * (float)(3 * (KC / 8) * seg_st);
#pragma unroll
        for (int c0 = 0; c0 < MAX_N; c0 += 16) {
          if (c0 < ncols) {                      // warp-uniform
            uint32_t v0[16];
            tmem_ld16_nowait(trow + (uint32_t)c0, v0);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 16; ++e)
              acc[c0 + e] = fmaf(__uint_as_float(v0[e]), seg_gain, i0 == 0 ? 0.f : acc[c0 + e]);
          }
        }
        tc_fence_before();
        mbar_arrive(&tempty[buf]);               // buffer may be overwritten by segment g+2
      }
      // ---- epilogue: bias [, affine], relu, 128-bit stores of this pixel's channel run ----
      const long long t_epi = p.dbg ? clock64() : 0;
      const int r_h = r / p.ct_w, r_w = r - r_h * p.ct_w;
      const int oh = h0 + r_h, ow = w0 + r_w;
      const bool pix_ok = (r_h < p.ct_h) && oh < p.Ho && ow < p.Wo;
      if (p.tma_store) {
        // TMEM-drained sums -> (+bias [*scale+shift], relu) -> swizzled smem tiles -> TMA
        // stores.  The TMA unit writes whole 128-byte lines asynchronously and clips ragged
        // tiles / the channel tail; the drain warps never wait on global memory.  Each warp
        // owns tile rows 2q, 2q+1 (its 32 TMEM lanes) and stores them itself: no CTA-level
        // barrier, only __syncwarp.  Ring of two 4 KB tiles per warp.
        const bool affine = p.scale != nullptr;
        const float lo_clip = p.relu ? 0.f : -CUDART_INF_F;
#pragma unroll
        for (int jg = 0; jg < MAX_N / 32; ++jg) {
          if (jg * 32 < ck.ch_count) {                  // warp-uniform
            if (lane == 0) {
              const long long t0 = p.dbg ? clock64() : 0;
              if (p.store_ring == 2) tma_store_wait_read_le1();   // tile used 2 stores ago is free
              else tma_store_wait_read_all();
              if (p.dbg) c_stw += clock64() - t0;
            }
            __syncwarp();
            const uint32_t tile_w = out_b + (uint32_t)((dgroup * 4 + q) * (4096 * p.store_ring) +
                                                       (p.store_ring == 2 ? (n_store & 1) * 4096 : 0));
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const int c = jg * 32 + k * 4;
              const float4 b0 = lds128(par + 4u * (uint32_t)c);
              float o[4] = {acc[c] + b0.x, acc[c + 1] + b0.y, acc[c + 2] + b0.z,
                            acc[c + 3] + b0.w};
              if (affine) {
                const float4 s0 = lds128(par + 4u * (uint32_t)(MAX_N + c));
                const float4 h0v = lds128(par + 4u * (uint32_t)(2 * MAX_N + c));
                o[0] = o[0] * s0.x + h0v.x; o[1] = o[1] * s0.y + h0v.y;
                o[2] = o[2] * s0.z + h0v.z; o[3] = o[3] * s0.w + h0v.w;
              }
              float4 v;
              v.x = fmaxf(o[0], lo_clip); v.y = fmaxf(o[1], lo_clip);
              v.z = fmaxf(o[2], lo_clip); v.w = fmaxf(o[3], lo_clip);
              sts128(tile_w + (uint32_t)(lane * 128 + ((k ^ (lane & 7)) << 4)), v);
            }
            fence_async_proxy();
            __syncwarp();
            if (lane == 0)
              tma_store_4d(tile_w, &p.tmY, ck.y_coff + jg * 32, w0 + q * p.sq_w, h0 + q * p.sq_h, img);
            ++n_store;
          }
        }
      } else if (pix_ok) {
        float* yrow =
            p.y + (((size_t)img * p.Ho + oh) * p.Wo + ow) * (size_t)p.y_cstride + ck.y_coff;
        // 256-bit stores: each thread writes whole 32-byte sectors of its pixel's channel run.
        // Branch-free per element: parameters come from smem (padded with bias 0 / scale 1).
        const bool wide = ((p.y_cstride | ck.y_coff | ck.ch_count) & 7) == 0;
        const bool affine = p.scale != nullptr;
        const float lo_clip = p.relu ? 0.f : -CUDART_INF_F;
#pragma unroll
        for (int c = 0; c < MAX_N; c += 8) {
          if (c < ck.ch_count) {
            float o[8];
            const float4 b0 = lds128(par + 4u * (uint32_t)c);
            const float4 b1 = lds128(par + 4u * (uint32_t)(c + 4));
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = acc[c + e] + bb[e];
            if (affine) {
              const float4 s0 = lds128(par + 4u * (uint32_t)(MAX_N + c));
              const float4 s1 = lds128(par + 4u * (uint32_t)(MAX_N + c + 4));
              const float4 h0v = lds128(par + 4u * (uint32_t)(2 * MAX_N + c));
              const float4 h1v = lds128(par + 4u * (uint32_t)(2 * MAX_N + c + 4));
              const float ss[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
              const float hh[8] = {h0v.x, h0v.y, h0v.z, h0v.w, h1v.x, h1v.y, h1v.z, h1v.w};
#pragma unroll
              for (int e = 0; e < 8; ++e) o[e] = o[e] * ss[e] + hh[e];
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], lo_clip);
            if (wide) {
              asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(yrow + c),
                           "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]), "f"(o[4]), "f"(o[5]),
                           "f"(o[6]), "f"(o[7])
                           : "memory");
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (c + e < ck.ch_count) yrow[c + e] = o[e];
            }
          }
        }
      }
      if (p.dbg) c_epi += clock64() - t_epi;
    }
    if (p.tma_store && lane == 0) tma_store_wait_all();
    if (p.dbg && threadIdx.x == 256) {   // group 0 only
      p.dbg[blockIdx.x * 12 + 4] = w_tfull;
      p.dbg[blockIdx.x * 12 + 7] = c_epi;
      p.dbg[blockIdx.x * 12 + 8] = c_stw;
      p.dbg[blockIdx.x * 12 + 10] = c_par;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// Split-K reduction: y[p][c] = act( (bias[c] + sum_s part[p][s*pitch + c]) [*scale + shift] ).
// Deterministic (fixed summation order), 128-bit loads/stores; the partials are L2-resident.
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ part, float* __restrict__ y,
                     const float* __restrict__ bias, const float* __restrict__ scale,
                     const float* __restrict__ shift, long long npix, int cout, int pitch,
                     int ksplit, int y_cstride, int y_coff, int relu) {
  const int c4n = cout / 4;
  const long long total = npix * c4n;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % c4n) * 4;
    const long long px = idx / c4n;
    float4 a = bias ? *reinterpret_cast<const float4*>(bias + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float* src = part + px * (long long)(ksplit * pitch) + c;
    for (int s2 = 0; s2 < ksplit; ++s2) {
      const float4 v = *reinterpret_cast<const float4*>(src + s2 * pitch);
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    if (scale) {
      const float4 sc = *reinterpret_cast<const float4*>(scale + c);
      const float4 sh = *reinterpret_cast<const float4*>(shift + c);
      a.x = a.x * sc.x + sh.x; a.y = a.y * sc.y + sh.y;
      a.z = a.z * sc.z + sh.z; a.w = a.w * sc.w + sh.w;
    }
    if (relu) {
      a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f);
    }
    *reinterpret_cast<float4*>(y + px * y_cstride + y_coff + c) = a;
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

struct ConvGroup {        // one conv reading the shared input; >= 1 chunks
  int ksize, Cout, y_coff, bias_base;
  int tap_begin = 0, tap_count = -1;   // tap sub-range (split-K); -1 = all ksize*ksize taps
  int kc_begin = 0, kc_count = -1;     // input-channel chunk sub-range (split-K); -1 = all Cin / KC
};

struct TcImpl {
  TcParams prm;
  int KC = 32;
  int Cin = 0;
  size_t smem_bytes = 0;
  dim3 grid;
  float* d_w = nullptr;        // packed weights: hi rows then lo rows, [rows][KC]
  float* d_bias = nullptr;     // concatenated per-group bias (or null)
  float* d_scale = nullptr;
  float* d_shift = nullptr;
  int rows_half = 0;
  int bias_total = 0;
  std::vector<ConvGroup> groups;
  std::vector<TcChunk> chunks;
  // split-K: the kernel writes `ksplit` partial sums into d_scratch [pixels][ksplit*pitch];
  // splitk_reduce_kernel adds them (+bias [,affine], relu) into the real output
  int ksplit = 1, pitch = 0, relu_final = 0, cout = 0, y_cstride_final = 0, y_coff_final = 0;
  long long npix = 0;
  float* d_scratch = nullptr;
  float* y_final = nullptr;
  int* d_sched = nullptr;      // static LPT schedule (see TcParams::sched)
  // gather mode: the input address is baked into the 1-D tensor map; the engine feeds the first
  // layer from several buffers (pipelined inputs), so maps are cached per address
  long long x_floats = 0;
  mutable std::vector<std::pair<const float*, CUtensorMap>> xmaps;
};

static inline float host_rn_tf32(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

static int encode_act_map(CUtensorMap* map, const float* x, int B, int H, int W, int C, int KC,
                          int box_w = TILE_W, int box_h = TILE_H) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(SQDET_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
  cuuint32_t box[4] = {(cuuint32_t)KC, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(x), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   KC == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[96];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled(activation) failed: CUresult %d", (int)r);
    return fail(SQDET_ERR_CUDA, buf);
  }
  return SQDET_OK;
}

static int encode_w_map(CUtensorMap* map, const float* w, int rows, int KC, int N) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(SQDET_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)KC, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)KC * 4};
  cuuint32_t box[2] = {(cuuint32_t)KC, (cuuint32_t)N};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   KC == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[96];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled(weights) failed: CUresult %d", (int)r);
    return fail(SQDET_ERR_CUDA, buf);
  }
  return SQDET_OK;
}

// Common planner: `groups` convs (same ksize rules as the fire pair) over one input.
// First-layer (gather) mode: the conv really is `ks x ks` over a 3-channel image with this
// stride / padding; plan_common is then called on the conv OUTPUT grid with a fake 1x1 group.
struct GatherSpec {
  int B_in, H_in, W_in, stride, pad_t, pad_l;
};

static int encode_flat_map(CUtensorMap* map, const float* x, long long n, int box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(SQDET_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[1] = {(cuuint64_t)n};
  cuuint64_t strides[1] = {0};
  cuuint32_t bx[1] = {(cuuint32_t)box};
  cuuint32_t estr[1] = {1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1, const_cast<float*>(x), dims, strides, bx,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[96];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled(flat input) failed: CUresult %d", (int)r);
    return fail(SQDET_ERR_CUDA, buf);
  }
  return SQDET_OK;
}

static int plan_common(TcImpl* im, int B, int H, int W, int Cin, const std::vector<ConvGroup>& groups,
                       int relu, bool has_affine, int y_cstride, const float* x_dev, float* y_dev,
                       const GatherSpec* gs = nullptr) {
  // A launch made only of 1x1 convs has no spatial structure: walk the B*H*W pixels as one flat
  // row in tiles of 128 consecutive pixels (no ragged image-edge tiles; e.g. 22x76x20 is 262
  // tiles instead of 300, which is two waves of 148 CTAs instead of three).
  bool flat = !gs;
  for (auto& g : groups) flat = flat && g.ksize == 1;
  if (flat) {
    W = B * H * W;
    H = 1;
    B = 1;
  }
  im->Cin = Cin;
  im->KC = (Cin % 32 == 0) ? 32 : 16;
  const int KC = im->KC;
  im->groups = groups;
  // uniform N over all chunks
  int maxc = 0;
  for (auto& g : groups) maxc = g.Cout > maxc ? g.Cout : maxc;
  int N = 0;
  {
    const int nsplit = (maxc + MAX_N - 1) / MAX_N;
    N = ((maxc + nsplit - 1) / nsplit + 15) / 16 * 16;
  }
  TcParams& P = im->prm;
  memset(&P, 0, sizeof P);
  im->chunks.clear();
  int row = 0;
  const int kch = Cin / KC;
  for (auto& g : groups) {
    for (int cb = 0; cb < g.Cout; cb += N) {
      TcChunk c;
      c.ksize = g.ksize;
      c.pad = (g.ksize - 1) / 2;
      c.w_row_base = row;
      c.ch_base = cb;
      c.ch_count = (g.Cout - cb) < N ? (g.Cout - cb) : N;
      c.y_coff = g.y_coff + cb;
      c.bias_base = g.bias_base + cb;
      c.tap_begin = g.tap_begin;
      c.tap_count = g.tap_count < 0 ? g.ksize * g.ksize : g.tap_count;
      c.kc_begin = g.kc_begin;
      c.kc_count = g.kc_count < 0 ? kch : g.kc_count;
      row += c.tap_count * c.kc_count * N;
      im->chunks.push_back(c);
    }
  }
  if ((int)im->chunks.size() > MAX_CHUNKS) return 0;   // not taken by this path
  im->rows_half = row;
  im->bias_total = 0;
  for (auto& g : groups) im->bias_total = (g.bias_base + g.Cout) > im->bias_total ? (g.bias_base + g.Cout) : im->bias_total;
  P.B = B; P.Ho = H; P.Wo = W;                      // stride-1 SAME: output grid == input grid
  P.ct_h = TILE_H; P.ct_w = TILE_W;
  P.tiles_h = (H + TILE_H - 1) / TILE_H;
  P.tiles_w = (W + TILE_W - 1) / TILE_W;
  P.sq_w = 0; P.sq_h = 2;                           // drain warp q stores tile rows 2q, 2q+1
  if (flat) {
    P.ct_h = 1; P.ct_w = TILE_M;
    P.tiles_h = 1; P.tiles_w = (W + TILE_M - 1) / TILE_M;
    P.sq_w = 32; P.sq_h = 0;
  }
  // TMA-store epilogue: needs every chunk to be a whole number of 32-channel groups unless it
  // ends at the tensor's last channel (where the TMA unit clips the tail).
  bool store_ok = (y_cstride % 4 == 0);
  for (auto& c : im->chunks)
    if ((c.ch_count % 32) != 0 && (c.y_coff + c.ch_count != y_cstride)) store_ok = false;
  for (auto& c : im->chunks)
    if (c.y_coff % 4 != 0) store_ok = false;
  if (!store_ok && !flat && !gs) {
    // Direct-store epilogue: any ct_h x ct_w <= 128 tile works, so pick the shape with the fewest
    // rounds of the persistent grid (ConvDet head on 22x76x20: 8x16 tiles = 900 split-K items =
    // 7 rounds on 148 SMs; 11x11 tiles = 840 items = 6 rounds), then the fewest tiles.
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long nch = (long long)im->chunks.size();
    auto rounds_of = [&](long long tiles) { return (tiles * nch + sms - 1) / sms; };
    long long best_tiles = (long long)B * P.tiles_h * P.tiles_w;
    long long best_rounds = rounds_of(best_tiles);
    for (int th = 1; th <= 32; ++th) {
      int twd = TILE_M / th;
      if (twd > 128) twd = 128;
      if (twd < 4) break;
      const long long tiles = (long long)B * ((H + th - 1) / th) * ((W + twd - 1) / twd);
      const long long rounds = rounds_of(tiles);
      if (rounds < best_rounds || (rounds == best_rounds && tiles < best_tiles * 9 / 10)) {
        best_rounds = rounds; best_tiles = tiles;
        P.ct_h = th; P.ct_w = twd;
        P.tiles_h = (H + th - 1) / th; P.tiles_w = (W + twd - 1) / twd;
      }
    }
  }
  P.kch = kch;
  P.N = N;

  // 36 chained MMAs per accumulation segment (3 MMAs per 8-wide K step).  Measured relative
  // error of one conv: 24 -> 4e-7, 48 -> 7e-7, 96 -> 1.3e-6 (fp32 SIMT accumulation: 1e-6 ..
  // 2e-6); 48 is 5% faster end to end than 24 but the truncation bias is systematic, and at
  // 48 the 50-layer ResNet body lands one box coordinate 8e-3 px from the fp32 reference
  // (the test bar is ~6e-3): 36 keeps the margin.  SQDET_TC_SEG overrides it.
  static const int env_seg = env_int("SQDET_TC_SEG", 0);
  P.seg_stages = env_seg > 0 ? env_seg : (KC == 32) ? 3 : 6;
  P.ntiles = B * P.tiles_h * P.tiles_w;
  P.y_cstride = y_cstride;
  P.relu = relu;
  P.lo_row_offset = row;
  P.nchunks = (int)im->chunks.size();
  for (int i = 0; i < P.nchunks; ++i) P.chunk[i] = im->chunks[i];
  const size_t stage = (size_t)TILE_M * KC * 4 + (size_t)2 * N * KC * 4;
  // Pipeline depth: as many stages as fit one CTA per SM (512 threads x 128 registers) after the
  // TMA-store staging; a ring of one staging tile per drain warp instead of two when that buys a
  // fourth stage.
  auto overhead_for = [&](int ring) {
    return (size_t)(1024 /*alignment*/ + 512 /*barriers*/ + 4 * 3 * MAX_N * 4 /*epilogue params*/ +
                    1024 + 8 * 4096 * ring /*store staging*/);
  };
  const size_t budget = 227 * 1024;
  int ring = 2;
  {
    const int s2 = (int)((budget - overhead_for(2)) / stage), s1 = (int)((budget - overhead_for(1)) / stage);
    if (s2 < 4 && s1 > s2) ring = 1;
  }
  P.store_ring = ring;
  const size_t overhead = overhead_for(ring);
  int stages = (int)((budget - overhead) / stage);
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  // TMEM: two accumulator buffers (2N columns) + one [a_hi | a_lo] slot (2*KC columns) per stage
  while (stages > 2 && 2 * N + stages * 2 * KC > 512) --stages;
  if (stages < 2 || 2 * N + stages * 2 * KC > 512) return 0;
  P.stages = stages;
  {
    int cols = 32;
    while (cols < 2 * N + stages * 2 * KC) cols <<= 1;
    P.tmem_cols = cols;
  }
  static const float env_comp = env_float("SQDET_TC_BIAS_COMP", 1.4e-8f);
  P.bias_comp = env_comp;
  im->smem_bytes = stages * stage + overhead;
  {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long items = (long long)P.ntiles * P.nchunks;
    const long long nctas = items < sms ? items : sms;
    im->grid = dim3((unsigned)nctas);
    // Static longest-processing-time-first schedule when chunks differ in cost (a fire expand
    // pair: 1x1 items of kch stages, 3x3 items of 9*kch): round-robin leaves e.g. 12 of 148 CTAs
    // with 7 expensive items against 6 (207 vs 182 stages on fire10); LPT hands those CTAs
    // fewer cheap items instead.
    bool differ = false;
    for (auto& c : im->chunks)
      if (c.tap_count * c.kc_count != im->chunks[0].tap_count * im->chunks[0].kc_count) differ = true;
    // (only when a CTA gets few items: with dozens per CTA round-robin is already balanced, and
    // keeping a tile's 1x1 and 3x3 items adjacent in time is better for L2 - measured on fire2/3)
    if (differ && items > nctas && items < 24 * nctas) {
      std::vector<int> order(im->chunks.size());
      for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
      auto cost_of = [&](int c) { return 2 * im->chunks[c].tap_count * im->chunks[c].kc_count + 3; };   // + epilogue
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost_of(a) > cost_of(b); });
      typedef std::pair<long long, int> Bin;     // (load, CTA id): least loaded first
      std::priority_queue<Bin, std::vector<Bin>, std::greater<Bin>> heap;
      for (int b = 0; b < (int)nctas; ++b) heap.push(Bin(0, b));
      std::vector<std::vector<int>> lists((size_t)nctas);
      for (int c : order)
        for (int t = 0; t < P.ntiles; ++t) {
          Bin b = heap.top();
          heap.pop();
          lists[(size_t)b.second].push_back(c * P.ntiles + t);
          b.first += cost_of(c);
          heap.push(b);
        }
      std::vector<int> sched((size_t)nctas + 1);
      int pos = (int)nctas + 1;
      for (int b = 0; b < (int)nctas; ++b) {
        sched[(size_t)b] = pos;
        pos += (int)lists[(size_t)b].size();
      }
      sched[(size_t)nctas] = pos;
      for (auto& l : lists) sched.insert(sched.end(), l.begin(), l.end());
      SQ_CUDA(cudaMalloc(&im->d_sched, sizeof(int) * sched.size()));
      SQ_CUDA(cudaMemcpy(im->d_sched, sched.data(), sizeof(int) * sched.size(), cudaMemcpyHostToDevice));
      P.sched = im->d_sched;
    }
  }
  P.y = y_dev;
  SQ_CUDA(cudaMalloc(&im->d_w, sizeof(float) * (size_t)row * 2 * KC));
  SQ_CUDA(cudaMemset(im->d_w, 0, sizeof(float) * (size_t)row * 2 * KC));
  SQ_CUDA(cudaMalloc(&im->d_bias, sizeof(float) * im->bias_total));
  SQ_CUDA(cudaMemset(im->d_bias, 0, sizeof(float) * im->bias_total));
  P.bias = im->d_bias;
  if (has_affine) {
    SQ_CUDA(cudaMalloc(&im->d_scale, sizeof(float) * im->bias_total));
    SQ_CUDA(cudaMalloc(&im->d_shift, sizeof(float) * im->bias_total));
    P.scale = im->d_scale;
    P.shift = im->d_shift;
  }
  int rc = 0;
  if (gs) {
    P.gather = 1;
    P.g_H = gs->H_in; P.g_W = gs->W_in; P.g_stride = gs->stride;
    P.g_pad_t = gs->pad_t; P.g_pad_l = gs->pad_l;
    P.g_ph = (P.ct_h - 1) * gs->stride + 3;
    // patch columns * 3 floats, + up to 3 floats of alignment shift, rounded to 16 bytes
    P.g_box = (((P.ct_w - 1) * gs->stride + 3) * 3 + 3 + 3) / 4 * 4;
    if ((long long)gs->B_in * gs->H_in * gs->W_in * 3 + 4096 >= (1LL << 31)) return 0;
    if (P.g_box > GATHER_PITCH || (size_t)P.g_ph * GATHER_PITCH * 4 > (size_t)TILE_M * KC * 4)
      return 0;                                       // patch must fit the stage's A region
    im->x_floats = (long long)gs->B_in * gs->H_in * gs->W_in * 3;
    rc = encode_flat_map(&P.tmX, x_dev, im->x_floats, P.g_box);
    if (rc) return rc;
    im->xmaps.emplace_back(x_dev, P.tmX);
  } else {
    rc = encode_act_map(&P.tmA, x_dev, B, H, W, Cin, KC, P.ct_w, P.ct_h);
    if (rc) return rc;
  }
  if (store_ok) {
    rc = flat ? encode_act_map(&P.tmY, y_dev, B, H, W, y_cstride, 32, 32, 1)
              : encode_act_map(&P.tmY, y_dev, B, H, W, y_cstride, 32, TILE_W, 2);   // per-warp rows
    if (rc) return rc;
  }
  P.tma_store = store_ok ? 1 : 0;
  rc = encode_w_map(&P.tmW, im->d_w, row * 2, KC, N);
  if (rc) return rc;
  // opt in to the full 227 KB once per DEVICE for every instantiation (the attribute is per
  // function and per device context, not per launch, so it must cover the largest plan)
  static unsigned long long attr_devs = 0ull;
  int attr_dev = 0;
  SQ_CUDA(cudaGetDevice(&attr_dev));
  if (attr_dev >= 64 || !((attr_devs >> attr_dev) & 1ull)) {
    SQ_CUDA(cudaFuncSetAttribute(conv_tc_kernel<32, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    SQ_CUDA(cudaFuncSetAttribute(conv_tc_kernel<16, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    SQ_CUDA(cudaFuncSetAttribute(conv_tc_kernel<32, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    if (attr_dev < 64) attr_devs |= 1ull << attr_dev;
  }
  return 1;
}

// Pack group `gi` weights (HWIO [k,k,Cin,Cout]) into the [chunk][tap][kchunk][N][KC] hi/lo rows.
static void pack_group(const TcImpl* im, int gi, const float* w_hwio, std::vector<float>& packed) {
  const int KC = im->KC, N = im->prm.N, Cin = im->Cin;
  const ConvGroup& g = im->groups[gi];
  const size_t lo_off = (size_t)im->rows_half * KC;
  // chunks of this group appear in order; find the first
  int ci = 0;
  for (int i = 0; i < gi; ++i) ci += (im->groups[i].Cout + N - 1) / N;
  for (int cb = 0; cb < g.Cout; cb += N, ++ci) {
    const TcChunk& c = im->chunks[ci];
    for (int tl = 0; tl < c.tap_count; ++tl)
      for (int kc = c.kc_begin; kc < c.kc_begin + c.kc_count; ++kc)
        for (int n = 0; n < c.ch_count; ++n) {
          const int tap = c.tap_begin + tl;
          const size_t rowi = (size_t)c.w_row_base + ((size_t)tl * c.kc_count + (kc - c.kc_begin)) * N + n;
          for (int k = 0; k < KC; ++k) {
            const float v = (kc * KC + k < Cin)
                                ? w_hwio[((size_t)tap * Cin + (size_t)kc * KC + k) * g.Cout + cb + n]
                                : 0.f;   // gather mode: K = 27 padded to 32
            const float hi = host_rn_tf32(v);
            packed[rowi * KC + k] = hi;
            packed[lo_off + rowi * KC + k] = host_rn_tf32(v - hi);
          }
        }
  }
}

static int launch_impl(const TcImpl* im, const float* x_dev, float* y_dev, cudaStream_t stream) {
  // the tensor map bakes in the activation address the plan was made for
  (void)x_dev;
  (void)y_dev;
  static const int debug = env_int("SQDET_TC_DEBUG", 0);
  TcParams prm = im->prm;
  if (prm.gather && x_dev) {
    bool found = false;
    for (auto& m : im->xmaps)
      if (m.first == x_dev) { prm.tmX = m.second; found = true; break; }
    if (!found) {
      CUtensorMap m;
      int rc = encode_flat_map(&m, x_dev, im->x_floats, prm.g_box);
      if (rc) return rc;
      if (im->xmaps.size() >= 8) im->xmaps.erase(im->xmaps.begin());
      im->xmaps.emplace_back(x_dev, m);
      prm.tmX = m;
    }
  }
  long long* dbg = nullptr;
  const int nb = (int)im->grid.x;
  if (debug) {
    SQ_CUDA(cudaMalloc(&dbg, sizeof(long long) * 12 * nb));
    SQ_CUDA(cudaMemsetAsync(dbg, 0, sizeof(long long) * 12 * nb, stream));
    prm.dbg = dbg;
  }
  if (prm.gather)
    SQ_CUDA(launch_kernel(conv_tc_kernel<32, true>, im->grid, dim3(NUM_THREADS), im->smem_bytes, stream,
                          prm));
  else if (im->KC == 32)
    SQ_CUDA(launch_kernel(conv_tc_kernel<32, false>, im->grid, dim3(NUM_THREADS), im->smem_bytes, stream,
                          prm));
  else
    SQ_CUDA(launch_kernel(conv_tc_kernel<16, false>, im->grid, dim3(NUM_THREADS), im->smem_bytes, stream,
                          prm));
  SQ_CHECK_LAUNCH("conv_tc_kernel");
  if (im->ksplit > 1) {
    const long long total = im->npix * (im->cout / 4);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    SQ_CUDA(launch_kernel(splitk_reduce_kernel, dim3((unsigned)blocks), dim3(256), 0, stream,
                          (const float*)im->d_scratch, im->y_final, (const float*)im->d_bias,
                          (const float*)im->d_scale, (const float*)im->d_shift, im->npix, im->cout,
                          im->pitch, im->ksplit, im->y_cstride_final, im->y_coff_final, im->relu_final));
    SQ_CHECK_LAUNCH("splitk_reduce_kernel");
  }
  if (debug) {
    std::vector<long long> h((size_t)12 * nb);
    SQ_CUDA(cudaStreamSynchronize(stream));
    SQ_CUDA(cudaMemcpy(h.data(), dbg, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    cudaFree(dbg);
    double a[12] = {0};
    for (int b = 0; b < nb; ++b)
      for (int k = 0; k < 12; ++k) a[k] += (double)h[(size_t)b * 12 + k] / nb;
    fprintf(stderr,
            "[tc] grid %d tile %dx%d ntiles %d%s smem %zu KC %d N %d kch %d chunks %d stages %d seg %d | per-CTA avg cycles: "
            "total %.0f stages %.0f | waits: producer(empty) %.0f mma(split) %.0f mma(tempty) %.0f "
            "splitter(full) %.0f drain(tfull) %.0f | epilogue %.0f (store-wait %.0f, params %.0f)\n",
            nb, prm.ct_h, prm.ct_w, prm.ntiles, prm.sched ? " LPT" : "", im->smem_bytes, im->KC, prm.N, prm.kch, prm.nchunks, prm.stages, prm.seg_stages,
            a[5], a[6], a[0], a[1], a[2], a[3], a[4], a[7], a[8], a[10]);
  }
  return SQDET_OK;
}

static void release_impl(void** impl) {
  if (!*impl) return;
  TcImpl* im = static_cast<TcImpl*>(*impl);
  cudaFree(im->d_w);
  cudaFree(im->d_bias);
  cudaFree(im->d_scale);
  cudaFree(im->d_shift);
  cudaFree(im->d_scratch);
  cudaFree(im->d_sched);
  delete im;
  *impl = nullptr;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
int tc_encode_act_map(CUtensorMap* map, const float* x, int B, int H, int W, int C, int KC,
                      int box_w, int box_h) {
  return encode_act_map(map, x, B, H, W, C, KC, box_w, box_h);
}
int tc_encode_w_map(CUtensorMap* map, const float* w, int rows, int KC, int N) {
  return encode_w_map(map, w, rows, KC, N);
}
int tc_encode_flat_map(CUtensorMap* map, const float* x, long long n, int box) {
  return encode_flat_map(map, x, n, box);
}

bool tc_conv_eligible(int Cin, int Cout, int size, int stride, int padding, int y_cstride,
                      int y_coff) {
  // shapes this path takes: stride-1 SAME, 1x1 or 3x3, Cin a multiple of 16, 16B-aligned stores
  if (stride != 1 || padding != SQDET_PAD_SAME || (size != 1 && size != 3)) return false;
  if (Cin % 16 != 0 || Cin < 16 || (y_cstride % 4) || (y_coff % 4) || (Cout % 4)) return false;
  return true;
}

int tc_conv_plan(TcConvPlan* plan, int B, int H, int W, int Cin, int Cout, int size, int stride,
                 int padding, int relu, bool has_affine, int y_cstride, int y_coff,
                 const float* x_dev, float* y_dev) {
  plan->enabled = false;
  // First layer: 3x3 conv over a 3-channel image (stride 1 or 2, SAME or VALID) -> gather mode
  if (Cin == 3 && size == 3 && (stride == 1 || stride == 2) && (Cout % 4) == 0 &&
      (y_cstride % 4) == 0 && (y_coff % 4) == 0) {
    const Geom gh = tf_geometry(H, size, stride, padding);
    const Geom gw = tf_geometry(W, size, stride, padding);
    if (gh.out <= 0 || gw.out <= 0) return 0;
    TcImpl* im = new TcImpl();
    GatherSpec gs{B, H, W, stride, gh.pad_before, gw.pad_before};
    std::vector<ConvGroup> groups = {{1, Cout, y_coff, 0}};   // one K block of 32 (27 real taps)
    int rc = plan_common(im, B, gh.out, gw.out, 32, groups, relu, has_affine, y_cstride, x_dev,
                         y_dev, &gs);
    if (rc <= 0) {
      void* p = im;
      release_impl(&p);
      return rc;
    }
    im->Cin = 27;          // weight packing: HWIO flattened is already [k = (dy, dx, c)][Cout]
    plan->enabled = true;
    plan->B = B; plan->H = H; plan->W = W; plan->Cin = Cin; plan->Cout = Cout;
    plan->size = size; plan->stride = stride; plan->relu = relu;
    plan->Ho = gh.out; plan->Wo = gw.out; plan->pad_t = gh.pad_before; plan->pad_l = gw.pad_before;
    plan->y_cstride = y_cstride; plan->y_coff = y_coff;
    plan->launches = 1;
    plan->impl = im;
    return 1;
  }
  if (!tc_conv_eligible(Cin, Cout, size, stride, padding, y_cstride, y_coff)) return 0;
  TcImpl* im = new TcImpl();
  // Split-K for 3x3 convs whose item count leaves the last round of the persistent grid mostly
  // idle (SqueezeDet's ConvDet head: 300 items on 148 SMs = 3 rounds for 2.03 rounds of work):
  // three partial convs over the filter rows, then a deterministic reduction.
  int ksplit = 1;
  {
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long ntiles = (long long)B * ((H + TILE_H - 1) / TILE_H) * ((W + TILE_W - 1) / TILE_W);
    const bool few_items = Cout <= MAX_N && ntiles < 4LL * sms && (ntiles % sms) != 0 &&
                           (double)(ntiles % sms) / sms < 0.5;
    if (size == 3 && few_items && Cin >= 96 && (Cout % 4) == 0) ksplit = 3;
  }
  std::vector<ConvGroup> groups;
  int rc;
  if (ksplit == 1) {
    groups = {{size, Cout, y_coff, 0}};
    rc = plan_common(im, B, H, W, Cin, groups, relu, has_affine, y_cstride, x_dev, y_dev);
  } else {
    const int pitch = (Cout + 7) / 8 * 8;
    im->ksplit = ksplit;
    im->pitch = pitch;
    im->relu_final = relu;
    im->cout = Cout;
    im->y_cstride_final = y_cstride;
    im->y_coff_final = y_coff;
    im->npix = (long long)B * H * W;
    im->y_final = y_dev;
    cudaError_t ce = cudaMalloc(&im->d_scratch, sizeof(float) * (size_t)im->npix * ksplit * pitch);
    if (ce != cudaSuccess) {
      delete im;
      return cuda_fail(ce, "cudaMalloc(split-K scratch)");
    }
    const int KCs = (Cin % 32 == 0) ? 32 : 16, kch_all = Cin / KCs;
    for (int s2 = 0; s2 < ksplit; ++s2) {
      ConvGroup g{size, Cout, s2 * pitch, 0};
      if (kch_all % ksplit != 0) {
        g.tap_begin = s2 * size;         // one filter row per partial (reads the input ksplit times)
        g.tap_count = size;
      } else {
        g.kc_begin = s2 * (kch_all / ksplit);   // one input-channel range per partial: every input
        g.kc_count = kch_all / ksplit;          // byte is read once (ConvDet: 329 -> ~130 MB of DRAM reads)
      }
      groups.push_back(g);
    }
    // partials: no bias / affine / relu in the conv epilogue (they are applied by the reduction)
    rc = plan_common(im, B, H, W, Cin, groups, 0, has_affine, ksplit * pitch, x_dev, im->d_scratch);
    if (rc > 0) im->prm.bias = nullptr, im->prm.scale = nullptr, im->prm.shift = nullptr;
  }
  if (rc <= 0) {
    void* p = im;
    release_impl(&p);
    return rc;
  }
  plan->enabled = true;
  plan->B = B; plan->H = H; plan->W = W; plan->Cin = Cin; plan->Cout = Cout;
  plan->size = size; plan->stride = stride; plan->relu = relu; plan->Ho = H; plan->Wo = W;
  plan->y_cstride = y_cstride; plan->y_coff = y_coff;
  plan->launches = im->ksplit > 1 ? 2 : 1;
  plan->impl = im;
  return 1;
}

int tc_fire_plan(TcFirePlan* plan, int B, int H, int W, int S, int E1, int E3, const float* q_dev,
                 float* y_dev) {
  plan->enabled = false;
  if (S % 16 != 0 || S < 16 || (E1 % 4) || (E3 % 4)) return 0;
  TcImpl* im = new TcImpl();
  std::vector<ConvGroup> groups = {{1, E1, 0, 0}, {3, E3, E1, E1}};
  int rc = plan_common(im, B, H, W, S, groups, 1, false, E1 + E3, q_dev, y_dev);
  if (rc <= 0) {
    void* p = im;
    release_impl(&p);
    return rc;
  }
  plan->enabled = true;
  plan->B = B; plan->H = H; plan->W = W; plan->S = S; plan->E1 = E1; plan->E3 = E3;
  plan->impl = im;
  return 1;
}

int tc_conv_pack_weights(TcConvPlan* plan, const float* w_hwio, const float* bias) {
  TcImpl* im = static_cast<TcImpl*>(plan->impl);
  std::vector<float> packed((size_t)im->rows_half * 2 * im->KC, 0.f);
  for (int gi = 0; gi < (int)im->groups.size(); ++gi) pack_group(im, gi, w_hwio, packed);
  SQ_CUDA(cudaMemcpy(im->d_w, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (bias)
    SQ_CUDA(cudaMemcpy(im->d_bias, bias, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int tc_conv_set_affine(TcConvPlan* plan, const float* scale, const float* shift) {
  TcImpl* im = static_cast<TcImpl*>(plan->impl);
  if (!im->d_scale) return fail(SQDET_ERR_STATE, "tc conv planned without an affine epilogue");
  SQ_CUDA(cudaMemcpy(im->d_scale, scale, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_shift, shift, sizeof(float) * plan->Cout, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int tc_fire_pack_weights(TcFirePlan* plan, const float* w_e1, const float* b_e1, const float* w_e3,
                         const float* b_e3) {
  TcImpl* im = static_cast<TcImpl*>(plan->impl);
  std::vector<float> packed((size_t)im->rows_half * 2 * im->KC, 0.f);
  pack_group(im, 0, w_e1, packed);
  pack_group(im, 1, w_e3, packed);
  SQ_CUDA(cudaMemcpy(im->d_w, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_bias, b_e1, sizeof(float) * plan->E1, cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_bias + plan->E1, b_e3, sizeof(float) * plan->E3, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int launch_conv_tc(const TcConvPlan& plan, const float* x_dev, float* y_dev, cudaStream_t stream) {
  return launch_impl(static_cast<const TcImpl*>(plan.impl), x_dev, y_dev, stream);
}

int launch_fire_expand_tc(const TcFirePlan& plan, const float* q_dev, float* y_dev,
                          cudaStream_t stream) {
  return launch_impl(static_cast<const TcImpl*>(plan.impl), q_dev, y_dev, stream);
}

void tc_conv_release(TcConvPlan* plan) {
  release_impl(&plan->impl);
  plan->enabled = false;
}
void tc_fire_release(TcFirePlan* plan) {
  release_impl(&plan->impl);
  plan->enabled = false;
}

int conv2d_tc_oneshot(const float* x_dev, const float* w_hwio_dev, const float* bias_dev,
                      const float* scale_dev, const float* shift_dev, float* y_dev, int B, int H,
                      int W, int Cin, int Cout, int size, int stride, int padding, int relu,
                      int y_cstride, int y_coff, cudaStream_t stream) {
  TcConvPlan plan;
  int rc = tc_conv_plan(&plan, B, H, W, Cin, Cout, size, stride, padding, relu,
                        scale_dev != nullptr, y_cstride, y_coff, x_dev, y_dev);
  if (rc < 0) return rc;
  if (rc == 0) {
    // shape not taken by the tensor-core path (e.g. conv1, Cin = 3): same dispatch as the engine
    ConvArgs a;
    a.x = x_dev; a.w = w_hwio_dev; a.bias = bias_dev; a.scale = scale_dev; a.shift = shift_dev;
    a.y = y_dev; a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.size = size;
    a.stride = stride; a.padding = padding; a.relu = relu; a.y_cstride = y_cstride; a.y_coff = y_coff;
    return launch_conv_simt(a, stream);
  }
  std::vector<float> w((size_t)size * size * Cin * Cout), b(Cout, 0.f), sc, sh;
  SQ_CUDA(cudaMemcpy(w.data(), w_hwio_dev, w.size() * sizeof(float), cudaMemcpyDeviceToHost));
  if (bias_dev) SQ_CUDA(cudaMemcpy(b.data(), bias_dev, Cout * sizeof(float), cudaMemcpyDeviceToHost));
  rc = tc_conv_pack_weights(&plan, w.data(), bias_dev ? b.data() : nullptr);
  if (!rc && scale_dev) {
    sc.resize(Cout); sh.resize(Cout);
    SQ_CUDA(cudaMemcpy(sc.data(), scale_dev, Cout * sizeof(float), cudaMemcpyDeviceToHost));
    SQ_CUDA(cudaMemcpy(sh.data(), shift_dev, Cout * sizeof(float), cudaMemcpyDeviceToHost));
    rc = tc_conv_set_affine(&plan, sc.data(), sh.data());
  }
  if (!rc) rc = launch_conv_tc(plan, x_dev, y_dev, stream);
  cudaError_t ce = cudaStreamSynchronize(stream);
  tc_conv_release(&plan);
  if (rc) return rc;
  if (ce != cudaSuccess) return cuda_fail(ce, "conv2d_tc_oneshot sync");
  return SQDET_OK;
}

}  // namespace sqdet
