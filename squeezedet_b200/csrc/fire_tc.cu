// The fire module as ONE kernel on tcgen05 (SQDET_MATH_TF32X3_TC):
//   squeeze 1x1 + bias + ReLU  ->  expand 1x1 || expand 3x3 + bias + ReLU  ->  channel concat
// Replaces SqueezeDet._fire_layer (src/nets/squeezeDet.py:81-106, squeezeDetPlus.py:81-106; the
// three _conv_layer calls of src/nn_skeleton.py:471-561 and the tf.concat) - the squeeze tensor
// never leaves the SM.
//
// Item = a 16 (h) x 8 (w) tile of output pixels of one image.  Per item:
//   squeeze : the 18 x 10 halo of the tile (SAME padding of the 3x3 expand) as two M tiles of
//             9 halo rows x 10 = 90 pixels each:  Q[90, S] = X[90, Cin] * Ws[Cin, S], the conv_tc.cu
//             pipeline (TMA box {32 ch, 10 w, 9 h} -> operand splitter -> [a_hi | a_lo] in TENSOR
//             MEMORY -> tcgen05.mma .ts form, 3xTF32, segments of 36 chained MMAs summed in fp32
//             registers by the drain warps).
//   Q tile  : the squeeze drain adds the bias, applies ReLU, forces halo pixels OUTSIDE the image to
//             0 (tf pads the post-ReLU squeeze tensor, not relu(bias)), splits q = q_hi + q_lo ONCE
//             and writes both halves to shared memory as [16-byte channel chunk][h 18][w 10][4 floats].
//   expand  : that layout is a K-major SWIZZLE_NONE UMMA operand whose 8-row core matrices are 8
//             consecutive w of one halo row (16 B apart), 8-row groups one halo row apart (SBO = 160 B),
//             K chunks LBO = 2880 B apart - so the A operand of filter tap (dy, dx) is the SAME tile
//             at start address + dy*160 + dx*16 (tools/desc_test.cu checks this on the hardware).
//             The nine taps therefore need no im2col, no re-split and no TMA re-fetch: tcgen05.mma
//             .ss form straight from the Q tile, B = packed hi/lo expand weights, resident in shared
//             memory for the whole launch when they fit (fire2/3: 80 KB), else streamed through a ring.
//             (conv_tc.cu's expand kernel re-fetched and re-split the squeeze tile once per tap: its
//             splitter, not the tensor pipe or HBM, bounded fire2-5.)
//   epilogue: accumulator segments -> fp32 registers (+bias, ReLU) -> swizzled staging -> TMA store
//             of {32 ch, 8 w, 4 h} boxes into the concat tensor.
// Roles (512 threads): warpgroups 0,1 = drains (squeeze drain of M tile g; expand drain of the
//   32-channel groups jg = g mod 2 of EVERY chunk; 176 registers), warps 8-10 and 12-14 = the two
//   operand splitter groups (alternate squeeze stages; only TMEM lanes 0..95 of a squeeze M tile hold
//   pixels, which frees the fourth warp of each warpgroup), warp 11 = TMA producer of both rings,
//   warp 15 = TMEM owner + MMA issuer.
// Order: with two Q buffers the MMA warp issues squeeze(i+1) BEFORE expand(i), so the squeeze drain
//   of the next item overlaps the expand MMAs of this one; with one buffer squeeze(i), expand(i).
// Roofline: HBM-bound for fire2-5 (AI 24-60 FLOP/B, SURVEY.md 8d); algorithmic bytes per pixel =
//   4*(Cin + E1 + E3), the squeeze tensor contributes nothing.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"
#include "fire_tc.cuh"
#include "tc_ptx.cuh"

namespace sqdet {
namespace {

constexpr int FF_THREADS = 512;
constexpr int FF_TH = 16, FF_TW = 8;               // output tile
constexpr int FF_HH = FF_TH + 2, FF_HW = FF_TW + 2;   // halo: 18 x 10
constexpr int FF_QROW = FF_HW * 16;                // bytes between halo rows of one channel chunk
constexpr int FF_QCH = FF_HH * FF_HW * 16;         // bytes between 16-byte channel chunks (2880)
constexpr int FF_MT_H = 9;                         // halo rows per squeeze M tile
constexpr int FF_MT_ROWS = FF_MT_H * FF_HW;        // 90 valid rows of the 128
constexpr int FF_SQ_A = 12288;                     // squeeze stage: A region (90 x 128 B, padded)
constexpr int FF_SEG = 12;                         // K steps (of 8) per accumulation segment = 36 MMAs
constexpr int FF_MAX_S = 64;
constexpr int KCE = 16;                            // K width of an expand weight tile (SWIZZLE_64B rows)
constexpr int FF_MAX_CHUNKS = 8;
constexpr int FF_MAX_RING = 4;
constexpr int FF_PAR_FLOATS = FF_MAX_S + 512;      // bias_sq | bias_e1 ++ bias_e3

struct FireChunk {
  int tile_base;   // first weight tile ([Ne][KCE] hi + lo) of this chunk
  int taps;        // 1 (expand1x1) or 9 (expand3x3)
  int y_coff;      // first output channel of this chunk in the concat tensor
};

struct FireParams {
  CUtensorMap tmX;     // input [B,H,W,Cin], box {32 ch, 10 w, 9 h, 1}, SWIZZLE_128B
  CUtensorMap tmWs;    // squeeze weights [Cin/32][hi S rows | ...][32], box {32, S}
  CUtensorMap tmWe;    // expand weight tiles, rows [tile][Ne][KCE], box {KCE, Ne}
  CUtensorMap tmY;     // output [B,H,W,E1+E3], box {32 ch, 8 w, 4 h, 1}, SWIZZLE_128B
  const float* bias_sq;
  const float* bias_e;     // [E1 + E3]
  int B, H, W, Cin, S, E1, E3;
  int tiles_h, tiles_w, ntiles;
  int Ne;                  // UMMA N of the expand MMAs (channels per chunk)
  int nchunks;
  int nsq, nq, nring;      // squeeze stages, Q buffers, expand-weight stages (resident: all tiles)
  int resident;
  int sq_seg;              // squeeze stages (32 channels each) per accumulation segment: 3, or 4 with sq_on_split
  int sq_on_split;         // 1: the two splitter groups drain the squeeze accumulators (single-segment squeezes,
                           // S = 16): takes 40 % of the work off the drain warpgroups, which bounded fire2/3
  int ntiles_w;            // expand weight tiles in total
  int lo_rows_sq, lo_rows_e;   // rows between the hi and the lo copy in the packed matrices
  int tmem_cols;
  int store_ring;
  float bias_comp;
  // shared-memory map (bytes from the 1024-aligned base)
  int off_q, q_half, q_bytes, off_sq, sq_stage, off_ew, ew_tile, off_out, off_par, off_bar;
  long long* dbg;
  FireChunk chunk[FF_MAX_CHUNKS];
};

// debug-only stall accounting (SQDET_TC_DEBUG=1): 32-bit cycle counters (a launch is < 2 s)
#define FF_WAIT(counter, bar, parity)                       \
  do {                                                      \
    if (p.dbg) {                                            \
      const uint32_t _t0 = (uint32_t)clock();               \
      mbar_wait(bar, parity);                               \
      counter += (uint32_t)clock() - _t0;                   \
    } else {                                                \
      mbar_wait(bar, parity);                               \
    }                                                       \
  } while (0)

// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// non-blocking probe: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

struct RingPos {        // position in a ring of n stages: stage index and mbarrier phase
  int s;
  uint32_t ph;
  __device__ __forceinline__ void next(int n) {
    if (++s == n) { s = 0; ph ^= 1u; }
  }
};

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FF_THREADS, 1)
fire_fused_kernel(const __grid_constant__ FireParams p) {
  extern __shared__ uint8_t smem_dyn[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                             ~uintptr_t(1023));
  const uint32_t smem_b = smem_u32(smem);
  const uint32_t q_b = smem_b + (uint32_t)p.off_q;
  const uint32_t sq_b = smem_b + (uint32_t)p.off_sq;
  const uint32_t ew_b = smem_b + (uint32_t)p.off_ew;
  const uint32_t out_b = smem_b + (uint32_t)p.off_out;
  const uint32_t par_b = smem_b + (uint32_t)p.off_par;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.off_bar);
  uint64_t* sfull = bars;                        // [nsq]  TMA -> splitter
  uint64_t* ssplit = bars + FF_MAX_RING;         // [nsq]  splitter -> MMA
  uint64_t* sempty = bars + 2 * FF_MAX_RING;     // [nsq]  MMA commit -> TMA
  uint64_t* efull = bars + 3 * FF_MAX_RING;      // [nring] TMA -> MMA (streamed expand weights); [0] = resident set
  uint64_t* eempty = bars + 4 * FF_MAX_RING;     // [nring] MMA commit -> TMA
  uint64_t* sqfull = bars + 5 * FF_MAX_RING;     // [2]  MMA commit -> squeeze drain of M tile mt
  uint64_t* sqempty = sqfull + 2;                // [2]  squeeze drain -> MMA
  uint64_t* qfull = sqfull + 4;                  // [2]  drains -> MMA (Q buffer written)
  uint64_t* qempty = sqfull + 6;                 // [2]  MMA commit -> drains (Q buffer read out)
  uint64_t* tfull = sqfull + 8;                  // [2]  MMA commit -> expand drain
  uint64_t* tempty = sqfull + 10;                // [2]  expand drains -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sqfull + 12);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int role = warp >> 2;   // 0,1 drains, 2 splitter A + TMA producer, 3 splitter B + MMA issuer
  const bool ctl = (warp & 3) == 3;                          // fourth warp of a splitter warpgroup
  const int S = p.S, Ne = p.Ne;
  const int kch = p.Cin >> 5;                    // 32-channel K chunks of the squeeze
  const int ksq = S >> 3;                        // K steps of 8 squeeze channels (expand K per tap)
  const int my_items = ((int)p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < FF_MAX_RING; ++s) {
      mbar_init(&sfull[s], 1);
      mbar_init(&ssplit[s], 96);
      mbar_init(&sempty[s], 1);
      mbar_init(&efull[s], 1);
      mbar_init(&eempty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&sqfull[b], 1);
      mbar_init(&sqempty[b], p.sq_on_split ? 96 : 128);
      mbar_init(&qfull[b], p.sq_on_split ? 192 : 256);
      mbar_init(&qempty[b], 1);
      mbar_init(&tfull[b], 1);
      mbar_init(&tempty[b], 256);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (role == 3 && ctl) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // TMEM columns: [0, 2S) squeeze accumulators (M tile 0 | 1), [2S, 2S + 2Ne) expand accumulators
  // (two buffers), then one [a_hi | a_lo] = 64-column A slot per squeeze stage
  const uint32_t col_e = (uint32_t)(2 * S), col_a = (uint32_t)(2 * S + 2 * Ne);

#define FF_TILE_DECODE(item_)                          \
  int tile_ = (item_);                                 \
  const int tw = tile_ % p.tiles_w;                    \
  tile_ /= p.tiles_w;                                  \
  const int th = tile_ % p.tiles_h;                    \
  const int img = tile_ / p.tiles_h;                   \
  const int h0 = th * FF_TH, w0 = tw * FF_TW;

  if (role >= 2) {
   // warpgroups 2 and 3: warps 8-10 / 12-14 = the two splitter groups (only TMEM lanes 0..95 of a
   // squeeze M tile hold pixels, so the fourth warp of each warpgroup is free for a control role)
   asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
   if (ctl) {
    if (role == 2) {
      // ================================ TMA producer ==========================================
      if (lane == 0) {
        RingPos rq{0, 0u}, re{0, 0u};
        const uint32_t bytes = (uint32_t)(FF_MT_ROWS * 128 + 2 * S * 128);
        const uint32_t half = (uint32_t)(Ne * KCE * 4);
        if (p.resident) {
          mbar_expect_tx(&efull[0], (uint32_t)p.ntiles_w * 2u * half);
          for (int t = 0; t < p.ntiles_w; ++t) {
            uint8_t* dst = smem + p.off_ew + (size_t)t * p.ew_tile;
            tma_load_2d(dst, &p.tmWe, &efull[0], 0, t * Ne);
            tma_load_2d(dst + half, &p.tmWe, &efull[0], 0, t * Ne + p.lo_rows_e);
          }
        }
        // One thread feeds BOTH rings without ever blocking on either (mbarrier.test_wait): each
        // ring is FIFO in the MMA warp's consumption order, and a full ring never holds back the other
        // (a blocking producer delayed the next item's squeeze stages behind the weight stream).
        int sq_k = 0, sq_seg0 = 0, sq_mt = 0, sq_kc = 0;       // next squeeze stage
        int ew_k = 0, ew_t = 0;                                // next expand weight tile
        bool sq_left = my_items > 0, ew_left = my_items > 0 && !p.resident;
        int tw = 0, th = 0, img = 0;
        bool decoded = false;
        while (sq_left || ew_left) {
          if (sq_left && mbar_test(&sempty[rq.s], rq.ph ^ 1u)) {
            if (!decoded) {
              int tile_ = (int)blockIdx.x + sq_k * (int)gridDim.x;
              tw = tile_ % p.tiles_w;
              tile_ /= p.tiles_w;
              th = tile_ % p.tiles_h;
              img = tile_ / p.tiles_h;
              decoded = true;
            }
            uint8_t* st = smem + p.off_sq + (size_t)rq.s * p.sq_stage;
            mbar_expect_tx(&sfull[rq.s], bytes);
            tma_load_4d(st, &p.tmX, &sfull[rq.s], sq_kc * 32, tw * FF_TW - 1,
                        th * FF_TH - 1 + FF_MT_H * sq_mt, img);
            tma_load_2d(st + FF_SQ_A, &p.tmWs, &sfull[rq.s], 0, sq_kc * S);
            tma_load_2d(st + FF_SQ_A + S * 128, &p.tmWs, &sfull[rq.s], 0, sq_kc * S + p.lo_rows_sq);
            rq.next(p.nsq);
            // advance (segment of 3 K chunks, M tile, K chunk): the MMA / splitter order
            if (++sq_kc == kch || sq_kc == sq_seg0 + p.sq_seg) {
              if (++sq_mt == 2) {
                sq_mt = 0;
                sq_seg0 += p.sq_seg;
                if (sq_seg0 >= kch) {
                  sq_seg0 = 0;
                  decoded = false;
                  if (++sq_k == my_items) sq_left = false;
                }
              }
              sq_kc = sq_seg0;
            }
          }
          if (ew_left && mbar_test(&eempty[re.s], re.ph ^ 1u)) {
            uint8_t* dst = smem + p.off_ew + (size_t)re.s * p.ew_tile;
            mbar_expect_tx(&efull[re.s], 2u * half);
            tma_load_2d(dst, &p.tmWe, &efull[re.s], 0, ew_t * Ne);
            tma_load_2d(dst + half, &p.tmWe, &efull[re.s], 0, ew_t * Ne + p.lo_rows_e);
            re.next(p.nring);
            if (++ew_t == p.ntiles_w) {
              ew_t = 0;
              if (++ew_k == my_items) ew_left = false;
            }
          }
        }
      }
    } else {
      // ================================ MMA issuer (warp 15) ==================================
      const uint32_t idesc_s = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(S >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
      const uint32_t idesc_e = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(Ne >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      // B descriptors (swizzled K-major tiles), high words; low word = LBO field | address >> 4
      const uint64_t dsw_hi = make_desc<32>(0) & 0xFFFFFFFF00000000ull;
      const uint32_t dsw_lo = (uint32_t)(make_desc<32>(0) & 0xFFFFFFFFull);
      const uint64_t dew_hi = make_desc<KCE>(0) & 0xFFFFFFFF00000000ull;
      const uint32_t dew_lo = (uint32_t)(make_desc<KCE>(0) & 0xFFFFFFFFull);
      // A descriptor of the Q tile: SWIZZLE_NONE, LBO = channel-chunk stride, SBO = halo-row stride
      const uint64_t dq_hi = ((uint64_t)(FF_QROW >> 4) << 32) | (1ull << 46);
      const uint32_t dq_lo = (uint32_t)(FF_QCH >> 4) << 16;
      RingPos rs{0, 0u}, re{0, 0u};
      uint32_t sq_use0 = 0u, sq_use1 = 0u, eg = 0u;
      uint32_t w_split = 0, w_sqempty = 0, w_qfull = 0, w_tempty = 0, w_efull = 0;
      const uint32_t t_begin = (uint32_t)clock();

      auto squeeze = [&]() {
        for (int seg0 = 0; seg0 < kch; seg0 += p.sq_seg)
          for (int mt = 0; mt < 2; ++mt) {
            const uint32_t use = mt ? sq_use1 : sq_use0;
            FF_WAIT(w_sqempty, &sqempty[mt], (use & 1u) ^ 1u);
            if (mt) ++sq_use1; else ++sq_use0;
            tc_fence_after();
            const uint32_t d_tmem = tmem_u + (uint32_t)(mt * S);
            for (int kc = seg0; kc < kch && kc < seg0 + p.sq_seg; ++kc) {
              FF_WAIT(w_split, &ssplit[rs.s], rs.ph);
              tc_fence_after();
              const uint32_t b_hi = dsw_lo | (((sq_b + (uint32_t)(rs.s * p.sq_stage + FF_SQ_A)) & 0x3FFFFu) >> 4);
              const uint32_t b_lo = b_hi + (uint32_t)((S * 128) >> 4);
              const uint32_t a_hi = tmem_u + col_a + (uint32_t)(rs.s * 64);
              const uint32_t a_lo = a_hi + 32u;
              if (elect_one()) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const uint64_t dbh = dsw_hi | (uint64_t)(b_hi + 2 * j);
                  const uint64_t dbl = dsw_hi | (uint64_t)(b_lo + 2 * j);
                  umma_tf32_ts(d_tmem, a_lo + 8 * j, dbh, idesc_s, (kc != seg0 || j != 0) ? 1u : 0u);
                  umma_tf32_ts(d_tmem, a_hi + 8 * j, dbl, idesc_s, 1u);
                  umma_tf32_ts(d_tmem, a_hi + 8 * j, dbh, idesc_s, 1u);
                }
                umma_commit(&sempty[rs.s]);
              }
              __syncwarp();
              rs.next(p.nsq);
            }
            if (elect_one()) umma_commit(&sqfull[mt]);
            __syncwarp();
          }
      };
      auto expand = [&](int k) {
        const int qb = (p.nq == 2) ? (k & 1) : 0;
        const uint32_t qn = (p.nq == 2) ? ((uint32_t)k >> 1) : (uint32_t)k;
        FF_WAIT(w_qfull, &qfull[qb], qn & 1u);
        tc_fence_after();
        const uint32_t qa = ((q_b + (uint32_t)(qb * p.q_bytes)) & 0x3FFFFu) >> 4;
        const uint32_t qlo_off = (uint32_t)p.q_half >> 4;
        const int tpt = S / KCE;                   // weight tiles (2 K steps each) per filter tap
        for (int c = 0; c < p.nchunks; ++c) {
          const FireChunk ck = p.chunk[c];
          const int nt = ck.taps * tpt;
          // tap (dy, dx) = the Q tile at + dy*160 + dx*16 bytes (1x1: the centre tap), in 16-byte units
          uint32_t tap_off = ck.taps == 1 ? (uint32_t)((FF_QROW + 16) >> 4) : 0u;
          int i = 0, dx = 0;
          uint32_t wb_res = ew_b + (uint32_t)(ck.tile_base * p.ew_tile);
          for (int t0 = 0; t0 < nt; t0 += FF_SEG / 2, ++eg) {      // segment = 6 tiles = 36 MMAs
            const uint32_t buf = eg & 1u;
            FF_WAIT(w_tempty, &tempty[buf], ((eg >> 1) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_u + col_e + buf * (uint32_t)Ne;
            const int t1 = (t0 + FF_SEG / 2 < nt) ? t0 + FF_SEG / 2 : nt;
            for (int t = t0; t < t1; ++t) {
              uint32_t wb;
              if (p.resident) {
                wb = wb_res;
                wb_res += (uint32_t)p.ew_tile;
              } else {
                FF_WAIT(w_efull, &efull[re.s], re.ph);
                tc_fence_after();
                wb = ew_b + (uint32_t)(re.s * p.ew_tile);
              }
              const uint32_t a_hi = dq_lo | (qa + tap_off + (uint32_t)(i * ((4 * FF_QCH) >> 4)));
              const uint32_t a_lo = a_hi + qlo_off;
              const uint32_t b_hi = dew_lo | ((wb & 0x3FFFFu) >> 4);
              const uint32_t b_lo = b_hi + (uint32_t)((Ne * KCE * 4) >> 4);
              if (elect_one()) {
#pragma unroll
                for (int j = 0; j < KCE / 8; ++j) {
                  const uint32_t ao = (uint32_t)(j * ((2 * FF_QCH) >> 4)), bo = (uint32_t)(2 * j);
                  umma_tf32_ss(d_tmem, dq_hi | (uint64_t)(a_lo + ao), dew_hi | (uint64_t)(b_hi + bo), idesc_e,
                               (t != t0 || j != 0) ? 1u : 0u);
                  umma_tf32_ss(d_tmem, dq_hi | (uint64_t)(a_hi + ao), dew_hi | (uint64_t)(b_lo + bo), idesc_e, 1u);
                  umma_tf32_ss(d_tmem, dq_hi | (uint64_t)(a_hi + ao), dew_hi | (uint64_t)(b_hi + bo), idesc_e, 1u);
                }
                if (!p.resident) umma_commit(&eempty[re.s]);
              }
              __syncwarp();
              if (!p.resident) re.next(p.nring);
              if (++i == tpt) {                    // next tap: dx + 1, or the start of the next halo row
                i = 0;
                if (ck.taps != 1) {
                  if (++dx == 3) { dx = 0; tap_off += (uint32_t)((FF_QROW - 32) >> 4); }
                  else tap_off += 1u;
                }
              }
            }
            if (elect_one()) umma_commit(&tfull[buf]);
            __syncwarp();
          }
        }
        if (elect_one()) umma_commit(&qempty[qb]);   // every MMA that reads this Q buffer has retired
        __syncwarp();
      };

      if (p.resident) {
        mbar_wait(&efull[0], 0u);
        tc_fence_after();
      }
      // step s: squeeze(s), then expand(s - look): look = 1 with two Q buffers
      const int look = p.nq == 2 ? 1 : 0;
      for (int s = 0; s < my_items + look; ++s) {
        if (s < my_items) squeeze();
        if (s >= look) expand(s - look);
      }
      if (p.dbg && lane == 0) {
        p.dbg[blockIdx.x * 16 + 2] = (uint32_t)clock() - t_begin;
        p.dbg[blockIdx.x * 16 + 3] = w_split;
        p.dbg[blockIdx.x * 16 + 4] = w_sqempty;
        p.dbg[blockIdx.x * 16 + 5] = w_qfull;
        p.dbg[blockIdx.x * 16 + 6] = w_tempty;
        p.dbg[blockIdx.x * 16 + 7] = w_efull;
      }
    }
   } else {
    // ================================ operand splitters =====================================
    const int sg = role - 2;                       // squeeze stages cnt with cnt % 2 == sg
    const int t = (warp & 3) * 32 + lane;          // row of the M tile = TMEM lane, 0..95
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    RingPos r{0, 0u};
    uint32_t cnt = 0u;
    uint32_t w_full = 0;
    // squeeze-drain duty (sq_on_split): this group's rows 0..89 of M tile sg = halo pixel (9 sg + t / 10, t % 10)
    const int hl = t / FF_HW, wx = t - hl * FF_HW;
    const bool row_ok = t < FF_MT_ROWS;
    const uint32_t q_off = (uint32_t)((FF_MT_H * sg + hl) * FF_QROW + wx * 16);
    uint32_t sqn = 0u;
    for (int k = 0; k < my_items; ++k) {
      for (int seg0 = 0; seg0 < kch; seg0 += p.sq_seg)
        for (int mt = 0; mt < 2; ++mt)
          for (int kc = seg0; kc < kch && kc < seg0 + p.sq_seg; ++kc, ++cnt, r.next(p.nsq)) {
            // both groups wait on EVERY stage in order: an mbarrier waiter that skips phases can
            // mistake phase n-2 for phase n (same parity) when TMA loads complete out of order
            FF_WAIT(w_full, &sfull[r.s], r.ph);
            if ((int)(cnt & 1u) != sg) continue;
            {
              const uint32_t arow = sq_b + (uint32_t)(r.s * p.sq_stage + t * 128);
              const int sw = t & 7;
              const uint32_t a_slot = tmem_base + lane_sel + col_a + (uint32_t)(r.s * 64);
#pragma unroll
              for (int hblk = 0; hblk < 2; ++hblk) {
                uint32_t hi[16], lo[16];
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) {
                  const float4 v = lds128(arow + (uint32_t)(((hblk * 4 + c4) ^ sw) << 4));
                  const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float h = rn_tf32(vv[e]);
                    hi[c4 * 4 + e] = __float_as_uint(h);
                    lo[c4 * 4 + e] = __float_as_uint(vv[e] - h);
                  }
                }
                tmem_st16(a_slot + (uint32_t)(hblk * 16), hi);
                tmem_st16(a_slot + (uint32_t)(32 + hblk * 16), lo);
              }
              tmem_wait_st();
            }
            tc_fence_before();
            mbar_arrive(&ssplit[r.s]);
          }
      if (p.sq_on_split) {
        // every stage of item k is split: drain its squeeze accumulator (ONE segment, S = 16) into the Q tile
        FF_TILE_DECODE((int)blockIdx.x + k * (int)gridDim.x);
        (void)img;
        const int qb = (p.nq == 2) ? (k & 1) : 0;
        const uint32_t qn = (p.nq == 2) ? ((uint32_t)k >> 1) : (uint32_t)k;
        mbar_wait(&qempty[qb], (qn & 1u) ^ 1u);       // the expand MMAs of this buffer's last item retired
        mbar_wait(&sqfull[sg], sqn & 1u);
        ++sqn;
        tc_fence_after();
        uint32_t v[16];
        const uint32_t trow = tmem_base + lane_sel + (uint32_t)(sg * S);
        tmem_ld16_nowait(trow, v);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive(&sqempty[sg]);
        const float gain = 1.f + p.bias_comp * (float)(12 * kch);
        const int gy = h0 - 1 + FF_MT_H * sg + hl, gx = w0 - 1 + wx;
        const bool inside = gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
        if (row_ok) {
          const uint32_t dst = q_b + (uint32_t)(qb * p.q_bytes) + q_off;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias_sq) + c4);   // L1-resident
            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
            float o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a = __uint_as_float(v[c4 * 4 + e]) * gain;
              o[e] = inside ? fmaxf(a + bb[e], 0.f) : 0.f;
            }
            float4 hi, lo;
            hi.x = rn_tf32(o[0]); hi.y = rn_tf32(o[1]); hi.z = rn_tf32(o[2]); hi.w = rn_tf32(o[3]);
            lo.x = o[0] - hi.x; lo.y = o[1] - hi.y; lo.z = o[2] - hi.z; lo.w = o[3] - hi.w;
            sts128(dst + (uint32_t)(c4 * FF_QCH), hi);
            sts128(dst + (uint32_t)(c4 * FF_QCH + p.q_half), lo);
          }
        }
        fence_async_proxy();
        mbar_arrive(&qfull[qb]);
      }
    }
    if (p.dbg && t == 0 && sg == 0) p.dbg[blockIdx.x * 16 + 8] = w_full;
   }
  } else {
    // ==================== drains: squeeze -> Q tile, expand -> output ========================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
    const int g = role;                          // drain group: squeeze M tile g, expand groups jg % 2 == g
    const int q = warp & 3;
    const int r = q * 32 + lane;                 // TMEM lane
    const int tt = threadIdx.x & 127;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    // epilogue parameters, the same for every item: squeeze bias, expand biases
    for (int i = g * 128 + tt; i < FF_PAR_FLOATS; i += 256) {
      float v = 0.f;
      if (i < FF_MAX_S) { if (i < S) v = __ldg(p.bias_sq + i); }
      else if (i - FF_MAX_S < p.E1 + p.E3) v = __ldg(p.bias_e + (i - FF_MAX_S));
      sts32(par_b + 4u * (uint32_t)i, v);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // squeeze drain geometry: row r of M tile g = halo pixel (9g + r / 10, r % 10)
    const int hl = r / FF_HW, wx = r - hl * FF_HW;
    const bool row_ok = r < FF_MT_ROWS;
    const uint32_t q_off = (uint32_t)((FF_MT_H * g + hl) * FF_QROW + wx * 16);
    uint32_t sqn = 0u, eg = 0u;
    int n_store = 0;
    uint32_t w_sqfull = 0, w_qempty = 0, w_tfull = 0, c_sq = 0, c_epi = 0, c_stw = 0;

    auto squeeze_drain = [&](int k) {
      FF_TILE_DECODE((int)blockIdx.x + k * (int)gridDim.x);
      (void)img;
      const int qb = (p.nq == 2) ? (k & 1) : 0;
      const uint32_t qn = (p.nq == 2) ? ((uint32_t)k >> 1) : (uint32_t)k;
      FF_WAIT(w_qempty, &qempty[qb], (qn & 1u) ^ 1u);   // the expand MMAs of this buffer's last item retired
      float acc[FF_MAX_S];
      for (int seg0 = 0; seg0 < kch; seg0 += p.sq_seg, ++sqn) {
        FF_WAIT(w_sqfull, &sqfull[g], sqn & 1u);
        tc_fence_after();
        const int nst = (kch - seg0) < p.sq_seg ? (kch - seg0) : p.sq_seg;
        // chained MMAs per accumulator column in this segment: 3 per K step
        const float gain = 1.f + p.bias_comp * (float)(12 * nst);
        const uint32_t trow = tmem_base + lane_sel + (uint32_t)(g * S);
#pragma unroll
        for (int c0 = 0; c0 < FF_MAX_S; c0 += 16) {
          if (c0 < S) {                            // warp-uniform
            uint32_t v[16];
            tmem_ld16_nowait(trow + (uint32_t)c0, v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 16; ++e)
              acc[c0 + e] = fmaf(__uint_as_float(v[e]), gain, seg0 == 0 ? 0.f : acc[c0 + e]);
          }
        }
        tc_fence_before();
        mbar_arrive(&sqempty[g]);
      }
      const uint32_t t0 = p.dbg ? (uint32_t)clock() : 0u;
      const int gy = h0 - 1 + FF_MT_H * g + hl, gx = w0 - 1 + wx;
      const bool inside = gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
      if (row_ok) {
        const uint32_t dst = q_b + (uint32_t)(qb * p.q_bytes) + q_off;
#pragma unroll
        for (int c4 = 0; c4 < FF_MAX_S / 4; ++c4) {
          if (c4 * 4 < S) {
            const float4 b = lds128(par_b + 16u * (uint32_t)c4);
            float o[4] = {acc[c4 * 4] + b.x, acc[c4 * 4 + 1] + b.y, acc[c4 * 4 + 2] + b.z,
                          acc[c4 * 4 + 3] + b.w};
            float4 hi, lo;
#pragma unroll
            for (int e = 0; e < 4; ++e) o[e] = inside ? fmaxf(o[e], 0.f) : 0.f;
            hi.x = rn_tf32(o[0]); hi.y = rn_tf32(o[1]); hi.z = rn_tf32(o[2]); hi.w = rn_tf32(o[3]);
            lo.x = o[0] - hi.x; lo.y = o[1] - hi.y; lo.z = o[2] - hi.z; lo.w = o[3] - hi.w;
            sts128(dst + (uint32_t)(c4 * FF_QCH), hi);
            sts128(dst + (uint32_t)(c4 * FF_QCH + p.q_half), lo);
          }
        }
      }
      fence_async_proxy();                         // the tensor core reads Q through the async proxy
      mbar_arrive(&qfull[qb]);
      if (p.dbg) c_sq += (uint32_t)clock() - t0;
    };

    auto expand_drain = [&](int k) {
      FF_TILE_DECODE((int)blockIdx.x + k * (int)gridDim.x);
      for (int c = 0; c < p.nchunks; ++c) {
        const FireChunk ck = p.chunk[c];
        const int nk = ck.taps * ksq;
        float acc[64];                             // groups jg = g and g + 2 of this chunk
        for (int kk0 = 0; kk0 < nk; kk0 += FF_SEG, ++eg) {
          const uint32_t buf = eg & 1u;
          FF_WAIT(w_tfull, &tfull[buf], (eg >> 1) & 1u);
          tc_fence_after();
          const int nks = (nk - kk0) < FF_SEG ? (nk - kk0) : FF_SEG;
          const float gain = 1.f + p.bias_comp * (float)(3 * nks);
          const uint32_t trow = tmem_base + lane_sel + col_e + buf * (uint32_t)Ne;
#pragma unroll
          for (int jj = 0; jj < 2; ++jj) {
            const int jg = g + 2 * jj;
            if (jg * 32 < Ne) {                    // warp-uniform
              uint32_t v0[16], v1[16];
              tmem_ld16_nowait(trow + (uint32_t)(jg * 32), v0);
              tmem_ld16_nowait(trow + (uint32_t)(jg * 32 + 16), v1);
              tmem_wait_ld();
#pragma unroll
              for (int e = 0; e < 16; ++e) {
                acc[jj * 32 + e] = fmaf(__uint_as_float(v0[e]), gain, kk0 == 0 ? 0.f : acc[jj * 32 + e]);
                acc[jj * 32 + 16 + e] =
                    fmaf(__uint_as_float(v1[e]), gain, kk0 == 0 ? 0.f : acc[jj * 32 + 16 + e]);
              }
            }
          }
          tc_fence_before();
          mbar_arrive(&tempty[buf]);
        }
        // ---- epilogue: + bias, ReLU, 32-pixel x 32-channel tile per warp -> TMA store --------
        const uint32_t t0 = p.dbg ? (uint32_t)clock() : 0u;
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int jg = g + 2 * jj;
          if (jg * 32 < Ne) {
            if (lane == 0) {
              const uint32_t t1 = p.dbg ? (uint32_t)clock() : 0u;
              if (p.store_ring == 2) tma_store_wait_read_le1();
              else tma_store_wait_read_all();
              if (p.dbg) c_stw += (uint32_t)clock() - t1;
            }
            __syncwarp();
            const uint32_t tile_w = out_b + (uint32_t)((g * 4 + q) * (4096 * p.store_ring) +
                                                       (p.store_ring == 2 ? (n_store & 1) * 4096 : 0));
            const uint32_t bias = par_b + 4u * (uint32_t)(FF_MAX_S + ck.y_coff + jg * 32);
#pragma unroll
            for (int kq = 0; kq < 8; ++kq) {
              const float4 b = lds128(bias + 16u * (uint32_t)kq);
              float4 v;
              v.x = fmaxf(acc[jj * 32 + kq * 4] + b.x, 0.f);
              v.y = fmaxf(acc[jj * 32 + kq * 4 + 1] + b.y, 0.f);
              v.z = fmaxf(acc[jj * 32 + kq * 4 + 2] + b.z, 0.f);
              v.w = fmaxf(acc[jj * 32 + kq * 4 + 3] + b.w, 0.f);
              sts128(tile_w + (uint32_t)(lane * 128 + ((kq ^ (lane & 7)) << 4)), v);
            }
            fence_async_proxy();
            __syncwarp();
            // TMEM lane 32q + l = output pixel (4q + l / 8, l % 8) of the tile = row l of the box
            if (lane == 0)
              tma_store_4d(tile_w, &p.tmY, ck.y_coff + jg * 32, w0, h0 + 4 * q, img);
            ++n_store;
          }
        }
        if (p.dbg) c_epi += (uint32_t)clock() - t0;
      }
    };

    const int look = p.nq == 2 ? 1 : 0;            // same order as the MMA warp
    for (int s = 0; s < my_items + look; ++s) {
      if (s < my_items && !p.sq_on_split) squeeze_drain(s);
      if (s >= look) expand_drain(s - look);
    }
    if (lane == 0) tma_store_wait_all();
    if (p.dbg && g == 0 && tt == 0) {
      p.dbg[blockIdx.x * 16 + 9] = w_sqfull;
      p.dbg[blockIdx.x * 16 + 10] = w_qempty;
      p.dbg[blockIdx.x * 16 + 11] = w_tfull;
      p.dbg[blockIdx.x * 16 + 12] = c_sq;
      p.dbg[blockIdx.x * 16 + 13] = c_epi;
      p.dbg[blockIdx.x * 16 + 14] = c_stw;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (role == 3 && ctl) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
struct FireImpl {
  FireParams prm;
  size_t smem_bytes = 0;
  dim3 grid;
  float* d_ws = nullptr;      // packed squeeze weights [Cin/32][S][32], hi rows then lo rows
  float* d_we = nullptr;      // packed expand weight tiles [tile][Ne][KCE], hi then lo
  float* d_bsq = nullptr;
  float* d_be = nullptr;
};

static inline float ff_rn_tf32(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

static void release_fire(void** impl) {
  if (!*impl) return;
  FireImpl* im = static_cast<FireImpl*>(*impl);
  cudaFree(im->d_ws);
  cudaFree(im->d_we);
  cudaFree(im->d_bsq);
  cudaFree(im->d_be);
  delete im;
  *impl = nullptr;
}

}  // namespace

int fused_fire_plan(FusedFirePlan* plan, int B, int H, int W, int Cin, int S, int E1, int E3,
                    const float* x_dev, float* y_dev) {
  plan->enabled = false;
  plan->impl = nullptr;
  static const int env_fused = env_int("SQDET_FUSED_FIRE", 1);
  if (!env_fused) return 0;
  // shapes this kernel takes (everything else stays on the squeeze + expand-pair launches)
  if (Cin % 32 != 0 || Cin < 32 || S % 16 != 0 || S < 16 || S > FF_MAX_S) return 0;
  if (E1 % 32 != 0 || E3 % 32 != 0 || E1 < 32 || E3 < 32 || E1 + E3 > 512) return 0;
  auto ne_of = [](int E) {
    const int ns = (E + 127) / 128;
    return (E % ns == 0 && (E / ns) % 32 == 0) ? E / ns : 0;
  };
  const int Ne = ne_of(E1);
  if (Ne == 0 || ne_of(E3) != Ne) return 0;
  FireImpl* im = new FireImpl();
  FireParams& P = im->prm;
  memset(&P, 0, sizeof P);
  P.B = B; P.H = H; P.W = W; P.Cin = Cin; P.S = S; P.E1 = E1; P.E3 = E3;
  P.tiles_h = (H + FF_TH - 1) / FF_TH;
  P.tiles_w = (W + FF_TW - 1) / FF_TW;
  P.ntiles = B * P.tiles_h * P.tiles_w;
  P.Ne = Ne;
  int tiles = 0;
  P.nchunks = 0;
  for (int cb = 0; cb < E1; cb += Ne) {
    P.chunk[P.nchunks++] = FireChunk{tiles, 1, cb};
    tiles += S / KCE;
  }
  for (int cb = 0; cb < E3; cb += Ne) {
    P.chunk[P.nchunks++] = FireChunk{tiles, 9, E1 + cb};
    tiles += 9 * (S / KCE);
  }
  P.ntiles_w = tiles;
  P.ew_tile = 2 * Ne * KCE * 4;
  P.q_half = (S / 4) * FF_QCH;
  P.q_bytes = 2 * P.q_half;
  P.sq_stage = FF_SQ_A + 2 * S * 128;
  static const float env_comp = env_float("SQDET_TC_BIAS_COMP", 1.4e-8f);
  P.bias_comp = env_comp;
  // shared-memory plan: the deepest configuration that fits 227 KB, in order of preference
  const int fixed = FF_PAR_FLOATS * 4 + 1024 /*barriers*/;
  const bool can_reside = (long long)tiles * P.ew_tile <= 120 * 1024;
  // squeeze drain on the splitter groups: single-segment squeezes with S = 16 (fire2/3: Cin <= 128 as
  // ONE segment of up to 4 stages = 48 chained MMAs).  OPT-IN: parity-green (tests/test_gpu_fire.py)
  // and -15 % / -6 % on fire2 / fire3 in the per-op timing (profiles/r2_fused_fire.txt), but the one
  // bench.py run made with it did not finish inside its time limit and the GPU budget of the round
  // ended before that could be explained - off until it is.
  static const int env_sqsplit = env_int("SQDET_FF_SQSPLIT", 0);
  P.sq_on_split = (S == 16 && Cin <= 128 && env_sqsplit) ? 1 : 0;
  P.sq_seg = P.sq_on_split ? 4 : 3;
  struct Cand { int nq, nsq, nring, store_ring; };
  // deepest squeeze ring first (measured: with 2-3 stages the MMA warp waits on the TMA -> splitter
  // latency at the start of every item), then two Q buffers, then the weight ring
  const Cand cands[] = {{2, 4, 4, 2}, {2, 4, 4, 1}, {2, 4, 3, 1}, {2, 3, 4, 1}, {2, 3, 3, 1}, {2, 3, 2, 1},
                        {1, 4, 4, 1}, {1, 3, 4, 1}, {1, 3, 3, 1}, {2, 2, 4, 1}, {2, 2, 3, 1}, {1, 2, 4, 1},
                        {1, 2, 3, 1}, {1, 2, 2, 1}};
  bool placed = false;
  for (int pass = 0; pass < 2 && !placed; ++pass) {
    const bool resident = pass == 0 && can_reside;   // weights resident first, else streamed
    if (pass == 0 && !resident) continue;
    for (const Cand& c : cands) {
      // the exact shared-memory map of this candidate (same arithmetic as below)
      auto up1k = [](long long v) { return (v + 1023) & ~1023LL; };
      long long off = up1k((long long)c.nsq * P.sq_stage);
      off = up1k(off + (resident ? (long long)tiles : (long long)c.nring) * P.ew_tile);
      off = up1k(off + 8LL * 4096 * c.store_ring);
      off = up1k(off + (long long)c.nq * P.q_bytes);
      off += fixed + 16 + 1024 /*base alignment*/;
      if (off > 232448) continue;
      if (2 * S + 2 * Ne + 64 * c.nsq > 512) continue;
      P.nq = c.nq; P.nsq = c.nsq; P.nring = resident ? 1 : c.nring; P.store_ring = c.store_ring;
      P.resident = resident ? 1 : 0;
      placed = true;
      break;
    }
  }
  if (!placed) { delete im; return 0; }
  {
    auto up = [](int v) { return (v + 1023) & ~1023; };
    int off = 0;
    P.off_sq = off;  off = up(off + P.nsq * P.sq_stage);
    P.off_ew = off;  off = up(off + (P.resident ? tiles : P.nring) * P.ew_tile);
    P.off_out = off; off = up(off + 8 * 4096 * P.store_ring);
    P.off_q = off;   off = up(off + P.nq * P.q_bytes);
    P.off_par = off; off += FF_PAR_FLOATS * 4;
    off = (off + 15) & ~15;
    P.off_bar = off; off += 1024;
    im->smem_bytes = (size_t)off + 1024;
    if (im->smem_bytes > 232448) { delete im; return 0; }
  }
  {
    int cols = 32;
    while (cols < 2 * S + 2 * Ne + 64 * P.nsq) cols <<= 1;
    P.tmem_cols = cols;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  im->grid = dim3((unsigned)(P.ntiles < sms ? P.ntiles : sms));
  void* pim = im;
  const size_t ws_floats = (size_t)(Cin / 32) * S * 32 * 2;
  const size_t we_floats = (size_t)tiles * Ne * KCE * 2;
  P.lo_rows_sq = (Cin / 32) * S;
  P.lo_rows_e = tiles * Ne;
  if (cudaMalloc(&im->d_ws, sizeof(float) * ws_floats) != cudaSuccess ||
      cudaMalloc(&im->d_we, sizeof(float) * we_floats) != cudaSuccess ||
      cudaMalloc(&im->d_bsq, sizeof(float) * S) != cudaSuccess ||
      cudaMalloc(&im->d_be, sizeof(float) * (E1 + E3)) != cudaSuccess) {
    release_fire(&pim);
    return fail(SQDET_ERR_CUDA, "fused_fire_plan: cudaMalloc failed");
  }
  cudaMemset(im->d_ws, 0, sizeof(float) * ws_floats);
  cudaMemset(im->d_we, 0, sizeof(float) * we_floats);
  cudaMemset(im->d_bsq, 0, sizeof(float) * S);
  cudaMemset(im->d_be, 0, sizeof(float) * (E1 + E3));
  P.bias_sq = im->d_bsq;
  P.bias_e = im->d_be;
  int rc = tc_encode_act_map(&P.tmX, x_dev, B, H, W, Cin, 32, FF_HW, FF_MT_H);
  if (!rc) rc = tc_encode_w_map(&P.tmWs, im->d_ws, 2 * P.lo_rows_sq, 32, S);
  if (!rc) rc = tc_encode_w_map(&P.tmWe, im->d_we, 2 * P.lo_rows_e, KCE, Ne);
  if (!rc) rc = tc_encode_act_map(&P.tmY, y_dev, B, H, W, E1 + E3, 32, FF_TW, 4);
  if (rc) {
    release_fire(&pim);
    return rc;
  }
  cudaError_t ce = cudaFuncSetAttribute(fire_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        232448);
  if (ce != cudaSuccess) {
    release_fire(&pim);
    return cuda_fail(ce, "cudaFuncSetAttribute(fire_fused_kernel)");
  }
  plan->enabled = true;
  plan->B = B; plan->H = H; plan->W = W; plan->Cin = Cin; plan->S = S; plan->E1 = E1; plan->E3 = E3;
  plan->impl = im;
  return 1;
}

int fused_fire_pack_weights(FusedFirePlan* plan, const float* w_sq, const float* b_sq,
                            const float* w_e1, const float* b_e1, const float* w_e3,
                            const float* b_e3) {
  FireImpl* im = static_cast<FireImpl*>(plan->impl);
  const FireParams& P = im->prm;
  const int Cin = P.Cin, S = P.S, E1 = P.E1, E3 = P.E3, Ne = P.Ne;
  // squeeze: HWIO [1,1,Cin,S] -> rows [kc][s][32 input channels], hi block then lo block
  std::vector<float> ws((size_t)2 * P.lo_rows_sq * 32, 0.f);
  for (int kc = 0; kc < Cin / 32; ++kc)
    for (int s = 0; s < S; ++s)
      for (int k = 0; k < 32; ++k) {
        const float v = w_sq[(size_t)(kc * 32 + k) * S + s];
        const float hi = ff_rn_tf32(v);
        const size_t row = (size_t)kc * S + s;
        ws[row * 32 + k] = hi;
        ws[((size_t)P.lo_rows_sq + row) * 32 + k] = ff_rn_tf32(v - hi);
      }
  // expand: tiles [chunk][tap][K chunk of KCE squeeze channels][Ne output channels][KCE]
  std::vector<float> we((size_t)2 * P.lo_rows_e * KCE, 0.f);
  for (int c = 0; c < P.nchunks; ++c) {
    const FireChunk& ck = P.chunk[c];
    const bool is3 = ck.taps == 9;
    const float* w = is3 ? w_e3 : w_e1;
    const int E = is3 ? E3 : E1;
    const int cb = ck.y_coff - (is3 ? E1 : 0);
    for (int tap = 0; tap < ck.taps; ++tap)
      for (int kc = 0; kc < S / KCE; ++kc)
        for (int n = 0; n < Ne; ++n)
          for (int k = 0; k < KCE; ++k) {
            const float v = w[((size_t)tap * S + (size_t)kc * KCE + k) * E + cb + n];
            const float hi = ff_rn_tf32(v);
            const size_t row = ((size_t)ck.tile_base + (size_t)tap * (S / KCE) + kc) * Ne + n;
            we[row * KCE + k] = hi;
            we[((size_t)P.lo_rows_e + row) * KCE + k] = ff_rn_tf32(v - hi);
          }
  }
  SQ_CUDA(cudaMemcpy(im->d_ws, ws.data(), ws.size() * sizeof(float), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_we, we.data(), we.size() * sizeof(float), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_bsq, b_sq, sizeof(float) * S, cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_be, b_e1, sizeof(float) * E1, cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMemcpy(im->d_be + E1, b_e3, sizeof(float) * E3, cudaMemcpyHostToDevice));
  return SQDET_OK;
}

int launch_fused_fire(const FusedFirePlan& plan, cudaStream_t stream) {
  const FireImpl* im = static_cast<const FireImpl*>(plan.impl);
  if (!im) return fail(SQDET_ERR_STATE, "no fused fire plan");
  FireParams prm = im->prm;
  static const int debug = env_int("SQDET_TC_DEBUG", 0);
  long long* dbg = nullptr;
  const int nb = (int)im->grid.x;
  if (debug) {
    SQ_CUDA(cudaMalloc(&dbg, sizeof(long long) * 16 * nb));
    SQ_CUDA(cudaMemsetAsync(dbg, 0, sizeof(long long) * 16 * nb, stream));
    prm.dbg = dbg;
  }
  SQ_CUDA(launch_kernel(fire_fused_kernel, im->grid, dim3(FF_THREADS), im->smem_bytes, stream, prm));
  SQ_CHECK_LAUNCH("fire_fused_kernel");
  if (debug) {
    std::vector<long long> h((size_t)16 * nb);
    SQ_CUDA(cudaStreamSynchronize(stream));
    SQ_CUDA(cudaMemcpy(h.data(), dbg, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
    cudaFree(dbg);
    double a[16] = {0};
    for (int b = 0; b < nb; ++b)
      for (int k = 0; k < 16; ++k) a[k] += (double)h[(size_t)b * 16 + k] / nb;
    fprintf(stderr,
            "[fire_tc] grid %d tiles %d Cin %d S %d E %d+%d Ne %d KCE %d chunks %d | nq %d nsq %d %s%d "
            "store_ring %d smem %zu | per-CTA avg cycles: mma total %.0f waits: split %.0f sqempty %.0f "
            "qfull %.0f tempty %.0f efull %.0f | producers wait-empty: sq %.0f ew %.0f | splitter(g0) "
            "wait-full %.0f | drain(g0) waits: sqfull %.0f qempty %.0f tfull %.0f work: sq-epi %.0f "
            "ex-epi %.0f (store-wait %.0f)\n",
            nb, prm.ntiles, prm.Cin, prm.S, prm.E1, prm.E3, prm.Ne, KCE, prm.nchunks, prm.nq,
            prm.nsq, prm.resident ? "resident tiles " : "ring ", prm.resident ? prm.ntiles_w : prm.nring,
            prm.store_ring, im->smem_bytes, a[2], a[3], a[4], a[5], a[6], a[7], a[0], a[1], a[8], a[9],
            a[10], a[11], a[12], a[13], a[14]);
  }
  return SQDET_OK;
}

void fused_fire_release(FusedFirePlan* plan) {
  release_fire(&plan->impl);
  plan->enabled = false;
}

int fire_fused_oneshot(const float* x_dev, const float* w_sq_dev, const float* b_sq_dev,
                       const float* w_e1_dev, const float* b_e1_dev, const float* w_e3_dev,
                       const float* b_e3_dev, float* y_dev, int B, int H, int W, int Cin, int S,
                       int E1, int E3, cudaStream_t stream) {
  FusedFirePlan plan;
  int rc = fused_fire_plan(&plan, B, H, W, Cin, S, E1, E3, x_dev, y_dev);
  if (rc < 0) return rc;
  if (rc == 0) return 1;
  std::vector<float> ws((size_t)Cin * S), w1((size_t)S * E1), w3((size_t)9 * S * E3), bs(S), b1(E1),
      b3(E3);
  auto pull = [](std::vector<float>& h, const float* d) {
    return cudaMemcpy(h.data(), d, h.size() * sizeof(float), cudaMemcpyDeviceToHost);
  };
  cudaError_t ce = pull(ws, w_sq_dev);
  if (ce == cudaSuccess) ce = pull(w1, w_e1_dev);
  if (ce == cudaSuccess) ce = pull(w3, w_e3_dev);
  if (ce == cudaSuccess) ce = pull(bs, b_sq_dev);
  if (ce == cudaSuccess) ce = pull(b1, b_e1_dev);
  if (ce == cudaSuccess) ce = pull(b3, b_e3_dev);
  if (ce != cudaSuccess) {
    fused_fire_release(&plan);
    return cuda_fail(ce, "fire_fused_oneshot: weight download");
  }
  rc = fused_fire_pack_weights(&plan, ws.data(), bs.data(), w1.data(), b1.data(), w3.data(), b3.data());
  if (!rc) rc = launch_fused_fire(plan, stream);
  ce = cudaStreamSynchronize(stream);
  fused_fire_release(&plan);
  if (rc) return rc;
  if (ce != cudaSuccess) return cuda_fail(ce, "fire_fused_oneshot sync");
  return SQDET_OK;
}

}  // namespace sqdet
