// Fused first layer: conv (Cin = 3, k x k, stride 2) + bias [+ frozen BN] + ReLU + 3x3/2
// max-pool in ONE kernel, fp32 FFMA.
//
// Replaces conv1 -> pool1 of every net (reference src/nets/squeezeDet.py:40-44,
// squeezeDetPlus.py:40-44, resnet50_convDet.py:41-46; layer code src/nn_skeleton.py:471-586).
// conv1's output is the largest tensor of the whole network (20 x 188 x 621 x 64 fp32 = 598 MB
// at the benchmark size); unfused it is written once and read once by pool1 (1.2 GB of the
// 4.7 GB a forward pass moves).  Here it never leaves shared memory.
//
// K = 27 (or 147) with Cin = 3 is too thin for a tensor-core tile and the layer is
// HBM-bound after fusion (reads 112 MB, writes 150 MB), so it stays on the FFMA pipe:
// exact fp32, same arithmetic as the reference's fp32 conv.
//
// CTA = one pooled tile of 4 x 16 pixels of one image:
//   input patch  (2*8+k) x (2*32+k) x 3 floats        -> smem (coalesced row loads, 0 = pad)
//   conv tile    9 x 33 conv pixels x Cout             -> registers (5 px x 16 ch per thread)
//                 -> +bias [*scale+shift], ReLU, -inf outside the image -> smem
//   pooled tile  4 x 16 x Cout, max over 3x3 windows   -> 128-bit coalesced global stores
// Threads: 64 per 16-channel group (Cout/16 groups).  Weights [k*k*3][Cout] live in smem.
#include <math_constants.h>

#include "common.cuh"

namespace sqdet {
namespace {

constexpr int PT_H = 4, PT_W = 16;                 // pooled tile
constexpr int CT_H = 2 * PT_H + 1, CT_W = 2 * PT_W + 1;   // 9 x 33 conv pixels (3x3/2 pool)
constexpr int CT_PIX = CT_H * CT_W;               // 297
constexpr int PIX_PER_THREAD = (CT_PIX + 63) / 64;  // 5

// Two IEEE fp32 FMAs per instruction (Blackwell FFMA2): identical results to two fmaf().
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b,
                                                    unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

struct ConvPoolParams {
  const float* x;       // [B,H,W,3]
  const float* w;       // [k,k,3,Cout]
  const float* bias;    // [Cout] or null
  const float* scale;   // [Cout] or null
  const float* shift;
  float* y;             // [B,Hp,Wp,Cout]
  int B, H, W, Cout;
  int Hc, Wc;           // conv output size
  int Hp, Wp;           // pooled output size
  int cpad_t, cpad_l;   // conv pad_before
  int ppad_t, ppad_l;   // pool pad_before
  int relu;
  int tiles_w, tiles_h;
};

template <int KS, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB)
conv_pool_simt_kernel(const ConvPoolParams p) {
  constexpr int PH = 2 * (CT_H - 1) + KS;          // input patch rows
  constexpr int PW = 2 * (CT_W - 1) + KS;          // input patch cols (pixels)
  constexpr int K = KS * KS * 3;
  extern __shared__ __align__(16) float sm[];
  float* s_patch = sm;                             // [PH][PW*3]
  float* s_w = s_patch + ((PH * PW * 3 + 3) & ~3); // [K][Cout]
  float* s_conv = s_w + K * p.Cout;                // [Cout/16][CT_PIX][16] (swizzled chunks)

  const int tid = threadIdx.x;
  const int nthreads = blockDim.x;
  int tile = blockIdx.x;
  const int tw = tile % p.tiles_w;
  tile /= p.tiles_w;
  const int th = tile % p.tiles_h;
  const int img = tile / p.tiles_h;
  const int ph0 = th * PT_H, pw0 = tw * PT_W;            // pooled origin
  const int ch0 = 2 * ph0 - p.ppad_t, cw0 = 2 * pw0 - p.ppad_l;   // conv origin
  const int iy0 = 2 * ch0 - p.cpad_t, ix0 = 2 * cw0 - p.cpad_l;   // input origin

  // ---- stage weights and the input patch with cp.async (fire-and-forget, so the ~20
  // row-segment loads per thread overlap instead of paying one L2 round trip each) ----
  for (int i = tid; i < K * p.Cout / 4; i += nthreads) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(s_w + i * 4);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p.w + i * 4) : "memory");
  }
  {
    const float* xin = p.x + (size_t)img * p.H * p.W * 3;
    const int wid = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    for (int row = wid; row < PH; row += nwarps) {       // one warp per patch row: coalesced
      const int iy = iy0 + row;
      const bool row_ok = iy >= 0 && iy < p.H;
      const float* src = xin + (size_t)(row_ok ? iy : 0) * p.W * 3;
#pragma unroll
      for (int it = 0; it < (PW * 3 + 31) / 32; ++it) {  // col counts floats (pixel*3 + c)
        const int col = lane + it * 32;
        if (col < PW * 3) {
          const int ixc = ix0 * 3 + col;
          const bool ok = row_ok && ixc >= 0 && ixc < p.W * 3;
          const unsigned dst = (unsigned)__cvta_generic_to_shared(s_patch + row * (PW * 3) + col);
          const int nbytes = ok ? 4 : 0;                 // 0 -> the 4 bytes are zero-filled
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst),
                       "l"(src + (ok ? ixc : 0)), "r"(nbytes)
                       : "memory");
        }
      }
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  // ---- conv: 5 pixels x 16 channels per thread ----
  const int cg = tid >> 6;                 // channel group (warp-uniform)
  const int l64 = tid & 63;
  unsigned long long acc2[PIX_PER_THREAD][8];      // 16 channels as 8 packed fp32 pairs
#pragma unroll
  for (int i = 0; i < PIX_PER_THREAD; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc2[i][c] = 0ull;
  int pbase[PIX_PER_THREAD];
#pragma unroll
  for (int i = 0; i < PIX_PER_THREAD; ++i) {
    int px = l64 + 64 * i;
    if (px >= CT_PIX) px = CT_PIX - 1;     // clamp (result discarded)
    const int cr = px / CT_W, cc = px - cr * CT_W;
    pbase[i] = (2 * cr * PW + 2 * cc) * 3;
  }
  const float* wg = s_w + cg * 16;
  for (int a = 0; a < KS; ++a) {
#pragma unroll
    for (int bc = 0; bc < KS * 3; ++bc) {          // (b, c) flattened: contiguous in the patch
      const int k = a * KS * 3 + bc;
      unsigned long long xx[PIX_PER_THREAD];
#pragma unroll
      for (int i = 0; i < PIX_PER_THREAD; ++i) {
        const unsigned xb = __float_as_uint(s_patch[pbase[i] + a * PW * 3 + bc]);
        xx[i] = ((unsigned long long)xb << 32) | xb;
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {       // 8 channels at a time: fewer live weights
        const ulonglong2 wa = *reinterpret_cast<const ulonglong2*>(wg + k * p.Cout + half * 8);
        const ulonglong2 wb = *reinterpret_cast<const ulonglong2*>(wg + k * p.Cout + half * 8 + 4);
        const unsigned long long wv[4] = {wa.x, wa.y, wb.x, wb.y};
#pragma unroll
        for (int i = 0; i < PIX_PER_THREAD; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c)
            acc2[i][half * 4 + c] = ffma2(xx[i], wv[c], acc2[i][half * 4 + c]);
      }
    }
  }
  float acc[PIX_PER_THREAD][16];
#pragma unroll
  for (int i = 0; i < PIX_PER_THREAD; ++i)
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      acc[i][2 * c] = __uint_as_float((unsigned)(acc2[i][c] & 0xffffffffull));
      acc[i][2 * c + 1] = __uint_as_float((unsigned)(acc2[i][c] >> 32));
    }

  // ---- epilogue 1: bias [, affine], relu, mask, conv tile -> smem ----
  {
    float bv[16], sv[16], hv[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      bv[c] = p.bias ? __ldg(p.bias + cg * 16 + c) : 0.f;
      sv[c] = p.scale ? __ldg(p.scale + cg * 16 + c) : 1.f;
      hv[c] = p.scale ? __ldg(p.shift + cg * 16 + c) : 0.f;
    }
    float* tile_c = s_conv + (size_t)cg * CT_PIX * 16;
#pragma unroll
    for (int i = 0; i < PIX_PER_THREAD; ++i) {
      const int px = l64 + 64 * i;
      if (px < CT_PIX) {
        const int cr = px / CT_W, cc = px - cr * CT_W;
        const int oh = ch0 + cr, ow = cw0 + cc;
        const bool ok = oh >= 0 && oh < p.Hc && ow >= 0 && ow < p.Wc;
        const int sw = (px >> 1) & 3;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float f = acc[i][j * 4 + e] + bv[j * 4 + e];
            if (p.scale) f = f * sv[j * 4 + e] + hv[j * 4 + e];
            if (p.relu) f = fmaxf(f, 0.f);
            o[e] = ok ? f : -CUDART_INF_F;      // tf.nn.max_pool ignores padded cells
          }
          *reinterpret_cast<float4*>(tile_c + px * 16 + ((j ^ sw) << 2)) =
              make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
  }
  __syncthreads();

  // ---- epilogue 2: 3x3/2 max-pool from smem, coalesced 128-bit stores ----
  const int chunks = p.Cout / 4;                   // 16-byte chunks per pooled pixel
  for (int u = tid; u < PT_H * PT_W * chunks; u += nthreads) {
    const int chunk = u % chunks, pp = u / chunks;
    const int py = pp / PT_W, pxp = pp - py * PT_W;
    const int ph = ph0 + py, pw = pw0 + pxp;
    if (ph >= p.Hp || pw >= p.Wp) continue;
    const int g = chunk >> 2, j = chunk & 3;
    const float* tile_c = s_conv + (size_t)g * CT_PIX * 16;
    float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        const int px = (2 * py + a) * CT_W + 2 * pxp + b;
        const float4 q = *reinterpret_cast<const float4*>(tile_c + px * 16 + ((j ^ ((px >> 1) & 3)) << 2));
        m.x = fmaxf(m.x, q.x); m.y = fmaxf(m.y, q.y);
        m.z = fmaxf(m.z, q.z); m.w = fmaxf(m.w, q.w);
      }
    *reinterpret_cast<float4*>(p.y + (((size_t)img * p.Hp + ph) * p.Wp + pw) * p.Cout + chunk * 4) = m;
  }
}

template <int KS>
size_t smem_bytes_for(int Cout) {
  constexpr int PH = 2 * (CT_H - 1) + KS, PW = 2 * (CT_W - 1) + KS;
  return sizeof(float) * ((size_t)((PH * PW * 3 + 3) & ~3) + (size_t)KS * KS * 3 * Cout +
                          (size_t)(Cout / 16) * CT_PIX * 16);
}

}  // namespace

bool conv_pool_simt_eligible(int Cin, int Cout, int ksize, int stride, int pool_size,
                             int pool_stride) {
  return Cin == 3 && (ksize == 3 || ksize == 7) && stride == 2 && pool_size == 3 &&
         pool_stride == 2 && Cout % 16 == 0 && Cout >= 16 && Cout <= 96;
}

int launch_conv_pool_simt(const float* x, const float* w, const float* bias, const float* scale,
                          const float* shift, float* y, int B, int H, int W, int Cout, int ksize,
                          int conv_padding, int relu, int pool_padding, cudaStream_t stream) {
  if (!conv_pool_simt_eligible(3, Cout, ksize, 2, 3, 2))
    return fail(SQDET_ERR_UNSUPPORTED, "conv+pool fusion: unsupported shape");
  const Geom ch = tf_geometry(H, ksize, 2, conv_padding), cw = tf_geometry(W, ksize, 2, conv_padding);
  if (ch.out <= 0 || cw.out <= 0) return fail(SQDET_ERR_INVALID_ARG, "conv+pool: empty conv output");
  const Geom ph = tf_geometry(ch.out, 3, 2, pool_padding), pw = tf_geometry(cw.out, 3, 2, pool_padding);
  if (ph.out <= 0 || pw.out <= 0) return fail(SQDET_ERR_INVALID_ARG, "conv+pool: empty pooled output");
  ConvPoolParams p;
  p.x = x; p.w = w; p.bias = bias; p.scale = scale; p.shift = shift; p.y = y;
  p.B = B; p.H = H; p.W = W; p.Cout = Cout;
  p.Hc = ch.out; p.Wc = cw.out; p.Hp = ph.out; p.Wp = pw.out;
  p.cpad_t = ch.pad_before; p.cpad_l = cw.pad_before;
  p.ppad_t = ph.pad_before; p.ppad_l = pw.pad_before;
  p.relu = relu;
  p.tiles_h = (p.Hp + PT_H - 1) / PT_H;
  p.tiles_w = (p.Wp + PT_W - 1) / PT_W;
  const unsigned grid = (unsigned)(B * p.tiles_h * p.tiles_w);
  const int threads = 64 * (Cout / 16);
  const size_t smem = ksize == 3 ? smem_bytes_for<3>(Cout) : smem_bytes_for<7>(Cout);
  if (smem > 232448) return fail(SQDET_ERR_UNSUPPORTED, "conv+pool: tile does not fit in smem");
#define SQ_LAUNCH_CP(KS_, NT_, MINB_)                                                          \
  do {                                                                                         \
    /* the opt-in is per device: remember which devices of this process already have it */    \
    static unsigned long long attr_devs = 0ull;                                                \
    int dev_ = 0;                                                                              \
    SQ_CUDA(cudaGetDevice(&dev_));                                                             \
    if (dev_ >= 64 || !((attr_devs >> dev_) & 1ull)) {                                         \
      SQ_CUDA(cudaFuncSetAttribute(conv_pool_simt_kernel<KS_, NT_, MINB_>,                     \
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));      \
      if (dev_ < 64) attr_devs |= 1ull << dev_;                                                \
    }                                                                                          \
    SQ_CUDA(launch_kernel(conv_pool_simt_kernel<KS_, NT_, MINB_>, grid, dim3(NT_), smem, stream, \
                          p));                                                               \
  } while (0)
  if (ksize == 3 && threads <= 256) SQ_LAUNCH_CP(3, 256, 2);
  else if (ksize == 3) SQ_LAUNCH_CP(3, 384, 1);
  else if (threads <= 256) SQ_LAUNCH_CP(7, 256, 1);
  else SQ_LAUNCH_CP(7, 384, 1);
#undef SQ_LAUNCH_CP
  SQ_CHECK_LAUNCH("conv_pool_simt_kernel");
  return SQDET_OK;
}

}  // namespace sqdet
