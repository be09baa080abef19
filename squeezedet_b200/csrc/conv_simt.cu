// fp32 FFMA implicit-GEMM convolution (SQDET_MATH_FP32_SIMT).
//
// Replaces tf.nn.conv2d + tf.nn.bias_add [+ tf.nn.batch_normalization] + tf.nn.relu
// (reference src/nn_skeleton.py:539-547, :441-449).  Handles every shape the four
// nets use (any k, stride, SAME/VALID, Cin incl. 3, strided channel-offset output for
// the fire concat).  It is the kernel for conv1 (Cin = 3: K = 27/147 is too thin for
// a tensor-core tile) and the on-device fp32 cross-check of the tcgen05 path.
//
// GEMM view: M = B*Ho*Wo output pixels, N = Cout, K = kh*kw*Cin ordered (u, v, c) —
// the row order of the HWIO weight tensor viewed as [K, Cout].
// CTA tile 64 x 64, K step 16, 256 threads, 4 x 4 outputs per thread.
#include "common.cuh"

namespace sqdet {
namespace {

constexpr int BM = 64, BN = 64, BK = 16, NT = 256;

template <bool VEC4>
__global__ void __launch_bounds__(NT)
conv_simt_kernel(const float* __restrict__ x, const float* __restrict__ w,
                 const float* __restrict__ bias, const float* __restrict__ scale,
                 const float* __restrict__ shift, float* __restrict__ y,
                 int B, int H, int W, int Cin, int Cout, int ksz, int stride,
                 int pad_t, int pad_l, int Ho, int Wo, int relu, int y_cstride,
                 int y_coff) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN];

  const int tid = threadIdx.x;
  const long long M = (long long)B * Ho * Wo;
  const int K = ksz * ksz * Cin;
  const long long m0 = (long long)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;

  // A-load role: this thread owns pixel (tid % 64) and k-quad (tid / 64).
  const int am = tid & 63;
  const int akq = tid >> 6;          // 0..3 -> k offsets akq*4 .. akq*4+3
  const long long mg = m0 + am;
  const bool m_ok = mg < M;
  int pn = 0, ph = 0, pw = 0;
  if (m_ok) {
    pw = (int)(mg % Wo);
    long long t = mg / Wo;
    ph = (int)(t % Ho);
    pn = (int)(t / Ho);
  }
  const int iy0 = ph * stride - pad_t;
  const int ix0 = pw * stride - pad_l;
  const float* xin = x + (long long)pn * H * W * Cin;

  // B-load role: row (tid / 16), 4 columns at (tid % 16) * 4.
  const int bk = tid >> 4;
  const int bn = (tid & 15) * 4;

  // compute role
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
    // ---- stage A (on-the-fly im2col) ----
    {
      const int kb = k0 + akq * 4;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (VEC4) {
        // Cin % 4 == 0: the 4 consecutive k share one tap and are contiguous in c.
        if (m_ok && kb < K) {
          const int tap = kb / Cin, c = kb - tap * Cin;
          const int u = tap / ksz, vv = tap - u * ksz;
          const int iy = iy0 + u, ix = ix0 + vv;
          if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
            const float4 q = *reinterpret_cast<const float4*>(
                xin + ((long long)iy * W + ix) * Cin + c);
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int k = kb + e;
          if (m_ok && k < K) {
            const int tap = k / Cin, c = k - tap * Cin;
            const int u = tap / ksz, vv = tap - u * ksz;
            const int iy = iy0 + u, ix = ix0 + vv;
            if (iy >= 0 && iy < H && ix >= 0 && ix < W)
              v[e] = __ldg(xin + ((long long)iy * W + ix) * Cin + c);
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) As[akq * 4 + e][am] = v[e];
    }
    // ---- stage B (weights [K, Cout]) ----
    {
      const int k = k0 + bk;
      float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k < K) {
        const float* wr = w + (long long)k * Cout + n0 + bn;
        if (VEC4 && (n0 + bn + 3 < Cout)) {
          q = *reinterpret_cast<const float4*>(wr);
        } else {
          if (n0 + bn + 0 < Cout) q.x = __ldg(wr + 0);
          if (n0 + bn + 1 < Cout) q.y = __ldg(wr + 1);
          if (n0 + bn + 2 < Cout) q.z = __ldg(wr + 2);
          if (n0 + bn + 3 < Cout) q.w = __ldg(wr + 3);
        }
      }
      *reinterpret_cast<float4*>(&Bs[bk][bn]) = q;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

  // ---- epilogue: bias, optional affine (frozen BN), relu, strided channel store ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
    float* yr = y + m * y_cstride + y_coff;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= Cout) continue;
      float v = acc[i][j];
      if (bias) v += __ldg(bias + n);
      if (scale) v = v * __ldg(scale + n) + __ldg(shift + n);
      if (relu) v = fmaxf(v, 0.f);
      yr[n] = v;
    }
  }
}

}  // namespace

int launch_conv_simt(const ConvArgs& a, cudaStream_t stream) {
  if (a.B <= 0 || a.H <= 0 || a.W <= 0 || a.Cin <= 0 || a.Cout <= 0 || a.size <= 0 ||
      a.stride <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "conv: non-positive dimension");
  if ((a.scale == nullptr) != (a.shift == nullptr))
    return fail(SQDET_ERR_INVALID_ARG, "conv: scale and shift must be given together");
  const Geom gh = tf_geometry(a.H, a.size, a.stride, a.padding);
  const Geom gw = tf_geometry(a.W, a.size, a.stride, a.padding);
  if (gh.out <= 0 || gw.out <= 0) return fail(SQDET_ERR_INVALID_ARG, "conv: empty output");
  if (a.y_coff < 0 || a.y_coff + a.Cout > a.y_cstride)
    return fail(SQDET_ERR_INVALID_ARG, "conv: output channel window out of range");
  const long long M = (long long)a.B * gh.out * gw.out;
  dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((a.Cout + BN - 1) / BN));
  const bool vec4 = (a.Cin % 4 == 0) && (a.Cout % 4 == 0) &&
                    ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(a.w) & 15) == 0);
  if (vec4)
    SQ_CUDA(launch_kernel(conv_simt_kernel<true>, grid, dim3(NT), 0, stream,
                          a.x, a.w, a.bias, a.scale, a.shift, a.y, a.B, a.H, a.W, a.Cin, a.Cout, a.size,
                          a.stride, gh.pad_before, gw.pad_before, gh.out, gw.out, a.relu, a.y_cstride,
                          a.y_coff));
  else
    SQ_CUDA(launch_kernel(conv_simt_kernel<false>, grid, dim3(NT), 0, stream,
                          a.x, a.w, a.bias, a.scale, a.shift, a.y, a.B, a.H, a.W, a.Cin, a.Cout, a.size,
                          a.stride, gh.pad_before, gw.pad_before, gh.out, gw.out, a.relu, a.y_cstride,
                          a.y_coff));
  SQ_CHECK_LAUNCH("conv_simt_kernel");
  return SQDET_OK;
}

}  // namespace sqdet
