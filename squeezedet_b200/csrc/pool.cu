// NHWC max-pool and residual add+relu: pure-bandwidth kernels, 128-bit vectorised.
//
// Replaces tf.nn.max_pool (reference src/nn_skeleton.py:580-583; SAME never reads the
// padding: out-of-image taps are skipped, which equals a -inf pad) and
// tf.nn.relu(a + b) (src/nets/resnet50_convDet.py:55).
// Roofline: HBM.  Algorithmic bytes = 4*(B*H*W*C + B*Ho*Wo*C); each input element is
// read ~(k/stride)^2 times but the re-reads hit L1/L2 (adjacent threads share rows).
#include <math_constants.h>
#include <stdlib.h>
#include "common.cuh"

namespace sqdet {
namespace {

__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

// One thread = one output pixel x 4 channels.
__global__ void __launch_bounds__(256)
maxpool_vec4_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W,
                    int C4, int k, int stride, int pad_t, int pad_l, int Ho, int Wo) {
  const long long total = (long long)B * Ho * Wo * C4;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(idx % C4);
    long long t = idx / C4;
    const int ow = (int)(t % Wo);
    t /= Wo;
    const int oh = (int)(t % Ho);
    const int n = (int)(t / Ho);
    const int iy0 = oh * stride - pad_t, ix0 = ow * stride - pad_l;
    float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
    const float4* xin = reinterpret_cast<const float4*>(x) + (long long)n * H * W * C4;
    for (int u = 0; u < k; ++u) {
      const int iy = iy0 + u;
      if (iy < 0 || iy >= H) continue;
      for (int v = 0; v < k; ++v) {
        const int ix = ix0 + v;
        if (ix < 0 || ix >= W) continue;
        const float4 q = __ldg(xin + ((long long)iy * W + ix) * C4 + c4);
        m.x = fmaxf(m.x, q.x); m.y = fmaxf(m.y, q.y);
        m.z = fmaxf(m.z, q.z); m.w = fmaxf(m.w, q.w);
      }
    }
    reinterpret_cast<float4*>(y)[idx] = m;
  }
}

// Stride-2 windows of 2x2 or 3x3 (every pool of the four nets): all K*K loads of a thread are
// issued before the first max (addresses clamped into the image, out-of-image taps replaced by -inf
// afterwards), 32-bit index arithmetic.  The generic kernel below branches around each tap, which
// serialises its loads (pool3: 3.39 TB/s -> see profiles/r2_pool.txt).
template <int K>
__global__ void __launch_bounds__(256)
maxpool_s2_vec4_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W,
                       int C4, int pad_t, int pad_l, int Ho, int Wo) {
  const int total = B * Ho * Wo * C4;
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int c4 = idx % C4;
    int t = idx / C4;
    const int ow = t % Wo;
    t /= Wo;
    const int oh = t % Ho;
    const int n = t / Ho;
    const int iy0 = oh * 2 - pad_t, ix0 = ow * 2 - pad_l;
    const int base = n * H * W;
    float4 q[K * K];
#pragma unroll
    for (int u = 0; u < K; ++u) {
      const int iy = min(max(iy0 + u, 0), H - 1);
#pragma unroll
      for (int v = 0; v < K; ++v) {
        const int ix = min(max(ix0 + v, 0), W - 1);
        q[u * K + v] = __ldg(x4 + (size_t)(base + iy * W + ix) * C4 + c4);
      }
    }
    float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
    for (int u = 0; u < K; ++u)
#pragma unroll
      for (int v = 0; v < K; ++v) {
        const bool ok = (unsigned)(iy0 + u) < (unsigned)H && (unsigned)(ix0 + v) < (unsigned)W;
        const float4 r = q[u * K + v];
        if (ok) {
          m.x = fmaxf(m.x, r.x); m.y = fmaxf(m.y, r.y);
          m.z = fmaxf(m.z, r.z); m.w = fmaxf(m.w, r.w);
        }
      }
    reinterpret_cast<float4*>(y)[idx] = m;
  }
}

__global__ void __launch_bounds__(256)
maxpool_scalar_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W,
                      int C, int k, int stride, int pad_t, int pad_l, int Ho, int Wo) {
  const long long total = (long long)B * Ho * Wo * C;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    long long t = idx / C;
    const int ow = (int)(t % Wo);
    t /= Wo;
    const int oh = (int)(t % Ho);
    const int n = (int)(t / Ho);
    const int iy0 = oh * stride - pad_t, ix0 = ow * stride - pad_l;
    float m = -CUDART_INF_F;
    for (int u = 0; u < k; ++u) {
      const int iy = iy0 + u;
      if (iy < 0 || iy >= H) continue;
      for (int v = 0; v < k; ++v) {
        const int ix = ix0 + v;
        if (ix < 0 || ix >= W) continue;
        m = fmaxf(m, __ldg(x + (((long long)n * H + iy) * W + ix) * C + c));
      }
    }
    y[idx] = m;
  }
}

__global__ void __launch_bounds__(256)
add_relu_kernel(const float* __restrict__ a, const float* __restrict__ b,
                float* __restrict__ y, long long n4, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) {
    const float4 p = ld_stream(reinterpret_cast<const float4*>(a) + i);
    const float4 q = ld_stream(reinterpret_cast<const float4*>(b) + i);
    float4 r;
    r.x = fmaxf(p.x + q.x, 0.f); r.y = fmaxf(p.y + q.y, 0.f);
    r.z = fmaxf(p.z + q.z, 0.f); r.w = fmaxf(p.w + q.w, 0.f);
    reinterpret_cast<float4*>(y)[i] = r;
  }
  if (i == 0) {  // tail (n not a multiple of 4)
    for (long long j = n4 * 4; j < n; ++j) y[j] = fmaxf(a[j] + b[j], 0.f);
  }
}

// uint8 BGR -> fp32, minus the per-channel mean: float32(double(u8) - mean), the value the
// reference feeds (src/demo.py:187-190: float32 image, float64 BGR_MEANS, cast at the feed).
// One thread = 4 pixels = 12 input bytes = three 128-bit output stores.
__global__ void __launch_bounds__(256)
u8_meansub_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, long long n_quads,
                  long long n_pixels, double m0, double m1, double m2) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_quads) return;
  const double mean[3] = {m0, m1, m2};
  if ((q + 1) * 4 <= n_pixels) {
    const uint3 w = *reinterpret_cast<const uint3*>(src + q * 12);     // 12 bytes, 4-aligned
    const unsigned words[3] = {w.x, w.y, w.z};
    float o[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const unsigned b = (words[i >> 2] >> (8 * (i & 3))) & 0xffu;
      o[i] = (float)((double)b - mean[i % 3]);
    }
    float4* d = reinterpret_cast<float4*>(dst + q * 12);
    d[0] = make_float4(o[0], o[1], o[2], o[3]);
    d[1] = make_float4(o[4], o[5], o[6], o[7]);
    d[2] = make_float4(o[8], o[9], o[10], o[11]);
  } else {
    for (long long px = q * 4; px < n_pixels; ++px)
      for (int c = 0; c < 3; ++c)
        dst[px * 3 + c] = (float)((double)src[px * 3 + c] - mean[c]);
  }
}

// uint8 BGR [H0, W0, 3] -> fp32 [H, W, 3]: cv2.resize (float32, INTER_LINEAR) and the mean
// subtraction, in the reference's two orders (src/demo.py:187-190: resize, then `- BGR_MEANS`
// in float64; src/dataset/imdb.py:87-91: float32 `-= BGR_MEANS`, then resize).  Restates
// oracle/preproc.py operation for operation (double sampling position, float32 weight, clamps,
// horizontal pass then vertical pass, round-to-nearest multiplies and adds, no contraction).
// One thread = one output pixel (3 channels); the 4 taps are 12 byte loads served by L1.
__global__ void __launch_bounds__(256)
resize_meansub_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, int H0, int W0,
                         int H, int W, double scale_x, double scale_y, double m0, double m1,
                         double m2, int sub_first) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)H * W) return;
  const int dx = (int)(idx % W), dy = (int)(idx / W);
  const double mean[3] = {m0, m1, m2};
  int sx, sx1, y0, y1;
  float fx, fy;
  bool x_edge = false;
  if (W == W0 && H == H0) {                    // cv2.resize returns a copy for equal sizes
    sx = sx1 = dx; y0 = y1 = dy; fx = 0.f; fy = 0.f; x_edge = true;
  } else {
    // explicit round-to-nearest ops: an FMA contraction here could move a sampling position
    // across an integer relative to the restatement
    const double px = __dsub_rn(__dmul_rn(__dadd_rn((double)dx, 0.5), scale_x), 0.5);
    const double py = __dsub_rn(__dmul_rn(__dadd_rn((double)dy, 0.5), scale_y), 0.5);
    const double flx = floor(px), fly = floor(py);
    sx = (int)flx;
    fx = (float)(px - flx);
    if (sx < 0) { sx = 0; fx = 0.f; }
    if (sx >= W0 - 1) { sx = W0 - 1; fx = 0.f; x_edge = true; }
    sx1 = min(sx + 1, W0 - 1);
    const int sy = (int)fly;
    fy = (float)(py - fly);
    y0 = min(max(sy, 0), H0 - 1);
    y1 = min(max(sy + 1, 0), H0 - 1);
  }
  const float a0 = __fsub_rn(1.f, fx), a1 = fx, b0 = __fsub_rn(1.f, fy), b1 = fy;
  const bool same = (W == W0 && H == H0);
  float o[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float t[2][2];
    const int ys[2] = {y0, y1}, xs[2] = {sx, sx1};
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const float v = (float)src[((long long)ys[r] * W0 + xs[q]) * 3 + c];
        t[r][q] = sub_first ? (float)((double)v - mean[c]) : v;
      }
    float row[2];
#pragma unroll
    for (int r = 0; r < 2; ++r)
      row[r] = x_edge ? t[r][0] : __fadd_rn(__fmul_rn(t[r][0], a0), __fmul_rn(t[r][1], a1));
    const float v = same ? row[0] : __fadd_rn(__fmul_rn(row[0], b0), __fmul_rn(row[1], b1));
    o[c] = sub_first ? v : (float)((double)v - mean[c]);
  }
  float* d = dst + idx * 3;
  d[0] = o[0]; d[1] = o[1]; d[2] = o[2];
}

}  // namespace

int launch_resize_meansub_u8(const uint8_t* src, int H0, int W0, float* dst, int H, int W,
                             double m0, double m1, double m2, int sub_first, cudaStream_t stream) {
  if (H0 <= 0 || W0 <= 0 || H <= 0 || W <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "resize_meansub_u8: non-positive image size");
  // cv::resize: inv_scale = dst / src, scale = 1 / inv_scale (both double)
  const double scale_x = 1.0 / ((double)W / (double)W0);
  const double scale_y = 1.0 / ((double)H / (double)H0);
  const long long n = (long long)H * W;
  resize_meansub_u8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(
      src, dst, H0, W0, H, W, scale_x, scale_y, m0, m1, m2, sub_first);
  SQ_CHECK_LAUNCH("resize_meansub_u8_kernel");
  return SQDET_OK;
}

int launch_u8_meansub(const uint8_t* src, float* dst, int64_t n_pixels, double m0, double m1,
                      double m2, cudaStream_t stream) {
  if (n_pixels <= 0) return fail(SQDET_ERR_INVALID_ARG, "u8_meansub: empty image");
  const long long quads = (n_pixels + 3) / 4;
  u8_meansub_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, stream>>>(src, dst, quads, n_pixels,
                                                                         m0, m1, m2);
  SQ_CHECK_LAUNCH("u8_meansub_kernel");
  return SQDET_OK;
}

int launch_maxpool(const float* x, float* y, int B, int H, int W, int C, int size,
                   int stride, int padding, cudaStream_t stream) {
  if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || size <= 0 || stride <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "maxpool: non-positive dimension");
  const Geom gh = tf_geometry(H, size, stride, padding);
  const Geom gw = tf_geometry(W, size, stride, padding);
  if (gh.out <= 0 || gw.out <= 0) return fail(SQDET_ERR_INVALID_ARG, "maxpool: empty output");
  const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(y) & 15) == 0);
  const long long total = (long long)B * gh.out * gw.out * (vec ? C / 4 : C);
  long long blocks = (total + 255) / 256;
  const long long cap = 148LL * 8 * 16;   // grid-stride beyond 16 waves of 8 CTAs/SM
  if (blocks > cap) blocks = cap;
  const long long in_elems = (long long)B * H * W * (C / 4);
  if (vec && stride == 2 && (size == 2 || size == 3) && total < (1LL << 30) &&
      in_elems < (1LL << 30)) {
    if (size == 3)
      SQ_CUDA(launch_kernel(maxpool_s2_vec4_kernel<3>, dim3((unsigned)blocks), dim3(256), 0, stream, x, y,
                            B, H, W, C / 4, gh.pad_before, gw.pad_before, gh.out, gw.out));
    else
      SQ_CUDA(launch_kernel(maxpool_s2_vec4_kernel<2>, dim3((unsigned)blocks), dim3(256), 0, stream, x, y,
                            B, H, W, C / 4, gh.pad_before, gw.pad_before, gh.out, gw.out));
  } else if (vec)
    SQ_CUDA(launch_kernel(maxpool_vec4_kernel, dim3((unsigned)blocks), dim3(256), 0, stream,
                          x, y, B, H, W, C / 4, size, stride, gh.pad_before, gw.pad_before, gh.out, gw.out));
  else
    SQ_CUDA(launch_kernel(maxpool_scalar_kernel, dim3((unsigned)blocks), dim3(256), 0, stream,
                          x, y, B, H, W, C, size, stride, gh.pad_before, gw.pad_before, gh.out, gw.out));
  SQ_CHECK_LAUNCH("maxpool_kernel");
  return SQDET_OK;
}

int launch_add_relu(const float* a, const float* b, float* y, int64_t n, cudaStream_t stream) {
  if (n <= 0) return fail(SQDET_ERR_INVALID_ARG, "add_relu: empty tensor");
  const bool aligned = (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
                          reinterpret_cast<uintptr_t>(y)) & 15) == 0);
  const long long n4 = aligned ? n / 4 : 0;
  long long threads = n4 > 0 ? n4 : 1;
  SQ_CUDA(launch_kernel(add_relu_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, stream, a, b, y, n4, n));
  SQ_CHECK_LAUNCH("add_relu_kernel");
  return SQDET_OK;
}

}  // namespace sqdet
