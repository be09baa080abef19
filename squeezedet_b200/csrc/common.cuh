// Shared declarations for libsqdet_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string>
#include "../../include/sqdet_b200.h"

namespace sqdet {

// ---- error plumbing (nothing throws across the C ABI) ---------------------------------
void set_error(const std::string& msg);
int  fail(int code, const std::string& msg);
int  cuda_fail(cudaError_t err, const char* what);

#define SQ_CUDA(expr)                                                   \
  do {                                                                  \
    cudaError_t _e = (expr);                                            \
    if (_e != cudaSuccess) return ::sqdet::cuda_fail(_e, #expr);        \
  } while (0)

#define SQ_CHECK_LAUNCH(what)                                           \
  do {                                                                  \
    cudaError_t _e = cudaGetLastError();                                \
    if (_e != cudaSuccess) return ::sqdet::cuda_fail(_e, what);         \
  } while (0)


// ---- environment switches (INTEGRATION.md §5) ---------------------------------------------
// Every SQDET_* variable the library reads goes through these, as the initializer of a
// function-local `static const`: read once, on first use, thread-safe.
inline const char* env_str(const char* name) { return getenv(name); }
inline int env_int(const char* name, int dflt) {
  const char* a = env_str(name);
  return a ? atoi(a) : dflt;
}
inline float env_float(const char* name, float dflt) {
  const char* a = env_str(name);
  return a ? (float)atof(a) : dflt;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                 cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- TF NHWC geometry (SURVEY App. A.1; tf.nn.conv2d / tf.nn.max_pool) ------------------
struct Geom {
  int out, pad_before, pad_after;
};
inline Geom tf_geometry(int in, int k, int stride, int padding) {
  Geom g;
  if (padding == SQDET_PAD_SAME) {
    g.out = (in + stride - 1) / stride;
    int total = (g.out - 1) * stride + k - in;
    if (total < 0) total = 0;
    g.pad_before = total / 2;
    g.pad_after = total - g.pad_before;
  } else {
    g.out = (in - k) / stride + 1;
    g.pad_before = g.pad_after = 0;
  }
  return g;
}

// ---- kernel launchers (each returns a status; asynchronous on `stream`) ----------------
struct ConvArgs {
  const float* x;       // [B,H,W,Cin]
  const float* w;       // [kh,kw,Cin,Cout] (HWIO)
  const float* bias;    // [Cout] or null
  const float* scale;   // [Cout] or null   (frozen BN: rsqrt(var+eps)*gamma)
  const float* shift;   // [Cout] or null   (beta - mean*scale)
  float* y;             // [B,Ho,Wo,y_cstride], this conv owns channels [y_coff, y_coff+Cout)
  int B, H, W, Cin, Cout, size, stride, padding, relu, y_cstride, y_coff;
};
int launch_conv_simt(const ConvArgs& a, cudaStream_t stream);

bool conv_pool_simt_eligible(int Cin, int Cout, int ksize, int stride, int pool_size,
                             int pool_stride);
int launch_conv_pool_simt(const float* x, const float* w, const float* bias, const float* scale,
                          const float* shift, float* y, int B, int H, int W, int Cout, int ksize,
                          int conv_padding, int relu, int pool_padding, cudaStream_t stream);

int launch_maxpool(const float* x, float* y, int B, int H, int W, int C, int size,
                   int stride, int padding, cudaStream_t stream);
int launch_resize_meansub_u8(const uint8_t* src, int H0, int W0, float* dst, int H, int W,
                             double m0, double m1, double m2, int sub_first, cudaStream_t stream);
int launch_u8_meansub(const uint8_t* src, float* dst, int64_t n_pixels, double m0, double m1,
                      double m2, cudaStream_t stream);
int launch_add_relu(const float* a, const float* b, float* y, int64_t n, cudaStream_t stream);

int launch_interpret(const float* preds, const float* anchors, float* boxes, float* probs,
                     int64_t* cls, int B, int grid_h, int grid_w, int K, int C,
                     int image_width, int image_height, float exp_thresh,
                     cudaStream_t stream);
int launch_rescale_boxes(float* boxes, const float* scales_xy, int B, int A, cudaStream_t stream);
int launch_topk_nms(const float* boxes, const float* probs, const int64_t* cls, int B,
                    int A, int classes, int top_n, float prob_thresh, float nms_thresh,
                    sqdet_det* dets, int32_t* counts, int max_dets, cudaStream_t stream);

}  // namespace sqdet
