// tcgen05 (5th-gen tensor core) convolution path: plans, weight packing, launchers.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sqdet {

// One convolution executed as an implicit GEMM on tcgen05 with the 3xTF32 split.
struct TcConvPlan {
  bool enabled = false;
  int B = 0, H = 0, W = 0, Cin = 0, Cout = 0, size = 1, stride = 1, relu = 1;
  int Ho = 0, Wo = 0, pad_t = 0, pad_l = 0;
  int y_cstride = 0, y_coff = 0;
  int launches = 1;              // 2 when the conv runs as split-K partials + reduction
  void* impl = nullptr;          // opaque device/host state (tensor maps, packed weights)
};

// The expand pair of a fire module (1x1 || 3x3 on the same squeeze tensor) fused into
// one kernel writing the channel-concatenated output.
struct TcFirePlan {
  bool enabled = false;
  int B = 0, H = 0, W = 0, S = 0, E1 = 0, E3 = 0;
  void* impl = nullptr;
};

bool tc_conv_eligible(int Cin, int Cout, int size, int stride, int padding, int y_cstride,
                      int y_coff);

// Returns 1 when the shape is taken by the tensor-core path (plan->enabled), 0 when it is
// left to the fp32 SIMT kernel, negative on error.
int tc_conv_plan(TcConvPlan* plan, int B, int H, int W, int Cin, int Cout, int size, int stride,
                 int padding, int relu, bool has_affine, int y_cstride, int y_coff,
                 const float* x_dev, float* y_dev);
int tc_fire_plan(TcFirePlan* plan, int B, int H, int W, int S, int E1, int E3,
                 const float* q_dev, float* y_dev);
int tc_conv_pack_weights(TcConvPlan* plan, const float* w_hwio, const float* bias);
int tc_conv_set_affine(TcConvPlan* plan, const float* scale, const float* shift);
int tc_fire_pack_weights(TcFirePlan* plan, const float* w_e1, const float* b_e1,
                         const float* w_e3, const float* b_e3);
int launch_conv_tc(const TcConvPlan& plan, const float* x_dev, float* y_dev, cudaStream_t stream);
int launch_fire_expand_tc(const TcFirePlan& plan, const float* q_dev, float* y_dev,
                          cudaStream_t stream);
void tc_conv_release(TcConvPlan* plan);
void tc_fire_release(TcFirePlan* plan);

// Tensor-map encoders shared by the tensor-core kernels: NHWC fp32 activation, box
// {KC ch, box_w, box_h, 1}, 128B (KC=32) / 64B (KC=16) swizzle; packed weight rows [rows][KC], box
// {KC, N}.  Return SQDET_OK or a negative status.
int tc_encode_act_map(CUtensorMap* map, const float* x, int B, int H, int W, int C, int KC,
                      int box_w, int box_h);
int tc_encode_w_map(CUtensorMap* map, const float* w, int rows, int KC, int N);
// a whole tensor as a 1-D array of floats, box = `box` floats (no swizzle)
int tc_encode_flat_map(CUtensorMap* map, const float* x, long long n, int box);

// Stage-isolated entry (sqdet_conv2d with SQDET_MATH_TF32X3_TC): plans, packs from device
// weights, launches, and releases; synchronises the stream (test/debug path, not the hot path).
int conv2d_tc_oneshot(const float* x_dev, const float* w_hwio_dev, const float* bias_dev,
                      const float* scale_dev, const float* shift_dev, float* y_dev, int B, int H,
                      int W, int Cin, int Cout, int size, int stride, int padding, int relu,
                      int y_cstride, int y_coff, cudaStream_t stream);

}  // namespace sqdet
