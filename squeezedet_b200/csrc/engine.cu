// libsqdet_b200 engine: graph builder, parameter store, executor and the C ABI.
//
// The reference's "framework" for this path is the TF-1.0 graph that the nets build
// through ModelSkeleton's layer constructors and run through sess.run
// (src/nn_skeleton.py:74-135, 374-586; src/nets/*.py; src/demo.py:193-199).  Here the
// Python facade records the same constructor calls into a plan (sqdet_add_*), and this
// file owns everything behind it: shape inference with TF geometry, activation and
// weight storage in HBM, BN folding to (scale, shift), kernel selection per op
// (tcgen05 3xTF32 implicit GEMM or fp32 SIMT), CUDA-graph capture of the whole forward,
// and the fused post-processing.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"
#include "fire_tc.cuh"
#include "first_tc.cuh"

namespace sqdet {

// ---------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
int cuda_fail(cudaError_t err, const char* what) {
  g_last_error = std::string("CUDA error: ") + cudaGetErrorString(err) + " in " + what;
  return SQDET_ERR_CUDA;
}

// ---------------------------------------------------------------------------------------
struct Tensor {
  std::string name;
  int B = 0, H = 0, W = 0, C = 0;
  float* dev = nullptr;         // owned (except tensor 0 when the caller feeds its own)
  bool external = false;
  bool materialized = true;     // false: produced and consumed inside a fused kernel only
  int64_t numel() const { return (int64_t)B * H * W * C; }
};

struct Param {
  std::string name;
  std::vector<int64_t> shape;
  std::vector<float> host;
  float* dev = nullptr;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

enum OpKind { OP_CONV, OP_POOL, OP_FIRE, OP_ADD_RELU };

struct ConvSpec {
  std::string name;
  int src = -1, dst = -1;
  int Cin = 0, Cout = 0, size = 1, stride = 1, padding = SQDET_PAD_SAME, relu = 1;
  int y_coff = 0;
  int p_kernel = -1, p_bias = -1, p_gamma = -1, p_beta = -1, p_mean = -1, p_var = -1;
  float* scale = nullptr;      // device, BN only
  float* shift = nullptr;
  TcConvPlan tc;               // tensor-core plan (valid when tc.enabled)
};

struct Op {
  OpKind kind;
  std::string name;
  std::vector<ConvSpec> convs;   // 1 for conv, 3 for fire (squeeze, expand1x1, expand3x3)
  int src = -1, src2 = -1, dst = -1;
  int size = 0, stride = 0, padding = 0;
  int64_t flops = 0, params = 0, min_bytes = 0;
  int launches = 0;
  TcFirePlan tcfire;             // fused expand pair (valid when tcfire.enabled)
  FusedFirePlan fused;           // whole fire module in one kernel (valid when fused.enabled)
  FirstTcPlan first_tc;          // first layer conv+pool on tcgen05 (valid when first_tc.enabled)
  bool skip = false;             // pool op whose work happens in the producer's epilogue
  int fused_pool_op = -1;        // index of the pool op fused into this first layer
  bool first_layer_fused = false;  // Cin=3 stride-2 conv + 3x3/2 pool as one FFMA kernel
  int out = -1;                  // tensor actually written (dst, or the fused pool's dst)
};

}  // namespace sqdet

using namespace sqdet;

struct sqdet_engine {
  sqdet_config cfg;
  int device = 0;
  bool finalized = false;
  bool params_dirty = true;
  std::vector<Tensor> tensors;
  std::vector<Param> params;
  std::map<std::string, int> param_index;
  std::vector<Op> ops;
  int preds = -1;
  int grid_h = 0, grid_w = 0;
  int64_t num_anchors = 0;
  std::vector<double> anchors_f64;
  float* d_anchors = nullptr;
  float* d_boxes = nullptr;
  float* d_probs = nullptr;
  int64_t* d_cls = nullptr;
  sqdet_det* d_dets = nullptr;
  int32_t* d_counts = nullptr;
  int max_dets = 0;
  float* d_input = nullptr;       // engine-owned input buffer (host-path + graph)
  // CUDA graphs of one forward, keyed by (input pointer, stream); small LRU-less cache
  struct GraphEntry {
    cudaGraphExec_t exec = nullptr;
    const float* input = nullptr;
    cudaStream_t stream = nullptr;
  };
  GraphEntry graphs[4];
  int graph_next = 0;
  bool use_graph = true;
  // pipelined host path (sqdet_submit / sqdet_wait), depth 2
  cudaStream_t copy_stream = nullptr;
  float* d_in_slot[2] = {nullptr, nullptr};       // slot 0 aliases tensors[0].dev
  uint8_t* d_u8_slot[2] = {nullptr, nullptr};
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr};
  cudaEvent_t ev_done[2] = {nullptr, nullptr};
  bool slot_used[2] = {false, false};
  long long n_submitted = 0, n_waited = 0;
  double bgr_means[3] = {103.939, 116.779, 123.68};   // config.py:72
  cudaStream_t own_stream = nullptr;
  std::vector<cudaEvent_t> prof_events;
  // eval-order rescale (src/eval.py:83-84): det_boxes / (x_scale, y_scale) BEFORE the filter
  float* d_scales = nullptr;      // [2 pipeline slots][B][2] device
  int scale_slot = 0;             // half read by the forward being enqueued
  bool rescale_on = false;
  // variable-size uint8 frames (sqdet_submit_frames): one staging buffer per pipeline slot
  uint8_t* d_frames[2] = {nullptr, nullptr};
  size_t frames_cap[2] = {0, 0};
  // multi-GPU: the ONE collective of the path, ncclAllGather of the result blob
  void* comm = nullptr;           // ncclComm_t
  bool comm_owned = false;
  int comm_nranks = 0, comm_rank = 0;
  uint8_t* d_gathered = nullptr;  // [nranks][blob_bytes]
  size_t blob_bytes = 0;
  bool gather_in_forward = false;
};

namespace sqdet {

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static int add_param(sqdet_engine* e, const std::string& name, std::vector<int64_t> shape) {
  auto it = e->param_index.find(name);
  if (it != e->param_index.end()) return it->second;
  Param p;
  p.name = name;
  p.shape = std::move(shape);
  p.host.assign((size_t)p.numel(), 0.f);
  e->params.push_back(std::move(p));
  const int idx = (int)e->params.size() - 1;
  e->param_index[name] = idx;
  return idx;
}

static int new_tensor(sqdet_engine* e, const std::string& name, int B, int H, int W, int C) {
  Tensor t;
  t.name = name;
  t.B = B; t.H = H; t.W = W; t.C = C;
  e->tensors.push_back(t);
  return (int)e->tensors.size() - 1;
}

static int check_build(sqdet_engine* e, int src) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (e->finalized) return fail(SQDET_ERR_STATE, "graph is frozen (already finalized)");
  if (src < 0 || src >= (int)e->tensors.size())
    return fail(SQDET_ERR_INVALID_ARG, "unknown source tensor id");
  return SQDET_OK;
}

// Describe one convolution reading tensor `src`; output geometry by TF rules.
static int make_conv(sqdet_engine* e, const std::string& name, int src, int filters, int size,
                     int stride, int padding, int relu, bool bn, bool with_bias,
                     ConvSpec* cs, int* Ho, int* Wo) {
  if (filters <= 0 || size <= 0 || stride <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "conv '" + name + "': non-positive filters/size/stride");
  if (padding != SQDET_PAD_SAME && padding != SQDET_PAD_VALID)
    return fail(SQDET_ERR_INVALID_ARG, "conv '" + name + "': padding must be SAME(0) or VALID(1)");
  const Tensor& in = e->tensors[src];
  const Geom gh = tf_geometry(in.H, size, stride, padding);
  const Geom gw = tf_geometry(in.W, size, stride, padding);
  if (gh.out <= 0 || gw.out <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "conv '" + name + "': kernel larger than input");
  cs->name = name;
  cs->src = src;
  cs->Cin = in.C;
  cs->Cout = filters;
  cs->size = size;
  cs->stride = stride;
  cs->padding = padding;
  cs->relu = relu;
  cs->p_kernel = add_param(e, name + "/kernels", {size, size, in.C, filters});
  if (!bn || with_bias) cs->p_bias = add_param(e, name + "/biases", {filters});
  if (bn) {
    // reference order of model_params: kernels, [biases], gamma, beta, mean, var
    cs->p_gamma = add_param(e, name + "/gamma", {filters});
    cs->p_beta = add_param(e, name + "/beta", {filters});
    cs->p_mean = add_param(e, name + "/mean", {filters});
    cs->p_var = add_param(e, name + "/var", {filters});
  }
  *Ho = gh.out;
  *Wo = gw.out;
  return SQDET_OK;
}

static void conv_cost(const sqdet_engine* e, const ConvSpec& c, int Ho, int Wo, Op* op) {
  const Tensor& in = e->tensors[c.src];
  const int64_t px = (int64_t)in.B * Ho * Wo;
  op->flops += 2LL * c.size * c.size * c.Cin * c.Cout * px;
  op->params += (int64_t)(1 + c.size * c.size * c.Cin) * c.Cout;
}

static int run_conv(sqdet_engine* e, const ConvSpec& c, const float* x_override,
                    cudaStream_t stream) {
  const Tensor& in = e->tensors[c.src];
  const Tensor& out = e->tensors[c.dst];
  const float* x = (c.src == 0 && x_override) ? x_override : in.dev;
  if (c.tc.enabled) return launch_conv_tc(c.tc, x, out.dev, stream);
  ConvArgs a;
  a.x = x;
  a.w = e->params[c.p_kernel].dev;
  a.bias = c.p_bias >= 0 ? e->params[c.p_bias].dev : nullptr;
  a.scale = c.scale;
  a.shift = c.shift;
  a.y = out.dev;
  a.B = in.B; a.H = in.H; a.W = in.W; a.Cin = c.Cin; a.Cout = c.Cout;
  a.size = c.size; a.stride = c.stride; a.padding = c.padding; a.relu = c.relu;
  a.y_cstride = out.C;
  a.y_coff = c.y_coff;
  return launch_conv_simt(a, stream);
}

static int run_op(sqdet_engine* e, const Op& op, const float* x_override, cudaStream_t stream) {
  if (op.skip) return SQDET_OK;
  switch (op.kind) {
    case OP_CONV:
      if (op.first_layer_fused) {
        const ConvSpec& c = op.convs[0];
        const Op& po = e->ops[op.fused_pool_op];
        const Tensor& in = e->tensors[c.src];
        const float* x = (c.src == 0 && x_override) ? x_override : in.dev;
        if (op.first_tc.enabled) return launch_first_tc(op.first_tc, x, stream);
        return launch_conv_pool_simt(x, e->params[c.p_kernel].dev,
                                     c.p_bias >= 0 ? e->params[c.p_bias].dev : nullptr, c.scale,
                                     c.shift, e->tensors[op.out].dev, in.B, in.H, in.W, c.Cout,
                                     c.size, c.padding, c.relu, po.padding, stream);
      }
      return run_conv(e, op.convs[0], x_override, stream);
    case OP_FIRE: {
      if (op.fused.enabled) return launch_fused_fire(op.fused, stream);
      int rc = run_conv(e, op.convs[0], x_override, stream);
      if (rc) return rc;
      if (op.tcfire.enabled)
        return launch_fire_expand_tc(op.tcfire, e->tensors[op.convs[1].src].dev,
                                     e->tensors[op.out].dev, stream);
      rc = run_conv(e, op.convs[1], nullptr, stream);
      if (rc) return rc;
      return run_conv(e, op.convs[2], nullptr, stream);
    }
    case OP_POOL: {
      const Tensor& in = e->tensors[op.src];
      const float* x = (op.src == 0 && x_override) ? x_override : in.dev;
      return launch_maxpool(x, e->tensors[op.dst].dev, in.B, in.H, in.W, in.C, op.size,
                            op.stride, op.padding, stream);
    }
    case OP_ADD_RELU: {
      const Tensor& a = e->tensors[op.src];
      return launch_add_relu(a.dev, e->tensors[op.src2].dev, e->tensors[op.dst].dev,
                             a.numel(), stream);
    }
  }
  return fail(SQDET_ERR_STATE, "unknown op kind");
}

// ---- NCCL, bound at run time (dlopen): the library must load on boxes without NCCL ----------
// Prototypes restated from nccl.h (stable since NCCL 2.0); ncclUniqueId is passed BY VALUE.
struct NcclId { char internal[128]; };
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
  if (g_nccl.handle) return SQDET_OK;
  static const char* const env = env_str("SQDET_NCCL_LIB");
  const char* cands[] = {env, "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* c : cands) {
    if (!c || !*c) continue;
    h = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) return fail(SQDET_ERR_UNSUPPORTED, "NCCL not found (set SQDET_NCCL_LIB to libnccl.so.2)");
  NcclApi a;
  a.handle = h;
  a.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
  a.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
  a.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
  a.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
  a.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllGather)
    return fail(SQDET_ERR_UNSUPPORTED, "NCCL library lacks the expected entry points");
  g_nccl = a;
  return SQDET_OK;
}
static int nccl_fail(int r, const char* what) {
  std::string m = std::string("NCCL error in ") + what + ": ";
  m += g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "unknown";
  return fail(SQDET_ERR_CUDA, m);
}

static int run_allgather(sqdet_engine* e, void* comm, cudaStream_t stream) {
  if (!comm) return fail(SQDET_ERR_STATE, "sqdet_allgather: no communicator attached");
  if (!e->d_gathered) return fail(SQDET_ERR_STATE, "sqdet_allgather: gather buffer missing");
  // records and counts are ONE contiguous blob (sqdet_finalize): one collective per step
  const int r = g_nccl.AllGather(e->d_dets, e->d_gathered, e->blob_bytes, /*ncclUint8*/ 1, comm,
                                 stream);
  if (r != 0) return nccl_fail(r, "ncclAllGather");
  return SQDET_OK;
}

static int run_postproc(sqdet_engine* e, cudaStream_t stream) {
  const sqdet_config& c = e->cfg;
  int rc = launch_interpret(e->tensors[e->preds].dev, e->d_anchors, e->d_boxes, e->d_probs,
                            e->d_cls, c.batch_size, e->grid_h, e->grid_w, c.anchors_per_grid,
                            c.classes, c.image_width, c.image_height, c.exp_thresh, stream);
  if (rc) return rc;
  if (e->rescale_on) {
    rc = launch_rescale_boxes(e->d_boxes, e->d_scales + (size_t)e->scale_slot * c.batch_size * 2,
                              c.batch_size, (int)e->num_anchors, stream);
    if (rc) return rc;
  }
  rc = launch_topk_nms(e->d_boxes, e->d_probs, e->d_cls, c.batch_size, (int)e->num_anchors,
                       c.classes, c.top_n_detection, c.prob_thresh, c.nms_thresh, e->d_dets,
                       e->d_counts, e->max_dets, stream);
  if (rc) return rc;
  if (e->gather_in_forward && e->comm) return run_allgather(e, e->comm, stream);
  return SQDET_OK;
}

// Upload parameters and derive what the kernels consume (BN scale/shift, TC packs).
static int prepare_params(sqdet_engine* e) {
  if (!e->params_dirty) return SQDET_OK;
  for (auto& p : e->params) {
    if (!p.dev) SQ_CUDA(cudaMalloc(&p.dev, sizeof(float) * (size_t)p.numel()));
    SQ_CUDA(cudaMemcpy(p.dev, p.host.data(), sizeof(float) * (size_t)p.numel(),
                       cudaMemcpyHostToDevice));
  }
  for (auto& op : e->ops) {
    for (auto& c : op.convs) {
      if (c.p_gamma >= 0) {
        // tf.nn.batch_normalization: inv = rsqrt(var+eps)*gamma; y = x*inv + (beta - mean*inv)
        const int n = c.Cout;
        std::vector<float> sc(n), sh(n);
        const auto& g = e->params[c.p_gamma].host;
        const auto& b = e->params[c.p_beta].host;
        const auto& m = e->params[c.p_mean].host;
        const auto& v = e->params[c.p_var].host;
        for (int i = 0; i < n; ++i) {
          const float inv = (1.0f / sqrtf(v[i] + e->cfg.batch_norm_epsilon)) * g[i];
          sc[i] = inv;
          sh[i] = b[i] - m[i] * inv;
        }
        if (!c.scale) SQ_CUDA(cudaMalloc(&c.scale, sizeof(float) * n));
        if (!c.shift) SQ_CUDA(cudaMalloc(&c.shift, sizeof(float) * n));
        SQ_CUDA(cudaMemcpy(c.scale, sc.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
        SQ_CUDA(cudaMemcpy(c.shift, sh.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
        if (c.tc.enabled) {
          int rc = tc_conv_set_affine(&c.tc, sc.data(), sh.data());
          if (rc) return rc;
        }
        if (op.first_tc.enabled && &c == &op.convs[0]) {
          int rc = first_tc_set_affine(&op.first_tc, sc.data(), sh.data());
          if (rc) return rc;
        }
      }
    }
  }
  // tensor-core weight packs
  for (auto& op : e->ops) {
    if (op.first_tc.enabled) {
      const ConvSpec& c = op.convs[0];
      const float* bias = c.p_bias >= 0 ? e->params[c.p_bias].host.data() : nullptr;
      int rc = first_tc_pack_weights(&op.first_tc, e->params[c.p_kernel].host.data(), bias);
      if (rc) return rc;
    }
    for (auto& c : op.convs) {
      const float* bias = c.p_bias >= 0 ? e->params[c.p_bias].host.data() : nullptr;
      if (!c.tc.enabled) continue;
      int rc = tc_conv_pack_weights(&c.tc, e->params[c.p_kernel].host.data(), bias);
      if (rc) return rc;
    }
    if (op.fused.enabled) {
      const ConvSpec& sq = op.convs[0];
      const ConvSpec& e1 = op.convs[1];
      const ConvSpec& e3 = op.convs[2];
      int rc = fused_fire_pack_weights(&op.fused, e->params[sq.p_kernel].host.data(),
                                       e->params[sq.p_bias].host.data(),
                                       e->params[e1.p_kernel].host.data(),
                                       e->params[e1.p_bias].host.data(),
                                       e->params[e3.p_kernel].host.data(),
                                       e->params[e3.p_bias].host.data());
      if (rc) return rc;
    }
    if (op.tcfire.enabled) {
      const ConvSpec& e1 = op.convs[1];
      const ConvSpec& e3 = op.convs[2];
      int rc = tc_fire_pack_weights(&op.tcfire, e->params[e1.p_kernel].host.data(),
                                    e->params[e1.p_bias].host.data(),
                                    e->params[e3.p_kernel].host.data(),
                                    e->params[e3.p_bias].host.data());
      if (rc) return rc;
    }
  }
  // cudaMemcpy from pageable host memory may return before its DMA has landed, and the forward
  // runs on non-blocking streams that do not wait for the legacy stream: every upload above (and
  // the plan-time ones of sqdet_finalize) must be complete before a kernel reads it
  SQ_CUDA(cudaStreamSynchronize(nullptr));
  e->params_dirty = false;
  // weights changed -> any captured graph still points at the same buffers, so it stays valid
  return SQDET_OK;
}

static void drop_graph(sqdet_engine* e) {
  for (auto& g : e->graphs) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g = sqdet_engine::GraphEntry();
  }
}

static int enqueue_all(sqdet_engine* e, const float* images_dev, cudaStream_t stream) {
  for (const auto& op : e->ops) {
    int rc = run_op(e, op, images_dev, stream);
    if (rc) return rc;
  }
  return run_postproc(e, stream);
}

static int forward_impl(sqdet_engine* e, const float* images_dev, cudaStream_t stream) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_forward before sqdet_finalize");
  if (!images_dev) return fail(SQDET_ERR_INVALID_ARG, "null images pointer");
  DeviceGuard guard(e->device);
  if (!guard.ok) return fail(SQDET_ERR_CUDA, "cannot select the engine's device");
  int rc = prepare_params(e);
  if (rc) return rc;
  e->scale_slot = (e->d_in_slot[1] && images_dev == e->d_in_slot[1]) ? 1 : 0;
  const bool can_graph = e->use_graph && stream != nullptr;   // legacy stream cannot capture
  if (!can_graph) return enqueue_all(e, images_dev, stream);
  sqdet_engine::GraphEntry* hit = nullptr;
  for (auto& g : e->graphs)
    if (g.exec && g.input == images_dev && g.stream == stream) hit = &g;
  if (!hit) {
    sqdet_engine::GraphEntry& slot = e->graphs[e->graph_next];
    e->graph_next = (e->graph_next + 1) % 4;
    if (slot.exec) cudaGraphExecDestroy(slot.exec);
    slot = sqdet_engine::GraphEntry();
    cudaGraph_t graph = nullptr;
    SQ_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    rc = enqueue_all(e, images_dev, stream);
    cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    if (rc) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (ce != cudaSuccess) return cuda_fail(ce, "cudaStreamEndCapture");
    ce = cudaGraphInstantiate(&slot.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return cuda_fail(ce, "cudaGraphInstantiate");
    slot.input = images_dev;
    slot.stream = stream;
    hit = &slot;
  }
  SQ_CUDA(cudaGraphLaunch(hit->exec, stream));
  return SQDET_OK;
}

}  // namespace sqdet

// =========================================================================================
//                                        C ABI
// =========================================================================================
extern "C" {

const char* sqdet_last_error(void) { return g_last_error.c_str(); }
const char* sqdet_version(void) { return "sqdet_b200 0.1 (sm_100a)"; }

int sqdet_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int sqdet_create(const sqdet_config* cfg, int device, sqdet_engine** out) {
  if (!cfg || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_create: null argument");
  if (cfg->batch_size <= 0 || cfg->image_height <= 0 || cfg->image_width <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_create: batch/image size must be positive");
  if (cfg->classes <= 0 || cfg->anchors_per_grid <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_create: classes/anchors_per_grid must be positive");
  if (cfg->math_mode != SQDET_MATH_FP32_SIMT && cfg->math_mode != SQDET_MATH_TF32X3_TC)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_create: unknown math_mode");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess) return cuda_fail(ce, "cudaGetDeviceCount (no CUDA device: this "
                                              "library has no CPU fallback)");
  if (device < 0 || device >= ndev)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_create: device index out of range");
  cudaDeviceProp prop;
  SQ_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(SQDET_ERR_UNSUPPORTED, "sqdet_create: this build targets sm_100a (B200) only");
  std::unique_ptr<sqdet_engine> e(new sqdet_engine());
  e->cfg = *cfg;
  e->device = device;
  new_tensor(e.get(), "image_input", cfg->batch_size, cfg->image_height, cfg->image_width, 3);
  *out = e.release();
  return SQDET_OK;
}

int sqdet_destroy(sqdet_engine* e) {
  if (!e) return SQDET_OK;
  DeviceGuard guard(e->device);
  drop_graph(e);
  for (auto& t : e->tensors)
    if (t.dev && !t.external) cudaFree(t.dev);
  for (auto& p : e->params)
    if (p.dev) cudaFree(p.dev);
  for (auto& op : e->ops) {
    for (auto& c : op.convs) {
      if (c.scale) cudaFree(c.scale);
      if (c.shift) cudaFree(c.shift);
      tc_conv_release(&c.tc);
    }
    tc_fire_release(&op.tcfire);
    fused_fire_release(&op.fused);
    first_tc_release(&op.first_tc);
  }
  cudaFree(e->d_anchors);
  cudaFree(e->d_boxes);
  cudaFree(e->d_probs);
  cudaFree(e->d_cls);
  cudaFree(e->d_dets);   // also owns d_counts (one blob); d_input aliases tensors[0].dev
  for (auto ev : e->prof_events) cudaEventDestroy(ev);
  for (int k = 0; k < 2; ++k) {
    if (k == 1 && e->d_in_slot[1]) cudaFree(e->d_in_slot[1]);
    if (e->d_u8_slot[k]) cudaFree(e->d_u8_slot[k]);
    if (e->ev_h2d[k]) cudaEventDestroy(e->ev_h2d[k]);
    if (e->ev_done[k]) cudaEventDestroy(e->ev_done[k]);
  }
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  cudaFree(e->d_scales);
  cudaFree(e->d_frames[0]);
  cudaFree(e->d_frames[1]);
  cudaFree(e->d_gathered);
  if (e->comm && e->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
  (void)cudaGetLastError();   // never leave a stale error for the next engine's launch checks
  delete e;
  return SQDET_OK;
}

int sqdet_add_conv(sqdet_engine* e, const char* layer_name, int src, int filters, int size,
                   int stride, int padding, int relu, int* out) {
  int rc = check_build(e, src);
  if (rc) return rc;
  if (!layer_name || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_conv: null argument");
  Op op;
  op.kind = OP_CONV;
  op.name = layer_name;
  ConvSpec cs;
  int Ho, Wo;
  rc = make_conv(e, layer_name, src, filters, size, stride, padding, relu, false, true, &cs,
                 &Ho, &Wo);
  if (rc) return rc;
  cs.dst = new_tensor(e, layer_name, e->tensors[src].B, Ho, Wo, filters);
  conv_cost(e, cs, Ho, Wo, &op);
  op.src = src;
  op.dst = cs.dst;
  op.convs.push_back(cs);
  e->ops.push_back(op);
  *out = cs.dst;
  return SQDET_OK;
}

int sqdet_add_conv_bn(sqdet_engine* e, const char* scope_name, int src, int filters, int size,
                      int stride, int relu, int conv_with_bias, int* out) {
  int rc = check_build(e, src);
  if (rc) return rc;
  if (!scope_name || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_conv_bn: null argument");
  Op op;
  op.kind = OP_CONV;
  op.name = scope_name;
  ConvSpec cs;
  int Ho, Wo;
  rc = make_conv(e, scope_name, src, filters, size, stride, SQDET_PAD_SAME, relu, true,
                 conv_with_bias != 0, &cs, &Ho, &Wo);
  if (rc) return rc;
  cs.dst = new_tensor(e, scope_name, e->tensors[src].B, Ho, Wo, filters);
  conv_cost(e, cs, Ho, Wo, &op);
  op.src = src;
  op.dst = cs.dst;
  op.convs.push_back(cs);
  e->ops.push_back(op);
  *out = cs.dst;
  return SQDET_OK;
}

int sqdet_add_pool(sqdet_engine* e, const char* layer_name, int src, int size, int stride,
                   int padding, int* out) {
  int rc = check_build(e, src);
  if (rc) return rc;
  if (!layer_name || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_pool: null argument");
  if (size <= 0 || stride <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_pool: non-positive size/stride");
  if (padding != SQDET_PAD_SAME && padding != SQDET_PAD_VALID)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_pool: padding must be SAME(0) or VALID(1)");
  const Tensor in = e->tensors[src];
  const Geom gh = tf_geometry(in.H, size, stride, padding);
  const Geom gw = tf_geometry(in.W, size, stride, padding);
  if (gh.out <= 0 || gw.out <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_pool: window larger than input");
  Op op;
  op.kind = OP_POOL;
  op.name = layer_name;
  op.src = src;
  op.size = size;
  op.stride = stride;
  op.padding = padding;
  op.dst = new_tensor(e, layer_name, in.B, gh.out, gw.out, in.C);
  e->ops.push_back(op);
  *out = op.dst;
  return SQDET_OK;
}

int sqdet_add_fire(sqdet_engine* e, const char* layer_name, int src, int s1x1, int e1x1,
                   int e3x3, int* out) {
  int rc = check_build(e, src);
  if (rc) return rc;
  if (!layer_name || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_fire: null argument");
  const std::string base(layer_name);
  Op op;
  op.kind = OP_FIRE;
  op.name = base;
  ConvSpec sq, x1, x3;
  int Ho, Wo;
  rc = make_conv(e, base + "/squeeze1x1", src, s1x1, 1, 1, SQDET_PAD_SAME, 1, false, true, &sq,
                 &Ho, &Wo);
  if (rc) return rc;
  sq.dst = new_tensor(e, base + "/squeeze1x1", e->tensors[src].B, Ho, Wo, s1x1);
  conv_cost(e, sq, Ho, Wo, &op);
  rc = make_conv(e, base + "/expand1x1", sq.dst, e1x1, 1, 1, SQDET_PAD_SAME, 1, false, true,
                 &x1, &Ho, &Wo);
  if (rc) return rc;
  rc = make_conv(e, base + "/expand3x3", sq.dst, e3x3, 3, 1, SQDET_PAD_SAME, 1, false, true,
                 &x3, &Ho, &Wo);
  if (rc) return rc;
  const int dst = new_tensor(e, base, e->tensors[src].B, Ho, Wo, e1x1 + e3x3);
  x1.dst = dst; x1.y_coff = 0;
  x3.dst = dst; x3.y_coff = e1x1;      // tf.concat([ex1x1, ex3x3], 3)  squeezeDet.py:106
  conv_cost(e, x1, Ho, Wo, &op);
  conv_cost(e, x3, Ho, Wo, &op);
  op.src = src;
  op.dst = dst;
  op.convs = {sq, x1, x3};
  e->ops.push_back(op);
  *out = dst;
  return SQDET_OK;
}

int sqdet_add_add_relu(sqdet_engine* e, const char* name, int a, int b, int* out) {
  int rc = check_build(e, a);
  if (rc) return rc;
  rc = check_build(e, b);
  if (rc) return rc;
  if (!name || !out) return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_add_relu: null argument");
  const Tensor ta = e->tensors[a], tb = e->tensors[b];
  if (ta.B != tb.B || ta.H != tb.H || ta.W != tb.W || ta.C != tb.C)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_add_add_relu: operand shapes differ");
  Op op;
  op.kind = OP_ADD_RELU;
  op.name = name;
  op.src = a;
  op.src2 = b;
  op.dst = new_tensor(e, name, ta.B, ta.H, ta.W, ta.C);
  e->ops.push_back(op);
  *out = op.dst;
  return SQDET_OK;
}

int sqdet_set_preds(sqdet_engine* e, int preds, const double* anchor_box, int64_t num_anchors) {
  int rc = check_build(e, preds);
  if (rc) return rc;
  if (!anchor_box) return fail(SQDET_ERR_INVALID_ARG, "sqdet_set_preds: null anchors");
  const Tensor& t = e->tensors[preds];
  const int K = e->cfg.anchors_per_grid, C = e->cfg.classes;
  if (t.C != K * (C + 1 + 4))
    return fail(SQDET_ERR_INVALID_ARG,
                "sqdet_set_preds: preds must have ANCHOR_PER_GRID*(CLASSES+1+4) channels");
  if (num_anchors != (int64_t)t.H * t.W * K)
    return fail(SQDET_ERR_INVALID_ARG,
                "sqdet_set_preds: len(ANCHOR_BOX) != grid_h*grid_w*ANCHOR_PER_GRID");
  e->preds = preds;
  e->grid_h = t.H;
  e->grid_w = t.W;
  e->num_anchors = num_anchors;
  e->anchors_f64.assign(anchor_box, anchor_box + num_anchors * 4);
  return SQDET_OK;
}

int sqdet_finalize(sqdet_engine* e) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (e->finalized) return fail(SQDET_ERR_STATE, "already finalized");
  if (e->preds < 0) return fail(SQDET_ERR_STATE, "sqdet_finalize before sqdet_set_preds");
  DeviceGuard guard(e->device);
  if (!guard.ok) return fail(SQDET_ERR_CUDA, "cannot select the engine's device");
  const sqdet_config& c = e->cfg;
  // result capacity
  const bool topn = c.top_n_detection > 0 && c.top_n_detection < e->num_anchors;
  e->max_dets = c.max_dets > 0 ? c.max_dets : (topn ? c.top_n_detection : 1024);
  if (topn && e->max_dets < c.top_n_detection)
    return fail(SQDET_ERR_INVALID_ARG, "max_dets smaller than TOP_N_DETECTION");
  if (topn && c.top_n_detection > 1024)
    return fail(SQDET_ERR_UNSUPPORTED, "TOP_N_DETECTION above 1024 is not supported");
  // First layer: a Cin = 3, stride-2 conv followed by a 3x3/2 max-pool that nobody else reads runs
  // as one kernel (both math modes); the un-pooled tensor is never materialised.
  for (auto& op : e->ops) op.out = op.dst;
  for (int i = 0; i + 1 < (int)e->ops.size(); ++i) {
    Op& prod = e->ops[i];
    Op& pool = e->ops[i + 1];
    if (prod.kind != OP_CONV || pool.kind != OP_POOL || pool.src != prod.dst) continue;
    const ConvSpec& cs = prod.convs[0];
    if (!conv_pool_simt_eligible(cs.Cin, cs.Cout, cs.size, cs.stride, pool.size, pool.stride))
      continue;
    int readers = 0;
    for (const auto& o : e->ops) {
      if (o.src == prod.dst || o.src2 == prod.dst) ++readers;
      for (const auto& c2 : o.convs)
        if (&o != &prod && c2.src == prod.dst) ++readers;
    }
    if (readers != 1 || prod.dst == e->preds) continue;
    prod.first_layer_fused = true;
    prod.fused_pool_op = i + 1;
    prod.out = pool.dst;
    pool.skip = true;
    e->tensors[prod.dst].materialized = false;
  }
  // activations
  for (size_t i = 0; i < e->tensors.size(); ++i) {
    Tensor& t = e->tensors[i];
    if (!t.materialized) continue;
    SQ_CUDA(cudaMalloc(&t.dev, sizeof(float) * (size_t)t.numel()));
  }
  e->d_input = e->tensors[0].dev;
  const int64_t A = e->num_anchors, B = c.batch_size;
  std::vector<float> anc((size_t)A * 4);
  for (size_t i = 0; i < anc.size(); ++i) anc[i] = (float)e->anchors_f64[i];   // fp64 -> fp32 cast
  SQ_CUDA(cudaMalloc(&e->d_anchors, sizeof(float) * anc.size()));
  SQ_CUDA(cudaMemcpy(e->d_anchors, anc.data(), sizeof(float) * anc.size(), cudaMemcpyHostToDevice));
  SQ_CUDA(cudaMalloc(&e->d_boxes, sizeof(float) * (size_t)(B * A * 4)));
  SQ_CUDA(cudaMalloc(&e->d_probs, sizeof(float) * (size_t)(B * A)));
  SQ_CUDA(cudaMalloc(&e->d_cls, sizeof(int64_t) * (size_t)(B * A)));
  // records and counts share ONE allocation: [B*max_dets records][B int32 counts] is the
  // blob a rank contributes to the N-GPU all-gather (squeezedet_b200/shard.py).
  {
    const size_t rec_bytes = sizeof(sqdet_det) * (size_t)(B * e->max_dets);
    void* blob = nullptr;
    SQ_CUDA(cudaMalloc(&blob, rec_bytes + sizeof(int32_t) * (size_t)B));
    e->d_dets = reinterpret_cast<sqdet_det*>(blob);
    e->d_counts = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(blob) + rec_bytes);
  }
  SQ_CUDA(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
  // per-op accounting + tensor-core planning
  for (auto& op : e->ops) {
    int64_t bytes = 0;
    op.launches = 0;
    if (op.kind == OP_CONV || op.kind == OP_FIRE) {
      bytes = 4 * e->tensors[op.src].numel() + 4 * e->tensors[op.out].numel() + 4 * op.params;
      if (op.first_layer_fused) {
        if (c.math_mode == SQDET_MATH_TF32X3_TC) {
          // first layer on tcgen05, pooled-pixel-major with the pool as a max over accumulators
          // (first_tc.cu); shapes it declines stay on the fused FFMA kernel
          ConvSpec& cs = op.convs[0];
          const Op& po = e->ops[op.fused_pool_op];
          int rc = first_tc_plan(&op.first_tc, e->tensors[cs.src].B, e->tensors[cs.src].H,
                                 e->tensors[cs.src].W, cs.Cout, cs.size, cs.stride, cs.padding,
                                 cs.relu, cs.p_gamma >= 0, po.size, po.stride, po.padding,
                                 e->tensors[op.out].dev);
          if (rc < 0) return rc;
        }
      } else if (c.math_mode == SQDET_MATH_TF32X3_TC) {
        if (op.kind == OP_CONV) {
          ConvSpec& cs = op.convs[0];
          int rc = tc_conv_plan(&cs.tc, e->tensors[cs.src].B, e->tensors[cs.src].H,
                                e->tensors[cs.src].W, cs.Cin, cs.Cout, cs.size, cs.stride,
                                cs.padding, cs.relu, cs.p_gamma >= 0, e->tensors[op.out].C,
                                cs.y_coff, e->tensors[cs.src].dev, e->tensors[op.out].dev);
          if (rc < 0) return rc;
        } else {
          ConvSpec& sq = op.convs[0];
          // The whole module as ONE kernel (fire_tc.cu) where it is the faster plan - measured on
          // SqueezeDet b=20 (profiles/r2_fused_fire.txt): the layers with a 16-channel squeeze and
          // thousands of tiles (fire2/3: -30 % / -17 %); deeper layers need their expand weights
          // streamed per tile and a 2x squeeze (two M tiles per halo), and lose to the squeeze
          // launch + fused expand pair.  SQDET_FUSED_FIRE: 0 never, 1 this rule, 2 every shape the
          // kernel takes, 3 every shape with >= 4 tiles per SM.
          static const int env_fused = env_int("SQDET_FUSED_FIRE", 1);
          if (env_fused && e->tensors[sq.src].dev != nullptr && sq.src != 0) {
            const Tensor& xin = e->tensors[sq.src];
            int sms = 148, dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const long long tiles = (long long)xin.B * ((xin.H + 15) / 16) * ((xin.W + 7) / 8);
            if (env_fused == 2 || (tiles >= 4LL * sms && (env_fused == 3 || sq.Cout <= 16))) {
              int rcf = fused_fire_plan(&op.fused, xin.B, xin.H, xin.W, xin.C, sq.Cout,
                                        op.convs[1].Cout, op.convs[2].Cout, xin.dev,
                                        e->tensors[op.out].dev);
              if (rcf < 0) return rcf;
            }
          }
          if (op.fused.enabled) {
            op.launches = 1;
            op.min_bytes = bytes;
            continue;
          }
          int rc = tc_conv_plan(&sq.tc, e->tensors[sq.src].B, e->tensors[sq.src].H,
                                e->tensors[sq.src].W, sq.Cin, sq.Cout, 1, 1, SQDET_PAD_SAME, 1,
                                false, e->tensors[sq.dst].C, 0, e->tensors[sq.src].dev,
                                e->tensors[sq.dst].dev);
          if (rc < 0) return rc;
          const Tensor& q = e->tensors[sq.dst];
          rc = tc_fire_plan(&op.tcfire, q.B, q.H, q.W, q.C, op.convs[1].Cout, op.convs[2].Cout,
                            q.dev, e->tensors[op.out].dev);
          if (rc < 0) return rc;
        }
      }
      if (op.kind == OP_CONV) op.launches = op.convs[0].tc.enabled ? op.convs[0].tc.launches : 1;
      else op.launches = 1 + (op.tcfire.enabled ? 1 : 2);
    } else if (op.kind == OP_POOL) {
      bytes = op.skip ? 0 : 4 * e->tensors[op.src].numel() + 4 * e->tensors[op.dst].numel();
      op.launches = op.skip ? 0 : 1;
    } else {
      bytes = 4 * 3 * e->tensors[op.dst].numel();
      op.launches = 1;
    }
    op.min_bytes = bytes;
  }
  e->finalized = true;
  e->params_dirty = true;
  return SQDET_OK;
}

int sqdet_num_params(sqdet_engine* e) { return e ? (int)e->params.size() : SQDET_ERR_INVALID_ARG; }

int sqdet_param_info(sqdet_engine* e, int index, char* name_buf, int name_cap, int64_t shape[4],
                     int* ndim) {
  if (!e || index < 0 || index >= (int)e->params.size())
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_param_info: bad index");
  const Param& p = e->params[index];
  if (name_buf && name_cap > 0) {
    strncpy(name_buf, p.name.c_str(), (size_t)name_cap - 1);
    name_buf[name_cap - 1] = 0;
  }
  if (shape)
    for (int i = 0; i < 4; ++i) shape[i] = i < (int)p.shape.size() ? p.shape[i] : 1;
  if (ndim) *ndim = (int)p.shape.size();
  return SQDET_OK;
}

int sqdet_set_param(sqdet_engine* e, const char* name, const float* data, const int64_t* shape,
                    int ndim) {
  if (!e || !name || !data || !shape)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_set_param: null argument");
  auto it = e->param_index.find(name);
  if (it == e->param_index.end())
    return fail(SQDET_ERR_NOT_FOUND, std::string("sqdet_set_param: no parameter named '") + name + "'");
  Param& p = e->params[it->second];
  bool same = ndim == (int)p.shape.size();
  for (int i = 0; same && i < ndim; ++i) same = shape[i] == p.shape[i];
  if (!same)
    return fail(SQDET_ERR_INVALID_ARG,
                std::string("sqdet_set_param: shape mismatch for '") + name + "'");
  memcpy(p.host.data(), data, sizeof(float) * (size_t)p.numel());
  e->params_dirty = true;
  return SQDET_OK;
}

int sqdet_num_tensors(sqdet_engine* e) { return e ? (int)e->tensors.size() : SQDET_ERR_INVALID_ARG; }

int sqdet_tensor_info(sqdet_engine* e, int id, char* name_buf, int name_cap, int64_t shape[4]) {
  if (!e || id < 0 || id >= (int)e->tensors.size())
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_tensor_info: bad id");
  const Tensor& t = e->tensors[id];
  if (name_buf && name_cap > 0) {
    strncpy(name_buf, t.name.c_str(), (size_t)name_cap - 1);
    name_buf[name_cap - 1] = 0;
  }
  if (shape) { shape[0] = t.B; shape[1] = t.H; shape[2] = t.W; shape[3] = t.C; }
  return SQDET_OK;
}

int sqdet_read_tensor(sqdet_engine* e, int id, float* host_out) {
  if (!e || id < 0 || id >= (int)e->tensors.size() || !host_out)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_read_tensor: bad argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_read_tensor before sqdet_finalize");
  DeviceGuard guard(e->device);
  SQ_CUDA(cudaDeviceSynchronize());
  const Tensor& t = e->tensors[id];
  if (!t.materialized)
    return fail(SQDET_ERR_NOT_FOUND, "tensor '" + t.name + "' is not materialised (fused into its consumer)");
  SQ_CUDA(cudaMemcpy(host_out, t.dev, sizeof(float) * (size_t)t.numel(), cudaMemcpyDeviceToHost));
  return SQDET_OK;
}

int sqdet_num_ops(sqdet_engine* e) { return e ? (int)e->ops.size() + 2 : SQDET_ERR_INVALID_ARG; }

int sqdet_op_info(sqdet_engine* e, int index, char* name_buf, int name_cap, int64_t* flops,
                  int64_t* params, int64_t* min_bytes) {
  if (!e || index < 0 || index >= (int)e->ops.size() + 2)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_op_info: bad index");
  std::string name;
  int64_t fl = 0, pa = 0, by = 0;
  const int nops = (int)e->ops.size();
  if (index < nops) {
    const Op& op = e->ops[index];
    name = op.name; fl = op.flops; pa = op.params; by = op.min_bytes;
  } else {
    const int64_t B = e->cfg.batch_size, A = e->num_anchors;
    if (index == nops) {
      name = "interpret_output";
      by = e->preds >= 0 ? 4 * e->tensors[e->preds].numel() + B * A * (16 + 4 + 8) : 0;
    } else {
      name = "filter_prediction";
      by = B * A * 4 + B * (int64_t)e->max_dets * (int64_t)sizeof(sqdet_det);
    }
  }
  if (name_buf && name_cap > 0) {
    strncpy(name_buf, name.c_str(), (size_t)name_cap - 1);
    name_buf[name_cap - 1] = 0;
  }
  if (flops) *flops = fl;
  if (params) *params = pa;
  if (min_bytes) *min_bytes = by;
  return SQDET_OK;
}

int sqdet_forward(sqdet_engine* e, const float* images_dev, void* stream) {
  return forward_impl(e, images_dev, (cudaStream_t)stream);
}

int sqdet_forward_profiled(sqdet_engine* e, const float* images_dev, void* stream_v,
                           float* op_ms) {
  if (!e || !op_ms) return fail(SQDET_ERR_INVALID_ARG, "sqdet_forward_profiled: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_forward_profiled before sqdet_finalize");
  if (!images_dev) return fail(SQDET_ERR_INVALID_ARG, "null images pointer");
  cudaStream_t stream = (cudaStream_t)stream_v;
  DeviceGuard guard(e->device);
  int rc = prepare_params(e);
  if (rc) return rc;
  const int n = (int)e->ops.size() + 2;
  while ((int)e->prof_events.size() < n + 1) {
    cudaEvent_t ev;
    SQ_CUDA(cudaEventCreate(&ev));
    e->prof_events.push_back(ev);
  }
  SQ_CUDA(cudaEventRecord(e->prof_events[0], stream));
  for (int i = 0; i < (int)e->ops.size(); ++i) {
    rc = run_op(e, e->ops[i], images_dev, stream);
    if (rc) return rc;
    SQ_CUDA(cudaEventRecord(e->prof_events[i + 1], stream));
  }
  const sqdet_config& c = e->cfg;
  rc = launch_interpret(e->tensors[e->preds].dev, e->d_anchors, e->d_boxes, e->d_probs, e->d_cls,
                        c.batch_size, e->grid_h, e->grid_w, c.anchors_per_grid, c.classes,
                        c.image_width, c.image_height, c.exp_thresh, stream);
  if (rc) return rc;
  if (e->rescale_on) {
    rc = launch_rescale_boxes(e->d_boxes, e->d_scales + (size_t)e->scale_slot * c.batch_size * 2,
                              c.batch_size, (int)e->num_anchors, stream);
    if (rc) return rc;
  }
  SQ_CUDA(cudaEventRecord(e->prof_events[n - 1], stream));
  rc = launch_topk_nms(e->d_boxes, e->d_probs, e->d_cls, c.batch_size, (int)e->num_anchors,
                       c.classes, c.top_n_detection, c.prob_thresh, c.nms_thresh, e->d_dets,
                       e->d_counts, e->max_dets, stream);
  if (rc) return rc;
  SQ_CUDA(cudaEventRecord(e->prof_events[n], stream));
  SQ_CUDA(cudaEventSynchronize(e->prof_events[n]));
  for (int i = 0; i < n; ++i)
    SQ_CUDA(cudaEventElapsedTime(&op_ms[i], e->prof_events[i], e->prof_events[i + 1]));
  return SQDET_OK;
}

int sqdet_results_dev(sqdet_engine* e, float** det_boxes, float** det_probs, int64_t** det_class,
                      sqdet_det** dets, int32_t** counts, int32_t* max_dets) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_results_dev before sqdet_finalize");
  if (det_boxes) *det_boxes = e->d_boxes;
  if (det_probs) *det_probs = e->d_probs;
  if (det_class) *det_class = e->d_cls;
  if (dets) *dets = e->d_dets;
  if (counts) *counts = e->d_counts;
  if (max_dets) *max_dets = e->max_dets;
  return SQDET_OK;
}

int sqdet_detect(sqdet_engine* e, const float* images, float* det_boxes, float* det_probs,
                 int64_t* det_class, sqdet_det* dets, int32_t* counts, void* stream_v) {
  if (!e || !images) return fail(SQDET_ERR_INVALID_ARG, "sqdet_detect: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_detect before sqdet_finalize");
  DeviceGuard guard(e->device);
  cudaStream_t stream = stream_v ? (cudaStream_t)stream_v : e->own_stream;
  const sqdet_config& c = e->cfg;
  const size_t in_bytes = sizeof(float) * (size_t)e->tensors[0].numel();
  SQ_CUDA(cudaMemcpyAsync(e->d_input, images, in_bytes, cudaMemcpyHostToDevice, stream));
  int rc = forward_impl(e, e->d_input, stream);
  if (rc) return rc;
  const size_t BA = (size_t)c.batch_size * (size_t)e->num_anchors;
  if (det_boxes)
    SQ_CUDA(cudaMemcpyAsync(det_boxes, e->d_boxes, sizeof(float) * BA * 4, cudaMemcpyDeviceToHost, stream));
  if (det_probs)
    SQ_CUDA(cudaMemcpyAsync(det_probs, e->d_probs, sizeof(float) * BA, cudaMemcpyDeviceToHost, stream));
  if (det_class)
    SQ_CUDA(cudaMemcpyAsync(det_class, e->d_cls, sizeof(int64_t) * BA, cudaMemcpyDeviceToHost, stream));
  if (dets)
    SQ_CUDA(cudaMemcpyAsync(dets, e->d_dets, sizeof(sqdet_det) * (size_t)c.batch_size * e->max_dets,
                            cudaMemcpyDeviceToHost, stream));
  if (counts)
    SQ_CUDA(cudaMemcpyAsync(counts, e->d_counts, sizeof(int32_t) * (size_t)c.batch_size,
                            cudaMemcpyDeviceToHost, stream));
  SQ_CUDA(cudaStreamSynchronize(stream));
  return SQDET_OK;
}

int sqdet_set_bgr_means(sqdet_engine* e, const double bgr_means[3]) {
  if (!e || !bgr_means) return fail(SQDET_ERR_INVALID_ARG, "sqdet_set_bgr_means: null argument");
  for (int i = 0; i < 3; ++i) e->bgr_means[i] = bgr_means[i];
  return SQDET_OK;
}

int sqdet_submit(sqdet_engine* e, const void* images, int img_type, sqdet_det* dets,
                 int32_t* counts) {
  if (!e || !images) return fail(SQDET_ERR_INVALID_ARG, "sqdet_submit: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_submit before sqdet_finalize");
  if (img_type != SQDET_IMG_F32 && img_type != SQDET_IMG_U8)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_submit: unknown img_type");
  if (e->n_submitted - e->n_waited >= 2)
    return fail(SQDET_ERR_STATE, "sqdet_submit: two batches already in flight; call sqdet_wait");
  DeviceGuard guard(e->device);
  const sqdet_config& c = e->cfg;
  const int slot = (int)(e->n_submitted & 1);
  const int64_t n_pix = (int64_t)c.batch_size * c.image_height * c.image_width;
  if (!e->copy_stream) {
    SQ_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    e->d_in_slot[0] = e->tensors[0].dev;
    SQ_CUDA(cudaMalloc(&e->d_in_slot[1], sizeof(float) * (size_t)n_pix * 3));
    for (int k = 0; k < 2; ++k) {
      SQ_CUDA(cudaEventCreateWithFlags(&e->ev_h2d[k], cudaEventDisableTiming));
      SQ_CUDA(cudaEventCreateWithFlags(&e->ev_done[k], cudaEventDisableTiming));
    }
  }
  if (img_type == SQDET_IMG_U8 && !e->d_u8_slot[slot])
    SQ_CUDA(cudaMalloc(&e->d_u8_slot[slot], (size_t)n_pix * 3));
  cudaStream_t cs = e->copy_stream, ks = e->own_stream;
  // the slot's input buffers are free once the forward that last read them has finished
  if (e->slot_used[slot]) SQ_CUDA(cudaStreamWaitEvent(cs, e->ev_done[slot], 0));
  if (img_type == SQDET_IMG_U8)
    SQ_CUDA(cudaMemcpyAsync(e->d_u8_slot[slot], images, (size_t)n_pix * 3, cudaMemcpyHostToDevice, cs));
  else
    SQ_CUDA(cudaMemcpyAsync(e->d_in_slot[slot], images, sizeof(float) * (size_t)n_pix * 3,
                            cudaMemcpyHostToDevice, cs));
  SQ_CUDA(cudaEventRecord(e->ev_h2d[slot], cs));
  SQ_CUDA(cudaStreamWaitEvent(ks, e->ev_h2d[slot], 0));
  int rc = SQDET_OK;
  if (img_type == SQDET_IMG_U8) {
    // on the COMPUTE stream: on the copy stream (to overlap the previous batch's forward) it was
    // measured slower, 2.08 vs 1.93 ms per step end to end - its CTAs wait for the persistent
    // one-CTA-per-SM kernels of that forward and then delay this batch's first layer
    rc = launch_u8_meansub(e->d_u8_slot[slot], e->d_in_slot[slot], n_pix, e->bgr_means[0],
                           e->bgr_means[1], e->bgr_means[2], ks);
    if (rc) return rc;
  }
  rc = forward_impl(e, e->d_in_slot[slot], ks);
  if (rc) return rc;
  if (dets)
    SQ_CUDA(cudaMemcpyAsync(dets, e->d_dets, sizeof(sqdet_det) * (size_t)c.batch_size * e->max_dets,
                            cudaMemcpyDeviceToHost, ks));
  if (counts)
    SQ_CUDA(cudaMemcpyAsync(counts, e->d_counts, sizeof(int32_t) * (size_t)c.batch_size,
                            cudaMemcpyDeviceToHost, ks));
  SQ_CUDA(cudaEventRecord(e->ev_done[slot], ks));
  e->slot_used[slot] = true;
  ++e->n_submitted;
  return SQDET_OK;
}

int sqdet_wait(sqdet_engine* e) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (e->n_waited >= e->n_submitted) return fail(SQDET_ERR_STATE, "sqdet_wait: nothing in flight");
  DeviceGuard guard(e->device);
  const int slot = (int)(e->n_waited & 1);
  SQ_CUDA(cudaEventSynchronize(e->ev_done[slot]));
  ++e->n_waited;
  return SQDET_OK;
}

int sqdet_launches_per_forward(sqdet_engine* e) {
  if (!e) return SQDET_ERR_INVALID_ARG;
  int n = 2 + (e->rescale_on ? 1 : 0);   // interpret [+ rescale] + filter (NCCL's own kernel not counted)
  for (const auto& op : e->ops) n += op.launches;
  return n;
}


// ---- eval-order rescale ---------------------------------------------------------------------------
int sqdet_set_box_scale(sqdet_engine* e, const float* xy_scales) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_set_box_scale before sqdet_finalize");
  DeviceGuard guard(e->device);
  const bool on = xy_scales != nullptr;
  if (on) {
    const size_t n = (size_t)e->cfg.batch_size * 2;
    for (size_t i = 0; i < n; ++i)
      if (!(xy_scales[i] > 0.f)) return fail(SQDET_ERR_INVALID_ARG, "sqdet_set_box_scale: scales must be positive");
    if (!e->d_scales) SQ_CUDA(cudaMalloc(&e->d_scales, sizeof(float) * n * 2));
    // synchronous: no forward may be in flight while the table changes (both pipeline halves)
    SQ_CUDA(cudaDeviceSynchronize());
    SQ_CUDA(cudaMemcpy(e->d_scales, xy_scales, sizeof(float) * n, cudaMemcpyHostToDevice));
    SQ_CUDA(cudaMemcpy(e->d_scales + n, xy_scales, sizeof(float) * n, cudaMemcpyHostToDevice));
    SQ_CUDA(cudaStreamSynchronize(nullptr));   // landed before the next forward's stream reads it
  }
  if (on != e->rescale_on) {
    e->rescale_on = on;
    drop_graph(e);           // the captured forward has one kernel more / less
  }
  return SQDET_OK;
}

// ---- variable-size uint8 frames in front of the path (SURVEY 8 f-1) --------------------------------
int sqdet_submit_frames(sqdet_engine* e, const uint8_t* const* frames, const int32_t* heights,
                        const int32_t* widths, int order, int rescale, sqdet_det* dets,
                        int32_t* counts) {
  if (!e || !frames || !heights || !widths)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_submit_frames: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_submit_frames before sqdet_finalize");
  if (order != SQDET_PRE_RESIZE_THEN_SUB && order != SQDET_PRE_SUB_THEN_RESIZE)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_submit_frames: order must be 0 (demo) or 1 (eval)");
  if (e->n_submitted - e->n_waited >= 2)
    return fail(SQDET_ERR_STATE, "sqdet_submit_frames: two batches already in flight; call sqdet_wait");
  DeviceGuard guard(e->device);
  const sqdet_config& c = e->cfg;
  const int B = c.batch_size;
  size_t total = 0;
  std::vector<size_t> off((size_t)B);
  for (int i = 0; i < B; ++i) {
    if (!frames[i] || heights[i] <= 0 || widths[i] <= 0)
      return fail(SQDET_ERR_INVALID_ARG, "sqdet_submit_frames: empty frame");
    off[(size_t)i] = total;
    total += ((size_t)heights[i] * widths[i] * 3 + 255) & ~(size_t)255;
  }
  const int slot = (int)(e->n_submitted & 1);
  const int64_t n_pix = (int64_t)B * c.image_height * c.image_width;
  if (!e->copy_stream) {
    SQ_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    e->d_in_slot[0] = e->tensors[0].dev;
    SQ_CUDA(cudaMalloc(&e->d_in_slot[1], sizeof(float) * (size_t)n_pix * 3));
    for (int k = 0; k < 2; ++k) {
      SQ_CUDA(cudaEventCreateWithFlags(&e->ev_h2d[k], cudaEventDisableTiming));
      SQ_CUDA(cudaEventCreateWithFlags(&e->ev_done[k], cudaEventDisableTiming));
    }
  }
  cudaStream_t cs = e->copy_stream, ks = e->own_stream;
  if (e->slot_used[slot]) SQ_CUDA(cudaStreamWaitEvent(cs, e->ev_done[slot], 0));
  if (e->frames_cap[slot] < total) {
    // growing the staging buffer: the slot's previous forward must be done with it
    if (e->slot_used[slot]) SQ_CUDA(cudaEventSynchronize(e->ev_done[slot]));
    cudaFree(e->d_frames[slot]);
    e->d_frames[slot] = nullptr;
    SQ_CUDA(cudaMalloc(&e->d_frames[slot], total));
    e->frames_cap[slot] = total;
  }
  for (int i = 0; i < B; ++i)
    SQ_CUDA(cudaMemcpyAsync(e->d_frames[slot] + off[(size_t)i], frames[i],
                            (size_t)heights[i] * widths[i] * 3, cudaMemcpyHostToDevice, cs));
  SQ_CUDA(cudaEventRecord(e->ev_h2d[slot], cs));
  // eval order: boxes go back to each frame's own pixel grid before the filter (eval.py:80-87)
  if (rescale) {
    std::vector<float> sc((size_t)B * 2);
    for (int i = 0; i < B; ++i) {
      // eval.py:72-74 / imdb.py:93-95: x_scale = mc.IMAGE_WIDTH / orig_w (Python floats = double)
      sc[(size_t)2 * i] = (float)((double)c.image_width / (double)widths[i]);
      sc[(size_t)2 * i + 1] = (float)((double)c.image_height / (double)heights[i]);
    }
    if (!e->rescale_on) {
      int rc = sqdet_set_box_scale(e, sc.data());      // first use: allocate + enable
      if (rc) return rc;
    }
    // this slot's half of the table, in stream order behind the forward that last read it
    SQ_CUDA(cudaMemcpyAsync(e->d_scales + (size_t)slot * B * 2, sc.data(), sizeof(float) * B * 2,
                            cudaMemcpyHostToDevice, ks));
  } else if (e->rescale_on) {
    int rc = sqdet_set_box_scale(e, nullptr);
    if (rc) return rc;
  }
  SQ_CUDA(cudaStreamWaitEvent(ks, e->ev_h2d[slot], 0));
  const size_t img_floats = (size_t)c.image_height * c.image_width * 3;
  for (int i = 0; i < B; ++i) {
    int rc = launch_resize_meansub_u8(e->d_frames[slot] + off[(size_t)i], heights[i], widths[i],
                                      e->d_in_slot[slot] + (size_t)i * img_floats, c.image_height,
                                      c.image_width, e->bgr_means[0], e->bgr_means[1],
                                      e->bgr_means[2], order == SQDET_PRE_SUB_THEN_RESIZE, ks);
    if (rc) return rc;
  }
  int rc = forward_impl(e, e->d_in_slot[slot], ks);
  if (rc) return rc;
  if (dets)
    SQ_CUDA(cudaMemcpyAsync(dets, e->d_dets, sizeof(sqdet_det) * (size_t)B * e->max_dets,
                            cudaMemcpyDeviceToHost, ks));
  if (counts)
    SQ_CUDA(cudaMemcpyAsync(counts, e->d_counts, sizeof(int32_t) * (size_t)B,
                            cudaMemcpyDeviceToHost, ks));
  SQ_CUDA(cudaEventRecord(e->ev_done[slot], ks));
  e->slot_used[slot] = true;
  ++e->n_submitted;
  return SQDET_OK;
}

// ---- multi-GPU: ONE all-gather of the filtered records ---------------------------------------------
int sqdet_comm_unique_id(void* id128) {
  if (!id128) return fail(SQDET_ERR_INVALID_ARG, "sqdet_comm_unique_id: null buffer");
  int rc = nccl_load();
  if (rc) return rc;
  NcclId id;
  const int r = g_nccl.GetUniqueId(&id);
  if (r != 0) return nccl_fail(r, "ncclGetUniqueId");
  memcpy(id128, id.internal, 128);
  return SQDET_OK;
}

static int comm_buffers(sqdet_engine* e) {
  e->blob_bytes = sizeof(sqdet_det) * (size_t)e->cfg.batch_size * e->max_dets +
                  sizeof(int32_t) * (size_t)e->cfg.batch_size;
  cudaFree(e->d_gathered);
  e->d_gathered = nullptr;
  SQ_CUDA(cudaMalloc(&e->d_gathered, e->blob_bytes * (size_t)e->comm_nranks));
  SQ_CUDA(cudaMemset(e->d_gathered, 0, e->blob_bytes * (size_t)e->comm_nranks));
  return SQDET_OK;
}

int sqdet_comm_init(sqdet_engine* e, int nranks, int rank, const void* id128) {
  if (!e || !id128) return fail(SQDET_ERR_INVALID_ARG, "sqdet_comm_init: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_comm_init before sqdet_finalize");
  if (nranks <= 0 || rank < 0 || rank >= nranks)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_comm_init: bad nranks/rank");
  if (e->comm) return fail(SQDET_ERR_STATE, "sqdet_comm_init: a communicator is already attached");
  int rc = nccl_load();
  if (rc) return rc;
  DeviceGuard guard(e->device);
  if (!guard.ok) return fail(SQDET_ERR_CUDA, "cannot select the engine's device");
  NcclId id;
  memcpy(id.internal, id128, 128);
  void* comm = nullptr;
  const int r = g_nccl.CommInitRank(&comm, nranks, id, rank);
  if (r != 0) return nccl_fail(r, "ncclCommInitRank");
  e->comm = comm;
  e->comm_owned = true;
  e->comm_nranks = nranks;
  e->comm_rank = rank;
  rc = comm_buffers(e);
  if (rc) return rc;
  // one eager collective so that channels / peer connections exist before any graph capture
  rc = run_allgather(e, e->comm, e->own_stream);
  if (rc) return rc;
  SQ_CUDA(cudaStreamSynchronize(e->own_stream));
  return SQDET_OK;
}

int sqdet_comm_attach(sqdet_engine* e, void* nccl_comm, int nranks, int rank) {
  if (!e || !nccl_comm) return fail(SQDET_ERR_INVALID_ARG, "sqdet_comm_attach: null argument");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_comm_attach before sqdet_finalize");
  if (nranks <= 0 || rank < 0 || rank >= nranks)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_comm_attach: bad nranks/rank");
  if (e->comm) return fail(SQDET_ERR_STATE, "sqdet_comm_attach: a communicator is already attached");
  int rc = nccl_load();
  if (rc) return rc;
  DeviceGuard guard(e->device);
  e->comm = nccl_comm;
  e->comm_owned = false;
  e->comm_nranks = nranks;
  e->comm_rank = rank;
  return comm_buffers(e);
}

int sqdet_comm_destroy(sqdet_engine* e) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  DeviceGuard guard(e->device);
  cudaDeviceSynchronize();
  drop_graph(e);
  if (e->comm && e->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
  e->comm = nullptr;
  e->comm_owned = false;
  e->gather_in_forward = false;
  cudaFree(e->d_gathered);
  e->d_gathered = nullptr;
  return SQDET_OK;
}

int sqdet_set_gather_in_forward(sqdet_engine* e, int on) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (on && !e->comm) return fail(SQDET_ERR_STATE, "sqdet_set_gather_in_forward: no communicator");
  if ((on != 0) != e->gather_in_forward) {
    e->gather_in_forward = on != 0;
    drop_graph(e);
  }
  return SQDET_OK;
}

int sqdet_allgather(sqdet_engine* e, void* nccl_comm, void* stream) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (!e->finalized) return fail(SQDET_ERR_STATE, "sqdet_allgather before sqdet_finalize");
  DeviceGuard guard(e->device);
  return run_allgather(e, nccl_comm ? nccl_comm : e->comm, (cudaStream_t)stream);
}

int sqdet_gathered_dev(sqdet_engine* e, void** gathered, int64_t* bytes_per_rank, int32_t* nranks) {
  if (!e) return fail(SQDET_ERR_INVALID_ARG, "null engine");
  if (!e->d_gathered) return fail(SQDET_ERR_STATE, "sqdet_gathered_dev: no communicator attached");
  if (gathered) *gathered = e->d_gathered;
  if (bytes_per_rank) *bytes_per_rank = (int64_t)e->blob_bytes;
  if (nranks) *nranks = e->comm_nranks;
  return SQDET_OK;
}

void* sqdet_engine_stream(sqdet_engine* e) { return e ? (void*)e->own_stream : nullptr; }

// ---- stage-isolated kernels ------------------------------------------------------------------
int sqdet_conv2d(const float* x_dev, const float* w_hwio_dev, const float* bias_dev,
                 const float* scale_dev, const float* shift_dev, float* y_dev, int B, int H, int W,
                 int Cin, int Cout, int size, int stride, int padding, int relu, int y_cstride,
                 int y_coff, int math_mode, void* stream) {
  if (!x_dev || !w_hwio_dev || !y_dev) return fail(SQDET_ERR_INVALID_ARG, "sqdet_conv2d: null pointer");
  if (padding != SQDET_PAD_SAME && padding != SQDET_PAD_VALID)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_conv2d: padding must be SAME(0) or VALID(1)");
  if (math_mode == SQDET_MATH_TF32X3_TC)
    return conv2d_tc_oneshot(x_dev, w_hwio_dev, bias_dev, scale_dev, shift_dev, y_dev, B, H, W,
                             Cin, Cout, size, stride, padding, relu, y_cstride, y_coff,
                             (cudaStream_t)stream);
  if (math_mode != SQDET_MATH_FP32_SIMT)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_conv2d: unknown math_mode");
  ConvArgs a;
  a.x = x_dev; a.w = w_hwio_dev; a.bias = bias_dev; a.scale = scale_dev; a.shift = shift_dev;
  a.y = y_dev; a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.size = size;
  a.stride = stride; a.padding = padding; a.relu = relu; a.y_cstride = y_cstride; a.y_coff = y_coff;
  return launch_conv_simt(a, (cudaStream_t)stream);
}

/* SqueezeDet._fire_layer as ONE stage-isolated call (src/nets/squeezeDet.py:81-106). */
int sqdet_fire(const float* x_dev, const float* w_sq_dev, const float* b_sq_dev,
               const float* w_e1_dev, const float* b_e1_dev, const float* w_e3_dev,
               const float* b_e3_dev, float* y_dev, int B, int H, int W, int Cin, int S, int E1,
               int E3, int math_mode, void* stream_v) {
  if (!x_dev || !w_sq_dev || !b_sq_dev || !w_e1_dev || !b_e1_dev || !w_e3_dev || !b_e3_dev || !y_dev)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_fire: null pointer");
  if (B <= 0 || H <= 0 || W <= 0 || Cin <= 0 || S <= 0 || E1 <= 0 || E3 <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_fire: non-positive dimension");
  if (math_mode != SQDET_MATH_FP32_SIMT && math_mode != SQDET_MATH_TF32X3_TC)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_fire: unknown math_mode");
  cudaStream_t stream = (cudaStream_t)stream_v;
  if (math_mode == SQDET_MATH_TF32X3_TC) {
    int rc = fire_fused_oneshot(x_dev, w_sq_dev, b_sq_dev, w_e1_dev, b_e1_dev, w_e3_dev, b_e3_dev,
                                y_dev, B, H, W, Cin, S, E1, E3, stream);
    if (rc != 1) return rc < 0 ? rc : SQDET_OK;   // 1 = shape not taken by the fused kernel
  }
  // un-fused: squeeze tensor through HBM, then the two expand convs into the concat tensor
  float* q = nullptr;
  SQ_CUDA(cudaMalloc(&q, sizeof(float) * (size_t)B * H * W * S));
  int rc = sqdet_conv2d(x_dev, w_sq_dev, b_sq_dev, nullptr, nullptr, q, B, H, W, Cin, S, 1, 1,
                        SQDET_PAD_SAME, 1, S, 0, math_mode, stream_v);
  if (!rc)
    rc = sqdet_conv2d(q, w_e1_dev, b_e1_dev, nullptr, nullptr, y_dev, B, H, W, S, E1, 1, 1,
                      SQDET_PAD_SAME, 1, E1 + E3, 0, math_mode, stream_v);
  if (!rc)
    rc = sqdet_conv2d(q, w_e3_dev, b_e3_dev, nullptr, nullptr, y_dev, B, H, W, S, E3, 3, 1,
                      SQDET_PAD_SAME, 1, E1 + E3, E1, math_mode, stream_v);
  cudaError_t ce = cudaStreamSynchronize(stream);
  cudaFree(q);
  if (rc) return rc;
  if (ce != cudaSuccess) return cuda_fail(ce, "sqdet_fire sync");
  return SQDET_OK;
}

int sqdet_maxpool_nhwc(const float* x_dev, float* y_dev, int B, int H, int W, int C, int size,
                       int stride, int padding, void* stream) {
  if (!x_dev || !y_dev) return fail(SQDET_ERR_INVALID_ARG, "sqdet_maxpool_nhwc: null pointer");
  if (padding != SQDET_PAD_SAME && padding != SQDET_PAD_VALID)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_maxpool_nhwc: padding must be SAME(0) or VALID(1)");
  return launch_maxpool(x_dev, y_dev, B, H, W, C, size, stride, padding, (cudaStream_t)stream);
}

int sqdet_preprocess_u8(const uint8_t* src_dev, int src_h, int src_w, float* dst_dev, int dst_h,
                        int dst_w, const double* bgr_means, int order, void* stream) {
  if (!src_dev || !dst_dev || !bgr_means)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_preprocess_u8: null pointer");
  if (order != SQDET_PRE_RESIZE_THEN_SUB && order != SQDET_PRE_SUB_THEN_RESIZE)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_preprocess_u8: order must be 0 (demo) or 1 (eval)");
  return launch_resize_meansub_u8(src_dev, src_h, src_w, dst_dev, dst_h, dst_w, bgr_means[0],
                                  bgr_means[1], bgr_means[2], order == SQDET_PRE_SUB_THEN_RESIZE,
                                  (cudaStream_t)stream);
}

int sqdet_interpret(const float* preds_dev, const float* anchors_f32_dev, float* det_boxes_dev,
                    float* det_probs_dev, int64_t* det_class_dev, int B, int grid_h, int grid_w,
                    int anchors_per_grid, int classes, int image_width, int image_height,
                    float exp_thresh, void* stream) {
  if (!preds_dev || !anchors_f32_dev || !det_boxes_dev || !det_probs_dev || !det_class_dev)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_interpret: null pointer");
  return launch_interpret(preds_dev, anchors_f32_dev, det_boxes_dev, det_probs_dev, det_class_dev,
                          B, grid_h, grid_w, anchors_per_grid, classes, image_width, image_height,
                          exp_thresh, (cudaStream_t)stream);
}

int sqdet_topk_nms(const float* boxes_dev, const float* probs_dev, const int64_t* cls_dev, int B,
                   int A, int classes, int top_n, float prob_thresh, float nms_thresh,
                   sqdet_det* dets_dev, int32_t* counts_dev, int max_dets, void* stream) {
  if (!boxes_dev || !probs_dev || !cls_dev || !dets_dev || !counts_dev)
    return fail(SQDET_ERR_INVALID_ARG, "sqdet_topk_nms: null pointer");
  return launch_topk_nms(boxes_dev, probs_dev, cls_dev, B, A, classes, top_n, prob_thresh,
                         nms_thresh, dets_dev, counts_dev, max_dets, (cudaStream_t)stream);
}

// ---- memory helpers ------------------------------------------------------------------------------
int sqdet_malloc(int device, int64_t bytes, void** out_dev) {
  if (!out_dev || bytes <= 0) return fail(SQDET_ERR_INVALID_ARG, "sqdet_malloc: bad argument");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SQDET_ERR_CUDA, "sqdet_malloc: cannot select device");
  SQ_CUDA(cudaMalloc(out_dev, (size_t)bytes));
  return SQDET_OK;
}
int sqdet_free(int device, void* dev) {
  DeviceGuard guard(device);
  if (dev) SQ_CUDA(cudaFree(dev));
  return SQDET_OK;
}
int sqdet_malloc_host(int64_t bytes, void** out_pinned) {
  if (!out_pinned || bytes <= 0) return fail(SQDET_ERR_INVALID_ARG, "sqdet_malloc_host: bad argument");
  SQ_CUDA(cudaMallocHost(out_pinned, (size_t)bytes));
  return SQDET_OK;
}
int sqdet_free_host(void* pinned) {
  if (pinned) SQ_CUDA(cudaFreeHost(pinned));
  return SQDET_OK;
}
int sqdet_memcpy_h2d(void* dst_dev, const void* src, int64_t bytes, void* stream) {
  if (!dst_dev || !src || bytes < 0) return fail(SQDET_ERR_INVALID_ARG, "sqdet_memcpy_h2d: bad argument");
  SQ_CUDA(cudaMemcpyAsync(dst_dev, src, (size_t)bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return SQDET_OK;
}
int sqdet_memcpy_d2h(void* dst, const void* src_dev, int64_t bytes, void* stream) {
  if (!dst || !src_dev || bytes < 0) return fail(SQDET_ERR_INVALID_ARG, "sqdet_memcpy_d2h: bad argument");
  SQ_CUDA(cudaMemcpyAsync(dst, src_dev, (size_t)bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return SQDET_OK;
}
int sqdet_stream_sync(int device, void* stream) {
  DeviceGuard guard(device);
  SQ_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return SQDET_OK;
}

}  // extern "C"
