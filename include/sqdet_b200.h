/*
 * sqdet_b200.h — C ABI of libsqdet_b200.so: the B200 (sm_100a) SqueezeDet
 * inference hot path (conv backbone -> ConvDet -> interpret_output ->
 * filter_prediction / NMS).
 *
 * The reference (BichenWuUCB/squeezeDet) has no FFI of its own: its boundary is
 * the Python object contract of `ModelSkeleton` driven through `sess.run`.  Each
 * entry point below therefore cites the reference *Python* interface it stands
 * in for (paths relative to the reference tree); the binding a maintainer would
 * add on the reference side is a ctypes stub, shown in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns an int status: 0 = SQDET_OK, negative = error;
 *     sqdet_last_error() gives the message of the calling thread's last failure.
 *     Nothing throws across this boundary.
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream).
 *   - "_dev" pointers are device memory on the engine's device, everything else
 *     is host memory.  The caller owns every pointer it passes; the engine owns
 *     its weights, activations and result buffers.
 *   - an engine is bound to one device and is NOT thread-safe (one engine per
 *     host thread / stream).  All launches go to the caller's stream; no hidden
 *     host synchronisation except in the functions documented as synchronous.
 *   - layouts are the reference's: activations NHWC fp32, kernels HWIO fp32,
 *     boxes (cx, cy, w, h) fp32, class ids int64.
 */
#ifndef SQDET_B200_H_
#define SQDET_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQDET_OK                 0
#define SQDET_ERR_INVALID_ARG   (-1)
#define SQDET_ERR_CUDA          (-2)
#define SQDET_ERR_UNSUPPORTED   (-3)
#define SQDET_ERR_STATE         (-4)   /* call order (e.g. forward before finalize) */
#define SQDET_ERR_NOT_FOUND     (-5)
#define SQDET_ERR_OVERFLOW      (-6)   /* threshold branch produced more boxes than capacity */

#define SQDET_PAD_SAME   0
#define SQDET_PAD_VALID  1

/* math_mode of the convolution kernels */
#define SQDET_MATH_FP32_SIMT   0   /* fp32 FFMA direct/implicit-GEMM kernels            */
#define SQDET_MATH_TF32X3_TC   1   /* tcgen05 tensor cores, 3xTF32 split (fp32-grade)    */

typedef struct sqdet_engine sqdet_engine;   /* opaque */

/* One filtered detection (28 bytes) — the element type of the N-GPU all-gather. */
typedef struct sqdet_det {
  int32_t anchor;   /* index into the image's [A] anchors ("kept-box index")           */
  int32_t cls;      /* class id                                                         */
  float   prob;     /* det_probs[anchor]                                                */
  float   cx, cy, w, h;
} sqdet_det;

/* The inference-relevant keys of the reference's `mc` EasyDict
 * (src/config/config.py:10-142, src/config/kitti_squeezeDet_config.py:9-43). */
typedef struct sqdet_config {
  int32_t batch_size;        /* mc.BATCH_SIZE   (static batch dim, nn_skeleton.py:81-84) */
  int32_t image_height;      /* mc.IMAGE_HEIGHT */
  int32_t image_width;       /* mc.IMAGE_WIDTH  */
  int32_t classes;           /* mc.CLASSES      */
  int32_t anchors_per_grid;  /* mc.ANCHOR_PER_GRID */
  int32_t top_n_detection;   /* mc.TOP_N_DETECTION */
  float   prob_thresh;       /* mc.PROB_THRESH  */
  float   nms_thresh;        /* mc.NMS_THRESH   */
  float   exp_thresh;        /* mc.EXP_THRESH   */
  float   batch_norm_epsilon;/* mc.BATCH_NORM_EPSILON */
  int32_t math_mode;         /* SQDET_MATH_*    */
  int32_t max_dets;          /* per-image record capacity; 0 = derive (top_n, else 1024) */
} sqdet_config;

/* ---- library ---------------------------------------------------------------------- */
const char* sqdet_last_error(void);
const char* sqdet_version(void);
/* Number of CUDA devices visible (0 without a GPU/driver); never fails. */
int sqdet_device_count(void);

/* ---- engine life cycle: replaces `Net(mc, gpu_id)` ---------------------------------
 * ModelSkeleton.__init__ (src/nn_skeleton.py:74-135) + the nets' constructors
 * (src/nets/squeezeDet.py:19-28).  `device` is the reference's `gpu_id`. */
int sqdet_create(const sqdet_config* cfg, int device, sqdet_engine** out);
int sqdet_destroy(sqdet_engine* e);

/* ---- graph construction: one call per reference layer constructor ------------------
 * Tensor ids: 0 is `image_input` [B,H,W,3]; every add_* returns a new id in *out.   */
/* ModelSkeleton._conv_layer (src/nn_skeleton.py:471-563): relu?(conv2d + bias).      */
int sqdet_add_conv(sqdet_engine* e, const char* layer_name, int src, int filters,
                   int size, int stride, int padding, int relu, int* out);
/* ModelSkeleton._conv_bn_layer (src/nn_skeleton.py:374-468): SAME conv [+bias] + frozen BN. */
int sqdet_add_conv_bn(sqdet_engine* e, const char* scope_name, int src, int filters,
                      int size, int stride, int relu, int conv_with_bias, int* out);
/* ModelSkeleton._pooling_layer (src/nn_skeleton.py:565-586): tf.nn.max_pool.          */
int sqdet_add_pool(sqdet_engine* e, const char* layer_name, int src, int size,
                   int stride, int padding, int* out);
/* SqueezeDet._fire_layer (src/nets/squeezeDet.py:81-106).                             */
int sqdet_add_fire(sqdet_engine* e, const char* layer_name, int src, int s1x1,
                   int e1x1, int e3x3, int* out);
/* tf.nn.relu(a + b) of the ResNet shortcuts (src/nets/resnet50_convDet.py:55).        */
int sqdet_add_add_relu(sqdet_engine* e, const char* name, int a, int b, int* out);
/* ModelSkeleton._add_interpretation_graph (src/nn_skeleton.py:142-283): declares
 * `preds` and mc.ANCHOR_BOX ([A,4] float64, as the reference stores it).              */
int sqdet_set_preds(sqdet_engine* e, int preds, const double* anchor_box, int64_t num_anchors);
/* Allocate activations / results, upload + pre-process parameters.  After this the
 * graph is frozen.  Parameters not yet set are zero.                                  */
int sqdet_finalize(sqdet_engine* e);

/* ---- parameters: replaces tf.train.Saver(model.model_params).restore ---------------
 * (src/demo.py:181-184, src/eval.py:205).  Names are the reference's TF variable
 * names: "<layer>/kernels" [kh,kw,Cin,Cout], "<layer>/biases" [Cout], BN
 * "<scope>/gamma|beta|mean|var" [Cout].  Callable before or after finalize.           */
int sqdet_num_params(sqdet_engine* e);
int sqdet_param_info(sqdet_engine* e, int index, char* name_buf, int name_cap,
                     int64_t shape[4], int* ndim);
int sqdet_set_param(sqdet_engine* e, const char* name, const float* data,
                    const int64_t* shape, int ndim);

/* ---- introspection (model_size_counter / flop_counter / activation_counter,
 * src/nn_skeleton.py:549-561) -------------------------------------------------------- */
int sqdet_num_tensors(sqdet_engine* e);
int sqdet_tensor_info(sqdet_engine* e, int id, char* name_buf, int name_cap,
                      int64_t shape[4]);
int sqdet_read_tensor(sqdet_engine* e, int id, float* host_out);   /* synchronous */
int sqdet_num_ops(sqdet_engine* e);
int sqdet_op_info(sqdet_engine* e, int index, char* name_buf, int name_cap,
                  int64_t* flops, int64_t* params, int64_t* min_bytes);

/* ---- execution: replaces sess.run([det_boxes, det_probs, det_class], feed_dict) ----
 * (src/demo.py:193-195, src/eval.py:75-77) and model.filter_prediction on every image
 * (src/demo.py:198-199, src/eval.py:86-87).                                           */
/* Asynchronous on `stream`: backbone + ConvDet + interpret_output + filter for the
 * whole batch.  images_dev [B,H,W,3] fp32 (BGR, mean-subtracted).                     */
int sqdet_forward(sqdet_engine* e, const float* images_dev, void* stream);
/* Same, but records a CUDA event around every op (not graph-captured) and returns
 * per-op milliseconds (synchronous).  op_ms has sqdet_num_ops() entries.              */
int sqdet_forward_profiled(sqdet_engine* e, const float* images_dev, void* stream,
                           float* op_ms);
/* Device result buffers of the last forward (valid until the next one):
 * det_boxes [B,A,4] f32, det_probs [B,A] f32, det_class [B,A] i64,
 * dets [B,max_dets] records, counts [B] i32.                                          */
int sqdet_results_dev(sqdet_engine* e, float** det_boxes, float** det_probs,
                      int64_t** det_class, sqdet_det** dets, int32_t** counts,
                      int32_t* max_dets);
/* Synchronous host-buffer call (the end-to-end path): H2D of images, forward, D2H of
 * whichever outputs are non-NULL.  Host buffers should be pinned for full speed.      */
int sqdet_detect(sqdet_engine* e, const float* images, float* det_boxes,
                 float* det_probs, int64_t* det_class, sqdet_det* dets,
                 int32_t* counts, void* stream);
/* Pipelined host-buffer path (depth 2): sqdet_submit enqueues H2D (own copy stream) ->
 * [uint8 -> fp32 - mc.BGR_MEANS on the GPU] -> forward -> D2H of the filtered records and
 * returns at once; sqdet_wait blocks until the OLDEST outstanding submit has delivered into its
 * dets/counts buffers.  With two submits in flight the copy of batch i+1 overlaps the compute
 * of batch i.  img_type SQDET_IMG_F32: [B,H,W,3] fp32 BGR, mean-subtracted (feed_dict
 * semantics, src/demo.py:190-195); SQDET_IMG_U8: [B,H,W,3] uint8 BGR exactly as cv2.imread /
 * cv2.resize leave it (src/demo.py:187-189) - the engine applies `im - mc.BGR_MEANS`
 * (src/demo.py:190, src/dataset/imdb.py:88).  Host buffers must stay valid (and should be
 * pinned) until the matching sqdet_wait.  SQDET_ERR_STATE if two submits are already pending. */
#define SQDET_IMG_F32 0
#define SQDET_IMG_U8  1
int sqdet_set_bgr_means(sqdet_engine* e, const double bgr_means[3]);   /* mc.BGR_MEANS */
int sqdet_submit(sqdet_engine* e, const void* images, int img_type, sqdet_det* dets,
                 int32_t* counts);
int sqdet_wait(sqdet_engine* e);
/* Variable-size frames in front of the path (SURVEY 8 f-1): B uint8 BGR frames exactly as
 * cv2.imread returns them, frame i = [heights[i], widths[i], 3].  The engine does
 * astype(float32) + cv2.resize(..., (mc.IMAGE_WIDTH, mc.IMAGE_HEIGHT)) (float32 INTER_LINEAR) +
 * `- mc.BGR_MEANS` in the reference order `order` (SQDET_PRE_RESIZE_THEN_SUB: src/demo.py:187-190;
 * SQDET_PRE_SUB_THEN_RESIZE: src/dataset/imdb.py:85-97) on the GPU, then the forward; same
 * depth-2 pipelining and sqdet_wait contract as sqdet_submit.  rescale != 0 additionally divides
 * every det box by (x_scale, y_scale) = (IMAGE_WIDTH / widths[i], IMAGE_HEIGHT / heights[i])
 * BEFORE filter_prediction, i.e. the order of src/eval.py:80-87.                            */
int sqdet_submit_frames(sqdet_engine* e, const uint8_t* const* frames,
                        const int32_t* heights, const int32_t* widths, int order,
                        int rescale, sqdet_det* dets, int32_t* counts);
/* src/eval.py:83-84 for callers that resize on the host: xy_scales = B pairs (x_scale,
 * y_scale), host memory; every later forward divides det_boxes[b,:,0::2] by x_scale and
 * [b,:,1::2] by y_scale (float32, as numpy does) between interpret_output and
 * filter_prediction, so det_boxes, the records and the NMS all live on the original image.
 * NULL switches it off.  Synchronous (waits for in-flight forwards).                       */
int sqdet_set_box_scale(sqdet_engine* e, const float* xy_scales);
/* Kernel launches issued by one sqdet_forward (for accounting).                        */
int sqdet_launches_per_forward(sqdet_engine* e);
/* The engine's own compute stream (cudaStream_t as void*): sqdet_detect / sqdet_submit run on
 * it; callers that order foreign work behind those calls record events on it.              */
void* sqdet_engine_stream(sqdet_engine* e);

/* ---- multi-GPU: the ONE collective of the path ---------------------------------------
 * The reference is single-device (`tf.device('/gpu:{}')`, src/nets/squeezeDet.py:21); the
 * path shards over the batch with no data-path exchange, and the only collective is an
 * ncclAllGather of each rank's result blob
 *     [batch * max_dets sqdet_det records][batch int32 counts]
 * NCCL is bound at run time (dlopen of libnccl.so.2, or $SQDET_NCCL_LIB).
 * sqdet_comm_unique_id: rank 0 creates the 128-byte ncclUniqueId; the launcher distributes it
 * (any host channel).  sqdet_comm_init: ncclCommInitRank on the engine's device (collective
 * over all ranks) + the [nranks][blob] receive buffer.  sqdet_comm_attach: use a communicator
 * the caller owns instead (ncclComm_t as void*).  sqdet_set_gather_in_forward(1): every
 * sqdet_forward / sqdet_submit then ends with the all-gather on the SAME stream, captured in
 * the forward's CUDA graph (no host code between filter and collective).  sqdet_allgather:
 * the collective alone on `stream` (comm NULL = the attached one).  sqdet_gathered_dev: the
 * receive buffer, rank-major.                                                              */
int sqdet_comm_unique_id(void* id128);
int sqdet_comm_init(sqdet_engine* e, int nranks, int rank, const void* id128);
int sqdet_comm_attach(sqdet_engine* e, void* nccl_comm, int nranks, int rank);
int sqdet_comm_destroy(sqdet_engine* e);
int sqdet_set_gather_in_forward(sqdet_engine* e, int on);
int sqdet_allgather(sqdet_engine* e, void* nccl_comm, void* stream);
int sqdet_gathered_dev(sqdet_engine* e, void** gathered_dev, int64_t* bytes_per_rank,
                       int32_t* nranks);

/* ---- stage-isolated kernels (device pointers, asynchronous on `stream`) -------------
 * `device` must be current-capable; buffers must live on it.                           */
/* tf.nn.conv2d + bias_add + relu (src/nn_skeleton.py:539-547); scale/shift optional
 * per-channel affine applied before relu (frozen BN, :447-449); y has `y_cstride`
 * channels per pixel and this conv writes channels [y_coff, y_coff+Cout).            */
int sqdet_conv2d(const float* x_dev, const float* w_hwio_dev, const float* bias_dev,
                 const float* scale_dev, const float* shift_dev, float* y_dev,
                 int B, int H, int W, int Cin, int Cout, int size, int stride,
                 int padding, int relu, int y_cstride, int y_coff, int math_mode,
                 void* stream);
/* SqueezeDet._fire_layer (src/nets/squeezeDet.py:81-106; same in squeezeDetPlus.py) as ONE
 * call: y[..., :E1] = relu(1x1_e1(q)+b), y[..., E1:] = relu(3x3_e3(q)+b), q = relu(1x1_s(x)+b).
 * x [B,H,W,Cin], kernels HWIO, y [B,H,W,E1+E3].  With SQDET_MATH_TF32X3_TC and a shape the
 * fused kernel takes (Cin % 32 == 0, S % 16 == 0, S <= 64, E % 32 == 0) this is ONE kernel
 * launch and the squeeze tensor never leaves the SM; other shapes run squeeze and expand
 * as separate launches.  Synchronises the stream (test / debug entry, not the hot path).    */
int sqdet_fire(const float* x_dev, const float* w_sq_dev, const float* b_sq_dev,
               const float* w_e1_dev, const float* b_e1_dev, const float* w_e3_dev,
               const float* b_e3_dev, float* y_dev, int B, int H, int W, int Cin, int S,
               int E1, int E3, int math_mode, void* stream);
/* tf.nn.max_pool NHWC (src/nn_skeleton.py:580-583).                                   */
int sqdet_maxpool_nhwc(const float* x_dev, float* y_dev, int B, int H, int W, int C,
                       int size, int stride, int padding, void* stream);
/* Image pre-processing in front of the path (SURVEY 8 f-1): uint8 BGR [src_h, src_w, 3] ->
 * fp32 [dst_h, dst_w, 3], cv2.resize's float32 INTER_LINEAR plus the mean subtraction.
 * order SQDET_PRE_RESIZE_THEN_SUB: src/demo.py:187-190 (astype(float32), resize, - BGR_MEANS);
 * order SQDET_PRE_SUB_THEN_RESIZE: src/dataset/imdb.py:87-91 (astype(float32), -= BGR_MEANS,
 * resize).  bgr_means: 3 doubles on the host.  dst may point into an engine input batch.  */
#define SQDET_PRE_RESIZE_THEN_SUB 0
#define SQDET_PRE_SUB_THEN_RESIZE 1
int sqdet_preprocess_u8(const uint8_t* src_dev, int src_h, int src_w, float* dst_dev,
                        int dst_h, int dst_w, const double* bgr_means, int order,
                        void* stream);
/* interpret_output (src/nn_skeleton.py:146-238,271-283; util.py:167-196,219-231).     */
int sqdet_interpret(const float* preds_dev, const float* anchors_f32_dev,
                    float* det_boxes_dev, float* det_probs_dev, int64_t* det_class_dev,
                    int B, int grid_h, int grid_w, int anchors_per_grid, int classes,
                    int image_width, int image_height, float exp_thresh, void* stream);
/* ModelSkeleton.filter_prediction + util.nms (src/nn_skeleton.py:696-734,
 * src/utils/util.py:32-76) for B images at once: boxes [B,A,4], probs [B,A],
 * cls [B,A] -> dets [B,max_dets], counts [B] (count<0: SQDET_ERR_OVERFLOW case).      */
int sqdet_topk_nms(const float* boxes_dev, const float* probs_dev,
                   const int64_t* cls_dev, int B, int A, int classes, int top_n,
                   float prob_thresh, float nms_thresh, sqdet_det* dets_dev,
                   int32_t* counts_dev, int max_dets, void* stream);

/* ---- tiny device-memory helpers so a ctypes caller needs nothing else -------------- */
int sqdet_malloc(int device, int64_t bytes, void** out_dev);
int sqdet_free(int device, void* dev);
int sqdet_malloc_host(int64_t bytes, void** out_pinned);
int sqdet_free_host(void* pinned);
int sqdet_memcpy_h2d(void* dst_dev, const void* src, int64_t bytes, void* stream);
int sqdet_memcpy_d2h(void* dst, const void* src_dev, int64_t bytes, void* stream);
int sqdet_stream_sync(int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* SQDET_B200_H_ */
