// interpret_output and filter_prediction / NMS on the GPU.
//
// interpret_kernel  : reference src/nn_skeleton.py:146-238,271-283 (+ util.py:167-196
//                     bbox_transform[_inv], util.py:219-231 safe_exp).  One thread per
//                     anchor; fp32, operation-for-operation (explicit _rn intrinsics so
//                     nvcc cannot contract a*b+c into an FMA the reference did not do).
// filter_kernel     : reference src/nn_skeleton.py:696-734 + src/utils/util.py:32-76.
//                     One CTA per image: radix-select of the top-N score, ordered
//                     compaction, bitonic sort (prob desc, anchor asc), all-pairs
//                     "suppressed-still-suppresses" NMS per class (the reference's rule,
//                     NOT greedy NMS), class-grouped output order.  IoU arithmetic is
//                     bit-exact with numpy float32 (IEEE mul/add/div, no FMA).
// Roofline: HBM / latency (B*A*(K*(C+5))/K*4 bytes in, <= B*top_n*28 bytes out).
#include <math_constants.h>
#include "common.cuh"

namespace sqdet {
namespace {

// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float safe_exp_ref(float w, float thresh, float slope) {
  // util.py:219-231: lin*(slope*(w-thresh+1)) + (1-lin)*exp(where(w>thresh, 0, w))
  const bool lin_b = w > thresh;
  const float lin = lin_b ? 1.f : 0.f;
  const float lin_out = __fmul_rn(slope, __fadd_rn(__fsub_rn(w, thresh), 1.f));
  const float exp_out = expf(lin_b ? 0.f : w);
  return __fadd_rn(__fmul_rn(lin, lin_out), __fmul_rn(__fsub_rn(1.f, lin), exp_out));
}

__global__ void __launch_bounds__(256)
interpret_kernel(const float* __restrict__ preds, const float* __restrict__ anchors,
                 float* __restrict__ boxes, float* __restrict__ probs,
                 long long* __restrict__ cls, int B, int A, int K, int C, float wm1,
                 float hm1, float exp_thresh, float slope) {
  const long long total = (long long)B * A;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int a = (int)(idx % A);
  const int b = (int)(idx / A);
  const int cell = a / K, k = a - cell * K;
  const int nch = K * (C + 5);
  const float* p = preds + ((long long)b * (A / K) + cell) * nch;

  // class probabilities: softmax over C logits (max-subtracted), nn_skeleton.py:151-161
  const float* lg = p + k * C;
  float mx = lg[0];
  for (int c = 1; c < C; ++c) mx = fmaxf(mx, lg[c]);
  float sum = 0.f;
  for (int c = 0; c < C; ++c) sum = __fadd_rn(sum, expf(__fsub_rn(lg[c], mx)));
  // confidence: sigmoid, nn_skeleton.py:164-170
  const float conf = __fdiv_rn(1.f, __fadd_rn(1.f, expf(-p[K * C + k])));
  float best = -CUDART_INF_F;
  int best_c = 0;
  for (int c = 0; c < C; ++c) {
    const float pc = __fmul_rn(__fdiv_rn(expf(__fsub_rn(lg[c], mx)), sum), conf);
    if (pc > best) { best = pc; best_c = c; }   // first maximum wins (tf.argmax)
  }

  // box decode, nn_skeleton.py:173-238
  const float* d = p + K * C + K + k * 4;
  const float4 an = *reinterpret_cast<const float4*>(anchors + (long long)a * 4);
  const float cx = __fadd_rn(an.x, __fmul_rn(d[0], an.z));
  const float cy = __fadd_rn(an.y, __fmul_rn(d[1], an.w));
  const float bw = __fmul_rn(an.z, safe_exp_ref(d[2], exp_thresh, slope));
  const float bh = __fmul_rn(an.w, safe_exp_ref(d[3], exp_thresh, slope));
  const float hw = __fdiv_rn(bw, 2.f), hh = __fdiv_rn(bh, 2.f);
  float xmin = __fsub_rn(cx, hw), ymin = __fsub_rn(cy, hh);
  float xmax = __fadd_rn(cx, hw), ymax = __fadd_rn(cy, hh);
  xmin = fminf(fmaxf(0.f, xmin), wm1);
  ymin = fminf(fmaxf(0.f, ymin), hm1);
  xmax = fmaxf(fminf(wm1, xmax), 0.f);
  ymax = fmaxf(fminf(hm1, ymax), 0.f);
  const float w = __fadd_rn(__fsub_rn(xmax, xmin), 1.f);
  const float h = __fadd_rn(__fsub_rn(ymax, ymin), 1.f);
  float4 o;
  o.x = __fadd_rn(xmin, __fmul_rn(0.5f, w));
  o.y = __fadd_rn(ymin, __fmul_rn(0.5f, h));
  o.z = w;
  o.w = h;
  reinterpret_cast<float4*>(boxes)[idx] = o;
  probs[idx] = best;
  cls[idx] = best_c;
}

// det_boxes[j, :, 0::2] /= x_scale; det_boxes[j, :, 1::2] /= y_scale  (reference src/eval.py:83-84):
// the rescale of ALL boxes to the original image that the reference applies BEFORE
// filter_prediction.  numpy divides the float32 array by the (weak) Python float in float32.
__global__ void __launch_bounds__(256)
rescale_boxes_kernel(float4* __restrict__ boxes, const float* __restrict__ scales, int A,
                     long long total) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int b = (int)(idx / A);
  const float xs = __ldg(scales + 2 * b), ys = __ldg(scales + 2 * b + 1);
  float4 v = boxes[idx];
  v.x = __fdiv_rn(v.x, xs); v.z = __fdiv_rn(v.z, xs);
  v.y = __fdiv_rn(v.y, ys); v.w = __fdiv_rn(v.w, ys);
  boxes[idx] = v;
}

// ------------------------------------------------------------------------------------------
constexpr int FT = 1024;          // threads of the filter CTA
constexpr int FCAP = 1024;        // max candidates per image

__device__ __forceinline__ unsigned order_key(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);   // larger float -> larger key
}

// centre-format IoU, util.py:42-54, numpy float32 semantics.
__device__ __forceinline__ float iou_ref(const float4 a, const float4 b) {
  const float ahw = __fmul_rn(0.5f, a.z), bhw = __fmul_rn(0.5f, b.z);
  const float ahh = __fmul_rn(0.5f, a.w), bhh = __fmul_rn(0.5f, b.w);
  const float lr = fmaxf(__fsub_rn(fminf(__fadd_rn(a.x, ahw), __fadd_rn(b.x, bhw)),
                                   fmaxf(__fsub_rn(a.x, ahw), __fsub_rn(b.x, bhw))), 0.f);
  const float tb = fmaxf(__fsub_rn(fminf(__fadd_rn(a.y, ahh), __fadd_rn(b.y, bhh)),
                                   fmaxf(__fsub_rn(a.y, ahh), __fsub_rn(b.y, bhh))), 0.f);
  const float inter = __fmul_rn(lr, tb);
  const float uni = __fsub_rn(__fadd_rn(__fmul_rn(a.z, a.w), __fmul_rn(b.z, b.w)), inter);
  return __fdiv_rn(inter, uni);
}

// Exclusive block scan of a 0/1 flag in thread order; returns this thread's offset and the
// block total.  Uses one ballot per warp + a 32-entry smem table.
__device__ __forceinline__ int block_scan_flag(bool flag, int* warp_tot, int& total) {
  const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  const int in_warp = __popc(bal & ((1u << lane) - 1u));
  __syncthreads();                       // protect warp_tot from the previous use
  if (lane == 0) warp_tot[wid] = __popc(bal);
  __syncthreads();
  int off = 0, tot = 0;
#pragma unroll
  for (int i = 0; i < FT / 32; ++i) {
    const int c = warp_tot[i];
    if (i < (int)wid) off += c;
    tot += c;
  }
  total = tot;
  return off + in_warp;
}

__global__ void __launch_bounds__(FT)
filter_kernel(const float* __restrict__ boxes, const float* __restrict__ probs,
              const long long* __restrict__ cls, int A, int classes, int top_n,
              float prob_thresh, float nms_thresh, sqdet_det* __restrict__ dets,
              int* __restrict__ counts, int max_dets) {
  __shared__ unsigned long long s_key[FCAP];   // (order_key << 32) | (~anchor)
  __shared__ float4 s_box[FCAP];
  __shared__ int s_cls[FCAP];
  __shared__ unsigned char s_keep[FCAP];
  __shared__ int s_hist[256];
  __shared__ int s_warp[FT / 32];
  __shared__ unsigned s_prefix;
  __shared__ int s_remaining;

  const int img = blockIdx.x;
  const int tid = threadIdx.x;
  const float* pr = probs + (long long)img * A;
  const float4* bx = reinterpret_cast<const float4*>(boxes) + (long long)img * A;
  const long long* cl = cls + (long long)img * A;
  sqdet_det* out = dets + (long long)img * max_dets;

  const bool topn_branch = (top_n > 0 && top_n < A);     // nn_skeleton.py:711
  int M = 0;                                              // number of candidates

  if (topn_branch) {
    // Each thread owns a contiguous run of `per` anchors, so one block scan orders the whole
    // image (17 runs of block scans per image were most of this kernel's 80 us).  Keys are
    // cached in registers when the run is short enough, else re-read from L2.
    constexpr int KCACHE = 24;
    const int per = (A + FT - 1) / FT;
    const int i_lo = tid * per, i_hi = min(A, i_lo + per);
    const bool cached = per <= KCACHE;
    unsigned kc[KCACHE];
    if (cached) {
#pragma unroll
      for (int j = 0; j < KCACHE; ++j)
        kc[j] = (i_lo + j < i_hi) ? order_key(pr[i_lo + j]) : 0u;
    }
    // ---- radix select: key of the top_n-th largest score --------------------------------
    if (tid == 0) { s_prefix = 0u; s_remaining = top_n; }
    unsigned mask = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) s_hist[tid] = 0;
      __syncthreads();
      const unsigned prefix = s_prefix;
      if (cached) {
#pragma unroll
        for (int j = 0; j < KCACHE; ++j) {
          const bool in = (i_lo + j < i_hi) && ((kc[j] & mask) == prefix);
          // warp-aggregated histogram: one atomic per distinct digit per warp
          const unsigned digit = (kc[j] >> shift) & 255u;
          const unsigned act = __ballot_sync(0xffffffffu, in);
          if (in) {
            const unsigned peers = __match_any_sync(act, digit);
            if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1))
              atomicAdd(&s_hist[digit], __popc(peers));
          }
        }
      } else {
        for (int i = i_lo; i < i_hi; ++i) {
          const unsigned k = order_key(pr[i]);
          if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & 255u], 1);
        }
      }
      __syncthreads();
      if (tid == 0) {
        int rem = s_remaining, d = 255;
        for (; d > 0; --d) {
          const int h = s_hist[d];
          if (h >= rem) break;
          rem -= h;
        }
        s_remaining = rem;                       // how many to take among digit d
        s_prefix = prefix | ((unsigned)d << shift);
      }
      mask |= 255u << shift;
      __syncthreads();
    }
    const unsigned T = s_prefix;
    const int take_eq = s_remaining;             // ties at T: lowest anchor ids first
    const int n_gt = top_n - take_eq;
    // ---- ordered compaction: [0,n_gt) scores > T, [n_gt, top_n) scores == T --------------
    int c_gt = 0, c_eq = 0;
    if (cached) {
#pragma unroll
      for (int j = 0; j < KCACHE; ++j)
        if (i_lo + j < i_hi) { c_gt += (kc[j] > T); c_eq += (kc[j] == T); }
    } else {
      for (int i = i_lo; i < i_hi; ++i) {
        const unsigned k = order_key(pr[i]);
        c_gt += (k > T);
        c_eq += (k == T);
      }
    }
    // exclusive block scan of (c_gt, c_eq) in thread order
    int o_gt, o_eq;
    {
      const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
      int v_gt = c_gt, v_eq = c_eq;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, v_gt, off);
        const int b2 = __shfl_up_sync(0xffffffffu, v_eq, off);
        if (lane >= (unsigned)off) { v_gt += a; v_eq += b2; }
      }
      __syncthreads();
      if (lane == 31) { s_warp[wid] = v_gt; s_hist[wid] = v_eq; }
      __syncthreads();
      int base_gt = 0, base_eq = 0;
      for (int w = 0; w < (int)wid; ++w) { base_gt += s_warp[w]; base_eq += s_hist[w]; }
      o_gt = base_gt + v_gt - c_gt;
      o_eq = base_eq + v_eq - c_eq;
    }
    auto place = [&](unsigned k, int i) {
      int slot = -1;
      if (k > T) slot = o_gt++;
      else if (k == T) { if (o_eq < take_eq) slot = n_gt + o_eq; ++o_eq; }
      if (slot >= 0) {
        s_key[slot] = ((unsigned long long)k << 32) | (unsigned)(~(unsigned)i);
        s_box[slot] = bx[i];
        s_cls[slot] = (int)cl[i];
      }
    };
    if (cached) {
#pragma unroll
      for (int j = 0; j < KCACHE; ++j)
        if (i_lo + j < i_hi && kc[j] >= T) place(kc[j], i_lo + j);
    } else {
      for (int i = i_lo; i < i_hi; ++i) place(order_key(pr[i]), i);
    }
    M = top_n;
    __syncthreads();
    // ---- bitonic sort, descending in (score, -anchor) ------------------------------------
    int P = 1;
    while (P < M) P <<= 1;
    for (int i = M + tid; i < P; i += FT) s_key[i] = 0ull;   // pads sort last
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {
      for (int strd = size >> 1; strd > 0; strd >>= 1) {
        for (int t = tid; t < P; t += FT) {
          const int partner = t ^ strd;
          if (partner > t) {
            const bool desc = ((t & size) == 0);
            const unsigned long long ka = s_key[t], kb = s_key[partner];
            if (desc ? (ka < kb) : (ka > kb)) {
              s_key[t] = kb; s_key[partner] = ka;
              const float4 tb4 = s_box[t]; s_box[t] = s_box[partner]; s_box[partner] = tb4;
              const int tc = s_cls[t]; s_cls[t] = s_cls[partner]; s_cls[partner] = tc;
            }
          }
        }
        __syncthreads();
      }
    }
  } else {
    // ---- threshold branch (nn_skeleton.py:716-720): probs > PROB_THRESH, original order ---
    int run = 0;
    bool overflow = false;
    for (int base = 0; base < A; base += FT) {
      const int i = base + tid;
      const bool ok = (i < A) && (pr[i] > prob_thresh);
      int tot;
      const int o = block_scan_flag(ok, s_warp, tot);
      const int slot = run + o;
      if (ok && slot < FCAP && slot < max_dets) {
        s_key[slot] = ((unsigned long long)order_key(pr[i]) << 32) | (unsigned)(~(unsigned)i);
        s_box[slot] = bx[i];
        s_cls[slot] = (int)cl[i];
      }
      run += tot;
    }
    if (run > FCAP || run > max_dets) overflow = true;
    if (overflow) {
      if (tid == 0) counts[img] = -1;
      for (int i = tid; i < max_dets; i += FT) {
        sqdet_det z; z.anchor = -1; z.cls = -1; z.prob = 0.f; z.cx = z.cy = z.w = z.h = 0.f;
        out[i] = z;
      }
      return;
    }
    M = run;
    __syncthreads();
  }

  // ---- NMS (util.py:56-76): j is dropped iff some higher-ranked same-class i overlaps ----
  for (int j = tid; j < M; j += FT) {
    const int cj = s_cls[j];
    bool keep = (cj >= 0 && cj < classes);
    if (keep) {
      const unsigned long long kj = s_key[j];
      const float4 bj = s_box[j];
      for (int i = 0; i < M; ++i) {
        if (i == j || s_cls[i] != cj || !(s_key[i] > kj)) continue;
        if (iou_ref(bj, s_box[i]) > nms_thresh) { keep = false; break; }
      }
    }
    s_keep[j] = keep ? 1 : 0;
  }
  __syncthreads();
  // ---- class-grouped output order (nn_skeleton.py:726-733) --------------------------------
  for (int j = tid; j < M; j += FT) {
    if (!s_keep[j]) continue;
    const int cj = s_cls[j];
    int pos = 0;
    for (int i = 0; i < M; ++i)
      pos += (s_keep[i] && (s_cls[i] < cj || (s_cls[i] == cj && i < j))) ? 1 : 0;
    const unsigned long long kj = s_key[j];
    const int anchor = (int)(~(unsigned)(kj & 0xffffffffull));
    sqdet_det r;
    r.anchor = anchor;
    r.cls = cj;
    r.prob = pr[anchor];
    const float4 b4 = s_box[j];
    r.cx = b4.x; r.cy = b4.y; r.w = b4.z; r.h = b4.w;
    out[pos] = r;
  }
  int my = 0;
  for (int j = tid; j < M; j += FT) my += s_keep[j];
  // total kept (block reduction through the scan helper's table)
  int tot = 0;
  {
    // reduce `my` over the block
    for (int o = 16; o > 0; o >>= 1) my += __shfl_xor_sync(0xffffffffu, my, o);
    __syncthreads();
    if ((tid & 31) == 0) s_warp[tid >> 5] = my;
    __syncthreads();
    for (int i = 0; i < FT / 32; ++i) tot += s_warp[i];
  }
  if (tid == 0) counts[img] = tot;
  for (int i = tot + tid; i < max_dets; i += FT) {   // deterministic padding
    sqdet_det z; z.anchor = -1; z.cls = -1; z.prob = 0.f; z.cx = z.cy = z.w = z.h = 0.f;
    out[i] = z;
  }
}

}  // namespace

int launch_interpret(const float* preds, const float* anchors, float* boxes, float* probs,
                     int64_t* cls, int B, int grid_h, int grid_w, int K, int C,
                     int image_width, int image_height, float exp_thresh,
                     cudaStream_t stream) {
  if (B <= 0 || grid_h <= 0 || grid_w <= 0 || K <= 0 || C <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "interpret: non-positive dimension");
  if ((reinterpret_cast<uintptr_t>(anchors) & 15) || (reinterpret_cast<uintptr_t>(boxes) & 15))
    return fail(SQDET_ERR_INVALID_ARG, "interpret: anchors/boxes must be 16-byte aligned");
  const int A = grid_h * grid_w * K;
  const long long total = (long long)B * A;
  // slope = np.exp(thresh) in float64, cast to fp32 where it meets the tensor (util.py:222)
  const float slope = (float)exp((double)exp_thresh);
  SQ_CUDA(launch_kernel(interpret_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream,
                        preds, anchors, boxes, probs, reinterpret_cast<long long*>(cls), B, A, K, C,
                        (float)(image_width - 1.0), (float)(image_height - 1.0), exp_thresh, slope));
  SQ_CHECK_LAUNCH("interpret_kernel");
  return SQDET_OK;
}

int launch_rescale_boxes(float* boxes, const float* scales_xy, int B, int A,
                         cudaStream_t stream) {
  if (B <= 0 || A <= 0) return fail(SQDET_ERR_INVALID_ARG, "rescale_boxes: non-positive dimension");
  if (reinterpret_cast<uintptr_t>(boxes) & 15)
    return fail(SQDET_ERR_INVALID_ARG, "rescale_boxes: boxes must be 16-byte aligned");
  const long long total = (long long)B * A;
  SQ_CUDA(launch_kernel(rescale_boxes_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0,
                        stream, reinterpret_cast<float4*>(boxes), scales_xy, A, total));
  SQ_CHECK_LAUNCH("rescale_boxes_kernel");
  return SQDET_OK;
}

int launch_topk_nms(const float* boxes, const float* probs, const int64_t* cls, int B,
                    int A, int classes, int top_n, float prob_thresh, float nms_thresh,
                    sqdet_det* dets, int32_t* counts, int max_dets, cudaStream_t stream) {
  if (B <= 0 || A <= 0 || classes <= 0 || max_dets <= 0)
    return fail(SQDET_ERR_INVALID_ARG, "topk_nms: non-positive dimension");
  if (reinterpret_cast<uintptr_t>(boxes) & 15)
    return fail(SQDET_ERR_INVALID_ARG, "topk_nms: boxes must be 16-byte aligned");
  const bool topn_branch = (top_n > 0 && top_n < A);
  if (topn_branch && (top_n > FCAP || top_n > max_dets))
    return fail(SQDET_ERR_UNSUPPORTED,
                "topk_nms: TOP_N_DETECTION above capacity (max 1024 and <= max_dets)");
  SQ_CUDA(launch_kernel(filter_kernel, dim3((unsigned)B), dim3(FT), 0, stream, boxes, probs,
                        reinterpret_cast<const long long*>(cls), A, classes, top_n, prob_thresh,
                        nms_thresh, dets, reinterpret_cast<int*>(counts), max_dets));
  SQ_CHECK_LAUNCH("filter_kernel");
  return SQDET_OK;
}

}  // namespace sqdet
