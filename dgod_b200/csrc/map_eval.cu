// COCO-style bbox mean average precision: per-image greedy matching and per-class precision / recall accumulation.
//
// Reference behaviour restated (torchmetrics MeanAveragePrecision(box_format="xyxy", iou_type="bbox") on its
// pycocotools backend: COCOeval.evaluateImg / accumulate, maskApi.c bbIou; no crowd ground truths, area range "all"):
//   * boxes go to xywh in fp32 (w = x2 - x1), then every IoU is computed in double:
//       w = min(dx + dw, gx + gw) - max(dx, gx), 0 if w <= 0; h likewise; i = w * h; u = dw * dh + gw * gh - i; i / u
//   * per (image, class): detections in descending score order (stable: ties keep input order), the first max_det
//     kept.  For each IoU threshold t, thr = min(t, 1 - 1e-10), each detection in turn takes the not yet matched GT of
//     its class with the largest IoU >= thr; on equal IoU the later GT wins.
//   * per class over all images: the kept detections in descending score order (ties: earlier image, then the order
//     above); tp / fp cumulative counts, rc = tp / npig, pr = tp / ((fp + tp) + eps), pr made non-increasing from the
//     right, and for each recall threshold r: q = pr[searchsorted(rc, r, left)], or 0 past the end.
// Every double operation is an explicit _rn intrinsic, so no contraction can move a value at a threshold.
#include "common.cuh"

namespace dgod {

constexpr int kMatchThreads = 256;
constexpr int kAccThreads = 512;
constexpr double kCocoEps = 2.220446049250313e-16;   // np.spacing(1)

struct XYWH {
  double x, y, w, h;
};

// torchvision box_convert(xyxy -> xywh) in fp32, widened to double as pycocotools receives it.
__device__ __forceinline__ XYWH to_xywh(float4 b) {
  return {(double)b.x, (double)b.y, (double)__fsub_rn(b.z, b.x), (double)__fsub_rn(b.w, b.y)};
}

// maskApi.c bbIou for one (detection, ground truth) pair, non-crowd.
__device__ __forceinline__ double bb_iou(const XYWH& d, const XYWH& g) {
  const double w = __dsub_rn(fmin(__dadd_rn(d.w, d.x), __dadd_rn(g.w, g.x)), fmax(d.x, g.x));
  if (w <= 0.0) return 0.0;
  const double h = __dsub_rn(fmin(__dadd_rn(d.h, d.y), __dadd_rn(g.h, g.y)), fmax(d.y, g.y));
  if (h <= 0.0) return 0.0;
  const double i = __dmul_rn(w, h);
  const double u = __dsub_rn(__dadd_rn(__dmul_rn(d.w, d.h), __dmul_rn(g.w, g.h)), i);
  return __ddiv_rn(i, u);
}

// IoUs of one detection with the GTs g = lane, lane + 32, ... of its label.  Kept out of line: the double division's
// slow path is a subroutine call, and inlined into the matching loop it makes ptxas spill the loop's state.
__device__ __noinline__ void iou_row(float4 det, int64_t label, const float4* s_gbox, const int64_t* s_glabel, int ng,
                                     int lane, double* w_iou) {
  const XYWH d = to_xywh(det);
  for (int g = lane; g < ng; g += 32)
    if (s_glabel[g] == label) w_iou[g] = bb_iou(d, to_xywh(s_gbox[g]));
}

// Candidate (iou, g) beats (bi, bg): a larger IoU, or the same IoU at a later GT (g = -1: no candidate).
__device__ __forceinline__ bool match_better(double iou, int g, double bi, int bg) {
  return g >= 0 && (bg < 0 || iou > bi || (iou == bi && g > bg));
}

// One CTA per image.  Shared memory: GT boxes, one IoU row per warp, GT labels, per-GT matched bits (one per
// threshold), detection labels, descending-score keys and the sort permutation.
__global__ void __launch_bounds__(kMatchThreads)
map_match_kernel(const float* __restrict__ det_boxes, const float* __restrict__ det_scores,
                 const int64_t* __restrict__ det_labels, const int* __restrict__ det_off,
                 const float* __restrict__ gt_boxes, const int64_t* __restrict__ gt_labels,
                 const int* __restrict__ gt_off, const double* __restrict__ iou_thr, int n_thr, int max_det,
                 int cap_d, int cap_g, int sort_n, uint32_t* __restrict__ tp_mask, uint8_t* __restrict__ kept) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* s_gbox = reinterpret_cast<float4*>(smem_raw);
  double* s_iou = reinterpret_cast<double*>(s_gbox + cap_g);
  int64_t* s_glabel = reinterpret_cast<int64_t*>(s_iou + (size_t)(kMatchThreads / 32) * cap_g);
  int64_t* s_label = s_glabel + cap_g;
  uint32_t* s_gtm = reinterpret_cast<uint32_t*>(s_label + cap_d);
  uint32_t* s_skey = s_gtm + cap_g;
  uint16_t* s_idx = reinterpret_cast<uint16_t*>(s_skey + cap_d);
  __shared__ double s_thr[32];

  const int img = blockIdx.x, tid = threadIdx.x;
  const int d0 = det_off[img], g0 = gt_off[img];
  // the caps are what the caller sized shared memory with; they hold for every image of a well-formed call
  const int nd = min(det_off[img + 1] - d0, cap_d), ng = min(gt_off[img + 1] - g0, cap_g);
  for (int i = tid; i < sort_n; i += kMatchThreads) {
    s_idx[i] = (uint16_t)i;
    if (i < nd) {
      s_label[i] = det_labels[d0 + i];
      // -0.0 and +0.0 tie (numpy compares them equal); ~ordered: ascending key = descending score
      s_skey[i] = ~float_ordered(__fadd_rn(det_scores[d0 + i], 0.0f));
    }
  }
  for (int g = tid; g < ng; g += kMatchThreads) {
    s_gbox[g] = ld_box(gt_boxes, g0 + g);
    s_glabel[g] = gt_labels[g0 + g];
    s_gtm[g] = 0u;
  }
  if (tid < n_thr) s_thr[tid] = fmin(iou_thr[tid], 1.0 - 1e-10);
  __syncthreads();

  // bitonic sort of the permutation by (label, descending score, index); slots >= nd sort last
  for (int k = 2; k <= sort_n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int q = tid; q < (sort_n >> 1); q += kMatchThreads) {
        const int i = 2 * q - (q & (j - 1)), l = i + j;
        const int a = s_idx[i], b = s_idx[l];
        bool a_gt_b;
        if (a >= nd || b >= nd) {
          a_gt_b = a > b;
        } else if (s_label[a] != s_label[b]) {
          a_gt_b = s_label[a] > s_label[b];
        } else if (s_skey[a] != s_skey[b]) {
          a_gt_b = s_skey[a] > s_skey[b];
        } else {
          a_gt_b = a > b;
        }
        if (a_gt_b == ((i & k) == 0)) {
          s_idx[i] = (uint16_t)b;
          s_idx[l] = (uint16_t)a;
        }
      }
      __syncthreads();
    }
  }

  // Runs of one label are matched by one warp each: detections in order, lanes over the GTs, one threshold at a time.
  const int lane = tid & 31, warp = tid >> 5, n_warps = kMatchThreads / 32;
  double* w_iou = s_iou + (size_t)warp * cap_g;       // this warp's IoUs of the current detection, one per GT
  int run = 0;
  for (int base = 0; base < nd; base += 32) {
    const int p = base + lane;
    const bool starts = p < nd && (p == 0 || s_label[s_idx[p]] != s_label[s_idx[p - 1]]);
    unsigned starts_mask = __ballot_sync(0xffffffffu, starts);
    while (starts_mask) {
      const int start = base + __ffs(starts_mask) - 1;
      starts_mask &= starts_mask - 1;
      if (run++ % n_warps != warp) continue;
      const int64_t label = s_label[s_idx[start]];
      for (int p2 = start; p2 < nd && s_label[s_idx[p2]] == label; ++p2) {
        const int i = s_idx[p2];
        const bool keep = p2 - start < max_det;
        uint32_t mask = 0u;
        if (keep) {
          iou_row(ld_box(det_boxes, d0 + i), label, s_gbox, s_glabel, ng, lane, w_iou);
          __syncwarp();
          for (int t = 0; t < n_thr; ++t) {
            double best = 0.0;
            int best_g = -1;
            for (int g = lane; g < ng; g += 32) {
              if (s_glabel[g] != label || ((s_gtm[g] >> t) & 1u)) continue;
              const double iou = w_iou[g];
              if (iou >= s_thr[t] && match_better(iou, g, best, best_g)) {
                best = iou;
                best_g = g;
              }
            }
            for (int off = 16; off > 0; off >>= 1) {
              const double o_iou = __shfl_xor_sync(0xffffffffu, best, off);
              const int o_g = __shfl_xor_sync(0xffffffffu, best_g, off);
              if (match_better(o_iou, o_g, best, best_g)) {
                best = o_iou;
                best_g = o_g;
              }
            }
            if (best_g >= 0) {
              mask |= 1u << t;
              if (lane == 0) s_gtm[best_g] |= 1u << t;
            }
            __syncwarp();
          }
        }
        if (lane == 0) {
          tp_mask[d0 + i] = mask;
          kept[d0 + i] = keep ? 1 : 0;
        }
      }
    }
  }
}

// Inclusive block scan over kAccThreads threads (op: sum or max); `total` receives the block-wide result.
template <typename T, typename Op>
__device__ __forceinline__ T block_scan(T v, Op op, T* s_warp, T& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 1; off < 32; off <<= 1) {
    const T o = __shfl_up_sync(0xffffffffu, v, off);
    if (lane >= off) v = op(o, v);
  }
  if (lane == 31) s_warp[warp] = v;
  __syncthreads();
  if (warp == 0) {
    T w = lane < kAccThreads / 32 ? s_warp[lane] : s_warp[0];
    for (int off = 1; off < kAccThreads / 32; off <<= 1) {
      const T o = __shfl_up_sync(0xffffffffu, w, off);
      if (lane >= off) w = op(o, w);
    }
    if (lane < kAccThreads / 32) s_warp[lane] = w;
  }
  __syncthreads();
  if (warp > 0) v = op(s_warp[warp - 1], v);
  total = s_warp[kAccThreads / 32 - 1];
  __syncthreads();
  return v;
}

struct SumOp {
  __device__ int operator()(int a, int b) const { return a + b; }
};
struct MaxOp {
  __device__ double operator()(double a, double b) const { return fmax(a, b); }
};

// One CTA per (class, IoU threshold): blockIdx.x = class, blockIdx.y = threshold.
__global__ void __launch_bounds__(kAccThreads)
map_accumulate_kernel(const uint32_t* __restrict__ tp_mask, const int* __restrict__ seg_off,
                      const int* __restrict__ gt_count, int n_cls, int n_rec_total, const double* __restrict__ rec_thr,
                      int n_rthr, double* __restrict__ precision, double* __restrict__ recall, double* __restrict__ ws_pr,
                      double* __restrict__ ws_rc) {
  __shared__ int s_isum[kAccThreads / 32];
  __shared__ double s_dmax[kAccThreads / 32];
  const int k = blockIdx.x, t = blockIdx.y, tid = threadIdx.x;
  const int s = seg_off[k], nd = seg_off[k + 1] - s, npig = gt_count[k];
  if (npig == 0) {                       // no ground truth: -1 everywhere, excluded from every mean
    for (int r = tid; r < n_rthr; r += kAccThreads) precision[((size_t)t * n_rthr + r) * n_cls + k] = -1.0;
    if (tid == 0) recall[(size_t)t * n_cls + k] = -1.0;
    return;
  }
  double* pr = ws_pr + (size_t)t * n_rec_total + s;
  double* rc = ws_rc + (size_t)t * n_rec_total + s;
  const double npig_d = (double)npig;
  int carry = 0;
  for (int c0 = 0; c0 < nd; c0 += kAccThreads) {
    const int i = c0 + tid;
    const int v = i < nd ? (int)((tp_mask[s + i] >> t) & 1u) : 0;
    int total;
    const int tp = block_scan(v, SumOp(), s_isum, total) + carry;
    carry += total;
    if (i < nd) {
      const double tpd = (double)tp;
      pr[i] = __ddiv_rn(tpd, __dadd_rn((double)(i + 1), kCocoEps));    // fp + tp = i + 1, exact
      rc[i] = __ddiv_rn(tpd, npig_d);
    }
  }
  __syncthreads();
  double run_max = 0.0;                  // precisions are >= 0
  for (int end = nd; end > 0; end -= kAccThreads) {
    const int i = end - 1 - tid;
    const double v = i >= 0 ? pr[i] : 0.0;
    double total;
    const double m = fmax(block_scan(v, MaxOp(), s_dmax, total), run_max);
    run_max = fmax(run_max, total);
    if (i >= 0) pr[i] = m;
  }
  __syncthreads();
  for (int r = tid; r < n_rthr; r += kAccThreads) {
    const double thr = rec_thr[r];
    int lo = 0, hi = nd;                 // first i with rc[i] >= thr
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (rc[mid] < thr) lo = mid + 1;
      else hi = mid;
    }
    precision[((size_t)t * n_rthr + r) * n_cls + k] = lo < nd ? pr[lo] : 0.0;
  }
  if (tid == 0) recall[(size_t)t * n_cls + k] = nd ? rc[nd - 1] : 0.0;
}

static int next_pow2_int(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

static size_t match_smem_bytes(int cap_d, int cap_g, int sort_n) {
  return (size_t)cap_g * (sizeof(float4) + (kMatchThreads / 32) * sizeof(double) + sizeof(int64_t) + sizeof(uint32_t)) +
         (size_t)cap_d * (sizeof(int64_t) + sizeof(uint32_t)) + (size_t)sort_n * sizeof(uint16_t);
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_map_match(const float* det_boxes, const float* det_scores, const int64_t* det_labels,
                              const int* det_offsets, const float* gt_boxes, const int64_t* gt_labels,
                              const int* gt_offsets, int n_img, int max_dets_per_image, int max_gts_per_image,
                              const double* iou_thresholds, int n_thr, int max_det, uint32_t* tp_mask, uint8_t* kept,
                              dgod_stream_t stream) {
  DGOD_REQUIRE(n_img >= 0, "dgod_map_match: negative image count");
  DGOD_REQUIRE(n_thr >= 1 && n_thr <= DGOD_MAP_MAX_IOU_THRESHOLDS, "dgod_map_match: 1..%d IoU thresholds, got %d",
               DGOD_MAP_MAX_IOU_THRESHOLDS, n_thr);
  DGOD_REQUIRE(max_det >= 1, "dgod_map_match: max_det must be >= 1, got %d", max_det);
  DGOD_REQUIRE(max_dets_per_image >= 0 && max_dets_per_image <= DGOD_MAP_MAX_DETS_PER_IMAGE,
               "dgod_map_match: at most %d detections per image, got %d", DGOD_MAP_MAX_DETS_PER_IMAGE,
               max_dets_per_image);
  DGOD_REQUIRE(max_gts_per_image >= 0 && max_gts_per_image <= DGOD_MAP_MAX_GTS_PER_IMAGE,
               "dgod_map_match: at most %d ground truths per image, got %d", DGOD_MAP_MAX_GTS_PER_IMAGE,
               max_gts_per_image);
  if (n_img == 0 || max_dets_per_image == 0) return DGOD_OK;
  DGOD_REQUIRE(det_boxes && det_scores && det_labels && det_offsets && gt_offsets && iou_thresholds && tp_mask && kept,
               "dgod_map_match: null pointer");
  DGOD_REQUIRE(max_gts_per_image == 0 || (gt_boxes && gt_labels), "dgod_map_match: null ground-truth pointer");
  DGOD_REQUIRE(aligned16(det_boxes) && aligned16(gt_boxes), "dgod_map_match: boxes must be 16-byte aligned");
  const int sort_n = next_pow2_int(max_dets_per_image);
  const size_t smem = match_smem_bytes(max_dets_per_image, max_gts_per_image, sort_n);
  static bool attr_set = false;          // idempotent; racing threads set the same value
  if (!attr_set) {
    DGOD_CUDA(cudaFuncSetAttribute(map_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)match_smem_bytes(DGOD_MAP_MAX_DETS_PER_IMAGE, DGOD_MAP_MAX_GTS_PER_IMAGE,
                                                         DGOD_MAP_MAX_DETS_PER_IMAGE)));
    attr_set = true;
  }
  map_match_kernel<<<n_img, kMatchThreads, smem, (cudaStream_t)stream>>>(
      det_boxes, det_scores, det_labels, det_offsets, gt_boxes, gt_labels, gt_offsets, iou_thresholds, n_thr, max_det,
      max_dets_per_image, max_gts_per_image, sort_n, tp_mask, kept);
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" size_t dgod_map_accumulate_workspace_bytes(int n_records, int n_thr) {
  if (n_records < 0 || n_thr < 0) return 0;
  return 2 * align_up((size_t)n_records * n_thr * sizeof(double), 256);
}

extern "C" int dgod_map_accumulate(const uint32_t* tp_mask, const int* seg_offsets, const int* gt_counts, int n_classes,
                                   int n_records, const double* rec_thresholds, int n_rec_thr, int n_thr,
                                   double* precision, double* recall, void* workspace, size_t workspace_bytes,
                                   dgod_stream_t stream) {
  DGOD_REQUIRE(n_classes >= 0 && n_records >= 0 && n_rec_thr >= 0, "dgod_map_accumulate: negative size");
  DGOD_REQUIRE(n_thr >= 1 && n_thr <= DGOD_MAP_MAX_IOU_THRESHOLDS, "dgod_map_accumulate: 1..%d IoU thresholds, got %d",
               DGOD_MAP_MAX_IOU_THRESHOLDS, n_thr);
  if (n_classes == 0) return DGOD_OK;
  DGOD_REQUIRE(seg_offsets && gt_counts && precision && recall && (n_records == 0 || tp_mask) &&
               (n_rec_thr == 0 || rec_thresholds),
               "dgod_map_accumulate: null pointer");
  if (workspace_bytes < dgod_map_accumulate_workspace_bytes(n_records, n_thr)) {
    set_error("dgod_map_accumulate: workspace of %zu bytes, %zu needed", workspace_bytes,
              dgod_map_accumulate_workspace_bytes(n_records, n_thr));
    return DGOD_ERR_WORKSPACE;
  }
  Workspace ws(workspace, workspace_bytes);
  double* pr = ws.take<double>((size_t)n_records * n_thr);
  double* rc = ws.take<double>((size_t)n_records * n_thr);
  map_accumulate_kernel<<<dim3(n_classes, n_thr), kAccThreads, 0, (cudaStream_t)stream>>>(
      tp_mask, seg_offsets, gt_counts, n_classes, n_records, rec_thresholds, n_rec_thr, precision, recall, pr, rc);
  DGOD_LAUNCHED();
  return DGOD_OK;
}
