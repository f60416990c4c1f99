// box_iou, Matcher and the fused IoU+Matcher+label kernel (SURVEY.md §8a rows A5, A6).
//
// Reference behaviour restated (TV = torchvision 0.26.0):
//   box_iou            TV ops/boxes.py:308-370
//   Matcher.__call__   TV models/detection/_utils.py:357-416
//   RPN labels         TV models/detection/rpn.py:193-229
//   RoI-head labels    TV models/detection/roi_heads.py:580-613
//
// Data layout: boxes are [n,4] fp32 xyxy rows (one 128-bit load per box); ground truths of a
// batch are concatenated with an offsets vector.  The [M,N] IoU matrix is never written: the
// per-prediction arg-max and the per-ground-truth row maximum (for allow_low_quality_matches)
// are both recomputed from the 16-byte box records, so the kernels move 16 B per box in and
// 8..40 B per box out — pure HBM/latency bound, no reuse to stage beyond the ground truths,
// which sit in shared memory.
#include "common.cuh"

namespace dgod {

constexpr int kMatchThreads = 256;
constexpr int kGtChunk = 256;  // ground truths staged per shared-memory pass

struct GtTile {
  float4 box[kGtChunk];
  float area[kGtChunk];
};

__device__ __forceinline__ void load_gt_tile(GtTile& t, const float* gt_boxes, int g0, int cnt) {
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    float4 b = ld_box(gt_boxes, g0 + i);
    t.box[i] = b;
    t.area[i] = box_area_exact(b.x, b.y, b.z, b.w);
  }
}

// ---------------------------------------------------------------------------- box_iou
__global__ void __launch_bounds__(256) box_iou_kernel(const float* __restrict__ b1, int n1,
                                                      const float* __restrict__ b2, int n2,
                                                      float* __restrict__ out) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)n1 * n2;
  if (t >= total) return;
  int i = (int)(t / n2), j = (int)(t % n2);
  float4 a = ld_box(b1, i), b = ld_box(b2, j);
  out[t] = iou_exact(a, box_area_exact(a.x, a.y, a.z, a.w), b, box_area_exact(b.x, b.y, b.z, b.w));
}

// ---------------------------------------------------------------------------- fused path
// The candidate slots of one image in the three layouts of dgod_iou_match.  Slot n < nb gets its outputs at out0 + n;
// it holds a box when n < nv: row b0 + n of `boxes` while n < n_prop, past that (padded layout) ground truth n - n_prop.
struct ImageSlots {
  int nb, nv, n_prop;
  long long b0, out0;
};

__device__ __forceinline__ ImageSlots image_slots(int img, int n_gt, const int32_t* __restrict__ box_offsets,
                                                  const int32_t* __restrict__ box_counts, int n_boxes, int n_slots) {
  ImageSlots s;
  if (box_offsets) {                       // ragged: image i owns boxes[box_offsets[i] .. box_offsets[i+1])
    s.b0 = s.out0 = box_offsets[img];
    s.nb = s.nv = s.n_prop = box_offsets[img + 1] - box_offsets[img];
  } else if (box_counts) {                 // padded [n_img, n_boxes] rows, the image's ground truths appended
    s.b0 = (long long)img * n_boxes;
    s.out0 = (long long)img * n_slots;
    s.n_prop = min(max(box_counts[img], 0), n_boxes);
    s.nb = n_slots;
    s.nv = min(s.n_prop + n_gt, n_slots);
  } else {                                 // one set of boxes shared by every image
    s.b0 = 0;
    s.out0 = (long long)img * n_boxes;
    s.nb = s.nv = s.n_prop = n_boxes;
  }
  return s;
}

__device__ __forceinline__ float4 slot_box(const ImageSlots& s, const float* __restrict__ boxes,
                                           const float* __restrict__ gt_boxes, int g0, int n) {
  return n < s.n_prop ? ld_box(boxes, s.b0 + n) : ld_box(gt_boxes, g0 + (n - s.n_prop));
}

// Pass 1 (allow_low_quality only): row maximum of the implicit IoU matrix per ground truth.
__global__ void __launch_bounds__(kMatchThreads)
iou_rowmax_kernel(const float* __restrict__ gt_boxes, const int32_t* __restrict__ gt_offsets,
                  const float* __restrict__ boxes, const int32_t* __restrict__ box_offsets,
                  const int32_t* __restrict__ box_counts, int n_boxes, int n_slots,
                  uint32_t* __restrict__ gt_max /* ordered keys, zero-initialised */) {
  __shared__ GtTile tile;
  __shared__ uint32_t smax[kGtChunk];
  const int img = blockIdx.y;
  const int g0 = gt_offsets[img], g1 = gt_offsets[img + 1];
  const ImageSlots s = image_slots(img, g1 - g0, box_offsets, box_counts, n_boxes, n_slots);
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x * blockDim.x >= s.nv) return;  // whole block idle (uniform)
  const bool active = n < s.nv;
  float4 bx = make_float4(0, 0, 0, 0);
  float ba = 0.f;
  if (active) {
    bx = slot_box(s, boxes, gt_boxes, g0, n);
    ba = box_area_exact(bx.x, bx.y, bx.z, bx.w);
  }
  for (int c0 = g0; c0 < g1; c0 += kGtChunk) {
    const int cnt = min(kGtChunk, g1 - c0);
    __syncthreads();
    load_gt_tile(tile, gt_boxes, c0, cnt);
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) smax[i] = 0u;
    __syncthreads();
    for (int m = 0; m < cnt; ++m) {
      uint32_t key = 0u;
      if (active) key = float_ordered(iou_exact_skip(tile.box[m], tile.area[m], bx, ba));
      key = __reduce_max_sync(0xffffffffu, key);
      if ((threadIdx.x & 31) == 0 && key > smax[m]) atomicMax(&smax[m], key);   // smax only grows: a stale read is safe
    }
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) atomicMax(&gt_max[c0 + i], smax[i]);
  }
}

// Pass 2: arg-max over ground truths, thresholds, low-quality restore, derived outputs.
__global__ void __launch_bounds__(kMatchThreads)
iou_match_kernel(const float* __restrict__ gt_boxes, const int64_t* __restrict__ gt_labels,
                 const int32_t* __restrict__ gt_offsets, const float* __restrict__ boxes,
                 const int32_t* __restrict__ box_offsets, const int32_t* __restrict__ box_counts, int n_boxes,
                 int n_slots, float high, float low,
                 const uint32_t* __restrict__ gt_max /* NULL when !allow_low_quality */,
                 int64_t* __restrict__ matched_idx, float* __restrict__ labels_f32,
                 int64_t* __restrict__ labels_i64, int64_t* __restrict__ clamped_idx,
                 float* __restrict__ matched_boxes) {
  __shared__ GtTile tile;
  __shared__ uint32_t smax[kGtChunk];
  const int img = blockIdx.y;
  const int g0 = gt_offsets[img], g1 = gt_offsets[img + 1];
  const ImageSlots s = image_slots(img, g1 - g0, box_offsets, box_counts, n_boxes, n_slots);
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x * blockDim.x >= s.nb) return;
  const bool active = n < s.nv;
  float4 bx = make_float4(0, 0, 0, 0);
  float ba = 0.f;
  if (active) {
    bx = slot_box(s, boxes, gt_boxes, g0, n);
    ba = box_area_exact(bx.x, bx.y, bx.z, bx.w);
  }
  float best = 0.f;
  int best_m = -1;
  bool tie_with_rowmax = false;
  for (int c0 = g0; c0 < g1; c0 += kGtChunk) {
    const int cnt = min(kGtChunk, g1 - c0);
    __syncthreads();
    load_gt_tile(tile, gt_boxes, c0, cnt);
    if (gt_max)
      for (int i = threadIdx.x; i < cnt; i += blockDim.x) smax[i] = gt_max[c0 + i];
    __syncthreads();
    if (active) {
      for (int m = 0; m < cnt; ++m) {
        float v = iou_exact_skip(tile.box[m], tile.area[m], bx, ba);
        // Tensor.max(dim=0) keeps the first maximal index; NaN wins like in torch.
        if (best_m < 0 || v > best || (v != v && best == best)) { best = v; best_m = c0 - g0 + m; }
        if (gt_max) tie_with_rowmax |= (float_ordered(v) == smax[m]);
      }
    }
  }
  if (n >= s.nb) return;
  const long long o = s.out0 + n;
  if (!active) {                           // padded layout: a slot past the image's candidates is ignored
    if (matched_idx) matched_idx[o] = -2;
    if (clamped_idx) clamped_idx[o] = 0;
    if (labels_f32) labels_f32[o] = -1.f;
    if (labels_i64) labels_i64[o] = -1;
    if (matched_boxes) reinterpret_cast<float4*>(matched_boxes)[o] = make_float4(0, 0, 0, 0);
    return;
  }
  long long idx;
  if (best_m < 0) {
    idx = -1;  // image without ground truth: everything is background
  } else {
    idx = best_m;
    if (best < low) idx = -1;                        // BELOW_LOW_THRESHOLD
    else if (best < high) idx = -2;                  // BETWEEN_THRESHOLDS (best >= low here)
    if (tie_with_rowmax) idx = best_m;               // set_low_quality_matches_
  }
  const long long cl = idx < 0 ? 0 : idx;
  if (matched_idx) matched_idx[o] = idx;
  if (clamped_idx) clamped_idx[o] = cl;
  if (labels_f32) labels_f32[o] = idx >= 0 ? 1.f : (idx == -1 ? 0.f : -1.f);
  if (labels_i64) {
    long long lab = 0;
    if (best_m >= 0) {
      lab = gt_labels ? gt_labels[g0 + cl] : 1;
      if (idx == -1) lab = 0;
      if (idx == -2) lab = -1;
    }
    labels_i64[o] = lab;
  }
  if (matched_boxes) {
    float4 r = make_float4(0, 0, 0, 0);
    if (best_m >= 0) r = ld_box(gt_boxes, g0 + cl);
    reinterpret_cast<float4*>(matched_boxes)[o] = r;
  }
}

// ---------------------------------------------------------------------------- Matcher on a matrix
__global__ void __launch_bounds__(256)
matrix_rowmax_kernel(const float* __restrict__ q, int m, int n, uint32_t* __restrict__ row_max) {
  __shared__ uint32_t s[8];
  const int r = blockIdx.x;
  uint32_t key = 0u;
  for (int j = threadIdx.x; j < n; j += blockDim.x) key = max(key, float_ordered(q[(size_t)r * n + j]));
  key = __reduce_max_sync(0xffffffffu, key);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = key;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) key = max(key, s[w]);
    row_max[r] = key;
  }
}

__global__ void __launch_bounds__(256)
matrix_match_kernel(const float* __restrict__ q, int m, int n, float high, float low,
                    const uint32_t* __restrict__ row_max, int64_t* __restrict__ matches) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  float best = q[j];
  int best_m = 0;
  bool tie = row_max && float_ordered(best) == row_max[0];
  for (int r = 1; r < m; ++r) {
    float v = q[(size_t)r * n + j];
    if (v > best || (v != v && best == best)) { best = v; best_m = r; }
    if (row_max) tie |= (float_ordered(v) == row_max[r]);
  }
  long long idx = best_m;
  if (best < low) idx = -1;
  else if (best < high) idx = -2;
  if (tie) idx = best_m;
  matches[j] = idx;
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_box_iou(const float* boxes1, int n1, const float* boxes2, int n2, float* iou,
                            dgod_stream_t stream) {
  DGOD_REQUIRE(n1 >= 0 && n2 >= 0, "dgod_box_iou: negative size");
  if (n1 == 0 || n2 == 0) return DGOD_OK;
  DGOD_REQUIRE(boxes1 && boxes2 && iou, "dgod_box_iou: null pointer");
  long long total = (long long)n1 * n2;
  box_iou_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(boxes1, n1, boxes2, n2, iou);
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" size_t dgod_matcher_workspace_bytes(int m) {
  return align_up((size_t)(m > 0 ? m : 1) * sizeof(uint32_t), 256);
}

extern "C" int dgod_matcher(const float* quality, int m, int n, double high_threshold,
                            double low_threshold, int allow_low_quality, int64_t* matches,
                            void* workspace, size_t workspace_bytes, dgod_stream_t stream) {
  // TV _utils.py:368-373: an empty matrix is an error, not an empty result.
  DGOD_REQUIRE(m > 0, "No ground-truth boxes available for one of the images during training");
  DGOD_REQUIRE(n > 0, "No proposal boxes available for one of the images during training");
  DGOD_REQUIRE(quality && matches, "dgod_matcher: null pointer");
  DGOD_REQUIRE(low_threshold <= high_threshold, "low_threshold should be <= high_threshold");
  cudaStream_t st = (cudaStream_t)stream;
  uint32_t* row_max = nullptr;
  if (allow_low_quality) {
    if (!workspace || workspace_bytes < dgod_matcher_workspace_bytes(m)) {
      set_error("dgod_matcher: workspace too small");
      return DGOD_ERR_WORKSPACE;
    }
    row_max = (uint32_t*)workspace;
    matrix_rowmax_kernel<<<m, 256, 0, st>>>(quality, m, n, row_max);
    DGOD_LAUNCHED();
  }
  matrix_match_kernel<<<cdiv(n, 256), 256, 0, st>>>(quality, m, n, (float)high_threshold,
                                                    (float)low_threshold, row_max, matches);
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" size_t dgod_iou_match_workspace_bytes(int n_img, int total_gt) {
  (void)n_img;
  return align_up((size_t)(total_gt > 0 ? total_gt : 1) * sizeof(uint32_t), 256);
}

extern "C" int dgod_iou_match(const float* gt_boxes, const int64_t* gt_labels,
                              const int32_t* gt_offsets, int n_img, int total_gt,
                              const float* boxes, const int32_t* box_offsets, const int32_t* box_counts,
                              int n_boxes, int max_boxes_per_img, double high_threshold, double low_threshold,
                              int allow_low_quality, int64_t* matched_idx, float* labels_f32,
                              int64_t* labels_i64, int64_t* clamped_idx, float* matched_boxes,
                              void* workspace, size_t workspace_bytes, dgod_stream_t stream) {
  DGOD_REQUIRE(n_img >= 0 && total_gt >= 0 && n_boxes >= 0 && max_boxes_per_img >= 0,
               "dgod_iou_match: negative size");
  DGOD_REQUIRE(low_threshold <= high_threshold, "low_threshold should be <= high_threshold");
  DGOD_REQUIRE(!(box_offsets && box_counts), "dgod_iou_match: box_offsets and box_counts are exclusive");
  if (n_img == 0 || max_boxes_per_img == 0 || (n_boxes == 0 && !box_counts)) return DGOD_OK;
  DGOD_REQUIRE(gt_offsets && (boxes || n_boxes == 0), "dgod_iou_match: null pointer");
  DGOD_REQUIRE(total_gt == 0 || gt_boxes, "dgod_iou_match: gt_boxes is null");
  DGOD_REQUIRE(!box_counts || max_boxes_per_img >= n_boxes, "dgod_iou_match: fewer slots than padded boxes");
  if (!box_offsets && !box_counts) max_boxes_per_img = n_boxes;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(cdiv(max_boxes_per_img, kMatchThreads), n_img);
  uint32_t* gt_max = nullptr;
  if (allow_low_quality && total_gt > 0) {
    if (!workspace || workspace_bytes < dgod_iou_match_workspace_bytes(n_img, total_gt)) {
      set_error("dgod_iou_match: workspace too small");
      return DGOD_ERR_WORKSPACE;
    }
    gt_max = (uint32_t*)workspace;
    DGOD_CUDA(cudaMemsetAsync(gt_max, 0, (size_t)total_gt * sizeof(uint32_t), st));
    iou_rowmax_kernel<<<grid, kMatchThreads, 0, st>>>(gt_boxes, gt_offsets, boxes, box_offsets,
                                                      box_counts, n_boxes, max_boxes_per_img, gt_max);
    DGOD_LAUNCHED();
  }
  iou_match_kernel<<<grid, kMatchThreads, 0, st>>>(
      gt_boxes, gt_labels, gt_offsets, boxes, box_offsets, box_counts, n_boxes, max_boxes_per_img,
      (float)high_threshold, (float)low_threshold, gt_max, matched_idx, labels_f32, labels_i64,
      clamped_idx, matched_boxes);
  DGOD_LAUNCHED();
  return DGOD_OK;
}
