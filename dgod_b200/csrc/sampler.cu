// BalancedPositiveNegativeSampler on the device without host synchronisation (SURVEY.md §8f rank 1;
// TV models/detection/_utils.py:11-71, used by the RPN loss fasterrcnn.py:119-123 and by
// RoIHeads.subsample TV roi_heads.py:615-622 <- fasterrcnn.py:272).
//
// Upstream draws `randperm(#pos)[:num_pos]` and `randperm(#neg)[:num_neg]` per image — a uniformly random subset of
// the positives and of the negatives — and returns boolean masks that the callers turn into index lists with
// torch.where (a host synchronisation each).  Here every candidate carries a uniform random key; the subset is "the k
// smallest keys of the class", found per image by a 4-pass 8-bit radix select over the key bits in ONE launch for the
// whole batch, and the survivors are written as fixed-capacity index lists in ascending index order (the order
// torch.where would give) plus validity masks.  Equal keys are resolved by ascending index.  Keys can be injected,
// which is how the tests force the selection the reference made.
//
// One 8-CTA cluster per image (a contiguous slice of the candidates per CTA, histograms summed through distributed
// shared memory): labels + keys are read 5 times (4 radix passes for both classes at once + the gather), L2 resident
// (155 520 anchors x 8 B per image).  Latency-bound; replaces two 155 k-wide torch.topk launches and their temporaries.
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace dgod {

constexpr int kSampThreads = 1024;

template <typename L> __device__ __forceinline__ int label_class(const L* __restrict__ labels, long long i);
// 1: positive (label >= 1), 0: negative (label == 0), -1: ignored
template <> __device__ __forceinline__ int label_class<float>(const float* __restrict__ labels, long long i) {
  const float v = __ldg(labels + i);
  return v >= 1.f ? 1 : (v == 0.f ? 0 : -1);
}
template <> __device__ __forceinline__ int label_class<int64_t>(const int64_t* __restrict__ labels, long long i) {
  const long long v = __ldg(labels + i);
  return v >= 1 ? 1 : (v == 0 ? 0 : -1);
}

constexpr int kSampUnroll = 4;          // independent (label, key) loads in flight per thread
constexpr int kSampCluster = 8;         // CTAs (one cluster) sharing the candidates of one image, a contiguous slice each
constexpr int kSampMaxList = 1024;      // survivors of both classes per image handled by the in-shared-memory sort

struct SampShared {
  unsigned hist[2][256];                // [class][digit], this CTA's slice
  unsigned warp[kSampThreads / 32];
  unsigned prefix[2], remaining[2], total[2], n_equal[2];
  unsigned cnt_below[2], cnt_eq[2];     // this slice: survivors-to-be below / at the k-th key, per class
  unsigned base_below[2], base_eq[2];
  unsigned n_list;
  int list[kSampMaxList];               // survivors of this slice, any order, then sorted by (class, index)
};

// class (1 positive, 0 negative, -1 ignored) and order-preserving key bits of element e
template <typename L>
__device__ __forceinline__ void load_elem(const L* __restrict__ labels, const float* __restrict__ keys, int e, int hi, int& cls,
                                          unsigned& key) {
  cls = -1;
  key = 0;
  if (e < hi) {
    cls = label_class<L>(labels, e);
    key = float_ordered(__ldg(keys + e));
  }
}

// One cluster of kSampCluster CTAs per image; CTA `rank` owns the contiguous slice [lo, hi) of the image's candidates, so
// "ascending index" across the cluster is "rank-major, then ascending inside the slice".
template <typename L>
__global__ void __cluster_dims__(kSampCluster, 1, 1) __launch_bounds__(kSampThreads)
balanced_sample_kernel(const L* __restrict__ labels, const float* __restrict__ keys, int n, int num_pos, int batch_size,
                       int cap_pos, int cap_neg, int64_t* __restrict__ pos_idx, uint8_t* __restrict__ pos_valid,
                       int64_t* __restrict__ neg_idx, uint8_t* __restrict__ neg_valid, int32_t* __restrict__ counts) {
  __shared__ SampShared sh;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), img = blockIdx.x / kSampCluster, tid = threadIdx.x;
  labels += (size_t)img * n;
  keys += (size_t)img * n;
  const int per = (n + kSampCluster - 1) / kSampCluster;
  const int lo = min(rank * per, n), hi = min(lo + per, n);
  int64_t* out_idx[2] = {neg_idx + (size_t)img * cap_neg, pos_idx + (size_t)img * cap_pos};
  uint8_t* out_valid[2] = {neg_valid + (size_t)img * cap_neg, pos_valid + (size_t)img * cap_pos};

  // ---- 4-pass radix select of the k-th smallest key of BOTH classes at once (class 1 = positives, 0 = negatives): local
  // histograms, summed over the cluster through distributed shared memory; every CTA takes the same decision
  unsigned prefix[2] = {0, 0}, mask = 0, k[2] = {0, 0};
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = tid; i < 512; i += kSampThreads) (&sh.hist[0][0])[i] = 0;
    __syncthreads();
    for (int e0 = lo + tid; e0 < hi; e0 += kSampThreads * kSampUnroll) {
      int cls[kSampUnroll];
      unsigned key[kSampUnroll];
#pragma unroll
      for (int u = 0; u < kSampUnroll; ++u) load_elem<L>(labels, keys, e0 + u * kSampThreads, hi, cls[u], key[u]);
#pragma unroll
      for (int u = 0; u < kSampUnroll; ++u)
        if (cls[u] >= 0 && (key[u] & mask) == (cls[u] ? prefix[1] : prefix[0]) && (pass == 0 || (cls[u] ? k[1] : k[0]) > 0))
          atomicAdd(&sh.hist[cls[u]][(key[u] >> shift) & 255u], 1u);
    }
    cluster.sync();                                        // all local histograms complete
    unsigned tot = 0;
    if (tid < 512)
      for (int r = 0; r < kSampCluster; ++r) tot += (&cluster.map_shared_rank(&sh, r)->hist[0][0])[tid];
    cluster.sync();                                        // everyone has read every histogram
    if (tid < 512) (&sh.hist[0][0])[tid] = tot;            // now the image-wide histogram, in every CTA
    __syncthreads();
    if (tid < 2 && pass == 0) {
      unsigned total = 0;
      for (int b = 0; b < 256; ++b) total += sh.hist[tid][b];
      sh.total[tid] = total;
    }
    __syncthreads();
    if (tid < 2) {
      const int c = tid;
      if (pass == 0) {
        // TV _utils.py:44-50: num_pos = min(#pos, batch * fraction); num_neg = min(#neg, batch - num_pos)
        const unsigned np = min((unsigned)num_pos, sh.total[1]);
        sh.remaining[c] = c == 1 ? np : min((unsigned)batch_size - np, sh.total[0]);
      }
      unsigned rem = sh.remaining[c], b = 0;
      if (rem > 0) {
        for (; b < 255; ++b) {
          if (sh.hist[c][b] >= rem) break;
          rem -= sh.hist[c][b];
        }
      }
      sh.prefix[c] = prefix[c] | (b << shift);
      sh.remaining[c] = rem;
      if (pass == 3) sh.n_equal[c] = sh.hist[c][b];        // elements whose key IS the k-th key
    }
    __syncthreads();
    if (pass == 0) {
      const unsigned np = min((unsigned)num_pos, sh.total[1]);
      k[1] = np;
      k[0] = min((unsigned)batch_size - np, sh.total[0]);
    }
    prefix[0] = sh.prefix[0]; prefix[1] = sh.prefix[1];
    mask |= 255u << shift;
    __syncthreads();
  }
  const unsigned kth[2] = {prefix[0], prefix[1]};
  const unsigned n_eq[2] = {sh.remaining[0], sh.remaining[1]};      // how many of the equals are taken
  const bool ties_cut = (k[0] > 0 && sh.n_equal[0] != n_eq[0]) || (k[1] > 0 && sh.n_equal[1] != n_eq[1]);
  if (tid == 0) {
    sh.n_list = 0;
    sh.cnt_below[0] = sh.cnt_below[1] = sh.cnt_eq[0] = sh.cnt_eq[1] = 0;
  }
  __syncthreads();

  if (!ties_cut && k[0] + k[1] <= (unsigned)kSampMaxList) {
    // ---- common case (distinct keys at the cut): one pass gathers this slice's survivors (everything <= the k-th key of
    // its class); the short list is sorted by (class, index) and lands behind the survivors of the lower ranks
    for (int e0 = lo + tid; e0 < hi; e0 += kSampThreads * kSampUnroll) {
      int cls[kSampUnroll];
      unsigned key[kSampUnroll];
#pragma unroll
      for (int u = 0; u < kSampUnroll; ++u) load_elem<L>(labels, keys, e0 + u * kSampThreads, hi, cls[u], key[u]);
#pragma unroll
      for (int u = 0; u < kSampUnroll; ++u)
        if (cls[u] >= 0 && (cls[u] ? k[1] : k[0]) > 0 && key[u] <= (cls[u] ? kth[1] : kth[0])) {
          sh.list[atomicAdd(&sh.n_list, 1u)] = (cls[u] << 30) | (e0 + u * kSampThreads);      // n < 2^30
          atomicAdd(&sh.cnt_below[cls[u]], 1u);
        }
    }
    __syncthreads();
    const unsigned m = sh.n_list;
    for (int i = (int)m + tid; i < kSampMaxList; i += kSampThreads) sh.list[i] = 0x7fffffff;
    __syncthreads();
    for (int size = 2; size <= kSampMaxList; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const int i = tid, j = i ^ stride;
        if (j > i) {
          const bool up = (i & size) == 0;
          const int a = sh.list[i], b = sh.list[j];
          if ((a > b) == up) { sh.list[i] = b; sh.list[j] = a; }
        }
        __syncthreads();
      }
    cluster.sync();                                        // every slice's counts are final
    unsigned before[2] = {0, 0};
    for (int r = 0; r < rank; ++r) {
      const SampShared* o = cluster.map_shared_rank(&sh, r);
      before[0] += o->cnt_below[0];
      before[1] += o->cnt_below[1];
    }
    const unsigned mine0 = sh.cnt_below[0];
    for (int i = tid; i < (int)m; i += kSampThreads) {
      const int v = sh.list[i], c = v >> 30, e = v & 0x3fffffff;
      const int pos = (int)(c ? before[1] : before[0]) + (c == 0 ? i : i - (int)mine0);
      int64_t* oi = c ? out_idx[1] : out_idx[0];
      uint8_t* ov = c ? out_valid[1] : out_valid[0];
      if (pos < (c ? cap_pos : cap_neg)) { oi[pos] = e; ov[pos] = 1; }
    }
  } else {
    // ---- equal keys at the cut (or more survivors than the list holds): count below / equal per slice, exchange, then an
    // ordered compaction chunk by chunk — everything below the k-th key of its class, and the first n_eq equal ones
    // image-wide, land in ascending index order
    for (int e0 = lo + tid; e0 < hi; e0 += kSampThreads) {
      int cls;
      unsigned key;
      load_elem<L>(labels, keys, e0, hi, cls, key);
      if (cls >= 0 && (cls ? k[1] : k[0]) > 0) {
        if (key < (cls ? kth[1] : kth[0])) atomicAdd(&sh.cnt_below[cls], 1u);
        else if (key == (cls ? kth[1] : kth[0])) atomicAdd(&sh.cnt_eq[cls], 1u);
      }
    }
    cluster.sync();
    if (tid < 2) {
      unsigned bb = 0, be = 0;
      for (int r = 0; r < rank; ++r) {
        const SampShared* o = cluster.map_shared_rank(&sh, r);
        bb += o->cnt_below[tid];
        be += o->cnt_eq[tid];
      }
      sh.base_below[tid] = bb;
      sh.base_eq[tid] = be;
    }
    __syncthreads();
    for (int c = 0; c < 2; ++c) {
      if (k[c] == 0) continue;
      const int capc = c ? cap_pos : cap_neg;
      int64_t* oi = c ? out_idx[1] : out_idx[0];
      uint8_t* ov = c ? out_valid[1] : out_valid[0];
      const unsigned kc = c ? kth[1] : kth[0], nq = c ? n_eq[1] : n_eq[0];
      for (int e0 = lo; e0 < hi; e0 += kSampThreads) {
        const int e = e0 + tid;
        int cls;
        unsigned key;
        load_elem<L>(labels, keys, e, hi, cls, key);
        const bool below = cls == c && key < kc, eq = cls == c && key == kc;
        const unsigned bal_b = __ballot_sync(0xffffffffu, below), bal_e = __ballot_sync(0xffffffffu, eq);
        if ((tid & 31) == 0) sh.warp[tid >> 5] = __popc(bal_b) | (__popc(bal_e) << 16);
        __syncthreads();
        unsigned before_b = 0, before_e = 0;
        for (int w = 0; w < (tid >> 5); ++w) { before_b += sh.warp[w] & 0xffffu; before_e += sh.warp[w] >> 16; }
        const unsigned lane_lt = (1u << (tid & 31)) - 1u;
        const unsigned eq_rank = sh.base_eq[c] + before_e + __popc(bal_e & lane_lt);
        if (below || (eq && eq_rank < nq)) {
          const unsigned pos = sh.base_below[c] + before_b + __popc(bal_b & lane_lt) + min(eq_rank, nq);
          if ((int)pos < capc) { oi[pos] = e; ov[pos] = 1; }
        }
        __syncthreads();
        if (tid == 0) {
          unsigned tb = 0, te = 0;
          for (int w = 0; w < kSampThreads / 32; ++w) { tb += sh.warp[w] & 0xffffu; te += sh.warp[w] >> 16; }
          sh.base_below[c] += tb;
          sh.base_eq[c] += te;
        }
        __syncthreads();
      }
    }
  }
  if (rank == 0) {
    for (int i = (int)k[0] + tid; i < cap_neg; i += kSampThreads) { out_idx[0][i] = 0; out_valid[0][i] = 0; }
    for (int i = (int)k[1] + tid; i < cap_pos; i += kSampThreads) { out_idx[1][i] = 0; out_valid[1][i] = 0; }
    if (tid == 0) { counts[2 * img] = (int)k[1]; counts[2 * img + 1] = (int)k[0]; }
  }
  cluster.sync();                                          // no CTA leaves while its shared memory may still be read
}

// ---- sampled RoIs of the RoI heads (TV roi_heads.py:615-678 from the sampler's output on): one CTA per image
constexpr int kRoiThreads = 512;
constexpr int kRoiMaxList = 1024;        // sampler capacity per class (and batch_size_per_image) handled per image

// number of entries of the ascending list a[0..n) below v
__device__ __forceinline__ int count_below(const int* a, int n, int v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// BoxCoder.encode_single (TV _utils.py:75-119) in the order of the torch composition (one rounding per operation)
__device__ __forceinline__ float4 encode_box(float4 gt, float4 p, float wx, float wy, float ww, float wh) {
  const float ex_w = __fsub_rn(p.z, p.x), ex_h = __fsub_rn(p.w, p.y);
  const float ex_cx = __fadd_rn(p.x, __fmul_rn(0.5f, ex_w)), ex_cy = __fadd_rn(p.y, __fmul_rn(0.5f, ex_h));
  const float gt_w = __fsub_rn(gt.z, gt.x), gt_h = __fsub_rn(gt.w, gt.y);
  const float gt_cx = __fadd_rn(gt.x, __fmul_rn(0.5f, gt_w)), gt_cy = __fadd_rn(gt.y, __fmul_rn(0.5f, gt_h));
  return make_float4(__fdiv_rn(__fmul_rn(wx, __fsub_rn(gt_cx, ex_cx)), ex_w),
                     __fdiv_rn(__fmul_rn(wy, __fsub_rn(gt_cy, ex_cy)), ex_h),
                     __fmul_rn(ww, logf(__fdiv_rn(gt_w, ex_w))), __fmul_rn(wh, logf(__fdiv_rn(gt_h, ex_h))));
}

__global__ void __launch_bounds__(kRoiThreads)
sample_rois_kernel(const int64_t* __restrict__ pos_idx, const uint8_t* __restrict__ pos_valid, int cap_pos,
                   const int64_t* __restrict__ neg_idx, const uint8_t* __restrict__ neg_valid, int cap_neg,
                   const int64_t* __restrict__ labels, const int64_t* __restrict__ clamped_idx, int n_slots,
                   const float* __restrict__ boxes, const int32_t* __restrict__ box_counts, int n_boxes,
                   const float* __restrict__ gt_boxes, const int32_t* __restrict__ gt_offsets, int batch_size,
                   float wx, float wy, float ww, float wh, float* __restrict__ s_props, int64_t* __restrict__ s_labels,
                   float* __restrict__ reg_targets) {
  __shared__ int pos[kRoiMaxList], neg[kRoiMaxList], sel[kRoiMaxList];
  __shared__ int n_pos, n_neg;
  const int img = blockIdx.x, tid = threadIdx.x;
  pos_idx += (size_t)img * cap_pos; pos_valid += (size_t)img * cap_pos;
  neg_idx += (size_t)img * cap_neg; neg_valid += (size_t)img * cap_neg;
  if (tid == 0) n_pos = n_neg = 0;
  __syncthreads();
  // the sampler's lists are ascending with the valid entries first
  for (int i = tid; i < cap_pos; i += kRoiThreads) {
    pos[i] = (int)pos_idx[i];
    if (pos_valid[i]) atomicAdd(&n_pos, 1);
  }
  for (int i = tid; i < cap_neg; i += kRoiThreads) {
    neg[i] = (int)neg_idx[i];
    if (neg_valid[i]) atomicAdd(&n_neg, 1);
  }
  __syncthreads();
  // merge of the two (disjoint) ascending lists = torch.sort of their concatenation (roi_heads.py:620 torch.where order)
  const int np = n_pos, nn = n_neg, n_sel = min(np + nn, batch_size);
  for (int i = tid; i < np; i += kRoiThreads) {
    const int r = i + count_below(neg, nn, pos[i]);
    if (r < batch_size) sel[r] = pos[i];
  }
  for (int i = tid; i < nn; i += kRoiThreads) {
    const int r = i + count_below(pos, np, neg[i]);
    if (r < batch_size) sel[r] = neg[i];
  }
  __syncthreads();
  const int g0 = gt_offsets[img], n_gt = gt_offsets[img + 1] - g0;
  const int n_prop = min(max(box_counts[img], 0), n_boxes);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = tid; s < batch_size; s += kRoiThreads) {
    const size_t o = (size_t)img * batch_size + s;
    float4 box = zero, gt = n_gt > 0 ? ld_box(gt_boxes, g0) : zero, enc_box = make_float4(0.f, 0.f, 1.f, 1.f);
    long long lab = -100;                  // an empty slot: cross_entropy's ignore_index, a zero box
    if (s < n_sel) {
      const int c = sel[s];
      box = enc_box = c < n_prop ? ld_box(boxes, (long long)img * n_boxes + c) : ld_box(gt_boxes, g0 + (c - n_prop));
      lab = labels[(size_t)img * n_slots + c];
      if (n_gt > 0) gt = ld_box(gt_boxes, g0 + clamped_idx[(size_t)img * n_slots + c]);
    }
    reinterpret_cast<float4*>(s_props)[o] = box;
    s_labels[o] = lab;
    // empty slots encode against (0,0,1,1) so that log() stays finite
    reinterpret_cast<float4*>(reg_targets)[o] = encode_box(gt, enc_box, wx, wy, ww, wh);
  }
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_balanced_sample(const void* labels, int labels_are_int64, const float* keys, int n_img, int n,
                                    int num_pos, int batch_size_per_image, int64_t* pos_idx, uint8_t* pos_valid,
                                    int64_t* neg_idx, uint8_t* neg_valid, int32_t* counts, dgod_stream_t stream) {
  DGOD_REQUIRE(n_img >= 0 && n >= 0 && num_pos >= 0 && batch_size_per_image >= num_pos, "dgod_balanced_sample: bad size");
  if (n_img == 0) return DGOD_OK;
  const int cap_pos = num_pos < n ? num_pos : n, cap_neg = batch_size_per_image < n ? batch_size_per_image : n;
  DGOD_REQUIRE(labels && keys && counts && (cap_pos == 0 || (pos_idx && pos_valid)) && (cap_neg == 0 || (neg_idx && neg_valid)),
               "dgod_balanced_sample: null pointer");
  if (labels_are_int64)
    balanced_sample_kernel<int64_t><<<n_img * kSampCluster, kSampThreads, 0, (cudaStream_t)stream>>>(
        (const int64_t*)labels, keys, n, num_pos, batch_size_per_image, cap_pos, cap_neg, pos_idx, pos_valid, neg_idx, neg_valid,
        counts);
  else
    balanced_sample_kernel<float><<<n_img * kSampCluster, kSampThreads, 0, (cudaStream_t)stream>>>(
        (const float*)labels, keys, n, num_pos, batch_size_per_image, cap_pos, cap_neg, pos_idx, pos_valid, neg_idx, neg_valid,
        counts);
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" int dgod_sample_rois(const int64_t* pos_idx, const uint8_t* pos_valid, int cap_pos, const int64_t* neg_idx,
                                const uint8_t* neg_valid, int cap_neg, const int64_t* labels, const int64_t* clamped_idx,
                                int n_img, int n_slots, const float* boxes, const int32_t* box_counts, int n_boxes,
                                const float* gt_boxes, const int32_t* gt_offsets, int batch_size_per_image, float wx,
                                float wy, float ww, float wh, float* s_props, int64_t* s_labels, float* reg_targets,
                                dgod_stream_t stream) {
  DGOD_REQUIRE(n_img >= 0 && n_slots >= 0 && n_boxes >= 0 && cap_pos >= 0 && cap_neg >= 0 && batch_size_per_image >= 0,
               "dgod_sample_rois: negative size");
  DGOD_REQUIRE(cap_pos <= kRoiMaxList && cap_neg <= kRoiMaxList && batch_size_per_image <= kRoiMaxList,
               "dgod_sample_rois: more than 1024 sampled RoIs per image");
  if (n_img == 0 || batch_size_per_image == 0) return DGOD_OK;
  DGOD_REQUIRE((cap_pos == 0 || (pos_idx && pos_valid)) && (cap_neg == 0 || (neg_idx && neg_valid)) && labels &&
                   clamped_idx && (boxes || n_boxes == 0) && box_counts && gt_offsets && s_props && s_labels &&
                   reg_targets,
               "dgod_sample_rois: null pointer");
  sample_rois_kernel<<<n_img, kRoiThreads, 0, (cudaStream_t)stream>>>(
      pos_idx, pos_valid, cap_pos, neg_idx, neg_valid, cap_neg, labels, clamped_idx, n_slots, boxes, box_counts, n_boxes,
      gt_boxes, gt_offsets, batch_size_per_image, wx, wy, ww, wh, s_props, s_labels, reg_targets);
  DGOD_LAUNCHED();
  return DGOD_OK;
}
