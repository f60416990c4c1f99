// The RPN head after its 3x3 convolution (TV models/detection/rpn.py RPNHead.forward; fasterrcnn.py:165), all levels in
// one launch each way.  Stock runs, per level, a broadcast bias add, relu_, two 1x1 convolutions and their bias adds,
// and in the backward two 1x1 dgrads, the accumulation add, threshold_backward, the bias reduction and two 1x1 wgrads:
// about eleven passes over the 256-channel map.  Here the forward reads the bias-free conv output c once and the
// backward reads c once and writes its gradient once.
//
//   forward   t = relu_(c + b)                        (ATen's add_ and clamp_min: bit-identical to the stock t)
//             obj[a]    = (sum_k W_cls[a][k] t[k]) + b_cls[a]      fp32 fma, k ascending
//             deltas[j] = (sum_k W_bbox[j][k] t[k]) + b_bbox[j]
//   backward  gt[k] = sum_o W[o][k] g[o]  (o = the A objectness then the 4A delta outputs, ascending)
//             gc[k] = t[k] <= 0 ? 0 : gt[k]           (threshold_backward, NaN included)
//             dW[o][k] = sum_p g[o] t[k],  db[k] = sum_p gc[k],  db_o = sum_p g[o]   over every pixel of every level
//
// t is never stored: the backward recomputes it from c.  Outputs are NCHW-contiguous [n, A, h, w] / [n, 4A, h, w] (what
// rpn_proposals reads); c and gc are NHWC.  C = 256 and A = 3 (torchvision's FPN width and anchors per location).
//
// Forward: a CTA stages 256 pixels x 32 channels of c in shared memory (cp.async, two stages) and each thread computes
// all 15 outputs of two pixels against the weights in shared memory (broadcast reads).
// Backward: a thread owns 4 channels (64 threads cover a pixel, so a pixel's 1 KB is one coalesced read), keeps its
// 15 x 4 weights and 15 x 4 weight-gradient sums in registers, and walks its pixels with a per-thread cp.async ring that
// keeps 8 pixels in flight.  The incoming gradients of 256 pixels are staged in shared memory per chunk.  Each CTA owns
// a fixed contiguous range of chunks and writes its partial sums; a finish kernel adds the partials in CTA order.  No
// float atomics: the results are the same bits on every run on the same device.
#include "common.cuh"

namespace dgod {

constexpr int kRhC = 256, kRhA = 3, kRhO = 5 * kRhA;
// packed parameter gradients: dW_cls [A, C], dW_bbox [4A, C], db [C], db_cls [A], db_bbox [4A]
constexpr int kRhParams = kRhO * kRhC + kRhC + kRhO;
constexpr int kRhPartStride = (kRhParams + 3) / 4 * 4;        // a CTA's partial sums: rows 16-byte aligned

struct RpnHeadLevels {
  const float* c[DGOD_MAX_LEVELS];
  float* obj[DGOD_MAX_LEVELS];           // forward outputs
  float* deltas[DGOD_MAX_LEVELS];
  const float* g_obj[DGOD_MAX_LEVELS];   // backward inputs
  const float* g_deltas[DGOD_MAX_LEVELS];
  float* gc[DGOD_MAX_LEVELS];            // backward output
  int hw[DGOD_MAX_LEVELS];
  int n_pix[DGOD_MAX_LEVELS];            // n_img * hw
  int tile0[DGOD_MAX_LEVELS + 1];        // first tile (forward) / chunk (backward) of each level
  int n_levels;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ int level_of(const RpnHeadLevels& L, int tile) {
  int lv = 0;
  while (lv + 1 < L.n_levels && tile >= L.tile0[lv + 1]) ++lv;
  return lv;
}

__device__ __forceinline__ float4 relu_bias(float4 c, float4 b) {
  return make_float4(clamp_min0(__fadd_rn(c.x, b.x)), clamp_min0(__fadd_rn(c.y, b.y)), clamp_min0(__fadd_rn(c.z, b.z)),
                     clamp_min0(__fadd_rn(c.w, b.w)));
}

__device__ __forceinline__ float fma4(float4 w, float4 t, float acc) {
  acc = __fmaf_rn(w.x, t.x, acc);
  acc = __fmaf_rn(w.y, t.y, acc);
  acc = __fmaf_rn(w.z, t.z, acc);
  return __fmaf_rn(w.w, t.w, acc);
}

// ---------------------------------------------------------------- forward
constexpr int kFwdThreads = 128, kFwdTile = 2 * kFwdThreads, kFwdKc = 32, kFwdRow = kFwdKc + 4;
constexpr int kFwdSmem = (kRhO * kRhC + kRhC + 2 * kFwdTile * kFwdRow) * 4;

__global__ void __launch_bounds__(kFwdThreads, 2)
rpn_head_fwd_kernel(const RpnHeadLevels L, const float* __restrict__ bias, const float* __restrict__ w_cls,
                    const float* __restrict__ b_cls, const float* __restrict__ w_bbox, const float* __restrict__ b_bbox) {
  extern __shared__ float4 smem4[];
  float4* w_s = smem4;                          // [kRhO][kRhC / 4]
  float4* b_s = w_s + kRhO * kRhC / 4;          // [kRhC / 4]
  float* t_s = reinterpret_cast<float*>(b_s + kRhC / 4);   // [2][kFwdTile][kFwdRow]
  const int tid = threadIdx.x;
  const int lv = level_of(L, blockIdx.x);
  const int p0 = (blockIdx.x - L.tile0[lv]) * kFwdTile;
  const int cnt = min(kFwdTile, L.n_pix[lv] - p0);
  const float* c = L.c[lv] + (size_t)p0 * kRhC;

  auto stage = [&](int kc) {
    float* dst = t_s + (kc & 1) * kFwdTile * kFwdRow;
#pragma unroll
    for (int j = 0; j < kFwdTile * kFwdKc / 4 / kFwdThreads; ++j) {
      const int idx = tid + j * kFwdThreads, px = idx >> 3, v = idx & 7;
      const bool ok = px < cnt;
      cp_async16(dst + px * kFwdRow + v * 4, ok ? c + (size_t)px * kRhC + kc * kFwdKc + v * 4 : c, ok);
    }
    cp_async_commit();
  };
  stage(0);
  for (int i = tid; i < kRhO * kRhC / 4; i += kFwdThreads) {
    const int o = i / (kRhC / 4), k = i % (kRhC / 4);
    w_s[i] = __ldg(reinterpret_cast<const float4*>(o < kRhA ? w_cls + o * kRhC : w_bbox + (o - kRhA) * kRhC) + k);
  }
  for (int i = tid; i < kRhC / 4; i += kFwdThreads) b_s[i] = __ldg(reinterpret_cast<const float4*>(bias) + i);

  float acc0[kRhO], acc1[kRhO];
#pragma unroll
  for (int o = 0; o < kRhO; ++o) acc0[o] = acc1[o] = 0.f;
  for (int kc = 0; kc < kRhC / kFwdKc; ++kc) {
    if (kc + 1 < kRhC / kFwdKc) {
      stage(kc + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float4* r0 = reinterpret_cast<const float4*>(t_s + ((kc & 1) * kFwdTile + tid) * kFwdRow);
    const float4* r1 = r0 + kFwdThreads * kFwdRow / 4;
#pragma unroll
    for (int k4 = 0; k4 < kFwdKc / 4; ++k4) {
      const int kv = kc * (kFwdKc / 4) + k4;
      const float4 b = b_s[kv];
      const float4 x0 = relu_bias(r0[k4], b), x1 = relu_bias(r1[k4], b);
#pragma unroll
      for (int o = 0; o < kRhO; ++o) {
        const float4 w = w_s[o * (kRhC / 4) + kv];
        acc0[o] = fma4(w, x0, acc0[o]);
        acc1[o] = fma4(w, x1, acc1[o]);
      }
    }
    __syncthreads();                            // the buffer is refilled two chunks on
  }
  const int hw = L.hw[lv];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int px = tid + h * kFwdThreads;
    if (px >= cnt) continue;
    const int p = p0 + px, n = p / hw, r = p - n * hw;
    const float* acc = h ? acc1 : acc0;
#pragma unroll
    for (int a = 0; a < kRhA; ++a) L.obj[lv][((size_t)n * kRhA + a) * hw + r] = __fadd_rn(acc[a], __ldg(b_cls + a));
#pragma unroll
    for (int j = 0; j < 4 * kRhA; ++j)
      L.deltas[lv][((size_t)n * 4 * kRhA + j) * hw + r] = __fadd_rn(acc[kRhA + j], __ldg(b_bbox + j));
  }
}

// ---------------------------------------------------------------- backward
constexpr int kBwdThreads = 128, kBwdChunk = 256, kBwdRing = 8, kBwdCtasPerSm = 2;
constexpr int kBwdGroupPix = kBwdChunk / (kBwdThreads / (kRhC / 4));   // pixels of one 64-thread group per chunk

__global__ void __launch_bounds__(kBwdThreads, kBwdCtasPerSm)
rpn_head_bwd_kernel(const RpnHeadLevels L, int n_chunks, const float* __restrict__ bias, const float* __restrict__ w_cls,
                    const float* __restrict__ w_bbox, float* __restrict__ partial) {
  __shared__ __align__(16) float g_s[kBwdChunk][16];        // the chunk's 15 incoming gradients per pixel (+1 pad)
  __shared__ __align__(16) float4 ring[kBwdRing][kBwdThreads];
  __shared__ float sb_s[kRhO][kBwdThreads];                 // per-thread sums of the incoming gradients
  pdl_trigger();                                             // the finish kernel is scheduled behind this grid
  const int tid = threadIdx.x, q = tid & (kRhC / 4 - 1), grp = tid / (kRhC / 4);
  float w[kRhO][4], dw[kRhO][4], db[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int o = 0; o < kRhO; ++o) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(o < kRhA ? w_cls + o * kRhC : w_bbox + (o - kRhA) * kRhC) + q);
    w[o][0] = v.x; w[o][1] = v.y; w[o][2] = v.z; w[o][3] = v.w;
    dw[o][0] = dw[o][1] = dw[o][2] = dw[o][3] = 0.f;
    sb_s[o][tid] = 0.f;
  }
  const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + q);
  const int ch0 = (int)((long long)blockIdx.x * n_chunks / gridDim.x);
  const int ch1 = (int)((long long)(blockIdx.x + 1) * n_chunks / gridDim.x);
  int lv = 0;
  for (int ch = ch0; ch < ch1; ++ch) {
    while (ch >= L.tile0[lv + 1]) ++lv;
    const int p0 = (ch - L.tile0[lv]) * kBwdChunk, cnt = min(kBwdChunk, L.n_pix[lv] - p0), hw = L.hw[lv];
    __syncthreads();                                         // the previous chunk's g_s is consumed
    for (int px = tid; px < kBwdChunk; px += kBwdThreads) {
      float g[kRhO];
      if (px < cnt) {
        const int p = p0 + px, n = p / hw, r = p - n * hw;
#pragma unroll
        for (int a = 0; a < kRhA; ++a) g[a] = L.g_obj[lv][((size_t)n * kRhA + a) * hw + r];
#pragma unroll
        for (int j = 0; j < 4 * kRhA; ++j) g[kRhA + j] = L.g_deltas[lv][((size_t)n * 4 * kRhA + j) * hw + r];
      } else {
#pragma unroll
        for (int o = 0; o < kRhO; ++o) g[o] = 0.f;
      }
#pragma unroll
      for (int o = 0; o < kRhO; ++o) {
        g_s[px][o] = g[o];
        sb_s[o][tid] = __fadd_rn(sb_s[o][tid], g[o]);
      }
      g_s[px][kRhO] = 0.f;
    }
    __syncthreads();
    const int lo = grp * kBwdGroupPix, hi = min(cnt, lo + kBwdGroupPix);
    const float* cp = L.c[lv] + (size_t)p0 * kRhC + 4 * q;
    float* gp = L.gc[lv] + (size_t)p0 * kRhC + 4 * q;
#pragma unroll
    for (int s = 0; s < kBwdRing; ++s) {
      if (lo + s < hi) cp_async16(&ring[s][tid], cp + (size_t)(lo + s) * kRhC, true);
      cp_async_commit();
    }
    for (int i = lo; i < hi; ++i) {
      const int slot = (i - lo) % kBwdRing;
      cp_async_wait<kBwdRing - 1>();
      const float4 cv = ring[slot][tid];
      const float t[4] = {clamp_min0(__fadd_rn(cv.x, b.x)), clamp_min0(__fadd_rn(cv.y, b.y)),
                          clamp_min0(__fadd_rn(cv.z, b.z)), clamp_min0(__fadd_rn(cv.w, b.w))};
      const float4* g4 = reinterpret_cast<const float4*>(g_s[i]);
      float g[16];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 v = g4[k];
        g[4 * k] = v.x; g[4 * k + 1] = v.y; g[4 * k + 2] = v.z; g[4 * k + 3] = v.w;
      }
      float gc[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float gt = __fmul_rn(w[0][j], g[0]);
#pragma unroll
        for (int o = 1; o < kRhO; ++o) gt = __fmaf_rn(w[o][j], g[o], gt);
        gc[j] = t[j] <= 0.f ? 0.f : gt;
        db[j] = __fadd_rn(db[j], gc[j]);
#pragma unroll
        for (int o = 0; o < kRhO; ++o) dw[o][j] = __fmaf_rn(g[o], t[j], dw[o][j]);
      }
      *reinterpret_cast<float4*>(gp + (size_t)i * kRhC) = make_float4(gc[0], gc[1], gc[2], gc[3]);
      if (i + kBwdRing < hi) cp_async16(&ring[slot][tid], cp + (size_t)(i + kBwdRing) * kRhC, true);
      cp_async_commit();
    }
    cp_async_wait<0>();
  }
  // group 1 hands its sums to group 0 through g_s (4096 floats), which adds them in a fixed order
  __syncthreads();
  float* red = &g_s[0][0];
  if (grp == 1) {
#pragma unroll
    for (int o = 0; o < kRhO; ++o)
#pragma unroll
      for (int j = 0; j < 4; ++j) red[(o * 4 + j) * (kRhC / 4) + q] = dw[o][j];
#pragma unroll
    for (int j = 0; j < 4; ++j) red[(kRhO * 4 + j) * (kRhC / 4) + q] = db[j];
  }
  __syncthreads();
  float* out = partial + (size_t)blockIdx.x * kRhPartStride;
  if (grp == 0) {
#pragma unroll
    for (int o = 0; o < kRhO; ++o)
      reinterpret_cast<float4*>(out + o * kRhC)[q] =
          make_float4(__fadd_rn(dw[o][0], red[(o * 4 + 0) * (kRhC / 4) + q]), __fadd_rn(dw[o][1], red[(o * 4 + 1) * (kRhC / 4) + q]),
                      __fadd_rn(dw[o][2], red[(o * 4 + 2) * (kRhC / 4) + q]), __fadd_rn(dw[o][3], red[(o * 4 + 3) * (kRhC / 4) + q]));
    reinterpret_cast<float4*>(out + kRhO * kRhC)[q] =
        make_float4(__fadd_rn(db[0], red[(kRhO * 4 + 0) * (kRhC / 4) + q]), __fadd_rn(db[1], red[(kRhO * 4 + 1) * (kRhC / 4) + q]),
                    __fadd_rn(db[2], red[(kRhO * 4 + 2) * (kRhC / 4) + q]), __fadd_rn(db[3], red[(kRhO * 4 + 3) * (kRhC / 4) + q]));
  }
  // the predictor bias sums over the CTA's threads: warp w takes outputs w, w + 4, ...; a fixed-shape pairwise tree
  for (int o = tid >> 5; o < kRhO; o += kBwdThreads / 32) {
    const int lane = tid & 31;
    float s = sb_s[o][lane];
#pragma unroll
    for (int k = 1; k < kBwdThreads / 32; ++k) s = __fadd_rn(s, sb_s[o][lane + 32 * k]);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, d));
    if (lane == 0) out[kRhO * kRhC + kRhC + o] = s;
  }
}

// out[i] = sum over the CTAs b of partial[b][i], b ascending within each of 8 warps (warp w takes b = w mod 8), the 8
// warp sums added in warp order.
constexpr int kFinishThreads = 256, kFinishCols = 32;

__global__ void __launch_bounds__(kFinishThreads)
rpn_head_finish_kernel(const float* __restrict__ partial, int n_parts, float* __restrict__ out) {
  __shared__ float s[kFinishThreads / 32][kFinishCols];
  pdl_wait();                                                // launched behind rpn_head_bwd_kernel
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, i = blockIdx.x * kFinishCols + lane;
  float acc = 0.f;
  if (i < kRhParams) {
#pragma unroll 4
    for (int b = warp; b < n_parts; b += kFinishThreads / 32) acc = __fadd_rn(acc, partial[(size_t)b * kRhPartStride + i]);
  }
  s[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < kRhParams) {
    float v = s[0][lane];
    for (int k = 1; k < kFinishThreads / 32; ++k) v = __fadd_rn(v, s[k][lane]);
    out[i] = v;
  }
}

static int bwd_ctas(int n_chunks) {
  int dev = 0, n_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return -1;
  return n_chunks < kBwdCtasPerSm * n_sm ? n_chunks : kBwdCtasPerSm * n_sm;
}

static int fill_levels(const char* fn, RpnHeadLevels& L, const float* const* c, int n_levels, const int* height,
                       const int* width, int n_img, int channels, int anchors, int tile, long long* total_tiles) {
  DGOD_REQUIRE(channels == kRhC && anchors == kRhA, "%s: only %d channels and %d anchors per location are supported, got "
               "%d and %d", fn, kRhC, kRhA, channels, anchors);
  DGOD_REQUIRE(n_levels >= 1 && n_levels <= DGOD_MAX_LEVELS, "%s: 1..%d levels expected, got %d", fn, DGOD_MAX_LEVELS,
               n_levels);
  DGOD_REQUIRE(c && height && width && n_img >= 0, "%s: null level table or negative batch", fn);
  L = RpnHeadLevels{};
  L.n_levels = n_levels;
  long long tiles = 0;
  for (int l = 0; l < n_levels; ++l) {
    DGOD_REQUIRE(height[l] >= 0 && width[l] >= 0, "%s: level %d has a negative size", fn, l);
    const long long hw = (long long)height[l] * width[l], np = hw * n_img;
    DGOD_REQUIRE(np <= INT32_MAX, "%s: level %d too large", fn, l);
    DGOD_REQUIRE(np == 0 || aligned16(c[l]), "%s: level %d: c must be a 16-byte aligned NHWC map", fn, l);
    L.c[l] = c[l];
    L.hw[l] = (int)hw;
    L.n_pix[l] = (int)np;
    L.tile0[l] = (int)tiles;
    tiles += (np + tile - 1) / tile;
    DGOD_REQUIRE(tiles <= INT32_MAX, "%s: too many pixels", fn);
  }
  L.tile0[n_levels] = (int)tiles;
  *total_tiles = tiles;
  return DGOD_OK;
}

}  // namespace dgod

using namespace dgod;

extern "C" size_t dgod_rpn_head_workspace_bytes(void) {
  const int g = bwd_ctas(INT32_MAX);
  return g > 0 ? (size_t)g * kRhPartStride * sizeof(float) + 256 : 0;
}

extern "C" int dgod_rpn_head_fwd(const float* const* c, int n_levels, const int* height, const int* width, int n_img,
                                 int channels, int anchors, const float* bias, const float* w_cls, const float* b_cls,
                                 const float* w_bbox, const float* b_bbox, float* const* objectness,
                                 float* const* deltas, dgod_stream_t stream) {
  RpnHeadLevels L;
  long long tiles = 0;
  const int rc = fill_levels("dgod_rpn_head_fwd", L, c, n_levels, height, width, n_img, channels, anchors, kFwdTile,
                             &tiles);
  if (rc != DGOD_OK) return rc;
  DGOD_REQUIRE(objectness && deltas && bias && w_cls && b_cls && w_bbox && b_bbox, "dgod_rpn_head_fwd: null pointer");
  DGOD_REQUIRE(aligned16(bias) && aligned16(w_cls) && aligned16(w_bbox), "dgod_rpn_head_fwd: bias and weights must be "
               "16-byte aligned");
  for (int l = 0; l < n_levels; ++l) {
    DGOD_REQUIRE(L.n_pix[l] == 0 || (objectness[l] && deltas[l]), "dgod_rpn_head_fwd: level %d: null output", l);
    L.obj[l] = objectness[l];
    L.deltas[l] = deltas[l];
  }
  if (tiles == 0) return DGOD_OK;
  DGOD_CUDA(cudaFuncSetAttribute(rpn_head_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdSmem));
  rpn_head_fwd_kernel<<<(unsigned)tiles, kFwdThreads, kFwdSmem, (cudaStream_t)stream>>>(L, bias, w_cls, b_cls, w_bbox,
                                                                                       b_bbox);
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" int dgod_rpn_head_bwd(const float* const* c, int n_levels, const int* height, const int* width, int n_img,
                                 int channels, int anchors, const float* bias, const float* w_cls, const float* w_bbox,
                                 const float* const* grad_objectness, const float* const* grad_deltas,
                                 float* const* grad_c, float* grad_params, void* workspace, size_t workspace_bytes,
                                 dgod_stream_t stream) {
  RpnHeadLevels L;
  long long chunks = 0;
  const int rc = fill_levels("dgod_rpn_head_bwd", L, c, n_levels, height, width, n_img, channels, anchors, kBwdChunk,
                             &chunks);
  if (rc != DGOD_OK) return rc;
  DGOD_REQUIRE(grad_objectness && grad_deltas && grad_c && grad_params && bias && w_cls && w_bbox,
               "dgod_rpn_head_bwd: null pointer");
  DGOD_REQUIRE(aligned16(bias) && aligned16(w_cls) && aligned16(w_bbox), "dgod_rpn_head_bwd: bias and weights must be "
               "16-byte aligned");
  for (int l = 0; l < n_levels; ++l) {
    DGOD_REQUIRE(L.n_pix[l] == 0 || (grad_objectness[l] && grad_deltas[l] && grad_c[l] && aligned16(grad_c[l])),
                 "dgod_rpn_head_bwd: level %d: null or misaligned gradient", l);
    L.g_obj[l] = grad_objectness[l];
    L.g_deltas[l] = grad_deltas[l];
    L.gc[l] = grad_c[l];
  }
  const int g = bwd_ctas(chunks > 0 ? (int)chunks : 1);
  DGOD_REQUIRE(g > 0, "dgod_rpn_head_bwd: cannot query the device");
  DGOD_REQUIRE(workspace && workspace_bytes >= (size_t)g * kRhPartStride * sizeof(float) && aligned16(workspace),
               "dgod_rpn_head_bwd: workspace too small or misaligned");
  float* partial = (float*)workspace;
  rpn_head_bwd_kernel<<<g, kBwdThreads, 0, (cudaStream_t)stream>>>(L, (int)chunks, bias, w_cls, w_bbox, partial);
  DGOD_LAUNCHED();
  DGOD_CUDA(launch_pdl(rpn_head_finish_kernel, dim3(cdiv(kRhParams, kFinishCols)), dim3(kFinishThreads), 0,
                       (cudaStream_t)stream, (const float*)partial, g, grad_params));
  DGOD_LAUNCHED();
  return DGOD_OK;
}
