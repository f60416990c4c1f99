// Native data movement at the backbone -> FPN boundary: the FPN's top-down merge (forward and backward) and the
// frozen stem's epilogue.  Every kernel is a streaming pass, bit-exact with the ATen composition it replaces.
//
// Reference behaviour restated (torchvision 0.26.0 ops/feature_pyramid_network.py, FeaturePyramidNetwork.forward;
// ATen UpSample.cuh / UpSampleNearest2d.cu, DilatedMaxPool2d.cu, TensorCompare.cu):
//   merge forward   last_inner = inner_lateral + F.interpolate(last_inner, size, mode="nearest")
//                   with inner_lateral = conv1x1(x) + bias (cuDNN conv, then a separate broadcast bias add):
//                   out = (lat + bias[c]) + coarse[sy(y), sx(x)], sy(y) = min(floor(y * (float)Hc / H), Hc - 1).
//   merge backward  upsample_nearest2d_backward sums, per coarse pixel, the fine pixels
//                   y in [ceil(yc * s), ceil((yc + 1) * s)) clamped to H, s = (float)H / Hc (likewise x), row-major
//                   into a float starting at 0; autograd then adds the coarse level's own (layer-block) gradient.
//   stem            max_pool2d(relu_(conv + shift), 3, 2, 1): relu_ is clamp_min (NaN passes), the max-pool keeps a
//                   value if it is > the running max or NaN, starting from -inf, window rows then columns.
// NHWC: one thread owns 4 consecutive channels of a pixel (128-bit accesses, C % 4 == 0); NCHW: one element.  The grid's
// y dimension walks output rows (n, y) or (n, c, y), its x dimension the elements of a row, both grid-stride.
#include "common.cuh"

namespace dgod {

// ATen's nearest_neighbor_compute_source_index / nearest_neighbor_bw_compute_source_index (UpSample.cuh)
__device__ __forceinline__ int nearest_src(float scale, int dst, int in_size) {
  return min((int)floorf(__fmul_rn((float)dst, scale)), in_size - 1);
}
__device__ __forceinline__ int nearest_bw_src(float scale, int dst, int out_size) {
  return min((int)ceilf(__fmul_rn((float)dst, scale)), out_size);
}

__device__ __forceinline__ float4 add4(float4 a, float4 b) {
  return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}

// clamp_min(v, 0) with NaN passed through (TensorCompare.cu), then the max-pool's update rule (DilatedMaxPool2d.cu)
__device__ __forceinline__ void relu_max(float& m, float v, float shift) {
  const float t = clamp_min0(__fadd_rn(v, shift));
  if (t > m || isnan(t)) m = t;
}

// ---------------------------------------------------------------------------- merge forward
// `lat` and `out` may be the same buffer: each element is read once, by the thread that writes it.
template <bool NHWC>
__global__ void __launch_bounds__(256)
fpn_merge_fwd_kernel(const float* lat, const float* __restrict__ bias, const float* __restrict__ coarse, float* out,
                     int rows, int H, int W, int Hc, int Wc, int C, float scale_h, float scale_w) {
  const int row_len = NHWC ? W * (C >> 2) : W;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int y = r % H, plane = r / H;               // plane = n (NHWC) or n * C + c (NCHW)
    const int sy = nearest_src(scale_h, y, Hc);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int C4 = C >> 2;
      const float4* __restrict__ b4 = reinterpret_cast<const float4*>(bias);
      const float4* crow = reinterpret_cast<const float4*>(coarse) + ((size_t)plane * Hc + sy) * Wc * C4;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x = j / C4, c4 = j - x * C4;
        const float4 l = reinterpret_cast<const float4*>(lat)[row + j];
        const float4 u = __ldg(crow + (size_t)nearest_src(scale_w, x, Wc) * C4 + c4);
        reinterpret_cast<float4*>(out)[row + j] = add4(add4(l, __ldg(b4 + c4)), u);
      }
    } else {
      const float bc = __ldg(bias + plane % C);
      const float* crow = coarse + ((size_t)plane * Hc + sy) * Wc;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x)
        out[row + j] = __fadd_rn(__fadd_rn(lat[row + j], bc), __ldg(crow + nearest_src(scale_w, j, Wc)));
    }
  }
}

// ---------------------------------------------------------------------------- merge backward
// g_coarse = g_lb + (sum of g_fine over the fine pixels that map to the coarse pixel); g_lb may be NULL (zero) and may be
// the same buffer as g_coarse.
template <bool NHWC>
__global__ void __launch_bounds__(256)
fpn_merge_bwd_kernel(const float* __restrict__ g_fine, const float* g_lb, float* g_coarse, int rows, int H, int W,
                     int Hc, int Wc, int C, float scale_h, float scale_w) {
  const int row_len = NHWC ? Wc * (C >> 2) : Wc;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int yc = r % Hc, plane = r / Hc;
    const int y0 = nearest_bw_src(scale_h, yc, H), y1 = nearest_bw_src(scale_h, yc + 1, H);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int C4 = C >> 2;
      const float4* __restrict__ g4 = reinterpret_cast<const float4*>(g_fine) + (size_t)plane * H * W * C4;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int xc = j / C4, c4 = j - xc * C4;
        const int x0 = nearest_bw_src(scale_w, xc, W), x1 = nearest_bw_src(scale_w, xc + 1, W);
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) s = add4(s, __ldg(g4 + ((size_t)y * W + x) * C4 + c4));
        if (g_lb) s = add4(reinterpret_cast<const float4*>(g_lb)[row + j], s);
        reinterpret_cast<float4*>(g_coarse)[row + j] = s;
      }
    } else {
      const float* __restrict__ gp = g_fine + (size_t)plane * H * W;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x0 = nearest_bw_src(scale_w, j, W), x1 = nearest_bw_src(scale_w, j + 1, W);
        float s = 0.f;
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) s = __fadd_rn(s, __ldg(gp + (size_t)y * W + x));
        if (g_lb) s = __fadd_rn(g_lb[row + j], s);
        g_coarse[row + j] = s;
      }
    }
  }
}

// ---------------------------------------------------------------------------- stem: shift + ReLU + 3x3/2 max-pool
template <bool NHWC>
__global__ void __launch_bounds__(256)
stem_pool_kernel(const float* __restrict__ conv, const float* __restrict__ shift, float* __restrict__ out, int rows,
                 int H, int W, int C, int Ho, int Wo) {
  const int row_len = NHWC ? Wo * (C >> 2) : Wo;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int yo = r % Ho, plane = r / Ho;
    const int y0 = max(2 * yo - 1, 0), y1 = min(2 * yo + 2, H);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int C4 = C >> 2;
      const float4* __restrict__ in4 = reinterpret_cast<const float4*>(conv) + (size_t)plane * H * W * C4;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int xo = j / C4, c4 = j - xo * C4;
        const int x0 = max(2 * xo - 1, 0), x1 = min(2 * xo + 2, W);
        const float4 sh = __ldg(reinterpret_cast<const float4*>(shift) + c4);
        float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) {
            const float4 v = __ldg(in4 + ((size_t)y * W + x) * C4 + c4);
            relu_max(m.x, v.x, sh.x); relu_max(m.y, v.y, sh.y); relu_max(m.z, v.z, sh.z); relu_max(m.w, v.w, sh.w);
          }
        reinterpret_cast<float4*>(out)[row + j] = m;
      }
    } else {
      const float sh = __ldg(shift + plane % C);
      const float* __restrict__ ip = conv + (size_t)plane * H * W;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x0 = max(2 * j - 1, 0), x1 = min(2 * j + 2, W);
        float m = -INFINITY;
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) relu_max(m, __ldg(ip + (size_t)y * W + x), sh);
        out[row + j] = m;
      }
    }
  }
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_fpn_merge_fwd(const float* lat, const float* bias, const float* coarse, float* out, int n, int h,
                                  int w, int hc, int wc, int c, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "dgod_fpn_merge_fwd: negative size");
  if ((long long)n * h * w * c == 0) return DGOD_OK;
  DGOD_REQUIRE(hc > 0 && wc > 0, "dgod_fpn_merge_fwd: empty coarse map");
  DGOD_REQUIRE(lat && bias && coarse && out, "dgod_fpn_merge_fwd: null pointer");
  const long long rows = channels_last ? (long long)n * h : (long long)n * c * h;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "dgod_fpn_merge_fwd: map too large");
  const float sh = (float)hc / (float)h, sw = (float)wc / (float)w;   // ATen: (float)input_size / output_size
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    DGOD_REQUIRE(c % 4 == 0, "dgod_fpn_merge_fwd: channels_last needs channels %% 4 == 0, got %d", c);
    DGOD_REQUIRE(aligned16(lat) && aligned16(bias) && aligned16(coarse) && aligned16(out),
                 "dgod_fpn_merge_fwd: channels_last needs 16-byte aligned pointers");
    fpn_merge_fwd_kernel<true><<<row_grid(rows, w * (c / 4)), 256, 0, st>>>(lat, bias, coarse, out, (int)rows, h, w, hc,
                                                                         wc, c, sh, sw);
  } else {
    fpn_merge_fwd_kernel<false><<<row_grid(rows, w), 256, 0, st>>>(lat, bias, coarse, out, (int)rows, h, w, hc, wc, c,
                                                                  sh, sw);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" int dgod_fpn_merge_bwd(const float* g_fine, const float* g_lb, float* g_coarse, int n, int h, int w, int hc,
                                  int wc, int c, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && hc >= 0 && wc >= 0 && c >= 0, "dgod_fpn_merge_bwd: negative size");
  if ((long long)n * hc * wc * c == 0) return DGOD_OK;
  DGOD_REQUIRE(h > 0 && w > 0, "dgod_fpn_merge_bwd: empty fine map");
  DGOD_REQUIRE(g_fine && g_coarse, "dgod_fpn_merge_bwd: null pointer");
  const long long rows = channels_last ? (long long)n * hc : (long long)n * c * hc;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "dgod_fpn_merge_bwd: map too large");
  const float sh = (float)h / (float)hc, sw = (float)w / (float)wc;   // ATen: (float)output_size / input_size
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    DGOD_REQUIRE(c % 4 == 0, "dgod_fpn_merge_bwd: channels_last needs channels %% 4 == 0, got %d", c);
    DGOD_REQUIRE(aligned16(g_fine) && aligned16(g_lb) && aligned16(g_coarse),
                 "dgod_fpn_merge_bwd: channels_last needs 16-byte aligned pointers");
    fpn_merge_bwd_kernel<true><<<row_grid(rows, wc * (c / 4)), 256, 0, st>>>(g_fine, g_lb, g_coarse, (int)rows, h, w,
                                                                          hc, wc, c, sh, sw);
  } else {
    fpn_merge_bwd_kernel<false><<<row_grid(rows, wc), 256, 0, st>>>(g_fine, g_lb, g_coarse, (int)rows, h, w, hc, wc, c,
                                                                   sh, sw);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" int dgod_stem_pool_fwd(const float* conv, const float* shift, float* out, int n, int h, int w, int c, int ho,
                                  int wo, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "dgod_stem_pool_fwd: negative size");
  DGOD_REQUIRE(ho == (h - 1) / 2 + 1 && wo == (w - 1) / 2 + 1 && h > 0 && w > 0,
               "dgod_stem_pool_fwd: output %dx%d is not the 3x3 / stride 2 / pad 1 pooling of %dx%d", ho, wo, h, w);
  if ((long long)n * c == 0) return DGOD_OK;
  DGOD_REQUIRE(conv && shift && out, "dgod_stem_pool_fwd: null pointer");
  const long long rows = channels_last ? (long long)n * ho : (long long)n * c * ho;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "dgod_stem_pool_fwd: map too large");
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    DGOD_REQUIRE(c % 4 == 0, "dgod_stem_pool_fwd: channels_last needs channels %% 4 == 0, got %d", c);
    DGOD_REQUIRE(aligned16(conv) && aligned16(shift) && aligned16(out),
                 "dgod_stem_pool_fwd: channels_last needs 16-byte aligned pointers");
    stem_pool_kernel<true><<<row_grid(rows, wo * (c / 4)), 256, 0, st>>>(conv, shift, out, (int)rows, h, w, c, ho, wo);
  } else {
    stem_pool_kernel<false><<<row_grid(rows, wo), 256, 0, st>>>(conv, shift, out, (int)rows, h, w, c, ho, wo);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}
