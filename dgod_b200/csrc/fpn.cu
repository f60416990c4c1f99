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
//
// bf16 maps (the same modules under torch.autocast(dtype=bfloat16)) compute in fp32 and round to bf16 (RNE) where ATen's
// bf16 ops round: the bias / shift (an fp32 parameter or buffer) is first rounded to bf16, as autocast casts a conv's
// bias before ATen adds it; every add's result is rounded; the upsample backward's window sum stays in its fp32
// accumulator and is rounded once, then added to the coarse level's own gradient and rounded again:
//   merge forward   out = bf16(bf16(lat + bf16(bias)) + coarse[sy, sx])
//   merge backward  g_coarse = bf16(g_lb + bf16(sum))
//   stem            max-pool of clamp_min(bf16(conv + bf16(shift)), 0), same update rule (exact on bf16 values)
// NHWC: one thread owns one 16-byte vector of a pixel's channels (4 fp32 or 8 bf16: C % 4 or C % 8 == 0); NCHW: one
// element.  The grid's y dimension walks output rows (n, y) or (n, c, y), its x dimension the elements of a row, both
// grid-stride.
#include "common.cuh"

namespace dgod {

// ATen's nearest_neighbor_compute_source_index / nearest_neighbor_bw_compute_source_index (UpSample.cuh)
__device__ __forceinline__ int nearest_src(float scale, int dst, int in_size) {
  return min((int)floorf(__fmul_rn((float)dst, scale)), in_size - 1);
}
__device__ __forceinline__ int nearest_bw_src(float scale, int dst, int out_size) {
  return min((int)ceilf(__fmul_rn((float)dst, scale)), out_size);
}

// clamp_min(v, 0) with NaN passed through (TensorCompare.cu), then the max-pool's update rule (DilatedMaxPool2d.cu);
// `shift` is already rounded to T
template <typename T>
__device__ __forceinline__ void relu_max(float& m, float v, float shift) {
  const float t = clamp_min0(round_to<T>(__fadd_rn(v, shift)));
  if (t > m || isnan(t)) m = t;
}

// ---------------------------------------------------------------------------- merge forward
// `lat` and `out` may be the same buffer: each element is read once, by the thread that writes it.
template <typename T, bool NHWC>
__global__ void __launch_bounds__(256)
fpn_merge_fwd_kernel(const T* lat, const float* __restrict__ bias, const T* __restrict__ coarse, T* out,
                     int rows, int H, int W, int Hc, int Wc, int C, float scale_h, float scale_w) {
  constexpr int N = Pack<T>::N;
  typedef typename Pack<T>::V V;
  const int row_len = NHWC ? W * (C >> Pack<T>::SHIFT) : W;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int y = r % H, plane = r / H;               // plane = n (NHWC) or n * C + c (NCHW)
    const int sy = nearest_src(scale_h, y, Hc);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int CV = C >> Pack<T>::SHIFT;
      const V* crow = reinterpret_cast<const V*>(coarse) + ((size_t)plane * Hc + sy) * Wc * CV;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x = j / CV, cv = j - x * CV;
        float l[N], u[N], b[N];
        Pack<T>::unpack(reinterpret_cast<const V*>(lat)[row + j], l);
        Pack<T>::unpack(__ldg(crow + (size_t)nearest_src(scale_w, x, Wc) * CV + cv), u);
        ldg_channels<N>(bias, cv, b);
#pragma unroll
        for (int k = 0; k < N; ++k) l[k] = __fadd_rn(round_to<T>(__fadd_rn(l[k], round_to<T>(b[k]))), u[k]);
        reinterpret_cast<V*>(out)[row + j] = Pack<T>::pack(l);
      }
    } else {
      const float bc = round_to<T>(__ldg(bias + plane % C));
      const T* crow = coarse + ((size_t)plane * Hc + sy) * Wc;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x)
        out[row + j] = from_f<T>(__fadd_rn(round_to<T>(__fadd_rn(to_f(lat[row + j]), bc)),
                                           to_f(__ldg(crow + nearest_src(scale_w, j, Wc)))));
    }
  }
}

// ---------------------------------------------------------------------------- merge backward
// g_coarse = g_lb + (sum of g_fine over the fine pixels that map to the coarse pixel); g_lb may be NULL (zero) and may be
// the same buffer as g_coarse.  The window sum stays fp32 and is rounded to T once, before the add.
template <typename T, bool NHWC>
__global__ void __launch_bounds__(256)
fpn_merge_bwd_kernel(const T* __restrict__ g_fine, const T* g_lb, T* g_coarse, int rows, int H, int W,
                     int Hc, int Wc, int C, float scale_h, float scale_w) {
  constexpr int N = Pack<T>::N;
  typedef typename Pack<T>::V V;
  const int row_len = NHWC ? Wc * (C >> Pack<T>::SHIFT) : Wc;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int yc = r % Hc, plane = r / Hc;
    const int y0 = nearest_bw_src(scale_h, yc, H), y1 = nearest_bw_src(scale_h, yc + 1, H);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int CV = C >> Pack<T>::SHIFT;
      const V* __restrict__ gv = reinterpret_cast<const V*>(g_fine) + (size_t)plane * H * W * CV;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int xc = j / CV, cv = j - xc * CV;
        const int x0 = nearest_bw_src(scale_w, xc, W), x1 = nearest_bw_src(scale_w, xc + 1, W);
        float s[N], v[N];
#pragma unroll
        for (int k = 0; k < N; ++k) s[k] = 0.f;
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) {
            Pack<T>::unpack(__ldg(gv + ((size_t)y * W + x) * CV + cv), v);
#pragma unroll
            for (int k = 0; k < N; ++k) s[k] = __fadd_rn(s[k], v[k]);
          }
        if (g_lb) {
          Pack<T>::unpack(reinterpret_cast<const V*>(g_lb)[row + j], v);
#pragma unroll
          for (int k = 0; k < N; ++k) s[k] = __fadd_rn(v[k], round_to<T>(s[k]));
        }
        reinterpret_cast<V*>(g_coarse)[row + j] = Pack<T>::pack(s);
      }
    } else {
      const T* __restrict__ gp = g_fine + (size_t)plane * H * W;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x0 = nearest_bw_src(scale_w, j, W), x1 = nearest_bw_src(scale_w, j + 1, W);
        float s = 0.f;
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) s = __fadd_rn(s, to_f(__ldg(gp + (size_t)y * W + x)));
        if (g_lb) s = __fadd_rn(to_f(g_lb[row + j]), round_to<T>(s));
        g_coarse[row + j] = from_f<T>(s);
      }
    }
  }
}

// ---------------------------------------------------------------------------- stem: shift + ReLU + 3x3/2 max-pool
template <typename T, bool NHWC>
__global__ void __launch_bounds__(256)
stem_pool_kernel(const T* __restrict__ conv, const float* __restrict__ shift, T* __restrict__ out, int rows,
                 int H, int W, int C, int Ho, int Wo) {
  constexpr int N = Pack<T>::N;
  typedef typename Pack<T>::V V;
  const int row_len = NHWC ? Wo * (C >> Pack<T>::SHIFT) : Wo;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const int yo = r % Ho, plane = r / Ho;
    const int y0 = max(2 * yo - 1, 0), y1 = min(2 * yo + 2, H);
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int CV = C >> Pack<T>::SHIFT;
      const V* __restrict__ in = reinterpret_cast<const V*>(conv) + (size_t)plane * H * W * CV;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int xo = j / CV, cv = j - xo * CV;
        const int x0 = max(2 * xo - 1, 0), x1 = min(2 * xo + 2, W);
        float sh[N], m[N], v[N];
        ldg_channels<N>(shift, cv, sh);
#pragma unroll
        for (int k = 0; k < N; ++k) {
          sh[k] = round_to<T>(sh[k]);
          m[k] = -INFINITY;
        }
        // The same columns in the same order; the bf16 instance walks the window from its first column (a form ptxas
        // compiles without a spill).
        for (int y = y0; y < y1; ++y)
          for (int x = N == 4 ? x0 : 2 * xo - 1; x < x1; ++x) {
            if (x < x0) continue;
            Pack<T>::unpack(__ldg(in + ((size_t)y * W + x) * CV + cv), v);
#pragma unroll
            for (int k = 0; k < N; ++k) relu_max<T>(m[k], v[k], sh[k]);
          }
        reinterpret_cast<V*>(out)[row + j] = Pack<T>::pack(m);
      }
    } else {
      const float sh = round_to<T>(__ldg(shift + plane % C));
      const T* __restrict__ ip = conv + (size_t)plane * H * W;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int x0 = max(2 * j - 1, 0), x1 = min(2 * j + 2, W);
        float m = -INFINITY;
        for (int y = y0; y < y1; ++y)
          for (int x = x0; x < x1; ++x) relu_max<T>(m, to_f(__ldg(ip + (size_t)y * W + x)), sh);
        out[row + j] = from_f<T>(m);
      }
    }
  }
}

}  // namespace dgod

using namespace dgod;

template <typename T>
static int fpn_merge_fwd(const char* fn, const T* lat, const float* bias, const T* coarse, T* out, int n, int h, int w,
                         int hc, int wc, int c, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "%s: negative size", fn);
  if ((long long)n * h * w * c == 0) return DGOD_OK;
  DGOD_REQUIRE(hc > 0 && wc > 0, "%s: empty coarse map", fn);
  DGOD_REQUIRE(lat && bias && coarse && out, "%s: null pointer", fn);
  const long long rows = channels_last ? (long long)n * h : (long long)n * c * h;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "%s: map too large", fn);
  const float sh = (float)hc / (float)h, sw = (float)wc / (float)w;   // ATen: (float)input_size / output_size
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    constexpr int N = Pack<T>::N;
    DGOD_REQUIRE(c % N == 0, "%s: channels_last needs channels %% %d == 0, got %d", fn, N, c);
    DGOD_REQUIRE(aligned16(lat) && aligned16(bias) && aligned16(coarse) && aligned16(out),
                 "%s: channels_last needs 16-byte aligned pointers", fn);
    fpn_merge_fwd_kernel<T, true><<<row_grid(rows, w * (c / N)), 256, 0, st>>>(lat, bias, coarse, out, (int)rows, h, w,
                                                                             hc, wc, c, sh, sw);
  } else {
    fpn_merge_fwd_kernel<T, false><<<row_grid(rows, w), 256, 0, st>>>(lat, bias, coarse, out, (int)rows, h, w, hc, wc,
                                                                      c, sh, sw);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

template <typename T>
static int fpn_merge_bwd(const char* fn, const T* g_fine, const T* g_lb, T* g_coarse, int n, int h, int w, int hc,
                         int wc, int c, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && hc >= 0 && wc >= 0 && c >= 0, "%s: negative size", fn);
  if ((long long)n * hc * wc * c == 0) return DGOD_OK;
  DGOD_REQUIRE(h > 0 && w > 0, "%s: empty fine map", fn);
  DGOD_REQUIRE(g_fine && g_coarse, "%s: null pointer", fn);
  const long long rows = channels_last ? (long long)n * hc : (long long)n * c * hc;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "%s: map too large", fn);
  const float sh = (float)h / (float)hc, sw = (float)w / (float)wc;   // ATen: (float)output_size / input_size
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    constexpr int N = Pack<T>::N;
    DGOD_REQUIRE(c % N == 0, "%s: channels_last needs channels %% %d == 0, got %d", fn, N, c);
    DGOD_REQUIRE(aligned16(g_fine) && aligned16(g_lb) && aligned16(g_coarse),
                 "%s: channels_last needs 16-byte aligned pointers", fn);
    fpn_merge_bwd_kernel<T, true><<<row_grid(rows, wc * (c / N)), 256, 0, st>>>(g_fine, g_lb, g_coarse, (int)rows, h,
                                                                              w, hc, wc, c, sh, sw);
  } else {
    fpn_merge_bwd_kernel<T, false><<<row_grid(rows, wc), 256, 0, st>>>(g_fine, g_lb, g_coarse, (int)rows, h, w, hc, wc,
                                                                       c, sh, sw);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

template <typename T>
static int stem_pool_fwd(const char* fn, const T* conv, const float* shift, T* out, int n, int h, int w, int c, int ho,
                         int wo, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "%s: negative size", fn);
  DGOD_REQUIRE(ho == (h - 1) / 2 + 1 && wo == (w - 1) / 2 + 1 && h > 0 && w > 0,
               "%s: output %dx%d is not the 3x3 / stride 2 / pad 1 pooling of %dx%d", fn, ho, wo, h, w);
  if ((long long)n * c == 0) return DGOD_OK;
  DGOD_REQUIRE(conv && shift && out, "%s: null pointer", fn);
  const long long rows = channels_last ? (long long)n * ho : (long long)n * c * ho;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX, "%s: map too large", fn);
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    constexpr int N = Pack<T>::N;
    DGOD_REQUIRE(c % N == 0, "%s: channels_last needs channels %% %d == 0, got %d", fn, N, c);
    DGOD_REQUIRE(aligned16(conv) && aligned16(shift) && aligned16(out),
                 "%s: channels_last needs 16-byte aligned pointers", fn);
    stem_pool_kernel<T, true><<<row_grid(rows, wo * (c / N)), 256, 0, st>>>(conv, shift, out, (int)rows, h, w, c, ho,
                                                                          wo);
  } else {
    stem_pool_kernel<T, false><<<row_grid(rows, wo), 256, 0, st>>>(conv, shift, out, (int)rows, h, w, c, ho, wo);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

extern "C" int dgod_fpn_merge_fwd(const float* lat, const float* bias, const float* coarse, float* out, int n, int h,
                                  int w, int hc, int wc, int c, int channels_last, dgod_stream_t stream) {
  return fpn_merge_fwd<float>("dgod_fpn_merge_fwd", lat, bias, coarse, out, n, h, w, hc, wc, c, channels_last, stream);
}

extern "C" int dgod_fpn_merge_fwd_bf16(const void* lat, const float* bias, const void* coarse, void* out, int n, int h,
                                       int w, int hc, int wc, int c, int channels_last, dgod_stream_t stream) {
  return fpn_merge_fwd<__nv_bfloat16>("dgod_fpn_merge_fwd_bf16", (const __nv_bfloat16*)lat, bias,
                                      (const __nv_bfloat16*)coarse, (__nv_bfloat16*)out, n, h, w, hc, wc, c,
                                      channels_last, stream);
}

extern "C" int dgod_fpn_merge_bwd(const float* g_fine, const float* g_lb, float* g_coarse, int n, int h, int w, int hc,
                                  int wc, int c, int channels_last, dgod_stream_t stream) {
  return fpn_merge_bwd<float>("dgod_fpn_merge_bwd", g_fine, g_lb, g_coarse, n, h, w, hc, wc, c, channels_last, stream);
}

extern "C" int dgod_fpn_merge_bwd_bf16(const void* g_fine, const void* g_lb, void* g_coarse, int n, int h, int w,
                                       int hc, int wc, int c, int channels_last, dgod_stream_t stream) {
  return fpn_merge_bwd<__nv_bfloat16>("dgod_fpn_merge_bwd_bf16", (const __nv_bfloat16*)g_fine,
                                      (const __nv_bfloat16*)g_lb, (__nv_bfloat16*)g_coarse, n, h, w, hc, wc, c,
                                      channels_last, stream);
}

extern "C" int dgod_stem_pool_fwd(const float* conv, const float* shift, float* out, int n, int h, int w, int c, int ho,
                                  int wo, int channels_last, dgod_stream_t stream) {
  return stem_pool_fwd<float>("dgod_stem_pool_fwd", conv, shift, out, n, h, w, c, ho, wo, channels_last, stream);
}

extern "C" int dgod_stem_pool_fwd_bf16(const void* conv, const float* shift, void* out, int n, int h, int w, int c,
                                       int ho, int wo, int channels_last, dgod_stream_t stream) {
  return stem_pool_fwd<__nv_bfloat16>("dgod_stem_pool_fwd_bf16", (const __nv_bfloat16*)conv, shift,
                                      (__nv_bfloat16*)out, n, h, w, c, ho, wo, channels_last, stream);
}
