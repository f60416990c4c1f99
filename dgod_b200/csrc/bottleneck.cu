// The elementwise epilogues of a ResNet Bottleneck whose convolutions have their frozen BatchNorm folded in: one streaming
// pass per convolution instead of ATen's bias add, residual add and ReLU passes.  Bit-exact with the ATen composition.
//
// Reference behaviour restated (torchvision 0.26.0 models/resnet.py, Bottleneck.forward, on convolutions that carry the
// folded shift as their bias; ATen Convolution.cpp adds a cuDNN convolution's bias in a separate add_ after the
// convolution, TensorCompare.cu):
//   conv1, conv2      out = relu_(conv(x) + s)
//   identity tail     out = relu_((conv3(y) + s) + x)
//   downsample tail   out = relu_((conv3(y) + s) + (conv_d(x) + t))
// relu_ is clamp_min(v, 0) (clamp_min0).  Each add is one fp32 rounding, in the order above.
// bf16 maps (the block under torch.autocast(dtype=bfloat16)): fp32 math, and every add's result rounded to bf16 (RNE);
// the fp32 shifts are rounded to bf16 first, as autocast casts the conv's bias before ATen's add_:
//   v = bf16(c + bf16(s)), then bf16(v + r) (identity tail) or bf16(v + bf16(r + bf16(t))) (downsample tail), relu_.
// dgod_bias_add_fwd is the fp32 SR_PLAIN instance without the ReLU: out = c + s (an FPN layer block's bias).
// NHWC: one thread owns one 16-byte vector of a pixel's channels (4 fp32 or 8 bf16: C % 4 or C % 8 == 0), the grid's y
// dimension walks the rows (n, y); NCHW: one element per thread, the grid's y dimension walks the planes (n, c).  Both
// grid-stride.
#include "common.cuh"

namespace dgod {

enum { SR_PLAIN = 0, SR_RESIDUAL = 1, SR_SHIFTED_RESIDUAL = 2 };

// The shifts s and t arrive rounded to T (a bf16 conv's bias is cast to bf16 by autocast and added by a separate add_).
template <typename T, int FORM, bool RELU>
__device__ __forceinline__ float shift_relu1(float c, float s, float r, float t) {
  float v = round_to<T>(__fadd_rn(c, s));
  if (FORM == SR_RESIDUAL) v = round_to<T>(__fadd_rn(v, r));
  if (FORM == SR_SHIFTED_RESIDUAL) v = round_to<T>(__fadd_rn(v, round_to<T>(__fadd_rn(r, t))));
  return RELU ? clamp_min0(v) : v;
}

template <typename T, bool NHWC, int FORM, bool RELU>
__global__ void __launch_bounds__(256)
shift_relu_kernel(const T* __restrict__ conv, const float* __restrict__ shift, const T* __restrict__ res,
                  const float* __restrict__ res_shift, T* __restrict__ out, int rows, int row_len, int C) {
  constexpr int N = Pack<T>::N;
  typedef typename Pack<T>::V V;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int CV = C >> Pack<T>::SHIFT;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int cv = j % CV;
        float v[N], s[N], q[N], t[N];
        Pack<T>::unpack(reinterpret_cast<const V*>(conv)[row + j], v);
        ldg_channels<N>(shift, cv, s);
#pragma unroll
        for (int k = 0; k < N; ++k) q[k] = t[k] = 0.f;
        if (FORM != SR_PLAIN) Pack<T>::unpack(reinterpret_cast<const V*>(res)[row + j], q);
        if (FORM == SR_SHIFTED_RESIDUAL) ldg_channels<N>(res_shift, cv, t);
#pragma unroll
        for (int k = 0; k < N; ++k) v[k] = shift_relu1<T, FORM, RELU>(v[k], round_to<T>(s[k]), q[k], round_to<T>(t[k]));
        reinterpret_cast<V*>(out)[row + j] = Pack<T>::pack(v);
      }
    } else {
      const int ch = r % C;
      const float s = round_to<T>(__ldg(shift + ch));
      const float t = FORM == SR_SHIFTED_RESIDUAL ? round_to<T>(__ldg(res_shift + ch)) : 0.f;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x)
        out[row + j] = from_f<T>(shift_relu1<T, FORM, RELU>(to_f(conv[row + j]), s, FORM != SR_PLAIN ? to_f(res[row + j]) : 0.f, t));
    }
  }
}

template <typename T, bool NHWC>
static void launch_shift_relu(int form, bool relu, dim3 grid, cudaStream_t st, const T* conv, const float* shift,
                              const T* res, const float* res_shift, T* out, int rows, int row_len, int c) {
  if (form == SR_PLAIN && !relu)
    shift_relu_kernel<T, NHWC, SR_PLAIN, false><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len, c);
  else if (form == SR_PLAIN)
    shift_relu_kernel<T, NHWC, SR_PLAIN, true><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len, c);
  else if (form == SR_RESIDUAL)
    shift_relu_kernel<T, NHWC, SR_RESIDUAL, true><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len,
                                                                        c);
  else
    shift_relu_kernel<T, NHWC, SR_SHIFTED_RESIDUAL, true><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows,
                                                                                 row_len, c);
}

template <typename T>
static int shift_relu_fwd(const char* fn, const T* conv, const float* shift, const T* res, const float* res_shift,
                          T* out, int n, int h, int w, int c, int channels_last, int relu, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "%s: negative size", fn);
  if ((long long)n * h * w * c == 0) return DGOD_OK;
  DGOD_REQUIRE(conv && shift && out, "%s: null pointer", fn);
  DGOD_REQUIRE(res || !res_shift, "%s: res_shift given without res", fn);
  DGOD_REQUIRE(relu || !res, "%s: the residual forms always end in the ReLU", fn);
  const long long rows = channels_last ? (long long)n * h : (long long)n * c;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX && (long long)h * w <= INT32_MAX,
               "%s: map too large", fn);
  const int form = res_shift ? SR_SHIFTED_RESIDUAL : res ? SR_RESIDUAL : SR_PLAIN;
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    constexpr int N = Pack<T>::N;
    DGOD_REQUIRE(c % N == 0, "%s: channels_last needs channels %% %d == 0, got %d", fn, N, c);
    DGOD_REQUIRE(aligned16(conv) && aligned16(shift) && aligned16(res) && aligned16(res_shift) && aligned16(out),
                 "%s: channels_last needs 16-byte aligned pointers", fn);
    const int row_len = w * (c / N);
    launch_shift_relu<T, true>(form, relu != 0, row_grid(rows, row_len), st, conv, shift, res, res_shift, out, (int)rows, row_len,
                               c);
  } else {
    launch_shift_relu<T, false>(form, relu != 0, row_grid(rows, h * w), st, conv, shift, res, res_shift, out, (int)rows, h * w, c);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_shift_relu_fwd(const float* conv, const float* shift, const float* res, const float* res_shift,
                                   float* out, int n, int h, int w, int c, int channels_last, dgod_stream_t stream) {
  return shift_relu_fwd<float>("dgod_shift_relu_fwd", conv, shift, res, res_shift, out, n, h, w, c, channels_last, 1,
                               stream);
}

extern "C" int dgod_bias_add_fwd(const float* conv, const float* bias, float* out, int n, int h, int w, int c,
                                 int channels_last, dgod_stream_t stream) {
  return shift_relu_fwd<float>("dgod_bias_add_fwd", conv, bias, nullptr, nullptr, out, n, h, w, c, channels_last, 0,
                               stream);
}

extern "C" int dgod_shift_relu_fwd_bf16(const void* conv, const float* shift, const void* res, const float* res_shift,
                                        void* out, int n, int h, int w, int c, int channels_last, dgod_stream_t stream) {
  return shift_relu_fwd<__nv_bfloat16>("dgod_shift_relu_fwd_bf16", (const __nv_bfloat16*)conv, shift,
                                       (const __nv_bfloat16*)res, res_shift, (__nv_bfloat16*)out, n, h, w, c,
                                       channels_last, 1, stream);
}
