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
// NHWC: one thread owns 4 consecutive channels of a pixel (128-bit accesses, C % 4 == 0), the grid's y dimension walks
// the rows (n, y); NCHW: one element per thread, the grid's y dimension walks the planes (n, c).  Both grid-stride.
#include "common.cuh"

namespace dgod {

enum { SR_PLAIN = 0, SR_RESIDUAL = 1, SR_SHIFTED_RESIDUAL = 2 };

template <int FORM>
__device__ __forceinline__ float shift_relu1(float c, float s, float r, float t) {
  float v = __fadd_rn(c, s);
  if (FORM == SR_RESIDUAL) v = __fadd_rn(v, r);
  if (FORM == SR_SHIFTED_RESIDUAL) v = __fadd_rn(v, __fadd_rn(r, t));
  return clamp_min0(v);
}

template <bool NHWC, int FORM>
__global__ void __launch_bounds__(256)
shift_relu_kernel(const float* __restrict__ conv, const float* __restrict__ shift, const float* __restrict__ res,
                  const float* __restrict__ res_shift, float* __restrict__ out, int rows, int row_len, int C) {
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const size_t row = (size_t)r * row_len;
    if (NHWC) {
      const int C4 = C >> 2;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x) {
        const int c4 = j % C4;
        const float4 v = reinterpret_cast<const float4*>(conv)[row + j];
        const float4 s = __ldg(reinterpret_cast<const float4*>(shift) + c4);
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f), t = q;
        if (FORM != SR_PLAIN) q = reinterpret_cast<const float4*>(res)[row + j];
        if (FORM == SR_SHIFTED_RESIDUAL) t = __ldg(reinterpret_cast<const float4*>(res_shift) + c4);
        reinterpret_cast<float4*>(out)[row + j] =
            make_float4(shift_relu1<FORM>(v.x, s.x, q.x, t.x), shift_relu1<FORM>(v.y, s.y, q.y, t.y),
                        shift_relu1<FORM>(v.z, s.z, q.z, t.z), shift_relu1<FORM>(v.w, s.w, q.w, t.w));
      }
    } else {
      const int ch = r % C;
      const float s = __ldg(shift + ch), t = FORM == SR_SHIFTED_RESIDUAL ? __ldg(res_shift + ch) : 0.f;
      for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < row_len; j += gridDim.x * blockDim.x)
        out[row + j] = shift_relu1<FORM>(conv[row + j], s, FORM != SR_PLAIN ? res[row + j] : 0.f, t);
    }
  }
}

template <bool NHWC>
static void launch_shift_relu(int form, dim3 grid, cudaStream_t st, const float* conv, const float* shift,
                              const float* res, const float* res_shift, float* out, int rows, int row_len, int c) {
  if (form == SR_PLAIN)
    shift_relu_kernel<NHWC, SR_PLAIN><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len, c);
  else if (form == SR_RESIDUAL)
    shift_relu_kernel<NHWC, SR_RESIDUAL><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len, c);
  else
    shift_relu_kernel<NHWC, SR_SHIFTED_RESIDUAL><<<grid, 256, 0, st>>>(conv, shift, res, res_shift, out, rows, row_len,
                                                                        c);
}

}  // namespace dgod

using namespace dgod;

extern "C" int dgod_shift_relu_fwd(const float* conv, const float* shift, const float* res, const float* res_shift,
                                   float* out, int n, int h, int w, int c, int channels_last, dgod_stream_t stream) {
  DGOD_REQUIRE(n >= 0 && h >= 0 && w >= 0 && c >= 0, "dgod_shift_relu_fwd: negative size");
  if ((long long)n * h * w * c == 0) return DGOD_OK;
  DGOD_REQUIRE(conv && shift && out, "dgod_shift_relu_fwd: null pointer");
  DGOD_REQUIRE(res || !res_shift, "dgod_shift_relu_fwd: res_shift given without res");
  const long long rows = channels_last ? (long long)n * h : (long long)n * c;
  DGOD_REQUIRE(rows <= INT32_MAX && (long long)w * c <= INT32_MAX && (long long)h * w <= INT32_MAX,
               "dgod_shift_relu_fwd: map too large");
  const int form = res_shift ? SR_SHIFTED_RESIDUAL : res ? SR_RESIDUAL : SR_PLAIN;
  cudaStream_t st = (cudaStream_t)stream;
  if (channels_last) {
    DGOD_REQUIRE(c % 4 == 0, "dgod_shift_relu_fwd: channels_last needs channels %% 4 == 0, got %d", c);
    DGOD_REQUIRE(aligned16(conv) && aligned16(shift) && aligned16(res) && aligned16(res_shift) && aligned16(out),
                 "dgod_shift_relu_fwd: channels_last needs 16-byte aligned pointers");
    const int row_len = w * (c / 4);
    launch_shift_relu<true>(form, row_grid(rows, row_len), st, conv, shift, res, res_shift, out, (int)rows, row_len, c);
  } else {
    launch_shift_relu<false>(form, row_grid(rows, h * w), st, conv, shift, res, res_shift, out, (int)rows, h * w, c);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}
