// Shared device/host helpers for the dgod_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/dgod_b200.h"

namespace dgod {

// ---------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launches;

#define DGOD_REQUIRE(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      ::dgod::set_error(__VA_ARGS__);           \
      return DGOD_ERR_ARG;                      \
    }                                           \
  } while (0)

#define DGOD_CUDA(expr)                                                              \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) {                                                         \
      ::dgod::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                        __FILE__, __LINE__);                                         \
      return DGOD_ERR_CUDA;                                                          \
    }                                                                                \
  } while (0)

// Call after every <<<>>> launch: counts it and surfaces launch-configuration errors.
#define DGOD_LAUNCHED()                                              \
  do {                                                               \
    ::dgod::g_launches.fetch_add(1, std::memory_order_relaxed);      \
    DGOD_CUDA(cudaGetLastError());                                   \
  } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over the caller's workspace (256-byte aligned slices).
struct Workspace {
  char* base;
  size_t size, used;
  Workspace(void* p, size_t n) : base((char*)p), size(n), used(0) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    T* r = (T*)(base + used);
    used += bytes;
    return r;
  }
  bool ok() const { return used <= size; }
};

// ---------------------------------------------------------------- exact fp32 box arithmetic
// torchvision's CPU ops never contract a*b+c; the __f*_rn intrinsics are never fused by nvcc,
// which keeps every IoU bit-identical to the oracle regardless of -fmad.

__device__ __forceinline__ float box_area_exact(float x1, float y1, float x2, float y2) {
  return __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));  // TV ops/boxes.py:299
}

// IoU in the operation order shared by box_iou (TV ops/boxes.py:336-339,369) and the CPU nms
// kernel (inter / (iarea + areas[j] - inter)); SURVEY.md §8c probed them bit-identical.
__device__ __forceinline__ float iou_exact(const float4 a, float area_a, const float4 b,
                                           float area_b) {
  float lx = fmaxf(a.x, b.x), ly = fmaxf(a.y, b.y);
  float rx = fminf(a.z, b.z), ry = fminf(a.w, b.w);
  float w = fmaxf(__fsub_rn(rx, lx), 0.f);
  float h = fmaxf(__fsub_rn(ry, ly), 0.f);
  float inter = __fmul_rn(w, h);
  float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  return __fdiv_rn(inter, uni);
}

// Same value, bit for bit, without the IEEE division for disjoint boxes: inter == +0 and a positive
// union give exactly +0 (the common case of an anchor far from a ground truth).
__device__ __forceinline__ float iou_exact_skip(const float4 a, float area_a, const float4 b,
                                                float area_b) {
  float lx = fmaxf(a.x, b.x), ly = fmaxf(a.y, b.y);
  float rx = fminf(a.z, b.z), ry = fminf(a.w, b.w);
  float w = fmaxf(__fsub_rn(rx, lx), 0.f);
  float h = fmaxf(__fsub_rn(ry, ly), 0.f);
  float inter = __fmul_rn(w, h);
  float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  if (inter == 0.f && uni > 0.f) return 0.f;
  return __fdiv_rn(inter, uni);
}

// Monotone map float -> uint32 (a < b  <=>  key(a) < key(b) for non-NaN values).
__device__ __forceinline__ uint32_t float_ordered(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float float_from_ordered(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

// ATen's relu_ on CUDA is clamp_min(v, 0) (TensorCompare.cu, launch_clamp_scalar): NaN passes through, everything else
// is ::max(v, 0), i.e. fmaxf — the same instruction, so signed zeros come out as ATen's do.
__device__ __forceinline__ float clamp_min0(float v) { return isnan(v) ? v : fmaxf(v, 0.f); }

// ---------------------------------------------------------------- storage types of the backbone epilogue kernels
// Maps are stored as T (float or __nv_bfloat16) and computed on in fp32 ("opmath", as ATen does for bf16).  A 16-byte
// access holds Pack<T>::N = 1 << Pack<T>::SHIFT values.  round_to<T> is the rounding an ATen op applies when its result
// is a T tensor: none for float, round-to-nearest-even for bf16 (c10::BFloat16(float) is __float2bfloat16 on sm_80+).
template <typename T> struct Pack;
template <> struct Pack<float> {
  static constexpr int N = 4, SHIFT = 2;
  typedef float4 V;
  __device__ __forceinline__ static void unpack(const float4 v, float (&f)[4]) {
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
  __device__ __forceinline__ static float4 pack(const float (&f)[4]) { return make_float4(f[0], f[1], f[2], f[3]); }
};
template <> struct Pack<__nv_bfloat16> {
  static constexpr int N = 8, SHIFT = 3;
  typedef uint4 V;
  __device__ __forceinline__ static void unpack(const uint4 v, float (&f)[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ static uint4 pack(const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
};

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <typename T> __device__ __forceinline__ float round_to(float v) { return to_f(from_f<T>(v)); }

// The N fp32 per-channel values (shifts, biases) that go with 16-byte map vector `i`: p must be 16-byte aligned.
template <int N>
__device__ __forceinline__ void ldg_channels(const float* __restrict__ p, int i, float (&f)[N]) {
#pragma unroll
  for (int k = 0; k < N / 4; ++k) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p) + i * (N / 4) + k);
    f[4 * k] = v.x; f[4 * k + 1] = v.y; f[4 * k + 2] = v.z; f[4 * k + 3] = v.w;
  }
}

// Streaming passes over [rows x row_len] maps: rows go to the grid's y dimension (at most 65535, the kernels stride over
// the rest), a row's elements to x in blocks of 256 threads.
static inline dim3 row_grid(long long rows, int row_len) {
  return dim3((unsigned)cdiv(row_len, 256), (unsigned)(rows < 65535 ? rows : 65535));
}

static inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

__device__ __forceinline__ float4 ld_box(const float* p, long long i) {
  return __ldg(reinterpret_cast<const float4*>(p) + i);
}

// Largest float f with (double)f <= t: `(double)x > t`  <=>  `x > f` for every float x.
static inline float float_round_down(double t) {
  float f = (float)t;
  if ((double)f > t) f = nextafterf(f, -INFINITY);
  return f;
}

// Programmatic dependent launch (griddepcontrol): a kernel launched with launch_pdl() may start while its predecessor in
// the stream is still running; it must call pdl_wait() before touching anything the predecessor wrote (the call returns
// when the predecessor grid has completed and its writes are visible).  pdl_trigger() in the predecessor lets the
// dependent's CTAs be scheduled as soon as every predecessor CTA has called it (or exited) and resources allow — what
// is saved is the launch latency and the dependent's prologue (barrier init, descriptor prefetch), a few us per boundary.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace dgod
