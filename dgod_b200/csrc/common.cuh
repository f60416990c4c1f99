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
