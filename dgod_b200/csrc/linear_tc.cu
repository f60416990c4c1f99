// fp32 matrix products on the tcgen05 tensor cores with fp32-level accuracy (3xTF32): the box head's fc6 / fc7
// Linear layers, forward and backward.
//
//   C[m, n] = epilogue( sum_k A[m, k] * B[n, k] )      A = op(a), B = op(b): a stored [m, k] or (a_trans) [k, m],
//                                                      b stored [n, k] or (b_trans) [k, n]
//   forward  Y  = X W^T (+ bias, ReLU)   a = X,  b = W                  (both K-major)
//   dgrad    dX = dY W  (* mask > 0)     a = dY, b = W, b_trans
//   wgrad    dW = dY^T X                 a = dY, a_trans, b = X, b_trans
//
// 3xTF32: every operand element x is split into hi = tf32_rna(x) and lo = tf32_rna(x - hi) (x - hi is exact, and both
// parts are exact tf32 values, so the tensor core's own fp32 -> tf32 reduction never matters); the accumulator receives
// A_hi B_lo + A_lo B_hi + A_hi B_hi, which carries the product to about the precision of an fp32 SGEMM.  Non-finite x
// split into (x, 0).  Where SGEMM's result is +-inf the split can give NaN (inf * 0 in a correction term whose other
// factor is exactly tf32-representable); every non-finite SGEMM result is non-finite here too, and vice versa.
//
// Two kernels per call:
//   split   a and b are split once into a caller-owned workspace, K-major, the K extent padded with zeros to a multiple
//           of 32.  The transposed operands (dgrad's W, wgrad's dY and X) are transposed by the same pass, so the
//           product kernel reads only K-major tiles.  The pass costs one read and two writes of each operand
//           (~0.6 GB of HBM traffic for fc6's X at 4096 RoIs, ~0.1 ms).
//   product persistent, warp-specialised, one CTA per SM.  Tiles of 128 x 256 (the largest single-CTA tcgen05 shape:
//           the operand reads of one 128x256x8 MMA are 96 B/clk against 128 B/clk of shared-memory bandwidth, a
//           128x128 tile would need all of it), K in blocks of 32 floats (one 128-byte swizzle row).
//           warp 8      TMA producer: hi and lo of the A and B tiles (96 KB a stage, 2 stages)
//           warp 9      TMEM allocation and the MMA issuer (one thread): 12 tcgen05.mma.kind::tf32 per K block into
//                       one of two TMEM accumulators (2 x 256 columns), alternating per K block
//           warps 0-7   epilogue: tcgen05.ld of each K block's partial product (thread = row; warp w reads the TMEM
//                       lanes of w % 4 and column half w / 4), summed in fp32 registers with round-to-nearest, then
//                       bias / ReLU / mask and 128-bit stores after the tile's last block.  The tensor core's own
//                       accumulation truncates: summed in TMEM over fc6's K = 12 544 the error grew to ~40x SGEMM's.
//           Tiles are dealt round-robin, n fastest: the CTAs that share an A block run together.
//           Tile counts at the box head's shapes (4096 RoIs): fc6 forward 32 x 4 = 128 tiles of K 12544 (one wave on
//           148 SMs, 86 % of them busy; split-K would give 1.7 waves of half the work, no better), fc6 dgrad 32 x 49 =
//           1568 tiles of K 1024, fc6 wgrad 8 x 49 = 392 tiles of K 4096 (2.65 waves).
//
// Bounds: any m >= 1, k >= 1; n % 32 == 0 (the epilogue stores 32-column chunks); pointers 16-byte aligned.  Rows past
// m and columns past n read as zero (TMA zero fill) and are not stored.
//
// Built with -DDGOD_DEBUG_WAITS, every mbarrier wait gives up after a bounded number of polls, records the barrier in
// g_linear_tc_timeout, prints it and ends its role, so a lost arrive ends the kernel instead of hanging the GPU.
#include "tmap.cuh"

namespace dgod {
namespace {

constexpr int BM = 128, BN = 256, BK = 32, STAGES = 2;
constexpr int A_TILE = BM * BK * 4, B_TILE = BN * BK * 4;       // 16 KB, 32 KB
constexpr int STAGE_BYTES = 2 * A_TILE + 2 * B_TILE;             // hi + lo of each: 96 KB
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;          // + alignment slack for the 1024-byte swizzle atoms
constexpr int TMEM_COLS = 2 * BN;                                // two fp32 accumulators of 128 lanes x 256 columns
constexpr int THREADS = 320;

#ifdef DGOD_DEBUG_WAITS
__device__ unsigned g_linear_tc_timeout;
#endif

__device__ __forceinline__ bool tc_wait(unsigned bar, unsigned parity) {
#ifdef DGOD_DEBUG_WAITS
  for (unsigned i = 0; i < (1u << 26); ++i) {
    unsigned ok;
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return true;
  }
  atomicExch(&g_linear_tc_timeout, bar | 0x80000000u);
  printf("linear_tc: mbarrier wait timed out (block %d, thread %d, barrier 0x%x, parity %u)\n", blockIdx.x, threadIdx.x,
         bar, parity);
  return false;
#else
  mbar_wait_s(bar, parity);
  return true;
#endif
}

__device__ __forceinline__ unsigned tf32_rna(float x) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ void split1(float x, float& hi, float& lo) {
  hi = __uint_as_float(tf32_rna(x));
  lo = isfinite(hi) ? __uint_as_float(tf32_rna(__fsub_rn(x, hi))) : 0.f;
}

// ---------------------------------------------------------------- split pass
// src [rows, k] -> hi / lo [rows, kp], zero-padded columns k .. kp-1.
__global__ void __launch_bounds__(256) split_kernel(const float* __restrict__ src, float* __restrict__ hi,
                                                    float* __restrict__ lo, long long rows, int k, int kp) {
  const long long total = rows * (long long)kp;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / kp;
    const int c = (int)(i - r * kp);
    float h = 0.f, l = 0.f;
    if (c < k) split1(__ldg(src + r * k + c), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}
// The same with 4 columns a thread when k % 4 == 0.
__global__ void __launch_bounds__(256) split4_kernel(const float4* __restrict__ src, float4* __restrict__ hi,
                                                     float4* __restrict__ lo, long long rows, int k4, int kp4) {
  const long long total = rows * (long long)kp4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / kp4;
    const int c = (int)(i - r * kp4);
    float4 h = make_float4(0.f, 0.f, 0.f, 0.f), l = h;
    if (c < k4) {
      const float4 v = __ldg(src + r * k4 + c);
      split1(v.x, h.x, l.x);
      split1(v.y, h.y, l.y);
      split1(v.z, h.z, l.z);
      split1(v.w, h.w, l.w);
    }
    hi[i] = h;
    lo[i] = l;
  }
}
// Transposing split: src [k, rows] -> hi / lo [rows, kp] through 32 x 32 shared-memory tiles.  grid (kp/32, rows/32).
__global__ void __launch_bounds__(256) split_t_kernel(const float* __restrict__ src, float* __restrict__ hi,
                                                      float* __restrict__ lo, int rows, int k, int kp) {
  __shared__ float t[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const int kk = c0 + j, r = r0 + tx;
    t[j][tx] = (kk < k && r < rows) ? __ldg(src + (size_t)kk * rows + r) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int r = r0 + j, kk = c0 + tx;
    if (r < rows) {
      float h, l;
      split1(t[tx][j], h, l);
      hi[(size_t)r * kp + kk] = h;
      lo[(size_t)r * kp + kk] = l;
    }
  }
}

// ---------------------------------------------------------------- tcgen05 helpers
// Shared-memory matrix descriptor of a K-major operand tile in the 128-byte swizzle layout the TMA writes: rows of
// 128 bytes, 8-row swizzle atoms of 1024 bytes (stride byte offset), the leading byte offset unused for this layout.
// Bits: start address >> 4 [0,14), leading byte offset >> 4 [16,30), stride byte offset >> 4 [32,46), descriptor
// version 1 [46,48), base offset 0 (atoms 1024-byte aligned), layout type SWIZZLE_128B = 2 [61,64).  A K step inside
// the 128-byte row advances the start address by its byte offset.
__device__ __forceinline__ unsigned long long sdesc(unsigned saddr) {
  return (unsigned long long)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((unsigned long long)(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
// Instruction descriptor of kind::tf32: D fp32 (bits [4,6) = 1), A and B tf32 (bits [7,10), [10,13) = 2), both
// K-major (bits 15, 16 = 0), N >> 3 at [17,23), M >> 4 at [24,29).
constexpr unsigned IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(BN >> 3) << 17) | ((unsigned)(BM >> 4) << 24);

__device__ __forceinline__ void mma_tf32(unsigned d_tmem, unsigned long long a, unsigned long long b, unsigned accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(a), "l"(b), "r"(IDESC), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit(unsigned bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(unsigned taddr, float (&v)[16]) {
  unsigned r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---------------------------------------------------------------- product kernel
struct Epilogue {
  const float* bias;   // [n] or nullptr
  const float* mask;   // [m, n] or nullptr: C *= (mask > 0)
  float* c;            // [m, n]
  int relu;
};

__global__ void __launch_bounds__(THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap ta_hi, const __grid_constant__ CUtensorMap ta_lo,
                 const __grid_constant__ CUtensorMap tb_hi, const __grid_constant__ CUtensorMap tb_lo, int m, int n, int kp,
                 Epilogue ep) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long full_bar[STAGES], empty_bar[STAGES], acc_full[2], acc_empty[2];
  __shared__ unsigned tmem_base_s;
  const unsigned smem = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mb = (m + BM - 1) / BM, nb = (n + BN - 1) / BN, n_tiles = mb * nb, kb_count = kp / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], 8);
    }
    mbar_fence_init();
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = tmem_base_s;

  if (warp == 8) {
    if (lane == 0) {                                   // ------------------------------ TMA producer
      tmap_prefetch(&ta_hi);
      tmap_prefetch(&ta_lo);
      tmap_prefetch(&tb_hi);
      tmap_prefetch(&tb_lo);
      int s = 0;
      unsigned ph = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int m0 = (t / nb) * BM, n0 = (t % nb) * BN;
        for (int kb = 0; kb < kb_count; ++kb) {
          if (!tc_wait(smem_u32(&empty_bar[s]), ph ^ 1)) goto done;
          mbar_expect_tx(&full_bar[s], STAGE_BYTES);
          unsigned char* st = smem_raw + (smem + s * STAGE_BYTES - smem_u32(smem_raw));
          tmap_load_2d(st, &ta_hi, kb * BK, m0, &full_bar[s]);
          tmap_load_2d(st + A_TILE, &ta_lo, kb * BK, m0, &full_bar[s]);
          tmap_load_2d(st + 2 * A_TILE, &tb_hi, kb * BK, n0, &full_bar[s]);
          tmap_load_2d(st + 2 * A_TILE + B_TILE, &tb_lo, kb * BK, n0, &full_bar[s]);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 9) {
    if (lane == 0) {                                   // ------------------------------ MMA issuer
      int s = 0;
      unsigned ph = 0;
      int q = 0;                                       // K blocks issued: accumulator buffer q & 1
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        for (int kb = 0; kb < kb_count; ++kb, ++q) {
          const int a = q & 1;
          if (!tc_wait(smem_u32(&acc_empty[a]), ((q >> 1) & 1) ^ 1)) goto done;
          if (!tc_wait(smem_u32(&full_bar[s]), ph)) goto done;
          tc_fence_after();
          const unsigned d = tmem + a * BN;
          const unsigned st = smem + s * STAGE_BYTES;
#pragma unroll
          for (int j = 0; j < BK / 8; ++j) {           // K = 8 per tf32 MMA: 32 bytes along the swizzled row
            const unsigned long long a_hi = sdesc(st + 32 * j), a_lo = sdesc(st + A_TILE + 32 * j);
            const unsigned long long b_hi = sdesc(st + 2 * A_TILE + 32 * j), b_lo = sdesc(st + 2 * A_TILE + B_TILE + 32 * j);
            // the two small correction terms first: each MMA's addition into the accumulator truncates, so the large
            // term comes last and is rounded once
            mma_tf32(d, a_hi, b_lo, j != 0);
            mma_tf32(d, a_lo, b_hi, 1);
            mma_tf32(d, a_hi, b_hi, 1);
          }
          mma_commit(smem_u32(&empty_bar[s]));        // frees the stage once these MMAs have read it
          mma_commit(smem_u32(&acc_full[a]));         // this K block's partial product is ready for the epilogue
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {                                             // ------------------------------ epilogue (warps 0-7)
    // Warp w reads TMEM lanes 32 (w % 4) .. + 31 (its rows) and columns 128 (w / 4) .. + 127 of the accumulator.  The
    // tensor core's accumulation truncates; summing each K block's partial product here in fp32 with round-to-nearest
    // keeps the error of a long K at the level of an fp32 SGEMM instead of growing with K.
    const int quarter = warp & 3, half = warp >> 2;
    int q = 0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const int m0 = (t / nb) * BM, n0 = (t % nb) * BN + half * (BN / 2);
      float acc[BN / 2];
#pragma unroll
      for (int i = 0; i < BN / 2; ++i) acc[i] = 0.f;
      for (int kb = 0; kb < kb_count; ++kb, ++q) {
        const int a = q & 1;
        if (!tc_wait(smem_u32(&acc_full[a]), (q >> 1) & 1)) goto done;
        tc_fence_after();
        const unsigned taddr = tmem + a * BN + half * (BN / 2) + ((unsigned)(quarter * 32) << 16);
#pragma unroll
        for (int ch = 0; ch < BN / 32; ++ch) {
          float v[16];
          tmem_ld16(taddr + ch * 16, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[ch * 16 + i] = __fadd_rn(acc[ch * 16 + i], v[i]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[a]);     // buffer read: the MMA warp may overwrite it
      }
      const int row = m0 + quarter * 32 + lane;
#pragma unroll
      for (int ch = 0; ch < BN / 64; ++ch) {
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = acc[ch * 32 + i];
        const int c0 = n0 + ch * 32;
        if (row < m && c0 < n) {
          if (ep.bias) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + c0) + i);
              v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
            }
          }
          if (ep.relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = v[i] > 0.f ? v[i] : (v[i] == v[i] ? 0.f : v[i]);   // NaN passes
          }
          const size_t off = (size_t)row * n + c0;
          if (ep.mask) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 g = __ldg(reinterpret_cast<const float4*>(ep.mask + off) + i);
              if (!(g.x > 0.f)) v[4 * i] = 0.f;
              if (!(g.y > 0.f)) v[4 * i + 1] = 0.f;
              if (!(g.z > 0.f)) v[4 * i + 2] = 0.f;
              if (!(g.w > 0.f)) v[4 * i + 3] = 0.f;
            }
          }
          float4* dst = reinterpret_cast<float4*>(ep.c + off);
#pragma unroll
          for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        }
      }
    }
  }
done:
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
  }
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
      (void)cudaGetLastError();
      n = 148;
    }
  }
  return n;
}

inline int kpad(int k) { return (k + BK - 1) / BK * BK; }

int split(const float* src, int trans, int rows, int k, float* hi, float* lo, cudaStream_t st) {
  const int kp = kpad(k);
  if (trans) {
    split_t_kernel<<<dim3(kp / 32, (rows + 31) / 32), 256, 0, st>>>(src, hi, lo, rows, k, kp);
  } else {
    const long long total = (long long)rows * kp;
    const int blocks = (int)std::min<long long>((total / ((k % 4 == 0) ? 4 : 1) + 255) / 256, 32LL * sm_count());
    if (k % 4 == 0)
      split4_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(src), reinterpret_cast<float4*>(hi),
                                            reinterpret_cast<float4*>(lo), rows, k / 4, kp / 4);
    else
      split_kernel<<<blocks, 256, 0, st>>>(src, hi, lo, rows, k, kp);
  }
  DGOD_LAUNCHED();
  return DGOD_OK;
}

}  // namespace
}  // namespace dgod

using namespace dgod;

extern "C" size_t dgod_linear_tc_workspace_bytes(int m, int n, int k) {
  if (m < 1 || n < 1 || k < 1) return 0;
  return 2 * ((size_t)m + (size_t)n) * (size_t)kpad(k) * sizeof(float) + 1024;
}

extern "C" int dgod_linear_tc(const float* a, int a_trans, const float* b, int b_trans, int m, int n, int k,
                              const float* bias, int relu, const float* mask, float* c, void* workspace,
                              size_t workspace_bytes, dgod_stream_t stream) {
  DGOD_REQUIRE(a && b && c && workspace, "dgod_linear_tc: a, b, c and workspace must not be NULL");
  DGOD_REQUIRE(m >= 1 && n >= 1 && k >= 1, "dgod_linear_tc: m, n, k must be >= 1 (got %d, %d, %d)", m, n, k);
  DGOD_REQUIRE(n % 32 == 0, "dgod_linear_tc: n must be a multiple of 32 (got %d)", n);
  DGOD_REQUIRE(workspace_bytes >= dgod_linear_tc_workspace_bytes(m, n, k),
               "dgod_linear_tc: workspace of %zu bytes, %zu needed", workspace_bytes, dgod_linear_tc_workspace_bytes(m, n, k));
  DGOD_REQUIRE(aligned16(a) && aligned16(b) && aligned16(c) && (!bias || aligned16(bias)) && (!mask || aligned16(mask)),
               "dgod_linear_tc: every pointer must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int kp = kpad(k);
  char* ws = (char*)(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
  float* a_hi = (float*)ws;
  float* a_lo = a_hi + (size_t)m * kp;
  float* b_hi = a_lo + (size_t)m * kp;
  float* b_lo = b_hi + (size_t)n * kp;
  int rc;
  if ((rc = split(a, a_trans, m, k, a_hi, a_lo, st)) != DGOD_OK) return rc;
  if ((rc = split(b, b_trans, n, k, b_hi, b_lo, st)) != DGOD_OK) return rc;
  CUtensorMap ta_hi, ta_lo, tb_hi, tb_lo;
  if ((rc = encode_f32_2d_sw128(&ta_hi, a_hi, m, kp, BM)) != DGOD_OK) return rc;
  if ((rc = encode_f32_2d_sw128(&ta_lo, a_lo, m, kp, BM)) != DGOD_OK) return rc;
  if ((rc = encode_f32_2d_sw128(&tb_hi, b_hi, n, kp, BN)) != DGOD_OK) return rc;
  if ((rc = encode_f32_2d_sw128(&tb_lo, b_lo, n, kp, BN)) != DGOD_OK) return rc;
  static bool attr = false;
  if (!attr) {
    DGOD_CUDA(cudaFuncSetAttribute(linear_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr = true;
  }
  const int tiles = ((m + BM - 1) / BM) * ((n + BN - 1) / BN);
  Epilogue ep{bias, mask, c, relu ? 1 : 0};
  linear_tc_kernel<<<std::min(tiles, sm_count()), THREADS, SMEM_BYTES, st>>>(ta_hi, ta_lo, tb_hi, tb_lo, m, n, kp, ep);
  DGOD_LAUNCHED();
  return DGOD_OK;
}
