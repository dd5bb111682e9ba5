// Shared device helpers for the icr_b200 kernels (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/icr_b200.h"

namespace icr {

constexpr float kNormEps = 1e-12f;  // F.normalize eps used by sentence-transformers cos_sim
constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- host-side error plumbing (api.cu) -------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
void count_launch();
// no-ops unless icr_profile_enable(1): CUDA events around the dominant kernel of a call
void profile_begin(int kernel_id, int mma_terms, cudaStream_t st);
void profile_end(cudaStream_t st);
constexpr int kKernelGemv = 1, kKernelGemm = 2;

#define ICR_CUDA_CHECK(expr)                                  \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return ::icr::cuda_fail(_e, #expr); \
  } while (0)

#define ICR_LAUNCH_CHECK()                                              \
  do {                                                                  \
    ::icr::count_launch();                                              \
    cudaError_t _e = cudaGetLastError();                                \
    if (_e != cudaSuccess) return ::icr::cuda_fail(_e, "kernel launch"); \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: each launcher remembers, per host
// thread, on which devices it has configured its kernel (a thread may serve cuda:0 and then cuda:1).
struct SmemAttrCache {
  unsigned long long devmask = 0;
};
// the same for launchers whose shared-memory need varies with the problem: remembers the largest size set per device
struct SmemSizeCache {
  size_t bytes[64] = {};
};
template <typename F>
inline int ensure_dyn_smem_size(SmemSizeCache& c, F func, size_t bytes) {
  int dev = 0;
  ICR_CUDA_CHECK(cudaGetDevice(&dev));
  const bool tracked = dev >= 0 && dev < 64;
  if (tracked && bytes <= c.bytes[dev]) return ICR_OK;
  ICR_CUDA_CHECK(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
  if (tracked) c.bytes[dev] = bytes;
  return ICR_OK;
}
template <typename F>
inline int ensure_dyn_smem(SmemAttrCache& c, F func, size_t bytes) {
  int dev = 0;
  ICR_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && ((c.devmask >> dev) & 1ull)) return ICR_OK;
  ICR_CUDA_CHECK(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
  if (dev >= 0 && dev < 64) c.devmask |= 1ull << dev;
  return ICR_OK;
}

// ---- candidate keys -----------------------------------------------------------------------
// A candidate is one 64-bit key: high word = order-preserving image of the fp32 score, low
// word = ~row. Larger key == better candidate: higher score first, lower row on ties. Key 0
// is "empty" (no finite score maps to it).
__host__ __device__ __forceinline__ uint32_t order_bits(float s) {
  s += 0.0f;  // -0.0 -> +0.0 so that equal scores compare equal
#ifdef __CUDA_ARCH__
  uint32_t b = __float_as_uint(s);
#else
  uint32_t b;
  memcpy(&b, &s, 4);
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float unorder_bits(uint32_t b) {
  b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  float s;
  memcpy(&s, &b, 4);
  return s;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float s, uint32_t row) {
  return (static_cast<uint64_t>(order_bits(s)) << 32) | static_cast<uint64_t>(~row);
}
__host__ __device__ __forceinline__ float key_score(uint64_t k) { return unorder_bits(static_cast<uint32_t>(k >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_row(uint64_t k) { return ~static_cast<uint32_t>(k); }

// ---- excluded rows ---------------------------------------------------------------------------
// `shared`: one byte per catalog row, the same for every query of a call. `bits`: per-query bitmap [ceil(N/32)][ld]
// (icr_query_exclusion_bits), row r excluded for query q when bit r % 32 of bits[r / 32][q] is set. The word index is
// outermost because the 32 rows of one epilogue block always share a word: 32 consecutive queries then read one
// 128-byte line (K2), and 32 consecutive rows of one query read one word (K2s, the selects).
// The kernels that accept a bitmap are separate instantiations (template flag BITS): the others compile to the
// shared-mask test alone.
struct Exclusions {
  const uint8_t* shared;
  const uint32_t* bits;
  int64_t ld;  // queries per word row of `bits`
  __device__ __forceinline__ uint32_t word(int64_t q, int64_t row32) const { return __ldg(bits + row32 * ld + q); }
  __device__ __forceinline__ bool bit(int64_t q, int64_t row) const { return (word(q, row >> 5) >> (row & 31)) & 1u; }
  template <bool BITS>
  __device__ __forceinline__ bool excluded(int64_t q, int64_t row) const {
    if (shared && shared[row]) return true;
    if constexpr (BITS) return bit(q, row);
    return false;
  }
};

// ---- vector loads -------------------------------------------------------------------------
// streaming 128-bit load: read-only path, do not allocate in L1 (catalog rows are used once)
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// Element traits: VEC elements per 16-byte load, expanded to fp32.
template <typename T>
struct Elem;
template <>
struct Elem<float> {
  static constexpr int VEC = 4;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = __uint_as_float(v.x);
    f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z);
    f[3] = __uint_as_float(v.w);
  }
  __device__ static __forceinline__ float to_f32(float x) { return x; }
  __device__ static __forceinline__ float from_f32(float x) { return x; }
};
template <>
struct Elem<__nv_bfloat16> {
  static constexpr int VEC = 8;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = bf16lo(v.x);
    f[1] = bf16hi(v.x);
    f[2] = bf16lo(v.y);
    f[3] = bf16hi(v.y);
    f[4] = bf16lo(v.z);
    f[5] = bf16hi(v.z);
    f[6] = bf16lo(v.w);
    f[7] = bf16hi(v.w);
  }
  __device__ static __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
  __device__ static __forceinline__ __nv_bfloat16 from_f32(float x) { return __float2bfloat16_rn(x); }
};

template <>
struct Elem<__half> {
  static constexpr int VEC = 8;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 p = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      f[2 * i] = p.x;
      f[2 * i + 1] = p.y;
    }
  }
  __device__ static __forceinline__ float to_f32(__half x) { return __half2float(x); }
  __device__ static __forceinline__ __half from_f32(float x) { return __float2half_rn(x); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
  return v;
}

// Transposing warp reduction: every lane holds V partial sums acc[0..V); on return lane l
// holds in acc[0] the full 32-lane sum of value index (l >> (5 - log2 V)). V shuffles in
// total instead of 5*V.
template <int V>
__device__ __forceinline__ void warp_transpose_reduce(float (&acc)[V], int lane) {
  static_assert(V == 1 || V == 2 || V == 4 || V == 8 || V == 16 || V == 32, "V must be a power of two <= 32");
  int off = 16;
#pragma unroll
  for (int n = V; n > 1; n >>= 1, off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = upper ? acc[i] : acc[i + n / 2];
      const float keep = upper ? acc[i + n / 2] : acc[i];
      acc[i] = keep + __shfl_xor_sync(kFull, send, off);
    }
  }
#pragma unroll
  for (; off > 0; off >>= 1) acc[0] += __shfl_xor_sync(kFull, acc[0], off);
}

// The same exchange pattern with max instead of +: on return lane l holds in acc[0] the maximum over the 32 lanes of value
// index (l >> (5 - log2 V)).
template <int V>
__device__ __forceinline__ void warp_transpose_max(float (&acc)[V], int lane) {
  static_assert(V == 1 || V == 2 || V == 4 || V == 8 || V == 16 || V == 32, "V must be a power of two <= 32");
  int off = 16;
#pragma unroll
  for (int n = V; n > 1; n >>= 1, off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = upper ? acc[i] : acc[i + n / 2];
      const float keep = upper ? acc[i + n / 2] : acc[i];
      acc[i] = fmaxf(keep, __shfl_xor_sync(kFull, send, off));
    }
  }
#pragma unroll
  for (; off > 0; off >>= 1) acc[0] = fmaxf(acc[0], __shfl_xor_sync(kFull, acc[0], off));
}

// ---- shared-memory bitonic sort of 64-bit keys, DESCENDING, n = power of two ------------------
// All threads of the CTA must call it; ends with __syncthreads().
__device__ __forceinline__ void block_bitonic_sort_desc(uint64_t* keys, int n) {
  __syncthreads();
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        // stride is a power of two: index arithmetic by mask/shift (an integer divide here costs more than the sort)
        const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a < b) == desc) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
      __syncthreads();
    }
  }
}

// warp-synchronous bitonic sort (descending) of n = power-of-two keys in shared memory
__device__ __forceinline__ void warp_bitonic_sort_desc(uint64_t* keys, int n, int lane) {
  __syncwarp();
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = lane; t < (n >> 1); t += 32) {
        const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a < b) == desc) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
      __syncwarp();
    }
  }
}

__host__ __device__ __forceinline__ int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// arguments of the MNRL kernels (mnrl.cu), filled by api.cu
struct MnrlArgs {
  const void* a;
  const void* p;
  int64_t lda, ldp;
  int B, D;
  int Bc;         // candidates: B, or G*B when positives were gathered across devices (tensor path only)
  int label_off;  // the positive of anchor i is candidate i + label_off
  float scale;
  // forward outputs / backward inputs
  float* lse;
  float* inv_a;
  float* inv_p;
  float* row_loss;        // [B] workspace
  unsigned int* counter;  // workspace, zeroed before the forward launch
  float* loss;
  // backward
  const float* grad_out;
  void* grad_a;
  void* grad_p;
  int64_t ldga, ldgp;
};

}  // namespace icr
