// K5: row inverse norms and the fp16 (hi|lo) operand planes of the fp32-parity tensor path.
#include "common.cuh"

namespace icr {

__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  const uint4 v = ldg_stream(p);
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

// one warp per row; 128-bit loads; inv = 1 / max(||x||, eps)   (torch F.normalize semantics)
// tau_init / ovf_init (optional, query side of a top-k call): the per-query threshold starts at -inf and the overflow flag at 0;
// written here so that the call needs no separate initialisation launch
template <typename T>
__global__ void __launch_bounds__(256) row_inv_norms_kernel(const T* __restrict__ x, int64_t rows, int64_t dim, int64_t ld,
                                                            float* __restrict__ inv, float* __restrict__ tau_init,
                                                            unsigned int* __restrict__ ovf_init) {
  constexpr int VEC = Elem<T>::VEC;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / VEC);
  for (int64_t r = warp; r < rows; r += nwarps) {
    const T* row = x + r * ld;
    float ss = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      float f[VEC];
      Elem<T>::unpack(ldg_stream(row + static_cast<int64_t>(v) * VEC), f);
#pragma unroll
      for (int i = 0; i < VEC; ++i) ss = fmaf(f[i], f[i], ss);
    }
    for (int e = nvec * VEC + lane; e < dim; e += 32) {
      const float f = Elem<T>::to_f32(row[e]);
      ss = fmaf(f, f, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) {
      inv[r] = 1.0f / fmaxf(sqrtf(ss), kNormEps);
      if (tau_init) tau_init[r] = -INFINITY;
      if (ovf_init) ovf_init[r] = 0u;
    }
    if (ovf_init && r == 0 && lane < 8) ovf_init[rows + lane] = 0u;  // the grid-barrier counters kept behind the flags
  }
}

// one warp per row: normalise (fp32), scale by 2^8, split into fp16 hi + fp16 lo.
// hi + lo carries ~22 significant bits of the normalised value; hi*hi + hi*lo + lo*hi on the
// tensor cores (fp32 accumulate) then reproduces the fp32 dot product to ~1e-6 relative.
__global__ void __launch_bounds__(256) split_f16_planes_kernel(const float* __restrict__ x, int64_t rows, int64_t dim, int64_t ld,
                                                               __half* __restrict__ planes, int64_t dim_pad) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t r = warp; r < rows; r += nwarps) {
    const float* row = x + r * ld;
    float ss = 0.f;
    for (int e = lane; e < dim; e += 32) {
      const float f = row[e];
      ss = fmaf(f, f, ss);
    }
    ss = warp_sum(ss);
    const float inv = 256.0f / fmaxf(sqrtf(ss), kNormEps);
    __half* hi = planes + r * (2 * dim_pad);
    __half* lo = hi + dim_pad;
    for (int e = lane; e < dim_pad; e += 32) {
      float v = (e < dim) ? row[e] * inv : 0.f;
      const __half h = __float2half_rn(v);
      const __half l = __float2half_rn(v - __half2float(h));
      hi[e] = h;
      lo[e] = l;
    }
  }
}

// One warp per row: the SCREENING operand of fp32 catalogs and queries. plane[r] = fp16(256 * x_r / max(|x_r|, eps)),
// zero-padded to dim_pad; inv[r] = 1 / max(|x_r|, eps) for the exact re-scoring of the few rows that pass the screen.
// A single fp16 plane carries 11 significant bits per element: the screened score differs from the exact cosine by
// at most 2^-10 (Cauchy-Schwarz over the two rounding-error vectors), which the caller turns into a safety band.
__global__ void __launch_bounds__(256) screen_plane_kernel(const float* __restrict__ x, int64_t rows, int64_t dim, int64_t ld,
                                                           __half* __restrict__ plane, int64_t dim_pad, float* __restrict__ inv_out,
                                                           float* __restrict__ tau_init, unsigned int* __restrict__ ovf_init) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / 4), nvec_pad = static_cast<int>(dim_pad / 4);
  for (int64_t r = warp; r < rows; r += nwarps) {
    const float* row = x + r * ld;
    float ss = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      const float4 f = ldg_stream_f4(row + 4 * v);
      ss = fmaf(f.x, f.x, fmaf(f.y, f.y, fmaf(f.z, f.z, fmaf(f.w, f.w, ss))));
    }
    ss = warp_sum(ss);
    const float inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
    if (lane == 0) {
      if (inv_out) inv_out[r] = inv;
      if (tau_init) tau_init[r] = -INFINITY;
      if (ovf_init) ovf_init[r] = 0u;
    }
    if (ovf_init && r == 0 && lane < 8) ovf_init[rows + lane] = 0u;  // the grid-barrier counters kept behind the flags
    const float sc = 256.0f * inv;
    __half* dst = plane + r * dim_pad;
    for (int v = lane; v < nvec_pad; v += 32) {
      float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
      if (v < nvec) f = *reinterpret_cast<const float4*>(row + 4 * v);  // second touch: L1/L2 hit
      const __half2 a = __floats2half2_rn(f.x * sc, f.y * sc), b = __floats2half2_rn(f.z * sc, f.w * sc);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&a);
      pk.y = *reinterpret_cast<const uint32_t*>(&b);
      *reinterpret_cast<uint2*>(dst + 4 * v) = pk;
    }
  }
}

int launch_screen_plane(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* plane, float* inv, cudaStream_t st, float* tau_init,
                        unsigned int* ovf_init) {
  if (rows == 0) return ICR_OK;
  const int64_t dim_pad = (dim + 63) / 64 * 64;
  const int64_t want = (rows + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  screen_plane_kernel<<<blocks, 256, 0, st>>>(x, rows, dim, ld, reinterpret_cast<__half*>(plane), dim_pad, inv, tau_init, ovf_init);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

int launch_row_inv_norms(const void* x, int64_t rows, int64_t dim, int64_t ld, int dtype, float* inv, cudaStream_t st, float* tau_init,
                         unsigned int* ovf_init) {
  if (rows == 0) return ICR_OK;
  const int threads = 256;
  const int64_t want = (rows + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  if (dtype == ICR_F32)
    row_inv_norms_kernel<float><<<blocks, threads, 0, st>>>(static_cast<const float*>(x), rows, dim, ld, inv, tau_init, ovf_init);
  else if (dtype == ICR_F16)
    row_inv_norms_kernel<__half><<<blocks, threads, 0, st>>>(static_cast<const __half*>(x), rows, dim, ld, inv, tau_init, ovf_init);
  else
    row_inv_norms_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>(static_cast<const __nv_bfloat16*>(x), rows, dim, ld, inv, tau_init, ovf_init);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

int launch_split_planes(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* planes, cudaStream_t st) {
  if (rows == 0) return ICR_OK;
  const int64_t dim_pad = (dim + 63) / 64 * 64;
  const int64_t want = (rows + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  split_f16_planes_kernel<<<blocks, 256, 0, st>>>(x, rows, dim, ld, reinterpret_cast<__half*>(planes), dim_pad);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

// two fp32 values -> one word of two 16-bit elements, round to nearest even (what torch's .to(bfloat16 / float16) does;
// fp16 overflows to +-inf and keeps subnormals)
template <typename OUT>
__device__ __forceinline__ uint32_t pack_rn(float lo, float hi);
template <>
__device__ __forceinline__ uint32_t pack_rn<__nv_bfloat16>(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
template <>
__device__ __forceinline__ uint32_t pack_rn<__half>(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// Catalog upload: fp32 rows as stored on disk -> the resident form (fp32, bf16 or fp16), optionally L2-normalised first.
// One warp per row, 128-bit loads.
template <typename OUT>
__global__ void __launch_bounds__(256) convert_rows_kernel(const float* __restrict__ x, int64_t rows, int64_t dim, int64_t ldx,
                                                           OUT* __restrict__ out, int64_t ldo, int normalize) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / 4);
  for (int64_t r = warp; r < rows; r += nwarps) {
    const float* row = x + r * ldx;
    float inv = 1.0f;
    if (normalize) {
      float ss = 0.f;
      for (int v = lane; v < nvec; v += 32) {
        const float4 f = *reinterpret_cast<const float4*>(row + 4 * v);
        ss = fmaf(f.x, f.x, fmaf(f.y, f.y, fmaf(f.z, f.z, fmaf(f.w, f.w, ss))));
      }
      ss = warp_sum(ss);
      inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
    }
    OUT* dst = out + r * ldo;
    for (int v = lane; v < nvec; v += 32) {
      float4 f = ldg_stream_f4(row + 4 * v);
      if (normalize) {
        f.x *= inv;
        f.y *= inv;
        f.z *= inv;
        f.w *= inv;
      }
      if constexpr (sizeof(OUT) == 4) {
        *reinterpret_cast<float4*>(dst + 4 * v) = f;
      } else {
        uint2 pk;
        pk.x = pack_rn<OUT>(f.x, f.y);
        pk.y = pack_rn<OUT>(f.z, f.w);
        *reinterpret_cast<uint2*>(dst + 4 * v) = pk;
      }
    }
  }
}

int launch_convert_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx, void* out, int64_t ldo, int out_dtype, int normalize,
                        cudaStream_t st) {
  if (rows == 0) return ICR_OK;
  const int64_t want = (rows + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  if (out_dtype == ICR_F32)
    convert_rows_kernel<float><<<blocks, 256, 0, st>>>(x, rows, dim, ldx, static_cast<float*>(out), ldo, normalize);
  else if (out_dtype == ICR_F16)
    convert_rows_kernel<__half><<<blocks, 256, 0, st>>>(x, rows, dim, ldx, static_cast<__half*>(out), ldo, normalize);
  else
    convert_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(x, rows, dim, ldx, static_cast<__nv_bfloat16*>(out), ldo, normalize);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

// ---- per-query exclusion bitmap (icr_query_exclusion_bits) ------------------------------------------------
// One warp per query scatters its CSR list into bits[row / 32][q]; rows outside [0, N) are ignored, duplicates are harmless.
__global__ void __launch_bounds__(256) query_exclusion_bits_kernel(const int64_t* __restrict__ offsets, const int64_t* __restrict__ rows,
                                                                   int64_t Q, int64_t N, uint32_t* __restrict__ bits) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  for (int64_t q = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); q < Q; q += nwarps) {
    const int64_t b = offsets[q], e = offsets[q + 1];
    for (int64_t i = b + lane; i < e; i += 32) {
      const int64_t r = rows[i];
      if (r >= 0 && r < N) atomicOr(bits + (r >> 5) * Q + q, 1u << (r & 31));
    }
  }
}

int launch_query_exclusion_bits(const int64_t* offsets, const int64_t* rows, int64_t Q, int64_t N, uint32_t* bits, cudaStream_t st) {
  ICR_CUDA_CHECK(cudaMemsetAsync(bits, 0, static_cast<size_t>((N + 31) / 32) * static_cast<size_t>(Q) * sizeof(uint32_t), st));
  const int64_t blocks = (Q + 7) / 8;
  query_exclusion_bits_kernel<<<static_cast<unsigned>(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, st>>>(offsets, rows, Q, N, bits);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

}  // namespace icr
