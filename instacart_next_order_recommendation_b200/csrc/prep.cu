// K5: row inverse norms and the fp16 (hi|lo) operand planes of the fp32-parity tensor path.
#include "common.cuh"
#include "rows.cuh"

namespace icr {

// one warp per row; 128-bit loads; inv = 1 / max(||x||, eps)   (torch F.normalize semantics)
// tau_init / ovf_init (optional, query side of a top-k call): the per-query threshold starts at -inf and the overflow flag at 0;
// written here so that the call needs no separate initialisation launch
template <typename T>
__global__ void __launch_bounds__(256) row_inv_norms_kernel(const T* __restrict__ x, int64_t rows, int64_t dim, int64_t ld,
                                                            float* __restrict__ inv, float* __restrict__ tau_init,
                                                            unsigned int* __restrict__ ovf_init) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / Elem<T>::VEC);
  for (int64_t r = warp; r < rows; r += nwarps) {
    const float ss = row_sumsq<T, true>(x + r * ld, nvec, dim, lane);
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

// One row of the SCREENING operand of fp32 catalogs and queries, by the calling warp: dst = fp16(256 * x / max(|x|, eps)),
// zero-padded to nvec_pad float4s (nvec = dim / 4, dim % 4 == 0), at plane + off; hands inv = 1 / max(|x|, eps) to on_inv (every
// lane) before it writes the plane row. The sum of squares takes a float4 as
// fmaf(x, fmaf(y, fmaf(z, fmaf(w, ss)))): it can differ from row_sumsq<float>'s norm in the last bit, so a catalog keeps the
// inverse norms of whichever of the two built it. STREAM as for row_sumsq.
// A single fp16 plane carries 11 significant bits per element: the screened score differs from the exact cosine by
// at most 2^-10 (Cauchy-Schwarz over the two rounding-error vectors), which the caller turns into a safety band.
template <bool STREAM, typename OnInv>
__device__ __forceinline__ void screen_row(const float* __restrict__ row, int nvec, int nvec_pad, __half* __restrict__ plane, int64_t off,
                                           int lane, OnInv on_inv) {
  const float ss = screen_sumsq<STREAM>(row, nvec, lane);
  const float inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
  on_inv(inv);
  const float sc = 256.0f * inv;
  __half* dst = plane + off;
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

// One warp per row: plane[r] = screen_row(x_r), zero-padded to dim_pad; inv[r] = 1 / max(|x_r|, eps) for the exact
// re-scoring of the few rows that pass the screen.
__global__ void __launch_bounds__(256) screen_plane_kernel(const float* __restrict__ x, int64_t rows, int64_t dim, int64_t ld,
                                                           __half* __restrict__ plane, int64_t dim_pad, float* __restrict__ inv_out,
                                                           float* __restrict__ tau_init, unsigned int* __restrict__ ovf_init) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / 4), nvec_pad = static_cast<int>(dim_pad / 4);
  for (int64_t r = warp; r < rows; r += nwarps) {
    screen_row<true>(x + r * ld, nvec, nvec_pad, plane, r * dim_pad, lane, [&](float inv) {
      if (lane == 0) {
        if (inv_out) inv_out[r] = inv;
        if (tau_init) tau_init[r] = -INFINITY;
        if (ovf_init) ovf_init[r] = 0u;
      }
      if (ovf_init && r == 0 && lane < 8) ovf_init[rows + lane] = 0u;  // the grid-barrier counters kept behind the flags
    });
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

// One row in the resident form (fp32, bf16 or fp16), optionally L2-normalised first, by the calling warp; dim % 4 == 0.
template <typename OUT>
__device__ __forceinline__ void convert_row(const float* row, int nvec, OUT* out, int64_t r, int64_t ldo, int normalize, int lane) {
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

// Catalog upload: fp32 rows as stored on disk -> the resident form (fp32, bf16 or fp16), optionally L2-normalised first.
// One warp per row, 128-bit loads.
template <typename OUT>
__global__ void __launch_bounds__(256) convert_rows_kernel(const float* __restrict__ x, int64_t rows, int64_t dim, int64_t ldx,
                                                           OUT* __restrict__ out, int64_t ldo, int normalize) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec = static_cast<int>(dim / 4);
  for (int64_t r = warp; r < rows; r += nwarps) convert_row<OUT>(x + r * ldx, nvec, out, r, ldo, normalize, lane);
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

// ---- int8 rows (icr_quantize_rows): one warp per row, the format of I8Rows -------------------------------------
__global__ void __launch_bounds__(256) quantize_rows_kernel(const float* __restrict__ x, int64_t rows, int dim, int64_t ldx,
                                                            int8_t* __restrict__ codes, int64_t ldc, float* __restrict__ factors,
                                                            float* __restrict__ tau_init, unsigned int* __restrict__ ovf_init) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nwords = static_cast<int>(ldc / 4);  // the padding up to the row stride is written as zero codes
  for (int64_t r = warp; r < rows; r += nwarps) {
    uint32_t* dst = reinterpret_cast<uint32_t*>(codes + r * ldc);
    const float f = I8Rows::quantize(x + r * ldx, dim, nwords, lane, [dst](int w, uint32_t word) { dst[w] = word; });
    if (lane == 0) {
      factors[r] = f;
      if (tau_init) tau_init[r] = -INFINITY;  // query side of a tensor-core top-k call, as row_inv_norms_kernel
      if (ovf_init) ovf_init[r] = 0u;
    }
    if (ovf_init && r == 0 && lane < 8) ovf_init[rows + lane] = 0u;  // the grid-barrier counters kept behind the flags
  }
}

int launch_quantize_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx, int8_t* codes, int64_t ldc, float* factors, cudaStream_t st,
                         float* tau_init, unsigned int* ovf_init) {
  if (rows == 0) return ICR_OK;
  const int64_t want = (rows + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  quantize_rows_kernel<<<blocks, 256, 0, st>>>(x, rows, static_cast<int>(dim), ldx, codes, ldc, factors, tau_init, ovf_init);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

// ---- in-place catalog updates (icr_update_rows) ------------------------------------------------------------
// One warp per source row i: catalog row dst_rows[i] (ignored outside [0, N)) receives x_i in the resident form and its
// derived data, through the same warp-level helpers as the bulk kernels, so each row is bit for bit what the bulk kernels
// write for it: convert_row, then screen_row (fp32 with a plane) or row_sumsq (otherwise) over the row just written
// (coherent loads after __syncwarp, which orders the warp's stores before its loads).
template <typename OUT>
__global__ void __launch_bounds__(256) update_rows_kernel(const float* __restrict__ x, int64_t M, int64_t dim, int64_t ldx,
                                                          const int64_t* __restrict__ dst_rows, int64_t N, OUT* rows, int64_t ld_rows,
                                                          __half* plane, int64_t dim_pad, float* __restrict__ inv_norms, int normalize) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nvec4 = static_cast<int>(dim / 4), nvec = static_cast<int>(dim / Elem<OUT>::VEC), nvec_pad = static_cast<int>(dim_pad / 4);
  for (int64_t i = warp; i < M; i += nwarps) {
    const int64_t r = dst_rows[i];
    if (r < 0 || r >= N) continue;  // warp-uniform
    convert_row<OUT>(x + i * ldx, nvec4, rows, r, ld_rows, normalize, lane);
    __syncwarp();
    const OUT* dst = rows + r * ld_rows;
    if constexpr (sizeof(OUT) == 4) {
      if (plane) {
        screen_row<false>(dst, nvec4, nvec_pad, plane, r * dim_pad, lane, [&](float inv) {
          if (lane == 0) inv_norms[r] = inv;
        });
        continue;
      }
    }
    const float ss = row_sumsq<OUT, false>(dst, nvec, dim, lane);
    if (lane == 0) inv_norms[r] = 1.0f / fmaxf(sqrtf(ss), kNormEps);
  }
}

__global__ void __launch_bounds__(256) update_rows_i8_kernel(const float* __restrict__ x, int64_t M, int dim, int64_t ldx,
                                                             const int64_t* __restrict__ dst_rows, int64_t N, int8_t* __restrict__ codes,
                                                             int64_t ldc, float* __restrict__ factors) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nwords = static_cast<int>(ldc / 4);
  for (int64_t i = warp; i < M; i += nwarps) {
    const int64_t r = dst_rows[i];
    if (r < 0 || r >= N) continue;
    uint32_t* dst = reinterpret_cast<uint32_t*>(codes + r * ldc);
    const float f = I8Rows::quantize(x + i * ldx, dim, nwords, lane, [dst](int w, uint32_t word) { dst[w] = word; });
    if (lane == 0) factors[r] = f;
  }
}

int launch_update_rows(const float* x, int64_t M, int64_t dim, int64_t ldx, const int64_t* dst_rows, int64_t N, int dtype, void* rows,
                       int64_t ld_rows, uint16_t* plane, float* inv_norms, int normalize, cudaStream_t st) {
  if (M == 0) return ICR_OK;
  const int64_t want = (M + 7) / 8;
  const int blocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  const int64_t dim_pad = (dim + 63) / 64 * 64;
  __half* pl = reinterpret_cast<__half*>(plane);
  if (dtype == ICR_I8)
    update_rows_i8_kernel<<<blocks, 256, 0, st>>>(x, M, static_cast<int>(dim), ldx, dst_rows, N, static_cast<int8_t*>(rows), ld_rows, inv_norms);
  else if (dtype == ICR_F32)
    update_rows_kernel<float><<<blocks, 256, 0, st>>>(x, M, dim, ldx, dst_rows, N, static_cast<float*>(rows), ld_rows, pl, dim_pad, inv_norms,
                                                      normalize);
  else if (dtype == ICR_F16)
    update_rows_kernel<__half><<<blocks, 256, 0, st>>>(x, M, dim, ldx, dst_rows, N, static_cast<__half*>(rows), ld_rows, nullptr, 0, inv_norms,
                                                       normalize);
  else
    update_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(x, M, dim, ldx, dst_rows, N, static_cast<__nv_bfloat16*>(rows), ld_rows,
                                                              nullptr, 0, inv_norms, normalize);
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
