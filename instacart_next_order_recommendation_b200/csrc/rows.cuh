// Per-row sums of squares, one warp per row, shared by the preparation kernels (prep.cu) and the candidate-list top-k
// (subset_topk.cu): a row's inverse norm is the same bits wherever it is computed.
#pragma once

#include "common.cuh"

namespace icr {

__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  const uint4 v = ldg_stream(p);
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

// One row's sum of squares, on every lane of the calling warp; its inverse norm is 1 / max(sqrt(ss), eps). Lane l
// sums, with fmaf in element order, the elements of its vectors l, l + 32, ... and then the elements past the last whole
// vector; then warp_sum. STREAM: read through the non-coherent streaming path (rows that no kernel writes meanwhile);
// icr_update_rows reads back the row it has just written and needs coherent loads.
template <typename T, bool STREAM>
__device__ __forceinline__ float row_sumsq(const T* __restrict__ row, int nvec, int64_t dim, int lane) {
  constexpr int VEC = Elem<T>::VEC;
  float ss = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float f[VEC];
    if constexpr (STREAM)
      Elem<T>::unpack(ldg_stream(row + static_cast<int64_t>(v) * VEC), f);
    else
      Elem<T>::unpack(*reinterpret_cast<const uint4*>(row + static_cast<int64_t>(v) * VEC), f);
#pragma unroll
    for (int i = 0; i < VEC; ++i) ss = fmaf(f[i], f[i], ss);
  }
  for (int e = nvec * VEC + lane; e < dim; e += 32) {
    const float f = Elem<T>::to_f32(row[e]);
    ss = fmaf(f, f, ss);
  }
  return warp_sum(ss);
}

// The sum of squares of an fp32 row as the screening plane takes it (screen_row, prep.cu), on every lane: nvec = dim / 4
// float4s, each as fmaf(x, fmaf(y, fmaf(z, fmaf(w, ss)))), then warp_sum. The inverse norm of an fp32 query on the
// tensor-core path, and so of its exact re-scoring, is 1 / max(sqrt(ss), eps) of this sum. STREAM as for row_sumsq.
template <bool STREAM>
__device__ __forceinline__ float screen_sumsq(const float* __restrict__ row, int nvec, int lane) {
  float ss = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float4 f;
    if constexpr (STREAM)
      f = ldg_stream_f4(row + 4 * v);
    else
      f = *reinterpret_cast<const float4*>(row + 4 * v);
    ss = fmaf(f.x, f.x, fmaf(f.y, f.y, fmaf(f.z, f.z, fmaf(f.w, f.w, ss))));
  }
  return warp_sum(ss);
}

}  // namespace icr
