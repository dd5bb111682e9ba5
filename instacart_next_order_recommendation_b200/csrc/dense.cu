// K2' (CUDA-core form): dense cosine similarity out[i][j] = <a_i, b_j> / (|a_i| |b_j|), fp32 accumulate.
// Serves the hook-compatible callers that really want the [Q, N] matrix
// (sentence_transformers.util.cos_sim as MNRL `similarity_fct` / evaluator `score_functions`).
#include "common.cuh"

namespace icr {

constexpr int kDT = 64;   // output tile edge
constexpr int kDK = 16;   // K slab

template <typename T>
__global__ void __launch_bounds__(256) cos_sim_dense_kernel(const T* __restrict__ a, int64_t Qa, int64_t lda,
                                                            const T* __restrict__ b, int64_t Nb, int64_t ldb, int D,
                                                            const float* __restrict__ inva, const float* __restrict__ invb,
                                                            float* __restrict__ out, int64_t ldo) {
  __shared__ float As[kDK][kDT + 4];
  __shared__ float Bs[kDK][kDT + 4];
  const int tid = threadIdx.x;
  const int64_t i0 = static_cast<int64_t>(blockIdx.y) * kDT, j0 = static_cast<int64_t>(blockIdx.x) * kDT;
  const int lr = tid >> 2, lk = (tid & 3) * 4;  // this thread stages row lr, k-offsets lk..lk+3
  const int ty = tid >> 4, tx = tid & 15;       // 16x16 threads, 4x4 outputs each
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < D; k0 += kDK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k0 + lk + e;
      const int64_t ra = i0 + lr, rb = j0 + lr;
      As[lk + e][lr] = (ra < Qa && k < D) ? Elem<T>::to_f32(a[ra * lda + k]) : 0.f;
      Bs[lk + e][lr] = (rb < Nb && k < D) ? Elem<T>::to_f32(b[rb * ldb + k]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kDK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w};
      const float br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = i0 + ty * 4 + i;
    if (r >= Qa) continue;
    const float ia = inva[r];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t c = j0 + tx * 4 + j;
      if (c < Nb) out[r * ldo + c] = acc[i][j] * ia * invb[c];
    }
  }
}

int launch_cos_sim_dense(const void* a, int64_t Qa, int64_t lda, const void* b, int64_t Nb, int64_t ldb, int D, int dtype,
                         const float* inva, const float* invb, float* out, int64_t ldo, cudaStream_t st) {
  if (Qa == 0 || Nb == 0) return ICR_OK;
  dim3 grid(static_cast<unsigned>((Nb + kDT - 1) / kDT), static_cast<unsigned>((Qa + kDT - 1) / kDT));
  if (dtype == ICR_F32)
    cos_sim_dense_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(a), Qa, lda, static_cast<const float*>(b), Nb, ldb, D, inva, invb, out, ldo);
  else if (dtype == ICR_F16)
    cos_sim_dense_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(a), Qa, lda, static_cast<const __half*>(b), Nb, ldb, D, inva, invb, out, ldo);
  else
    cos_sim_dense_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(a), Qa, lda, static_cast<const __nv_bfloat16*>(b), Nb, ldb, D, inva, invb, out, ldo);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

}  // namespace icr
