// K3: MultipleNegativesRankingLoss forward / backward, one kernel each.
//
//   loss = mean_i [ logsumexp_j( s * <a^_i, p^_j> ) - s * <a^_i, p^_i> ],  x^ = x / max(|x|, eps)
//
// Forward : normalise + in-batch similarity + scale + online log-sum-exp + cross-entropy + mean,
//           fused; the [B,B] score matrix is never materialised.
// Backward: recomputes the scores tile by tile (cheaper than storing them), forms
//           G = (softmax - I) * s * dL/dloss / B, the two products G P^ and G^T A^, and the
//           normalisation Jacobian (I - x^ x^T)/|x| in the same kernel.
// All arithmetic is fp32 whatever the storage dtype (the reference trains under fp16 autocast,
// src/training/train_sbert.py:232; a native-bf16 loss is 1.5e-2 off, SURVEY §8c).
//
// Replaces sentence_transformers.losses.MultipleNegativesRankingLoss.forward + autograd
// (constructed at reference src/training/train_sbert.py:182-185).
#include "common.cuh"

namespace icr {

constexpr int kMnrlThreads = 256;
constexpr int kMnrlWarps = kMnrlThreads / 32;

// Four elements per lane and load for EVERY storage type (16-byte loads of fp32, 8-byte loads of bf16 / fp16): with eight
// 16-bit elements per load a 384-wide row is 48 vectors, i.e. a second chunk with half the lanes idle and 16 instead of 12
// accumulators per row pair - the 16-bit kernels ran 1.6x slower than the fp32 ones on the same batch (profiles/r02_notes.md).
template <typename T>
struct MVec {
  static constexpr int VEC = 4;
  __device__ static __forceinline__ void load(const T* p, float* f) {
    if constexpr (sizeof(T) == 4) {
      Elem<float>::unpack(ldg_stream(p), f);
    } else {
      uint2 w;
      asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(w.x), "=r"(w.y) : "l"(p));
      const T* h = reinterpret_cast<const T*>(&w);
#pragma unroll
      for (int i = 0; i < 4; ++i) f[i] = Elem<T>::to_f32(h[i]);
    }
  }
};

template <typename T, int NCV>
struct MnrlCfg {
  static constexpr int VEC = MVec<T>::VEC;
  static constexpr int EPL = NCV * VEC;                              // elements per lane of one row
  static constexpr int TM = EPL <= 12 ? 8 : (EPL <= 24 ? 4 : 2);     // tile rows per CTA
};


// load this lane's slice of a row as fp32: vector c of the slice is vector (c*32 + lane) of the row
template <typename T, int NCV>
__device__ __forceinline__ void load_slice(const T* row, int nvec, int lane, float (&y)[NCV * MVec<T>::VEC]) {
  constexpr int VEC = MVec<T>::VEC;
#pragma unroll
  for (int c = 0; c < NCV; ++c) {
    const int v = c * 32 + lane;
    if (v < nvec) {
      MVec<T>::load(row + static_cast<int64_t>(v) * VEC, &y[c * VEC]);
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) y[c * VEC + i] = 0.f;
    }
  }
}

// MODE 0: forward (tile = anchors, stream = positives)
// MODE 1: backward; blockIdx.x < tiles -> tile = anchors (writes grad_a), else tile = positives (grad_p)
// TMV: tile rows per CTA (0 = the default of MnrlCfg). Small batches take TMV = 2: at B = 256 the default tiles (4-8 rows)
// make only 32-64 CTAs and each walks all B stream rows serially - a latency-bound 40 us per kernel for 50 MFLOP.
template <typename T, int NCV, int MODE, int TMV = 0>
__global__ void __launch_bounds__(kMnrlThreads) mnrl_kernel(MnrlArgs g) {
  using C = MnrlCfg<T, NCV>;
  constexpr int VEC = C::VEC, EPL = C::EPL, TM = TMV ? TMV : C::TM;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int D = g.D, B = g.B;
  const int nvec = D / VEC;
  const int dpad = NCV * 32 * VEC;  // padded row length in shared memory
  float* xt = reinterpret_cast<float*>(smem_raw);        // [TM][dpad] normalised tile rows
  float* red = xt + TM * dpad;                           // bwd: [TM][dpad] reduced gradient; fwd: scratch
  float* xinv = red + TM * dpad;                         // [TM]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tiles = (B + TM - 1) / TM;
  const bool tile_is_anchor = (MODE == 0) || (static_cast<int>(blockIdx.x) < tiles);
  const int tile = tile_is_anchor ? blockIdx.x : blockIdx.x - tiles;
  const int row0 = tile * TM;
  const T* X = static_cast<const T*>(tile_is_anchor ? g.a : g.p);
  const T* Y = static_cast<const T*>(tile_is_anchor ? g.p : g.a);
  const int64_t ldx = tile_is_anchor ? g.lda : g.ldp;
  const int64_t ldy = tile_is_anchor ? g.ldp : g.lda;

  // ---- stage normalised tile rows -----------------------------------------------------------
  for (int r = warp; r < TM; r += kMnrlWarps) {
    float x[EPL];
    const bool live = row0 + r < B;
    if (live) load_slice<T, NCV>(X + static_cast<int64_t>(row0 + r) * ldx, nvec, lane, x);
    else {
#pragma unroll
      for (int i = 0; i < EPL; ++i) x[i] = 0.f;
    }
    float inv;
    if (MODE == 0) {
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < EPL; ++i) ss = fmaf(x[i], x[i], ss);
      ss = warp_sum(ss);
      inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
      if (live && lane == 0) g.inv_a[row0 + r] = inv;
    } else {
      inv = live ? (tile_is_anchor ? g.inv_a[row0 + r] : g.inv_p[row0 + r]) : 0.f;
    }
    if (lane == 0) xinv[r] = inv;
#pragma unroll
    for (int c = 0; c < NCV; ++c)
#pragma unroll
      for (int i = 0; i < VEC; ++i) xt[r * dpad + (c * 32 + lane) * VEC + i] = x[c * VEC + i] * inv;
  }
  for (int i = tid; i < TM * dpad; i += kMnrlThreads) red[i] = 0.f;
  __syncthreads();

  // ---- stream the other matrix ----------------------------------------------------------------
  float m[TM], l[TM], diag[TM];       // forward: online log-sum-exp state (replicated in all lanes)
  float acc[MODE == 1 ? TM : 1][EPL]; // backward: this warp's partial gradient w.r.t. normalised rows
#pragma unroll
  for (int r = 0; r < TM; ++r) {
    m[r] = -INFINITY;
    l[r] = 0.f;
    diag[r] = 0.f;
  }
  if (MODE == 1) {
#pragma unroll
    for (int r = 0; r < TM; ++r)
#pragma unroll
      for (int i = 0; i < EPL; ++i) acc[r][i] = 0.f;
  }
  const float coef = (MODE == 1) ? (g.grad_out ? g.grad_out[0] : 1.0f) * g.scale / static_cast<float>(B) : 0.f;  // null: dL/dloss = 1
  float tile_lse[TM];
  if (MODE == 1) {
#pragma unroll
    for (int r = 0; r < TM; ++r) tile_lse[r] = (tile_is_anchor && row0 + r < B) ? g.lse[row0 + r] : 0.f;
  }

  // JB stream rows per iteration: their loads, dot products and warp reductions are independent chains, so one
  // warp keeps several L2 round trips and shuffle trees in flight instead of paying each latency in turn
  constexpr int JB = EPL <= 16 ? 4 : 2;
  for (int j0 = warp * JB; j0 < B; j0 += kMnrlWarps * JB) {
    float y[JB][EPL];
    float yinv[JB], stream_lse[JB];
#pragma unroll
    for (int b = 0; b < JB; ++b) {
      const int j = j0 + b;
      if (j < B) {
        load_slice<T, NCV>(Y + static_cast<int64_t>(j) * ldy, nvec, lane, y[b]);
      } else {
#pragma unroll
        for (int i = 0; i < EPL; ++i) y[b][i] = 0.f;
      }
      yinv[b] = 0.f;
      stream_lse[b] = 0.f;
      if (MODE == 1 && j < B) {
        yinv[b] = tile_is_anchor ? g.inv_p[j] : g.inv_a[j];
        stream_lse[b] = tile_is_anchor ? 0.f : g.lse[j];
      }
    }
    if (MODE == 0) {
      float ss[JB];
#pragma unroll
      for (int b = 0; b < JB; ++b) {
        ss[b] = 0.f;
#pragma unroll
        for (int i = 0; i < EPL; ++i) ss[b] = fmaf(y[b][i], y[b][i], ss[b]);
      }
#pragma unroll
      for (int b = 0; b < JB; ++b) ss[b] = warp_sum(ss[b]);
#pragma unroll
      for (int b = 0; b < JB; ++b) {
        yinv[b] = 1.0f / fmaxf(sqrtf(ss[b]), kNormEps);
        if (blockIdx.x == 0 && lane == 0 && j0 + b < B) g.inv_p[j0 + b] = yinv[b];
      }
    }
    float dot[JB][TM];
#pragma unroll
    for (int b = 0; b < JB; ++b)
#pragma unroll
      for (int r = 0; r < TM; ++r) dot[b][r] = 0.f;
#pragma unroll
    for (int c = 0; c < NCV; ++c) {
#pragma unroll
      for (int h = 0; h < VEC / 4; ++h) {
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          const float4 xv = *reinterpret_cast<const float4*>(xt + r * dpad + (c * 32 + lane) * VEC + h * 4);
#pragma unroll
          for (int b = 0; b < JB; ++b) {
            dot[b][r] = fmaf(xv.x, y[b][c * VEC + h * 4 + 0], dot[b][r]);
            dot[b][r] = fmaf(xv.y, y[b][c * VEC + h * 4 + 1], dot[b][r]);
            dot[b][r] = fmaf(xv.z, y[b][c * VEC + h * 4 + 2], dot[b][r]);
            dot[b][r] = fmaf(xv.w, y[b][c * VEC + h * 4 + 3], dot[b][r]);
          }
        }
      }
    }
#pragma unroll
    for (int b = 0; b < JB; ++b)
#pragma unroll
      for (int r = 0; r < TM; ++r) dot[b][r] = warp_sum(dot[b][r]);

#pragma unroll
    for (int b = 0; b < JB; ++b) {
      const int j = j0 + b;
      if (j >= B) continue;
      if (MODE == 0) {
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          const float s = g.scale * dot[b][r] * yinv[b];
          const float mn = fmaxf(m[r], s);
          l[r] = l[r] * __expf(m[r] - mn) + __expf(s - mn);
          m[r] = mn;
          if (j == row0 + r) diag[r] = s;
        }
      } else {
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          const float s = g.scale * dot[b][r] * yinv[b];
          const float lse = tile_is_anchor ? tile_lse[r] : stream_lse[b];
          float w = __expf(s - lse) - ((j == row0 + r) ? 1.f : 0.f);
          w *= coef * yinv[b];  // d/d(x^_r) += w * y_j  (y^_j = y_j * yinv)
#pragma unroll
          for (int i = 0; i < EPL; ++i) acc[r][i] = fmaf(w, y[b][i], acc[r][i]);
        }
      }
    }
  }

  if (MODE == 0) {
    // ---- combine the warps' (m, l, diag) and finish the rows ------------------------------------
    float* sm = red;                          // [warps][TM]
    float* sl = red + kMnrlWarps * TM;
    float* sd = sl + kMnrlWarps * TM;
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < TM; ++r) {
        sm[warp * TM + r] = m[r];
        sl[warp * TM + r] = l[r];
        sd[warp * TM + r] = diag[r];
      }
    }
    __syncthreads();
    if (tid < TM && row0 + tid < B) {
      float mm = -INFINITY, dd = 0.f;
      for (int w = 0; w < kMnrlWarps; ++w) {
        mm = fmaxf(mm, sm[w * TM + tid]);
        dd += sd[w * TM + tid];
      }
      float ll = 0.f;
      for (int w = 0; w < kMnrlWarps; ++w) ll += sl[w * TM + tid] * __expf(sm[w * TM + tid] - mm);
      const float lse = mm + logf(ll);
      g.lse[row0 + tid] = lse;
      g.row_loss[row0 + tid] = lse - dd;
    }
    // ---- deterministic mean by the last CTA to finish -------------------------------------------
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(g.counter, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last && warp == 0) {
      __threadfence();
      float s = 0.f;
      for (int i = lane; i < B; i += 32) s += __ldcg(g.row_loss + i);
      s = warp_sum(s);
      if (lane == 0) {
        g.loss[0] = s / static_cast<float>(B);
        *g.counter = 0u;
      }
    }
  } else {
    // ---- reduce the warps' partial gradients in a fixed order (deterministic) -------------------
    for (int w = 0; w < kMnrlWarps; ++w) {
      if (warp == w) {
#pragma unroll
        for (int r = 0; r < TM; ++r)
#pragma unroll
          for (int c = 0; c < NCV; ++c)
#pragma unroll
            for (int i = 0; i < VEC; ++i) red[r * dpad + (c * 32 + lane) * VEC + i] += acc[r][c * VEC + i];
      }
      __syncthreads();
    }
    // ---- normalisation Jacobian: dx = (dx^ - x^ <x^, dx^>) / |x| -------------------------------
    T* G = static_cast<T*>(tile_is_anchor ? g.grad_a : g.grad_p);
    const int64_t ldg = tile_is_anchor ? g.ldga : g.ldgp;
    for (int r = warp; r < TM; r += kMnrlWarps) {
      if (row0 + r >= B) continue;
      float pr = 0.f;
      for (int e = lane; e < D; e += 32) pr = fmaf(xt[r * dpad + e], red[r * dpad + e], pr);
      pr = warp_sum(pr);
      const float inv = xinv[r];
      for (int e = lane; e < D; e += 32)
        G[static_cast<int64_t>(row0 + r) * ldg + e] = Elem<T>::from_f32((red[r * dpad + e] - xt[r * dpad + e] * pr) * inv);
    }
  }
}

template <typename T, int NCV, int TMV>
static int launch_mnrl_tm(const MnrlArgs& g, bool bwd, cudaStream_t st) {
  using C = MnrlCfg<T, NCV>;
  constexpr int TM = TMV ? TMV : C::TM;
  const int dpad = NCV * 32 * C::VEC;
  const size_t smem = (2 * TM * dpad + TM + 8 + 3 * kMnrlWarps * TM) * sizeof(float);
  const int tiles = (g.B + TM - 1) / TM;
  if (!bwd) {
    if (smem > 48 * 1024) ICR_CUDA_CHECK(cudaFuncSetAttribute(mnrl_kernel<T, NCV, 0, TMV>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    mnrl_kernel<T, NCV, 0, TMV><<<tiles, kMnrlThreads, smem, st>>>(g);
  } else {
    if (smem > 48 * 1024) ICR_CUDA_CHECK(cudaFuncSetAttribute(mnrl_kernel<T, NCV, 1, TMV>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    mnrl_kernel<T, NCV, 1, TMV><<<2 * tiles, kMnrlThreads, smem, st>>>(g);
  }
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

template <typename T, int NCV>
static int launch_mnrl(const MnrlArgs& g, bool bwd, cudaStream_t st) {
  using C = MnrlCfg<T, NCV>;
  // fewer CTAs than SMs with the default tile: spread the batch over 2-row tiles
  if (C::TM > 2 && (g.B + C::TM - 1) / C::TM < 148) return launch_mnrl_tm<T, NCV, 2>(g, bwd, st);
  return launch_mnrl_tm<T, NCV, 0>(g, bwd, st);
}

// out[i] = x[i] * s[0] for two equally sized buffers at once (the two gradients of a step scaled by the incoming dL/dloss)
template <typename T>
__global__ void __launch_bounds__(256) scale2_kernel(const T* __restrict__ x0, const T* __restrict__ x1, int64_t n, const float* __restrict__ s,
                                                     T* __restrict__ o0, T* __restrict__ o1) {
  const float f = s[0];
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    o0[i] = Elem<T>::from_f32(Elem<T>::to_f32(x0[i]) * f);
    o1[i] = Elem<T>::from_f32(Elem<T>::to_f32(x1[i]) * f);
  }
}

int launch_scale2(const void* x0, const void* x1, int64_t n, int dtype, const float* s, void* o0, void* o1, cudaStream_t st) {
  if (n == 0) return ICR_OK;
  const int64_t want = (n + 255) / 256;
  const int blocks = static_cast<int>(want < 148 * 8 ? want : 148 * 8);
  if (dtype == ICR_F32)
    scale2_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(x0), static_cast<const float*>(x1), n, s, static_cast<float*>(o0),
                                                 static_cast<float*>(o1));
  else if (dtype == ICR_F16)
    scale2_kernel<__half><<<blocks, 256, 0, st>>>(static_cast<const __half*>(x0), static_cast<const __half*>(x1), n, s, static_cast<__half*>(o0),
                                                  static_cast<__half*>(o1));
  else
    scale2_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x0), static_cast<const __nv_bfloat16*>(x1), n, s,
                                                         static_cast<__nv_bfloat16*>(o0), static_cast<__nv_bfloat16*>(o1));
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

int launch_mnrl_dispatch(const MnrlArgs& g, int dtype, bool bwd, cudaStream_t st) {
  const int vec = 4;
  const int nvec = g.D / vec;
  const int ncv = (nvec + 31) / 32;
#define ICR_MNRL_CASE(T, N) \
  if (ncv <= N) return launch_mnrl<T, N>(g, bwd, st)
  if (dtype == ICR_F32) {
    ICR_MNRL_CASE(float, 1);
    ICR_MNRL_CASE(float, 2);
    ICR_MNRL_CASE(float, 3);
    ICR_MNRL_CASE(float, 6);
  } else if (dtype == ICR_F16) {
    ICR_MNRL_CASE(__half, 1);
    ICR_MNRL_CASE(__half, 2);
    ICR_MNRL_CASE(__half, 3);
    ICR_MNRL_CASE(__half, 6);
  } else {
    ICR_MNRL_CASE(__nv_bfloat16, 1);
    ICR_MNRL_CASE(__nv_bfloat16, 2);
    ICR_MNRL_CASE(__nv_bfloat16, 3);
    ICR_MNRL_CASE(__nv_bfloat16, 6);
  }
#undef ICR_MNRL_CASE
  set_error("mnrl: embedding dim %d too large (max 768 on the CUDA-core path)", g.D);
  return ICR_ERR_ARG;
}

}  // namespace icr
