// Finishing steps of a query's selection, shared by the select kernels (select_hist.cu) and the tail of the single-launch
// swapped GEMM kernel (gemm_topk.cu): exact fp32 re-scoring of screened candidates, the whole-catalog ranking of a query
// whose screening band overflowed, and the ordered emit of the k best keys. All of them work on one warp's (sc, rw) arrays
// in shared memory (select_lean.cuh).
#pragma once

#include "common.cuh"
#include "select_args.cuh"
#include "select_warp.cuh"
#include "select_lean.cuh"

namespace icr {

__device__ __forceinline__ uint64_t canonical_from_raw(uint64_t raw) {
  const float f = __uint_as_float(static_cast<uint32_t>(raw >> 32));
  return (static_cast<uint64_t>(order_bits(f)) << 32) | (raw & 0xFFFFFFFFull);
}


// ---- exact re-scoring of screened candidates (fp32 catalogs) -------------------------------------------------------
// cos(q, row) = <q, c_row> * qinv * cinv[row] in fp32 FMAs on the rows as the caller stores them: the arithmetic of the
// GEMV path (K1), so both paths return the same scores. RB rows are scored at once: RB * NV independent 16-byte loads
// per lane are in flight before the first FMA (the candidates' rows are scattered over the L2-resident catalog).
template <int NV, int RB>
__device__ __forceinline__ void score_rows_fixed(const float* __restrict__ qrow, const float* const (&rows)[RB], float (&acc)[RB], int lane) {
  float4 qv[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) qv[v] = __ldg(reinterpret_cast<const float4*>(qrow) + v * 32 + lane);
  float4 c[RB][NV];
#pragma unroll
  for (int u = 0; u < RB; ++u)
#pragma unroll
    for (int v = 0; v < NV; ++v) {  // a candidate's row is read once per query: do not allocate it in L1
      const uint4 w = ldg_stream(reinterpret_cast<const float4*>(rows[u]) + v * 32 + lane);
      c[u][v] = make_float4(__uint_as_float(w.x), __uint_as_float(w.y), __uint_as_float(w.z), __uint_as_float(w.w));
    }
#pragma unroll
  for (int u = 0; u < RB; ++u) {
    float s = 0.f;
#pragma unroll
    for (int v = 0; v < NV; ++v) s = fmaf(qv[v].x, c[u][v].x, fmaf(qv[v].y, c[u][v].y, fmaf(qv[v].z, c[u][v].z, fmaf(qv[v].w, c[u][v].w, s))));
    acc[u] = s;
  }
}

// partial dot products of 8 rows with the query (any D % 4 == 0); lane sums are combined by the caller.
// 12 independent 16-byte loads per lane in flight (4 rows x 3 vectors at D = 384, 2 x 6 at D = 768): with 16 resident warps
// per SM that is ~100 KB outstanding, enough to cover the L2 latency, and the kernel stays within 128 registers.
template <bool WIDE = false>
__device__ __forceinline__ void score_rows8(const float* __restrict__ qrow, const float* const (&rows)[8], int D, float (&acc)[8], int lane) {
  // real loops (unroll 1): fully unrolled, the scheduler hoists every batch's loads to the top and the kernel needs 250 registers
  if (D == 384) {
    if (WIDE) {  // all 8 rows at once: 24 loads per lane in flight (the re-scoring kernel, ~170 registers)
      score_rows_fixed<3, 8>(qrow, rows, acc, lane);
      return;
    }
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      const float* r[4];
      float t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) r[u] = h ? rows[4 + u] : rows[u];
      score_rows_fixed<3, 4>(qrow, r, t, lane);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        acc[u] = h ? acc[u] : t[u];
        acc[4 + u] = h ? t[u] : 0.f;
      }
    }
    return;
  }
  if (D == 768) {
#pragma unroll 1
    for (int h = 0; h < 4; ++h) {
      const float* r[2];
      float t[2];
      r[0] = h == 0 ? rows[0] : (h == 1 ? rows[2] : (h == 2 ? rows[4] : rows[6]));
      r[1] = h == 0 ? rows[1] : (h == 1 ? rows[3] : (h == 2 ? rows[5] : rows[7]));
      score_rows_fixed<6, 2>(qrow, r, t, lane);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        acc[2 * u] = h == u ? t[0] : (h < u ? 0.f : acc[2 * u]);
        acc[2 * u + 1] = h == u ? t[1] : (h < u ? 0.f : acc[2 * u + 1]);
      }
    }
    return;
  }
#pragma unroll
  for (int u = 0; u < 8; ++u) acc[u] = 0.f;
  const int nvec = D >> 2;
#pragma unroll 1
  for (int v = lane; v < nvec; v += 32) {
    const float4 qv = __ldg(reinterpret_cast<const float4*>(qrow) + v);
    float4 c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) c[u] = __ldg(reinterpret_cast<const float4*>(rows[u]) + v);
#pragma unroll
    for (int u = 0; u < 8; ++u) acc[u] = fmaf(qv.x, c[u].x, fmaf(qv.y, c[u].y, fmaf(qv.z, c[u].z, fmaf(qv.w, c[u].w, acc[u]))));
  }
}

// sel[i] <- exact key of the row held in sel[i], for i = first, first + stride, ... in batches of 8 (one warp)
template <bool WIDE = false>
__device__ __forceinline__ void warp_rescore(uint64_t* sel, int m, int first_batch, int batch_stride, int64_t q, const HistSelectArgs& a, int lane) {
  const float* qrow = a.rs_q + q * a.rs_ldq;
  const float qi = a.rs_qinv[q];
  for (int b0 = first_batch * 8; b0 < m; b0 += batch_stride * 8) {
    const float* rows[8];
    uint32_t rid[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      rid[u] = key_row(sel[min(b0 + u, m - 1)]);
      rows[u] = a.rs_cat + static_cast<int64_t>(rid[u]) * a.rs_ldc;
    }
    float acc[8];
    score_rows8<WIDE>(qrow, rows, a.rs_D, acc, lane);
    warp_transpose_reduce<8>(acc, lane);  // lane l: full sum of row (l >> 2)
    const int u = lane >> 2;
    uint32_t my_row = rid[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) my_row = (u == j) ? rid[j] : my_row;
    __syncwarp();
    if ((lane & 3) == 0 && b0 + u < m) sel[b0 + u] = make_key(acc[0] * qi * __ldg(a.rs_cinv + my_row), my_row);
  }
  __syncwarp();
}

template <bool WIDE>
__device__ __forceinline__ void ls_rescore(uint32_t* sc, const uint32_t* rw, int m, int64_t q, const HistSelectArgs& a, int lane) {
  const float* qrow = a.rs_q + q * a.rs_ldq;
  const float qi = a.rs_qinv[q];
  for (int b0 = 0; b0 < m; b0 += 8) {
    const float* rows[8];
    uint32_t rid[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      rid[u] = ~rw[min(b0 + u, m - 1)];
      rows[u] = a.rs_cat + static_cast<int64_t>(rid[u]) * a.rs_ldc;
    }
    float acc[8];
    score_rows8<WIDE>(qrow, rows, a.rs_D, acc, lane);
    warp_transpose_reduce<8>(acc, lane);  // lane l: full sum of row (l >> 2)
    const int u = lane >> 2;
    uint32_t my_row = rid[0];
#pragma unroll
    for (int j = 1; j < 8; ++j) my_row = (u == j) ? rid[j] : my_row;
    if ((lane & 3) == 0 && b0 + u < m) sc[b0 + u] = order_bits(acc[0] * qi * __ldg(a.rs_cinv + my_row));
  }
  __syncwarp();
}

// Exact ranking of the WHOLE catalog for one query by one warp (only for queries whose screening band overflowed: more
// near-ties around the k-th score than the carry holds). Leaves the k best exact keys in sc/rw, returns their number.
template <bool XB = false>
__device__ __forceinline__ int ls_rank_catalog(uint32_t* sc, uint32_t* rw, int buf_cap, uint32_t* hist, int64_t q, const HistSelectArgs& a, int lane) {
  const float* qrow = a.rs_q + q * a.rs_ldq;
  const float qi = a.rs_qinv[q];
  const unsigned lt = (1u << lane) - 1u;
  const int k = a.k;
  int n = 0;
  uint32_t fs = 0u, fr = 0u;  // keys <= (fs, fr) cannot be among the k best any more
  for (int64_t r0 = 0; r0 < a.rs_N; r0 += 8) {
    const float* rows[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) rows[u] = a.rs_cat + min(r0 + u, a.rs_N - 1) * a.rs_ldc;
    float acc[8];
    score_rows8(qrow, rows, a.rs_D, acc, lane);
    warp_transpose_reduce<8>(acc, lane);
    const int64_t row = r0 + (lane >> 2);
    bool ok = (lane & 3) == 0 && row < a.rs_N && !a.excl().excluded<XB>(q, row);
    uint32_t s1 = 0, r1 = 0;
    if (ok) {
      s1 = order_bits(acc[0] * qi * __ldg(a.rs_cinv + row));
      r1 = ~static_cast<uint32_t>(row);
      ok = pair_gt(s1, r1, fs, fr);
    }
    const unsigned mk = __ballot_sync(kFull, ok);
    if (ok) {
      const int pos = n + __popc(mk & lt);
      sc[pos] = s1;
      rw[pos] = r1;
    }
    n += __popc(mk);
    if (n > buf_cap - 8) {
      __syncwarp();
      float t;
      n = ls_reduce(sc, rw, n, k, 0.f, hist, &t);  // exact keys: exactly k survive
      uint32_t ms = 0xFFFFFFFFu, mr = 0xFFFFFFFFu;
      for (int i = lane; i < n; i += 32)
        if (pair_gt(ms, mr, sc[i], rw[i])) {
          ms = sc[i];
          mr = rw[i];
        }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const uint32_t os = __shfl_xor_sync(kFull, ms, o), orr = __shfl_xor_sync(kFull, mr, o);
        if (pair_gt(ms, mr, os, orr)) {
          ms = os;
          mr = orr;
        }
      }
      fs = ms;
      fr = mr;
    }
  }
  __syncwarp();
  float t;
  return ls_reduce(sc, rw, n, k, 0.f, hist, &t);
}

// Ordered output of the k best of the `kept` (<= 512) keys. Up to 128 keys (the usual case: k <= 100 results plus a few
// keys of the screening band) are sorted as 64-bit keys by a warp bitonic network in the idle histogram array - rank counting
// is O(kept^2) and was half of the re-scoring kernel's time; beyond 128 each lane rank-counts four of its keys at a time.
__device__ __forceinline__ void ls_emit_ranked(const uint32_t* sc, const uint32_t* rw, int kept, int k, float scale, int64_t q, const HistSelectArgs& a,
                                               uint32_t* hist, int lane) {
  if (kept <= 128) {
    uint64_t* keys = reinterpret_cast<uint64_t*>(hist);  // kHsBins * 4 bytes = 128 keys
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = lane + 32 * u;
      keys[i] = i < kept ? ((static_cast<uint64_t>(sc[i]) << 32) | rw[i]) : 0ull;
    }
    warp_bitonic_sort_desc(keys, 128, lane);
    for (int i = lane; i < k; i += 32) {
      const bool ok = i < kept;
      const uint64_t key = ok ? keys[i] : 0ull;
      a.out_scores[q * k + i] = ok ? unorder_bits(static_cast<uint32_t>(key >> 32)) * scale : -INFINITY;
      a.out_ids[q * k + i] = ok ? static_cast<int64_t>(~static_cast<uint32_t>(key)) + a.id_offset : -1;
    }
    return;
  }
  for (int base = lane; base < kept; base += 128) {
    uint32_t s1[4], r1[4];
    int rank[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + 32 * u;
      s1[u] = i < kept ? sc[i] : 0xFFFFFFFFu;
      r1[u] = i < kept ? rw[i] : 0xFFFFFFFFu;
      rank[u] = 0;
    }
#pragma unroll 2
    for (int j = 0; j < kept; ++j) {
      const uint32_t s2 = sc[j], r2 = rw[j];
#pragma unroll
      for (int u = 0; u < 4; ++u) rank[u] += (pair_gt(s2, r2, s1[u], r1[u]) || (j < base + 32 * u && s2 == s1[u] && r2 == r1[u])) ? 1 : 0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (base + 32 * u < kept && rank[u] < k) {
        a.out_scores[q * k + rank[u]] = unorder_bits(s1[u]) * scale;
        a.out_ids[q * k + rank[u]] = static_cast<int64_t>(~r1[u]) + a.id_offset;
      }
    }
  }
  for (int i = min(kept, k) + lane; i < k; i += 32) {
    a.out_scores[q * k + i] = -INFINITY;
    a.out_ids[q * k + i] = -1;
  }
}

}  // namespace icr
