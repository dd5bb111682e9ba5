// K7: cosine top-k over per-query candidate lists (icr_cos_topk_subset). Query q ranks only the catalog rows
// rows[offsets[q] .. offsets[q+1]) of a CSR list, so a call reads about nnz rows of the catalog, not N.
//
// Two launches, no host round trip:
//   subset_prep_kernel   one warp per query: its inverse norm (fp32: the screening helper of the tensor-core path; 16-bit:
//       row_sumsq) or its int8 codes and factor (I8Rows), the merge ticket reset, the (-inf, -1) rows of an empty list, and
//       for every chunk the query that holds the chunk's first entry.
//   subset_topk_kernel   one warp per chunk of `chunk` consecutive CSR entries, whatever the list lengths (a 1M-row list
//       is cut into many chunks, a thousand 10-row lists share a few): the warp scores the entries of each query in the
//       chunk eight rows at a time - ls_rank_catalog's loop walking a list - and keeps the best keys in a shared-memory
//       buffer held against a running floor. A query wholly inside the chunk is finished there. A query that spans chunks
//       leaves its k best keys of each chunk in a workspace slot; the last of its pieces to arrive (a per-query ticket,
//       atom.add.acq_rel.gpu) merges the slots and writes the sorted top-k.
// Scores are those of the exact ranking paths: fp32 rows score_rows8 * qinv * cinv (the tensor-core path's re-scoring,
// bit for bit), 16-bit rows fp32 FMAs on the values * both inverse norms, int8 rows fp32(S) * f_row with S the exact code
// dot product and the score key * f_query (K1's int8 arithmetic).
#include "common.cuh"
#include "rows.cuh"
#include "select_finish.cuh"

namespace icr {

constexpr int kSubWarps = 4;           // warps (= chunks) per CTA
constexpr int kSubCap = 1024;          // keys buffered per warp (> ICR_MAX_K + one window of 32)
constexpr int kSubGroup = 8;           // slots read together by a merge
constexpr int64_t kSubTargetWarps = 148 * 8;
constexpr int64_t kSubChunkMax = 4096;

struct SubsetArgs {
  const void* q;
  int64_t ldq;
  int64_t Q;
  const void* cat;
  int64_t N;
  int64_t ldc;
  int D;
  const float* cinv;  // row inverse norms (int8: the row factors)
  const int64_t* offsets;
  const int64_t* rows;
  int64_t nnz;
  int k;
  int chunk_log2;  // entries per chunk = 1 << chunk_log2
  int64_t nchunks;
  int64_t id_offset;
  float* out_scores;
  int64_t* out_ids;
  // workspace
  float* qinv;         // [Q] query inverse norms (int8: query factors)
  int8_t* qcodes;      // [Q][D] int8 query codes
  unsigned int* ticket;  // [Q]
  int* chunk_first;    // [nchunks]
  uint64_t* slots;     // [nchunks][2][k]: slot 0 = the query that entered the chunk from before, 1 = the one leaving it
};

// log2 of the entries per chunk (a power of two: the kernels divide by shifts): enough chunks to give every SM a few
// warps, at least 4k entries per chunk so that the slots stay a fraction of the list (2 * ceil(nnz / chunk) * k keys
// <= nnz / 2 + 2k), at most kSubChunkMax.
static int subset_chunk_log2(int64_t nnz, int k) {
  int64_t c = (nnz + kSubTargetWarps - 1) / kSubTargetWarps;
  const int64_t lo = 4 * k > 64 ? 4 * k : 64;
  if (c < lo) c = lo;
  if (c > kSubChunkMax) c = kSubChunkMax;
  int s = 5;
  while ((int64_t{1} << s) < c) ++s;
  return s;
}

struct SubsetWs {
  size_t qinv, qcodes, ticket, chunk_first, slots, total;
  int chunk_log2;
  int64_t nchunks;
};

static SubsetWs subset_ws_layout(int64_t Q, int64_t nnz, int64_t D, int dtype, int k) {
  SubsetWs L{};
  L.chunk_log2 = subset_chunk_log2(nnz, k);
  L.nchunks = nnz > 0 ? ((nnz - 1) >> L.chunk_log2) + 1 : 0;
  size_t o = 0;
  L.qinv = o;
  o += align_up(static_cast<size_t>(Q) * sizeof(float), 256);
  L.qcodes = o;
  if (dtype == ICR_I8) o += align_up(static_cast<size_t>(Q) * static_cast<size_t>(D), 256);
  L.ticket = o;
  o += align_up(static_cast<size_t>(Q) * sizeof(unsigned int), 256);
  L.chunk_first = o;
  o += align_up(static_cast<size_t>(L.nchunks) * sizeof(int), 256);
  L.slots = o;
  o += align_up(static_cast<size_t>(L.nchunks) * 2 * static_cast<size_t>(k) * sizeof(uint64_t), 256);
  L.total = o > 256 ? o : 256;
  return L;
}

size_t subset_workspace_bytes(int64_t Q, int64_t nnz, int64_t D, int dtype, int k) { return subset_ws_layout(Q, nnz, D, dtype, k).total; }

// ---- query preparation --------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) subset_prep_kernel(SubsetArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t q = warp; q < a.Q; q += nwarps) {
    const int64_t b = __ldg(a.offsets + q), e = __ldg(a.offsets + q + 1);
    if (b >= e) {  // an empty list owns no chunk: its rows are written here
      for (int i = lane; i < a.k; i += 32) {
        a.out_scores[q * a.k + i] = -INFINITY;
        a.out_ids[q * a.k + i] = -1;
      }
    } else {
      const int64_t mask = (int64_t{1} << a.chunk_log2) - 1;
      for (int64_t c = ((b + mask) >> a.chunk_log2) + lane; (c << a.chunk_log2) < e; c += 32) a.chunk_first[c] = static_cast<int>(q);
    }
    float inv;
    if constexpr (std::is_same_v<T, int8_t>) {
      uint32_t* dst = reinterpret_cast<uint32_t*>(a.qcodes + q * a.D);
      inv = I8Rows::quantize(static_cast<const float*>(a.q) + q * a.ldq, a.D, a.D / 4, lane, [dst](int w, uint32_t word) { dst[w] = word; });
    } else if constexpr (std::is_same_v<T, float>) {
      // the tensor-core path's query norm (screen_row), which its exact re-scoring multiplies by
      const float ss = screen_sumsq<true>(static_cast<const float*>(a.q) + q * a.ldq, a.D / 4, lane);
      inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
    } else {
      const float ss = row_sumsq<T, true>(static_cast<const T*>(a.q) + q * a.ldq, a.D / Elem<T>::VEC, a.D, lane);
      inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
    }
    if (lane == 0) {
      a.qinv[q] = inv;
      a.ticket[q] = 0u;
    }
  }
}

// ---- scoring of 8 listed rows (lane l ends with the key of row l >> 2) ---------------------------------------------
template <typename T>
__device__ __forceinline__ void score_rows8_elem(const T* __restrict__ qrow, const T* const (&rows)[8], int D, float (&acc)[8], int lane) {
  constexpr int VEC = Elem<T>::VEC;
  const int nvec = D / VEC;
#pragma unroll
  for (int u = 0; u < 8; ++u) acc[u] = 0.f;
  for (int v = lane; v < nvec; v += 32) {
    float qf[VEC];
    Elem<T>::unpack(__ldg(reinterpret_cast<const uint4*>(qrow) + v), qf);
    uint4 c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) c[u] = ldg_stream(rows[u] + static_cast<int64_t>(v) * VEC);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float f[VEC];
      Elem<T>::unpack(c[u], f);
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[u] = fmaf(qf[i], f[i], acc[u]);
    }
  }
}

__device__ __forceinline__ void score_rows8_i8(const int8_t* __restrict__ qcodes, const int8_t* const (&rows)[8], int D, int (&acc)[8], int lane) {
  const int nvec = D / 16;
#pragma unroll
  for (int u = 0; u < 8; ++u) acc[u] = 0;
  for (int v = lane; v < nvec; v += 32) {
    const uint4 qv = __ldg(reinterpret_cast<const uint4*>(qcodes) + v);
    uint4 c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) c[u] = ldg_stream(rows[u] + static_cast<int64_t>(v) * 16);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      int s = acc[u];
      s = __dp4a(static_cast<int>(c[u].x), static_cast<int>(qv.x), s);
      s = __dp4a(static_cast<int>(c[u].y), static_cast<int>(qv.y), s);
      s = __dp4a(static_cast<int>(c[u].z), static_cast<int>(qv.z), s);
      acc[u] = __dp4a(static_cast<int>(c[u].w), static_cast<int>(qv.w), s);
    }
  }
}

// order bits of the ranking key of rid[lane >> 2] (valid on lanes with lane & 3 == 0)
template <typename T>
__device__ __forceinline__ uint32_t score_keys8(const SubsetArgs& a, int64_t q, float qi, const uint32_t (&rid)[8], uint32_t my_row, int lane) {
  if constexpr (std::is_same_v<T, int8_t>) {
    const int8_t* rows[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) rows[u] = static_cast<const int8_t*>(a.cat) + static_cast<int64_t>(rid[u]) * a.ldc;
    int acc[8];
    score_rows8_i8(a.qcodes + q * a.D, rows, a.D, acc, lane);
    warp_transpose_reduce<8, int>(acc, lane);
    return order_bits(I8Rows::key(acc[0], __ldg(a.cinv + my_row)));
  } else {
    const T* rows[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) rows[u] = static_cast<const T*>(a.cat) + static_cast<int64_t>(rid[u]) * a.ldc;
    float acc[8];
    const T* qrow = static_cast<const T*>(a.q) + q * a.ldq;
    if constexpr (std::is_same_v<T, float>) score_rows8(qrow, rows, a.D, acc, lane);  // the arithmetic of ls_rescore / ls_rank_catalog
    else score_rows8_elem<T>(qrow, rows, a.D, acc, lane);
    warp_transpose_reduce<8>(acc, lane);
    return order_bits(acc[0] * qi * __ldg(a.cinv + my_row));
  }
}

// ---- selection helpers ---------------------------------------------------------------------------------------------
// the smallest kept key (every key <= it can no longer be among the k best once the buffer holds k keys)
__device__ __forceinline__ void warp_floor(const uint32_t* sc, const uint32_t* rw, int n, int lane, uint32_t& fs, uint32_t& fr) {
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

// appends the keys of the lanes with `ok`; squeezes the buffer to the k best and raises the floor when fewer than
// `room` free places are left
__device__ __forceinline__ void warp_append(bool ok, uint32_t s1, uint32_t r1, uint32_t* sc, uint32_t* rw, uint32_t* hist, int& n, int k, int room,
                                            uint32_t& fs, uint32_t& fr, int lane) {
  const unsigned mk = __ballot_sync(kFull, ok);
  if (ok) {
    const int pos = n + __popc(mk & ((1u << lane) - 1u));
    sc[pos] = s1;
    rw[pos] = r1;
  }
  n += __popc(mk);
  if (n > kSubCap - room) {
    __syncwarp();
    float t;
    n = ls_reduce(sc, rw, n, k, 0.f, hist, &t);
    warp_floor(sc, rw, n, lane, fs, fr);
  }
}

// Ordered output of the k best of the `kept` keys: out(i, key) for i < k, key 0 past the kept ones. ls_emit_ranked's
// two regimes: a warp bitonic sort of up to 128 keys in the idle histogram, rank counting beyond.
template <typename Out>
__device__ __forceinline__ void subset_emit(const uint32_t* sc, const uint32_t* rw, int kept, int k, uint32_t* hist, int lane, Out out) {
  if (kept <= 128) {
    uint64_t* keys = reinterpret_cast<uint64_t*>(hist);
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = lane + 32 * u;
      keys[i] = i < kept ? ((static_cast<uint64_t>(sc[i]) << 32) | rw[i]) : 0ull;
    }
    warp_bitonic_sort_desc(keys, 128, lane);
    for (int i = lane; i < k; i += 32) out(i, i < kept ? keys[i] : 0ull);
    __syncwarp();
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
    for (int u = 0; u < 4; ++u)
      if (base + 32 * u < kept && rank[u] < k) out(rank[u], (static_cast<uint64_t>(s1[u]) << 32) | r1[u]);
  }
  for (int i = min(kept, k) + lane; i < k; i += 32) out(i, 0ull);
  __syncwarp();
}

__device__ __forceinline__ void emit_final(const SubsetArgs& a, const uint32_t* sc, const uint32_t* rw, int kept, int64_t q, float scale, uint32_t* hist,
                                           int lane) {
  float* os = a.out_scores + q * a.k;
  int64_t* oi = a.out_ids + q * a.k;
  const int64_t off = a.id_offset;
  subset_emit(sc, rw, kept, a.k, hist, lane, [&](int i, uint64_t key) {
    os[i] = key ? unorder_bits(static_cast<uint32_t>(key >> 32)) * scale : -INFINITY;
    oi[i] = key ? static_cast<int64_t>(~static_cast<uint32_t>(key)) + off : -1;
  });
}

// slot of query q's piece in chunk c: 0 if the query entered the chunk from an earlier one, 1 if it starts inside it
__device__ __forceinline__ uint64_t* subset_slot(const SubsetArgs& a, int64_t c, int64_t qb) {
  return a.slots + (c * 2 + (qb < (c << a.chunk_log2) ? 0 : 1)) * a.k;
}

// ---- the top-k kernel: one warp per chunk of CSR entries ------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kSubWarps * 32) subset_topk_kernel(SubsetArgs a) {
  constexpr bool I8 = std::is_same_v<T, int8_t>;
  __shared__ __align__(16) uint32_t s_sc[kSubWarps][kSubCap];
  __shared__ __align__(16) uint32_t s_rw[kSubWarps][kSubCap];
  __shared__ __align__(16) uint32_t s_hist[kSubWarps][kHsBins];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = static_cast<int64_t>(blockIdx.x) * kSubWarps + warp;
  if (c >= a.nchunks) return;
  uint32_t* sc = s_sc[warp];
  uint32_t* rw = s_rw[warp];
  uint32_t* hist = s_hist[warp];
  const int k = a.k;
  const int64_t e0 = c << a.chunk_log2, e1 = min(e0 + (int64_t{1} << a.chunk_log2), a.nnz);
  for (int64_t q = a.chunk_first[c]; q < a.Q; ++q) {
    const int64_t qb = __ldg(a.offsets + q), qe = __ldg(a.offsets + q + 1);
    if (qb >= e1) break;
    const int64_t pb = max(qb, e0), pe = min(qe, e1);
    if (pb >= pe) continue;  // an empty list between two others
    const float qi = __ldg(a.qinv + q);
    int n = 0;
    uint32_t fs = 0u, fr = 0u;  // floor: keys <= (fs, fr) cannot be among the k best any more
    for (int64_t b0 = pb; b0 < pe; b0 += 32) {
      // 32 entries per window: lane j reads entry b0 + j; rows outside [0, N) are ignored
      const int64_t r = b0 + lane < pe ? __ldg(a.rows + b0 + lane) : -1;
      const bool valid = r >= 0 && r < a.N;
      const unsigned vm = __ballot_sync(kFull, valid);
      if (!vm) continue;
      const uint32_t rfirst = __shfl_sync(kFull, static_cast<uint32_t>(r), __ffs(vm) - 1);  // stands in for an invalid entry
      const uint32_t rr = valid ? static_cast<uint32_t>(r) : rfirst;
      for (int g = 0; g < 32; g += 8) {
        if (((vm >> g) & 0xFFu) == 0u) continue;
        uint32_t rid[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) rid[u] = __shfl_sync(kFull, rr, g + u);
        const int u = lane >> 2;
        uint32_t my_row = rid[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) my_row = (u == j) ? rid[j] : my_row;
        const uint32_t s1 = score_keys8<T>(a, q, qi, rid, my_row, lane);
        const uint32_t r1 = ~my_row;
        const bool ok = (lane & 3) == 0 && ((vm >> (g + u)) & 1u) && pair_gt(s1, r1, fs, fr);
        warp_append(ok, s1, r1, sc, rw, hist, n, k, 8, fs, fr, lane);
      }
    }
    __syncwarp();
    float t;
    n = ls_reduce(sc, rw, n, k, 0.f, hist, &t);
    const float scale = I8 ? qi : 1.0f;  // int8: score = key * f_query
    const int64_t c0 = qb >> a.chunk_log2, c1 = (qe - 1) >> a.chunk_log2;
    if (c0 == c1) {  // the whole list is in this chunk
      emit_final(a, sc, rw, n, q, scale, hist, lane);
      continue;
    }
    uint64_t* slot = subset_slot(a, c, qb);
    subset_emit(sc, rw, n, k, hist, lane, [slot](int i, uint64_t key) { slot[i] = key; });
    __threadfence();
    __syncwarp();
    unsigned int prev = 0;
    if (lane == 0) asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(prev) : "l"(a.ticket + q) : "memory");
    prev = __shfl_sync(kFull, prev, 0);
    if (prev != static_cast<unsigned int>(c1 - c0)) continue;
    __threadfence();
    // the last piece: merge the sorted slots of chunks c0 .. c1, kSubGroup at a time. A slot's keys are sorted, so its
    // first window of 32 usually settles it; later windows are read only while a whole window beats the floor
    n = 0;
    fs = fr = 0u;
    for (int64_t cg = c0; cg <= c1; cg += kSubGroup) {
      uint64_t key[kSubGroup];
#pragma unroll
      for (int j = 0; j < kSubGroup; ++j) key[j] = (cg + j <= c1 && lane < k) ? __ldcg(subset_slot(a, cg + j, qb) + lane) : 0ull;
#pragma unroll
      for (int j = 0; j < kSubGroup; ++j) {
        uint32_t s1 = static_cast<uint32_t>(key[j] >> 32), r1 = static_cast<uint32_t>(key[j]);
        bool ok = key[j] != 0ull && pair_gt(s1, r1, fs, fr);
        bool more = __ballot_sync(kFull, ok) >> 31;
        warp_append(ok, s1, r1, sc, rw, hist, n, k, 32, fs, fr, lane);
        for (int w = 32; more && w < k; w += 32) {
          const uint64_t kw = lane + w < k ? __ldcg(subset_slot(a, cg + j, qb) + lane + w) : 0ull;
          s1 = static_cast<uint32_t>(kw >> 32);
          r1 = static_cast<uint32_t>(kw);
          ok = kw != 0ull && pair_gt(s1, r1, fs, fr);
          more = __ballot_sync(kFull, ok) >> 31;
          warp_append(ok, s1, r1, sc, rw, hist, n, k, 32, fs, fr, lane);
        }
      }
    }
    __syncwarp();
    n = ls_reduce(sc, rw, n, k, 0.f, hist, &t);
    emit_final(a, sc, rw, n, q, scale, hist, lane);
  }
}

// ---- host side ------------------------------------------------------------------------------------------------------
template <typename T>
static int launch_subset_t(const SubsetArgs& a, cudaStream_t st) {
  const int64_t want = (a.Q + 7) / 8;
  const int pblocks = static_cast<int>(want < 148 * 16 ? want : 148 * 16);
  subset_prep_kernel<T><<<pblocks, 256, 0, st>>>(a);
  ICR_LAUNCH_CHECK();
  if (a.nchunks == 0) return ICR_OK;
  const int64_t blocks = (a.nchunks + kSubWarps - 1) / kSubWarps;
  profile_begin(kKernelGemv, 1, st);
  subset_topk_kernel<T><<<static_cast<unsigned int>(blocks), kSubWarps * 32, 0, st>>>(a);
  profile_end(st);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

int launch_subset_topk(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D, int dtype,
                       const float* cat_inv_norms, const int64_t* offsets, const int64_t* rows, int64_t nnz, int k, int64_t row_offset,
                       float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const SubsetWs L = subset_ws_layout(Q, nnz, D, dtype, k);
  if (workspace_bytes < L.total || !workspace) {
    set_error("cos_topk_subset: workspace %zu bytes < required %zu", workspace_bytes, L.total);
    return ICR_ERR_WORKSPACE;
  }
  if (Q == 0) return ICR_OK;
  char* base = static_cast<char*>(workspace);
  SubsetArgs a{};
  a.q = queries;
  a.ldq = ldq;
  a.Q = Q;
  a.cat = catalog;
  a.N = N;
  a.ldc = ldc;
  a.D = static_cast<int>(D);
  a.cinv = cat_inv_norms;
  a.offsets = offsets;
  a.rows = rows;
  a.nnz = nnz;
  a.k = k;
  a.chunk_log2 = L.chunk_log2;
  a.nchunks = L.nchunks;
  a.id_offset = row_offset;
  a.out_scores = out_scores;
  a.out_ids = out_ids;
  a.qinv = reinterpret_cast<float*>(base + L.qinv);
  a.qcodes = reinterpret_cast<int8_t*>(base + L.qcodes);
  a.ticket = reinterpret_cast<unsigned int*>(base + L.ticket);
  a.chunk_first = reinterpret_cast<int*>(base + L.chunk_first);
  a.slots = reinterpret_cast<uint64_t*>(base + L.slots);
  if (dtype == ICR_F32) return launch_subset_t<float>(a, st);
  if (dtype == ICR_BF16) return launch_subset_t<__nv_bfloat16>(a, st);
  if (dtype == ICR_F16) return launch_subset_t<__half>(a, st);
  return launch_subset_t<int8_t>(a, st);
}

}  // namespace icr
