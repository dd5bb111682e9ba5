// K1: streaming cosine GEMV with fused top-k for small query batches (Q <= 7 per pass).
//
// HBM-bound by design: every catalog row is read exactly once; the row's squared norm is accumulated from
// the same data (or, for a single query against a catalog that carries precomputed inverse norms, the 32 bytes of
// norms ride into the ring with their slab). Scores never reach HBM:
// each CTA keeps, per query, a shared-memory candidate list guarded by a running threshold (the CTA's k-th
// best so far) and emits its k best keys; the last CTA to finish merges the per-CTA lists in the same launch
// (no second kernel on the batch-1 latency path).
//
// Two ways of moving the rows:
//   gemv_ring_kernel  (default, contiguous catalogs): a producer warp streams 8-row slabs with 1-D bulk async
//       copies (cp.async.bulk, the TMA engine) into a shared-memory ring guarded by mbarriers; eight consumer
//       warps read slabs with conflict-free 128-bit shared loads. The whole ring (up to 192 KB per SM) is in
//       flight from the first microsecond, independent of consumer register pressure. Every CTA owns one ring
//       filling of slabs; the rest of the catalog is handed out in chunks from a device-wide counter, so the
//       slowest SM does not hold up the request's tail.
//   gemv_topk_kernel  (row-strided catalogs): 128-bit ld.global.nc.L1::no_allocate, RB rows x 3 vectors per
//       lane in flight.
//
// Replaces, for one request: torch.tensor(catalog) + F.normalize x2 + torch.mm + argsort
// (reference src/inference/serve_recommendations.py:213-215 via sentence_transformers.util.cos_sim).
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "peer.cuh"
#include "ptx.cuh"
#include "select_warp.cuh"

namespace icr {

constexpr int kGemvThreads = 256;  // compute threads of either kernel
constexpr int kGemvWarps = kGemvThreads / 32;
constexpr int kGemvUnroll = 3;   // 16-byte vectors per lane per row kept in flight (direct-load kernel)
constexpr int kMergeSel = 256;   // >= ICR_MAX_K: output buffer of the in-kernel merge
constexpr int kMaxSlots = 64;
constexpr int kRingThreads = kGemvThreads + 32;  // + the producer warp

#ifdef ICR_TRACE  // development builds only (ICR_NVCC_DEFS=-DICR_TRACE): per-CTA globaltimer stamps of the ring kernel
__device__ unsigned long long g_trace[296 * 8];
#define ICR_STAMP(i)                                                      \
  do {                                                                    \
    if ((threadIdx.x & 255) == 0 && threadIdx.x < 256) {                  \
      unsigned long long t_;                                              \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));              \
      g_trace[blockIdx.x * 8 + (i)] = t_;                                 \
    }                                                                     \
  } while (0)
__device__ unsigned long long g_trace_merge[8];
#define ICR_MSTAMP(i)                                                     \
  do {                                                                    \
    if (threadIdx.x == 0) {                                               \
      unsigned long long t_;                                              \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));              \
      g_trace_merge[i] = t_;                                              \
    }                                                                     \
  } while (0)
#else
#define ICR_STAMP(i) do {} while (0)
#define ICR_MSTAMP(i) do {} while (0)
#endif

struct GemvArgs {
  const void* cat;
  int64_t N;
  int64_t ldc;
  int D;
  const void* q;  // [Q][D] same dtype as the catalog (int8 catalogs: fp32 queries, quantised by every CTA)
  int64_t ldq;
  int Q;
  const uint8_t* mask;  // optional exclusion mask
  const float* cat_inv;  // optional precomputed 1 / max(|row|, eps) (icr_row_inv_norms): single-query ring kernel skips the norm FMAs
  int k;
  int64_t rows_per_cta;
  uint64_t* part_keys;  // [Q][gridDim.x][k]
  int* part_cnt;        // [Q][gridDim.x]
  int q0;               // first query of this pass
  int ring_slots;       // ring kernel: slots of kSlabRows rows
  // in-kernel merge by the last CTA (skipped when out_scores is null)
  float* out_scores;           // [Q][k]
  int64_t* out_ids;            // [Q][k]
  int64_t id_offset;
  unsigned int* done_counter;  // zero before the first launch; the merging CTA resets it
  // ring kernel: rows are handed out as slabs. Every CTA owns `static_slabs` slabs up front (its ring is in flight before
  // the first atomic returns); the rest of the catalog is pulled in chunks of kProducers slabs from a device-wide counter
  // (done_counter[1], same reset rule), so that no SM is still streaming while the others sit in the tail of the request
  unsigned int* chunk_counter;
  int static_slabs;
#ifdef ICR_TRACE
  int dbg;  // development builds: ICR_K1_DBG bit 0 = consumers skip the arithmetic, bit 1 = static row blocks only, bit 2 = 8-slot ring
#endif
  // sharded request (peer_on): out_scores / out_ids are a staging area for this shard's lists; the merging CTA pushes them to
  // every peer, waits for theirs and writes the global top-k to fin_scores / fin_ids (one pass only: Q <= 7, q0 = 0)
  int peer_on;
  float* fin_scores;
  int64_t* fin_ids;
  PeerTail peer;
  // per-query exclusions (XB kernels): Exclusions::bits of this call's queries, query a.q0 + t at column a.q0 + t
  const uint32_t* xbits;
  int64_t xld;
};

// barrier over the 256 compute threads: the whole CTA in the direct kernel, a named barrier in the ring kernel
template <bool NAMED>
__device__ __forceinline__ void compute_sync() {
  if (NAMED) ptx::named_sync(1, kGemvThreads);
  else __syncthreads();
}

// shared-memory carve-up common to both kernels (after `prefix` bytes used by the ring)
template <int QT>
struct GemvSmem {
  // candidate keys per query held in shared memory (>= k + the rows scored between two threshold refreshes)
  static constexpr int CAND = QT == 1 ? 1024 : (QT <= 3 ? 768 : 512);
  uint64_t* cand;       // [QT][CAND]
  uint64_t* sel;        // [QT][kMergeSel]  selection output (threshold refresh, merge fallback)
  float* qs;            // [QT][dpad]
  int* ncand;           // [QT]
  float* tau;           // [QT]
  int* list_cnt;        // [512]   merge: per-query floor slots and counters
  unsigned int* hist;   // [QT][kHsBins]
  __device__ GemvSmem(unsigned char* base, int dpad) {
    cand = reinterpret_cast<uint64_t*>(base);
    sel = cand + QT * CAND;
    qs = reinterpret_cast<float*>(sel + QT * kMergeSel);
    ncand = reinterpret_cast<int*>(qs + QT * dpad);
    tau = reinterpret_cast<float*>(ncand + QT);
    list_cnt = reinterpret_cast<int*>(tau + QT);
    hist = reinterpret_cast<unsigned int*>(list_cnt + 512);
  }
  static size_t bytes(int D) {
    return static_cast<size_t>(QT) * (CAND * 8 + kMergeSel * 8 + kHsBins * 4 + 8) + static_cast<size_t>(QT) * D * 4 + 512 * 4 + 16;
  }
};

// floats of the query area per query (GemvSmem::qs): the fp32 row for the float kernels; the int8 kernels stage D / 4 packed
// words and keep the query factors in the last 8 floats of the area (i8_query_factors), so each query gets 8 floats more
template <typename T>
__host__ __device__ constexpr int query_area(int D) { return std::is_same_v<T, int8_t> ? D / 4 + 8 : D; }

// ---- stage the L2-normalised queries in shared memory (fp32) ----------------------------------------
// One warp per query; the row is fetched with 16-byte loads issued back to back (one memory round trip: this
// sits on the critical path of a batch-1 request, before the first FMA).
template <typename T, int QT>
__device__ __forceinline__ void stage_queries(const GemvArgs& a, float* qs, int dpad, int nq, int warp, int lane) {
  constexpr int VEC = Elem<T>::VEC;
  constexpr int U = 4;
  const int nvec = dpad / VEC;
  const T* qg = static_cast<const T*>(a.q);
  for (int t = warp; t < QT; t += kGemvWarps) {
    float* dst = qs + t * dpad;
    if (t < nq) {
      const uint4* qrow = reinterpret_cast<const uint4*>(qg + static_cast<int64_t>(a.q0 + t) * a.ldq);
      float ss = 0.f;
      for (int vb = lane; vb < nvec; vb += 32 * U) {
        uint4 x[U];
#pragma unroll
        for (int u = 0; u < U; ++u) x[u] = (vb + 32 * u < nvec) ? __ldg(qrow + vb + 32 * u) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (vb + 32 * u < nvec) {
            float f[VEC];
            Elem<T>::unpack(x[u], f);
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
              dst[(vb + 32 * u) * VEC + i] = f[i];
              ss = fmaf(f[i], f[i], ss);
            }
          }
        }
      }
      ss = warp_sum(ss);
      const float inv = 1.0f / fmaxf(sqrtf(ss), kNormEps);
      __syncwarp();
      for (int e = lane; e < dpad; e += 32) dst[e] *= inv;
    } else {
      for (int e = lane; e < dpad; e += 32) dst[e] = 0.f;
    }
  }
}

// accumulate one 16-byte vector of RB rows against QT queries (+ the rows' squared norms unless NORMS: precomputed)
template <typename T, int RB, int QT, bool NORMS = false>
__device__ __forceinline__ void fma_vector(const uint4 (&c)[RB], const float* qs, int dpad, int v, float (&acc)[RB * (QT + (NORMS ? 0 : 1))]) {
  constexpr int VEC = Elem<T>::VEC;
  float qv[QT][VEC];
#pragma unroll
  for (int t = 0; t < QT; ++t) {
#pragma unroll
    for (int h = 0; h < VEC / 4; ++h) {
      const float4 x = *reinterpret_cast<const float4*>(qs + t * dpad + v * VEC + h * 4);
      qv[t][h * 4 + 0] = x.x;
      qv[t][h * 4 + 1] = x.y;
      qv[t][h * 4 + 2] = x.z;
      qv[t][h * 4 + 3] = x.w;
    }
  }
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    float f[VEC];
    Elem<T>::unpack(c[r], f);
#pragma unroll
    for (int t = 0; t < QT; ++t) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[t * RB + r] = fmaf(f[i], qv[t][i], acc[t * RB + r]);
    }
    if (!NORMS) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[QT * RB + r] = fmaf(f[i], f[i], acc[QT * RB + r]);
    }
  }
}

// transposing reduction of the RB*(QT+1) partial sums, then threshold test and candidate append
// NORMS: lane r (< RB) brings the precomputed inverse norm of row r0 + r in `inv_lane`
// XB: per-query exclusions, one scattered bitmap load for the (few) scores that beat the threshold
template <int RB, int QT, bool NORMS = false, bool XB = false>
__device__ __forceinline__ void reduce_and_append(float (&acc)[RB * (QT + (NORMS ? 0 : 1))], const GemvArgs& a, GemvSmem<QT>& sm, int nq, int64_t r0,
                                                  int64_t row_limit, int lane, float inv_lane = 0.f) {
  constexpr int V = RB * (QT + (NORMS ? 0 : 1));
  constexpr int SH = (V == 32) ? 0 : (V == 16 ? 1 : (V == 8 ? 2 : 3));  // lane -> value index shift
  warp_transpose_reduce<V>(acc, lane);
  const int idx = lane >> SH;  // value index owned by this lane
  const int t = idx / RB, r = idx % RB;
  // squared norm of row r lives in the lane group of index QT*RB + r
  const float ss = NORMS ? 0.f : __shfl_sync(kFull, acc[0], (QT * RB + r) << SH);
  const float inv = NORMS ? __shfl_sync(kFull, inv_lane, r) : (1.0f / fmaxf(sqrtf(ss), kNormEps));
  const int64_t row = r0 + r;
  if (t < nq && (lane & ((1 << SH) - 1)) == 0 && row < row_limit) {
    const bool excluded = a.mask && a.mask[row];
    const float score = acc[0] * inv;
    if (!excluded && score > sm.tau[t] && !(XB && Exclusions{nullptr, a.xbits, a.xld}.bit(a.q0 + t, row))) {
      const int pos = atomicAdd(&sm.ncand[t], 1);
      if (pos < GemvSmem<QT>::CAND) sm.cand[t * GemvSmem<QT>::CAND + pos] = make_key(score, static_cast<uint32_t>(row));
    }
  }
}

// ---- int8 rows (ICR_I8) ----------------------------------------------------------------------------------
// Each CTA quantises its queries from the fp32 rows (I8Rows) in the prologue, so a request stays one launch. The codes are
// staged as packed words [QT][D / 4] at the start of the query area (query_area<int8_t>: QT * (D / 4 + 8) floats); the query
// factors sit in its last 8 floats, behind the codes, where the merging CTA reads them back to scale the k final keys.
template <int QT>
__device__ __forceinline__ float* i8_query_factors(GemvSmem<QT>& sm) { return reinterpret_cast<float*>(sm.ncand) - 8; }

template <int QT>
__device__ __forceinline__ void stage_queries_i8(const GemvArgs& a, GemvSmem<QT>& sm, int D, int nq, int warp, int lane) {
  const int nwords = D / 4;
  const float* qg = static_cast<const float*>(a.q);
  for (int t = warp; t < QT; t += kGemvWarps) {
    uint32_t* dst = reinterpret_cast<uint32_t*>(sm.qs) + t * nwords;
    float f = 0.f;
    if (t < nq) {
      f = I8Rows::quantize(qg + static_cast<int64_t>(a.q0 + t) * a.ldq, D, nwords, lane, [dst](int w, uint32_t word) { dst[w] = word; });
    } else {
      for (int w = lane; w < nwords; w += 32) dst[w] = 0u;
    }
    if (lane == 0) i8_query_factors(sm)[t] = f;
  }
}

// int8 counterpart of fma_vector: exact int32 dot products, four codes per __dp4a. The accumulators are laid out as
// [VT][RB] like the float kernels'; slots t >= QT (the norm slot the int8 kernels keep for QT > 1, so that V stays a power
// of two) stay zero.
template <int RB, int QT, int VT>
__device__ __forceinline__ void dp4a_vector(const uint4 (&c)[RB], const float* qs, int dpad, int v, int (&acc)[RB * VT]) {
  const uint32_t* qw = reinterpret_cast<const uint32_t*>(qs);
  uint4 qv[QT];
#pragma unroll
  for (int t = 0; t < QT; ++t) qv[t] = *reinterpret_cast<const uint4*>(qw + t * (dpad / 4) + v * 4);
#pragma unroll
  for (int r = 0; r < RB; ++r) {
#pragma unroll
    for (int t = 0; t < QT; ++t) {
      int s = acc[t * RB + r];
      s = __dp4a(static_cast<int>(c[r].x), static_cast<int>(qv[t].x), s);
      s = __dp4a(static_cast<int>(c[r].y), static_cast<int>(qv[t].y), s);
      s = __dp4a(static_cast<int>(c[r].z), static_cast<int>(qv[t].z), s);
      acc[t * RB + r] = __dp4a(static_cast<int>(c[r].w), static_cast<int>(qv[t].w), s);
    }
  }
}

// one 16-byte vector of RB rows, whichever the element type (float kernels: fma_vector; int8: dp4a_vector)
template <typename T, int RB, int QT, bool NORMS, int VT, typename A>
__device__ __forceinline__ void accumulate_vector(const uint4 (&c)[RB], const float* qs, int dpad, int v, A (&acc)[RB * VT]) {
  if constexpr (std::is_same_v<T, int8_t>) dp4a_vector<RB, QT, VT>(c, qs, dpad, v, acc);
  else fma_vector<T, RB, QT, NORMS>(c, qs, dpad, v, acc);
}

// int8 counterpart of reduce_and_append: integer reduction, then key = fp32(S) * f_row (I8Rows::key). Lane r (< RB) brings
// the factor of row r0 + r in `f_lane`.
template <int RB, int QT, int VT, bool XB>
__device__ __forceinline__ void reduce_and_append_i8(int (&acc)[RB * VT], const GemvArgs& a, GemvSmem<QT>& sm, int nq, int64_t r0,
                                                     int64_t row_limit, int lane, float f_lane) {
  constexpr int V = RB * VT;
  constexpr int SH = (V == 32) ? 0 : (V == 16 ? 1 : (V == 8 ? 2 : 3));
  warp_transpose_reduce<V>(acc, lane);
  const int idx = lane >> SH;
  const int t = idx / RB, r = idx % RB;
  const float f = __shfl_sync(kFull, f_lane, r);
  const int64_t row = r0 + r;
  if (t < nq && (lane & ((1 << SH) - 1)) == 0 && row < row_limit) {
    const bool excluded = a.mask && a.mask[row];
    const float key = I8Rows::key(acc[0], f);
    if (!excluded && key > sm.tau[t] && !(XB && Exclusions{nullptr, a.xbits, a.xld}.bit(a.q0 + t, row))) {
      const int pos = atomicAdd(&sm.ncand[t], 1);
      if (pos < GemvSmem<QT>::CAND) sm.cand[t * GemvSmem<QT>::CAND + pos] = make_key(key, static_cast<uint32_t>(row));
    }
  }
}

// the score the merge writes for a key of query t: the key itself, or for int8 rows key * f_query
template <bool I8, int QT>
__device__ __forceinline__ float out_score(uint64_t key, GemvSmem<QT>& sm, int t) {
  if constexpr (I8) return __fmul_rn(key_score(key), i8_query_factors(sm)[t]);
  else return key_score(key);
}

// If a list could overflow during the next block of rows (or at the end), keep its k best and raise tau.
// One warp per query (QT <= 7 < 8 warps), histogram selection instead of a sort: no CTA-wide barrier inside, and
// every query of the pass is handled at the same time. The final lists are sorted (k keys only) for the merge.
template <int QT, bool NAMED>
__device__ __forceinline__ void refresh_thresholds(const GemvArgs& a, GemvSmem<QT>& sm, int nq, bool last, int block_rows, int tid,
                                                   bool early = false) {
  constexpr int CAND = GemvSmem<QT>::CAND;
  const int warp = tid >> 5, lane = tid & 31;
  if (warp < nq) {
    const int t = warp;
    const int n = min(sm.ncand[t], CAND);
    if (last || n > CAND - block_rows || (early && n >= 2 * a.k + 32)) {
      uint64_t* keys = sm.cand + t * CAND;
      uint64_t* sel = sm.sel + t * kMergeSel;
      int kept = min(n, a.k);
      uint64_t kth = ~0ull;
      if (n <= 64 || n <= a.k) {  // short list: order it by rank counting
        warp_rank_sort_desc(keys, n, sel, kept, lane);
        for (int i = lane; i < kept; i += 32) keys[i] = sel[i];
        if (kept > 0) kth = sel[kept - 1];
      } else {
        warp_select_topk(keys, n, a.k, sel, sm.hist + t * kHsBins, lane);  // k best, unordered
        __syncwarp();
        if (last) {  // the merge wants sorted lists
          warp_rank_sort_desc(sel, kept, keys, kept, lane);
          kth = keys[kept - 1];
        } else {
          for (int i = lane; i < kept; i += 32) {
            keys[i] = sel[i];
            kth = sel[i] < kth ? sel[i] : kth;
          }
          kth = warp_min_u64(kth);
        }
      }
      if (lane == 0) {
        sm.ncand[t] = kept;
        sm.tau[t] = (kept >= a.k) ? key_score(kth) : -INFINITY;
      }
    }
  }
  compute_sync<NAMED>();
}

// Rank (0 = largest) of `mine` among the distinct keys[0..n) in shared memory, by counting. One function, not inlined, shared by
// the threshold refresh, the list emit and the final merge of the single-query kernel: the tail of a request runs once per
// launch, the merge on ONE CTA, and after another model's kernels have run in between its instructions come from DRAM
// (~0.1 us per 128-byte line: 350 straight-line instructions of merge measured 5.5 us cold against 2 us warm). Code every CTA
// has just executed is resident in the SM when the merge needs it.
__device__ __noinline__ int cta_key_rank(const uint64_t* keys, int n, uint64_t mine) {
  int rank = 0;
#pragma unroll 4
  for (int j = 0; j < n; ++j) rank += (keys[j] > mine) ? 1 : 0;
  return rank;
}

// Single-query kernels: the whole CTA orders a list of <= 256 candidates (thread i ranks key i), instead of one warp doing
// it while seven wait at the barrier (the first refresh, 64 keys after 64 rows, held the CTA for ~1 us).
template <bool NAMED>
__device__ __forceinline__ void refresh_single(const GemvArgs& a, GemvSmem<1>& sm, int block_rows, int tid, bool early) {
  constexpr int CAND = GemvSmem<1>::CAND;
  const int n = min(sm.ncand[0], CAND);
  if (!(n > CAND - block_rows || (early && n >= 2 * a.k + 32))) return;  // uniform: ncand was read after a barrier
  if (n > kGemvThreads) {
    refresh_thresholds<1, NAMED>(a, sm, 1, false, block_rows, tid, early);
    return;
  }
  const uint64_t mine = tid < n ? sm.cand[tid] : 0ull;
  const int rank = tid < n ? cta_key_rank(sm.cand, n, mine) : n;
  compute_sync<NAMED>();  // every thread has read the list
  if (rank < a.k) sm.cand[rank] = mine;
  if (rank == a.k - 1) sm.tau[0] = key_score(mine);
  if (tid == 0) sm.ncand[0] = min(n, a.k);
  compute_sync<NAMED>();
}

// Merge of the G per-CTA lists of query t by a group of GT threads (gtid = index in the group); LISTS * GT >= G.
template <int QT, int GT, int LISTS, bool I8, typename Sync>
__device__ __forceinline__ void merge_query(const GemvArgs& a, GemvSmem<QT>& sm, int t, int gtid, Sync sync) {
  constexpr int kGemvCand = GemvSmem<QT>::CAND;
  const int k = a.k, G = gridDim.x, lane = gtid & 31;
  uint64_t* buf = sm.cand + t * GemvSmem<QT>::CAND;  // heads first, then the gathered candidates
  uint64_t* floor_slot = reinterpret_cast<uint64_t*>(sm.list_cnt) + t;
  int* counter = sm.list_cnt + 64 + t;
  const int64_t slot0 = static_cast<int64_t>(a.q0 + t) * G;
  uint64_t my_head[LISTS];
  int my_cnt[LISTS];
#pragma unroll
  for (int j = 0; j < LISTS; ++j) {  // all loads independent and issued back to back
    const int c = gtid + j * GT;
    my_cnt[j] = (c < G) ? __ldcg(a.part_cnt + slot0 + c) : 0;
    my_head[j] = (c < G) ? __ldcg(a.part_keys + (slot0 + c) * k) : 0ull;  // garbage if the list is empty: masked next
  }
#pragma unroll
  for (int j = 0; j < LISTS; ++j) {
    const int c = gtid + j * GT;
    if (my_cnt[j] <= 0) my_head[j] = 0ull;
    if (c < G) buf[c] = my_head[j];
  }
  if (gtid == 0) {
    *counter = 0;
    *floor_slot = 0ull;  // stays 0 when fewer than k lists are non-empty
  }
  sync();
  ICR_MSTAMP(1);
#pragma unroll
  for (int j = 0; j < LISTS; ++j) {
    if (my_head[j] != 0ull) {
      int rank = 0;
#pragma unroll 8
      for (int i = 0; i < G; ++i) rank += (buf[i] > my_head[j]) ? 1 : 0;
      if (rank == k - 1) *floor_slot = my_head[j];
    }
  }
  sync();
  const uint64_t head_floor = *floor_slot;
  sync();  // everyone has read the floor and is done with the heads in `buf`
  ICR_MSTAMP(2);
  // Lists are sorted, so the entries of a list that reach the floor form a prefix: each qualifying list (at most k
  // of them) is walked by its thread in chunks of 4 independent loads until an entry falls below the floor.
#pragma unroll
  for (int j = 0; j < LISTS; ++j) {
    if (my_head[j] != 0ull && my_head[j] >= head_floor) {
      const uint64_t* list = a.part_keys + (slot0 + gtid + j * GT) * k;
      {
        const int pos = atomicAdd(counter, 1);
        if (pos < kGemvCand) buf[pos] = my_head[j];
      }
      bool more = true;
      for (int i = 1; more && i < my_cnt[j]; i += 4) {
        uint64_t key[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) key[u] = (i + u < my_cnt[j]) ? __ldcg(list + i + u) : 0ull;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (more && key[u] != 0ull && key[u] >= head_floor) {
            const int pos = atomicAdd(counter, 1);
            if (pos < kGemvCand) buf[pos] = key[u];
          } else {
            more = false;
          }
        }
      }
    }
  }
  sync();
  ICR_MSTAMP(3);
  int n = *counter;
  const int64_t qo = static_cast<int64_t>(a.q0 + t) * k;
  if (n <= kGemvCand) {
    for (int i = gtid; i < n; i += GT) {
      const uint64_t key = buf[i];
      int rank = 0;
#pragma unroll 8
      for (int j = 0; j < n; ++j) rank += (buf[j] > key) ? 1 : 0;
      if (rank < k) {
        a.out_scores[qo + rank] = out_score<I8>(key, sm, t);
        a.out_ids[qo + rank] = static_cast<int64_t>(key_row(key)) + a.id_offset;
      }
    }
    for (int i = n + gtid; i < k; i += GT) {  // fewer than k eligible rows in the whole catalog
      a.out_scores[qo + i] = -INFINITY;
      a.out_ids[qo + i] = -1;
    }
  } else if (gtid < 32) {
    // overflow (possible only for k > 32): exact streaming merge by one warp, list by list
    uint64_t* sel = sm.sel + t * kMergeSel;
    unsigned int* hist = sm.hist + t * kHsBins;
    n = 0;
    for (int c = 0; c < G; ++c) {
      const int cnt = __ldcg(a.part_cnt + slot0 + c);
      if (cnt == 0) continue;
      if (n + cnt > kGemvCand) {
        warp_select_topk(buf, n, k, sel, hist, lane);
        for (int i = lane; i < k; i += 32) buf[i] = sel[i];
        n = k;
        __syncwarp();
      }
      for (int i = lane; i < cnt; i += 32) buf[n + i] = __ldcg(a.part_keys + (slot0 + c) * k + i);
      n += cnt;
      __syncwarp();
    }
    int kept = n;
    if (n > k) {
      warp_select_topk(buf, n, k, sel, hist, lane);
      kept = k;
    } else {
      for (int i = lane; i < n; i += 32) sel[i] = buf[i];
    }
    __syncwarp();
    const int P = next_pow2(kept < 2 ? 2 : kept);
    for (int i = kept + lane; i < P; i += 32) sel[i] = 0ull;
    warp_bitonic_sort_desc(sel, P, lane);
    for (int i = lane; i < k; i += 32) {
      const bool ok = i < kept;
      a.out_scores[qo + i] = ok ? out_score<I8>(sel[i], sm, t) : -INFINITY;
      a.out_ids[qo + i] = ok ? static_cast<int64_t>(key_row(sel[i])) + a.id_offset : -1;
    }
    __syncwarp();
  }
}

// "flat" tail of a single-query request with short lists (k <= 16, at most 256 CTAs and 10 keys per merging thread): every CTA
// leaves its k best keys sorted and zero-padded to k, so the merging CTA fetches the whole [G][k] block and the G list heads
// in ONE memory round trip of independent loads (the walk over list tails in dependent chunks was 2.7 us of a 24 us
// request). A key can only be among the k best if it reaches `floor`, the largest over the 8 warps of the k-th largest of a
// warp's 32 heads (ranked by counting over shuffles - a short loop, not a sorting network: this code starts from a cold
// instruction cache): k distinct keys >= floor exist. What survives (typically 50-100 keys) is ranked by counting, which
// yields the sorted output positions directly.
constexpr int kFlatPer = 10;  // keys per merging thread: k <= 16 at 148 CTAs
constexpr int kFlatSurv = 256;
__device__ __forceinline__ bool flat_tail(const GemvArgs& a, int nq) {
  return nq == 1 && a.k <= 16 && gridDim.x <= kGemvThreads && static_cast<int>(gridDim.x) * a.k <= kFlatPer * kGemvThreads &&
         a.out_scores != nullptr;
}

// returns false when more keys than the buffer holds reach the floor (the caller then takes the general merge)
template <int QT, bool I8, typename Sync>
__device__ __forceinline__ bool merge_query_flat(const GemvArgs& a, GemvSmem<QT>& sm, int tid, Sync sync) {
  const int k = a.k, G = gridDim.x, tot = G * k, lane = tid & 31, warp = tid >> 5;
  uint64_t* surv = sm.cand;  // [kFlatSurv]
  uint64_t* warp_floor = reinterpret_cast<uint64_t*>(sm.list_cnt);  // [8]
  int* counter = sm.list_cnt + 64;
  const int64_t slot0 = static_cast<int64_t>(a.q0) * G;
  const uint64_t* keys_g = a.part_keys + slot0 * k;
  uint64_t key[kFlatPer];
#pragma unroll
  for (int j = 0; j < kFlatPer; ++j) {
    const int e = tid + j * kGemvThreads;
    key[j] = e < tot ? __ldcg(keys_g + e) : 0ull;
  }
  uint64_t head = tid < G ? __ldcg(keys_g + static_cast<int64_t>(tid) * k) : 0ull;
  int head_rank = 0;  // among the warp's 32 heads; empty lists (0) tie and are ordered by lane, so the ranks are a permutation
#pragma unroll 4
  for (int i = 0; i < 32; ++i) {
    const uint64_t o = __shfl_sync(kFull, head, i);
    head_rank += (o > head || (o == head && i < lane)) ? 1 : 0;
  }
  if (head_rank == k - 1) warp_floor[warp] = head;  // 0 when the warp holds fewer than k non-empty lists
  if (tid == 0) *counter = 0;
  sync();
  ICR_MSTAMP(1);
  uint64_t floor_key = 0ull;
#pragma unroll
  for (int w = 0; w < kGemvWarps; ++w) floor_key = warp_floor[w] > floor_key ? warp_floor[w] : floor_key;
#pragma unroll
  for (int j = 0; j < kFlatPer; ++j) {
    if (key[j] != 0ull && key[j] >= floor_key) {
      const int pos = atomicAdd(counter, 1);
      if (pos < kFlatSurv) surv[pos] = key[j];
    }
  }
  sync();
  ICR_MSTAMP(2);
  const int n = *counter;
  if (n > kFlatSurv) {
    sync();  // everyone has read the counter before the general merge re-uses it
    return false;
  }
  const int64_t qo = static_cast<int64_t>(a.q0) * k;
  if (tid < n) {
    const uint64_t mine = surv[tid];
    const int rank = cta_key_rank(surv, n, mine);
    if (rank < k) {
      a.out_scores[qo + rank] = out_score<I8>(mine, sm, 0);
      a.out_ids[qo + rank] = static_cast<int64_t>(key_row(mine)) + a.id_offset;
    }
  }
  for (int i = n + tid; i < k; i += kGemvThreads) {  // fewer than k eligible rows in the whole catalog
    a.out_scores[qo + i] = -INFINITY;
    a.out_ids[qo + i] = -1;
  }
  ICR_MSTAMP(3);
  return true;
}

// ---- sharded request: exchange + global merge in the tail of the merging CTA ------------------------------------------------
// The shard's nq sorted lists (just written to out_scores / out_ids, global ids) go to slot `rank` of every peer's buffer
// (exchange.cu: layout and protocol), the epoch is published, and once every rank's lists are in the local buffer the `world`
// lists of each query are merged: they are sorted, so the rank of a key is its own position plus, per other list, the number
// of keys ahead of it - a binary search (7 steps for k = 100) instead of a selection. Equal keys (shards that overlap) are
// ordered by rank, so the ranks stay a permutation. No second launch, no host round trip: the request ends in this kernel.
template <int QT, bool NAMED>
__device__ __forceinline__ void peer_tail_merge(const GemvArgs& a, GemvSmem<QT>& sm, int nq, int tid) {
  const PeerTail& p = a.peer;
  const int k = a.k, W = p.world, tot = W * k;
  peer_push(p, a.out_scores, a.out_ids, static_cast<int64_t>(nq) * k, tid, kGemvThreads);
  __threadfence_system();
  compute_sync<NAMED>();
  peer_publish(p, tid);
  peer_wait(p, tid);
  compute_sync<NAMED>();
  const float* ls = reinterpret_cast<const float*>(p.peer_base[p.rank] + p.scores_off);
  const int64_t* li = reinterpret_cast<const int64_t*>(p.peer_base[p.rank] + p.ids_off);
  uint64_t* buf = sm.cand;  // QT * CAND keys, one query at a time (the launcher checked world * k against it)
  for (int t = 0; t < nq; ++t) {
    for (int i = tid; i < tot; i += kGemvThreads) {
      const int g = i / k, j = i - g * k;
      const int64_t off = (static_cast<int64_t>(g) * nq + t) * k + j;
      const int64_t id = __ldcg(li + off);
      const float sc = __ldcg(ls + off);
      buf[i] = id < 0 ? 0ull : make_key(sc, static_cast<uint32_t>(id));
    }
    compute_sync<NAMED>();
    int valid = 0;  // eligible candidates of all shards together (every thread counts: W short searches)
    for (int r = 0; r < W; ++r) {
      const uint64_t* list = buf + r * k;
      int lo = 0, hi = k;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (list[mid] != 0ull) lo = mid + 1;
        else hi = mid;
      }
      valid += lo;
    }
    for (int i = tid; i < tot; i += kGemvThreads) {
      const uint64_t key = buf[i];
      if (key == 0ull) continue;
      const int g = i / k;
      int rank = i - g * k;
      for (int r = 0; r < W; ++r) {
        if (r == g) continue;
        const uint64_t* list = buf + r * k;
        int lo = 0, hi = k;  // first position whose key does not come before `key`
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          const uint64_t o = list[mid];
          if (o > key || (o == key && r < g)) lo = mid + 1;
          else hi = mid;
        }
        rank += lo;
      }
      if (rank < k) {
        a.fin_scores[t * k + rank] = key_score(key);
        a.fin_ids[t * k + rank] = static_cast<int64_t>(key_row(key));
      }
    }
    for (int i = valid + tid; i < k; i += kGemvThreads) {  // fewer than k eligible rows in the whole catalog
      a.fin_scores[t * k + i] = -INFINITY;
      a.fin_ids[t * k + i] = -1;
    }
    compute_sync<NAMED>();
  }
}

// ---- emit this CTA's lists; the last CTA to finish merges all of them -----------------------------------
// `pending`: the caller has not run the final threshold refresh (ring kernel): it happens here, and on a flat tail the whole
// CTA ranks the (<= 256) candidates by counting and stores the k best straight into the global list - one warp ordering
// ~50 keys alone took 1.4-1.9 us per CTA, on the critical path of the slowest one.
template <int QT, bool NAMED, bool I8 = false>
__device__ __forceinline__ void emit_and_merge(const GemvArgs& a, GemvSmem<QT>& sm, int nq, bool has_rows, int tid, bool pending = false) {
  const int lane = tid & 31, warp = tid >> 5;
  const int k = a.k, G = gridDim.x;
  const bool flat = QT == 1 && flat_tail(a, nq);
  bool emitted = false;
  if (pending) {
    const int n0 = min(sm.ncand[0], GemvSmem<QT>::CAND);
    if (flat && n0 <= kGemvThreads) {
      const uint64_t mine = tid < n0 ? sm.cand[tid] : 0ull;
      const int rank = tid < n0 ? cta_key_rank(sm.cand, n0, mine) : n0;
      const int64_t slot = static_cast<int64_t>(a.q0) * G + blockIdx.x;
      const int kept = min(n0, k);
      if (tid < n0 && rank < k) a.part_keys[slot * k + rank] = mine;
      if (tid >= kept && tid < k) a.part_keys[slot * k + tid] = 0ull;
      if (tid == 0) a.part_cnt[slot] = kept;
      emitted = true;
    } else {
      refresh_thresholds<QT, NAMED>(a, sm, nq, true, 0, tid);
    }
  }
  if (!emitted) {
    for (int t = 0; t < nq; ++t) {
      const int n = has_rows ? sm.ncand[t] : 0;
      const int64_t slot = static_cast<int64_t>(a.q0 + t) * G + blockIdx.x;
      for (int i = tid; i < n; i += kGemvThreads) a.part_keys[slot * k + i] = sm.cand[t * GemvSmem<QT>::CAND + i];
      if (flat)  // the flat merge reads whole lists without their counts
        for (int i = n + tid; i < k; i += kGemvThreads) a.part_keys[slot * k + i] = 0ull;
      if (tid == 0) a.part_cnt[slot] = n;
    }
  }
  if (a.out_scores == nullptr) return;  // the caller merges the per-CTA lists with a separate select launch

  // The barrier orders the CTA's list writes before thread 0's ticket, whose release (cumulative, device scope) publishes them;
  // its acquire side orders the merging CTA's reads (after the second barrier) behind every earlier ticket. One acq_rel
  // atomic instead of fence + atomic + fence: the two stand-alone fences were ~0.4 us each on the request's critical path.
  ICR_STAMP(5);
  compute_sync<NAMED>();
  int* is_last = sm.list_cnt + 128;
  if (tid == 0) {
    unsigned int prev;
    asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(prev) : "l"(a.done_counter) : "memory");
    *is_last = (prev == static_cast<unsigned int>(G) - 1u) ? 1 : 0;
  }
  compute_sync<NAMED>();
  ICR_STAMP(6);
  if (!*is_last) return;
  ICR_MSTAMP(0);

  // Every per-CTA list is sorted, so the k best list HEADS are k distinct keys >= head_floor (the k-th largest
  // head) and no key below head_floor can be among the k best overall: typically ~2k of the G*k keys survive.
  // Ranks are found by counting (n^2 comparisons on shared-memory broadcasts, spread over the group's threads),
  // which also yields the sorted output positions directly. One query: the whole CTA works on it. Several
  // queries: one warp each, side by side.
  if (nq == 1) {
    if (!flat || !merge_query_flat<QT, I8>(a, sm, tid, [] { compute_sync<NAMED>(); }))
      merge_query<QT, kGemvThreads, 2, I8>(a, sm, 0, tid, [] { compute_sync<NAMED>(); });
  } else if (nq <= 4) {  // two warps per query, each pair on its own named barrier
    const int t = warp >> 1;
    if (t < nq) merge_query<QT, 64, 5, I8>(a, sm, t, tid & 63, [t] { ptx::named_sync(2 + t, 64); });
  } else if (warp < nq) {
    merge_query<QT, 32, 10, I8>(a, sm, warp, lane, [] { __syncwarp(); });
  }
  compute_sync<NAMED>();
  ICR_MSTAMP(4);
  if (a.peer_on) peer_tail_merge<QT, NAMED>(a, sm, nq, tid);
  if (tid == 0) {  // ready for the next launch that shares this workspace
    *a.done_counter = 0u;
    *a.chunk_counter = 0u;
  }
}

// =====================================================================================================
// direct-load kernel: RB rows per warp batch, QT queries per pass; V = RB * (QT + 1) in {16, 32}
// =====================================================================================================
template <typename T, int RB, int QT, bool XB = false>
__global__ void __launch_bounds__(kGemvThreads) gemv_topk_kernel(GemvArgs a) {
  constexpr bool I8 = std::is_same_v<T, int8_t>;  // int8 rows: fp32 queries quantised here, factors in a.cat_inv
  using Acc = std::conditional_t<I8, int, float>;
  constexpr int VEC = Elem<T>::VEC;
  constexpr int V = RB * (QT + 1);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nvec = a.D / VEC;
  const int dpad = nvec * VEC;
  GemvSmem<QT> sm(smem_raw, query_area<T>(dpad));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const T* cat = static_cast<const T*>(a.cat);
  const int nq = min(QT, a.Q - a.q0);

  if constexpr (I8) stage_queries_i8<QT>(a, sm, dpad, nq, warp, lane);
  else stage_queries<T, QT>(a, sm.qs, dpad, nq, warp, lane);
  if (tid < QT) {
    sm.ncand[tid] = 0;
    sm.tau[tid] = -INFINITY;
  }
  __syncthreads();

  const int64_t row_begin = static_cast<int64_t>(blockIdx.x) * a.rows_per_cta;
  const int64_t row_end = min(a.N, row_begin + a.rows_per_cta);
  constexpr int kBlockRows = kGemvWarps * RB * 4;  // rows between two threshold refreshes

  for (int64_t blk = row_begin; blk < row_end; blk += kBlockRows) {
    const int64_t blk_end = min(row_end, blk + kBlockRows);
    for (int64_t r0 = blk + warp * RB; r0 < blk_end; r0 += kGemvWarps * RB) {
      Acc acc[V];
#pragma unroll
      for (int i = 0; i < V; ++i) acc[i] = 0;
      for (int vb = 0; vb < nvec; vb += 32 * kGemvUnroll) {
        uint4 c[kGemvUnroll][RB];
#pragma unroll
        for (int u = 0; u < kGemvUnroll; ++u) {
          const int v = vb + u * 32 + lane;
#pragma unroll
          for (int r = 0; r < RB; ++r) {
            if (v < nvec && r0 + r < blk_end) c[u][r] = ldg_stream(cat + (r0 + r) * a.ldc + static_cast<int64_t>(v) * VEC);
            else c[u][r] = make_uint4(0, 0, 0, 0);
          }
        }
#pragma unroll
        for (int u = 0; u < kGemvUnroll; ++u) {
          const int v = vb + u * 32 + lane;
          if (v < nvec) accumulate_vector<T, RB, QT, false, QT + 1>(c[u], sm.qs, dpad, v, acc);
        }
      }
      if constexpr (I8) {
        const float f_lane = (lane < RB && r0 + lane < blk_end) ? __ldg(a.cat_inv + r0 + lane) : 0.f;
        reduce_and_append_i8<RB, QT, QT + 1, XB>(acc, a, sm, nq, r0, blk_end, lane, f_lane);
      } else {
        reduce_and_append<RB, QT, false, XB>(acc, a, sm, nq, r0, blk_end, lane);
      }
    }
    __syncthreads();
    refresh_thresholds<QT, false>(a, sm, nq, blk + kBlockRows >= row_end, kBlockRows, tid);
  }
  emit_and_merge<QT, false, I8>(a, sm, nq, row_begin < row_end, tid);
}

// =====================================================================================================
// ring kernel: producer warp + bulk async copies into a shared-memory ring, 8 consumer warps
// =====================================================================================================
template <typename T, int QT, bool NORMS = false, bool XB = false>
__global__ void __launch_bounds__(kRingThreads, 1) gemv_ring_kernel(GemvArgs a) {
  // int8 rows: fp32 queries quantised here; the row factors always come precomputed (NORMS), and for QT > 1 the unused norm
  // slot of the accumulators is kept so that V stays a power of two
  constexpr bool I8 = std::is_same_v<T, int8_t>;
  using Acc = std::conditional_t<I8, int, float>;
  static_assert(!NORMS || QT == 1 || I8, "precomputed norms: single-query kernel only (V must stay a power of two)");
  static_assert(!I8 || NORMS, "int8 rows come with their factors");
  constexpr int VEC = Elem<T>::VEC;
  constexpr int RB = (QT == 7) ? 4 : 8;  // rows reduced together (V = RB * (QT + 1) <= 32) = rows per ring slot
  constexpr int kSlabRows = RB;
  constexpr int VT = (NORMS && QT == 1) ? 1 : QT + 1;  // accumulator slots per row: the queries (+ the norm)
  constexpr int V = RB * VT;
  extern __shared__ __align__(128) unsigned char ring_smem_raw[];
  const int nvec = a.D / VEC;
  const int dpad = nvec * VEC;
  const int row_bytes = a.D * static_cast<int>(sizeof(T));
  const int slot_bytes = kSlabRows * row_bytes;
  const int NS = a.ring_slots;
  unsigned char* ring = ring_smem_raw;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + static_cast<size_t>(NS) * slot_bytes);
  uint64_t* empty_bar = full_bar + kMaxSlots;
  int64_t* slot_row = reinterpret_cast<int64_t*>(empty_bar + kMaxSlots);  // first catalog row of the slab in a slot (producer -> consumer)
  // precomputed inverse norms of the slab's rows, copied next to it (NORMS): a global load per slab from the consumer waited
  // behind the whole ring's worth of queued catalog reads - 3.7 us of an 18 us stream on a cold 76 MB catalog
  float* slot_inv = reinterpret_cast<float*>(slot_row + kMaxSlots);  // [kMaxSlots][8]
  GemvSmem<QT> sm(reinterpret_cast<unsigned char*>(slot_inv + kMaxSlots * 8), query_area<T>(dpad));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nq = min(QT, a.Q - a.q0);
  constexpr int kProducers = 4;
  const int64_t total_slabs = (a.N + kSlabRows - 1) / kSlabRows;

  ICR_STAMP(0);
  if (tid < NS) {
    ptx::mbar_init(ptx::smem_u32(&full_bar[tid]), 1);
    ptx::mbar_init(ptx::smem_u32(&empty_bar[tid]), 1);
    ptx::mbar_fence_init();
  }
  __syncthreads();  // the only CTA-wide barrier: the producer warp never joins another one
  ICR_STAMP(1);

  if (warp == kGemvWarps) {
    // ================= producer: the whole ring is in flight before the first FMA =================
    // kProducers lanes issue the copies, lane j those of local slabs j, j + kProducers, ...: with 768-byte rows a slab is
    // 6 KB and one lane's wait / expect / copy loop (~450 cycles per slab) was what held the stream at 58 % of the
    // HBM rate. NS is a multiple of 8, so the lanes own disjoint slot sets (slot = local slab % NS) and every slot still
    // has exactly one producer and one consumer; slot and parity advance incrementally (no division per slab).
    //
    // Which catalog slab a local slab is: the first static_slabs are the CTA's own block, after that each step of the four
    // lanes takes one chunk of kProducers consecutive slabs from the device-wide counter (the first dynamic chunk is the
    // CTA's index, so nothing waits for an atomic before the ring is full; lane 0 fetches the NEXT chunk before it blocks
    // on the ring). The row of a slot travels in slot_row[]; -1 = nothing in this slot, -2 = end of the stream. The end
    // markers fill one whole iteration of the eight consumer warps, so all of them leave the loop in the same iteration.
    if (lane < kProducers) {
      const unsigned int G = gridDim.x;
      const int static_steps = a.static_slabs / kProducers;
      const int64_t dyn_base = static_cast<int64_t>(G) * a.static_slabs;
      const char* cat = static_cast<const char*>(a.cat);
      int slot = lane;  // lane < kProducers <= NS
      uint32_t parity = 0;
      unsigned int nx = blockIdx.x;
      int tail = -1;  // >= 0: padding / end steps still to emit
      for (int step = 0;; ++step) {
        int64_t slab = -1;
        if (tail < 0) {
          int64_t first;
          if (step < static_steps) {
            first = static_cast<int64_t>(blockIdx.x) * a.static_slabs + static_cast<int64_t>(step) * kProducers;
          } else {
            const unsigned int cur = __shfl_sync(0xFu, nx, 0);
            first = dyn_base + static_cast<int64_t>(cur) * kProducers;
            if (lane == 0 && first < total_slabs) nx = G + atomicAdd(a.chunk_counter, 1u);
          }
          if (first >= total_slabs) tail = (step & 1) ? 3 : 2;  // odd: a step of empty slots completes the iteration first
          else if (first + lane < total_slabs) slab = first + lane;
        }
        if (tail >= 0) {
          if (tail == 0) break;
          slab = (tail == 3) ? -1 : -2;
          --tail;
        }
        ptx::mbar_wait(ptx::smem_u32(&empty_bar[slot]), parity ^ 1u);
        const uint32_t fb = ptx::smem_u32(&full_bar[slot]);
        if (slab >= 0) {
          const int64_t row0 = slab * kSlabRows;
          const int64_t rows = a.N - row0 < kSlabRows ? a.N - row0 : kSlabRows;
          const uint32_t bytes = static_cast<uint32_t>(rows) * static_cast<uint32_t>(row_bytes);
          *reinterpret_cast<volatile int64_t*>(&slot_row[slot]) = row0;
          const bool inv_too = NORMS && rows == kSlabRows;  // whole slabs only (16-byte granules); the last one loads them itself
          ptx::mbar_expect_tx(fb, bytes + (inv_too ? kSlabRows * 4u : 0u));
          ptx::bulk_g2s(ptx::smem_u32(ring + static_cast<size_t>(slot) * slot_bytes), cat + row0 * row_bytes, bytes, fb);
          if (inv_too) ptx::bulk_g2s(ptx::smem_u32(slot_inv + slot * 8), a.cat_inv + row0, kSlabRows * 4u, fb);
        } else {
          *reinterpret_cast<volatile int64_t*>(&slot_row[slot]) = slab;
          ptx::mbar_arrive(fb);  // release: the marker is visible to the consumer that acquires this phase
        }
        slot += kProducers;
        if (slot >= NS) {
          slot -= NS;
          parity ^= 1u;
        }
      }
    }
    return;
  }

  // ================= consumers =================
  if constexpr (I8) stage_queries_i8<QT>(a, sm, dpad, nq, warp, lane);
  else stage_queries<T, QT>(a, sm.qs, dpad, nq, warp, lane);
  if (tid < QT) {
    sm.ncand[tid] = 0;
    sm.tau[tid] = -INFINITY;
  }
  compute_sync<true>();
  ICR_STAMP(2);

  constexpr int kItersPerRefresh = 4;
  constexpr int kBlockRows = kItersPerRefresh * kGemvWarps * kSlabRows;
  int slot = warp;  // local slab b = it * 8 + warp lives in slot b % NS; NS is a multiple of 8: advance by 8, wrap, flip the parity
  uint32_t parity = 0;
  for (int it = 0;; ++it) {
    ptx::mbar_wait(ptx::smem_u32(&full_bar[slot]), parity);
    if (it == 0) ICR_STAMP(3);
    const int64_t r0 = *reinterpret_cast<volatile int64_t*>(&slot_row[slot]);
#ifdef ICR_TRACE
    if (r0 >= 0 && !(a.dbg & 1)) {
#else
    if (r0 >= 0) {
#endif
      const unsigned char* slab = ring + static_cast<size_t>(slot) * slot_bytes;
      constexpr int g = 0;
      Acc acc[V];
#pragma unroll
      for (int i = 0; i < V; ++i) acc[i] = 0;
      float inv_lane = 0.f;
      if (NORMS && lane < RB && r0 + lane < a.N) inv_lane = (r0 + RB <= a.N) ? slot_inv[slot * 8 + lane] : __ldg(a.cat_inv + r0 + lane);
      const int nfull = nvec & ~31;  // vectors covered by iterations in which every lane has one
      for (int v = lane; v < nfull; v += 32) {
        uint4 c[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          // rows past the end of the catalog were not copied: stale ring bytes, masked by row_limit below
          c[r] = *reinterpret_cast<const uint4*>(slab + static_cast<size_t>(g * RB + r) * row_bytes + static_cast<size_t>(v) * 16);
        }
        accumulate_vector<T, RB, QT, NORMS, VT>(c, sm.qs, dpad, v, acc);
      }
      if (nvec - nfull == 16) {
        // Half-filled last iteration (768-byte and 256-byte bf16 rows, ...): instead of idling 16 lanes, the two
        // half-warps split the ROWS of the tail — lanes 0-15 take rows 0,2,4,.., lanes 16-31 rows 1,3,5,.. — and
        // the partial sums are folded into the full-width accumulators with predicated adds (static indices).
        constexpr int HB = RB / 2;
        const int h = lane >> 4, v = nfull + (lane & 15);
        uint4 c[HB];
#pragma unroll
        for (int i = 0; i < HB; ++i)
          c[i] = *reinterpret_cast<const uint4*>(slab + static_cast<size_t>(g * RB + 2 * i + h) * row_bytes + static_cast<size_t>(v) * 16);
        Acc tacc[HB * VT];
#pragma unroll
        for (int i = 0; i < HB * VT; ++i) tacc[i] = 0;
        accumulate_vector<T, HB, QT, NORMS, VT>(c, sm.qs, dpad, v, tacc);
#pragma unroll
        for (int t = 0; t < VT; ++t)
#pragma unroll
          for (int i = 0; i < HB; ++i) {
            acc[t * RB + 2 * i] += h == 0 ? tacc[t * HB + i] : Acc(0);
            acc[t * RB + 2 * i + 1] += h == 1 ? tacc[t * HB + i] : Acc(0);
          }
      } else if (lane < nvec - nfull) {
        const int v = nfull + lane;
        uint4 c[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r)
          c[r] = *reinterpret_cast<const uint4*>(slab + static_cast<size_t>(g * RB + r) * row_bytes + static_cast<size_t>(v) * 16);
        accumulate_vector<T, RB, QT, NORMS, VT>(c, sm.qs, dpad, v, acc);
      }
      if constexpr (I8) reduce_and_append_i8<RB, QT, VT, XB>(acc, a, sm, nq, r0 + g * RB, a.N, lane, inv_lane);
      else reduce_and_append<RB, QT, NORMS, XB>(acc, a, sm, nq, r0 + g * RB, a.N, lane, inv_lane);
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&empty_bar[slot]));
    slot += kGemvWarps;
    if (slot >= NS) {
      slot -= NS;
      parity ^= 1u;
    }
    if (r0 == -2) break;  // the end markers fill one whole iteration: every warp leaves here together
    // early thresholds (as soon as a list holds 2k + 32 keys) keep the final list short: the selection at the end
    // of the stream is on the critical path of a request, the ones in the middle hide behind the ring
    if ((it + 1) % kItersPerRefresh == 0 || it == 0) {
      compute_sync<true>();
      if constexpr (QT == 1) refresh_single<true>(a, sm, kBlockRows, tid, true);
      else refresh_thresholds<QT, true>(a, sm, nq, false, kBlockRows, tid, true);
    }
  }
  compute_sync<true>();
  ICR_STAMP(4);
  emit_and_merge<QT, true, I8>(a, sm, nq, true, tid, true);
  ICR_STAMP(7);
}

// ---- host side --------------------------------------------------------------------------------------------
constexpr size_t kSmemBudget = 227 * 1024 - 1024;

template <typename T, int RB, int QT, bool XB>
static int launch_direct(const GemvArgs& a, int grid, cudaStream_t st) {
  const size_t smem = GemvSmem<QT>::bytes(query_area<T>(a.D));
  static thread_local SmemSizeCache configured;  // per device (ADVICE r1): a thread may serve several GPUs
  if (smem > 48 * 1024) {
    const int rc = ensure_dyn_smem_size(configured, gemv_topk_kernel<T, RB, QT, XB>, smem);
    if (rc) return rc;
  }
  profile_begin(kKernelGemv, 1, st);
  gemv_topk_kernel<T, RB, QT, XB><<<grid, kGemvThreads, smem, st>>>(a);
  profile_end(st);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

template <typename T, int QT>
static int ring_slots_for(int D) {
  const size_t fixed = GemvSmem<QT>::bytes(query_area<T>(D)) + 3 * kMaxSlots * sizeof(uint64_t) + kMaxSlots * 8 * sizeof(float) + 128;
  const size_t slot = static_cast<size_t>(QT == 7 ? 4 : 8) * D * sizeof(T);
  if (fixed + kGemvWarps * slot > kSmemBudget) return 0;
  const size_t n = (kSmemBudget - fixed) / slot;
  // A multiple of the consumer-warp count, so that every slot is only ever consumed by ONE warp (batch b goes to
  // warp b % 8 and slot b % NS): a slot shared by two warps would let the later one wait on a phase parity that an
  // mbarrier reports as already complete before the earlier phase has even been filled.
  // Short rows make small slabs: what has to stay constant is the BYTES in flight per SM (~190 KB keeps the HBM
  // pipe full; the 96 KB that 16 slabs of 768-byte rows amount to streamed at 54 % of the HBM rate), so the ring
  // takes as many slots as fit, in multiples of the warp count.
  size_t slots = n / kGemvWarps * kGemvWarps;
  if (slots > static_cast<size_t>(kMaxSlots)) slots = kMaxSlots;
  return static_cast<int>(slots);
}

template <typename T, int QT, bool NORMS, bool XB>
static int launch_ring(GemvArgs a, int grid, cudaStream_t st) {
  a.ring_slots = ring_slots_for<T, QT>(a.D);
  {
    // up-front share of every CTA: one ring filling, or less when the catalog is too small for that (whole chunks only)
    const int64_t total_slabs = (a.N + (QT == 7 ? 4 : 8) - 1) / (QT == 7 ? 4 : 8);
    const int64_t share = total_slabs / grid / 4 * 4;
    a.static_slabs = static_cast<int>(share < a.ring_slots ? share : a.ring_slots);
#ifdef ICR_TRACE
    a.dbg = getenv("ICR_K1_DBG") ? atoi(getenv("ICR_K1_DBG")) : 0;
    if (a.dbg & 4) a.ring_slots = 8;
    if (a.dbg & 2) a.static_slabs = static_cast<int>((total_slabs + grid - 1) / grid + 3) / 4 * 4;
#endif
  }
  const size_t smem = static_cast<size_t>(a.ring_slots) * (QT == 7 ? 4 : 8) * a.D * sizeof(T) + 3 * kMaxSlots * sizeof(uint64_t) + kMaxSlots * 8 * sizeof(float) + GemvSmem<QT>::bytes(query_area<T>(a.D)) + 128;
  static thread_local SmemSizeCache configured;  // per device
  {
    const int rc = ensure_dyn_smem_size(configured, gemv_ring_kernel<T, QT, NORMS, XB>, smem);
    if (rc) return rc;
  }
  profile_begin(kKernelGemv, 1, st);
  gemv_ring_kernel<T, QT, NORMS, XB><<<grid, kRingThreads, smem, st>>>(a);
  profile_end(st);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

static bool g_force_direct = false;  // tuning / test hook, see icr_debug_set

void gemv_force_direct(bool on) { g_force_direct = on; }

template <typename T>
static int ring_slots_q(int qt, int D) {
  return qt == 1 ? ring_slots_for<T, 1>(D) : (qt == 3 ? ring_slots_for<T, 3>(D) : ring_slots_for<T, 7>(D));
}

// contiguous rows, 16-byte aligned slabs and a ring of at least 4 slots -> bulk-copy ring kernel
static bool ring_ok(int64_t ldc, int D, int dtype, int qt) {
  if (g_force_direct || ldc != D) return false;
  int slots;
  if (dtype == ICR_F32) slots = ring_slots_q<float>(qt, D);
  else if (dtype == ICR_BF16) slots = ring_slots_q<__nv_bfloat16>(qt, D);
  else if (dtype == ICR_I8) slots = ring_slots_q<int8_t>(qt, D);
  else slots = ring_slots_q<__half>(qt, D);
  // one slot per warp (no load/compute overlap inside a warp) still wins for 1-3 queries per pass; 4-7 queries
  // (4-row slabs) want two slots per warp
  return qt == 7 ? slots >= 2 * kGemvWarps : slots >= kGemvWarps;
}

// the tail of a sharded request merges `world` lists of k keys per query in the candidate area of the merging CTA: one pass
// (Q <= 7) and world * k keys must fit
bool gemv_peer_tail_fits(int Q, int k, int world) {
  if (Q < 1 || Q > 7) return false;
  const int qt = Q == 1 ? 1 : (Q <= 3 ? 3 : 7);
  const int cap = qt == 1 ? GemvSmem<1>::CAND : (qt == 3 ? 3 * GemvSmem<3>::CAND : 7 * GemvSmem<7>::CAND);
  return world * k <= cap;
}

int gemv_grid(int64_t N) {
  // one CTA per SM for the ring kernel, two for the direct kernel; at least 64 rows per CTA. The workspace is
  // sized for the larger of the two.
  int64_t g = (N + 63) / 64;
  if (g > 148 * 2) g = 148 * 2;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

// one pass of qt (1, 3 or 7) queries
template <typename T, bool XB>
static int launch_gemv_pass(const GemvArgs& a, int qt, bool ring, int g, cudaStream_t st) {
  if (qt == 1) return ring ? (a.cat_inv ? launch_ring<T, 1, true, XB>(a, g, st) : launch_ring<T, 1, false, XB>(a, g, st)) : launch_direct<T, 8, 1, XB>(a, g, st);
  if (qt == 3) return ring ? launch_ring<T, 3, false, XB>(a, g, st) : launch_direct<T, 8, 3, XB>(a, g, st);
  return ring ? launch_ring<T, 7, false, XB>(a, g, st) : launch_direct<T, 4, 7, XB>(a, g, st);
}

// int8 rows: the ring kernels always take the precomputed factors
template <bool XB>
static int launch_gemv_pass_i8(const GemvArgs& a, int qt, bool ring, int g, cudaStream_t st) {
  if (qt == 1) return ring ? launch_ring<int8_t, 1, true, XB>(a, g, st) : launch_direct<int8_t, 8, 1, XB>(a, g, st);
  if (qt == 3) return ring ? launch_ring<int8_t, 3, true, XB>(a, g, st) : launch_direct<int8_t, 8, 3, XB>(a, g, st);
  return ring ? launch_ring<int8_t, 7, true, XB>(a, g, st) : launch_direct<int8_t, 4, 7, XB>(a, g, st);
}

// Runs ceil(Q/7) passes (one for Q <= 7). part_keys/part_cnt sized [Q][grid][k] / [Q][grid].
// xbits: per-query exclusions of these Q queries (Exclusions::bits with ld xld), or null.
int launch_gemv_topk(const void* cat, int64_t N, int64_t ldc, int D, int dtype, const void* q, int64_t ldq, int Q,
                     const uint8_t* mask, const uint32_t* xbits, int64_t xld, int k, uint64_t* part_keys, int* part_cnt, int grid, float* out_scores, int64_t* out_ids,
                     int64_t id_offset, unsigned int* done_counter, cudaStream_t st, const float* cat_inv, const PeerTail* peer, float* fin_scores,
                     int64_t* fin_ids) {
  GemvArgs a{};
  if (peer) {
    a.peer_on = 1;
    a.peer = *peer;
    a.fin_scores = fin_scores;
    a.fin_ids = fin_ids;
  }
  // the ring kernel copies the inverse norms with 16-byte bulk copies; an unaligned array falls back to norms from the rows
  // (int8 factors cannot be recovered from the codes: icr_cos_topk requires them 16-byte aligned)
  a.cat_inv = (dtype == ICR_I8 || (reinterpret_cast<uintptr_t>(cat_inv) & 15) == 0) ? cat_inv : nullptr;
  a.cat = cat;
  a.N = N;
  a.ldc = ldc;
  a.D = D;
  a.q = q;
  a.ldq = ldq;
  a.Q = Q;
  a.mask = mask;
  a.xbits = xbits;
  a.xld = xld;
  a.k = k;
  a.part_keys = part_keys;
  a.part_cnt = part_cnt;
  a.out_scores = out_scores;
  a.out_ids = out_ids;
  a.id_offset = id_offset;
  a.done_counter = done_counter;
  a.chunk_counter = done_counter + 1;
  for (int q0 = 0; q0 < Q;) {
    a.q0 = q0;
    const int rem = Q - q0;
    const int qt = rem == 1 ? 1 : (rem <= 3 ? 3 : 7);
    const bool ring = ring_ok(ldc, D, dtype, qt);
    // the ring kernel owns a whole SM (its ring is the SM's shared memory): one CTA per SM
    const int g = ring ? (grid < 148 ? grid : 148) : grid;
    a.rows_per_cta = (N + g - 1) / g;
    int rc;
    if (dtype == ICR_F32) rc = xbits ? launch_gemv_pass<float, true>(a, qt, ring, g, st) : launch_gemv_pass<float, false>(a, qt, ring, g, st);
    else if (dtype == ICR_BF16) rc = xbits ? launch_gemv_pass<__nv_bfloat16, true>(a, qt, ring, g, st) : launch_gemv_pass<__nv_bfloat16, false>(a, qt, ring, g, st);
    else if (dtype == ICR_I8) rc = xbits ? launch_gemv_pass_i8<true>(a, qt, ring, g, st) : launch_gemv_pass_i8<false>(a, qt, ring, g, st);
    else rc = xbits ? launch_gemv_pass<__half, true>(a, qt, ring, g, st) : launch_gemv_pass<__half, false>(a, qt, ring, g, st);
    if (rc != ICR_OK) return rc;
    q0 += qt;
  }
  return ICR_OK;
}

}  // namespace icr

#ifdef ICR_TRACE
extern "C" int icr_debug_read_trace(unsigned long long* out, int n) {
  return static_cast<int>(cudaMemcpyFromSymbol(out, icr::g_trace, sizeof(unsigned long long) * n));
}
extern "C" int icr_debug_read_merge_trace(unsigned long long* out) {
  return static_cast<int>(cudaMemcpyFromSymbol(out, icr::g_trace_merge, sizeof(unsigned long long) * 8));
}
#endif
