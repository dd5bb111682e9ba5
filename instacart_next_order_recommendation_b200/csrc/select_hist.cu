// Warp-per-query exact top-k selection by histogram partitioning (no full sort).
//
// The GEMM epilogue leaves, per query and phase, a few hundred candidate keys spread over a handful of
// segments, plus the k keys carried from earlier phases. Only the k largest matter, so instead of sorting
// everything (select.cu) one warp per query
//   1. gathers the keys into shared memory (all loads independent, coalesced 8-byte lanes),
//   2. bins them linearly over [min key, max key] into 256 bins (shared-memory histogram),
//   3. scans the histogram from the top to find the bin holding the k-th largest key,
//   4. moves keys above that bin straight to the output, compacts the keys of that bin in place, and
//      either sorts those few (<= 64) or repeats 2-4 on them with 256x finer bins.
// Keys are distinct 64-bit values (score bits, ~row), so ties in score are resolved exactly by row and the
// refinement always terminates. The final phase sorts the k selected keys; earlier phases only need the set
// and its minimum (the new threshold tau).
#include "common.cuh"
#include "ptx.cuh"
#include "select_args.cuh"
#include "select_warp.cuh"
#define ICR_ST_OWNER 1  // this translation unit owns the trace counters of select_lean.cuh
#include "peer.cuh"
#include "select_lean.cuh"
#include "select_finish.cuh"

namespace icr {

#ifndef ICR_HS_WARPS
#define ICR_HS_WARPS 4
#endif
constexpr int kHsWarps = ICR_HS_WARPS;  // queries per CTA, 11 KB of shared memory each (tuning: profiles/r01_notes.md)
constexpr int kHsSel = 512;       // >= 2 * ICR_MAX_K: the k results, or k + the band capacity of screened keys

// flat candidate t of query q from the dense matrix or the shard lists -> key; false if there is none
template <bool XB = false>
__device__ __forceinline__ bool front_fetch(const HistSelectArgs& a, int64_t q, int t, int count, uint64_t& key) {
  key = 0ull;
  if (t >= count) return false;
  if (a.dense) {
    if (a.excl().excluded<XB>(q, t)) return false;
    key = make_key(__ldcs(a.dense + q * a.dense_ld + t), static_cast<uint32_t>(t));
    return true;
  }
  const int g = t / a.list_k, i = t - g * a.list_k;
  const int64_t off = (static_cast<int64_t>(g) * a.Q + q) * a.list_k + i;
  const int64_t id = __ldcs(a.list_ids + off);
  if (id < 0) return false;
  key = make_key(__ldcs(a.list_scores + off), static_cast<uint32_t>(id));
  return true;
}
__device__ __forceinline__ int front_count(const HistSelectArgs& a) {
  return a.dense ? a.dense_rows : (a.list_scores ? a.list_g * a.list_k : 0);
}

struct LsSmem {
  uint32_t sc[kHsWarps][kLsCap];
  uint32_t rw[kHsWarps][kLsCap];
  uint32_t hist[kHsWarps][kHsBins];
};

// XB: the call excludes rows per query (HistSelectArgs::xbits); only the dense front end reads the bitmap
template <bool XB>
__global__ void __launch_bounds__(kHsWarps * 32, 24 / kHsWarps) select_hist_kernel(HistSelectArgs a) {
  extern __shared__ __align__(16) unsigned char hs_raw[];
  LsSmem& sm = *reinterpret_cast<LsSmem*>(hs_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * kHsWarps + warp;
  if (q >= a.Q) return;  // whole warps leave; nothing below synchronises across warps
  uint32_t* sc = sm.sc[warp];
  uint32_t* rw = sm.rw[warp];
  uint32_t* hist = sm.hist[warp];
  const int k = a.k;
  const bool screened = a.band > 0.f;
  const int kc = screened ? a.kc : k;  // keys carried between phases
  const int cap = min(a.seg_cap, a.seg_stride);
  const unsigned lt = (1u << lane) - 1u;
  float tau = -INFINITY;
  bool lost = false;  // screened keys inside the band were dropped for lack of room: exact ranking at the end
  int kept = 0;
  ICR_ST_BEGIN();

  if (a.dense && !a.carry_in && a.nseg == 0 && a.dense_rows <= kLsCap) {
    // ---- first phase of K2: the query's whole row of the dense score matrix is fetched with all 32 loads per lane in
    // flight at once; without a mask key i is simply catalog row i (no compaction) ----
    const float* row = a.dense + q * a.dense_ld;
    float f[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int t = lane + 32 * j;
      f[j] = t < a.dense_rows ? __ldcs(row + t) : 0.f;
    }
    int n = 0;
    if (a.mask == nullptr && !XB) {  // key i = catalog row i
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int t = lane + 32 * j;
        sc[t] = order_bits(f[j]);
        rw[t] = ~static_cast<uint32_t>(t);
      }
      n = a.dense_rows;
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int t = lane + 32 * j;
        const bool valid = t < a.dense_rows && !a.excl().excluded<XB>(q, t);
        const unsigned m = __ballot_sync(kFull, valid);
        if (valid) {
          const int pos = n + __popc(m & lt);
          sc[pos] = order_bits(f[j]);
          rw[pos] = ~static_cast<uint32_t>(t);
        }
        n += __popc(m);
      }
    }
    __syncwarp();
    ICR_ST_MARK(8);
    kept = ls_reduce(sc, rw, n, k, a.band, hist, &tau);
    ICR_ST_MARK(14);
  } else {
    // squeeze: reduce to the keys that can still matter (buffer nearly full, or the end); only screened keys can leave
    // more than kc - too many near-ties - and then the query is ranked exactly at the end
#define ICR_SQUEEZE(n_)                                        \
  do {                                                         \
    n_ = ls_reduce(sc, rw, n_, k, a.band, hist, &tau);         \
    if (n_ > kc) {                                             \
      lost = true;                                             \
      n_ = kc;                                                 \
    }                                                          \
  } while (0)
    int n = 0;
    if (a.carry_in) {
      n = min(a.carry_cnt_in[q], kc);
      for (int i = lane; i < n; i += 32) {
        const uint64_t key = a.carry_in[q * kc + i];
        sc[i] = static_cast<uint32_t>(key >> 32);
        rw[i] = static_cast<uint32_t>(key);
      }
    }
    if (const int count = front_count(a)) {
      for (int base = 0; base < count; base += 32 * 8) {
        if (kLsCap - n < 32 * 8) {
          __syncwarp();
          ICR_SQUEEZE(n);
        }
        uint64_t key[8];
        bool ok[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) ok[u] = front_fetch<XB>(a, q, base + u * 32 + lane, count, key[u]);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const unsigned m = __ballot_sync(kFull, ok[u]);
          if (ok[u]) {
            const int pos = n + __popc(m & lt);
            sc[pos] = static_cast<uint32_t>(key[u] >> 32);
            rw[pos] = static_cast<uint32_t>(key[u]);
          }
          n += __popc(m);
        }
      }
    }
    ICR_ST_MARK(8);
    const uint64_t* qbase = a.seg_keys + q * a.nseg * static_cast<int64_t>(a.seg_stride);
    // Segment lengths of up to 255 segments are fetched at once (independent loads) and prefix-summed in shared memory
    // (the prefix array lives in hist[], idle until the selection). The keys are then copied SEGMENT by segment, eight
    // segments per step: lanes l and l + 32 take keys l and l + 32 of each segment, so a step issues 16 independent loads per
    // lane and costs ~12 instructions per segment. (Gathering by flat key index - binary search or a per-lane segment cursor -
    // cost ~40 instructions per KEY with divergent loops: a third of the kernel's instructions.)
    int* pref = reinterpret_cast<int*>(hist);
    constexpr int kPref = kHsBins - 1;
    for (int g0 = 0; g0 < a.nseg; g0 += kPref) {
      const int ng = min(kPref, a.nseg - g0);
      bool have_pref = false, squeezed = false;
      int sgm = 0, step = 8;
      while (sgm < ng) {
        if (!have_pref) {
          __syncwarp();
#pragma unroll 4
          for (int i = lane; i < ng; i += 32) pref[i] = min(__ldg(a.seg_cnt + q * a.nseg + g0 + i), cap);
          __syncwarp();
          int carry = 0;
          for (int b0 = 0; b0 < ng; b0 += 32) {
            const int v = (b0 + lane < ng) ? pref[b0 + lane] : 0;
            int incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int u = __shfl_up_sync(kFull, incl, o);
              if (lane >= o) incl += u;
            }
            if (b0 + lane < ng) pref[b0 + lane] = carry + incl - v;
            carry += __shfl_sync(kFull, incl, 31);
          }
          if (lane == 0) pref[ng] = carry;
          have_pref = true;
          __syncwarp();
        }
        const int e = min(sgm + step, ng);
        const int p0 = pref[sgm], gtot = pref[e] - p0;
        if (n + gtot > kLsCap) {
          if (!squeezed) {  // make room: keep what can still matter (the selection overwrites the prefix array)
            ICR_SQUEEZE(n);
            have_pref = false;
            squeezed = true;
            continue;
          }
          step = 1;  // a group of (nearly full) segments larger than the buffer: one segment at a time (kc + cap <= kLsCap)
          squeezed = false;
          continue;
        }
        squeezed = false;
        uint64_t v[8][2];
        int c[8], b[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int sg = sgm + u;
          const bool ok = sg < e;
          b[u] = ok ? pref[sg] - p0 : 0;
          c[u] = ok ? pref[sg + 1] - pref[sg] : 0;
          const uint64_t* seg = qbase + static_cast<int64_t>(g0 + (ok ? sg : sgm)) * a.seg_stride;
          v[u][0] = lane < c[u] ? __ldcs(seg + lane) : 0ull;
          v[u][1] = lane + 32 < c[u] ? __ldcs(seg + lane + 32) : 0ull;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int i = lane + 32 * h;
            if (i < c[u]) {
              const uint32_t hi = static_cast<uint32_t>(v[u][h] >> 32);
              sc[n + b[u] + i] = a.raw_keys ? order_bits(__uint_as_float(hi)) : hi;
              rw[n + b[u] + i] = static_cast<uint32_t>(v[u][h]);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {  // segments longer than 64 keys: the rest, 32 at a time
          if (c[u] > 64) {
            const uint64_t* seg = qbase + static_cast<int64_t>(g0 + sgm + u) * a.seg_stride;
            for (int i = 64 + lane; i < c[u]; i += 32) {
              const uint64_t key = __ldcs(seg + i);
              const uint32_t hi = static_cast<uint32_t>(key >> 32);
              sc[n + b[u] + i] = a.raw_keys ? order_bits(__uint_as_float(hi)) : hi;
              rw[n + b[u] + i] = static_cast<uint32_t>(key);
            }
          }
        }
        n += gtot;
        sgm = e;
      }
      __syncwarp();
    }
    __syncwarp();
    ICR_ST_MARK(9);
    kept = n;
    ICR_SQUEEZE(kept);
#undef ICR_SQUEEZE
    ICR_ST_MARK(14);
  }
  if (kept > kc) {  // (first-phase path) only screened keys can leave more than kc
    lost = true;
    kept = kc;
  }
  if (screened && lost && lane == 0) a.overflow[q] = 1u;

  if (a.carry_out) {
    for (int i = lane; i < kept; i += 32) a.carry_out[q * kc + i] = (static_cast<uint64_t>(sc[i]) << 32) | rw[i];
    if (lane == 0) a.carry_cnt_out[q] = kept;
  }
  if (a.tau_out && lane == 0) a.tau_out[q] = tau;
  ICR_ST_MARK(10);
  if (a.out_scores && !screened) {  // screened keys: rescore_rank_kernel finishes from the carry
    const float scale = a.out_scale * (a.out_qscale ? a.out_qscale[q] : 1.0f);
    ls_emit_ranked(sc, rw, kept, k, scale, q, a, hist, lane);
    ICR_ST_MARK(11);
  }
}

// ---- screened keys, last step: exact re-scoring of the carried candidates and the ordered top-k -----------------------
// Its own kernel because its needs differ from the select's: no staging buffer (4 KB of keys per query, 9 KB with the
// fallback's buffer) and ~170 registers for 24 independent 16-byte loads per lane - the candidates' rows are scattered over
// the catalog, and the gather is bound by the bytes in flight, not by instructions.
constexpr int kRsCap = kLsCap;  // keys per query: the carry (<= 512), or the buffer of the whole-catalog ranking
struct RsSmem {
  uint32_t sc[kHsWarps][kRsCap];
  uint32_t rw[kHsWarps][kRsCap];
  uint32_t hist[kHsWarps][kHsBins];
};

// Tried and dropped: staging the rows with 1-D bulk async copies (cp.async.bulk, two 18 KB halves per warp, 5 warps per SM =
// 180 KB in flight). 426 us instead of 184: only 740 queries are in flight chip-wide instead of 1,776, and every catalog row
// is wanted by ~23 queries - with fewer of them running at the same time the 76 MB of fp32 rows (more than one die's share of
// the L2) are fetched from DRAM once per wave of queries (13 waves instead of 6).
#ifndef ICR_RS_MINB
#define ICR_RS_MINB 3  // CTAs per SM the kernel is compiled for: 3 -> up to 170 registers
#endif
#ifndef ICR_RS_WIDE
#define ICR_RS_WIDE 1  // 1: 8 rows x 3 vectors = 24 loads per lane in flight (D = 384); 0: 4 x 3
#endif
template <bool XB>
__global__ void __launch_bounds__(kHsWarps * 32, ICR_RS_MINB) rescore_rank_kernel(HistSelectArgs a) {
  __shared__ __align__(16) RsSmem sm;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * kHsWarps + warp;
  if (q >= a.Q) return;
  uint32_t* sc = sm.sc[warp];
  uint32_t* rw = sm.rw[warp];
  int kept;
  ICR_ST_BEGIN();
  if (a.overflow[q]) {
    kept = ls_rank_catalog<XB>(sc, rw, kRsCap, sm.hist[warp], q, a, lane);
  } else {
    kept = min(a.carry_cnt_in[q], a.kc);
    for (int i = lane; i < kept; i += 32) rw[i] = static_cast<uint32_t>(a.carry_in[q * a.kc + i]);
    __syncwarp();
    ls_rescore<(ICR_RS_WIDE != 0)>(sc, rw, kept, q, a, lane);
  }
  ICR_ST_MARK(12);
  ls_emit_ranked(sc, rw, kept, a.k, 1.0f, q, a, sm.hist[warp], lane);
  ICR_ST_MARK(13);
}

#ifdef ICR_SELECT_TRACE
}  // namespace icr
extern "C" int icr_debug_select_trace(unsigned long long* out16, int reset) {
  if (out16 && cudaMemcpyFromSymbol(out16, icr::g_sel_trace, sizeof(icr::g_sel_trace)) != cudaSuccess) return -6;
  if (reset) {
    unsigned long long z[16] = {};
    if (cudaMemcpyToSymbol(icr::g_sel_trace, z, sizeof(z)) != cudaSuccess) return -6;
  }
  return 0;
}
namespace icr {
#endif

// ---- block-per-query variant for small batches --------------------------------------------------------------
// With a few dozen queries the warp-per-query kernel leaves the GPU idle while each warp walks thousands of keys on
// its own (the swapped GEMM kernel produces one short segment per chunk and CTA: hundreds per query). Here a CTA of
// 256 threads owns a query: block-wide gather, block-wide histogram partition down to <= 1024 keys, then one warp
// finishes with warp_select_topk. Same inputs, outputs and exactness as select_hist_kernel.
constexpr int kBsThreads = 256;
constexpr int kBsCap = 6144;    // keys buffered per query at once (two buffers: 96 KB)
constexpr int kBsPref = 1024;   // segments per gather round

struct BsSmem {
  uint64_t buf[kBsCap];
  uint64_t bnd[kBsCap];
  uint64_t sel[kHsSel];
  uint64_t red[2 * (kBsThreads / 32)];
  unsigned int hist[kHsBins];
  int pref[kBsPref + 1];
  int misc[8];
};

// k largest of cur[0..n) -> sm.sel[0..k) (unordered); n > k. `cur` is sm.buf; sm.bnd is scratch.
__device__ __forceinline__ void block_select_topk(BsSmem& sm, int n, int k, int tid) {
  const int warp = tid >> 5, lane = tid & 31;
  uint64_t* cur = sm.buf;
  uint64_t* other = sm.bnd;
  int need = k, nsel = 0, len = n;
  for (;;) {
    if (len <= 1024) {
      if (warp == 0) {
        if (need == len) {
          for (int i = lane; i < len; i += 32) sm.sel[nsel + i] = cur[i];
        } else {
          warp_select_topk(cur, len, need, sm.sel + nsel, sm.hist, lane);
        }
      }
      __syncthreads();
      return;
    }
    uint64_t mn = ~0ull, mx = 0ull;
    for (int i = tid; i < len; i += kBsThreads) {
      const uint64_t key = cur[i];
      mn = key < mn ? key : mn;
      mx = key > mx ? key : mx;
    }
    mn = warp_min_u64(mn);
    mx = warp_max_u64(mx);
    if (lane == 0) {
      sm.red[warp] = mn;
      sm.red[kBsThreads / 32 + warp] = mx;
    }
    if (tid < kHsBins) sm.hist[tid] = 0u;
    __syncthreads();
    mn = sm.red[0];
    mx = sm.red[kBsThreads / 32];
#pragma unroll
    for (int w = 1; w < kBsThreads / 32; ++w) {
      mn = sm.red[w] < mn ? sm.red[w] : mn;
      mx = sm.red[kBsThreads / 32 + w] > mx ? sm.red[kBsThreads / 32 + w] : mx;
    }
    const uint64_t range = mx - mn;
    const int bits = 64 - __clzll(static_cast<long long>(range | 1ull));
    const int shift = bits > 8 ? bits - 8 : 0;
    for (int i = tid; i < len; i += kBsThreads) atomicAdd(&sm.hist[255 - static_cast<int>((cur[i] - mn) >> shift)], 1u);
    __syncthreads();
    if (warp == 0) {  // cumulative counts from the top bin: lane L owns t in [8L, 8L+8)
      unsigned int local[8], lsum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        local[j] = sm.hist[lane * 8 + j];
        lsum += local[j];
      }
      unsigned int incl = lsum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += v;
      }
      unsigned int c = incl - lsum;
      if (c < static_cast<unsigned int>(need) && static_cast<unsigned int>(need) <= incl) {
        int t_star = -1;
        unsigned int above = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (t_star < 0 && c + local[j] >= static_cast<unsigned int>(need)) {
            t_star = lane * 8 + j;
            above = c;
          }
          c += local[j];
        }
        sm.misc[0] = 255 - t_star;
        sm.misc[1] = static_cast<int>(above);
      }
      if (lane == 0) {
        sm.misc[2] = nsel;
        sm.misc[3] = 0;
      }
    }
    __syncthreads();
    const int b_star = sm.misc[0];
    for (int i = tid; i < len; i += kBsThreads) {
      const uint64_t key = cur[i];
      const int bin = static_cast<int>((key - mn) >> shift);
      if (bin > b_star) sm.sel[atomicAdd(&sm.misc[2], 1)] = key;
      else if (bin == b_star) other[atomicAdd(&sm.misc[3], 1)] = key;
    }
    __syncthreads();
    nsel = sm.misc[2];
    need -= sm.misc[1];
    const int nb = sm.misc[3];
    __syncthreads();  // misc is rewritten in the next round
    if (need == nb) {
      for (int i = tid; i < nb; i += kBsThreads) sm.sel[nsel + i] = other[i];
      __syncthreads();
      return;
    }
    uint64_t* t = cur;
    cur = other;
    other = t;
    len = nb;
    if (cur != sm.buf && len <= 1024) {  // the warp-level finish works in place on `cur`; keep it simple: move back
      for (int i = tid; i < len; i += kBsThreads) sm.buf[i] = cur[i];
      __syncthreads();
      cur = sm.buf;
      other = sm.bnd;
    }
  }
}

// keep the kk best of sm.buf[0..n) (n > kk): they end up in sm.sel[0..kk) AND sm.buf[0..kk). Returns the smallest kept key.
__device__ __forceinline__ uint64_t block_truncate(BsSmem& sm, int n, int kk, int tid) {
  block_select_topk(sm, n, kk, tid);
  uint64_t mn = ~0ull;
  for (int i = tid; i < kk; i += kBsThreads) {
    const uint64_t key = sm.sel[i];
    sm.buf[i] = key;
    mn = key < mn ? key : mn;
  }
  mn = warp_min_u64(mn);
  __syncthreads();  // sm.red is free (block_select_topk ended with a barrier)
  if ((tid & 31) == 0) sm.red[tid >> 5] = mn;
  __syncthreads();
  mn = sm.red[0];
#pragma unroll
  for (int w = 1; w < kBsThreads / 32; ++w) mn = sm.red[w] < mn ? sm.red[w] : mn;
  __syncthreads();
  return mn;
}

// Exact ranking of the whole catalog for one query by one CTA (screening-band overflow only; see warp_rank_catalog).
// Leaves the result keys in sm.sel[0..return value).
template <bool XB>
__device__ __forceinline__ int block_rank_catalog(BsSmem& sm, int64_t q, const HistSelectArgs& a, int tid) {
  const int warp = tid >> 5, lane = tid & 31;
  const float* qrow = a.rs_q + q * a.rs_ldq;
  const float qi = a.rs_qinv[q];
  const int k = a.k;
  constexpr int kWarps = kBsThreads / 32;
  int n = 0;
  uint64_t floor_key = 0ull;
  __syncthreads();
  if (tid == 0) sm.misc[4] = 0;
  __syncthreads();
  for (int64_t r0 = 0; r0 < a.rs_N; r0 += 8 * kWarps) {
    const int64_t w0 = r0 + warp * 8;
    const float* rows[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) rows[u] = a.rs_cat + min(w0 + u, a.rs_N - 1) * a.rs_ldc;
    float acc[8];
    score_rows8(qrow, rows, a.rs_D, acc, lane);
    warp_transpose_reduce<8>(acc, lane);
    const int64_t row = w0 + (lane >> 2);
    bool ok = (lane & 3) == 0 && row < a.rs_N && !a.excl().excluded<XB>(q, row);
    uint64_t key = 0ull;
    if (ok) {
      key = make_key(acc[0] * qi * __ldg(a.rs_cinv + row), static_cast<uint32_t>(row));
      ok = key > floor_key;
    }
    if (ok) sm.buf[atomicAdd(&sm.misc[4], 1)] = key;
    __syncthreads();
    n = sm.misc[4];
    if (n > kBsCap - 8 * kWarps) {
      floor_key = block_truncate(sm, n, k, tid);
      n = k;
      if (tid == 0) sm.misc[4] = k;
    }
    __syncthreads();
  }
  if (n > k) {
    block_select_topk(sm, n, k, tid);
    return k;
  }
  for (int i = tid; i < n; i += kBsThreads) sm.sel[i] = sm.buf[i];
  __syncthreads();
  return n;
}

template <bool XB>
__global__ void __launch_bounds__(kBsThreads) select_block_kernel(HistSelectArgs a) {
  extern __shared__ __align__(16) unsigned char bs_raw[];
  BsSmem& sm = *reinterpret_cast<BsSmem*>(bs_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t q = blockIdx.x;
  const int k = a.k;
  const int kc = a.band > 0.f ? a.kc : k;  // keys kept between phases
  const int cap = min(a.seg_cap, a.seg_stride);
  int n = 0;
  uint64_t cut_max = 0ull;  // largest "smallest kept key" of any truncation (meaningful in thread 0's view after block_truncate)
  if (a.carry_in) {
    n = min(a.carry_cnt_in[q], kc);
    for (int i = tid; i < n; i += kBsThreads) sm.buf[i] = a.carry_in[q * kc + i];
  }
  if (const int count = front_count(a)) {
    const unsigned lt = (1u << lane) - 1u;
    __syncthreads();
    for (int base = 0; base < count; base += kBsThreads * 4) {
      if (kBsCap - n < kBsThreads * 4) {
        cut_max = max(cut_max, block_truncate(sm, n, kc, tid));
        n = kc;
      }
      if (tid == 0) sm.misc[4] = n;
      __syncthreads();
      uint64_t key[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) ok[u] = front_fetch<XB>(a, q, base + u * kBsThreads + tid, count, key[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const unsigned m = __ballot_sync(kFull, ok[u]);
        int wbase = 0;
        if (lane == 0 && m) wbase = atomicAdd(&sm.misc[4], __popc(m));
        wbase = __shfl_sync(kFull, wbase, 0);
        if (ok[u]) sm.buf[wbase + __popc(m & lt)] = key[u];
      }
      __syncthreads();
      n = sm.misc[4];
      __syncthreads();
    }
  }
  const uint64_t* qbase = a.seg_keys + q * a.nseg * static_cast<int64_t>(a.seg_stride);
  for (int g0 = 0; g0 < a.nseg; g0 += kBsPref) {
    const int ng = min(kBsPref, a.nseg - g0);
    int top = 1;
    while (top * 2 <= ng) top *= 2;
    __syncthreads();
    for (int i = tid; i < ng; i += kBsThreads) sm.pref[i] = min(__ldg(a.seg_cnt + q * a.nseg + g0 + i), cap);
    __syncthreads();
    if (warp == 0) {
      int carry = 0;
      for (int b0 = 0; b0 < ng; b0 += 32) {
        const int v = (b0 + lane < ng) ? sm.pref[b0 + lane] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int u = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += u;
        }
        if (b0 + lane < ng) sm.pref[b0 + lane] = carry + incl - v;
        carry += __shfl_sync(kFull, incl, 31);
      }
      if (lane == 0) sm.pref[ng] = carry;
    }
    __syncthreads();
    const int total = sm.pref[ng];
    int done = 0;
    while (done < total) {
      if (kBsCap - n < kBsThreads) {  // buffer full: keep the kc best and go on
        cut_max = max(cut_max, block_truncate(sm, n, kc, tid));
        n = kc;
      }
      const int take = min(kBsCap - n, total - done);
      for (int i0 = 0; i0 < take; i0 += kBsThreads * 4) {
        uint64_t v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * kBsThreads + tid;
          v[u] = 0ull;
          if (i < take) {
            const int idx = done + i;
            int sg = 0;
            for (int step = top; step > 0; step >>= 1)
              if (sg + step < ng && sm.pref[sg + step] <= idx) sg += step;
            v[u] = __ldcs(qbase + static_cast<int64_t>(g0 + sg) * a.seg_stride + (idx - sm.pref[sg]));
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * kBsThreads + tid;
          if (i < take) sm.buf[n + i] = a.raw_keys ? canonical_from_raw(v[u]) : v[u];
        }
      }
      n += take;
      done += take;
      __syncthreads();
    }
  }
  __syncthreads();
  int kept = n;
  if (a.band > 0.f) {
    // ---- screened keys (see select_hist_kernel) ---------------------------------------------------------------------
    if (n > kc) {
      cut_max = max(cut_max, block_truncate(sm, n, kc, tid));  // the kc best in sm.sel and sm.buf[0..kc)
      kept = kc;
    } else {
      for (int i = tid; i < n; i += kBsThreads) sm.sel[i] = sm.buf[i];
      __syncthreads();
    }
    if (warp == 0) {
      float tau = -INFINITY;
      int m = kept;
      if (kept >= k) {
        uint64_t kth = ~0ull;
        if (kept > k) {
          warp_select_topk(sm.buf, kept, k, sm.buf + kHsSel, sm.hist, lane);
          for (int i = lane; i < k; i += 32) kth = sm.buf[kHsSel + i] < kth ? sm.buf[kHsSel + i] : kth;
        } else {
          for (int i = lane; i < k; i += 32) kth = sm.sel[i] < kth ? sm.sel[i] : kth;
        }
        kth = warp_min_u64(kth);
        tau = key_score(kth) - a.band;
        const uint64_t t_key = static_cast<uint64_t>(order_bits(tau)) << 32;
        if (cut_max >= t_key && lane == 0) a.overflow[q] = 1u;
        const unsigned lt = (1u << lane) - 1u;
        m = 0;
        for (int b0 = 0; b0 < kept; b0 += 32) {
          const int i = b0 + lane;
          const uint64_t key = i < kept ? sm.sel[i] : 0ull;
          const bool keep = i < kept && key >= t_key;
          const unsigned mk = __ballot_sync(kFull, keep);
          if (keep) sm.sel[m + __popc(mk & lt)] = key;
          m += __popc(mk);
        }
      }
      if (lane == 0) {
        sm.misc[5] = m;
        if (a.tau_out) a.tau_out[q] = tau;
      }
    }
    __syncthreads();
    kept = sm.misc[5];
    if (a.carry_out) {
      for (int i = tid; i < kept; i += kBsThreads) a.carry_out[q * kc + i] = sm.sel[i];
      if (tid == 0) a.carry_cnt_out[q] = kept;
    }
    if (a.out_scores) {
      if (a.overflow[q]) kept = block_rank_catalog<XB>(sm, q, a, tid);
      else warp_rescore(sm.sel, kept, warp, kBsThreads / 32, q, a, lane);
      __syncthreads();
      for (int i = tid; i < kept; i += kBsThreads) {  // kept <= kHsSel: rank counting, as below
        const uint64_t key = sm.sel[i];
        int rank = 0;
        for (int j = 0; j < kept; ++j) rank += (sm.sel[j] > key || (sm.sel[j] == key && j < i)) ? 1 : 0;  // the index orders exact duplicates
        if (rank < k) {
          a.out_scores[q * k + rank] = key_score(key);
          a.out_ids[q * k + rank] = static_cast<int64_t>(key_row(key)) + a.id_offset;
        }
      }
      for (int i = kept + tid; i < k; i += kBsThreads) {
        a.out_scores[q * k + i] = -INFINITY;
        a.out_ids[q * k + i] = -1;
      }
    }
    return;
  }
  if (n > k) {
    block_select_topk(sm, n, k, tid);
    kept = k;
  } else {
    for (int i = tid; i < n; i += kBsThreads) sm.sel[i] = sm.buf[i];
    __syncthreads();
  }
  if (a.carry_out) {
    for (int i = tid; i < kept; i += kBsThreads) a.carry_out[q * k + i] = sm.sel[i];
    if (tid == 0) a.carry_cnt_out[q] = kept;
  }
  // every thread ranks one selected key (kept <= 256): the minimum is the new threshold, the ranks the output order
  const bool mine = tid < kept;
  const uint64_t key = mine ? sm.sel[tid] : 0ull;
  int rank = 0;
  if (mine)
    for (int j = 0; j < kept; ++j) rank += (sm.sel[j] > key || (sm.sel[j] == key && j < tid)) ? 1 : 0;  // the index orders exact duplicates
  if (a.tau_out && mine && rank == kept - 1) a.tau_out[q] = (kept >= k) ? key_score(key) : -INFINITY;
  if (a.tau_out && kept == 0 && tid == 0) a.tau_out[q] = -INFINITY;
  if (a.out_scores) {
    const float scale = a.out_scale * (a.out_qscale ? a.out_qscale[q] : 1.0f);
    if (mine) {
      a.out_scores[q * k + rank] = key_score(key) * scale;
      a.out_ids[q * k + rank] = static_cast<int64_t>(key_row(key)) + a.id_offset;
    }
    for (int i = kept + tid; i < k; i += kBsThreads) {
      a.out_scores[q * k + i] = -INFINITY;
      a.out_ids[q * k + i] = -1;
    }
  }
}


// ---- K4f: shard-candidate exchange and merge in ONE kernel ----------------------------------------------------------------
// Every rank calls it with its own [Q][k] (score, global id) lists. The CTAs push them into slot `rank` of every peer's
// buffer over NVLink (protocol and layout: exchange.cu), the last CTA to finish its part publishes the epoch to the peers, and
// then EVERY CTA waits until the local buffer holds all ranks' lists of this epoch and merges its share of the queries from
// it, one warp per query (the list path of the select above). One launch instead of push + merge, and no host round trip
// between the two; every CTA waits, so the grid must be co-resident (sized from the occupancy, launched cooperatively).
struct PeerMergeArgs {
  const float* scores;  // this rank's candidates, [Q][k]
  const int64_t* ids;
  PeerTail peer;
  HistSelectArgs sel;  // list_scores / list_ids = the local buffer's slot of this epoch, list_g = world
};

__global__ void __launch_bounds__(kHsWarps * 32, 24 / kHsWarps) peer_exchange_merge_kernel(const PeerMergeArgs m) {
  extern __shared__ __align__(16) unsigned char hs_raw[];
  LsSmem& sm = *reinterpret_cast<LsSmem*>(hs_raw);
  __shared__ bool is_last;
  const PeerTail& p = m.peer;
  const HistSelectArgs& a = m.sel;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  peer_push(p, m.scores, m.ids, a.Q * a.list_k, static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<size_t>(gridDim.x) * blockDim.x);
  __threadfence_system();
  __syncthreads();
  unsigned int* ticket = reinterpret_cast<unsigned int*>(p.peer_base[p.rank] + kPeerTicketOff);
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (is_last) {
    __threadfence_system();
    peer_publish(p, threadIdx.x);
    if (threadIdx.x == 0) *ticket = 0u;  // every CTA of this launch has taken its ticket
  }
  peer_wait(p, threadIdx.x);
  __syncthreads();

  uint32_t* sc = sm.sc[warp];
  uint32_t* rw = sm.rw[warp];
  uint32_t* hist = sm.hist[warp];
  const int k = a.k, count = a.list_g * a.list_k;
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t q = static_cast<int64_t>(blockIdx.x) * kHsWarps + warp; q < a.Q; q += static_cast<int64_t>(gridDim.x) * kHsWarps) {
    int n = 0;
    float tau;
    for (int base = 0; base < count; base += 32 * 8) {
      if (kLsCap - n < 32 * 8) {
        __syncwarp();
        n = min(ls_reduce(sc, rw, n, k, 0.f, hist, &tau), k);
      }
      uint64_t key[8];
      bool ok[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) ok[u] = front_fetch(a, q, base + u * 32 + lane, count, key[u]);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const unsigned mk = __ballot_sync(kFull, ok[u]);
        if (ok[u]) {
          const int pos = n + __popc(mk & lt);
          sc[pos] = static_cast<uint32_t>(key[u] >> 32);
          rw[pos] = static_cast<uint32_t>(key[u]);
        }
        n += __popc(mk);
      }
    }
    __syncwarp();
    const int kept = min(ls_reduce(sc, rw, n, k, 0.f, hist, &tau), k);  // identical (score, id) pairs can leave more than k: any k of them
    ls_emit_ranked(sc, rw, kept, k, 1.0f, q, a, hist, lane);
    __syncwarp();
  }
}

int launch_peer_exchange_merge(const float* scores, const int64_t* ids, int64_t Q, int k, const PeerTail& peer, float* os, int64_t* oi,
                               cudaStream_t st) {
  if (Q == 0) return ICR_OK;
  static thread_local SmemAttrCache cache;  // per device
  int rc = ensure_dyn_smem(cache, peer_exchange_merge_kernel, sizeof(LsSmem));
  if (rc) return rc;
  static thread_local int resident[64] = {};  // co-resident CTAs per device
  int dev = 0;
  ICR_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (resident[dev] == 0) {
    int per_sm = 0, sms = 0;
    ICR_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, peer_exchange_merge_kernel, kHsWarps * 32, sizeof(LsSmem)));
    ICR_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    resident[dev] = per_sm * sms > 0 ? per_sm * sms : 1;
  }
  PeerMergeArgs m{};
  m.scores = scores;
  m.ids = ids;
  m.peer = peer;
  m.sel.k = k;
  m.sel.Q = Q;
  m.sel.out_scores = os;
  m.sel.out_ids = oi;
  m.sel.out_scale = 1.0f;
  m.sel.list_scores = reinterpret_cast<const float*>(peer.peer_base[peer.rank] + peer.scores_off);
  m.sel.list_ids = reinterpret_cast<const int64_t*>(peer.peer_base[peer.rank] + peer.ids_off);
  m.sel.list_g = peer.world;
  m.sel.list_k = k;
  int64_t grid = (Q + kHsWarps - 1) / kHsWarps;
  if (grid > resident[dev]) grid = resident[dev];
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(kHsWarps * 32);
  cfg.dynamicSmemBytes = sizeof(LsSmem);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ICR_CUDA_CHECK(cudaLaunchKernelEx(&cfg, peer_exchange_merge_kernel, m));
  count_launch();
  return ICR_OK;
}

// K4: merge of G shard lists of k_in (score, id) pairs per query, [G][Q][k_in] -> sorted top k_out per query
int launch_merge_lists(const float* cs, const int64_t* ci, int64_t Q, int G, int k_in, int k_out, float* os, int64_t* oi,
                       cudaStream_t st) {
  if (Q == 0) return ICR_OK;
  HistSelectArgs a{};
  a.k = k_out;
  a.Q = Q;
  a.out_scores = os;
  a.out_ids = oi;
  a.out_scale = 1.0f;
  a.list_scores = cs;
  a.list_ids = ci;
  a.list_g = G;
  a.list_k = k_in;
  return run_select(a, Q, st);
}

// batches of up to this many queries take the block-per-query select, larger ones a warp per query
constexpr int64_t kSelectBlockMaxQ = 512;

template <bool XB>
static int run_select_impl(const HistSelectArgs& a, int64_t Q, cudaStream_t st) {
  static thread_local SmemAttrCache warp_cache, block_cache;  // per device
  int rc = ensure_dyn_smem(warp_cache, select_hist_kernel<XB>, sizeof(LsSmem));
  if (rc) return rc;
  if (Q <= kSelectBlockMaxQ) {
    if ((rc = ensure_dyn_smem(block_cache, select_block_kernel<XB>, sizeof(BsSmem)))) return rc;
    select_block_kernel<XB><<<static_cast<unsigned>(Q), kBsThreads, sizeof(BsSmem), st>>>(a);
    ICR_LAUNCH_CHECK();
    return ICR_OK;
  }
  const unsigned grid = static_cast<unsigned>((Q + kHsWarps - 1) / kHsWarps);
  select_hist_kernel<XB><<<grid, kHsWarps * 32, sizeof(LsSmem), st>>>(a);
  ICR_LAUNCH_CHECK();
  if (a.band > 0.f && a.out_scores) {
    // screened keys: the select left the candidates within the band in carry_out; re-score them exactly and rank
    if (!a.carry_out || !a.carry_cnt_out) {
      set_error("select: the final phase of a screened search needs a carry buffer for its candidates");
      return ICR_ERR_ARG;
    }
    HistSelectArgs r = a;
    r.carry_in = a.carry_out;
    r.carry_cnt_in = a.carry_cnt_out;
    rescore_rank_kernel<XB><<<grid, kHsWarps * 32, 0, st>>>(r);
    ICR_LAUNCH_CHECK();
  }
  return ICR_OK;
}

int run_select(const HistSelectArgs& a, int64_t Q, cudaStream_t st) {
  return a.xbits ? run_select_impl<true>(a, Q, st) : run_select_impl<false>(a, Q, st);
}

}  // namespace icr
