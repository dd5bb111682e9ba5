// K2: cosine scoring as a tcgen05 / TMEM tensor-core GEMM whose epilogue never writes scores:
// it filters them against a per-query threshold and appends the few survivors as candidate keys.
//
//   S[256 queries, 256 catalog rows] = A[256, K] * B[256, K]^T      per CTA PAIR (cta_group::2, fp32 accumulate)
//
//  * Two CTAs of a cluster (one TPC) work as a pair: each owns 128 queries (its half of M) and loads only
//    HALF of every catalog tile (128 of the 256 rows); one elected thread of the leader CTA issues
//    tcgen05.mma.cta_group::2 (M=256, N=256, K=16) which reads both CTAs' shared memory and writes a
//    128-lane x 256-column fp32 accumulator into EACH CTA's TMEM. Halving the B traffic per SM is what
//    takes this loop off the L2-bandwidth limit (profiles/r01_notes.md).
//  * Operands arrive by TMA (cp.async.bulk.tensor.2d.cta_group::2, 128-byte swizzle) into a shared-memory
//    ring guarded by mbarriers (transaction bytes of both CTAs land on the leader's "full" barrier;
//    tcgen05.commit multicasts "empty" to both). Two TMEM accumulators let the epilogue of tile i overlap
//    the MMAs of tile i+1.
//  * Queries sit on the M axis: after tcgen05.ld every epilogue thread owns ONE query (its TMEM lane) and
//    sees 32 catalog scores per load. A score survives if it beats the thread's threshold tau — the k-th
//    best score of the catalog rows already ranked in earlier phases (an exact lower bound of the final
//    k-th score). The append is predicated, not branched: ~8 instructions per score.
//  * The catalog is walked in phases of geometrically growing row ranges; between phases the select kernel
//    (select.cu) folds the survivors into the running top-k and publishes the new tau. If a thread's
//    candidate segment fills up anyway (adversarially ordered catalogs), its warp sorts the segment in
//    shared memory, keeps the k best and raises that thread's tau: exact for any input.
//  * fp32 catalogs are swept with ONE MMA term on fp16 screening planes: rows are L2-normalised, scaled by 2^8 and
//    rounded to fp16 (prep.cu). Screened scores are within a known band of the exact ones (select_args.cuh), so the
//    thresholds sit that band below the k-th best, and the last select re-scores the rows inside it exactly in fp32
//    (rescore_rank_kernel). bf16 and fp16 catalogs take one MMA term on the raw rows and multiply by the two inverse
//    norms in the epilogue.
//  * The dense K2' path (DENSE, icr_cos_sim_dense) keeps fp32 parity for fp32 inputs: rows are split into fp16
//    hi + lo planes, and hi*hi + hi*lo + lo*hi accumulated in fp32 reproduces the fp32 dot product to ~1e-6 relative
//    (profiles/r01_split_precision.txt). Each pipeline stage holds the four plane tiles of one 64-wide K block, so no
//    plane is fetched twice.
//
// Replaces cos_sim [Q,N] -> torch.topk(100) -> Python heap of sentence-transformers'
// InformationRetrievalEvaluator (built at reference src/training/train_sbert.py:197-202) and the
// cos_sim -> np.argsort loops of src/baselines/content_based.py:54-63.
#include "select_args.cuh"
#include "select_lean.cuh"
#include "select_finish.cuh"
#include "tc.cuh"  // BM, BN, BK, tile geometry, PTX wrappers, tensor maps

namespace icr {

constexpr int kRingBytes = 192 * 1024;
constexpr int kSegCapMax = 512;      // candidate keys per (query, chunk, column half) segment: 256 for k <= 128, else 512
// warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warp 3 idle, warps 4.. epilogue. With 8 epilogue warps (two per
// scheduler) warps 4-7 filter accumulator columns 0-127 and warps 8-11 columns 128-255 of the same 128 queries.
// Epilogue warps per CTA, in sets of four (a warp may only read the TMEM lane quarter warp_id % 4); with two sets each
// filters half of a tile's columns. Measured (profiles/r01_notes.md): the three-term kernel is tensor-bound and does
// best with four (fewer segments for the select); the one-term kernels are epilogue-latency-bound and want two warps
// per scheduler.
#ifndef ICR_EPI_WARPS_F32
#define ICR_EPI_WARPS_F32 4
#endif
#ifndef ICR_EPI_WARPS_BF16
#define ICR_EPI_WARPS_BF16 8
#endif
__host__ __device__ constexpr int epi_warps(int terms) { return terms == 3 ? ICR_EPI_WARPS_F32 : ICR_EPI_WARPS_BF16; }
constexpr int kEpiWarps = 8;  // upper bound, for buffer sizes
constexpr int kEpiCols = BN;
constexpr int kGemmThreads = 128 + kEpiWarps * 32;
constexpr int kTmemCols = 512;      // two 256-column fp32 accumulators
constexpr int kMaxStages = 6;
constexpr int kAStatMaxKB = 6;       // A-stationary variant: up to 6 K blocks (D <= 384) of queries stay resident

struct GemmArgs {
  int Q, N;
  int k;
  int kb_per_term;  // 64-element K blocks of the embedding dimension
  int plane_stride; // element offset of the lo plane inside a row (plane path)
  int tile_begin, tile_end;  // catalog tiles [begin, end) of this phase
  int chunks;                // balanced tile ranges, see chunk_first_tile
  int qblocks;               // blocks of 256 queries
  float acc_scale;           // 2^-16 for the plane path, 1 for bf16 / fp16 rows
  const float* tau;          // [Q]
  const float* qinv;         // [Q]  (bf16 / fp16 rows) or null
  const float* cinv;         // [N]  (bf16 / fp16 rows) or null
  const uint8_t* mask;       // [N] or null
  uint64_t* cand;            // [Q][chunks * 2][seg_cap]   (segment = query x chunk x column half)
  int* cand_cnt;             // [Q][chunks * 2]
  int seg_cap;
  float* dense_out;          // K2' mode: write every score to dense_out[q * dense_ld + row] instead of filtering
  int64_t dense_ld;
  uint64_t* compact_scratch; // [gridDim.x][kEpiWarps][kSegCapMax] global scratch of the (rare) in-kernel compaction
  int qpad;                  // swapped kernel: queries rounded up to a multiple of 32 (the MMA's N)
  int dense_raw;             // dense mode stores raw-unit scores (no per-query factor): first phase of the top-k path
  // swapped kernel, single-launch mode: the thresholds are bootstrapped inside the kernel (see gemm_swap_kernel)
  int boot;                  // 0 = off, else the number of bootstrap tiles per chunk (its first tiles, streamed twice)
  float* gmax;               // [qpad][4 * gridDim.x] group maxima of the bootstrap tiles
  unsigned int* gsync;       // [3] grid-barrier counters, zero before the launch
  int fuse_select;           // swapped kernel, single-launch mode: the select runs in the kernel's tail (swap_select_tail)
  int boot_coarse;           // K2 single-launch mode: ONE maximum per (bootstrap tile, column group) instead of one per 32 scores
  float band;                // screened scores (MODE 2): tau already sits `band` below the k-th best; 0 = exact scores
  unsigned int* overflow;    // [Q] screened scores: set when a segment cannot be cut back without losing keys of the band
  const uint32_t* xbits;     // per-query exclusions (Exclusions::bits, ld = xld): read by the XB instantiations only
  int64_t xld;
};

// chunk c of a phase covers tiles [first(c), first(c+1)): sizes differ by at most one tile
__device__ __forceinline__ int chunk_first_tile(const GemmArgs& g, int c) {
  return g.tile_begin + static_cast<int>(static_cast<int64_t>(c) * (g.tile_end - g.tile_begin) / g.chunks);
}

__device__ __forceinline__ uint32_t order_bits_canonical(float s) {  // s must not be -0.0
  const uint32_t b = __float_as_uint(s);
  return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}
// segment ("raw") key <-> ordered key
__device__ __forceinline__ uint64_t canonical_key(uint64_t raw) {
  const float f = __uint_as_float(static_cast<uint32_t>(raw >> 32)) + 0.0f;  // -0.0 -> +0.0: equal scores, equal keys
  return (static_cast<uint64_t>(order_bits_canonical(f)) << 32) | (raw & 0xFFFFFFFFull);
}
__device__ __forceinline__ uint64_t raw_key(uint64_t key) {
  return (static_cast<uint64_t>(__float_as_uint(unorder_bits(static_cast<uint32_t>(key >> 32)))) << 32) | (key & 0xFFFFFFFFull);
}

struct SegState {
  uint64_t* seg;    // this thread's candidate segment (global)
  int cnt;
  uint32_t tau_ob;  // order_bits of the threshold: a score survives iff order_bits(score) > tau_ob
};

// Any lane whose segment could overflow during the next 32 scores gets it compacted by the whole warp.
// `scratch` is global memory (L2-resident): this path only runs when the running threshold fails to prune, e.g. a
// catalog sorted by similarity to the query, so it trades speed for 16-32 KB of shared memory.
__device__ __forceinline__ void compact_full_segments(SegState& s, uint64_t* scratch, int cap, int k, int lane, float band,
                                                      unsigned int* overflow, int q_lane0) {
  unsigned need = __ballot_sync(kFull, s.cnt > cap - 32);
  while (need) {
    const int L = __ffs(need) - 1;
    need &= need - 1;
    uint64_t* seg = reinterpret_cast<uint64_t*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(s.seg), L));
    const int n = __shfl_sync(kFull, s.cnt, L);
    __syncwarp();
    const int P = cap <= 256 ? 256 : kSegCapMax;  // power of two for the sorting network
    for (int i = lane; i < P; i += 32) scratch[i] = (i < n) ? canonical_key(__ldcg(seg + i)) : 0ull;
    warp_bitonic_sort_desc(scratch, P, lane);
    int kept = n < k ? n : k;
    uint32_t t_new = (n >= k) ? static_cast<uint32_t>(scratch[k - 1] >> 32) : 0u;
    if (band > 0.f && n >= k) {
      // screened scores: every key within `band` of the segment's k-th best may still belong to the exact top-k
      t_new = order_bits(unorder_bits(t_new) - band);
      const uint64_t t_key = static_cast<uint64_t>(t_new) << 32;
      int c = 0;
      for (int i = lane; i < n; i += 32) c += (scratch[i] >= t_key) ? 1 : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
      kept = c;
      if (kept > cap - 64) {  // too many near-ties to carry: this query is ranked exactly over the whole catalog at the end
        if (lane == 0) overflow[q_lane0 + L] = 1u;
        kept = k;
      }
    }
    for (int i = lane; i < kept; i += 32) seg[i] = raw_key(scratch[i]);
    if (lane == L) {
      s.cnt = kept;
      s.tau_ob = max(s.tau_ob, t_new);
    }
    __syncwarp();
  }
}

// predicated append of a raw key (score bits, ~row): no branch, so a warp whose lanes disagree pays nothing extra
__device__ __forceinline__ void append_if(SegState& s, float sc, float tau_f, uint32_t nrow) {
  uint32_t inc;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.gt.f32 p, %2, %3;\n"
      "@p st.global.v2.u32 [%1], {%4, %5};\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(inc)
      : "l"(s.seg + s.cnt), "f"(sc), "f"(tau_f), "r"(nrow), "r"(__float_as_uint(sc))
      : "memory");
  s.cnt += static_cast<int>(inc);
}

// MODE 5 (int8 rows): the accumulators are exact s32 dot products; converted once after each TMEM load (__int2float_rn, the
// rounding K1 applies too), every consumer below reads fp32 bits as for the other modes
template <int MODE>
__device__ __forceinline__ void acc_to_f32(uint32_t (&r)[32]) {
  if constexpr (MODE == 5) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__int2float_rn(static_cast<int>(r[j])));
  }
}
// the one-term MMA of a mode: kind::i8 for int8 rows, kind::f16 (f16 / bf16 operands) otherwise
template <int MODE>
__device__ __forceinline__ void umma_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (MODE == 5) umma_i8_pair(d_tmem, adesc, bdesc, idesc, accumulate);
  else umma_f16_pair(d_tmem, adesc, bdesc, idesc, accumulate);
}
// instruction descriptor bits 4-12: D format (1 = F32, 2 = S32) and the A / B formats (kind::f16: 0 = F16, 1 = BF16;
// kind::i8: 1 = signed 8-bit)
template <int MODE>
__host__ __device__ constexpr uint32_t idesc_formats() {
  return MODE == 5 ? ((2u << 4) | (1u << 7) | (1u << 10)) : ((1u << 4) | ((MODE == 1 ? 1u : 0u) << 7) | ((MODE == 1 ? 1u : 0u) << 10));
}

// Per-query exclusions (XB kernels): the accumulators of the rows that this thread's bitmap word `w` excludes become -inf
// before any filter, maximum or bound sees them. Every filter is a strict ">", which never admits -inf (not even against
// the first phase's tau = -inf), so the fast paths stay as they are; a warp whose 32 words are all zero skips the selects.
__device__ __forceinline__ void exclude32(uint32_t (&r)[32], uint32_t w) {
  if (__any_sync(kFull, w != 0u)) {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = ((w >> j) & 1u) ? 0xff800000u : r[j];
  }
}

// Bootstrap threshold from the k-th largest group maximum `ks` (order bits): one ulp below it, minus the screening band.
// XB kernels: a query with fewer than k eligible groups (rows excluded) has a k-th maximum of -inf, and its threshold
// is -inf rather than the NaN one ulp below -inf would give (which no score passes).
// A k-th maximum of exactly 0 (a zero query: every key is 0) steps over the image of -0.0, which no score maps to and which
// no zero score would pass, to the largest negative float.
template <bool XB>
__device__ __forceinline__ float boot_tau(uint32_t ks, float band) {
  if (XB && ks <= order_bits(-INFINITY)) return -INFINITY;
  const uint32_t below = ks == 0x80000000u ? 0x7ffffffeu : ks - 1u;
  return unorder_bits(ks > 1u ? below : ks) - band;
}

// Filter 32 accumulator columns (catalog rows rbase .. rbase+31) of this thread's query.
// Segments hold RAW keys: (accumulator-unit score bits, ~row); the select kernel turns them into ordered keys when
// it gathers them. Scores are in "raw" units - the accumulator itself (plane path) or accumulator * catalog inverse
// norm (bf16 path); the per-query positive factor (2^-16, or the query's inverse norm) does not change the order
// within a query and is applied once, to the k final scores, by the select kernel.
// cmax / cmin: largest / smallest catalog inverse norm of these 32 rows (SCALED: the bf16 and fp16 row paths).
template <bool SCALED>
__device__ __forceinline__ void filter32(const uint32_t (&r)[32], SegState& s, const float* cinv32, float cmax, float cmin, int rbase,
                                         bool fast, int N, const uint8_t* mask) {
  const float tau_f = unorder_bits(s.tau_ob);  // NaN for dead lanes: every comparison below is false
  if (fast) {
    // Survivors are rare once the threshold has converged (k / rows-seen per score), so the 32 accumulators are
    // screened together: one max tree + one warp vote (~1.1 instructions per score; the bf16 path bounds the scaled
    // maximum with the block's extreme inverse norms instead of scaling 32 scores). Only when SOME lane of the warp
    // has a survivor are the scores scaled and appended - with positions from a prefix sum over the 32 predicates,
    // so the 32 predicated stores are independent of each other (no serial counter chain).
    float m[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) m[j] = fmaxf(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
#pragma unroll
    for (int w = 8; w > 0; w >>= 1)
#pragma unroll
      for (int j = 0; j < w; ++j) m[j] = fmaxf(m[j], m[j + w]);
    const float bound = SCALED ? fmaxf(m[0] * cmax, m[0] * cmin) : m[0];
    if (__any_sync(kFull, bound > tau_f)) {
      float sc[32];
      if (SCALED) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 ci = *reinterpret_cast<const float4*>(cinv32 + j);
          sc[j] = __uint_as_float(r[j]) * ci.x;
          sc[j + 1] = __uint_as_float(r[j + 1]) * ci.y;
          sc[j + 2] = __uint_as_float(r[j + 2]) * ci.z;
          sc[j + 3] = __uint_as_float(r[j + 3]) * ci.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) sc[j] = __uint_as_float(r[j]);
      }
      int off[33];
      off[0] = s.cnt;
#pragma unroll
      for (int g = 0; g < 4; ++g) {  // prefix sums: depth 3 inside a group of 8, one add between groups
        int inc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) inc[j] = (sc[g * 8 + j] > tau_f) ? 1 : 0;
        const int s01 = inc[0] + inc[1], s23 = inc[2] + inc[3], s45 = inc[4] + inc[5], s67 = inc[6] + inc[7];
        const int b = off[g * 8];
        off[g * 8 + 1] = b + inc[0];
        off[g * 8 + 2] = b + s01;
        off[g * 8 + 3] = b + s01 + inc[2];
        const int b4 = b + s01 + s23;
        off[g * 8 + 4] = b4;
        off[g * 8 + 5] = b4 + inc[4];
        off[g * 8 + 6] = b4 + s45;
        off[g * 8 + 7] = b4 + s45 + inc[6];
        off[g * 8 + 8] = b4 + s45 + s67;
      }
      const uint32_t nrow0 = ~static_cast<uint32_t>(rbase);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.gt.f32 p, %1, %2;\n"
            "@p st.global.v2.u32 [%0], {%3, %4};\n"
            "}\n" ::"l"(s.seg + off[j]),
            "f"(sc[j]), "f"(tau_f), "r"(nrow0 - j), "r"(__float_as_uint(sc[j]))
            : "memory");
      }
      s.cnt = off[32];
    }
    // Tried in round 2 and dropped: appending quad by quad (one more vote per quad, four chained predicated appends in the
    // quads that have a survivor) instead of 32-wide prefix sums. At C2's survivor density nearly every quad is taken and the
    // chained appends are latency-bound: the 163-tile launch went from 272 to 286 us. Likewise parking the block in shared memory
    // and letting every lane walk only the quads whose maximum beats its threshold (~140 instructions instead of ~275, but a
    // per-lane loop of dependent ffs -> LDS -> compare -> store steps): 421 -> 519 us for the single-launch C2 sweep. The
    // prefix-sum form below has more instructions and all of them independent, which is what this epilogue needs.
  } else {
    // last (partial) tile of the catalog, or an exclusion mask: rows are checked one by one
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int row = rbase + j;
      if (row < N && !(mask && mask[row])) {
        const float sc = SCALED ? __uint_as_float(r[j]) * cinv32[j] : __uint_as_float(r[j]);
        append_if(s, sc, tau_f, ~static_cast<uint32_t>(row));
      }
    }
  }
}

// K2' (dense cos_sim): same main loop, the epilogue scales and stores all 32 scores of a batch to this query's row.
template <bool SCALED>
__device__ __forceinline__ void dense_store32(const uint32_t (&r)[32], float* out_row, float qscale, const float* cinv32, int ncols,
                                              bool vec_ok) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = SCALED ? __uint_as_float(r[j]) * qscale * cinv32[j] : __uint_as_float(r[j]) * qscale;
  if (ncols >= 32 && vec_ok) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(out_row + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < ncols) out_row[j] = v[j];
  }
}

constexpr int kK2BootCap = 640;  // block maxima per query the in-kernel bootstrap of K2 can rank

// Barrier over the epilogue warps of every CTA of the grid (all CTAs co-resident: one per SM, grid <= 148): named barrier 2
// joins this CTA's epilogue warps, one thread counts the CTA in and waits. Traps after ~2 s instead of hanging the GPU.
__device__ __forceinline__ void k2_grid_barrier(unsigned int* counter, unsigned int ctas, int ewarp, int ewarps) {
  asm volatile("bar.sync 2, %0;" ::"r"(ewarps * 32) : "memory");
  if (ewarp == 0 && (threadIdx.x & 31) == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= ctas) break;
      __nanosleep(100);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 2000000000ull) __trap();
    }
    __threadfence();
  }
  asm volatile("bar.sync 2, %0;" ::"r"(ewarps * 32) : "memory");
}

// MODE = 3: fp16 hi/lo planes, three MMA terms (fp32 parity of every score): instantiated for the dense K2' path only;
// MODE = 1: raw bf16 rows, one term, inverse norms applied in the epilogue;
// MODE = 2: one fp16 plane of the normalised fp32 rows, one term: SCREENING scores (select_args.cuh), the survivors
//           of the whole sweep are re-scored exactly by the last select;
// MODE = 4: raw fp16 rows, one term, inverse norms applied in the epilogue: MODE 1 with fp16 operands. fp16 x fp16
//           products are exact in fp32, so the scores are those of fp32 arithmetic on the fp16 values: no band, no
//           re-scoring.
// MODE = 5: int8 rows (ICR_I8), one kind::i8 term (K = 32 codes = 32 bytes, the bytes of one f16 MMA step, so the tiles,
//           swizzle and descriptor advance are those of a 16-bit matrix of D / 2 columns); the s32 accumulators become
//           fp32 once (acc_to_f32) and are scaled by the catalog's factors: keys fp32(S) * f_row, exactly K1's.
// SCALED (MODE 1, 4 and 5): exact scores, multiplied by the catalog's inverse norms (int8: factors) in the epilogue.
// ASTAT (bf16, D <= 384): the work item's 128 query rows stay resident in shared memory for all of its catalog
// tiles ("A-stationary"), so the ring streams catalog tiles only: 31 instead of 62 B/cycle/SM of L2 traffic,
// which is the difference between L2-bound and tensor-bound for one-term MMAs (profiles/r01_notes.md).
// XB (filtering kernels only): the call excludes rows per query (GemmArgs::xbits).
template <int MODE, bool ASTAT, bool DENSE, bool XB = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_topk_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const GemmArgs g) {
  constexpr int TERMS = (MODE == 3) ? 3 : 1;
  static_assert(!ASTAT || TERMS == 1, "A-stationary is a one-term variant");
  static_assert(!XB || !DENSE, "dense scores are filtered by the select");
  constexpr bool SCALED = (MODE == 1 || MODE == 4 || MODE == 5);  // exact scores scaled by the catalog's inverse norms in the epilogue
  constexpr int EW = epi_warps(TERMS), EH = EW / 4, ECOLS = BN / EH;  // epilogue warps, column groups, columns per warp
  constexpr int kStageTiles = ASTAT ? 1 : ((TERMS == 3) ? 4 : 2);  // B | A_hi A_lo B_hi B_lo | A B
  constexpr int kStageBytes = kStageTiles * kTileBytes;
  constexpr int kAResidentBytes = ASTAT ? kAStatMaxKB * kTileBytes : 0;
  constexpr int kStages = (kRingBytes - kAResidentBytes) / kStageBytes;  // 6 | 3 | 6
  static_assert(kStages <= kMaxStages, "barrier array too small");

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // 128-byte-swizzled tiles need 1024-byte alignment; the allocation carries 1 KB of slack for this.
  // Both CTAs of the pair compute the same offset (same kernel, same static layout).
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* a_resident = smem;                    // ASTAT: kb-th K block of the queries at kb * kTileBytes
  unsigned char* stage_base = smem + kAResidentBytes;
  float* cinv_all = reinterpret_cast<float*>(smem + kRingBytes);                    // 8 warps x 128 floats
  uint64_t* bars = reinterpret_cast<uint64_t*>(cinv_all + EW * ECOLS);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tfull_bar = bars + 2 * kMaxStages;
  uint64_t* tempty_bar = bars + 2 * kMaxStages + 2;
  uint64_t* afull_bar = bars + 2 * kMaxStages + 4;   // ASTAT: resident queries loaded
  uint64_t* aempty_bar = bars + 2 * kMaxStages + 5;  // ASTAT: every MMA of the work item has read them
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 6);
  uint32_t* boot_s = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 7);  // [EW][kK2BootCap + kHsBins], boot mode only

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader of the pair
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int KB = g.kb_per_term;
  const int items = g.qblocks * g.chunks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);   // leader's arrive.expect_tx; data of both CTAs arrives as tx bytes
      mbar_init(smem_u32(&empty_bar[s]), 1);  // one multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&tfull_bar[a]), 1);   // one multicast tcgen05.commit
      mbar_init(smem_u32(&tempty_bar[a]), 2 * EW);  // the epilogue warps of both CTAs (used in the leader only)
    }
    mbar_init(smem_u32(afull_bar), 1);
    mbar_init(smem_u32(aempty_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_b) : "memory");
  }
  if (warp == 2) tmem_alloc_pair(smem_u32(tmem_ptr), kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // peer barriers are initialised and its TMEM allocated before anything crosses CTAs
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0 && lane == 0) {
    // ================= TMA producer (both CTAs; each loads its own queries and its half of B) =================
    int stage = 0;
    uint32_t phase = 0, a_phase = 0;
    // boot mode (g.boot > 0): pass 0 streams only the first g.boot tiles of every work item (the epilogue takes group maxima
    // from them and the thresholds are computed in the kernel), pass 1 the whole items
    for (int pass = g.boot > 0 ? 0 : 1; pass < 2; ++pass)
    for (int w = pair; w < items; w += npairs) {
      const int chunk = w / g.qblocks, qb = w - chunk * g.qblocks;
      const int t0 = chunk_first_tile(g, chunk), t1 = pass == 0 ? t0 + g.boot : chunk_first_tile(g, chunk + 1);
      const int qrow = qb * (2 * BM) + static_cast<int>(rank) * BM;
      if (ASTAT) {
        // the previous work item's MMAs must have finished reading the resident queries
        mbar_wait(smem_u32(aempty_bar), a_phase ^ 1);
        const uint32_t ab = smem_u32(afull_bar);
        if (rank == 0) mbar_expect_tx(ab, 2 * KB * kTileBytes);
        for (int kb = 0; kb < KB; ++kb) tma_load_2d_pair(smem_u32(a_resident + kb * kTileBytes), &tma_a, kb * BK, qrow, ab);
        a_phase ^= 1;
      }
      for (int tile = t0; tile < t1; ++tile) {
        const int crow = tile * BN + static_cast<int>(rank) * BNH;
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full_bar[stage]);
          if (rank == 0) mbar_expect_tx(fb, 2 * kStageBytes);
          const uint32_t sa = smem_u32(stage_base + stage * kStageBytes);
          if (ASTAT) {
            tma_load_2d_pair(sa, &tma_b, kb * BK, crow, fb);
          } else if (TERMS == 3) {
            tma_load_2d_pair(sa, &tma_a, kb * BK, qrow, fb);
            tma_load_2d_pair(sa + kTileBytes, &tma_a, g.plane_stride + kb * BK, qrow, fb);
            tma_load_2d_pair(sa + 2 * kTileBytes, &tma_b, kb * BK, crow, fb);
            tma_load_2d_pair(sa + 3 * kTileBytes, &tma_b, g.plane_stride + kb * BK, crow, fb);
          } else {
            tma_load_2d_pair(sa, &tma_a, kb * BK, qrow, fb);
            tma_load_2d_pair(sa + kTileBytes, &tma_b, kb * BK, crow, fb);
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ================= MMA issuer (leader CTA only) =================
    // The WHOLE warp walks the loop and one elected lane issues: descriptors, barrier addresses and loop state are
    // then warp-uniform values (uniform registers), not per-thread values that must be moved into uniform
    // registers before every tcgen05 instruction. With a single-lane branch that traffic made the issue loop,
    // not the tensor pipe, the limit of the one-term kernels (4 MMAs per stage): profiles/r01_notes.md.
    // instruction descriptor: D=f32, A/B = f16 or bf16, K-major both, N=256, M=256 (two CTAs x 128)
    const uint32_t idesc = idesc_formats<MODE>() | (static_cast<uint32_t>(BN >> 3) << 17) | (static_cast<uint32_t>((2 * BM) >> 4) << 24);
    // descriptors differ only in the 16-byte-unit start address (shared memory is < 256 KB: no carry out of the field)
    const uint64_t a_res0 = smem_desc_sw128(smem_u32(a_resident));
    const uint64_t st0 = smem_desc_sw128(smem_u32(stage_base));
    constexpr uint64_t kTileUnits = kTileBytes >> 4, kStageUnits = kStageBytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0, a_phase = 0;
    for (int pass = g.boot > 0 ? 0 : 1; pass < 2; ++pass)
    for (int w = pair; w < items; w += npairs) {
      const int chunk = w / g.qblocks;
      const int t0 = chunk_first_tile(g, chunk), t1 = pass == 0 ? t0 + g.boot : chunk_first_tile(g, chunk + 1);
      if (ASTAT) {
        mbar_wait(smem_u32(afull_bar), a_phase);
        tc_fence_after();
        a_phase ^= 1;
      }
      for (int tile = t0; tile < t1; ++tile) {
        mbar_wait(smem_u32(&tempty_bar[acc]), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint64_t sd = st0 + static_cast<uint64_t>(stage) * kStageUnits;
          if (elect_one()) {
            if (ASTAT) {
              const uint64_t adesc = a_res0 + static_cast<uint64_t>(kb) * kTileUnits, bdesc = sd;
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4) {
                // advancing 16 elements (32 bytes) along K inside the swizzle atom = +2 in the 16-byte address field
                const uint64_t o = static_cast<uint64_t>(k4 * 2);
                umma_pair<MODE>(d_tmem, adesc + o, bdesc + o, idesc, (kb | k4) != 0 ? 1u : 0u);
              }
            } else if (TERMS == 3) {
              const uint64_t a_hi = sd, a_lo = sd + kTileUnits, b_hi = sd + 2 * kTileUnits, b_lo = sd + 3 * kTileUnits;
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4) {
                const uint64_t o = static_cast<uint64_t>(k4 * 2);
                umma_f16_pair(d_tmem, a_hi + o, b_hi + o, idesc, (kb | k4) != 0 ? 1u : 0u);
                umma_f16_pair(d_tmem, a_hi + o, b_lo + o, idesc, 1u);
                umma_f16_pair(d_tmem, a_lo + o, b_hi + o, idesc, 1u);
              }
            } else {
              const uint64_t adesc = sd, bdesc = sd + kTileUnits;
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4) {
                const uint64_t o = static_cast<uint64_t>(k4 * 2);
                umma_pair<MODE>(d_tmem, adesc + o, bdesc + o, idesc, (kb | k4) != 0 ? 1u : 0u);
              }
            }
            umma_commit_pair(smem_u32(&empty_bar[stage]));  // frees the stage in both CTAs when these MMAs have read it
            if (kb == KB - 1) umma_commit_pair(smem_u32(&tfull_bar[acc]));  // accumulator complete -> both epilogues
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
      if (ASTAT) {
        if (elect_one()) umma_commit_pair(smem_u32(aempty_bar));  // resident queries may be overwritten in both CTAs
        __syncwarp();
      }
    }
  } else if (warp >= 4 && warp < 4 + EW) {
    // ================= epilogue: threshold filter, one query per thread =================
    const int ew = (warp - 4) & 3;   // TMEM lane quarter this warp may read (hardware rule: warp id % 4)
    const int half = (warp - 4) >> 2;  // which 128 accumulator columns of every tile this warp filters
    uint64_t* scratch = g.compact_scratch + (static_cast<int64_t>(blockIdx.x) * EW + (warp - 4)) * kSegCapMax;
    float* cinv_s = cinv_all + (warp - 4) * ECOLS;
    const int cap = g.seg_cap;
    int acc = 0;
    uint32_t acc_phase = 0;
    // XB: this query's bitmap words, one per 32-row block of the ECOLS columns a tile gives this warp. The next tile's words
    // are loaded while the current tile is filtered (xw) and staged at the start of each tile in this warp's share of the
    // bootstrap's ranking buffer (idle outside the ranking): xs[u * 32 + lane] = word of block u.
    uint32_t* xs = boot_s + (warp - 4) * (kK2BootCap + kHsBins);
    uint32_t xw[ECOLS / 32];
    auto load_words = [&](int q, bool live, int row0) {
      if constexpr (XB) {
#pragma unroll
        for (int u = 0; u < ECOLS / 32; ++u)
          xw[u] = (live && row0 + u * 32 < g.N) ? Exclusions{nullptr, g.xbits, g.xld}.word(q, (row0 >> 5) + u) : 0u;
      }
    };
    auto stage_words = [&]() {
      if constexpr (XB) {
#pragma unroll
        for (int u = 0; u < ECOLS / 32; ++u) xs[u * 32 + lane] = xw[u];
        __syncwarp();
      }
    };
    if (!DENSE && g.boot > 0) {
      // ---- single-launch mode, pass 0: group maxima of the first g.boot tiles of every work item ----------------------
      // A thread owns one query and sees 32 catalog scores per TMEM load: the maximum of each such block is the score of
      // a distinct row, so the k-th largest of a query's block maxima (chunks * g.boot * 8 of them) is a lower bound of its
      // final k-th best score. The whole grid meets at a barrier, every epilogue warp ranks the maxima of its share of the
      // queries and publishes tau, a second barrier, and pass 1 filters the whole catalog against those thresholds: the
      // dense first phase, one sparse phase and the two selects between them (a third of the C2 step) are gone.
      // boot_coarse: one maximum per tile and column group (ECOLS rows) - a large catalog streamed by ONE query block would
      // otherwise bring more maxima per query than the in-kernel ranking holds (C4 shard, Q = 128: 148 chunks x 8 per tile)
      const int per_tile = g.boot_coarse ? 1 : (ECOLS / 32);
      const int gstride = g.chunks * g.boot * EH * per_tile;
      for (int w = pair; w < items; w += npairs) {
        const int chunk = w / g.qblocks, qb = w - chunk * g.qblocks;
        const int t0 = chunk_first_tile(g, chunk);
        const int q = qb * (2 * BM) + static_cast<int>(rank) * BM + ew * 32 + lane;
        const bool live = q < g.Q;
        float* gq = g.gmax + static_cast<int64_t>(live ? q : 0) * gstride + (chunk * g.boot * EH + half) * per_tile;
        load_words(q, live, t0 * BN + half * ECOLS);
        for (int bt = 0; bt < g.boot; ++bt) {
          float m_tile = -INFINITY;
          const int row0 = (t0 + bt) * BN + half * ECOLS;
          stage_words();
          if (bt + 1 < g.boot) load_words(q, live, row0 + BN);
          if (SCALED) {
            __syncwarp();
#pragma unroll
            for (int u = 0; u < ECOLS / 32; ++u) {
              const int i = u * 32 + lane;
              cinv_s[i] = (row0 + i < g.N) ? __ldg(g.cinv + row0 + i) : 0.f;
            }
            __syncwarp();
          }
          mbar_wait(smem_u32(&tfull_bar[acc]), acc_phase);
          tc_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(acc * BN + half * ECOLS);
          const bool plain = (row0 + ECOLS <= g.N) && (g.mask == nullptr);
#pragma unroll 1
          for (int cb = 0; cb < ECOLS / 32; ++cb) {
            uint32_t r[32];
            tmem_ld32(taddr + cb * 32, r);
            tmem_ld_wait(r);
            acc_to_f32<MODE>(r);
            if (XB) exclude32(r, xs[cb * 32 + lane]);  // an excluded row must not be a block's maximum: the k-th maximum stays a lower bound
            float m = -INFINITY;
            if (plain) {
#pragma unroll
              for (int j = 0; j < 32; ++j) m = fmaxf(m, SCALED ? __uint_as_float(r[j]) * cinv_s[cb * 32 + j] : __uint_as_float(r[j]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int row = row0 + cb * 32 + j;
                if (row < g.N && !(g.mask && g.mask[row]))
                  m = fmaxf(m, SCALED ? __uint_as_float(r[j]) * cinv_s[cb * 32 + j] : __uint_as_float(r[j]));
              }
            }
            m_tile = fmaxf(m_tile, m);
            if (live && !g.boot_coarse) gq[bt * (EH * (ECOLS / 32)) + cb] = m;
          }
          if (live && g.boot_coarse) gq[bt * EH] = m_tile;
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(smem_u32(&tempty_bar[acc]), 0);
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
      }
      k2_grid_barrier(g.gsync, gridDim.x, warp - 4, EW);
      uint32_t* bsc = boot_s + (warp - 4) * (kK2BootCap + kHsBins);
      uint32_t* bhist = bsc + kK2BootCap;
      const int nwarps = static_cast<int>(gridDim.x) * EW;
      for (int j = blockIdx.x * EW + (warp - 4); j < g.Q; j += nwarps) {
        for (int i = lane; i < gstride; i += 32) bsc[i] = order_bits(__ldcg(g.gmax + static_cast<int64_t>(j) * gstride + i));
        __syncwarp();
        uint32_t ks, kr;
        ls_kth(bsc, bsc, gstride, g.k, bhist, lane, ks, kr);  // only the k-th VALUE matters: the tie-break word is the value itself
        // the filter is a strict ">" and the bootstrap rows are filtered again in pass 1: one ulp below the k-th maximum
        if (lane == 0) const_cast<float*>(g.tau)[j] = boot_tau<XB>(ks, g.band);
        __syncwarp();
      }
      k2_grid_barrier(g.gsync + 1, gridDim.x, warp - 4, EW);
    }
    for (int w = pair; w < items; w += npairs) {
      const int chunk = w / g.qblocks, qb = w - chunk * g.qblocks;
      const int t0 = chunk_first_tile(g, chunk), t1 = chunk_first_tile(g, chunk + 1);
      const int q = qb * (2 * BM) + static_cast<int>(rank) * BM + ew * 32 + lane;
      const bool live = q < g.Q;
      const int64_t seg_index = (static_cast<int64_t>(live ? q : 0) * g.chunks + chunk) * EH + half;
      SegState s;
      s.seg = g.cand + seg_index * cap;
      s.cnt = 0;
      constexpr bool dense = DENSE;  // compile-time: the top-k instantiation keeps its register budget
      s.tau_ob = (live && !dense) ? order_bits(__ldcg(g.tau + q)) : 0xFFFFFFFFu;
      float* out_q = dense ? g.dense_out + static_cast<int64_t>(live ? q : 0) * g.dense_ld : nullptr;
      load_words(q, live, t0 * BN + half * ECOLS);
      const float qscale = dense ? (g.dense_raw ? 1.0f : g.acc_scale * ((SCALED && live) ? g.qinv[q] : 1.0f)) : 0.f;
      const bool vec_ok = dense && (g.dense_ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.dense_out) & 15) == 0);
      for (int tile = t0; tile < t1; ++tile) {
        const int row0 = tile * BN + half * ECOLS;
        stage_words();
        if (tile + 1 < t1) load_words(q, live, row0 + BN);
        float cmax_l = 1.f, cmin_l = 1.f;  // lane u: extremes of the inverse norms of 32-row block u
        if (SCALED) {
          // stage this warp's catalog inverse norms once per tile (read back as shared-memory broadcasts), with
          // the extremes of every 32-row block for the screening bound
          static_assert(ECOLS / 32 <= 32, "one lane per 32-row block");
          __syncwarp();
#pragma unroll
          for (int u = 0; u < ECOLS / 32; ++u) {
            const int i = u * 32 + lane;
            const float ci = (row0 + i < g.N) ? __ldg(g.cinv + row0 + i) : 0.f;
            cinv_s[i] = ci;
            const float mx = warp_max(ci), mn = -warp_max(-ci);
            if (lane == u) {
              cmax_l = mx;
              cmin_l = mn;
            }
          }
          __syncwarp();
        }
        mbar_wait(smem_u32(&tfull_bar[acc]), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(acc * BN + half * ECOLS);
        const bool fast = (row0 + ECOLS <= g.N) && (g.mask == nullptr);
        uint32_t ra[32], rb[32];
        tmem_ld32(taddr, ra);
#pragma unroll 1
        for (int cb = 0; cb < ECOLS / 32; cb += 2) {
          // the next 32 columns are in flight while the current 32 are filtered
          tmem_ld_wait(ra);
          acc_to_f32<MODE>(ra);
          tmem_ld32(taddr + (cb + 1) * 32, rb);
          if (dense) {
            if (live) dense_store32<SCALED>(ra, out_q + row0 + cb * 32, qscale, cinv_s + cb * 32, g.N - (row0 + cb * 32), vec_ok);
          } else {
            compact_full_segments(s, scratch, cap, g.k, lane, g.band, g.overflow, q - lane);
            if (XB) exclude32(ra, xs[cb * 32 + lane]);
            filter32<SCALED>(ra, s, cinv_s + cb * 32, __shfl_sync(kFull, cmax_l, cb), __shfl_sync(kFull, cmin_l, cb), row0 + cb * 32, fast,
                           g.N, g.mask);
          }
          tmem_ld_wait(rb);
          acc_to_f32<MODE>(rb);
          if (cb + 2 < ECOLS / 32) tmem_ld32(taddr + (cb + 2) * 32, ra);
          if (dense) {
            if (live) dense_store32<SCALED>(rb, out_q + row0 + (cb + 1) * 32, qscale, cinv_s + (cb + 1) * 32, g.N - (row0 + (cb + 1) * 32), vec_ok);
          } else {
            compact_full_segments(s, scratch, cap, g.k, lane, g.band, g.overflow, q - lane);
            if (XB) exclude32(rb, xs[(cb + 1) * 32 + lane]);
            filter32<SCALED>(rb, s, cinv_s + (cb + 1) * 32, __shfl_sync(kFull, cmax_l, cb + 1), __shfl_sync(kFull, cmin_l, cb + 1),
                           row0 + (cb + 1) * 32, fast, g.N, g.mask);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(smem_u32(&tempty_bar[acc]), 0);  // accumulator drained: tell the leader's MMA thread
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
      if (live && !dense) g.cand_cnt[seg_index] = s.cnt;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA may exit (or free TMEM) while its peer can still reach it
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}


// =====================================================================================================
// K2s: "swapped" kernel for small query batches (Q <= 256 and the queries fit in ~half of shared memory).
//
// Below the ridge (Q < ~256) the path is HBM-bound, but with queries on the MMA's M axis every catalog tile costs
// a full M=256 MMA whatever Q is, and half of the ring re-streams the same queries from L2. Here the roles are
// swapped: the CATALOG tile is the M operand (256 rows per pair, 128 per CTA), the QUERIES are the N operand
// (N = Q rounded up to 32), loaded once and resident in shared memory. MMA time scales with Q, the whole ring
// carries catalog bytes only, and the epilogue sees 128 x Q scores per CTA and tile instead of 128 x 256.
// Epilogue thread = catalog row (TMEM lane); per-query thresholds live in shared memory; survivors go to the
// (query, chunk, CTA) segment through a shared-memory counter. Same phases, segments and select as K2.
// =====================================================================================================
constexpr int kBootCap = 640;  // group maxima per query the in-kernel bootstrap can rank (4 per CTA: up to 160 CTAs)
constexpr size_t kSwapBootBytes = 4 * (2 * kBootCap + kHsBins) * sizeof(uint32_t);  // per epilogue warp: values, indices, histogram
constexpr int kSwapMaxStages = 12;
constexpr int kSwapThreads = 256;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 3 idle, 4-7 epilogue
// Resident queries may take 64 KB of the ring's shared memory: that leaves >= 8 catalog stages, and a 5-stage ring loses to K2 on
// catalogs that stream from HBM (C4 shard, Q = 128: 0.49 against 0.46 ms, profiles/r02_notes.md). A catalog small enough to
// sit in L2 does not need the deep ring: up to 100 KB there, which takes the single-launch path to Q = 256 at D = 384.
constexpr int kSwapResidentMax = 64 * 1024;
constexpr int kSwapResidentMaxSmallCatalog = 100 * 1024;
constexpr int64_t kSmallCatalogBytes = 96ll << 20;

__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// Barrier over the epilogue warps of EVERY CTA of the grid (all co-resident: one CTA per SM, grid <= 148). The counter is
// zero before the launch and counts CTAs. A barrier that cannot complete (a CTA that never became resident) traps after
// ~2 s instead of hanging the GPU.
__device__ __forceinline__ void swap_grid_barrier(unsigned int* counter, unsigned int ctas, int et) {
  epi_sync();  // this CTA's global writes are done
  if (et == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= ctas) break;
      __nanosleep(100);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 2000000000ull) __trap();
    }
    __threadfence();
  }
  epi_sync();
}

// ---- single-launch mode, last step: the select runs in the tail of the GEMM kernel ----------------------------------------
// After a third grid barrier every query's survivors are complete, and CTA b finishes queries b, b + gridDim.x, ... with its
// four epilogue warps: the lengths of the query's 2 * chunks segments (one per CTA: many segments, a handful of keys) are
// prefix-summed, the keys gathered by flat index (every thread finds its keys' segments by binary search: all loads of a
// round independent), ranked by counting - which orders them - and cut at the k-th key (minus the screening band); screened
// keys are re-scored exactly (8 rows per warp and batch, every load of a batch in flight at once), ranked again and written
// out. What select_block_kernel and its launch did in 13-23 us beside a 29 us GEMM on the 49,688-row catalog.
//
// The code is deliberately SMALL: it runs once per launch on a few CTAs, so its instructions come from L2 or DRAM, ~0.1 us
// per 128-byte line - a first version that called the histogram selection (ls_reduce, ~4,000 instructions) per query was
// slower than the separate select launch. The host only asks for the tail when the expected number of survivors per query is
// far below its buffer; a query that exceeds it anyway (or whose screening band overflows) takes the general routines on
// warp 0 - slow, exact.
constexpr int kTailSegs = 160;   // 2 * chunks <= 160 segments per query (5 per lane of warp 0)
constexpr int kTailCap = 1024;   // keys of one query ranked in shared memory (two 8 KB arrays in the idle operand ring)

// rank (0 = largest) of `mine` among the distinct keys[0..n): one small loop shared by both rankings of the tail
__device__ __noinline__ int tail_rank(const uint64_t* keys, int n, uint64_t mine) {
  int rank = 0;
#pragma unroll 4
  for (int j = 0; j < n; ++j) rank += (keys[j] > mine) ? 1 : 0;
  return rank;
}

// dst[rank of src[i]] = src[i] for all i < n, by the 128 epilogue threads (n <= kTailCap)
__device__ __forceinline__ void tail_order(const uint64_t* src, uint64_t* dst, int n, int et) {
  for (int i = et; i < n; i += 128) {
    const uint64_t key = src[i];
    dst[tail_rank(src, n, key)] = key;
  }
  epi_sync();
}

template <bool XB>
__device__ __noinline__ void swap_select_tail(unsigned int* gsync, const HistSelectArgs& a, unsigned char* ring, int ew, int lane, int et) {
  swap_grid_barrier(gsync, gridDim.x, et);
  uint64_t* kin = reinterpret_cast<uint64_t*>(ring);               // [kTailCap] gathered keys
  uint64_t* kso = kin + kTailCap;                                   // [kTailCap] the same in descending order
  int* start = reinterpret_cast<int*>(kso + kTailCap);              // [kTailSegs + 1] first flat index of each segment
  uint32_t* sc = reinterpret_cast<uint32_t*>(start + kTailSegs + 8);  // general routines (warp 0 only): [kLsCap] x 2 + histogram
  uint32_t* rw = sc + kLsCap;
  uint32_t* hist = rw + kLsCap;
  const int k = a.k, nseg = a.nseg;
  const bool screened = a.band > 0.f;
  const int kc = screened ? a.kc : k;
  const int cap = min(a.seg_cap, a.seg_stride);
  for (int64_t q = blockIdx.x; q < a.Q; q += gridDim.x) {
    const uint64_t* qbase = a.seg_keys + q * nseg * static_cast<int64_t>(a.seg_stride);
    if (ew == 0) {
      int c[5];
      int mine = 0;
#pragma unroll
      for (int u = 0; u < 5; ++u) {
        const int sg = lane * 5 + u;
        c[u] = sg < nseg ? min(__ldcg(a.seg_cnt + q * nseg + sg), cap) : 0;
        mine += c[u];
      }
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += v;
      }
      int run = incl - mine;
#pragma unroll
      for (int u = 0; u < 5; ++u) {
        start[lane * 5 + u] = run;
        run += c[u];
      }
      if (lane == 31) start[kTailSegs] = run;
    }
    epi_sync();
    const int total = start[kTailSegs];
    if (total <= kTailCap) {
      for (int base = 0; base < total; base += 4 * 128) {
        uint64_t raw[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int i = base + j * 128 + et;
          raw[j] = 0ull;
          if (i < total) {
            int sg = 0;
#pragma unroll
            for (int step = 128; step > 0; step >>= 1)
              if (sg + step < kTailSegs && start[sg + step] <= i) sg += step;
            raw[j] = __ldcg(qbase + static_cast<int64_t>(sg) * a.seg_stride + (i - start[sg]));
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int i = base + j * 128 + et;
          if (i < total) kin[i] = (static_cast<uint64_t>(order_bits(__uint_as_float(static_cast<uint32_t>(raw[j] >> 32)))) << 32) | (raw[j] & 0xFFFFFFFFull);
        }
      }
      epi_sync();
      tail_order(kin, kso, total, et);
      int kept = min(total, k);
      bool lost = false;
      if (screened) {
        if (total >= k) {  // every key within the band below the k-th best screened score goes on to the exact re-scoring
          const uint64_t t_key = static_cast<uint64_t>(order_bits(key_score(kso[k - 1]) - a.band)) << 32;
          int lo = k, hi = total;  // first position whose key falls below the threshold
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (kso[mid] >= t_key) lo = mid + 1;
            else hi = mid;
          }
          kept = lo;
        }
        lost = kept > kc || __ldcg(a.overflow + q) != 0u;
      }
      if (!screened) {
        const float scale = a.out_scale * (a.out_qscale ? a.out_qscale[q] : 1.0f);
        for (int i = et; i < k; i += 128) {
          const bool ok = i < kept;
          a.out_scores[q * k + i] = ok ? key_score(kso[i]) * scale : -INFINITY;
          a.out_ids[q * k + i] = ok ? static_cast<int64_t>(key_row(kso[i])) + a.id_offset : -1;
        }
      } else if (lost) {  // too many near-ties inside the band: rank the whole catalog for this query
        if (ew == 0) {
          const int kr = ls_rank_catalog<XB>(sc, rw, kLsCap, hist, q, a, lane);
          ls_emit_ranked(sc, rw, kr, k, 1.0f, q, a, hist, lane);
        }
      } else {
        warp_rescore<true>(kso, kept, ew, 4, q, a, lane);  // kso[i] <- exact (score, row) of its row
        epi_sync();
        tail_order(kso, kin, kept, et);
        for (int i = et; i < k; i += 128) {
          const bool ok = i < kept;
          a.out_scores[q * k + i] = ok ? key_score(kin[i]) : -INFINITY;
          a.out_ids[q * k + i] = ok ? static_cast<int64_t>(key_row(kin[i])) + a.id_offset : -1;
        }
      }
    } else if (ew == 0) {
      // more survivors than the buffer holds: the general routines, segment by segment with squeezes in between
      float tau = -INFINITY;
      bool lost = false;
      int n = 0;
      for (int sg = 0; sg < nseg; ++sg) {
        const int cs = start[sg + 1] - start[sg];
        if (n + cs > kLsCap) {
          __syncwarp();
          n = ls_reduce(sc, rw, n, k, a.band, hist, &tau);
          if (n > kc) {
            lost = true;
            n = kc;
          }
        }
        const uint64_t* seg = qbase + static_cast<int64_t>(sg) * a.seg_stride;
        for (int i = lane; i < cs; i += 32) {
          const uint64_t raw = __ldcg(seg + i);
          sc[n + i] = order_bits(__uint_as_float(static_cast<uint32_t>(raw >> 32)));
          rw[n + i] = static_cast<uint32_t>(raw);
        }
        n += cs;
      }
      __syncwarp();
      int kept = ls_reduce(sc, rw, n, k, a.band, hist, &tau);
      if (kept > kc) {
        lost = true;
        kept = kc;
      }
      if (screened) {
        if (lost || __ldcg(a.overflow + q) != 0u) kept = ls_rank_catalog<XB>(sc, rw, kLsCap, hist, q, a, lane);
        else ls_rescore<false>(sc, rw, kept, q, a, lane);
        ls_emit_ranked(sc, rw, kept, k, 1.0f, q, a, hist, lane);
      } else {
        ls_emit_ranked(sc, rw, kept, k, a.out_scale * (a.out_qscale ? a.out_qscale[q] : 1.0f), q, a, hist, lane);
      }
    }
    epi_sync();  // the buffers are free for the CTA's next query
  }
}

// Per-query exclusions of the swapped kernel (XB): a warp's 32 rows share one bitmap word per query. Lane l loads the words
// of queries l, l + 32, ... for the tile's row block (coalesced) into this warp's share of the bootstrap buffer, xs[query]
// (idle outside the bootstrap's ranking); row `lane` of the warp is excluded for query j when bit `lane` of xs[j] is set
// (broadcast reads).
// The boot tiles load their words before the epilogue waits for the accumulator and store them after it; the filtering tiles
// load the next tile's words while the current one is filtered.
__device__ __forceinline__ void load_swap_words(uint32_t (&w)[8], const GemmArgs& g, int row32, int lane) {
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const int q = b * 32 + lane;
    w[b] = (b * 32 < g.qpad && q < g.Q && row32 * 32 < g.N) ? Exclusions{nullptr, g.xbits, g.xld}.word(q, row32) : 0u;
  }
}
__device__ __forceinline__ void store_swap_words(uint32_t* xs, const uint32_t (&w)[8], int qpad, int lane) {
  __syncwarp();
#pragma unroll
  for (int b = 0; b < 8; ++b)
    if (b * 32 < qpad) xs[b * 32 + lane] = w[b];
  __syncwarp();
}
// bit j: query jb + j excludes row `lane` of this warp
__device__ __forceinline__ uint32_t swap_excluded32(const uint32_t* xs, int jb, int lane) {
  uint32_t m = 0u;
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const uint4 w = *reinterpret_cast<const uint4*>(xs + jb + j);
    m |= ((w.x >> lane) & 1u) << j;
    m |= ((w.y >> lane) & 1u) << (j + 1);
    m |= ((w.z >> lane) & 1u) << (j + 2);
    m |= ((w.w >> lane) & 1u) << (j + 3);
  }
  return m;
}

template <int MODE, bool XB = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kSwapThreads, 1)
gemm_swap_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_c, const GemmArgs g,
                 const __grid_constant__ HistSelectArgs sel) {
  constexpr bool SCALED = (MODE == 1 || MODE == 4 || MODE == 5);  // exact scores scaled by the catalog's inverse norms in the epilogue
  constexpr int kStageBytes = kTileBytes;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int KB = g.kb_per_term;
  const int QH = g.qpad >> 1;              // query rows held by each CTA of the pair
  const int qtile_bytes = QH * 128;        // one 64-element K block of them (multiple of 2 KB)
  const int res_bytes = KB * qtile_bytes;
  int stages = (kRingBytes - res_bytes) / kStageBytes;
  if (stages > kSwapMaxStages) stages = kSwapMaxStages;
  unsigned char* q_res = smem;  // K block kb at q_res + kb * qtile_bytes
  unsigned char* stage_base = smem + res_bytes;
  float* tau_s = reinterpret_cast<float*>(smem + kRingBytes);  // [256] per-query thresholds (raw units)
  int* cnt_s = reinterpret_cast<int*>(tau_s + 256);             // [256] keys in this CTA's segment of each query
  int* flag_s = cnt_s + 256;                                    // [4]   some segment is close to its capacity
  uint64_t* bars = reinterpret_cast<uint64_t*>(flag_s + 4);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kSwapMaxStages;
  uint64_t* tfull_bar = bars + 2 * kSwapMaxStages;
  uint64_t* tempty_bar = bars + 2 * kSwapMaxStages + 2;
  uint64_t* qfull_bar = bars + 2 * kSwapMaxStages + 4;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kSwapMaxStages + 5);
  uint32_t* boot_s = reinterpret_cast<uint32_t*>(bars + 2 * kSwapMaxStages + 6);  // [4 warps][2 * kBootCap + kHsBins], boot mode only

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int items = g.chunks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&tfull_bar[a]), 1);
      mbar_init(smem_u32(&tempty_bar[a]), 2 * 4);  // four epilogue warps in each CTA
    }
    mbar_init(smem_u32(qfull_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_q) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tma_c) : "memory");
  }
  if (warp == 2) tmem_alloc_pair(smem_u32(tmem_ptr), kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0 && lane == 0) {
    // ================= TMA producer =================
    const uint32_t qb = smem_u32(qfull_bar);
    if (rank == 0) mbar_expect_tx(qb, 2 * res_bytes);
    for (int kb = 0; kb < KB; ++kb)
      tma_load_2d_pair(smem_u32(q_res + kb * qtile_bytes), &tma_q, kb * BK, static_cast<int>(rank) * QH, qb);
    int stage = 0;
    uint32_t phase = 0;
    for (int w = pair; w < items; w += npairs) {
      const int t0 = chunk_first_tile(g, w), t1 = chunk_first_tile(g, w + 1);
      for (int tt = t0 - g.boot; tt < t1; ++tt) {  // boot mode: the chunk's first g.boot tiles are streamed twice (see the epilogue)
        const int tile = tt < t0 ? tt + g.boot : tt;
        const int crow = tile * BN + static_cast<int>(rank) * BNH;
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full_bar[stage]);
          if (rank == 0) mbar_expect_tx(fb, 2 * kStageBytes);
          const uint32_t sa = smem_u32(stage_base + stage * kStageBytes);
          tma_load_2d_pair(sa, &tma_c, kb * BK, crow, fb);
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ================= MMA issuer: whole warp walks the loop, one elected lane issues =================
    const uint32_t idesc = idesc_formats<MODE>() | (static_cast<uint32_t>(g.qpad >> 3) << 17) | (static_cast<uint32_t>(BN >> 4) << 24);
    const uint64_t qd0 = smem_desc_sw128(smem_u32(q_res));
    const uint64_t cd0 = smem_desc_sw128(smem_u32(stage_base));
    constexpr uint64_t kStageUnits = kStageBytes >> 4;
    const uint64_t qunits = static_cast<uint64_t>(qtile_bytes >> 4);
    mbar_wait(smem_u32(qfull_bar), 0);
    tc_fence_after();
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = pair; w < items; w += npairs) {
      const int t0 = chunk_first_tile(g, w), t1 = chunk_first_tile(g, w + 1);
      for (int tt = t0 - g.boot; tt < t1; ++tt) {
        mbar_wait(smem_u32(&tempty_bar[acc]), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * 256);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint64_t cdesc = cd0 + static_cast<uint64_t>(stage) * kStageUnits;
          const uint64_t qdesc = qd0 + static_cast<uint64_t>(kb) * qunits;
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4) {
              const uint64_t o = static_cast<uint64_t>(k4 * 2);
              umma_pair<MODE>(d_tmem, cdesc + o, qdesc + o, idesc, (kb | k4) != 0 ? 1u : 0u);
            }
            umma_commit_pair(smem_u32(&empty_bar[stage]));
            if (kb == KB - 1) umma_commit_pair(smem_u32(&tfull_bar[acc]));
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = catalog row, columns = queries =================
    const int ew = warp & 3, et = threadIdx.x - 128;
    const int cap = g.seg_cap;
    uint64_t* scratch = g.compact_scratch + (static_cast<int64_t>(blockIdx.x) * kEpiWarps + ew) * kSegCapMax;
    uint32_t* xs = boot_s + ew * (2 * kBootCap + kHsBins);  // XB: [qpad] staged bitmap words (see stage_swap_words)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int w = pair; w < items; w += npairs) {
      const int t0 = chunk_first_tile(g, w), t1 = chunk_first_tile(g, w + 1);
      const int64_t seg0 = static_cast<int64_t>(w) * 2 + rank;  // + q * chunks * 2
      if (g.boot) {
        // ---- single-launch mode: bootstrap the thresholds from the chunk's first g.boot tiles ------------------------
        // Every epilogue warp takes the maximum of its rows (32 per tile) for each query: 4 * gridDim.x group maxima per query, each
        // the score of a distinct catalog row, so the k-th largest of them is a lower bound of the final k-th best score
        // (k <= 4 * gridDim.x is the host's condition for this mode). After a grid barrier the warps of all CTAs rank the
        // maxima of their share of the queries and publish tau; after a second barrier the chunk - including its first
        // tile, streamed again - is filtered as in the phased path. Two launches (first-phase GEMM + select) and, for small
        // catalogs, most of the call's latency disappear (profiles/r02_notes.md).
        const int gstride = 4 * static_cast<int>(gridDim.x);
        float best[8];  // lane l: running maximum of this warp's rows for query 32 * b + l (qpad <= 256)
#pragma unroll
        for (int b = 0; b < 8; ++b) best[b] = -INFINITY;
        for (int bt = 0; bt < g.boot; ++bt) {
          const int row = (t0 + bt) * BN + static_cast<int>(rank) * BNH + ew * 32 + lane;
          const bool valid = row < g.N && !(g.mask && g.mask[row]);
          const float cinv_r = SCALED ? (row < g.N ? __ldg(g.cinv + row) : 0.f) : 1.0f;
          uint32_t xw[8];
          if (XB) load_swap_words(xw, g, (row - lane) >> 5, lane);
          mbar_wait(smem_u32(&tfull_bar[acc]), acc_phase);
          tc_fence_after();
          if (XB) store_swap_words(xs, xw, g.qpad, lane);
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(acc * 256);
#pragma unroll
          for (int b = 0; b < 8; ++b) {
            if (b * 32 < g.qpad) {
              uint32_t r[32];
              tmem_ld32(taddr + b * 32, r);
              tmem_ld_wait(r);
              acc_to_f32<MODE>(r);
              float sc[32];
              const uint32_t xm = XB ? swap_excluded32(xs, b * 32, lane) : 0u;  // excluded (row, query) pairs do not bound anything
#pragma unroll
              for (int j = 0; j < 32; ++j) sc[j] = (valid && !((xm >> j) & 1u)) ? __uint_as_float(r[j]) * cinv_r : -INFINITY;
              warp_transpose_max<32>(sc, lane);  // lane l: the maximum over this warp's rows for query 32 * b + l
              best[b] = fmaxf(best[b], sc[0]);
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(smem_u32(&tempty_bar[acc]), 0);
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
#pragma unroll
        for (int b = 0; b < 8; ++b)
          if (b * 32 + lane < g.Q) g.gmax[static_cast<int64_t>(b * 32 + lane) * gstride + blockIdx.x * 4 + ew] = best[b];
        swap_grid_barrier(g.gsync, gridDim.x, et);
        uint32_t* bsc = boot_s + ew * (2 * kBootCap + kHsBins);
        uint32_t* brw = bsc + kBootCap;
        uint32_t* bhist = brw + kBootCap;
        for (int j = blockIdx.x * 4 + ew; j < g.Q; j += gstride) {
          for (int i = lane; i < gstride; i += 32) {
            bsc[i] = order_bits(__ldcg(g.gmax + static_cast<int64_t>(j) * gstride + i));
            brw[i] = ~static_cast<uint32_t>(i);
          }
          __syncwarp();
          uint32_t ks, kr;
          ls_kth(bsc, brw, gstride, g.k, bhist, lane, ks, kr);
          // the filter is a strict ">", and the bootstrap rows are filtered again: the threshold sits one ulp BELOW the k-th
          // group maximum so that the row it came from (and its exact ties) survive
          if (lane == 0) const_cast<float*>(g.tau)[j] = boot_tau<XB>(ks, g.band);
          __syncwarp();
        }
        swap_grid_barrier(g.gsync + 1, gridDim.x, et);
      }
      for (int j = et; j < 256; j += 128) {
        tau_s[j] = j < g.Q ? __ldcg(g.tau + j) : INFINITY;
        cnt_s[j] = 0;
      }
      if (et == 0) flag_s[0] = 0;
      epi_sync();
      const int wrow0 = static_cast<int>(rank) * BNH + ew * 32;  // this warp's first row of a tile
      uint32_t xw[8];  // XB: the words of the next tile, loaded while the current one is filtered
      if (XB) load_swap_words(xw, g, (t0 * BN + wrow0) >> 5, lane);
      for (int tile = t0; tile < t1; ++tile) {
        const int row = tile * BN + wrow0 + lane;
        const bool valid = row < g.N && !(g.mask && g.mask[row]);
        const float cinv_r = SCALED ? (row < g.N ? __ldg(g.cinv + row) : 0.f) : 1.0f;
        const uint32_t nrow = ~static_cast<uint32_t>(row);
        if (XB) {
          store_swap_words(xs, xw, g.qpad, lane);
          if (tile + 1 < t1) load_swap_words(xw, g, ((tile + 1) * BN + wrow0) >> 5, lane);
        }
        mbar_wait(smem_u32(&tfull_bar[acc]), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + static_cast<uint32_t>(acc * 256);
        for (int jb = 0; jb < g.qpad; jb += 32) {
          uint32_t r[32];
          tmem_ld32(taddr + jb, r);
          tmem_ld_wait(r);
          acc_to_f32<MODE>(r);
          float sc[32];
          unsigned m = 0;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 t4 = *reinterpret_cast<const float4*>(tau_s + jb + j);  // broadcast reads
            sc[j] = __uint_as_float(r[j]) * cinv_r;
            sc[j + 1] = __uint_as_float(r[j + 1]) * cinv_r;
            sc[j + 2] = __uint_as_float(r[j + 2]) * cinv_r;
            sc[j + 3] = __uint_as_float(r[j + 3]) * cinv_r;
            m |= (sc[j] > t4.x ? 1u : 0u) << j;
            m |= (sc[j + 1] > t4.y ? 1u : 0u) << (j + 1);
            m |= (sc[j + 2] > t4.z ? 1u : 0u) << (j + 2);
            m |= (sc[j + 3] > t4.w ? 1u : 0u) << (j + 3);
          }
          if (!valid) m = 0;
          if (XB && __any_sync(kFull, xs[jb + lane] != 0u)) m &= ~swap_excluded32(xs, jb, lane);
          if (__any_sync(kFull, m != 0)) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (m & (1u << j)) {
                const int q = jb + j;
                const int pos = atomicAdd(&cnt_s[q], 1);
                if (pos < cap) {
                  uint64_t* seg = g.cand + (static_cast<int64_t>(q) * g.chunks * 2 + seg0) * cap;
                  seg[pos] = (static_cast<uint64_t>(__float_as_uint(sc[j])) << 32) | nrow;
                }
                if (pos >= cap - 129) flag_s[0] = 1;
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(smem_u32(&tempty_bar[acc]), 0);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
        // A tile adds at most 128 keys per query to this CTA's segments: any segment that could overflow during
        // the next tile is cut back to its k best now, which also raises that query's threshold in this CTA.
        epi_sync();
        if (flag_s[0]) {
          for (int q = ew; q < g.Q; q += 4) {
            const int n = min(cnt_s[q], cap);
            if (n > cap - 128) {
              uint64_t* seg = g.cand + (static_cast<int64_t>(q) * g.chunks * 2 + seg0) * cap;
              const int P = cap <= 256 ? 256 : kSegCapMax;
              for (int i = lane; i < P; i += 32) scratch[i] = (i < n) ? canonical_key(__ldcg(seg + i)) : 0ull;
              warp_bitonic_sort_desc(scratch, P, lane);
              int kept = n < g.k ? n : g.k;
              float t_new = (n >= g.k) ? unorder_bits(static_cast<uint32_t>(scratch[g.k - 1] >> 32)) : -INFINITY;
              if (g.band > 0.f && n >= g.k) {  // screened scores: keep the whole band below the segment's k-th best
                t_new -= g.band;
                const uint64_t t_key = static_cast<uint64_t>(order_bits(t_new)) << 32;
                int c = 0;
                for (int i = lane; i < n; i += 32) c += (scratch[i] >= t_key) ? 1 : 0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
                kept = c;
                if (kept > cap - 136) {  // no room for another tile (<= 128 keys): exact ranking of this query at the end
                  if (lane == 0) g.overflow[q] = 1u;
                  kept = g.k;
                }
              }
              for (int i = lane; i < kept; i += 32) seg[i] = raw_key(scratch[i]);
              if (lane == 0) {
                cnt_s[q] = kept;
                tau_s[q] = fmaxf(tau_s[q], t_new);
              }
              __syncwarp();
            }
          }
          epi_sync();
          if (et == 0) flag_s[0] = 0;
          epi_sync();
        }
      }
      for (int j = et; j < g.Q; j += 128) g.cand_cnt[static_cast<int64_t>(j) * g.chunks * 2 + seg0] = min(cnt_s[j], cap);
      epi_sync();
    }
    if (g.fuse_select) swap_select_tail<XB>(g.gsync + 2, sel, smem, ew, lane, et);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}

// ---- host side ---------------------------------------------------------------------------------------
int launch_row_inv_norms(const void* x, int64_t rows, int64_t dim, int64_t ld, int dtype, float* inv, cudaStream_t st, float* tau_init = nullptr,
                         unsigned int* ovf_init = nullptr);
int launch_split_planes(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* planes, cudaStream_t st);
int launch_screen_plane(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* plane, float* inv, cudaStream_t st, float* tau_init = nullptr,
                        unsigned int* ovf_init = nullptr);
int launch_quantize_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx, int8_t* codes, int64_t ldc, float* factors, cudaStream_t st,
                         float* tau_init = nullptr, unsigned int* ovf_init = nullptr);

constexpr size_t kGemmSmemBytes = static_cast<size_t>(kRingBytes) + 4 * BN * sizeof(float) +  // EW * ECOLS = 4 * BN inverse norms
                                 
                                  (2 * kMaxStages + 6) * sizeof(uint64_t) + 16 + kEpiWarps * (kK2BootCap + kHsBins) * sizeof(uint32_t) + 1024;
// 256 + 32: a whole 256-row tile of a first phase (threshold -inf, every row survives) fits without tripping the
// in-kernel cut-back, whose margin is 32 keys
static int seg_cap_for(int k) { return k <= 128 ? 288 : kSegCapMax; }
static_assert(kGemmSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
constexpr size_t kSwapSmemBytes = static_cast<size_t>(kRingBytes) + 2 * 256 * 4 + 16 + (2 * kSwapMaxStages + 6) * sizeof(uint64_t) + 16 + kSwapBootBytes + 1024;
static_assert(kSwapSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA may use");

// top-k path: MODE 2 (one-term screening + exact re-scoring of the survivors) on fp32 catalogs, MODE 1 on bf16 ones,
// MODE 4 on fp16 ones, MODE 5 on int8 ones
static int mode_for(int dtype) { return dtype == ICR_F32 ? 2 : (dtype == ICR_BF16 ? 1 : (dtype == ICR_I8 ? 5 : 4)); }
// The tile geometry sees an int8 row of D codes as a 16-bit row of D / 2 elements (the same bytes): swap_applies, the
// bootstrap plans, the K-block count ceil(D / 128) and the A-stationary limit (D <= 768) all follow from the true bytes.
static int64_t geometry_dim(int64_t D, int dtype) { return dtype == ICR_I8 ? D / 2 : D; }
// keys carried per query between phases: k exact keys, or k + room for the screening band (select_args.cuh)
static int carry_cap(int k, int mode) {
  if (mode != 2) return k;
  const int kc = k + (k > 32 ? k : 32);
  return kc < 512 ? kc : 512;
}

// the swapped kernel applies when one block of queries is small enough to stay resident next to a useful ring
static bool swap_applies(int64_t Q, int64_t N, int64_t D) {
  if (Q > 256) return false;
  const int64_t qpad = (Q + 31) / 32 * 32;
  const int64_t kb = (D + BK - 1) / BK;
  const int64_t res = kb * (qpad / 2) * 128;
  const int64_t sweep_bytes = N * ((D + BK - 1) / BK * BK) * 2;
  return res <= (sweep_bytes <= kSmallCatalogBytes ? kSwapResidentMaxSmallCatalog : kSwapResidentMax);
}

struct Phase {
  int tile_begin, tile_end, chunks;
};

// Phases of geometrically growing tile ranges. tau after a phase is the exact k-th score of all rows seen,
// so a phase that multiplies the rows seen by g admits ~k*ln(g) (at most ~k*(g-1)) survivors per query.
// swapped kernel: its epilogue work is small (128 x Q scores per tile), so it affords denser survivors in exchange
// for fewer phases - every phase costs a launch of the GEMM and of the select (~25 us for a small batch)
constexpr int kSwapGrowth = 32;
constexpr int kK2First = 4, kSwapFirst = 8;  // tiles of the first phase, at least
static int plan_phases(int64_t N, int qblocks, int k, Phase* out, int max_phases, bool swap, int begin0 = 0) {
  const int T = static_cast<int>((N + BN - 1) / BN);
  // K2: 8, or 32 for ONE query block on a catalog that streams from HBM: there every phase costs ~35-45 us of small
  // GEMM + select beside a stream of a few hundred us, and 3 sparse phases beat 4 (profiles/r02_c4_phase_sweep.txt)
  const int k2_growth = (qblocks == 1 && T >= 2048) ? 32 : 8;
  const int growth = swap ? kSwapGrowth : k2_growth;
  const int npairs = kNumSMs / 2;
  int first = (2 * k + BN - 1) / BN;
  if (first < kK2First) first = kK2First;
  if (swap && first < kSwapFirst) first = kSwapFirst;
  int n = 0, begin = 0, end = first < T ? first : T;
  if (begin0 > 0) {  // rows of tiles [0, begin0) were scored densely: the sparse phases start behind them
    begin = begin0;
    const int64_t next = static_cast<int64_t>(begin0) * growth;
    end = next < T ? static_cast<int>(next) : T;
  }
  while (begin < T && n < max_phases) {
    if (n == max_phases - 1) end = T;
    const int tiles = end - begin;
    // enough work items to fill the machine twice, few enough survivors per segment to stay far from its capacity:
    // phase 0 admits every row (rows per chunk <= cap, i.e. cap/2 per column half); later phases expect
    // ~(growth-1)*k survivors per query, spread over 2*chunks segments, kept under a quarter of the capacity
    const int cap = seg_cap_for(k);
    int chunks = (2 * npairs + qblocks - 1) / qblocks;
    const int by_load = (n == 0 && begin0 == 0) ? (tiles * BN + cap - 1) / cap : ((growth - 1) * k + cap / 2 - 1) / (cap / 2);
    if (chunks < by_load) chunks = by_load;
    if (chunks > tiles) chunks = tiles;
    if (chunks < 1) chunks = 1;
    // work items go round-robin to the pairs; pick the chunk count (near the floor computed above) whose
    // busiest pair has the least tiles: rounds * ceil(tiles / chunks)
    int best = chunks;
    int64_t best_load = -1;
    for (int c = chunks; c <= tiles && c < chunks + 24; ++c) {
      const int64_t rounds = (static_cast<int64_t>(qblocks) * c + npairs - 1) / npairs;
      const int64_t load = rounds * ((tiles + c - 1) / c);
      if (best_load < 0 || load < best_load) {
        best_load = load;
        best = c;
      }
    }
    out[n].tile_begin = begin;
    out[n].tile_end = end;
    out[n].chunks = best;
    ++n;
    begin = end;
    const int64_t next = static_cast<int64_t>(end) * growth;
    end = next < T ? static_cast<int>(next) : T;
  }
  return n;
}

constexpr int kMaxPhases = 16;
// Rows of the first tiles are scored densely in the first phase of the (non-swapped) top-k path (profiles/r01_notes.md):
// 4 tiles, or 16 for one query block on a catalog that streams from HBM (one sparse phase less, see plan_phases)
static int dense0_tiles(int64_t Q, int64_t N) { return (Q <= 2 * BM && (N + BN - 1) / BN >= 2048) ? 16 : 4; }

// kernel variants: 1 = bf16 streaming both operands, 2 = bf16 with resident queries, 5 / 6 = fp16 screen plane streaming /
// resident queries, 8 / 9 = fp16 rows streaming / resident queries, 10 / 11 = int8 rows streaming / resident queries,
// 4 / 7 / 3 / 12 = swapped kernel (small batches) on bf16 / the screen plane / fp16 rows / int8 rows; DENSE only: 0 = fp16
// hi|lo planes, three MMA terms (K2' on fp32 inputs)
#define ICR_GEMM_VARIANTS(X, DENSE, XB)            \
  X(1, (gemm_topk_kernel<1, false, DENSE, XB>))    \
  X(2, (gemm_topk_kernel<1, true, DENSE, XB>))     \
  X(5, (gemm_topk_kernel<2, false, DENSE, XB>))    \
  X(6, (gemm_topk_kernel<2, true, DENSE, XB>))     \
  X(8, (gemm_topk_kernel<4, false, DENSE, XB>))    \
  X(9, (gemm_topk_kernel<4, true, DENSE, XB>))     \
  X(10, (gemm_topk_kernel<5, false, DENSE, XB>))   \
  X(11, (gemm_topk_kernel<5, true, DENSE, XB>))

// Launch helper of the GEMM kernels. The single-launch modes (g.boot > 0) synchronise the whole grid through a counter in
// global memory, which needs every CTA resident at once: those launches carry the cooperative attribute, so the driver
// rejects a grid that cannot be co-resident and never starts one piecemeal beside kernels of other streams. A driver that
// refuses the attribute on a cluster kernel gets the plain launch (the grid is sized to one CTA per SM either way).
template <typename... KArgs, typename... Args>
static void launch_gemm_grid(void (*kernel)(KArgs...), int grid, int threads, size_t smem, cudaStream_t st, bool coop, Args&&... args) {
  static thread_local bool refused = false;
  if (coop && !refused) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(threads));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
    if (e == cudaSuccess) return;
    if (e != cudaErrorNotSupported && e != cudaErrorInvalidValue && e != cudaErrorInvalidConfiguration &&
        e != cudaErrorCooperativeLaunchTooLarge)
      return;  // left for ICR_LAUNCH_CHECK
    (void)cudaGetLastError();
    if (e != cudaErrorCooperativeLaunchTooLarge) refused = true;
  }
  kernel<<<grid, threads, smem, st>>>(KArgs(args)...);
}

// launches instantiation `which` of the queries-on-M kernel, DENSE (K2' / first phase) or filtering (XB: with per-query
// exclusions)
template <bool DENSE, bool XB = false>
static int launch_gemm_variant(int which, int grid, const CUtensorMap& map_a, const CUtensorMap& map_b, const GemmArgs& g, cudaStream_t st) {
  static thread_local SmemAttrCache cache[12];
  int rc = ICR_OK;
#define ICR_SET(ID, K) \
  if (which == ID) rc = ensure_dyn_smem(cache[ID], K, kGemmSmemBytes);
  ICR_GEMM_VARIANTS(ICR_SET, DENSE, XB)
  if constexpr (DENSE) ICR_SET(0, (gemm_topk_kernel<3, false, true>))
#undef ICR_SET
  if (rc) return rc;
  const int terms = which == 0 ? 3 : 1;
  profile_begin(kKernelGemm, terms, st);
  const int threads = 128 + epi_warps(terms) * 32;
#define ICR_RUN(ID, K) \
  if (which == ID) launch_gemm_grid(K, grid, threads, kGemmSmemBytes, st, g.boot > 0, map_a, map_b, g);
  ICR_GEMM_VARIANTS(ICR_RUN, DENSE, XB)
  if constexpr (DENSE) ICR_RUN(0, (gemm_topk_kernel<3, false, true>))
#undef ICR_RUN
  profile_end(st);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

template <bool XB = false>
static int launch_swap_variant(int which, int grid, const CUtensorMap& map_q, const CUtensorMap& map_c, const GemmArgs& g, cudaStream_t st,
                               const HistSelectArgs& sel = HistSelectArgs{}) {
  static thread_local SmemAttrCache cache[4];
  int rc = ICR_OK;
  if (which == 4) rc = ensure_dyn_smem(cache[0], gemm_swap_kernel<1, XB>, kSwapSmemBytes);
  if (which == 7) rc = ensure_dyn_smem(cache[1], gemm_swap_kernel<2, XB>, kSwapSmemBytes);
  if (which == 3) rc = ensure_dyn_smem(cache[2], gemm_swap_kernel<4, XB>, kSwapSmemBytes);
  if (which == 12) rc = ensure_dyn_smem(cache[3], gemm_swap_kernel<5, XB>, kSwapSmemBytes);
  if (rc) return rc;
  profile_begin(kKernelGemm, 1, st);
  if (which == 4) launch_gemm_grid(gemm_swap_kernel<1, XB>, grid, kSwapThreads, kSwapSmemBytes, st, g.boot > 0, map_q, map_c, g, sel);
  if (which == 7) launch_gemm_grid(gemm_swap_kernel<2, XB>, grid, kSwapThreads, kSwapSmemBytes, st, g.boot > 0, map_q, map_c, g, sel);
  if (which == 3) launch_gemm_grid(gemm_swap_kernel<4, XB>, grid, kSwapThreads, kSwapSmemBytes, st, g.boot > 0, map_q, map_c, g, sel);
  if (which == 12) launch_gemm_grid(gemm_swap_kernel<5, XB>, grid, kSwapThreads, kSwapSmemBytes, st, g.boot > 0, map_q, map_c, g, sel);
  profile_end(st);
  ICR_LAUNCH_CHECK();
  return ICR_OK;
}

struct GemmWs {
  size_t q_planes, c_planes, qinv, cinv, tau, overflow, carry[2], carry_cnt[2], cand, cand_cnt, scratch, dense0, gmax, total;
  int max_chunks, seg_cap, kc;
  int boot_pairs;  // > 0: single-launch swapped path with in-kernel threshold bootstrap on this many CTA pairs
  int boot_tiles;  // bootstrap tiles per chunk
  int k2_boot_chunks, k2_boot_tiles;  // > 0: single-launch K2 (queries on M) with in-kernel bootstrap
  int k2_boot_coarse;                 // its maxima are per tile and column group (k2_boot_plan)
};

// Single-launch mode of K2: one phase over the whole catalog, `chunks` tile ranges per query block, the first `tiles` tiles of
// every work item scored twice (once for the block maxima the thresholds come from). The bootstrap rows are chosen so that
// ~kK2BootTarget keys per query pass the threshold (N * k / rows); the mode needs 2k..kK2BootCap block maxima per query and
// re-streams at most a quarter of a chunk - i.e. it serves catalogs of up to a few hundred thousand rows, where the phased
// path spends a third of its time on the two bootstrap phases and their selects; larger catalogs keep the phased path.
constexpr int kK2BootTarget = 550;  // profiles/r02_k2_boot_target_sweep_*.txt
static int k2_boot_plan(int64_t Q, int64_t N, int64_t D, int k, int* chunks_out, int* coarse_out = nullptr) {
  if (coarse_out) *coarse_out = 0;
  if (swap_applies(Q, N, D)) return 0;
  const int T = static_cast<int>((N + BN - 1) / BN);
  const int qblocks = static_cast<int>((Q + 2 * BM - 1) / (2 * BM));
  const int npairs = kNumSMs / 2;
  int c0 = (2 * npairs + qblocks - 1) / qblocks;
  const int by_load = (kK2BootTarget + 71) / 72;  // survivors spread over 2 * chunks segments, kept under a quarter of their capacity
  if (c0 < by_load) c0 = by_load;
  if (c0 > T) c0 = T;
  int best = c0;
  int64_t best_load = -1;
  for (int c = c0; c <= T && c < c0 + 24; ++c) {
    const int64_t rounds = (static_cast<int64_t>(qblocks) * c + npairs - 1) / npairs;
    const int64_t load = rounds * ((T + c - 1) / c);
    if (best_load < 0 || load < best_load) {
      best_load = load;
      best = c;
    }
  }
  const int64_t want_rows = N * k / kK2BootTarget;
  int tiles = static_cast<int>((want_rows + static_cast<int64_t>(BN) * best - 1) / (static_cast<int64_t>(BN) * best));
  if (tiles < 1) tiles = 1;
  while (best * tiles * (BN / 32) < 2 * k) ++tiles;
  if (best * tiles * (BN / 32) > kK2BootCap) {
    // Too many 32-score block maxima for the in-kernel ranking. ONE query block on a catalog that streams from HBM (C4 shard,
    // Q = 65...256) is worth a coarser bootstrap: one maximum per tile and column group, as many bootstrap tiles as the
    // ranking holds. Fewer sampled rows let more keys pass (C4 shard, k = 100: ~1,650 per query instead of ~550), but the
    // four sparse phases with their selects that this replaces cost ~100 us beside a 0.33 ms stream.
    const int eh = epi_warps(1) / 4;
    const int qblocks1 = static_cast<int>((Q + 2 * BM - 1) / (2 * BM));
    int ct = kK2BootCap / (best * eh);
    if (ct > tiles) ct = tiles;
    if (qblocks1 != 1 || T < 2048 || ct < 1 || best * ct * eh < 2 * k) return 0;
    if (static_cast<double>(N) * k / (static_cast<double>(BN) * best * ct) > 2500.0) return 0;  // survivors per query the segments and the select take in their stride
    if (ct * 4 > T / best) return 0;
    if (coarse_out) *coarse_out = 1;
    *chunks_out = best;
    return ct;
  }
  // at most a quarter of a chunk is scored twice; half for a catalog the L2 holds, where the second read is cheap and the
  // phased path's extra launches are the larger cost (Q = 512 on the 49,688-row catalog: 74 chunks of 2-3 tiles)
  const int64_t dp = (D + 63) / 64 * 64;
  const bool l2_sized = N * dp * 2 <= (96ll << 20);
  if (tiles * (l2_sized ? 2 : 4) > T / best) return 0;
  *chunks_out = best;
  return tiles;
}

// Single-launch mode of the swapped kernel: one chunk per CTA pair, thresholds bootstrapped in the kernel from 4 group maxima
// per CTA. Needs at least k groups (and leaves headroom: 2k), at most kBootCap, and one chunk per pair.
// The bootstrap threshold lets ~N * k / (rows scored in the bootstrap) keys per query through: the number of bootstrap tiles per
// chunk is chosen so that this stays near 4,000 (cheap for the select, far from the segments' capacity), and the mode is
// refused when that would re-stream more than a quarter of a chunk.
static int boot_pairs_for(int64_t Q, int64_t N, int64_t D, int k, int* boot_tiles) {
  if (!swap_applies(Q, N, D)) return 0;
  const int64_t T = (N + BN - 1) / BN;
  const int pairs = static_cast<int>(T < kNumSMs / 2 ? T : kNumSMs / 2);
  const int groups = 8 * pairs;  // 2 CTAs x 4 epilogue warps
  if (groups < 2 * k || groups > kBootCap) return 0;
  const int64_t want_rows = N / 4000 * k;
  int tiles = static_cast<int>((want_rows + static_cast<int64_t>(BN) * pairs - 1) / (static_cast<int64_t>(BN) * pairs));
  if (tiles < 1) tiles = 1;
  const int64_t per_chunk = T / pairs;  // the shortest chunk
  if (tiles > 1 && tiles * 4 > per_chunk) return 0;
  if (boot_tiles) *boot_tiles = tiles;
  return pairs;
}

static GemmWs gemm_ws_layout(int64_t Q, int64_t N, int64_t D, int dtype, int k, int have_planes, int have_cinv) {
  GemmWs w{};
  const int mode = mode_for(dtype);
  D = geometry_dim(D, dtype);
  const int qblocks = static_cast<int>((Q + 2 * BM - 1) / (2 * BM));
  Phase ph[kMaxPhases];
  const bool swap = swap_applies(Q, N, D);
  const bool dense0 = !swap;  // K2 scores its first tiles densely (see launch_gemm_topk)
  const int np = plan_phases(N, qblocks, k, ph, kMaxPhases, swap, dense0 ? dense0_tiles(Q, N) : 0);
  int maxc = 1;
  for (int i = 0; i < np; ++i) maxc = ph[i].chunks > maxc ? ph[i].chunks : maxc;
  w.boot_tiles = 0;
  w.boot_pairs = boot_pairs_for(Q, N, D, k, &w.boot_tiles);
  if (w.boot_pairs > maxc) maxc = w.boot_pairs;
  w.k2_boot_chunks = 0;
  w.k2_boot_coarse = 0;
  w.k2_boot_tiles = k2_boot_plan(Q, N, D, k, &w.k2_boot_chunks, &w.k2_boot_coarse);
  if (w.k2_boot_chunks > maxc) maxc = w.k2_boot_chunks;
  w.max_chunks = maxc;
  const int64_t dp = (D + 63) / 64 * 64;  // elements of a screen-plane row
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes, 1024);
    return o;
  };
  w.q_planes = take(mode == 2 ? static_cast<size_t>(Q) * dp * 2 : (mode == 5 ? static_cast<size_t>(Q) * D * 2 : 0));  // int8: query codes
  w.c_planes = take((mode == 2 && !have_planes) ? static_cast<size_t>(N) * dp * 2 : 0);
  w.qinv = take(static_cast<size_t>(Q) * 4);
  w.cinv = take(!have_cinv ? static_cast<size_t>(N) * 4 : 0);
  w.tau = take(static_cast<size_t>(Q) * 4);
  w.overflow = take(static_cast<size_t>(Q) * 4 + 32);  // + the grid-barrier counters of the boot mode (zeroed with the flags)
  w.kc = carry_cap(k, mode);
  for (int i = 0; i < 2; ++i) {
    w.carry[i] = take(static_cast<size_t>(Q) * w.kc * 8);
    w.carry_cnt[i] = take(static_cast<size_t>(Q) * 4);
  }
  w.seg_cap = seg_cap_for(k);
  const int halves = swap ? 2 : epi_warps(1) / 4;
  w.cand = take(static_cast<size_t>(Q) * maxc * halves * w.seg_cap * 8);
  w.cand_cnt = take(static_cast<size_t>(Q) * maxc * halves * 4);
  w.scratch = take(static_cast<size_t>(kNumSMs) * kEpiWarps * kSegCapMax * 8);  // in-kernel compaction scratch
  w.dense0 = take(dense0 ? static_cast<size_t>(Q) * dense0_tiles(Q, N) * BN * 4 : 0);
  size_t gmax_bytes = w.boot_pairs ? static_cast<size_t>((Q + 31) / 32 * 32) * 8 * w.boot_pairs * 4 : 0;
  if (w.k2_boot_tiles) gmax_bytes = static_cast<size_t>(Q) * w.k2_boot_chunks * w.k2_boot_tiles * (BN / 32) * 4;  // upper bound for the coarse form
  w.gmax = take(gmax_bytes);
  w.total = off + 1024;
  return w;
}

bool gemm_topk_supported(int64_t Q, int64_t N, int64_t D, int dtype, int k, const uint8_t* mask) {
  (void)mask;
  if (Q < 1 || N < 1 || k > ICR_MAX_K) return false;
  if (dtype != ICR_F32 && D % 8 != 0) return false;
  if (N > (static_cast<int64_t>(1) << 31) - BN || Q > (static_cast<int64_t>(1) << 30)) return false;
  return true;
}

size_t gemm_topk_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int have_planes) {
  // sized without cached inverse norms so that one figure covers both cases
  return gemm_ws_layout(Q, N, D, dtype, k, have_planes, 0).total;
}

// the filtering GEMM launches of a call, with or without per-query exclusions
static int launch_filter(bool swap, int which, int grid, const CUtensorMap& map_a, const CUtensorMap& map_b, const GemmArgs& g, cudaStream_t st,
                         const HistSelectArgs& sel = HistSelectArgs{}) {
  if (swap) return g.xbits ? launch_swap_variant<true>(which, grid, map_a, map_b, g, st, sel) : launch_swap_variant<false>(which, grid, map_a, map_b, g, st, sel);
  return g.xbits ? launch_gemm_variant<false, true>(which, grid, map_a, map_b, g, st) : launch_gemm_variant<false, false>(which, grid, map_a, map_b, g, st);
}

int launch_gemm_topk(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D,
                     int dtype, const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* mask, const uint32_t* xbits, int k,
                     int64_t row_offset, float* out_scores, int64_t* out_ids, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int mode = mode_for(dtype);
  const GemmWs L = gemm_ws_layout(Q, N, D, dtype, k, cat_planes != nullptr, cat_inv_norms != nullptr);
  if (ws_bytes < L.total) {
    set_error("gemm_topk: workspace %zu < %zu", ws_bytes, L.total);
    return ICR_ERR_WORKSPACE;
  }
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~static_cast<uintptr_t>(1023));
  const int qblocks = static_cast<int>((Q + 2 * BM - 1) / (2 * BM));
  const int64_t dp = (D + 63) / 64 * 64;
  int rc;
  GemmArgs g{};
  g.Q = static_cast<int>(Q);
  g.N = static_cast<int>(N);
  g.k = k;
  g.qblocks = qblocks;
  g.mask = mask;
  g.xbits = xbits;
  g.xld = Q;
  g.tau = reinterpret_cast<float*>(base + L.tau);
  g.overflow = reinterpret_cast<unsigned int*>(base + L.overflow);
  g.cand = reinterpret_cast<uint64_t*>(base + L.cand);
  g.cand_cnt = reinterpret_cast<int*>(base + L.cand_cnt);
  g.seg_cap = L.seg_cap;
  g.compact_scratch = reinterpret_cast<uint64_t*>(base + L.scratch);
  // what every select of this call shares
  HistSelectArgs sa{};
  sa.Q = Q;
  sa.k = k;
  sa.kc = L.kc;
  sa.seg_keys = g.cand;
  sa.seg_cnt = g.cand_cnt;
  sa.seg_stride = sa.seg_cap = g.seg_cap;
  sa.id_offset = row_offset;
  sa.raw_keys = 1;  // the only producer of segments is the GEMM epilogue
  sa.xbits = xbits;
  sa.xld = Q;
  CUtensorMap map_a, map_b;
  const void* q_operand = queries;  // what the TMA map of the swapped kernel is built over
  int64_t q_cols = D, q_ld = ldq;
  // the query-side preparation kernels also initialise tau (-inf: phase 0 admits every row), the overflow flags and the
  // grid-barrier counters behind them
  if (mode == 2) {
    uint16_t* qp = reinterpret_cast<uint16_t*>(base + L.q_planes);
    float* qinv = reinterpret_cast<float*>(base + L.qinv);
    if ((rc = launch_screen_plane(static_cast<const float*>(queries), Q, D, ldq, qp, qinv, st, const_cast<float*>(g.tau), g.overflow))) return rc;
    const uint16_t* cp = cat_planes;
    const float* cinv = cat_inv_norms;
    if (!cp) {
      uint16_t* built = reinterpret_cast<uint16_t*>(base + L.c_planes);
      float* built_inv = cinv ? nullptr : reinterpret_cast<float*>(base + L.cinv);
      if ((rc = launch_screen_plane(static_cast<const float*>(catalog), N, D, ldc, built, built_inv, st))) return rc;
      cp = built;
      if (!cinv) cinv = built_inv;
    } else if (!cinv) {
      float* built_inv = reinterpret_cast<float*>(base + L.cinv);
      if ((rc = launch_row_inv_norms(catalog, N, D, ldc, dtype, built_inv, st))) return rc;
      cinv = built_inv;
    }
    if ((rc = make_map(&map_a, qp, Q, dp, dp, false))) return rc;
    if ((rc = make_map(&map_b, cp, N, dp, dp, false))) return rc;
    g.kb_per_term = static_cast<int>(dp / BK);
    g.plane_stride = 0;
    g.acc_scale = 1.0f / 65536.0f;
    g.band = kScreenBandRaw;
    q_operand = qp;
    q_cols = q_ld = dp;
    sa.band = kScreenBandRaw;
    sa.overflow = g.overflow;
    sa.rs_q = static_cast<const float*>(queries);
    sa.rs_ldq = ldq;
    sa.rs_cat = static_cast<const float*>(catalog);
    sa.rs_ldc = ldc;
    sa.rs_N = N;
    sa.rs_D = static_cast<int>(D);
    sa.rs_qinv = qinv;
    sa.rs_cinv = cinv;
    sa.mask = mask;  // the exact ranking of an overflowed query walks the catalog itself
  } else if (mode == 5) {
    // int8 rows: the fp32 queries are quantised into the workspace (I8Rows, as K1 and icr_quantize_rows do), their factors
    // are the query scale of the select; the catalog's factors are required (icr_cos_topk checked them)
    int8_t* qc = reinterpret_cast<int8_t*>(base + L.q_planes);
    float* qinv = reinterpret_cast<float*>(base + L.qinv);
    if ((rc = launch_quantize_rows(static_cast<const float*>(queries), Q, D, ldq, qc, D, qinv, st, const_cast<float*>(g.tau), g.overflow))) return rc;
    const int64_t d2 = D / 2;  // D % 16 == 0: the codes as a 16-bit matrix of D / 2 columns
    if ((rc = make_map(&map_a, qc, Q, d2, d2, false))) return rc;
    if ((rc = make_map(&map_b, catalog, N, d2, ldc / 2, false))) return rc;
    g.kb_per_term = static_cast<int>((d2 + BK - 1) / BK);
    g.plane_stride = 0;
    g.acc_scale = 1.0f;
    g.qinv = qinv;
    g.cinv = cat_inv_norms;
    q_operand = qc;
    q_cols = q_ld = d2;
  } else {
    float* qinv = reinterpret_cast<float*>(base + L.qinv);
    if ((rc = launch_row_inv_norms(queries, Q, D, ldq, dtype, qinv, st, const_cast<float*>(g.tau), g.overflow))) return rc;
    const float* cinv = cat_inv_norms;
    if (!cinv) {
      float* built = reinterpret_cast<float*>(base + L.cinv);
      if ((rc = launch_row_inv_norms(catalog, N, D, ldc, dtype, built, st))) return rc;
      cinv = built;
    }
    if ((rc = make_map(&map_a, queries, Q, D, ldq, mode == 1))) return rc;
    if ((rc = make_map(&map_b, catalog, N, D, ldc, mode == 1))) return rc;
    g.kb_per_term = static_cast<int>((D + BK - 1) / BK);
    g.plane_stride = 0;
    g.acc_scale = 1.0f;
    g.qinv = qinv;
    g.cinv = cinv;
  }
  sa.out_scale = g.acc_scale;
  sa.out_qscale = g.qinv;
  const bool swap = swap_applies(Q, N, geometry_dim(D, dtype));
  const bool astat = g.kb_per_term <= kAStatMaxKB;
  int which;
  if (swap) which = mode == 1 ? 4 : (mode == 4 ? 3 : (mode == 5 ? 12 : 7));
  else if (mode == 2) which = astat ? 6 : 5;
  else if (mode == 1) which = astat ? 2 : 1;
  else if (mode == 5) which = astat ? 11 : 10;
  else which = astat ? 9 : 8;
  if (swap) {
    g.qpad = static_cast<int>((Q + 31) / 32 * 32);
    if ((rc = make_map(&map_a, q_operand, Q, q_cols, q_ld, mode == 1, g.qpad / 2))) return rc;
  }

  if (L.boot_pairs > 0) {
    // ---- single launch over the whole catalog: thresholds bootstrapped in the kernel, then one select ----
    g.boot = L.boot_tiles;
    g.gmax = reinterpret_cast<float*>(base + L.gmax);
    g.gsync = g.overflow + Q;  // zeroed by the query preparation kernel together with the flags
    g.tile_begin = 0;
    g.tile_end = static_cast<int>((N + BN - 1) / BN);
    g.chunks = L.boot_pairs;
    HistSelectArgs sp = sa;
    sp.nseg = g.chunks * 2;
    sp.carry_out = mode == 2 ? reinterpret_cast<uint64_t*>(base + L.carry[0]) : nullptr;
    sp.carry_cnt_out = mode == 2 ? reinterpret_cast<int*>(base + L.carry_cnt[0]) : nullptr;
    sp.out_scores = out_scores;
    sp.out_ids = out_ids;
    // The select moves into the kernel's tail when a query's survivors are expected to be few: the bootstrap threshold is the
    // k-th largest of `groups` maxima of 32 rows each, so ~N * k / (32 * groups * boot_tiles) rows pass it (plus the screening
    // band's share): that has to stay under a third of the tail's buffer (a query that overflows it anyway is still exact). Larger cases (catalogs that
    // stream from HBM, where the select is a few percent of the call) keep the separate select launch.
    const double expect = static_cast<double>(N) * k / (256.0 * L.boot_pairs * L.boot_tiles);
    // One CTA finishes one query at a time: more queries than CTAs means rounds, which only short lists (k <= 32) afford
    // (Q = 256 on the 49,688-row catalog: k = 10 75 us against 89 us with the select launch, k = 100 134 against 118).
    const bool one_round = Q <= 2 * L.boot_pairs || k <= 32;
    g.fuse_select = (one_round && sp.nseg <= kTailSegs && expect <= kTailCap / 3 && (mode != 2 || D % 4 == 0)) ? 1 : 0;
    if ((rc = launch_filter(true, which, 2 * L.boot_pairs, map_a, map_b, g, st, sp))) return rc;
    if (g.fuse_select) return ICR_OK;
    return run_select(sp, Q, st);
  }

  if (L.k2_boot_tiles > 0) {
    // ---- K2, single launch over the whole catalog (thresholds bootstrapped in the kernel), then one select ----
    g.boot = L.k2_boot_tiles;
    g.boot_coarse = L.k2_boot_coarse;
    g.gmax = reinterpret_cast<float*>(base + L.gmax);
    g.gsync = g.overflow + Q;
    g.tile_begin = 0;
    g.tile_end = static_cast<int>((N + BN - 1) / BN);
    g.chunks = L.k2_boot_chunks;
    const int items = qblocks * g.chunks;
    const int pairs = items < kNumSMs / 2 ? items : kNumSMs / 2;
    if ((rc = launch_filter(false, which, 2 * pairs, map_a, map_b, g, st))) return rc;
    HistSelectArgs sp = sa;
    sp.nseg = g.chunks * (epi_warps(1) / 4);
    sp.carry_out = mode == 2 ? reinterpret_cast<uint64_t*>(base + L.carry[0]) : nullptr;
    sp.carry_cnt_out = mode == 2 ? reinterpret_cast<int*>(base + L.carry_cnt[0]) : nullptr;
    sp.out_scores = out_scores;
    sp.out_ids = out_ids;
    return run_select(sp, Q, st);
  }

  // ---- first phase, dense: rows of the first dense0_tiles() tiles have no threshold to beat yet, so every score would
  // be appended through uncoalesced 8-byte stores (measured: 27 us per tile). They are written as a dense [Q, 1024]
  // score matrix instead (full 128-byte lines) and the select builds its keys from that.
  Phase ph[kMaxPhases];
  const int T = static_cast<int>((N + BN - 1) / BN);
  const bool dense0 = !swap;  // K2 only
  int done_phases = 0;
  if (dense0) {
    const int kDense0Tiles = dense0_tiles(Q, N);
    const int T0 = T < kDense0Tiles ? T : kDense0Tiles;
    float* d0 = reinterpret_cast<float*>(base + L.dense0);
    GemmArgs gd = g;
    gd.tile_begin = 0;
    gd.tile_end = T0;
    gd.chunks = T0;
    gd.dense_out = d0;
    gd.dense_ld = static_cast<int64_t>(kDense0Tiles) * BN;
    gd.dense_raw = 1;
    const int items = qblocks * T0;
    const int pairs = items < kNumSMs / 2 ? items : kNumSMs / 2;
    if ((rc = launch_gemm_variant<true>(which, 2 * pairs, map_a, map_b, gd, st))) return rc;
    const bool last = (T0 >= T);
    HistSelectArgs s0 = sa;
    s0.nseg = 0;
    const bool keep0 = !last || mode == 2;  // a screened search hands its final candidates to the re-scoring kernel through the carry
    s0.carry_out = keep0 ? reinterpret_cast<uint64_t*>(base + L.carry[0]) : nullptr;
    s0.carry_cnt_out = keep0 ? reinterpret_cast<int*>(base + L.carry_cnt[0]) : nullptr;
    s0.tau_out = last ? nullptr : const_cast<float*>(g.tau);
    s0.out_scores = last ? out_scores : nullptr;
    s0.out_ids = last ? out_ids : nullptr;
    s0.dense = d0;
    s0.dense_ld = gd.dense_ld;
    s0.dense_rows = static_cast<int>(N < static_cast<int64_t>(T0) * BN ? N : static_cast<int64_t>(T0) * BN);
    s0.mask = mask;
    if ((rc = run_select(s0, Q, st))) return rc;
    if (last) return ICR_OK;
    done_phases = 1;
  }
  const int np = plan_phases(N, qblocks, k, ph, kMaxPhases, swap, dense0 ? dense0_tiles(Q, N) : 0);
  for (int pp = 0; pp < np; ++pp) {
    const int p = pp + done_phases;  // index for the carry ping-pong
    g.tile_begin = ph[pp].tile_begin;
    g.tile_end = ph[pp].tile_end;
    g.chunks = ph[pp].chunks;
    const int items = qblocks * g.chunks;
    const int pairs = items < kNumSMs / 2 ? items : kNumSMs / 2;
    const int grid = 2 * pairs;  // whole CTA pairs (cluster dims 2x1x1)
    if ((rc = launch_filter(swap, which, grid, map_a, map_b, g, st))) return rc;
    const bool last = (pp == np - 1);
    const int cur = p & 1, prev = cur ^ 1;
    HistSelectArgs sp = sa;
    sp.nseg = g.chunks * (swap ? 2 : epi_warps(1) / 4);
    sp.carry_in = p > 0 ? reinterpret_cast<uint64_t*>(base + L.carry[prev]) : nullptr;
    sp.carry_cnt_in = p > 0 ? reinterpret_cast<int*>(base + L.carry_cnt[prev]) : nullptr;
    const bool keep = !last || mode == 2;
    sp.carry_out = keep ? reinterpret_cast<uint64_t*>(base + L.carry[cur]) : nullptr;
    sp.carry_cnt_out = keep ? reinterpret_cast<int*>(base + L.carry_cnt[cur]) : nullptr;
    sp.tau_out = last ? nullptr : const_cast<float*>(g.tau);
    sp.out_scores = last ? out_scores : nullptr;  // raw key scores -> cosines (or exact re-scoring) on the way out
    sp.out_ids = last ? out_ids : nullptr;
    if ((rc = run_select(sp, Q, st))) return rc;
  }
  return ICR_OK;
}

// ---- K2': dense cosine similarity out[q][n] on the same tensor-core main loop -----------------------------
size_t gemm_dense_workspace_bytes(int64_t Qa, int64_t Nb, int64_t D, int dtype) {
  const int64_t dp2 = 2 * ((D + 63) / 64 * 64);
  size_t b = 4096;
  if (dtype == ICR_F32) b += align_up(static_cast<size_t>(Qa) * dp2 * 2, 1024) + align_up(static_cast<size_t>(Nb) * dp2 * 2, 1024);
  else b += align_up(static_cast<size_t>(Qa) * 4, 1024) + align_up(static_cast<size_t>(Nb) * 4, 1024);
  return b;
}

int launch_gemm_dense(const void* a, int64_t Qa, int64_t lda, const void* b, int64_t Nb, int64_t ldb, int64_t D, int dtype, float* out,
                      int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (ws_bytes < gemm_dense_workspace_bytes(Qa, Nb, D, dtype)) {
    set_error("gemm_dense: workspace too small");
    return ICR_ERR_WORKSPACE;
  }
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~static_cast<uintptr_t>(1023));
  const int64_t dp = (D + 63) / 64 * 64;
  const int qblocks = static_cast<int>((Qa + 2 * BM - 1) / (2 * BM));
  const int tiles = static_cast<int>((Nb + BN - 1) / BN);
  int rc;
  GemmArgs g{};
  g.Q = static_cast<int>(Qa);
  g.N = static_cast<int>(Nb);
  g.k = 1;
  g.qblocks = qblocks;
  g.seg_cap = 256;
  g.dense_out = out;
  g.dense_ld = ldo;
  g.tile_begin = 0;
  g.tile_end = tiles;
  CUtensorMap map_a, map_b;
  int which;
  if (dtype == ICR_F32) {
    uint16_t* ap = reinterpret_cast<uint16_t*>(base);
    uint16_t* bp = reinterpret_cast<uint16_t*>(base + align_up(static_cast<size_t>(Qa) * 2 * dp * 2, 1024));
    if ((rc = launch_split_planes(static_cast<const float*>(a), Qa, D, lda, ap, st))) return rc;
    if ((rc = launch_split_planes(static_cast<const float*>(b), Nb, D, ldb, bp, st))) return rc;
    if ((rc = make_map(&map_a, ap, Qa, 2 * dp, 2 * dp, false))) return rc;
    if ((rc = make_map(&map_b, bp, Nb, 2 * dp, 2 * dp, false))) return rc;
    g.kb_per_term = static_cast<int>(dp / BK);
    g.plane_stride = static_cast<int>(dp);
    g.acc_scale = 1.0f / 65536.0f;
    which = 0;
  } else {
    float* qinv = reinterpret_cast<float*>(base);
    float* cinv = reinterpret_cast<float*>(base + align_up(static_cast<size_t>(Qa) * 4, 1024));
    if ((rc = launch_row_inv_norms(a, Qa, D, lda, dtype, qinv, st))) return rc;
    if ((rc = launch_row_inv_norms(b, Nb, D, ldb, dtype, cinv, st))) return rc;
    const bool bf16 = dtype == ICR_BF16;
    if ((rc = make_map(&map_a, a, Qa, D, lda, bf16))) return rc;
    if ((rc = make_map(&map_b, b, Nb, D, ldb, bf16))) return rc;
    g.kb_per_term = static_cast<int>((D + BK - 1) / BK);
    g.acc_scale = 1.0f;
    g.qinv = qinv;
    g.cinv = cinv;
    const bool astat = g.kb_per_term <= kAStatMaxKB;
    which = bf16 ? (astat ? 2 : 1) : (astat ? 9 : 8);
  }
  // work items: (query block, chunk of tiles); enough chunks to fill the pairs a few times over
  const int npairs = kNumSMs / 2;
  int chunks = (3 * npairs + qblocks - 1) / qblocks;
  if (chunks > tiles) chunks = tiles;
  if (chunks < 1) chunks = 1;
  g.chunks = chunks;
  const int items = qblocks * chunks;
  const int grid = 2 * (items < npairs ? items : npairs);
  return launch_gemm_variant<true>(which, grid, map_a, map_b, g, st);
}

}  // namespace icr
