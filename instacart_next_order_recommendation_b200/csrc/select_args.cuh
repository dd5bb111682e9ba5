// Arguments of the selection kernels (select_hist.cu), shared with their callers (gemm_topk.cu, api.cu).
#pragma once

#include "common.cuh"

namespace icr {

// Screening mode of fp32 catalogs. The tensor-core sweep scores with ONE fp16 plane per operand (11 significant
// bits): screened = accumulator / 65536 differs from the exact cosine by at most eps = 2 * 2^-11 (Cauchy-Schwarz over
// the two rounding-error vectors, |x_lo| <= 2^-11 |x|) + the fp32 accumulation error of the tensor cores (< 5e-5 for
// K <= 4096). A row of the exact top-k therefore has a screened score >= (k-th best screened score) - 2 eps, so the
// selection keeps every key within `band` = 2 eps (+ margin) below the k-th screened score, and only those few rows
// (k + ~10 on a 50k-row catalog) are re-scored exactly in fp32. Raw units: accumulator = 65536 * cosine.
constexpr float kScreenBandRaw = 140.0f;  // 2 * (64.05 + 3.0) raw units = 2.05e-3 in cosine, rounded up

struct HistSelectArgs {
  const uint64_t* seg_keys;  // [Q][nseg][seg_stride]
  const int* seg_cnt;        // [Q][nseg]
  int nseg;
  int seg_stride;
  int seg_cap;
  const uint64_t* carry_in;  // [Q][kc] or null
  const int* carry_cnt_in;   // [Q]
  uint64_t* carry_out;       // [Q][kc] or null (unsorted set)
  int* carry_cnt_out;        // [Q]
  float* tau_out;            // [Q] or null
  float* out_scores;         // [Q][k] or null (sorted descending)
  int64_t* out_ids;          // [Q][k]
  int64_t id_offset;
  int k;
  int kc;                    // keys carried per query: k (exact keys) or k + band capacity (screened keys)
  int64_t Q;
  float out_scale;          // final score = key score * out_scale * (out_qscale ? out_qscale[q] : 1)
  const float* out_qscale;  // [Q] or null
  int raw_keys;             // segments hold (score bits, ~row) as the GEMM epilogue writes them; carry keys are ordered
  // dense front end (first phase of K2): instead of segments, row q of a [Q][dense_ld] score matrix holds the raw
  // scores of catalog rows 0 .. dense_rows-1; rows flagged in `mask` are skipped
  const float* dense;
  int64_t dense_ld;
  int dense_rows;
  const uint8_t* mask;
  // list front end (K4 shard merge): G lists of list_k (score, id) pairs per query, laid out [G][Q][list_k]; id < 0 = empty
  const float* list_scores;
  const int64_t* list_ids;
  int list_g, list_k;
  // ---- screened keys (band > 0): see kScreenBandRaw --------------------------------------------------------------
  float band;               // raw units; 0 = keys carry exact scores
  unsigned int* overflow;   // [Q] set when more keys than kc fall inside the band (or a GEMM segment could not be cut
                            // back): the final phase then ranks the whole catalog for that query, exactly
  // exact re-scoring in the final phase: fp32 rows of both operands and their inverse norms
  const float* rs_q;        // [Q][rs_D], row stride rs_ldq
  int64_t rs_ldq;
  const float* rs_cat;      // [rs_N][rs_D], row stride rs_ldc
  int64_t rs_ldc;
  int64_t rs_N;
  int rs_D;
  const float* rs_qinv;     // [Q]
  const float* rs_cinv;     // [rs_N]
  // per-query exclusions (Exclusions::bits, ld = Q): read by the dense front end and the whole-catalog rankings of the
  // BITS instantiations only; the segments of the GEMM epilogue are already filtered
  const uint32_t* xbits;
  int64_t xld;
  __device__ __forceinline__ Exclusions excl() const { return Exclusions{mask, xbits, xld}; }
};

int run_select(const HistSelectArgs& a, int64_t Q, cudaStream_t st);

}  // namespace icr
