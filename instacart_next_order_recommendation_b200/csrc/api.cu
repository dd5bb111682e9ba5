// extern "C" entry points of libicr_b200.so (declared in include/icr_b200.h).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "peer.cuh"

namespace icr {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return ICR_ERR_CUDA;
}
void count_launch() { ++g_launches; }

// ---- optional timing of the dominant kernel (bench.py's roofline leg) -------------------------
static thread_local bool g_prof_on = false;
static thread_local int g_prof_kernel = 0, g_prof_terms = 1;
static thread_local std::vector<cudaEvent_t> g_prof_events;  // pairs: begin, end
static thread_local size_t g_prof_used = 0;

void profile_begin(int kernel_id, int mma_terms, cudaStream_t st) {
  if (!g_prof_on) return;
  if (g_prof_used + 2 > g_prof_events.size()) {
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
    g_prof_events.push_back(a);
    g_prof_events.push_back(b);
  }
  g_prof_kernel = kernel_id;
  g_prof_terms = mma_terms;
  cudaEventRecord(g_prof_events[g_prof_used], st);
}
void profile_end(cudaStream_t st) {
  if (!g_prof_on || g_prof_used + 2 > g_prof_events.size()) return;
  cudaEventRecord(g_prof_events[g_prof_used + 1], st);
  g_prof_used += 2;
}

// kernels' host launchers (defined in the other translation units)
int launch_row_inv_norms(const void* x, int64_t rows, int64_t dim, int64_t ld, int dtype, float* inv, cudaStream_t st, float* tau_init = nullptr,
                         unsigned int* ovf_init = nullptr);
int launch_split_planes(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* planes, cudaStream_t st);
int launch_screen_plane(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* plane, float* inv, cudaStream_t st, float* tau_init = nullptr,
                        unsigned int* ovf_init = nullptr);
int launch_convert_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx, void* out, int64_t ldo, int out_dtype, int normalize,
                        cudaStream_t st);
int launch_peer_exchange_merge(const float* scores, const int64_t* ids, int64_t Q, int k, const PeerTail& peer, float* os, int64_t* oi,
                               cudaStream_t st);
bool gemv_peer_tail_fits(int Q, int k, int world);
int launch_peer_exchange(const float* scores, const int64_t* ids, int64_t n, int rank, int world, const uint64_t* peer_buffers, uint32_t epoch,
                         int64_t n_max, cudaStream_t st);
int gemv_grid(int64_t N);
int launch_gemv_topk(const void* cat, int64_t N, int64_t ldc, int D, int dtype, const void* q, int64_t ldq, int Q,
                     const uint8_t* mask, const uint32_t* xbits, int64_t xld, int k, uint64_t* part_keys, int* part_cnt, int grid, float* out_scores, int64_t* out_ids,
                     int64_t id_offset, unsigned int* done_counter, cudaStream_t st, const float* cat_inv, const PeerTail* peer = nullptr,
                     float* fin_scores = nullptr, int64_t* fin_ids = nullptr);
size_t select_scratch_bytes(int64_t Q, int nseg, int seg_cap, int k);
int launch_select(const uint64_t* seg_keys, const int* seg_cnt, int64_t Q, int nseg, int seg_stride, int seg_cap,
                  const uint64_t* carry_in, const int* carry_cnt_in, uint64_t* carry_out, int* carry_cnt_out,
                  float* tau_out, float* out_scores, int64_t* out_ids, int64_t id_offset, int k, void* scratch,
                  size_t scratch_bytes, cudaStream_t st);
int launch_merge_lists(const float* cs, const int64_t* ci, int64_t Q, int G, int k_in, int k_out, float* os, int64_t* oi,
                       cudaStream_t st);
int launch_cos_sim_dense(const void* a, int64_t Qa, int64_t lda, const void* b, int64_t Nb, int64_t ldb, int D, int dtype,
                         const float* inva, const float* invb, float* out, int64_t ldo, cudaStream_t st);
// GEMM path (gemm_topk.cu)
size_t gemm_topk_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int have_planes);
int launch_gemm_topk(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D,
                     int dtype, const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* mask, const uint32_t* xbits, int k,
                     int64_t row_offset, float* out_scores, int64_t* out_ids, void* ws, size_t ws_bytes, cudaStream_t st);
bool gemm_topk_supported(int64_t Q, int64_t N, int64_t D, int dtype, int k, const uint8_t* mask);
size_t gemm_dense_workspace_bytes(int64_t Qa, int64_t Nb, int64_t D, int dtype);
int launch_gemm_dense(const void* a, int64_t Qa, int64_t lda, const void* b, int64_t Nb, int64_t ldb, int64_t D, int dtype, float* out,
                      int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st);
// the tensor-core dense path pays off once there is a tile's worth of work; below that the CUDA-core kernel wins
static bool dense_use_gemm(int64_t Qa, int64_t Nb, int64_t D, int dtype) {
  if (dtype != ICR_F32 && D % 8 != 0) return false;
  return Qa >= 64 && Nb >= 1024;
}

int launch_mnrl_dispatch(const MnrlArgs& g, int dtype, bool bwd, cudaStream_t st);
int launch_scale2(const void* x0, const void* x1, int64_t n, int dtype, const float* s, void* o0, void* o1, cudaStream_t st);
// tensor-core MNRL (mnrl_tc.cu)
bool mnrl_tc_applies(int64_t B, int64_t Bc, int64_t D);
size_t mnrl_tc_workspace_bytes(int64_t B, int64_t Bc, int64_t D);
int launch_mnrl_tc(const MnrlArgs& m, int dtype, int mode, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_query_exclusion_bits(const int64_t* offsets, const int64_t* rows, int64_t Q, int64_t N, uint32_t* bits, cudaStream_t st);
int launch_ir_metrics(const int64_t* ids, int64_t Q, int K, int64_t ld, const int64_t* rel_offsets, const int64_t* rel_rows,
                      const int32_t* n_relevant, const int32_t* kinds, const int32_t* ks, int M, double* per_query, double* means,
                      cudaStream_t st);

static int elem_size(int dtype) { return dtype == ICR_F32 ? 4 : 2; }
static int vec_elems(int dtype) { return dtype == ICR_F32 ? 4 : 8; }

static int check_matrix(const char* name, const void* p, int64_t rows, int64_t dim, int64_t ld, int dtype) {
  if (dtype != ICR_F32 && dtype != ICR_BF16 && dtype != ICR_F16) {
    set_error("%s: unsupported dtype %d (0 = f32, 1 = bf16, 2 = f16)", name, dtype);
    return ICR_ERR_DTYPE;
  }
  if (rows < 0 || dim <= 0 || ld < dim) {
    set_error("%s: bad shape rows=%lld dim=%lld ld=%lld", name, (long long)rows, (long long)dim, (long long)ld);
    return ICR_ERR_ARG;
  }
  if (rows > 0 && p == nullptr) {
    set_error("%s: null pointer", name);
    return ICR_ERR_ARG;
  }
  if (dim % vec_elems(dtype) != 0) {
    set_error("%s: embedding dim %lld must be a multiple of %d for 16-byte vector access", name, (long long)dim, vec_elems(dtype));
    return ICR_ERR_ALIGN;
  }
  if ((reinterpret_cast<uintptr_t>(p) & 15) != 0 || (ld * elem_size(dtype)) % 16 != 0) {
    set_error("%s: base pointer and row stride must be 16-byte aligned", name);
    return ICR_ERR_ALIGN;
  }
  return ICR_OK;
}

static int check_device() {
  int dev = 0;
  ICR_CUDA_CHECK(cudaGetDevice(&dev));
  static thread_local int cached_dev = -1, cached_ok = 0;
  if (dev != cached_dev) {
    int major = 0;
    ICR_CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    cached_dev = dev;
    cached_ok = (major == 10);
  }
  if (!cached_ok) {
    set_error("device %d is not compute capability 10.x (B200); there is no fallback path", dev);
    return ICR_ERR_DEVICE;
  }
  return ICR_OK;
}

constexpr int kGemvQueryChunk = 252;  // queries per GEMV workspace round (multiple of 7)

static size_t gemv_ws_bytes(int64_t Q, int64_t N, int k) {
  const int grid = gemv_grid(N);
  const int64_t qc = Q < kGemvQueryChunk ? Q : kGemvQueryChunk;
  size_t b = 0;
  b += align_up(static_cast<size_t>(qc) * grid * k * sizeof(uint64_t), 256);
  b += align_up(static_cast<size_t>(qc) * grid * sizeof(int), 256);
  b += align_up(select_scratch_bytes(qc, grid, k, k), 256);
  return b + 512;  // + the merge counter
}

}  // namespace icr

using namespace icr;

extern "C" {

int icr_abi_version(void) { return ICR_ABI_VERSION; }
const char* icr_last_error_string(void) { return g_err; }
int icr_last_launch_count(void) { return g_launches; }

int icr_device_supported(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return ICR_ERR_CUDA;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return ICR_ERR_CUDA;
  return major == 10 ? 1 : 0;
}

int icr_profile_enable(int on) {
  g_prof_on = on != 0;
  g_prof_used = 0;
  return ICR_OK;
}

int icr_profile_collect(float* total_ms, int* launches, int* kernel_id, int* mma_terms) {
  float sum = 0.f;
  for (size_t i = 0; i + 1 < g_prof_used; i += 2) {
    ICR_CUDA_CHECK(cudaEventSynchronize(g_prof_events[i + 1]));
    float ms = 0.f;
    ICR_CUDA_CHECK(cudaEventElapsedTime(&ms, g_prof_events[i], g_prof_events[i + 1]));
    sum += ms;
  }
  if (total_ms) *total_ms = sum;
  if (launches) *launches = static_cast<int>(g_prof_used / 2);
  if (kernel_id) *kernel_id = g_prof_kernel;
  if (mma_terms) *mma_terms = g_prof_terms;
  g_prof_used = 0;
  return ICR_OK;
}

int icr_row_inv_norms(const void* x, int64_t rows, int64_t dim, int64_t ld, int dtype, float* inv_norms, void* stream) {
  g_launches = 0;
  int rc = check_matrix("row_inv_norms.x", x, rows, dim, ld, dtype);
  if (rc) return rc;
  if ((rc = check_device())) return rc;
  if (rows > 0 && !inv_norms) {
    set_error("row_inv_norms: null output");
    return ICR_ERR_ARG;
  }
  return launch_row_inv_norms(x, rows, dim, ld, dtype, inv_norms, static_cast<cudaStream_t>(stream));
}

int64_t icr_planes_row_elems(int64_t dim) { return 2 * ((dim + 63) / 64 * 64); }

int icr_split_f16_planes(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* planes, void* stream) {
  g_launches = 0;
  int rc = check_matrix("split_f16_planes.x", x, rows, dim, ld, ICR_F32);
  if (rc) return rc;
  if ((rc = check_device())) return rc;
  if (rows > 0 && (!planes || (reinterpret_cast<uintptr_t>(planes) & 127))) {
    set_error("split_f16_planes: planes must be non-null and 128-byte aligned");
    return ICR_ERR_ALIGN;
  }
  return launch_split_planes(x, rows, dim, ld, planes, static_cast<cudaStream_t>(stream));
}

int64_t icr_screen_plane_row_elems(int64_t dim) { return (dim + 63) / 64 * 64; }

int icr_screen_plane(const float* x, int64_t rows, int64_t dim, int64_t ld, uint16_t* plane, float* inv_norms, void* stream) {
  g_launches = 0;
  int rc = check_matrix("screen_plane.x", x, rows, dim, ld, ICR_F32);
  if (rc) return rc;
  if ((rc = check_device())) return rc;
  if (rows > 0 && (!plane || (reinterpret_cast<uintptr_t>(plane) & 127))) {
    set_error("screen_plane: plane must be non-null and 128-byte aligned");
    return ICR_ERR_ALIGN;
  }
  return launch_screen_plane(x, rows, dim, ld, plane, inv_norms, static_cast<cudaStream_t>(stream));
}

static int resolve_path(int path, int64_t Q, int64_t N, int64_t D, int dtype, int k, const uint8_t* mask) {
  if (path == ICR_PATH_GEMV || path == ICR_PATH_GEMM) return path;
  // small batches are HBM-bound GEMVs; larger ones are tensor-core work. bf16 and fp16 rows have the same bytes and the
  // same MMA rate, so every threshold below treats them alike
  int gemv_max_q = (dtype == ICR_F32) ? 7 : 3;
  // The tensor-core pipeline costs ~55 us of launches and selects on top of its stream, but streams a large catalog
  // closer to the HBM rate than the multi-query GEMV passes (measured, profiles/r01_notes.md): crossover ~256 MB
  // for 4-7 queries, ~640 MB for 2-3.
  const double cat_bytes = static_cast<double>(N) * static_cast<double>(D) * (dtype == ICR_F32 ? 4.0 : 2.0);
  if (cat_bytes >= 256e6 && gemv_max_q > 3) gemv_max_q = 3;
  // 2 GB catalogs, whole call: fp32 rows, 2-3 queries: one GEMV pass 0.36 ms against 0.40 ms on the tensor path (the pass
  // re-uses each row for all its queries and fp32 needs no unpacking); bf16 rows: 0.43 ms against 0.39 ms
  if (cat_bytes >= 640e6) gemv_max_q = (dtype == ICR_F32) ? 3 : 1;
  // rows shorter than 512 bytes leave the GEMV kernel instruction-bound even for one query (per-row reduction and
  // threshold test against 256 bytes of FMAs: 20 % of the HBM rate measured at D=128 bf16); the swapped tensor-core
  // kernel streams such a catalog at 74 % with the query padded to N=32
  if (cat_bytes >= 640e6 && D * (dtype == ICR_F32 ? 4 : 2) < 512) gemv_max_q = 0;
  if (Q > gemv_max_q && gemm_topk_supported(Q, N, D, dtype, k, mask)) return ICR_PATH_GEMM;
  return ICR_PATH_GEMV;
}

size_t icr_cos_topk_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int path, int have_planes) {
  path &= ~ICR_PATH_WS_RESIDENT;
  if (Q <= 0 || N <= 0 || k <= 0) return 256;
  if (path == ICR_PATH_AUTO) {
    const size_t a = gemv_ws_bytes(Q, N, k);
    const size_t b = gemm_topk_supported(Q, N, D, dtype, k, nullptr) ? gemm_topk_workspace_bytes(Q, N, D, dtype, k, have_planes) : 0;
    return a > b ? a : b;
  }
  if (path == ICR_PATH_GEMM) return gemm_topk_workspace_bytes(Q, N, D, dtype, k, have_planes);
  return gemv_ws_bytes(Q, N, k);
}

// `peer` != null (request-sized sharded call on the GEMV path, gemv_peer_tail_fits): the exchange and the global merge happen
// in the tail of the scoring kernel; out_* then receive the GLOBAL top-k and stage_* hold the shard's own lists.
// `excl_bits` (per-query exclusions, [ceil(N/32)][Q]) is null on the sharded entry.
static int cos_topk_impl(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D,
                         int dtype, const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* exclude_mask,
                         const uint32_t* excl_bits, int k,
                         int64_t row_offset, int path, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                         void* stream, const PeerTail* peer, float* stage_scores, int64_t* stage_ids) {
  int rc;
  if ((rc = check_matrix("cos_topk.queries", queries, Q, D, ldq, dtype))) return rc;
  if ((rc = check_matrix("cos_topk.catalog", catalog, N, D, ldc, dtype))) return rc;
  if (k < 1 || k > ICR_MAX_K) {
    set_error("cos_topk: k=%d outside [1, %d]", k, ICR_MAX_K);
    return ICR_ERR_K;
  }
  if (N >= 0xffffffffll) {
    set_error("cos_topk: a shard holds at most 2^32-2 rows (got %lld)", (long long)N);
    return ICR_ERR_ARG;
  }
  if (Q > 0 && (!out_scores || !out_ids)) {
    set_error("cos_topk: null output");
    return ICR_ERR_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(excl_bits) & 3) != 0) {
    set_error("cos_topk: excl_bits must be 4-byte aligned");
    return ICR_ERR_ALIGN;
  }
  if ((rc = check_device())) return rc;
  if (Q == 0) return ICR_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool ws_resident = (path & ICR_PATH_WS_RESIDENT) != 0;
  path &= ~ICR_PATH_WS_RESIDENT;
  const int p = resolve_path(path, Q, N, D, dtype, k, exclude_mask);
  const size_t need = icr_cos_topk_workspace_bytes(Q, N, D, dtype, k, p, cat_planes != nullptr);
  if (workspace_bytes < need || (need > 256 && !workspace)) {
    set_error("cos_topk: workspace %zu bytes < required %zu", workspace_bytes, need);
    return ICR_ERR_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
    set_error("cos_topk: workspace must be 256-byte aligned");
    return ICR_ERR_ALIGN;
  }
  if (p == ICR_PATH_GEMM) {
    if (!gemm_topk_supported(Q, N, D, dtype, k, exclude_mask)) {
      set_error("cos_topk: GEMM path does not support this problem (Q=%lld N=%lld D=%lld k=%d mask=%d)", (long long)Q,
                (long long)N, (long long)D, k, exclude_mask != nullptr);
      return ICR_ERR_ARG;
    }
    return launch_gemm_topk(queries, Q, ldq, catalog, N, ldc, D, dtype, cat_planes, cat_inv_norms, exclude_mask, excl_bits, k, row_offset,
                            out_scores, out_ids, workspace, workspace_bytes, st);
  }
  if (N == 0) {
    // nothing eligible: (-inf, -1) everywhere, produced by a select over zero segments
  }
  // ---- GEMV path: rounds of <= kGemvQueryChunk queries share the workspace -----------------------
  if (D > 4096) {
    set_error("cos_topk: GEMV path supports D <= 4096 (got %lld)", (long long)D);
    return ICR_ERR_ARG;
  }
  const int grid = gemv_grid(N);
  const int64_t qc = Q < kGemvQueryChunk ? Q : kGemvQueryChunk;
  char* w = static_cast<char*>(workspace);
  uint64_t* part_keys = reinterpret_cast<uint64_t*>(w);
  w += align_up(static_cast<size_t>(qc) * grid * k * sizeof(uint64_t), 256);
  int* part_cnt = reinterpret_cast<int*>(w);
  w += align_up(static_cast<size_t>(qc) * grid * sizeof(int), 256);
  w += align_up(select_scratch_bytes(qc, grid, k, k), 256);
  unsigned int* done_counter = reinterpret_cast<unsigned int*>(w);
  const size_t esz = elem_size(dtype);
  // the last CTA of every GEMV launch merges the per-CTA lists itself (no select launch on the latency path)
  if (!ws_resident) ICR_CUDA_CHECK(cudaMemsetAsync(done_counter, 0, 2 * sizeof(unsigned int), st));  // ticket + slab-chunk counter
  if (peer)  // the merging CTA of the one GEMV launch also exchanges and merges (gemv_topk.cu peer_tail_merge)
    return launch_gemv_topk(catalog, N, ldc, static_cast<int>(D), dtype, queries, ldq, static_cast<int>(Q), exclude_mask, nullptr, 0, k, part_keys, part_cnt,
                            grid, stage_scores, stage_ids, row_offset, done_counter, st, cat_inv_norms, peer, out_scores, out_ids);
  for (int64_t q0 = 0; q0 < Q; q0 += qc) {
    const int nq = static_cast<int>(Q - q0 < qc ? Q - q0 : qc);
    const char* qptr = static_cast<const char*>(queries) + q0 * ldq * esz;
    rc = launch_gemv_topk(catalog, N, ldc, static_cast<int>(D), dtype, qptr, ldq, nq, exclude_mask, excl_bits ? excl_bits + q0 : nullptr, Q, k,
                          part_keys, part_cnt, grid,
                          out_scores + q0 * k, out_ids + q0 * k, row_offset, done_counter, st, cat_inv_norms);
    if (rc) return rc;
  }
  return ICR_OK;
}

int icr_cos_topk_excl(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D,
                      int dtype, const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* exclude_mask,
                      const uint32_t* excl_bits, int k, int64_t row_offset, int path, float* out_scores, int64_t* out_ids, void* workspace,
                      size_t workspace_bytes, void* stream) {
  g_launches = 0;
  return cos_topk_impl(queries, Q, ldq, catalog, N, ldc, D, dtype, cat_planes, cat_inv_norms, exclude_mask, excl_bits, k, row_offset, path,
                       out_scores, out_ids, workspace, workspace_bytes, stream, nullptr, nullptr, nullptr);
}

int icr_cos_topk(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D,
                 int dtype, const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* exclude_mask, int k,
                 int64_t row_offset, int path, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                 void* stream) {
  return icr_cos_topk_excl(queries, Q, ldq, catalog, N, ldc, D, dtype, cat_planes, cat_inv_norms, exclude_mask, nullptr, k, row_offset, path,
                           out_scores, out_ids, workspace, workspace_bytes, stream);
}

int icr_query_exclusion_bits(const int64_t* offsets, const int64_t* rows, int64_t Q, int64_t N, uint32_t* bits, void* stream) {
  g_launches = 0;
  if (Q < 0 || N < 0 || N >= 0xffffffffll || (Q > 0 && !offsets) || (Q > 0 && N > 0 && !bits) || (reinterpret_cast<uintptr_t>(bits) & 3)) {
    set_error("query_exclusion_bits: bad arguments Q=%lld N=%lld (offsets, and bits for N > 0, must be non-null; bits 4-byte aligned)",
              (long long)Q, (long long)N);
    return ICR_ERR_ARG;
  }
  int rc;
  if ((rc = check_device())) return rc;
  if (Q == 0 || N == 0) return ICR_OK;
  return launch_query_exclusion_bits(offsets, rows, Q, N, bits, static_cast<cudaStream_t>(stream));
}

static int check_peer_args(const char* who, int64_t n, int rank, int world, const uint64_t* peer_buffers, uint32_t epoch, int64_t n_max) {
  if (world < 1 || world > ICR_MAX_PEERS || rank < 0 || rank >= world || n < 0 || n > n_max || !peer_buffers || epoch == 0) {
    set_error("%s: bad arguments n=%lld n_max=%lld rank=%d world=%d (<= %d) epoch=%u", who, (long long)n, (long long)n_max, rank, world,
              ICR_MAX_PEERS, epoch);
    return ICR_ERR_ARG;
  }
  for (int p = 0; p < world; ++p) {
    if (peer_buffers[p] == 0 || (peer_buffers[p] & 255)) {
      set_error("%s: buffer of rank %d is null or not 256-byte aligned", who, p);
      return ICR_ERR_ALIGN;
    }
  }
  return ICR_OK;
}

int icr_peer_exchange_merge(const float* scores, const int64_t* ids, int64_t Q, int k, int rank, int world, const uint64_t* peer_buffers,
                            uint32_t epoch, int64_t n_max, float* out_scores, int64_t* out_ids, void* stream) {
  g_launches = 0;
  int rc;
  if (Q < 0 || k < 1 || k > ICR_MAX_K) {
    set_error("peer_exchange_merge: bad arguments Q=%lld k=%d", (long long)Q, k);
    return ICR_ERR_ARG;
  }
  if ((rc = check_peer_args("peer_exchange_merge", Q * k, rank, world, peer_buffers, epoch, n_max))) return rc;
  if (Q > 0 && (!scores || !ids || !out_scores || !out_ids || (reinterpret_cast<uintptr_t>(scores) & 3) || (reinterpret_cast<uintptr_t>(ids) & 7))) {
    set_error("peer_exchange_merge: null or misaligned candidates / outputs");
    return ICR_ERR_ARG;
  }
  if ((rc = check_device())) return rc;
  const PeerTail tail = make_peer_tail(rank, world, peer_buffers, epoch, n_max);
  return launch_peer_exchange_merge(scores, ids, Q, k, tail, out_scores, out_ids, static_cast<cudaStream_t>(stream));
}

static size_t sharded_stage_bytes(int64_t Q, int k) {
  const size_t n = static_cast<size_t>(Q > 0 ? Q : 0) * static_cast<size_t>(k > 0 ? k : 0);
  return align_up(n * sizeof(float), 256) + align_up(n * sizeof(int64_t), 256);
}

size_t icr_cos_topk_sharded_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int path, int have_planes) {
  return align_up(icr_cos_topk_workspace_bytes(Q, N, D, dtype, k, path, have_planes), 256) + sharded_stage_bytes(Q, k);
}

int icr_cos_topk_sharded(const void* queries, int64_t Q, int64_t ldq, const void* catalog, int64_t N, int64_t ldc, int64_t D, int dtype,
                         const uint16_t* cat_planes, const float* cat_inv_norms, const uint8_t* exclude_mask, int k, int64_t row_offset,
                         int path, int rank, int world, const uint64_t* peer_buffers, uint32_t epoch, int64_t n_max, float* out_scores,
                         int64_t* out_ids, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc;
  if (k < 1 || k > ICR_MAX_K) {
    set_error("cos_topk_sharded: k=%d outside [1, %d]", k, ICR_MAX_K);
    return ICR_ERR_K;
  }
  if ((rc = check_peer_args("cos_topk_sharded", Q * k, rank, world, peer_buffers, epoch, n_max))) return rc;
  const size_t local_ws = align_up(icr_cos_topk_workspace_bytes(Q, N, D, dtype, k, path & ~ICR_PATH_WS_RESIDENT, cat_planes != nullptr), 256);
  if (!workspace || workspace_bytes < local_ws + sharded_stage_bytes(Q, k)) {
    set_error("cos_topk_sharded: workspace %zu bytes < required %zu", workspace_bytes, local_ws + sharded_stage_bytes(Q, k));
    return ICR_ERR_WORKSPACE;
  }
  if (Q == 0) return ICR_OK;  // nothing to exchange either: every rank passes the same Q
  float* stage_scores = reinterpret_cast<float*>(static_cast<char*>(workspace) + local_ws);
  int64_t* stage_ids = reinterpret_cast<int64_t*>(static_cast<char*>(workspace) + local_ws + align_up(static_cast<size_t>(Q) * k * sizeof(float), 256));
  const PeerTail tail = make_peer_tail(rank, world, peer_buffers, epoch, n_max);
  const int p = resolve_path(path & ~ICR_PATH_WS_RESIDENT, Q, N, D, dtype, k, exclude_mask);
  if (p == ICR_PATH_GEMV && gemv_peer_tail_fits(static_cast<int>(Q < 8 ? Q : 8), k, world))  // one launch for the whole sharded request
    return cos_topk_impl(queries, Q, ldq, catalog, N, ldc, D, dtype, cat_planes, cat_inv_norms, exclude_mask, nullptr, k, row_offset, path, out_scores, out_ids,
                         workspace, local_ws, stream, &tail, stage_scores, stage_ids);
  // otherwise the shard's lists go to the staging area and the exchange + merge kernel writes the outputs
  rc = cos_topk_impl(queries, Q, ldq, catalog, N, ldc, D, dtype, cat_planes, cat_inv_norms, exclude_mask, nullptr, k, row_offset, path, stage_scores, stage_ids,
                     workspace, local_ws, stream, nullptr, nullptr, nullptr);
  if (rc) return rc;
  return launch_peer_exchange_merge(stage_scores, stage_ids, Q, k, tail, out_scores, out_ids, static_cast<cudaStream_t>(stream));
}

size_t icr_cos_sim_dense_workspace_bytes(int64_t Qa, int64_t Nb, int64_t D, int dtype) {
  if (Qa > 0 && Nb > 0 && dense_use_gemm(Qa, Nb, D, dtype)) return gemm_dense_workspace_bytes(Qa, Nb, D, dtype) + 1024;
  return align_up(static_cast<size_t>(Qa > 0 ? Qa : 0) * 4, 256) + align_up(static_cast<size_t>(Nb > 0 ? Nb : 0) * 4, 256) + 256;
}

int icr_cos_sim_dense(const void* a, int64_t Qa, int64_t lda, const void* b, int64_t Nb, int64_t ldb, int64_t D, int dtype,
                      float* out, int64_t ldo, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc;
  if ((rc = check_matrix("cos_sim_dense.a", a, Qa, D, lda, dtype))) return rc;
  if ((rc = check_matrix("cos_sim_dense.b", b, Nb, D, ldb, dtype))) return rc;
  if (ldo < Nb || (Qa > 0 && Nb > 0 && !out)) {
    set_error("cos_sim_dense: bad output (ldo=%lld, Nb=%lld)", (long long)ldo, (long long)Nb);
    return ICR_ERR_ARG;
  }
  if ((rc = check_device())) return rc;
  if (Qa == 0 || Nb == 0) return ICR_OK;
  const size_t need = icr_cos_sim_dense_workspace_bytes(Qa, Nb, D, dtype);
  if (workspace_bytes < need || !workspace) {
    set_error("cos_sim_dense: workspace %zu bytes < required %zu", workspace_bytes, need);
    return ICR_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dense_use_gemm(Qa, Nb, D, dtype)) return launch_gemm_dense(a, Qa, lda, b, Nb, ldb, D, dtype, out, ldo, workspace, workspace_bytes, st);
  float* inva = static_cast<float*>(workspace);
  float* invb = reinterpret_cast<float*>(static_cast<char*>(workspace) + align_up(static_cast<size_t>(Qa) * 4, 256));
  if ((rc = launch_row_inv_norms(a, Qa, D, lda, dtype, inva, st))) return rc;
  if ((rc = launch_row_inv_norms(b, Nb, D, ldb, dtype, invb, st))) return rc;
  return launch_cos_sim_dense(a, Qa, lda, b, Nb, ldb, static_cast<int>(D), dtype, inva, invb, out, ldo, st);
}

size_t icr_topk_merge_workspace_bytes(int64_t Q, int G, int k_in, int k_out) {
  (void)Q;
  (void)G;
  (void)k_in;
  (void)k_out;
  return 256;
}

int icr_topk_merge(const float* cand_scores, const int64_t* cand_ids, int64_t Q, int G, int k_in, int k_out, float* out_scores,
                   int64_t* out_ids, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  (void)workspace;
  (void)workspace_bytes;
  if (Q < 0 || G < 1 || k_in < 1 || k_out < 1 || k_out > ICR_MAX_K) {
    set_error("topk_merge: bad arguments Q=%lld G=%d k_in=%d k_out=%d", (long long)Q, G, k_in, k_out);
    return ICR_ERR_ARG;
  }
  if (Q > 0 && (!cand_scores || !cand_ids || !out_scores || !out_ids)) {
    set_error("topk_merge: null pointer");
    return ICR_ERR_ARG;
  }
  // candidate ids travel in the 32-bit half of the selection keys: the caller (ShardedCatalog) bounds the catalog below 2^32 - 1
  // rows; ids at or above that would come back truncated, so the contract is stated here and enforced on the host side
  int rc;
  if ((rc = check_device())) return rc;
  return launch_merge_lists(cand_scores, cand_ids, Q, G, k_in, k_out, out_scores, out_ids, static_cast<cudaStream_t>(stream));
}

// the CUDA-core kernels hold a row slice per lane: D <= 768; wider rows take the tensor path at any batch size
static bool mnrl_use_tc(int64_t B, int64_t D, int dtype) {
  (void)dtype;
  if (mnrl_tc_applies(B, B, D)) return true;
  const int64_t simt_max = 768;
  return D > simt_max && D % 8 == 0 && D <= 4096 && B >= 2;
}

size_t icr_mnrl_workspace_bytes(int64_t B, int64_t D) {
  // sized for either element type: the wider-row rule differs between them, the tensor path's need is the larger one
  if (B > 0 && D > 0 && (mnrl_use_tc(B, D, ICR_F32) || mnrl_use_tc(B, D, ICR_BF16))) return mnrl_tc_workspace_bytes(B, B, D);
  return align_up(static_cast<size_t>(B > 0 ? B : 0) * sizeof(float), 256) + 256;
}

static int mnrl_common(const void* a, int64_t lda, const void* p, int64_t ldp, int64_t B, int64_t D, int dtype, void* workspace,
                       size_t workspace_bytes) {
  int rc;
  if ((rc = check_matrix("mnrl.anchors", a, B, D, lda, dtype))) return rc;
  if ((rc = check_matrix("mnrl.positives", p, B, D, ldp, dtype))) return rc;
  if (B < 1 || B > (1 << 24)) {
    set_error("mnrl: batch %lld outside [1, 2^24]", (long long)B);
    return ICR_ERR_ARG;
  }
  if (!workspace || workspace_bytes < icr_mnrl_workspace_bytes(B, D)) {
    set_error("mnrl: workspace %zu bytes < required %zu", workspace_bytes, icr_mnrl_workspace_bytes(B, D));
    return ICR_ERR_WORKSPACE;
  }
  return check_device();
}

int icr_mnrl_fwd(const void* a, int64_t lda, const void* p, int64_t ldp, int64_t B, int64_t D, int dtype, float scale,
                 float* loss, float* lse, float* inv_a, float* inv_p, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = mnrl_common(a, lda, p, ldp, B, D, dtype, workspace, workspace_bytes);
  if (rc) return rc;
  if (!loss || !lse || !inv_a || !inv_p) {
    set_error("mnrl_fwd: null output");
    return ICR_ERR_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MnrlArgs g{};
  g.a = a;
  g.p = p;
  g.lda = lda;
  g.ldp = ldp;
  g.B = g.Bc = static_cast<int>(B);
  g.D = static_cast<int>(D);
  g.scale = scale;
  g.lse = lse;
  g.inv_a = inv_a;
  g.inv_p = inv_p;
  g.counter = static_cast<unsigned int*>(workspace);
  g.row_loss = reinterpret_cast<float*>(static_cast<char*>(workspace) + 256);
  g.loss = loss;
  if (mnrl_use_tc(B, D, dtype)) return launch_mnrl_tc(g, dtype, 0, workspace, workspace_bytes, st);
  ICR_CUDA_CHECK(cudaMemsetAsync(g.counter, 0, sizeof(unsigned int), st));
  return launch_mnrl_dispatch(g, dtype, false, st);
}

int icr_mnrl_bwd(const void* a, int64_t lda, const void* p, int64_t ldp, int64_t B, int64_t D, int dtype, float scale,
                 const float* lse, const float* inv_a, const float* inv_p, const float* grad_out, void* grad_a, int64_t ldga,
                 void* grad_p, int64_t ldgp, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = mnrl_common(a, lda, p, ldp, B, D, dtype, workspace, workspace_bytes);
  if (rc) return rc;
  if (!lse || !inv_a || !inv_p || !grad_out || !grad_a || !grad_p || ldga < D || ldgp < D) {
    set_error("mnrl_bwd: null pointer or bad gradient stride");
    return ICR_ERR_ARG;
  }
  MnrlArgs g{};
  g.a = a;
  g.p = p;
  g.lda = lda;
  g.ldp = ldp;
  g.B = g.Bc = static_cast<int>(B);
  g.D = static_cast<int>(D);
  g.scale = scale;
  g.lse = const_cast<float*>(lse);
  g.inv_a = const_cast<float*>(inv_a);
  g.inv_p = const_cast<float*>(inv_p);
  g.grad_out = grad_out;
  g.grad_a = grad_a;
  g.grad_p = grad_p;
  g.ldga = ldga;
  g.ldgp = ldgp;
  if (mnrl_use_tc(B, D, dtype)) return launch_mnrl_tc(g, dtype, 1, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  return launch_mnrl_dispatch(g, dtype, true, static_cast<cudaStream_t>(stream));
}

int icr_convert_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx, void* out, int64_t ldo, int out_dtype, int normalize,
                     void* stream) {
  g_launches = 0;
  int rc = check_matrix("convert_rows.x", x, rows, dim, ldx, ICR_F32);
  if (rc) return rc;
  if (out_dtype != ICR_F32 && out_dtype != ICR_BF16 && out_dtype != ICR_F16) {
    set_error("convert_rows: unsupported output dtype %d", out_dtype);
    return ICR_ERR_DTYPE;
  }
  const int64_t osz = out_dtype == ICR_F32 ? 4 : 2;
  if (rows > 0 && (!out || ldo < dim || (reinterpret_cast<uintptr_t>(out) & 15) || (ldo * osz) % 8 != 0)) {
    set_error("convert_rows: output must be non-null, 16-byte aligned, row stride >= dim and a multiple of 8 bytes");
    return ICR_ERR_ALIGN;
  }
  if ((rc = check_device())) return rc;
  return launch_convert_rows(x, rows, dim, ldx, out, ldo, out_dtype, normalize ? 1 : 0, static_cast<cudaStream_t>(stream));
}

size_t icr_peer_buffer_bytes(int64_t n_max, int world) {
  size_t total = 0;
  if (n_max < 0 || world < 1) return 0;
  peer_layout(n_max, world, 0, nullptr, nullptr, &total);
  return total;
}

int icr_peer_exchange(const float* scores, const int64_t* ids, int64_t n, int rank, int world, const uint64_t* peer_buffers, uint32_t epoch,
                      int64_t n_max, size_t* scores_off, size_t* ids_off, void* stream) {
  g_launches = 0;
  if (world < 1 || world > ICR_MAX_PEERS || rank < 0 || rank >= world || n < 0 || n > n_max || !peer_buffers || epoch == 0) {
    set_error("peer_exchange: bad arguments n=%lld n_max=%lld rank=%d world=%d (<= %d) epoch=%u", (long long)n, (long long)n_max, rank, world,
              ICR_MAX_PEERS, epoch);
    return ICR_ERR_ARG;
  }
  for (int p = 0; p < world; ++p) {
    if (peer_buffers[p] == 0 || (peer_buffers[p] & 255)) {
      set_error("peer_exchange: buffer of rank %d is null or not 256-byte aligned", p);
      return ICR_ERR_ALIGN;
    }
  }
  if (n > 0 && (!scores || !ids || (reinterpret_cast<uintptr_t>(scores) & 3) || (reinterpret_cast<uintptr_t>(ids) & 7))) {
    set_error("peer_exchange: null or misaligned candidates");
    return ICR_ERR_ARG;
  }
  int rc;
  if ((rc = check_device())) return rc;
  peer_layout(n_max, world, epoch, scores_off, ids_off, nullptr);
  return launch_peer_exchange(scores, ids, n, rank, world, peer_buffers, epoch, n_max, static_cast<cudaStream_t>(stream));
}

int icr_ir_metrics(const int64_t* ids, int64_t Q, int K, int64_t ld_ids, const int64_t* rel_offsets, const int64_t* rel_rows,
                   const int32_t* n_relevant, const int32_t* kinds, const int32_t* ks, int M, double* per_query, double* means,
                   void* stream) {
  g_launches = 0;
  if (Q < 0 || K < 1 || K > ICR_MAX_K || ld_ids < K || M < 1 || M > ICR_MAX_METRICS || !kinds || !ks) {
    set_error("ir_metrics: bad arguments Q=%lld K=%d ld=%lld M=%d (K <= %d, M <= %d)", (long long)Q, K, (long long)ld_ids, M, ICR_MAX_K,
              ICR_MAX_METRICS);
    return ICR_ERR_ARG;
  }
  for (int m = 0; m < M; ++m) {
    if (kinds[m] < ICR_METRIC_ACCURACY || kinds[m] > ICR_METRIC_MAP_RETRIEVED || ks[m] < 1) {
      set_error("ir_metrics: metric %d has kind %d, k %d", m, kinds[m], ks[m]);
      return ICR_ERR_ARG;
    }
  }
  if (!means || (Q > 0 && (!ids || !rel_offsets || !n_relevant || !per_query))) {
    set_error("ir_metrics: null pointer");
    return ICR_ERR_ARG;
  }
  int rc;
  if ((rc = check_device())) return rc;
  return launch_ir_metrics(ids, Q, K, ld_ids, rel_offsets, rel_rows, n_relevant, kinds, ks, M, per_query, means,
                           static_cast<cudaStream_t>(stream));
}

// forward and backward in one call: loss plus the gradients for dL/dloss = 1 (the caller scales them by the incoming
// gradient). One prep instead of two on the tensor path, one host round trip instead of two on both.
int icr_mnrl_fwd_bwd(const void* a, int64_t lda, const void* p, int64_t ldp, int64_t B, int64_t D, int dtype, float scale, float* loss,
                     float* lse, float* inv_a, float* inv_p, void* grad_a, int64_t ldga, void* grad_p, int64_t ldgp, void* workspace,
                     size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = mnrl_common(a, lda, p, ldp, B, D, dtype, workspace, workspace_bytes);
  if (rc) return rc;
  if (!loss || !lse || !inv_a || !inv_p || !grad_a || !grad_p || ldga < D || ldgp < D) {
    set_error("mnrl_fwd_bwd: null pointer or bad gradient stride");
    return ICR_ERR_ARG;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MnrlArgs g{};
  g.a = a;
  g.p = p;
  g.lda = lda;
  g.ldp = ldp;
  g.B = g.Bc = static_cast<int>(B);
  g.D = static_cast<int>(D);
  g.scale = scale;
  g.lse = lse;
  g.inv_a = inv_a;
  g.inv_p = inv_p;
  g.loss = loss;
  g.grad_out = nullptr;  // dL/dloss = 1
  g.grad_a = grad_a;
  g.grad_p = grad_p;
  g.ldga = ldga;
  g.ldgp = ldgp;
  if (mnrl_use_tc(B, D, dtype)) return launch_mnrl_tc(g, dtype, 2, workspace, workspace_bytes, st);
  g.counter = static_cast<unsigned int*>(workspace);
  g.row_loss = reinterpret_cast<float*>(static_cast<char*>(workspace) + 256);
  ICR_CUDA_CHECK(cudaMemsetAsync(g.counter, 0, sizeof(unsigned int), st));
  if ((rc = launch_mnrl_dispatch(g, dtype, false, st))) return rc;
  return launch_mnrl_dispatch(g, dtype, true, st);
}

// the autograd glue's only arithmetic: both gradients of icr_mnrl_fwd_bwd times the incoming dL/dloss (a device scalar)
int icr_mnrl_scale_grads(const void* grad_a, const void* grad_p, int64_t n, int dtype, const float* grad_out, void* out_a, void* out_p,
                         void* stream) {
  g_launches = 0;
  if (n < 0 || (dtype != ICR_F32 && dtype != ICR_BF16 && dtype != ICR_F16) || (n > 0 && (!grad_a || !grad_p || !grad_out || !out_a || !out_p))) {
    set_error("mnrl_scale_grads: bad arguments (n=%lld dtype=%d)", (long long)n, dtype);
    return ICR_ERR_ARG;
  }
  int rc;
  if ((rc = check_device())) return rc;
  return launch_scale2(grad_a, grad_p, n, dtype, grad_out, out_a, out_p, static_cast<cudaStream_t>(stream));
}

// ---- rectangular form: B anchors against Bc >= B candidates, the positive of anchor i at column i + label_offset ----
size_t icr_mnrl_rect_workspace_bytes(int64_t B, int64_t Bc, int64_t D) {
  if (B < 1 || Bc < 1 || D < 1) return 0;
  return mnrl_tc_workspace_bytes(B, Bc, D);
}

static int mnrl_rect_common(const void* a, int64_t lda, const void* c, int64_t ldc, int64_t B, int64_t Bc, int64_t label_offset, int64_t D,
                            int dtype, void* workspace, size_t workspace_bytes) {
  int rc;
  if ((rc = check_matrix("mnrl.anchors", a, B, D, lda, dtype))) return rc;
  if ((rc = check_matrix("mnrl.candidates", c, Bc, D, ldc, dtype))) return rc;
  if (B < 1 || Bc < 2 || label_offset < 0 || label_offset + B > Bc || D % 8 != 0 || D > 4096 || B > 65536 || Bc > (1 << 20)) {
    set_error("mnrl (rectangular): need 1 <= B <= 65536, label_offset + B <= Bc <= 2^20, D %% 8 == 0, D <= 4096; got B=%lld Bc=%lld offset=%lld D=%lld",
              (long long)B, (long long)Bc, (long long)label_offset, (long long)D);
    return ICR_ERR_ARG;
  }
  if (!workspace || workspace_bytes < icr_mnrl_rect_workspace_bytes(B, Bc, D)) {
    set_error("mnrl (rectangular): workspace %zu bytes < required %zu", workspace_bytes, icr_mnrl_rect_workspace_bytes(B, Bc, D));
    return ICR_ERR_WORKSPACE;
  }
  return check_device();
}

int icr_mnrl_fwd_rect(const void* a, int64_t lda, const void* c, int64_t ldc, int64_t B, int64_t Bc, int64_t label_offset, int64_t D, int dtype,
                      float scale, float* loss, float* lse, float* inv_a, float* inv_c, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = mnrl_rect_common(a, lda, c, ldc, B, Bc, label_offset, D, dtype, workspace, workspace_bytes);
  if (rc) return rc;
  if (!loss || !lse || !inv_a || !inv_c) {
    set_error("mnrl_fwd_rect: null output");
    return ICR_ERR_ARG;
  }
  MnrlArgs g{};
  g.a = a;
  g.p = c;
  g.lda = lda;
  g.ldp = ldc;
  g.B = static_cast<int>(B);
  g.Bc = static_cast<int>(Bc);
  g.label_off = static_cast<int>(label_offset);
  g.D = static_cast<int>(D);
  g.scale = scale;
  g.lse = lse;
  g.inv_a = inv_a;
  g.inv_p = inv_c;
  g.loss = loss;
  return launch_mnrl_tc(g, dtype, 0, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int icr_mnrl_bwd_rect(const void* a, int64_t lda, const void* c, int64_t ldc, int64_t B, int64_t Bc, int64_t label_offset, int64_t D, int dtype,
                      float scale, const float* lse, const float* inv_a, const float* inv_c, const float* grad_out, void* grad_a, int64_t ldga,
                      void* grad_c, int64_t ldgc, void* workspace, size_t workspace_bytes, void* stream) {
  g_launches = 0;
  int rc = mnrl_rect_common(a, lda, c, ldc, B, Bc, label_offset, D, dtype, workspace, workspace_bytes);
  if (rc) return rc;
  if (!lse || !inv_a || !inv_c || !grad_out || !grad_a || !grad_c || ldga < D || ldgc < D) {
    set_error("mnrl_bwd_rect: null pointer or bad gradient stride");
    return ICR_ERR_ARG;
  }
  MnrlArgs g{};
  g.a = a;
  g.p = c;
  g.lda = lda;
  g.ldp = ldc;
  g.B = static_cast<int>(B);
  g.Bc = static_cast<int>(Bc);
  g.label_off = static_cast<int>(label_offset);
  g.D = static_cast<int>(D);
  g.scale = scale;
  g.lse = const_cast<float*>(lse);
  g.inv_a = const_cast<float*>(inv_a);
  g.inv_p = const_cast<float*>(inv_c);
  g.grad_out = grad_out;
  g.grad_a = grad_a;
  g.grad_p = grad_c;
  g.ldga = ldga;
  g.ldgp = ldgc;
  return launch_mnrl_tc(g, dtype, 1, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
