// tcgen05 / TMEM / TMA building blocks shared by the tensor-core kernels (gemm_topk.cu, mnrl_tc.cu): PTX wrappers for
// CTA-pair MMAs (cta_group::2), mbarriers, 2-D TMA tile loads with 128-byte swizzle, TMEM loads, and the host-side
// tensor-map encoder. sm_100a only.
#pragma once

#include <cuda.h>

#include "common.cuh"

namespace icr {

constexpr int BM = 128;          // M rows per CTA (TMEM lanes); 256 per pair
constexpr int BN = 256;          // N rows per tile (TMEM columns of one accumulator)
constexpr int BNH = BN / 2;      // N rows of a tile loaded by each CTA of the pair
constexpr int BK = 64;           // K elements per pipeline stage = one 128-byte swizzle atom of 16-bit elements
constexpr int kTileBytes = 128 * BK * 2;  // every operand tile in shared memory is 128 rows x 128 bytes
constexpr uint32_t kSpinLimit = 1u << 24;
constexpr int kNumSMs = 148;

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n"
      ".reg .b32 ra;\n"
      "mapa.shared::cluster.u32 ra, %0, %1;\n"
      // default (.release at CTA scope): a cluster-scope release here costs a MEMBAR + L1 invalidate per tile and
      // nothing needs it — the TMEM reads are ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
      "}\n" ::"r"(bar), "r"(cta)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (spin > kSpinLimit) __trap();  // a protocol bug must abort the launch, not hang the GPU
  }
}
// TMA tile load of a CTA pair: data lands in THIS CTA's shared memory, the transaction bytes are
// credited to the barrier at the same offset in the pair's leader (peer bit of the address cleared)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// int8 operands (signed 8-bit A and B, s32 accumulate): K = 32 elements per instruction, the 32 bytes of one f16 step
__device__ __forceinline__ void umma_i8_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once all MMAs issued so far have completed) on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(static_cast<uint16_t>(3))
               : "memory");
}
// one lane of a converged warp (warp-uniform predicate)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// wait for the outstanding tcgen05.ld of this thread; the registers are tied to the wait so that no use of
// them can be scheduled above it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                 "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                 "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                 "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// K-major operand tile in shared memory, rows of 128 bytes, 128-byte swizzle, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);  // start address, 16-byte units
  d |= static_cast<uint64_t>(1) << 16;                   // leading byte offset (ignored for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;           // stride byte offset between 8-row groups
  d |= static_cast<uint64_t>(1) << 46;                   // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                   // SWIZZLE_128B
  return d;
}

// ---- host side: tensor maps ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D map over a row-major [rows, cols] matrix of 16-bit elements, box = [128 rows, 64 cols], 128B swizzle
inline int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld_elems, bool bf16, int box_rows = 128) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return ICR_ERR_CUDA;
  }
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld_elems) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims,
                         strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", static_cast<int>(r), (long long)rows,
              (long long)cols, (long long)ld_elems);
    return ICR_ERR_CUDA;
  }
  return ICR_OK;
}
}  // namespace icr
