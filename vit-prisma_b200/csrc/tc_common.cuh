// tc_common.cuh -- tcgen05 / TMEM / TMA / mbarrier PTX wrappers, tile configuration and tensor-map construction shared by
// the tensor-core kernels of this library (gemm_tc.cu, sae_fused.cu).  sm_100a only.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace {


// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug turns into a trap (-> CUDA error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  for (;;) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      printf("gemm_tc: mbarrier wait timed out (block %d,%d thread %d bar %u parity %u)\n", blockIdx.x, blockIdx.y, threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
template <int KIND>  // 0: kind::f16 (bf16 in), 1: kind::tf32
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (KIND == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle (cute::UMMA::SmemDescriptor):
//   [0,14)  start address >> 4        [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   [32,46) stride byte offset >> 4   = 1024 B between 8-row groups (rows are 128 B, stored densely by TMA)
//   [46,48) descriptor version = 1 (sm_100)      [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

constexpr int TC_BM = 128;
constexpr int TC_THREADS = 192;

template <typename T, int NPASS, int BN, int STAGES>
struct TcCfg {
  static constexpr int ES = sizeof(T);
  static constexpr int BK = 128 / ES;       // elements per 128-byte k-slab
  static constexpr int UMMA_K_BYTES = 32;   // one tcgen05.mma consumes 32 bytes of K per row
  static constexpr int A_BYTES = TC_BM * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int NOP = NPASS == 3 ? 2 : 1;  // operand copies per matrix (hi [+ lo])
  static constexpr int STAGE_BYTES = NOP * (A_BYTES + B_BYTES);
  static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
  static constexpr int SMEM_BYTES = RING_BYTES + 1024 /*alignment slack*/ + 256 /*barriers + tmem ptr*/;
  static constexpr uint32_t FMT = sizeof(T) == 2 ? 1u : 2u;  // F16F32Format: BF16 = 1, TF32 = 2
  // cute::UMMA::InstrDescriptor: c_format F32 [4,6) | a_format [7,10) | b_format [10,13) | a/b K-major (0) | N>>3 [17,23) | M>>4 [24,29)
  static constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

constexpr int TC_F16 = 2;   // make_map dtype of the fp16 operands (PB_F32 / PB_BF16 for the others)

// 2-D map over a row-major [rows, cols] matrix with row stride ld (elements); box = [box_rows, 128 bytes]
int make_map(CUtensorMap* map, const void* ptr, int dtype, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { pb_set_error("gemm_tc: cuTensorMapEncodeTiled entry point unavailable"); return PB_ECUDA; }
  const int es = dtype == PB_F32 ? 4 : 2;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * es};
  cuuint32_t box[2] = {(cuuint32_t)(128 / es), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = fn(map, dtype == PB_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : dtype == PB_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim,
                   gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    pb_set_error("gemm_tc: cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld", (int)rc, (long long)rows, (long long)cols, (long long)ld);
    return PB_ECUDA;
  }
  return PB_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// CTA pairs (tcgen05 cta_group::2): shared by gemm_tc_pair.cuh and the fused SAE encoder (sae_fused.cu)
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;            // shared::cluster address of the same offset in CTA rank 0 of the pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}
// TMA load whose complete_tx lands on the LEADER's barrier (both CTAs execute it)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar & PEER_BIT_MASK), "r"(c0), "r"(c1)
      : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (KIND == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// arrive::one on the barrier at this offset in BOTH CTAs once the MMAs issued so far have completed
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  const uint16_t mask = 0x3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
               : "memory");
}
// arrive on the barrier at this offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 remote;\n\t"
      "mapa.shared::cluster.u32 remote, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remote];\n\t}" ::"r"(bar),
      "r"(rank)
      : "memory");
}

}  // namespace
