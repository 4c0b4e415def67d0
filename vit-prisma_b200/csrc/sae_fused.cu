// sae_fused.cu -- fused SAE encoder -> TopK for sm_100a: the dense pre-activation matrix hidden_pre [tokens, d_sae] is never
// written to HBM (reference sae/sae.py:557-581 `sae_in @ W_enc + b_enc` followed by TopK.forward :795-808 `torch.topk`).
//
// Approximate-then-rescore, exact by construction:
//   1. k_enc_cand     persistent tcgen05 GEMM, ONE kind::f16 pass over the fp16 shadows sae_in_h / W_encT_h (f16_cand: round to
//                     nearest, saturate, flush below 2^-14; fp32 accumulate), 128 x 256 tiles, accumulators double-buffered in
//                     TMEM.  The epilogue never stores the tile: every thread owns one token row x 128 feature columns of it
//                     (TMEM's native layout) and keeps that segment's C_KEEP largest values as packed keys (order-preserving
//                     int of the value, the low 7 bits replaced by the column inside the segment) with branch-free networks, then writes
//                     C_KEEP x 4 bytes.  Per token: d_sae / 128 segments x C_KEEP keys (6 KB at d_sae = 24576) instead of a
//                     98 KB dense row.
//   2. k_cand_select  one CTA per token: the m_cand best keys of the row (threshold from per-thread bests, rank by counting),
//                     EXACT fp32 re-evaluation of those m_cand pre-activations (FFMA dot products against W_encT rows),
//                     exact top-k of the re-scored values (ties -> lower index, sorted descending), and a proof that no
//                     feature outside the candidate set can belong to the exact top-k:
//                         ub(best key not selected, or last kept key of a segment whose keys were all selected) + E_row < tau_k
//                     where E_row bounds |fp16 product - exact| by Cauchy-Schwarz on the operand residuals plus the fp32
//                     accumulation (DESIGN.md section 4).  Rows that fail the proof go on a list.
//   3. k_topk_fallback  persistent, normally finds the list empty: recomputes a listed row's 'd_sae' pre-activations exactly and
//                     selects from all of them.  Correctness therefore never depends on the approximation; only speed does.
// Outputs are those of pb_sae_topk: idx int32 / val fp32 [rows][k] sorted by value, feat_count[f] += selections.
#include "tc_common.cuh"
#include "gemm_epi.cuh"
#include <limits.h>

namespace {

__device__ __forceinline__ int f2ord(float v) {           // monotone float -> signed int
  const int k = __float_as_int(v);
  return k ^ ((k >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord2f(int k) { return __int_as_float(k ^ ((k >> 31) & 0x7fffffff)); }
__device__ __forceinline__ bool key_gt_f(float va, int ia, float vb, int ib) { return va > vb || (va == vb && ia < ib); }

#ifndef PB_ENC_PAIR_DEFAULT
#define PB_ENC_PAIR_DEFAULT 0      // flipped to 1 once measured faster on the B200 (profiles/r02_sae_notes.md)
#endif
constexpr int FZ_BN = 256;       // tile columns
constexpr int FZ_STAGES = 4;     // 4 x (16 KB A + 32 KB B) = 192 KB operand ring
constexpr int FZ_NEPI = 8;       // epilogue warps: 4 TMEM lane quarters x 2 column halves
constexpr int FZ_SEG = 128;      // columns per thread segment (= FZ_BN / 2)
constexpr int FZ_THREADS = 64 + FZ_NEPI * 32;
using FzCfg = TcCfg<uint16_t, 1, FZ_BN, FZ_STAGES>;    // fp16 operands: 64 elements per 128-byte k-slab
// kind::f16 instruction descriptor: c_format F32 [4,6) | a_format = b_format = F16 (0) | K-major | N>>3 [17,23) | M>>4 [24,29)
constexpr uint32_t FZ_IDESC = (1u << 4) | ((uint32_t)(FZ_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
constexpr int FZ_SMEM = FzCfg::RING_BYTES + 1024 + 256;

// Insert x into s[0, N) (sorted descending) and drop the smallest of the N + 1: 2N - 1 integer min / max.
template <int N>
__device__ __forceinline__ void key_insert(int (&s)[N], int x) {
#pragma unroll
  for (int i = 0; i < N - 1; ++i) {
    const int hi = max(s[i], x);
    x = min(s[i], x);
    s[i] = hi;
  }
  s[N - 1] = max(s[N - 1], x);
}
__device__ __forceinline__ void key_cas(int& a, int& b) {        // a >= b afterwards
  const int hi = max(a, b);
  b = min(a, b);
  a = hi;
}

// One epilogue warp's share of one finished accumulator: thread = one token row x one 128-feature segment; keeps the segment's
// C_KEEP largest pre-activations as packed keys and writes them.  `release` is called once the accumulator has been read.
// Grouped selection: each group of 4 consecutive columns is sorted (5 compare-exchanges) and its r-th largest key goes to a list
// of floor(C_KEEP / r) slots.  If a group's r-th key is among the segment's C_KEEP largest, so are the r - 1 keys above it, so at
// most floor(C_KEEP / r) r-th keys are; each list therefore keeps every key of its rank that belongs to the top C_KEEP.  Keys are
// distinct (the low 7 bits are the column), and the lists are merged once per segment: the same C_KEEP keys, sorted descending,
// as a plain insertion network, at 9.5 instead of 15 min / max per element for C_KEEP = 8.
template <int C_KEEP, typename Release>
__device__ __forceinline__ void enc_cand_epilogue(uint32_t tmem_base, int ab, int quarter, int cbase, int lane, int m0, int n0, int M, int N,
                                                  const float* __restrict__ bias, int* __restrict__ cand, Release release) {
  constexpr int N2 = C_KEEP / 2, N3 = C_KEEP / 3, N4 = C_KEEP / 4;
  const int nseg = N / FZ_SEG;
  const int row = m0 + quarter * 32 + lane;
  const bool seg_in = (n0 + cbase) < N;          // N % 128 == 0: a segment is entirely inside or outside the matrix
  int s[C_KEEP], s2[N2], s3[N3], s4[N4];
#pragma unroll
  for (int i = 0; i < C_KEEP; ++i) s[i] = INT_MIN;
#pragma unroll
  for (int i = 0; i < N2; ++i) s2[i] = INT_MIN;
#pragma unroll
  for (int i = 0; i < N3; ++i) s3[i] = INT_MIN;
#pragma unroll
  for (int i = 0; i < N4; ++i) s4[i] = INT_MIN;
#pragma unroll 1
  for (int c = 0; c < FZ_SEG / 32; ++c) {
    uint32_t r[32];
    tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * FZ_BN + cbase + c * 32), r);
    tmem_ld_wait();
    if (c == FZ_SEG / 32 - 1) {                  // last read of this accumulator: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) release();
    }
    if (seg_in) {
      const float* bp = bias + n0 + cbase + c * 32;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float bb[4];
        ld4(bp + 4 * q, bb);                     // same address in every lane: one broadcast transaction
        int x[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = (f2ord(__uint_as_float(r[4 * q + j]) + bb[j]) & ~127) | (c * 32 + 4 * q + j);
        key_cas(x[0], x[1]); key_cas(x[2], x[3]); key_cas(x[0], x[2]); key_cas(x[1], x[3]); key_cas(x[1], x[2]);
        key_insert(s, x[0]);
        key_insert(s2, x[1]);
        key_insert(s3, x[2]);
        key_insert(s4, x[3]);
      }
    }
  }
  if (seg_in && row < M) {
#pragma unroll
    for (int i = 0; i < N2; ++i) key_insert(s, s2[i]);
#pragma unroll
    for (int i = 0; i < N3; ++i) key_insert(s, s3[i]);
#pragma unroll
    for (int i = 0; i < N4; ++i) key_insert(s, s4[i]);
    int* dst = cand + ((int64_t)row * nseg + (n0 + cbase) / FZ_SEG) * C_KEEP;
    if (C_KEEP % 4 == 0) {
#pragma unroll
      for (int i = 0; i < C_KEEP / 4; ++i) reinterpret_cast<int4*>(dst)[i] = make_int4(s[4 * i], s[4 * i + 1], s[4 * i + 2], s[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < C_KEEP / 2; ++i) reinterpret_cast<int2*>(dst)[i] = make_int2(s[2 * i], s[2 * i + 1]);
    }
  }
}

template <int C_KEEP>
__global__ void __launch_bounds__(FZ_THREADS, 1)
k_enc_cand(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int K, int M, int N,
           const float* __restrict__ bias, int* __restrict__ cand, int num_m_tiles, int num_n_tiles) {
  using C = FzCfg;
  pb_pdl_trigger();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = smem_u32(smem_raw);
  const uint32_t ring = (smem0 + 1023u) & ~1023u;
  const uint32_t bar_base = ring + C::RING_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (FZ_STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * FZ_STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * FZ_STAGES + 2 + a); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * FZ_STAGES + 4);
  volatile uint32_t* tmem_ptr_generic = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem0));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (K + C::BK - 1) / C::BK;
  const int num_tiles = num_m_tiles * num_n_tiles;
  // m-fastest raster: the CTAs in flight share one 256-feature slab of the dictionary and walk the token tiles, so W_encT
  // (75 MB at d_sae = 24576) streams from HBM once while sae_in (12.6 MB) stays L2-resident.
  auto tile_m = [&](int tile) { return tile % num_m_tiles; };
  auto tile_n = [&](int tile) { return tile / num_m_tiles; };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < FZ_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), FZ_NEPI); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"((uint32_t)(2 * FZ_BN)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_generic;
  pb_pdl_wait();            // barriers initialised, TMEM allocated, tensor maps prefetched: now the prep kernel's sae_in must be complete

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = tile_m(tile) * TC_BM, n0 = tile_n(tile) * FZ_BN;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % FZ_STAGES;
          const uint32_t ph = (it / FZ_STAGES) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), C::STAGE_BYTES);
          const uint32_t sa = ring + s * C::STAGE_BYTES;
          tma_load_2d(sa, &tmA, full_bar(s), kb * C::BK, m0);
          tma_load_2d(sa + C::A_BYTES, &tmB, full_bar(s), kb * C::BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: one kind::f16 pass =====================
    if (lane == 0) {
      uint32_t it = 0;
      int li = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++li) {
        const int ab = li & 1;
        const uint32_t aph = (li >> 1) & 1;
        mbar_wait(tempty_bar(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * FZ_BN);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % FZ_STAGES;
          const uint32_t ph = (it / FZ_STAGES) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = ring + s * C::STAGE_BYTES;
          const uint32_t sb = sa + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < 128 / C::UMMA_K_BYTES; ++k) {
            const uint32_t koff = k * C::UMMA_K_BYTES;
            tc_mma<0>(d_tmem, make_smem_desc(sa + koff), make_smem_desc(sb + koff), FZ_IDESC, (kb | k) != 0 ? 1u : 0u);
          }
          tc_commit(empty_bar(s));
        }
        tc_commit(tfull_bar(ab));
      }
    }
  } else {
    // ===================== epilogue: per-row, per-128-column top-C_KEEP as packed keys =====================
    const int e = warp - 2;
    const int quarter = warp & 3;          // TMEM lane quarter this warp may read
    const int cbase = (e >> 2) * FZ_SEG;   // column half of the tile
    int li = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++li) {
      const int m0 = tile_m(tile) * TC_BM, n0 = tile_n(tile) * FZ_BN;
      const int ab = li & 1;
      const uint32_t aph = (li >> 1) & 1;
      mbar_wait(tfull_bar(ab), aph);
      tc_fence_after();
      enc_cand_epilogue<C_KEEP>(tmem_base, ab, quarter, cbase, lane, m0, n0, M, N, bias, cand, [&] { mbar_arrive(tempty_bar(ab)); });
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * FZ_BN)) : "memory");
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2, protocol of gemm_tc_pair.cuh): the two CTAs of a cluster compute a 256-token x 256-feature
// tile with one MMA stream issued by the leader; each CTA loads its own 128 token rows and HALF of the dictionary tile, so the
// per-SM operand ingest drops from 48 KB to 32 KB per k-block (the one-CTA kernel runs the tensor pipe at 76 % of its active cycles
// because its 67 B/clk/SM operand demand exceeds what TMA delivers, profiles/r02_sae_notes.md).  Six 32 KB stages.
constexpr int FZP_STAGES = 6;
constexpr int FZP_A_BYTES = TC_BM * 128, FZP_BH_BYTES = (FZ_BN / 2) * 128, FZP_STAGE_BYTES = FZP_A_BYTES + FZP_BH_BYTES;
constexpr int FZP_SMEM = FZP_STAGES * FZP_STAGE_BYTES + 1024 + 256;
constexpr uint32_t FZP_IDESC = (1u << 4) | ((uint32_t)(FZ_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);   // f16, M = 256 across the pair

template <int C_KEEP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FZ_THREADS, 1)
k_enc_cand_pair(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh, int K, int M, int N,
                const float* __restrict__ bias, int* __restrict__ cand, int num_m_tiles /* of 256 rows */, int num_n_tiles) {
  pb_pdl_trigger();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = smem_u32(smem_raw);
  const uint32_t ring = (smem0 + 1023u) & ~1023u;
  const uint32_t bar_base = ring + FZP_STAGES * FZP_STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                            // used in the leader only
  auto empty_bar = [&](int s) { return bar_base + 8u * (FZP_STAGES + s); };            // one per CTA
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * FZP_STAGES + a); };        // one per CTA
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * FZP_STAGES + 2 + a); };   // used in the leader only
  const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * FZP_STAGES + 4);
  volatile uint32_t* tmem_ptr_generic = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - smem0));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  constexpr int BK = 64;                                   // fp16 elements per 128-byte k-slab
  const int num_kb = (K + BK - 1) / BK;
  const int num_tiles = num_m_tiles * num_n_tiles;
  auto tile_m = [&](int tile) { return tile % num_m_tiles; };        // m-fastest raster, as in k_enc_cand
  auto tile_n = [&](int tile) { return tile / num_m_tiles; };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmBh);
    for (int s = 0; s < FZP_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * FZ_NEPI); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr), "r"((uint32_t)(2 * FZ_BN)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                        // peer barriers initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_generic;
  pb_pdl_wait();

  if (warp == 0) {
    if (lane == 0) {                                         // TMA producer (both CTAs)
      uint32_t it = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += n_clusters) {
        const int m0 = tile_m(tile) * 256 + (int)rank * TC_BM;
        const int n0 = tile_n(tile) * FZ_BN + (int)rank * (FZ_BN / 2);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % FZP_STAGES;
          const uint32_t ph = (it / FZP_STAGES) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          if (leader) mbar_expect_tx(full_bar(s), 2u * FZP_STAGE_BYTES);   // bytes of BOTH CTAs land on the leader's barrier
          const uint32_t sa = ring + s * FZP_STAGE_BYTES;
          tma_load_2d_pair(sa, &tmA, full_bar(s), kb * BK, m0);
          tma_load_2d_pair(sa + FZP_A_BYTES, &tmBh, full_bar(s), kb * BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {                               // MMA issuer (leader only): one kind::f16 pass
      uint32_t it = 0;
      int li = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += n_clusters, ++li) {
        const int ab = li & 1;
        const uint32_t aph = (li >> 1) & 1;
        mbar_wait(tempty_bar(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * FZ_BN);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % FZP_STAGES;
          const uint32_t ph = (it / FZP_STAGES) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = ring + s * FZP_STAGE_BYTES;
          const uint32_t sb = sa + FZP_A_BYTES;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            tc_mma_pair<0>(d_tmem, make_smem_desc(sa + 32 * k), make_smem_desc(sb + 32 * k), FZP_IDESC, (kb | k) != 0 ? 1u : 0u);
          tc_commit_pair(empty_bar(s));
        }
        tc_commit_pair(tfull_bar(ab));
      }
    }
  } else {
    const int e = warp - 2;
    const int quarter = warp & 3;
    const int cbase = (e >> 2) * FZ_SEG;
    int li = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += n_clusters, ++li) {
      const int m0 = tile_m(tile) * 256 + (int)rank * TC_BM, n0 = tile_n(tile) * FZ_BN;
      const int ab = li & 1;
      const uint32_t aph = (li >> 1) & 1;
      mbar_wait(tfull_bar(ab), aph);
      tc_fence_after();
      enc_cand_epilogue<C_KEEP>(tmem_base, ab, quarter, cbase, lane, m0, n0, M, N, bias, cand, [&] { mbar_arrive_remote(tempty_bar(ab), 0); });
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                        // the peer may still be reading its half of TMEM / our shared memory
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * FZ_BN)) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// exact fp32 dot products of one shared-memory row with rows of W (16-byte loads, one warp per dot, two dots in flight)
__device__ __forceinline__ float warp_dot(const float4* __restrict__ a4, const float4* __restrict__ w4, int nvec, int lane) {
  float acc = 0.f;
  for (int i = lane; i < nvec; i += 32) {
    const float4 a = a4[i], w = __ldg(w4 + i);
    acc = fmaf(a.x, w.x, acc); acc = fmaf(a.y, w.y, acc); acc = fmaf(a.z, w.z, acc); acc = fmaf(a.w, w.w, acc);
  }
  return warp_sum(acc);
}
__device__ __forceinline__ void warp_dot2(const float4* __restrict__ a4, const float4* __restrict__ w0, const float4* __restrict__ w1, int nvec,
                                          int lane, float& o0, float& o1) {
  float x = 0.f, y = 0.f;
  for (int i = lane; i < nvec; i += 32) {
    const float4 a = a4[i], u = __ldg(w0 + i), v = __ldg(w1 + i);
    x = fmaf(a.x, u.x, x); x = fmaf(a.y, u.y, x); x = fmaf(a.z, u.z, x); x = fmaf(a.w, u.w, x);
    y = fmaf(a.x, v.x, y); y = fmaf(a.y, v.y, y); y = fmaf(a.z, v.z, y); y = fmaf(a.w, v.w, y);
  }
  o0 = warp_sum(x);
  o1 = warp_sum(y);
}

constexpr int SEL_MAX_CAND = 128;   // most candidates one row may re-score before it gives up and takes the exact path
constexpr int SEL_EXTEND = 16;      // candidates added per extension round
constexpr int SEL_TAU_RANK = 96;    // the gather threshold keeps at least this many keys (typically 1.2-1.5x as many)
constexpr int SEL_SLOTS = 512;      // gathered keys that can be sorted; more (massive ties) -> exact path

__device__ __forceinline__ unsigned long long sel_pack(int key, int pos) {    // orders like (key descending-first, pos ascending-first)
  return ((unsigned long long)((unsigned)key ^ 0x80000000u) << 32) | (unsigned)(0xFFFFFFFFu - (unsigned)pos);
}
__device__ __forceinline__ int sel_key(unsigned long long it) { return (int)((unsigned)(it >> 32) ^ 0x80000000u); }
__device__ __forceinline__ int sel_pos(unsigned long long it) { return (int)(0xFFFFFFFFu - (unsigned)it); }

// One CTA (256 threads) per token row.  dynamic smem: a_row[d]
//   1. threshold: every warp bitonic-sorts its 32 per-thread bests (= segment maxima) in registers and reports its q-th largest;
//      the smallest report is a key with at least SEL_TAU_RANK keys of the row at or above it;
//   2. gather the keys >= threshold (packed with their position) and bitonic-sort them in shared memory (256 or 512 slots);
//   3. rounds: exactly re-score the first m_cur sorted candidates (m_cand, then +16 per round), take the exact top-k of those,
//      and try to prove no other feature can beat the k-th:   ub(best key not yet re-scored) + E_row < tau_k.  Most rows are
//      proven in the first round; a row that runs out of sorted candidates (or whose segment kept-lists saturate) is listed.
// (The first version ranked by counting -- 256^2 + G^2 shared-memory compares per row -- and was ALU-bound at 205 us per launch,
//  75 % issue-active, with the re-scoring gathers a small part of it: profiles/r02_sae_notes.md.)
template <int SPT>
__global__ void __launch_bounds__(256) k_cand_select(const int* __restrict__ cand, int nseg, int c_keep, const float* __restrict__ sae_in,
                                                     const float* __restrict__ W_encT, const float* __restrict__ b_enc,
                                                     const float* __restrict__ wnorm_max, float err_scale, int d, int k, int m_cand,
                                                     int* __restrict__ out_idx, float* __restrict__ out_val, float* __restrict__ feat_count,
                                                     int* __restrict__ fb_count, int* __restrict__ fb_rows, int* __restrict__ stats) {
  pb_pdl();
  extern __shared__ __align__(16) unsigned char sm_raw[];
  float* a_row = reinterpret_cast<float*>(sm_raw);
  __shared__ unsigned long long items[SEL_SLOTS];
  __shared__ int ex_idx[SEL_MAX_CAND], win_idx[64], warp_tau[8];
  __shared__ float ex_val[SEL_MAX_CAND];
  __shared__ float red[2][8];
  __shared__ int g_n, u_below, sat_key;
  __shared__ float tau_exact, a_norm, a_lo_norm;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int row = blockIdx.x;
  const int nvec = d >> 2;
  const int nkeys = nseg * c_keep;

  // ---- the token's encoder input -> shared memory; ||a|| and ||a - f16_cand(a)|| for the error bound
  {
    const float4* src = reinterpret_cast<const float4*>(sae_in + (int64_t)row * d);
    float4* dst = reinterpret_cast<float4*>(a_row);
    float nsq = 0.f, lsq = 0.f;
    for (int i = t; i < nvec; i += 256) {
      const float4 v = src[i];
      dst[i] = v;
      nsq += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      const float vv[4] = {v.x, v.y, v.z, v.w};
      lsq += st4_f16_cand(nullptr, vv);
    }
    nsq = warp_sum(nsq);
    lsq = warp_sum(lsq);
    if (lane == 0) { red[0][warp] = nsq; red[1][warp] = lsq; }
  }
  // ---- keys of this row.  Thread t owns WHOLE segments t, t + 256, ... (their c_keep keys, sorted descending by the GEMM
  // epilogue), so a thread's best key is the largest segment maximum it holds.
  int key[SPT][8];
  int bk = INT_MIN;
  const int* kr = cand + (int64_t)row * nkeys;
#pragma unroll
  for (int i = 0; i < SPT; ++i) {
    const int sg = t + 256 * i;
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      int2 v = make_int2(INT_MIN, INT_MIN);
      if (sg < nseg && j < c_keep) v = *reinterpret_cast<const int2*>(kr + sg * c_keep + j);
      key[i][j] = v.x;
      key[i][j + 1] = v.y;
    }
    bk = max(bk, key[i][0]);
  }
  // ---- threshold.  Warp w holds cnt_w = clamp(nthr - 32 w, 0, 32) valid bests (nthr = threads that own a segment); its quota
  // q_w = ceil(m_tau cnt_w / nthr) of them are >= its q_w-th largest, and the quotas add up to >= m_tau.
  {
    int v = bk;                                     // bitonic sort across the warp, descending: lane i ends with the i-th largest
#pragma unroll
    for (int kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll
      for (int j = kk >> 1; j > 0; j >>= 1) {
        const int o = __shfl_xor_sync(0xffffffffu, v, j);
        const bool keep_max = ((lane & kk) == 0) == ((lane & j) == 0);
        v = keep_max ? max(v, o) : min(v, o);
      }
    }
    const int nthr = min(256, nseg);
    const int m_tau = min(SEL_TAU_RANK, nthr);
    const int cnt_w = max(0, min(32, nthr - 32 * warp));
    const int q_w = (m_tau * cnt_w + nthr - 1) / nthr;
    const int rep = __shfl_sync(0xffffffffu, v, max(q_w - 1, 0));
    if (lane == 0) warp_tau[warp] = q_w > 0 ? rep : INT_MAX;
  }
  if (t == 0) { g_n = 0; u_below = INT_MIN; }
  __syncthreads();
  if (t == 0) {
    float s0 = 0.f, s1 = 0.f;
    for (int i = 0; i < 8; ++i) { s0 += red[0][i]; s1 += red[1][i]; }
    a_norm = sqrtf(s0);
    a_lo_norm = sqrtf(s1);
  }
  int tau = INT_MAX;
#pragma unroll
  for (int w = 0; w < 8; ++w) tau = min(tau, warp_tau[w]);
  // ---- gather
  int lower = INT_MIN;                              // best key of this thread below tau
#pragma unroll
  for (int i = 0; i < SPT; ++i) {
    const int sg = t + 256 * i;
    if (sg < nseg) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j < c_keep) {
          if (key[i][j] >= tau) {
            const int slot = atomicAdd(&g_n, 1);
            if (slot < SEL_SLOTS) items[slot] = sel_pack(key[i][j], sg * c_keep + j);
          } else {
            lower = max(lower, key[i][j]);
          }
        }
      }
    }
  }
  if (lower != INT_MIN) atomicMax(&u_below, lower);
  __syncthreads();
  const bool overflow = g_n > SEL_SLOTS;            // only with massive ties (e.g. constant rows): such rows take the exact path
  const int G = min(g_n, SEL_SLOTS);
  const int n_sort = G <= 256 ? 256 : SEL_SLOTS;
  for (int i = G + t; i < n_sort; i += 256) items[i] = 0ull;     // padding sorts last
  __syncthreads();
  // ---- bitonic sort of items[0, n_sort), descending
  for (int kk = 2; kk <= n_sort; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int p = t; p < (n_sort >> 1); p += 256) {
        const int i = 2 * j * (p / j) + (p % j);
        const int o = i + j;
        const unsigned long long x = items[i], y = items[o];
        const bool desc = (i & kk) == 0;
        if ((x < y) == desc) { items[i] = y; items[o] = x; }
      }
      __syncthreads();
    }
  }
  const int Gs = min(G, SEL_MAX_CAND);
  const float4* a4 = reinterpret_cast<const float4*>(a_row);
  int m_prev = 0, m_cur = min(m_cand, Gs);
  bool ok = false;
  for (;;) {
    if (t == 0) sat_key = INT_MIN;
    // ---- exact re-evaluation of candidates [m_prev, m_cur): hidden_pre[f] = <sae_in, W_enc[:, f]> + b_enc[f]   (sae.py:568-574)
    for (int c = m_prev + 2 * warp; c < m_cur; c += 16) {
      const unsigned long long it0 = items[c];
      const int f0 = (sel_pos(it0) / c_keep) * FZ_SEG + (sel_key(it0) & 127);
      if (c + 1 < m_cur) {
        const unsigned long long it1 = items[c + 1];
        const int f1 = (sel_pos(it1) / c_keep) * FZ_SEG + (sel_key(it1) & 127);
        float v0, v1;
        warp_dot2(a4, reinterpret_cast<const float4*>(W_encT + (int64_t)f0 * d), reinterpret_cast<const float4*>(W_encT + (int64_t)f1 * d), nvec,
                  lane, v0, v1);
        if (lane == 0) { ex_val[c] = v0 + b_enc[f0]; ex_idx[c] = f0; ex_val[c + 1] = v1 + b_enc[f1]; ex_idx[c + 1] = f1; }
      } else {
        const float v0 = warp_dot(a4, reinterpret_cast<const float4*>(W_encT + (int64_t)f0 * d), nvec, lane);
        if (lane == 0) { ex_val[c] = v0 + b_enc[f0]; ex_idx[c] = f0; }
      }
    }
    __syncthreads();
    // ---- exact top-k among the first m_cur candidates (sorted descending, ties -> lower index)
    if (t < m_cur) {
      const float v = ex_val[t];
      const int f = ex_idx[t];
      int rank = 0;
      for (int j = 0; j < m_cur; ++j) rank += key_gt_f(ex_val[j], ex_idx[j], v, f) ? 1 : 0;
      if (rank < k) {
        out_idx[(int64_t)row * k + rank] = f;
        out_val[(int64_t)row * k + rank] = v;
        win_idx[rank] = f;
        if (rank == k - 1) tau_exact = v;
      }
    }
    // a segment whose c_keep kept keys were ALL re-scored may have dropped a value as large as its last kept key
    if (m_cur > 0) {
      const int key_m = sel_key(items[m_cur - 1]);
      int sat = INT_MIN;
#pragma unroll
      for (int i = 0; i < SPT; ++i) {
        if (t + 256 * i < nseg) {
          int last = key[i][3];                    // last kept key of the segment: slot c_keep - 1
          if (c_keep == 6) last = key[i][5];
          if (c_keep == 8) last = key[i][7];
          if (last >= key_m) sat = max(sat, last);
        }
      }
      if (sat != INT_MIN) atomicMax(&sat_key, sat);
    }
    __syncthreads();
    // ---- proof of completeness for this round
    {
      const int u_rest = m_cur < G ? sel_key(items[m_cur]) : u_below;                      // best key not re-scored
      const int u = max(u_rest, sat_key);
      const float u_val = u == INT_MIN ? -INFINITY : ord2f((u & ~127) | 127);               // upper end of the key's value bucket
      // |fp16 product - exact| <= ||a_lo|| max||w|| + ||a|| max||w_lo|| (operands, Cauchy-Schwarz, per row, lo = x - f16_cand(x))
      //                          + d 2^-22 ||a|| max||w||                 (fp32 accumulation in the tensor core: DESIGN.md section 4)
      const float E = err_scale * (a_lo_norm * wnorm_max[0] + a_norm * wnorm_max[1] + (float)d * 2.3841858e-7f * a_norm * wnorm_max[0]) +
                      fabsf(tau_exact) * 1.2207031e-4f;
      ok = !overflow && m_cur >= k && (u_val + E < tau_exact);
    }
    if (ok || m_cur >= Gs) break;
    __syncthreads();                                // everybody has read sat_key / tau_exact of this round
    m_prev = m_cur;
    m_cur = min(m_cur + SEL_EXTEND, Gs);
  }
  if (ok) {
    if (t < k && feat_count) atomicAdd(feat_count + win_idx[t], 1.0f);
    if (stats && t == 0) atomicAdd(stats, m_cur);                 // candidates re-scored, summed over the proven rows
  } else if (t == 0) {
    fb_rows[atomicAdd(fb_count, 1)] = row;
  }
}

// Exact path for listed rows: hidden row recomputed with FFMA into this CTA's scratch row, then exact selection from all F values.
// dynamic smem: a_row[d] | cand_v[cap] | cand_i[cap]
__global__ void __launch_bounds__(256) k_topk_fallback(const int* __restrict__ fb_count, const int* __restrict__ fb_rows,
                                                       const float* __restrict__ sae_in, const float* __restrict__ W_encT,
                                                       const float* __restrict__ b_enc, float* __restrict__ scratch, int d, int F, int k, int cap,
                                                       int* __restrict__ out_idx, float* __restrict__ out_val, float* __restrict__ feat_count) {
  pb_pdl();
  const int n_items = *fb_count;
  if (n_items == 0) return;
  extern __shared__ __align__(16) unsigned char sm_raw[];
  float* a_row = reinterpret_cast<float*>(sm_raw);
  float* cand_v = a_row + d;
  int* cand_i = reinterpret_cast<int*>(cand_v + cap);
  __shared__ float best_v[256];
  __shared__ int best_i[256];
  __shared__ float tau_v;
  __shared__ int tau_i, cand_n;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int nvec = d >> 2;
  float* h = scratch + (int64_t)blockIdx.x * F;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int row = fb_rows[item];
    __syncthreads();
    for (int i = t; i < nvec; i += 256) reinterpret_cast<float4*>(a_row)[i] = reinterpret_cast<const float4*>(sae_in + (int64_t)row * d)[i];
    if (t == 0) cand_n = 0;
    __syncthreads();
    const float4* a4 = reinterpret_cast<const float4*>(a_row);
    for (int f = 2 * warp; f < F; f += 16) {
      float v0, v1;
      warp_dot2(a4, reinterpret_cast<const float4*>(W_encT + (int64_t)f * d), reinterpret_cast<const float4*>(W_encT + (int64_t)(f + 1) * d), nvec, lane,
                v0, v1);
      if (lane == 0) { h[f] = v0 + b_enc[f]; h[f + 1] = v1 + b_enc[f + 1]; }
    }
    __syncthreads();
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int p = t; p < F; p += 256) {
      const float v = h[p];
      if (key_gt_f(v, p, bv, bi)) { bv = v; bi = p; }
    }
    best_v[t] = bv;
    best_i[t] = bi;
    __syncthreads();
    {
      int rank = 0;
      for (int j = 0; j < 256; ++j) rank += key_gt_f(best_v[j], best_i[j], bv, bi) ? 1 : 0;
      if (rank == min(k, 256) - 1) { tau_v = bv; tau_i = bi; }
    }
    __syncthreads();
    const float tv = tau_v;
    const int ti = tau_i;
    for (int p = t; p < F; p += 256) {
      const float v = h[p];
      if (!key_gt_f(tv, ti, v, p)) {
        const int slot = atomicAdd(&cand_n, 1);
        if (slot < cap) { cand_v[slot] = v; cand_i[slot] = p; }
      }
    }
    __syncthreads();
    const int C = min(cand_n, cap);
    for (int c = t; c < C; c += 256) {
      const float cv = cand_v[c];
      const int ci = cand_i[c];
      int rank = 0;
      for (int j = 0; j < C; ++j) rank += key_gt_f(cand_v[j], cand_i[j], cv, ci) ? 1 : 0;
      if (rank < k) {
        out_idx[(int64_t)row * k + rank] = ci;
        out_val[(int64_t)row * k + rank] = cv;
        if (feat_count) atomicAdd(feat_count + ci, 1.0f);
      }
    }
  }
}

// out[0] = max_f ||W[f, :]||_2, out[1] = max_f ||W[f, :] - f16_cand(W[f, :])||_2 (atomic max on the bit patterns: norms are
// non-negative), and the fp16 shadow W_h[f, :] = f16_cand(W[f, :]) (row stride f16_ld(d)) when W_h is given; out must be zeroed
// by the caller
__global__ void __launch_bounds__(256) k_rownorm_max(const float* __restrict__ W, int F, int d, float* __restrict__ out, uint16_t* __restrict__ W_h) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  float best = 0.f, best_lo = 0.f;
  for (int f = blockIdx.x * nw + warp; f < F; f += gridDim.x * nw) {
    const float4* w4 = reinterpret_cast<const float4*>(W + (int64_t)f * d);
    float s = 0.f, l = 0.f;
    for (int i = lane; i < nvec; i += 32) {
      const float4 v = w4[i];
      s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      const float vv[4] = {v.x, v.y, v.z, v.w};
      l += st4_f16_cand(W_h ? W_h + (int64_t)f * f16_ld(d) + 4 * i : nullptr, vv);
    }
    best = fmaxf(best, warp_sum(s));
    best_lo = fmaxf(best_lo, warp_sum(l));
  }
  if (lane == 0 && best > 0.f) {
    atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(sqrtf(best)));
    atomicMax(reinterpret_cast<unsigned int*>(out) + 1, __float_as_uint(sqrtf(best_lo)));
  }
}

// PB_ENC_PAIR=0 forces the one-CTA kernel, =1 the CTA-pair kernel (default: pairs when at least two 256-token tiles exist)
static int enc_pair_mode() {
  const char* v = getenv("PB_ENC_PAIR");       // read per call: tests flip it inside one process
  return v && *v ? atoi(v) : -1;
}

template <int C_KEEP>
int launch_enc_cand_pair(const PbSaeEncode* e, cudaStream_t st) {
  CUtensorMap tmA, tmBh;
  PB_TRY(make_map(&tmA, e->sae_in_h, TC_F16, e->rows, e->d, f16_ld(e->d), TC_BM));
  PB_TRY(make_map(&tmBh, e->W_encT_h, TC_F16, e->F, e->d, f16_ld(e->d), FZ_BN / 2));       // box = this CTA's half of the dictionary tile
  auto kern = k_enc_cand_pair<C_KEEP>;
  static bool attr_done = false;
  if (!attr_done) {
    PB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FZP_SMEM));
    attr_done = true;
  }
  const int num_m = (e->rows + 255) / 256, num_n = (e->F + FZ_BN - 1) / FZ_BN;
  int clusters = pb_sm_count() / 2;
  if (clusters > num_m * num_n) clusters = num_m * num_n;
  PB_LAUNCH_PDL(kern, 2 * clusters, FZ_THREADS, FZP_SMEM, st, tmA, tmBh, e->d, e->rows, e->F, e->b_enc, e->cand, num_m, num_n);
  return PB_OK;
}

template <int C_KEEP>
int launch_enc_cand(const PbSaeEncode* e, cudaStream_t st) {
  const int pm = enc_pair_mode();
  if (pm == 1 || (pm < 0 && PB_ENC_PAIR_DEFAULT && e->rows >= 512)) return launch_enc_cand_pair<C_KEEP>(e, st);
  CUtensorMap tmA, tmB;
  PB_TRY(make_map(&tmA, e->sae_in_h, TC_F16, e->rows, e->d, f16_ld(e->d), TC_BM));
  PB_TRY(make_map(&tmB, e->W_encT_h, TC_F16, e->F, e->d, f16_ld(e->d), FZ_BN));
  auto kern = k_enc_cand<C_KEEP>;
  static bool attr_done = false;
  if (!attr_done) {
    PB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FZ_SMEM));
    attr_done = true;
  }
  const int num_m = (e->rows + TC_BM - 1) / TC_BM, num_n = (e->F + FZ_BN - 1) / FZ_BN;
  int grid = pb_sm_count();
  if (grid > num_m * num_n) grid = num_m * num_n;
  PB_LAUNCH_PDL(kern, grid, FZ_THREADS, FZ_SMEM, st, tmA, tmB, e->d, e->rows, e->F, e->b_enc, e->cand, num_m, num_n);
  return PB_OK;
}

template <int SPT>
int launch_select(const PbSaeEncode* e, int nseg, float scale, cudaStream_t st) {
  const size_t smem = sizeof(float) * e->d;
  PB_LAUNCH_PDL(k_cand_select<SPT>, e->rows, 256, smem, st, (const int*)e->cand, nseg, e->c_keep, e->sae_in, e->W_encT, e->b_enc, e->enc_norm_max, scale,
                e->d, e->k, e->m_cand, e->idx, e->val, e->feat_count, e->fb_count, e->fb_rows, e->fb_count + 1);
  return PB_OK;
}

}  // namespace

extern "C" int pb_sae_fused_workspace(int32_t rows, int32_t F, int32_t c_keep, int64_t* cand_bytes, int64_t* fb_scratch_bytes) {
  PB_CHECK_ARG(rows >= 0 && F > 0 && F % FZ_SEG == 0 && (c_keep == 4 || c_keep == 6 || c_keep == 8) && cand_bytes && fb_scratch_bytes,
               "pb_sae_fused_workspace: needs d_sae %% 128 == 0 and c_keep in {4, 6, 8}");
  *cand_bytes = (int64_t)rows * (F / FZ_SEG) * c_keep * 4;
  *fb_scratch_bytes = (int64_t)2 * pb_sm_count() * F * 4;
  return PB_OK;
}

extern "C" int pb_sae_encode_topk_fused(const PbSaeEncode* e, pb_stream_t stream) {
  PB_CHECK_ARG(e && e->sae_in && e->W_encT && e->sae_in_h && e->W_encT_h && e->b_enc && e->cand && e->enc_norm_max && e->idx && e->val &&
                   e->fb_count && e->fb_rows,
               "pb_sae_encode_topk_fused: missing pointers");
  PB_CHECK_ARG(e->rows >= 0 && e->d >= 32 && e->d % 4 == 0 && e->d <= 8192 && e->F % FZ_SEG == 0 && e->F >= FZ_SEG,
               "pb_sae_encode_topk_fused: needs d_in %% 4 == 0, 32 <= d_in <= 8192, d_sae %% 128 == 0 (d=%d F=%d)", e->d, e->F);
  PB_CHECK_ARG(e->c_keep == 4 || e->c_keep == 6 || e->c_keep == 8, "pb_sae_encode_topk_fused: c_keep must be 4, 6 or 8");
  PB_CHECK_ARG(e->k >= 1 && e->k <= 64 && e->k <= e->m_cand && e->m_cand <= SEL_MAX_CAND && e->k <= e->F,
               "pb_sae_encode_topk_fused: needs k <= 64 and k <= m_cand <= %d", SEL_MAX_CAND);
  PB_CHECK_ARG(pb_aligned16(e->sae_in) && pb_aligned16(e->W_encT) && pb_aligned16(e->sae_in_h) && pb_aligned16(e->W_encT_h) &&
                   pb_aligned16(e->b_enc) && pb_aligned16(e->cand),
               "pb_sae_encode_topk_fused: operands must be 16-byte aligned");
  const int nkeys = e->F / FZ_SEG * e->c_keep;
  PB_CHECK_ARG(e->F / FZ_SEG <= 256 * 4, "pb_sae_encode_topk_fused: d_sae=%d too large for the selection kernel (max 131072)", e->F);
  PB_CHECK_ARG(e->cand_bytes >= (int64_t)e->rows * nkeys * 4, "pb_sae_encode_topk_fused: candidate buffer too small");
  if (e->rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int phases = (e->phases & 7) ? e->phases : (e->phases | 7);
  if (phases & 1) {
    if (e->c_keep == 4) PB_TRY(launch_enc_cand<4>(e, st));
    else if (e->c_keep == 6) PB_TRY(launch_enc_cand<6>(e, st));
    else PB_TRY(launch_enc_cand<8>(e, st));
  }
  if (phases & 2) {
    if (!(phases & 8)) PB_CUDA(cudaMemsetAsync(e->fb_count, 0, 2 * sizeof(int), st));    // [0] rows on the exact path, [1] candidates re-scored
    const float coef = e->err_coef > 0.f ? e->err_coef : 1.05f;       // safety factor on the Cauchy-Schwarz bound (norms evaluated in fp32)
    const int nseg = e->F / FZ_SEG, spt = (nseg + 255) / 256;
    if (spt <= 1) PB_TRY(launch_select<1>(e, nseg, coef, st));
    else if (spt <= 2) PB_TRY(launch_select<2>(e, nseg, coef, st));
    else PB_TRY(launch_select<4>(e, nseg, coef, st));
  }
  if (phases & 4) {
    PB_CHECK_ARG(e->fb_scratch && e->fb_scratch_bytes >= (int64_t)e->F * 4, "pb_sae_encode_topk_fused: fallback scratch missing");
    int grid = (int)(e->fb_scratch_bytes / ((int64_t)e->F * 4));
    if (grid > 2 * pb_sm_count()) grid = 2 * pb_sm_count();
    int cap = ((e->F + 255) / 256) * e->k;
    if (cap > e->F) cap = e->F;
    const size_t smem = sizeof(float) * e->d + 8 * (size_t)cap;
    PB_CHECK_ARG(smem <= 200 * 1024, "pb_sae_encode_topk_fused: k=%d x d_sae=%d too large for the exact-path candidate buffer", e->k, e->F);
    static size_t attr_smem = 0;
    if (smem > 48 * 1024 && smem > attr_smem) {
      PB_CUDA(cudaFuncSetAttribute(k_topk_fallback, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_smem = smem;
    }
    PB_LAUNCH_PDL(k_topk_fallback, grid, 256, smem, st, (const int*)e->fb_count, (const int*)e->fb_rows, e->sae_in, e->W_encT, e->b_enc, e->fb_scratch,
                  e->d, e->F, e->k, cap, e->idx, e->val, e->feat_count);
  }
  return PB_OK;
}

extern "C" int pb_rownorm_max(const float* W, int32_t F, int32_t d, float* out, void* W_h, pb_stream_t stream) {
  PB_CHECK_ARG(W && out && F >= 0 && d > 0 && d % 4 == 0, "pb_rownorm_max: bad arguments");
  PB_CHECK_ARG(pb_aligned16(W_h), "pb_rownorm_max: W_h must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  PB_CUDA(cudaMemsetAsync(out, 0, 2 * sizeof(float), st));
  if (F == 0) return PB_OK;
  int grid = pb_sm_count() * 4;
  if (grid > (F + 7) / 8) grid = (F + 7) / 8;
  k_rownorm_max<<<grid, 256, 0, st>>>(W, F, d, out, reinterpret_cast<uint16_t*>(W_h));
  PB_LAUNCH_CHECK();
  return PB_OK;
}

int pb_abi_sizeof_fused(int which) { return which == 9 ? (int)sizeof(PbSaeEncode) : -1; }
