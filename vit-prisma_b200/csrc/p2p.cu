// p2p.cu -- data-parallel SAE training over NVLink 5 / NVSwitch peer memory, no NCCL on the data path.
//
// One process per GPU (torchrun).  Buffers that peers must see (gradients, parameters, a few small vectors and the
// barrier flags) are cudaMalloc'd here and exported with CUDA IPC handles; the host side (vit_prisma/b200/p2p.py)
// swaps the 64-byte handles through torch.distributed once at start-up -- that exchange is the only use of a
// collective library.  Every step then runs:
//
//   local forward / backward (sae.cu)                      -> this rank's gW_dec, gW_encT, gb_enc, gb_dec, fired, xsum
//   k_p2p_barrier                                          (all ranks' gradients are complete)
//   k_p2p_reduce_scatter: rank r owns feature rows [r*F/N, (r+1)*F/N): it LOADS those rows from every peer's gradient
//        buffers (16-byte peer loads over NVLink), sums them into its own buffer, accumulates ||.||^2 of the reduced slice,
//        and reduces the small vectors (gb_enc, gb_dec, fired) fully; publishes its norm partial to every peer
//   k_p2p_barrier                                          (norm partials visible, all peer reads of this step done)
//   k_p2p_adam_allgather: global clip coefficient, decoder-parallel-gradient removal, Adam and row renorm on the OWNED rows
//        (Adam state is therefore sharded 1/N), then STORES the updated rows into every peer's parameter buffers
//   k_p2p_barrier                                          (all parameters updated everywhere)
//
// The gradient is the SUM over ranks: each rank's local gradient already carries the 1/(global tokens) factor of the
// mean loss, and the batch statistics the loss needs (column mean of x, sae.py:145) are reduced across ranks first.
#include "common.cuh"

#define PB_MAX_RANKS 8

// NVSwitch multicast (mc.cu): one instruction reads the SUM of every rank's copy / writes every rank's copy
__device__ __forceinline__ float4 mc_ld_reduce4(const float* mc_addr) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(mc_addr)
               : "memory");
  return v;
}
__device__ __forceinline__ void mc_st4(float* mc_addr, const float (&v)[4]) {
  asm volatile("multimem.st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");   // weak: the flag barrier's system fence publishes it
}
__device__ __forceinline__ void mc_st1(float* mc_addr, float v) {
  asm volatile("multimem.st.global.f32 [%0], %1;" ::"l"(mc_addr), "f"(v) : "memory");
}

struct P2PTables {
  int rank, world;
  float* gW_dec[PB_MAX_RANKS];
  float* gW_encT[PB_MAX_RANKS];
  float* gb_enc[PB_MAX_RANKS];
  float* gb_dec[PB_MAX_RANKS];
  float* fired[PB_MAX_RANKS];
  float* xsum[PB_MAX_RANKS];
  float* W_dec[PB_MAX_RANKS];
  float* W_encT[PB_MAX_RANKS];
  float* W_encT_lo[PB_MAX_RANKS];
  float* b_enc[PB_MAX_RANKS];
  float* norm_parts[PB_MAX_RANKS];   // [world] floats on every rank
  unsigned int* flags[PB_MAX_RANKS]; // [world] arrival epochs on every rank
};

// ------------------------------------------------------------------------------------------- memory
extern "C" int pb_p2p_alloc(int64_t bytes, void** dev_ptr, unsigned char* handle64) {
  PB_CHECK_ARG(bytes > 0 && dev_ptr && handle64, "pb_p2p_alloc: bad arguments");
  PB_CUDA(cudaMalloc(dev_ptr, (size_t)bytes));
  PB_CUDA(cudaMemset(*dev_ptr, 0, (size_t)bytes));
  cudaIpcMemHandle_t h;
  PB_CUDA(cudaIpcGetMemHandle(&h, *dev_ptr));
  static_assert(sizeof(h) == 64, "CUDA IPC handle is 64 bytes");
  memcpy(handle64, &h, 64);
  return PB_OK;
}
extern "C" int pb_p2p_open(const unsigned char* handle64, void** peer_ptr) {
  PB_CHECK_ARG(handle64 && peer_ptr, "pb_p2p_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  PB_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return PB_OK;
}
extern "C" int pb_p2p_close(void* peer_ptr) {
  PB_CUDA(cudaIpcCloseMemHandle(peer_ptr));
  return PB_OK;
}
extern "C" int pb_p2p_free(void* dev_ptr) {
  PB_CUDA(cudaFree(dev_ptr));
  return PB_OK;
}

// ------------------------------------------------------------------------------------------- barrier
// Thread r stores this rank's epoch into peer r's flag slot [rank] (system-scope release) and waits until peer r's
// epoch has arrived in our own slot [r] (acquire).  Stream order makes everything before the barrier kernel visible.
__global__ void k_p2p_barrier(P2PTables t, unsigned int epoch) {
  const int r = threadIdx.x;
  if (r < t.world) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(t.flags[r] + t.rank), "r"(epoch) : "memory");
    const unsigned int* mine = t.flags[t.rank] + r;
    const long long t0 = clock64();
    for (;;) {
      unsigned int v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if ((int)(v - epoch) >= 0) break;
      if (clock64() - t0 > 20000000000LL) {   // ~10 s: a peer died; fail loudly instead of hanging the box
        printf("p2p barrier timeout: rank %d waiting for rank %d at epoch %u (have %u)\n", t.rank, r, epoch, v);
        __trap();
      }
    }
    __threadfence_system();
  }
}

// sum of d floats from every rank's xsum into this rank's xsum_global (batch mean of x across the global batch)
__global__ void k_p2p_sum_small(P2PTables t, float* __restrict__ out, int which, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int r = 0; r < t.world; ++r) {
      const float* src = which == 0 ? t.xsum[r] : which == 1 ? t.gb_enc[r] : which == 2 ? t.gb_dec[r] : t.fired[r];
      acc += src[i];
    }
    out[i] = acc;
  }
}

// gb_enc [F], gb_dec [d], fired [F] summed over ranks in one launch (three launches of k_p2p_sum_small + a memset before:
// four dependent ~4 us launches in front of the reduce-scatter); thread 0 also resets the step's accumulators
__global__ void __launch_bounds__(256) k_p2p_sum_small3(P2PTables t, float* __restrict__ gb_enc_red, float* __restrict__ gb_dec_red,
                                                       float* __restrict__ fired_red, int F, int d, float* __restrict__ part_accum) {
  if (blockIdx.x == 0 && threadIdx.x < 4) part_accum[threadIdx.x] = 0.f;   // [0] gradient-norm partial of the owned slice
  const int n = 2 * F + d;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int which = i < F ? 0 : i < 2 * F ? 1 : 2;
    const int j = which == 0 ? i : which == 1 ? i - F : i - 2 * F;
    float acc = 0.f;
    for (int r = 0; r < t.world; ++r) acc += (which == 0 ? t.gb_enc[r] : which == 1 ? t.fired[r] : t.gb_dec[r])[j];
    (which == 0 ? gb_enc_red : which == 1 ? fired_red : gb_dec_red)[j] = acc;
  }
}

// ------------------------------------------------------------------------------------------- reduce-scatter + norm
// rows [f0, f1) of both gradient matrices: own += sum of peers; partial ||g||^2 -> every peer's norm_parts[rank]
// One gradient array's owned slice: own[i] = sum over ranks of that rank's copy, owner first then (rank + j) % world -- a fixed order per row; returns this thread's share of ||.||^2.
// W = compile-time rank count (ranks >= t.world are skipped when W is the generic PB_MAX_RANKS), U = elements per trip.
template <int W, int U>
__device__ __forceinline__ float rs_peer_slice(const P2PTables& t, int m, int64_t base4, int64_t n4, float4* __restrict__ own, int64_t tid,
                                               int64_t stride) {
  // slot j holds rank (t.rank + j) % world: at any instant the 8 GPUs pull from 8 different peers (a permutation through the
  // switch) instead of all hitting rank 0, then rank 1, ...; the sum therefore runs owner-first, in the same order every step
  const float4* src[W];
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const int r = (t.rank + j) % t.world;
    src[j] = j < t.world ? reinterpret_cast<const float4*>(m == 0 ? t.gW_dec[r] : t.gW_encT[r]) + base4 : nullptr;
  }
  float nsq = 0.f;
  int64_t i = tid;
  for (; i + (U - 1) * stride < n4; i += U * stride) {
    float4 v[U][W];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int r = 0; r < W; ++r)
        if (r < t.world) v[u][r] = src[r][i + u * stride];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float4 acc = v[u][0];
#pragma unroll
      for (int r = 1; r < W; ++r)
        if (r < t.world) { acc.x += v[u][r].x; acc.y += v[u][r].y; acc.z += v[u][r].z; acc.w += v[u][r].w; }
      own[i + u * stride] = acc;
      nsq += acc.x * acc.x + acc.y * acc.y + acc.z * acc.z + acc.w * acc.w;
    }
  }
  for (; i < n4; i += stride) {
    float4 acc = src[0][i];
#pragma unroll
    for (int r = 1; r < W; ++r)
      if (r < t.world) { const float4 b = src[r][i]; acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w; }
    own[i] = acc;
    nsq += acc.x * acc.x + acc.y * acc.y + acc.z * acc.z + acc.w * acc.w;
  }
  return nsq;
}

// W / U: compile-time rank count and elements per trip of the peer-load path (0 / 0 = the multicast path).  One instantiation per
// case: as one kernel with a runtime switch the four unrolled bodies cost 254 registers (one CTA per SM).
template <int W, int U>
__global__ void __launch_bounds__(256, 3) k_p2p_reduce_scatter(P2PTables t, int f0, int f1, int d, const float* __restrict__ gb_enc_red,
                                                              const float* __restrict__ gb_dec_red, int F, float* __restrict__ part_accum,
                                                              const float* __restrict__ mc_gW_dec, const float* __restrict__ mc_gW_encT) {
  const int64_t n4 = (int64_t)(f1 - f0) * d / 4;
  const int64_t base4 = (int64_t)f0 * d / 4;
  float nsq = 0.f;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  for (int m = 0; m < 2; ++m) {
    float4* own = reinterpret_cast<float4*>(m == 0 ? t.gW_dec[t.rank] : t.gW_encT[t.rank]) + base4;
    const float* mc = m == 0 ? mc_gW_dec : mc_gW_encT;
    if constexpr (W == 0) {
      // summed inside the switch: this slice crosses NVLink once.  A multimem load is a round trip through the switch (several
      // microseconds): four independent loads per thread keep enough bytes in flight (one per trip ran at 270 GB/s, r2d_bench2).
      const float* src = mc + 4 * base4;
      int64_t i = tid;
      for (; i + 3 * stride < n4; i += 4 * stride) {
        const float4 a0 = mc_ld_reduce4(src + 4 * i), a1 = mc_ld_reduce4(src + 4 * (i + stride)), a2 = mc_ld_reduce4(src + 4 * (i + 2 * stride)),
                     a3 = mc_ld_reduce4(src + 4 * (i + 3 * stride));
        own[i] = a0; own[i + stride] = a1; own[i + 2 * stride] = a2; own[i + 3 * stride] = a3;
        nsq += a0.x * a0.x + a0.y * a0.y + a0.z * a0.z + a0.w * a0.w + a1.x * a1.x + a1.y * a1.y + a1.z * a1.z + a1.w * a1.w +
               a2.x * a2.x + a2.y * a2.y + a2.z * a2.z + a2.w * a2.w + a3.x * a3.x + a3.y * a3.y + a3.z * a3.z + a3.w * a3.w;
      }
      for (; i < n4; i += stride) {
        const float4 a = mc_ld_reduce4(src + 4 * i);
        own[i] = a;
        nsq += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
      }
      continue;
    }
    // peer loads (NVLink): a load from a peer is a ~2 us round trip, so eight 16-byte loads per thread are issued before the first
    // is consumed -- all ranks' copies of U = 8 / world consecutive elements (adding them one by one inside a runtime-bounded
    // loop ran at 489 GB/s at 8 ranks, r2g_bench8_peer; one element per trip at 2 ranks at 409 GB/s, r2i_bench2).
    if constexpr (W != 0) nsq += rs_peer_slice<W, U>(t, m, base4, n4, own, tid, stride);
  }
  // small vectors are fully reduced on every rank; only rank 0 counts their norm so the global sum counts them once
  if (t.rank == 0) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < F; i += gridDim.x * blockDim.x) nsq += gb_enc_red[i] * gb_enc_red[i];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d; i += gridDim.x * blockDim.x) nsq += gb_dec_red[i] * gb_dec_red[i];
  }
  nsq = warp_sum(nsq);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = nsq;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int i = 0; i < 8; ++i) a += red[i];
    atomicAdd(part_accum, a);
  }
}
__global__ void k_p2p_publish_norm(P2PTables t, float* part_accum) {
  const int r = threadIdx.x;
  if (r < t.world) t.norm_parts[r][t.rank] = *part_accum;     // peer store
}

struct SaeScalarsP2P { float loss_sum, gnorm_sq, clip_coef, mse, l0, pos_count, grad_norm, reserved; };

// after the norm barrier: total norm, clip coefficient, global loss statistics
__global__ void k_p2p_finalize(P2PTables t, SaeScalarsP2P* sc, float max_norm, float inv_elems_global, float inv_rows_global) {
  float tot = 0.f;
  for (int r = 0; r < t.world; ++r) tot += t.norm_parts[t.rank][r];
  const float norm = sqrtf(tot);
  sc->gnorm_sq = tot;
  sc->grad_norm = norm;
  sc->clip_coef = max_norm > 0.f ? fminf(1.f, max_norm / (norm + 1e-6f)) : 1.f;
  sc->mse = sc->loss_sum * inv_elems_global;      // this rank's share of the global mean (ranks' shares add up)
  sc->l0 = sc->pos_count * inv_rows_global;
}

// ------------------------------------------------------------------------------------------- Adam on owned rows + all-gather
struct AdamHyperP2P { float lr, beta1, beta2, eps, bc1, bc2_sqrt; };
__device__ __forceinline__ float adam_upd(float p, float gr, float& m, float& v, const AdamHyperP2P& h) {   // same arithmetic as sae.cu adam_update
  m = h.beta1 * m + (1.f - h.beta1) * gr;
  v = h.beta2 * v + (1.f - h.beta2) * gr * gr;
  float sq, rc;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
  const float denom = fmaf(sq, __frcp_rn(h.bc2_sqrt), h.eps);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(denom));
  return fmaf(-(h.lr * __frcp_rn(h.bc1)) * m, rc, p);
}

template <int CHUNKS>
__global__ void __launch_bounds__(256) k_p2p_adam_allgather(P2PTables t, int f0, int f1, int d, const float* __restrict__ gb_enc_red,
                                                           float* __restrict__ m_dec, float* __restrict__ v_dec, float* __restrict__ m_enc,
                                                           float* __restrict__ v_enc, float* __restrict__ m_be, float* __restrict__ v_be,
                                                           const SaeScalarsP2P* __restrict__ sc, AdamHyperP2P h, float* __restrict__ mc_W_dec,
                                                           float* __restrict__ mc_W_encT, float* __restrict__ mc_b_enc, int defer_dec) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  const float clip = sc->clip_coef;
  float* W_dec = t.W_dec[t.rank];
  float* W_encT = t.W_encT[t.rank];
  const float* gWd = t.gW_dec[t.rank];
  const float* gWe = t.gW_encT[t.rank];
  // destination j = rank (t.rank + j) % world: every GPU addresses a different peer at a time (permutation traffic through the switch)
  float *wdec_rot[PB_MAX_RANKS], *wenc_rot[PB_MAX_RANKS], *wlo_rot[PB_MAX_RANKS];
#pragma unroll
  for (int j = 0; j < PB_MAX_RANKS; ++j) {
    const int r = (t.rank + j) % t.world;
    wdec_rot[j] = t.W_dec[r]; wenc_rot[j] = t.W_encT[r]; wlo_rot[j] = t.W_encT_lo[r];
  }
  for (int f = f0 + blockIdx.x * nw + warp; f < f1; f += gridDim.x * nw) {
    const int64_t base = (int64_t)f * d;
    float w[CHUNKS][4], gq[CHUNKS][4];
    float par = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        ld4(W_dec + base + 4 * c4, w[i]);
        ld4(gWd + base + 4 * c4, gq[i]);
#pragma unroll
        for (int q = 0; q < 4; ++q) { gq[i][q] *= clip; par = fmaf(gq[i][q], w[i][q], par); }
      } else {
        w[i][0] = w[i][1] = w[i][2] = w[i][3] = gq[i][0] = gq[i][1] = gq[i][2] = gq[i][3] = 0.f;
      }
    }
    par = warp_sum(par);
    float nsq = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        float mm[4], vv[4];
        ld4(m_dec + base + 4 * c4, mm);
        ld4(v_dec + base + 4 * c4, vv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          w[i][q] = adam_upd(w[i][q], gq[i][q] - par * w[i][q], mm[q], vv[q], h);
          nsq += w[i][q] * w[i][q];
        }
        st4(m_dec + base + 4 * c4, mm);
        st4(v_dec + base + 4 * c4, vv);
      }
    }
    const float inv_nrm = 1.f / sqrtf(warp_sum(nsq));
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
#pragma unroll
        for (int q = 0; q < 4; ++q) w[i][q] = w[i][q] * inv_nrm;
        if (defer_dec) st4(W_dec + base + 4 * c4, w[i]);                                   // own copy only: pb_p2p_push_dec sends it later
        else if (mc_W_dec) mc_st4(mc_W_dec + base + 4 * c4, w[i]);                         // all-gather: one multicast store
        else for (int j = 0; j < t.world; ++j) st4(wdec_rot[j] + base + 4 * c4, w[i]);     // all-gather: peer stores, own copy first
      }
    }
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        float p[4], gr[4], mm[4], vv[4], lo[4];
        ld4(W_encT + base + 4 * c4, p);
        ld4(gWe + base + 4 * c4, gr);
        ld4(m_enc + base + 4 * c4, mm);
        ld4(v_enc + base + 4 * c4, vv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          p[q] = adam_upd(p[q], gr[q] * clip, mm[q], vv[q], h);
          lo[q] = tf32_lo(p[q]);
        }
        st4(m_enc + base + 4 * c4, mm);
        st4(v_enc + base + 4 * c4, vv);
        if (mc_W_encT) {
          mc_st4(mc_W_encT + base + 4 * c4, p);
        } else {
          for (int j = 0; j < t.world; ++j) {
            st4(wenc_rot[j] + base + 4 * c4, p);
            if (wlo_rot[j]) st4(wlo_rot[j] + base + 4 * c4, lo);             // tf32 residual plane: dense 3xTF32 encoder only
          }
        }
      }
    }
    if (lane == 0) {
      float mm = m_be[f], vv = v_be[f];
      const float nb = adam_upd(t.b_enc[t.rank][f], gb_enc_red[f] * clip, mm, vv, h);
      m_be[f] = mm;
      v_be[f] = vv;
      if (mc_b_enc) mc_st1(mc_b_enc + f, nb);
      else for (int r = 0; r < t.world; ++r) t.b_enc[r][f] = nb;
    }
  }
}

// replicated tiny updates: b_dec Adam (identical inputs on every rank -> identical result) and the dead-feature counters
__global__ void __launch_bounds__(256) k_p2p_small_updates(P2PTables t, float* __restrict__ b_dec,
                                                          const float* __restrict__ gb_dec_red, float* __restrict__ m_bd,
                                                          float* __restrict__ v_bd, const float* __restrict__ fired_red,
                                                          float* __restrict__ since_fired, float* __restrict__ act_freq,
                                                          const SaeScalarsP2P* __restrict__ sc, AdamHyperP2P h, int d, int F) {
  const float clip = sc->clip_coef;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < F; i += gridDim.x * blockDim.x) {
    if (i < d) {
      float mm = m_bd[i], vv = v_bd[i];
      b_dec[i] = adam_upd(b_dec[i], gb_dec_red[i] * clip, mm, vv, h);
      m_bd[i] = mm;
      v_bd[i] = vv;
    }
    if (since_fired) since_fired[i] = fired_red[i] > 0.f ? 0.f : since_fired[i] + 1.f;
    if (act_freq) act_freq[i] += fired_red[i];
  }
}

// ------------------------------------------------------------------------------------------- C ABI
static int fill_tables(const PbP2PStep* s, P2PTables* t) {
  PB_CHECK_ARG(s && s->world >= 1 && s->world <= PB_MAX_RANKS && s->rank >= 0 && s->rank < s->world, "pb_p2p: bad rank/world");
  t->rank = s->rank;
  t->world = s->world;
  for (int r = 0; r < s->world; ++r) {
    t->gW_dec[r] = s->gW_dec[r]; t->gW_encT[r] = s->gW_encT[r]; t->gb_enc[r] = s->gb_enc[r]; t->gb_dec[r] = s->gb_dec[r];
    t->fired[r] = s->fired[r]; t->xsum[r] = s->xsum[r]; t->W_dec[r] = s->W_dec[r]; t->W_encT[r] = s->W_encT[r];
    t->W_encT_lo[r] = s->W_encT_lo[r]; t->b_enc[r] = s->b_enc[r]; t->norm_parts[r] = s->norm_parts[r]; t->flags[r] = s->flags[r];
  }
  return PB_OK;
}

extern "C" int pb_p2p_barrier(const PbP2PStep* s, uint32_t epoch, pb_stream_t stream) {
  P2PTables t;
  PB_TRY(fill_tables(s, &t));
  k_p2p_barrier<<<1, 32, 0, (cudaStream_t)stream>>>(t, epoch);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// xsum_global[d] = sum over ranks of xsum (call after a barrier that follows pb_sae_prep on every rank)
extern "C" int pb_p2p_sum_xsum(const PbP2PStep* s, float* xsum_global, pb_stream_t stream) {
  P2PTables t;
  PB_TRY(fill_tables(s, &t));
  k_p2p_sum_small<<<(s->d + 255) / 256, 256, 0, (cudaStream_t)stream>>>(t, xsum_global, 0, s->d);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

extern "C" int pb_p2p_reduce_scatter(const PbP2PStep* s, pb_stream_t stream) {
  P2PTables t;
  PB_TRY(fill_tables(s, &t));
  PB_CHECK_ARG(s->gb_enc_red && s->gb_dec_red && s->fired_red && s->part_accum, "pb_p2p_reduce_scatter: reduction buffers missing");
  PB_CHECK_ARG((s->F % s->world) == 0 && (((int64_t)(s->F / s->world) * s->d) % 4) == 0, "pb_p2p_reduce_scatter: F must divide evenly by world");
  cudaStream_t st = (cudaStream_t)stream;
  const int per = s->F / s->world, f0 = s->rank * per, f1 = f0 + per;
  k_p2p_sum_small3<<<(2 * s->F + s->d + 255) / 256, 256, 0, st>>>(t, s->gb_enc_red, s->gb_dec_red, s->fired_red, s->F, s->d, s->part_accum);
  PB_LAUNCH_CHECK();
  PB_CHECK_ARG(!s->mc_gW_dec == !s->mc_gW_encT, "pb_p2p_reduce_scatter: both multicast gradient views or none");
#define PB_RS(W_, U_) k_p2p_reduce_scatter<W_, U_><<<pb_sm_count() * 3, 256, 0, st>>>(t, f0, f1, s->d, s->gb_enc_red, s->gb_dec_red, s->F, s->part_accum, s->mc_gW_dec, s->mc_gW_encT)
  if (s->mc_gW_dec) PB_RS(0, 0);
  else if (s->world == 2) PB_RS(2, 4);
  else if (s->world == 4) PB_RS(4, 2);
  else if (s->world == 8) PB_RS(8, 1);
  else PB_RS(PB_MAX_RANKS, 1);
#undef PB_RS
  PB_LAUNCH_CHECK();
  k_p2p_publish_norm<<<1, 32, 0, st>>>(t, s->part_accum);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

extern "C" int pb_p2p_adam_allgather(const PbP2PStep* s, pb_stream_t stream) {
  P2PTables t;
  PB_TRY(fill_tables(s, &t));
  PB_CHECK_ARG(s->m_dec && s->v_dec && s->m_enc && s->v_enc && s->m_be && s->v_be && s->m_bd && s->v_bd && s->scalars && s->b_dec,
               "pb_p2p_adam_allgather: optimizer state missing");
  PB_CHECK_ARG(s->step >= 1, "pb_p2p_adam_allgather: step counter starts at 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int per = s->F / s->world, f0 = s->rank * per, f1 = f0 + per;
  AdamHyperP2P h;
  h.lr = s->lr; h.beta1 = s->beta1; h.beta2 = s->beta2; h.eps = s->adam_eps;
  h.bc1 = 1.f - powf(s->beta1, (float)s->step);
  h.bc2_sqrt = sqrtf(1.f - powf(s->beta2, (float)s->step));
  k_p2p_finalize<<<1, 1, 0, st>>>(t, (SaeScalarsP2P*)s->scalars, s->max_grad_norm, 1.f / ((float)s->global_rows * (float)s->d),
                                  1.f / (float)s->global_rows);
  PB_LAUNCH_CHECK();
  const int d = s->d;
  int grid = pb_sm_count() * 4;
  if (grid > (per + 7) / 8) grid = (per + 7) / 8;
  PB_CHECK_ARG((!s->mc_W_dec == !s->mc_W_encT) && (!s->mc_W_dec == !s->mc_b_enc), "pb_p2p_adam_allgather: all three multicast parameter views or none");
#define PB_P2P_ADAM(CH) k_p2p_adam_allgather<CH><<<grid, 256, 0, st>>>(t, f0, f1, d, s->gb_enc_red, s->m_dec, s->v_dec, s->m_enc, s->v_enc, s->m_be, s->v_be, (const SaeScalarsP2P*)s->scalars, h, s->mc_W_dec, s->mc_W_encT, s->mc_b_enc, s->defer_dec)
  const int nvec = d / 4;
  if (d % 4 != 0 || nvec > 384) { pb_set_error("pb_p2p_adam_allgather: d_in=%d unsupported", d); return PB_EUNSUPPORTED; }
  if (nvec <= 32) PB_P2P_ADAM(1);
  else if (nvec <= 64) PB_P2P_ADAM(2);
  else if (nvec <= 128) PB_P2P_ADAM(4);
  else if (nvec <= 192) PB_P2P_ADAM(6);
  else if (nvec <= 256) PB_P2P_ADAM(8);
  else PB_P2P_ADAM(12);
#undef PB_P2P_ADAM
  PB_LAUNCH_CHECK();
  k_p2p_small_updates<<<(s->F + 255) / 256, 256, 0, st>>>(t, s->b_dec, s->gb_dec_red, s->m_bd, s->v_bd, s->fired_red, s->since_fired,
                                                        s->act_freq, (const SaeScalarsP2P*)s->scalars, h, d, s->F);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// Deferred half of the all-gather: the owned W_dec rows -> every peer (or one multicast store).  The next step needs W_dec only at
// its decode, ~0.35 ms after the encoder matrix, so this runs on a side stream under the next step's prep / encoder GEMM / select.
__global__ void __launch_bounds__(256) k_p2p_push_dec(P2PTables t, int f0, int f1, int d, float* __restrict__ mc_W_dec) {
  const int64_t n4 = (int64_t)(f1 - f0) * d / 4, base4 = (int64_t)f0 * d / 4;
  const float4* own = reinterpret_cast<const float4*>(t.W_dec[t.rank]) + base4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = own[i];
    if (mc_W_dec) {
      const float w[4] = {v.x, v.y, v.z, v.w};
      mc_st4(mc_W_dec + 4 * (base4 + i), w);
    } else {
      for (int j = 1; j < t.world; ++j)                                   // rotated: a different peer per GPU at any instant
        (reinterpret_cast<float4*>(t.W_dec[(t.rank + j) % t.world]) + base4)[i] = v;
    }
  }
}

extern "C" int pb_p2p_push_dec(const PbP2PStep* s, pb_stream_t stream) {
  P2PTables t;
  PB_TRY(fill_tables(s, &t));
  const int per = s->F / s->world, f0 = s->rank * per, f1 = f0 + per;
  k_p2p_push_dec<<<pb_sm_count() * 2, 256, 0, (cudaStream_t)stream>>>(t, f0, f1, s->d, s->mc_W_dec);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

int pb_abi_sizeof_fused(int which);  // sae_fused.cu
int pb_abi_sizeof_p2p(int which) { return which == 8 ? (int)sizeof(PbP2PStep) : pb_abi_sizeof_fused(which); }
