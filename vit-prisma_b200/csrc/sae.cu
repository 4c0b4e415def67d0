// sae.cu -- TopK sparse-autoencoder forward / training step (reference sae/sae.py:32-645,
// sae/train_sae.py:278-411) as HBM-bound sm_100a kernels around one tensor-core GEMM.
//
// Data layout in HBM (all fp32, F = d_sae, d = d_in, Bt = tokens per step):
//   W_encT [F][d]   encoder, stored feature-major (the nn.Parameter W_enc [d,F] is a transposed VIEW of it):
//                   K-major B operand of the encoder GEMM, and one contiguous row per feature for the optimizer
//   W_dec  [F][d]   decoder rows (unit norm on entry to every step)
//   idx/val [Bt][k] TopK support of hidden_pre per token (sorted by value, descending) -- the only "feature_acts"
//                   the training step ever materialises; the dense [Bt][F] form exists only on request
//   csc_*           the same support transposed (per feature: the tokens that selected it) for the weight gradients
//
// Step = prep -> encoder GEMM (gemm_tc.cu, 3xTF32) -> topk -> decode+loss+d_hidden -> csc build ->
//        per-feature gradients (+global grad-norm partials) -> finalize (clip coefficient) ->
//        fused clip + decoder-parallel-gradient removal + Adam + decoder row renorm + dead-feature counters.
// No host synchronisation anywhere: scalars (loss, norm, clip coefficient) live in a device struct.
#include "common.cuh"
#include <stdlib.h>
#include "tc_common.cuh"

// ---------------------------------------------------------------------------------------------
// device scalars of one step
struct SaeScalars {
  float loss_sum;      // sum_b sum_c (out-x)^2 / nf[b]            (mse = loss_sum / (Bt*d))
  float gnorm_sq;      // sum of squares of all gradient entries (pre-clip)
  float clip_coef;     // min(1, max_norm / (norm + 1e-6))
  float mse;           // loss_sum / (Bt*d)
  float l0;            // mean number of positive activations per token
  float pos_count;     // accumulator for l0
  float grad_norm;     // sqrt(gnorm_sq)
  float reserved;
};

// ---------------------------------------------------------------------------------------------
// 1. prep: run-time input normalisation + decoder-bias subtraction (sae.py:78-87, 557-566)
//    layer_norm mode: mu = mean(x); xc = x - mu; std = unbiased std(xc); xn = xc / (std + 1e-5)
//    sae_in = xn - b_dec ;  sae_in_lo = tf32 residual (A operand of the 3xTF32 encoder GEMM) ;
//    sae_in_h = f16_cand(sae_in), row stride f16_ld(d) (A operand of the fused encoder's candidate GEMM)
//    xsum[c] += x[b,c]  (batch mean for _compute_mse_loss's centring, sae.py:145)
// one warp per token row; row kept in registers.
template <int CHUNKS>
__global__ void __launch_bounds__(256) k_sae_prep(const float* __restrict__ x, const float* __restrict__ b_dec, float* __restrict__ sae_in,
                                                  float* __restrict__ sae_in_lo, uint16_t* __restrict__ sae_in_h, float* __restrict__ mu_out,
                                                  float* __restrict__ std_out, int rows, int d, int norm_mode, float eps) {
  pb_pdl();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int nvec = d >> 2;
  const float* xr = x + (int64_t)row * d;
  float v[CHUNKS][4];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) {
    const int c4 = i * 32 + lane;
    if (c4 < nvec) { ld4(xr + 4 * c4, v[i]); sum += (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]); }
    else v[i][0] = v[i][1] = v[i][2] = v[i][3] = 0.f;
  }
  float mu = 0.f, inv = 1.f, sd = 1.f;
  if (norm_mode == 1) {  // layer_norm
    mu = warp_sum(sum) / (float)d;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { v[i][j] -= mu; sq += v[i][j] * v[i][j]; }
      }
    }
    sd = sqrtf(warp_sum(sq) / (float)(d - 1));   // torch.std: Bessel-corrected
    inv = 1.f / (sd + eps);
  } else if (norm_mode == 2) {  // constant_norm_rescale: x * sqrt(d) / ||x||
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sq += v[i][j] * v[i][j];
    sd = sqrtf(warp_sum(sq)) / sqrtf((float)d);   // x_out = x_norm * sd
    inv = 1.f / sd;
  }
  if (lane == 0) {
    if (mu_out) mu_out[row] = mu;
    if (std_out) std_out[row] = sd;
  }
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) {
    const int c4 = i * 32 + lane;
    if (c4 < nvec) {
      float bd[4], o[4], lo[4];
      ld4(b_dec + 4 * c4, bd);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        o[j] = (norm_mode == 1 ? v[i][j] / (sd + eps) : v[i][j] * inv) - bd[j];
        lo[j] = tf32_lo(o[j]);
      }
      (void)inv;
      st4(sae_in + (int64_t)row * d + 4 * c4, o);
      if (sae_in_lo) st4(sae_in_lo + (int64_t)row * d + 4 * c4, lo);
      if (sae_in_h) st4_f16_cand(sae_in_h + (int64_t)row * f16_ld(d) + 4 * c4, o);
    }
  }
}

// column sums: out[c] += sum_r x[r,c]   (rows split across CTAs, one atomic per column per CTA)
__global__ void __launch_bounds__(256) k_colsum(const float* __restrict__ x, float* __restrict__ out, int rows, int d, int rows_per_cta) {
  pb_pdl();
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float acc = 0.f;
    for (int r = r0; r < r1; ++r) acc += x[(int64_t)r * d + c];
    atomicAdd(out + c, acc);
  }
}

// ---------------------------------------------------------------------------------------------
// 2. top-k per row (sae.py:795-808 torch.topk(x, k, dim=-1), values sorted descending)
// Exact selection without sorting the row:
//   (a) each of 256 threads scans its strided share of the row and keeps its best key;
//   (b) tau = k-th best of the 256 thread-bests: at least k row elements are >= tau, so every true
//       top-k element is >= tau (keys = (value, lower index wins) are totally ordered -> no tie trouble);
//   (c) elements >= tau are gathered (typically ~k, at most IPT*k) and ranked by counting;
//       rank < k writes slot `rank`, which also leaves the output sorted.
// Rows longer than 256*IPT are cut into segments (grid.y); a second launch merges the per-segment winners.
__device__ __forceinline__ bool key_gt(float va, int ia, float vb, int ib) { return va > vb || (va == vb && ia < ib); }

template <int IPT>
__global__ void __launch_bounds__(256) k_topk(const float* __restrict__ vals, const int* __restrict__ idx_map, int64_t row_stride, int F,
                                              int seg_len, int k, int* __restrict__ out_idx, float* __restrict__ out_val,
                                              int64_t out_row_stride, float* __restrict__ feat_count, int cand_cap) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* best_v = reinterpret_cast<float*>(smem_raw);       // [256]
  int* best_i = reinterpret_cast<int*>(best_v + 256);        // [256]
  float* cand_v = reinterpret_cast<float*>(best_i + 256);    // [cand_cap]
  int* cand_i = reinterpret_cast<int*>(cand_v + cand_cap);   // [cand_cap]
  __shared__ float tau_v;
  __shared__ int tau_i, cand_n;
  const int t = threadIdx.x;
  const int row = blockIdx.x, seg = blockIdx.y;
  const int s0 = seg * seg_len, s1 = min(F, s0 + seg_len);
  const float* vr = vals + (int64_t)row * row_stride;
  const int* mr = idx_map ? idx_map + (int64_t)row * row_stride : nullptr;

  float v[IPT];
  float bv = -INFINITY;
  int bi = 0x7fffffff;
#pragma unroll
  for (int i = 0; i < IPT; ++i) {
    const int p = s0 + t + 256 * i;
    v[i] = p < s1 ? vr[p] : -INFINITY;
    const int gi = p < s1 ? (mr ? mr[p] : p) : 0x7fffffff;
    if (key_gt(v[i], gi, bv, bi)) { bv = v[i]; bi = gi; }
  }
  best_v[t] = bv;
  best_i[t] = bi;
  if (t == 0) cand_n = 0;
  __syncthreads();
  {
    int rank = 0;
    for (int j = 0; j < 256; ++j) rank += key_gt(best_v[j], best_i[j], bv, bi) ? 1 : 0;
    const int kk = min(k, 256);
    if (rank == kk - 1) { tau_v = bv; tau_i = bi; }
  }
  __syncthreads();
  const float tv = tau_v;
  const int ti = tau_i;
#pragma unroll
  for (int i = 0; i < IPT; ++i) {
    const int p = s0 + t + 256 * i;
    if (p < s1) {
      const int gi = mr ? mr[p] : p;
      if (!key_gt(tv, ti, v[i], gi)) {  // key >= tau
        const int slot = atomicAdd(&cand_n, 1);
        if (slot < cand_cap) { cand_v[slot] = v[i]; cand_i[slot] = gi; }
      }
    }
  }
  __syncthreads();
  const int C = min(cand_n, cand_cap);
  for (int c = t; c < C; c += 256) {
    const float cv = cand_v[c];
    const int ci = cand_i[c];
    int rank = 0;
    for (int j = 0; j < C; ++j) rank += key_gt(cand_v[j], cand_i[j], cv, ci) ? 1 : 0;
    if (rank < k) {
      const int64_t o = (int64_t)row * out_row_stride + (int64_t)seg * k + rank;
      out_idx[o] = ci;
      out_val[o] = cv;
      if (feat_count) atomicAdd(feat_count + ci, 1.0f);
    }
  }
  // segments shorter than k (only possible for a ragged last segment): pad so the merge pass ignores them
  if (C < k) {
    for (int r = C + t; r < k; r += 256) {
      const int64_t o = (int64_t)row * out_row_stride + (int64_t)seg * k + r;
      out_idx[o] = 0x7fffffff;
      out_val[o] = -INFINITY;
    }
  }
}

// dense feature_acts [rows][F] = scatter(relu(val)) -- only when a caller wants the dense tensor (API / hooks)
__global__ void __launch_bounds__(256) k_scatter_acts(const int* __restrict__ idx, const float* __restrict__ val, float* __restrict__ dense,
                                                      int rows, int k, int F, int relu) {
  const int64_t n = (int64_t)rows * k;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / k);
    float v = val[e];
    if (relu) v = fmaxf(v, 0.f);
    dense[(int64_t)r * F + idx[e]] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// 3. sparse decode + loss + gradient wrt the selected pre-activations (one warp per token)
//    out_n  = sum_j relu(val_j) W_dec[idx_j] + b_dec           (sae.py:583-592)
//    out    = out_n * std + mu                                 (run_time_activation_ln_out, :89-90)
//    nf     = || x - mean_batch(x) ||_2                        (:145-147)
//    mse   += sum_c (out - x)^2 / nf ;  g = dL/d out_n = 2 (out - x) std / (nf Bt d)   (:148, mean over all elements)
//    dval_j = (val_j > 0) * <g, W_dec[idx_j]>                  (backward of decode + ReLU on the TopK support)
template <int CHUNKS>
__global__ void __launch_bounds__(256) k_sae_decode(const float* __restrict__ x, const float* __restrict__ xsum, const float* __restrict__ mu,
                                                    const float* __restrict__ sd, const int* __restrict__ idx, const float* __restrict__ val,
                                                    const float* __restrict__ W_dec, const float* __restrict__ b_dec,
                                                    float* __restrict__ sae_out, float* __restrict__ g_out, float* __restrict__ dval,
                                                    SaeScalars* __restrict__ sc, int rows, int d, int k, int norm_mode, int training,
                                                    float inv_rows) {
  pb_pdl();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const bool active = row < rows;
  const int nvec = d >> 2;
  float loss_part = 0.f, pos_part = 0.f;
  if (active) {
    const int* ir = idx + (int64_t)row * k;
    const float* vr = val + (int64_t)row * k;
    float acc[CHUNKS][4];
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) ld4(b_dec + 4 * c4, acc[i]);
      else acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    }
    // The k decoder rows of a token are independent gathers (L2 latency each): the support is read 32 entries at a time into lanes
    // and broadcast, and the row loop is unrolled so several rows' loads are in flight.  A selected value that is not positive
    // contributes a = 0 (its row is still read: rare, and it keeps the loop free of data-dependent branches).
    for (int j0 = 0; j0 < k; j0 += 32) {
      const int jn = min(32, k - j0);
      const int my_i = lane < jn ? ir[j0 + lane] : 0;
      const float my_a = lane < jn ? fmaxf(vr[j0 + lane], 0.f) : 0.f;
      pos_part += (float)__popc(__ballot_sync(0xffffffffu, my_a > 0.f));
#pragma unroll 4
      for (int j = 0; j < jn; ++j) {
        const float a = __shfl_sync(0xffffffffu, my_a, j);
        const float* wr = W_dec + (int64_t)__shfl_sync(0xffffffffu, my_i, j) * d;
#pragma unroll
        for (int i = 0; i < CHUNKS; ++i) {
          const int c4 = i * 32 + lane;
          if (c4 < nvec) {
            float w[4];
            ld4(wr + 4 * c4, w);
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[i][q] = fmaf(a, w[q], acc[i][q]);
          }
        }
      }
    }
    const float m = norm_mode ? mu[row] : 0.f;
    const float s = norm_mode ? sd[row] : 1.f;
    // pass A: out, centred norm
    float nsq = 0.f;
    float e[CHUNKS][4];
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        float xv[4], xs[4], o[4];
        ld4(x + (int64_t)row * d + 4 * c4, xv);
        ld4(xsum + 4 * c4, xs);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          o[q] = norm_mode == 1 ? acc[i][q] * s + m : (norm_mode == 2 ? acc[i][q] * s : acc[i][q]);
          const float xc = xv[q] - xs[q] * inv_rows;
          nsq += xc * xc;
          e[i][q] = o[q] - xv[q];
        }
        if (sae_out) st4(sae_out + (int64_t)row * d + 4 * c4, o);
      } else {
        e[i][0] = e[i][1] = e[i][2] = e[i][3] = 0.f;
      }
    }
    const float nf = sqrtf(warp_sum(nsq));
    float esq = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i)
#pragma unroll
      for (int q = 0; q < 4; ++q) esq += e[i][q] * e[i][q];
    loss_part = warp_sum(esq) / nf;
    if (training) {
      // g = dL/d out_n ;  L = sum (out - x)^2 / nf / (rows*d)
      const float gs = 2.f * s * inv_rows / ((float)d * nf);
#pragma unroll
      for (int i = 0; i < CHUNKS; ++i) {
        const int c4 = i * 32 + lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) e[i][q] *= gs;
        if (c4 < nvec) st4(g_out + (int64_t)row * d + 4 * c4, e[i]);
      }
      for (int j0 = 0; j0 < k; j0 += 32) {
        const int jn = min(32, k - j0);
        const int my_i = lane < jn ? ir[j0 + lane] : 0;
        const bool my_on = lane < jn && vr[j0 + lane] > 0.f;      // ReLU backward on the TopK support
        float my_dot = 0.f;
#pragma unroll 4
        for (int j = 0; j < jn; ++j) {
          const float* wr = W_dec + (int64_t)__shfl_sync(0xffffffffu, my_i, j) * d;
          float dot = 0.f;
#pragma unroll
          for (int i = 0; i < CHUNKS; ++i) {
            const int c4 = i * 32 + lane;
            if (c4 < nvec) {
              float w[4];
              ld4(wr + 4 * c4, w);
#pragma unroll
              for (int q = 0; q < 4; ++q) dot = fmaf(e[i][q], w[q], dot);
            }
          }
          dot = warp_sum(dot);
          if (lane == j) my_dot = dot;
        }
        if (lane < jn) dval[(int64_t)row * k + j0 + lane] = my_on ? my_dot : 0.f;
      }
    }
  }
  // one atomic pair per CTA
  __shared__ float red[2][8];
  const int w = threadIdx.x >> 5;
  if (lane == 0) { red[0][w] = active ? loss_part : 0.f; red[1][w] = active ? pos_part : 0.f; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += red[0][i]; b += red[1][i]; }
    atomicAdd(&sc->loss_sum, a);
    atomicAdd(&sc->pos_count, b);
  }
}

// ---------------------------------------------------------------------------------------------
// 4. CSC build: feat_count (float, from k_topk) -> offsets (exclusive scan) ; fill entries
// One CTA of 1024 threads; thread t owns the contiguous run [t * per, (t + 1) * per) of the counts (per = ceil(F / 1024) rounded up to
// a multiple of 4): 16-byte loads, a register prefix inside the run, ONE block scan of the 1024 run totals, 16-byte stores.
// (v1 walked its run with dependent scalar loads: 35 us; v2 block-scanned 1024-count chunks: 96 barriers, 15 us.)
template <int PER>
__global__ void __launch_bounds__(1024) k_scan_counts(const float* __restrict__ cnt, int* __restrict__ off, int* __restrict__ cursor, int F) {
  pb_pdl();
  __shared__ int wtot[32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int base = t * PER;
  int v[PER];
#pragma unroll
  for (int i = 0; i < PER; i += 4) {
    const int p = base + i;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p + 3 < F) c = *reinterpret_cast<const float4*>(cnt + p);
    else {
      if (p < F) c.x = cnt[p];
      if (p + 1 < F) c.y = cnt[p + 1];
      if (p + 2 < F) c.z = cnt[p + 2];
    }
    v[i] = (int)c.x; v[i + 1] = (int)c.y; v[i + 2] = (int)c.z; v[i + 3] = (int)c.w;
  }
  int run = 0;
#pragma unroll
  for (int i = 0; i < PER; ++i) { const int x = v[i]; v[i] = run; run += x; }       // exclusive prefix inside the run
  int x = run;                                                                         // inclusive scan of the run totals
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) wtot[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = wtot[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    wtot[lane] = w;
  }
  __syncthreads();
  const int excl = (warp ? wtot[warp - 1] : 0) + x - run;
#pragma unroll
  for (int i = 0; i < PER; i += 4) {
    const int p = base + i;
    const int4 o4 = make_int4(excl + v[i], excl + v[i + 1], excl + v[i + 2], excl + v[i + 3]);
    if (p + 3 < F) {
      *reinterpret_cast<int4*>(off + p) = o4;
      *reinterpret_cast<int4*>(cursor + p) = o4;
    } else {
      const int o[4] = {o4.x, o4.y, o4.z, o4.w};
      for (int j = 0; j < 4; ++j)
        if (p + j < F) { off[p + j] = o[j]; cursor[p + j] = o[j]; }
    }
  }
  if (t == 1023) off[F] = wtot[31];
}
__global__ void __launch_bounds__(256) k_csc_fill(const int* __restrict__ idx, int* __restrict__ cursor, int* __restrict__ entries, int64_t n) {
  pb_pdl();
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int f = idx[e];
    const int pos = atomicAdd(cursor + f, 1);
    entries[pos] = (int)e;
  }
}

// ---------------------------------------------------------------------------------------------
// 5. per-feature gradients (one warp per feature, persistent grid)
//    gW_dec[f]  = sum_{tokens b selecting f} relu(val) g[b]          (d loss / d W_dec row)
//    gW_encT[f] = sum dval * sae_in[b]                                (d loss / d W_enc column)
//    gb_enc[f]  = sum dval
//    gbdec2    += gb_enc[f] * W_encT[f]     (the -b_dec path through sae_in = xn - b_dec: d sae_in = W_enc dpre)
//    fired[f]   = number of tokens with relu(val) > 0 ; gnorm_sq += all squares
// Entry order inside a feature list comes from atomics, so the fp32 sums are order-nondeterministic at the
// 1e-7 level; the list is therefore sorted by token index first (lists are short: mean Bt*k/F).
constexpr int SAE_LONG_LIST = 32;    // lists longer than a warp are split into chunks across warps (k_sae_grads_long)
constexpr int SAE_LONG_CHUNK = 32;   // entries per work item of the long-list kernel
struct SaeWorkHeader { int n_chunks, n_long, next_f, pad; };   // followed in memory by work_feats[F] and work_chunks[2 * capacity]
constexpr int SAE_CLAIM = 4;         // features a warp claims per trip to the dynamic queue

template <int CHUNKS>
__global__ void __launch_bounds__(256) k_sae_grads(const int* __restrict__ off, int* __restrict__ entries, const float* __restrict__ val,
                                                   const float* __restrict__ dval, const float* __restrict__ g, const float* __restrict__ sae_in,
                                                   const float* __restrict__ W_encT, float* __restrict__ gW_dec, float* __restrict__ gW_encT,
                                                   float* __restrict__ gb_enc, float* __restrict__ gbdec2, float* __restrict__ fired,
                                                   SaeScalars* __restrict__ sc, int F, int d, int k, SaeWorkHeader* __restrict__ work,
                                                   int* __restrict__ work_feats, int* __restrict__ work_chunks) {
  pb_pdl();
  extern __shared__ __align__(16) float sm_bd[];  // [d] per-CTA partial of gbdec2
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  for (int c = threadIdx.x; c < d; c += blockDim.x) sm_bd[c] = 0.f;
  __syncthreads();
  float nsq = 0.f;
  float bd[CHUNKS][4];
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) bd[i][0] = bd[i][1] = bd[i][2] = bd[i][3] = 0.f;
  // dynamic queue: list lengths vary (mean Bt*k/F, long tail), and with a static feature -> warp map the CTA waited at its final
  // barrier for its slowest warp (9.9 barrier-stall cycles per issue, profiles/r02_sae_step_ncu_summary.txt)
  for (;;) {
    int fbase = 0;
    if (lane == 0) fbase = atomicAdd(&work->next_f, SAE_CLAIM);
    fbase = __shfl_sync(0xffffffffu, fbase, 0);
    if (fbase >= F) break;
   for (int f = fbase; f < min(F, fbase + SAE_CLAIM); ++f) {
    const int e0 = off[f], e1 = off[f + 1];
    const int len = e1 - e0;
    if (len > SAE_LONG_LIST) {
      // hot feature (selected by many tokens -- with real activations a handful of features fire on almost every token):
      // one warp walking thousands of entries would be the tail of the whole step (measured 2.4 ms).  Zero its rows, queue
      // its list in chunks of SAE_LONG_CHUNK entries for k_sae_grads_long, count its norm in k_sae_norm_long.
#pragma unroll
      for (int i = 0; i < CHUNKS; ++i) {
        const int c4 = i * 32 + lane;
        if (c4 < nvec) {
          const float z4[4] = {0.f, 0.f, 0.f, 0.f};
          st4(gW_dec + (int64_t)f * d + 4 * c4, z4);
          st4(gW_encT + (int64_t)f * d + 4 * c4, z4);
        }
      }
      const int nchunks = (len + SAE_LONG_CHUNK - 1) / SAE_LONG_CHUNK;
      int base = 0, lslot = 0;
      if (lane == 0) {
        gb_enc[f] = 0.f;
        fired[f] = 0.f;
        base = atomicAdd(&work->n_chunks, nchunks);
        lslot = atomicAdd(&work->n_long, 1);
        work_feats[lslot] = f;
      }
      base = __shfl_sync(0xffffffffu, base, 0);
      for (int c = lane; c < nchunks; c += 32) {
        work_chunks[2 * (base + c)] = f;
        work_chunks[2 * (base + c) + 1] = e0 + c * SAE_LONG_CHUNK;
      }
      continue;
    }
    // The whole list (<= 32 entries) lives in the warp: lane i loads entry i, its sorted slot is the number of smaller entries
    // (rank by counting: entries are distinct; token order makes the fp32 sums deterministic), then lane i loads ITS entry's
    // activation / d(pre-activation) / token row index.  The accumulation loop below only shuffles those out of registers, so the
    // row gathers of consecutive entries are independent loads in flight together.  (Before: entry -> val / dval -> rows was a chain
    // of three dependent L2 round trips PER PAIR of entries, ~8 us per feature: profiles/r02_sae_notes.md.)
    int my_b = 0;
    float my_a = 0.f, my_dp = 0.f;
    {
      const int mine = lane < len ? entries[e0 + lane] : 0x7fffffff;
      int rank = 0;
#pragma unroll
      for (int j = 0; j < 32; ++j) rank += __shfl_sync(0xffffffffu, mine, j) < mine ? 1 : 0;
      // lane `rank` must hold `mine`: invert the permutation with one shuffle per lane (lane j looks for the lane whose rank is j)
      int src = 0;
#pragma unroll
      for (int j = 0; j < 32; ++j) src = (__shfl_sync(0xffffffffu, rank, j) == lane && j < len) ? j : src;
      const int sorted = __shfl_sync(0xffffffffu, mine, src);
      if (lane < len) {
        my_b = sorted / k;
        my_a = fmaxf(val[sorted], 0.f);
        my_dp = dval[sorted];
      }
    }
    float ad[CHUNKS][4], ae[CHUNKS][4];
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) ad[i][0] = ad[i][1] = ad[i][2] = ad[i][3] = ae[i][0] = ae[i][1] = ae[i][2] = ae[i][3] = 0.f;
    float gbe = 0.f;
    const float npos = (float)__popc(__ballot_sync(0xffffffffu, my_a > 0.f));
#pragma unroll 2
    for (int j = 0; j < len; ++j) {
      const float a = __shfl_sync(0xffffffffu, my_a, j), dp = __shfl_sync(0xffffffffu, my_dp, j);
      const int b = __shfl_sync(0xffffffffu, my_b, j);
      gbe += dp;
      const float* gr = g + (int64_t)b * d;
      const float* sr = sae_in + (int64_t)b * d;
#pragma unroll
      for (int i = 0; i < CHUNKS; ++i) {
        const int c4 = i * 32 + lane;
        if (c4 < nvec) {
          float gv[4], sv[4];
          ld4(gr + 4 * c4, gv);
          ld4(sr + 4 * c4, sv);
#pragma unroll
          for (int q = 0; q < 4; ++q) { ad[i][q] = fmaf(a, gv[q], ad[i][q]); ae[i][q] = fmaf(dp, sv[q], ae[i][q]); }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        st4(gW_dec + (int64_t)f * d + 4 * c4, ad[i]);
        st4(gW_encT + (int64_t)f * d + 4 * c4, ae[i]);
#pragma unroll
        for (int q = 0; q < 4; ++q) nsq += ad[i][q] * ad[i][q] + ae[i][q] * ae[i][q];
        if (gbe != 0.f) {
          float w[4];
          ld4(W_encT + (int64_t)f * d + 4 * c4, w);
#pragma unroll
          for (int q = 0; q < 4; ++q) bd[i][q] = fmaf(gbe, w[q], bd[i][q]);
        }
      }
    }
    if (lane == 0) {
      gb_enc[f] = gbe;
      fired[f] = npos;
      nsq += gbe * gbe;
    }
   }
  }
  // the -b_dec path, sum_f gb_enc[f] W_encT[f]: per-lane register partials over this warp's features, one shared-memory
  // reduction per CTA (the per-feature shared atomics of the first version cost 24 x 64 cycles of the LSU per feature -- the
  // whole kernel ran at the ATOMS rate, profiles/r02_sae_notes.md)
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) {
    const int c4 = i * 32 + lane;
    if (c4 < nvec) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (bd[i][q] != 0.f) atomicAdd(&sm_bd[4 * c4 + q], bd[i][q]);
    }
  }
  nsq = warp_sum(nsq);
  __shared__ float red[8];
  if (lane == 0) red[warp] = nsq;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int i = 0; i < nw; ++i) a += red[i];
    atomicAdd(&sc->gnorm_sq, a);
  }
  for (int c = threadIdx.x; c < d; c += blockDim.x)
    if (sm_bd[c] != 0.f) atomicAdd(gbdec2 + c, sm_bd[c]);
}

// 5b. hot features: one warp per chunk of SAE_LONG_CHUNK list entries, partial rows added with 16-byte red.global.add
template <int CHUNKS>
__global__ void __launch_bounds__(256) k_sae_grads_long(const int* __restrict__ off, const int* __restrict__ entries, const float* __restrict__ val,
                                                        const float* __restrict__ dval, const float* __restrict__ g,
                                                        const float* __restrict__ sae_in, const float* __restrict__ W_encT,
                                                        float* __restrict__ gW_dec, float* __restrict__ gW_encT, float* __restrict__ gb_enc,
                                                        float* __restrict__ gbdec2, float* __restrict__ fired, int d, int k,
                                                        const SaeWorkHeader* __restrict__ work, const int* __restrict__ work_chunks) {
  pb_pdl();
  extern __shared__ __align__(16) float sm_bd[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  const int n_items = work->n_chunks;
  if (n_items == 0) return;
  for (int c = threadIdx.x; c < d; c += blockDim.x) sm_bd[c] = 0.f;
  __syncthreads();
  float bd[CHUNKS][4];
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) bd[i][0] = bd[i][1] = bd[i][2] = bd[i][3] = 0.f;
  for (int item = blockIdx.x * nw + warp; item < n_items; item += gridDim.x * nw) {
    const int f = work_chunks[2 * item], p0 = work_chunks[2 * item + 1];
    const int p1 = min(off[f + 1], p0 + SAE_LONG_CHUNK);
    float ad[CHUNKS][4], ae[CHUNKS][4];
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) ad[i][0] = ad[i][1] = ad[i][2] = ad[i][3] = ae[i][0] = ae[i][1] = ae[i][2] = ae[i][3] = 0.f;
    const int n = p1 - p0;                                   // <= SAE_LONG_CHUNK = 32: one entry per lane
    int my_b = 0;
    float my_a = 0.f, my_dp = 0.f;
    if (lane < n) {
      const int e = entries[p0 + lane];
      my_b = e / k;
      my_a = fmaxf(val[e], 0.f);
      my_dp = dval[e];
    }
    float gbe = 0.f;
    const float npos = (float)__popc(__ballot_sync(0xffffffffu, my_a > 0.f));
#pragma unroll 2
    for (int j = 0; j < n; ++j) {
      const float a = __shfl_sync(0xffffffffu, my_a, j), dp = __shfl_sync(0xffffffffu, my_dp, j);
      const int b = __shfl_sync(0xffffffffu, my_b, j);
      gbe += dp;
      const float* gr = g + (int64_t)b * d;
      const float* sr = sae_in + (int64_t)b * d;
#pragma unroll
      for (int i = 0; i < CHUNKS; ++i) {
        const int c4 = i * 32 + lane;
        if (c4 < nvec) {
          float gv[4], sv[4];
          ld4(gr + 4 * c4, gv);
          ld4(sr + 4 * c4, sv);
#pragma unroll
          for (int q = 0; q < 4; ++q) { ad[i][q] = fmaf(a, gv[q], ad[i][q]); ae[i][q] = fmaf(dp, sv[q], ae[i][q]); }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        atomicAdd(reinterpret_cast<float4*>(gW_dec + (int64_t)f * d + 4 * c4), make_float4(ad[i][0], ad[i][1], ad[i][2], ad[i][3]));
        atomicAdd(reinterpret_cast<float4*>(gW_encT + (int64_t)f * d + 4 * c4), make_float4(ae[i][0], ae[i][1], ae[i][2], ae[i][3]));
        if (gbe != 0.f) {
          float w[4];
          ld4(W_encT + (int64_t)f * d + 4 * c4, w);
#pragma unroll
          for (int q = 0; q < 4; ++q) bd[i][q] = fmaf(gbe, w[q], bd[i][q]);
        }
      }
    }
    if (lane == 0) {
      atomicAdd(gb_enc + f, gbe);
      atomicAdd(fired + f, npos);
    }
  }
#pragma unroll
  for (int i = 0; i < CHUNKS; ++i) {
    const int c4 = i * 32 + lane;
    if (c4 < nvec) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (bd[i][q] != 0.f) atomicAdd(&sm_bd[4 * c4 + q], bd[i][q]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < d; c += blockDim.x)
    if (sm_bd[c] != 0.f) atomicAdd(gbdec2 + c, sm_bd[c]);
}

// 5c. squared norm of the completed hot-feature rows (not additive over chunks, so it waits for 5b)
__global__ void __launch_bounds__(256) k_sae_norm_long(const float* __restrict__ gW_dec, const float* __restrict__ gW_encT,
                                                       const float* __restrict__ gb_enc, SaeScalars* __restrict__ sc, int d,
                                                       const SaeWorkHeader* __restrict__ work, const int* __restrict__ work_feats) {
  pb_pdl();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int n = work->n_long;
  float nsq = 0.f;
  for (int li = blockIdx.x * nw + warp; li < n; li += gridDim.x * nw) {
    const int f = work_feats[li];
    for (int c = lane; c < d; c += 32) {
      const float a = gW_dec[(int64_t)f * d + c], b = gW_encT[(int64_t)f * d + c];
      nsq += a * a + b * b;
    }
    if (lane == 0) nsq += gb_enc[f] * gb_enc[f];
  }
  nsq = warp_sum(nsq);
  if (lane == 0 && nsq != 0.f) atomicAdd(&sc->gnorm_sq, nsq);
}

__global__ void k_sae_gbdec(const float* __restrict__ gcol, const float* __restrict__ gbdec2, float* __restrict__ gb_dec, int d) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < d) gb_dec[c] = gcol[c] - gbdec2[c];
}

// 6. finalize: gb_dec = colsum(g) - gbdec2 ; total norm ; clip coefficient (train_sae.py:394-397)
__global__ void __launch_bounds__(256) k_sae_finalize(const float* __restrict__ gcol, const float* __restrict__ gbdec2, float* __restrict__ gb_dec,
                                                      SaeScalars* __restrict__ sc, int d, float max_norm, float inv_elems, float inv_rows) {
  pb_pdl();
  __shared__ float red[8];
  float s = 0.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float v = gcol[c] - gbdec2[c];
    gb_dec[c] = v;
    s += v * v;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = sc->gnorm_sq;
    for (int i = 0; i < 8; ++i) t += red[i];
    const float norm = sqrtf(t);
    sc->gnorm_sq = t;
    sc->grad_norm = norm;
    sc->clip_coef = max_norm > 0.f ? fminf(1.f, max_norm / (norm + 1e-6f)) : 1.f;
    sc->mse = sc->loss_sum * inv_elems;
    sc->l0 = sc->pos_count * inv_rows;
  }
}

// ---------------------------------------------------------------------------------------------
// 7. optimizer: clip -> remove decoder-parallel gradient -> Adam -> unit-norm decoder rows (+ counters)
//    (train_sae.py:394-401, sae.py:275-297, torch.optim.Adam defaults betas (0.9, 0.999), eps 1e-8, no weight decay)
//    The row renorm is the *next* step's set_decoder_norm_to_unit_norm() (train_sae.py:307) applied early; forward
//    and backward of every later step see identical numbers.
struct AdamHyper { float lr, beta1, beta2, eps, bc1, bc2_sqrt; };  // bc1 = 1-beta1^t, bc2_sqrt = sqrt(1-beta2^t)

// torch.optim.Adam (single tensor, no amsgrad / weight decay): m, v exactly as torch computes them; the parameter update
// -(lr / bc1) m / (sqrt(v) / bc2_sqrt + eps) uses MUFU sqrt / reciprocal approximations (relative error ~1e-7 of an update that is
// itself ~lr relative to the parameter: 1e-10 on the parameter, against a 1e-4 parity bar).  The IEEE sqrt + two divisions of the
// first version were ~30 of the ~45 instructions per element and made the optimizer issue-bound (profiles/r02_sae_notes.md).
__device__ __forceinline__ float adam_update(float p, float gr, float& m, float& v, const AdamHyper& h) {
  m = h.beta1 * m + (1.f - h.beta1) * gr;
  v = h.beta2 * v + (1.f - h.beta2) * gr * gr;
  float sq, rc;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
  const float denom = fmaf(sq, __frcp_rn(h.bc2_sqrt), h.eps);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(denom));
  return fmaf(-(h.lr * __frcp_rn(h.bc1)) * m, rc, p);
}

template <int CHUNKS>
__global__ void __launch_bounds__(256) k_sae_adam_rows(float* __restrict__ W_dec, float* __restrict__ W_encT, float* __restrict__ W_encT_lo,
                                                       float* __restrict__ b_enc, const float* __restrict__ gW_dec,
                                                       const float* __restrict__ gW_encT, const float* __restrict__ gb_enc,
                                                       float* __restrict__ m_dec, float* __restrict__ v_dec, float* __restrict__ m_enc,
                                                       float* __restrict__ v_enc, float* __restrict__ m_be, float* __restrict__ v_be,
                                                       const float* __restrict__ fired, float* __restrict__ since_fired,
                                                       float* __restrict__ act_freq, const SaeScalars* __restrict__ sc, AdamHyper h,
                                                       int F, int d, int renorm, float* __restrict__ enc_norm_max,
                                                       uint16_t* __restrict__ W_encT_h) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  const float clip = sc->clip_coef;
  float enc_best = 0.f, enc_best_lo = 0.f;
  for (int f = blockIdx.x * nw + warp; f < F; f += gridDim.x * nw) {
    const int64_t base = (int64_t)f * d;
    // ---- decoder row
    float w[CHUNKS][4], gq[CHUNKS][4];
    float par = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        ld4(W_dec + base + 4 * c4, w[i]);
        ld4(gW_dec + base + 4 * c4, gq[i]);
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
          const float gr = gq[i][q] - par * w[i][q];
          w[i][q] = adam_update(w[i][q], gr, mm[q], vv[q], h);
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
        if (renorm) {
#pragma unroll
          for (int q = 0; q < 4; ++q) w[i][q] = w[i][q] * inv_nrm;
        }
        st4(W_dec + base + 4 * c4, w[i]);
      }
    }
    // ---- encoder row (feature-major)
    float esq = 0.f, elo = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        float p[4], gr[4], mm[4], vv[4], lo[4];
        ld4(W_encT + base + 4 * c4, p);
        ld4(gW_encT + base + 4 * c4, gr);
        ld4(m_enc + base + 4 * c4, mm);
        ld4(v_enc + base + 4 * c4, vv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          p[q] = adam_update(p[q], gr[q] * clip, mm[q], vv[q], h);
          lo[q] = tf32_lo(p[q]);
          esq = fmaf(p[q], p[q], esq);
        }
        elo += st4_f16_cand(W_encT_h ? W_encT_h + (int64_t)f * f16_ld(d) + 4 * c4 : nullptr, p);
        st4(W_encT + base + 4 * c4, p);
        st4(m_enc + base + 4 * c4, mm);
        st4(v_enc + base + 4 * c4, vv);
        if (W_encT_lo) st4(W_encT_lo + base + 4 * c4, lo);
      }
    }
    if (enc_norm_max) { enc_best = fmaxf(enc_best, warp_sum(esq)); enc_best_lo = fmaxf(enc_best_lo, warp_sum(elo)); }
    if (lane == 0) {
      float mm = m_be[f], vv = v_be[f];
      b_enc[f] = adam_update(b_enc[f], gb_enc[f] * clip, mm, vv, h);
      m_be[f] = mm;
      v_be[f] = vv;
      // dead-feature bookkeeping (train_sae.py:356-361)
      if (since_fired) since_fired[f] = fired[f] > 0.f ? 0.f : since_fired[f] + 1.f;
      if (act_freq) act_freq[f] += fired[f];
    }
  }
  // largest encoder-column norm after the update (error bound of the fused encoder's fp16 pass); norms are >= 0 so the
  // bit pattern orders like the value
  if (enc_norm_max && lane == 0 && enc_best > 0.f) {
    atomicMax(reinterpret_cast<unsigned int*>(enc_norm_max), __float_as_uint(sqrtf(enc_best)));
    atomicMax(reinterpret_cast<unsigned int*>(enc_norm_max) + 1, __float_as_uint(sqrtf(enc_best_lo)));
  }
}

// ---- 7b. the same update as a bulk-copy pipeline ---------------------------------------------------------------------
// k_sae_adam_rows keeps a feature's rows in registers: its loads are issued in four dependent waves per feature (w,g -> m,v ->
// encoder row), 16 warps per SM, and it reaches 0.63 of the HBM copy bandwidth.  Here one producer lane streams every feature's
// EIGHT rows (W_dec, gW_dec, m_dec, v_dec, W_encT, gW_encT, m_enc, v_enc: 8 x d x 4 bytes) into a shared-memory ring with
// cp.async.bulk (completion on an mbarrier), one consumer warp per ring slot updates its feature in place, and the six result rows go
// back with cp.async.bulk stores.  The bytes in flight per SM are set by the ring depth (S x 24 KB at d = 768), not by registers.
// One consumer warp per ring slot (block = 32 x (1 + S) threads): iteration i and iteration i + S then belong to the SAME warp, so a
// warp never waits for phase p + 1 of a slot's "full" barrier before it has itself consumed phase p.  (With more warps than slots a
// warp could start waiting a whole phase early; mbarrier parity is one bit, the early waiter saw "already complete" and read a slot
// another warp was still updating -- the first 12-warp version deadlocked in run r2d.)
constexpr int AB_MAX_STAGES = 12;
constexpr int AB_THREADS = 32 * (1 + AB_MAX_STAGES);

__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}

template <int CHUNKS>
__global__ void __launch_bounds__(AB_THREADS, 1)
k_sae_adam_bulk(float* __restrict__ W_dec, float* __restrict__ W_encT, float* __restrict__ b_enc, const float* __restrict__ gW_dec,
                const float* __restrict__ gW_encT, const float* __restrict__ gb_enc, float* __restrict__ m_dec, float* __restrict__ v_dec,
                float* __restrict__ m_enc, float* __restrict__ v_enc, float* __restrict__ m_be, float* __restrict__ v_be,
                const float* __restrict__ fired, float* __restrict__ since_fired, float* __restrict__ act_freq,
                const SaeScalars* __restrict__ sc, AdamHyper h, int F, int d, int renorm, float* __restrict__ enc_norm_max, int S,
                float* __restrict__ b_dec, const float* __restrict__ gb_dec, float* __restrict__ m_bd, float* __restrict__ v_bd,
                uint16_t* __restrict__ W_encT_h) {
  pb_pdl_trigger();
  extern __shared__ __align__(128) unsigned char ab_smem[];
  const uint32_t s0 = smem_u32(ab_smem);
  const uint32_t row_bytes = (uint32_t)d * 4u, stage_bytes = 8u * row_bytes;
  auto full_bar = [&](int s) { return s0 + 8u * s; };
  auto empty_bar = [&](int s) { return s0 + 8u * (S + s); };
  const uint32_t data0 = s0 + 256u;                       // barriers live in the first 256 bytes (S <= 16)
  float* data_generic = reinterpret_cast<float*>(ab_smem + 256);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_mine = F > (int)blockIdx.x ? (F - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pb_pdl_wait();                                   // gradients / clip coefficient of the preceding kernels are complete
  if (warp == 0) {
    if (blockIdx.x == 0 && b_dec) {                 // the decoder bias (d values): this warp, before it turns producer
      const float clip0 = sc->clip_coef;
      for (int c = lane; c < d; c += 32) {
        float mm = m_bd[c], vv = v_bd[c];
        b_dec[c] = adam_update(b_dec[c], gb_dec[c] * clip0, mm, vv, h);
        m_bd[c] = mm;
        v_bd[c] = vv;
      }
    }
    if (lane == 0) {
      for (int i = 0; i < n_mine; ++i) {
        const int s = i % S;
        const uint32_t ph = (uint32_t)(i / S) & 1u;
        const int64_t base = (int64_t)(blockIdx.x + (int64_t)i * gridDim.x) * d;
        mbar_wait(empty_bar(s), ph ^ 1u);
        mbar_expect_tx(full_bar(s), stage_bytes);
        const uint32_t dst = data0 + (uint32_t)s * stage_bytes;
        bulk_load(dst + 0 * row_bytes, W_dec + base, row_bytes, full_bar(s));
        bulk_load(dst + 1 * row_bytes, gW_dec + base, row_bytes, full_bar(s));
        bulk_load(dst + 2 * row_bytes, m_dec + base, row_bytes, full_bar(s));
        bulk_load(dst + 3 * row_bytes, v_dec + base, row_bytes, full_bar(s));
        bulk_load(dst + 4 * row_bytes, W_encT + base, row_bytes, full_bar(s));
        bulk_load(dst + 5 * row_bytes, gW_encT + base, row_bytes, full_bar(s));
        bulk_load(dst + 6 * row_bytes, m_enc + base, row_bytes, full_bar(s));
        bulk_load(dst + 7 * row_bytes, v_enc + base, row_bytes, full_bar(s));
      }
    }
    return;
  }
  const int nvec = d >> 2;
  const float clip = sc->clip_coef;
  float enc_best = 0.f, enc_best_lo = 0.f;
  for (int i = warp - 1; i < n_mine; i += S) {
    const int s = i % S;
    const uint32_t ph = (uint32_t)(i / S) & 1u;
    const int f = blockIdx.x + i * gridDim.x;
    const int64_t base = (int64_t)f * d;
    // per-feature scalars: in flight while the rows arrive
    float be = 0.f, gbe = 0.f, mbe = 0.f, vbe = 0.f, fr = 0.f, sf = 0.f, af = 0.f;
    if (lane == 0) {
      be = b_enc[f]; gbe = gb_enc[f]; mbe = m_be[f]; vbe = v_be[f]; fr = fired[f];
      if (since_fired) sf = since_fired[f];
      if (act_freq) af = act_freq[f];
    }
    mbar_wait(full_bar(s), ph);
    float* st = data_generic + (size_t)s * 8 * d;
    float *wd = st, *gd = st + d, *md = st + 2 * d, *vd = st + 3 * d, *we = st + 4 * d, *ge = st + 5 * d, *me = st + 6 * d, *ve = st + 7 * d;
    // ---- decoder row: clip, remove the component parallel to the (unit-norm) row, Adam, renormalise
    float w[CHUNKS][4], gq[CHUNKS][4];
    float par = 0.f;
#pragma unroll
    for (int c = 0; c < CHUNKS; ++c) {
      const int c4 = c * 32 + lane;
      if (c4 < nvec) {
        ld4(wd + 4 * c4, w[c]);
        ld4(gd + 4 * c4, gq[c]);
#pragma unroll
        for (int q = 0; q < 4; ++q) { gq[c][q] *= clip; par = fmaf(gq[c][q], w[c][q], par); }
      } else {
        w[c][0] = w[c][1] = w[c][2] = w[c][3] = gq[c][0] = gq[c][1] = gq[c][2] = gq[c][3] = 0.f;
      }
    }
    par = warp_sum(par);
    float nsq = 0.f;
#pragma unroll
    for (int c = 0; c < CHUNKS; ++c) {
      const int c4 = c * 32 + lane;
      if (c4 < nvec) {
        float mm[4], vv[4];
        ld4(md + 4 * c4, mm);
        ld4(vd + 4 * c4, vv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float gr = gq[c][q] - par * w[c][q];
          w[c][q] = adam_update(w[c][q], gr, mm[q], vv[q], h);
          nsq += w[c][q] * w[c][q];
        }
        st4(md + 4 * c4, mm);
        st4(vd + 4 * c4, vv);
      }
    }
    const float inv_nrm = 1.f / sqrtf(warp_sum(nsq));
#pragma unroll
    for (int c = 0; c < CHUNKS; ++c) {
      const int c4 = c * 32 + lane;
      if (c4 < nvec) {
        if (renorm) {
#pragma unroll
          for (int q = 0; q < 4; ++q) w[c][q] = w[c][q] * inv_nrm;
        }
        st4(wd + 4 * c4, w[c]);
      }
    }
    // ---- encoder row
    float esq = 0.f, elo = 0.f;
#pragma unroll
    for (int c = 0; c < CHUNKS; ++c) {
      const int c4 = c * 32 + lane;
      if (c4 < nvec) {
        float p[4], gr[4], mm[4], vv[4];
        ld4(we + 4 * c4, p);
        ld4(ge + 4 * c4, gr);
        ld4(me + 4 * c4, mm);
        ld4(ve + 4 * c4, vv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          p[q] = adam_update(p[q], gr[q] * clip, mm[q], vv[q], h);
          esq = fmaf(p[q], p[q], esq);
        }
        elo += st4_f16_cand(W_encT_h ? W_encT_h + (int64_t)f * f16_ld(d) + 4 * c4 : nullptr, p);   // fp16 shadow: from registers
        st4(we + 4 * c4, p);
        st4(me + 4 * c4, mm);
        st4(ve + 4 * c4, vv);
      }
    }
    enc_best = fmaxf(enc_best, warp_sum(esq));
    enc_best_lo = fmaxf(enc_best_lo, warp_sum(elo));
    __syncwarp();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes above -> visible to the bulk-copy engine
    __syncwarp();
    if (lane == 0) {
      const uint32_t src = data0 + (uint32_t)s * stage_bytes;
      bulk_store(W_dec + base, src + 0 * row_bytes, row_bytes);
      bulk_store(m_dec + base, src + 2 * row_bytes, row_bytes);
      bulk_store(v_dec + base, src + 3 * row_bytes, row_bytes);
      bulk_store(W_encT + base, src + 4 * row_bytes, row_bytes);
      bulk_store(m_enc + base, src + 6 * row_bytes, row_bytes);
      bulk_store(v_enc + base, src + 7 * row_bytes, row_bytes);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      // bias + dead-feature bookkeeping (train_sae.py:356-361) while the stores drain
      b_enc[f] = adam_update(be, gbe * clip, mbe, vbe, h);
      m_be[f] = mbe;
      v_be[f] = vbe;
      if (since_fired) since_fired[f] = fr > 0.f ? 0.f : sf + 1.f;
      if (act_freq) act_freq[f] = af + fr;
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the ring slot has been read: hand it back
      mbar_arrive(empty_bar(s));
    }
  }
  if (enc_norm_max && lane == 0 && enc_best > 0.f) {
    atomicMax(reinterpret_cast<unsigned int*>(enc_norm_max), __float_as_uint(sqrtf(enc_best)));
    atomicMax(reinterpret_cast<unsigned int*>(enc_norm_max) + 1, __float_as_uint(sqrtf(enc_best_lo)));
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__global__ void __launch_bounds__(256) k_sae_adam_vec(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                      float* __restrict__ v, const SaeScalars* __restrict__ sc, AdamHyper h, int n) {
  const float clip = sc->clip_coef;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float mm = m[i], vv = v[i];
    p[i] = adam_update(p[i], g[i] * clip, mm, vv, h);
    m[i] = mm;
    v[i] = vv;
  }
}

// row norms -> unit (set_decoder_norm_to_unit_norm, sae.py:275-277) as a standalone op
template <int CHUNKS>
__global__ void __launch_bounds__(256) k_unit_rows(float* __restrict__ W, float* __restrict__ W_lo, int F, int d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nvec = d >> 2;
  for (int f = blockIdx.x * nw + warp; f < F; f += gridDim.x * nw) {
    float w[CHUNKS][4];
    float nsq = 0.f;
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        ld4(W + (int64_t)f * d + 4 * c4, w[i]);
#pragma unroll
        for (int q = 0; q < 4; ++q) nsq += w[i][q] * w[i][q];
      }
    }
    const float nrm = sqrtf(warp_sum(nsq));
#pragma unroll
    for (int i = 0; i < CHUNKS; ++i) {
      const int c4 = i * 32 + lane;
      if (c4 < nvec) {
        float lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { w[i][q] = w[i][q] / nrm; lo[q] = tf32_lo(w[i][q]); }
        st4(W + (int64_t)f * d + 4 * c4, w[i]);
        if (W_lo) st4(W_lo + (int64_t)f * d + 4 * c4, lo);
      }
    }
  }
}

// =============================================================================================
// host side
// =============================================================================================
static int chunks_for(int d) {
  if (d % 4 != 0) return -1;
  const int nvec = d / 4;
  if (nvec <= 32) return 1;
  if (nvec <= 64) return 2;
  if (nvec <= 128) return 4;
  if (nvec <= 192) return 6;
  if (nvec <= 256) return 8;
  if (nvec <= 384) return 12;
  return -1;
}
#define PB_DISPATCH_CHUNKS(CH, CALL)                                                   \
  switch (CH) {                                                                        \
    case 1: { constexpr int C_ = 1; CALL; } break;                                     \
    case 2: { constexpr int C_ = 2; CALL; } break;                                     \
    case 4: { constexpr int C_ = 4; CALL; } break;                                     \
    case 6: { constexpr int C_ = 6; CALL; } break;                                     \
    case 8: { constexpr int C_ = 8; CALL; } break;                                     \
    case 12: { constexpr int C_ = 12; CALL; } break;                                   \
    default: pb_set_error("sae: d_in=%d unsupported (needs d %% 4 == 0 and d <= 1536)", d); return PB_EUNSUPPORTED; \
  }

static int persistent_grid(int warps_per_cta, int items) {
  int ctas = pb_sm_count() * 4;
  const int need = (items + warps_per_cta - 1) / warps_per_cta;
  if (ctas > need) ctas = need;
  return ctas < 1 ? 1 : ctas;
}

extern "C" int pb_sae_prep(const float* x, const float* b_dec, float* sae_in, float* sae_in_lo, void* sae_in_h, float* mu, float* sd, float* xsum,
                           int32_t rows, int32_t d, int32_t norm_mode, pb_stream_t stream) {
  PB_CHECK_ARG(x && b_dec && sae_in && rows >= 0 && d > 0, "pb_sae_prep: bad arguments");
  PB_CHECK_ARG(norm_mode == 0 || (mu && sd), "pb_sae_prep: mu/std buffers required when normalising");
  if (rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int ch = chunks_for(d);
  PB_DISPATCH_CHUNKS(ch, PB_LAUNCH_PDL(k_sae_prep<C_>, (rows + 7) / 8, 256, 0, st, x, b_dec, sae_in, sae_in_lo, reinterpret_cast<uint16_t*>(sae_in_h), mu, sd, rows,
                                          d, norm_mode, 1e-5f));
  if (xsum) {
    PB_CUDA(cudaMemsetAsync(xsum, 0, sizeof(float) * d, st));
    const int rpc = 8;
    k_colsum<<<(rows + rpc - 1) / rpc, 256, 0, st>>>(x, xsum, rows, d, rpc);     // after a memset: a plain launch
    PB_LAUNCH_CHECK();
  }
  return PB_OK;
}

static int launch_topk(const float* vals, const int* map, int64_t row_stride, int F, int seg_len, int nseg, int k, int* oi, float* ov,
                       int64_t out_stride, float* feat_count, int rows, cudaStream_t st) {
  const int ipt_needed = (seg_len + 255) / 256;
  const int ipt = ipt_needed <= 8 ? 8 : ipt_needed <= 24 ? 24 : ipt_needed <= 48 ? 48 : 96;
  int cap = ipt * k;
  if (cap > seg_len) cap = seg_len;
  if (cap < k) cap = k;
  const size_t smem = 256 * 8 + (size_t)cap * 8;
  if (smem > 200 * 1024) { pb_set_error("pb_sae_topk: k=%d too large for the candidate buffer", k); return PB_EUNSUPPORTED; }
  dim3 grid(rows, nseg);
#define PB_TOPK(IPT)                                                                                                      \
  do {                                                                                                                    \
    auto kern = k_topk<IPT>;                                                                                              \
    if (smem > 48 * 1024) PB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
    kern<<<grid, 256, smem, st>>>(vals, map, row_stride, F, seg_len, k, oi, ov, out_stride, feat_count, cap);             \
  } while (0)
  if (ipt == 8) PB_TOPK(8);
  else if (ipt == 24) PB_TOPK(24);
  else if (ipt == 48) PB_TOPK(48);
  else PB_TOPK(96);
#undef PB_TOPK
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// hidden_pre [rows][F] -> idx/val [rows][k]; feat_count[F] (float) += selections; scratch: 2 * rows * nseg * k * 4 bytes
extern "C" int pb_sae_topk(const float* hidden_pre, int32_t rows, int32_t F, int32_t k, int32_t* idx, float* val, float* feat_count,
                           void* scratch, int64_t scratch_bytes, pb_stream_t stream) {
  PB_CHECK_ARG(hidden_pre && idx && val && rows >= 0 && F > 0 && k > 0 && k <= F, "pb_sae_topk: bad arguments");
  PB_CHECK_ARG(k <= 256, "pb_sae_topk: k=%d > 256 unsupported", k);
  if (rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int SEG = 256 * 96;
  if (F <= SEG) return launch_topk(hidden_pre, nullptr, F, F, F, 1, k, idx, val, k, feat_count, rows, st);
  const int nseg = (F + SEG - 1) / SEG;
  const int seg_len = ((F + nseg - 1) / nseg + 255) / 256 * 256;
  const int64_t need = (int64_t)rows * nseg * k * 8;
  PB_CHECK_ARG(scratch && scratch_bytes >= need, "pb_sae_topk: scratch too small (%lld < %lld)", (long long)scratch_bytes, (long long)need);
  int* ci = (int*)scratch;
  float* cv = (float*)(ci + (int64_t)rows * nseg * k);
  PB_TRY(launch_topk(hidden_pre, nullptr, F, F, seg_len, nseg, k, ci, cv, (int64_t)nseg * k, nullptr, rows, st));
  return launch_topk(cv, ci, (int64_t)nseg * k, nseg * k, nseg * k, 1, k, idx, val, k, feat_count, rows, st);
}

extern "C" int pb_sae_scatter_acts(const int32_t* idx, const float* val, float* dense, int32_t rows, int32_t k, int32_t F, int32_t relu,
                                   pb_stream_t stream) {
  PB_CHECK_ARG(idx && val && dense && rows >= 0, "pb_sae_scatter_acts: bad arguments");
  if (rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  PB_CUDA(cudaMemsetAsync(dense, 0, sizeof(float) * (size_t)rows * F, st));
  k_scatter_acts<<<pb_sm_count() * 4, 256, 0, st>>>(idx, val, dense, rows, k, F, relu);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// PbSaeStep: every pointer of one training / inference step (device memory owned by the caller)
__global__ void k_sae_fwd_scalars(SaeScalars* sc, float inv_elems, float inv_rows) {
  sc->mse = sc->loss_sum * inv_elems;
  sc->l0 = sc->pos_count * inv_rows;
}

// every accumulator a training step starts from zero, in one launch (they were six memsets / fills on the stream)
__global__ void __launch_bounds__(256) k_sae_step_reset(float* __restrict__ feat_count, int F, float* __restrict__ scalars, float* __restrict__ gcol,
                                                        float* __restrict__ gbdec2, int d, int* __restrict__ work_hdr, int* __restrict__ fb_count) {
  pb_pdl();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (int f = i; f < F; f += gridDim.x * blockDim.x) feat_count[f] = 0.f;
  if (i < d) { gcol[i] = 0.f; gbdec2[i] = 0.f; }
  if (i < 8) scalars[i] = 0.f;
  if (i < 4 && work_hdr) work_hdr[i] = 0;
  if (i < 2 && fb_count) fb_count[i] = 0;
}

extern "C" int pb_sae_step_reset(const PbSaeStep* s, int32_t* fb_count, pb_stream_t stream) {
  PB_CHECK_ARG(s && s->feat_count && s->scalars && s->gcol && s->gbdec2, "pb_sae_step_reset: missing pointers");
  PB_CHECK_ARG(!s->work || s->work_bytes >= (int64_t)sizeof(SaeWorkHeader), "pb_sae_step_reset: work buffer too small");
  const int n = s->F > s->d ? s->F : s->d;
  int grid = (n + 255) / 256;
  if (grid > pb_sm_count() * 2) grid = pb_sm_count() * 2;
  if (grid * 256 < s->d) grid = (s->d + 255) / 256;
  PB_LAUNCH_PDL(k_sae_step_reset, grid, 256, 0, (cudaStream_t)stream, s->feat_count, s->F, (float*)s->scalars, s->gcol, s->gbdec2, s->d, (int*)s->work, fb_count);
  return PB_OK;
}

extern "C" int pb_sae_decode(const PbSaeStep* s, pb_stream_t stream) {
  PB_CHECK_ARG(s && s->x && s->xsum && s->idx && s->val && s->W_dec && s->b_dec && s->scalars, "pb_sae_decode: missing pointers");
  PB_CHECK_ARG(!s->training || (s->g && s->dval), "pb_sae_decode: training needs g and dval buffers");
  if (s->rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int d = s->d, ch = chunks_for(d);
  PB_DISPATCH_CHUNKS(ch, PB_LAUNCH_PDL(k_sae_decode<C_>, (s->rows + 7) / 8, 256, 0, st,
      s->x, s->xsum, s->mu, s->sd, s->idx, s->val, s->W_dec, s->b_dec, s->sae_out, s->g, s->dval, (SaeScalars*)s->scalars, s->rows, d, s->k,
      s->norm_mode, s->training, 1.f / (float)(s->global_rows > 0 ? s->global_rows : s->rows)));
  if (!s->training) {  // inference: publish mse / l0 now (the training path does it in k_sae_finalize)
    k_sae_fwd_scalars<<<1, 1, 0, st>>>((SaeScalars*)s->scalars, 1.f / ((float)s->rows * (float)d), 1.f / (float)s->rows);
    PB_LAUNCH_CHECK();
  }
  return PB_OK;
}

extern "C" int pb_sae_backward(const PbSaeStep* s, pb_stream_t stream) {
  PB_CHECK_ARG(s && s->idx && s->val && s->dval && s->g && s->sae_in && s->W_encT && s->feat_count && s->csc_off && s->csc_cursor &&
               s->csc_entries && s->gW_dec && s->gW_encT && s->gb_enc && s->gb_dec && s->gcol && s->gbdec2 && s->fired && s->scalars,
               "pb_sae_backward: missing pointers");
  if (s->rows == 0) return PB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int d = s->d, F = s->F, ch = chunks_for(d);
  {
    const int per = ((F + 1023) / 1024 + 3) / 4 * 4;
    PB_CHECK_ARG(per <= 128, "pb_sae_backward: d_sae=%d too large for the offset scan (max 131072)", F);
    if (per <= 8) PB_LAUNCH_PDL(k_scan_counts<8>, 1, 1024, 0, st, s->feat_count, s->csc_off, s->csc_cursor, F);
    else if (per <= 24) PB_LAUNCH_PDL(k_scan_counts<24>, 1, 1024, 0, st, s->feat_count, s->csc_off, s->csc_cursor, F);
    else if (per <= 48) PB_LAUNCH_PDL(k_scan_counts<48>, 1, 1024, 0, st, s->feat_count, s->csc_off, s->csc_cursor, F);
    else if (per <= 64) PB_LAUNCH_PDL(k_scan_counts<64>, 1, 1024, 0, st, s->feat_count, s->csc_off, s->csc_cursor, F);
    else PB_LAUNCH_PDL(k_scan_counts<128>, 1, 1024, 0, st, s->feat_count, s->csc_off, s->csc_cursor, F);
  }
  const int64_t n = (int64_t)s->rows * s->k;
  PB_LAUNCH_PDL(k_csc_fill, pb_sm_count() * 4, 256, 0, st, (const int*)s->idx, s->csc_cursor, s->csc_entries, n);
  if (!s->pre_zeroed) {
    PB_CUDA(cudaMemsetAsync(s->gcol, 0, sizeof(float) * d, st));
    PB_CUDA(cudaMemsetAsync(s->gbdec2, 0, sizeof(float) * d, st));
  }
  const int rpc = 8;     // 512 CTAs at 4096 rows: the 32-row version ran 128 CTAs of 32 dependent-latency trips (10.7 us)
  PB_LAUNCH_PDL(k_colsum, (s->rows + rpc - 1) / rpc, 256, 0, st, (const float*)s->g, s->gcol, s->rows, d, rpc);
  // work area for hot features: header | work_feats[F] | work_chunks[2 * (rows*k / CHUNK + F + 1)]
  const int64_t cap = n / SAE_LONG_CHUNK + F + 1;
  const int64_t need = (int64_t)sizeof(SaeWorkHeader) + 4 * (int64_t)F + 8 * cap;
  PB_CHECK_ARG(s->work && s->work_bytes >= need, "pb_sae_backward: work buffer too small (%lld < %lld bytes)", (long long)s->work_bytes,
               (long long)need);
  SaeWorkHeader* wh = (SaeWorkHeader*)s->work;
  int* work_feats = (int*)(wh + 1);
  int* work_chunks = work_feats + F;
  if (!s->pre_zeroed) PB_CUDA(cudaMemsetAsync(wh, 0, sizeof(SaeWorkHeader), st));
  const int grid = persistent_grid(8, F);
  PB_DISPATCH_CHUNKS(ch, PB_LAUNCH_PDL(k_sae_grads<C_>, grid, 256, sizeof(float) * d, st, s->csc_off, s->csc_entries, s->val, s->dval, s->g, s->sae_in,
                                       s->W_encT, s->gW_dec, s->gW_encT, s->gb_enc, s->gbdec2, s->fired, (SaeScalars*)s->scalars, F, d, s->k, wh,
                                       work_feats, work_chunks));
  PB_DISPATCH_CHUNKS(ch, PB_LAUNCH_PDL(k_sae_grads_long<C_>, pb_sm_count() * 4, 256, sizeof(float) * d, st, s->csc_off, s->csc_entries, s->val, s->dval,
                                       s->g, s->sae_in, s->W_encT, s->gW_dec, s->gW_encT, s->gb_enc, s->gbdec2, s->fired, d, s->k, wh, work_chunks));
  if (!s->dist) {
    PB_LAUNCH_PDL(k_sae_norm_long, pb_sm_count(), 256, 0, st, s->gW_dec, s->gW_encT, s->gb_enc, (SaeScalars*)s->scalars, d, wh, work_feats);
  }
  if (s->dist) {  // data parallel: only the local gb_dec; norm / clip happen after the peer reduction (p2p.cu)
    k_sae_gbdec<<<(d + 255) / 256, 256, 0, st>>>(s->gcol, s->gbdec2, s->gb_dec, d);
    PB_LAUNCH_CHECK();
    return PB_OK;
  }
  PB_LAUNCH_PDL(k_sae_finalize, 1, 256, 0, st, s->gcol, s->gbdec2, s->gb_dec, (SaeScalars*)s->scalars, d, s->max_grad_norm,
                1.f / ((float)s->rows * (float)d), 1.f / (float)s->rows);
  return PB_OK;
}

extern "C" int pb_sae_adam(const PbSaeStep* s, pb_stream_t stream) {
  PB_CHECK_ARG(s && s->W_dec && s->W_encT && s->b_enc && s->b_dec && s->gW_dec && s->gW_encT && s->gb_enc && s->gb_dec && s->m_dec &&
               s->v_dec && s->m_enc && s->v_enc && s->m_be && s->v_be && s->m_bd && s->v_bd && s->fired && s->scalars,
               "pb_sae_adam: missing pointers");
  PB_CHECK_ARG(s->step >= 1, "pb_sae_adam: step counter starts at 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int d = s->d, F = s->F, ch = chunks_for(d);
  AdamHyper h;
  h.lr = s->lr; h.beta1 = s->beta1; h.beta2 = s->beta2; h.eps = s->adam_eps;
  h.bc1 = 1.f - powf(s->beta1, (float)s->step);
  h.bc2_sqrt = sqrtf(1.f - powf(s->beta2, (float)s->step));
  const int grid = persistent_grid(8, F);
  if (s->enc_norm_max) PB_CUDA(cudaMemsetAsync(s->enc_norm_max, 0, 2 * sizeof(float), st));
  static int bulk_mode = -1;        // PB_SAE_ADAM=rows forces the register kernel (A/B measurements)
  if (bulk_mode < 0) { const char* e = getenv("PB_SAE_ADAM"); bulk_mode = (e && !strcmp(e, "rows")) ? 0 : 1; }
  if (bulk_mode && !s->W_encT_lo && d % 4 == 0 && d >= 64) {      // no tf32 residual plane to maintain: the bulk-copy pipeline
    const size_t stage = (size_t)8 * d * 4;
    int S = (int)((200 * 1024) / stage);
    if (S > 12) S = 12;
    if (S >= 3) {
      const size_t smem = 256 + (size_t)S * stage;
      int g2 = pb_sm_count();
      if (g2 > F) g2 = F;
#define PB_ADAM_BULK(CH)                                                                                                              \
  do {                                                                                                                                \
    auto kern = k_sae_adam_bulk<CH>;                                                                                                  \
    PB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                                     \
    PB_LAUNCH_PDL(kern, g2, 32 * (1 + S), smem, st, s->W_dec, s->W_encT, s->b_enc, s->gW_dec, s->gW_encT, s->gb_enc, s->m_dec, s->v_dec, s->m_enc, \
                  s->v_enc, s->m_be, s->v_be, s->fired, s->since_fired, s->act_freq, (const SaeScalars*)s->scalars,                    \
                  h, F, d, s->renorm_decoder, s->enc_norm_max, S, s->b_dec, s->gb_dec, s->m_bd, s->v_bd,                                \
                  reinterpret_cast<uint16_t*>(s->W_encT_h));                                                                          \
  } while (0)
      switch (ch) {
        case 1: PB_ADAM_BULK(1); break;
        case 2: PB_ADAM_BULK(2); break;
        case 4: PB_ADAM_BULK(4); break;
        case 6: PB_ADAM_BULK(6); break;
        case 8: PB_ADAM_BULK(8); break;
        case 12: PB_ADAM_BULK(12); break;
        default: pb_set_error("sae: d_in=%d unsupported", d); return PB_EUNSUPPORTED;
      }
#undef PB_ADAM_BULK
      return PB_OK;
    }
  }
  PB_DISPATCH_CHUNKS(ch, (k_sae_adam_rows<C_><<<grid, 256, 0, st>>>(s->W_dec, s->W_encT, s->W_encT_lo, s->b_enc, s->gW_dec, s->gW_encT, s->gb_enc,
                                                                     s->m_dec, s->v_dec, s->m_enc, s->v_enc, s->m_be, s->v_be, s->fired,
                                                                     s->since_fired, s->act_freq, (const SaeScalars*)s->scalars, h,
                                                                     F, d, s->renorm_decoder, s->enc_norm_max,
                                                                     reinterpret_cast<uint16_t*>(s->W_encT_h))));
  PB_LAUNCH_CHECK();
  k_sae_adam_vec<<<(d + 255) / 256, 256, 0, st>>>(s->b_dec, s->gb_dec, s->m_bd, s->v_bd, (const SaeScalars*)s->scalars, h, d);
  PB_LAUNCH_CHECK();
  return PB_OK;
}

extern "C" int pb_unit_norm_rows(float* W, float* W_lo, int32_t F, int32_t d, pb_stream_t stream) {
  PB_CHECK_ARG(W && F >= 0 && d > 0, "pb_unit_norm_rows: bad arguments");
  if (F == 0) return PB_OK;
  const int ch = chunks_for(d);
  cudaStream_t st = (cudaStream_t)stream;
  PB_DISPATCH_CHUNKS(ch, (k_unit_rows<C_><<<persistent_grid(8, F), 256, 0, st>>>(W, W_lo, F, d)));
  PB_LAUNCH_CHECK();
  return PB_OK;
}

// normalised MSE of an arbitrary reconstruction (dense / hooked route of SparseAutoencoder.forward, sae.py:144-149)
__global__ void __launch_bounds__(256) k_sae_mse_rows(const float* __restrict__ x, const float* __restrict__ xsum, const float* __restrict__ out,
                                                      float* __restrict__ acc, int rows, int d, float inv_rows) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  float part = 0.f;
  if (row < rows) {
    float nsq = 0.f, esq = 0.f;
    for (int c = lane; c < d; c += 32) {
      const float xv = x[(int64_t)row * d + c];
      const float xc = xv - xsum[c] * inv_rows;
      const float e = out[(int64_t)row * d + c] - xv;
      nsq += xc * xc;
      esq += e * e;
    }
    part = warp_sum(esq) / sqrtf(warp_sum(nsq));
  }
  if (lane == 0 && row < rows) atomicAdd(acc, part);
}
__global__ void k_scale_scalar(float* v, float s) { v[0] *= s; }

extern "C" int pb_sae_mse(const float* x, const float* out, float* xsum_scratch, float* result, int32_t rows, int32_t d, pb_stream_t stream) {
  PB_CHECK_ARG(x && out && xsum_scratch && result && rows > 0 && d > 0, "pb_sae_mse: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  PB_CUDA(cudaMemsetAsync(xsum_scratch, 0, sizeof(float) * d, st));
  PB_CUDA(cudaMemsetAsync(result, 0, sizeof(float), st));
  const int rpc = 32;
  k_colsum<<<(rows + rpc - 1) / rpc, 256, 0, st>>>(x, xsum_scratch, rows, d, rpc);
  PB_LAUNCH_CHECK();
  k_sae_mse_rows<<<(rows + 7) / 8, 256, 0, st>>>(x, xsum_scratch, out, result, rows, d, 1.f / (float)rows);
  PB_LAUNCH_CHECK();
  k_scale_scalar<<<1, 1, 0, st>>>(result, 1.f / ((float)rows * (float)d));
  PB_LAUNCH_CHECK();
  return PB_OK;
}

int pb_abi_sizeof_p2p(int which);  // p2p.cu
int pb_abi_sizeof_sae(int which) {
  if (which == 6) return (int)sizeof(PbSaeStep);
  if (which == 7) return (int)sizeof(SaeScalars);
  return pb_abi_sizeof_p2p(which);
}
