// common.cuh -- shared helpers for libprisma_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include "../../include/prisma_b200.h"

// ------------------------------------------------------------------ errors
void pb_set_error(const char* fmt, ...);

#define PB_CHECK_ARG(cond, ...)                                   \
  do {                                                            \
    if (!(cond)) {                                                \
      pb_set_error(__VA_ARGS__);                                  \
      return PB_EINVAL;                                           \
    }                                                             \
  } while (0)

#define PB_CUDA(call)                                                                  \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess) {                                                          \
      pb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return PB_ECUDA;                                                                 \
    }                                                                                  \
  } while (0)

extern unsigned long long g_pb_launches;  // kernels launched by this library (pb_launch_count)

#define PB_LAUNCH_CHECK()                                                              \
  do {                                                                                 \
    ++g_pb_launches;                                                                   \
    cudaError_t e__ = cudaGetLastError();                                              \
    if (e__ != cudaSuccess) {                                                          \
      pb_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return PB_ECUDA;                                                                 \
    }                                                                                  \
  } while (0)

#define PB_TRY(expr)                \
  do {                              \
    int rc__ = (expr);              \
    if (rc__ != PB_OK) return rc__; \
  } while (0)

int pb_sm_count();  // cached multiprocessor count of the current device

// ------------------------------------------------------------------ dtypes
typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float ld_as_float(const float* p) { return *p; }
__device__ __forceinline__ float ld_as_float(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void st_from_float(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_from_float(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
// value as it will read back after a store in T (bf16 rounding made explicit)
template <typename T> __device__ __forceinline__ float round_to(float v);
template <> __device__ __forceinline__ float round_to<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_to<bf16>(float v) {
  return __bfloat162float(__float2bfloat16_rn(v));
}

// 4-element vector access (16 B for float, 8 B for bf16)
struct alignas(8) bf16x4 { __nv_bfloat162 lo, hi; };
__device__ __forceinline__ void ld4(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void ld4(const bf16* p, float (&v)[4]) {
  bf16x4 t = *reinterpret_cast<const bf16x4*>(p);
  float2 a = __bfloat1622float2(t.lo), b = __bfloat1622float2(t.hi);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void st4(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void st4(bf16* p, const float (&v)[4]) {
  bf16x4 t;
  t.lo = __floats2bfloat162_rn(v[0], v[1]);
  t.hi = __floats2bfloat162_rn(v[2], v[3]);
  *reinterpret_cast<bf16x4*>(p) = t;
}

// tf32 split: hi = x with the 13 low mantissa bits cleared (what kind::tf32 consumes),
// lo = x - hi (exact in fp32).
__device__ __forceinline__ float tf32_trunc(float x) {
  return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
}
// low plane of the 3xTF32 split: x - hi, itself rounded to the NEAREST tf32 so that the tensor core's truncating read of the
// plane is exact.  A truncated lo loses up to 2^-20 |x| per element, always in the same direction, so the error of a K-term dot
// product grows like K (measured 2.6e-5 at K = 3072); rounded, it is +-2^-21 |x| and averages out (profiles/r01_gemm_notes.md).
__device__ __forceinline__ float tf32_lo(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x - tf32_trunc(x)));
  return __uint_as_float(r);
}

// fp16 operand of the fused encoder's candidate GEMM (sae_in_h, W_encT_h): round to nearest, saturate to +-65504, and flush
// results below 2^-14 in magnitude to zero.  Every producer of the fp16 shadows and every residual norm of the error bound uses
// this one conversion.  The flush makes the software residual x - f16_val(h) exact whatever the tensor core does with fp16
// subnormals; saturation turns an overflow into a huge residual, so the bound fails and the row takes the exact path.
__device__ __forceinline__ uint16_t f16_cand(float x) {
  uint16_t h;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(h) : "f"(x));
  return (h & 0x7c00u) == 0 ? (uint16_t)0 : h;
}
__device__ __forceinline__ float f16_val(uint16_t h) { return __half2float(__ushort_as_half(h)); }
// row stride (elements) of the fp16 shadows: rows padded to 16 bytes, as the tensor maps require
__host__ __device__ __forceinline__ int f16_ld(int d) { return (d + 7) & ~7; }
// four consecutive fp16 operands (8 bytes) + the sum of squares of their residuals
__device__ __forceinline__ float st4_f16_cand(uint16_t* p, const float v[4]) {
  const uint16_t h0 = f16_cand(v[0]), h1 = f16_cand(v[1]), h2 = f16_cand(v[2]), h3 = f16_cand(v[3]);
  if (p) *reinterpret_cast<uint2*>(p) = make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
  const float r0 = v[0] - f16_val(h0), r1 = v[1] - f16_val(h1), r2 = v[2] - f16_val(h2), r3 = v[3] - f16_val(h3);
  return r0 * r0 + r1 * r1 + r2 * r2 + r3 * r3;
}

// ------------------------------------------------------------- activations
// Matches torch: F.gelu (erf), F.silu, F.relu and the closed forms in
// reference models/activation_fns.py:19-47.
__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case PB_ACT_RELU: return fmaxf(x, 0.f);
    case PB_ACT_GELU: return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
    case PB_ACT_SILU: return x / (1.f + expf(-x));
    case PB_ACT_GELU_NEW: {
      float inner = 0.79788456080286535588f * (x + 0.044715f * x * x * x);
      return 0.5f * x * (1.f + tanhf(inner));
    }
    case PB_ACT_GELU_FAST: return 0.5f * x * (1.f + tanhf(x * 0.7978845608f * (1.f + 0.044715f * x * x)));
    case PB_ACT_QUICK_GELU: return x / (1.f + expf(-1.702f * x));
    case PB_ACT_TANH_RELU: return tanhf(fmaxf(x, 0.f));
    case PB_ACT_EXP: return expf(x);
    default: return x;
  }
}

// ------------------------------------------------------------ reductions
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ------------------------------------------------- programmatic dependent launch (PDL)
// The SAE training step is ~15 short dependent kernels; launched back to back they leave the GPU idle for a few microseconds at
// every boundary (grid launch latency + block ramp-up).  With the programmatic-stream-serialization attribute the NEXT kernel's
// blocks are dispatched as soon as every block of the current kernel has executed `griddepcontrol.launch_dependents` (first thing
// each kernel does) and then park in `griddepcontrol.wait` until the current kernel has completed and flushed -- so correctness
// is exactly stream order, only the dispatch latency is hidden.  PB_PDL=0 in the environment launches plainly (A/B, debugging).
__device__ __forceinline__ void pb_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pb_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pb_pdl() { pb_pdl_trigger(); pb_pdl_wait(); }

bool pb_pdl_enabled();   // library.cu-level switch (PB_PDL environment variable, default on)

template <typename... KArgs, typename... Args>
static inline cudaError_t pb_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pb_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#define PB_LAUNCH_PDL(kern, grid, block, smem, st, ...)                                  \
  do {                                                                                   \
    cudaError_t le__ = pb_launch_pdl(kern, dim3(grid), dim3(block), (size_t)(smem), st, __VA_ARGS__); \
    ++g_pb_launches;                                                                     \
    if (le__ != cudaSuccess) {                                                           \
      pb_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(le__)); \
      return PB_ECUDA;                                                                   \
    }                                                                                    \
  } while (0)
