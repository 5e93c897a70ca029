// Shared device/host helpers for libpbmc (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "pbmc.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libpbmc is written for sm_100a (B200) only"
#endif

namespace pbmc {

// ---------------------------------------------------------------- host-side error plumbing
void set_last_cuda_error(cudaError_t e, const char* where);

#define PBMC_CHECK_LAUNCH(where)                         \
  do {                                                   \
    cudaError_t _e = cudaPeekAtLastError();              \
    if (_e != cudaSuccess) {                             \
      ::pbmc::set_last_cuda_error(_e, where);            \
      return PBMC_ERR_CUDA;                              \
    }                                                    \
  } while (0)

#define PBMC_CUDA(call)                                  \
  do {                                                   \
    cudaError_t _e = (call);                             \
    if (_e != cudaSuccess) {                             \
      ::pbmc::set_last_cuda_error(_e, #call);            \
      return PBMC_ERR_CUDA;                              \
    }                                                    \
  } while (0)

// Kernel launch with optional programmatic stream serialization: the kernel may become resident while its predecessor in
// the stream drains and must execute griddepcontrol.wait before it touches anything the predecessor (or, transitively,
// anything earlier) wrote or still reads.  Without the attribute griddepcontrol.* are no-ops.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_maybe_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                           Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------- device math
// exact-erf GELU, nn.GELU() default (pytorch_networks_convae.py:751): x * Phi(x).
// Branch-free evaluation: Phi(-t) = 2^q(t) for t = |x| with q a degree-8 minimax fit of log2(Phi(-t)) on
// [0, 6.6] (absolute error of Phi and of t*Phi < 1.5e-8 before rounding, below fp32's 6e-8 |x|; x * Phi(-6.6) < 2e-10, so clamping t is exact in
// fp32), Phi(x) = 1 - Phi(-x) for x > 0.  12 instructions instead of erff's two selected polynomials;
// fp32 result within 2.6e-7 absolute of the float64 value (tools/fit_gelu.py regenerates and checks the fit).
__device__ __forceinline__ float gelu_erf(float x) {
  const float t = fminf(fabsf(x), 6.6f);
  float q = -2.2756834377020336e-06f;
  q = fmaf(q, t, 3.296563960267106e-05f);
  q = fmaf(q, t, -0.000157266929481836f);
  q = fmaf(q, t, -0.0002025088577467934f);
  q = fmaf(q, t, 0.007142822415561599f);
  q = fmaf(q, t, -0.05254646501180134f);
  q = fmaf(q, t, -0.4591930475265861f);
  q = fmaf(q, t, -1.1511069423662477f);
  q = fmaf(q, t, -0.9999999590055544f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(q));
  // x * Phi(x) = max(x, 0) - |x| * Phi(-|x|): one FMNMX + one FFMA instead of compare, predicated subtract, multiply
  return fmaf(-fabsf(x), e, fmaxf(x, 0.f));
}

// Two GELUs at once on the packed fp32x2 pipe (FFMA2, sm_100): same polynomial, same rounding per lane as
// gelu_erf -- the results are bit-identical to two scalar calls, at half the FMA issue slots.
__device__ __forceinline__ uint64_t f2_pack(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
  const uint64_t t = f2_pack(fminf(fabsf(x0), 6.6f), fminf(fabsf(x1), 6.6f));
  uint64_t q = f2_pack(-2.2756834377020336e-06f, -2.2756834377020336e-06f);
#define PBMC_F2C(c) f2_pack(c, c)
  q = f2_fma(q, t, PBMC_F2C(3.296563960267106e-05f));
  q = f2_fma(q, t, PBMC_F2C(-0.000157266929481836f));
  q = f2_fma(q, t, PBMC_F2C(-0.0002025088577467934f));
  q = f2_fma(q, t, PBMC_F2C(0.007142822415561599f));
  q = f2_fma(q, t, PBMC_F2C(-0.05254646501180134f));
  q = f2_fma(q, t, PBMC_F2C(-0.4591930475265861f));
  q = f2_fma(q, t, PBMC_F2C(-1.1511069423662477f));
  q = f2_fma(q, t, PBMC_F2C(-0.9999999590055544f));
#undef PBMC_F2C
  float q0, q1, e0, e1;
  f2_unpack(q, q0, q1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(q0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(q1));
  x0 = fmaf(-fabsf(x0), e0, fmaxf(x0, 0.f));
  x1 = fmaf(-fabsf(x1), e1, fmaxf(x1, 0.f));
}

// NP packed pairs of exact-erf GELUs in lock step: the same polynomial and rounding as gelu_erf2 (common.cuh),
// written so that the NP dependent FFMA2 chains are interleaved in program order.
template <int NP>
__device__ __forceinline__ void gelu_erf2n(float* x) {
  uint64_t t[NP], q[NP];
#pragma unroll
  for (int k = 0; k < NP; ++k) {
    t[k] = f2_pack(fminf(fabsf(x[2 * k]), 6.6f), fminf(fabsf(x[2 * k + 1]), 6.6f));
    q[k] = f2_pack(-2.2756834377020336e-06f, -2.2756834377020336e-06f);
  }
#define PBMC_F2STEP(c)                                          \
  _Pragma("unroll") for (int k = 0; k < NP; ++k) q[k] = f2_fma(q[k], t[k], f2_pack(c, c));
  PBMC_F2STEP(3.296563960267106e-05f)
  PBMC_F2STEP(-0.000157266929481836f)
  PBMC_F2STEP(-0.0002025088577467934f)
  PBMC_F2STEP(0.007142822415561599f)
  PBMC_F2STEP(-0.05254646501180134f)
  PBMC_F2STEP(-0.4591930475265861f)
  PBMC_F2STEP(-1.1511069423662477f)
  PBMC_F2STEP(-0.9999999590055544f)
#undef PBMC_F2STEP
#pragma unroll
  for (int k = 0; k < NP; ++k) {
    float q0, q1, e0, e1;
    f2_unpack(q[k], q0, q1);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(q0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(q1));
    const float a = x[2 * k], b = x[2 * k + 1];
    x[2 * k] = fmaf(-fabsf(a), e0, fmaxf(a, 0.f));
    x[2 * k + 1] = fmaf(-fabsf(b), e1, fmaxf(b, 0.f));
  }
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// source index for a padded coordinate; returns -1 for a zero-padded tap
__device__ __forceinline__ int pad_index(int i, int n, int mode) {
  if (i >= 0 && i < n) return i;
  if (mode == PBMC_PAD_REPLICATE) return i < 0 ? 0 : n - 1;
  if (mode == PBMC_PAD_REFLECT) {
    int r = i < 0 ? -i : 2 * (n - 1) - i;
    return r < 0 ? 0 : (r >= n ? n - 1 : r);
  }
  return -1;
}

// Per-channel (scale, shift) of a fused GroupNorm: y = x*a + b, from raw (sum, sum^2).
// torch.nn.GroupNorm semantics: biased variance, eps = 1e-5 (pytorch_networks_convae.py:788).
__device__ __forceinline__ void gn_coeffs(const double* stats2, double inv_count, float gamma, float beta, float& a,
                                          float& b) {
  double mean = stats2[0] * inv_count;
  double var = stats2[1] * inv_count - mean * mean;
  if (var < 0.0) var = 0.0;
  double rstd = rsqrt(var + 1e-5);
  double ad = rstd * (double)gamma;
  a = (float)ad;
  b = (float)((double)beta - mean * ad);
}

// PBMC_XFORM_SCALE: 2^-s with 2^(s-1) <= rms < 2^s, rms over all nblk*4 channels of one sample from its (sum, sum^2) per
// block; 1 for an all-zero source.  A power of two, so scaling the source by it (and the output back) is exact.
__device__ __forceinline__ float scale_src_factor(const double* st, int nblk, size_t plane_px) {
  double ss = 0.0;
  for (int k = 0; k < nblk; ++k) ss += __ldcg(st + 2 * k + 1);
  int ex = 0;
  frexp(sqrt(ss / ((double)nblk * 4.0 * (double)plane_px)), &ex);
  ex = ex < -64 ? -64 : (ex > 64 ? 64 : ex);
  return ldexpf(1.f, -ex);
}
__device__ __forceinline__ float4 xform4(float4 v, const float* a4, const float* b4, int xform) {
  if (xform == PBMC_XFORM_NONE) return v;
  if (xform != PBMC_XFORM_GELU) {
    v.x = fmaf(v.x, a4[0], b4[0]);
    v.y = fmaf(v.y, a4[1], b4[1]);
    v.z = fmaf(v.z, a4[2], b4[2]);
    v.w = fmaf(v.w, a4[3], b4[3]);
  }
  if (xform != PBMC_XFORM_GN) {
    v.x = gelu_erf(v.x);
    v.y = gelu_erf(v.y);
    v.z = gelu_erf(v.z);
    v.w = gelu_erf(v.w);
  }
  return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// non-negative floats order like their bit patterns
__device__ __forceinline__ void atomic_max_nonneg(uint32_t* addr, float v) { atomicMax(addr, __float_as_uint(v)); }

}  // namespace pbmc
