// Layout conversion, network-input synthesis, AvgPool2d(2,2) and bicubic up-sampling.
#include <cuda_fp16.h>

#include "common.cuh"

namespace pbmc {

// ---------------------------------------------------------------- NCHW <-> blocked
__global__ void pack_nchw_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int CB, size_t plane) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  const int cb = blockIdx.y, b = blockIdx.z;
  float v[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const int c = cb * 4 + l;
    v[l] = c < C ? __ldg(src + ((size_t)b * C + c) * plane + i) : 0.f;
  }
  *reinterpret_cast<float4*>(dst + (((size_t)b * CB + cb) * plane + i) * 4) = make_float4(v[0], v[1], v[2], v[3]);
}

__global__ void unpack_nchw_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int CB, size_t plane) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  const int cb = blockIdx.y, b = blockIdx.z;
  const float4 v = ldg4(src + (((size_t)b * CB + cb) * plane + i) * 4);
  const float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const int c = cb * 4 + l;
    if (c < C) dst[((size_t)b * C + c) * plane + i] = a[l];
  }
}

// blocked -> NCHW with the producer's GroupNorm(+GELU) applied (FluidLayer.forward tail, :796-797)
__global__ void finalize_nchw_kernel(const pbmc_src S, float* __restrict__ dst, int C, size_t plane) {
  const int cb = blockIdx.y, b = blockIdx.z;
  __shared__ float a4[4], b4[4];
  if (threadIdx.x < 4) {
    float a = 1.f, bb = 0.f;
    if (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN)
      gn_coeffs(S.stats + ((size_t)b * S.nblk + cb) * 2, S.inv_count, S.gamma[cb * 4 + threadIdx.x],
                S.beta[cb * 4 + threadIdx.x], a, bb);
    a4[threadIdx.x] = a;
    b4[threadIdx.x] = bb;
  }
  __syncthreads();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  float4 v = ldg4(S.ptr + (((size_t)b * S.nblk + cb) * plane + i) * 4);
  v = xform4(v, a4, b4, S.xform);
  const float a[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const int c = cb * 4 + l;
    if (c < C) dst[((size_t)b * C + c) * plane + i] = a[l];
  }
}

// ---------------------------------------------------------------- A1: network input
// TS.forward, pytorch_networks_convae.py:379-407.  log10(clip(exp(z),1e-8,1)) is evaluated as
// clamp(z*log10(e), -8, 0): identical in exact arithmetic, and free of the exp->log10 round trip.
// `zero` / `zero_words`: scratch of the forward that follows (statistics accumulators, grid-barrier counters, the CFL
// maximum) cleared here, grid-stride, instead of by memset nodes in front of conv[0] -- two links less on the rollout's
// critical chain.  NULL outside the rollout.
__global__ void build_input_kernel(const float* __restrict__ T, const float* __restrict__ xc,
                                   const float* __restrict__ yc, const float* __restrict__ ycc,
                                   const pbmc_member* __restrict__ mem, float* __restrict__ inp, float* __restrict__ V,
                                   size_t plane, uint32_t* __restrict__ zero, size_t zero_words) {
  // no-ops unless launched with programmatic stream serialization (the rollout does, behind the stencil)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (zero != nullptr) {
    const size_t nthr = (size_t)gridDim.x * gridDim.y * blockDim.x;
    for (size_t w = (size_t)blockIdx.y * gridDim.x * blockDim.x + i; w < zero_words; w += nthr) zero[w] = 0u;
  }
  if (i >= plane) return;
  const int b = blockIdx.y;
  const pbmc_member m = mem[b];
  const float t = __ldg(T + (size_t)b * plane + i);
  const float z = m.ln_fkt * (0.0f - t) + m.ln_fkp * (1.0f - __ldg(ycc + i));
  const float l10 = fminf(fmaxf(z * 0.43429448190325182765f, -8.0f), 0.0f);
  float4 c0 = make_float4(__ldg(xc + i) * 0.25f, __ldg(yc + i) * 0.25f, l10 * 0.125f, m.raq_nd);
  float4 c1 = make_float4(m.fkt_nd, m.fkp_nd, t, 0.f);
  *reinterpret_cast<float4*>(inp + (((size_t)b * 2 + 0) * plane + i) * 4) = c0;
  *reinterpret_cast<float4*>(inp + (((size_t)b * 2 + 1) * plane + i) * 4) = c1;
  if (V != nullptr) V[(size_t)b * plane + i] = fminf(fmaxf(expf(z), 1e-8f), 1.0f);
}

// ---------------------------------------------------------------- A5: AvgPool2d(2,2), floor
__global__ void avgpool2_kernel(const pbmc_src S, float* __restrict__ dst, int H, int W, int Ho, int Wo) {
  const int cb = blockIdx.y, b = blockIdx.z;
  __shared__ float a4[4], b4[4];
  if (threadIdx.x < 4) {
    float a = 1.f, bb = 0.f;
    if (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN)
      gn_coeffs(S.stats + ((size_t)b * S.nblk + cb) * 2, S.inv_count, S.gamma[cb * 4 + threadIdx.x],
                S.beta[cb * 4 + threadIdx.x], a, bb);
    a4[threadIdx.x] = a;
    b4[threadIdx.x] = bb;
  }
  __syncthreads();
  const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= (size_t)Ho * Wo) return;
  const int oy = (int)(o / Wo), ox = (int)(o % Wo);
  const float* base = S.ptr + ((size_t)b * S.nblk + cb) * (size_t)H * W * 4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      float4 v = ldg4(base + ((size_t)(2 * oy + dy) * W + 2 * ox + dx) * 4);
      v = xform4(v, a4, b4, S.xform);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  s.x *= 0.25f; s.y *= 0.25f; s.z *= 0.25f; s.w *= 0.25f;
  *reinterpret_cast<float4*>(dst + (((size_t)b * S.nblk + cb) * (size_t)Ho * Wo + o) * 4) = s;
}

// ---------------------------------------------------------------- A5: bicubic up-sampling
// nn.Upsample(size, mode="bicubic"): align_corners=False, A = -0.75, source index
// scale*(dst+0.5)-0.5 NOT clamped, the four taps clamped to [0, n-1].
constexpr int BU_TW = 128, BU_TH = 8;  // output tile; 256 threads, four output pixels (float4 each) per thread
constexpr int BU_MAX_SW = BU_TW + 4, BU_MAX_SH = BU_TH + 4;

__device__ __forceinline__ void cubic_w(float t, float w[4]) {
  const float A = -0.75f;
  const float x0 = t + 1.f, x1 = t, x2 = 1.f - t, x3 = 2.f - t;
  w[0] = ((A * x0 - 5.f * A) * x0 + 8.f * A) * x0 - 4.f * A;
  w[1] = ((A + 2.f) * x1 - (A + 3.f)) * x1 * x1 + 1.f;
  w[2] = ((A + 2.f) * x2 - (A + 3.f)) * x2 * x2 + 1.f;
  w[3] = ((A * x3 - 5.f * A) * x3 + 8.f * A) * x3 - 4.f * A;
}

__device__ __forceinline__ int src_floor(int d, float scale, float& t) {
  const float s = scale * ((float)d + 0.5f) - 0.5f;
  const float f = floorf(s);
  t = s - f;
  return (int)f;
}

// Separable in shared memory, same association as oracle/ref_numpy.bicubic_upsample (rows first, then columns):
//   pass 1  colv[r][c] = sum_ky wy_r[ky] * src[cy_r[ky]][c]      for the 8 output rows x the tile's source columns
//   pass 2  out[r][x]  = sum_kx wx_x[kx] * colv[r][cx_x[kx]]
// i.e. 4 + <=4 shared-memory reads per output instead of 16 (the first version was shared-memory bound: 16.6 us per level).
// STAGED: the output is written as the conv[1] operand image (PBMC_LAYOUT_STAGED16, include/pbmc.h) instead of
// blocked fp32: fp16 hi | lo of every value, [row][part][chunk][position][8 channels], with the replicate-padded
// columns -1 / W at positions 0 / W+1, so that the row conv kernel stages it with four bulk copies per row.
template <bool STAGED>
__global__ void __launch_bounds__(256) bicubic_kernel(const pbmc_src S, float* __restrict__ dst, int Hs, int Ws, int H, int W,
                                                      float sy_scale, float sx_scale) {
  __shared__ float4 tile[BU_MAX_SH][BU_MAX_SW];
  __shared__ float4 colv[BU_TH][BU_MAX_SW];
  __shared__ float a4[4], b4[4];
  __shared__ float wy_s[BU_TH][4];
  __shared__ int cy_s[BU_TH][4];
  const int cb = blockIdx.z % S.nblk, b = blockIdx.z / S.nblk;
  const int tid = threadIdx.x;
  const int ox0 = blockIdx.x * BU_TW, oy0 = blockIdx.y * BU_TH;
  const int ox1 = min(ox0 + BU_TW, W) - 1, oy1 = min(oy0 + BU_TH, H) - 1;
  float tdum;
  // source footprint of this output tile (taps -1..+2 around the floor), clamped like the taps are
  const int fx0 = max(src_floor(ox0, sx_scale, tdum) - 1, 0), fx1 = min(src_floor(ox1, sx_scale, tdum) + 2, Ws - 1);
  const int fy0 = max(src_floor(oy0, sy_scale, tdum) - 1, 0), fy1 = min(src_floor(oy1, sy_scale, tdum) + 2, Hs - 1);
  const int fw = fx1 - fx0 + 1, fh = fy1 - fy0 + 1;  // <= BU_T? + 4 because scale <= 1
  if (tid < 4) {
    float a = 1.f, bb = 0.f;
    if (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN)
      gn_coeffs(S.stats + ((size_t)b * S.nblk + cb) * 2, S.inv_count, S.gamma[cb * 4 + tid], S.beta[cb * 4 + tid], a, bb);
    a4[tid] = a;
    b4[tid] = bb;
  }
  if (tid >= 32 && tid < 32 + BU_TH) {
    const int r = tid - 32, oy = min(oy0 + r, H - 1);
    float ty, wy[4];
    const int iy = src_floor(oy, sy_scale, ty);
    cubic_w(ty, wy);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      wy_s[r][k] = wy[k];
      cy_s[r][k] = min(max(iy - 1 + k, 0), Hs - 1) - fy0;
    }
  }
  __syncthreads();
  const float* base = S.ptr + ((size_t)b * S.nblk + cb) * (size_t)Hs * Ws * 4;
  for (int e = tid; e < fw * fh; e += 256) {
    const int r = e / fw, c = e - r * fw;
    float4 v = ldg4(base + ((size_t)(fy0 + r) * Ws + fx0 + c) * 4);
    tile[r][c] = xform4(v, a4, b4, S.xform);
  }
  __syncthreads();
  const int nrow = oy1 - oy0 + 1;
  for (int e = tid; e < nrow * fw; e += 256) {
    const int r = e / fw, c = e - r * fw;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const float w = wy_s[r][ky];
      const float4 v = tile[cy_s[r][ky]][c];
      acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y); acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
    }
    colv[r][c] = acc;
  }
  __syncthreads();
  const int ty_ = tid >> 5, lane = tid & 31;
  const int oy = oy0 + ty_;
  if (oy >= H) return;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ox = ox0 + lane + 32 * j;
    if (ox >= W) break;
    float tx, wx[4];
    const int ix = src_floor(ox, sx_scale, tx);
    cubic_w(tx, wx);
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int kx = 0; kx < 4; ++kx) {
      const float4 v = colv[ty_][min(max(ix - 1 + kx, 0), Ws - 1) - fx0];
      o.x = fmaf(wx[kx], v.x, o.x); o.y = fmaf(wx[kx], v.y, o.y); o.z = fmaf(wx[kx], v.z, o.z); o.w = fmaf(wx[kx], v.w, o.w);
    }
    if (!STAGED) {
      *reinterpret_cast<float4*>(dst + (((size_t)b * S.nblk + cb) * (size_t)H * W + (size_t)oy * W + ox) * 4) = o;
    } else {
      // channels cb*4 .. cb*4+3 of chunk cb>>1: 8 bytes at byte (cb&1)*8 of the position's 16-byte cell
      const __half2 h01 = __floats2half2_rn(o.x, o.y), h23 = __floats2half2_rn(o.z, o.w);
      const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
      const __half2 l01 = __floats2half2_rn(o.x - f01.x, o.y - f01.y), l23 = __floats2half2_rn(o.z - f23.x, o.w - f23.y);
      const uint2 hi = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
      const uint2 lo = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
      const size_t Wp = (size_t)((W + 127) / 128 * 128 + 2);
      unsigned char* row = reinterpret_cast<unsigned char*>(dst) + ((size_t)b * H + oy) * 4 * Wp * 16;
      const size_t plane_hi = (size_t)(cb >> 1) * Wp * 16, plane_lo = (size_t)(2 + (cb >> 1)) * Wp * 16;
      const size_t cell = (size_t)(ox + 1) * 16 + (size_t)(cb & 1) * 8;
      *reinterpret_cast<uint2*>(row + plane_hi + cell) = hi;
      *reinterpret_cast<uint2*>(row + plane_lo + cell) = lo;
      if (ox == 0) {
        *reinterpret_cast<uint2*>(row + plane_hi + cell - 16) = hi;
        *reinterpret_cast<uint2*>(row + plane_lo + cell - 16) = lo;
      }
      if (ox == W - 1) {
        *reinterpret_cast<uint2*>(row + plane_hi + cell + 16) = hi;
        *reinterpret_cast<uint2*>(row + plane_lo + cell + 16) = lo;
      }
    }
  }
}

}  // namespace pbmc

using namespace pbmc;

extern "C" int pbmc_pack_nchw(const float* src, float* dst, int B, int C, int H, int W, void* stream) {
  if (!src || !dst) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(dst)) return PBMC_ERR_MISALIGNED;
  const size_t plane = (size_t)H * W;
  dim3 grid((unsigned)((plane + 255) / 256), (C + 3) / 4, B);
  pack_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, C, (C + 3) / 4, plane);
  PBMC_CHECK_LAUNCH("pack_nchw_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_unpack_nchw(const float* src, float* dst, int B, int C, int H, int W, void* stream) {
  if (!src || !dst) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(src)) return PBMC_ERR_MISALIGNED;
  const size_t plane = (size_t)H * W;
  dim3 grid((unsigned)((plane + 255) / 256), (C + 3) / 4, B);
  unpack_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, C, (C + 3) / 4, plane);
  PBMC_CHECK_LAUNCH("unpack_nchw_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_finalize_nchw(const pbmc_src* S, float* dst, int B, int C, int H, int W, void* stream) {
  if (!S || !S->ptr || !dst) return PBMC_ERR_NULL_POINTER;
  if (S->layout != PBMC_LAYOUT_BLOCKED) return PBMC_ERR_UNSUPPORTED;
  if ((S->xform == PBMC_XFORM_GN_GELU || S->xform == PBMC_XFORM_GN) && (!S->stats || !S->gamma || !S->beta)) return PBMC_ERR_NULL_POINTER;
  if (S->xform < PBMC_XFORM_NONE || S->xform > PBMC_XFORM_GELU) return PBMC_ERR_UNSUPPORTED;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || S->nblk != (C + 3) / 4) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(S->ptr)) return PBMC_ERR_MISALIGNED;
  const size_t plane = (size_t)H * W;
  dim3 grid((unsigned)((plane + 255) / 256), S->nblk, B);
  finalize_nchw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*S, dst, C, plane);
  PBMC_CHECK_LAUNCH("finalize_nchw_kernel");
  return PBMC_OK;
}

namespace pbmc {
int build_input_enqueue(const float* T, const float* xc, const float* yc, const float* ycc, const pbmc_member* members, float* inp,
                        float* V, int B, int H, int W, void* zero, size_t zero_bytes, cudaStream_t st, bool pdl) {
  if (!T || !xc || !yc || !ycc || !members || !inp) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(inp) || (zero_bytes & 3) != 0) return PBMC_ERR_MISALIGNED;
  const size_t plane = (size_t)H * W;
  dim3 grid((unsigned)((plane + 255) / 256), B);
  PBMC_CUDA(launch_maybe_pdl(build_input_kernel, grid, dim3(256), 0, st, pdl, T, xc, yc, ycc, members, inp, V, plane,
                             reinterpret_cast<uint32_t*>(zero), zero_bytes / 4));
  PBMC_CHECK_LAUNCH("build_input_kernel");
  return PBMC_OK;
}
}  // namespace pbmc

extern "C" int pbmc_build_input(const float* T, const float* xc, const float* yc, const float* ycc,
                                const pbmc_member* members, float* inp, float* V, int B, int H, int W, void* stream) {
  return pbmc::build_input_enqueue(T, xc, yc, ycc, members, inp, V, B, H, W, nullptr, 0, (cudaStream_t)stream, false);
}

extern "C" int pbmc_avgpool2(const pbmc_src* S, float* dst, int B, int H, int W, void* stream) {
  if (!S || !S->ptr || !dst) return PBMC_ERR_NULL_POINTER;
  if (S->layout != PBMC_LAYOUT_BLOCKED) return PBMC_ERR_UNSUPPORTED;
  if ((S->xform == PBMC_XFORM_GN_GELU || S->xform == PBMC_XFORM_GN) && (!S->stats || !S->gamma || !S->beta)) return PBMC_ERR_NULL_POINTER;
  if (S->xform < PBMC_XFORM_NONE || S->xform > PBMC_XFORM_GELU) return PBMC_ERR_UNSUPPORTED;
  const int Ho = H / 2, Wo = W / 2;
  if (B <= 0 || Ho <= 0 || Wo <= 0 || S->nblk <= 0) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(S->ptr) || !aligned16(dst)) return PBMC_ERR_MISALIGNED;
  dim3 grid((unsigned)(((size_t)Ho * Wo + 255) / 256), S->nblk, B);
  avgpool2_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*S, dst, H, W, Ho, Wo);
  PBMC_CHECK_LAUNCH("avgpool2_kernel");
  return PBMC_OK;
}

static int bicubic_launch(const pbmc_src* S, void* dst, int B, int Hs, int Ws, int H, int W, bool staged, void* stream) {
  if (!S || !S->ptr || !dst) return PBMC_ERR_NULL_POINTER;
  if ((S->xform == PBMC_XFORM_GN_GELU || S->xform == PBMC_XFORM_GN) && (!S->stats || !S->gamma || !S->beta)) return PBMC_ERR_NULL_POINTER;
  if (S->xform < PBMC_XFORM_NONE || S->xform > PBMC_XFORM_GELU) return PBMC_ERR_UNSUPPORTED;
  if (B <= 0 || Hs <= 0 || Ws <= 0 || H < Hs || W < Ws || S->nblk <= 0) return PBMC_ERR_BAD_SHAPE;  // up-sampling only
  if (S->layout != PBMC_LAYOUT_BLOCKED) return PBMC_ERR_UNSUPPORTED;
  if (staged && S->nblk != 4) return PBMC_ERR_UNSUPPORTED;  // the staged image is one 16-channel K group
  if (!aligned16(S->ptr) || !aligned16(dst)) return PBMC_ERR_MISALIGNED;
  dim3 grid(cdiv(W, BU_TW), cdiv(H, BU_TH), B * S->nblk);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  if (staged)
    bicubic_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(*S, reinterpret_cast<float*>(dst), Hs, Ws, H, W, (float)Hs / (float)H,
                                                                 (float)Ws / (float)W);
  else
    bicubic_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(*S, reinterpret_cast<float*>(dst), Hs, Ws, H, W, (float)Hs / (float)H,
                                                                  (float)Ws / (float)W);
  PBMC_CHECK_LAUNCH("bicubic_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_bicubic_up(const pbmc_src* S, float* dst, int B, int Hs, int Ws, int H, int W, void* stream) {
  return bicubic_launch(S, dst, B, Hs, Ws, H, W, false, stream);
}
extern "C" int pbmc_bicubic_up_staged(const pbmc_src* S, void* dst, int B, int Hs, int Ws, int H, int W, void* stream) {
  return bicubic_launch(S, dst, B, Hs, Ws, H, W, true, stream);
}
extern "C" int pbmc_staged_width(int W) { return W > 0 ? (W + 127) / 128 * 128 + 2 : 0; }
extern "C" size_t pbmc_staged_bytes(int B, int H, int W) {
  return (B > 0 && H > 0 && W > 0) ? (size_t)B * H * 4 * (size_t)pbmc_staged_width(W) * 16 : 0;
}
