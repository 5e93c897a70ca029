// A7: network head -- zero-mean, stream-function curl, wall boundary conditions,
// velocity un-scaling and the CFL reduction max|u|,|v| in ONE pass.
//   pytorch_networks_convae.py:1343       y - mean(y, (2,3))
//   :1357-1370                            a = y0*a_bound; u = d a/d row; v = -d a/d col (central, interior)
//   :1372-1386                            replicate pad; u side columns / v wall rows negated; corners 0
//   :341-352, :411-412                    u,v *= scaler
//   :524-525, :556  (ADNet)               max|u|,|v| over [1:-1,1:-1]
#include "common.cuh"

namespace pbmc {

__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ y, const double* __restrict__ chan_sum,
                                                   const pbmc_member* __restrict__ mem, float a_bound, int head_kind,
                                                   int p_pred, float* __restrict__ u, float* __restrict__ v,
                                                   float* __restrict__ p, uint32_t* __restrict__ uvmax, int H, int W) {
  // no-ops unless launched with programmatic stream serialization (api.cu does, behind conv[3])
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int b = blockIdx.z;
  const int gx = blockIdx.x * 32 + threadIdx.x;
  const int gy = blockIdx.y * 8 + threadIdx.y;
  const size_t plane = (size_t)H * W;
  const float* yb = y + (size_t)b * plane * 4;
  const float sc = mem ? mem[b].scaler : 1.0f;
  float m = 0.f;  // |u|,|v| candidate for the CFL reduction
  if (gx < W && gy < H) {
    const size_t o = (size_t)b * plane + (size_t)gy * W + gx;
    const double inv_n = 1.0 / (double)plane;
    if (head_kind == PBMC_HEAD_CURL) {
      // value of the replicate-padded interior field at (i, j) == interior value at the clamped index
      const int ci = min(max(gy, 1), H - 2), cj = min(max(gx, 1), W - 2);
      // the mean cancels in the differences; it is not subtracted (closer to the fp64 result)
      float uu = 0.5f * a_bound * (__ldg(yb + ((size_t)(ci + 1) * W + cj) * 4) - __ldg(yb + ((size_t)(ci - 1) * W + cj) * 4));
      float vv = -0.5f * a_bound * (__ldg(yb + ((size_t)ci * W + cj + 1) * 4) - __ldg(yb + ((size_t)ci * W + cj - 1) * 4));
      const bool xwall = (gx == 0 || gx == W - 1), ywall = (gy == 0 || gy == H - 1);
      if (xwall) uu = -uu;
      if (ywall) vv = -vv;
      if (xwall && ywall) { uu = 0.f; vv = 0.f; }
      uu *= sc;
      vv *= sc;
      u[o] = uu;
      v[o] = vv;
      if (p_pred && p) p[o] = __ldg(yb + ((size_t)gy * W + gx) * 4 + 1) - (float)(chan_sum[(size_t)b * 4 + 1] * inv_n);
      if (!xwall && !ywall) m = fmaxf(fabsf(uu), fabsf(vv));
    } else {
      const float4 yv = ldg4(yb + ((size_t)gy * W + gx) * 4);
      const float uu = (yv.x - (float)(chan_sum[(size_t)b * 4 + 0] * inv_n)) * sc;
      const float vv = (yv.y - (float)(chan_sum[(size_t)b * 4 + 1] * inv_n)) * sc;
      u[o] = uu;
      v[o] = vv;
      if (p_pred && p) p[o] = yv.z - (float)(chan_sum[(size_t)b * 4 + 2] * inv_n);
      if (gx > 0 && gx < W - 1 && gy > 0 && gy < H - 1) m = fmaxf(fabsf(uu), fabsf(vv));
    }
  }
  if (uvmax != nullptr) {
    __shared__ float red[8];
    m = warp_max(m);
    const int tid = threadIdx.y * 32 + threadIdx.x;
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    if (tid < 8) {
      float t = red[tid];
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) t = fmaxf(t, __shfl_xor_sync(0xffu, t, o));
      if (tid == 0) atomic_max_nonneg(uvmax + b, t);
    }
  }
}

int head_enqueue(const float* y, const double* chan_sum, const pbmc_member* members, float a_bound, int head_kind, int p_pred,
                 float* u, float* v, float* p, uint32_t* uvmax, int B, int H, int W, cudaStream_t st, bool pdl) {
  if (!y || !chan_sum || !u || !v) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;
  if (head_kind != PBMC_HEAD_CURL && head_kind != PBMC_HEAD_MAE) return PBMC_ERR_UNSUPPORTED;
  if (!aligned16(y)) return PBMC_ERR_MISALIGNED;
  dim3 grid(cdiv(W, 32), cdiv(H, 8), B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  PBMC_CUDA(launch_maybe_pdl(head_kernel, grid, dim3(32, 8), 0, st, pdl, y, chan_sum, members, a_bound, head_kind, p_pred, u, v, p,
                             uvmax, H, W));
  PBMC_CHECK_LAUNCH("head_kernel");
  return PBMC_OK;
}

}  // namespace pbmc

extern "C" int pbmc_head(const float* y, const double* chan_sum, const pbmc_member* members, float a_bound,
                         int head_kind, int p_pred, float* u, float* v, float* p, uint32_t* uvmax, int B, int H, int W,
                         void* stream) {
  return pbmc::head_enqueue(y, chan_sum, members, a_bound, head_kind, p_pred, u, v, p, uvmax, B, H, W, (cudaStream_t)stream, false);
}
