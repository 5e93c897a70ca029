// A4: the eight boundary regions of BoundaryLearnedConvolution2D (pytorch_networks_convae.py:1022-1065), one launch.
//
// The reference computes nine bias-free VALID convolutions with separate weights (interior, 4 edge strips of
// pad = k rows/columns for k = 3, k + 1 for k = 5, 4 corners) and stitches them with torch.cat.  Seen from one output
// pixel (i, j) of the H x W result (p = (k-1)/2) that is a single k x k window whose POSITION and WEIGHT SET depend on
// the pixel's row class and column class:
//   rows   i <  p      "bottom" weights, window rows  H - pad + i ..          (the strip computed from the LAST input
//                                                                             rows lands at output row 0, :1060)
//          i >= H - p  "top" weights,    window rows  i - (H - p) ..
//          else        centre,           window rows  i - p ..
//   cols   j <  p      "left",           window cols  j ..
//          j >= W - p  "right",          window cols  (W - pad) + j - (W - p) ..
//          else        centre,           window cols  j - p ..
// The (centre, centre) pixels are an ordinary 'same' convolution restricted to outputs whose window stays inside the
// image: pbmc_conv_fwd (tensor cores, any padding mode) computes them for the WHOLE image first.  This kernel then
// overwrites the ring of width p with the eight edge / corner regions -- and repairs the statistics the first kernel
// accumulated over its (wrong) ring values: every ring pixel subtracts its old value's contribution to the GroupNorm
// sums / channel sums and adds the new one.  Two launches per layer instead of nine convs + three cats + a reduction.
//
// Work: 2p(W + H - 2p) pixels x k^2 C_in C_out MACs -- 0.5 % of the layer at 128 x 506 -- so plain FFMA: a CTA takes 8
// ring pixels; per source it stages the pixels' windows in shared memory with the producer's GroupNorm + GELU applied
// (once per tap, not once per MAC), then thread (pixel, c_out) accumulates over taps and input channels; filters come
// from L2 as 128-bit loads of 4 input channels, contiguous across the 16 c_out lanes.
#include "common.cuh"

namespace pbmc {

constexpr int E9_PX = 8;          // ring pixels per CTA
constexpr int E9_THREADS = E9_PX * 16;
constexpr int E9_MAXC = 128;      // channels per source (32 blocks); wider sources are split by the caller

struct Edge9Params {
  pbmc_src src[PBMC_MAX_SRC];
  int nsrc, B, H, W, cout_blks, k, epi_act, cin_blks;
  const float* wedge;   // [8 regions][cin_blks][k*k][16 c_out][4 c_in]
  const float* bias;    // [16] (zero padded)
  float* out;           // [B][cout_blks][H][W][4]
  double* out_stats;    // [B][cout_blks][2] or NULL
  double* out_chan_sum; // [B][cout_blks*4] or NULL
};

// region index in `wedge`: 0 top_left, 1 top_right, 2 bottom_left, 3 bottom_right, 4 top, 5 bottom, 6 left, 7 right
// ("top" = the reference's name: weights applied to the FIRST input rows, whose result lands in the LAST output rows)
__device__ __forceinline__ int edge9_region(int rowc, int colc) {  // class: 0 low index, 1 centre, 2 high index
  // rowc 0 (output rows < p) uses the LAST input rows = "bottom"; rowc 2 uses the FIRST = "top"
  if (rowc == 0) return colc == 0 ? 2 : (colc == 2 ? 3 : 5);
  if (rowc == 2) return colc == 0 ? 0 : (colc == 2 ? 1 : 4);
  return colc == 0 ? 6 : 7;
}

__global__ void __launch_bounds__(E9_THREADS) conv_edge9_kernel(const __grid_constant__ Edge9Params p) {
  extern __shared__ __align__(16) float win[];  // [E9_PX][k*k][16] transformed window values of the current source
  __shared__ float xa[PBMC_MAX_SRC][E9_MAXC], xb[PBMC_MAX_SRC][E9_MAXC];
  __shared__ double red[E9_THREADS / 32][4][3];
  const int tid = threadIdx.x, px = tid >> 4, co = tid & 15;
  const int b = blockIdx.y;
  const int H = p.H, W = p.W, k = p.k, pd = (k - 1) / 2, pad = k == 5 ? k + 1 : k, kk = k * k;
  const long ring = 2L * pd * W + 2L * pd * (H - 2 * pd);
  const size_t plane = (size_t)H * W;
  // programmatic dependent launch (no-ops otherwise): everything below reads what the interior conv (or earlier) wrote;
  // the next kernel of the chain does its own griddepcontrol.wait before it reads this kernel's output
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // GroupNorm coefficients of every transformed source
  for (int e = tid; e < p.nsrc * E9_MAXC; e += E9_THREADS) {
    const int s = e / E9_MAXC, c = e % E9_MAXC;
    const pbmc_src& S = p.src[s];
    float a = 1.f, bb = 0.f;
    if (s < p.nsrc && (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN) && c < S.nblk * 4)
      gn_coeffs(S.stats + ((size_t)b * S.nblk + (c >> 2)) * 2, S.inv_count, S.gamma[c], S.beta[c], a, bb);
    xa[s][c] = a;
    xb[s][c] = bb;
  }

  // this thread's ring pixel: output position, window origin, weight set
  const long q = (long)blockIdx.x * E9_PX + px;
  const bool on = q < ring;
  int i = 0, j = 0;
  if (on) {
    if (q < (long)pd * W) { i = (int)(q / W); j = (int)(q % W); }
    else if (q < 2L * pd * W) { const long r = q - (long)pd * W; i = H - pd + (int)(r / W); j = (int)(r % W); }
    else { const long r = q - 2L * pd * W; i = pd + (int)(r / (2 * pd)); const int jj = (int)(r % (2 * pd)); j = jj < pd ? jj : W - 2 * pd + jj; }
  }
  const int rowc = i < pd ? 0 : (i >= H - pd ? 2 : 1), colc = j < pd ? 0 : (j >= W - pd ? 2 : 1);
  const int r0 = rowc == 0 ? H - pad + i : (rowc == 2 ? i - (H - pd) : i - pd);
  const int c0 = colc == 0 ? j : (colc == 2 ? (W - pad) + j - (W - pd) : j - pd);
  const int region = edge9_region(rowc, colc);
  __syncthreads();

  float acc = 0.f;
  int cb0 = 0;  // channel-block offset of the current 16-channel chunk in the concatenation
  for (int s = 0; s < p.nsrc; ++s) {
    const pbmc_src& S = p.src[s];
    for (int c4 = 0; c4 < S.nblk; c4 += 4) {  // 16-channel chunks of the source
      const int nb = min(4, S.nblk - c4);
      // ---- stage: every (pixel, tap, block) of this chunk, producer transform applied
      for (int e = tid; e < E9_PX * kk * nb; e += E9_THREADS) {
        const int blk = e % nb, t = (e / nb) % kk, pp = e / (nb * kk);
        // window origin of pixel pp: recomputed from its ring index (cheap integer work, no shared table)
        const long qq = (long)blockIdx.x * E9_PX + pp;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (qq < ring) {
          int ii, jj2;
          if (qq < (long)pd * W) { ii = (int)(qq / W); jj2 = (int)(qq % W); }
          else if (qq < 2L * pd * W) { const long r = qq - (long)pd * W; ii = H - pd + (int)(r / W); jj2 = (int)(r % W); }
          else { const long r = qq - 2L * pd * W; ii = pd + (int)(r / (2 * pd)); const int j3 = (int)(r % (2 * pd)); jj2 = j3 < pd ? j3 : W - 2 * pd + j3; }
          const int rc = ii < pd ? 0 : (ii >= H - pd ? 2 : 1), cc = jj2 < pd ? 0 : (jj2 >= W - pd ? 2 : 1);
          const int rr0 = rc == 0 ? H - pad + ii : (rc == 2 ? ii - (H - pd) : ii - pd);
          const int cc0 = cc == 0 ? jj2 : (cc == 2 ? (W - pad) + jj2 - (W - pd) : jj2 - pd);
          const int y = rr0 + t / k, x = cc0 + t % k;
          v = ldg4(S.ptr + (((size_t)b * S.nblk + c4 + blk) * plane + (size_t)y * W + x) * 4);
          v = xform4(v, &xa[s][(c4 + blk) * 4], &xb[s][(c4 + blk) * 4], S.xform);
        }
        *reinterpret_cast<float4*>(win + ((size_t)pp * kk + t) * 16 + blk * 4) = v;
      }
      __syncthreads();
      // ---- accumulate: thread (pixel, c_out) over taps x input channels of this chunk
      if (on) {
        const float* wr = p.wedge + ((size_t)region * p.cin_blks + cb0) * kk * 64 + co * 4;
        const float* wp = win + (size_t)px * kk * 16;
        for (int blk = 0; blk < nb; ++blk) {
#pragma unroll 5
          for (int t = 0; t < kk; ++t) {
            const float4 w4 = ldg4(wr + ((size_t)blk * kk + t) * 64);
            const float4 a4 = *reinterpret_cast<const float4*>(wp + t * 16 + blk * 4);
            acc = fmaf(a4.x, w4.x, acc);
            acc = fmaf(a4.y, w4.y, acc);
            acc = fmaf(a4.z, w4.z, acc);
            acc = fmaf(a4.w, w4.w, acc);
          }
        }
      }
      __syncthreads();
      cb0 += nb;
    }
  }

  // ---- write the ring pixel, repair the statistics (old value out, new value in)
  double d1 = 0.0, d2 = 0.0;
  const bool cw = on && co < p.cout_blks * 4;
  if (cw) {
    float o = acc + __ldg(p.bias + co);
    if (p.epi_act == PBMC_ACT_GELU) o = gelu_erf(o);
    float* dst = p.out + (((size_t)b * p.cout_blks + (co >> 2)) * plane + (size_t)i * W + j) * 4 + (co & 3);
    const float old = *dst;
    *dst = o;
    d1 = (double)o - (double)old;
    d2 = (double)o * (double)o - (double)old * (double)old;
  }
  if (p.out_stats != nullptr || p.out_chan_sum != nullptr) {
    // a warp = 2 pixels x 16 c_out: channel sums over the 2 pixels, block sums also over the 4 channels of a block
    double c1 = d1 + __shfl_xor_sync(0xffffffffu, d1, 16);
    double b1 = c1, b2 = d2 + __shfl_xor_sync(0xffffffffu, d2, 16);
    b1 += __shfl_xor_sync(0xffffffffu, b1, 1); b1 += __shfl_xor_sync(0xffffffffu, b1, 2);
    b2 += __shfl_xor_sync(0xffffffffu, b2, 1); b2 += __shfl_xor_sync(0xffffffffu, b2, 2);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane < 16 && (lane & 3) == 0) { red[warp][lane >> 2][0] = b1; red[warp][lane >> 2][1] = b2; }
    if (p.out_chan_sum != nullptr && lane < 4 && lane < p.cout_blks * 4) red[warp][lane][2] = c1;  // head conv: c_out <= 4
    __syncthreads();
    if (tid < 8 && (tid >> 1) < p.cout_blks && p.out_stats != nullptr) {
      double t = 0.0;
      for (int w = 0; w < E9_THREADS / 32; ++w) t += red[w][tid >> 1][tid & 1];
      if (t != 0.0) atomicAdd(p.out_stats + ((size_t)b * p.cout_blks + (tid >> 1)) * 2 + (tid & 1), t);
    }
    if (p.out_chan_sum != nullptr && tid >= 32 && tid < 36 && tid - 32 < p.cout_blks * 4) {
      double t = 0.0;
      for (int w = 0; w < E9_THREADS / 32; ++w) t += red[w][tid - 32][2];
      if (t != 0.0) atomicAdd(p.out_chan_sum + (size_t)b * p.cout_blks * 4 + (tid - 32), t);
    }
  }
}

}  // namespace pbmc

using namespace pbmc;

extern "C" int pbmc_conv_edge9(const pbmc_edge9_desc* d, void* stream) {
  if (!d) return PBMC_ERR_NULL_POINTER;
  if (d->nsrc <= 0 || d->nsrc > PBMC_MAX_SRC || d->B <= 0 || d->cout <= 0) return PBMC_ERR_BAD_SHAPE;
  if (d->ksize != 3 && d->ksize != 5) return PBMC_ERR_UNSUPPORTED;
  if (d->cout > 16) return PBMC_ERR_UNSUPPORTED;  // one 16-wide c_out tile (all the surrogate's learned layers)
  const int pad = d->ksize == 5 ? 6 : 3;
  if (d->H < pad || d->W < pad) return PBMC_ERR_BAD_SHAPE;  // the reference's strips would overlap
  if (!d->wedge || !d->bias || !d->out) return PBMC_ERR_NULL_POINTER;
  if (!aligned16(d->wedge) || !aligned16(d->out)) return PBMC_ERR_MISALIGNED;
  if (d->out_chan_sum != nullptr && d->cout > 4) return PBMC_ERR_UNSUPPORTED;
  Edge9Params p;
  int cin_blks = 0;
  for (int s = 0; s < d->nsrc; ++s) {
    const pbmc_src& S = d->src[s];
    if (!S.ptr) return PBMC_ERR_NULL_POINTER;
    if (!aligned16(S.ptr)) return PBMC_ERR_MISALIGNED;
    if (S.nblk <= 0 || S.nblk * 4 > E9_MAXC || S.layout != PBMC_LAYOUT_BLOCKED) return PBMC_ERR_UNSUPPORTED;
    if (S.xform < PBMC_XFORM_NONE || S.xform > PBMC_XFORM_GELU) return PBMC_ERR_UNSUPPORTED;
    if ((S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN) && (!S.stats || !S.gamma || !S.beta)) return PBMC_ERR_NULL_POINTER;
    p.src[s] = S;
    cin_blks += S.nblk;
  }
  p.nsrc = d->nsrc; p.B = d->B; p.H = d->H; p.W = d->W; p.cout_blks = (d->cout + 3) / 4; p.k = d->ksize; p.epi_act = d->epi_act;
  p.cin_blks = cin_blks;
  p.wedge = d->wedge; p.bias = d->bias; p.out = d->out; p.out_stats = d->out_stats; p.out_chan_sum = d->out_chan_sum;
  const int pd = (d->ksize - 1) / 2;
  const long ring = 2L * pd * d->W + 2L * pd * (d->H - 2 * pd);
  const size_t smem = (size_t)E9_PX * d->ksize * d->ksize * 16 * sizeof(float);
  dim3 grid((unsigned)((ring + E9_PX - 1) / E9_PX), d->B);
  if (grid.y > 65535) return PBMC_ERR_BAD_SHAPE;
  conv_edge9_kernel<<<grid, E9_THREADS, smem, (cudaStream_t)stream>>>(p);
  PBMC_CHECK_LAUNCH("conv_edge9_kernel");
  return PBMC_OK;
}
