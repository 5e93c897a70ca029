// tcgen05 / TMEM implicit-GEMM convolution for sm_100a (the hot 16-channel-out shapes).
//
// Same contract as conv_ffma.cu (sources with fused GroupNorm+GELU on load, padding folded into
// the load coordinates, bias / GELU / GroupNorm statistics in the epilogue), restating
//   SymmetricConv2d.forward symmetric_layers_torch.py:113-138, nn.Conv2d heads
//   pytorch_networks_convae.py:1263-1309, FluidLayer :790-799, concat :1327/:1332,
// but the contraction runs on the 5th-generation tensor cores:
//
//   GEMM view      D[pixel, c_out] += A[pixel, (tap, c_in)] * B[(tap, c_in), c_out]
//   M = 128 pixels (one TMEM lane each), N = 16 output channels, K = 8 (tf32) per tcgen05.mma
//   A: the input tile (+halo) is staged ONCE in shared memory as channel-chunk planes
//      plane[chunk][pos] = 16 B (4 channels of one pixel), pos = row * PW + col of the halo tile.
//      This is the UMMA "K-major, no swizzle" canonical layout with 8-row groups 128 B apart
//      (SBO) and K chunks one plane apart (LBO), so the operand of filter tap (dy, dx) is the
//      SAME planes addressed at start + (dy * PW + dx) * 16 B: im2col is a descriptor offset,
//      no data is replicated.  An M-tile is a run of 128 consecutive positions; positions in
//      the halo columns compute junk rows that the epilogue discards (TW / PW efficiency).
//   B: packed filters [part][c_in block][tap][16 c_out][4 c_in] (hi / lo parts), K-major.
//   D: NMT accumulators of 16 columns each in TMEM; read back with tcgen05.ld 32x32b.x16.
//
// fp32-grade accuracy on tf32 tensor cores ("3xTF32"): a = a_hi + a_lo, b = b_hi + b_lo with
// hi = round-to-tf32, lo = exact remainder; D = a_hi b_hi + a_lo b_hi + a_hi b_lo (fp32 accumulate
// in TMEM).  The dropped a_lo b_lo term is ~2^-22 relative.  MODE 1 (single tf32 pass) is the
// fast / low-precision variant.
#include <cuda_bf16.h>
#include <stdlib.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc05.cuh"

namespace pbmc {

constexpr int CU_THREADS = 256;
constexpr int CU_STAGE = 4;  // channel blocks (4 channels each) per smem stage = 16 input channels

// Operand modes.  Every tcgen05.mma here reads a 128 x 32 B A-tile from shared memory for only
// N = 16 columns of math, so the instruction is shared-memory-read bound (~32 cycles at 128 B/clk,
// measured) and the number of MMAs per pixel is what matters:
//   TF32X3  a = tf32 hi + lo, 3 passes, K = 8 per MMA   -> 6 MMAs per 16 input channels per tap
//   F16X2   a = fp16 hi + lo, 3 passes, K = 16 per MMA  -> 3 MMAs (same ~2^-22 product error: 11+11 bits)
//   BF16    single bf16 pass, K = 16 per MMA            -> 1 MMA  (the stated-looser-bound variant)
enum { CU_TF32X3 = 0, CU_F16X2 = 1, CU_BF16 = 2 };
template <int MODE> struct UmmaMode;
template <> struct UmmaMode<CU_TF32X3> { static constexpr int PARTS = 2, BPC = 1; static constexpr uint32_t FMT = 2, KIND_F16 = 0; };
template <> struct UmmaMode<CU_F16X2> { static constexpr int PARTS = 2, BPC = 2; static constexpr uint32_t FMT = 0, KIND_F16 = 1; };
template <> struct UmmaMode<CU_BF16> { static constexpr int PARTS = 1, BPC = 2; static constexpr uint32_t FMT = 1, KIND_F16 = 1; };

struct ConvUmmaParams {
  pbmc_src src[PBMC_MAX_SRC];
  int nsrc, B, H, W;
  int cout_blks, cin_blks, pad_mode, epi_act;
  const void* wpk;  // [parts][cin chunks][taps][16 c_out][16 B of c_in]
  const float* wscale;  // 2^-e: the image holds the filters times 2^e (ops.prescale_pow2)
  const float* bias;
  float* out;
  double* out_stats;
  double* out_chan_sum;
};

template <int KS, int TW, int TH, int NMT, int MODE>
struct UmmaGeom {
  static constexpr int PARTS = UmmaMode<MODE>::PARTS, BPC = UmmaMode<MODE>::BPC;
  static constexpr int CPS = CU_STAGE / BPC;  // 16 B chunks per stage
  static constexpr int P = KS / 2;
  static constexpr int PW = TW + KS - 1;
  static constexpr int NPOS_IN = (TH + KS - 1) * PW;
  static constexpr int PLANE = ((NMT * 128 + (KS - 1) * PW + (KS - 1)) + 7) / 8 * 8;  // positions per plane (16 B each)
  static constexpr int TAPS = KS * KS;
  static constexpr int B_BYTES = PARTS * CPS * TAPS * 256;
  static constexpr int A_BYTES = PARTS * CPS * PLANE * 16;
  static_assert(TH * PW <= NMT * 128, "M-tiles do not cover the output tile");
  static_assert(NMT * 16 <= 512, "TMEM has 512 columns");
};

template <int KS, int TW, int TH, int NMT, int MODE>
__global__ void __launch_bounds__(CU_THREADS, (MODE == CU_TF32X3 ? 1 : (NMT <= 4 ? 3 : 2))) conv_umma_kernel(const ConvUmmaParams p) {
  using G = UmmaGeom<KS, TW, TH, NMT, MODE>;
  using MD = UmmaMode<MODE>;
  constexpr int PW = G::PW, PLANE = G::PLANE, TAPS = G::TAPS, P = G::P, PARTS = G::PARTS, BPC = G::BPC, CPS = G::CPS;
  constexpr uint32_t TMEM_COLS = NMT * 16 <= 32 ? 32 : (NMT * 16 <= 64 ? 64 : (NMT * 16 <= 128 ? 128 : (NMT * 16 <= 256 ? 256 : 512)));
  constexpr uint32_t IDESC = cu_idesc(MD::FMT);
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);                 // [0,8)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 8);       // [8,12)
  double* red = reinterpret_cast<double*>(smem + 16);                // 8 warps x 16 doubles = 1024 B
  uint4* Bs = reinterpret_cast<uint4*>(smem + 1152);                 // [PARTS][CPS][TAPS][16 rows] x 16 B
  uint4* As = reinterpret_cast<uint4*>(smem + 1152 + G::B_BYTES);    // [PARTS][CPS][PLANE] x 16 B
  float* xf_a = reinterpret_cast<float*>(smem + 1152 + G::B_BYTES + G::A_BYTES);
  float* xf_b = xf_a + p.cin_blks * 4;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const int H = p.H, W = p.W;
  const size_t plane_px = (size_t)H * W;

  // ---- one-time setup: mbarrier, TMEM, GroupNorm coefficients, zero the never-loaded slack
  if (tid == 0) {
    mbar_init(smem_u32(bar), 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), TMEM_COLS);
  {
    int c0 = 0;
    for (int s = 0; s < p.nsrc; ++s) {
      const pbmc_src& S = p.src[s];
      for (int c = tid; c < S.nblk * 4; c += CU_THREADS) {
        float a = 1.f, bb = 0.f;
        if (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN)
          gn_coeffs(S.stats + ((size_t)b * S.nblk + (c >> 2)) * 2, S.inv_count, S.gamma[c], S.beta[c], a, bb);
        xf_a[c0 + c] = a;
        xf_b[c0 + c] = bb;
      }
      c0 += S.nblk * 4;
    }
  }
  for (int e = tid; e < PARTS * CPS * (PLANE - G::NPOS_IN); e += CU_THREADS) {
    const int pl = e / (PLANE - G::NPOS_IN), o = e % (PLANE - G::NPOS_IN);
    As[pl * PLANE + G::NPOS_IN + o] = make_uint4(0u, 0u, 0u, 0u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t a_base = smem_u32(As), b_base = smem_u32(Bs), bar_addr = smem_u32(bar);

  uint32_t n_commits = 0;
  int gblk0 = 0;
  for (int s = 0; s < p.nsrc; ++s) {
    const pbmc_src S = p.src[s];
    for (int cb = 0; cb < S.nblk; cb += CU_STAGE) {
      const int nb = min(CU_STAGE, S.nblk - cb);  // even (checked on the host)
      const int nch = (nb + BPC - 1) / BPC;       // real 16 B chunks in this stage
      const int nks = (nch + 1) / 2;              // K-steps (a K-step is two chunks; an odd tail chunk is zero-padded)
      if (n_commits > 0) {  // the previous stage's MMAs must have finished reading smem
        mbar_wait(bar_addr, (n_commits - 1) & 1);
        tc_fence_after();
      }
      // ---- A: input tile (+halo), transform + padding folded in, converted to the operand format
      const int nchp = 2 * nks;  // chunks written (incl. a zero pad chunk)
      constexpr int ITERS = (G::NPOS_IN + CU_THREADS - 1) / CU_THREADS;
      for (int ch = 0; ch < nchp; ++ch) {
        // all global loads of this chunk are issued before any of the (long) transform math
        float4 raw[ITERS][BPC];
        uint32_t valid = 0;
#pragma unroll
        for (int it = 0; it < ITERS; ++it) {
          const int pos = tid + it * CU_THREADS;
          const int r = pos / PW, c = pos % PW;
          const int sy = pad_index(y0 + r - P, H, p.pad_mode);
          const int sx = pad_index(x0 + c - P, W, p.pad_mode);
          const bool ok = pos < G::NPOS_IN && sy >= 0 && sx >= 0 && ch < nch;
          valid |= (ok ? 1u : 0u) << it;
#pragma unroll
          for (int j = 0; j < BPC; ++j) {
            raw[it][j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok) raw[it][j] = ldg4(S.ptr + (((size_t)b * S.nblk + cb + ch * BPC + j) * plane_px + (size_t)sy * W + sx) * 4);
          }
        }
#pragma unroll
        for (int it = 0; it < ITERS; ++it) {
          const int pos = tid + it * CU_THREADS;
          if (pos >= G::NPOS_IN) break;
          float v[4 * BPC];
#pragma unroll
          for (int j = 0; j < BPC; ++j) {
            float4 t = raw[it][j];
            if ((valid >> it) & 1u) {
              const int chn = (gblk0 + cb + ch * BPC + j) * 4;
              t = xform4(t, xf_a + chn, xf_b + chn, S.xform);
            }
            v[4 * j + 0] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
          }
          if (MODE == CU_TF32X3) {
            float h[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) h[q] = tf32_rna(v[q]);
            As[ch * PLANE + pos] = make_uint4(__float_as_uint(h[0]), __float_as_uint(h[1]), __float_as_uint(h[2]), __float_as_uint(h[3]));
            As[(CPS + ch) * PLANE + pos] = make_uint4(__float_as_uint(v[0] - h[0]), __float_as_uint(v[1] - h[1]),
                                                      __float_as_uint(v[2] - h[2]), __float_as_uint(v[3] - h[3]));
          } else if (MODE == CU_F16X2) {
            uint4 hi, lo;
            split_f16(v, hi, lo);
            As[ch * PLANE + pos] = hi;
            As[(CPS + ch) * PLANE + pos] = lo;
          } else {
            As[ch * PLANE + pos] = pack_bf16(v);
          }
        }
      }
      // ---- B: [part][chunk][tap][16 rows] for this stage (zero chunk if the K-step is padded)
      {
        const int gch0 = (gblk0 + cb) / BPC;           // first global chunk of the stage
        const int tot_ch = p.cin_blks / BPC;           // chunks per part in the packed image
        for (int e = tid; e < PARTS * nchp * TAPS * 16; e += CU_THREADS) {
          const int part = e / (nchp * TAPS * 16), rem = e % (nchp * TAPS * 16);
          const int ch = rem / (TAPS * 16), o = rem % (TAPS * 16);
          uint4 w = make_uint4(0u, 0u, 0u, 0u);
          if (ch < nch) w = __ldg(reinterpret_cast<const uint4*>(p.wpk) + ((size_t)part * tot_ch + gch0 + ch) * (TAPS * 16) + o);
          Bs[(part * CPS + ch) * (TAPS * 16) + o] = w;
        }
      }
      fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      __syncthreads();
      // ---- MMA issue: one thread; im2col == descriptor start offset.  M-tiles are the INNER loop so
      // consecutive MMAs hit different accumulators (no back-to-back dependent accumulation).
      if (tid == 0) {
        tc_fence_after();
        constexpr uint32_t A_LBO = PLANE * 16, B_LBO = TAPS * 256, SBO = 128;
        constexpr uint32_t A_PART = CPS * PLANE * 16, B_PART = CPS * TAPS * 256;
        const bool first_stage = (n_commits == 0);
        for (int t = 0; t < TAPS; ++t) {
          const int dy = t / KS, dx = t % KS;
          for (int ks = 0; ks < nks; ++ks) {
            const uint32_t a_tap = a_base + (uint32_t)(2 * ks) * A_LBO + (uint32_t)(dy * PW + dx) * 16;
            const uint32_t b_hi = b_base + (uint32_t)((2 * ks) * TAPS + t) * 256;
            const uint64_t bd_hi = umma_desc(b_hi, B_LBO, SBO), bd_lo = umma_desc(b_hi + B_PART, B_LBO, SBO);
            const uint32_t acc0 = (first_stage && t == 0 && ks == 0) ? 0u : 1u;
#pragma unroll
            for (int m = 0; m < NMT; ++m)
              umma_ss<MD::KIND_F16>(tmem_base + (uint32_t)m * 16, umma_desc(a_tap + (uint32_t)m * 2048, A_LBO, SBO), bd_hi, IDESC, acc0);
            if (PARTS == 2) {
#pragma unroll
              for (int m = 0; m < NMT; ++m)
                umma_ss<MD::KIND_F16>(tmem_base + (uint32_t)m * 16, umma_desc(a_tap + A_PART + (uint32_t)m * 2048, A_LBO, SBO), bd_hi,
                                      IDESC, 1u);
#pragma unroll
              for (int m = 0; m < NMT; ++m)
                umma_ss<MD::KIND_F16>(tmem_base + (uint32_t)m * 16, umma_desc(a_tap + (uint32_t)m * 2048, A_LBO, SBO), bd_lo, IDESC, 1u);
            }
          }
        }
        umma_commit(bar_addr);  // implies tcgen05.fence::before_thread_sync
      }
      ++n_commits;
    }
    gblk0 += S.nblk;
  }
  mbar_wait(bar_addr, (n_commits - 1) & 1);
  tc_fence_after();

  // ---- epilogue: TMEM -> registers, bias / activation, coalesced float4 stores, statistics
  const int lg = warp & 3, wg = warp >> 2;
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f}, cs[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) cs[c] = 0.f;
  float bias[16];
  const float wsc = __ldg(p.wscale);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q < p.cout_blks) bq = ldg4(p.bias + q * 4);
    bias[q * 4 + 0] = bq.x; bias[q * 4 + 1] = bq.y; bias[q * 4 + 2] = bq.z; bias[q * 4 + 3] = bq.w;
  }
  for (int m = wg; m < NMT; m += 2) {
    float v[16];
    tmem_ld16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)m * 16, v);
    const int q = m * 128 + lg * 32 + lane;
    const int r = q / PW, c = q % PW;
    const int gy = y0 + r, gx = x0 + c;
    if (r < TH && c < TW && gy < H && gx < W) {
#pragma unroll
      for (int qb = 0; qb < 4; ++qb) {
        if (qb < p.cout_blks) {
          float4 o = make_float4(fmaf(v[qb * 4 + 0], wsc, bias[qb * 4 + 0]), fmaf(v[qb * 4 + 1], wsc, bias[qb * 4 + 1]),
                                 fmaf(v[qb * 4 + 2], wsc, bias[qb * 4 + 2]), fmaf(v[qb * 4 + 3], wsc, bias[qb * 4 + 3]));
          if (p.epi_act == PBMC_ACT_GELU) {
            o.x = gelu_erf(o.x); o.y = gelu_erf(o.y); o.z = gelu_erf(o.z); o.w = gelu_erf(o.w);
          }
          *reinterpret_cast<float4*>(p.out + (((size_t)b * p.cout_blks + qb) * plane_px + (size_t)gy * W + gx) * 4) = o;
          s1[qb] += (o.x + o.y) + (o.z + o.w);
          s2[qb] += (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
          cs[qb * 4 + 0] += o.x; cs[qb * 4 + 1] += o.y; cs[qb * 4 + 2] += o.z; cs[qb * 4 + 3] += o.w;
        }
      }
    }
  }
  constexpr int NWARP = CU_THREADS / 32;
  if (p.out_stats != nullptr) {
#pragma unroll
    for (int qb = 0; qb < 4; ++qb) {
      const double a = warp_sum((double)s1[qb]);
      const double c2 = warp_sum((double)s2[qb]);
      if (lane == 0) { red[(warp * 4 + qb) * 2] = a; red[(warp * 4 + qb) * 2 + 1] = c2; }
    }
    __syncthreads();
    if (tid < 8 && (tid >> 1) < p.cout_blks) {
      double t = 0.0;
      for (int w = 0; w < NWARP; ++w) t += red[(w * 4 + (tid >> 1)) * 2 + (tid & 1)];
      atomicAdd(p.out_stats + ((size_t)b * p.cout_blks + (tid >> 1)) * 2 + (tid & 1), t);
    }
    __syncthreads();
  }
  if (p.out_chan_sum != nullptr) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const double a = warp_sum((double)cs[c]);
      if (lane == 0) red[warp * 16 + c] = a;
    }
    __syncthreads();
    if (tid < p.cout_blks * 4) {
      double t = 0.0;
      for (int w = 0; w < NWARP; ++w) t += red[w * 16 + tid];
      atomicAdd(p.out_chan_sum + (size_t)b * p.cout_blks * 4 + tid, t);
    }
  }
  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int KS, int TW, int TH, int NMT, int MODE>
static int launch_umma(const ConvUmmaParams& p, cudaStream_t st) {
  using G = UmmaGeom<KS, TW, TH, NMT, MODE>;
  const size_t smem = 1152 + G::B_BYTES + G::A_BYTES + (size_t)p.cin_blks * 8 * sizeof(float);
  if (smem > 227 * 1024) return PBMC_ERR_UNSUPPORTED;
  static bool attr_set = false;
  if (!attr_set) {
    PBMC_CUDA(cudaFuncSetAttribute(conv_umma_kernel<KS, TW, TH, NMT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid(cdiv(p.W, TW), cdiv(p.H, TH), p.B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  conv_umma_kernel<KS, TW, TH, NMT, MODE><<<grid, CU_THREADS, smem, st>>>(p);
  PBMC_CHECK_LAUNCH("conv_umma_kernel");
  return PBMC_OK;
}

bool conv_umma_supported(const pbmc_conv_desc& d) {
  if (d.ksize != 3 && d.ksize != 5) return false;
  if (d.cout > 16) return false;
  for (int s = 0; s < d.nsrc; ++s)
    if (d.src[s].nblk % 2 != 0) return false;  // operand chunks / K-steps pair 4-channel blocks
  return true;
}

int conv_umma_dispatch(const pbmc_conv_desc& d, cudaStream_t st) {
  ConvUmmaParams p;
  int cin = 0;
  for (int s = 0; s < d.nsrc; ++s) {
    p.src[s] = d.src[s];
    cin += d.src[s].nblk;
  }
  p.nsrc = d.nsrc; p.B = d.B; p.H = d.H; p.W = d.W;
  p.cout_blks = (d.cout + 3) / 4;
  p.cin_blks = cin;
  p.pad_mode = d.pad_mode; p.epi_act = d.epi_act;
  p.bias = d.bias; p.out = d.out; p.out_stats = d.out_stats; p.out_chan_sum = d.out_chan_sum;
  // wpk_umma holds three operand images back to back (see ops.pack_conv_weight_umma), then the prescale tail:
  //   [tf32 hi|lo : 2*cin*taps*256 B][fp16 hi|lo : cin/2*taps*512 B][bf16 : cin/2*taps*256 B][float 2^-e, 0, 0, 0]
  const size_t taps = (size_t)d.ksize * d.ksize;
  const char* base = reinterpret_cast<const char*>(d.wpk_umma);
  if (!aligned16(base)) return PBMC_ERR_MISALIGNED;
  const size_t off_f16 = 2 * (size_t)cin * taps * 256, off_bf16 = off_f16 + (size_t)(cin / 2) * taps * 512;
  p.wscale = reinterpret_cast<const float*>(base + off_bf16 + (size_t)(cin / 2) * taps * 256);
  if (d.impl == PBMC_CONV_UMMA_3XTF32) {
    p.wpk = base;
    return d.ksize == 3 ? launch_umma<3, 64, 15, 8, CU_TF32X3>(p, st) : launch_umma<5, 64, 15, 8, CU_TF32X3>(p, st);
  }
  if (d.impl == PBMC_CONV_UMMA_F16X2) {
    p.wpk = base + off_f16;
    return d.ksize == 3 ? launch_umma<3, 64, 15, 8, CU_F16X2>(p, st) : launch_umma<5, 64, 15, 8, CU_F16X2>(p, st);
  }
  if (d.impl == PBMC_CONV_UMMA_BF16) {
    p.wpk = base + off_bf16;
    return d.ksize == 3 ? launch_umma<3, 64, 15, 8, CU_BF16>(p, st) : launch_umma<5, 64, 15, 8, CU_BF16>(p, st);
  }
  return PBMC_ERR_UNSUPPORTED;
}

}  // namespace pbmc
