// Time-multiplexed row-streaming tcgen05 / TMEM convolution for sm_100a ("mux"): the single-group
// (c_in <= 16), 3x3 convs of the surrogate -- every trunk FluidLayer, conv[0], conv[2], conv[3]: 27 of
// the 28 convs of a forward.  Same operator contract and the same GEMM view as conv_row.cu
//   SymmetricConv2d.forward symmetric_layers_torch.py:113-138, nn.Conv2d heads
//   pytorch_networks_convae.py:1263-1309, FluidLayer :790-799
//   M = 128 output columns, N = 48 = (dy, c_out), K = 16 input channels, one accumulator D_r per INPUT row,
//   out[y][x][co] = bias + sum_dy D_{y+dy}[x][(dy, co)]
// but a different execution plan.  conv_row.cu dedicates warps to roles (12 producer, 8 epilogue) and
// pipelines them through an 8-stage ring; its in-kernel timelines (tools/rowtrace.py) show every role
// latency-bound on its own serial chain (a producer group needs ~3500 clk per row: GroupNorm+GELU, fp16
// hi/lo split, STS, proxy fence, barrier), ~5000 clk of ramp on either side of only 16 stages, and the
// issue slots 35 % busy.  Here the warps are NOT specialised:
//   phase 1  all 20 worker warps are producers.  Five groups of 4 warps each take TWO consecutive input
//            rows at a time (one thread = one column of both rows: twice the instruction-level parallelism,
//            one fence + barrier round per two rows) and stage them as fp16 hi|lo K-major planes.  ALL input
//            rows of the CTA stay resident in shared memory (<= 24 rows x 8.5 KB): no ring, no back-pressure.
//   MMA      one warp issues the 9 tcgen05.mma of a row as soon as that row is staged (tensor pipe is
//            asynchronous: it overlaps phase 1), accumulating into a ring of 10 TMEM accumulators.
//   phase 2  the same 20 warps become five epilogue sets (TMEM lane quarter = warp & 3), set e takes output
//            rows e, e+5, ...: 3 TMEM loads, bias (+GELU), store, GroupNorm / zero-mean partial sums.
// A group that runs out of input rows starts on the epilogue while the others still produce.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "tc05.cuh"

namespace pbmc {

constexpr int CM_SETS = 5;                         // groups of 4 warps
constexpr int CM_WORKERS = 4 * CM_SETS;            // 20 worker warps
constexpr int CM_NMMA = 2;
constexpr int CM_MMA_WARP = CM_WORKERS;            // + the MMA issuers (row ri by issuer ri % CM_NMMA; the first one owns TMEM)
constexpr int CM_THREADS = (CM_WORKERS + CM_NMMA) * 32;
constexpr int CM_MAXR = 24;                        // input rows per CTA (all resident in shared memory)
constexpr int CM_ND = 10;                          // TMEM accumulator ring
constexpr int CM_N = 48;                           // (dy, c_out)
constexpr int CM_PLANE = 136;                      // positions per K-chunk plane (128 + 2 halo, rounded up to 8)
constexpr int CM_HDR = 2048;
// registers are granted to a CTA in units of 4 warps: 22 warps count as 24 -> 80 per thread
constexpr int CM_MAXNREG = 80;

struct ConvMuxParams {
  const float* in;      // [B][nblk][H][W][4]
  const double* stats;  // producer's GroupNorm sums (xform != NONE)
  const float* gamma;
  const float* beta;
  double inv_count;
  int nblk, xform;
  int B, H, W;
  int cout_blks, pad_mode, epi_act;
  int rpc;           // output rows per CTA (<= CM_MAXR - 2)
  const void* wpk;   // [dx][part][2 K-chunks][48 rows (dy, c_out)][8 c_in] 16-bit
  const float* wscale;  // 2^-e: the image holds the filters times 2^e (ops.prescale_pow2)
  const float* bias;
  float* out;
  double* out_stats;
  double* out_chan_sum;
  unsigned long long* trace;  // developer timeline (PBMC_ROW_TRACE builds only), else NULL
};

#ifdef PBMC_ROW_TRACE
#define CM_TR(slot)                                                                                  \
  do {                                                                                               \
    if (p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (slot) < 4096) \
      p.trace[(slot)] = clock64();                                                                   \
  } while (0)
#else
#define CM_TR(slot) \
  do {              \
  } while (0)
#endif

__device__ __forceinline__ void cm_worker_bar() { asm volatile("bar.sync 1, %0;" ::"n"(CM_WORKERS * 32) : "memory"); }

template <int PARTS>
__global__ void __maxnreg__(CM_MAXNREG) conv_mux_kernel(const __grid_constant__ ConvMuxParams p) {
  constexpr int KS = 3, P = 1, N = CM_N, ND = CM_ND, PLANE = CM_PLANE;
  constexpr int PART_BYTES = 2 * PLANE * 16, STAGE_BYTES = PARTS * PART_BYTES;
  constexpr int B_TILE = 2 * N * 16, B_GROUP = KS * PARTS * B_TILE;
  constexpr uint32_t FMT = PARTS == 2 ? 0u : 1u;  // fp16 hi|lo split, or one bf16 pass
  constexpr uint32_t IDESC = row_idesc(FMT, N);
  static_assert(8 * (CM_MAXR + 2 * ND) <= 448, "barrier area");
  static_assert(ND * N <= 512, "TMEM has 512 columns");
  extern __shared__ __align__(128) unsigned char smem[];
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 448);
  double* red = reinterpret_cast<double*>(smem + 512);        // 20 warps x 8 doubles
  float* bias_s = reinterpret_cast<float*>(smem + 1792);      // 16 floats (zero padded)
  float* xf_a = reinterpret_cast<float*>(smem + 1856);        // GroupNorm scale / shift of the 16 input channels
  float* xf_b = reinterpret_cast<float*>(smem + 1920);
  float* wsc_s = reinterpret_cast<float*>(smem + 1984);       // epilogue factor 2^-e (times 2^s for a SCALE source)
  unsigned char* Bs = smem + CM_HDR;
  unsigned char* As = Bs + B_GROUP;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z;
  const int x0 = blockIdx.y * 128;
  const int y0 = blockIdx.x * p.rpc;
  const int H = p.H, W = p.W;
  const int nrows = min(p.rpc, H - y0);
  const int nin = nrows + KS - 1;
  const int nb = min(p.nblk, 4);
  const size_t plane_px = (size_t)H * W;
  const uint32_t bar0 = smem_u32(smem);
  auto a_full = [&](uint32_t r) { return bar0 + r * 8u; };
  auto d_full = [&](uint32_t d) { return bar0 + (uint32_t)(CM_MAXR + d) * 8u; };
  auto d_empty = [&](uint32_t d) { return bar0 + (uint32_t)(CM_MAXR + ND + d) * 8u; };

  // ---- worker geometry (needed before the set-up barrier: the first rows are requested right away)
  const int g = warp >> 2, wq = warp & 3;
  const int i = wq * 32 + lane;  // position in the staged row = input column x0 - 1 + i
  const int gxp = x0 - P + i;
  const int sx = pad_index(gxp, W, p.pad_mode);
  const bool col_ok = gxp < W + P && sx >= 0;  // columns past the image feed masked outputs only
  const int hch = lane & 15, he = lane >> 4;   // halo positions 128, 129: warp 0 of a group, lane = (position, channel)
  const int gxh = x0 - P + 128 + he;
  const int hsx = pad_index(gxh, W, p.pad_mode);
  const bool h_on = warp < CM_WORKERS && wq == 0 && gxh < W + P && hsx >= 0 && (hch >> 2) < nb;
  const float* in_b = p.in + (size_t)b * p.nblk * plane_px * 4;
  const float* cbase = in_b + (size_t)(sx < 0 ? 0 : sx) * 4;
  const float* hbase = in_b + (size_t)(hch >> 2) * plane_px * 4 + (size_t)(hsx < 0 ? 0 : hsx) * 4 + (hch & 3);
  const size_t pstride = plane_px * 4, rstride = (size_t)W * 4;
  struct Row {
    float4 v0, v1, v2, v3;
    float h;
    bool ok;
  };
  auto load_row = [&](int ri, Row& R) {
    const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
    R.ok = sy >= 0;
    const size_t ro = (size_t)(sy < 0 ? 0 : sy) * rstride;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    R.v0 = R.v1 = R.v2 = R.v3 = z;
    R.h = 0.f;
    if (col_ok && sy >= 0) {
      const float* c = cbase + ro;
      R.v0 = ldg4(c);
      if (nb > 1) R.v1 = ldg4(c + pstride);
      if (nb > 2) R.v2 = ldg4(c + 2 * pstride);
      if (nb > 3) R.v3 = ldg4(c + 3 * pstride);
    }
    if (h_on && sy >= 0) R.h = __ldg(hbase + ro);
  };

  // ---- one-time setup
  if (tid == 0) {
    CM_TR(0);
    for (int r = 0; r < CM_MAXR; ++r) mbar_init(a_full(r), 4);  // the 4 warps of the group that stages the row
    for (int d = 0; d < ND; ++d) {
      mbar_init(d_full(d), 1);        // tcgen05.commit
      mbar_init(d_empty(d), 4 * KS);  // 4 warps x the KS output rows that read D_d
    }
    fence_mbar_init();
  }
  if (warp == CM_MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 512);
  {
    if (tid < 16) bias_s[tid] = tid < p.cout_blks * 4 ? __ldg(p.bias + tid) : 0.f;
    const uint4* wsrc = reinterpret_cast<const uint4*>(p.wpk);
    uint4* wdst = reinterpret_cast<uint4*>(Bs);
    for (int e = tid; e < B_GROUP / 16; e += CM_THREADS) wdst[e] = __ldg(wsrc + e);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");  // no-op unless launched with programmatic serialization
  Row ra;
  if (warp < CM_WORKERS && g < nin) load_row(g, ra);  // the group's first row is requested before the set-up barrier
  const bool do_x = p.xform == PBMC_XFORM_GN_GELU;
  if (tid < 16) {
    float a = 1.f, bb = 0.f;
    if (do_x && tid < nb * 4) gn_coeffs(p.stats + ((size_t)b * p.nblk + (tid >> 2)) * 2, p.inv_count, p.gamma[tid], p.beta[tid], a, bb);
    if (p.xform == PBMC_XFORM_SCALE) a = scale_src_factor(p.stats + (size_t)b * p.nblk * 2, p.nblk, plane_px);
    xf_a[tid] = a;
    xf_b[tid] = bb;
    if (tid == 0) *wsc_s = p.xform == PBMC_XFORM_SCALE ? __ldg(p.wscale) / a : __ldg(p.wscale);  // powers of two: exact
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tid == 0) CM_TR(1);

  if (warp < CM_WORKERS) {
    // ================================================================ workers: stage rows, drain accumulators
    // Group g stages input rows g, g+5, ... and owns output rows g, g+5, ...  After every staged row it takes ONE
    // of its output rows if that row's accumulators are already complete (non-blocking test), so the TMEM ring
    // keeps draining while the MMA warp works through the staged rows; once a warp has no input rows left it
    // waits for its remaining output rows.  (The 4 warps of a group may interleave differently: every barrier
    // only counts arrivals.)
    const uint32_t as_addr = smem_u32(As) + (uint32_t)i * 16u;
    const uint32_t h_off = (uint32_t)(((hch >> 3) * PLANE + 128 + he) * 16 + (hch & 7) * 2);
    const float h_a = xf_a[hch], h_b = xf_b[hch];
    const bool tr_lane = lane == 0 && wq == 0;
    (void)tr_lane;
    auto sts = [](uint32_t addr, uint4 q) {
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
    };
    const uint32_t xfa_addr = smem_u32(xf_a), xfb_addr = smem_u32(xf_b);
    auto stage_row = [&](int ri, const Row& R) {
      if (tr_lane) CM_TR(100 + g * 64 + 4 * (ri / CM_SETS));
      float v[16] = {R.v0.x, R.v0.y, R.v0.z, R.v0.w, R.v1.x, R.v1.y, R.v1.z, R.v1.w,
                     R.v2.x, R.v2.y, R.v2.z, R.v2.w, R.v3.x, R.v3.y, R.v3.z, R.v3.w};
      float hv = R.h;
      if (p.xform == PBMC_XFORM_SCALE) {  // exact power-of-two scale: out-of-image taps stay zero
        const float s_a = xf_a[0];
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] *= s_a;
        hv *= s_a;
      }
      if (do_x) {
        // GroupNorm + GELU, branch-free: out-of-image taps are masked back to zero afterwards
        const bool keep = R.ok && col_ok;
        const bool all_keep = __all_sync(0xffffffffu, keep) && nb == 4;  // interior warp: nothing to mask (warp-uniform)
#pragma unroll
        for (int j = 0; j < 4; j += 2) {
          if (j < nb) {
            float4 a0, b0, a1, b1;
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a0.x), "=f"(a0.y), "=f"(a0.z), "=f"(a0.w) : "r"(xfa_addr + j * 16));
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b0.x), "=f"(b0.y), "=f"(b0.z), "=f"(b0.w) : "r"(xfb_addr + j * 16));
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a1.x), "=f"(a1.y), "=f"(a1.z), "=f"(a1.w) : "r"(xfa_addr + j * 16 + 16));
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(b1.x), "=f"(b1.y), "=f"(b1.z), "=f"(b1.w) : "r"(xfb_addr + j * 16 + 16));
            float x8[8];
            x8[0] = fmaf(v[4 * j + 0], a0.x, b0.x); x8[1] = fmaf(v[4 * j + 1], a0.y, b0.y);
            x8[2] = fmaf(v[4 * j + 2], a0.z, b0.z); x8[3] = fmaf(v[4 * j + 3], a0.w, b0.w);
            x8[4] = fmaf(v[4 * j + 4], a1.x, b1.x); x8[5] = fmaf(v[4 * j + 5], a1.y, b1.y);
            x8[6] = fmaf(v[4 * j + 6], a1.z, b1.z); x8[7] = fmaf(v[4 * j + 7], a1.w, b1.w);
            gelu_erf2n<4>(x8);
            if (all_keep) {
#pragma unroll
              for (int e = 0; e < 8; ++e) v[4 * j + e] = x8[e];
            } else {
              const bool keep1 = keep && j + 1 < nb;  // absent blocks of a partial group stay exactly zero
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                v[4 * j + e] = keep ? x8[e] : 0.f;
                v[4 * j + 4 + e] = keep1 ? x8[4 + e] : 0.f;
              }
            }
          }
        }
        if (h_on) {
          float hx[2] = {fmaf(hv, h_a, h_b), 0.f};
          gelu_erf2n<1>(hx);
          hv = R.ok ? hx[0] : 0.f;
        }
      }
      if (tr_lane) CM_TR(101 + g * 64 + 4 * (ri / CM_SETS));
      const uint32_t sa = as_addr + (uint32_t)ri * (uint32_t)STAGE_BYTES;
      if (PARTS == 2) {
        uint4 h0, l0, h1, l1;
        split_f16(v, h0, l0);
        split_f16(v + 8, h1, l1);
        sts(sa, h0);
        sts(sa + PLANE * 16, h1);
        sts(sa + 2 * PLANE * 16, l0);
        sts(sa + 3 * PLANE * 16, l1);
      } else {
        sts(sa, pack_bf16(v));
        sts(sa + PLANE * 16, pack_bf16(v + 8));
      }
      if (wq == 0) {
        const uint32_t ha = smem_u32(As) + (uint32_t)ri * (uint32_t)STAGE_BYTES + h_off;
        if (PARTS == 2) {
          const __half hh = __float2half_rn(hv);
          const __half hl = __float2half_rn(hv - __half2float(hh));
          asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__half_as_ushort(hh)) : "memory");
          asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha + (uint32_t)PART_BYTES), "h"(__half_as_ushort(hl)) : "memory");
        } else {
          asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__bfloat16_as_ushort(__float2bfloat16_rn(hv))) : "memory");
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full((uint32_t)ri));
      if (tr_lane) CM_TR(102 + g * 64 + 4 * (ri / CM_SETS));
    };

    const int q = wq;
    const int col = q * 32 + lane, gx = x0 + col;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    float cs[4] = {0.f, 0.f, 0.f, 0.f};  // zero-mean sums: only the c_out <= 4 head conv asks for them
    const bool want_cs = p.out_chan_sum != nullptr;
    const int cout_blks = p.cout_blks;
    const bool epi_gelu = p.epi_act == PBMC_ACT_GELU;
    const uint32_t bias_addr = smem_u32(bias_s);
    const uint32_t wsc_addr = smem_u32(wsc_s);
    float* const obase = p.out + (((size_t)b * cout_blks) * plane_px + (size_t)y0 * W + gx) * 4;
    const size_t blk_stride = plane_px * 4;
    const bool col_in = gx < W;
    auto worker_loop = [&](auto lean_tag) {
      constexpr bool LEAN = decltype(lean_tag)::value;
      // Output row yo reads D_yo .. D_{yo+KS-1}.  Each issuer commits its own rows in order, so the last CM_NMMA
      // of them (one per issuer) cover all KS.
      auto dfull_bar = [&](int r) { return d_full((uint32_t)r % ND); };
      auto dfull_par = [&](int r) { return ((uint32_t)r / ND) & 1u; };
      auto epi_ready = [&](int yo) {
        bool ok = true;
#pragma unroll
        for (int k = 0; k < (CM_NMMA < KS ? CM_NMMA : KS); ++k) ok = ok && mbar_test(dfull_bar(yo + KS - 1 - k), dfull_par(yo + KS - 1 - k));
        return ok;
      };
      auto epi_row = [&](int yo) {
#pragma unroll
        for (int k = (CM_NMMA < KS ? CM_NMMA : KS) - 1; k >= 0; --k) mbar_wait_parked(dfull_bar(yo + KS - 1 - k), dfull_par(yo + KS - 1 - k));
        tc_fence_after();
        if (tr_lane) CM_TR(1200 + 3 * yo);
        const uint32_t s_lo = (uint32_t)yo % ND;
        float* orow = obase + (size_t)yo * W * 4;
        // two halves of 8 output channels: 24 live accumulator registers instead of 48
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
          uint32_t r[KS][8];
          uint32_t sl = s_lo;
#pragma unroll
          for (int dy = 0; dy < KS; ++dy) {
            tmem_ld8_issue(lane_addr + sl * (uint32_t)N + (uint32_t)(dy * 16 + hq * 8), r[dy]);
            if (++sl == (uint32_t)ND) sl = 0;
          }
#pragma unroll
          for (int dy = 0; dy < KS; ++dy) tmem_ld_wait8(r[dy]);
          if (hq == 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              // D_{yo+dy} is read by output rows yo+dy-KS+1 .. yo+dy; rows < 0 do not exist, so row 0 arrives for them
              sl = s_lo;
#pragma unroll
              for (int dy = 0; dy < KS; ++dy) {
                mbar_arrive_n(d_empty(sl), yo == 0 ? (uint32_t)(KS - dy) : 1u);
                if (++sl == (uint32_t)ND) sl = 0;
              }
            }
            if (tr_lane) CM_TR(1201 + 3 * yo);
          }
          if (col_in) {
#pragma unroll
            for (int qh = 0; qh < 2; ++qh) {
              const int qb = 2 * hq + qh;
              if (LEAN || qb < cout_blks) {
                float4 bq;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bq.x), "=f"(bq.y), "=f"(bq.z), "=f"(bq.w) : "r"(bias_addr + qb * 16));
                const float bias4[4] = {bq.x, bq.y, bq.z, bq.w};
                float wsc;  // re-read per block: a register held across the loop spills under the register cap
                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(wsc) : "r"(wsc_addr));
                float o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float a = __uint_as_float(r[0][qh * 4 + e]);
#pragma unroll
                  for (int dy = 1; dy < KS; ++dy) a += __uint_as_float(r[dy][qh * 4 + e]);
                  a = fmaf(a, wsc, bias4[e]);
                  if (!LEAN && epi_gelu) a = gelu_erf(a);
                  o[e] = a;
                }
                *reinterpret_cast<float4*>(orow + qb * blk_stride) = make_float4(o[0], o[1], o[2], o[3]);
                s1[qb] += (o[0] + o[1]) + (o[2] + o[3]);
                s2[qb] = fmaf(o[0], o[0], fmaf(o[1], o[1], fmaf(o[2], o[2], fmaf(o[3], o[3], s2[qb]))));
                if (!LEAN && qb == 0 && want_cs) { cs[0] += o[0]; cs[1] += o[1]; cs[2] += o[2]; cs[3] += o[3]; }
              }
            }
          }
        }
        if (tr_lane) CM_TR(1202 + 3 * yo);
      };
      int ri = g, yo = g;
      while (ri < nin) {
        stage_row(ri, ra);
        ri += CM_SETS;
        if (ri < nin) load_row(ri, ra);  // after the fence: its MEMBAR would wait for freshly issued loads
        if (yo < nrows && epi_ready(yo)) {
          epi_row(yo);
          yo += CM_SETS;
        }
      }
      for (; yo < nrows; yo += CM_SETS) epi_row(yo);
    };
    if (cout_blks == 4 && !epi_gelu && !want_cs)
      worker_loop(std::true_type{});
    else
      worker_loop(std::false_type{});

    if (tid == 0) CM_TR(3);
    if (p.out_stats != nullptr) {
#pragma unroll
      for (int qb = 0; qb < 4; ++qb) {
        const double a = warp_sum((double)s1[qb]);
        const double c2 = warp_sum((double)s2[qb]);
        if (lane == 0) { red[(warp * 4 + qb) * 2] = a; red[(warp * 4 + qb) * 2 + 1] = c2; }
      }
      cm_worker_bar();
      if (tid < 8 && (tid >> 1) < p.cout_blks) {
        double t = 0.0;
        for (int w = 0; w < CM_WORKERS; ++w) t += red[(w * 4 + (tid >> 1)) * 2 + (tid & 1)];
        atomicAdd(p.out_stats + ((size_t)b * p.cout_blks + (tid >> 1)) * 2 + (tid & 1), t);
      }
      cm_worker_bar();
    }
    if (want_cs) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const double a = warp_sum((double)cs[c]);
        if (lane == 0) red[warp * 4 + c] = a;
      }
      cm_worker_bar();
      if (tid < 4) {
        double t = 0.0;
        for (int w = 0; w < CM_WORKERS; ++w) t += red[w * 4 + tid];
        atomicAdd(p.out_chan_sum + (size_t)b * 4 + tid, t);
      }
    }
  } else {
    // ================================================================ MMA issuer: row ri as soon as it is staged
    const bool leader = elect_one();
    constexpr uint32_t A_LBO = PLANE * 16, B_LBO = N * 16, SBO = 128;
    const uint64_t a_desc0 = umma_desc(smem_u32(As), A_LBO, SBO), b_desc0 = umma_desc(smem_u32(Bs), B_LBO, SBO);
    // Rows are independent accumulations (one accumulator per input row), so CM_NMMA warps issue alternate rows:
    // the ~450 clk of barrier / uniform-datapath latency around each row's 9 MMAs (tools/muxtrace.py) would
    // otherwise leave the tensor pipe idle a third of the time.  tcgen05.commit tracks the issuing thread's MMAs.
    for (int ri = warp - CM_MMA_WARP; ri < nin; ri += CM_NMMA) {
      const uint32_t ds = (uint32_t)ri % ND;
      if (ri >= ND) mbar_wait_parked(d_empty(ds), (((uint32_t)ri / ND) & 1u) ^ 1u);  // first ND rows: the ring is free
      mbar_wait_parked(a_full((uint32_t)ri), 0u);
      tc_fence_after();
      if (leader) {
        CM_TR(1400 + 2 * ri);
        const uint32_t dcol = tmem_base + ds * (uint32_t)N;
        const uint64_t a_s = a_desc0 + (uint64_t)((uint32_t)ri * (uint32_t)(STAGE_BYTES >> 4));
#pragma unroll
        for (int dx = 0; dx < KS; ++dx) {
          const uint64_t a_hi = a_s + (uint64_t)dx;  // one position = 16 B
          const uint64_t b_hi = b_desc0 + (uint64_t)(dx * PARTS * (B_TILE >> 4));
          umma_ss<1>(dcol, a_hi, b_hi, IDESC, (uint32_t)dx);
          if (PARTS == 2) {
            umma_ss<1>(dcol, a_hi + (uint64_t)(PART_BYTES >> 4), b_hi, IDESC, 1u);
            umma_ss<1>(dcol, a_hi, b_hi + (uint64_t)(B_TILE >> 4), IDESC, 1u);
          }
        }
        umma_commit(d_full(ds));  // D_ri complete
        CM_TR(1401 + 2 * ri);
      }
      __syncwarp();
    }
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (tid == 0) CM_TR(2);
  if (warp == CM_MMA_WARP) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

#ifdef PBMC_ROW_TRACE
static unsigned long long* g_mux_trace = nullptr;
extern "C" void pbmc_debug_set_mux_trace(void* dev_buf) { g_mux_trace = reinterpret_cast<unsigned long long*>(dev_buf); }
#endif

// Output rows per CTA: minimise waves x (fixed cost + staging rounds + epilogue rounds), in clocks measured with
// tools/muxtrace.py (a staging round = 5 groups x 1 row, an epilogue round = 5 rows).
static int choose_rpc_mux(int units, int H, int max_ctas, bool gelu) {
  const long avail = max_ctas > 0 ? max_ctas : 148;
  int best = 1;
  double best_cost = 1e30;
  for (int r = 1; r <= CM_MAXR - 2 && r <= H; ++r) {
    const long ctas = (long)units * cdiv(H, r);
    const long waves = (ctas + avail - 1) / avail;
    const int rounds1 = cdiv(r + 2, CM_SETS), rounds2 = cdiv(r, CM_SETS);  // one row per group and round
    const double cost = (double)waves * (4000.0 + rounds1 * (gelu ? 2800.0 : 1800.0) + rounds2 * 1000.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = r; }
  }
  return best;
}

template <int PARTS>
static int launch_mux(ConvMuxParams& p, int max_ctas, cudaStream_t st, bool pdl) {
  constexpr int STAGE_BYTES = PARTS * 2 * CM_PLANE * 16, B_GROUP = 3 * PARTS * (2 * CM_N * 16);
  static bool attr_set = false;
  if (!attr_set) {
    PBMC_CUDA(cudaFuncSetAttribute(conv_mux_kernel<PARTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int nstrips = cdiv(p.W, 128);
  p.rpc = choose_rpc_mux(nstrips * p.B, p.H, max_ctas, p.xform == PBMC_XFORM_GN_GELU);
  const size_t smem = CM_HDR + (size_t)B_GROUP + (size_t)(p.rpc + 2) * STAGE_BYTES;
  if (smem > 227 * 1024) return PBMC_ERR_UNSUPPORTED;
  dim3 grid(cdiv(p.H, p.rpc), nstrips, p.B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  // With programmatic dependent launch the set-up (barriers, TMEM, filters) runs while the producer kernel drains; the
  // kernel reads its producer's outputs only after griddepcontrol.wait.
  PBMC_CUDA(launch_maybe_pdl(conv_mux_kernel<PARTS>, grid, dim3(CM_THREADS), smem, st, pdl, p));
  PBMC_CHECK_LAUNCH("conv_mux_kernel");
  return PBMC_OK;
}

// AUTO picks the mux kernel only when its whole grid is resident at once (<= one CTA per SM of the budget): it was
// built for the short strips of a single 512^2 field; for batches that run in waves the pipelined row kernel is faster
// (32 x 256^2: 109 vs 124 us, tools/kbench.py).
bool conv_mux_one_wave(const pbmc_conv_desc& d) {
  const int nstrips = cdiv(d.W, 128);
  const int rpc = choose_rpc_mux(nstrips * d.B, d.H, d.max_ctas, d.src[0].xform == PBMC_XFORM_GN_GELU);
  return (long)nstrips * d.B * cdiv(d.H, rpc) <= (d.max_ctas > 0 ? d.max_ctas : 148);
}

// one source of at most 16 channels, 3x3, c_out <= 16, input either raw or GroupNorm+GELU of its producer
bool conv_mux_supported(const pbmc_conv_desc& d) {
  if (d.ksize != 3 || d.cout > 16 || d.nsrc != 1 || d.src[0].layout != PBMC_LAYOUT_BLOCKED) return false;
  if (d.src[0].nblk < 1 || d.src[0].nblk > 4) return false;
  if (d.src[0].xform != PBMC_XFORM_NONE && d.src[0].xform != PBMC_XFORM_GN_GELU && d.src[0].xform != PBMC_XFORM_SCALE) return false;
  if (d.out_chan_sum != nullptr && d.cout > 4) return false;  // per-channel sums: head conv only
  return true;
}

// wpk_row holds two operand images back to back (ops.pack_conv_weight_row), one 16-channel group here, then the prescale tail:
//   [fp16 hi|lo : 3 * 2 * 1536 B][bf16 : 3 * 1536 B][float 2^-e, 0, 0, 0]
int conv_mux_dispatch(const pbmc_conv_desc& d, cudaStream_t st, bool pdl) {
  ConvMuxParams p;
  const pbmc_src& S = d.src[0];
  p.in = S.ptr; p.stats = S.stats; p.gamma = S.gamma; p.beta = S.beta; p.inv_count = S.inv_count;
  p.nblk = S.nblk; p.xform = S.xform;
  p.B = d.B; p.H = d.H; p.W = d.W;
  p.cout_blks = (d.cout + 3) / 4;
  p.pad_mode = d.pad_mode; p.epi_act = d.epi_act;
  p.rpc = 1;
  p.bias = d.bias; p.out = d.out; p.out_stats = d.out_stats; p.out_chan_sum = d.out_chan_sum;
  p.trace = nullptr;
#ifdef PBMC_ROW_TRACE
  p.trace = g_mux_trace;
#endif
  const char* base = reinterpret_cast<const char*>(d.wpk_row);
  if (!base) return PBMC_ERR_NULL_POINTER;
  if (!aligned16(base)) return PBMC_ERR_MISALIGNED;
  const size_t off_bf16 = (size_t)3 * 2 * (2 * CM_N * 16);
  p.wscale = reinterpret_cast<const float*>(base + off_bf16 + (size_t)3 * (2 * CM_N * 16));
  if (d.impl == PBMC_CONV_MUX_F16X2) {
    p.wpk = base;
    return launch_mux<2>(p, d.max_ctas, st, pdl);
  }
  if (d.impl == PBMC_CONV_MUX_BF16) {
    p.wpk = base + off_bf16;
    return launch_mux<1>(p, d.max_ctas, st, pdl);
  }
  return PBMC_ERR_UNSUPPORTED;
}

}  // namespace pbmc
