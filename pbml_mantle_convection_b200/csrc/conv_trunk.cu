// Persistent trunk kernel for sm_100a: the R FluidLayers of ONE pyramid level in ONE launch.
//   NewFluidNet.forward trunk   pytorch_networks_convae.py:1321-1327  (for r in range(R): y1 = convs[l][r](y1))
//   FluidLayer.forward          :790-799   conv -> GroupNorm(4 ch / group, eps 1e-5) -> exact GELU
//   SymmetricConv2d.forward     symmetric_layers_torch.py:113-138 (mirrored filters expanded at pack time)
// Same GEMM and the same per-layer plan as conv_mux.cu (M = 128 output columns, N = 48 = (dy, c_out), K = 16,
// one TMEM accumulator per INPUT row, all input rows of the CTA resident in shared memory as fp16 hi|lo planes,
// GroupNorm + GELU of the producer applied while a row is staged, statistics of the output in the epilogue) --
// what changes is the life time of a CTA.  A 512^2 layer is ~25 k clk of work per CTA wrapped in ~9 k clk of launch
// ramp / drain and ~4 k clk of set-up and teardown (TMEM allocation, barrier init, filter copy; tools/muxtrace.py,
// profiles/r1_muxtrace_512.txt).  Here a CTA keeps its strip for all R layers:
//   * TMEM, the mbarriers (their phases simply keep counting) and the staging buffers live across layers;
//   * the NEXT layer's filters are copied into a second shared-memory buffer by the idle MMA warps while the
//     current layer runs;
//   * GroupNorm is a reduction over the whole image, so layer r + 1 can only start when every CTA has finished
//     layer r: a grid-wide arrive/poll counter (one per sample: samples are independent) in global memory.  The
//     barrier also publishes the neighbours' boundary rows; everything read after it comes from L2 (ld.global.cg:
//     L1 may still hold the lines of two layers ago, the ping-pong buffer's previous content).
// Tried and withdrawn (round 2, profiles/r2_ncu_trunk_512_remap.txt): a staging map in which warp q owns channel block q of
// the whole row (GroupNorm coefficients in registers, no ld.shared while staging).  It cut the LSU shared-memory
// wavefronts by 20 % (5.1 M -> 4.1 M per launch) but needed 21 % more instructions (8-byte stores, four positions per
// lane) and was SLOWER: 72.7 vs 66.6 us per 4-layer launch at 512^2.  The kernel is bound by issued instructions and the
// hand-off latencies between its phases, not by the shared-memory pipe.
// Every CTA of the launch must be resident at once (the dispatcher only takes the kernel when the grid fits the
// caller's CTA budget; the rollout's per-level budgets sum to <= 148).  A CTA that waits longer than 2 s traps.
#include <stdlib.h>

#include "common.cuh"
#include "tc05.cuh"

namespace pbmc {

// Six groups (832 threads at 72 registers, three staging rounds instead of four at 16 input rows) were measured against
// five: 68.6 vs 68.6 us per 4-layer launch at 148 CTAs, 85.1 vs 85.0 at 96 -- fewer rounds, each slower by the same
// factor: the staging rounds are bound by issued instructions, not by their number.
constexpr int CT_SETS = 5;                       // groups of 4 worker warps
constexpr int CT_WORKERS = 4 * CT_SETS;          // 20 worker warps
constexpr int CT_NMMA = 2;                       // MMA issuer warps (alternate rows); the first one owns TMEM
constexpr int CT_MMA_WARP = CT_WORKERS;
constexpr int CT_THREADS = (CT_WORKERS + CT_NMMA) * 32;
constexpr int CT_MAXR = 24;                      // input rows per CTA (all resident in shared memory)
constexpr int CT_ND = 10;                        // TMEM accumulator ring
constexpr int CT_N = 48;                         // (dy, c_out)
constexpr int CT_PLANE = 136;                    // positions per K-chunk plane (128 + 2 halo, rounded up to 8)
constexpr int CT_HDR = 2432;                     // barriers, TMEM slot, reduction scratch, raw-row barriers, coefficients

struct TrunkLayerDev {
  const float* in;       // [B][4][H][W][4] raw producer output (or the level's input for layer 0)
  const double* stats;   // [B][4][2] GroupNorm sums of `in` (NULL: `in` is used as it is)
  const float* gamma;    // [16] affine of `in`'s GroupNorm
  const float* beta;
  const void* wpk;       // this layer's filters, row-kernel operand image (one 16-channel group)
  const float* wscale;   // 2^-e: the image holds the filters times 2^e (ops.prescale_pow2)
  const float* bias;     // [16]
  float* out;            // [B][4][H][W][4] raw output
  double* out_stats;     // [B][4][2], zeroed before the launch
};

struct ConvTrunkParams {
  TrunkLayerDev L[PBMC_MAX_REPEATS];
  double inv_count;      // 1 / (4 * H * W)
  unsigned int* sync;    // [B] arrive counters, zeroed before the launch
  int R, B, H, W, pad_mode, rpc;
};

// BULK loader (opt-in, pbmc_trunk_desc.loader; correct, measured 15 % slower than the thread loader, see include/pbmc.h):
// the raw input rows of a layer are copied into shared memory by the TMA engine (cp.async.bulk, one copy
// per 4-channel plane and row, all rows of the layer requested up front by ONE thread right after the grid barrier) --
// each row lands in the very stage slot its operand image will occupy (4 planes x 130 positions x 16 B of fp32 = the
// size of the fp16 hi|lo image), the group that owns the row waits for its mbarrier, reads its pixels from shared memory,
// and writes the GroupNorm+GELU'd, split operand image over them.  No global load, no address arithmetic and no
// prefetch registers in the workers; the copies run ahead of the staging by as many rows as the layer has.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ float4 lds4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

__device__ __forceinline__ void ct_worker_bar() { asm volatile("bar.sync 1, %0;" ::"n"(CT_WORKERS * 32) : "memory"); }
__device__ __forceinline__ void ct_mma_bar() { asm volatile("bar.sync 2, %0;" ::"n"(CT_NMMA * 32) : "memory"); }
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

template <int PARTS, bool BULK>
__global__ void __maxnreg__(CT_SETS <= 5 ? 80 : 72) conv_trunk_kernel(const __grid_constant__ ConvTrunkParams p) {
  constexpr int KS = 3, P = 1, N = CT_N, ND = CT_ND, PLANE = CT_PLANE;
  constexpr int PART_BYTES = 2 * PLANE * 16, STAGE_BYTES = PARTS * PART_BYTES;
  constexpr int B_TILE = 2 * N * 16, B_GROUP = KS * PARTS * B_TILE;
  constexpr uint32_t FMT = PARTS == 2 ? 0u : 1u;  // fp16 hi|lo split, or one bf16 pass
  constexpr uint32_t IDESC = row_idesc(FMT, N);
  static_assert(8 * (CT_MAXR + 2 * ND) <= 448, "barrier area");
  static_assert(!BULK || PARTS == 2, "the raw fp32 row fills exactly the fp16 hi|lo stage slot");
  static_assert(512 + CT_WORKERS * 64 <= 2048 && 2048 + 8 * CT_MAXR <= 2240, "reduction scratch, raw-row barriers");
  static_assert(ND * N <= 512, "TMEM has 512 columns");
  static_assert(B_GROUP % 128 == 0, "operand buffers stay 128-byte aligned");
  extern __shared__ __align__(128) unsigned char smem[];
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 448);
  double* red = reinterpret_cast<double*>(smem + 512);        // CT_WORKERS warps x 8 doubles
  float* bias_s = reinterpret_cast<float*>(smem + 2240);      // 16 floats
  float* xf_a = reinterpret_cast<float*>(smem + 2304);        // GroupNorm scale / shift of the 16 input channels
  float* xf_b = reinterpret_cast<float*>(smem + 2368);
  unsigned char* Bs = smem + CT_HDR;                          // two filter buffers: layer l uses Bs + (l & 1) * B_GROUP
  unsigned char* As = Bs + 2 * B_GROUP;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z;
  const int x0 = blockIdx.y * 128;
  const int y0 = blockIdx.x * p.rpc;
  const int H = p.H, W = p.W, R = p.R;
  const int nrows = min(p.rpc, H - y0);
  const int nin = nrows + KS - 1;
  const size_t plane_px = (size_t)H * W;
  const uint32_t bar0 = smem_u32(smem);
  auto a_full = [&](uint32_t r) { return bar0 + r * 8u; };
  auto d_full = [&](uint32_t d) { return bar0 + (uint32_t)(CT_MAXR + d) * 8u; };
  auto d_empty = [&](uint32_t d) { return bar0 + (uint32_t)(CT_MAXR + ND + d) * 8u; };
  auto raw_full = [&](uint32_t r) { return bar0 + 2048u + r * 8u; };  // BULK: the raw row r of this layer has landed

  // ---- one-time set-up: barriers, TMEM, layer 0's filters / bias / GroupNorm coefficients
  if (tid == 0) {
    for (int r = 0; r < CT_MAXR; ++r) {
      mbar_init(a_full(r), 4);  // the 4 warps of the group that stages the row
      if (BULK) mbar_init(raw_full(r), 1);  // one arrive.expect_tx (+ the bytes of the row's four bulk copies)
    }
    for (int d = 0; d < ND; ++d) {
      mbar_init(d_full(d), 1);        // tcgen05.commit
      mbar_init(d_empty(d), 4 * KS);  // 4 warps x the KS output rows that read D_d
    }
    fence_mbar_init();
  }
  if (warp == CT_MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 512);
  {
    const uint4* wsrc = reinterpret_cast<const uint4*>(p.L[0].wpk);
    uint4* wdst = reinterpret_cast<uint4*>(Bs);
    for (int e = tid; e < B_GROUP / 16; e += CT_THREADS) wdst[e] = __ldg(wsrc + e);
  }
  auto load_coeffs = [&](int l) {  // threads 0..15 of the CTA; the statistics come from L2 (written by other CTAs)
    const TrunkLayerDev& Ld = p.L[l];
    float a = 1.f, bb = 0.f;
    if (Ld.stats != nullptr) {
      const double* s2 = Ld.stats + ((size_t)b * 4 + (tid >> 2)) * 2;
      const double mean = __ldcg(s2) * p.inv_count;
      double var = __ldcg(s2 + 1) * p.inv_count - mean * mean;
      if (var < 0.0) var = 0.0;
      const double ad = rsqrt(var + 1e-5) * (double)__ldg(Ld.gamma + tid);
      a = (float)ad;
      bb = (float)((double)__ldg(Ld.beta + tid) - mean * ad);
    }
    xf_a[tid] = a;
    xf_b[tid] = bb;
    bias_s[tid] = __ldg(Ld.bias + tid);
  };
  // Everything above (barriers, TMEM, layer 0's filters) may overlap the drain of the previous kernel in the stream when the
  // launch carries programmatic stream serialization (api.cu: the level-0 kernel behind conv[0]); without it a no-op.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tid < 16) load_coeffs(0);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < CT_WORKERS) {
    // ================================================================ workers: stage rows, drain accumulators
    const int g = warp >> 2, wq = warp & 3;
    const int i = wq * 32 + lane;  // position in the staged row = input column x0 - 1 + i
    const int gxp = x0 - P + i;
    const int sx = pad_index(gxp, W, p.pad_mode);
    const bool col_ok = gxp < W + P && sx >= 0;  // columns past the image feed masked outputs only
    const int hch = lane & 15, he = lane >> 4;   // halo positions 128, 129: warp 0 of a group, lane = (position, channel)
    const int gxh = x0 - P + 128 + he;
    const int hsx = pad_index(gxh, W, p.pad_mode);
    const bool h_on = wq == 0 && gxh < W + P && hsx >= 0;
    const size_t in_boff = (size_t)b * 4 * plane_px * 4;
    const size_t c_off = in_boff + (size_t)(sx < 0 ? 0 : sx) * 4;
    const size_t h_off_g = in_boff + (size_t)(hch >> 2) * plane_px * 4 + (size_t)(hsx < 0 ? 0 : hsx) * 4 + (hch & 3);
    const size_t pstride = plane_px * 4, rstride = (size_t)W * 4;
    struct Row {
      float4 v0, v1, v2, v3;
      float h;
      bool ok;
    };
    const uint32_t as_addr = smem_u32(As) + (uint32_t)i * 16u;
    const uint32_t h_off = (uint32_t)(((hch >> 3) * PLANE + 128 + he) * 16 + (hch & 7) * 2);
    auto sts = [](uint32_t addr, uint4 q) {
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
    };
    const uint32_t xfa_addr = smem_u32(xf_a), xfb_addr = smem_u32(xf_b);
    const int col = wq * 32 + lane, gx = x0 + col;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(wq * 32) << 16);
    const uint32_t bias_addr = smem_u32(bias_s);
    const size_t blk_stride = plane_px * 4;
    const bool col_in = gx < W;
    const size_t o_off = (((size_t)b * 4) * plane_px + (size_t)y0 * W + gx) * 4;
    const unsigned int nctas = gridDim.x * gridDim.y;
    // BULK loader geometry: the in-image part of positions 0..129 (input columns x0-1 .. x0+128) is copied, a padded
    // position reads the position its padding rule points at
    constexpr uint32_t RAWP = PLANE * 16;  // plane stride of a raw row inside its stage slot
    const int i_lo = x0 == 0 ? 1 : 0, i_hi = min(129, W - x0), ncols = i_hi - i_lo + 1;
    const uint32_t raw_pos = (uint32_t)((sx < 0 ? 0 : sx) - (x0 - P)) * 16u;
    const uint32_t raw_hpos = (uint32_t)(hch >> 2) * RAWP + (uint32_t)((hsx < 0 ? 0 : hsx) - (x0 - P)) * 16u + (uint32_t)(hch & 3) * 4u;
    auto group_bar = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(3 + g) : "memory"); };
    // all raw rows of layer l, requested by lanes 0..3 of warp 0 (one 4-channel plane each) right after the grid barrier
    auto request_rows = [&](int l) {
      if (warp != 0 || lane >= 4) return;
      asm volatile("fence.proxy.async;" ::: "memory");  // other CTAs' (generic-proxy) stores, acquired at the barrier, before the async-proxy reads
      const float* src_pl = p.L[l].in + (((size_t)b * 4 + lane) * plane_px + (size_t)(x0 - P + i_lo)) * 4;
      const uint32_t dst_pl = smem_u32(As) + (uint32_t)lane * RAWP + (uint32_t)i_lo * 16u;
      for (int ri = 0; ri < nin; ++ri) {
        const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
        if (sy < 0) continue;  // a zero-padded row: nothing to copy, the workers stage zeros
        if (lane == 0) mbar_expect_tx(raw_full((uint32_t)ri), (uint32_t)(4 * ncols * 16));
        bulk_g2s(dst_pl + (uint32_t)ri * (uint32_t)STAGE_BYTES, src_pl + (size_t)sy * W * 4, (uint32_t)(ncols * 16), raw_full((uint32_t)ri));
      }
    };
    if (BULK) request_rows(0);

    for (int l = 0; l < R; ++l) {
      const TrunkLayerDev& Ld = p.L[l];
      const bool do_x = Ld.stats != nullptr;
      const float* in_c = Ld.in + c_off;
      const float* in_h = Ld.in + h_off_g;
      const uint32_t apar = (uint32_t)l & 1u;  // a_full(ri) completes once per layer
      const int gb = l * nin;                  // running row index of this layer's input row 0 (TMEM ring position)
      auto load_row = [&](int ri, Row& Rw) {
        const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
        Rw.ok = sy >= 0;
        const size_t ro = (size_t)(sy < 0 ? 0 : sy) * rstride;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        Rw.v0 = Rw.v1 = Rw.v2 = Rw.v3 = z;
        Rw.h = 0.f;
        if (BULK) {
          if (sy >= 0) {
            mbar_wait_parked(raw_full((uint32_t)ri), apar);  // the row's four planes have landed in its stage slot
            const uint32_t base = smem_u32(As) + (uint32_t)ri * (uint32_t)STAGE_BYTES;
            if (col_ok) {
              Rw.v0 = lds4(base + raw_pos);
              Rw.v1 = lds4(base + RAWP + raw_pos);
              Rw.v2 = lds4(base + 2 * RAWP + raw_pos);
              Rw.v3 = lds4(base + 3 * RAWP + raw_pos);
            }
            if (h_on) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(Rw.h) : "r"(base + raw_hpos) : "memory");
          }
          return;
        }
        if (col_ok && sy >= 0) {
          const float* c = in_c + ro;
          Rw.v0 = ldcg4(c);
          Rw.v1 = ldcg4(c + pstride);
          Rw.v2 = ldcg4(c + 2 * pstride);
          Rw.v3 = ldcg4(c + 3 * pstride);
        }
        if (h_on && sy >= 0) Rw.h = __ldcg(in_h + ro);
      };
      // the group's first row is requested before the layer's GroupNorm coefficients are computed (threads 0..15: two
      // L2 reads and a double-precision rsqrt each), so that the two latencies overlap
      Row ra;
      int ri = g, yo = g;
      if (ri < nin) load_row(ri, ra);
      if (l > 0) {
        if (tid < 16) load_coeffs(l);
        ct_worker_bar();
      }
      const float h_a = xf_a[hch], h_b = xf_b[hch];
      auto stage_row = [&](int ri, const Row& Rw) {
        float v[16] = {Rw.v0.x, Rw.v0.y, Rw.v0.z, Rw.v0.w, Rw.v1.x, Rw.v1.y, Rw.v1.z, Rw.v1.w,
                       Rw.v2.x, Rw.v2.y, Rw.v2.z, Rw.v2.w, Rw.v3.x, Rw.v3.y, Rw.v3.z, Rw.v3.w};
        float hv = Rw.h;
        if (do_x) {
          // GroupNorm + GELU, branch-free: out-of-image taps are masked back to zero afterwards
          const bool keep = Rw.ok && col_ok;
          const bool all_keep = __all_sync(0xffffffffu, keep);  // interior warp: nothing to mask (warp-uniform)
#pragma unroll
          for (int j = 0; j < 4; j += 2) {
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
#pragma unroll
              for (int e = 0; e < 8; ++e) v[4 * j + e] = keep ? x8[e] : 0.f;
            }
          }
          if (h_on) {
            float hx[2] = {fmaf(hv, h_a, h_b), 0.f};
            gelu_erf2n<1>(hx);
            hv = Rw.ok ? hx[0] : 0.f;
          }
        }
        const uint32_t sa = as_addr + (uint32_t)ri * (uint32_t)STAGE_BYTES;
        if (BULK) group_bar();  // every thread of the group has read its pixels of the raw row: now it may be overwritten
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
      };

      float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
      float* const obase = Ld.out + o_off;
      const float wsc = __ldg(Ld.wscale);
      // Output row yo reads D_yo .. D_{yo+KS-1} (running indices gb + ...).  Each issuer commits its own rows in order,
      // so the last CT_NMMA of them (one per issuer) cover all KS.
      auto dfull_bar = [&](int r) { return d_full((uint32_t)(gb + r) % ND); };
      auto dfull_par = [&](int r) { return ((uint32_t)(gb + r) / ND) & 1u; };
      auto epi_ready = [&](int yo) {
        bool ok = true;
#pragma unroll
        for (int k = 0; k < CT_NMMA; ++k) ok = ok && mbar_test(dfull_bar(yo + KS - 1 - k), dfull_par(yo + KS - 1 - k));
        return ok;
      };
      auto epi_row = [&](int yo) {
#pragma unroll
        for (int k = CT_NMMA - 1; k >= 0; --k) mbar_wait_parked(dfull_bar(yo + KS - 1 - k), dfull_par(yo + KS - 1 - k));
        tc_fence_after();
        const uint32_t s_lo = (uint32_t)(gb + yo) % ND;
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
              // D_{yo+dy} is read by output rows yo+dy-KS+1 .. yo+dy; the rows above the strip (< 0) and below it
              // (>= nrows) do not exist, so the first / last row arrives for them: every accumulator's "empty"
              // phase completes, which the next layer's MMAs wait for
              sl = s_lo;
#pragma unroll
              for (int dy = 0; dy < KS; ++dy) {
                const uint32_t cnt = 1u + (yo == 0 ? (uint32_t)(KS - 1 - dy) : 0u) + (yo == nrows - 1 ? (uint32_t)dy : 0u);
                mbar_arrive_n(d_empty(sl), cnt);
                if (++sl == (uint32_t)ND) sl = 0;
              }
            }
          }
          if (col_in) {
#pragma unroll
            for (int qh = 0; qh < 2; ++qh) {
              const int qb = 2 * hq + qh;
              float4 bq;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bq.x), "=f"(bq.y), "=f"(bq.z), "=f"(bq.w) : "r"(bias_addr + qb * 16));
              const float bias4[4] = {bq.x, bq.y, bq.z, bq.w};
              float o[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float a = __uint_as_float(r[0][qh * 4 + e]);
#pragma unroll
                for (int dy = 1; dy < KS; ++dy) a += __uint_as_float(r[dy][qh * 4 + e]);
                o[e] = fmaf(a, wsc, bias4[e]);
              }
              *reinterpret_cast<float4*>(orow + qb * blk_stride) = make_float4(o[0], o[1], o[2], o[3]);
              s1[qb] += (o[0] + o[1]) + (o[2] + o[3]);
              s2[qb] = fmaf(o[0], o[0], fmaf(o[1], o[1], fmaf(o[2], o[2], fmaf(o[3], o[3], s2[qb]))));
            }
          }
        }
      };

      while (ri < nin) {
        stage_row(ri, ra);
        ri += CT_SETS;
        if (ri < nin) load_row(ri, ra);  // after the fence: its MEMBAR would wait for freshly issued loads
        if (yo < nrows && epi_ready(yo)) {
          epi_row(yo);
          yo += CT_SETS;
        }
      }
      for (; yo < nrows; yo += CT_SETS) epi_row(yo);

      // ---- GroupNorm sums of this layer's output: warp -> CTA (double) -> one atomic per (block, moment)
#pragma unroll
      for (int qb = 0; qb < 4; ++qb) {
        const double a = warp_sum((double)s1[qb]);
        const double c2 = warp_sum((double)s2[qb]);
        if (lane == 0) { red[(warp * 4 + qb) * 2] = a; red[(warp * 4 + qb) * 2 + 1] = c2; }
      }
      ct_worker_bar();  // every output row of the CTA is stored, red[] is complete
      if (warp == 0) {
        // one warp finishes the layer for the CTA: lane = (quarter of the 20 warps, moment) adds five partial sums, two
        // shuffles fold the quarters, lanes 0..7 issue the atomics ...
        static_assert(CT_WORKERS % 4 == 0, "four quarters of CT_SETS warps");
        const int m = lane & 7, q = lane >> 3;
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < CT_SETS; ++w) t += red[((q * CT_SETS + w) * 4 + (m >> 1)) * 2 + (m & 1)];
        t += __shfl_xor_sync(0xffffffffu, t, 8);
        t += __shfl_xor_sync(0xffffffffu, t, 16);
        if (lane < 8) atomicAdd(Ld.out_stats + ((size_t)b * 4 + (m >> 1)) * 2 + (m & 1), t);
        if (l + 1 < R) {
          // ... and takes the CTA through the grid-wide barrier of this sample's CTAs: every output row and every statistics
          // contribution of layer l is in L2 before anybody starts layer l + 1 (cooperative-groups pattern: CTA barrier
          // above, fence, arrive + poll by one thread, CTA barrier below)
          __threadfence();
          __syncwarp();
          if (lane == 0) {
            atomicAdd(p.sync + b, 1u);
            const unsigned int target = (unsigned int)(l + 1) * nctas;
            if (ld_acquire_gpu_u32(p.sync + b) < target) {
              const long long t0 = clock64();
              while (ld_acquire_gpu_u32(p.sync + b) < target) {
                __nanosleep(20);
                if (clock64() - t0 > 4000000000ll) __trap();  // ~2 s: some CTA of the launch is not resident
              }
            }
            __threadfence();
          }
        }
      }
      if (l + 1 < R) {
        ct_worker_bar();
        if (BULK) request_rows(l + 1);
      }
    }
  } else {
    // ================================================================ MMA issuers: row ri as soon as it is staged
    const bool leader = elect_one();
    const int mw = warp - CT_MMA_WARP, mt = mw * 32 + lane;
    constexpr uint32_t A_LBO = PLANE * 16, B_LBO = N * 16, SBO = 128;
    const uint64_t a_desc0 = umma_desc(smem_u32(As), A_LBO, SBO);
    for (int l = 0; l < R; ++l) {
      const uint64_t b_desc0 = umma_desc(smem_u32(Bs + (l & 1) * B_GROUP), B_LBO, SBO);
      const uint32_t apar = (uint32_t)l & 1u;
      const int gb = l * nin;
      // Rows are independent accumulations (one accumulator per input row), so the issuers take alternate rows;
      // tcgen05.commit tracks the issuing thread's MMAs.
      for (int ri = mw; ri < nin; ri += CT_NMMA) {
        const uint32_t gri = (uint32_t)(gb + ri);
        const uint32_t ds = gri % ND;
        if (gri >= (uint32_t)ND) mbar_wait_parked(d_empty(ds), ((gri / ND) & 1u) ^ 1u);  // first ND rows: the ring is free
        mbar_wait_parked(a_full((uint32_t)ri), apar);
        tc_fence_after();
        if (leader) {
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
        }
        __syncwarp();
      }
      if (l + 1 < R) {
        // next layer's filters into the other buffer (its last readers, layer l - 1's MMAs, completed before the
        // previous grid barrier); visible to the tensor core's proxy before either issuer goes on
        const uint4* wsrc = reinterpret_cast<const uint4*>(p.L[l + 1].wpk);
        uint4* wdst = reinterpret_cast<uint4*>(Bs + ((l + 1) & 1) * B_GROUP);
        for (int e = mt; e < B_GROUP / 16; e += CT_NMMA * 32) wdst[e] = __ldg(wsrc + e);
        fence_proxy_async_smem();
        ct_mma_bar();
      }
    }
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == CT_MMA_WARP) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

// Output rows per CTA: the whole grid must be resident at once (ctas <= avail); among those, minimise
// fixed cost + staging rounds + epilogue rounds (clocks from tools/muxtrace.py, as conv_mux.cu).
// clocks of one layer for a CTA that owns `rpc` output rows (0: more rows than shared memory holds)
double conv_trunk_layer_cost(int rpc) {
  if (rpc < 1 || rpc > CT_MAXR - 2) return 0.0;
  const int rounds1 = cdiv(rpc + 2, CT_SETS), rounds2 = cdiv(rpc, CT_SETS);
  return 1500.0 + rounds1 * 2800.0 + rounds2 * 1000.0;
}

static int choose_rpc_trunk(int units, int H, int avail) {
  int best = 0;
  double best_cost = 1e30;
  for (int r = 1; r <= CT_MAXR - 2 && r <= H; ++r) {
    const long ctas = (long)units * cdiv(H, r);
    if (ctas > avail) continue;
    const double cost = conv_trunk_layer_cost(r);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = r; }
  }
  return best;
}

bool conv_trunk_supported(const pbmc_trunk_desc& t) {
  if (t.R < 1 || t.R > PBMC_MAX_REPEATS || t.B < 1 || t.H < 1 || t.W < 1) return false;
  if (t.src0.nblk != 4 || t.src0.layout != PBMC_LAYOUT_BLOCKED) return false;
  if (t.src0.xform != PBMC_XFORM_NONE && t.src0.xform != PBMC_XFORM_GN_GELU) return false;
  if (t.impl != PBMC_CONV_AUTO && t.impl != PBMC_CONV_MUX_F16X2 && t.impl != PBMC_CONV_MUX_BF16 && t.impl != PBMC_CONV_ROW_F16X2 &&
      t.impl != PBMC_CONV_ROW_BF16)
    return false;
  for (int r = 0; r < t.R; ++r)
    if (t.layers[r].cout != 16 || t.layers[r].ksize != 3 || t.layers[r].cin_blks != 4 || !t.layers[r].wpk_row) return false;
  const int avail = t.max_ctas > 0 ? t.max_ctas : 148;
  if (avail > 148) return false;
  return choose_rpc_trunk(cdiv(t.W, 128) * t.B, t.H, avail) > 0;
}

template <int PARTS, bool BULK>
static int launch_trunk(ConvTrunkParams& p, cudaStream_t st, bool pdl) {
  constexpr int STAGE_BYTES = PARTS * 2 * CT_PLANE * 16, B_GROUP = 3 * PARTS * (2 * CT_N * 16);
  static bool attr_set = false;
  if (!attr_set) {
    PBMC_CUDA(cudaFuncSetAttribute(conv_trunk_kernel<PARTS, BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const size_t smem = CT_HDR + (size_t)2 * B_GROUP + (size_t)(p.rpc + 2) * STAGE_BYTES;
  if (smem > 227 * 1024) return PBMC_ERR_UNSUPPORTED;
  dim3 grid(cdiv(p.H, p.rpc), cdiv(p.W, 128), p.B);
  PBMC_CUDA(launch_maybe_pdl(conv_trunk_kernel<PARTS, BULK>, grid, dim3(CT_THREADS), smem, st, pdl, p));
  PBMC_CHECK_LAUNCH("conv_trunk_kernel");
  return PBMC_OK;
}

// wpk_row of a layer: [fp16 hi|lo : 3 * 2 * 1536 B][bf16 : 3 * 1536 B][float 2^-e, 0, 0, 0] (ops.pack_conv_weight_row, one
// 16-channel group)
int conv_trunk_dispatch(const pbmc_trunk_desc& t, cudaStream_t st, bool pdl) {
  if (!conv_trunk_supported(t)) return PBMC_ERR_UNSUPPORTED;
  if (!t.src0.ptr || !t.ping[0] || !t.ping[1] || !t.stats || !t.sync) return PBMC_ERR_NULL_POINTER;
  if (!aligned16(t.src0.ptr) || !aligned16(t.ping[0]) || !aligned16(t.ping[1])) return PBMC_ERR_MISALIGNED;
  const bool bf16 = t.impl == PBMC_CONV_MUX_BF16 || t.impl == PBMC_CONV_ROW_BF16;
  const size_t off_bf16 = (size_t)3 * 2 * (2 * CT_N * 16);
  ConvTrunkParams p;
  p.R = t.R; p.B = t.B; p.H = t.H; p.W = t.W; p.pad_mode = t.pad_mode;
  p.inv_count = 1.0 / (4.0 * (double)t.H * (double)t.W);
  p.sync = t.sync;
  const int avail = t.max_ctas > 0 ? t.max_ctas : 148;
  p.rpc = choose_rpc_trunk(cdiv(t.W, 128) * t.B, t.H, avail);
  for (int r = 0; r < t.R; ++r) {
    const pbmc_layer& Lh = t.layers[r];
    TrunkLayerDev& Ld = p.L[r];
    if (!Lh.bias || !aligned16(Lh.wpk_row)) return PBMC_ERR_NULL_POINTER;
    if (r == 0) {
      const bool x = t.src0.xform == PBMC_XFORM_GN_GELU;
      if (x && (!t.src0.stats || !t.src0.gamma || !t.src0.beta)) return PBMC_ERR_NULL_POINTER;
      Ld.in = t.src0.ptr; Ld.stats = x ? t.src0.stats : nullptr; Ld.gamma = t.src0.gamma; Ld.beta = t.src0.beta;
    } else {
      const pbmc_layer& Lp = t.layers[r - 1];
      if (!Lp.gamma || !Lp.beta) return PBMC_ERR_NULL_POINTER;
      Ld.in = t.ping[(r - 1) & 1]; Ld.stats = t.stats + (size_t)(r - 1) * t.B * 8; Ld.gamma = Lp.gamma; Ld.beta = Lp.beta;
    }
    Ld.wpk = reinterpret_cast<const char*>(Lh.wpk_row) + (bf16 ? off_bf16 : 0);
    Ld.wscale = reinterpret_cast<const float*>(reinterpret_cast<const char*>(Lh.wpk_row) + off_bf16 + (size_t)3 * (2 * CT_N * 16));
    Ld.bias = Lh.bias;
    Ld.out = t.ping[r & 1];
    Ld.out_stats = t.stats + (size_t)r * t.B * 8;
  }
  if (!t.pre_zeroed) {
    PBMC_CUDA(cudaMemsetAsync(t.sync, 0, (size_t)t.B * sizeof(unsigned int), st));
    PBMC_CUDA(cudaMemsetAsync(t.stats, 0, (size_t)t.R * t.B * 8 * sizeof(double), st));
  }
  if (bf16) return launch_trunk<1, false>(p, st, pdl);
  return t.loader == PBMC_TRUNK_LOADER_BULK ? launch_trunk<2, true>(p, st, pdl) : launch_trunk<2, false>(p, st, pdl);
}

}  // namespace pbmc
