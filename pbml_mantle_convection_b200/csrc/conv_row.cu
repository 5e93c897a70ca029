// Row-streaming, warp-specialised tcgen05 / TMEM implicit-GEMM convolution for sm_100a.
//
// Same operator contract as conv_ffma.cu / conv_umma.cu (sources with the producer's GroupNorm+GELU
// fused into the load, padding folded into the load coordinates, bias / GELU / GroupNorm statistics /
// zero-mean sums in the epilogue), restating
//   SymmetricConv2d.forward symmetric_layers_torch.py:113-138, nn.Conv2d heads
//   pytorch_networks_convae.py:1263-1309, FluidLayer :790-799, concat :1327/:1332.
//
// GEMM view (k = KS, P = k/2).  A CTA owns a strip of 128 output columns x `rpc` output rows and
// streams the strip's input rows through a shared-memory ring.  For ONE input row r (128 + k - 1
// positions, staged once as fp16 hi|lo channel-chunk planes = UMMA K-major / no-swizzle canonical
// layout) and one 16-channel input group, k tcgen05.mma (x3 for the hi/lo split) with
//     M = 128 output columns, N = k*16 = (dy, c_out), K = 16 input channels
// accumulate   D_r[x][(dy, co)] += sum_{dx, ci} X[r][x + dx][ci] * W[dy][dx][ci][co]
// where the dx shift is the A descriptor's start address (+dx*16 B) and ALL k vertical taps ride in
// the N dimension: the A tile is read from shared memory once per (dx, pass) instead of once per tap
// (tcgen05.mma with N = 16 is shared-memory-read bound, see conv_umma.cu).  Output row y is then
//     out[y][x][co] = bias + sum_dy D_{y+dy}[x][(dy, co)]
// i.e. k TMEM loads from the SAME lane -- no shuffles, no junk lanes, no halo columns in M.
// D_r live in a TMEM ring of ND accumulators (N columns each).
//
// Warp roles:  epilogue sets of 4 warps (output rows dealt round-robin; TMEM lane quarter = warp & 3),
// then the producers (NPG groups of 128 threads, one thread per position plus the k-1 halo positions,
// round-robin over stages, loads two stages ahead), last warp = MMA issuer (one elected lane) + TMEM allocator.
// Tried and withdrawn for the several-groups variant (round 2; tools/conv1_time.py): raw fp32 rows
// streamed by cp.async.bulk into a second shared-memory ring so that the producers neither compute addresses nor hold
// prefetch registers.  Bit-identical, and no faster: 66.6 us with one copying lane, 58.5 us with one lane per channel plane,
// 59.4 us with a 12-stage ring, against 58.3 us for the register-prefetch producers -- half of the producers' time then
// went into waiting for their row (ncu source view), with ALL inputs resident in L2 as well (aliased sources, no flush:
// 60.4 us), so it is the bulk-copy path's rate for 2 KB copies (about four per 800 clk per SM) that paces it, not DRAM.
// Also tried: FIVE producer groups (one epilogue set, no bulk-copy warp: 25 warps, which the register file holds at 72
// registers per thread): 61.4-63.5 us against 58.3 us with four -- more staging warps only crowd the issue slots and the
// shared-memory pipe they share with the MMA operand fetches.
// Pipelines: a_full/a_empty (producers <-> MMA, NSTAGE smem stages; one stage = one input row of one
// 16-channel group), d_full/d_empty (MMA <-> epilogue, ND accumulators; D_r is released by the k output
// rows that read it).
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "tc05.cuh"

namespace pbmc {

// Role split (template parameter NPG of the kernel): 5 sets of 4 warps are divided between epilogue and producers.
//   NPG = 3: two epilogue sets (alternate output rows) + three producer groups -- one 16-channel group per row, where an
//            output row is due after every stage;
//   NPG = 4: one epilogue set + four producer groups -- several groups per row (conv[1]: 7 stages per output row), where
//            the epilogue idles and the producers' serial per-stage chain sets the pace.
constexpr int CR_SETS = 5;
constexpr int CR_MMA_WARP = 4 * CR_SETS;      // warps 0 .. 4*EPI_SETS-1 epilogue, then 4*NPG producer warps, then the MMA issuer
constexpr int CR_TMA_WARP = CR_MMA_WARP + 1;  // one lane bulk-copies the stages of operand-image (STAGED16) sources
constexpr int CR_THREADS = (CR_TMA_WARP + 1) * 32;
constexpr int CR_NT = 8;                                // stages of the bulk-copy ring (power of two)
constexpr int CR_MAXG = 24;
constexpr int CR_SMEM_HDR = 2176;

struct ConvRowParams {
  pbmc_src src[PBMC_MAX_SRC];
  int nsrc, B, H, W;
  int cout_blks, pad_mode, epi_act;
  int ngroups;  // 16-channel K groups over the concatenated sources
  int cin_ch;   // padded channel count of the concatenation (sum nblk * 4)
  int rpc;      // output rows per CTA
  int max_ctas; // CTA budget (0 = whole GPU)
  int has_staged;  // some source is an operand image: the bulk-copy ring is allocated
  const void* wpk;  // [group][dx][part][2 K-chunks][N = k*16 rows (dy, c_out)][8 c_in] 16-bit
  const float* wscale;  // 2^-e: the image holds the filters times 2^e (ops.prescale_pow2)
  const float* bias;
  float* out;
  double* out_stats;
  double* out_chan_sum;
  unsigned long long* trace;  // developer timeline (PBMC_ROW_TRACE builds only), else NULL
};

struct RowGroup {
  const float* base;  // first block of the group for this sample
  int nb;             // real 4-channel blocks (1..4); the rest of the 16 channels are zero
  int xform;
  int chan0;          // first channel in the xf_a / xf_b tables
  int staged;         // PBMC_LAYOUT_STAGED16: base = this sample's fp16 hi|lo operand image, rows are bulk-copied
};

// MERGE (k = 3, fp16 hi|lo): the hi*hi and hi*lo products share ONE N = 96 MMA -- B = [W_hi ; W_lo] stacked along N, so A_hi is
// fetched from shared memory once for both (the MMA is operand-fetch bound: 4 KB of A + 1.5 KB of B per N = 48 MMA at
// 128 B/clk) -- followed by the N = 48 MMA A_lo * W_hi on the first half: 6 MMAs and 37.5 KB of operand reads per stage
// instead of 9 and 49.5 KB.  An accumulator is then 96 columns, [0,48) = hi*hi + lo*hi and [48,96) = hi*lo, summed by the
// epilogue; the ring shrinks to 5 accumulators.
template <int KS, int PARTS, bool MERGE = false>
struct RowGeom {
  static_assert(!MERGE || (KS == 3 && PARTS == 2), "merged passes: 3x3, fp16 hi|lo only");
  static constexpr int P = KS / 2;
  static constexpr int N = KS * 16;
  static constexpr int DN = MERGE ? 2 * N : N;      // TMEM columns of one accumulator
  static constexpr int PWS = 128 + KS - 1;
  static constexpr int PLANE = (PWS + 7) / 8 * 8;   // positions per K-chunk plane (16 B each)
  static constexpr int PART_BYTES = 2 * PLANE * 16;  // two K chunks (8 channels each)
  static constexpr int STAGE_BYTES = PARTS * PART_BYTES;
  static constexpr int NSTAGE = 8;
  // accumulator ring: the MMA warp may run ND - KS rows ahead of the epilogue (measured with tools/probe:
  // dependent accumulation into the same TMEM columns costs nothing, one N = 48 MMA is ~44 clk)
  static constexpr int ND = MERGE ? 5 : (KS == 3 ? 10 : 6);
  static constexpr uint32_t TMEM_COLS = ND * DN <= 256 ? 256 : 512;
  static constexpr int B_TILE = 2 * N * 16;  // one (group, dx, part) operand: [2 chunks][N rows][16 B]
  static constexpr int B_GROUP = KS * PARTS * B_TILE;
  static_assert(ND * DN <= 512, "TMEM has 512 columns");
  static_assert(ND >= KS + 1, "the MMA must be able to run ahead of the epilogue");
};

#ifdef PBMC_ROW_TRACE
#define CR_TR(slot)                                                                              \
  do {                                                                                           \
    if (p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (slot) < 4096) \
      p.trace[(slot)] = clock64();                                                               \
  } while (0)
#else
#define CR_TR(slot) \
  do {              \
  } while (0)
#endif

template <int NWARPS>
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NWARPS * 32) : "memory"); }

__device__ __forceinline__ float xform1(float v, float a, float b, int xform) {
  if (xform == PBMC_XFORM_NONE) return v;
  if (xform != PBMC_XFORM_GELU) v = fmaf(v, a, b);
  if (xform != PBMC_XFORM_GN) v = gelu_erf(v);
  return v;
}

template <int KS, int PARTS, int NPG>
__global__ void __launch_bounds__(CR_THREADS, 1) conv_row_kernel(const __grid_constant__ ConvRowParams p) {
  constexpr bool MERGE = NPG == 4 && KS == 3 && PARTS == 2;  // the several-groups-per-row variant (conv[1]) merges two passes
  using G = RowGeom<KS, PARTS, MERGE>;
  constexpr int CR_NPG = NPG, EPI_SETS = CR_SETS - NPG, CR_EPI_WARPS = 4 * EPI_SETS;
  static_assert(NPG >= 1 && EPI_SETS >= 1, "role split");
  constexpr int P = G::P, N = G::N, DN = G::DN, NSTAGE = G::NSTAGE, ND = G::ND, PLANE = G::PLANE;
  static_assert(8 * (2 * NSTAGE + 2 * ND + 2 * CR_NT) <= 448, "barrier area");
  static_assert((NSTAGE & (NSTAGE - 1)) == 0, "NSTAGE must be a power of two");
  constexpr uint32_t FMT = PARTS == 2 ? 0u : 1u;  // fp16 hi|lo split, or one bf16 pass
  constexpr uint32_t IDESC = row_idesc(FMT, N);
  constexpr uint32_t IDESC2 = row_idesc(FMT, 2 * N);  // MERGE: A_hi x [W_hi ; W_lo]
  extern __shared__ __align__(128) unsigned char smem[];
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 448);  // barriers occupy [0, 8 * (2 NSTAGE + 2 ND))
  RowGroup* gtab = reinterpret_cast<RowGroup*>(smem + 512);
  double* red = reinterpret_cast<double*>(smem + 1152);             // 8 warps x 8 doubles
  float* bias_s = reinterpret_cast<float*>(smem + 1152 + 512);      // 16 floats (zero padded)
  int* nslist = reinterpret_cast<int*>(smem + 1152 + 512 + 64);     // the groups the producer warps stage (not bulk-copied), then their count
  uint32_t* stg_mask = reinterpret_cast<uint32_t*>(smem + 1152 + 512 + 64 + 4 * (CR_MAXG + 1));  // bit g: group g is an operand image
  unsigned char* Bs = smem + CR_SMEM_HDR;
  unsigned char* As = Bs + (size_t)p.ngroups * G::B_GROUP;
  float* xf_a = reinterpret_cast<float*>(As + (size_t)(NSTAGE + (p.has_staged ? CR_NT : 0)) * G::STAGE_BYTES);
  float* xf_b = xf_a + p.cin_ch;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z;
  const int x0 = blockIdx.y * 128;
  const int y0 = blockIdx.x * p.rpc;
  const int H = p.H, W = p.W;
  const int nrows = min(p.rpc, H - y0);
  const int nin = nrows + KS - 1;
  const int NG = p.ngroups;
  const int total = nin * NG;  // stage st = (input row ri, 16-channel group g), row-major: st = ri * NG + g
  const size_t plane_px = (size_t)H * W;
  const uint32_t bar0 = smem_u32(smem);
  auto a_full = [&](uint32_t s) { return bar0 + s * 8u; };
  auto a_empty = [&](uint32_t s) { return bar0 + (uint32_t)(NSTAGE + s) * 8u; };
  auto d_full = [&](uint32_t d) { return bar0 + (uint32_t)(2 * NSTAGE + d) * 8u; };
  auto d_empty = [&](uint32_t d) { return bar0 + (uint32_t)(2 * NSTAGE + ND + d) * 8u; };
  // Operand-image sources get their own ring (stages NSTAGE .. NSTAGE+CR_NT-1) and barriers: every barrier then has one
  // kind of waiter that sees all of its phases in order (a parity wait is unsound for a waiter that skips phases).
  auto t_full = [&](uint32_t s) { return bar0 + (uint32_t)(2 * NSTAGE + 2 * ND + s) * 8u; };
  auto t_empty = [&](uint32_t s) { return bar0 + (uint32_t)(2 * NSTAGE + 2 * ND + CR_NT + s) * 8u; };

  // ---- one-time setup
  if (tid == 0) {
    CR_TR(0);
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(a_full(s), 4);   // the 4 warps of the producer group that owns the stage
      mbar_init(a_empty(s), 1);  // tcgen05.commit
    }
    for (int d = 0; d < ND; ++d) {
      mbar_init(d_full(d), 1);        // tcgen05.commit
      mbar_init(d_empty(d), 4 * KS);  // 4 epilogue warps x the KS output rows that read D_d
    }
    for (int s = 0; s < CR_NT; ++s) {
      mbar_init(t_full(s), 1);   // arrive.expect_tx of the copying lane (+ the bytes of the four bulk copies)
      mbar_init(t_empty(s), 1);  // tcgen05.commit
    }
    fence_mbar_init();
    int g = 0, c0 = 0;
    for (int s = 0; s < p.nsrc; ++s) {
      const pbmc_src& S = p.src[s];
      for (int cb = 0; cb < S.nblk; cb += 4, ++g) {
        RowGroup gi;
        gi.base = S.ptr + ((size_t)b * S.nblk + cb) * plane_px * 4;
        gi.nb = min(4, S.nblk - cb);
        gi.xform = S.xform;
        gi.chan0 = c0 + cb * 4;
        gi.staged = S.layout == PBMC_LAYOUT_STAGED16;
        if (gi.staged)  // [H][part][chunk][Wp][8] halves per sample
          gi.base = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(S.ptr) +
                                                   (size_t)b * H * 4 * (size_t)((W + 127) / 128 * 128 + 2) * 16);
        gtab[g] = gi;
      }
      c0 += S.nblk * 4;
    }
    int nns = 0;
    uint32_t mask = 0;
    for (int q = 0; q < g; ++q) {
      if (gtab[q].staged) mask |= 1u << q;
      else nslist[nns++] = q;
    }
    nslist[CR_MAXG] = nns;
    *stg_mask = mask;
  }
  if (warp == CR_MMA_WARP) tmem_alloc(smem_u32(tmem_slot), G::TMEM_COLS);
  {
    // filters and bias are constants of the network: copied before the programmatic-dependent-launch wait
    if (tid < 16) bias_s[tid] = tid < p.cout_blks * 4 ? __ldg(p.bias + tid) : 0.f;
    const uint4* wsrc = reinterpret_cast<const uint4*>(p.wpk);
    uint4* wdst = reinterpret_cast<uint4*>(Bs);
    if (MERGE) {
      // [group][dx][part][chunk][48 rows] -> [group][dx][chunk][96 rows: hi 0..47 | lo 48..95]: one N = 96 operand per (group, dx)
      for (int e = tid; e < NG * (G::B_GROUP / 16); e += CR_THREADS) {
        const int q = e / (2 * N), row = e - q * (2 * N);  // q = (group, dx, part), row = chunk * N + r
        const int part = q & 1, chunk = row >= N;
        wdst[(q >> 1) * (4 * N) + chunk * (2 * N) + part * N + (row - chunk * N)] = __ldg(wsrc + e);
      }
    } else {
      for (int e = tid; e < NG * (G::B_GROUP / 16); e += CR_THREADS) wdst[e] = __ldg(wsrc + e);
    }
  }
  // Everything above overlaps the tail of the previous kernel in the stream when this kernel was launched with
  // programmatic stream serialization; the producer's outputs (activations, GroupNorm sums) are read only below.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  {
    int c0 = 0;
    for (int s = 0; s < p.nsrc; ++s) {
      const pbmc_src& S = p.src[s];
      for (int c = tid; c < S.nblk * 4; c += CR_THREADS) {
        float a = 1.f, bb = 0.f;
        if (S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN)
          gn_coeffs(S.stats + ((size_t)b * S.nblk + (c >> 2)) * 2, S.inv_count, S.gamma[c], S.beta[c], a, bb);
        xf_a[c0 + c] = a;
        xf_b[c0 + c] = bb;
      }
      c0 += S.nblk * 4;
    }
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next kernel may start its own prologue
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tid == 0) CR_TR(1);

  if (warp < CR_EPI_WARPS) {
    // ================================================================ epilogue: EPI_SETS sets of 4 warps,
    // set e takes output rows yo = e, e + EPI_SETS, ...; thread = output column (TMEM lane quarter = warp & 3)
    const int eset = warp >> 2, q = warp & 3;
    const int col = q * 32 + lane, gx = x0 + col;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    float cs[4] = {0.f, 0.f, 0.f, 0.f};  // zero-mean sums: only the c_out <= 4 head conv asks for them
    const bool want_cs = p.out_chan_sum != nullptr;
    const int cout_blks = p.cout_blks;
    const bool epi_gelu = p.epi_act == PBMC_ACT_GELU;
    const uint32_t bias_addr = smem_u32(bias_s);
    const float wsc = __ldg(p.wscale);
    float* orow = p.out + (((size_t)b * cout_blks) * plane_px + (size_t)(y0 + eset) * W + gx) * 4;
    const size_t blk_stride = plane_px * 4, row_stride = (size_t)EPI_SETS * W * 4;
    const bool col_in = gx < W;
    // The epilogue's instruction stream is the busiest in the CTA (ncu: half of all issued instructions), so
    // the common shape -- 16 outputs, no activation, no channel sums -- gets a loop with nothing else in it.
    auto row_loop = [&](auto lean_tag) {
      constexpr bool LEAN = decltype(lean_tag)::value;
      // ring positions advance by EPI_SETS rows per iteration
      uint32_t s_lo = (uint32_t)eset % ND, s_hi = (uint32_t)(eset + KS - 1) % ND, par_hi = ((uint32_t)(eset + KS - 1) / ND) & 1u;
      for (int yo = eset; yo < nrows; yo += EPI_SETS) {
        mbar_wait_parked(d_full(s_hi), par_hi);  // the last input row this output row needs (commits are in order)
        tc_fence_after();
        if ((tid & 127) == 0) CR_TR(1200 + 3 * yo);
        uint32_t r[KS][16];
        uint32_t sl = s_lo;
#pragma unroll
        for (int dy = 0; dy < KS; ++dy) {
          tmem_ld16_issue(lane_addr + sl * (uint32_t)DN + (uint32_t)(dy * 16), r[dy]);
          if (++sl == (uint32_t)ND) sl = 0;
        }
#pragma unroll
        for (int dy = 0; dy < KS; ++dy) tmem_ld_wait16(r[dy]);
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
        if ((tid & 127) == 0) CR_TR(1201 + 3 * yo);
        if (col_in) {
#pragma unroll
          for (int qb = 0; qb < 4; ++qb) {
            if (LEAN || qb < cout_blks) {
              float4 bq;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bq.x), "=f"(bq.y), "=f"(bq.z), "=f"(bq.w) : "r"(bias_addr + qb * 16));
              const float bias4[4] = {bq.x, bq.y, bq.z, bq.w};
              float o[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float a = __uint_as_float(r[0][qb * 4 + e]);
#pragma unroll
                for (int dy = 1; dy < KS; ++dy) a += __uint_as_float(r[dy][qb * 4 + e]);
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
        orow += row_stride;
        s_lo += EPI_SETS; if (s_lo >= (uint32_t)ND) s_lo -= ND;
        s_hi += EPI_SETS; if (s_hi >= (uint32_t)ND) { s_hi -= ND; par_hi ^= 1u; }
        if ((tid & 127) == 0) CR_TR(1202 + 3 * yo);
      }
    };
    // MERGE: an accumulator is [0,48) = hi*hi + lo*hi | [48,96) = hi*lo; two halves of 8 output channels keep 48 values live
    auto row_loop_merged = [&]() {
      uint32_t s_lo = (uint32_t)eset % ND, s_hi = (uint32_t)(eset + KS - 1) % ND, par_hi = ((uint32_t)(eset + KS - 1) / ND) & 1u;
      for (int yo = eset; yo < nrows; yo += EPI_SETS) {
        mbar_wait_parked(d_full(s_hi), par_hi);
        tc_fence_after();
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
          uint32_t ra[KS][8], rb[KS][8];
          uint32_t sl = s_lo;
#pragma unroll
          for (int dy = 0; dy < KS; ++dy) {
            tmem_ld8_issue(lane_addr + sl * (uint32_t)DN + (uint32_t)(dy * 16 + hq * 8), ra[dy]);
            tmem_ld8_issue(lane_addr + sl * (uint32_t)DN + (uint32_t)(N + dy * 16 + hq * 8), rb[dy]);
            if (++sl == (uint32_t)ND) sl = 0;
          }
#pragma unroll
          for (int dy = 0; dy < KS; ++dy) { tmem_ld_wait8(ra[dy]); tmem_ld_wait8(rb[dy]); }
          if (hq == 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              sl = s_lo;
#pragma unroll
              for (int dy = 0; dy < KS; ++dy) {
                mbar_arrive_n(d_empty(sl), yo == 0 ? (uint32_t)(KS - dy) : 1u);
                if (++sl == (uint32_t)ND) sl = 0;
              }
            }
          }
          if (col_in) {
#pragma unroll
            for (int qh = 0; qh < 2; ++qh) {
              const int qb = 2 * hq + qh;
              if (qb < cout_blks) {
                float4 bq;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bq.x), "=f"(bq.y), "=f"(bq.z), "=f"(bq.w) : "r"(bias_addr + qb * 16));
                const float bias4[4] = {bq.x, bq.y, bq.z, bq.w};
                float o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float a = __uint_as_float(ra[0][qh * 4 + e]), c = __uint_as_float(rb[0][qh * 4 + e]);
#pragma unroll
                  for (int dy = 1; dy < KS; ++dy) {
                    a += __uint_as_float(ra[dy][qh * 4 + e]);
                    c += __uint_as_float(rb[dy][qh * 4 + e]);
                  }
                  a = fmaf(a + c, wsc, bias4[e]);
                  if (epi_gelu) a = gelu_erf(a);
                  o[e] = a;
                }
                *reinterpret_cast<float4*>(orow + qb * blk_stride) = make_float4(o[0], o[1], o[2], o[3]);
                s1[qb] += (o[0] + o[1]) + (o[2] + o[3]);
                s2[qb] = fmaf(o[0], o[0], fmaf(o[1], o[1], fmaf(o[2], o[2], fmaf(o[3], o[3], s2[qb]))));
                if (qb == 0 && want_cs) { cs[0] += o[0]; cs[1] += o[1]; cs[2] += o[2]; cs[3] += o[3]; }
              }
            }
          }
        }
        orow += row_stride;
        s_lo += EPI_SETS; if (s_lo >= (uint32_t)ND) s_lo -= ND;
        s_hi += EPI_SETS; if (s_hi >= (uint32_t)ND) { s_hi -= ND; par_hi ^= 1u; }
      }
    };
    if (MERGE)
      row_loop_merged();
    else if (cout_blks == 4 && !epi_gelu && !want_cs)
      row_loop(std::true_type{});
    else
      row_loop(std::false_type{});
    if (tid == 0) CR_TR(3);
    if (p.out_stats != nullptr) {
#pragma unroll
      for (int qb = 0; qb < 4; ++qb) {
        const double a = warp_sum((double)s1[qb]);
        const double c2 = warp_sum((double)s2[qb]);
        if (lane == 0) { red[(warp * 4 + qb) * 2] = a; red[(warp * 4 + qb) * 2 + 1] = c2; }
      }
      epi_bar_sync<CR_EPI_WARPS>();
      if (tid < 8 && (tid >> 1) < p.cout_blks) {
        double t = 0.0;
        for (int w = 0; w < CR_EPI_WARPS; ++w) t += red[(w * 4 + (tid >> 1)) * 2 + (tid & 1)];
        atomicAdd(p.out_stats + ((size_t)b * p.cout_blks + (tid >> 1)) * 2 + (tid & 1), t);
      }
      epi_bar_sync<CR_EPI_WARPS>();
    }
    if (want_cs) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const double a = warp_sum((double)cs[c]);
        if (lane == 0) red[warp * 4 + c] = a;
      }
      epi_bar_sync<CR_EPI_WARPS>();
      if (tid < 4) {
        double t = 0.0;
        for (int w = 0; w < CR_EPI_WARPS; ++w) t += red[w * 4 + tid];
        atomicAdd(p.out_chan_sum + (size_t)b * 4 + tid, t);
      }
    }
  } else if (warp < CR_MMA_WARP) {
    // ================================================================ producers: NPG groups of 128 threads,
    // one thread per position; group pg owns stages pg, pg + NPG, ...  Warp 0 of a group also produces the
    // KS-1 halo positions (one channel per lane).  Loads run TWO stages ahead and are issued right after
    // the stage's fence: fence.proxy.async is MEMBAR + FENCE.VIEW.ASYNC, and the MEMBAR would otherwise wait
    // for freshly issued prefetch loads.
    const int pw = warp - CR_EPI_WARPS;
    const int pg = pw >> 2, wq = pw & 3;
    if (lane == 0 && wq == 0) CR_TR(4 + pg);
    const int i = wq * 32 + lane;
    const int gxp = x0 - P + i;
    const int sx = pad_index(gxp, W, p.pad_mode);
    const bool col_ok = gxp < W + P && sx >= 0;  // columns past the image feed masked outputs only
    constexpr int HITEMS = ((KS - 1) * 16 + 31) / 32;
    const bool tr_lane = lane == 0 && wq == 0;
    (void)tr_lane;
    int hsx[HITEMS];
    bool hok[HITEMS];
#pragma unroll
    for (int k = 0; k < HITEMS; ++k) {
      const int item = lane + 32 * k, e = item >> 4;
      const int gxh = x0 - P + 128 + e;
      hsx[k] = pad_index(gxh, W, p.pad_mode);
      hok[k] = wq == 0 && e < KS - 1 && gxh < W + P && hsx[k] >= 0;
    }
    struct Buf {
      float4 v[4];
      float h[HITEMS];
      bool ok;
    };
    auto load_stage = [&](int ri, int g, Buf& B) {
      const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
      const RowGroup gi = gtab[g];
      B.ok = sy >= 0;
      const bool ok = col_ok && sy >= 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        B.v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok && j < gi.nb) B.v[j] = ldg4(gi.base + ((size_t)j * plane_px + (size_t)sy * W + sx) * 4);
      }
#pragma unroll
      for (int k = 0; k < HITEMS; ++k) {
        const int ch = (lane + 32 * k) & 15;
        B.h[k] = 0.f;
        if (hok[k] && sy >= 0 && (ch >> 2) < gi.nb)
          B.h[k] = __ldg(gi.base + ((size_t)(ch >> 2) * plane_px + (size_t)sy * W + hsx[k]) * 4 + (ch & 3));
      }
    };
    auto process = [&](int st, int g, Buf& B) {
      if (tr_lane) CR_TR(100 + pg * 300 + 4 * (st / CR_NPG));
      const RowGroup gi = gtab[g];
      float v[16];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[4 * j + 0] = B.v[j].x; v[4 * j + 1] = B.v[j].y; v[4 * j + 2] = B.v[j].z; v[4 * j + 3] = B.v[j].w;
      }
      float hv[HITEMS];
#pragma unroll
      for (int k = 0; k < HITEMS; ++k) hv[k] = B.h[k];
      if (B.ok && gi.xform != PBMC_XFORM_NONE) {
        const float4* a4 = reinterpret_cast<const float4*>(xf_a + gi.chan0);
        const float4* b4 = reinterpret_cast<const float4*>(xf_b + gi.chan0);
        const bool do_gn = gi.xform != PBMC_XFORM_GELU, do_gelu = gi.xform != PBMC_XFORM_GN;
        if (col_ok) {
          if (gi.nb == 4 && gi.xform == PBMC_XFORM_GN_GELU) {
            // the trunk's shape, branch-free: 16 independent GN+GELU chains that the scheduler can interleave
            // (a lone warp is latency-bound on the 10-FMA polynomial: 706 clk per 16 values vs 325 clk of issue)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 a = a4[j], bb = b4[j];
              v[4 * j + 0] = fmaf(v[4 * j + 0], a.x, bb.x); v[4 * j + 1] = fmaf(v[4 * j + 1], a.y, bb.y);
              v[4 * j + 2] = fmaf(v[4 * j + 2], a.z, bb.z); v[4 * j + 3] = fmaf(v[4 * j + 3], a.w, bb.w);
            }
#pragma unroll
            for (int c = 0; c < 16; c += 2) gelu_erf2(v[c], v[c + 1]);  // packed fp32x2 FMAs, bit-identical to gelu_erf
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (j < gi.nb) {  // absent blocks of a partial group stay exactly zero
                if (do_gn) {
                  const float4 a = a4[j], bb = b4[j];
                  v[4 * j + 0] = fmaf(v[4 * j + 0], a.x, bb.x); v[4 * j + 1] = fmaf(v[4 * j + 1], a.y, bb.y);
                  v[4 * j + 2] = fmaf(v[4 * j + 2], a.z, bb.z); v[4 * j + 3] = fmaf(v[4 * j + 3], a.w, bb.w);
                }
                if (do_gelu) {
#pragma unroll
                  for (int e = 0; e < 4; ++e) v[4 * j + e] = gelu_erf(v[4 * j + e]);
                }
              }
            }
          }
        }
#pragma unroll
        for (int k = 0; k < HITEMS; ++k) {
          const int ch = (lane + 32 * k) & 15;
          if (hok[k] && (ch >> 2) < gi.nb) {
            if (do_gn) hv[k] = fmaf(hv[k], xf_a[gi.chan0 + ch], xf_b[gi.chan0 + ch]);
            if (do_gelu) hv[k] = gelu_erf(hv[k]);
          }
        }
      }
      const uint32_t slot = (uint32_t)st & (NSTAGE - 1);
      unsigned char* stage_b = As + (size_t)slot * G::STAGE_BYTES;
      uint4* stage = reinterpret_cast<uint4*>(stage_b);
      if (tr_lane) CR_TR(101 + pg * 300 + 4 * (st / CR_NPG));
      mbar_wait_parked(a_empty(slot), (((uint32_t)st / NSTAGE) & 1u) ^ 1u);
      if (tr_lane) CR_TR(102 + pg * 300 + 4 * (st / CR_NPG));
      if (PARTS == 2) {
        uint4 h0, l0, h1, l1;
        split_f16(v, h0, l0);
        split_f16(v + 8, h1, l1);
        stage[i] = h0;
        stage[PLANE + i] = h1;
        stage[2 * PLANE + i] = l0;
        stage[3 * PLANE + i] = l1;
      } else {
        stage[i] = pack_bf16(v);
        stage[PLANE + i] = pack_bf16(v + 8);
      }
      if (wq == 0) {
#pragma unroll
        for (int k = 0; k < HITEMS; ++k) {
          const int item = lane + 32 * k, e = item >> 4, ch = item & 15;
          if (e < KS - 1) {
            const size_t off = ((size_t)(ch >> 3) * PLANE + 128 + e) * 16 + (size_t)(ch & 7) * 2;
            if (PARTS == 2) {
              const __half h = __float2half_rn(hv[k]);
              const __half l = __float2half_rn(hv[k] - __half2float(h));
              *reinterpret_cast<__half*>(stage_b + off) = h;
              *reinterpret_cast<__half*>(stage_b + G::PART_BYTES + off) = l;
            } else {
              *reinterpret_cast<__nv_bfloat16*>(stage_b + off) = __float2bfloat16_rn(hv[k]);
            }
          }
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full(slot));
      if (tr_lane) CR_TR(103 + pg * 300 + 4 * (st / CR_NPG));
    };
    auto advance = [&](int& ri, int& g) {
      g += CR_NPG;
      while (g >= NG) { g -= NG; ++ri; }
    };
    // ---- fast path: ONE full 16-channel group (every trunk layer and the two last head convs: 25 of the 28 convs
    // of a forward).  A stage is then simply an input row; everything that does not change from row to row is
    // hoisted, the body is straight-line: the generic loop below spends ~330 instructions per stage on
    // bookkeeping and the stage rate of a CTA is bounded by exactly this serial, single-warp chain.
    if (NG == 1 && gtab[0].nb == 4 && !gtab[0].staged && (gtab[0].xform == PBMC_XFORM_NONE || gtab[0].xform == PBMC_XFORM_GN_GELU)) {
      const RowGroup gi = gtab[0];
      const bool do_x = gi.xform == PBMC_XFORM_GN_GELU;
      const size_t pstride = plane_px * 4;
      const float* cb0 = gi.base + (size_t)(sx < 0 ? 0 : sx) * 4;  // this thread's column, channel block 0
      const float* cb1 = cb0 + pstride;
      const float* cb2 = cb1 + pstride;
      const float* cb3 = cb2 + pstride;
      // halo (warp 0 of the group, KS == 3: lane = (extra position e, channel ch))
      const int hch = lane & 15, he = lane >> 4;
      const bool h_on = wq == 0 && hok[0];
      const float* hbase = gi.base + (size_t)(hch >> 2) * pstride + (size_t)(h_on ? hsx[0] : 0) * 4 + (hch & 3);
      const float h_a = do_x ? xf_a[gi.chan0 + hch] : 1.f, h_b = do_x ? xf_b[gi.chan0 + hch] : 0.f;
      const uint32_t h_off = (uint32_t)(((hch >> 3) * PLANE + 128 + he) * 16 + (hch & 7) * 2);
      const uint32_t as_addr = smem_u32(As) + (uint32_t)i * 16u;
      const uint32_t xfa_addr = smem_u32(xf_a + gi.chan0), xfb_addr = smem_u32(xf_b + gi.chan0);
      const size_t rstride = (size_t)W * 4;
      struct FBuf {
        float4 v0, v1, v2, v3;
        float h;
        bool ok;
      };
      auto fload = [&](int ri, FBuf& B) {
        const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
        B.ok = sy >= 0;
        const size_t ro = (size_t)(sy < 0 ? 0 : sy) * rstride;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        B.v0 = B.v1 = B.v2 = B.v3 = z;
        B.h = 0.f;
        if (col_ok && sy >= 0) {
          B.v0 = ldg4(cb0 + ro); B.v1 = ldg4(cb1 + ro); B.v2 = ldg4(cb2 + ro); B.v3 = ldg4(cb3 + ro);
        }
        if (h_on && sy >= 0) B.h = __ldg(hbase + ro);
      };
      auto fproc = [&](int st, FBuf& B) {
        if (tr_lane) CR_TR(100 + pg * 300 + 8 * (st / CR_NPG));
        float v[16] = {B.v0.x, B.v0.y, B.v0.z, B.v0.w, B.v1.x, B.v1.y, B.v1.z, B.v1.w,
                       B.v2.x, B.v2.y, B.v2.z, B.v2.w, B.v3.x, B.v3.y, B.v3.z, B.v3.w};
        float hv = B.h;
        if (do_x && B.ok) {
          if (col_ok) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float4 a, bb;
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(xfa_addr + j * 16));
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bb.x), "=f"(bb.y), "=f"(bb.z), "=f"(bb.w) : "r"(xfb_addr + j * 16));
              v[4 * j + 0] = fmaf(v[4 * j + 0], a.x, bb.x); v[4 * j + 1] = fmaf(v[4 * j + 1], a.y, bb.y);
              v[4 * j + 2] = fmaf(v[4 * j + 2], a.z, bb.z); v[4 * j + 3] = fmaf(v[4 * j + 3], a.w, bb.w);
            }
#pragma unroll
            for (int c2 = 0; c2 < 16; c2 += 2) gelu_erf2(v[c2], v[c2 + 1]);
          }
          if (h_on) hv = gelu_erf(fmaf(hv, h_a, h_b));
        }
        const uint32_t slot = (uint32_t)st & (NSTAGE - 1);
        const uint32_t sa = as_addr + slot * (uint32_t)G::STAGE_BYTES;
        if (tr_lane) CR_TR(101 + pg * 300 + 8 * (st / CR_NPG));
        if (st >= NSTAGE) mbar_wait_parked(a_empty(slot), (((uint32_t)st / NSTAGE) & 1u) ^ 1u);  // first pass: ring is free
        if (tr_lane) CR_TR(102 + pg * 300 + 8 * (st / CR_NPG));
        auto sts = [](uint32_t addr, uint4 q) {
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
        };
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
        if (wq == 0 && he < KS - 1) {
          const uint32_t ha = smem_u32(As) + slot * (uint32_t)G::STAGE_BYTES + h_off;
          if (PARTS == 2) {
            const __half hh = __float2half_rn(hv);
            const __half hl = __float2half_rn(hv - __half2float(hh));
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__half_as_ushort(hh)) : "memory");
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha + (uint32_t)G::PART_BYTES), "h"(__half_as_ushort(hl)) : "memory");
          } else {
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__bfloat16_as_ushort(__float2bfloat16_rn(hv))) : "memory");
          }
        }
        if (tr_lane) CR_TR(104 + pg * 300 + 8 * (st / CR_NPG));
        fence_proxy_async_smem();
        if (tr_lane) CR_TR(105 + pg * 300 + 8 * (st / CR_NPG));
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full(slot));
        if (tr_lane) CR_TR(103 + pg * 300 + 8 * (st / CR_NPG));
      };
      static_assert(KS == 3 || HITEMS == 2, "halo lanes");
      if (KS == 3) {
        FBuf f0, f1;
        if (tr_lane) CR_TR(8 + pg);
        if (pg < nin) fload(pg, f0);
        if (pg + CR_NPG < nin) fload(pg + CR_NPG, f1);
        for (int st = pg; st < nin; st += 2 * CR_NPG) {
          fproc(st, f0);
          if (st + 2 * CR_NPG < nin) fload(st + 2 * CR_NPG, f0);
          if (tr_lane) CR_TR(106 + pg * 300 + 8 * (st / CR_NPG));
          if (st + CR_NPG < nin) {
            fproc(st + CR_NPG, f1);
            if (st + 3 * CR_NPG < nin) fload(st + 3 * CR_NPG, f1);
          }
        }
        goto producer_done;
      }
    }
    // ---- lean path for several groups / partial groups (conv[1]: 7 sources, conv[0]: 8 of 16 channels) with
    // xform NONE or GN+GELU per group: same straight-line body, the group's few parameters travel with the buffer
    if (KS == 3) {
      bool simple = true;
      for (int g = 0; g < NG; ++g) simple = simple && (gtab[g].xform == PBMC_XFORM_NONE || gtab[g].xform == PBMC_XFORM_GN_GELU);
      if (simple) {
        const size_t pstride = plane_px * 4;
        const size_t coff = (size_t)(sx < 0 ? 0 : sx) * 4;
        const int hch = lane & 15, he = lane >> 4;
        const bool h_on = wq == 0 && hok[0];
        const size_t hoff = (size_t)(hch >> 2) * pstride + (size_t)(h_on ? hsx[0] : 0) * 4 + (hch & 3);
        const uint32_t h_off = (uint32_t)(((hch >> 3) * PLANE + 128 + he) * 16 + (hch & 7) * 2);
        const uint32_t as_addr = smem_u32(As) + (uint32_t)i * 16u;
        const uint32_t xfa0 = smem_u32(xf_a), xfb0 = smem_u32(xf_b);
        const size_t rstride = (size_t)W * 4;
        struct GBuf {
          float4 v0, v1, v2, v3;
          float h;
          int chan0;  // >= 0: GN+GELU with the tables at chan0; -1: plain
          int nb;
        };
        auto gload = [&](int ri, int g, GBuf& B) {
          const int sy = pad_index(y0 - P + ri, H, p.pad_mode);
          const RowGroup gi = gtab[g];
          B.chan0 = (gi.xform == PBMC_XFORM_GN_GELU && sy >= 0) ? gi.chan0 : -1;
          B.nb = gi.nb;
          const size_t ro = (size_t)(sy < 0 ? 0 : sy) * rstride;
          const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
          B.v0 = B.v1 = B.v2 = B.v3 = z;
          B.h = 0.f;
          const float* cb = gi.base + coff + ro;
          if (col_ok && sy >= 0) {
            B.v0 = ldg4(cb);
            if (gi.nb > 1) B.v1 = ldg4(cb + pstride);
            if (gi.nb > 2) B.v2 = ldg4(cb + 2 * pstride);
            if (gi.nb > 3) B.v3 = ldg4(cb + 3 * pstride);
          }
          if (h_on && sy >= 0 && (hch >> 2) < gi.nb) B.h = __ldg(gi.base + hoff + ro);
        };
        auto gproc = [&](int st, GBuf& B) {
          if (tr_lane && st / CR_NPG < 37) CR_TR(100 + pg * 300 + 8 * (st / CR_NPG));
          float v[16] = {B.v0.x, B.v0.y, B.v0.z, B.v0.w, B.v1.x, B.v1.y, B.v1.z, B.v1.w,
                         B.v2.x, B.v2.y, B.v2.z, B.v2.w, B.v3.x, B.v3.y, B.v3.z, B.v3.w};
          float hv = B.h;
          if (B.chan0 >= 0) {
            if (col_ok) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (j < B.nb) {
                  float4 a, bb;
                  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(xfa0 + (B.chan0 + 4 * j) * 4));
                  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(bb.x), "=f"(bb.y), "=f"(bb.z), "=f"(bb.w) : "r"(xfb0 + (B.chan0 + 4 * j) * 4));
                  v[4 * j + 0] = fmaf(v[4 * j + 0], a.x, bb.x); v[4 * j + 1] = fmaf(v[4 * j + 1], a.y, bb.y);
                  v[4 * j + 2] = fmaf(v[4 * j + 2], a.z, bb.z); v[4 * j + 3] = fmaf(v[4 * j + 3], a.w, bb.w);
                  gelu_erf2(v[4 * j + 0], v[4 * j + 1]);
                  gelu_erf2(v[4 * j + 2], v[4 * j + 3]);
                }
              }
            }
            if (h_on && (hch >> 2) < B.nb) hv = gelu_erf(fmaf(hv, xf_a[B.chan0 + hch], xf_b[B.chan0 + hch]));
          }
          const uint32_t slot = (uint32_t)st & (NSTAGE - 1);
          const uint32_t sa = as_addr + slot * (uint32_t)G::STAGE_BYTES;
          if (tr_lane && st / CR_NPG < 37) CR_TR(101 + pg * 300 + 8 * (st / CR_NPG));
          if (st >= NSTAGE) mbar_wait_parked(a_empty(slot), (((uint32_t)st / NSTAGE) & 1u) ^ 1u);  // first pass: ring is free
          if (tr_lane && st / CR_NPG < 37) CR_TR(102 + pg * 300 + 8 * (st / CR_NPG));
          auto sts = [](uint32_t addr, uint4 q) {
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
          };
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
          if (wq == 0 && he < KS - 1) {
            const uint32_t ha = smem_u32(As) + slot * (uint32_t)G::STAGE_BYTES + h_off;
            if (PARTS == 2) {
              const __half hh = __float2half_rn(hv);
              const __half hl = __float2half_rn(hv - __half2float(hh));
              asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__half_as_ushort(hh)) : "memory");
              asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha + (uint32_t)G::PART_BYTES), "h"(__half_as_ushort(hl)) : "memory");
            } else {
              asm volatile("st.shared.b16 [%0], %1;" ::"r"(ha), "h"(__bfloat16_as_ushort(__float2bfloat16_rn(hv))) : "memory");
            }
          }
          if (tr_lane && st / CR_NPG < 37) CR_TR(104 + pg * 300 + 8 * (st / CR_NPG));
          fence_proxy_async_smem();
          if (tr_lane && st / CR_NPG < 37) CR_TR(105 + pg * 300 + 8 * (st / CR_NPG));
          __syncwarp();
          if (lane == 0) mbar_arrive(a_full(slot));
          if (tr_lane && st / CR_NPG < 37) CR_TR(103 + pg * 300 + 8 * (st / CR_NPG));
        };
        // The producer warps stage the groups that are not operand images (nslist), in (row, group) order, the k-th
        // such stage in slot k % NSTAGE of their own ring; group pg takes k = pg, pg + NPG, ...
        const int nns = nslist[CR_MAXG];
        const int total_ns = nin * nns;
        GBuf g0, g1;
        auto kload = [&](int k, GBuf& B) {
          const int ri = k / nns;
          gload(ri, nslist[k - ri * nns], B);
        };
        if (pg < total_ns) kload(pg, g0);
        if (pg + CR_NPG < total_ns) kload(pg + CR_NPG, g1);
        for (int k = pg; k < total_ns; k += 2 * CR_NPG) {
          gproc(k, g0);
          if (k + 2 * CR_NPG < total_ns) kload(k + 2 * CR_NPG, g0);
          if (tr_lane && k / CR_NPG < 37) CR_TR(106 + pg * 300 + 8 * (k / CR_NPG));
          if (k + CR_NPG < total_ns) {
            gproc(k + CR_NPG, g1);
            if (k + 3 * CR_NPG < total_ns) kload(k + 3 * CR_NPG, g1);
          }
        }
        goto producer_done;
      }
    }
    {
    Buf b0, b1;
    int cg = pg, cri = 0;  // (row, group) of the stage processed next
    while (cg >= NG) { cg -= NG; ++cri; }
    int lri = cri, lg = cg;  // (row, group) of the stage loaded next
    if (pg < total) load_stage(lri, lg, b0);
    advance(lri, lg);
    if (pg + CR_NPG < total) load_stage(lri, lg, b1);
    advance(lri, lg);
    for (int st = pg; st < total; st += 2 * CR_NPG) {
      process(st, cg, b0);
      if (st + 2 * CR_NPG < total) load_stage(lri, lg, b0);
      advance(lri, lg);
      advance(cri, cg);
      if (st + CR_NPG < total) {
        process(st + CR_NPG, cg, b1);
        if (st + 3 * CR_NPG < total) load_stage(lri, lg, b1);
        advance(lri, lg);
        advance(cri, cg);
      }
    }
    }
  producer_done:;
  } else if (warp == CR_MMA_WARP) {
    // ================================================================ MMA issuer
    // The whole warp walks the (uniform) pipeline state; one elected lane issues tcgen05.mma / commit.
    // This warp's serial instruction stream bounds the stage rate, so everything is incremental: descriptors
    // are base + small constant (the 14-bit address field cannot carry: smem < 256 KB), and the barrier of
    // the NEXT stage is tested (non-blocking) before the current stage's MMAs are issued, so its latency hides
    // behind the (back-pressured, ~400 clk) issue of 9 MMAs.
    // Stage (ri, g) lives in the producers' ring (its pk-th stage) or, for an operand-image group, in the bulk-copy
    // ring (its tk-th stage); with no such group pk is simply the stage number.
    const bool leader = elect_one();
    constexpr uint32_t A_LBO = PLANE * 16, B_LBO = (MERGE ? 2 * N : N) * 16, SBO = 128;
    const uint64_t a_desc0 = umma_desc(smem_u32(As), A_LBO, SBO), b_desc0 = umma_desc(smem_u32(Bs), B_LBO, SBO);
    const uint32_t smask = *stg_mask;
    auto sel = [&](int g, uint32_t pk, uint32_t tk, uint32_t& full, uint32_t& par, uint32_t& sidx, uint32_t& empty) {
      if ((smask >> g) & 1u) {
        const uint32_t s = tk & (CR_NT - 1);
        full = t_full(s); par = (tk / CR_NT) & 1u; sidx = NSTAGE + s; empty = t_empty(s);
      } else {
        const uint32_t s = pk & (NSTAGE - 1);
        full = a_full(s); par = (pk / NSTAGE) & 1u; sidx = s; empty = a_empty(s);
      }
    };
    if (smask == 0u) {
      // no operand-image group: the stage number is the ring position (this loop is the pace-maker of every plain
      // conv; the general one below costs ~10 % more per stage)
      uint32_t ds = 0, d_par = 0;
      int st = 0;
      bool ready = total > 0 && mbar_test(a_full(0), 0u);
      for (int ri = 0; ri < nin; ++ri) {
        if (ri >= ND) mbar_wait(d_empty(ds), d_par ^ 1u);  // first ND rows: the ring is free
        const uint32_t dcol = tmem_base + ds * (uint32_t)DN;
        for (int g = 0; g < NG; ++g, ++st) {
          const uint32_t slot = (uint32_t)st & (NSTAGE - 1);
          if (!ready) mbar_wait(a_full(slot), ((uint32_t)st / NSTAGE) & 1u);
          tc_fence_after();
          ready = (st + 1 < total) && mbar_test(a_full((uint32_t)(st + 1) & (NSTAGE - 1)), ((uint32_t)(st + 1) / NSTAGE) & 1u);
          if (leader) {
            CR_TR(1400 + 2 * st);
            const uint64_t a_s = a_desc0 + (uint64_t)(slot * (uint32_t)(G::STAGE_BYTES >> 4));
            const uint64_t b_s = b_desc0 + (uint64_t)((uint32_t)g * (uint32_t)(G::B_GROUP >> 4));
#pragma unroll
            for (int dx = 0; dx < KS; ++dx) {
              const uint64_t a_hi = a_s + (uint64_t)dx;  // one position = 16 B
              const uint64_t b_hi = b_s + (uint64_t)(dx * PARTS * (G::B_TILE >> 4));
              if (MERGE) {
                umma_ss<1>(dcol, a_hi, b_hi, IDESC2, (uint32_t)(g | dx));                          // A_hi x [W_hi ; W_lo] -> 96 columns
                umma_ss<1>(dcol, a_hi + (uint64_t)(G::PART_BYTES >> 4), b_hi, IDESC, 1u);          // A_lo x W_hi -> the first 48
              } else {
                umma_ss<1>(dcol, a_hi, b_hi, IDESC, (uint32_t)(g | dx));
                if (PARTS == 2) {
                  umma_ss<1>(dcol, a_hi + (uint64_t)(G::PART_BYTES >> 4), b_hi, IDESC, 1u);
                  umma_ss<1>(dcol, a_hi, b_hi + (uint64_t)(G::B_TILE >> 4), IDESC, 1u);
                }
              }
            }
            umma_commit(a_empty(slot));                // frees the smem stage once these MMAs have read it
            if (g == NG - 1) umma_commit(d_full(ds));  // D_ri complete
            CR_TR(1401 + 2 * st);
          }
        }
        if (++ds == (uint32_t)ND) { ds = 0; d_par ^= 1u; }
      }
    } else {
      uint32_t ds = 0, d_par = 0, pk = 0, tk = 0;
      int st = 0;
      uint32_t full = 0, par = 0, sidx = 0, empty = 0;
      if (total > 0) sel(0, 0u, 0u, full, par, sidx, empty);
      bool ready = total > 0 && mbar_test(full, par);
      for (int ri = 0; ri < nin; ++ri) {
        if (ri >= ND) mbar_wait(d_empty(ds), d_par ^ 1u);  // first ND rows: the ring is free
        const uint32_t dcol = tmem_base + ds * (uint32_t)DN;
        for (int g = 0; g < NG; ++g, ++st) {
          if (!ready) mbar_wait(full, par);
          tc_fence_after();
          const uint32_t c_sidx = sidx, c_empty = empty;
          if ((smask >> g) & 1u) ++tk; else ++pk;
          if (st + 1 < total) {
            sel(g + 1 == NG ? 0 : g + 1, pk, tk, full, par, sidx, empty);
            ready = mbar_test(full, par);
          }
          if (leader) {
            CR_TR(1400 + 2 * st);
            const uint64_t a_s = a_desc0 + (uint64_t)(c_sidx * (uint32_t)(G::STAGE_BYTES >> 4));
            const uint64_t b_s = b_desc0 + (uint64_t)((uint32_t)g * (uint32_t)(G::B_GROUP >> 4));
  #pragma unroll
            for (int dx = 0; dx < KS; ++dx) {
              const uint64_t a_hi = a_s + (uint64_t)dx;  // one position = 16 B
              const uint64_t b_hi = b_s + (uint64_t)(dx * PARTS * (G::B_TILE >> 4));
              if (MERGE) {
                umma_ss<1>(dcol, a_hi, b_hi, IDESC2, (uint32_t)(g | dx));                          // A_hi x [W_hi ; W_lo] -> 96 columns
                umma_ss<1>(dcol, a_hi + (uint64_t)(G::PART_BYTES >> 4), b_hi, IDESC, 1u);          // A_lo x W_hi -> the first 48
              } else {
                umma_ss<1>(dcol, a_hi, b_hi, IDESC, (uint32_t)(g | dx));
                if (PARTS == 2) {
                  umma_ss<1>(dcol, a_hi + (uint64_t)(G::PART_BYTES >> 4), b_hi, IDESC, 1u);
                  umma_ss<1>(dcol, a_hi, b_hi + (uint64_t)(G::B_TILE >> 4), IDESC, 1u);
                }
              }
            }
            umma_commit(c_empty);                      // frees the smem stage once these MMAs have read it
            if (g == NG - 1) umma_commit(d_full(ds));  // D_ri complete
            CR_TR(1401 + 2 * st);
          }
        }
        if (++ds == (uint32_t)ND) { ds = 0; d_par ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ================================================================ bulk-copy lane: operand-image (STAGED16) groups
    // The TMA engine copies a row's four operand planes (128 + 2 positions x 16 B each) from the source straight into
    // a stage of the second ring: no thread touches the data, no proxy fence (async proxy on both sides), and the
    // copies run up to CR_NT stages ahead of the MMAs.  Replicate padding only (checked on the host): the padded
    // columns are part of the image, a padded row is the clamped row.
    const uint32_t smask = *stg_mask;
    if (lane == 0 && smask != 0u) {
      constexpr uint32_t ROW_BYTES = (uint32_t)G::PWS * 16u;
      const size_t wp16 = (size_t)((W + 127) / 128 * 128 + 2) * 16;  // bytes of one plane row of an operand image
      uint32_t tk = 0;
      for (int ri = 0; ri < nin; ++ri) {
        const int sy = min(max(y0 - P + ri, 0), H - 1);
        for (int g = 0; g < NG; ++g) {
          if (!((smask >> g) & 1u)) continue;
          const uint32_t s = tk & (CR_NT - 1);
          if (tk >= (uint32_t)CR_NT) mbar_wait_parked(t_empty(s), ((tk / CR_NT) & 1u) ^ 1u);
          const uint32_t bar = t_full(s);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2u * PARTS * ROW_BYTES) : "memory");
          const unsigned char* srow = reinterpret_cast<const unsigned char*>(gtab[g].base) + (size_t)sy * 4 * wp16 + (size_t)x0 * 16;
          const uint32_t sa0 = smem_u32(As) + (uint32_t)(NSTAGE + s) * (uint32_t)G::STAGE_BYTES;
#pragma unroll
          for (int pl = 0; pl < 2 * PARTS; ++pl)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             sa0 + (uint32_t)(pl * PLANE * 16)),
                         "l"(srow + (size_t)pl * wp16), "r"(ROW_BYTES), "r"(bar)
                         : "memory");
          ++tk;
        }
      }
    }
    __syncwarp();
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (tid == 0) CR_TR(2);
  if (warp == CR_MMA_WARP) {
    __syncwarp();
    tmem_dealloc(tmem_base, G::TMEM_COLS);
  }
}

#ifdef PBMC_ROW_TRACE
static unsigned long long* g_row_trace = nullptr;
extern "C" void pbmc_debug_set_row_trace(void* dev_buf) { g_row_trace = reinterpret_cast<unsigned long long*>(dev_buf); }
#endif

// rows per CTA: minimise waves * (rows + halo + fixed per-CTA cost in row units)
static int choose_rpc(int units, int H, int ks, int max_ctas) {
  if (max_ctas > 0) {
    // a share of the GPU: the fewest rows per CTA that stay within the CTA budget (the conv runs next to others)
    for (int r = 1; r <= H; ++r)
      if ((long)units * cdiv(H, r) <= max_ctas || r == H) return r;
  }
  int best = 1;
  double best_cost = 1e30;
  for (int r = 1; r <= 64 && r <= H; ++r) {
    const long ctas = (long)units * cdiv(H, r);
    const long waves = (ctas + 147) / 148;
    const double cost = (double)waves * (r + ks - 1 + 6.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = r; }
  }
  return best;
}

template <int KS, int PARTS, int NPG>
static int launch_row_npg(ConvRowParams& p, cudaStream_t st, bool pdl) {
  using G = RowGeom<KS, PARTS>;
  const size_t smem = CR_SMEM_HDR + (size_t)p.ngroups * G::B_GROUP + (size_t)(G::NSTAGE + (p.has_staged ? CR_NT : 0)) * G::STAGE_BYTES +
                      (size_t)p.cin_ch * 8;
  if (smem > 227 * 1024) return PBMC_ERR_UNSUPPORTED;
  static bool attr_set = false;
  if (!attr_set) {
    PBMC_CUDA(cudaFuncSetAttribute(conv_row_kernel<KS, PARTS, NPG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int nstrips = cdiv(p.W, 128);
  p.rpc = choose_rpc(nstrips * p.B, p.H, KS, p.max_ctas);
  dim3 grid(cdiv(p.H, p.rpc), nstrips, p.B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  PBMC_CUDA(launch_maybe_pdl(conv_row_kernel<KS, PARTS, NPG>, grid, dim3(CR_THREADS), smem, st, pdl, p));
  PBMC_CHECK_LAUNCH("conv_row_kernel");
  return PBMC_OK;
}

template <int KS, int PARTS>
static int launch_row(ConvRowParams& p, cudaStream_t st, bool pdl) {
  // several K groups per input row (conv[1]): four producer groups, one epilogue set; else three and two
  const bool heavy = p.ngroups >= 3;
  return heavy ? launch_row_npg<KS, PARTS, 4>(p, st, pdl) : launch_row_npg<KS, PARTS, 3>(p, st, pdl);
}

static int row_groups(const pbmc_conv_desc& d) {
  int g = 0;
  for (int s = 0; s < d.nsrc; ++s) g += (d.src[s].nblk + 3) / 4;
  return g;
}

bool conv_row_supported(const pbmc_conv_desc& d) {
  if (d.ksize != 3 && d.ksize != 5) return false;
  if (d.cout > 16) return false;
  if (d.out_chan_sum != nullptr && d.cout > 4) return false;  // per-channel sums: head conv only
  const int ng = row_groups(d);
  if (ng > CR_MAXG) return false;
  int cin = 0;
  for (int s = 0; s < d.nsrc; ++s) cin += d.src[s].nblk * 4;
  const size_t n = (size_t)d.ksize * 16, b_group = (size_t)d.ksize * 2 * (2 * n * 16);
  const size_t plane = ((128 + d.ksize - 1) + 7) / 8 * 8;
  bool staged = false;
  for (int s = 0; s < d.nsrc; ++s) staged = staged || d.src[s].layout == PBMC_LAYOUT_STAGED16;
  const size_t smem = CR_SMEM_HDR + ng * b_group + (size_t)(8 + (staged ? CR_NT : 0)) * (2 * 2 * plane * 16) + (size_t)cin * 8;
  return smem <= 227 * 1024;
}

// wpk_row holds two operand images back to back (ops.pack_conv_weight_row), then the prescale tail:
//   [fp16 hi|lo : groups * k * 2 * (2*N*16) B][bf16 : groups * k * (2*N*16) B][float 2^-e, 0, 0, 0]
int conv_row_dispatch(const pbmc_conv_desc& d, cudaStream_t st, bool pdl) {
  ConvRowParams p;
  int cin = 0;
  for (int s = 0; s < d.nsrc; ++s) {
    p.src[s] = d.src[s];
    cin += d.src[s].nblk * 4;
  }
  p.nsrc = d.nsrc; p.B = d.B; p.H = d.H; p.W = d.W;
  p.cout_blks = (d.cout + 3) / 4;
  p.pad_mode = d.pad_mode; p.epi_act = d.epi_act;
  p.ngroups = row_groups(d);
  p.cin_ch = cin;
  p.rpc = 1;
  p.max_ctas = d.max_ctas;
  p.has_staged = 0;
  for (int s = 0; s < d.nsrc; ++s) p.has_staged |= d.src[s].layout == PBMC_LAYOUT_STAGED16;
  p.trace = nullptr;
#ifdef PBMC_ROW_TRACE
  p.trace = g_row_trace;
#endif
  p.bias = d.bias; p.out = d.out; p.out_stats = d.out_stats; p.out_chan_sum = d.out_chan_sum;
  for (int s = 0; s < d.nsrc; ++s) {
    if (d.src[s].layout == PBMC_LAYOUT_BLOCKED) continue;
    // staged operand images go through the lean multi-group producer path of the fp16 hi|lo kernel only
    if (d.src[s].layout != PBMC_LAYOUT_STAGED16 || d.ksize != 3 || d.pad_mode != PBMC_PAD_REPLICATE || d.impl != PBMC_CONV_ROW_F16X2 ||
        d.src[s].nblk != 4 || d.src[s].xform != PBMC_XFORM_NONE)
      return PBMC_ERR_UNSUPPORTED;
    for (int t = 0; t < d.nsrc; ++t)
      if (d.src[t].xform != PBMC_XFORM_NONE && d.src[t].xform != PBMC_XFORM_GN_GELU) return PBMC_ERR_UNSUPPORTED;
  }
  const char* base = reinterpret_cast<const char*>(d.wpk_row);
  if (!base) return PBMC_ERR_NULL_POINTER;
  if (!aligned16(base)) return PBMC_ERR_MISALIGNED;
  const size_t n = (size_t)d.ksize * 16;
  const size_t off_bf16 = (size_t)p.ngroups * d.ksize * 2 * (2 * n * 16);
  p.wscale = reinterpret_cast<const float*>(base + off_bf16 + (size_t)p.ngroups * d.ksize * (2 * n * 16));
  if (d.impl == PBMC_CONV_ROW_F16X2) {
    p.wpk = base;
    return d.ksize == 3 ? launch_row<3, 2>(p, st, pdl) : launch_row<5, 2>(p, st, pdl);
  }
  if (d.impl == PBMC_CONV_ROW_BF16) {
    p.wpk = base + off_bf16;
    return d.ksize == 3 ? launch_row<3, 1>(p, st, pdl) : launch_row<5, 1>(p, st, pdl);
  }
  return PBMC_ERR_UNSUPPORTED;
}

}  // namespace pbmc
