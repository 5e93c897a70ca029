// A8/A9: explicit advection-diffusion update of T with the CFL time step, one HBM pass.
//   ADNet.forward          pytorch_networks_convae.py:522-568
//     forced wall coords   :532-535      one-sided differences :537-545 (FD kernels :183-214)
//     upwind advection     :547-548      non-uniform central diffusion :550-552
//     dt                   :554-559      update + replicate pad + wall rows :561-567
//   TS boundary rows/cols  :468-471      (idempotent on top of ADNet's own BCs)
// Algorithmic traffic: read T,u,v + write T' = 16 B per cell (fp32).  The CFL reduction
// max|u|,|v| of the interior is produced in the same pass (warp shuffle -> block -> one
// atomicMax per CTA), so a following step (or sweep) never needs a separate reduction pass.
#include <stdlib.h>

#include "common.cuh"

namespace pbmc {

constexpr int ST_BX = 32, ST_BY = 8, ST_RPT = 4;  // block threads, rows per thread
constexpr int ST_TH = ST_BY * ST_RPT;             // 32-row tile

struct StencilParams {
  const float* T; const float* u; const float* v; const float* xcoef; const float* ycoef;
  const pbmc_member* mem; const uint32_t* uvmax_in; uint32_t* uvmax_out; float* T_out; double* dt_out;
  double dx_min, cn_max, dt_fixed;
  int member_stride, H, W;
  // row-slab extras (pbmc_advect_diffuse_slab): rows outside [store_lo, store_hi) are ghost rows and are not
  // written; the first / last owned row is ALSO stored into the neighbour rank's ghost row (peer memory)
  int store_lo, store_hi, push_up_row, push_down_row;
  float* push_up;
  float* push_down;
};

// Cross-rank state of the flag-synchronised slab step (pbmc_advect_diffuse_slab_sync): the global CFL reduction and the
// ordering of the halo pushes happen INSIDE the update kernel, through 8-byte slots in peer-mapped memory.
struct SlabSyncArgs {
  pbmc_slab_sync* self;
  pbmc_slab_sync* peer[PBMC_MAX_RANKS];  // every rank's block (own included), as mapped into this device's address space
  int rank, world;
};

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Wait until every rank has published its max|u|,|v| for step `s` (tag == s) in THIS rank's slots and return the
// global maximum (float bits).  Lane r polls rank r's slot; the acquire also orders the neighbours' ghost-row stores
// of step s - 1 (issued before their release) before this step's reads.  Whole warp calls it.
__device__ __forceinline__ uint32_t slab_wait_global_max(pbmc_slab_sync* self, uint32_t s, int world) {
  const int lane = threadIdx.x & 31;
  uint32_t bits = 0u;
  if (lane < world) {
    const unsigned long long* slot = &self->slot[s & 1u][lane];
    unsigned long long v = ld_acquire_sys_u64(slot);
    if ((uint32_t)(v >> 32) != s) {
      const unsigned long long t0 = globaltimer_ns();
      do {
        __nanosleep(64);
        v = ld_acquire_sys_u64(slot);
        if ((uint32_t)(v >> 32) != s && globaltimer_ns() - t0 > 10000000000ull) {
          // 10 s without the peer's publication: record WHO is missing (bit r = rank r, bit 31 = failed) and go on
          // with what is there -- the host checks `failed` at its next synchronisation point and raises; the context
          // stays usable, so the sync blocks can be read for the post-mortem
          atomicOr(&self->failed, 0x80000000u | (1u << lane));
          break;
        }
      } while ((uint32_t)(v >> 32) != s);
    }
    bits = (uint32_t)v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) bits = max(bits, __shfl_xor_sync(0xffffffffu, bits, o));
  return bits;
}

// Publish `bits` as this rank's max for step `s` into slot[s & 1][rank] of every rank (threads 0 .. world-1 of a CTA).
__device__ __forceinline__ void slab_publish(const SlabSyncArgs& a, uint32_t s, uint32_t bits) {
  if ((int)threadIdx.x < a.world) {
    __threadfence_system();
    st_release_sys_u64(&a.peer[threadIdx.x]->slot[s & 1u][a.rank], ((unsigned long long)s << 32) | (unsigned long long)bits);
  }
}

__device__ __forceinline__ double cfl_dt(double uvm, double dx_min, double cn_max) {
  // :557-559 verbatim (dt_diffuse reduces to dx_min^2/4)
  const double dt_adv = 0.5 * cn_max * dx_min / uvm;
  const double dt_dif = 0.5 * ((dx_min * dx_min) * (dx_min * dx_min)) / (dx_min * dx_min + dx_min * dx_min);
  return fmin(dt_adv, dt_dif);
}

template <int VEC>
__global__ void __launch_bounds__(ST_BX* ST_BY) stencil_kernel(const StencilParams p) {
  constexpr int TW = ST_BX * VEC;
  constexpr int PITCH = TW + 8;  // body at [4, 4+TW), halos at 3 and 4+TW; rows stay 16B aligned
  __shared__ __align__(16) float Ts[ST_TH + 2][PITCH];
  __shared__ float idxl[TW], idxr[TW], idxc[TW];  // 1/dx_left, 1/dx_right, 1/(0.5 dx_r + 0.5 dx_l) per column
  __shared__ float idyt[ST_TH], idyb[ST_TH], idyc[ST_TH];
  __shared__ float dt_s;
  __shared__ float red[ST_BY];

  const int H = p.H, W = p.W, b = blockIdx.z;
  const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * ST_BX + tx;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * ST_TH;
  const size_t plane = (size_t)H * W;
  const float* Tb = p.T + (size_t)b * plane;
  const float* ub = p.u + (size_t)b * plane;
  const float* vb = p.v + (size_t)b * plane;

  // ---- issue the u,v loads first: they stay in flight while the T tile is staged
  float uu[ST_RPT][VEC], vv[ST_RPT][VEC];
  const int gx = x0 + tx * VEC;
#pragma unroll
  for (int r = 0; r < ST_RPT; ++r) {
    const int gy = y0 + ty + r * ST_BY;
    const bool in = gy > 0 && gy < H - 1 && gx < W;
    if (VEC == 4) {
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), c = a;
      if (in) {
        a = __ldcs(reinterpret_cast<const float4*>(ub + (size_t)gy * W + gx));
        c = __ldcs(reinterpret_cast<const float4*>(vb + (size_t)gy * W + gx));
      }
      uu[r][0] = a.x; uu[r][VEC > 1 ? 1 : 0] = a.y; uu[r][VEC > 2 ? 2 : 0] = a.z; uu[r][VEC > 3 ? 3 : 0] = a.w;
      vv[r][0] = c.x; vv[r][VEC > 1 ? 1 : 0] = c.y; vv[r][VEC > 2 ? 2 : 0] = c.z; vv[r][VEC > 3 ? 3 : 0] = c.w;
    } else {
      uu[r][0] = in ? __ldcs(ub + (size_t)gy * W + gx) : 0.f;
      vv[r][0] = in ? __ldcs(vb + (size_t)gy * W + gx) : 0.f;
    }
  }

  // ---- T tile with a one-cell halo
  if (VEC == 4) {
    for (int e = tid; e < (ST_TH + 2) * ST_BX; e += ST_BX * ST_BY) {
      const int r = e / ST_BX, c4 = e % ST_BX;
      const int gy = y0 + r - 1, gxx = x0 + c4 * 4;
      if (gy >= 0 && gy < H && gxx < W)
        *reinterpret_cast<float4*>(&Ts[r][4 + c4 * 4]) = __ldg(reinterpret_cast<const float4*>(Tb + (size_t)gy * W + gxx));
    }
  } else {
    for (int e = tid; e < (ST_TH + 2) * TW; e += ST_BX * ST_BY) {
      const int r = e / TW, c = e % TW;
      const int gy = y0 + r - 1, gxx = x0 + c;
      if (gy >= 0 && gy < H && gxx < W) Ts[r][4 + c] = __ldg(Tb + (size_t)gy * W + gxx);
    }
  }
  if (tid < 2 * (ST_TH + 2)) {
    const int r = tid >> 1, side = tid & 1;
    const int gy = y0 + r - 1, gxx = side ? x0 + TW : x0 - 1;
    if (gy >= 0 && gy < H && gxx >= 0 && gxx < W) Ts[r][side ? 4 + TW : 3] = __ldg(Tb + (size_t)gy * W + gxx);
  }
  // ---- inverse spacings, precomputed in double by pbmc_stencil_coefs: [3][n] = 1/d_minus, 1/d_plus, 1/(0.5 d_plus + 0.5 d_minus)
  for (int c = tid; c < TW; c += ST_BX * ST_BY) {
    const int j = x0 + c;
    if (j > 0 && j < W - 1) {
      idxl[c] = __ldg(p.xcoef + j); idxr[c] = __ldg(p.xcoef + W + j); idxc[c] = __ldg(p.xcoef + 2 * W + j);
    }
  }
  for (int r = tid; r < ST_TH; r += ST_BX * ST_BY) {
    const int i = y0 + r;
    if (i > 0 && i < H - 1) {
      idyt[r] = __ldg(p.ycoef + i); idyb[r] = __ldg(p.ycoef + H + i); idyc[r] = __ldg(p.ycoef + 2 * H + i);
    }
  }
  if (tid == 0) {
    double dt = p.dt_fixed;
    if (!(dt > 0.0)) dt = cfl_dt((double)__uint_as_float(p.uvmax_in[(size_t)b * p.member_stride]), p.dx_min, p.cn_max);
    dt_s = (float)dt;
    if (p.dt_out != nullptr && blockIdx.x == 0 && blockIdx.y == 0) p.dt_out[b] = dt;
  }
  __syncthreads();

  const float dt = dt_s;
  const float raq = p.mem ? p.mem[b].raq : 0.f;
  float m = 0.f;
  float* To = p.T_out + (size_t)b * plane;
#pragma unroll
  for (int r = 0; r < ST_RPT; ++r) {
    const int lr = ty + r * ST_BY;  // local row in [0, ST_TH)
    const int gy = y0 + lr;
    if (gy >= H || gx >= W) continue;
    float o[VEC];
    if (gy == 0) {
#pragma unroll
      for (int k = 0; k < VEC; ++k) o[k] = 1.0f;  // hot bottom wall (:566, :468)
    } else if (gy == H - 1) {
#pragma unroll
      for (int k = 0; k < VEC; ++k) o[k] = 0.0f;  // cold top wall (:567, :469)
    } else {
      const float iyt = idyt[lr], iyb = idyb[lr], iyc = idyc[lr];
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const int c = tx * VEC + k, j = x0 + c;
        o[k] = 0.f;
        if (j > 0 && j < W - 1) {
          const float Tc = Ts[lr + 1][4 + c];
          const float Tl = (Tc - Ts[lr + 1][3 + c]) * idxl[c];
          const float Tr = (Ts[lr + 1][5 + c] - Tc) * idxr[c];
          const float Tt = (Tc - Ts[lr][4 + c]) * iyt;
          const float Tbm = (Ts[lr + 2][4 + c] - Tc) * iyb;
          const float u_ = uu[r][k], v_ = vv[r][k];
          const float Tx = u_ > 0.f ? Tl : (u_ < 0.f ? Tr : 0.f);
          const float Ty = v_ > 0.f ? Tt : (v_ < 0.f ? Tbm : 0.f);
          const float lap = (Tr - Tl) * idxc[c] + (Tbm - Tt) * iyc;
          o[k] = Tc + dt * (-u_ * Tx - v_ * Ty + lap + raq);
          m = fmaxf(m, fmaxf(fabsf(u_), fabsf(v_)));
        }
      }
      // side columns copy their interior neighbour (replicate pad :565, :470-471)
      if (VEC == 4) {
        if (gx == 0) o[0] = o[VEC > 1 ? 1 : 0];
        if (gx + VEC == W) o[VEC - 1] = o[VEC > 1 ? VEC - 2 : 0];
      }
    }
    if (VEC == 4) {
      __stcs(reinterpret_cast<float4*>(To + (size_t)gy * W + gx),
             make_float4(o[0], o[VEC > 1 ? 1 : 0], o[VEC > 2 ? 2 : 0], o[VEC > 3 ? 3 : 0]));
    } else {
      const int j = gx;
      if (j > 0 && j < W - 1) {
        To[(size_t)gy * W + j] = o[0];
        if (gy > 0 && gy < H - 1) {
          if (j == 1) To[(size_t)gy * W] = o[0];
          if (j == W - 2) To[(size_t)gy * W + W - 1] = o[0];
        }
      } else if (gy == 0 || gy == H - 1) {
        To[(size_t)gy * W + j] = o[0];
      }
    }
  }
  if (p.uvmax_out != nullptr) {
    m = warp_max(m);
    if (tx == 0) red[ty] = m;
    __syncthreads();
    if (tid < ST_BY) {
      float t = red[tid];
#pragma unroll
      for (int o2 = ST_BY / 2; o2 > 0; o2 >>= 1) t = fmaxf(t, __shfl_xor_sync((1u << ST_BY) - 1u, t, o2));
      if (tid == 0) atomic_max_nonneg(p.uvmax_out + (size_t)b * p.member_stride, t);
    }
  }
}

// ---- register-marching form of the same update for 16-byte aligned rows (W % 4 == 0): a warp owns a strip of
// 128 columns (one float4 per lane) and walks down `rpw` rows keeping rows r-1, r, r+1 of T in registers; the
// left / right neighbours of a lane's four cells come from the adjacent lanes by shuffle (the strip's two halo
// columns by one predicated scalar load each).  No shared memory, no block barrier: every row is one 128-bit
// load of T, u and v and one 128-bit store, with the next row's loads in flight during the arithmetic --
// 16 B per cell-update of HBM traffic plus 2/rpw of a row of T for the strip's top and bottom halo.
//
// SYNC (pbmc_advect_diffuse_slab_sync, one rank of a row-decomposed grid): no collective call surrounds the kernel.
//   start  every warp waits until all ranks' maxima for THIS step (tag = steps_done + 1) stand in this rank's slots
//          -> global max -> dt; the same acquire makes the neighbours' ghost rows of the previous step visible;
//   end    warp maxima -> local accumulator; the CTA that finishes last publishes (tag + 1, local max) into every
//          rank's slot of the other parity and advances steps_done.  Two parities suffice: a rank can only
//          overwrite parity (s & 1) at the end of step s + 1, which it enters only after every rank has published
//          step s + 1's value, i.e. after every rank has finished step s and consumed the tags of step s.
template <bool SYNC>
__global__ void __launch_bounds__(128, 6) stencil_march_kernel(const StencilParams p, int rpw, const SlabSyncArgs sa) {
  // no-ops unless launched with programmatic stream serialization (the rollout does, behind the head kernel)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int H = p.H, W = p.W, b = blockIdx.z;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int x0 = (blockIdx.x * 32 + lane) * 4;
  const int y0 = (blockIdx.y * 4 + warp) * rpw;
  uint32_t step = 0u, gmax_bits = 0u;
  if (SYNC) {
    step = *reinterpret_cast<volatile const unsigned int*>(&sa.self->steps_done) + 1u;
    gmax_bits = slab_wait_global_max(sa.self, step, sa.world);
  }
  if (!SYNC && y0 >= H) return;  // whole warp
  const bool warp_on = y0 < H;
  const int y1 = min(y0 + rpw, H);
  const bool act = x0 < W;              // W % 4 == 0: a lane's four columns are all inside or all outside
  const int xs = act ? x0 : W - 4;      // inactive lanes shadow the last float4 (they take part in the shuffles)
  const size_t plane = (size_t)H * W;
  const float* Tb = p.T + (size_t)b * plane;
  const float* ub = p.u + (size_t)b * plane;
  const float* vb = p.v + (size_t)b * plane;
  float* To = p.T_out + (size_t)b * plane;

  double dtd = p.dt_fixed;
  if (!(dtd > 0.0))
    dtd = cfl_dt((double)__uint_as_float(SYNC ? gmax_bits : __ldg(p.uvmax_in + (size_t)b * p.member_stride)), p.dx_min, p.cn_max);
  const float dt = (float)dtd;
  if (p.dt_out != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) p.dt_out[b] = dtd;
  const float raq = p.mem ? p.mem[b].raq : 0.f;
  float m = 0.f;
  if (warp_on) {
  const float4 ixl = ldg4(p.xcoef + xs), ixr = ldg4(p.xcoef + W + xs), ixc = ldg4(p.xcoef + 2 * W + xs);
  const float xl[4] = {ixl.x, ixl.y, ixl.z, ixl.w}, xr[4] = {ixr.x, ixr.y, ixr.z, ixr.w}, xcn[4] = {ixc.x, ixc.y, ixc.z, ixc.w};
  const bool need_l = lane == 0 && x0 > 0, need_r = (lane == 31 || x0 + 4 >= W) && x0 + 4 < W;

  auto row4 = [&](const float* base, int r) { return __ldcs(reinterpret_cast<const float4*>(base + (size_t)r * W + xs)); };
  auto rowT = [&](int r) { return __ldg(reinterpret_cast<const float4*>(Tb + (size_t)r * W + xs)); };
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  // rows r-1, r, r+1 of T; u, v, the two halo scalars and the y coefficients of row r
  float4 Tm = y0 > 0 ? rowT(y0 - 1) : zero4, Tc = rowT(y0), Tp = y0 + 1 < H ? rowT(y0 + 1) : zero4;
  float4 uc = row4(ub, y0), vc = row4(vb, y0);
  float hl = need_l ? __ldg(Tb + (size_t)y0 * W + x0 - 1) : 0.f, hr = need_r ? __ldg(Tb + (size_t)y0 * W + x0 + 4) : 0.f;
  float cyt = __ldg(p.ycoef + y0), cyb = __ldg(p.ycoef + H + y0), cyc = __ldg(p.ycoef + 2 * H + y0);
  for (int r = y0; r < y1; ++r) {
    // next row's operands first: they are in flight during this row's arithmetic
    const int rn = r + 1;
    const bool more = rn < y1;
    float4 Tn = zero4, un = zero4, vn = zero4;
    float hln = 0.f, hrn = 0.f, cytn = 0.f, cybn = 0.f, cycn = 0.f;
    if (rn + 1 < H && more) Tn = rowT(rn + 1);
    if (more) {
      un = row4(ub, rn);
      vn = row4(vb, rn);
      if (need_l) hln = __ldg(Tb + (size_t)rn * W + x0 - 1);
      if (need_r) hrn = __ldg(Tb + (size_t)rn * W + x0 + 4);
      cytn = __ldg(p.ycoef + rn); cybn = __ldg(p.ycoef + H + rn); cycn = __ldg(p.ycoef + 2 * H + rn);
    }
    float left = __shfl_up_sync(0xffffffffu, Tc.w, 1), right = __shfl_down_sync(0xffffffffu, Tc.x, 1);
    if (need_l) left = hl;
    if (need_r) right = hr;
    float o[4];
    if (r == 0) {
      o[0] = o[1] = o[2] = o[3] = 1.0f;  // hot bottom wall (:566, :468)
    } else if (r == H - 1) {
      o[0] = o[1] = o[2] = o[3] = 0.0f;  // cold top wall (:567, :469)
    } else {
      const float tc[6] = {left, Tc.x, Tc.y, Tc.z, Tc.w, right};
      const float tm[4] = {Tm.x, Tm.y, Tm.z, Tm.w}, tp[4] = {Tp.x, Tp.y, Tp.z, Tp.w};
      const float u4[4] = {uc.x, uc.y, uc.z, uc.w}, v4[4] = {vc.x, vc.y, vc.z, vc.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int j = x0 + k;
        o[k] = 0.f;
        if (j > 0 && j < W - 1) {
          const float c = tc[k + 1];
          const float Tl = (c - tc[k]) * xl[k];
          const float Tr = (tc[k + 2] - c) * xr[k];
          const float Tt = (c - tm[k]) * cyt;
          const float Tbm = (tp[k] - c) * cyb;
          const float u_ = u4[k], v_ = v4[k];
          const float Tx = u_ > 0.f ? Tl : (u_ < 0.f ? Tr : 0.f);
          const float Ty = v_ > 0.f ? Tt : (v_ < 0.f ? Tbm : 0.f);
          const float lap = (Tr - Tl) * xcn[k] + (Tbm - Tt) * cyc;
          o[k] = c + dt * (-u_ * Tx - v_ * Ty + lap + raq);
          m = fmaxf(m, fmaxf(fabsf(u_), fabsf(v_)));
        }
      }
      // side columns copy their interior neighbour (replicate pad :565, :470-471)
      if (x0 == 0) o[0] = o[1];
      if (x0 + 4 == W) o[3] = o[2];
    }
    if (act && r >= p.store_lo && r < p.store_hi) {
      const float4 o4 = make_float4(o[0], o[1], o[2], o[3]);
      __stcs(reinterpret_cast<float4*>(To + (size_t)r * W + x0), o4);
      // fused halo exchange: the slab's boundary rows go straight into the neighbours' ghost rows over NVLink
      if (r == p.push_up_row && p.push_up != nullptr) *reinterpret_cast<float4*>(p.push_up + x0) = o4;
      if (r == p.push_down_row && p.push_down != nullptr) *reinterpret_cast<float4*>(p.push_down + x0) = o4;
    }
    Tm = Tc; Tc = Tp; Tp = Tn;
    uc = un; vc = vn; hl = hln; hr = hrn; cyt = cytn; cyb = cybn; cyc = cycn;
  }
  if (!act) m = 0.f;
  }  // warp_on
  if (!SYNC) {
    if (p.uvmax_out != nullptr) {
      m = warp_max(m);
      if (lane == 0 && m > 0.f) atomic_max_nonneg(p.uvmax_out + (size_t)b * p.member_stride, m);
    }
    return;
  }
  // ---- SYNC epilogue: local max, CTA count, and -- by the CTA that finishes last -- the publication for the next step
  __shared__ uint32_t s_last, s_bits;
  m = warp_max(m);
  if (lane == 0 && m > 0.f) atomic_max_nonneg(&sa.self->local_max, m);
  // Only a warp that stored rows into a NEIGHBOUR's memory needs the system-scope fence (its stores must be performed
  // over NVLink before the CTA is counted); everything else this CTA wrote is local and ordered by the fence + atomic of
  // thread 0 below.  (MEMBAR.SC.SYS in every thread of every CTA cost microseconds per step.)
  const bool pushed = warp_on && ((p.push_up != nullptr && p.push_up_row >= y0 && p.push_up_row < y1) ||
                                  (p.push_down != nullptr && p.push_down_row >= y0 && p.push_down_row < y1));
  if (pushed) __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t total = gridDim.x * gridDim.y * gridDim.z;
    __threadfence();  // the CTA's atomicMax / stores (observed through the barrier) before its count
    const uint32_t prev = atomicAdd(&sa.self->ctas_done, 1u);
    s_last = prev == total - 1u;
    if (s_last) {
      __threadfence();
      s_bits = atomicExch(&sa.self->local_max, 0u);
      sa.self->ctas_done = 0u;
    }
  }
  __syncthreads();
  if (s_last) {
    slab_publish(sa, step + 1u, s_bits);
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      *reinterpret_cast<volatile unsigned int*>(&sa.self->steps_done) = step;
    }
  }
}

// First publication of a run (and after every change of the velocity field): this rank's max|u|,|v| -- left in
// self->local_max by uvmax_kernel -- goes out with tag steps_done + 1.
__global__ void slab_publish_kernel(const SlabSyncArgs sa) {
  __shared__ uint32_t s_bits;
  const uint32_t step = *reinterpret_cast<volatile const unsigned int*>(&sa.self->steps_done) + 1u;
  if (threadIdx.x == 0) s_bits = atomicExch(&sa.self->local_max, 0u);
  __syncthreads();
  slab_publish(sa, step, s_bits);
}

// ---- stand-alone interior max|u|,|v| (only when no producer supplied it)
__global__ void __launch_bounds__(256) uvmax_kernel(const float* __restrict__ u, const float* __restrict__ v,
                                                    uint32_t* __restrict__ out, int member_stride, int H, int W) {
  const int b = blockIdx.y;
  const size_t plane = (size_t)H * W;
  float m = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / W), c = (int)(i % W);
    if (r > 0 && r < H - 1 && c > 0 && c < W - 1)
      m = fmaxf(m, fmaxf(fabsf(__ldg(u + (size_t)b * plane + i)), fabsf(__ldg(v + (size_t)b * plane + i))));
  }
  __shared__ float red[8];
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 8) {
    float t = red[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) t = fmaxf(t, __shfl_xor_sync(0xffu, t, o));
    if (threadIdx.x == 0) atomic_max_nonneg(out + (size_t)b * member_stride, t);
  }
}

// ---- general form: coordinates (and optionally RaQ) given as fields, exactly ADNet's inputs tensor
__global__ void __launch_bounds__(256) stencil_fields_kernel(const float* __restrict__ T, const float* __restrict__ u,
                                                             const float* __restrict__ v, const double* __restrict__ xc,
                                                             const double* __restrict__ yc, size_t coord_stride,
                                                             const float* __restrict__ raq_field, const pbmc_member* mem,
                                                             const uint32_t* uvmax_in, int member_stride,
                                                             const double* dx_min_dev, double cn_max,
                                                             const double* dt_fixed_dev, float* __restrict__ T_out,
                                                             double* dt_out, int H, int W) {
  const int b = blockIdx.z;
  const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
  __shared__ float dt_s;
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    double dt = dt_fixed_dev ? *dt_fixed_dev : 0.0;
    if (!(dt > 0.0)) dt = cfl_dt((double)__uint_as_float(uvmax_in[(size_t)b * member_stride]), *dx_min_dev, cn_max);
    dt_s = (float)dt;
    if (dt_out != nullptr && blockIdx.x == 0 && blockIdx.y == 0) dt_out[b] = dt;
  }
  __syncthreads();
  if (i >= H || j >= W) return;
  const size_t plane = (size_t)H * W;
  const float* Tb = T + (size_t)b * plane;
  const double* xb = xc + (size_t)b * coord_stride;
  const double* yb = yc + (size_t)b * coord_stride;
  float* To = T_out + (size_t)b * plane;
  if (i == 0) { To[j] = 1.f; return; }
  if (i == H - 1) { To[(size_t)i * W + j] = 0.f; return; }
  if (j == 0 || j == W - 1) return;  // written by the neighbouring interior cell
  // spacings in double: differences of O(1) coordinates lose ~1e-5 relative accuracy in float
  auto X = [&](int ii, int jj) { return jj == 0 ? 0.0 : (jj == W - 1 ? 4.0 : __ldg(xb + (size_t)ii * W + jj)); };
  auto Y = [&](int ii, int jj) { return ii == 0 ? 0.0 : (ii == H - 1 ? 1.0 : __ldg(yb + (size_t)ii * W + jj)); };
  const float dxl = (float)(X(i, j) - X(i, j - 1)), dxr = (float)(X(i, j + 1) - X(i, j));
  const float dyt = (float)(Y(i, j) - Y(i - 1, j)), dyb = (float)(Y(i + 1, j) - Y(i, j));
  const size_t c = (size_t)i * W + j;
  const float Tc = Tb[c];
  const float Tl = (Tc - Tb[c - 1]) / dxl, Tr = (Tb[c + 1] - Tc) / dxr;
  const float Tt = (Tc - Tb[c - W]) / dyt, Tbm = (Tb[c + W] - Tc) / dyb;
  const float u_ = u[(size_t)b * plane + c], v_ = v[(size_t)b * plane + c];
  const float Tx = u_ > 0.f ? Tl : (u_ < 0.f ? Tr : 0.f);
  const float Ty = v_ > 0.f ? Tt : (v_ < 0.f ? Tbm : 0.f);
  const float lap = (Tr - Tl) / (0.5f * dxr + 0.5f * dxl) + (Tbm - Tt) / (0.5f * dyb + 0.5f * dyt);
  const float raq = raq_field ? __ldg(raq_field + (size_t)b * plane + c) : (mem ? mem[b].raq : 0.f);
  const float o = Tc + dt_s * (-u_ * Tx - v_ * Ty + lap + raq);
  To[c] = o;
  if (j == 1) To[(size_t)i * W] = o;
  if (j == W - 2) To[(size_t)i * W + W - 1] = o;
}

// ---- inverse spacings of one coordinate axis, from double coordinates with forced wall values (:532-545)
__global__ void stencil_coefs_kernel(const double* __restrict__ c, int n, double lo, double hi, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float a = 0.f, b = 0.f, d = 0.f;
  if (i > 0 && i < n - 1) {
    const double cm = (i - 1 == 0) ? lo : c[i - 1], cp = (i + 1 == n - 1) ? hi : c[i + 1], ci = c[i];
    const double dm = ci - cm, dp = cp - ci;
    a = (float)(1.0 / dm); b = (float)(1.0 / dp); d = (float)(1.0 / (0.5 * dp + 0.5 * dm));
  }
  out[i] = a; out[n + i] = b; out[2 * n + i] = d;
}

// ---- A10: advect_wi_gaia.py:624-629
__global__ void clamp_T_kernel(float* __restrict__ T, int core_cool, int H, int W) {
  const int b = blockIdx.z;
  const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
  if (i >= H || j >= W) return;
  float* Tb = T + (size_t)b * H * W;
  const int js = j == 0 ? 1 : (j == W - 1 ? W - 2 : j);
  float t = Tb[(size_t)i * W + js];
  if (i == 0 && !core_cool) t = 1.f;
  if (i == H - 1) t = 0.f;
  t = fminf(fmaxf(t, 0.f), 2.f);
  Tb[(size_t)i * W + j] = t;
}

// ---- A11: row means (profile) and mean-T in double
__global__ void __launch_bounds__(256) row_mean_kernel(const float* __restrict__ T, double* __restrict__ prof, int H, int W) {
  const int i = blockIdx.x, b = blockIdx.y;
  const float* row = T + ((size_t)b * H + i) * W;
  double s = 0.0;
  for (int j = threadIdx.x; j < W; j += 256) s += (double)__ldg(row + j);
  __shared__ double red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    prof[(size_t)b * H + i] = t / (double)W;
  }
}
__global__ void __launch_bounds__(256) prof_mean_kernel(const double* __restrict__ prof, double* __restrict__ meanT, int H) {
  const int b = blockIdx.x;
  double s = 0.0;
  for (int i = threadIdx.x; i < H; i += 256) s += prof[(size_t)b * H + i];
  __shared__ double red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    meanT[b] = t / (double)H;
  }
}

}  // namespace pbmc

using namespace pbmc;

extern "C" int pbmc_stencil_coefs(const double* coord, int n, double wall_lo, double wall_hi, float* coef, void* stream) {
  if (!coord || !coef) return PBMC_ERR_NULL_POINTER;
  if (n < 3) return PBMC_ERR_BAD_SHAPE;
  stencil_coefs_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(coord, n, wall_lo, wall_hi, coef);
  PBMC_CHECK_LAUNCH("stencil_coefs_kernel");
  return PBMC_OK;
}

// pdl: the plain (non-slab) marching kernel is launched with programmatic stream serialization
static int advect_diffuse_launch(const float* T, const float* u, const float* v, const float* x, const float* y,
                                 const pbmc_member* members, const uint32_t* uvmax_in, int member_stride, double dx_min,
                                 double cn_max, double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int B, int H,
                                 int W, int has_up, int has_down, float* peer_up, float* peer_down, void* stream, bool pdl,
                                 const SlabSyncArgs* sync = nullptr) {
  if (!T || !u || !v || !x || !y || !T_out) return PBMC_ERR_NULL_POINTER;
  if (!(dt_fixed > 0.0) && !uvmax_in && !sync) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3 || (member_stride != 0 && member_stride != 1)) return PBMC_ERR_BAD_SHAPE;
  if (T == T_out) return PBMC_ERR_UNSUPPORTED;  // out-of-place only (neighbours are read)
  const bool slab = has_up || has_down || peer_up || peer_down || sync != nullptr;
  StencilParams p{T, u, v, x, y, members, uvmax_in, uvmax_out, T_out, dt_out, dx_min, cn_max, dt_fixed, member_stride, H, W,
                  has_up ? 1 : 0, has_down ? H - 1 : H, has_up ? 1 : -1, has_down ? H - 2 : -1, peer_up, peer_down};
  const bool vec = (W % 4 == 0) && aligned16(T) && aligned16(u) && aligned16(v) && aligned16(T_out);
  if (vec && aligned16(x)) {
    if ((peer_up && !aligned16(peer_up)) || (peer_down && !aligned16(peer_down))) return PBMC_ERR_MISALIGNED;
    // Rows per warp.  The grid runs in waves of (resident CTAs per SM) x (SMs) CTAs and every CTA takes the same time
    // (~ rpw + a few rows of fixed cost), so the sweep time is waves x (rpw + c): pick the rpw in [4, 128] that minimises it
    // (ties: the larger one, 2/rpw of a row is re-read as halo).  The old rule (fill 148 x 16 warps, at most 64 rows)
    // left a 4096 x 8192 slab at 1.47 waves: 65 % of the HBM peak against 77 % for the 8192^2 grid.
    const int strips = cdiv(W, 128);
    static int cap[2] = {0, 0};
    int& capacity = cap[sync != nullptr ? 1 : 0];
    if (capacity == 0) {
      int per_sm = 0, dev = 0, sms = 148;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      if (sync != nullptr)
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stencil_march_kernel<true>, 128, 0);
      else
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, stencil_march_kernel<false>, 128, 0);
      capacity = (per_sm > 0 ? per_sm : 5) * sms;
    }
    int rpw = 4;
    double best = 1e30;
    for (int r = 4; r <= 128; ++r) {
      const long ctas = (long)strips * cdiv(H, 4 * r) * B;
      const long waves = (ctas + capacity - 1) / capacity;
      const double cost = (double)waves * (r + 3.0);
      if (cost <= best + 1e-9) { best = cost; rpw = r; }
    }
    dim3 grid(strips, cdiv(H, 4 * rpw), B);
    if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
    if (sync != nullptr) {
      stencil_march_kernel<true><<<grid, 128, 0, (cudaStream_t)stream>>>(p, rpw, *sync);
    } else {
      PBMC_CUDA(launch_maybe_pdl(stencil_march_kernel<false>, grid, dim3(128), 0, (cudaStream_t)stream, pdl, p, rpw, SlabSyncArgs{}));
    }
    PBMC_CHECK_LAUNCH("stencil_march_kernel");
    return PBMC_OK;
  }
  if (slab || sync) return PBMC_ERR_UNSUPPORTED;  // the slab form needs 16-byte aligned rows (W % 4 == 0)
  const int TW = vec ? ST_BX * 4 : ST_BX;
  dim3 grid(cdiv(W, TW), cdiv(H, ST_TH), B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  if (vec)
    stencil_kernel<4><<<grid, dim3(ST_BX, ST_BY), 0, (cudaStream_t)stream>>>(p);
  else
    stencil_kernel<1><<<grid, dim3(ST_BX, ST_BY), 0, (cudaStream_t)stream>>>(p);
  PBMC_CHECK_LAUNCH("stencil_kernel");
  return PBMC_OK;
}

namespace pbmc {
int advect_diffuse_enqueue(const float* T, const float* u, const float* v, const float* x, const float* y,
                           const pbmc_member* members, const uint32_t* uvmax_in, int member_stride, double dx_min, double cn_max,
                           double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int B, int H, int W, cudaStream_t st,
                           bool pdl) {
  return advect_diffuse_launch(T, u, v, x, y, members, uvmax_in, member_stride, dx_min, cn_max, dt_fixed, T_out, uvmax_out,
                               dt_out, B, H, W, 0, 0, nullptr, nullptr, st, pdl);
}
}  // namespace pbmc

extern "C" int pbmc_advect_diffuse(const float* T, const float* u, const float* v, const float* x, const float* y,
                                   const pbmc_member* members, const uint32_t* uvmax_in, int member_stride,
                                   double dx_min, double cn_max, double dt_fixed, float* T_out, uint32_t* uvmax_out,
                                   double* dt_out, int B, int H, int W, void* stream) {
  return advect_diffuse_enqueue(T, u, v, x, y, members, uvmax_in, member_stride, dx_min, cn_max, dt_fixed, T_out, uvmax_out,
                                dt_out, B, H, W, (cudaStream_t)stream, false);
}

extern "C" int pbmc_advect_diffuse_slab(const float* T, const float* u, const float* v, const float* x, const float* y,
                                        const pbmc_member* members, const uint32_t* uvmax_in, double dx_min, double cn_max,
                                        double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int H, int W,
                                        int has_up, int has_down, float* peer_up_ghost_row, float* peer_down_ghost_row,
                                        void* stream) {
  if ((peer_up_ghost_row && !has_up) || (peer_down_ghost_row && !has_down)) return PBMC_ERR_BAD_SHAPE;
  return advect_diffuse_launch(T, u, v, x, y, members, uvmax_in, 0, dx_min, cn_max, dt_fixed, T_out, uvmax_out, dt_out, 1, H, W,
                               has_up, has_down, peer_up_ghost_row, peer_down_ghost_row, stream, false);
}

static int make_sync_args(pbmc_slab_sync* self, pbmc_slab_sync* const* peers_h, int rank, int world, SlabSyncArgs& a) {
  if (!self || !peers_h) return PBMC_ERR_NULL_POINTER;
  if (world < 1 || world > PBMC_MAX_RANKS || rank < 0 || rank >= world) return PBMC_ERR_BAD_SHAPE;
  a.self = self; a.rank = rank; a.world = world;
  for (int r = 0; r < PBMC_MAX_RANKS; ++r) a.peer[r] = nullptr;
  for (int r = 0; r < world; ++r) {
    if (!peers_h[r]) return PBMC_ERR_NULL_POINTER;
    if (reinterpret_cast<uintptr_t>(peers_h[r]) & 7) return PBMC_ERR_MISALIGNED;
    a.peer[r] = peers_h[r];
  }
  return PBMC_OK;
}

extern "C" int pbmc_slab_sync_publish(const float* u, const float* v, int H, int W, pbmc_slab_sync* self,
                                      pbmc_slab_sync* const* peers_h, int rank, int world, void* stream) {
  if (!u || !v) return PBMC_ERR_NULL_POINTER;
  if (H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;
  SlabSyncArgs a;
  const int rc = make_sync_args(self, peers_h, rank, world, a);
  if (rc != PBMC_OK) return rc;
  // interior rows 1 .. H-2 of the local array = this rank's owned non-wall rows (local rows 0 / H-1 are ghosts or walls)
  const size_t plane = (size_t)H * W;
  const unsigned nb = (unsigned)min((size_t)1184, (plane + 255) / 256);
  uvmax_kernel<<<dim3(nb, 1), 256, 0, (cudaStream_t)stream>>>(u, v, &self->local_max, 0, H, W);
  PBMC_CHECK_LAUNCH("uvmax_kernel");
  slab_publish_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a);
  PBMC_CHECK_LAUNCH("slab_publish_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_advect_diffuse_slab_sync(const float* T, const float* u, const float* v, const float* x, const float* y,
                                             const pbmc_member* members, double dx_min, double cn_max, float* T_out,
                                             double* dt_out, int H, int W, int has_up, int has_down,
                                             float* peer_up_ghost_row, float* peer_down_ghost_row, pbmc_slab_sync* self,
                                             pbmc_slab_sync* const* peers_h, int rank, int world, void* stream) {
  if ((peer_up_ghost_row && !has_up) || (peer_down_ghost_row && !has_down)) return PBMC_ERR_BAD_SHAPE;
  SlabSyncArgs a;
  const int rc = make_sync_args(self, peers_h, rank, world, a);
  if (rc != PBMC_OK) return rc;
  return advect_diffuse_launch(T, u, v, x, y, members, nullptr, 0, dx_min, cn_max, 0.0, T_out, nullptr, dt_out, 1, H, W, has_up,
                               has_down, peer_up_ghost_row, peer_down_ghost_row, stream, false, &a);
}

extern "C" int pbmc_uvmax(const float* u, const float* v, uint32_t* uvmax, int member_stride, int B, int H, int W,
                          void* stream) {
  if (!u || !v || !uvmax) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3 || (member_stride != 0 && member_stride != 1)) return PBMC_ERR_BAD_SHAPE;
  const size_t plane = (size_t)H * W;
  const unsigned nb = (unsigned)min((size_t)1184, (plane + 255) / 256);
  uvmax_kernel<<<dim3(nb, B), 256, 0, (cudaStream_t)stream>>>(u, v, uvmax, member_stride, H, W);
  PBMC_CHECK_LAUNCH("uvmax_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_advect_diffuse_fields(const float* T, const float* u, const float* v, const double* xc,
                                          const double* yc, size_t coord_batch_stride, const float* raq_field,
                                          const pbmc_member* members, const uint32_t* uvmax_in, int member_stride,
                                          const double* dx_min_dev, double cn_max, const double* dt_fixed_dev,
                                          float* T_out, double* dt_out, int B, int H, int W, void* stream) {
  if (!T || !u || !v || !xc || !yc || !T_out) return PBMC_ERR_NULL_POINTER;
  if (!dt_fixed_dev && (!uvmax_in || !dx_min_dev)) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3 || (member_stride != 0 && member_stride != 1)) return PBMC_ERR_BAD_SHAPE;
  if (coord_batch_stride != 0 && coord_batch_stride != (size_t)H * W) return PBMC_ERR_BAD_SHAPE;
  if (T == T_out) return PBMC_ERR_UNSUPPORTED;
  dim3 grid(cdiv(W, 32), cdiv(H, 8), B);
  if (grid.y > 65535 || grid.z > 65535) return PBMC_ERR_BAD_SHAPE;
  stencil_fields_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(T, u, v, xc, yc, coord_batch_stride, raq_field,
                                                                       members, uvmax_in, member_stride, dx_min_dev,
                                                                       cn_max, dt_fixed_dev, T_out, dt_out, H, W);
  PBMC_CHECK_LAUNCH("stencil_fields_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_clamp_T(float* T, int core_cool, int B, int H, int W, void* stream) {
  if (!T) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;
  dim3 grid(cdiv(W, 32), cdiv(H, 8), B);
  clamp_T_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(T, core_cool, H, W);
  PBMC_CHECK_LAUNCH("clamp_T_kernel");
  return PBMC_OK;
}

extern "C" int pbmc_diagnostics(const float* T, double* prof, double* meanT, int B, int H, int W, void* stream) {
  if (!T || !prof || !meanT) return PBMC_ERR_NULL_POINTER;
  if (B <= 0 || H <= 0 || W <= 0 || H > 65535 * 16) return PBMC_ERR_BAD_SHAPE;
  row_mean_kernel<<<dim3(H, B), 256, 0, (cudaStream_t)stream>>>(T, prof, H, W);
  PBMC_CHECK_LAUNCH("row_mean_kernel");
  prof_mean_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(prof, meanT, H);
  PBMC_CHECK_LAUNCH("prof_mean_kernel");
  return PBMC_OK;
}
