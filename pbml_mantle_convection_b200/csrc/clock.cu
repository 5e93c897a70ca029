// Per-member simulated-time clock of a clocked rollout (pbmc_rollout_clocked): the reference driver's loop
// `while t < t_end: step; t += dt; log mean-T; if t > save_t: snapshot` (advect_wi_gaia.py:583-668) evaluated on the
// device behind every time step, so a captured k-step graph runs each member to its own t_end with no host involvement.
//
// Two launches per step, both on the rollout's stream and without programmatic dependent launch:
//   apply   grid (parts, B): reads the clock (writes only its scratch partials).  Frozen member: restores its output
//           T slot from its input slot.  Active member: per-CTA partial sum of the new T (fixed order) and, when a snapshot is due
//           (t + dt > save_t, computed identically by every CTA), the copy of T, u, v (, p) into the member's next ring
//           slot -- skipped when every slot holds an undrained snapshot.
//   commit  one block: fixed-order sum of the partials -> meanT_seq, then t / steps / save_t / snapshot counters /
//           active flag; the dt_seq rows of frozen members are zeroed.
// A member's clock is written by commit only, after apply has finished reading it: no CTA can see a half-updated clock.
#include "common.cuh"

namespace pbmc {

namespace {

constexpr int CLK_THREADS = 256;

// the decision of this step, from the clock as it was before the step (identical in apply and commit)
__device__ __forceinline__ bool clock_active(const pbmc_member_clock& c) { return c.t < c.t_end && c.steps < c.max_steps; }
__device__ __forceinline__ bool clock_ring_full(const pbmc_member_clock& c, int slots) { return c.snaps - c.drained >= slots; }

__global__ void __launch_bounds__(CLK_THREADS) clock_apply_kernel(pbmc_member_clock* __restrict__ clk, const float* __restrict__ Tin,
                                                                  float* __restrict__ Tout, const float* __restrict__ u,
                                                                  const float* __restrict__ v, const float* __restrict__ p,
                                                                  const double* __restrict__ dt_row, float* __restrict__ ring,
                                                                  int slots, int nch, size_t n, size_t chunk) {
  __shared__ double red[CLK_THREADS / 32];
  const int m = blockIdx.y, part = blockIdx.x;
  const int B = gridDim.y;
  const pbmc_member_clock c = clk[m];
  const size_t lo = (size_t)part * chunk, hi = lo + chunk < n ? lo + chunk : n;
  const size_t base = (size_t)m * n;
  const bool vec = (n & 3) == 0;  // every member plane and chunk boundary is then 16-byte aligned
  if (!clock_active(c)) {
    // frozen: the stencil has overwritten the output slot; the input slot (written one step earlier) is intact
    if (vec) {
      for (size_t i = lo + 4 * threadIdx.x; i < hi; i += 4 * CLK_THREADS)
        *reinterpret_cast<float4*>(Tout + base + i) = *reinterpret_cast<const float4*>(Tin + base + i);
    } else {
      for (size_t i = lo + threadIdx.x; i < hi; i += CLK_THREADS) Tout[base + i] = Tin[base + i];
    }
    return;
  }
  const double t_new = c.t + dt_row[m];
  const bool snap = t_new > c.save_t && !clock_ring_full(c, slots);
  float* dst = snap ? ring + ((size_t)(c.snaps % slots) * B + m) * nch * n : nullptr;
  double s = 0.0;
  if (vec) {
    for (size_t i = lo + 4 * threadIdx.x; i < hi; i += 4 * CLK_THREADS) {
      const float4 t4 = *reinterpret_cast<const float4*>(Tout + base + i);
      s += ((double)t4.x + (double)t4.y) + ((double)t4.z + (double)t4.w);
      if (snap) {
        *reinterpret_cast<float4*>(dst + i) = t4;
        *reinterpret_cast<float4*>(dst + n + i) = *reinterpret_cast<const float4*>(u + base + i);
        *reinterpret_cast<float4*>(dst + 2 * n + i) = *reinterpret_cast<const float4*>(v + base + i);
        if (nch == 4) *reinterpret_cast<float4*>(dst + 3 * n + i) = *reinterpret_cast<const float4*>(p + base + i);
      }
    }
  } else {
    for (size_t i = lo + threadIdx.x; i < hi; i += CLK_THREADS) {
      const float t1 = Tout[base + i];
      s += (double)t1;
      if (snap) {
        dst[i] = t1;
        dst[n + i] = u[base + i];
        dst[2 * n + i] = v[base + i];
        if (nch == 4) dst[3 * n + i] = p[base + i];
      }
    }
  }
  // fixed-order block reduction: warp tree, then warp 0 over the warp sums
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    double w = threadIdx.x < CLK_THREADS / 32 ? red[threadIdx.x] : 0.0;
    w = warp_sum(w);
    // the partials are the only clock words this kernel writes; only commit reads them
    if (threadIdx.x == 0) clk[m].part[part] = w;
  }
}

// one warp per member (strided), lane 0 writes
__global__ void __launch_bounds__(CLK_THREADS) clock_commit_kernel(pbmc_member_clock* __restrict__ clk, double* __restrict__ dt_row,
                                                                   double* __restrict__ meanT_row, double* __restrict__ meta, int slots,
                                                                   int parts, double inv_n, int B) {
  const int lane = threadIdx.x & 31;
  for (int m = threadIdx.x >> 5; m < B; m += CLK_THREADS / 32) {
    pbmc_member_clock* c = clk + m;
    if (!clock_active(*c)) {
      if (lane == 0) {
        dt_row[m] = 0.0;  // so the caller's time bookkeeping (sum of dt rows) stays right
        c->active = 0;
      }
      continue;
    }
    double s = 0.0;
    for (int q = lane; q < parts; q += 32) s += c->part[q];  // lane q sums partials q, q + 32, ...: fixed order
    s = warp_sum(s);
    if (lane == 0) {
      meanT_row[m] = s * inv_n;
      const double t_new = c->t + dt_row[m];
      c->steps += 1;
      if (t_new > c->save_t) {
        if (!clock_ring_full(*c, slots)) {
          const int slot = (int)(c->snaps % slots);
          meta[((size_t)slot * B + m) * 2 + 0] = (double)c->steps;
          meta[((size_t)slot * B + m) * 2 + 1] = t_new;
          c->snaps += 1;
        } else {
          c->overflow = 1;
        }
        c->save_t = t_new + c->save_every;
      }
      c->t = t_new;
      c->active = clock_active(*c) ? 1 : 0;
    }
  }
}

}  // namespace

int clock_parts(size_t n) {
  const size_t p = (n + 4095) / 4096;
  return (int)(p < 1 ? 1 : (p > PBMC_CLOCK_PARTS ? PBMC_CLOCK_PARTS : p));
}

// Step i of a clocked rollout, enqueued behind its stencil: Tin / Tout are the step's input and output slots, dt_row /
// meanT_row the step's rows ([B] each) of dt_seq / meanT_seq.
int clock_enqueue(pbmc_member_clock* clk, const float* Tin, float* Tout, const float* u, const float* v, const float* p,
                  double* dt_row, double* meanT_row, float* ring, double* meta, int slots, int B, int H, int W,
                  cudaStream_t st) {
  const size_t n = (size_t)H * W;
  const int parts = clock_parts(n);
  size_t chunk = (n + parts - 1) / parts;
  chunk = (chunk + 3) & ~(size_t)3;
  const int nch = p ? 4 : 3;
  clock_apply_kernel<<<dim3(parts, B), CLK_THREADS, 0, st>>>(clk, Tin, Tout, u, v, p, dt_row, ring, slots, nch, n, chunk);
  PBMC_CHECK_LAUNCH("clock_apply_kernel");
  clock_commit_kernel<<<1, CLK_THREADS, 0, st>>>(clk, dt_row, meanT_row, meta, slots, parts, 1.0 / (double)n, B);
  PBMC_CHECK_LAUNCH("clock_commit_kernel");
  return PBMC_OK;
}

}  // namespace pbmc
