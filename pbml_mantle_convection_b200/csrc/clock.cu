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
//
// With a member queue (pbmc_rollout_queued) the same two launches also refill the slots whose member stops at this step
// (include/pbmc.h states the rule): apply, after its partial sum and snapshot copy, overwrites the CTA's cells of the
// output slot with the queued member's T0; commit writes the new clock, the member row, slot_member, next and the
// member_seq / snap_member tags.  Both take "this step stops the member" from clock_stops and the queue entry from the
// same rank (slots with a lower index that stop too), so every CTA and the commit kernel agree.  Without a queue
// (Q = 0) neither kernel touches any of this.
#include <string.h>

#include "common.cuh"

namespace pbmc {

namespace {

constexpr int CLK_THREADS = 256;

// the decision of this step, from the clock as it was before the step (identical in apply and commit)
__device__ __forceinline__ bool clock_active(const pbmc_member_clock& c) { return c.t < c.t_end && c.steps < c.max_steps; }
__device__ __forceinline__ bool clock_ring_full(const pbmc_member_clock& c, int slots) { return c.snaps - c.drained >= slots; }
// whether this step stops the member: active before it, and not after t += dt, steps += 1 (what commit then computes)
__device__ __forceinline__ bool clock_stops(const pbmc_member_clock& c, double dt) {
  return clock_active(c) && !(c.t + dt < c.t_end && c.steps + 1 < c.max_steps);
}

__global__ void __launch_bounds__(CLK_THREADS) clock_apply_kernel(pbmc_member_clock* __restrict__ clk, const float* __restrict__ Tin,
                                                                  float* __restrict__ Tout, const float* __restrict__ u,
                                                                  const float* __restrict__ v, const float* __restrict__ p,
                                                                  const double* __restrict__ dt_row, float* __restrict__ ring,
                                                                  int slots, int nch, size_t n, size_t chunk, const pbmc_member_queue qu) {
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
  // queue: this member stops here and the queue holds an entry for the slot -> its T0 replaces the new T once read
  // (block-uniform: every thread reads the same clocks, dt row and next)
  const float* T0q = nullptr;
  if (qu.Q > 0 && clock_stops(c, dt_row[m])) {
    int r = 0;
    for (int b0 = 0; b0 < m; b0 += CLK_THREADS) {
      const int o = b0 + (int)threadIdx.x;
      r += __syncthreads_count(o < m && clock_stops(clk[o], dt_row[o]));
    }
    const int64_t q = *qu.next + r;
    if (q < qu.Q) T0q = qu.T0 + (size_t)q * n;
  }
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
      if (T0q) *reinterpret_cast<float4*>(Tout + base + i) = *reinterpret_cast<const float4*>(T0q + i);
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
      if (T0q) Tout[base + i] = T0q[i];
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

// one warp per member (strided), lane 0 writes.  Queue (qu.Q > 0): `stops` (dynamic shared memory, [B]) holds
// clock_stops of every slot, taken before any clock is written; members / seq_row are the member rows and this step's
// member_seq row.
__global__ void __launch_bounds__(CLK_THREADS) clock_commit_kernel(pbmc_member_clock* __restrict__ clk, double* __restrict__ dt_row,
                                                                   double* __restrict__ meanT_row, double* __restrict__ meta, int slots,
                                                                   int parts, double inv_n, int B, const pbmc_member_queue qu,
                                                                   pbmc_member* __restrict__ members, int64_t* __restrict__ seq_row) {
  extern __shared__ int stops[];
  const int lane = threadIdx.x & 31;
  const bool queued = qu.Q > 0;
  int64_t next = 0;
  if (queued) {
    next = *qu.next;
    for (int m = threadIdx.x; m < B; m += CLK_THREADS) stops[m] = clock_stops(clk[m], dt_row[m]) ? 1 : 0;
    __syncthreads();
  }
  for (int m = threadIdx.x >> 5; m < B; m += CLK_THREADS / 32) {
    pbmc_member_clock* c = clk + m;
    if (!clock_active(*c)) {
      if (lane == 0) {
        dt_row[m] = 0.0;  // so the caller's time bookkeeping (sum of dt rows) stays right
        c->active = 0;
        if (queued) seq_row[m] = -1;
      }
      continue;
    }
    double s = 0.0;
    for (int q = lane; q < parts; q += 32) s += c->part[q];  // lane q sums partials q, q + 32, ...: fixed order
    s = warp_sum(s);
    int r = 0;  // rank among the slots that stop at this step (the apply kernel's count)
    if (queued && stops[m]) {
      for (int o = lane; o < m; o += 32) r += stops[o];
      r = __reduce_add_sync(0xffffffffu, r);
    }
    if (lane == 0) {
      const int64_t who = queued ? qu.slot_member[m] : -1;
      if (queued) seq_row[m] = who;
      meanT_row[m] = s * inv_n;
      const double t_new = c->t + dt_row[m];
      c->steps += 1;
      if (t_new > c->save_t) {
        if (!clock_ring_full(*c, slots)) {
          const int slot = (int)(c->snaps % slots);
          meta[((size_t)slot * B + m) * 2 + 0] = (double)c->steps;
          meta[((size_t)slot * B + m) * 2 + 1] = t_new;
          if (queued) qu.snap_member[(size_t)slot * B + m] = who;
          c->snaps += 1;
        } else {
          c->overflow = 1;
        }
        c->save_t = t_new + c->save_every;
      }
      c->t = t_new;
      c->active = clock_active(*c) ? 1 : 0;
      if (queued && stops[m] && next + r < qu.Q) {
        const int64_t q = next + r;  // the slot's next member, from step i + 1 on
        c->t = qu.t0[q];
        c->t_end = qu.t_end[q];
        c->save_t = 0.0;
        c->save_every = qu.save_every[q];
        c->steps = qu.n_step0[q];
        c->max_steps = qu.max_steps[q];
        c->active = 1;
        members[m] = qu.params[q];
        qu.slot_member[m] = q;
      }
    }
  }
  if (queued) {
    __syncthreads();  // every thread has read next
    if (threadIdx.x == 0) {
      int64_t k = 0;
      for (int m = 0; m < B; ++m) k += stops[m];
      *qu.next = next + k < qu.Q ? next + k : qu.Q;
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
// queue (NULL: none): the rollout's member queue, members its member rows, seq_row the step's row of member_seq.
int clock_enqueue(pbmc_member_clock* clk, const float* Tin, float* Tout, const float* u, const float* v, const float* p,
                  double* dt_row, double* meanT_row, float* ring, double* meta, int slots, int B, int H, int W,
                  const pbmc_member_queue* queue, pbmc_member* members, int64_t* seq_row, cudaStream_t st) {
  const size_t n = (size_t)H * W;
  const int parts = clock_parts(n);
  size_t chunk = (n + parts - 1) / parts;
  chunk = (chunk + 3) & ~(size_t)3;
  const int nch = p ? 4 : 3;
  pbmc_member_queue qu;
  memset(&qu, 0, sizeof(qu));  // Q = 0: no queue
  if (queue) qu = *queue;
  const size_t smem = queue ? (size_t)B * sizeof(int) : 0;
  clock_apply_kernel<<<dim3(parts, B), CLK_THREADS, 0, st>>>(clk, Tin, Tout, u, v, p, dt_row, ring, slots, nch, n, chunk, qu);
  PBMC_CHECK_LAUNCH("clock_apply_kernel");
  clock_commit_kernel<<<1, CLK_THREADS, smem, st>>>(clk, dt_row, meanT_row, meta, slots, parts, 1.0 / (double)n, B, qu, members,
                                                     seq_row);
  PBMC_CHECK_LAUNCH("clock_commit_kernel");
  return PBMC_OK;
}

}  // namespace pbmc
