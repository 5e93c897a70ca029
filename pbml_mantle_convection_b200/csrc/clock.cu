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
//
// With a diagnostics descriptor (pbmc_rollout_diagnosed) the same two launches also log the wall fluxes and the rms
// velocity of every step and stop members at a statistical steady state (include/pbmc.h states the definitions): apply
// reads u and v on the pass that sums T and writes five more per-CTA partials (the sums of rows 0, 1, H-2, H-1 of T and
// the interior sum of u^2 + v^2); commit sums them in a fixed order, writes flux_seq / vrms_seq, pushes (meanT, q_top,
// vrms) into the slot's history ring and scans the ring with the member's warp.  A member found steady after step s
// stops at step s + 1 through clock_stops, so the queue's refill rule needs nothing new.  Without a descriptor
// (dg.part == NULL, block-uniform) neither kernel touches any of this.
//
// With chains (pbmc_rollout_chained) a stopping slot whose member has a successor hands its T over in place: apply
// skips the T0 overwrite and stores the slot's new T into the successor's T0 row on the same pass; commit loads the
// successor's clock and member row.  The refill rank counts only the stopping slots without a successor, and queue
// entries come from the heads list.  Without chains (ch.succ == NULL, block-uniform) neither kernel touches any of this.
#include <string.h>

#include "common.cuh"

namespace pbmc {

namespace {

constexpr int CLK_THREADS = 256;

constexpr int DIAG_SUMS = 5;  // per-CTA partials of a descriptor: rows 0, 1, H-2, H-1 of T, interior u^2 + v^2

// the member's PBMC_STEADY_* state (always NONE without a descriptor)
__device__ __forceinline__ int steady_of(const pbmc_diag_desc& dg, int m) { return dg.steady ? dg.steady[m] : PBMC_STEADY_NONE; }
// the decision of this step, from the clock (and steady state) as it was before the step (identical in apply and commit)
__device__ __forceinline__ bool clock_active(const pbmc_member_clock& c, int st) {
  return st != PBMC_STEADY_STOPPED && c.t < c.t_end && c.steps < c.max_steps;
}
__device__ __forceinline__ bool clock_ring_full(const pbmc_member_clock& c, int slots) { return c.snaps - c.drained >= slots; }
// whether this step stops the member: active before it, and either found steady after the previous step or not active
// after t += dt, steps += 1 (what commit then computes)
__device__ __forceinline__ bool clock_stops(const pbmc_member_clock& c, double dt, int st) {
  return clock_active(c, st) && (st == PBMC_STEADY_FOUND || !(c.t + dt < c.t_end && c.steps + 1 < c.max_steps));
}
// the successor of the member in slot m (-1: none, or no chains)
__device__ __forceinline__ int64_t chain_succ(const pbmc_member_chain& ch, const pbmc_member_queue& qu, int m) {
  if (!ch.succ) return -1;
  const int64_t w = qu.slot_member[m];
  return w < 0 ? -1 : ch.succ[w];
}
// the queue entry that head rank j (next + r) stands for
__device__ __forceinline__ int64_t head_entry(const pbmc_member_chain& ch, int64_t j) { return ch.succ ? ch.heads[j] : j; }

// cell e (column col) of a member plane into the descriptor's sums; rb / rt = first cell of rows H-2 / H-1 (H >= 3:
// for H = 3 row 1 goes into both r1 and rb)
__device__ __forceinline__ void diag_cell(size_t e, int col, float t, float u, float v, size_t W, size_t rb, size_t rt,
                                          double (&a)[DIAG_SUMS]) {
  if (e < 2 * W) {
    if (e < W) a[0] += (double)t;
    else a[1] += (double)t;
  }
  if (e >= rb) {
    if (e < rt) a[2] += (double)t;
    else a[3] += (double)t;
  }
  if (e >= W && e < rt && col != 0 && col != (int)W - 1) a[4] += (double)u * (double)u + (double)v * (double)v;
}

// four blocks per SM: the descriptor's sums fit in the 64 registers the kernel had without them (no spills)
__global__ void __launch_bounds__(CLK_THREADS, 4)
    clock_apply_kernel(pbmc_member_clock* __restrict__ clk, const float* __restrict__ Tin, float* __restrict__ Tout,
                       const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ p,
                       const double* __restrict__ dt_row, float* __restrict__ ring, int slots, int nch, size_t n, size_t chunk,
                       int W, const pbmc_member_queue qu, const pbmc_diag_desc dg, const pbmc_member_chain ch) {
  __shared__ double red[1 + DIAG_SUMS][CLK_THREADS / 32];
  const int m = blockIdx.y, part = blockIdx.x;
  const int B = gridDim.y;
  const pbmc_member_clock c = clk[m];
  const size_t lo = (size_t)part * chunk, hi = lo + chunk < n ? lo + chunk : n;
  const size_t base = (size_t)m * n;
  const bool vec = (n & 3) == 0;  // every member plane and chunk boundary is then 16-byte aligned
  const bool diag = dg.part != nullptr;
  const int st = steady_of(dg, m);
  if (!clock_active(c, st)) {
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
  // queue: this member stops here.  With a successor its new T stays and is also stored into the successor's T0 row
  // (hand = true); otherwise, when the queue holds a head for the slot, that head's T0 replaces the new T once read
  // (block-uniform: every thread reads the same clocks, dt row, slot members and next).  One pointer for both: the
  // kernel has no register to spare
  float* T0q = nullptr;
  bool hand = false;
  if (qu.Q > 0 && clock_stops(c, dt_row[m], st)) {
    const int64_t succ = chain_succ(ch, qu, m);
    if (succ >= 0) {
      T0q = const_cast<float*>(qu.T0) + (size_t)succ * n;  // written for chains only (include/pbmc.h)
      hand = true;
    } else {
      int r = 0;
      for (int b0 = 0; b0 < m; b0 += CLK_THREADS) {
        const int o = b0 + (int)threadIdx.x;
        r += __syncthreads_count(o < m && clock_stops(clk[o], dt_row[o], steady_of(dg, o)) && chain_succ(ch, qu, o) < 0);
      }
      const int64_t j = *qu.next + r;
      if (j < (ch.succ ? ch.K : qu.Q)) T0q = const_cast<float*>(qu.T0) + (size_t)head_entry(ch, j) * n;
    }
  }
  double s = 0.0;
  double a[DIAG_SUMS] = {0.0, 0.0, 0.0, 0.0, 0.0};  // descriptor sums (diag only)
  const size_t Ws = (size_t)W, rb = n - 2 * Ws, rt = n - Ws;
  if (vec) {
    const size_t i0 = lo + 4 * threadIdx.x;
    int col = diag ? (int)(i0 % Ws) : 0;  // column of cell i, advanced with the stride (W >= 3: one wrap at most)
    const int col_step = (int)((4 * CLK_THREADS) % Ws);
    for (size_t i = i0; i < hi; i += 4 * CLK_THREADS) {
      const float4 t4 = *reinterpret_cast<const float4*>(Tout + base + i);
      s += ((double)t4.x + (double)t4.y) + ((double)t4.z + (double)t4.w);
      if (hand) *reinterpret_cast<float4*>(T0q + i) = t4;  // here: t4 is not kept live across the diagnostics
      float4 u4, v4;
      if (snap || diag) {
        u4 = *reinterpret_cast<const float4*>(u + base + i);
        v4 = *reinterpret_cast<const float4*>(v + base + i);
      }
      if (snap) {
        *reinterpret_cast<float4*>(dst + i) = t4;
        *reinterpret_cast<float4*>(dst + n + i) = u4;
        *reinterpret_cast<float4*>(dst + 2 * n + i) = v4;
        if (nch == 4) *reinterpret_cast<float4*>(dst + 3 * n + i) = *reinterpret_cast<const float4*>(p + base + i);
      }
      if (diag) {
        const float tt[4] = {t4.x, t4.y, t4.z, t4.w}, uu[4] = {u4.x, u4.y, u4.z, u4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int cj = col + j;
          if (cj >= W) cj -= W;
          diag_cell(i + j, cj, tt[j], uu[j], vv[j], Ws, rb, rt, a);
        }
        col += col_step;
        if (col >= W) col -= W;
      }
      if (T0q && !hand) *reinterpret_cast<float4*>(Tout + base + i) = *reinterpret_cast<const float4*>(T0q + i);
    }
  } else {
    const size_t i0 = lo + threadIdx.x;
    int col = diag ? (int)(i0 % Ws) : 0;
    const int col_step = (int)(CLK_THREADS % Ws);
    for (size_t i = i0; i < hi; i += CLK_THREADS) {
      const float t1 = Tout[base + i];
      s += (double)t1;
      if (hand) T0q[i] = t1;
      if (snap) {
        dst[i] = t1;
        dst[n + i] = u[base + i];
        dst[2 * n + i] = v[base + i];
        if (nch == 4) dst[3 * n + i] = p[base + i];
      }
      if (diag) {
        diag_cell(i, col, t1, u[base + i], v[base + i], Ws, rb, rt, a);
        col += col_step;
        if (col >= W) col -= W;
      }
      if (T0q && !hand) Tout[base + i] = T0q[i];
    }
  }
  // fixed-order block reduction: warp tree, then warp 0 over the warp sums
  s = warp_sum(s);
  if (diag) {
#pragma unroll
    for (int k = 0; k < DIAG_SUMS; ++k) a[k] = warp_sum(a[k]);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = s;
    if (diag) {
#pragma unroll
      for (int k = 0; k < DIAG_SUMS; ++k) red[1 + k][threadIdx.x >> 5] = a[k];
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    double w = threadIdx.x < CLK_THREADS / 32 ? red[0][threadIdx.x] : 0.0;
    w = warp_sum(w);
    // the partials are the only clock words this kernel writes; only commit reads them
    if (threadIdx.x == 0) clk[m].part[part] = w;
    if (diag) {
#pragma unroll
      for (int k = 0; k < DIAG_SUMS; ++k) {
        double x = threadIdx.x < CLK_THREADS / 32 ? red[1 + k][threadIdx.x] : 0.0;
        x = warp_sum(x);
        if (threadIdx.x == 0) dg.part[((size_t)m * DIAG_SUMS + k) * PBMC_CLOCK_PARTS + part] = x;
      }
    }
  }
}

// one warp per member (strided), lane 0 writes.  Queue (qu.Q > 0): `stops` (dynamic shared memory, [B]) holds
// clock_stops of every slot, taken before any clock is written (1: the slot takes a head, 2: its member has a successor);
// members / seq_row are the member rows and this step's member_seq row.  Descriptor (dg.part != NULL): dg.flux_seq /
// dg.vrms_seq are this step's rows.
__global__ void __launch_bounds__(CLK_THREADS) clock_commit_kernel(pbmc_member_clock* __restrict__ clk, double* __restrict__ dt_row,
                                                                   double* __restrict__ meanT_row, double* __restrict__ meta, int slots,
                                                                   int parts, double inv_n, int H, int W, int B,
                                                                   const pbmc_member_queue qu,
                                                                   pbmc_member* __restrict__ members, int64_t* __restrict__ seq_row,
                                                                   const pbmc_diag_desc dg, const pbmc_member_chain ch) {
  extern __shared__ int stops[];
  const int lane = threadIdx.x & 31;
  const bool queued = qu.Q > 0;
  const bool diag = dg.part != nullptr;
  int64_t next = 0;
  if (queued) {
    next = *qu.next;
    for (int m = threadIdx.x; m < B; m += CLK_THREADS)
      stops[m] = clock_stops(clk[m], dt_row[m], steady_of(dg, m)) ? (chain_succ(ch, qu, m) >= 0 ? 2 : 1) : 0;
    __syncthreads();
  }
  for (int m = threadIdx.x >> 5; m < B; m += CLK_THREADS / 32) {
    pbmc_member_clock* c = clk + m;
    const int st = steady_of(dg, m);
    if (!clock_active(*c, st)) {
      if (lane == 0) {
        dt_row[m] = 0.0;  // so the caller's time bookkeeping (sum of dt rows) stays right
        c->active = 0;
        if (queued) seq_row[m] = -1;
        if (diag) {
          dg.flux_seq[2 * m] = dg.flux_seq[2 * m + 1] = 0.0;
          dg.vrms_seq[m] = 0.0;
        }
      }
      continue;
    }
    double s = 0.0;
    for (int q = lane; q < parts; q += 32) s += c->part[q];  // lane q sums partials q, q + 32, ...: fixed order
    s = warp_sum(s);
    double a[DIAG_SUMS] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (diag) {
#pragma unroll
      for (int k = 0; k < DIAG_SUMS; ++k) {
        const double* pk = dg.part + ((size_t)m * DIAG_SUMS + k) * PBMC_CLOCK_PARTS;
        for (int q = lane; q < parts; q += 32) a[k] += pk[q];  // same fixed order
        a[k] = warp_sum(a[k]);
      }
    }
    int r = 0;  // rank among the slots that stop at this step and take a head (the apply kernel's count)
    if (queued && stops[m] == 1) {
      for (int o = lane; o < m; o += 32) r += stops[o] == 1;
      r = __reduce_add_sync(0xffffffffu, r);
    }
    int scan = 0;  // the member goes on and its history ring holds `window` values: evaluate the criterion
    if (lane == 0) {
      const int64_t who = queued ? qu.slot_member[m] : -1;
      if (queued) seq_row[m] = who;
      const double mean = s * inv_n;
      meanT_row[m] = mean;
      double q_top = 0.0, vrms = 0.0;
      if (diag) {
        const double rows = (double)W;
        q_top = -(a[3] / rows - a[2] / rows) * dg.inv_dy_top;
        vrms = sqrt(a[4] / ((double)(H - 2) * (double)(W - 2)));
        dg.flux_seq[2 * m] = -(a[1] / rows - a[0] / rows) * dg.inv_dy_bot;
        dg.flux_seq[2 * m + 1] = q_top;
        dg.vrms_seq[m] = vrms;
      }
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
      bool running = clock_active(*c, PBMC_STEADY_NONE);
      if (st == PBMC_STEADY_FOUND) {
        // the step after the one the criterion held for: stop here; reported steady unless t_end / max_steps stop it too
        dg.steady[m] = running ? PBMC_STEADY_STOPPED : PBMC_STEADY_NONE;
        running = false;
      }
      c->active = running ? 1 : 0;
      int64_t q = -1;  // the slot's next member, from step i + 1 on: the successor, or the head of rank r
      if (queued && stops[m] == 2) q = ch.succ[who];
      else if (queued && stops[m] == 1 && next + r < (ch.succ ? ch.K : qu.Q)) q = head_entry(ch, next + r);
      if (q >= 0) {
        c->t = qu.t0[q];
        c->t_end = qu.t_end[q];
        c->save_t = 0.0;
        c->save_every = qu.save_every[q];
        c->steps = qu.n_step0[q];
        c->max_steps = qu.max_steps[q];
        c->active = 1;
        members[m] = qu.params[q];
        qu.slot_member[m] = q;
        if (diag) {
          dg.steady[m] = PBMC_STEADY_NONE;
          if (dg.hist_n) dg.hist_n[m] = 0;
        }
      }
      if (diag && dg.window > 0 && running) {
        const int64_t h = dg.hist_n[m];
        double* e = dg.hist + ((size_t)m * dg.window + (size_t)(h % dg.window)) * 3;
        e[0] = mean;
        e[1] = q_top;
        e[2] = vrms;
        dg.hist_n[m] = h + 1;
        scan = h + 1 >= dg.window;
      }
    }
    if (__shfl_sync(0xffffffffu, scan, 0)) {
      __syncwarp();  // lane 0's push is visible to the warp
      // one series at a time: min / max are exact, so the lanes' order does not matter
      bool steady = true;
      for (int k = 0; k < 3; ++k) {
        double mn = INFINITY, mx = -INFINITY;
        bool finite = true;
        for (int j = lane; j < dg.window; j += 32) {
          const double x = dg.hist[((size_t)m * dg.window + j) * 3 + k];
          finite = finite && isfinite(x);
          mn = fmin(mn, x);
          mx = fmax(mx, x);
        }
        for (int o = 16; o > 0; o >>= 1) {
          mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
          mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        // rounded sub / mul intrinsics: never contracted into an fma, so the host replays the same decision
        steady = steady && __all_sync(0xffffffffu, finite) &&
                 __dsub_rn(mx, mn) <= __dmul_rn(dg.rtol, fmax(fabs(mx), fabs(mn)));
      }
      if (lane == 0) {
        if (steady) dg.steady[m] = PBMC_STEADY_FOUND;
      }
    }
  }
  if (queued) {
    __syncthreads();  // every thread has read next
    if (threadIdx.x == 0) {
      int64_t k = 0;
      for (int m = 0; m < B; ++m) k += stops[m] == 1;
      const int64_t K = ch.succ ? ch.K : qu.Q;
      *qu.next = next + k < K ? next + k : K;
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
// diag (NULL: none): the diagnostics descriptor with flux_seq / vrms_seq pointing at the step's rows.
// chain (NULL: none; only with a queue): the queue's successor and head lists.
int clock_enqueue(pbmc_member_clock* clk, const float* Tin, float* Tout, const float* u, const float* v, const float* p,
                  double* dt_row, double* meanT_row, float* ring, double* meta, int slots, int B, int H, int W,
                  const pbmc_member_queue* queue, pbmc_member* members, int64_t* seq_row, const pbmc_diag_desc* diag,
                  const pbmc_member_chain* chain, cudaStream_t st) {
  const size_t n = (size_t)H * W;
  const int parts = clock_parts(n);
  size_t chunk = (n + parts - 1) / parts;
  chunk = (chunk + 3) & ~(size_t)3;
  const int nch = p ? 4 : 3;
  pbmc_member_queue qu;
  memset(&qu, 0, sizeof(qu));  // Q = 0: no queue
  if (queue) qu = *queue;
  pbmc_diag_desc dg;
  memset(&dg, 0, sizeof(dg));  // part = NULL: no diagnostics
  if (diag) dg = *diag;
  pbmc_member_chain ch;
  memset(&ch, 0, sizeof(ch));  // succ = NULL: no chains
  if (chain) ch = *chain;
  const size_t smem = queue ? (size_t)B * sizeof(int) : 0;
  clock_apply_kernel<<<dim3(parts, B), CLK_THREADS, 0, st>>>(clk, Tin, Tout, u, v, p, dt_row, ring, slots, nch, n, chunk, W, qu,
                                                             dg, ch);
  PBMC_CHECK_LAUNCH("clock_apply_kernel");
  clock_commit_kernel<<<1, CLK_THREADS, smem, st>>>(clk, dt_row, meanT_row, meta, slots, parts, 1.0 / (double)n, H, W, B, qu, members,
                                                     seq_row, dg, ch);
  PBMC_CHECK_LAUNCH("clock_commit_kernel");
  return PBMC_OK;
}

}  // namespace pbmc
