"""Device-resident rollouts: B independent members (varying Ra / initial T) advanced together.

This is the GAIA-free form of the reference's hot loop (advect_wi_gaia.py:583-668 around
`ts_net(...)`, i.e. `TS.forward`'s loop pytorch_networks_convae.py:377-473): T, u, v and dt
never leave the device; a whole block of time steps is one CUDA graph.  Each member keeps its
own CFL time step (the reference runs one member per process; ADNet's batch-global amax,
:556, is not inherited here -- use `per_member_dt=False` for that behaviour).

Run to a simulated end time (`start_clock` / `drain`): each member carries a clock in device memory that the device
advances after every step (pbmc_rollout_clocked): a member runs `while t < t_end` like the reference driver
(advect_wi_gaia.py:583), logs mean-T after every step and takes its snapshots at the exact steps where `t > save_t`;
once stopped it is frozen (T bit-identical, dt rows 0) while the others go on.  The host reads the logs once per block.

Sweeps larger than the batch (`start_sweep`): Q members run through the B slots; when a slot's member stops, the device
puts the next queued member into it inside the same graph (pbmc_rollout_queued), so no slot idles while the queue holds
members.

Per-step diagnostics and the steady stop (`start_clock(..., diagnostics=True)` or `steady=(window, rtol)`, the same for
`start_sweep`): the same launches also log the wall heat fluxes q_bot / q_top and the rms velocity of every step
(pbmc_rollout_diagnosed; include/pbmc.h defines them), and with `steady` a member stops one step after its meanT, q_top
and vrms have each varied by at most rtol (relative) over the last `window` steps.

Parameter continuation (`start_sweep(..., continue_from=...)`): a member may start from the T its predecessor stopped
with, handed over on the device in the predecessor's slot (pbmc_rollout_chained), so a ladder of parameters follows one
branch of steady states without a host round-trip between rungs.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L
from . import ops
from .engine import Grid, RolloutState


def synthetic_grid(H, W):
    """Cell-centre coordinates of the box [0,4]x[0,1] (SURVEY.md section 8d); at 128x506 this is
    the reference's GAIA grid (prepare_gaia_ini.py:24-25).  float64 numpy [H,W] pair."""
    x = np.empty(W)
    y = np.empty(H)
    x[0], x[-1] = 0.0, 4.0
    x[1:-1] = (np.arange(1, W - 1) - 0.5) * 4.0 / (W - 2)
    y[0], y[-1] = 0.0, 1.0
    y[1:-1] = (np.arange(1, H - 1) - 0.5) / (H - 2)
    return np.broadcast_to(x[None, :], (H, W)).copy(), np.broadcast_to(y[:, None], (H, W)).copy()


def synthetic_T0(H, W, seed=1):
    """Conductive profile + 1 % noise with the wall rows/columns enforced (SURVEY.md section 8d)."""
    _, yc = synthetic_grid(H, W)
    T = (1.0 - yc) + 0.01 * np.random.default_rng(seed).random((H, W))
    T[0, :], T[-1, :] = 1.0, 0.0
    T[:, 0], T[:, -1] = T[:, 1], T[:, -2]
    return T


_W = lambda name: getattr(L.MemberClock, name).offset // 8  # 8-byte word of a pbmc_member_clock field
_T, _T_END, _SAVE_T, _SAVE_EVERY = _W("t"), _W("t_end"), _W("save_t"), _W("save_every")
_STEPS, _MAX_STEPS, _SNAPS, _DRAINED = _W("steps"), _W("max_steps"), _W("snaps"), _W("drained")
_ACTIVE, _OVERFLOW = 2 * _W("active"), 2 * _W("active") + 1  # int32 words
_HDR = _W("part")  # the counters; the partial sums after them are device scratch
_NO_LIMIT = 1 << 62


class MemberClocks:
    """Device buffers of a clocked rollout: one pbmc_member_clock per member (as a [B, words] float64 tensor, viewed as
    int64 / int32 for the integer fields), meanT_seq (indexed like dt_seq) and the snapshot ring with its metadata."""

    def __init__(self, B, H, W, rows, p_pred, slots, device):
        words = C.sizeof(L.MemberClock) // 8
        self.clock = torch.zeros(B, words, dtype=torch.float64, device=device)
        self.meanT_seq = torch.zeros(rows, B, dtype=torch.float64, device=device)
        self.nch = 4 if p_pred else 3
        self.slots = int(slots)
        self.ring = torch.zeros(self.slots, B, self.nch, H, W, dtype=torch.float32, device=device)
        self.meta = torch.zeros(self.slots, B, 2, dtype=torch.float64, device=device)

    def key(self):
        return ("clock", self.clock.data_ptr(), self.meanT_seq.data_ptr(), self.ring.data_ptr(), self.meta.data_ptr(), self.slots)


class SweepQueue:
    """Device buffers of a sweep's member queue (pbmc_member_queue): the queued members' T0, parameter rows and clock
    starts, `next`, the slot each member is in and the member_seq / snap_member tags.  `desc` is the C struct.  With
    chains also the heads and successors of pbmc_member_chain; `chain` is that C struct (its K is set per sweep)."""

    def __init__(self, Q, B, H, W, rows, slots, device):
        f64 = lambda n: torch.zeros(n, dtype=torch.float64, device=device)
        i64 = lambda *n: torch.full(n, -1, dtype=torch.int64, device=device)
        self.Q, self.B, self.slots = int(Q), int(B), int(slots)
        self.T0 = torch.zeros(Q, H, W, dtype=torch.float32, device=device)
        self.params = torch.zeros(Q, C.sizeof(L.Member) // 4, dtype=torch.float32, device=device)
        self.t0, self.t_end, self.save_every = f64(Q), f64(Q), f64(Q)
        self.n_step0, self.max_steps = i64(Q), i64(Q)
        self.next, self.slot_member = i64(1), i64(B)
        self.member_seq, self.snap_member = i64(rows, B), i64(self.slots, B)
        d = self.desc = L.MemberQueue()
        for name in ("T0", "params", "t0", "t_end", "save_every", "n_step0", "max_steps", "next", "slot_member", "member_seq",
                     "snap_member"):
            setattr(d, name, L.ptr(getattr(self, name)))
        d.Q = self.Q
        self.heads, self.succ = i64(Q), i64(Q)
        self.chain = L.MemberChain()
        self.chain.heads, self.chain.succ = L.ptr(self.heads), L.ptr(self.succ)

    def key(self):
        d = self.desc
        return ("queue", d.T0, d.params, d.t0, d.t_end, d.save_every, d.n_step0, d.max_steps, d.next, d.slot_member,
                d.member_seq, d.snap_member, d.Q)

    def chain_key(self):
        return ("chain", self.chain.heads, self.chain.succ, self.chain.K)  # K is a launch argument


class MemberDiagnostics:
    """Device buffers of the per-step diagnostics and the steady criterion (pbmc_diag_desc): flux_seq [rows, B, 2] =
    (q_bot, q_top) and vrms_seq [rows, B], indexed like dt_seq; each slot's history ring of (meanT, q_top, vrms) with its
    count, the PBMC_STEADY_* state per slot and the partials scratch.  window = 0: diagnostics only.  `desc` is the C
    struct."""

    def __init__(self, B, rows, window, rtol, grid, device):
        f64 = lambda *n: torch.zeros(n, dtype=torch.float64, device=device)
        self.window, self.rtol = int(window), float(rtol)
        self.flux_seq, self.vrms_seq = f64(rows, B, 2), f64(rows, B)
        self.hist = f64(B, self.window, 3) if self.window else None
        self.hist_n = torch.zeros(B, dtype=torch.int64, device=device)
        self.steady = torch.zeros(B, dtype=torch.int32, device=device)
        self.part = f64(B, 5, L.CLOCK_PARTS)
        y = grid.y1d64  # row coordinates, walls forced to 0 and 1
        d = self.desc = L.DiagDesc()
        d.inv_dy_bot, d.inv_dy_top = 1.0 / float(y[1] - y[0]), 1.0 / float(y[-1] - y[-2])
        d.window, d.rtol = self.window, self.rtol
        for name in ("flux_seq", "vrms_seq", "hist", "hist_n", "steady", "part"):
            setattr(d, name, L.ptr(getattr(self, name)))

    def reset(self):
        """A clock starts: no history, nobody steady."""
        self.hist_n.zero_()
        self.steady.zero_()

    def key(self):
        d = self.desc
        return ("diag", d.flux_seq, d.vrms_seq, d.hist, d.hist_n, d.steady, d.part, self.window, self.rtol)


def _steady_args(diagnostics, steady):
    """(window, rtol) of start_clock / start_sweep's arguments, None without diagnostics."""
    if steady is None:
        return (0, 0.0) if diagnostics else None
    window, rtol = steady
    if isinstance(window, bool) or int(window) != window or not 1 <= int(window) <= L.STEADY_MAX_WINDOW:
        raise ValueError(f"steady window must be an integer in [1, {L.STEADY_MAX_WINDOW}], got {window!r}")
    rtol = float(rtol)
    if not (math.isfinite(rtol) and rtol >= 0.0):
        raise ValueError(f"steady rtol must be finite and >= 0, got {rtol!r}")
    return int(window), rtol


def _continue_from(continue_from, Q, can_step):
    """start_sweep's continue_from checked against the Q members (can_step: whether each could take a step): int64 [Q]."""
    if len(continue_from) != Q:
        raise ValueError(f"continue_from has {len(continue_from)} entries for {Q} members")
    cf = np.empty(Q, dtype=np.int64)
    for q, p in enumerate(continue_from):
        if isinstance(p, (bool, np.bool_)) or not isinstance(p, (int, np.integer)):
            raise ValueError(f"continue_from[{q}] must be an integer member index or -1, got {p!r}")
        if not -1 <= p < q:
            raise ValueError(f"continue_from[{q}] = {p}: a member continues from an earlier member (0 <= p < {q}) or -1")
        cf[q] = p
    preds = cf[cf >= 0]
    if len(np.unique(preds)) != len(preds):
        dup = sorted({int(p) for p in preds if (preds == p).sum() > 1})
        raise ValueError(f"members {dup} are continued by more than one member")
    chained = cf >= 0
    chained[preds] = True
    bad = np.flatnonzero(chained & ~can_step)
    if len(bad):
        raise ValueError(f"members {bad.tolist()} are in a chain but would take no step (t0 >= t_end or n_step >= "
                         "max_steps): the chain would break")
    return cf


class EnsembleRollout:
    """B members on one GPU.  `params`: list of (RaQ, gamma=fkt, beta=fkp), one per member."""

    def __init__(self, net, H, W, params, device, xc=None, yc=None, cn_max=0.99, per_member_dt=True, max_steps=4096):
        self.net, self.device = net, torch.device(device)
        self.B, self.H, self.W = len(params), H, W
        if xc is None:
            xc, yc = synthetic_grid(H, W)
        xc_t, yc_t = torch.as_tensor(xc, dtype=torch.float64), torch.as_tensor(yc, dtype=torch.float64)
        self.grid = Grid(xc_t, yc_t, yc_t, self.device)
        if not self.grid.separable:
            raise NotImplementedError("EnsembleRollout needs a separable (tensor-product) grid; use TS for general fields")
        self.members = ops.make_members(params, self.device)
        self.engine = net._engine(self.device)
        self.state = RolloutState(self.grid, self.members, self.B, 2, max_steps, cn_max, per_member_dt, net.p_pred,
                                  self.device)
        self.max_steps = max_steps
        self.n_done = 0
        self.time = torch.zeros(self.B, dtype=torch.float64, device=self.device)
        self._graphs = {}
        self._stream = torch.cuda.Stream(self.device)
        self._clk = None      # MemberClocks while a clock runs (start_clock)
        self._clocks = None   # the last MemberClocks (its buffers, and so its graphs, serve the next clock of that ring size)
        self._pending = None  # (first dt_seq row, steps) of the block not drained yet
        self._queue = None    # SweepQueue of the last sweep (its buffers, and so its graphs, serve the next one of that shape)
        self._sweep = None    # host bookkeeping while a sweep runs (start_sweep)
        self._diag = None     # MemberDiagnostics while a clock runs with diagnostics
        self._diags = {}      # (window, rtol) -> MemberDiagnostics: buffers, and so graphs, kept for the next clock

    # ------------------------------------------------------------------ state
    def set_T(self, T0):
        """T0: [B,H,W] (numpy or tensor, any float dtype)."""
        T0 = torch.as_tensor(T0).to(self.device, torch.float32).reshape(self.B, self.H, self.W)
        self.state.T_seq[self.n_done % 2].copy_(T0)

    @property
    def T(self):
        return self.state.T_seq[self.n_done % 2]

    # ------------------------------------------------------------------ stepping
    def step(self, n=1):
        """Enqueue n time steps directly (no graph)."""
        done = 0
        self.engine = self.net._engine(self.device)  # picks up a changed net.conv_impl
        if self._clk is not None and n > self.max_steps:
            raise ValueError("a clocked rollout advances at most max_steps steps between two drain() calls")
        while done < n:
            # dt history is written relative to first_step (rows first-1 .. first-1+k-1 of max_steps + 1); restart the
            # index every call
            first = 1 + (self.n_done % 2)
            k = min(n - done, self.max_steps)
            self._begin_block(first - 1, k)
            self.engine.rollout(self.state, first, k, clock=self._clk, queue=self._run_queue(), diag=self._diag,
                                chain=self._run_chain())
            self.time += self.state.dt_seq[first - 1:first - 1 + k].sum(0)
            self.n_done += k
            done += k

    def graph(self, steps_per_graph):
        """Capture (once per (k, slot parity)) and return the CUDA graph of k time steps starting
        from the current T slot.  Replaying it advances the state by k steps."""
        k = int(steps_per_graph)
        if k < 1 or k > self.max_steps - 1:
            raise ValueError("steps_per_graph out of range")
        self.engine = self.net._engine(self.device)  # picks up a changed net.conv_impl
        par = self.n_done % 2
        # the graph bakes in packed-weight and workspace addresses and the conv implementation: key on them too
        key = (k, par) + self.engine.graph_key(self.B, self.H, self.W)
        clk, qu, dg, ch = self._clk, self._run_queue(), self._diag, self._run_chain()
        if clk is not None:
            key = key + clk.key()  # a clocked graph: its own entry (t_end, save_every live in device memory)
        if qu is not None:
            key = key + qu.key()  # a sweep's graph: refills only rewrite device memory
        if dg is not None:
            key = key + dg.key()  # window and rtol are launch arguments
        if ch is not None:
            key = key + qu.chain_key()
        if key not in self._graphs:
            # eager warm-up (module load + func attributes outside capture) on saved state: what a step may rewrite
            saved = [self.state.T_seq] + ([clk.clock] if clk is not None else []) + \
                    ([self.members, qu.next, qu.slot_member] if qu is not None else []) + \
                    ([t for t in (dg.hist, dg.hist_n, dg.steady) if t is not None] if dg is not None else []) + \
                    ([qu.T0] if ch is not None else [])  # a hand-off writes the successor's T0 row
            copies = [t.clone() for t in saved]
            self.engine.rollout(self.state, 1 + par, 1, clock=clk, queue=qu, diag=dg, chain=ch)
            for t, c in zip(saved, copies):
                t.copy_(c)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.engine.rollout(self.state, 1 + par, k, clock=clk, queue=qu, diag=dg, chain=ch)
            self._graphs[key] = g
        return self._graphs[key]

    def run(self, n_steps, steps_per_graph=None, track_time=True):
        """Advance n_steps.  With steps_per_graph=k (divides n_steps) the work is k-step CUDA-graph replays.
        track_time=False skips the (tiny, torch-side) accumulation of simulated time."""
        if not steps_per_graph:
            return self.step(n_steps)
        k = int(steps_per_graph)
        if n_steps % k:
            raise ValueError("n_steps must be a multiple of steps_per_graph")
        if self._clk is not None and n_steps != k:
            raise ValueError("a clocked rollout runs one block (n_steps == steps_per_graph) between two drain() calls")
        for _ in range(n_steps // k):
            par = self.n_done % 2
            g = self.graph(k)
            self._begin_block(par, k)
            g.replay()
            if track_time:
                self.time += self.state.dt_seq[par:par + k].sum(0)
            self.n_done += k

    # ------------------------------------------------------------------ outputs
    def fields(self):
        """(u, v, p, V) of the last step, float32 [B,H,W].  With a clock, a frozen member's entries are the surrogate's
        output for its frozen T -- the velocities of a step it does not take, not those of its last step; its snapshots
        hold the right ones."""
        s = self.state
        return s.u, s.v, s.p, s.V

    def last_dt(self):
        return self.state.dt_seq

    def diagnostics(self):
        """mean-T [B], profile T(y) [B,H], gradient dT/dy [B,H-1] as float64 tensors
        (advect_wi_gaia.py:547,647; load_advection_results notebook :322-323, r -> the run's y)."""
        mean, prof = ops.diagnostics(self.T.contiguous())
        y = self.grid.y1d64.to(self.device)
        dprof = (prof[:, 1:] - prof[:, :-1]) / (y[1:] - y[:-1])[None]
        return mean, prof, dprof

    # ------------------------------------------------------------------ run to a simulated end time
    def _per_member(self, x, dtype=np.float64):
        return np.broadcast_to(np.asarray(x, dtype=dtype), (self.B,)).copy()

    def start_clock(self, t_end, save_every=0.0, t0=None, max_steps=None, n_step=0, snap_slots=None, steps_per_graph=10,
                    diagnostics=False, steady=None):
        """Give every member a clock (each argument a scalar or one value per member): the following steps run member m
        `while t[m] < t_end[m] and steps[m] < max_steps[m]` (advect_wi_gaia.py:583), log mean-T after every step and take a
        snapshot (T, u, v, p) whenever t > save_t (save_t = 0 at the start, then t + save_every).
          t0         start time (default: `self.time`; given, it also becomes `self.time`)
          n_step     step count at the start (the reference's n_step), max_steps an absolute limit on it (None: none)
          snap_slots snapshot-ring slots per member (default steps_per_graph: a ring drained once per block never fills)
          diagnostics  also log the wall heat fluxes q_bot, q_top and the rms velocity of every step (drain())
          steady     (window, rtol), 1 <= window <= 1024, rtol finite >= 0: diagnostics, and a member stops one step after
                     the last `window` values of each of its meanT, q_top and vrms satisfy max - min <= rtol * max(|max|,
                     |min|) (include/pbmc.h, pbmc_diag_desc); a member stopped so is reported `steady`
        Then alternate `run(k, steps_per_graph=k)` (or `step(n)`) and `drain()` until `any_active()` is False.
        The clock's device buffers (and so its captured graphs) outlive stop_clock(): the next start_clock() or
        start_sweep() with the same ring size reuses them, re-initialised, and captures nothing new."""
        dg = self._new_diag(diagnostics, steady)
        clk = self._new_clock(snap_slots, steps_per_graph)
        if t0 is None:
            t0 = self.time.cpu().numpy()
        t0 = self._per_member(t0)
        steps0 = self._per_member(n_step, np.int64)
        t_end, save_every = self._per_member(t_end), self._per_member(save_every)
        max_steps = self._per_member(_NO_LIMIT if max_steps is None else max_steps, np.int64)
        c = torch.zeros(clk.clock.shape, dtype=torch.float64)
        c[:, _T], c[:, _T_END], c[:, _SAVE_T], c[:, _SAVE_EVERY] = (torch.from_numpy(a) for a in (t0, t_end, np.zeros(self.B), save_every))
        ci = c.view(torch.int64)
        ci[:, _STEPS], ci[:, _MAX_STEPS] = torch.from_numpy(steps0), torch.from_numpy(max_steps)
        active = (t0 < t_end) & (steps0 < max_steps)
        c.view(torch.int32)[:, _ACTIVE] = torch.from_numpy(active.astype(np.int32))
        clk.clock.copy_(c)
        self.time.copy_(torch.from_numpy(t0))
        self._clk, self._diag = clk, dg
        self._pending = None
        self._sweep = None
        self._host_t, self._host_steps, self._host_active = t0, steps0, active
        self._t_end, self._max_steps = t_end, max_steps

    def _new_clock(self, snap_slots, steps_per_graph):
        """The MemberClocks for a clock with this ring size: the current one when it fits (its graphs stay valid)."""
        slots = int(snap_slots if snap_slots is not None else steps_per_graph)
        if slots < 1:
            raise ValueError("snap_slots must be >= 1")
        if not self.state.per_member_dt and self.B > 1:
            raise L.PbmcError("a clock needs per_member_dt=True when B > 1: with a batch-global dt a frozen member would "
                              "still set the others' time step")
        clk = self._clocks
        if clk is None or clk.slots != slots:
            self._graphs = {k: g for k, g in self._graphs.items() if "clock" not in k}  # graphs of the old buffers
            clk = MemberClocks(self.B, self.H, self.W, self.state.dt_seq.shape[0], self.state.p is not None, slots, self.device)
            self._clocks = clk
        return clk

    def _new_diag(self, diagnostics, steady):
        """The MemberDiagnostics of start_clock / start_sweep's arguments (None: none), reset; cached per (window, rtol)."""
        wr = _steady_args(diagnostics, steady)
        if wr is None:
            return None
        dg = self._diags.get(wr)
        if dg is None:
            dg = self._diags[wr] = MemberDiagnostics(self.B, self.state.dt_seq.shape[0], wr[0], wr[1], self.grid, self.device)
        dg.reset()
        return dg

    def start_sweep(self, T0, params, t_end, save_every=0.0, t0=0.0, max_steps=None, n_step=0, snap_slots=None,
                    steps_per_graph=10, diagnostics=False, steady=None, continue_from=None):
        """Run Q members (`params`: Q tuples (RaQ, gamma, beta); T0: [Q, H, W]) through this ensemble's B slots, each
        `while t < t_end and steps < max_steps` on its own clock as in start_clock (t_end, save_every, t0, max_steps,
        n_step: scalars or one value per member).  When a slot's member stops, the device puts the next queued member
        into the slot before the following step (include/pbmc.h, pbmc_rollout_queued: of the slots stopping at one step,
        the lower slot index takes the earlier member), inside the same graph.  Members that would take no step are
        finished here and never enter the queue; the first B queued members start in slots 0 .. B - 1 in member order,
        and with fewer queued members than slots the other slots stay frozen.  Then alternate `run(k, steps_per_graph=k)` and `drain()` until `any_active()` is False.
        The slots' T and member rows are rewritten by the sweep (`members` holds the last members afterwards), and
        `time` keeps summing each slot's dt rows: per-member times come from drain().  A second sweep with the same
        number of queued members and ring size reuses the buffers and the captured graphs.
        diagnostics / steady: as in start_clock; a slot's history and steady state start afresh with each member.
        continue_from: None, or one entry per member: p (0 <= p < q, no p twice) makes member q start from the T member p
        had after its last step, in p's slot, at p's stop step whatever stopped p (include/pbmc.h, pbmc_member_chain);
        -1 starts q from T0[q] as without it.  T0[q] of a continued member is ignored.  Members with -1 are chain heads
        and go through the queue rule above among themselves; a member in a chain must be able to take a step
        (ValueError otherwise: it would break the chain).  A continued member's first drained block also carries
        `start_T`, its float32 start field."""
        dg = self._new_diag(diagnostics, steady)
        Qa = len(params)
        bc = lambda x, dt=np.float64: np.broadcast_to(np.asarray(x, dtype=dt), (Qa,)).copy()
        t0, t_end, save_every = bc(t0), bc(t_end), bc(save_every)
        steps0 = bc(n_step, np.int64)
        max_steps = bc(_NO_LIMIT if max_steps is None else max_steps, np.int64)
        can_step = (t0 < t_end) & (steps0 < max_steps)
        cf = None if continue_from is None else _continue_from(continue_from, Qa, can_step)
        T0 = torch.as_tensor(T0).to(torch.float32).reshape(Qa, self.H, self.W)
        index = np.flatnonzero(can_step)  # queue entry -> member
        Q = len(index)
        heads = np.arange(Q)  # queue entries of the chain heads (all entries without chains)
        if cf is not None and Q:
            entry = np.full(Qa, -1, dtype=np.int64)
            entry[index] = np.arange(Q)
            pred = cf[index]  # each entry's predecessor member, -1: a head
            heads = np.flatnonzero(pred < 0)
            succ = np.full(Q, -1, dtype=np.int64)
            succ[entry[pred[pred >= 0]]] = np.flatnonzero(pred >= 0)
        clk = self._new_clock(snap_slots, steps_per_graph)
        qu = self._queue
        if Q and (qu is None or qu.Q != Q or qu.slots != clk.slots):
            self._graphs = {k: g for k, g in self._graphs.items() if "queue" not in k}
            qu = self._queue = SweepQueue(Q, self.B, self.H, self.W, self.state.dt_seq.shape[0], clk.slots, self.device)
        K = len(heads)
        n0 = min(self.B, K)
        active = np.arange(self.B) < n0
        c = torch.zeros(clk.clock.shape, dtype=torch.float64)
        if Q:
            sel = torch.from_numpy(index)
            qu.T0.copy_(T0[sel])
            qu.params.copy_(ops.make_members([params[i] for i in index], self.device))
            for name, a in (("t0", t0), ("t_end", t_end), ("save_every", save_every), ("n_step0", steps0), ("max_steps", max_steps)):
                getattr(qu, name).copy_(torch.from_numpy(a[index]))
            qu.next.fill_(n0)
            qu.slot_member.copy_(torch.from_numpy(np.where(active, heads[np.minimum(np.arange(self.B), n0 - 1)], -1)))
            qu.member_seq.fill_(-1)
            qu.snap_member.fill_(-1)
            if cf is not None:
                qu.heads[:K].copy_(torch.from_numpy(heads))
                qu.succ.copy_(torch.from_numpy(succ))
                qu.chain.K = K
            # slots without a member keep head 0's T and row (finite input to the surrogate); their clocks stay inactive
            fill = torch.from_numpy(heads[np.minimum(np.arange(self.B), n0 - 1)]).to(self.device)
            self.state.T_seq[self.n_done % 2].copy_(qu.T0[fill])
            self.members.copy_(qu.params[fill])
            first = index[heads[:n0]]
            c[:n0, _T], c[:n0, _T_END] = torch.from_numpy(t0[first]), torch.from_numpy(t_end[first])
            c[:n0, _SAVE_EVERY] = torch.from_numpy(save_every[first])
            ci = c.view(torch.int64)
            ci[:n0, _STEPS], ci[:n0, _MAX_STEPS] = torch.from_numpy(steps0[first]), torch.from_numpy(max_steps[first])
        c.view(torch.int32)[:, _ACTIVE] = torch.from_numpy(active.astype(np.int32))
        clk.clock.copy_(c)
        self.time.copy_(c[:, _T])
        self._clk, self._diag = clk, dg
        self._pending = None
        self._sweep = {"index": index, "Q": Q, "K": K, "next": n0, "t": t0, "steps": steps0, "t_end": t_end,
                       "max_steps": max_steps, "chained": cf is not None and Q > 0,
                       # continued members whose start field drain() has not reported yet: member -> queue entry
                       "unstarted": {int(index[e]): int(e) for e in range(Q) if cf is not None and cf[index[e]] >= 0}}
        self._host_active = active

    def stop_clock(self):
        """Back to unclocked stepping.  Also ends a sweep.  The clock's buffers and graphs stay cached for the next
        start_clock() / start_sweep() with the same ring size."""
        self._clk = None
        self._diag = None
        self._pending = None
        self._sweep = None

    def _run_queue(self):
        """The SweepQueue the next steps run with (None: no sweep, or a sweep whose members all finished on the host)."""
        return self._queue if self._sweep is not None and self._sweep["Q"] else None

    def _run_chain(self):
        """The MemberChain the next steps run with (None: no sweep, or a sweep without continue_from)."""
        return self._queue.chain if self._sweep is not None and self._sweep["chained"] else None

    def set_t_end(self, t_end):
        """New end time(s) between blocks: written to the device clock, no re-capture.  A stopped member whose t is now
        below its t_end takes steps again, unless the steady criterion stopped it."""
        self._require_clock(sweep=False)
        self._t_end = self._per_member(t_end)
        self._host_active = (self._host_t < self._t_end) & (self._host_steps < self._max_steps)
        if self._diag is not None:
            self._host_active &= self._diag.steady.cpu().numpy() != L.STEADY_STOPPED
        self._clk.clock[:, _T_END].copy_(torch.from_numpy(self._t_end))
        self._clk.clock.view(torch.int32)[:, _ACTIVE].copy_(torch.from_numpy(self._host_active.astype(np.int32)))

    def set_save_every(self, save_every):
        """New snapshot interval(s) between blocks (applies from the next snapshot on)."""
        self._require_clock(sweep=False)
        self._clk.clock[:, _SAVE_EVERY].copy_(torch.from_numpy(self._per_member(save_every)))

    def any_active(self):
        """Whether a member still takes steps (in a sweep: or waits in the queue), from the counters the last drain()
        read (no device access)."""
        self._require_clock()
        sw = self._sweep
        return bool(self._host_active.any()) or (sw is not None and sw["next"] < sw["K"])

    def read_clock(self):
        """The device clocks as numpy arrays: t, t_end, save_t, steps, snaps, drained, active, overflow (synchronises).
        In a sweep (one clock per slot) also slot_member (the member in each slot, -1: none) and next (queued members
        placed so far; with continue_from, chain heads placed so far).  With diagnostics also steady (the slot's member
        was stopped by the steady criterion)."""
        self._require_clock()
        c = self._clk.clock[:, :_HDR].cpu()
        ci, ci32 = c.view(torch.int64), c.view(torch.int32)
        out = {"t": c[:, _T].numpy(), "t_end": c[:, _T_END].numpy(), "save_t": c[:, _SAVE_T].numpy(),
               "steps": ci[:, _STEPS].numpy(), "snaps": ci[:, _SNAPS].numpy(), "drained": ci[:, _DRAINED].numpy(),
               "active": ci32[:, _ACTIVE].numpy() != 0, "overflow": ci32[:, _OVERFLOW].numpy() != 0}
        if self._diag is not None:
            out["steady"] = self._diag.steady.cpu().numpy() == L.STEADY_STOPPED
        if self._sweep is not None:
            qu = self._run_queue()
            out["slot_member"] = self._member_of(qu.slot_member.cpu().numpy() if qu is not None else np.full(self.B, -1))
            out["next"] = int(qu.next.item()) if qu is not None else 0
        return out

    def _member_of(self, entries):
        """Queue entries (-1: none) -> member indices of the sweep (-1: none)."""
        return np.append(self._sweep["index"], -1)[entries]

    def drain(self):
        """Logs of the block run since the last drain, one dict per member:
          dt, t, meanT  float64 [n] over the n steps the member took (t after each step, mean of T after each step)
          steps         int64 [n], the step numbers
          snapshots     list of dicts (step, t, T, u, v, p) in the order taken; fields float32 numpy [H,W] (p None without p_pred)
        Copies only the counters, the block's rows and the filled ring slots to the host.  Raises if a member's snapshot
        ring overflowed (a snapshot was due while every slot held an undrained one: drain more often or use more slots).
        In a sweep: a dict {member index: logs} over the members that took a step in the block, each with the fields
        above plus `finished` (the member has stopped); t is the cumsum of the member's dt from its own t0.
        With diagnostics, also q_bot, q_top, vrms (float64 [n], one per step taken) and steady (the member has been
        stopped by the steady criterion).  In a sweep with continue_from, a continued member's first dict also has
        start_T: the float32 [H,W] field it started from (its predecessor's T after its last step)."""
        self._require_clock()
        clk = self._clk
        ck = self.read_clock()
        if ck["overflow"].any():
            bad = np.flatnonzero(ck["overflow"]).tolist()
            raise L.PbmcError(f"snapshot ring overflow for members {bad}: a snapshot was due while all {clk.slots} slots held "
                              "undrained snapshots (it was skipped); drain() after every block or pass a larger snap_slots")
        if self._sweep is not None:
            return self._drain_sweep(ck)
        n = ck["steps"] - self._host_steps
        nmax = int(n.max()) if self.B else 0
        if nmax > 0:
            if self._pending is None or nmax > self._pending[1]:
                raise L.PbmcError("clock counters do not match the block that was run")
            lo = self._pending[0]
            dts = self.state.dt_seq[lo:lo + nmax].cpu().numpy()
            mts = clk.meanT_seq[lo:lo + nmax].cpu().numpy()
            if self._diag is not None:
                fls = self._diag.flux_seq[lo:lo + nmax].cpu().numpy()
                vrs = self._diag.vrms_seq[lo:lo + nmax].cpu().numpy()
        _, ring, meta = self._ring_entries(ck)
        out, r = [], 0
        for m in range(self.B):
            k = int(n[m])
            d = {"dt": dts[:k, m].copy() if k else np.zeros(0), "meanT": mts[:k, m].copy() if k else np.zeros(0),
                 "steps": np.arange(self._host_steps[m] + 1, ck["steps"][m] + 1, dtype=np.int64)}
            # the device's own sequence of double additions t += dt, so d["t"][-1] == the clock's t bit for bit
            d["t"] = np.cumsum(np.concatenate(([self._host_t[m]], d["dt"])))[1:]
            snaps = []
            for _ in range(int(ck["snaps"][m] - ck["drained"][m])):
                f = ring[r]
                snaps.append({"step": int(meta[r, 0]), "t": float(meta[r, 1]), "T": f[0], "u": f[1], "v": f[2],
                              "p": f[3] if clk.nch == 4 else None})
                r += 1
            d["snapshots"] = snaps
            if self._diag is not None:
                d["q_bot"] = fls[:k, m, 0].copy() if k else np.zeros(0)
                d["q_top"] = fls[:k, m, 1].copy() if k else np.zeros(0)
                d["vrms"] = vrs[:k, m].copy() if k else np.zeros(0)
                d["steady"] = bool(ck["steady"][m])
            out.append(d)
        clk.clock.view(torch.int64)[:, _DRAINED].copy_(torch.from_numpy(ck["snaps"].copy()))
        self._host_t, self._host_steps, self._host_active = ck["t"].copy(), ck["steps"].copy(), ck["active"].copy()
        self._pending = None
        return out

    def _ring_entries(self, ck):
        """(slot, ring slot) of every undrained snapshot, slot-major, oldest first, and their ring / meta contents."""
        clk = self._clk
        pairs = [(m, j % clk.slots) for m in range(self.B) for j in range(int(ck["drained"][m]), int(ck["snaps"][m]))]
        if not pairs:
            return pairs, None, None
        mi = torch.tensor([m for m, _ in pairs], device=self.device)
        si = torch.tensor([j for _, j in pairs], device=self.device)
        return pairs, clk.ring[si, mi].cpu().numpy(), clk.meta[si, mi].cpu().numpy()

    def _drain_sweep(self, ck):
        sw, clk, qu, dg = self._sweep, self._clk, self._run_queue(), self._diag
        out = {}
        if qu is None:
            self._pending = None
            return out
        pairs, ring, meta = self._ring_entries(ck)
        steps = {}
        if self._pending is not None:
            lo, k = self._pending
            seq = self._member_of(qu.member_seq[lo:lo + k].cpu().numpy())
            dts = self.state.dt_seq[lo:lo + k].cpu().numpy()
            mts = clk.meanT_seq[lo:lo + k].cpu().numpy()
            if dg is not None:
                fls, vrs = dg.flux_seq[lo:lo + k].cpu().numpy(), dg.vrms_seq[lo:lo + k].cpu().numpy()
            for m in np.unique(seq[seq >= 0]):
                j, s = np.nonzero(seq == m)  # row-major: in step order (a member runs in one slot)
                steps[int(m)] = (dts[j, s].copy(), mts[j, s].copy())
                if dg is not None:
                    steps[int(m)] += (fls[j, s, 0].copy(), fls[j, s, 1].copy(), vrs[j, s].copy())
        snaps = {}
        if pairs:
            owner = self._member_of(qu.snap_member.cpu().numpy())
            for r, (s, j) in enumerate(pairs):
                f = ring[r]
                snaps.setdefault(int(owner[j, s]), []).append(
                    {"step": int(meta[r, 0]), "t": float(meta[r, 1]), "T": f[0], "u": f[1], "v": f[2],
                     "p": f[3] if clk.nch == 4 else None})
        running = set(ck["slot_member"][ck["active"]].tolist())
        for m in sorted(set(steps) | set(snaps)):
            dt, mt = steps.get(m, (np.zeros(0), np.zeros(0)))[:2]
            h_t, h_n = sw["t"][m], sw["steps"][m]
            d = {"dt": dt, "meanT": mt, "steps": np.arange(h_n + 1, h_n + 1 + len(dt), dtype=np.int64)}
            d["t"] = np.cumsum(np.concatenate(([h_t], dt)))[1:]  # the device's own additions: == its clock bit for bit
            d["snapshots"] = snaps.get(m, [])
            d["finished"] = m not in running
            if len(dt):
                sw["t"][m], sw["steps"][m] = d["t"][-1], d["steps"][-1]
            if dg is not None:
                d["q_bot"], d["q_top"], d["vrms"] = steps[m][2:] if m in steps else (np.zeros(0),) * 3
                # a refill resets the slot's steady state, so it is read from the clock: a member stops either at its
                # t_end / max_steps or, before both, by the criterion (the limits take precedence at the same step)
                d["steady"] = bool(d["finished"] and sw["t"][m] < sw["t_end"][m] and sw["steps"][m] < sw["max_steps"][m])
            out[m] = d
        started = [m for m in out if m in sw["unstarted"]]
        if started:  # written by the hand-off into the member's T0 row, which nothing overwrites afterwards
            rows = qu.T0[torch.tensor([sw["unstarted"].pop(m) for m in started], device=self.device)].cpu().numpy()
            for m, f in zip(started, rows):
                out[m]["start_T"] = f
        occupied = ck["slot_member"] >= 0
        who = ck["slot_member"][occupied]
        if not (np.array_equal(sw["steps"][who], ck["steps"][occupied]) and np.array_equal(sw["t"][who], ck["t"][occupied])):
            raise L.PbmcError("clock counters do not match the block that was run")
        clk.clock.view(torch.int64)[:, _DRAINED].copy_(torch.from_numpy(ck["snaps"].copy()))
        sw["next"] = ck["next"]
        self._host_active = ck["active"].copy()
        self._pending = None
        return out

    def _require_clock(self, sweep=True):
        if self._clk is None:
            raise RuntimeError("no clock: call start_clock() first")
        if not sweep and self._sweep is not None:
            raise RuntimeError("a sweep's per-member t_end and save_every are fixed by start_sweep()")

    def _begin_block(self, first_row, k):
        if self._clk is None:
            return
        if self._pending is not None:
            raise RuntimeError("drain() the previous block first: its per-step rows would be overwritten")
        self._pending = (first_row, k)
