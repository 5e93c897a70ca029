"""Slab-decomposed SURROGATE time step: one large grid, rows split over the ranks (SURVEY.md section 8e row 3, BASELINE
config 5 "stretch").  The reference has nothing like it -- its rollout is one device, batch 1
(advect_wi_gaia.py:422-425); what is decomposed here is exactly its per-step arithmetic:

    TS.forward body          pytorch_networks_convae.py:379-473   (input build -> stokes net -> un-scale -> ADNet -> BCs)
    NewFluidNet.forward      :1315-1388                            (conv0, pyramid of FluidLayers, conv[1..3], curl head)
    ADNet.forward            :522-568                              (advection-diffusion + ONE CFL dt for the whole grid)

Decomposition.  Rank r owns n = H / world contiguous rows of every full-resolution field (n divisible by 2^(levels-1), so
that every pyramid level splits at the same physical boundaries and 2x2 pooling never straddles two ranks) and n / 2^l rows of
level l.  Every local array carries G = 3 ghost rows per INTERNAL side (wall sides carry none): 1 for the 3x3 convolutions
and the curl, 3 for the bicubic up-sampling (taps floor(s)-1 .. floor(s)+2 of the coarse row s; with power-of-two ratios the
interpolation is translation invariant, so up-sampling the local array gives the global result on every row that is at
least 3 coarse rows away from an internal array end).  An operator is applied to the WHOLE local array with its ordinary
border handling: what it writes into the ghost rows is wrong by construction and is replaced by the neighbours' owned
rows in the exchange that follows every layer (the same contract as `multigpu.SlabStencil`).

What crosses ranks per forward (all tiny, latency bound; SURVEY.md 8e):
  * after every conv layer: G boundary rows each way (halo), and an all-reduce(SUM) of the layer's GroupNorm sums
    (2 x 4 doubles per sample) -- GroupNorm is a whole-image reduction (:788); the local sums are first corrected for the
    ghost rows (their locally computed values are subtracted before the exchange overwrites them);
  * once per forward: all-reduce(SUM) of conv[3]'s channel sums (zero-mean, :1343) and all-reduce(MAX) of max|u|,|v| (:556).
Everything else -- the kernels, the fused GroupNorm+GELU on load, incremental pooling -- is the single-GPU path's
operator set (`ops.*` over the C ABI), driven layer by layer from Python.  This is the FUNCTIONAL form of the row
(correct on any number of ranks, memory scales with 1/world); the collectives are `torch.distributed` calls, not yet
folded into the kernels like the stencil's (`pbmc_advect_diffuse_slab_sync`).
"""
from __future__ import annotations

import threading

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from . import ops
from .engine import pack_network
from .multigpu import cfl_dt  # noqa: F401  (re-exported for callers that want the host-side formula)

GHOST = 3


# ------------------------------------------------------------------------------------------------ communication layer
class DistComm:
    """torch.distributed (NCCL on the GPU box, gloo in the CPU tests)."""

    def __init__(self, group=None):
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def allreduce(self, t, op="sum"):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == "sum" else dist.ReduceOp.MAX, group=self.group)
        return t

    def exchange(self, send_up, send_down):
        """send_up / send_down: contiguous tensors for the neighbour towards row 0 / towards row H-1 (None at a wall).
        Returns (from_up, from_down)."""
        ops_, out = [], [None, None]
        if send_up is not None:
            out[0] = torch.empty_like(send_up)
            ops_ += [dist.P2POp(dist.isend, send_up, self.rank - 1, self.group), dist.P2POp(dist.irecv, out[0], self.rank - 1, self.group)]
        if send_down is not None:
            out[1] = torch.empty_like(send_down)
            ops_ += [dist.P2POp(dist.isend, send_down, self.rank + 1, self.group), dist.P2POp(dist.irecv, out[1], self.rank + 1, self.group)]
        if ops_:
            for w in dist.batch_isend_irecv(ops_):
                w.wait()
        return out[0], out[1]


class ThreadComm:
    """`world` ranks as threads of ONE process (single-GPU and CPU tests): a shared mailbox and a barrier.  On one GPU
    every rank enqueues on the same stream, so the copies below are ordered like real communication would be."""

    class Shared:
        def __init__(self, world):
            self.world, self.box, self.barrier = world, [None] * world, threading.Barrier(world)

    def __init__(self, shared, rank):
        self.s, self.rank, self.world = shared, rank, shared.world

    def allreduce(self, t, op="sum"):
        self.s.box[self.rank] = t.clone()
        self.s.barrier.wait()
        acc = self.s.box[0].clone()
        for r in range(1, self.world):
            acc = acc + self.s.box[r] if op == "sum" else torch.maximum(acc, self.s.box[r])
        self.s.barrier.wait()
        t.copy_(acc)
        return t

    def exchange(self, send_up, send_down):
        self.s.box[self.rank] = (None if send_up is None else send_up.clone(), None if send_down is None else send_down.clone())
        self.s.barrier.wait()
        from_up = self.s.box[self.rank - 1][1] if send_up is not None else None
        from_down = self.s.box[self.rank + 1][0] if send_down is not None else None
        self.s.barrier.wait()
        return from_up, from_down


# ------------------------------------------------------------------------------------------------ the decomposed step
class SlabSurrogate:
    """One rank's share of the surrogate time step on an H x W grid split into `comm.world` row slabs.

    net: a (non-learned, c_h = 16-style) NewFluidNet on `device`; x1d [W], y1d [H]: the separable grid's coordinates;
    params: (RaQ, gamma, beta).  State: `T` (local [1, rows, W] float32, ghost rows valid)."""

    def __init__(self, net, H, W, x1d, y1d, params, comm, device, cn_max=0.99):
        if net.r_p == "learned":
            raise NotImplementedError("SlabSurrogate covers zeros / replicate / reflect padding; a learned-boundary network "
                                      "(r_p='learned') runs on one GPU per grid (TS, EnsembleRollout)")
        self.net, self.comm, self.device = net, comm, torch.device(device)
        self.H, self.W, self.cn_max = H, W, float(cn_max)
        self.rank, self.world = comm.rank, comm.world
        Lv = net.levels
        if H % self.world or (H // self.world) % (1 << (Lv - 1)):
            raise ValueError(f"H = {H} must split into {self.world} slabs of a multiple of 2^(levels-1) = {1 << (Lv - 1)} rows")
        self.n = H // self.world
        if self.n >> (Lv - 1) < GHOST:
            raise ValueError("slabs too thin: the coarsest level needs at least 3 owned rows per rank")
        self.up, self.down = self.rank > 0, self.rank < self.world - 1
        self.gu, self.gd = GHOST * int(self.up), GHOST * int(self.down)
        self.lo, self.hi = self.rank * self.n, (self.rank + 1) * self.n
        self.pk = pack_network(net, self.device)
        self.pad = {"constant": "zeros"}.get(net.r_p, net.r_p)
        x = np.asarray(x1d, dtype=np.float64).copy()
        y = np.asarray(y1d, dtype=np.float64).copy()
        dev = self.device
        l0, l1 = self.lo - self.gu, self.hi + self.gd
        f32 = lambda a: torch.tensor(a, dtype=torch.float32, device=dev)
        self.xc = f32(np.broadcast_to(x[None, :], (l1 - l0, W)).copy())
        self.yc = f32(np.broadcast_to(y[l0:l1, None], (l1 - l0, W)).copy())
        xw, yw = x.copy(), y.copy()
        xw[0], xw[-1], yw[0], yw[-1] = 0.0, 4.0, 0.0, 1.0  # forced wall coordinates, :532-535
        self.dx_min = float((xw[1:-1] - xw[:-2]).min())  # :555 (x spacing only)
        self.xcoef = ops.stencil_coefs(torch.tensor(xw, dtype=torch.float64, device=dev), 0.0, 4.0)
        self.ycoef = ops.stencil_coefs(torch.tensor(yw, dtype=torch.float64, device=dev), 0.0, 1.0)[:, l0:l1].contiguous()
        self.members = ops.make_members([tuple(params)], dev)
        self.T = None
        self.time, self.n_steps = 0.0, 0

    # ---------------------------------------------------------------- helpers on local arrays (rows = dim -3 blocked / -2 plain)
    def rows_at(self, l):
        return (self.n >> l) + self.gu + self.gd

    def _owned(self, t, dim, l=0):
        return t.narrow(dim, self.gu, self.n >> l)

    def refresh_ghosts(self, t, dim, l=0):
        """Replace the ghost rows of a local array by the neighbours' owned boundary rows (in place)."""
        n = self.n >> l
        su = t.narrow(dim, self.gu, GHOST).contiguous() if self.up else None
        sd = t.narrow(dim, self.gu + n - GHOST, GHOST).contiguous() if self.down else None
        fu, fd = self.comm.exchange(su, sd)
        if self.up:
            t.narrow(dim, 0, GHOST).copy_(fu)
        if self.down:
            t.narrow(dim, self.gu + n, GHOST).copy_(fd)
        return t

    def _ghost_sums(self, yb, csum=False):
        """What the conv epilogue accumulated for the ghost rows of `yb` (they were computed locally, from padding):
        (sum, sum^2) per (sample, block), or per-channel sums."""
        parts = ([yb.narrow(2, 0, self.gu)] if self.up else []) + ([yb.narrow(2, yb.shape[2] - self.gd, self.gd)] if self.down else [])
        if not parts:
            return None
        g = torch.cat(parts, 2)
        return ops.chan_sums(g) if csum else ops.block_stats(g)

    def _layer(self, lay, sources, l, epi_act=L.ACT_NONE, want_stats=True, want_csum=False):
        """One conv layer on local arrays: conv over the whole local array, statistics restricted to the owned rows and
        all-reduced, ghost rows refreshed.  Returns (out blocked, global stats | None, global channel sums | None)."""
        yb, st, cs = ops.conv_fwd(sources, lay.wpk, lay.bias, lay.cout, lay.ksize, self.pad, epi_act=epi_act, want_stats=want_stats,
                                  want_chan_sum=want_csum, impl=self.net.conv_impl, wpk_umma=lay.wpk_umma, wpk_row=lay.wpk_row)
        if want_stats:
            g = self._ghost_sums(yb)
            if g is not None:
                st = st - g
            self.comm.allreduce(st, "sum")
        if want_csum:
            g = self._ghost_sums(yb, csum=True)
            if g is not None:
                cs = cs - g
            self.comm.allreduce(cs, "sum")
        self.refresh_ghosts(yb, 2, l)
        return yb, st, cs

    def _src(self, yb, st, lay, l):
        """A layer's output as the next operator's input: GroupNorm (GLOBAL statistics and count) + GELU fused on load."""
        s = ops.Source(yb, L.XFORM_GN_GELU, st, lay.gamma, lay.beta)
        s.inv_count = 1.0 / (4.0 * (self.H >> l) * (self.W >> l))
        return s

    # ---------------------------------------------------------------- NewFluidNet.forward on the slab (:1315-1388)
    def forward(self, inp_b):
        """inp_b: blocked local input [1, 2, rows, W, 4] (ghosts valid) -> (u, v, p local [1, rows, W], global max|u|,|v| bits)."""
        net, pk, H, W = self.net, self.pk, self.H, self.W
        Lv, R = net.levels, net.repeats
        y0, st0, _ = self._layer(pk.conv0, [ops.Source(inp_b)], 0)
        x_in = self._src(y0, st0, pk.conv0, 0)
        srcs, pooled_owned = [], None
        for l in range(Lv):
            if l == 0:
                cur = x_in
            else:
                # pool^l(x_in), incrementally and on OWNED rows only (slab boundaries are multiples of 2^l): :1321-1322
                prev = ops.Source(self._owned(x_in.t, 2, 0).contiguous(), x_in.xform, x_in.stats, x_in.gamma, x_in.beta) if l == 1 \
                    else ops.Source(pooled_owned)
                prev.inv_count = x_in.inv_count if l == 1 else 0.0
                pooled_owned = ops.avgpool2(prev)
                loc = pooled_owned.new_zeros(tuple(pooled_owned.shape[:2]) + (self.rows_at(l),) + tuple(pooled_owned.shape[3:]))
                self._owned(loc, 2, l).copy_(pooled_owned)
                cur = ops.Source(self.refresh_ghosts(loc, 2, l))
            for r in range(R):
                yb, st, _ = self._layer(pk.trunk[l][r], [cur], l)
                cur = self._src(yb, st, pk.trunk[l][r], l)
            if l == 0:
                srcs.append(cur)
            else:
                # bicubic up-sampling of the LOCAL array (exact away from internal array ends, see the module docstring),
                # then the fine rows [lo - G, hi + G) of it
                upl = ops.bicubic_up(cur, self.rows_at(l) << l, W)
                a = (self.gu << l) - self.gu
                srcs.append(ops.Source(upl.narrow(2, a, self.rows_at(0)).contiguous()))
        srcs.append(ops.Source(inp_b))
        y1, st1, _ = self._layer(pk.conv1, srcs, 0)
        y2, _, _ = self._layer(pk.conv2, [self._src(y1, st1, pk.conv1, 0)], 0, epi_act=L.ACT_GELU, want_stats=False)
        y3, _, cs = self._layer(pk.conv3, [ops.Source(y2)], 0, want_stats=False, want_csum=True)
        # the head kernel divides the channel sums by ITS (local) pixel count: rescale the global sums accordingly
        cs_local = (cs * (float(self.rows_at(0)) / float(H))).contiguous()
        u, v, p, uvmax = ops.head(y3, cs_local, self.members, net.a_bound, L.HEAD_CURL if net.loss_type == "curl" else L.HEAD_MAE,
                                  net.p_pred, want_uvmax=True)
        self.comm.allreduce(uvmax, "max")  # non-negative float bits order like integers
        return u, v, p, uvmax

    # ---------------------------------------------------------------- TS.forward body on the slab (:379-473)
    def set_T(self, T_full):
        """Every rank passes the whole [H, W] field (tests, small grids); the local slab with ghosts is kept."""
        T_full = torch.as_tensor(T_full)
        self.T = T_full[self.lo - self.gu:self.hi + self.gd].to(self.device, torch.float32).reshape(1, -1, self.W).contiguous().clone()

    def step(self):
        """One time step; returns dt (device double tensor [1]).  Leaves u, v, p (local) in self.u / self.v / self.p."""
        inp_b, _ = ops.build_input(self.T, self.xc, self.yc, self.yc, self.members)
        self.u, self.v, self.p, uvmax = self.forward(inp_b)
        dt = torch.zeros(1, dtype=torch.float64, device=self.device)
        T_new = torch.empty_like(self.T)
        if self.world == 1:
            ops.advect_diffuse(self.T, self.u, self.v, self.xcoef, self.ycoef, self.members, uvmax, self.dx_min, self.cn_max,
                               per_member_dt=False, T_out=T_new, dt_out=dt)
        else:
            T_new.copy_(self.T)  # the kernel never writes the array's first / last row where that is a ghost row
            ops.advect_diffuse_slab(self.T, self.u, self.v, self.xcoef, self.ycoef, self.members, uvmax, self.dx_min, self.cn_max,
                                    T_new, dt, self.up, self.down)
            self.refresh_ghosts(T_new, 1)
        self.T = T_new
        self.n_steps += 1
        return dt

    def gather(self, t, dim=1):
        """Whole-grid field on every rank from a local array (owned rows of all ranks, in rank order)."""
        own = self._owned(t, dim).contiguous()
        if self.world == 1:
            return own
        if isinstance(self.comm, DistComm):
            bufs = [torch.empty_like(own) for _ in range(self.world)]
            dist.all_gather(bufs, own, group=self.comm.group)
            return torch.cat(bufs, dim)
        s = self.comm.s
        s.box[self.rank] = own.clone()
        s.barrier.wait()
        out = torch.cat(list(s.box), dim)
        s.barrier.wait()
        return out
