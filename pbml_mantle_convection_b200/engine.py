"""Host-side runtime for the surrogate: weight repacking, the `pbmc_net` descriptor, workspace
and stream-context ownership, and CUDA-graph capture of whole time steps.

Mirrors what the reference does implicitly through ATen (`NewFluidNet.forward`,
pytorch_networks_convae.py:1315-1388; `TS.forward`, :354-475) but with all device work
enqueued by two C calls (`pbmc_surrogate_forward`, `pbmc_rollout`).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from . import ops


class _PackedLayer:
    def __init__(self, w_full, bias, gamma, beta, src_channels, dev, w_edge=None):
        cout, _, k, _ = w_full.shape
        self.wpk = ops.pack_conv_weight(w_full.to(dev), src_channels)
        self.bias = ops.pad_vec(bias, cout, dev)
        self.gamma = ops.pad_vec(gamma, cout, dev, 1.0) if gamma is not None else None
        self.beta = ops.pad_vec(beta, cout, dev, 0.0) if beta is not None else None
        self.cin_blks = sum(ops.nblk(c) for c in src_channels)
        self.cout, self.ksize = cout, k
        self.wpk_umma = (ops.pack_conv_weight_umma(w_full.to(dev), src_channels)
                         if ops.umma_supported(cout, src_channels) else None)
        self.wpk_row = (ops.pack_conv_weight_row(w_full.to(dev), src_channels)
                        if ops.row_supported(cout, k, src_channels) else None)
        # learned 9-region conv: w_full is the interior filter bank, w_edge the eight edge / corner banks
        self.wedge = ops.pack_edge9_weights([w.to(dev) for w in w_edge], src_channels) if w_edge is not None else None

    def c(self):
        s = L.Layer()
        s.wpk, s.wpk_umma, s.bias = L.ptr(self.wpk), L.ptr(self.wpk_umma), L.ptr(self.bias)
        s.wpk_row = L.ptr(self.wpk_row)
        s.gamma, s.beta = L.ptr(self.gamma), L.ptr(self.beta)
        s.cin_blks, s.cout, s.ksize = self.cin_blks, self.cout, self.ksize
        return s


class PackedNetwork:
    """Repacked filters / bias / GroupNorm affine of every layer of a NewFluidNet: conv0, trunk[l][r], conv1, conv2, conv3
    as `_PackedLayer`s (learned-boundary nets: interior filters, edge filter image `wedge` and learnable bias).  Needs no
    library context: the fused engine and the slab-decomposed surrogate both start from it."""


def pack_network(m, dev) -> PackedNetwork:
    from .symmetric_layers_torch import _check_conv_supported, full_weight

    f32 = lambda t: None if t is None else t.detach().to(dev, torch.float32)

    def learned(conv, gamma, beta, src_channels):
        # BoundaryLearnedConvolution2D: regions in conv._REGIONS order = interior, then ops.EDGE9_REGIONS
        wf = [f32(full_weight(getattr(conv, name))) for name in conv._REGIONS]
        return _PackedLayer(wf[0], f32(conv.learnable_bias).reshape(-1), gamma, beta, src_channels, dev, wf[1:])

    def fluid(fl, cin):
        conv, gn = fl.layers[0], fl.layers[1]
        if m.r_p == "learned":
            return learned(conv, f32(gn.weight), f32(gn.bias), [cin])
        _check_conv_supported(conv)  # dilation / stride / groups != 1 would silently compute another operator
        w = f32(conv.weight)
        if getattr(conv, "symmetry", None) is not None:
            w = ops.expand_symmetric(w, conv.out_channels)
        return _PackedLayer(w, f32(conv.bias), f32(gn.weight), f32(gn.bias), [cin], dev)

    pk = PackedNetwork()
    pk.conv0 = fluid(m.conv[0], m.c_i)
    pk.trunk = [[fluid(m.convs[l][r], m.c_h) for r in range(m.repeats)] for l in range(m.levels)]
    c1, c2, c3 = m.conv[1], m.conv[2], m.conv[3]
    if m.r_p == "learned":
        pk.conv1 = learned(c1, f32(m.gn[0].weight), f32(m.gn[0].bias), [m.c_h] * m.levels + [m.c_i])
        pk.conv2 = learned(c2, None, None, [m.c_h])
        pk.conv3 = learned(c3, None, None, [m.c_h])
        return pk
    for c in (c1, c2, c3):
        _check_conv_supported(c)
    pk.conv1 = _PackedLayer(f32(c1.weight), f32(c1.bias), f32(m.gn[0].weight), f32(m.gn[0].bias),
                            [m.c_h] * m.levels + [m.c_i], dev)
    pk.conv2 = _PackedLayer(f32(c2.weight), f32(c2.bias), None, None, [m.c_h], dev)
    pk.conv3 = _PackedLayer(f32(c3.weight), f32(c3.bias), None, None, [m.c_h], dev)
    return pk


def shape_desc(m):
    """pbmc_net of `m` with its shape fields and flags only (no weights): enough for the host-side queries
    (pbmc_workspace_bytes, pbmc_trunk_cta_budgets), no device needed."""
    n = L.Net()
    n.levels, n.repeats, n.c_i, n.c_h, n.c_o = m.levels, m.repeats, m.c_i, m.c_h, m.c_o
    learned = m.r_p == "learned"
    n.ksize = m.conv[0].layers[0].k if learned else m.conv[0].layers[0].kernel_size[0]
    n.pad_mode = 0 if learned else L.PAD[m.r_p]  # learned: not used (the interior convs run with zeros padding)
    n.flags = L.NET_LEARNED if learned else 0
    return n


def fused_supported(m, B, H, W) -> bool:
    """Whether the fused engine (pbmc_surrogate_forward / pbmc_rollout) takes network `m` at this size."""
    return L.load().pbmc_workspace_bytes(C.byref(shape_desc(m)), B, H, W) > 0


class SurrogateEngine:
    """Owns everything device-side that belongs to ONE network instance on ONE device."""

    def __init__(self, net, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.PbmcError("the surrogate runs on CUDA only (no CPU fallback)")
        L.load()
        self.net_module = net
        self._key = None
        self._ctx = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(L.load().pbmc_ctx_create(C.byref(self._ctx)), "pbmc_ctx_create")
        self._ws = {}
        self.conv_impl = "auto"
        self.trunk_mode = "auto"  # "auto": persistent per-level trunk kernel where it fits; "per_layer": one launch per layer
        self.up_staged = False    # True: up-sampled levels written as conv[1]'s operand image, staged by TMA bulk copies
        self.refresh()

    def __del__(self):
        try:
            if self._ctx:
                L.load().pbmc_ctx_destroy(self._ctx)
        except Exception:
            pass

    # -------------------------------------------------------------- weights
    def _weights_key(self):
        """Identity + version of every parameter tensor.  Called on every forward, so it walks a cached list of
        the (sub)modules' parameter dicts instead of Module.parameters() (0.1 ms of Python per call for the 108
        tensors of the primary net); assigning a NEW Parameter object to a submodule is still seen, replacing a
        submodule after construction is not (call refresh(force=True))."""
        dicts = self.__dict__.get("_param_dicts")
        if dicts is None:
            dicts = self._param_dicts = [m._parameters for m in self.net_module.modules() if m._parameters]
        return tuple((p.data_ptr(), p._version) for d in dicts for p in d.values() if p is not None)

    def refresh(self, force=False):
        """(Re)pack weights if any parameter changed (load_state_dict, .double(), .to())."""
        if force:
            self.__dict__.pop("_param_dicts", None)
        key = self._weights_key()
        if not force and key == self._key:
            return
        pk = pack_network(self.net_module, self.device)
        self.conv0, self.trunk, self.conv1, self.conv2, self.conv3 = pk.conv0, pk.trunk, pk.conv1, pk.conv2, pk.conv3
        self._key = key
        self._build_desc()

    def _build_desc(self):
        m = self.net_module
        n = shape_desc(m)
        n.ksize = self.conv0.ksize
        n.head_kind = L.HEAD_CURL if m.loss_type == "curl" else L.HEAD_MAE
        n.p_pred = int(bool(m.p_pred))
        n.conv_impl = L.CONV_IMPL[self.conv_impl]
        n.flags |= L.TRUNK_MODE[self.trunk_mode] | (L.NET_UP_STAGED if self.up_staged else 0)
        n.a_bound = float(m.a_bound)
        n.conv0 = self.conv0.c()
        for l in range(m.levels):
            for r in range(m.repeats):
                n.trunk[l * L.MAX_REPEATS + r] = self.trunk[l][r].c()
        n.conv1, n.conv2, n.conv3 = self.conv1.c(), self.conv2.c(), self.conv3.c()
        if m.r_p == "learned":
            n.wedge_conv0 = L.ptr(self.conv0.wedge)
            for l in range(m.levels):
                for r in range(m.repeats):
                    n.wedge_trunk[l * L.MAX_REPEATS + r] = L.ptr(self.trunk[l][r].wedge)
            n.wedge_conv1, n.wedge_conv2, n.wedge_conv3 = (L.ptr(x.wedge) for x in (self.conv1, self.conv2, self.conv3))
        self.desc = n

    def set_conv_impl(self, impl):
        if impl not in L.CONV_IMPL:
            raise ValueError(impl)
        self.conv_impl = impl
        self._build_desc()

    def set_trunk_mode(self, mode, up_staged=None):
        if mode not in L.TRUNK_MODE:
            raise ValueError(mode)
        self.trunk_mode = mode
        if up_staged is not None:
            self.up_staged = bool(up_staged)
        self._build_desc()

    # -------------------------------------------------------------- workspace
    def workspace(self, B, H, W):
        """One workspace per (B, H, W), kept for the life of the engine: captured CUDA graphs (TS plans, ensemble graphs)
        hold its raw address, so a buffer is never freed or replaced while the engine lives.  `release_workspaces()` is
        the explicit way to give the memory back (every graph captured on this engine must be dropped first)."""
        k = (B, H, W)
        ws = self._ws.get(k)
        if ws is None:
            nbytes = L.load().pbmc_workspace_bytes(C.byref(self.desc), B, H, W)
            if nbytes == 0:
                raise L.PbmcError(f"unsupported network/grid configuration for the fused engine: B={B} H={H} W={W}")
            ws = self._ws[k] = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return ws

    def release_workspaces(self):
        self._ws = {}

    def graph_key(self, B, H, W, refresh=True):
        """Everything a captured graph of this engine bakes in besides its own buffers: packed-weight identity, conv
        implementation, workspace address.  A change in any of them must force a re-capture.  refresh=False: the caller
        has just called refresh() (the parameter walk costs ~30 us for the primary network's 108 tensors)."""
        if refresh:
            self.refresh()
        return (self._key, self.conv_impl, self.trunk_mode, self.up_staged, self.workspace(B, H, W).data_ptr())

    # -------------------------------------------------------------- forward
    def forward_blocked(self, inp_blocked, members=None, want_uvmax=False):
        """inp_blocked [B, ceil(c_i/4), H, W, 4] -> (u, v, p|None, uvmax|None), plain [B,H,W] float32."""
        self.refresh()
        m = self.net_module
        B, _, H, W, _ = inp_blocked.shape
        ws = self.workspace(B, H, W)
        dev = self.device
        u = torch.empty(B, H, W, dtype=torch.float32, device=dev)
        v = torch.empty_like(u)
        p = torch.empty_like(u) if m.p_pred else None
        uvmax = torch.zeros(B, dtype=torch.int32, device=dev) if want_uvmax else None
        L.check(L.load().pbmc_surrogate_forward(self._ctx, C.byref(self.desc), L.ptr(inp_blocked), L.ptr(members), L.ptr(u),
                                                L.ptr(v), L.ptr(p), L.ptr(uvmax), L.ptr(ws), ws.numel(), B, H, W,
                                                L.stream_ptr(dev)), "pbmc_surrogate_forward")
        return u, v, p, uvmax

    def rollout(self, state, first_step, n_steps, clock=None, queue=None, diag=None, chain=None):
        """Enqueue n_steps time steps on `state` (a RolloutState).  No host sync.  clock: a rollout.MemberClocks (the
        per-member run-to-time clock, pbmc_rollout_clocked) or None (pbmc_rollout); queue (with a clock only): a
        rollout.SweepQueue whose members refill the slots that stop (pbmc_rollout_queued); diag (with a clock only): a
        rollout.MemberDiagnostics, per-step wall fluxes / rms velocity and the steady stop (pbmc_rollout_diagnosed);
        chain (with a queue only): a _lib.MemberChain whose members continue from their predecessors
        (pbmc_rollout_chained)."""
        self.refresh()
        s = state
        ws = self.workspace(s.B, s.H, s.W)
        args = (self._ctx, C.byref(self.desc), L.ptr(s.members), L.ptr(s.xc), L.ptr(s.yc), L.ptr(s.ycc), L.ptr(s.xcoef),
                L.ptr(s.ycoef), float(s.dx_min), float(s.cn_max), int(s.per_member_dt), L.ptr(s.T_seq), s.nslots,
                int(first_step), int(n_steps), L.ptr(s.dt_seq), int(s.dt_seq.shape[0]), L.ptr(s.u), L.ptr(s.v), L.ptr(s.p),
                L.ptr(s.V), L.ptr(ws), ws.numel(), s.B, s.H, s.W)
        if clock is None:
            if diag is not None:
                raise ValueError("diagnostics need a clock")
            L.check(L.load().pbmc_rollout(*args, L.stream_ptr(self.device)), "pbmc_rollout")
            return
        clk = (L.ptr(clock.clock), L.ptr(clock.meanT_seq), L.ptr(clock.ring), L.ptr(clock.meta), int(clock.slots))
        if chain is not None:
            L.check(L.load().pbmc_rollout_chained(*args, *clk, C.byref(queue.desc),
                                                  C.byref(diag.desc) if diag is not None else None, C.byref(chain),
                                                  L.stream_ptr(self.device)), "pbmc_rollout_chained")
        elif diag is not None:
            L.check(L.load().pbmc_rollout_diagnosed(*args, *clk, C.byref(queue.desc) if queue is not None else None,
                                                    C.byref(diag.desc), L.stream_ptr(self.device)), "pbmc_rollout_diagnosed")
        elif queue is not None:
            L.check(L.load().pbmc_rollout_queued(*args, *clk, C.byref(queue.desc), L.stream_ptr(self.device)),
                    "pbmc_rollout_queued")
        else:
            L.check(L.load().pbmc_rollout_clocked(*args, *clk, L.stream_ptr(self.device)), "pbmc_rollout_clocked")


class Grid:
    """Device copies of the cell-centre coordinates + what the stencil needs from them."""

    def __init__(self, xc, yc, ycc, device):
        xc64 = xc.detach().to("cpu", torch.float64).reshape(xc.shape[-2], xc.shape[-1])
        yc64 = yc.detach().to("cpu", torch.float64).reshape(yc.shape[-2], yc.shape[-1])
        ycc64 = ycc.detach().to("cpu", torch.float64).reshape(ycc.shape[-2], ycc.shape[-1])
        self.H, self.W = xc64.shape
        self.xc = xc64.float().to(device).contiguous()
        self.yc = yc64.float().to(device).contiguous()
        self.ycc = self.yc if ycc is yc else ycc64.float().to(device).contiguous()
        # separable?  (x depends on the column only, y on the row only) -- checked once, on the host
        self.separable = bool((xc64 == xc64[0:1, :]).all() and (yc64 == yc64[:, 0:1]).all())
        xf = xc64.clone()
        xf[:, 0], xf[:, -1] = 0.0, 4.0  # ADNet forces the wall coordinates, pytorch_networks_convae.py:532-533
        dx_l = xf[1:-1, 1:-1] - xf[1:-1, :-2]
        self.dx_min = float(dx_l.min())  # :555
        self.xc64 = xc64.to(device).contiguous()  # float64 fields for the general (non-separable) stencil
        self.yc64 = yc64.to(device).contiguous()
        self.y1d64 = yc64[:, 0].clone()
        self.y1d64[0], self.y1d64[-1] = 0.0, 1.0
        self.xcoef = ops.stencil_coefs(xc64[0, :].to(device), 0.0, 4.0)  # [3, W] inverse spacings (:532-545)
        self.ycoef = ops.stencil_coefs(yc64[:, 0].to(device), 0.0, 1.0)  # [3, H]
        self.dx_min_dev = torch.tensor([self.dx_min], dtype=torch.float64, device=device)


class RolloutState:
    """Device-resident state of B independent (or batch-coupled) rollouts."""

    def __init__(self, grid: Grid, members: torch.Tensor, B, nslots, max_steps, cn_max, per_member_dt, p_pred, device):
        self.B, self.H, self.W = B, grid.H, grid.W
        self.xc, self.yc, self.ycc, self.dx_min = grid.xc, grid.yc, grid.ycc, grid.dx_min
        self.xcoef, self.ycoef = grid.xcoef, grid.ycoef
        self.members = members
        self.nslots = nslots
        self.cn_max, self.per_member_dt = cn_max, per_member_dt
        f = lambda: torch.empty(B, self.H, self.W, dtype=torch.float32, device=device)
        self.T_seq = torch.empty(nslots, B, self.H, self.W, dtype=torch.float32, device=device)
        # step i writes row i - 1; a chunk may start at first_step = 2 (odd slot parity): max_steps + 1 rows
        self.dt_seq = torch.zeros(max(max_steps, 1) + 1, B, dtype=torch.float64, device=device)
        self.u, self.v, self.V = f(), f(), f()
        self.p = f() if p_pred else None
