"""Drop-in modules for the surrogate time-stepping path (reference: pytorch_networks_convae.py).

Same class names, constructor signatures, `state_dict` layout and call signatures as the
reference's `FluidLayer` (:702-799), `BoundaryLearnedConvolution2D` (:802-1065),
`NewFluidNet` (:1068-1388), `FluidNet` (:1392-1697), `ADNet` (:478-568) and `TS` (:266-475);
the `forward` bodies enqueue hand-written sm_100a kernels through the C ABI (libpbmc.so).

Differences a user can observe:
  * CUDA only.  A CPU tensor / missing library raises -- there is no fallback path.
  * Arithmetic is float32 (tensor-core variants selectable per network); inputs of any float
    dtype are accepted and outputs come back in the input dtype, so `.double()` models and
    float64 state (advect_wi_gaia.py:348,430,468) keep working.
  * The grid size is taken from the input; the reference's hard-coded 128x506
    (:414-417, :1222-1229) is not inherited.
  * Inference only (the rollout runs under torch.no_grad(), advect_wi_gaia.py:589).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib as L
from . import ops
from .engine import Grid, RolloutState, SurrogateEngine, fused_supported
from .symmetric_layers_torch import SymmetricConv2d, conv_module_forward, full_weight

_ACTS = {"selu": nn.SELU, "tanh": nn.Tanh, "elu": nn.ELU, "silu": nn.SiLU, "relu": nn.ReLU, "gelu": nn.GELU}


def count_parameters(model):
    """pytorch_networks_convae.py:105-115."""
    return sum(p.numel() for p in model.parameters() if p.requires_grad)


def _make_act(act_fn):
    if act_fn == "sine":
        raise NotImplementedError("act_fn='sine' is not part of the rollout path")
    return _ACTS[act_fn]()


def _sym_counts(c_o):
    # pytorch_networks_convae.py:755-757
    return {"h": int(c_o / 4) if c_o > 4 else int(c_o / 2), "v": 0, "hv": 0}


def _require_cuda_device(dev):
    if dev.type != "cuda":
        raise L.PbmcError("TS runs on CUDA only: there is no CPU implementation of this path")


def _require_gelu(mod):
    if not isinstance(mod.act, nn.GELU):
        raise NotImplementedError("the B200 path fuses exact-erf GELU (act_fn='gelu', advect_wi_gaia.py:247); "
                                  f"{type(mod.act).__name__} is not implemented")


class BoundaryLearnedConvolution2D(nn.Module):
    """Nine bias-free 'valid' convolutions (interior, 4 edges, 4 corners) stitched together
    plus a learnable bias (reference :802-1065).  NB the reference places the strip computed
    from the LAST input rows at output row 0 (`cat([bottom, x, top], dim=2)`, :1060)."""

    _REGIONS = ("conv", "conv_top_left", "conv_top_right", "conv_bottom_left", "conv_bottom_right", "conv_top",
                "conv_bottom", "conv_left", "conv_right")

    def __init__(self, c_i, c_o, k, stride=1, use_symm=False):
        super().__init__()
        self.c_i, self.c_o, self.k = c_i, c_o, k
        for name in self._REGIONS:
            if use_symm:
                conv = SymmetricConv2d(c_i, c_o, k, bias=False, padding="valid", symmetry=_sym_counts(c_o))
            else:
                conv = nn.Conv2d(in_channels=c_i, out_channels=c_o, kernel_size=k, padding="valid", bias=False)
            setattr(self, name, conv)
        self.learnable_bias = nn.Parameter(torch.zeros(1, c_o, 1, 1))

    # ---- kernel path (bc_x = bc_y = 1, c_o <= 16): two launches over blocked sources, see include/pbmc.h (A4)
    def _packed(self, src_channels, dev):
        """Interior filters as the conv kernels' images, the eight boundary filter sets as the edge kernel's image, the
        learnable bias -- cached on the module, rebuilt when any parameter changes (in place or by re-assignment)."""
        ws = [getattr(self, n).weight for n in self._REGIONS]
        key = (tuple((w.data_ptr(), w._version) for w in ws), self.learnable_bias.data_ptr(), self.learnable_bias._version,
               tuple(src_channels), str(dev))
        c = self.__dict__.get("_pbmc_pack9")
        if c is None or c["key"] != key:
            wf = [full_weight(getattr(self, n)).detach().to(dev, torch.float32) for n in self._REGIONS]
            c = {"key": key, "wpk": ops.pack_conv_weight(wf[0], list(src_channels)),
                 "row": ops.pack_conv_weight_row(wf[0], list(src_channels)) if ops.row_supported(self.c_o, self.k, list(src_channels)) else None,
                 "wedge": ops.pack_edge9_weights(wf[1:], list(src_channels)),
                 "bias": ops.pad_vec(self.learnable_bias.detach().reshape(-1), self.c_o, dev)}
            self.__dict__["_pbmc_pack9"] = c  # plain attribute: not a parameter, not a buffer, not in the state_dict
        return c

    def kernel_path_ok(self, H, W, src_channels, bc_x=1, bc_y=1):
        pad = self.k + 1 if self.k == 5 else self.k
        return (bc_x == 1 and bc_y == 1 and self.c_o <= 16 and self.k in (3, 5) and H >= pad and W >= pad
                and all(c <= 128 for c in src_channels) and len(src_channels) <= L.MAX_SRC)

    def forward_blocked(self, sources, src_channels, epi_act=L.ACT_NONE, want_stats=True, want_chan_sum=False):
        """sources: ops.Source list (concat order, producer transforms fused) -> (out blocked, stats, chan_sum)."""
        pk = self._packed(src_channels, sources[0].t.device)
        return ops.conv_learned9(sources, pk["wpk"], pk["row"], pk["wedge"], pk["bias"], self.c_o, self.k, epi_act=epi_act,
                                 want_stats=want_stats, want_chan_sum=want_chan_sum)

    def forward(self, x, bc_x=1, bc_y=1):
        if x.is_cuda and self.kernel_path_ok(x.shape[-2], x.shape[-1], [self.c_i], bc_x, bc_y):
            yb, _, _ = self.forward_blocked([ops.Source(ops.pack_nchw(x))], [self.c_i], want_stats=False)
            return ops.unpack_nchw(yb, self.c_o).to(x.dtype)
        k = self.k
        pad_x = k + 1 + (bc_x - 1) if k == 5 else k + (bc_x - 1)
        pad_y = k + 1 + (bc_y - 1) if k == 5 else k + (bc_y - 1)
        run = lambda name, t: conv_module_forward(getattr(self, name), t.contiguous())
        first_r, last_r = x[:, :, :pad_y], x[:, :, -pad_y:]
        from_first = torch.cat([run("conv_top_left", first_r[..., :pad_x]), run("conv_top", first_r),
                                run("conv_top_right", first_r[..., -pad_x:])], 3)
        from_last = torch.cat([run("conv_bottom_left", last_r[..., :pad_x]), run("conv_bottom", last_r),
                               run("conv_bottom_right", last_r[..., -pad_x:])], 3)
        mid = torch.cat([run("conv_left", x[..., :pad_x]), run("conv", x), run("conv_right", x[..., -pad_x:])], 3)
        out = torch.cat([from_last, mid, from_first], 2)  # row order as in the reference (:1060)
        return out + self.learnable_bias.detach().to(out.dtype)


class FluidLayer(nn.Module):
    """conv -> GroupNorm(4 channels per group) -> activation -> Dropout (reference :702-799)."""

    def __init__(self, c_i: int, c_o: int, act_fn: str = "selu", r_p="zeros", use_symm=False, dilation=1, f=3,
                 drop_rate=0.0):
        super().__init__()
        self.layers = nn.ModuleList()
        self.r_p = "constant" if r_p == "zeros" else r_p
        self.act = _make_act(act_fn)
        self.dropout = torch.nn.Dropout(drop_rate)
        if r_p == "learned":
            self.layers.append(BoundaryLearnedConvolution2D(c_i, c_o, k=f, use_symm=use_symm))
        elif use_symm:
            self.layers.append(SymmetricConv2d(c_i, c_o, kernel_size=f, padding="same", dilation=dilation,
                                               padding_mode=r_p, symmetry=_sym_counts(c_o)))
        else:
            self.layers.append(nn.Conv2d(c_i, c_o, kernel_size=f, padding="same", dilation=dilation, padding_mode=r_p))
        self.layers.append(torch.nn.GroupNorm(int(c_o / min(4, c_o)), c_o))

    def forward(self, inputs, bc_x=1, bc_y=1):
        _require_gelu(self)
        if self.dropout.p != 0.0 and self.training:
            raise NotImplementedError("dropout>0 in training mode is outside the inference path")
        conv, gn = self.layers[0], self.layers[1]
        c_o = gn.num_channels
        if c_o > 4 and c_o % 4 != 0:
            raise NotImplementedError("GroupNorm groups must coincide with 4-channel blocks (c_o % 4 == 0)")
        dev = inputs.device
        if self.r_p == "learned" and inputs.is_cuda and conv.kernel_path_ok(inputs.shape[-2], inputs.shape[-1], [conv.c_i], bc_x, bc_y):
            yb, stats, _ = conv.forward_blocked([ops.Source(ops.pack_nchw(inputs))], [conv.c_i])
        elif self.r_p == "learned":
            y = conv(inputs, bc_x=bc_x, bc_y=bc_y)
            yb = ops.pack_nchw(y)
            # statistics of the stitched tensor: one more pass through the conv-free reduction
            stats = _stats_of_blocked(yb, c_o)
        else:
            from .symmetric_layers_torch import _check_conv_supported
            _check_conv_supported(conv)
            k = conv.kernel_size[0]
            w = full_weight(conv).detach().to(dev, torch.float32)
            wpk = ops.pack_conv_weight(w, [conv.in_channels])
            bias = ops.pad_vec(conv.bias, c_o, dev)
            yb, stats, _ = ops.conv_fwd([ops.Source(ops.pack_nchw(inputs))], wpk, bias, c_o, k, conv.padding_mode,
                                        want_stats=True, impl="ffma")
        src = ops.Source(yb, L.XFORM_GN_GELU, stats, ops.pad_vec(gn.weight, c_o, dev, 1.0), ops.pad_vec(gn.bias, c_o, dev),
                         channels_per_group=min(4, c_o))
        return ops.finalize_nchw(src, c_o).to(inputs.dtype)


def _stats_of_blocked(yb, c_o):
    """(sum, sum^2) per (sample, 4-channel block) of a blocked tensor, float64 (host-side helper
    for the stitched learned-boundary output; tiny reduction, stays on the device)."""
    y64 = yb.double()
    return torch.stack([y64.sum(dim=(2, 3, 4)), (y64 * y64).sum(dim=(2, 3, 4))], -1).contiguous()


class _FluidNetBase(nn.Module):
    """Shared constructor of NewFluidNet / FluidNet (reference :1123-1313 / :1447-1637)."""

    _HEAD_PADDING_CURL = (1, 1)

    def __init__(self, levels: int, c_i: int, c_h: int, c_o: int, device, act_fn: str = "selu", r_p="zeros",
                 loss_type="mae", use_symm=False, dilation=1, a_bound=4.0, use_cosine=False, repeats=3, use_skip=False,
                 f=3, p_pred=True, spectral_conv=False, blurr=False, drop_rate=0.0, factor=2):
        super().__init__()
        if spectral_conv:
            raise NotImplementedError("spectral_conv=True is outside the rollout path (advect_wi_gaia.py:253)")
        if blurr:
            raise NotImplementedError("blurr=True is outside the rollout path (advect_wi_gaia.py:255)")
        if factor != 2:
            raise NotImplementedError("pooling factor 2 is the only one used (advect_wi_gaia.py:307)")
        self.conv = nn.ModuleList()
        self.gn = nn.ModuleList()
        self.unpool = nn.ModuleList()
        self.levels, self.loss_type, self.a_bound = levels, loss_type, a_bound
        self.use_cosine, self.repeats, self.use_skip, self.p_pred = use_cosine, repeats, use_skip, p_pred
        self.c_h, self.c_i, self.c_o = c_h, c_i, c_o
        self.blurrer = None
        self.r_p = "constant" if r_p == "zeros" else r_p
        self.act = _make_act(act_fn)
        self.conv.append(FluidLayer(c_i, c_h, act_fn, r_p, use_symm, dilation, f=f, drop_rate=drop_rate))
        self.pool = nn.AvgPool2d((factor, factor), stride=factor)
        for _ in range(1, levels):
            # kept for structural parity; the kernels up-sample to the INPUT's size, whatever it is
            self.unpool.append(nn.Upsample(size=(128, 506), mode="bicubic"))
        self.convs = nn.ModuleList()
        for _l in range(levels):
            self.convs.append(nn.ModuleList(
                [FluidLayer(c_h, c_h, act_fn, r_p, use_symm, dilation, f=f, drop_rate=drop_rate) for _ in range(repeats)]))
        head_pad = self._HEAD_PADDING_CURL if loss_type == "curl" else (1, 1)
        if self.r_p != "learned":
            self.conv.append(nn.Conv2d(c_h * levels + c_i, c_h, kernel_size=3, padding=head_pad, dilation=dilation,
                                       padding_mode=r_p, stride=1))
        else:
            self.conv.append(BoundaryLearnedConvolution2D(c_h * levels + c_i, c_h, k=f, use_symm=use_symm))
        self.gn.append(torch.nn.GroupNorm(int(c_h / 4), c_h))
        for co in (c_h, c_o):
            if self.r_p != "learned":
                self.conv.append(nn.Conv2d(c_h, co, kernel_size=3, padding=(1, 1), dilation=1, padding_mode=r_p, stride=1))
            else:
                self.conv.append(BoundaryLearnedConvolution2D(c_h, co, k=f, use_symm=use_symm))
        self._engines = {}
        self.conv_impl = "auto"  # "auto" | "ffma" | "umma_3xtf32" | "umma_bf16"
        self.trunk_mode = "auto"  # "auto": one persistent launch per pyramid level where it fits | "per_layer"
        self.up_staged = False    # True: conv[1] stages the up-sampled levels with TMA bulk copies (see include/pbmc.h)
        self.use_cuda_graph = True  # learned-boundary networks: replay the module-level forward as one CUDA graph

    # nn.Module bookkeeping: engines hold device buffers, never parameters
    def _engine(self, device) -> SurrogateEngine:
        key = str(device)
        eng = self._engines.get(key)
        if eng is None:
            eng = self._engines[key] = SurrogateEngine(self, device)
        if eng.conv_impl != self.conv_impl:
            eng.set_conv_impl(self.conv_impl)
        if eng.trunk_mode != self.trunk_mode or eng.up_staged != bool(self.up_staged):
            eng.set_trunk_mode(self.trunk_mode, self.up_staged)
        return eng

    def __getstate__(self):  # engines are not picklable / deep-copyable
        d = dict(self.__dict__)
        d["_engines"] = {}
        d.pop("_learned_plan", None)
        return d

    def _r_p_name(self):
        return "zeros" if self.r_p == "constant" else self.r_p

    def _check_fused(self, inputs):
        _require_gelu(self)
        if not inputs.is_cuda:
            raise L.PbmcError("NewFluidNet/FluidNet run on CUDA only: there is no CPU implementation of this path")
        if inputs.dim() != 4 or inputs.shape[1] != self.c_i:
            raise ValueError(f"expected inputs [B,{self.c_i},H,W], got {tuple(inputs.shape)}")
        if self.training and any(m.dropout.p != 0.0 for m in self.modules() if isinstance(m, FluidLayer)):
            raise NotImplementedError("dropout>0 in training mode is outside the inference path")


class NewFluidNet(_FluidNetBase):
    """Multi-level conv surrogate T-features -> (u, v, p) (reference :1068-1388)."""

    def forward(self, inputs):
        self._check_fused(inputs)
        if self.r_p == "learned":
            return _forward_learned_replayed(self, inputs, head_bc=1, wall_bcs=True)
        eng = self._engine(inputs.device)
        eng.net_module = self
        u, v, p, _ = eng.forward_blocked(ops.pack_nchw(inputs))
        return _shape_outputs(self, u, v, p, inputs.dtype)


def _shape_outputs(net, u, v, p, dtype):
    u, v = u.to(dtype), v.to(dtype)
    if p is not None:
        p = p.to(dtype)
        if net.loss_type != "curl":
            p = p[:, None]  # reference returns y[:, 2:3] for the mae head (:1349)
    return u, v, p


class FluidNet(_FluidNetBase):
    """Variant whose head conv enlarges the field by one ring and which returns the raw curl
    without wall BCs (reference :1392-1697).  Like the reference it only runs with
    r_p='learned' and loss_type='curl' (:1659-1661)."""

    _HEAD_PADDING_CURL = (2, 2)

    def forward(self, inputs):
        self._check_fused(inputs)
        if self.r_p != "learned" or self.loss_type != "curl":
            raise TypeError("FluidNet.forward needs r_p='learned' and loss_type='curl' (the reference skips conv[1] "
                            "otherwise and fails, pytorch_networks_convae.py:1659-1661)")
        return _forward_learned_replayed(self, inputs, head_bc=2, wall_bcs=False)


class _LearnedPlan:
    """Captured CUDA graph of one (input shape, dtype, parameters) configuration of a learned-boundary network."""


def _forward_learned_replayed(net, inputs, head_bc, wall_bcs):
    """The module-level forward of a learned-boundary network is ~1000 small launches (9 region convs + stitching per
    layer): 26 ms of host time per call for the paper's network at 128x506 whatever the kernels do.  From the third
    call with the same input shape, dtype and parameter versions the whole forward is replayed as ONE CUDA graph
    (call 1 runs eagerly and fills the packed-filter caches, call 2 captures); the result is what the eager path
    returns, bit for bit.  Any parameter update (in place or by re-assignment) starts over.  If capture is impossible
    the eager path stays in use -- the same kernels, launched one by one."""
    if not net.use_cuda_graph or torch.cuda.is_current_stream_capturing():
        return _forward_learned(net, inputs, head_bc, wall_bcs)
    key = (tuple(inputs.shape), inputs.dtype, str(inputs.device), head_bc, wall_bcs, net.training,
           tuple((q.data_ptr(), q._version) for q in net.parameters()))
    pl = net.__dict__.get("_learned_plan")
    if pl is None or pl.key != key:
        pl = _LearnedPlan()
        pl.key, pl.calls, pl.graph, pl.failed = key, 0, None, False
        net.__dict__["_learned_plan"] = pl
    pl.calls += 1
    if pl.failed or pl.calls == 1:
        return _forward_learned(net, inputs, head_bc, wall_bcs)
    if pl.graph is None:
        try:
            pl.x = inputs.detach().clone()
            torch.cuda.synchronize(inputs.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                pl.out = _forward_learned(net, pl.x, head_bc, wall_bcs)
            pl.graph = g
        except Exception:  # not capturable on this build / driver: keep launching the kernels one by one
            pl.failed, pl.graph = True, None
            torch.cuda.synchronize(inputs.device)
            return _forward_learned(net, inputs, head_bc, wall_bcs)
    pl.x.copy_(inputs)
    pl.graph.replay()
    return tuple(None if o is None else o.clone() for o in pl.out)  # callers own what they get


def _learned_blocked_ok(net, H, W, head_bc, wall_bcs):
    """The all-blocked kernel path of a learned-boundary NewFluidNet: every layer's 9-region conv as two launches."""
    if head_bc != 1 or not wall_bcs or net.c_h % 4 or net.c_h > 16 or net.c_o > 4:
        return False
    h, w = H, W
    for l in range(net.levels):
        if not net.convs[l][0].layers[0].kernel_path_ok(h, w, [net.c_h]):
            return False
        h, w = h // 2, w // 2
    return net.conv[1].kernel_path_ok(H, W, [net.c_h] * net.levels + [net.c_i])


def _forward_learned_blocked(net, inputs):
    """NewFluidNet with learned boundaries (reference :1315-1388 with BoundaryLearnedConvolution2D layers, SURVEY.md 8f N1):
    activations stay in the blocked layout from the first conv to the head; every FluidLayer is TWO launches (interior
    conv with the producer's GroupNorm + GELU fused into its load and the statistics in its epilogue, then the ring
    kernel); pooling is incremental, the up-sampled levels and the raw input are conv[1]'s source list (never
    concatenated); zero-mean + curl + wall BCs are the head kernel."""
    B, _, H, W = inputs.shape
    dev, c_h, c_i = inputs.device, net.c_h, net.c_i
    gnp = lambda gn, c: (ops.pad_vec(gn.weight, c, dev, 1.0), ops.pad_vec(gn.bias, c, dev))

    def fluid(fl, sources, chans):
        yb, st, _ = fl.layers[0].forward_blocked(sources, chans)
        g, b_ = gnp(fl.layers[1], c_h)
        return ops.Source(yb, L.XFORM_GN_GELU, st, g, b_)

    inp_b = ops.pack_nchw(inputs)
    x_in = fluid(net.conv[0], [ops.Source(inp_b)], [c_i])
    srcs, level_in = [], x_in
    for l in range(net.levels):
        if l > 0:
            level_in = ops.Source(ops.avgpool2(level_in))  # pool^l(x_in), incrementally (identical composition, :1321-1322)
        y1 = level_in
        for r in range(net.repeats):
            y1 = fluid(net.convs[l][r], [y1], [c_h])
        srcs.append(y1 if l == 0 else ops.Source(ops.bicubic_up(y1, H, W)))
    srcs.append(ops.Source(inp_b))
    y1b, st1, _ = net.conv[1].forward_blocked(srcs, [c_h] * net.levels + [c_i])
    g0, b0 = gnp(net.gn[0], c_h)
    y2b, _, _ = net.conv[2].forward_blocked([ops.Source(y1b, L.XFORM_GN_GELU, st1, g0, b0)], [c_h], epi_act=L.ACT_GELU,
                                            want_stats=False)
    y3b, _, csum = net.conv[3].forward_blocked([ops.Source(y2b)], [c_h], want_stats=False, want_chan_sum=True)
    u, v, p, _ = ops.head(y3b, csum, None, net.a_bound, L.HEAD_CURL if net.loss_type == "curl" else L.HEAD_MAE, net.p_pred,
                          want_uvmax=False)
    return _shape_outputs(net, u, v, p, inputs.dtype)


def _forward_learned(net, inputs, head_bc, wall_bcs):
    """Learned-boundary networks (SURVEY.md section 8f N1).  NewFluidNet on grids every level of which holds the
    reference's boundary strips runs all-blocked (two launches per layer, `_forward_learned_blocked`); FluidNet (head
    conv enlarged by bc_x = bc_y = 2) and degenerate sizes run layer by layer through the module-level forwards."""
    B, _, H, W = inputs.shape
    if _learned_blocked_ok(net, H, W, head_bc, wall_bcs):
        return _forward_learned_blocked(net, inputs)
    dev = inputs.device
    x_in = net.conv[0](inputs)
    feats = []
    pooled = ops.pack_nchw(x_in)
    for l in range(net.levels):
        if l > 0:
            pooled = ops.avgpool2(ops.Source(pooled))
        y1 = ops.unpack_nchw(pooled, net.c_h)
        for r in range(net.repeats):
            y1 = net.convs[l][r](y1)
        if l > 0:
            y1 = ops.unpack_nchw(ops.bicubic_up(ops.Source(ops.pack_nchw(y1)), H, W), net.c_h)
        feats.append(y1.float())
    y = torch.cat(feats + [inputs.float()], 1)
    y = net.conv[1](y, bc_x=head_bc, bc_y=head_bc)
    c_h = net.c_h
    yb = ops.pack_nchw(y)
    src = ops.Source(yb, L.XFORM_GN_GELU, _stats_of_blocked(yb, c_h), ops.pad_vec(net.gn[0].weight, c_h, dev, 1.0),
                     ops.pad_vec(net.gn[0].bias, c_h, dev))
    y = ops.finalize_nchw(src, c_h)
    y = ops.finalize_nchw(ops.Source(ops.pack_nchw(net.conv[2](y)), L.XFORM_GELU), c_h)
    y = net.conv[3](y)
    Hh, Wh = y.shape[-2:]
    yb = ops.pack_nchw(y)
    csum = yb.double().sum(dim=(2, 3)).reshape(B, -1).contiguous()
    if wall_bcs:
        u, v, p, _ = ops.head(yb, csum, None, net.a_bound, L.HEAD_CURL if net.loss_type == "curl" else L.HEAD_MAE,
                              net.p_pred, want_uvmax=False)
        return _shape_outputs(net, u, v, p, inputs.dtype)
    # FluidNet: plain central differences of the enlarged stream function, no BCs (:1694-1697)
    ym = y - y.mean(dim=(2, 3), keepdim=True)
    a = ym[:, 0] * net.a_bound
    p = ym[:, 1] if net.p_pred else None
    u = 0.5 * (a[:, 2:, 1:-1] - a[:, :-2, 1:-1])
    v = -0.5 * (a[:, 1:-1, 2:] - a[:, 1:-1, :-2])
    return u.to(inputs.dtype), v.to(inputs.dtype), (p.to(inputs.dtype) if p is not None else None)


class Unet(nn.Module):
    """U-Net variant of the surrogate used as a time stepper: (x, y, dt, parameters, viscosity, T, u_prev, v_prev) ->
    (u, v, p, T_next) (reference :1700-2068; SURVEY.md section 8f N4).  Same constructor, module tree and `state_dict`
    keys/shapes as the reference.  `forward` runs on the module-level kernels (FluidLayer = conv + GroupNorm + GELU
    through libpbmc, incremental 2x2 pooling, bicubic up-sampling, curl head); it is not yet one fused DAG like
    NewFluidNet's.  The learned-boundary variant (r_p="learned": every conv is the 9-region conv, the first one enlarging the
    width through `bc_x=4`) runs on the same path: two launches per 9-region conv, the bc_x=4 layer as the 9-call composite."""

    def __init__(self, levels: int, c_i: int, c_h: int, c_o: int, device=torch.device("cpu"), act_fn: str = "gelu",
                 r_p="replicate", loss_type="curl", use_symm=False, dilation=1, a_bound=10.0, use_cosine=False, repeats=2,
                 use_skip=False, f=5, p_pred=False, spectral_conv=False, blurr=False, drop_rate=0.0):
        super().__init__()
        if spectral_conv:
            raise NotImplementedError("spectral_conv=True is outside the rollout path (advect_wi_gaia.py:253)")
        if blurr:
            raise NotImplementedError("blurr=True is outside the rollout path (advect_wi_gaia.py:255)")
        self.conv, self.gn = nn.ModuleList(), nn.ModuleList()
        self.levels, self.loss_type, self.a_bound = levels, loss_type, a_bound
        self.use_cosine, self.repeats, self.use_skip, self.p_pred = use_cosine, repeats, use_skip, p_pred
        self.c_i, self.c_o, self.f = c_i, c_o, f
        self.blurrer = None
        self.r_p = "constant" if r_p == "zeros" else r_p
        self.act = _make_act(act_fn)
        layer = lambda ci, co: FluidLayer(ci, co, act_fn, r_p, use_symm, dilation, f=f, drop_rate=drop_rate)
        for r in range(repeats):
            self.conv.append(layer(c_i if r == 0 else c_h, c_h))
        self.pool = nn.AvgPool2d((2, 2), stride=2)
        # down path: level 1 keeps c_h channels, every further level doubles them (:1866-1895)
        self.convs = nn.ModuleList()
        w = c_h
        for l in range(1, levels):
            self.convs.append(nn.ModuleList([layer(w // 2 if (r == 0 and l > 1) else w, w) for r in range(repeats)]))
            w *= 2
        w //= 2
        # up path: concat(skip of w/2 channels, up-sampled w channels) -> w/2 (:1897-1935)
        self.upconvs = nn.ModuleList()
        for _l in range(levels - 2, 0, -1):
            self.upconvs.append(nn.ModuleList([layer(w + w // 2 if r == 0 else w // 2, w // 2) for r in range(repeats)]))
            w //= 2
        self.c_head = w
        for ci, co in ((2 * w, w), (w, w), (w, c_o)):
            if self.r_p != "learned":
                self.conv.append(nn.Conv2d(ci, co, kernel_size=f, padding="same", dilation=dilation if ci == 2 * w else 1,
                                           padding_mode=r_p, stride=1))
            else:
                self.conv.append(BoundaryLearnedConvolution2D(ci, co, k=f, use_symm=use_symm))
            if ci == 2 * w:
                self.gn.append(torch.nn.GroupNorm(int(w / 4), w))

    def forward(self, inputs):
        _require_gelu(self)
        if not inputs.is_cuda:
            raise L.PbmcError("Unet runs on CUDA only: there is no CPU implementation of this path")
        if inputs.dim() != 4 or inputs.shape[1] != self.c_i:
            raise ValueError(f"expected inputs [B,{self.c_i},H,W], got {tuple(inputs.shape)}")
        learned = self.r_p == "learned"
        dev, dtype, R = inputs.device, inputs.dtype, self.repeats
        blocked = lambda t: ops.Source(ops.pack_nchw(t))
        pool = lambda t: ops.unpack_nchw(ops.avgpool2(blocked(t)), t.shape[1])
        up = lambda t, size: ops.unpack_nchw(ops.bicubic_up(blocked(t), int(size[0]), int(size[1])), t.shape[1])
        # non-learned: 3 padded columns each side (:1990-1991); learned: the first 9-region conv enlarges the width by the
        # same 3 columns itself (bc_x=4, bc_y=1, :1994-1996)
        x = [inputs.float() if learned else torch.nn.functional.pad(inputs.float(), (3, 3, 0, 0), mode=self.r_p)]
        for r in range(R):
            x[0] = self.conv[r](x[0], bc_x=4, bc_y=1) if (learned and r == 0) else self.conv[r](x[0])
        for l in range(1, self.levels):
            t = pool(x[l - 1])
            for r in range(R):
                t = self.convs[l - 1][r](t)
            x.append(t)
        xu = x[-1]
        for l_i, l in enumerate(range(self.levels - 2, 0, -1)):
            xu = torch.cat((x[l], up(xu, x[l].shape[-2:])), 1)
            for r in range(R):
                xu = self.upconvs[l_i][r](xu)
        y = torch.cat((up(xu, x[0].shape[-2:]), x[0]), 1)
        c = self.c_head
        head = (lambda m, t: m(t)) if learned else conv_module_forward  # 9-region conv modules / plain conv modules
        yb = ops.pack_nchw(head(self.conv[R], y))
        y = ops.finalize_nchw(ops.Source(yb, L.XFORM_GN_GELU, _stats_of_blocked(yb, c), ops.pad_vec(self.gn[0].weight, c, dev, 1.0),
                                         ops.pad_vec(self.gn[0].bias, c, dev)), c)
        y = ops.finalize_nchw(ops.Source(ops.pack_nchw(head(self.conv[R + 1], y)), L.XFORM_GELU), c)
        y = head(self.conv[R + 2], y)
        y = (y - y.mean(dim=(2, 3), keepdim=True))[..., 3:-3].contiguous()  # mean over the PADDED width, then crop (:2025)
        if self.loss_type in ("mae", "mass"):
            p = y[:, 3:4].to(dtype) if self.p_pred else None
            return y[:, 0:1].to(dtype), y[:, 1:2].to(dtype), p, y[:, 2:3].to(dtype)
        if self.loss_type != "curl":
            raise ValueError(self.loss_type)
        if self.c_o > 4:
            raise NotImplementedError("the curl head reads one 4-channel block (a, T, p)")
        # curl + wall BCs in the head kernel (channel 0 = stream function); with zero channel sums its "p" output is
        # channel 1 unchanged, which here is the temperature (:2041)
        yb = ops.pack_nchw(y)
        zero_sums = torch.zeros(y.shape[0], 4, dtype=torch.float64, device=dev)
        u, v, T, _ = ops.head(yb, zero_sums, None, self.a_bound, L.HEAD_CURL, True, want_uvmax=False)
        p = y[:, 2].to(dtype) if self.p_pred else None
        return u.to(dtype), v.to(dtype), p, torch.clip(T, 0.0, 1.5).to(dtype)


class ADNet(nn.Module):
    """Explicit upwind-advection / central-diffusion update with the CFL time step
    (reference :478-568).  `forward(inputs[B,6,H,W], dt=None, T_prev=None) -> (T[B,1,H,W], dt)`;
    channels = (u, v, T, RaQ, x, y).  As in the reference, dt is ONE scalar over the batch (:556)
    and the wall coordinates of `inputs` are overwritten in place (:532-535)."""

    def __init__(self, device, r_p="zeros", CN_max=0.1):
        super().__init__()
        self.device = device
        self.CN_max = CN_max

    def forward(self, inputs, dt=None, T_prev=None):
        if not inputs.is_cuda:
            raise L.PbmcError("ADNet runs on CUDA only: there is no CPU implementation of this path")
        B, _, H, W = inputs.shape
        dtype = inputs.dtype
        inputs[:, 4, :, 0] = 0.0
        inputs[:, 4, :, -1] = 4.0
        inputs[:, 5, 0, :] = 0.0
        inputs[:, 5, -1, :] = 1.0
        f32 = lambda t: t.contiguous().float()
        u, v = f32(inputs[:, 0]), f32(inputs[:, 1])
        T = f32(inputs[:, 2] if T_prev is None else T_prev.reshape(B, H, W))
        raq = f32(inputs[:, 3])
        xc, yc = inputs[:, 4].contiguous().double(), inputs[:, 5].contiguous().double()
        dx_min = (inputs[:, 4, 1:-1, 1:-1] - inputs[:, 4, 1:-1, :-2]).double().amin().reshape(1).contiguous()  # :555
        dt_dev = None
        uvmax = None
        if dt is None:
            uvmax = ops.uvmax_reduce(u, v, batch_global=True)
        else:
            dt_dev = torch.as_tensor(dt, dtype=torch.float64, device=inputs.device).reshape(1).contiguous()
        T_out, dt_out = ops.advect_diffuse_fields(T, u, v, xc, yc, raq, None, uvmax, dx_min, self.CN_max,
                                                  per_member_dt=False, dt_fixed_dev=dt_dev)
        dt_ret = dt if dt is not None else dt_out[0].to(dtype)
        return T_out[:, None].to(dtype), dt_ret


class _FusedPlan:
    """Cached device buffers + CUDA graph of one TS.forward configuration."""


class TS(nn.Module):
    """Evaluation wrapper that advances T by `ts` surrogate steps (reference :266-475).
    Same constructor and 15-argument `forward`; returns `(x, dts, u, v, p, V)` exactly like the
    reference: `x[i]` / `dts[i]` for every step, and the last step's fields."""

    def __init__(self, stokes, ad, device, ts=8, advection_scheme=2, scale=True, p_pred=True, net="fluidnet"):
        super().__init__()
        self.stokes, self.ad, self.ts, self.device = stokes, ad, ts, device
        self.advection_scheme, self.scale, self.p_pred, self.net = advection_scheme, scale, p_pred, net
        self._grid_key, self._grid = None, None
        self._plan_key, self._plan = None, None
        self._early_plan = None
        self.use_cuda_graph = True  # replay the whole call (convert in, ts steps, convert out) as one CUDA graph

    def _get_grid(self, xc, yc, ycc, dev):
        """Grid-derived device data (coordinates, stencil coefficients, dx_min) is built once per grid.
        Fast check: same tensor objects as last time; otherwise the values are compared (a driver that
        re-creates equal coordinate tensors every step must not rebuild -- or re-capture -- anything)."""
        key = tuple((t.data_ptr(), t._version, tuple(t.shape), str(t.device)) for t in (xc, yc, ycc))
        if key == self._grid_key:
            return self._grid
        if self._grid is not None and all(a.shape == b.shape and a.dtype == b.dtype and a.device == b.device and torch.equal(a, b)
                                          for a, b in zip((xc, yc, ycc), self._grid_src)):
            self._grid_key = key
            return self._grid
        self._grid, self._grid_key = Grid(xc, yc, ycc, dev), key
        self._grid_src = tuple(t.detach().clone() for t in (xc, yc, ycc))
        return self._grid

    # ------------------------------------------------------------------ fused, device-resident path
    def _forward_fused(self, T_prev, grid, prm, prm_nd, B, H, W, dev, cn_max, early_copied=False):
        """`ts` steps of build-input -> surrogate -> un-scale -> advect/diffuse -> BCs through pbmc_rollout.
        All device buffers of one (shape, ts, dtype, weights) configuration are cached in a plan; from the
        second call on, the dtype conversions and the ts steps replay as ONE CUDA graph, so a call costs one
        host->device copy of T, one graph launch and the result clones -- no allocation, no per-kernel launch."""
        stokes, n, dtype = self.stokes, self.ts, T_prev.dtype
        eng = stokes._engine(dev)
        _require_gelu(stokes)  # (the per-call part of stokes._check_fused; the input here is built on the device)
        if stokes.training and any(m.dropout.p != 0.0 for m in stokes.modules() if isinstance(m, FluidLayer)):
            raise NotImplementedError("dropout>0 in training mode is outside the inference path")
        eng.refresh()
        key = (B, H, W, n, dtype, id(grid), id(eng), eng.graph_key(B, H, W, refresh=False), float(cn_max), bool(stokes.p_pred))
        pl = self._plan if key == self._plan_key else None
        if pl is None:
            pl = _FusedPlan()
            pl.members_key = None
            pl.members = torch.zeros(B, 8, dtype=torch.float32, device=dev)
            pl.state = RolloutState(grid, pl.members, B, n + 1, n, cn_max, per_member_dt=False, p_pred=stokes.p_pred,
                                    device=dev)
            pl.T_in = torch.empty(B, H, W, dtype=dtype, device=dev)
            # all results of a call live in ONE buffer (T of every step | u, v, V, (p) | dt of every step), so that
            # handing the caller its own copy is one clone instead of three
            nf = 4 if stokes.p_pred else 3
            pl.n_T, pl.n_f = n * B * H * W, nf * B * H * W
            pl.out = torch.empty(pl.n_T + pl.n_f + n, dtype=dtype, device=dev)
            pl.split = lambda buf: (buf[:pl.n_T].view(n, B, 1, H, W), buf[pl.n_T + pl.n_f:],
                                    buf[pl.n_T:pl.n_T + pl.n_f].view(nf, B, 1, H, W))
            pl.T_out, pl.dt_out, pl.f_out = pl.split(pl.out)
            pl.graph, pl.calls = None, 0
            self._plan, self._plan_key = pl, key
        # `forward` may already have copied T into the cached plan and REPLAYED its graph speculatively, so that all of the
        # bookkeeping above overlapped the device work; the replay counts only if this call resolved to that very plan
        # with unchanged parameters (otherwise its results are discarded: it only wrote the plan's own buffers)
        spec_ok = getattr(self, "_spec_plan", None) is pl and early_copied and pl is self._early_plan
        if (prm, prm_nd) != pl.members_key:
            pl.members.copy_(ops.make_members([prm] * B, "cpu", nd_override=[prm_nd] * B))
            pl.members_key = (prm, prm_nd)
            spec_ok = False
        if not early_copied or pl is not self._early_plan:
            pl.T_in.copy_(T_prev.reshape(B, H, W), non_blocking=True)
        self._early_plan = self._spec_plan = None

        def body():
            st = pl.state
            st.T_seq[0].copy_(pl.T_in)
            eng.rollout(st, 1, n)
            pl.T_out.copy_(st.T_seq[1:n + 1].unsqueeze(2))
            pl.dt_out.copy_(st.dt_seq[:n, 0])
            pl.f_out[0].copy_(st.u.unsqueeze(1))
            pl.f_out[1].copy_(st.v.unsqueeze(1))
            pl.f_out[2].copy_(st.V.unsqueeze(1))
            if stokes.p_pred:
                pl.f_out[3].copy_(st.p.unsqueeze(1))

        pl.calls += 1
        if not self.use_cuda_graph or pl.calls == 1:
            body()  # first call: eager (module load, function attributes), also the warm-up the capture needs
        else:
            if pl.graph is None:
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    body()
                pl.graph = g
                spec_ok = False
            if not spec_ok:
                pl.graph.replay()
        T_all, dt_all, f_all = pl.split(pl.out.clone())  # callers own what they get
        x = {0: T_prev if T_prev.is_cuda else pl.T_in.clone().view(T_prev.shape)}
        dts = {}
        for i in range(1, n + 1):
            x[i] = T_all[i - 1]
            dts[i] = dt_all[i - 1]
        p = f_all[3] if stokes.p_pred else None
        if p is not None and not self.p_pred:
            p = p[:, 0]
        return x, dts, f_all[0], f_all[1], p, f_all[2]

    @torch.no_grad()
    def _forward_unet(self, T_prev, ycc, raq_nd, fkt_nd, fkp_nd, raq, fkt, fkp, xc, yc, u_prev, v_prev, dt):
        """U-Net time stepper (reference :419-451): the network predicts T directly; u_prev, v_prev and dt are inputs and
        stay what the caller passed for all `ts` steps; no advection kernel, no dt out; u, v are returned as predicted
        (the caller un-scales them, advect_wi_gaia.py:751-767).  Any grid size (the reference views to 128x506)."""
        if u_prev is None or v_prev is None or dt is None:
            raise ValueError("net='unet' needs u_prev, v_prev and dt")
        dev = torch.device(self.device)
        _require_cuda_device(dev)
        dtype = T_prev.dtype
        H, W = T_prev.shape[-2:]
        grid = self._get_grid(xc, yc, ycc, dev)
        def f32(t):  # [1,1,H,W] fields as the reference concatenates them (:419-441); a scalar dt is broadcast
            t = torch.as_tensor(t).to(dev, torch.float32)
            return t.expand(1, 1, H, W) if t.numel() == 1 else t.reshape(1, 1, H, W)

        members = ops.make_members([(float(raq), float(fkt), float(fkp))], dev,
                                   nd_override=[(float(raq_nd), float(fkt_nd), float(fkp_nd))])
        up, vp, dtf = f32(u_prev), f32(v_prev), f32(dt)
        x, u, v, V = {0: T_prev.to(dev)}, None, None, None
        Tc = x[0].reshape(1, H, W).float().contiguous()
        for i in range(1, self.ts + 1):
            # channels of the shared input builder: x/4, y/4, log10(clip V)/8, raq_nd, fkt_nd, fkp_nd, T
            c7 = ops.unpack_nchw(ops.build_input(Tc, grid.xc, grid.yc, grid.ycc, members)[0], 7)
            V = c7[:, 2:3]
            inp = torch.cat((c7[:, 0:2], dtf, c7[:, 3:6], V, c7[:, 6:7], up, vp), 1)
            u, v, _, T = self.stokes(inp)
            Tn = T.reshape(1, 1, H, W).float().clone()
            Tn[:, :, 0, :] = 1
            Tn[:, :, -1, :] = 0
            Tn[:, :, :, 0:1] = Tn[:, :, :, 1:2]
            Tn[:, :, :, -1:] = Tn[:, :, :, -2:-1]
            x[i] = Tn.to(dtype)
            Tc = Tn.reshape(1, H, W).contiguous()
        return x, {}, u.reshape(1, 1, H, W).to(dtype), v.reshape(1, 1, H, W).to(dtype), None, V.to(dtype)

    @torch.no_grad()
    def forward(self, T_prev, sdf, sdf2, ycc, raq_nd, fkt_nd, fkp_nd, raq, fkt, fkp, xc, yc, u_prev=None, v_prev=None,
                dt=None):
        if self.net == "unet":
            return self._forward_unet(T_prev, ycc, raq_nd, fkt_nd, fkp_nd, raq, fkt, fkp, xc, yc, u_prev, v_prev, dt)
        if self.net not in ("newfluidnet", "fluidnet"):
            raise ValueError(self.net)
        dev = torch.device(self.device)
        _require_cuda_device(dev)
        stokes = self.stokes
        dtype = T_prev.dtype
        B = T_prev.shape[0] if T_prev.dim() == 4 else 1
        H, W = T_prev.shape[-2:]
        # The host->device copy of T is the first thing the device needs: if the cached plan fits this call's shape and
        # dtype it is enqueued before the (tens of microseconds of) host-side bookkeeping below, which then overlaps it.
        early, pl0 = False, self._plan
        self._spec_plan = None
        if pl0 is not None and pl0.T_in.dtype == dtype and tuple(pl0.T_in.shape) == (B, H, W) and T_prev.numel() == B * H * W:
            pl0.T_in.copy_(T_prev.reshape(B, H, W), non_blocking=True)
            early = True
            if self.use_cuda_graph and pl0.graph is not None and self.ad is not None and not torch.cuda.is_current_stream_capturing():
                # speculative replay: the device starts on this call's T at once; _forward_fused verifies below that the
                # call really resolves to this plan (same grid, weights, parameters) and otherwise redoes it
                pl0.graph.replay()
                self._spec_plan = pl0
        self._early_plan = pl0 if early else None
        grid = self._get_grid(xc, yc, ycc, dev)
        fl = lambda t: float(t)
        advect = self.ad is not None and self.net == "newfluidnet"
        # learned-boundary nets: where the engine's ring kernel takes every level (else the per-step path below)
        fused = (isinstance(stokes, NewFluidNet) and grid.separable
                 and (stokes.r_p != "learned" or fused_supported(stokes, B, H, W)))
        cn_max = self.ad.CN_max if advect else 0.0
        n = self.ts
        if fused and advect:
            # whole loop device-resident: one C call enqueues ts steps (batch-global dt like ADNet, :556)
            return self._forward_fused(T_prev, grid, (fl(raq), fl(fkt), fl(fkp)), (fl(raq_nd), fl(fkt_nd), fl(fkp_nd)), B, H, W,
                                       dev, cn_max, early_copied=early)
        members = ops.make_members([(fl(raq), fl(fkt), fl(fkp))] * B, dev, nd_override=[(fl(raq_nd), fl(fkt_nd), fl(fkp_nd))] * B)
        T0 = T_prev.to(dev)
        x, dts = {0: T0}, {}
        Tc = T0.reshape(B, H, W).float().contiguous()
        u = v = p = V = None
        for i in range(1, n + 1):
            inp, V = ops.build_input(Tc, grid.xc, grid.yc, grid.ycc, members, want_V=True)
            uu, vv, pp = stokes(ops.unpack_nchw(inp, 7))
            s = members[:, 6].reshape(B, 1, 1)
            u, v, p = (uu.float() * s).contiguous(), (vv.float() * s).contiguous(), pp
            if advect:
                uvmax = ops.uvmax_reduce(u, v, batch_global=True)
                if grid.separable:
                    Tc, dt_i, _ = ops.advect_diffuse(Tc, u, v, grid.xcoef, grid.ycoef, members, uvmax, grid.dx_min,
                                                     cn_max, per_member_dt=False)
                else:
                    Tc, dt_i = ops.advect_diffuse_fields(Tc, u, v, grid.xc64, grid.yc64, None, members, uvmax,
                                                         grid.dx_min_dev, cn_max, per_member_dt=False)
                x[i] = Tc[:, None].to(dtype)
                dts[i] = dt_i[0].to(dtype)
        u = u.reshape(-1, 1, u.shape[-2], u.shape[-1]).to(dtype)
        v = v.reshape(-1, 1, v.shape[-2], v.shape[-1]).to(dtype)
        if self.p_pred and p is not None:
            p = p.reshape(-1, 1, p.shape[-2], p.shape[-1]).to(dtype)
        elif p is not None:
            p = p.to(dtype)
        return x, dts, u, v, p, V[:, None].to(dtype)
