"""Tensor-level wrappers over the C ABI (one Python function per `pbmc_*` operator).

These are the building blocks the drop-in modules use for their stand-alone `forward`s and
that the `-m gpu` parity tests call directly.  All tensors are float32 CUDA tensors owned by
PyTorch; the wrappers only allocate outputs and pass pointers + the current stream.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib as L


def _chk_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise L.PbmcError("this operator has no CPU implementation; pass CUDA tensors")


def nblk(c):
    return (int(c) + 3) // 4


# ------------------------------------------------------------------ weights
def expand_symmetric(w_unique: torch.Tensor, c_out: int) -> torch.Tensor:
    """Full filter bank of a SymmetricConv2d with symmetry {'h': h} (symmetric_layers_torch.py:118-138):
    [unique..., x-mirrored copies of the first h/2]."""
    n_mirror = c_out - w_unique.shape[0]
    if n_mirror == 0:
        return w_unique
    return torch.cat([w_unique, torch.flip(w_unique[:n_mirror], (3,))], 0)


def pack_conv_weight(w_full: torch.Tensor, src_channels) -> torch.Tensor:
    """[Co, Ci, k, k] -> float32 [ceil(Co/16)][cin_blks][k*k][4][16] (layout in include/pbmc.h).
    `src_channels`: channels contributed by each conv source, in concat order; each source is
    padded to a multiple of 4 input lanes (zero weights)."""
    Co, Ci, k, _ = w_full.shape
    assert sum(src_channels) == Ci, (src_channels, Ci)
    parts, c0 = [], 0
    for c in src_channels:
        wpart = w_full[:, c0:c0 + c]
        pad = nblk(c) * 4 - c
        if pad:
            wpart = torch.cat([wpart, wpart.new_zeros(Co, pad, k, k)], 1)
        parts.append(wpart)
        c0 += c
    w = torch.cat(parts, 1).float()
    cg = (Co + 15) // 16
    if cg * 16 != Co:
        w = torch.cat([w, w.new_zeros(cg * 16 - Co, w.shape[1], k, k)], 0)
    cb = w.shape[1] // 4
    w = w.reshape(cg, 16, cb, 4, k * k).permute(0, 2, 4, 3, 1).contiguous()  # [cg][cb][tap][ci][co]
    return w


def tf32_round(x: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest (ties away) float32 -> tf32 (10-bit mantissa), result still float32 -- cvt.rna.tf32.f32."""
    bits = x.contiguous().view(torch.int32)
    return ((bits + 0x1000) & -8192).view(torch.float32)


def pow2(e: torch.Tensor) -> torch.Tensor:
    """2^e as float32, built from the exponent bits (exact; e integer in [-126, 127])."""
    return ((e.to(torch.int32).reshape(1) + 127) << 23).view(torch.float32)


def prescale_pow2(w: torch.Tensor):
    """Tensor-core weight images hold w * 2^e, one e per layer, so that max|w| * 2^e lies in [2^14, 2^15): the fp16 hi part
    then uses fp16's whole range and the lo part stays normal for weights down to 2^-18 of the largest, whatever the
    layer's own scale (all-zero weights: e = 0).  Returns (w * 2^e, the image's 16-byte tail = float32 [2^-e, 0, 0, 0]),
    which the kernels' epilogues apply as fmaf(acc, 2^-e, bias).  Computed on w's device without a host sync."""
    mant, ex = torch.frexp(w.abs().amax())
    e = torch.where(mant > 0, 15 - ex, torch.zeros_like(ex)).clamp(-126, 126)
    tail = torch.cat([pow2(-e), w.new_zeros(3)])
    return w * pow2(e), tail


def umma_supported(cout: int, src_channels) -> bool:
    """Shapes the tcgen05 conv kernel takes (csrc/conv_umma.cu): <= 16 outputs, every source an even number of 4-channel blocks."""
    return cout <= 16 and all(nblk(c) % 2 == 0 for c in src_channels)


def pack_conv_weight_umma(w_full: torch.Tensor, src_channels) -> torch.Tensor:
    """[Co<=16, Ci, k, k] -> uint8 buffer holding the three K-major B-operand images of csrc/conv_umma.cu:
         tf32 : float32  [2 (hi, lo)][cin_blks  ][k*k][16 c_out][4 c_in]   hi = tf32(w),  lo = w - hi
         fp16 : float16  [2 (hi, lo)][cin_blks/2][k*k][16 c_out][8 c_in]   hi = fp16(w),  lo = fp16(w - hi)
         bf16 : bfloat16 [1         ][cin_blks/2][k*k][16 c_out][8 c_in]
         tail : float32  [4] = [2^-e, 0, 0, 0]
       back to back (offsets are multiples of 16 B); w here is the layer's filters times 2^e (prescale_pow2)."""
    Co, Ci, k, _ = w_full.shape
    assert Co <= 16 and sum(src_channels) == Ci
    parts, c0 = [], 0
    for c in src_channels:
        wpart = w_full[:, c0:c0 + c]
        pad = nblk(c) * 4 - c
        if pad:
            wpart = torch.cat([wpart, wpart.new_zeros(Co, pad, k, k)], 1)
        parts.append(wpart)
        c0 += c
    w, tail = prescale_pow2(torch.cat(parts, 1).float())
    if Co < 16:
        w = torch.cat([w, w.new_zeros(16 - Co, w.shape[1], k, k)], 0)
    cb = w.shape[1] // 4
    assert cb % 2 == 0
    w4 = w.reshape(16, cb, 4, k * k).permute(1, 3, 0, 2).contiguous()  # [cb][tap][co][4]
    hi = tf32_round(w4)
    img_tf32 = torch.stack([hi, w4 - hi], 0).contiguous()
    w8 = w.reshape(16, cb // 2, 8, k * k).permute(1, 3, 0, 2).contiguous()  # [cb/2][tap][co][8]
    h16 = w8.half()
    img_f16 = torch.stack([h16, (w8 - h16.float()).half()], 0).contiguous()
    img_bf16 = w8.bfloat16().contiguous()
    as_bytes = lambda t: t.view(torch.uint8).reshape(-1)
    return torch.cat([as_bytes(img_tf32), as_bytes(img_f16), as_bytes(img_bf16), as_bytes(tail)]).contiguous()


def row_supported(cout: int, ksize: int, src_channels) -> bool:
    """Shapes the row-streaming tcgen05 kernel takes (csrc/conv_row.cu): k in {3, 5}, <= 16 outputs, and
    the whole filter bank resident in shared memory next to the 4-stage input ring."""
    if cout > 16 or ksize not in (3, 5):
        return False
    groups = sum((nblk(c) + 3) // 4 for c in src_channels)
    n = ksize * 16
    plane = (128 + ksize - 1 + 7) // 8 * 8
    smem = 2176 + groups * ksize * 2 * (2 * n * 16) + 8 * (2 * 2 * plane * 16) + sum(nblk(c) * 4 for c in src_channels) * 8
    return groups <= 24 and smem <= 227 * 1024


def pack_conv_weight_row(w_full: torch.Tensor, src_channels) -> torch.Tensor:
    """[Co<=16, Ci, k, k] -> uint8 buffer with the two K-major B-operand images of csrc/conv_row.cu:
         fp16 : [group][dx][2 (hi, lo)][2 K-chunks][N = k*16 rows (dy, c_out)][8 c_in]   hi = fp16(w), lo = fp16(w - hi)
         bf16 : [group][dx][1         ][2 K-chunks][N rows][8 c_in]
         tail : float32 [4] = [2^-e, 0, 0, 0]
       back to back, w here being the layer's filters times 2^e (prescale_pow2).  A group is 16 input channels of ONE
       source (each source is zero-padded to a multiple of 16 channels), in concat order; the vertical tap dy rides in the
       MMA's N dimension."""
    Co, Ci, k, _ = w_full.shape
    assert Co <= 16 and sum(src_channels) == Ci
    parts, c0 = [], 0
    for c in src_channels:
        wpart = w_full[:, c0:c0 + c]
        pad = (nblk(c) + 3) // 4 * 16 - c
        if pad:
            wpart = torch.cat([wpart, wpart.new_zeros(Co, pad, k, k)], 1)
        parts.append(wpart)
        c0 += c
    w, tail = prescale_pow2(torch.cat(parts, 1).float())
    if Co < 16:
        w = torch.cat([w, w.new_zeros(16 - Co, w.shape[1], k, k)], 0)
    G = w.shape[1] // 16
    # (co, g, chunk, e, dy, dx) -> (g, dx, chunk, dy, co, e)
    w6 = w.reshape(16, G, 2, 8, k, k).permute(1, 5, 2, 4, 0, 3).contiguous()
    h16 = w6.half()
    img_f16 = torch.stack([h16, (w6 - h16.float()).half()], 2).contiguous()  # (g, dx, part, chunk, dy, co, e)
    img_bf16 = w6.bfloat16().contiguous()
    as_bytes = lambda t: t.view(torch.uint8).reshape(-1)
    return torch.cat([as_bytes(img_f16), as_bytes(img_bf16), as_bytes(tail)]).contiguous()


def pad_vec(v, c: int, device, fill=0.0) -> torch.Tensor:
    """[c] -> float32 [ceil(c/4)*4] on `device` (v=None: all `fill`)."""
    out = torch.full((nblk(c) * 4,), fill, dtype=torch.float32, device=device)
    if v is not None:
        out[:c] = v.detach().to(device, torch.float32).reshape(-1)
    return out


# ------------------------------------------------------------------ layout
def pack_nchw(x: torch.Tensor) -> torch.Tensor:
    _chk_cuda(x)
    x = x.contiguous().float()
    B, Cc, H, W = x.shape
    out = torch.empty(B, nblk(Cc), H, W, 4, dtype=torch.float32, device=x.device)
    L.check(L.load().pbmc_pack_nchw(L.ptr(x), L.ptr(out), B, Cc, H, W, L.stream_ptr(x.device)), "pbmc_pack_nchw")
    return out


def unpack_nchw(xb: torch.Tensor, Cc: int) -> torch.Tensor:
    _chk_cuda(xb)
    B, CB, H, W, _ = xb.shape
    out = torch.empty(B, Cc, H, W, dtype=torch.float32, device=xb.device)
    L.check(L.load().pbmc_unpack_nchw(L.ptr(xb), L.ptr(out), B, Cc, H, W, L.stream_ptr(xb.device)), "pbmc_unpack_nchw")
    return out


class Source:
    """A conv/pool/upsample input: blocked tensor + the producer's fused GroupNorm(+GELU)."""

    def __init__(self, t, xform=L.XFORM_NONE, stats=None, gamma=None, beta=None, channels_per_group=4):
        self.t, self.xform, self.stats, self.gamma, self.beta = t, xform, stats, gamma, beta
        B, CB, H, W, _ = t.shape
        self.nblk = CB
        self.inv_count = 1.0 / (channels_per_group * H * W) if xform in (L.XFORM_GN_GELU, L.XFORM_GN) else 0.0

    def c(self):
        return L.make_src(self.t, self.nblk, self.xform, self.stats, self.gamma, self.beta, self.inv_count)


class StagedSource:
    """A 16-channel conv input in PBMC_LAYOUT_STAGED16 (fp16 hi|lo operand image, see include/pbmc.h): what
    `bicubic_up(..., staged=True)` returns.  Only the row conv kernel reads it (3x3, replicate padding)."""

    def __init__(self, buf, B, H, W):
        self.t, self.B, self.H, self.W = buf, B, H, W
        self.nblk, self.xform = 4, L.XFORM_NONE

    def c(self):
        return L.make_src(self.t, 4, L.XFORM_NONE, layout=L.LAYOUT_STAGED16)


def finalize_nchw(src: Source, Cc: int) -> torch.Tensor:
    B, CB, H, W, _ = src.t.shape
    out = torch.empty(B, Cc, H, W, dtype=torch.float32, device=src.t.device)
    s = src.c()
    L.check(L.load().pbmc_finalize_nchw(C.byref(s), L.ptr(out), B, Cc, H, W, L.stream_ptr(out.device)), "pbmc_finalize_nchw")
    return out


# ------------------------------------------------------------------ conv
def conv_fwd(sources, wpk, bias, cout, ksize, pad_mode, epi_act=L.ACT_NONE, want_stats=False, want_chan_sum=False,
             impl="auto", wpk_umma=None, out=None, stats=None, csum=None, wpk_row=None, max_ctas=0):
    """Returns (out_blocked, stats|None, chan_sum|None).  `out`/`stats`/`csum` may be preallocated
    (statistics ACCUMULATE into the given buffers, as in the C ABI).  `max_ctas`: CTA budget (0 = the whole GPU)."""
    t0 = sources[0].t
    B, _, H, W, _ = t0.shape
    dev = t0.device
    cob = nblk(cout)
    if out is None:
        out = torch.empty(B, cob, H, W, 4, dtype=torch.float32, device=dev)
    if stats is None and want_stats:
        stats = torch.zeros(B, cob, 2, dtype=torch.float64, device=dev)
    if csum is None and want_chan_sum:
        csum = torch.zeros(B, cob * 4, dtype=torch.float64, device=dev)
    d = L.ConvDesc()
    d.nsrc = len(sources)
    for i, s in enumerate(sources):
        d.src[i] = s.c()
    d.B, d.H, d.W, d.cout, d.ksize = B, H, W, int(cout), int(ksize)
    d.pad_mode = L.PAD[pad_mode] if isinstance(pad_mode, str) else int(pad_mode)
    d.epi_act, d.impl, d.max_ctas = int(epi_act), L.CONV_IMPL[impl], int(max_ctas)
    d.wpk, d.wpk_umma, d.bias, d.out = L.ptr(wpk), L.ptr(wpk_umma), L.ptr(bias), L.ptr(out)
    d.wpk_row = L.ptr(wpk_row)
    d.out_stats, d.out_chan_sum = L.ptr(stats), L.ptr(csum)
    L.check(L.load().pbmc_conv_fwd(C.byref(d), L.stream_ptr(dev)), "pbmc_conv_fwd")
    return out, stats, csum


EDGE9_REGIONS = ("conv_top_left", "conv_top_right", "conv_bottom_left", "conv_bottom_right", "conv_top", "conv_bottom",
                 "conv_left", "conv_right")  # order of the filter sets in the edge kernel's image (reference names)


def pack_edge9_weights(w_regions, src_channels) -> torch.Tensor:
    """Eight full filter banks [Co<=16, Ci, k, k] (order EDGE9_REGIONS) -> float32 [8][cin_blks][k*k][16 c_out][4 c_in]
    for pbmc_conv_edge9; input channels follow the concatenation of the sources, each padded to whole 4-channel blocks."""
    assert len(w_regions) == 8
    out = []
    for w in w_regions:
        Co, Ci, k, _ = w.shape
        assert Co <= 16 and sum(src_channels) == Ci
        parts, c0 = [], 0
        for c in src_channels:
            wp = w[:, c0:c0 + c].float()
            pad = nblk(c) * 4 - c
            if pad:
                wp = torch.cat([wp, wp.new_zeros(Co, pad, k, k)], 1)
            parts.append(wp)
            c0 += c
        wf = torch.cat(parts, 1)
        if Co < 16:
            wf = torch.cat([wf, wf.new_zeros(16 - Co, wf.shape[1], k, k)], 0)
        nb = wf.shape[1] // 4
        # (co, blk, e, dy, dx) -> (blk, tap, co, e)
        out.append(wf.reshape(16, nb, 4, k * k).permute(1, 3, 0, 2).contiguous())
    return torch.stack(out, 0).contiguous()


def conv_edge9(sources, wedge, bias, cout, ksize, epi_act, out, stats=None, csum=None):
    """Second launch of the learned 9-region convolution (pbmc_conv_edge9): overwrite the ring of `out` (already holding the
    interior conv of pbmc_conv_fwd over the same sources) with the eight boundary regions; repair stats / csum."""
    B, _, H, W, _ = out.shape
    d = L.Edge9Desc()
    d.nsrc = len(sources)
    for i, s in enumerate(sources):
        d.src[i] = s.c()
    d.B, d.H, d.W, d.cout, d.ksize, d.epi_act = B, H, W, int(cout), int(ksize), int(epi_act)
    d.wedge, d.bias, d.out = L.ptr(wedge), L.ptr(bias), L.ptr(out)
    d.out_stats, d.out_chan_sum = L.ptr(stats), L.ptr(csum)
    L.check(L.load().pbmc_conv_edge9(C.byref(d), L.stream_ptr(out.device)), "pbmc_conv_edge9")
    return out


def conv_learned9(sources, wpk, wrow, wedge, bias, cout, ksize, epi_act=L.ACT_NONE, want_stats=False, want_chan_sum=False,
                  impl="auto"):
    """BoundaryLearnedConvolution2D (bc = 1) over blocked sources in two launches: interior filters through pbmc_conv_fwd
    (tensor cores where the shape allows), the ring through pbmc_conv_edge9.  Returns (out, stats|None, chan_sum|None)."""
    out, stats, csum = conv_fwd(sources, wpk, bias, cout, ksize, "zeros", epi_act=epi_act, want_stats=want_stats,
                                want_chan_sum=want_chan_sum, impl=impl, wpk_row=wrow)
    conv_edge9(sources, wedge, bias, cout, ksize, epi_act, out, stats, csum)
    return out, stats, csum


def block_stats(yb):
    """(sum, sum^2) per (sample, 4-channel block) of a blocked tensor [B, CB, h, W, 4], float64 [B, CB, 2]: the quantity the
    conv epilogues accumulate, here for a FEW rows (ghost-row corrections of the slab-decomposed surrogate) with torch
    reductions."""
    g = yb.double()
    return torch.stack([g.sum(dim=(2, 3, 4)), (g * g).sum(dim=(2, 3, 4))], -1)


def chan_sums(yb):
    """Per-channel sums of a blocked tensor [B, CB, h, W, 4] -> float64 [B, CB * 4]."""
    return yb.double().sum(dim=(2, 3)).reshape(yb.shape[0], -1)


def trunk_fwd(src: Source, layers, pad_mode, impl="auto", max_ctas=0, ping=None, stats=None, sync=None, loader="threads"):
    """The R FluidLayers of one pyramid level in ONE persistent launch (pbmc_trunk_fwd, csrc/conv_trunk.cu).
    `layers`: objects with .wpk_row, .bias, .gamma, .beta, .cout, .ksize, .cin_blks (engine._PackedLayer) -- each layer's
    GroupNorm affine is applied by ITS consumer.  Returns (raw output of the last layer [B,4,H,W,4], its GroupNorm sums
    [B,4,2], all sums [R,B,4,2]); raises PbmcError(unsupported) if the grid cannot be resident at once."""
    t0 = src.t
    B, CB, H, W, _ = t0.shape
    dev = t0.device
    R = len(layers)
    arr = (L.Layer * R)()
    for r, lay in enumerate(layers):
        arr[r].wpk, arr[r].wpk_umma, arr[r].wpk_row = L.ptr(getattr(lay, "wpk", None)), None, L.ptr(lay.wpk_row)
        arr[r].bias, arr[r].gamma, arr[r].beta = L.ptr(lay.bias), L.ptr(lay.gamma), L.ptr(lay.beta)
        arr[r].cin_blks, arr[r].cout, arr[r].ksize = lay.cin_blks, lay.cout, lay.ksize
    if ping is None:
        ping = [torch.empty(B, 4, H, W, 4, dtype=torch.float32, device=dev) for _ in range(2)]
    if stats is None:
        stats = torch.empty(R, B, 4, 2, dtype=torch.float64, device=dev)
    if sync is None:
        sync = torch.empty(B, dtype=torch.int32, device=dev)
    t = L.TrunkDesc()
    t.src0, t.layers = src.c(), arr
    t.ping[0], t.ping[1] = L.ptr(ping[0]), L.ptr(ping[1])
    t.stats, t.sync = L.ptr(stats), L.ptr(sync)
    t.R, t.B, t.H, t.W = R, B, H, W
    t.pad_mode = L.PAD[pad_mode] if isinstance(pad_mode, str) else int(pad_mode)
    t.impl, t.max_ctas, t.pre_zeroed = L.CONV_IMPL[impl], int(max_ctas), 0
    t.loader = {"threads": 0, "bulk": 1}[loader]
    L.check(L.load().pbmc_trunk_fwd(C.byref(t), L.stream_ptr(dev)), "pbmc_trunk_fwd")
    return ping[(R - 1) & 1], stats[R - 1], stats


# ------------------------------------------------------------------ pyramid
def avgpool2(src: Source) -> torch.Tensor:
    B, CB, H, W, _ = src.t.shape
    out = torch.empty(B, CB, H // 2, W // 2, 4, dtype=torch.float32, device=src.t.device)
    s = src.c()
    L.check(L.load().pbmc_avgpool2(C.byref(s), L.ptr(out), B, H, W, L.stream_ptr(out.device)), "pbmc_avgpool2")
    return out


def bicubic_up(src: Source, H: int, W: int, staged: bool = False):
    B, CB, Hs, Ws, _ = src.t.shape
    s = src.c()
    if staged:
        lib = L.load()
        buf = torch.zeros(lib.pbmc_staged_bytes(B, H, W), dtype=torch.uint8, device=src.t.device)
        L.check(lib.pbmc_bicubic_up_staged(C.byref(s), L.ptr(buf), B, Hs, Ws, H, W, L.stream_ptr(buf.device)), "pbmc_bicubic_up_staged")
        return StagedSource(buf, B, H, W)
    out = torch.empty(B, CB, H, W, 4, dtype=torch.float32, device=src.t.device)
    L.check(L.load().pbmc_bicubic_up(C.byref(s), L.ptr(out), B, Hs, Ws, H, W, L.stream_ptr(out.device)), "pbmc_bicubic_up")
    return out


# ------------------------------------------------------------------ members
def member_values(raq, fkt, fkp):
    """Host-side per-run constants (advect_wi_gaia.py:443-460, pytorch_networks_convae.py:343-350), in double."""
    raq, fkt, fkp = float(raq), float(fkt), float(fkp)
    raq_nd = (raq - 0.12624371) / (9.70723344 - 0.12624371)
    fkt_nd = (math.log10(fkt) - 6.00352841978384) / (9.888820429862925 - 6.00352841978384)
    fkp_nd = (math.log10(fkp) - 0.005251646002323797) / (1.9927988938926755 - 0.005251646002323797)
    scaler = math.exp(raq / 10 * 1.80167667 + math.log(fkt) * 0.4330392 + math.log(fkp) * -0.46052953) * 5
    return [raq_nd, fkt_nd, fkp_nd, math.log(fkt), math.log(fkp), raq, scaler, 0.0]


def make_members(params, device, nd_override=None) -> torch.Tensor:
    """params: iterable of (raq, fkt, fkp).  Returns a float32 [B, 8] tensor laid out as pbmc_member[B].
    nd_override: optional iterable of (raq_nd, fkt_nd, fkp_nd) when the caller supplies its own
    normalised values (TS.forward takes them as arguments)."""
    rows = [member_values(*p) for p in params]
    if nd_override is not None:
        for r, nd in zip(rows, nd_override):
            r[0], r[1], r[2] = float(nd[0]), float(nd[1]), float(nd[2])
    return torch.tensor(rows, dtype=torch.float64).float().to(device).contiguous()


# ------------------------------------------------------------------ input / head / stencil
def build_input(T, xc, yc, ycc, members, want_V=False):
    """T [B,H,W]; xc,yc,ycc [H,W]; members [B,8] -> (inp blocked [B,2,H,W,4], V|None)."""
    _chk_cuda(T, xc, yc, ycc, members)
    B, H, W = T.shape
    inp = torch.empty(B, 2, H, W, 4, dtype=torch.float32, device=T.device)
    V = torch.empty(B, H, W, dtype=torch.float32, device=T.device) if want_V else None
    L.check(L.load().pbmc_build_input(L.ptr(T), L.ptr(xc), L.ptr(yc), L.ptr(ycc), L.ptr(members), L.ptr(inp), L.ptr(V), B,
                                      H, W, L.stream_ptr(T.device)), "pbmc_build_input")
    return inp, V


def head(y_blocked, chan_sum, members, a_bound, head_kind, p_pred, want_uvmax=True):
    B, _, H, W, _ = y_blocked.shape
    dev = y_blocked.device
    u = torch.empty(B, H, W, dtype=torch.float32, device=dev)
    v = torch.empty_like(u)
    p = torch.empty_like(u) if p_pred else None
    uvmax = torch.zeros(B, dtype=torch.int32, device=dev) if want_uvmax else None
    L.check(L.load().pbmc_head(L.ptr(y_blocked), L.ptr(chan_sum), L.ptr(members), float(a_bound), int(head_kind),
                               int(bool(p_pred)), L.ptr(u), L.ptr(v), L.ptr(p), L.ptr(uvmax), B, H, W, L.stream_ptr(dev)),
            "pbmc_head")
    return u, v, p, uvmax


def uvmax_reduce(u, v, batch_global=False):
    B, H, W = u.shape
    out = torch.zeros(B, dtype=torch.int32, device=u.device)
    L.check(L.load().pbmc_uvmax(L.ptr(u), L.ptr(v), L.ptr(out), 0 if batch_global else 1, B, H, W, L.stream_ptr(u.device)),
            "pbmc_uvmax")
    return out


def stencil_coefs(coord64, wall_lo, wall_hi):
    """1-D cell coordinates (float64 CUDA tensor [n]) -> float32 [3, n] inverse spacings
    (1/d_minus, 1/d_plus, 1/(0.5 d_plus + 0.5 d_minus)) with ADNet's forced wall values."""
    _chk_cuda(coord64)
    coord64 = coord64.contiguous().double()
    n = coord64.numel()
    out = torch.empty(3, n, dtype=torch.float32, device=coord64.device)
    L.check(L.load().pbmc_stencil_coefs(L.ptr(coord64), n, float(wall_lo), float(wall_hi), L.ptr(out),
                                        L.stream_ptr(coord64.device)), "pbmc_stencil_coefs")
    return out


def advect_diffuse(T, u, v, xcoef, ycoef, members, uvmax, dx_min, cn_max, per_member_dt=True, dt_fixed=0.0,
                   want_uvmax_out=False, T_out=None, dt_out=None, uv_out=None):
    """Fast separable-grid step.  xcoef [3,W], ycoef [3,H] from stencil_coefs.
    Returns (T_out [B,H,W], dt [B] float64, uvmax_out|None)."""
    _chk_cuda(T, u, v, xcoef, ycoef)
    assert xcoef.shape == (3, T.shape[2]) and ycoef.shape == (3, T.shape[1])
    B, H, W = T.shape
    dev = T.device
    T_out = torch.empty_like(T) if T_out is None else T_out
    dt_out = torch.empty(B, dtype=torch.float64, device=dev) if dt_out is None else dt_out
    if uv_out is None and want_uvmax_out:
        uv_out = torch.zeros(B, dtype=torch.int32, device=dev)
    L.check(L.load().pbmc_advect_diffuse(L.ptr(T), L.ptr(u), L.ptr(v), L.ptr(xcoef), L.ptr(ycoef), L.ptr(members), L.ptr(uvmax),
                                         1 if per_member_dt else 0, float(dx_min), float(cn_max), float(dt_fixed),
                                         L.ptr(T_out), L.ptr(uv_out), L.ptr(dt_out), B, H, W, L.stream_ptr(dev)),
            "pbmc_advect_diffuse")
    return T_out, dt_out, uv_out


def advect_diffuse_slab(T, u, v, xcoef, ycoef, members, uvmax, dx_min, cn_max, T_out, dt_out, has_up, has_down,
                        peer_up_row_ptr=0, peer_down_row_ptr=0, dt_fixed=0.0, uv_out=None):
    """One rank's row slab of a decomposed grid (T, u, v [1,rows,W] with ghost rows).  peer_*_row_ptr: raw device
    addresses (ints) of the neighbours' ghost rows in THEIR T_out (peer memory), 0 = no fused push."""
    _chk_cuda(T, u, v, xcoef, ycoef, T_out)
    _, H, W = T.shape
    assert xcoef.shape == (3, W) and ycoef.shape == (3, H) and T.shape[0] == 1
    L.check(L.load().pbmc_advect_diffuse_slab(L.ptr(T), L.ptr(u), L.ptr(v), L.ptr(xcoef), L.ptr(ycoef), L.ptr(members),
                                              L.ptr(uvmax), float(dx_min), float(cn_max), float(dt_fixed), L.ptr(T_out),
                                              L.ptr(uv_out), L.ptr(dt_out), H, W, int(bool(has_up)), int(bool(has_down)),
                                              int(peer_up_row_ptr) or None, int(peer_down_row_ptr) or None,
                                              L.stream_ptr(T.device)), "pbmc_advect_diffuse_slab")
    return T_out, dt_out


SLAB_SYNC_BYTES = C.sizeof(L.SlabSync)


def _peer_array(peer_ptrs):
    if isinstance(peer_ptrs, C.Array):  # already marshalled (per-step callers build it once)
        return peer_ptrs
    return (C.c_void_p * len(peer_ptrs))(*[int(q) for q in peer_ptrs])


def peer_array(peer_ptrs):
    """ctypes array of the ranks' pbmc_slab_sync addresses, to be built once and passed to the per-step calls."""
    return _peer_array(peer_ptrs)


def slab_sync_publish(u, v, self_ptr, peer_ptrs, rank):
    """First publication of a flag-synchronised slab run: this rank's max|u|,|v| (owned interior rows of the local
    [1,rows,W] arrays) goes into every rank's slot with tag steps_done + 1 (pbmc_slab_sync_publish)."""
    _chk_cuda(u, v)
    _, H, W = u.shape
    L.check(L.load().pbmc_slab_sync_publish(L.ptr(u), L.ptr(v), H, W, int(self_ptr), _peer_array(peer_ptrs), int(rank),
                                            len(peer_ptrs), L.stream_ptr(u.device)), "pbmc_slab_sync_publish")


def advect_diffuse_slab_sync(T, u, v, xcoef, ycoef, members, dx_min, cn_max, T_out, dt_out, has_up, has_down,
                             peer_up_row_ptr, peer_down_row_ptr, self_ptr, peer_ptrs, rank):
    """One time step of one rank's slab with the dt reduction and the halo exchange inside the kernel
    (pbmc_advect_diffuse_slab_sync): no collective call, one launch.  self_ptr / peer_ptrs: device addresses of the
    ranks' pbmc_slab_sync blocks (peer-mapped memory)."""
    _chk_cuda(T, u, v, xcoef, ycoef, T_out)
    _, H, W = T.shape
    assert xcoef.shape == (3, W) and ycoef.shape == (3, H) and T.shape[0] == 1
    L.check(L.load().pbmc_advect_diffuse_slab_sync(L.ptr(T), L.ptr(u), L.ptr(v), L.ptr(xcoef), L.ptr(ycoef), L.ptr(members),
                                                   float(dx_min), float(cn_max), L.ptr(T_out), L.ptr(dt_out), H, W,
                                                   int(bool(has_up)), int(bool(has_down)), int(peer_up_row_ptr) or None,
                                                   int(peer_down_row_ptr) or None, int(self_ptr), _peer_array(peer_ptrs),
                                                   int(rank), len(peer_ptrs), L.stream_ptr(T.device)),
            "pbmc_advect_diffuse_slab_sync")
    return T_out, dt_out


def advect_diffuse_fields(T, u, v, xc, yc, raq_field, members, uvmax, dx_min_dev, cn_max, per_member_dt=False,
                          dt_fixed_dev=None):
    """General form (coordinates as float64 fields, RaQ optionally a field; ADNet.forward semantics)."""
    B, H, W = T.shape
    assert xc.dtype == torch.float64 and yc.dtype == torch.float64
    dev = T.device
    T_out = torch.empty_like(T)
    dt_out = torch.empty(B, dtype=torch.float64, device=dev)
    stride = 0 if xc.dim() == 2 or xc.shape[0] == 1 else H * W
    L.check(L.load().pbmc_advect_diffuse_fields(L.ptr(T), L.ptr(u), L.ptr(v), L.ptr(xc), L.ptr(yc), stride, L.ptr(raq_field),
                                                L.ptr(members), L.ptr(uvmax), 1 if per_member_dt else 0,
                                                L.ptr(dx_min_dev), float(cn_max), L.ptr(dt_fixed_dev), L.ptr(T_out),
                                                L.ptr(dt_out), B, H, W, L.stream_ptr(dev)), "pbmc_advect_diffuse_fields")
    return T_out, dt_out


def clamp_T(T, core_cool=False):
    B, H, W = T.shape
    L.check(L.load().pbmc_clamp_T(L.ptr(T), int(bool(core_cool)), B, H, W, L.stream_ptr(T.device)), "pbmc_clamp_T")
    return T


def diagnostics(T):
    """T [B,H,W] float32 -> (mean_T [B], profile [B,H]) float64 on device (SURVEY.md section 8a A11)."""
    B, H, W = T.shape
    prof = torch.empty(B, H, dtype=torch.float64, device=T.device)
    mean = torch.empty(B, dtype=torch.float64, device=T.device)
    L.check(L.load().pbmc_diagnostics(L.ptr(T), L.ptr(prof), L.ptr(mean), B, H, W, L.stream_ptr(T.device)), "pbmc_diagnostics")
    return mean, prof
