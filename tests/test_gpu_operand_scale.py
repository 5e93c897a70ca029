"""Operand magnitude: the convolutions must not care how large or small weights and inputs are.

The fp16 hi+lo split (f16x2 kernels, persistent trunk) has fp16's exponent range: a weight or input far from 1 loses
relative precision (subnormal lo part below 2^-3 relative to fp16's unit) or overflows (above 65504), while the tf32, bf16
and FFMA paths keep fp32's range.  The checks here use operands away from unit scale, and per element, where a relative
L2 over the whole tensor would average a magnitude-dependent error away:
  a. multiplying a layer's weights and bias by 2^k multiplies its output by exactly 2^k (every implementation);
  b. at any weight scale each output element is within 2^-19 (|w| * |x| + |b|) of the float64 oracle;
  c. the module-level drop-in takes inputs of any magnitude;
  d. whole networks with every conv scaled by 2^k meet the parity rule max(1e-5, 1.5 x the reference's own fp32 noise),
     with that noise computed here on the same scaled weights.
"""
import functools

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from oracle import ref_torch as RT
from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import ops
from pbml_mantle_convection_b200.symmetric_layers_torch import TENSOR_CORE_MIN_SIDE, SymmetricConv2d, conv_module_forward, full_weight
from tests._util import field_bound, load, load_learned_case, load_weights, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PARAMS = (6.79733173, 475523342.0, 2.58574662)

ALL_IMPLS = ["ffma", "umma_3xtf32", "umma_f16x2", "umma_bf16", "row_f16x2", "row_bf16", "mux_f16x2", "mux_bf16"]
F16X2_IMPLS = ["umma_f16x2", "row_f16x2", "mux_f16x2"]

# (B, source channels, Co, H, W, k, pad, GN_GELU on the first source): single-source shapes of CONV_CASES / ROW_CASES /
# MUX_CASES (tests/test_gpu_ops.py), the c_out = 2 head with its channel sums, k = 5, and a three-source concat whose first
# source carries its producer's GroupNorm + GELU (mux requests of multi-source / 5x5 shapes run the row kernel)
CASES = [
    (1, [16], 16, 40, 70, 3, "replicate", False),
    (1, [16], 2, 24, 40, 3, "replicate", False),
    (1, [16], 16, 21, 66, 5, "zeros", False),
    (2, [16, 16, 8], 16, 26, 45, 3, "reflect", True),
]


def cu(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device=DEV)


def f32(a):
    """The float64 value of a's float32 rounding: what the kernels are given."""
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def _operands(case, seed):
    B, chans, Co, H, W, k, pad, gn = case
    r = np.random.default_rng(seed)
    xs = [r.standard_normal((B, c, H, W)) for c in chans]
    w = f32(r.standard_normal((Co, sum(chans), k, k)) / np.sqrt(sum(chans) * k * k))
    b = f32(r.standard_normal(Co))
    g0, be0 = f32(1 + 0.2 * r.standard_normal(chans[0])), f32(0.2 * r.standard_normal(chans[0]))
    srcs = []
    for i, x in enumerate(xs):
        xb = ops.pack_nchw(cu(x))
        if i == 0 and gn:
            st = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
            srcs.append(ops.Source(xb, L.XFORM_GN_GELU, st, cu(g0), cu(be0)))
        else:
            srcs.append(ops.Source(xb))
    return srcs, w, b


def _conv(case, srcs, w, b, impl):
    B, chans, Co, H, W, k, pad, gn = case
    wt = cu(w)
    wum = ops.pack_conv_weight_umma(wt, chans) if ops.umma_supported(Co, chans) else None
    wrow = ops.pack_conv_weight_row(wt, chans) if ops.row_supported(Co, k, chans) else None
    return ops.conv_fwd(srcs, ops.pack_conv_weight(wt, chans), ops.pad_vec(cu(b), Co, DEV), Co, k, pad, want_stats=True,
                        want_chan_sum=Co <= 4, impl=impl, wpk_umma=wum, wpk_row=wrow)


def _assert_scaled(y0, yk, k, what):
    """yk == 2^k y0 bit for bit (both float32 tensors)."""
    ok = torch.equal(yk, y0 * 2.0**k)
    if not ok:
        d = (yk.double() - y0.double() * 2.0**k).abs().max().item() / max(y0.abs().max().item() * 2.0**k, 1e-300)
        pytest.fail(f"{what}: 2^{k}-scaled weights do not give a 2^{k}-scaled output (max deviation {d:.2e} of max|y|)")


def _assert_sums(s0, sk, factor, what):
    """sk == factor * s0 up to the order of the double-precision atomics, which may differ between two launches"""
    if s0 is None:
        return
    a, b = s0.double() * factor, sk.double()
    for i in range(a.shape[-1]):  # each moment on its own scale
        ai, bi = a[..., i], b[..., i]
        assert torch.allclose(bi, ai, rtol=1e-12, atol=1e-12 * float(ai.abs().max()) + 1e-300), what


def _gn_factor(k, dev):
    """GroupNorm sums are (sum, sum of squares): they scale by (2^k, 4^k)."""
    return torch.tensor([2.0**k, 4.0**k], dtype=torch.float64, device=dev)


SCALES_EXACT = [-20, -12, -6, -3, 3, 8]


@pytest.mark.parametrize("impl", ALL_IMPLS)
@pytest.mark.parametrize("case", CASES)
def test_weight_scale_equivariance(case, impl):
    """conv(x; 2^k w, 2^k b) == 2^k conv(x; w, b) exactly: a power-of-two scale is exact in every format, so an
    implementation whose result depends on it loses precision with the weights' magnitude (FFMA, tf32 and bf16 are the
    controls that show the property holds for a correct kernel).  GroupNorm sums scale by 4^k, channel sums by 2^k."""
    srcs, w, b = _operands(case, 11)
    y0, st0, cs0 = _conv(case, srcs, w, b, impl)
    for k in SCALES_EXACT:
        yk, stk, csk = _conv(case, srcs, w * 2.0**k, b * 2.0**k, impl)
        _assert_scaled(y0, yk, k, f"{impl} {case}")
        _assert_sums(st0, stk, _gn_factor(k, DEV), "GroupNorm sums")
        _assert_sums(cs0, csk, 2.0**k, "channel sums")


class _Lay:
    """What ops.trunk_fwd reads of an engine._PackedLayer."""

    def __init__(self, w, b, g, be):
        self.wpk = ops.pack_conv_weight(cu(w), [16])
        self.wpk_row = ops.pack_conv_weight_row(cu(w), [16])
        self.bias, self.gamma, self.beta = ops.pad_vec(cu(b), 16, DEV), cu(g), cu(be)
        self.cin_blks, self.cout, self.ksize = 4, 16, 3


def _trunk_case(seed=140, B=1, H=40, W=130, R=4):
    r = np.random.default_rng(seed)
    x = r.standard_normal((B, 16, H, W))
    ws = [f32(r.standard_normal((16, 16, 3, 3)) / 12) for _ in range(R)]
    bs = [f32(0.3 * r.standard_normal(16)) for _ in range(R)]
    gs = [f32(1 + 0.2 * r.standard_normal(16)) for _ in range(R)]
    bes = [f32(0.2 * r.standard_normal(16)) for _ in range(R)]
    xb = ops.pack_nchw(cu(x))
    st0 = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
    src = ops.Source(xb, L.XFORM_GN_GELU, st0, cu(gs[0]), cu(bes[0]))
    return src, ws, bs, gs, bes


def _trunk(src, ws, bs, gs, bes, loader, impl="auto"):
    lays = [_Lay(w, b, g, be) for w, b, g, be in zip(ws, bs, gs, bes)]
    B, _, H, W, _ = src.t.shape
    ping = [torch.empty(B, 4, H, W, 4, dtype=torch.float32, device=DEV) for _ in range(2)]
    out, st_last, st_all = ops.trunk_fwd(src, lays, "replicate", impl=impl, ping=ping, loader=loader)
    return out.clone(), st_last.clone(), st_all.clone(), ping, lays


@pytest.mark.parametrize("loader", ["threads", "bulk"])
def test_trunk_weight_scale_equivariance(loader):
    """The persistent trunk kernel, last layer's weights and bias scaled by 2^k (scaling an inner layer is not exact:
    GroupNorm's eps then enters the next layer's input)."""
    src, ws, bs, gs, bes = _trunk_case()
    y0, s0, sa0, _, _ = _trunk(src, ws, bs, gs, bes, loader)
    for k in SCALES_EXACT:
        yk, sk, sak, _, _ = _trunk(src, ws[:-1] + [ws[-1] * 2.0**k], bs[:-1] + [bs[-1] * 2.0**k], gs, bes, loader)
        _assert_scaled(y0, yk, k, f"trunk ({loader} loader)")
        _assert_sums(s0, sk, _gn_factor(k, DEV), "GroupNorm sums")
        _assert_sums(sa0[:-1], sak[:-1], 1.0, "GroupNorm sums of the unscaled layers")


@pytest.mark.parametrize("k,chans,cout", [(3, [16], 16), (5, [16], 1), (5, [16, 16, 8], 16)])
def test_learned9_weight_scale_equivariance(k, chans, cout):
    """BoundaryLearnedConvolution2D as interior conv (tensor cores where the shape allows) + FFMA ring kernel."""
    r = np.random.default_rng(5 + k + cout)
    B, H, W = 1, 24, 40
    ci = sum(chans)
    xs = [r.standard_normal((B, c, H, W)) for c in chans]
    wts = {n: f32(r.standard_normal((cout, ci, k, k)) / (k * np.sqrt(ci))) for n in ("conv",) + ops.EDGE9_REGIONS}
    bias = f32(0.3 * r.standard_normal(cout))
    srcs = [ops.Source(ops.pack_nchw(cu(x))) for x in xs]

    def run(s):
        wm = cu(wts["conv"] * s)
        wedge = ops.pack_edge9_weights([cu(wts[n] * s) for n in ops.EDGE9_REGIONS], chans)
        wrow = ops.pack_conv_weight_row(wm, chans) if ops.row_supported(cout, k, chans) else None
        return ops.conv_learned9(srcs, ops.pack_conv_weight(wm, chans), wrow, wedge, ops.pad_vec(cu(bias * s), cout, DEV), cout,
                                 k, want_stats=True, want_chan_sum=cout <= 4)

    y0, st0, cs0 = run(1.0)
    for e in SCALES_EXACT:
        yk, stk, csk = run(2.0**e)
        _assert_scaled(y0, yk, e, f"learned9 k={k} {chans}->{cout}")
        _assert_sums(st0, stk, _gn_factor(e, DEV), "GroupNorm sums")
        _assert_sums(cs0, csk, 2.0**e, "channel sums")


# ------------------------------------------------------------------------------------------------ b. per-element accuracy
SCALES_ACC = [-12, -6, 0, 6]
ELEM_BOUND = 2.0**-19
L2_BOUND = 3e-6


def _check_elements(y, ref, absref, what):
    """|y - ref| <= 2^-19 (|w| * |x| + |b|) per element, and rel-L2 <= 3e-6 per output channel."""
    y = np.asarray(y, np.float64)
    assert np.isfinite(y).all(), what
    ratio = np.abs(y - ref) / np.maximum(absref, 1e-300)
    worst = float(ratio.max())
    assert worst <= ELEM_BOUND, f"{what}: worst element error {worst:.2e} x (|w|*|x|+|b|) > 2^-19"
    for c in range(y.shape[1]):
        e = relerr(y[:, c], ref[:, c])
        assert e <= L2_BOUND, f"{what}: channel {c} rel-L2 {e:.2e}"


def _source_values(srcs, case):
    """float64 values the kernels read from each source (GroupNorm + GELU of the first one in float64)."""
    B, chans, Co, H, W, k, pad, gn = case
    vals = []
    for i, s in enumerate(srcs):
        x = ops.unpack_nchw(s.t, chans[i]).double().cpu().numpy()
        if i == 0 and gn:
            x = RN.gelu(RN.group_norm(x, s.gamma.double().cpu().numpy(), s.beta.double().cpu().numpy(), chans[0] // 4))
        vals.append(x)
    return np.concatenate(vals, 1)


@pytest.mark.parametrize("impl", F16X2_IMPLS)
@pytest.mark.parametrize("case", CASES)
def test_f16x2_accuracy_at_any_weight_scale(case, impl):
    B, chans, Co, H, W, k, pad, gn = case
    srcs, w, b = _operands(case, 13)
    x = _source_values(srcs, case)
    for e in SCALES_ACC:
        we, be = w * 2.0**e, b * 2.0**e
        y, _, _ = _conv(case, srcs, we, be, impl)
        ref = RN.conv2d_same(x, we, be, pad)
        absref = RN.conv2d_same(np.abs(x), np.abs(we), np.abs(be), pad)
        _check_elements(ops.unpack_nchw(y, Co).cpu().numpy(), ref, absref, f"{impl} {case} weights x 2^{e}")


@pytest.mark.parametrize("impl", F16X2_IMPLS)
def test_f16x2_accuracy_channels_of_different_magnitude(impl):
    """A c_out = 2 head whose stream-function and pressure channels differ in weight magnitude by 2^10: one prescale
    exponent per layer must still serve the small channel."""
    case = (1, [16], 2, 48, 70, 3, "replicate", False)
    srcs, w, b = _operands(case, 17)
    w[1] *= 2.0**-10
    b[1] *= 2.0**-10
    x = _source_values(srcs, case)
    for e in SCALES_ACC:
        we, be = w * 2.0**e, b * 2.0**e
        y, _, _ = _conv(case, srcs, we, be, impl)
        ref = RN.conv2d_same(x, we, be, "replicate")
        absref = RN.conv2d_same(np.abs(x), np.abs(we), np.abs(be), "replicate")
        _check_elements(ops.unpack_nchw(y, 2).cpu().numpy(), ref, absref, f"{impl} head weights x 2^{e}")


@pytest.mark.parametrize("loader", ["threads", "bulk"])
def test_trunk_accuracy_at_any_weight_scale(loader):
    """Last trunk layer against the float64 conv of the input the kernel read: GroupNorm + GELU of the device's own
    previous layer (finalize_nchw applies the same transform)."""
    src, ws, bs, gs, bes = _trunk_case()
    R = len(ws)
    for e in SCALES_ACC:
        we, be = ws[-1] * 2.0**e, bs[-1] * 2.0**e
        y, _, st_all, ping, lays = _trunk(src, ws[:-1] + [we], bs[:-1] + [be], gs, bes, loader)
        prev = ops.Source(ping[(R - 2) & 1], L.XFORM_GN_GELU, st_all[R - 2], lays[R - 2].gamma, lays[R - 2].beta)
        x = ops.finalize_nchw(prev, 16).double().cpu().numpy()
        ref = RN.conv2d_same(x, we, be, "replicate")
        absref = RN.conv2d_same(np.abs(x), np.abs(we), np.abs(be), "replicate")
        _check_elements(ops.unpack_nchw(y, 16).cpu().numpy(), ref, absref, f"trunk ({loader}) last layer x 2^{e}")


def _scale_source(x):
    """x [B, C, H, W] as a PBMC_XFORM_SCALE source: blocked tensor + its (sum, sum^2) per (sample, block)."""
    xb = ops.pack_nchw(cu(x))
    st = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
    return ops.Source(xb, L.XFORM_SCALE, st)


@pytest.mark.parametrize("impl", ["mux_f16x2", "mux_bf16"])
@pytest.mark.parametrize("Co,pad", [(16, "replicate"), (2, "zeros")])
def test_scale_source_mode_any_input_magnitude(Co, pad, impl):
    """PBMC_XFORM_SCALE (the network's conv[3] source): the mux kernel scales the source by 2^-s per sample, s from the
    source's rms, and the output back by 2^s.  Inputs 2^-24 ... 2^20 (beyond fp16's range) against the float64 oracle;
    two samples of very different magnitude in one launch."""
    r = np.random.default_rng(Co + 3)
    x0 = f32(r.standard_normal((2, 16, 40, 150)))
    w = f32(r.standard_normal((Co, 16, 3, 3)) / 12)
    b = f32(r.standard_normal(Co))
    for j in [-24, -16, 0, 16, 20]:
        x = x0 * np.array([2.0**j, 2.0**-j]).reshape(2, 1, 1, 1)
        y, _, _ = ops.conv_fwd([_scale_source(x)], ops.pack_conv_weight(cu(w), [16]), ops.pad_vec(cu(b), Co, DEV), Co, 3, pad,
                               want_chan_sum=Co <= 4, impl=impl, wpk_row=ops.pack_conv_weight_row(cu(w), [16]))
        y = ops.unpack_nchw(y, Co).cpu().numpy()
        ref = RN.conv2d_same(x, w, b, pad)
        if impl == "mux_f16x2":
            _check_elements(y, ref, RN.conv2d_same(np.abs(x), np.abs(w), np.abs(b), pad), f"SCALE source x 2^{j}")
        else:  # single bf16 pass: its own stated bound, now at any magnitude
            assert np.isfinite(y).all() and relerr(y, ref) < 1e-2, (j, relerr(y, ref))


def test_scale_source_mode_is_refused_where_not_implemented():
    """Only the mux kernel implements PBMC_XFORM_SCALE; every other request is refused, never ignored."""
    r = np.random.default_rng(2)
    x, w = r.standard_normal((1, 16, 20, 30)), f32(r.standard_normal((16, 16, 3, 3)) / 12)
    wt = cu(w)
    args = dict(wpk_umma=ops.pack_conv_weight_umma(wt, [16]), wpk_row=ops.pack_conv_weight_row(wt, [16]))
    for impl in ["ffma", "umma_3xtf32", "umma_f16x2", "umma_bf16", "row_f16x2", "row_bf16"]:
        with pytest.raises(L.PbmcError, match="unsupported"):
            ops.conv_fwd([_scale_source(x)], ops.pack_conv_weight(wt, [16]), torch.zeros(16, device=DEV), 16, 3, "zeros",
                         impl=impl, **args)
    with pytest.raises(L.PbmcError, match="unsupported"):  # 5x5: the mux kernel does not take the shape
        w5 = cu(r.standard_normal((16, 16, 5, 5)) / 20)
        ops.conv_fwd([_scale_source(x)], ops.pack_conv_weight(w5, [16]), torch.zeros(16, device=DEV), 16, 5, "zeros",
                     impl="mux_f16x2", wpk_row=ops.pack_conv_weight_row(w5, [16]))
    with pytest.raises(L.PbmcError):  # the pyramid operators do not take it either
        ops.avgpool2(_scale_source(x))


# ------------------------------------------------------------------------------------------------ c. module-level inputs
def _module(kind):
    torch.manual_seed(3)
    if kind == "symmetric":
        m = SymmetricConv2d(16, 16, 3, padding=1, padding_mode="replicate", symmetry={"h": 4})
    else:
        m = nn.Conv2d(16, 16, 3, padding=1, padding_mode="replicate")
    return m.to(DEV)


@pytest.mark.parametrize("j", [-16, 0, 16, 20])
@pytest.mark.parametrize("kind", ["symmetric", "conv2d"])
def test_module_forward_any_input_magnitude(kind, j):
    """conv_module_forward on the tensor cores (>= TENSOR_CORE_MIN_SIDE) with inputs scaled by 2^j."""
    m = _module(kind)
    side = max(64, TENSOR_CORE_MIN_SIDE)
    x = torch.randn(2, 16, side, side + 6, generator=torch.Generator().manual_seed(j + 40), dtype=torch.float64) * 2.0**j
    x = x.float().double()
    with torch.no_grad():
        y = (m(x.float().to(DEV)) if kind == "symmetric" else conv_module_forward(m, x.float().to(DEV))).double().cpu()
        w64, b64 = full_weight(m).detach().double().cpu(), m.bias.detach().double().cpu()
    ref = F.conv2d(F.pad(x, (1, 1, 1, 1), mode="replicate"), w64, b64)
    assert torch.isfinite(y).all(), f"{kind}: non-finite output at input scale 2^{j}"
    e = relerr(y.numpy(), ref.numpy())
    assert e <= L2_BOUND, f"{kind}: rel-L2 {e:.2e} at input scale 2^{j}"


# ------------------------------------------------------------------------------------------------ d. networks
NET_SCALES = [-6, -3, 3]


def _scale_convs(sd, k):
    """Every conv weight and bias (learnable biases included) times 2^k; GroupNorm affines unchanged."""
    gn = lambda name: ".layers.1." in name or name.startswith("gn.")
    return {n: (np.asarray(v) * 2.0**k if not gn(n) else np.asarray(v)) for n, v in sd.items()}


@functools.lru_cache(maxsize=None)
def _primary_oracle(k):
    g, spec = load("roll128"), RN.NetSpec()
    sd = _scale_convs(load_weights("roll128"), k)
    inp, _ = RN.build_input(g["T0"][None, None], g["xc"], g["yc"], g["yc"], *PARAMS)
    x = torch.tensor(inp)
    r64 = RT.net_forward(RT.prepare_weights(sd, spec), spec, x)
    r32 = RT.net_forward(RT.prepare_weights(sd, spec, torch.float32), spec, x.float())
    noise = [relerr(a.double().numpy(), b.numpy()) for a, b in zip(r32, r64)]
    return sd, inp, [a.numpy() for a in r64], noise


@pytest.mark.parametrize("impl", ["ffma", "umma_3xtf32", "umma_f16x2", "row_f16x2", "mux_f16x2", "auto"])
@pytest.mark.parametrize("k", NET_SCALES)
def test_primary_network_with_scaled_weights(k, impl):
    sd, inp, ref, noise = _primary_oracle(k)
    spec = RN.NetSpec()
    net = P.NewFluidNet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p=spec.r_p, loss_type=spec.loss_type,
                        use_symm=spec.use_symm, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({n: torch.tensor(v) for n, v in sd.items()})
    net.conv_impl = impl
    net = net.to(DEV).eval()
    with torch.no_grad():
        out = net(torch.tensor(inp, device=DEV))
    errs = [relerr(o[0].cpu().numpy(), r[0]) for o, r in zip(out, ref)]
    print(f"[2^{k} {impl}] rel-L2 (u, v, p) {errs}; reference fp32 noise {noise}")
    for name, e, nz in zip("uvp", errs, noise):
        assert e <= field_bound(nz), (name, e, field_bound(nz))


@pytest.mark.parametrize("k", NET_SCALES)
def test_learned_network_with_scaled_weights(k):
    spec, inp, _, w = load_learned_case("learned_k5")
    sd = _scale_convs(w, k)
    u64, v64, _ = RN.learned_net_forward(sd, spec, inp)
    u32, v32, _ = RN.learned_net_forward({n: np.asarray(a, np.float32) for n, a in sd.items()}, spec, inp.astype(np.float32))
    noise = {"u": relerr(u32, u64), "v": relerr(v32, v64)}
    net = P.NewFluidNet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p="learned", loss_type="curl",
                        use_symm=False, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({n: torch.tensor(v) for n, v in sd.items()})
    net = net.to(DEV).eval()
    x = torch.tensor(inp, device=DEV)
    u, v, _, _ = net._engine(torch.device(DEV)).forward_blocked(ops.pack_nchw(x))
    errs = {"u": relerr(u.cpu().numpy(), u64), "v": relerr(v.cpu().numpy(), v64)}
    print(f"[learned_k5 2^{k}] fused engine rel-L2 {errs}; reference fp32 noise {noise}")
    for n in errs:
        assert errs[n] <= field_bound(noise[n]), (n, errs[n], noise[n])
    for call in range(3):  # the module call: eager, capture + replay, replay
        u, v, _ = net(x)
        errs = {"u": relerr(u.cpu().numpy(), u64), "v": relerr(v.cpu().numpy(), v64)}
        print(f"[learned_k5 2^{k}] net(x) call {call} rel-L2 {errs}")
        for n in errs:
            assert errs[n] <= field_bound(noise[n]), (call, n, errs[n], noise[n])


def test_ts_rollout_with_scaled_weights():
    """TS(ts=5) at 128 x 506 with every conv scaled by 2^-6, against the float64 rollout of the oracle; the bounds are
    those of tests/test_gpu_net.py with the reference's fp32 noise taken on the same scaled weights."""
    from tests.test_gpu_net import T_bound, _ts_call

    g, spec = load("ts128x506"), RN.NetSpec()
    sd = _scale_convs(load_weights("ts128x506"), -6)
    xc, yc = RN.synthetic_grid(128, 506)
    T0 = RN.synthetic_T0(128, 506, seed=int(g["T0_seed"]))

    def oracle(dtype):
        t = lambda a: torch.tensor(a, dtype=dtype)
        return RT.rollout(RT.prepare_weights(sd, spec, dtype), spec, t(T0)[None, None], t(xc), t(yc), *PARAMS, 5)

    T64, dts64, u64, v64, p64, _, _ = oracle(torch.float64)
    T32, dts32, u32, v32, p32, _, _ = oracle(torch.float32)
    nT = float((T32.double() - T64).abs().max())
    ndt = max(abs(a / b - 1) for a, b in zip(dts32, dts64))
    nf = {n: relerr(a.double().numpy(), b.numpy()) for n, a, b in (("u", u32, u64), ("v", v32, v64), ("p", p32, p64))}
    net = P.NewFluidNet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p=spec.r_p, loss_type=spec.loss_type,
                        use_symm=spec.use_symm, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({n: torch.tensor(v) for n, v in sd.items()})
    net = net.to(DEV).eval()
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=5, scale=True, p_pred=True, net="newfluidnet")
    x, dts, u, v, p, _ = _ts_call(ts, T0, xc, yc)
    eT = float(np.abs(x[5][0, 0].cpu().numpy() - T64[0, 0].numpy()).max())
    edt = max(abs(float(dts[i]) / dts64[i - 1] - 1) for i in range(1, 6))
    ef = {n: relerr(a[0, 0].cpu().numpy(), b[0].numpy()) for n, a, b in (("u", u, u64), ("v", v, v64), ("p", p, p64))}
    print(f"ts 2^-6: max|dT5| {eT:.2e} (noise {nT:.2e}), dt rel {edt:.2e} (noise {ndt:.2e}), fields {ef} (noise {nf})")
    assert eT <= T_bound(nT)
    assert edt <= max(3e-5, 1.5 * ndt)
    for n in ef:
        assert ef[n] <= field_bound(nf[n]), (n, ef[n], nf[n])
