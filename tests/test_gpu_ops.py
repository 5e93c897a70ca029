"""Operator-level parity on the GPU: every C-ABI kernel against the numpy oracle on the same
seeded inputs (float64 oracle, float32 kernels; tolerances are relative L2 unless noted)."""
import numpy as np
import pytest
import torch

from oracle import ref_numpy as RN
from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import ops
from tests._util import load, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float32, device=DEV)


def c64(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device=DEV)


def xco(xc):
    return ops.stencil_coefs(c64(xc[0]), 0.0, 4.0)


def yco(yc):
    return ops.stencil_coefs(c64(yc[:, 0]), 0.0, 1.0)


def rng(seed):
    return np.random.default_rng(seed)


def test_library_is_loaded_from_tree():
    lib = L.load()
    assert lib.pbmc_version() == 3 and L.LIB_PATH.endswith("pbml_mantle_convection_b200/libpbmc.so")


@pytest.mark.parametrize("shape", [(1, 7, 16, 16), (2, 16, 33, 50), (3, 1, 5, 7), (1, 103, 20, 24)])
def test_pack_unpack_roundtrip(shape):
    x = rng(0).standard_normal(shape).astype(np.float32)
    xb = ops.pack_nchw(cu(x))
    B, C, H, W = shape
    assert tuple(xb.shape) == (B, (C + 3) // 4, H, W, 4)
    ref = np.zeros((B, (C + 3) // 4 * 4, H, W), np.float32)
    ref[:, :C] = x
    ref = ref.reshape(B, -1, 4, H, W).transpose(0, 1, 3, 4, 2)
    assert np.array_equal(xb.cpu().numpy(), ref)
    assert np.array_equal(ops.unpack_nchw(xb, C).cpu().numpy(), x)


CONV_CASES = [
    # (B, Ci, Co, H, W, k, pad)
    (1, 16, 16, 40, 70, 3, "replicate"),
    (2, 16, 16, 8, 64, 3, "zeros"),
    (1, 16, 16, 37, 129, 3, "reflect"),
    (2, 7, 16, 19, 23, 3, "replicate"),
    (1, 16, 2, 24, 40, 3, "replicate"),
    (1, 8, 8, 17, 31, 3, "zeros"),
    (1, 16, 16, 21, 66, 5, "zeros"),
    (1, 16, 1, 12, 30, 5, "reflect"),
    (1, 32, 32, 16, 20, 3, "replicate"),
    (1, 16, 16, 3, 3, 3, "replicate"),
    (1, 16, 16, 1, 5, 3, "zeros"),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_plain(case):
    B, Ci, Co, H, W, k, pad = case
    r = rng(1)
    x = r.standard_normal((B, Ci, H, W))
    w = r.standard_normal((Co, Ci, k, k)) / np.sqrt(Ci * k * k)
    b = r.standard_normal(Co)
    ref = RN.conv2d_same(x, w, b, pad)
    wpk = ops.pack_conv_weight(cu(w), [Ci])
    out, stats, csum = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], wpk, ops.pad_vec(cu(b), Co, DEV), Co, k, pad,
                                    want_stats=True, want_chan_sum=True, impl="ffma")
    y = ops.unpack_nchw(out, Co).cpu().numpy()
    assert relerr(y, ref) < 2e-6
    # statistics: per (sample, 4-channel block) sum and sum of squares, per-channel sums
    cb = (Co + 3) // 4
    refp = np.zeros((B, cb * 4, H, W))
    refp[:, :Co] = ref
    rs = refp.reshape(B, cb, -1)
    st = stats.cpu().numpy()
    assert np.allclose(st[..., 0], rs.sum(-1), rtol=1e-5, atol=1e-4 * np.sqrt(rs.shape[-1]))
    assert np.allclose(st[..., 1], (rs**2).sum(-1), rtol=1e-5)
    assert np.allclose(csum.cpu().numpy(), refp.sum((2, 3)), rtol=1e-5, atol=1e-4 * np.sqrt(H * W))


UMMA_CASES = [
    (1, 16, 16, 40, 70, 3, "replicate"),
    (2, 16, 16, 15, 64, 3, "zeros"),
    (1, 16, 16, 37, 129, 3, "reflect"),
    (2, 7, 16, 19, 23, 3, "replicate"),
    (1, 16, 2, 24, 40, 3, "replicate"),
    (1, 8, 8, 17, 31, 3, "zeros"),
    (1, 16, 16, 21, 66, 5, "zeros"),
    (1, 16, 1, 12, 30, 5, "reflect"),
    (1, 32, 16, 16, 20, 3, "replicate"),
    (1, 16, 16, 3, 3, 3, "replicate"),
    (1, 16, 16, 1, 5, 3, "zeros"),
    (1, 16, 16, 128, 128, 3, "replicate"),
]


@pytest.mark.parametrize("impl,tol", [("umma_3xtf32", 3e-6), ("umma_f16x2", 3e-6), ("umma_bf16", 1e-2)])
@pytest.mark.parametrize("case", UMMA_CASES)
def test_conv_umma(case, impl, tol):
    """tcgen05 implicit-GEMM conv: the hi+lo split modes are fp32-grade against the float64 oracle;
    the single-pass bf16 mode carries its own (stated) bound: 2^-9 per operand -> <= 1e-2 rel-L2."""
    B, Ci, Co, H, W, k, pad = case
    r = rng(21)
    x = r.standard_normal((B, Ci, H, W))
    w = r.standard_normal((Co, Ci, k, k)) / np.sqrt(Ci * k * k)
    b = r.standard_normal(Co)
    ref = RN.conv2d_same(x, w, b, pad)
    wpk, wum = ops.pack_conv_weight(cu(w), [Ci]), ops.pack_conv_weight_umma(cu(w), [Ci])
    out, stats, csum = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], wpk, ops.pad_vec(cu(b), Co, DEV), Co, k, pad,
                                    want_stats=True, want_chan_sum=True, impl=impl, wpk_umma=wum)
    y = ops.unpack_nchw(out, Co).cpu().numpy()
    assert relerr(y, ref) < tol, relerr(y, ref)
    if impl == "umma_bf16":
        ref = y.astype(np.float64)  # statistics are checked against the kernel's own output
    cb = (Co + 3) // 4
    refp = np.zeros((B, cb * 4, H, W))
    refp[:, :Co] = ref
    rs = refp.reshape(B, cb, -1)
    st = stats.cpu().numpy()
    assert np.allclose(st[..., 0], rs.sum(-1), rtol=1e-5, atol=1e-4 * np.sqrt(rs.shape[-1]))
    assert np.allclose(st[..., 1], (rs**2).sum(-1), rtol=1e-5)
    assert np.allclose(csum.cpu().numpy(), refp.sum((2, 3)), rtol=1e-5, atol=1e-4 * np.sqrt(H * W))
    # lanes of the padded output channels stay exactly zero-biased (weights are zero there)
    if Co % 4:
        assert np.all(out[:, -1, :, :, Co % 4:].cpu().numpy() == 0)


ROW_CASES = UMMA_CASES + [
    (1, 4, 16, 9, 140, 3, "replicate"),      # one 4-channel block; two column strips
    (1, 12, 16, 30, 300, 3, "reflect"),      # three blocks; three strips, partial last strip
    (2, 40, 16, 70, 130, 3, "zeros"),        # three K groups, last one half full; many rows per CTA
    (1, 16, 16, 200, 256, 3, "replicate"),   # exact strips, accumulator ring wraps many times
    (1, 16, 16, 64, 128, 5, "replicate"),
    # >= 3 K groups per row: four producer groups + one epilogue set, merged hi*hi / hi*lo MMA (fp16 hi|lo, k = 3)
    (1, 48, 2, 33, 140, 3, "reflect"),       # c_out = 2 with the zero-mean channel sums, two strips
    (1, 64, 12, 20, 129, 3, "replicate"),    # three output blocks, one column in the second strip
    (1, 48, 16, 1, 5, 3, "zeros"),           # a single row
    (1, 103, 16, 150, 128, 3, "replicate"),  # conv[1]'s channel count; the 5-deep accumulator ring wraps many times
    (2, 48, 16, 40, 64, 5, "zeros"),         # k = 5 with three groups (four producer groups, passes not merged)
]


@pytest.mark.parametrize("impl,tol", [("row_f16x2", 3e-6), ("row_bf16", 1e-2)])
@pytest.mark.parametrize("case", ROW_CASES)
def test_conv_row(case, impl, tol):
    """Row-streaming warp-specialised tcgen05 conv (csrc/conv_row.cu): fp16 hi+lo split is fp32-grade
    against the float64 oracle; the single-pass bf16 mode carries its own stated bound."""
    B, Ci, Co, H, W, k, pad = case
    r = rng(23)
    x = r.standard_normal((B, Ci, H, W))
    w = r.standard_normal((Co, Ci, k, k)) / np.sqrt(Ci * k * k)
    b = r.standard_normal(Co)
    ref = RN.conv2d_same(x, w, b, pad)
    assert ops.row_supported(Co, k, [Ci])
    wpk, wrow = ops.pack_conv_weight(cu(w), [Ci]), ops.pack_conv_weight_row(cu(w), [Ci])
    want_cs = Co <= 4  # the row kernel produces the zero-mean channel sums only for the (c_out <= 4) head conv
    out, stats, csum = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], wpk, ops.pad_vec(cu(b), Co, DEV), Co, k, pad,
                                    want_stats=True, want_chan_sum=want_cs, impl=impl, wpk_row=wrow)
    y = ops.unpack_nchw(out, Co).cpu().numpy()
    assert relerr(y, ref) < tol, relerr(y, ref)
    if impl == "row_bf16":
        ref = y.astype(np.float64)
    cb = (Co + 3) // 4
    refp = np.zeros((B, cb * 4, H, W))
    refp[:, :Co] = ref
    rs = refp.reshape(B, cb, -1)
    st = stats.cpu().numpy()
    assert np.allclose(st[..., 0], rs.sum(-1), rtol=1e-5, atol=1e-4 * np.sqrt(rs.shape[-1]))
    assert np.allclose(st[..., 1], (rs**2).sum(-1), rtol=1e-5)
    if want_cs:
        assert np.allclose(csum.cpu().numpy(), refp.sum((2, 3)), rtol=1e-5, atol=1e-4 * np.sqrt(H * W))
    if Co % 4:
        assert np.all(out[:, -1, :, :, Co % 4:].cpu().numpy() == 0)


MUX_CASES = [
    (1, 16, 16, 17, 31, 3, "replicate"),
    (2, 16, 16, 40, 300, 3, "reflect"),      # three strips, partial last strip
    (1, 16, 16, 33, 128, 3, "zeros"),        # zero padding: out-of-image taps stay zero
    (1, 7, 16, 50, 140, 3, "replicate"),     # conv[0]: 7 input channels (two blocks, one lane empty)
    (1, 4, 16, 9, 140, 3, "zeros"),          # one block
    (1, 16, 2, 64, 64, 3, "replicate"),      # conv[3]: c_out = 2 with the zero-mean channel sums
    (1, 16, 16, 1, 5, 3, "zeros"),
    (1, 16, 16, 3, 3, 3, "replicate"),
    (3, 16, 16, 200, 256, 3, "replicate"),   # several waves; accumulator ring wraps
    (1, 16, 12, 23, 129, 3, "replicate"),    # one column in the second strip
]


@pytest.mark.parametrize("impl,tol", [("mux_f16x2", 3e-6), ("mux_bf16", 1e-2)])
@pytest.mark.parametrize("case", MUX_CASES)
def test_conv_mux(case, impl, tol):
    """Time-multiplexed row kernel (csrc/conv_mux.cu): same arithmetic as the row kernel, fp32-grade with
    the fp16 hi+lo split; single-pass bf16 with its stated bound."""
    B, Ci, Co, H, W, k, pad = case
    r = rng(29)
    x = r.standard_normal((B, Ci, H, W))
    w = r.standard_normal((Co, Ci, k, k)) / np.sqrt(Ci * k * k)
    b = r.standard_normal(Co)
    ref = RN.conv2d_same(x, w, b, pad)
    wpk, wrow = ops.pack_conv_weight(cu(w), [Ci]), ops.pack_conv_weight_row(cu(w), [Ci])
    want_cs = Co <= 4
    out, stats, csum = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], wpk, ops.pad_vec(cu(b), Co, DEV), Co, k, pad,
                                    want_stats=True, want_chan_sum=want_cs, impl=impl, wpk_row=wrow)
    y = ops.unpack_nchw(out, Co).cpu().numpy()
    assert relerr(y, ref) < tol, relerr(y, ref)
    if impl == "mux_bf16":
        ref = y.astype(np.float64)
    cb = (Co + 3) // 4
    refp = np.zeros((B, cb * 4, H, W))
    refp[:, :Co] = ref
    rs = refp.reshape(B, cb, -1)
    st = stats.cpu().numpy()
    assert np.allclose(st[..., 0], rs.sum(-1), rtol=1e-5, atol=1e-4 * np.sqrt(rs.shape[-1]))
    assert np.allclose(st[..., 1], (rs**2).sum(-1), rtol=1e-5)
    if want_cs:
        assert np.allclose(csum.cpu().numpy(), refp.sum((2, 3)), rtol=1e-5, atol=1e-4 * np.sqrt(H * W))
    if Co % 4:
        assert np.all(out[:, -1, :, :, Co % 4:].cpu().numpy() == 0)


@pytest.mark.parametrize("pad", ["replicate", "zeros", "reflect"])
@pytest.mark.parametrize("H,W", [(26, 45), (61, 200)])
def test_conv_mux_fused_groupnorm_gelu_and_epilogue_gelu(H, W, pad):
    """conv -> [GN+GELU folded into the mux kernel's row staging] -> conv + GELU epilogue (the conv[1] -> conv[2] shape)."""
    r = rng(31)
    B = 2
    x0 = r.standard_normal((B, 16, H, W))
    w1, b1 = r.standard_normal((16, 16, 3, 3)) / 12, r.standard_normal(16)
    g1, be1 = 1 + 0.2 * r.standard_normal(16), 0.2 * r.standard_normal(16)
    w2, b2 = r.standard_normal((16, 16, 3, 3)) / 12, r.standard_normal(16)
    y1 = RN.conv2d_same(x0, w1, b1, pad)
    a1 = RN.gelu(RN.group_norm(y1, g1, be1, 4))
    ref = RN.gelu(RN.conv2d_same(a1, w2, b2, pad))
    y1b, st1, _ = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x0)))], ops.pack_conv_weight(cu(w1), [16]), ops.pad_vec(cu(b1), 16, DEV),
                               16, 3, pad, want_stats=True, impl="mux_f16x2", wpk_row=ops.pack_conv_weight_row(cu(w1), [16]))
    assert relerr(ops.unpack_nchw(y1b, 16).cpu().numpy(), y1) < 3e-6
    out, _, _ = ops.conv_fwd([ops.Source(y1b, L.XFORM_GN_GELU, st1, cu(g1), cu(be1))], ops.pack_conv_weight(cu(w2), [16]),
                             ops.pad_vec(cu(b2), 16, DEV), 16, 3, pad, epi_act=L.ACT_GELU, impl="mux_f16x2",
                             wpk_row=ops.pack_conv_weight_row(cu(w2), [16]))
    assert relerr(ops.unpack_nchw(out, 16).cpu().numpy(), ref) < 5e-6


def _conv_37x150(impl, max_ctas):
    """One 16 -> 16 3x3 conv of a 37 x 150 field (two 128-column strips) under a CTA budget, against the float64 oracle."""
    r = rng(5)
    x, w, b = r.standard_normal((1, 16, 37, 150)), r.standard_normal((16, 16, 3, 3)) / 12, r.standard_normal(16)
    out, _, _ = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], ops.pack_conv_weight(cu(w), [16]), ops.pad_vec(cu(b), 16, DEV),
                             16, 3, "replicate", impl=impl, wpk_row=ops.pack_conv_weight_row(cu(w), [16]), max_ctas=max_ctas)
    err = relerr(ops.unpack_nchw(out, 16).cpu().numpy(), RN.conv2d_same(x, w, b, "replicate"))
    assert err < 3e-6, err


# CTA budget -> the rows per CTA that choose_rpc_mux (csrc/conv_mux.cu) picks for 2 strips x 37 rows: 1, 2, 3, 4, 5, 6, 7, 8,
# 10, 13 and 19 rows, i.e. one to five staging rounds of the five worker groups and a TMEM accumulator ring (10) that wraps
@pytest.mark.parametrize("max_ctas", [148, 38, 26, 20, 16, 14, 12, 10, 8, 6, 2])
def test_conv_mux_any_rows_per_cta(max_ctas):
    """Rows per CTA is a scheduling choice: the mux kernel gives the same result for any of them."""
    _conv_37x150("mux_f16x2", max_ctas)


# CTA budget -> rows per CTA of choose_rpc (csrc/conv_row.cu), the smallest r with 2 * ceil(37 / r) <= budget: 1, 2, 3, 10 and
# 37 rows; from 7 rows on the 8-stage operand ring wraps, from 9 rows on the 10-accumulator ring as well
@pytest.mark.parametrize("max_ctas", [148, 38, 26, 8, 2])
def test_conv_row_any_rows_per_cta(max_ctas):
    """The strip decomposition (rows per CTA) is a scheduling choice: results must not depend on it."""
    _conv_37x150("row_f16x2", max_ctas)


def test_conv_gelu_epilogue():
    r = rng(2)
    x, w, b = r.standard_normal((1, 16, 20, 30)), r.standard_normal((16, 16, 3, 3)) / 12, r.standard_normal(16)
    ref = RN.gelu(RN.conv2d_same(x, w, b, "replicate"))
    out, _, _ = ops.conv_fwd([ops.Source(ops.pack_nchw(cu(x)))], ops.pack_conv_weight(cu(w), [16]), ops.pad_vec(cu(b), 16, DEV),
                             16, 3, "replicate", epi_act=L.ACT_GELU, impl="ffma")
    assert relerr(ops.unpack_nchw(out, 16).cpu().numpy(), ref) < 2e-6


@pytest.mark.parametrize("Co,pad", [(16, "replicate"), (3, "zeros")])
def test_conv_row_several_groups_gelu_epilogue_and_channel_sums(Co, pad):
    """The several-groups variant of the row kernel (merged MMA passes, 96-column accumulators read in two halves) with
    everything its epilogue can be asked for: GELU, partial output blocks, GroupNorm sums, zero-mean channel sums."""
    r = rng(31)
    B, H, W, chans = 2, 37, 150, [16, 16, 16, 7]
    xs = [r.standard_normal((B, c, H, W)) for c in chans]
    w, b = r.standard_normal((Co, sum(chans), 3, 3)) / 20, r.standard_normal(Co)
    ref = RN.gelu(RN.conv2d_same(np.concatenate(xs, 1), w, b, pad))
    srcs = [ops.Source(ops.pack_nchw(cu(x))) for x in xs]
    out, stats, csum = ops.conv_fwd(srcs, ops.pack_conv_weight(cu(w), chans), ops.pad_vec(cu(b), Co, DEV), Co, 3, pad,
                                    epi_act=L.ACT_GELU, want_stats=True, want_chan_sum=Co <= 4, impl="row_f16x2",
                                    wpk_row=ops.pack_conv_weight_row(cu(w), chans))
    y = ops.unpack_nchw(out, Co).cpu().numpy()
    assert relerr(y, ref) < 3e-6, relerr(y, ref)
    cb = (Co + 3) // 4
    refp = np.zeros((B, cb * 4, H, W))
    refp[:, :Co] = ref
    rs = refp.reshape(B, cb, -1)
    st = stats.cpu().numpy()
    assert np.allclose(st[..., 0], rs.sum(-1), rtol=1e-5, atol=1e-4 * np.sqrt(rs.shape[-1]))
    assert np.allclose(st[..., 1], (rs**2).sum(-1), rtol=1e-5)
    if Co <= 4:
        assert np.allclose(csum.cpu().numpy(), refp.sum((2, 3)), rtol=1e-5, atol=1e-4 * np.sqrt(H * W))


@pytest.mark.parametrize("impl", ["ffma", "umma_3xtf32", "umma_f16x2", "row_f16x2", "mux_f16x2"])
def test_fluid_layer_chain_with_fused_groupnorm_and_concat(impl):
    """conv -> [GN+GELU fused into the next load] -> conv over a 3-source concat (one plain source)."""
    r = rng(3)
    B, H, W = 2, 26, 45
    x0 = r.standard_normal((B, 16, H, W))
    xin = r.standard_normal((B, 7, H, W))
    w1, b1 = r.standard_normal((16, 16, 3, 3)) / 12, r.standard_normal(16)
    g1, be1 = 1 + 0.2 * r.standard_normal(16), 0.2 * r.standard_normal(16)
    w2, b2 = r.standard_normal((16, 39, 3, 3)) / 18, r.standard_normal(16)
    y1 = RN.conv2d_same(x0, w1, b1, "replicate")
    a1 = RN.gelu(RN.group_norm(y1, g1, be1, 4))
    ref = RN.conv2d_same(np.concatenate([a1, x0, xin], 1), w2, b2, "replicate")

    x0b, xinb = ops.pack_nchw(cu(x0)), ops.pack_nchw(cu(xin))
    y1b, st1, _ = ops.conv_fwd([ops.Source(x0b)], ops.pack_conv_weight(cu(w1), [16]), ops.pad_vec(cu(b1), 16, DEV), 16, 3,
                               "replicate", want_stats=True, impl=impl, wpk_umma=ops.pack_conv_weight_umma(cu(w1), [16]),
                               wpk_row=ops.pack_conv_weight_row(cu(w1), [16]))
    srcs = [ops.Source(y1b, L.XFORM_GN_GELU, st1, cu(g1), cu(be1)), ops.Source(x0b), ops.Source(xinb)]
    out, _, _ = ops.conv_fwd(srcs, ops.pack_conv_weight(cu(w2), [16, 16, 7]), ops.pad_vec(cu(b2), 16, DEV), 16, 3,
                             "replicate", impl=impl, wpk_umma=ops.pack_conv_weight_umma(cu(w2), [16, 16, 7]),
                             wpk_row=ops.pack_conv_weight_row(cu(w2), [16, 16, 7]))
    assert relerr(ops.unpack_nchw(out, 16).cpu().numpy(), ref) < 5e-6
    # stand-alone finalize == GN + GELU
    fin = ops.finalize_nchw(ops.Source(y1b, L.XFORM_GN_GELU, st1, cu(g1), cu(be1)), 16).cpu().numpy()
    assert relerr(fin, a1) < 3e-6


def _decode_staged(buf, B, H, W):
    """PBMC_LAYOUT_STAGED16 -> (hi + lo) as [B, 16, H, W+2] float64 (columns -1 .. W) and the raw halves."""
    Wp = (W + 127) // 128 * 128 + 2
    h = buf.view(torch.float16).view(B, H, 2, 2, Wp, 8)[:, :, :, :, :W + 2]          # [B, H, part, chunk, pos, 8]
    v = h.double().permute(0, 2, 3, 5, 1, 4).reshape(B, 2, 16, H, W + 2)            # [B, part, ch, H, pos]
    return (v[:, 0] + v[:, 1]).cpu().numpy(), h


@pytest.mark.parametrize("hs,ws,H,W", [(15, 31, 50, 77), (64, 64, 128, 128), (63, 126, 128, 506), (8, 8, 8, 8)])
def test_bicubic_staged_layout(hs, ws, H, W):
    """The up-sampled levels written as conv[1]'s operand image: hi + lo reproduces the blocked fp32 result to fp16^2
    precision, and positions 0 / W+1 hold the replicate-padded columns."""
    r = rng(41)
    x = r.standard_normal((2, 16, hs, ws))
    src = ops.Source(ops.pack_nchw(cu(x)))
    ref = ops.unpack_nchw(ops.bicubic_up(src, H, W), 16).cpu().numpy().astype(np.float64)
    st = ops.bicubic_up(src, H, W, staged=True)
    got, _ = _decode_staged(st.t, 2, H, W)
    assert np.abs(got[..., 1:W + 1] - ref).max() <= 2.0 ** -21 * max(1.0, np.abs(ref).max())
    assert np.array_equal(got[..., 0], got[..., 1]) and np.array_equal(got[..., W + 1], got[..., W])


@pytest.mark.parametrize("B,H,W", [(1, 40, 130), (2, 33, 256), (1, 70, 300)])
def test_conv_row_staged_sources_bit_identical(B, H, W):
    """conv[1]'s shape: [GN+GELU level 0, up-sampled levels, raw inputs].  With the up-sampled levels given as
    operand images (bulk-copied into the stage by the TMA engine) the result is bit-identical to the blocked path,
    and both match the float64 oracle."""
    r = rng(43)
    x0 = r.standard_normal((B, 16, H, W))
    lv = [r.standard_normal((B, 16, H // 2, W // 2)), r.standard_normal((B, 16, H // 4, W // 4))]
    xin = r.standard_normal((B, 7, H, W))
    g0, be0 = 1 + 0.2 * r.standard_normal(16), 0.2 * r.standard_normal(16)
    w, b = r.standard_normal((16, 55, 3, 3)) / 22, r.standard_normal(16)
    x0b = ops.pack_nchw(cu(x0))
    st0 = torch.stack([x0b.double().sum((2, 3, 4)), (x0b.double() ** 2).sum((2, 3, 4))], -1).contiguous()
    lsrc = [ops.Source(ops.pack_nchw(cu(a))) for a in lv]
    ups_b = [ops.Source(ops.bicubic_up(s_, H, W)) for s_ in lsrc]
    ups_s = [ops.bicubic_up(s_, H, W, staged=True) for s_ in lsrc]
    first, last = ops.Source(x0b, L.XFORM_GN_GELU, st0, cu(g0), cu(be0)), ops.Source(ops.pack_nchw(cu(xin)))
    ch = [16, 16, 16, 7]
    wpk, wrow = ops.pack_conv_weight(cu(w), ch), ops.pack_conv_weight_row(cu(w), ch)
    outs = []
    for ups in (ups_b, ups_s):
        o, stt, _ = ops.conv_fwd([first, *ups, last], wpk, ops.pad_vec(cu(b), 16, DEV), 16, 3, "replicate", want_stats=True,
                                 impl="row_f16x2", wpk_row=wrow)
        outs.append((o.clone(), stt.clone()))
    assert torch.equal(outs[0][0], outs[1][0])
    a0 = RN.gelu(RN.group_norm(x0, g0, be0, 4))
    upr = [ops.unpack_nchw(u_.t, 16).cpu().numpy().astype(np.float64) for u_ in ups_b]
    ref = RN.conv2d_same(np.concatenate([a0, *upr, xin], 1), w, b, "replicate")
    assert relerr(ops.unpack_nchw(outs[1][0], 16).cpu().numpy(), ref) < 5e-6
    # the other kernels refuse the operand-image layout instead of misreading it
    with pytest.raises(L.PbmcError):
        ops.conv_fwd([first, *ups_s, last], wpk, ops.pad_vec(cu(b), 16, DEV), 16, 3, "replicate", impl="ffma")
    with pytest.raises(L.PbmcError):
        ops.conv_fwd([first, *ups_s, last], wpk, ops.pad_vec(cu(b), 16, DEV), 16, 3, "zeros", impl="row_f16x2", wpk_row=wrow)


@pytest.mark.parametrize("H,W", [(16, 16), (15, 31), (50, 77), (2, 3)])
def test_avgpool_floor(H, W):
    x = rng(4).standard_normal((2, 16, H, W))
    out = ops.avgpool2(ops.Source(ops.pack_nchw(cu(x))))
    assert tuple(out.shape) == (2, 4, H // 2, W // 2, 4)
    assert relerr(ops.unpack_nchw(out, 16).cpu().numpy(), RN.avg_pool2(x)) < 1e-6


def test_avgpool_with_fused_groupnorm():
    r = rng(5)
    x = r.standard_normal((2, 16, 20, 34)) * 3 + 1
    g, be = 1 + 0.2 * r.standard_normal(16), 0.2 * r.standard_normal(16)
    ref = RN.avg_pool2(RN.gelu(RN.group_norm(x, g, be, 4)))
    xb = ops.pack_nchw(cu(x))
    st = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
    out = ops.avgpool2(ops.Source(xb, L.XFORM_GN_GELU, st, cu(g), cu(be)))
    assert relerr(ops.unpack_nchw(out, 16).cpu().numpy(), ref) < 3e-6


@pytest.mark.parametrize("hs,ws,H,W", [(15, 31, 50, 77), (64, 64, 128, 128), (4, 15, 128, 506), (8, 8, 8, 8), (1, 1, 9, 9),
                                       (63, 126, 128, 506)])
def test_bicubic(hs, ws, H, W):
    x = rng(6).standard_normal((1, 8, hs, ws))
    out = ops.bicubic_up(ops.Source(ops.pack_nchw(cu(x))), H, W)
    y = ops.unpack_nchw(out, 8).cpu().numpy()
    assert relerr(y, RN.bicubic_upsample(x, (H, W))) < 3e-6


def test_bicubic_matches_golden_torch():
    g = load("ops")
    out = ops.bicubic_up(ops.Source(ops.pack_nchw(cu(g["bic_x"]))), 50, 77)
    assert relerr(ops.unpack_nchw(out, 3).cpu().numpy(), g["bic_y"]) < 3e-6
    pl = ops.avgpool2(ops.Source(ops.pack_nchw(cu(g["bic_x"]))))
    assert relerr(ops.unpack_nchw(pl, 3).cpu().numpy(), g["pool_y"]) < 1e-6


def test_build_input():
    H, W, B = 40, 56, 3
    xc, yc = RN.synthetic_grid(H, W)
    prm = [(6.79733173, 475523342.0, 2.58574662), (0.5, 1.2e6, 1.1), (9.0, 7e9, 90.0)]
    T = np.stack([RN.synthetic_T0(H, W, seed=s) for s in range(B)])
    T[1] *= 1.7  # exercise the clip(V, 1e-8, 1) branches
    members = ops.make_members(prm, DEV)
    inp, V = ops.build_input(cu(T), cu(xc), cu(yc), cu(yc), members, want_V=True)
    got = ops.unpack_nchw(inp, 7).cpu().numpy()
    for b in range(B):
        ref, Vr = RN.build_input(T[b][None, None], xc, yc, yc, *prm[b])
        assert np.abs(got[b] - ref[0]).max() < 3e-6
        assert np.abs(V[b].cpu().numpy() - Vr[0, 0]).max() < 2e-6
    assert np.all(inp[:, 1, :, :, 3].cpu().numpy() == 0)


@pytest.mark.parametrize("H,W", [(20, 28), (33, 65), (3, 3)])
def test_head_curl(H, W):
    r = rng(7)
    B = 2
    y = r.standard_normal((B, 2, H, W))
    spec = RN.NetSpec()
    u_ref, v_ref, p_ref = RN.curl_head(y.copy(), spec)
    prm = [(6.79733173, 475523342.0, 2.58574662), (1.0, 1e7, 2.0)]
    members = ops.make_members(prm, DEV)
    yb = ops.pack_nchw(cu(y))
    csum = torch.tensor(np.pad(y.sum((2, 3)), ((0, 0), (0, 2))), dtype=torch.float64, device=DEV)
    u, v, p, uvmax = ops.head(yb, csum, members, spec.a_bound, L.HEAD_CURL, True)
    for b in range(B):
        s = RN.velocity_scaler(*prm[b])
        assert np.abs(u[b].cpu().numpy() - u_ref[b] * s).max() <= 2e-6 * np.abs(u_ref[b] * s).max() + 1e-30
        assert np.abs(v[b].cpu().numpy() - v_ref[b] * s).max() <= 2e-6 * np.abs(v_ref[b] * s).max() + 1e-30
        assert np.abs(p[b].cpu().numpy() - p_ref[b]).max() < 1e-5
        if H > 2 and W > 2:
            m = max(np.abs(u_ref[b, 1:-1, 1:-1]).max(), np.abs(v_ref[b, 1:-1, 1:-1]).max()) * s
            got = uvmax[b:b + 1].view(torch.float32).item()
            assert abs(got - m) <= 2e-6 * m
    # wall structure is exact
    un = u.cpu().numpy()
    assert np.all(un[:, 1:-1, 0] == -un[:, 1:-1, 1])
    assert np.all(un[:, 0, 0] == 0) and np.all(v.cpu().numpy()[:, -1, -1] == 0)


def test_head_mae():
    r = rng(8)
    y = r.standard_normal((2, 3, 12, 20))
    yb = ops.pack_nchw(cu(y))
    csum = torch.tensor(np.pad(y.sum((2, 3)), ((0, 0), (0, 1))), dtype=torch.float64, device=DEV)
    u, v, p, _ = ops.head(yb, csum, None, 10.0, L.HEAD_MAE, True, want_uvmax=False)
    ym = y - y.mean((2, 3), keepdims=True)
    assert np.abs(u.cpu().numpy() - ym[:, 0]).max() < 1e-5 and np.abs(p.cpu().numpy() - ym[:, 2]).max() < 1e-5


def _adnet_case(H, W, B, seed, scale=50.0):
    r = rng(seed)
    xc, yc = RN.synthetic_grid(H, W)
    u = r.standard_normal((B, H, W)) * scale
    v = r.standard_normal((B, H, W)) * scale
    u[0, min(5, H - 2), min(5, W - 2)] = 0.0
    T = r.random((B, H, W))
    return xc, yc, u, v, T


@pytest.mark.parametrize("H,W,B", [(40, 56, 2), (33, 65, 1), (128, 506, 1), (3, 3, 1), (64, 512, 2), (35, 130, 1)])
def test_stencil_vs_oracle(H, W, B):
    """fast separable kernel (vector path when W % 4 == 0) incl. the fused CFL reduction."""
    xc, yc, u, v, T = _adnet_case(H, W, B, 9)
    raq = 3.5
    members = ops.make_members([(raq, 1e7, 2.0)] * B, DEV)
    uvmax = ops.uvmax_reduce(cu(u), cu(v), batch_global=True)
    xf = xc.copy()
    xf[:, 0], xf[:, -1] = 0, 4
    dx_min = (xf[1:-1, 1:-1] - xf[1:-1, :-2]).min() if W > 2 else 1.0
    Tn, dt, uv_out = ops.advect_diffuse(cu(T), cu(u), cu(v), xco(xc), yco(yc), members, uvmax, dx_min, 0.99,
                                        per_member_dt=False, want_uvmax_out=True)
    # oracle in float64 on the float32-rounded inputs (isolates kernel arithmetic from input rounding)
    f = lambda a: a.astype(np.float32).astype(np.float64)
    Tr, dtr = RN.adnet_forward(f(u), f(v), f(T), np.float64(np.float32(raq)), xc, yc, 0.99)
    Tr = RN.apply_T_bcs(Tr)
    assert abs(dt[0].item() - dtr) <= 1e-6 * dtr
    got = Tn.cpu().numpy()
    # upwind switches at u == 0 exactly, inputs are identical => same branch everywhere
    assert np.abs(got - Tr).max() < 5e-6 * max(1.0, np.abs(Tr).max())
    m = max(np.abs(f(u)[:, 1:-1, 1:-1]).max(), np.abs(f(v)[:, 1:-1, 1:-1]).max())
    assert uv_out.view(torch.float32)[0].item() == pytest.approx(m, rel=1e-7)
    # wall structure
    assert np.all(got[:, 0, :] == 1) and np.all(got[:, -1, :] == 0)
    assert np.all(got[:, 1:-1, 0] == got[:, 1:-1, 1]) and np.all(got[:, 1:-1, -1] == got[:, 1:-1, -2])


def test_stencil_golden_reference():
    """against vectors produced by the reference's ADNet itself (B=2, batch-global dt; fixed dt)."""
    g = load("ops")
    u, v, T = g["ad_u"][:, 0], g["ad_v"][:, 0], g["ad_T"][:, 0]
    xc, yc = g["ad_xc"], g["ad_yc"]
    members = ops.make_members([(float(g["ad_raq"]), 1e7, 2.0)] * 2, DEV)
    uvmax = ops.uvmax_reduce(cu(u), cu(v), batch_global=True)
    xf = xc.copy()
    xf[:, 0], xf[:, -1] = 0, 4
    dx_min = (xf[1:-1, 1:-1] - xf[1:-1, :-2]).min()
    Tn, dt, _ = ops.advect_diffuse(cu(T), cu(u), cu(v), xco(xc), yco(yc), members, uvmax, dx_min, 0.99,
                                   per_member_dt=False)
    assert abs(dt[0].item() - float(g["ad_dt"])) < 1e-6 * float(g["ad_dt"])
    assert np.abs(Tn.cpu().numpy() - g["ad_Tn"][:, 0]).max() < 2e-5  # float32 inputs: |u| dt/dx ~ 0.5 => ~1e-6 expected
    Tn2, dt2, _ = ops.advect_diffuse(cu(T), cu(u), cu(v), xco(xc), yco(yc), members, None, dx_min, 0.99,
                                     per_member_dt=False, dt_fixed=1e-4)
    assert dt2[0].item() == 1e-4
    assert np.abs(Tn2.cpu().numpy() - g["ad_Tn_fixed_dt"][:, 0]).max() < 2e-4
    # general-fields kernel gives the same answer
    dxm = torch.tensor([dx_min], dtype=torch.float64, device=DEV)
    Tn3, dt3 = ops.advect_diffuse_fields(cu(T), cu(u), cu(v), c64(xc), c64(yc), None, members, uvmax, dxm, 0.99)
    assert np.abs(Tn3.cpu().numpy() - Tn.cpu().numpy()).max() < 2e-6 and dt3[0].item() == dt[0].item()


def test_stencil_per_member_dt():
    H, W, B = 32, 64, 3
    xc, yc, u, v, T = _adnet_case(H, W, B, 10)
    u[1] *= 10
    v[2] *= 0.01
    u[2] *= 0.01
    members = ops.make_members([(1.0, 1e7, 2.0), (2.0, 1e7, 2.0), (3.0, 1e7, 2.0)], DEV)
    uvmax = ops.uvmax_reduce(cu(u), cu(v), batch_global=False)
    xf = xc.copy()
    xf[:, 0], xf[:, -1] = 0, 4
    dx_min = (xf[1:-1, 1:-1] - xf[1:-1, :-2]).min()
    Tn, dt, _ = ops.advect_diffuse(cu(T), cu(u), cu(v), xco(xc), yco(yc), members, uvmax, dx_min, 0.99,
                                   per_member_dt=True)
    f = lambda a: a.astype(np.float32).astype(np.float64)
    for b in range(B):
        Tr, dtr = RN.adnet_forward(f(u[b:b + 1]), f(v[b:b + 1]), f(T[b:b + 1]), float(b + 1), xc, yc, 0.99)
        assert abs(dt[b].item() - dtr) <= 1e-6 * dtr
        assert np.abs(Tn[b].cpu().numpy() - RN.apply_T_bcs(Tr)[0]).max() < 5e-6


def test_stencil_large_grid_properties():
    """BASELINE config 3 size (8192^2): properties that need no oracle run -- zero velocity
    and linear T(y) on the non-uniform grid is a fixed point of the diffusion operator; wall
    rows/columns exact; CFL reduction equals torch's own max."""
    H = W = 8192
    xc, yc = RN.synthetic_grid(H, W)
    y1 = cu(yc[:, 0])
    T = (1.0 - y1)[None, :, None].expand(1, H, W).contiguous()
    z = torch.zeros(1, H, W, device=DEV)
    members = ops.make_members([(0.0, 1e7, 2.0)], DEV)
    uv = torch.zeros(1, dtype=torch.int32, device=DEV)
    dx_min = 2.0 / (W - 2)
    Tn, dt, _ = ops.advect_diffuse(T, z, z, xco(xc), yco(yc), members, uv, dx_min, 0.99)
    assert dt[0].item() == pytest.approx(0.25 * dx_min**2, rel=1e-12)  # diffusive limit when max|u| = 0
    assert (Tn[0, 1:-1, 1:-1] - T[0, 1:-1, 1:-1]).abs().max().item() < 1e-6
    assert torch.all(Tn[0, 0] == 1) and torch.all(Tn[0, -1] == 0)
    u = torch.randn(1, H, W, device=DEV) * 1e5  # fast enough that the advective limit binds at this resolution
    v = torch.randn(1, H, W, device=DEV) * 1e5
    Tn2, dt2, uvo = ops.advect_diffuse(T, u, v, xco(xc), yco(yc), members, ops.uvmax_reduce(u, v), dx_min, 0.99,
                                       want_uvmax_out=True)
    m = max(u[0, 1:-1, 1:-1].abs().max().item(), v[0, 1:-1, 1:-1].abs().max().item())
    assert uvo.view(torch.float32)[0].item() == m
    assert 0.5 * 0.99 * dx_min / m < 0.25 * dx_min**2
    assert dt2[0].item() == pytest.approx(0.5 * 0.99 * dx_min / m, rel=1e-6)
    assert torch.all(Tn2[0, 1:-1, 0] == Tn2[0, 1:-1, 1]) and torch.isfinite(Tn2).all()


def test_clamp_and_diagnostics():
    r = rng(11)
    T = r.standard_normal((2, 30, 44)) * 2
    t = cu(T)
    ops.clamp_T(t)
    ref = T.astype(np.float32).copy()
    ref[:, 0, :], ref[:, -1, :] = 1, 0
    ref[:, :, 0], ref[:, :, -1] = ref[:, :, 1], ref[:, :, -2]
    ref = np.clip(ref, 0, 2)
    assert np.array_equal(t.cpu().numpy(), ref)
    mean, prof = ops.diagnostics(t)
    assert np.allclose(prof.cpu().numpy(), ref.astype(np.float64).mean(-1), rtol=1e-12)
    assert np.allclose(mean.cpu().numpy(), ref.astype(np.float64).mean((1, 2)), rtol=1e-12)


def test_error_codes_on_device():
    x = torch.zeros(1, 1, 8, 8, 4, device=DEV)
    with pytest.raises(L.PbmcError, match="unsupported"):
        ops.conv_fwd([ops.Source(x)], torch.zeros(1, 1, 49, 4, 16, device=DEV), torch.zeros(4, device=DEV), 4, 7, "zeros")
    with pytest.raises(L.PbmcError):  # reflect needs size > pad
        ops.conv_fwd([ops.Source(torch.zeros(1, 1, 1, 8, 4, device=DEV))], torch.zeros(1, 1, 9, 4, 16, device=DEV),
                     torch.zeros(4, device=DEV), 4, 3, "reflect")


class _Lay:
    """Minimal stand-in for engine._PackedLayer (what ops.trunk_fwd reads)."""

    def __init__(self, w, b, g, be):
        self.wpk = ops.pack_conv_weight(cu(w), [16])
        self.wpk_row = ops.pack_conv_weight_row(cu(w), [16])
        self.bias, self.gamma, self.beta = ops.pad_vec(cu(b), 16, DEV), cu(g).float().contiguous(), cu(be).float().contiguous()
        self.cin_blks, self.cout, self.ksize = 4, 16, 3


@pytest.mark.parametrize("B,H,W,R,pad,xform0,max_ctas", [
    (1, 40, 130, 4, "replicate", True, 0), (2, 33, 256, 3, "zeros", False, 0), (1, 70, 300, 4, "reflect", True, 0),
    (1, 64, 64, 4, "replicate", True, 3), (1, 7, 9, 2, "replicate", True, 2), (3, 50, 77, 1, "replicate", False, 0),
    (1, 128, 128, 6, "replicate", True, 0)])
@pytest.mark.parametrize("loader", ["threads", "bulk"])
def test_trunk_persistent_kernel(B, H, W, R, pad, xform0, max_ctas, loader):
    """pbmc_trunk_fwd: R FluidLayers (conv -> GroupNorm -> GELU, pytorch_networks_convae.py:790-799, :1323-1324) in one
    persistent launch with a grid-wide barrier per layer, against (a) the float64 numpy oracle and (b) the same layers
    launched one by one through pbmc_conv_fwd (same arithmetic per output; only the order of the double-precision
    statistics atomics differs)."""
    r = rng(100 + H + R)
    x = r.standard_normal((B, 16, H, W))
    ws = [r.standard_normal((16, 16, 3, 3)) / 12 for _ in range(R)]
    bs = [0.3 * r.standard_normal(16) for _ in range(R)]
    gs = [1 + 0.2 * r.standard_normal(16) for _ in range(R)]
    bes = [0.2 * r.standard_normal(16) for _ in range(R)]
    g0, be0 = 1 + 0.2 * r.standard_normal(16), 0.2 * r.standard_normal(16)
    # oracle
    a = RN.gelu(RN.group_norm(x, g0, be0, 4)) if xform0 else x
    raws = []
    for i in range(R):
        y = RN.conv2d_same(a, ws[i], bs[i], pad)
        raws.append(y)
        a = RN.gelu(RN.group_norm(y, gs[i], bes[i], 4))
    lays = [_Lay(ws[i], bs[i], gs[i], bes[i]) for i in range(R)]
    xb = ops.pack_nchw(cu(x))
    if xform0:
        st0 = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
        src = ops.Source(xb, L.XFORM_GN_GELU, st0, cu(g0).float(), cu(be0).float())
    else:
        src = ops.Source(xb)
    out, st_last, st_all = ops.trunk_fwd(src, lays, pad, impl="mux_f16x2", max_ctas=max_ctas, loader=loader)
    got = ops.unpack_nchw(out, 16).cpu().numpy()
    assert relerr(got, raws[-1]) < 6e-6, relerr(got, raws[-1])
    ref_st = np.stack([raws[-1].reshape(B, 4, -1).sum(-1), (raws[-1] ** 2).reshape(B, 4, -1).sum(-1)], -1)
    assert np.allclose(st_last.cpu().numpy(), ref_st, rtol=2e-5, atol=1e-4 * H * W)
    fin = ops.finalize_nchw(ops.Source(out, L.XFORM_GN_GELU, st_last, lays[-1].gamma, lays[-1].beta), 16).cpu().numpy()
    assert relerr(fin, a) < 6e-6
    # layer by layer through pbmc_conv_fwd
    s = src
    for i in range(R):
        yb, sti, _ = ops.conv_fwd([s], lays[i].wpk, lays[i].bias, 16, 3, pad, want_stats=True, impl="mux_f16x2", wpk_row=lays[i].wpk_row)
        # (per-thread partial sums are float32 and the rows per CTA differ between the two kernels: ~1e-7 relative)
        assert np.allclose(st_all[i].cpu().numpy(), sti.cpu().numpy(), rtol=3e-6, atol=3e-6 * H * W)
        s = ops.Source(yb, L.XFORM_GN_GELU, sti, lays[i].gamma, lays[i].beta)
    assert (yb - out).abs().max().item() <= 2e-6 * max(1.0, float(yb.abs().max()))
    # twice in a row: scratch is re-zeroed by the call, same result bit for bit up to the statistics' atomic order
    out2, _, _ = ops.trunk_fwd(src, lays, pad, impl="mux_f16x2", max_ctas=max_ctas, loader=loader)
    if loader == "bulk":  # the two loaders feed the same arithmetic
        out3, _, _ = ops.trunk_fwd(src, lays, pad, impl="mux_f16x2", max_ctas=max_ctas, loader="threads")
        assert (out3 - out).abs().max().item() <= 2e-6 * max(1.0, float(out.abs().max()))
    assert (out2 - out).abs().max().item() <= 2e-6 * max(1.0, float(out.abs().max()))


def test_trunk_refuses_a_grid_that_cannot_be_resident():
    lays = [_Lay(np.zeros((16, 16, 3, 3)), np.zeros(16), np.ones(16), np.zeros(16))]
    x = torch.zeros(1, 4, 512, 512, 4, device=DEV)
    with pytest.raises(L.PbmcError):
        ops.trunk_fwd(ops.Source(x), lays, "replicate", max_ctas=8)  # 4 strips x >= 24 chunks of <= 22 rows


@pytest.mark.parametrize("k,chans,cout,B,H,W,epi_gelu,csum", [
    (3, [16], 16, 2, 40, 52, False, False), (5, [16], 16, 1, 37, 130, False, False), (5, [16, 16, 16, 7], 16, 1, 20, 28, False, False),
    (3, [7], 16, 2, 9, 11, False, False), (5, [16], 16, 1, 6, 6, True, False), (5, [16], 1, 2, 24, 31, False, True),
    (3, [16], 2, 1, 33, 140, False, True), (5, [87], 16, 1, 16, 20, False, False)])
def test_conv_learned9_two_launches(k, chans, cout, B, H, W, epi_gelu, csum):
    """BoundaryLearnedConvolution2D (pytorch_networks_convae.py:1022-1065, bc = 1) as pbmc_conv_fwd (interior filters, whole
    image) + pbmc_conv_edge9 (ring of width (k-1)/2 from the eight boundary filter sets, row swap of :1060 included;
    statistics of the first launch repaired): output, GroupNorm sums and channel sums against the float64 oracle, with
    multi-source concatenation, a fused producer transform on the first source, wide (> 16 channel) sources, GELU epilogue
    and the smallest legal image (one strip high)."""
    r = rng(7 * k + H + cout)
    ci = sum(chans)
    xs = [r.standard_normal((B, c, H, W)) for c in chans]
    g0, be0 = 1 + 0.2 * r.standard_normal(chans[0]), 0.2 * r.standard_normal(chans[0])
    use_x = chans[0] % 4 == 0
    x0 = RN.gelu(RN.group_norm(xs[0], g0, be0, chans[0] // 4)) if use_x else xs[0]
    xcat = np.concatenate([x0] + xs[1:], 1)
    names = ("conv",) + ops.EDGE9_REGIONS
    sd = {n + ".weight": r.standard_normal((cout, ci, k, k)) / (k * np.sqrt(ci)) for n in names}
    sd["learnable_bias"] = 0.3 * r.standard_normal((1, cout, 1, 1))
    ref = RN.boundary_learned_conv(xcat, sd, "", k, cout)
    if epi_gelu:
        ref = RN.gelu(ref)
    srcs = []
    for n_, (c, x) in enumerate(zip(chans, xs)):
        xb = ops.pack_nchw(cu(x))
        if n_ == 0 and use_x:
            st = torch.stack([xb.double().sum((2, 3, 4)), (xb.double() ** 2).sum((2, 3, 4))], -1).contiguous()
            srcs.append(ops.Source(xb, L.XFORM_GN_GELU, st, ops.pad_vec(cu(g0), c, DEV, 1.0), ops.pad_vec(cu(be0), c, DEV)))
        else:
            srcs.append(ops.Source(xb))
    wm = cu(sd["conv.weight"])
    wedge = ops.pack_edge9_weights([cu(sd[n + ".weight"]) for n in ops.EDGE9_REGIONS], chans)
    bias = ops.pad_vec(cu(sd["learnable_bias"].reshape(-1)), cout, DEV)
    wrow = ops.pack_conv_weight_row(wm, chans) if ops.row_supported(cout, k, chans) else None
    out, st, cs = ops.conv_learned9(srcs, ops.pack_conv_weight(wm, chans), wrow, wedge, bias, cout, k,
                                    epi_act=L.ACT_GELU if epi_gelu else L.ACT_NONE, want_stats=True, want_chan_sum=csum)
    got = ops.unpack_nchw(out, cout).cpu().numpy()
    assert got.shape == ref.shape and relerr(got, ref) < 6e-6, relerr(got, ref)
    p = (k - 1) // 2
    ring = np.ones((H, W), bool)
    ring[p:H - p, p:W - p] = False
    assert relerr(got[..., ring], ref[..., ring]) < 3e-6  # the FFMA ring by itself
    cob = (cout + 3) // 4
    refp = np.concatenate([ref, np.zeros((B, cob * 4 - cout, H, W))], 1).reshape(B, cob, 4 * H * W)
    ref_st = np.stack([refp.sum(-1), (refp ** 2).sum(-1)], -1)
    assert np.allclose(st.cpu().numpy(), ref_st, rtol=3e-5, atol=2e-5 * H * W)
    if csum:
        assert np.allclose(cs.cpu().numpy()[:, :cout], ref.sum((2, 3)), rtol=3e-5, atol=2e-5 * H * W)
