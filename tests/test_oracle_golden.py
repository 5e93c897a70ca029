"""Pin both oracle restatements against vectors produced by the real reference
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import ref_numpy as RN
from oracle import ref_torch as RT
from tests._util import LEARNED_CASES, UNET_CASES, VARIANTS, at, load, load_learned_case, load_unet_case, load_weights, relerr, spec_from_variant, split_weights


def test_ops_adnet():
    g = load("ops")
    Tn, dt = RN.adnet_forward(g["ad_u"][:, 0], g["ad_v"][:, 0], g["ad_T"][:, 0], float(g["ad_raq"]), g["ad_xc"],
                              g["ad_yc"], 0.99)
    assert np.abs(Tn - g["ad_Tn"][:, 0]).max() == 0.0
    assert dt == float(g["ad_dt"])
    Tn2, _ = RN.adnet_forward(g["ad_u"][:, 0], g["ad_v"][:, 0], g["ad_T"][:, 0], float(g["ad_raq"]), g["ad_xc"],
                              g["ad_yc"], 0.99, dt=1e-4)
    assert np.abs(Tn2 - g["ad_Tn_fixed_dt"][:, 0]).max() < 1e-15
    t = lambda a: torch.tensor(a)
    Tt, dtt = RT.adnet(t(g["ad_u"][:, 0]), t(g["ad_v"][:, 0]), t(g["ad_T"][:, 0]), float(g["ad_raq"]), t(g["ad_xc"]),
                       t(g["ad_yc"]), 0.99)
    assert np.abs(Tt.numpy() - g["ad_Tn"][:, 0]).max() < 1e-14
    assert abs(float(dtt) - float(g["ad_dt"])) < 1e-18


def test_ops_bicubic_pool():
    g = load("ops")
    assert np.abs(RN.bicubic_upsample(g["bic_x"], (50, 77)) - g["bic_y"]).max() < 1e-13
    assert np.abs(RN.avg_pool2(g["bic_x"]) - g["pool_y"]).max() == 0.0


@pytest.mark.parametrize("tag,k,co,symm", [("blc3", 3, 8, False), ("blc5", 5, 8, False), ("blc3s", 3, 16, True)])
def test_ops_boundary_learned(tag, k, co, symm):
    g = load("ops")
    sd = split_weights(g, tag + "_w::")
    y = RN.boundary_learned_conv(g[tag + "_x"], sd, "", k, co, use_symm=symm)
    assert relerr(y, g[tag + "_y"]) < 1e-14
    if tag == "blc3":
        y2 = RN.boundary_learned_conv(g[tag + "_x"], sd, "", k, co, bc_x=2, bc_y=2)
        assert y2.shape == g["blc3_y_bc2"].shape and relerr(y2, g["blc3_y_bc2"]) < 1e-14


@pytest.mark.parametrize("tag", VARIANTS)
def test_variants_numpy(tag):
    g = load(tag)
    spec = spec_from_variant(g)
    u, v, p = RN.newfluidnet_forward(split_weights(g), spec, g["inp"])
    assert relerr(u, g["u"]) < 1e-12 and relerr(v, g["v"]) < 1e-12
    if "p" in g:
        assert relerr(p, g["p"]) < 1e-12


@pytest.mark.parametrize("tag", ["var_reflect_sym", "var_replicate_odd", "var_zeros_nosym"])
def test_variants_torch_port(tag):
    g = load(tag)
    spec = spec_from_variant(g)
    W = RT.prepare_weights(split_weights(g), spec)
    u, v, p = RT.net_forward(W, spec, torch.tensor(g["inp"]))
    assert relerr(u.numpy(), g["u"]) < 1e-12 and relerr(v.numpy(), g["v"]) < 1e-12
    assert relerr(p.numpy(), g["p"]) < 1e-12


def test_rollout_torch_port_100_steps():
    g = load("roll128")
    spec = RN.NetSpec()
    W = RT.prepare_weights(load_weights("roll128"), spec)
    raq, fkt, fkp = g["params"]
    T, dts, u, v, p, V, snaps = RT.rollout(W, spec, torch.tensor(g["T0"])[None, None], torch.tensor(g["xc"]),
                                           torch.tensor(g["yc"]), float(raq), float(fkt), float(fkp), 100,
                                           keep=(1, 10, 100))
    for i in (1, 10, 100):
        assert np.abs(snaps[i][0, 0].numpy() - g[f"T{i}"]).max() < 1e-9
    assert np.allclose(dts, g["dts"], rtol=1e-9)
    mT, Tp, dTp = RN.diagnostics(T[0, 0].numpy(), g["yc"][:, 0])
    assert abs(mT - float(g["meanT"])) < 1e-12 and np.abs(Tp - g["Tprof"]).max() < 1e-10


def test_rollout_numpy_10_steps_small():
    g = load("roll64x96")
    spec = RN.NetSpec(levels=4)
    raq, fkt, fkp = g["params"]
    T, dts, u, v, p, V, snaps = RN.ts_rollout(load_weights("roll64x96"), spec, g["T0"][None, None], g["xc"], g["yc"],
                                              raq, fkt, fkp, 10, keep=(1, 10))
    assert np.abs(snaps[1][0, 0] - g["T1"]).max() < 1e-12
    assert np.abs(snaps[10][0, 0] - g["T10"]).max() < 1e-10
    assert np.allclose(dts, g["dts"], rtol=1e-10)


def test_unmodified_TS_128x506():
    """The reference's fields are stored at the sample indices g["idx"]."""
    g = load("ts128x506")
    spec = RN.NetSpec()
    W = RT.prepare_weights(load_weights("ts128x506"), spec)
    raq, fkt, fkp = g["params"]
    xc, yc = RN.synthetic_grid(128, 506)
    T0 = RN.synthetic_T0(128, 506, seed=int(g["T0_seed"]))
    T, dts, u, v, p, V, snaps = RT.rollout(W, spec, torch.tensor(T0)[None, None], torch.tensor(xc), torch.tensor(yc),
                                           float(raq), float(fkt), float(fkp), 5, keep=(1, 5))
    idx = g["idx"]
    assert np.abs(at(snaps[1][0, 0].numpy(), idx) - g["T1"]).max() < 1e-10
    assert np.abs(at(snaps[5][0, 0].numpy(), idx) - g["T5"]).max() < 1e-9
    assert relerr(at(u[0].numpy(), idx), g["u5"]) < 1e-9 and relerr(at(p[0].numpy(), idx), g["p5"]) < 1e-9
    assert np.abs(at(V[0, 0].numpy(), idx) - g["V5"]).max() < 1e-12
    assert np.allclose(dts, g["dts"], rtol=1e-9)


@pytest.mark.parametrize("tag", UNET_CASES)
def test_unet_restatement_against_reference(tag):
    """SURVEY.md section 8f N4: the U-Net time-stepper surrogate (reference :1985-2068), float64."""
    spec, inp, outs, sd = load_unet_case(tag)
    res = dict(zip("uvpT", RN.unet_forward(sd, spec, inp)))
    assert (res["p"] is None) == ("p" not in outs)
    for n, ref in outs.items():
        assert res[n].shape == ref.shape and relerr(res[n], ref) < 1e-13, n


@pytest.mark.parametrize("tag", LEARNED_CASES)
def test_learned_network_restatement_against_reference(tag):
    """SURVEY.md section 8f N1: whole learned-boundary networks (NewFluidNet :1315-1388, FluidNet :1639-1697), float64."""
    spec, inp, outs, sd = load_learned_case(tag)
    res = dict(zip("uvp", RN.learned_net_forward(sd, spec, inp, fluidnet=tag == "learned_fluidnet")))
    assert (res["p"] is None) == ("p" not in outs)
    for n, ref in outs.items():
        assert res[n].shape == ref.shape and relerr(res[n], ref) < 1e-13, n
