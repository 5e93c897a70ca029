"""Network / rollout parity on the GPU through the drop-in module API (which calls the C ABI).

Tolerance for one float32 forward (SURVEY.md section 8c, "parity metric caveat"): the reference's
OWN float32 forward differs from its float64 forward by `ref_fp32_noise` (stored with the
golden vectors; 3.7e-5 / 7.2e-5 / 1.4e-6 rel-L2 for u / v / p at 128^2), so the bound is
    rel_L2(new_fp32, ref_fp64) <= max(1e-5, 1.5 * rel_L2(ref_fp32, ref_fp64))     per field.
Rollout diagnostics (mean-T, T(y) profile) must agree within 1e-4 after 100 steps (north_star).
"""
import numpy as np
import pytest
import torch

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from oracle import ref_torch as RT
from pbml_mantle_convection_b200 import _lib as L
from tests._util import VARIANTS, at, field_bound, load, load_weights, noise, relerr, spec_from_variant, split_weights

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
PARAMS = (6.79733173, 475523342.0, 2.58574662)


def make_net(spec, weights, impl="auto", cls=P.NewFluidNet):
    net = cls(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p=spec.r_p, loss_type=spec.loss_type,
              use_symm=spec.use_symm, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({k: torch.tensor(v) for k, v in weights.items()})
    net.conv_impl = impl
    return net.to(DEV).eval()


def fwd_bound(noise):
    return np.maximum(1e-5, 1.5 * np.asarray(noise))


def T_bound(ref_noise):
    """max|T_new - T_ref|: T is O(1), so north_star's 1e-5 relative is 1e-5 absolute; widened to 3 x the reference's own
    fp32-vs-fp64 max-abs distance at the same step where that is larger (the upwind side switch (u > 0) / (u < 0),
    pytorch_networks_convae.py:547-548, turns a 1-ulp change of u near 0 into a different one-sided difference)."""
    return max(1e-5, 3.0 * float(ref_noise))


def pinned_oracle(g, full):
    """`full`: {golden name: full-grid field of the float64 oracle (oracle/ref_torch.py)}.  A full-size golden stores the
    reference's own fields only at the sample indices g["idx"]; the oracle must meet them there (it restates the reference
    to round-off, tests/test_oracle_golden.py) before the GPU result is compared with it over the whole grid."""
    out = {k: a.numpy() for k, a in full.items()}
    for k, a in out.items():
        assert relerr(at(a, g["idx"]), g[k]) < 1e-9, k
    return out


def dt_bound(nz):
    """relative error of the CFL dt = that of max|u|,|v| at ONE cell: 1.5 x the largest fp32 noise the reference itself
    shows on dt over the stored steps, floor 3e-5 (the per-cell velocity noise is ~1e-4, see the u, v entries)."""
    return max(3e-5, 1.5 * max(float(v["dt_rel"]) for k, v in nz.items() if k.startswith("step")))


IMPLS = ["ffma", "umma_3xtf32", "umma_f16x2", "row_f16x2", "mux_f16x2"]


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("tag", VARIANTS)
def test_variants_forward(tag, impl):
    """zeros / reflect / replicate padding, symmetric and plain filters, odd sizes, mae head, k=5."""
    g = load(tag)
    spec = spec_from_variant(g)
    net = make_net(spec, split_weights(g), impl=impl)
    inp = torch.tensor(g["inp"], device=DEV)  # float64 in, float64 out (module is .double() like the reference)
    u, v, p = net(inp)
    assert u.dtype == torch.float64 and tuple(u.shape) == g["u"].shape
    nz = noise(tag)
    res = {"u": u, "v": v, "p": p}
    assert (p is None) == ("p" not in g)
    errs = {n: relerr(res[n].cpu().numpy(), g[n]) for n in nz}
    print(f"[{tag}/{impl}] rel-L2 vs reference fp64: {errs}; reference fp32 noise: {nz}")
    for n in nz:
        assert tuple(res[n].shape) == g[n].shape and errs[n] <= field_bound(nz[n]), (n, errs[n], nz[n])


@pytest.mark.parametrize("impl", IMPLS)
def test_forward_128_against_reference_golden(impl):
    g = load("roll128")
    spec = RN.NetSpec()
    net = make_net(spec, load_weights("roll128"), impl=impl)
    inp, _ = RN.build_input(g["T0"][None, None], g["xc"], g["yc"], g["yc"], *PARAMS)
    u, v, p = net(torch.tensor(inp, device=DEV))
    s = RN.velocity_scaler(*PARAMS)
    errs = np.array([relerr(u[0].cpu().numpy() * s, g["u1"]), relerr(v[0].cpu().numpy() * s, g["v1"]),
                     relerr(p[0].cpu().numpy(), g["p1"])])
    print(f"[{impl}] rel-L2 (u,v,p) new fp32 vs reference fp64:", errs, " reference fp32 noise:", g["ref_fp32_noise"])
    assert np.all(errs <= fwd_bound(g["ref_fp32_noise"])), (errs, g["ref_fp32_noise"])


@pytest.mark.parametrize("impl", ["umma_bf16", "row_bf16"])
def test_forward_128_bf16_variant_bound(impl):
    """bf16-operand conv variant (north_star: "bf16 conv variants get their own stated looser bound").
    Stated bound for one forward at 128^2: rel-L2(p) <= 2e-2 -- and NOTHING is claimed for u, v: they are finite
    differences of the stream function, which amplifies the relative error of the net output by
    ~|a|/|delta a| ~ 600 (the reference's own fp32 run already shows 3.7e-5 / 7.2e-5 from a 5.8e-7 output
    error), so operands with 8 mantissa bits (measured 1.7e-3 per conv) give velocities 30-50 % off.  The bf16
    variant is a pressure-only / throughput-probe variant; the tensor-core path that meets the fp32 parity
    bound on u, v is the fp16 hi+lo split.  The velocity errors are printed, and only required to be finite."""
    g = load("roll128")
    net = make_net(RN.NetSpec(), load_weights("roll128"), impl=impl)
    inp, _ = RN.build_input(g["T0"][None, None], g["xc"], g["yc"], g["yc"], *PARAMS)
    u, v, p = net(torch.tensor(inp, device=DEV))
    s = RN.velocity_scaler(*PARAMS)
    errs = np.array([relerr(u[0].cpu().numpy() * s, g["u1"]), relerr(v[0].cpu().numpy() * s, g["v1"]),
                     relerr(p[0].cpu().numpy(), g["p1"])])
    print(f"[{impl}] rel-L2 (u,v,p) vs reference fp64:", errs)
    assert errs[2] < 2e-2 and np.isfinite(errs).all()


def _ts_call(ts, T0, xc, yc, params=PARAMS, dtype=torch.float64):
    H, W = T0.shape[-2:]
    t = lambda a: torch.tensor(a, dtype=dtype)
    nd = RN.nondim_params(*params)
    return ts(t(T0).view(-1, 1, H, W), None, None, t(yc).view(1, 1, H, W), t(nd[0]), t(nd[1]), t(nd[2]), t(params[0]),
              t(params[1]), t(params[2]), t(xc).view(1, 1, H, W), t(yc).view(1, 1, H, W))


def test_TS_dropin_unmodified_reference_128x506():
    """Same call as advect_wi_gaia.py:590-593 (CPU float64 tensors in), against the UNMODIFIED reference TS(ts=5)."""
    g = load("ts128x506")
    spec, w = RN.NetSpec(), load_weights("ts128x506")
    xc, yc = RN.synthetic_grid(128, 506)
    T0 = RN.synthetic_T0(128, 506, seed=int(g["T0_seed"]))
    T5, _dts, u5, v5, p5, V5, snaps = RT.rollout(RT.prepare_weights(w, spec), spec, torch.tensor(T0)[None, None], torch.tensor(xc),
                                                 torch.tensor(yc), *PARAMS, 5, keep=(1,))
    ref = pinned_oracle(g, {"T1": snaps[1][0, 0], "T5": T5[0, 0], "u5": u5[0], "v5": v5[0], "p5": p5[0], "V5": V5[0, 0]})
    net = make_net(spec, w, impl="auto")
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=5, scale=True, p_pred=True, net="newfluidnet")
    x, dts, u, v, p, V = _ts_call(ts, T0, xc, yc)
    assert sorted(x.keys()) == [0, 1, 2, 3, 4, 5] and sorted(dts.keys()) == [1, 2, 3, 4, 5]
    assert tuple(x[5].shape) == (1, 1, 128, 506) and x[5].dtype == torch.float64 and dts[1].dim() == 0
    assert tuple(u.shape) == (1, 1, 128, 506) and tuple(p.shape) == (1, 1, 128, 506) and tuple(V.shape) == (1, 1, 128, 506)
    nz = noise("ts128x506")
    eT1, eT5 = np.abs(x[1][0, 0].cpu().numpy() - ref["T1"]).max(), np.abs(x[5][0, 0].cpu().numpy() - ref["T5"]).max()
    got_dts = np.array([float(dts[i]) for i in range(1, 6)])
    edt = np.abs(got_dts / g["dts"] - 1).max()
    eu, ev, ep = (relerr(a[0, 0].cpu().numpy(), ref[k]) for a, k in ((u, "u5"), (v, "v5"), (p, "p5")))
    eV = np.abs(V[0, 0].cpu().numpy() - ref["V5"]).max()
    print(f"ts128x506: max|dT1| {eT1:.2e} max|dT5| {eT5:.2e} dt rel {edt:.2e} u5 {eu:.2e} v5 {ev:.2e} p5 {ep:.2e} V5 {eV:.2e}; noise {nz}")
    assert eT1 <= T_bound(nz["step1"]["T_maxabs"]) and eT5 <= T_bound(nz["step5"]["T_maxabs"])
    assert edt <= dt_bound(nz)
    assert eu <= field_bound(nz["step5"]["u"]) and ev <= field_bound(nz["step5"]["v"]) and ep <= field_bound(nz["step5"]["p"])
    assert eV <= max(2e-6, 3 * nz["step5"]["V_maxabs"])  # float32 exp of z ~ -20..0


def test_TS_cached_graph_path_equals_eager_and_tracks_arguments():
    """TS.forward replays one CUDA graph from the second call on (cached buffers).  Every call must still
    see ITS arguments (new T, new Ra), return tensors the caller owns, and equal the eager path bit for bit."""
    g = load("roll64x96")
    spec = RN.NetSpec(levels=4)
    net = make_net(spec, load_weights("roll64x96"), impl="auto")
    mk = lambda: P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=2, scale=True, p_pred=True, net="newfluidnet")
    ts_g, ts_e = mk(), mk()
    ts_e.use_cuda_graph = False
    T0 = g["T0"]
    T1 = np.clip(T0 + 0.05 * np.sin(np.arange(T0.shape[1]) / 7.0)[None, :], 0.0, 1.0)
    P2 = (3.2, 2.0e7, 5.0)
    calls = [(T0, PARAMS), (T1, PARAMS), (T0, P2), (T1, P2), (T0, PARAMS)]
    kept = []
    for T, prm in calls:
        a = _ts_call(ts_g, T, g["xc"], g["yc"], params=prm)
        b = _ts_call(ts_e, T, g["xc"], g["yc"], params=prm)
        for ta, tb in [(a[0][1], b[0][1]), (a[0][2], b[0][2]), (a[2], b[2]), (a[3], b[3]), (a[4], b[4]), (a[5], b[5]),
                       (a[1][1], b[1][1]), (a[1][2], b[1][2])]:
            assert ta.dtype == torch.float64 and torch.equal(ta, tb)
        kept.append((a[0][2].clone(), a[0][2]))
    assert ts_g._plan.graph is not None and ts_e._plan.graph is None
    for snap, live in kept:  # results of earlier calls were not overwritten by later replays
        assert torch.equal(snap, live)
    # different arguments gave different results (the graph did not freeze its first inputs)
    assert not torch.equal(kept[0][1], kept[1][1]) and not torch.equal(kept[0][1], kept[2][1])
    assert torch.equal(kept[0][1], kept[4][1])


@pytest.mark.parametrize("impl", IMPLS)
def test_rollout_100_steps_diagnostics(impl):
    """BASELINE config 1 (128x128, 100 steps): T fields and mean-T / profile diagnostics vs the reference."""
    g = load("roll128")
    net = make_net(RN.NetSpec(), load_weights("roll128"), impl=impl)
    ens = P.EnsembleRollout(net, 128, 128, [PARAMS], DEV, cn_max=0.99)
    ens.set_T(g["T0"][None])
    snaps = {}
    done = 0
    for upto in (1, 10, 100):
        ens.step(upto - done)
        done = upto
        snaps[upto] = ens.T[0].cpu().numpy().astype(np.float64)
    nz = noise("roll128")
    errs = {i: float(np.abs(snaps[i] - g[f"T{i}"]).max()) for i in (1, 10, 100)}
    print(f"[{impl}] max|dT| after 1/10/100 steps: {errs}; reference fp32 noise: { {i: nz[f'step{i}']['T_maxabs'] for i in (1, 10, 100)} }")
    for i in (1, 10, 100):
        assert errs[i] <= T_bound(nz[f"step{i}"]["T_maxabs"]), (i, errs[i])
    mean, prof, dprof = ens.diagnostics()
    assert abs(mean[0].item() - float(g["meanT"])) < 1e-4
    assert np.abs(prof[0].cpu().numpy() - g["Tprof"]).max() < 1e-4
    scale = np.abs(g["dTprof"]).max()
    assert np.abs(dprof[0].cpu().numpy() - g["dTprof"]).max() < 1e-3 * scale
    assert abs(ens.time[0].item() - g["dts"].sum()) <= dt_bound(nz) * g["dts"].sum()


def test_graph_replay_equals_eager():
    spec = RN.NetSpec(levels=4)
    w = load_weights("roll64x96")
    g = load("roll64x96")
    net = make_net(spec, w, impl="ffma")
    outs = []
    for mode in ("eager", "graph2", "graph5"):
        ens = P.EnsembleRollout(net, 64, 96, [PARAMS], DEV)
        ens.set_T(g["T0"][None])
        if mode == "eager":
            ens.step(10)
        else:
            ens.run(10, steps_per_graph=int(mode[5:]))
        outs.append((ens.T.clone(), ens.time.clone()))
    assert np.abs(outs[0][0].cpu().numpy()[0] - g["T10"]).max() <= T_bound(noise("roll64x96")["step10"]["T_maxabs"])
    for T, t in outs[1:]:
        # identical kernels and order; only the GroupNorm atomics may reorder (double) => ~1e-7
        assert (T - outs[0][0]).abs().max().item() < 2e-6
        assert abs(t[0].item() - outs[0][1][0].item()) < 1e-6 * outs[0][1][0].item()


def test_ensemble_members_are_independent():
    """B members with different (Ra, gamma, beta, T0) == B separate B=1 rollouts (per-member dt)."""
    spec = RN.NetSpec(levels=4)
    net = make_net(spec, load_weights("roll64x96"), impl="ffma")
    prm = [PARAMS, (0.9, 3.0e6, 1.5), (9.1, 5.0e9, 60.0)]
    H, W = 64, 96
    T0 = np.stack([RN.synthetic_T0(H, W, seed=1 + m) for m in range(3)])
    ens = P.EnsembleRollout(net, H, W, prm, DEV)
    ens.set_T(T0)
    ens.step(4)
    for m in range(3):
        one = P.EnsembleRollout(net, H, W, [prm[m]], DEV)
        one.set_T(T0[m:m + 1])
        one.step(4)
        assert (one.T[0] - ens.T[m]).abs().max().item() < 2e-6
        assert abs(one.time[0].item() - ens.time[m].item()) <= 1e-6 * one.time[0].item()
    # and against the float64 oracle for one non-default member
    W64 = RT.prepare_weights(load_weights("roll64x96"), spec)
    xc, yc = RN.synthetic_grid(H, W)
    Tr, dts, *_ = RT.rollout(W64, spec, torch.tensor(T0[1])[None, None], torch.tensor(xc), torch.tensor(yc), *prm[1], 4)
    assert np.abs(ens.T[1].cpu().numpy() - Tr[0, 0].numpy()).max() < 1e-5  # T is O(1): north_star's 1e-5
    assert abs(ens.time[1].item() - sum(dts)) < 1e-4 * sum(dts)  # dt follows max|u| at one cell (fp32 noise ~3e-5, dt_bound)


def test_full_size_512_against_reference_golden():
    """BASELINE config 2 grid (512x512, batch 1): fields of the first forward and T after 3 steps against the REFERENCE
    (tests/golden/roll512.npz, float64, written by make_golden.py fullsize), bound = the per-case noise rule."""
    g, nz = load("roll512"), noise("roll512")
    spec, w = RN.NetSpec(), load_weights("roll128")  # same spec and seed as roll128
    H = W = 512
    T0 = RN.synthetic_T0(H, W, seed=int(g["T0_seed"]))
    W64 = RT.prepare_weights(w, spec)
    xc, yc = (torch.tensor(a) for a in RN.synthetic_grid(H, W))
    T1, _, u1, v1, p1, _, _ = RT.rollout(W64, spec, torch.tensor(T0)[None, None], xc, yc, *PARAMS, 1)
    T3 = RT.rollout(W64, spec, T1, xc, yc, *PARAMS, 2)[0]
    ref = pinned_oracle(g, {"u1": u1[0], "v1": v1[0], "p1": p1[0], "T1": T1[0, 0], "T3": T3[0, 0]})
    net = make_net(spec, w, impl="auto")
    ens = P.EnsembleRollout(net, H, W, [PARAMS], DEV)
    ens.set_T(T0[None])
    ens.run(1)
    u, v, p, V = ens.fields()
    e1 = {n: relerr(a[0].cpu().numpy(), ref[n + "1"]) for n, a in (("u", u), ("v", v), ("p", p))}
    eT1 = float(np.abs(ens.T[0].cpu().numpy() - ref["T1"]).max())
    ens.run(2)
    eT3 = float(np.abs(ens.T[0].cpu().numpy() - ref["T3"]).max())
    et = abs(ens.time[0].item() - g["dts"].sum()) / g["dts"].sum()
    print(f"roll512: step-1 rel-L2 {e1}, max|dT1| {eT1:.2e}, max|dT3| {eT3:.2e}, time rel {et:.2e}; reference fp32 noise {nz}")
    for n in "uvp":
        assert e1[n] <= field_bound(nz["step1"][n]), (n, e1[n])
    assert eT1 <= T_bound(nz["step1"]["T_maxabs"]) and eT3 <= T_bound(nz["step3"]["T_maxabs"])
    assert et <= dt_bound(nz)


def test_ensemble_256_members_against_reference_golden():
    """BASELINE config 4 (256x256 members with different Ra / gamma / beta / initial T, per-member dt): 4 members advanced
    together for 3 steps against 4 separate B = 1 runs of the REFERENCE (tests/golden/ens256.npz)."""
    g, nz = load("ens256"), noise("ens256")
    spec, w = RN.NetSpec(), load_weights("roll128")
    H = W = 256
    prm = [tuple(r) for r in g["params"]]
    T0 = np.stack([RN.synthetic_T0(H, W, seed=int(s)) for s in g["T0_seeds"]])
    W64 = RT.prepare_weights(w, spec)
    xc, yc = (torch.tensor(a) for a in RN.synthetic_grid(H, W))
    ref = {}
    for m in range(len(prm)):
        T3, _, u3, v3, p3, _, _ = RT.rollout(W64, spec, torch.tensor(T0[m])[None, None], xc, yc, *prm[m], 3)
        ref.update({f"m{m}_u3": u3[0], f"m{m}_v3": v3[0], f"m{m}_p3": p3[0], f"m{m}_T3": T3[0, 0]})
    ref = pinned_oracle(g, ref)
    net = make_net(spec, w, impl="auto")
    ens = P.EnsembleRollout(net, H, W, prm, DEV)
    ens.set_T(T0)
    ens.run(3)
    u, v, p, V = ens.fields()
    for m in range(len(prm)):
        n_m = nz[f"m{m}"]
        e = {n: relerr(a[m].cpu().numpy(), ref[f"m{m}_{n}3"]) for n, a in (("u", u), ("v", v), ("p", p))}
        eT = float(np.abs(ens.T[m].cpu().numpy() - ref[f"m{m}_T3"]).max())
        et = abs(ens.time[m].item() - g[f"m{m}_dts"].sum()) / g[f"m{m}_dts"].sum()
        print(f"ens256 member {m}: rel-L2 {e}, max|dT3| {eT:.2e}, time rel {et:.2e}; reference fp32 noise {n_m}")
        for n in "uvp":
            assert e[n] <= field_bound(n_m[n]), (m, n, e[n])
        assert eT <= T_bound(n_m["T_maxabs"]) and et <= max(3e-5, 1.5 * n_m["dt_rel"])


def test_module_level_layers():
    """Stand-alone FluidLayer / SymmetricConv2d / BoundaryLearnedConvolution2D / ADNet forwards."""
    g = load("ops")
    for tag, k, ci, co, symm in (("blc3", 3, 5, 8, False), ("blc5", 5, 4, 8, False), ("blc3s", 3, 6, 16, True)):
        m = P.BoundaryLearnedConvolution2D(ci, co, k, use_symm=symm).double()
        m.load_state_dict({kk: torch.tensor(v) for kk, v in split_weights(g, tag + "_w::").items()})
        m = m.to(DEV)
        y = m(torch.tensor(g[tag + "_x"], device=DEV))
        assert tuple(y.shape) == g[tag + "_y"].shape and relerr(y.cpu().numpy(), g[tag + "_y"]) < 3e-6
        if tag == "blc3":
            y2 = m(torch.tensor(g[tag + "_x"], device=DEV), bc_x=2, bc_y=2)
            assert tuple(y2.shape) == g["blc3_y_bc2"].shape and relerr(y2.cpu().numpy(), g["blc3_y_bc2"]) < 3e-6
    # ADNet drop-in: inputs [B,6,H,W] float64, batch-global dt, in-place wall coordinates
    u, v, T = g["ad_u"], g["ad_v"], g["ad_T"]
    B, _, H, W = u.shape
    xc = np.broadcast_to(g["ad_xc"], (B, 1, H, W))
    yc = np.broadcast_to(g["ad_yc"], (B, 1, H, W))
    inp = torch.tensor(np.concatenate([u, v, T, np.full_like(u, float(g["ad_raq"])), xc, yc], 1), device=DEV)
    ad = P.ADNet(DEV, CN_max=0.99)
    Tn, dt = ad(inp)
    assert tuple(Tn.shape) == (B, 1, H, W) and Tn.dtype == torch.float64
    assert abs(float(dt) - float(g["ad_dt"])) < 1e-6 * float(g["ad_dt"])
    assert np.abs(Tn.cpu().numpy() - g["ad_Tn"]).max() < 2e-5
    assert inp[0, 4, 3, -1].item() == 4.0 and inp[0, 5, -1, 3].item() == 1.0  # reference side effect, :532-535
    Tn2, dt2 = ad(inp, dt=torch.tensor(1e-4, dtype=torch.float64))
    assert np.abs(Tn2.cpu().numpy() - g["ad_Tn_fixed_dt"]).max() < 2e-4
    # FluidLayer stand-alone == conv + GN + GELU (numpy oracle)
    torch.manual_seed(1)
    fl = P.FluidLayer(7, 16, "gelu", "replicate", True, 1, f=3).double().to(DEV)
    x = torch.randn(2, 7, 18, 27, dtype=torch.float64, device=DEV)
    sd = {k: t.detach().cpu().numpy() for k, t in fl.state_dict().items()}
    ref = RN.fluid_layer(x.cpu().numpy(), sd, "", 16, RN.NetSpec())
    assert relerr(fl(x).cpu().numpy(), ref) < 5e-6


def test_learned_boundary_network_runs_and_matches_oracle_layers():
    """SURVEY.md section 8f N1 (secondary config), small: learned 9-region convs, k=5, c_o=1, through NewFluidNet."""
    torch.manual_seed(2)
    net = P.NewFluidNet(2, 7, 8, 1, DEV, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10,
                        repeats=1, f=5, p_pred=False).double().to(DEV).eval()
    x = torch.randn(1, 7, 24, 32, dtype=torch.float64, device=DEV)
    u, v, p = net(x)
    assert p is None and tuple(u.shape) == (1, 24, 32) and torch.isfinite(u).all() and torch.isfinite(v).all()
    # first layer against the numpy oracle of the 9-region conv + GN + GELU
    sd = {k: t.detach().cpu().numpy() for k, t in net.state_dict().items()}
    y = RN.boundary_learned_conv(x.cpu().numpy(), sd, "conv.0.layers.0.", 5, 8)
    ref = RN.gelu(RN.group_norm(y, sd["conv.0.layers.1.weight"], sd["conv.0.layers.1.bias"], 2))
    assert relerr(net.conv[0](x).cpu().numpy(), ref) < 5e-6


@pytest.mark.parametrize("k,ci,co", [(5, 16, 16), (3, 7, 16), (5, 16, 1)])
def test_learned_boundary_conv_tensor_core_interior(k, ci, co):
    """At the sizes real grids have (>= 32 rows and columns) the interior region of the 9-region conv runs on the
    tensor-core kernels (fp16 hi+lo), the strips on the FFMA kernel; packed filters are cached on the modules and
    follow in-place weight updates."""
    torch.manual_seed(3)
    m = P.BoundaryLearnedConvolution2D(ci, co, k).double().to(DEV)
    with torch.no_grad():
        m.learnable_bias.normal_()
    x = torch.randn(2, ci, 40, 48, dtype=torch.float64, device=DEV)
    sd = {kk: t.detach().cpu().numpy() for kk, t in m.state_dict().items()}
    ref = RN.boundary_learned_conv(x.cpu().numpy(), sd, "", k, co)
    assert relerr(m(x).cpu().numpy(), ref) < 5e-6
    assert relerr(m(x).cpu().numpy(), ref) < 5e-6  # second call: cached filter images
    with torch.no_grad():
        m.conv.weight.mul_(0.5)  # in-place update: the cache must notice
    sd = {kk: t.detach().cpu().numpy() for kk, t in m.state_dict().items()}
    assert relerr(m(x).cpu().numpy(), RN.boundary_learned_conv(x.cpu().numpy(), sd, "", k, co)) < 5e-6


def test_learned_network_graph_replay_equals_eager_and_tracks_weights():
    """From the third call on a learned-boundary network replays its forward as one CUDA graph: same bits as the eager
    calls, new inputs are picked up, and a weight update re-captures."""
    torch.manual_seed(4)
    net = P.NewFluidNet(2, 7, 8, 1, DEV, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10,
                        repeats=2, f=5, p_pred=False).to(DEV).eval()
    x1 = torch.randn(1, 7, 40, 48, device=DEV)
    x2 = torch.randn(1, 7, 40, 48, device=DEV)
    net.use_cuda_graph = False
    e1, e2 = net(x1), net(x2)
    net.use_cuda_graph = True
    net(x1), net(x1)  # eager, capture + replay
    r1, r2 = net(x1), net(x2)
    plan = net.__dict__["_learned_plan"]
    assert plan.graph is not None and not plan.failed
    for a, b in ((e1, r1), (e2, r2)):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[2] is None and b[2] is None
    with torch.no_grad():
        net.conv[2].conv.weight.mul_(1.5)
    net.use_cuda_graph = False
    e3 = net(x1)
    net.use_cuda_graph = True
    outs = [net(x1) for _ in range(3)]
    assert net.__dict__["_learned_plan"] is not plan
    assert not torch.equal(e3[0], e1[0])
    for o in outs:
        assert torch.equal(o[0], e3[0]) and torch.equal(o[1], e3[1])


def test_no_silent_fallback_on_gpu_box():
    with pytest.raises(L.PbmcError):
        P.NewFluidNet(2, 7, 16, 2, DEV, act_fn="gelu", r_p="replicate", loss_type="curl", use_symm=True,
                      repeats=1)(torch.zeros(1, 7, 16, 16))  # CPU tensor on a CUDA model: refuse, do not fall back


def test_driver_per_step_and_resident_agree(tmp_path):
    """driver.attempt (one TS call per step, host round trip, advect_wi_gaia.py:583-668) and driver.attempt_resident
    (EnsembleRollout, k steps per CUDA graph) log the same simulated times and mean temperatures."""
    from pbml_mantle_convection_b200 import driver as D

    g = load("roll64x96")
    spec = RN.NetSpec(levels=4)
    net = make_net(spec, load_weights("roll64x96"), impl="auto")
    H, W = g["T0"].shape
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    xcc, ycc = t64(g["xc"]).view(1, 1, H, W), t64(g["yc"]).view(1, 1, H, W)
    nd = RN.nondim_params(*PARAMS)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=True, net="newfluidnet")
    t_a, n_a, (snap_a, TS_a, tv_a, Tv_a) = D.attempt(ts, t64(g["T0"]).view(1, 1, H, W), xcc, ycc, t64(PARAMS[0]), t64(PARAMS[1]),
                                                    t64(PARAMS[2]), t64(nd[0]), t64(nd[1]), t64(nd[2]), t_end=1.0,
                                                    out_dir=str(tmp_path / "a"), max_steps=12, save_every=0.0)
    ens = P.EnsembleRollout(net, H, W, [PARAMS], DEV, xc=g["xc"], yc=g["yc"], cn_max=0.99, per_member_dt=False)
    ens.set_T(g["T0"][None])
    t_b, n_b, (snap_b, TS_b, tv_b, Tv_b) = D.attempt_resident(ens, xcc, ycc, t_end=1.0, out_dir=str(tmp_path / "b"), max_steps=12,
                                                             check_every=4, save_every=0.0)
    assert n_a == 12 and n_b == 12
    assert np.allclose(tv_a["ML"], tv_b["ML"], rtol=1e-6)
    # the reference's 10-step golden T is matched by both (same bound as the rollout test)
    assert np.abs(snap_a["ML"]["T"][10].reshape(H, W) - g["T10"]).max() <= T_bound(noise("roll64x96")["step10"]["T_maxabs"])
    assert abs(Tv_a["ML"][12] - Tv_b["ML"][12]) < 1e-6  # block-end sample of the resident path == per-step value
    assert np.abs(snap_a["ML"]["T"][-1] - snap_b["ML"]["T"][-1]).max() < 1e-6
    assert snap_b["ML"]["v"][-1].shape == (H * W, 3) and len(snap_b["ML"]["T"]) == 1 + 3  # initial + one per block
    for sub in ("a", "b"):
        assert (tmp_path / sub / "snapshots_ML.pkl").exists() and (tmp_path / sub / "T_vec_ML.pkl").exists()


def test_forward_with_tma_staged_levels_is_bit_identical():
    """net.up_staged = True (pbmc_net.flags & PBMC_NET_UP_STAGED): the up-sampled levels are written as conv[1]'s fp16
    hi|lo operand image and staged by TMA bulk copies (api.cu / conv_row.cu bulk-copy lane).  Same arithmetic, so the
    forward must not change by one bit; the persistent and the per-layer trunk agree to the statistics' atomic order."""
    torch.manual_seed(0)
    net = P.NewFluidNet(4, 7, 16, 2, DEV, act_fn="gelu", r_p="replicate", loss_type="curl", use_symm=True, a_bound=10,
                        repeats=2, f=3, p_pred=True).to(DEV).eval()
    x = torch.randn(2, 7, 70, 150, generator=torch.Generator().manual_seed(1)).to(DEV)
    net.trunk_mode = "per_layer"
    ref = net(x)
    net.up_staged = True
    got = net(x)
    for a, b in zip(ref, got):
        assert torch.equal(a, b)
    net.up_staged, net.trunk_mode = False, "auto"
    per = net(x)
    for a, b in zip(ref, per):
        assert (a - b).abs().max().item() <= 1e-5 * float(a.abs().max())


def test_TS_without_adnet_is_the_ML_STOKES_mode():
    """advect_wi_gaia.py:486-500: `TS(model_uvp, None, ...)` -- the surrogate only supplies (u, v, p, V) to an external
    energy solver; no T is advanced, `dts` stays empty (reference :453: the ADNet branch is skipped)."""
    g, nz = load("roll64x96"), noise("roll64x96")["step1"]
    net = make_net(RN.NetSpec(levels=4), load_weights("roll64x96"), impl="auto")
    ts = P.TS(net, None, DEV, ts=1, scale=True, p_pred=True, net="newfluidnet")
    x, dts, u, v, p, V = _ts_call(ts, g["T0"], g["xc"], g["yc"])
    H, W = g["T0"].shape
    assert sorted(x.keys()) == [0] and dts == {} and tuple(u.shape) == (1, 1, H, W) and u.dtype == torch.float64
    for name, a, ref in (("u", u, g["u1"]), ("v", v, g["v1"]), ("p", p, g["p1"])):
        assert relerr(a[0, 0].cpu().numpy(), ref) <= field_bound(nz[name]), name
    assert np.abs(V[0, 0].cpu().numpy() - g["V1"]).max() <= max(2e-6, 3 * nz["V_maxabs"])
