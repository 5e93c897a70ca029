"""Learned-boundary networks (r_p="learned", SURVEY.md section 8f N1) through the fused, device-resident engine: the DAG of
pbmc_surrogate_forward / pbmc_rollout with a ring-kernel launch behind every conv.  Parity rule of DESIGN section 3: per
output field rel-L2 <= max(1e-5, 1.5 x the reference's own fp32-vs-fp64 distance on the case), T within 1e-5, dt within
3e-5 relative.  The paper configuration has no golden of the reference; it is held to the oracle with the noise of
learned_k5 (same k = 5 and head)."""
import numpy as np
import pytest
import torch

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from pbml_mantle_convection_b200 import _lib as L, engine, ops
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_T0, synthetic_grid
from tests._util import field_bound, load, load_learned_case, noise, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PARAMS = tuple(float(x) for x in load("roll64x96")["params"])  # (RaQ, gamma, beta) of the smoke / rollout golden


def _net(spec, w=None, seed=0):
    torch.manual_seed(seed)
    net = P.NewFluidNet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p="learned", loss_type="curl",
                        use_symm=False, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    if w is not None:
        net.load_state_dict({k: torch.tensor(v) for k, v in w.items()})
    else:  # random weights, learnable biases included (they start at zero)
        with torch.no_grad():
            for m in net.modules():
                if isinstance(m, P.BoundaryLearnedConvolution2D):
                    m.learnable_bias.normal_(0.0, 0.1)
    return net.to(DEV).eval()


def _sd(net):
    return {k: t.detach().cpu().numpy() for k, t in net.state_dict().items()}


PAPER = RN.NetSpec(levels=5, c_i=7, c_h=16, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0, repeats=6,
                   f=5, p_pred=False)


def _case(tag):
    if tag == "paper":
        net = _net(PAPER, seed=11)
        inp = np.random.default_rng(11).standard_normal((1, 7, 96, 160))  # coarsest level 6 x 10: exactly the k = 5 strip
        u, v, p = RN.learned_net_forward(_sd(net), PAPER, inp)
        return net, inp, {"u": u, "v": v}, noise("learned_k5")
    spec, inp, outs, w = load_learned_case(tag)
    return _net(spec, w), inp, outs, noise(tag)


@pytest.mark.parametrize("tag", ["learned_k5", "learned_k3_p", "paper"])
def test_engine_forward_against_reference(tag):
    net, inp, outs, nz = _case(tag)
    B, _, H, W = inp.shape
    assert engine.fused_supported(net, B, H, W)
    u, v, p, _ = net._engine(torch.device(DEV)).forward_blocked(ops.pack_nchw(torch.tensor(inp, device=DEV)))
    res = {"u": u, "v": v, "p": p}
    errs = {n: relerr(res[n].cpu().numpy(), ref) for n, ref in outs.items()}
    print(f"[{tag}] fused engine rel-L2 vs fp64: {errs}; reference fp32 noise: {nz}")
    for n, ref in outs.items():
        assert tuple(res[n].shape) == ref.shape
        assert errs[n] <= field_bound(nz[n]), (n, errs[n])


# ------------------------------------------------------------------------------------------------ TS on a learned net
def _oracle_rollout(sd, spec, T0, xc, yc, n_steps, CN_max=0.99):
    """TS.forward's loop restated in float64 with the learned network: build_input -> learned_net_forward -> velocity
    scaler -> adnet_forward -> apply_T_bcs."""
    raq, fkt, fkp = PARAMS
    T, Ts, dts = T0, {}, []
    for i in range(1, n_steps + 1):
        inp, V = RN.build_input(T, xc, yc, yc, raq, fkt, fkp)
        u, v, p = RN.learned_net_forward(sd, spec, inp)
        s = RN.velocity_scaler(raq, fkt, fkp)
        u, v = u * s, v * s
        Tn, dt = RN.adnet_forward(u, v, T[:, 0], raq, xc, yc, CN_max)
        T = RN.apply_T_bcs(Tn)[:, None]
        Ts[i] = T
        dts.append(float(dt))
    return Ts, np.asarray(dts), u, v, p


def _ts_call(ts, T0, xc, yc):
    raq, fkt, fkp = PARAMS
    H, W = T0.shape
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    nd = RN.nondim_params(raq, fkt, fkp)
    out = ts(t64(T0).view(1, 1, H, W), None, None, t64(yc).view(1, 1, H, W), t64(nd[0]), t64(nd[1]), t64(nd[2]), t64(raq),
             t64(fkt), t64(fkp), t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W))
    torch.cuda.synchronize()
    return out


def _learned_k3_p():
    spec, _, _, w = load_learned_case("learned_k3_p")  # k = 3, p predicted, 2 levels
    return spec, _net(spec, w)


def test_ts_learned_rollout_against_oracle():
    spec, net = _learned_k3_p()
    H, W = 64, 96
    xc, yc = synthetic_grid(H, W)
    T0 = synthetic_T0(H, W)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=10, scale=True, p_pred=True, net="newfluidnet")
    Ts, dts_ref, u_ref, v_ref, p_ref = _oracle_rollout(_sd(net), spec, T0[None, None], xc, yc, 10)
    nz = noise("learned_k3_p")
    for call in range(2):  # eager, then capture + replay of the fused plan
        x, dts, u, v, p, V = _ts_call(ts, T0, xc, yc)
        assert ts._plan is not None, "a supported learned net must take the fused rollout"
        if call == 1:
            assert ts._plan.graph is not None and ts._plan.calls == 2
        errs = {"u": relerr(u[0, 0].cpu().numpy(), u_ref[0]), "v": relerr(v[0, 0].cpu().numpy(), v_ref[0]),
                "p": relerr(p[0, 0].cpu().numpy(), p_ref[0])}
        eT = {i: float(np.abs(x[i].cpu().numpy() - Ts[i]).max()) for i in (1, 10)}
        edt = max(abs(float(dts[i]) - dts_ref[i - 1]) / dts_ref[i - 1] for i in range(1, 11))
        print(f"[TS learned call {call}] rel-L2 {errs}; max|dT| {eT}; dt rel {edt:.2e}")
        for n in "uvp":
            assert errs[n] <= field_bound(nz[n]), (call, n, errs[n])
        assert eT[1] <= 1e-5 and eT[10] <= 1e-5, (call, eT)
        assert edt <= 3e-5, (call, edt)


def test_ts_learned_weight_update_recaptures():
    """A parameter changed in place between two TS calls changes the result, to what a fresh TS computes."""
    _, net = _learned_k3_p()
    H, W = 64, 96
    xc, yc = synthetic_grid(H, W)
    T0 = synthetic_T0(H, W)
    mk = lambda: P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=3, scale=True, p_pred=True, net="newfluidnet")
    ts = mk()
    _ts_call(ts, T0, xc, yc)
    before = _ts_call(ts, T0, xc, yc)  # graph replay
    old_graph = ts._plan.graph
    assert old_graph is not None
    with torch.no_grad():
        net.conv[2].conv_top.weight.mul_(1.5)  # an edge filter set: only the ring kernel reads it
        net.conv[0].layers[0].learnable_bias.add_(0.05)
    after = _ts_call(ts, T0, xc, yc)
    after2 = _ts_call(ts, T0, xc, yc)
    fresh = _ts_call(mk(), T0, xc, yc)
    assert ts._plan.graph is not old_graph
    assert not torch.equal(after[2], before[2])
    for a in (after, after2):
        assert relerr(a[2].cpu().numpy(), fresh[2].cpu().numpy()) < 1e-6
        assert relerr(a[3].cpu().numpy(), fresh[3].cpu().numpy()) < 1e-6
        assert float((a[0][3] - fresh[0][3]).abs().max()) < 1e-6


def test_ts_learned_unsupported_shape_keeps_the_per_step_path():
    """Shapes the ring kernel does not take go through TS's per-step path, as before: a learned k = 5 net with 32 hidden
    channels (one ring-kernel tile holds 16 output channels) gives what the per-step composition gives.  On a grid whose
    coarsest level is shorter than the k = 5 strip the reference's 9-region conv itself has no valid form: TS still refuses
    it in the module-level forward, as before, and builds no fused plan."""
    spec = RN.NetSpec(levels=2, c_i=7, c_h=32, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0,
                      repeats=1, f=5, p_pred=False)
    net = _net(spec, seed=5)
    H, W = 40, 56
    assert not engine.fused_supported(net, 1, H, W)
    xc, yc = synthetic_grid(H, W)
    T0 = synthetic_T0(H, W)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=2, scale=True, p_pred=False, net="newfluidnet")
    x, dts, u, v, p, V = _ts_call(ts, T0, xc, yc)
    assert ts._plan is None
    # the per-step composition of TS.forward's loop
    grid = engine.Grid(torch.tensor(xc), torch.tensor(yc), torch.tensor(yc), torch.device(DEV))
    nd = RN.nondim_params(*PARAMS)
    members = ops.make_members([PARAMS], DEV, nd_override=[tuple(float(t) for t in nd)])
    Tc = torch.tensor(T0, dtype=torch.float64).to(DEV).reshape(1, H, W).float().contiguous()
    for i in (1, 2):
        inp, _ = ops.build_input(Tc, grid.xc, grid.yc, grid.ycc, members, want_V=True)
        uu, vv, _ = net(ops.unpack_nchw(inp, 7))
        s = members[:, 6].reshape(1, 1, 1)
        uu, vv = (uu.float() * s).contiguous(), (vv.float() * s).contiguous()
        uvmax = ops.uvmax_reduce(uu, vv, batch_global=True)
        Tc, _, _ = ops.advect_diffuse(Tc, uu, vv, grid.xcoef, grid.ycoef, members, uvmax, grid.dx_min, 0.99,
                                      per_member_dt=False)
        assert float((x[i][:, 0].float() - Tc).abs().max()) <= 1e-6, i
    # (up to the order of the statistics' double-precision atomics)
    assert relerr(u[:, 0].cpu().numpy(), uu.cpu().numpy()) <= 1e-6 and relerr(v[:, 0].cpu().numpy(), vv.cpu().numpy()) <= 1e-6

    spec5, _, _, w = load_learned_case("learned_k5")  # 3 levels, k = 5
    small = _net(spec5, w)
    Hs, Ws = 20, 28  # coarsest level 5 x 7: shorter than the 6-row strip
    assert not engine.fused_supported(small, 1, Hs, Ws)
    xs, ys = synthetic_grid(Hs, Ws)
    ts5 = P.TS(small, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=False, net="newfluidnet")
    with pytest.raises(L.PbmcError):
        _ts_call(ts5, synthetic_T0(Hs, Ws), xs, ys)
    assert ts5._plan is None


# ------------------------------------------------------------------------------------------------ ensemble
def test_ensemble_rollout_learned():
    _, net = _learned_k3_p()
    H, W = 64, 96
    params = [PARAMS, (PARAMS[0] * 0.6, PARAMS[1] * 3.0, PARAMS[2]), (PARAMS[0], PARAMS[1] * 0.3, PARAMS[2] * 0.5),
              (PARAMS[0] * 1.3, PARAMS[1], PARAMS[2] * 2.0)]
    T0 = np.stack([synthetic_T0(H, W, seed=s) for s in range(4)])
    nz = noise("learned_k3_p")

    def run(ps, T, mode):
        ens = EnsembleRollout(net, H, W, ps, DEV, per_member_dt=True, max_steps=64)
        ens.set_T(T)
        if mode == "step":
            ens.step(10)
        else:
            ens.run(10, steps_per_graph=5)
        torch.cuda.synchronize()
        u, v, p, V = ens.fields()
        return ens.T.clone(), u.clone(), v.clone(), p.clone(), ens.time.clone()

    full = run(params, T0, "step")
    graphed = run(params, T0, "graph")
    for b in range(4):
        one = run([params[b]], T0[b:b + 1], "step")
        assert float((full[0][b] - one[0][0]).abs().max()) <= 1e-5, b
        for k, n in ((1, "u"), (2, "v"), (3, "p")):
            assert relerr(full[k][b].cpu().numpy(), one[k][0].cpu().numpy()) <= field_bound(nz[n]), (b, n)
        assert abs(float(full[4][b]) - float(one[4][0])) <= 3e-5 * abs(float(one[4][0])), b
    assert float((full[0] - graphed[0]).abs().max()) <= 1e-5
    for k, n in ((1, "u"), (2, "v"), (3, "p")):
        assert relerr(graphed[k].cpu().numpy(), full[k].cpu().numpy()) <= field_bound(nz[n]), n
    # the ring kernel adds its statistics with double-precision atomics from many CTAs: the order (and so the last bits)
    # may differ from run to run, so bit-identity of the graphed and the direct run is reported, not asserted
    same = all(torch.equal(a, b) for a, b in zip(full[:4], graphed[:4]))
    print(f"[ensemble learned] run(10, steps_per_graph=5) bit-identical to step(10): {same}")
    # members with different parameters really differ (per-member dt and scaler)
    assert len({float(t) for t in full[4]}) > 1


def test_driver_per_step_and_resident_agree_learned(tmp_path):
    """driver.attempt (TS, one call per step) and driver.attempt_resident (EnsembleRollout, k steps per CUDA graph) run a
    learned net and log the same simulated times and temperatures."""
    from pbml_mantle_convection_b200 import driver as D

    _, net = _learned_k3_p()
    H, W = 64, 96
    xc, yc = synthetic_grid(H, W)
    T0 = synthetic_T0(H, W)
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    xcc, ycc = t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W)
    nd = RN.nondim_params(*PARAMS)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=True, net="newfluidnet")
    t_a, n_a, (snap_a, _, tv_a, Tv_a) = D.attempt(ts, t64(T0).view(1, 1, H, W), xcc, ycc, t64(PARAMS[0]), t64(PARAMS[1]),
                                                  t64(PARAMS[2]), t64(nd[0]), t64(nd[1]), t64(nd[2]), t_end=1.0,
                                                  out_dir=str(tmp_path / "a"), max_steps=8, save_every=0.0)
    assert ts._plan is not None  # the fused rollout, not the per-step composition
    ens = P.EnsembleRollout(net, H, W, [PARAMS], DEV, xc=xc, yc=yc, cn_max=0.99, per_member_dt=False)
    ens.set_T(T0[None])
    t_b, n_b, (snap_b, _, tv_b, Tv_b) = D.attempt_resident(ens, xcc, ycc, t_end=1.0, out_dir=str(tmp_path / "b"), max_steps=8,
                                                           check_every=4, save_every=0.0)
    assert n_a == 8 and n_b == 8
    assert np.allclose(tv_a["ML"], tv_b["ML"], rtol=3e-5)
    assert abs(Tv_a["ML"][8] - Tv_b["ML"][8]) < 1e-5
    assert np.abs(snap_a["ML"]["T"][-1] - snap_b["ML"]["T"][-1]).max() < 1e-5
