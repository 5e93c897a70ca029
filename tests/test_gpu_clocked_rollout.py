"""Run-to-time clock of the device-resident rollout (pbmc_rollout_clocked, EnsembleRollout.start_clock / drain,
driver.attempt_ensemble) on the GPU: agreement with the reference's per-step loop (driver.attempt with TS(ts=1)), frozen
members, per-step mean-T, snapshots at every step, a full snapshot ring, other grid shapes and networks, and no re-capture
when t_end changes."""
import numpy as np
import pytest
import torch

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import driver as D
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_grid
from tests._util import load_weights, noise, relerr
from tests.test_gpu_net import PARAMS, T_bound, dt_bound, make_net

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
PRM = [PARAMS, (0.9, 3.0e6, 1.5), (9.1, 5.0e9, 60.0)]
H, W = 64, 96


def _net():
    return make_net(RN.NetSpec(levels=4), load_weights("roll64x96"), impl="auto")


def _T0(B, H=H, W=W):
    return np.stack([RN.synthetic_T0(H, W, seed=1 + m) for m in range(B)])


def _ens(net, B=3, **kw):
    ens = EnsembleRollout(net, H, W, PRM[:B], DEV, **kw)
    ens.set_T(_T0(B))
    return ens


def _save_steps(t_vec, save_every):
    """Steps (1-based) at which the reference takes a snapshot, and the smallest relative margin of its comparisons."""
    save_t, steps, margin = 0.0, [], np.inf
    for j, t in enumerate(t_vec[1:], start=1):
        margin = min(margin, abs(t - save_t) / t)
        if t > save_t:
            steps.append(j)
            save_t = t + save_every
    return steps, margin


def test_attempt_ensemble_agrees_with_per_step_reference_loop(tmp_path):
    net = _net()
    xc, yc = synthetic_grid(H, W)
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    xcc, ycc = t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W)
    T0 = _T0(3)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=True, net="newfluidnet")

    def per_step(m, out, **kw):
        nd = RN.nondim_params(*PRM[m])
        return D.attempt(ts, t64(T0[m]).view(1, 1, H, W), xcc, ycc, *(t64(x) for x in PRM[m]), *(t64(x) for x in nd),
                         out_dir=str(tmp_path / out), **kw)

    # the reference's own times (a snapshot every step) choose t_end / save_every with a margin of >= 1e-4 relative on every
    # stop and save comparison, so that fp32 dt noise (~3e-5) cannot flip a step
    stop = [9, 11, 13]
    t_end, save_every, every_step = [], [], []
    for m in range(3):
        _, _, (snaps, _, tv, _) = per_step(m, f"probe{m}", t_end=np.inf, max_steps=stop[m] + 3, save_every=0.0)
        tv = np.array(tv["ML"], dtype=np.float64)
        every_step.append(np.stack(snaps["ML"]["T"]))  # T after every step (index 0: initial)
        t_end.append(0.5 * (tv[stop[m]] + tv[stop[m] + 1]))  # the member takes stop + 1 steps
        assert min(abs(tv[1:] - t_end[m]) / t_end[m]) >= 1e-4
        for f in (2.5, 2.3, 2.7, 2.1, 2.9, 3.3):
            se = f * (tv[stop[m] + 1] - tv[0]) / (stop[m] + 1)
            _, margin = _save_steps(tv[:stop[m] + 2], se)
            if margin >= 1e-4:
                break
        assert margin >= 1e-4, m
        save_every.append(se)
    ref = [per_step(m, f"ref{m}", t_end=t_end[m], save_every=save_every[m]) for m in range(3)]

    ens = EnsembleRollout(net, H, W, PRM, DEV, xc=xc, yc=yc, cn_max=0.99)
    ens.set_T(T0)
    t_e, n_e, logs = D.attempt_ensemble(ens, xcc, ycc, t_end=t_end, out_dir=str(tmp_path / "ens"), save_every=save_every,
                                        check_every=4)
    bound = dt_bound(noise("roll64x96"))
    for m in range(3):
        t_a, n_a, (snap_a, TS_a, tv_a, Tv_a) = ref[m]
        snap_e, TS_e, tv_e, Tv_e = logs[m]
        assert n_a == n_e[m] == stop[m] + 1
        tv_a, tv_e = np.array(tv_a["ML"], dtype=np.float64), np.array(tv_e["ML"], dtype=np.float64)
        assert tv_a.shape == tv_e.shape and np.all(np.abs(tv_e - tv_a) <= bound * np.maximum(tv_a, 1e-300))
        assert np.abs(np.array(Tv_e["ML"], dtype=np.float64) - np.array(Tv_a["ML"], dtype=np.float64)).max() <= 1e-6
        assert len(TS_e["ML"]) == n_a
        steps, _ = _save_steps(tv_a, save_every[m])
        assert len(snap_a["ML"]["T"]) == len(snap_e["ML"]["T"]) == 1 + len(steps)
        for s, Te, Ta in zip(steps, snap_e["ML"]["T"][1:], snap_a["ML"]["T"][1:]):
            # the snapshot is the T of step s: nearest of every step's T, and within T_bound of the reference's
            d = np.abs(every_step[m].reshape(len(every_step[m]), -1) - Te[None]).max(axis=1)
            assert int(np.argmin(d)) == s, (m, s, d)
            assert np.abs(Te - Ta).max() <= T_bound(noise("roll64x96")["step10"]["T_maxabs"])
        for name in ("snapshots_ML.pkl", "t_vec_ML.pkl", "T_vec_ML.pkl", "TS_vec_ML.pkl"):
            assert (tmp_path / "ens" / f"member_{m}" / name).exists()


def test_frozen_members_stay_frozen():
    ens = _ens(_net())
    ens.step(2)
    t2 = ens.time.cpu().numpy()
    ens.start_clock([t2[0] * 2.0, np.inf, np.inf])  # member 0 stops after about two more steps
    k, frozen_T = 4, None
    for blk in range(3):
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k)
        logs = ens.drain()
        if blk == 0:
            assert 0 < len(logs[0]["dt"]) < k and len(logs[1]["dt"]) == k
            frozen_T = ens.T[0].clone()
        else:
            assert len(logs[0]["dt"]) == 0 and logs[0]["snapshots"] == [] and len(logs[0]["meanT"]) == 0
            assert torch.equal(ens.T[0], frozen_T)
            assert (ens.state.dt_seq[par:par + k, 0] == 0).all()
            assert len(logs[1]["dt"]) == k
    ck = ens.read_clock()
    assert not ck["active"][0] and ck["active"][1]
    tt = ens.time.cpu().numpy()
    assert np.all(np.abs(ck["t"] - tt) <= 1e-12 * tt)
    assert ens.any_active()


def test_mean_T_per_step():
    ens = _ens(_net())
    ens.start_clock(np.inf)
    for _ in range(2):
        ens.run(5, steps_per_graph=5)
        logs = ens.drain()
        for m in range(3):
            assert len(logs[m]["meanT"]) == 5
            assert abs(logs[m]["meanT"][-1] - ens.T[m].double().mean().item()) <= 1e-12


def test_snapshot_every_step_matches_unclocked_steps():
    net = _net()
    ens, ref = _ens(net), _ens(net)
    ens.start_clock(np.inf, save_every=0.0, steps_per_graph=4)
    snaps = []
    for _ in range(2):
        ens.run(4, steps_per_graph=4)
        logs = ens.drain()
        for m in range(3):
            assert [s["step"] for s in logs[m]["snapshots"]] == list(logs[m]["steps"])
            assert [s["t"] for s in logs[m]["snapshots"]] == list(logs[m]["t"])
        snaps.append(logs)
    for blk in range(2):
        for j in range(4):
            ref.step(1)
            u, v, p, _ = ref.fields()
            for m in range(3):
                s = snaps[blk][m]["snapshots"][j]
                assert s["step"] == 4 * blk + j + 1
                assert np.abs(s["T"] - ref.T[m].cpu().numpy()).max() < 2e-6
                for name, f in (("u", u), ("v", v), ("p", p)):
                    assert relerr(s[name], f[m].cpu().numpy()) <= 1e-5, (blk, j, m, name)


def test_full_ring_skips_and_raises_without_writing_past_it():
    ens = _ens(_net())
    ens.start_clock(np.inf, save_every=0.0, snap_slots=2)
    clk = ens._clk
    sentinel = -12345.0
    ring = torch.full((clk.slots + 2,) + tuple(clk.ring.shape[1:]), sentinel, dtype=torch.float32, device=DEV)
    meta = torch.full((clk.slots + 2,) + tuple(clk.meta.shape[1:]), sentinel, dtype=torch.float64, device=DEV)
    clk.ring, clk.meta = ring[1:-1], meta[1:-1]  # guard slots on both sides
    ens.run(4, steps_per_graph=4)  # four snapshots due, two slots, no drain in between
    with pytest.raises(L.PbmcError, match="overflow"):
        ens.drain()
    torch.cuda.synchronize()
    for g in (ring[0], ring[-1]):
        assert (g == sentinel).all()
    for g in (meta[0], meta[-1]):
        assert (g == sentinel).all()
    assert (meta[1:-1, :, 0].cpu().numpy() == [[1.0] * 3, [2.0] * 3]).all()  # steps 1 and 2 were kept
    ck = ens.read_clock()
    assert ck["overflow"].all() and (ck["snaps"] == 2).all() and (ck["steps"] == 4).all()


def _learned_small():
    spec = RN.NetSpec(levels=3, c_i=7, c_h=16, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0,
                      repeats=2, f=5, p_pred=False)
    torch.manual_seed(5)
    net = P.NewFluidNet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p="learned", loss_type="curl",
                        use_symm=False, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    with torch.no_grad():
        for mod in net.modules():
            if isinstance(mod, P.BoundaryLearnedConvolution2D):
                mod.learnable_bias.normal_(0.0, 0.1)
    return net.to(DEV).eval()


@pytest.mark.parametrize("case", ["primary_128x506", "learned_k5"])
def test_clocked_equals_unclocked_on_other_shapes(case):
    net, (h, w) = (_net(), (128, 506)) if case == "primary_128x506" else (_learned_small(), (H, W))
    outs = []
    for clocked in (False, True):
        ens = EnsembleRollout(net, h, w, PRM[:2], DEV)
        ens.set_T(_T0(2, h, w))
        if clocked:
            ens.start_clock(np.inf, save_every=0.0, steps_per_graph=5)
        for _ in range(2):
            ens.run(5, steps_per_graph=5)
            if clocked:
                logs = ens.drain()
                assert all(len(d["dt"]) == 5 and len(d["snapshots"]) == 5 for d in logs)
        outs.append((ens.T.clone(), ens.time.clone()))
    (T_a, t_a), (T_b, t_b) = outs
    assert (T_a - T_b).abs().max().item() < 2e-6
    assert ((t_a - t_b).abs() <= 1e-6 * t_a).all()


def test_changing_t_end_needs_no_recapture():
    ens = _ens(_net())
    ens.step(1)
    t1 = ens.time.cpu().numpy()
    ens.start_clock(t1 * 2.5)  # every member stops within the first block of 4
    ens.run(4, steps_per_graph=4)
    logs = ens.drain()
    assert all(0 < len(d["dt"]) < 4 for d in logs) and not ens.any_active()
    n_graphs = len(ens._graphs)
    ens.run(4, steps_per_graph=4)
    assert all(len(d["dt"]) == 0 for d in ens.drain())
    ens.set_t_end(np.inf)
    assert ens.any_active()
    ens.run(4, steps_per_graph=4)
    assert all(len(d["dt"]) == 4 for d in ens.drain())
    assert len(ens._graphs) == n_graphs
