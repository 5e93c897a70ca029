"""Parameter-continuation chains on the GPU (pbmc_rollout_chained, EnsembleRollout.start_sweep(continue_from=...),
driver.attempt_sweep(continue_from=...)): the slot sequence of the chained rule, hand-offs that keep T bit for bit, each
member against that member run alone from its start field, hand-offs at steady stops, all-heads chains against the
sweep without chains, no re-capture, and the paper's learned network."""
import numpy as np
import pytest
import torch

from pbml_mantle_convection_b200 import driver as D
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_grid
from tests._util import noise
from tests.test_chain_cpu import chain_rule
from tests.test_diag_cpu import first_steady
from tests.test_gpu_clocked_rollout import PRM, _net
from tests.test_gpu_diag import _pick_rtol, _series
from tests.test_gpu_net import T_bound, dt_bound
from tests.test_gpu_sweep import _T0, _alone, _paper_net

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
H, W = 64, 96
PRM9 = [(PRM[q % 3][0] * (1.0 + 0.05 * q), PRM[q % 3][1], PRM[q % 3][2]) for q in range(9)]  # distinct member rows
# Q = 9 over B = 3: chains 0 -> 3 -> 6 -> 8 (length 4), 1 -> 5 (2), 4 -> 7 (2) and 2 (1).  Members 0, 1 and 2 stop after
# step 2 together (two hand-offs, and slot 2 takes the last head, 4); 3 and 5 stop after step 4 (3 hands over to 6, 5
# finds no head left and its slot freezes) while the chains 4 -> 7 and 6 -> 8 go on
CF = [-1, -1, -1, 0, -1, 1, 3, 4, 6]
MAX_STEPS = [2, 2, 2, 2, 3, 2, 3, 2, 2]
B, K = 3, 4


def _sweep(ens, T0, params, k, **kw):
    """start_sweep(**kw) and blocks of k steps until no member is left: (member_seq rows, {member: [drained dicts]},
    graph count after every block)."""
    ens.start_sweep(T0, params, kw.pop("t_end", np.inf), save_every=0.0, steps_per_graph=k, **kw)
    seq, logs, graphs = [], {q: [] for q in range(len(params))}, []
    while ens.any_active():
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k)
        seq += ens._member_of(ens._queue.member_seq[par:par + k].cpu().numpy()).tolist()
        for q, d in ens.drain().items():
            logs[q].append(d)
        graphs.append(len(ens._graphs))
    while seq and seq[-1] == [-1] * ens.B:
        seq.pop()
    return seq, logs, graphs


def _cat(blocks, fields=("dt", "t", "meanT", "steps")):
    return {f: np.concatenate([b[f] for b in blocks]) for f in fields if f in blocks[0]}


def _start_fields(T0, logs, cf):
    """Each member's start field: T0 for a head, the drained start_T (float32) for a continued member."""
    out = []
    for q in range(len(cf)):
        if cf[q] < 0:
            assert "start_T" not in logs[q][0]
            out.append(T0[q])
        else:
            assert "start_T" in logs[q][0] and all("start_T" not in b for b in logs[q][1:]), q
            out.append(logs[q][0]["start_T"].astype(np.float64))
    return np.stack(out)


def test_chained_slots_start_fields_and_members_run_alone(tmp_path):
    net = _net()
    Q = len(CF)
    T0 = _T0(Q)
    with torch.no_grad():
        ens = EnsembleRollout(net, H, W, PRM9[:B], DEV)
        seq, logs, _ = _sweep(ens, T0, PRM9, K, max_steps=MAX_STEPS, continue_from=CF)
        assert seq == chain_rule(MAX_STEPS, CF, B)
        starts = _start_fields(T0, logs, CF)
        ref = _alone(net, starts, PRM9, tmp_path, "alone", t_end=np.inf, save_every=0.0, max_steps=MAX_STEPS, check_every=K)
    bound_dt, bound_T = dt_bound(noise("roll64x96")), T_bound(noise("roll64x96")["step10"]["T_maxabs"])
    exact = 0
    for q in range(Q):
        d = _cat(logs[q])
        snaps = [s for b in logs[q] for s in b["snapshots"]]
        assert [b["finished"] for b in logs[q]] == [False] * (len(logs[q]) - 1) + [True]
        assert list(d["steps"]) == list(range(1, MAX_STEPS[q] + 1)) and ref[q][1] == MAX_STEPS[q]
        p = CF[q]
        if p >= 0:
            # the hand-off kept T bit for bit: q starts from p's T after p's last step in this run ...
            last_p = [s for b in logs[p] for s in b["snapshots"]][-1]
            assert last_p["step"] == MAX_STEPS[p] and np.array_equal(logs[q][0]["start_T"], last_p["T"]), q
            # ... which is p's final T run alone from p's start field (to the fp32 noise of two runs)
            exact += int(np.array_equal(logs[q][0]["start_T"], ref[p][3]))
            assert np.abs(logs[q][0]["start_T"] - ref[p][3]).max() <= bound_T, q
        _, _, (snap_a, _, tv_a, Tv_a), T_a = ref[q]
        assert tv_a["ML"][0] == 0.0 and Tv_a["ML"][0] == starts[q].astype(np.float32).astype(np.float64).reshape(-1).mean()
        tv_a, Tv_a = np.array(tv_a["ML"][1:], dtype=np.float64), np.array(Tv_a["ML"][1:], dtype=np.float64)
        assert np.all(np.abs(d["t"] - tv_a) <= bound_dt * tv_a), q
        assert np.abs(d["meanT"] - Tv_a).max() <= 1e-6, q
        assert [s["step"] for s in snaps] == list(d["steps"]) and [s["t"] for s in snaps] == list(d["t"])
        for s, Ta in zip(snaps, snap_a["ML"]["T"][1:]):
            assert np.abs(s["T"].astype(np.float64).reshape(-1) - Ta).max() <= bound_T, (q, s["step"])
    print(f"start fields bit-identical to the predecessor's final T run alone: {exact} of {sum(p >= 0 for p in CF)}")
    # the driver's pickles: attempt_sweep against attempt_ensemble alone from each member's start field
    with torch.no_grad():
        t_e, n_e, logs_e = D.attempt_sweep(ens, T0, PRM9, *synthetic_grid(H, W), t_end=np.inf,
                                           out_dir=str(tmp_path / "sweep"), save_every=0.0, max_steps=MAX_STEPS,
                                           check_every=K, continue_from=CF)
    for q in range(Q):
        assert n_e[q] == MAX_STEPS[q]
        snap_e, TS_e, tv_e, Tv_e = logs_e[q]
        snap_a, _, tv_a, Tv_a = ref[q][2]
        assert len(tv_e["ML"]) == len(tv_a["ML"]) == len(Tv_e["ML"]) == MAX_STEPS[q] + 1 and len(TS_e["ML"]) == MAX_STEPS[q]
        tv_a, tv_e = np.array(tv_a["ML"], dtype=np.float64), np.array(tv_e["ML"], dtype=np.float64)
        assert np.all(np.abs(tv_e - tv_a) <= bound_dt * np.maximum(tv_a, 1e-300)), q
        assert np.abs(np.array(Tv_e["ML"], dtype=np.float64) - np.array(Tv_a["ML"], dtype=np.float64)).max() <= 1e-6, q
        assert len(snap_e["ML"]["T"]) == len(snap_a["ML"]["T"]) == MAX_STEPS[q] + 1
        for Te, Ta in zip(snap_e["ML"]["T"], snap_a["ML"]["T"]):
            assert np.abs(Te - Ta).max() <= bound_T, q
        for name in ("snapshots_ML.pkl", "t_vec_ML.pkl", "T_vec_ML.pkl", "TS_vec_ML.pkl"):
            assert (tmp_path / "sweep" / f"member_{q}" / name).exists()


def test_hand_offs_at_steady_stops():
    net, window, N = _net(), 3, 16
    Q = len(CF)
    T0 = _T0(Q)
    with torch.no_grad():
        ens = EnsembleRollout(net, H, W, PRM9[:B], DEV)
        _, probe, _ = _sweep(ens, T0, PRM9, K, max_steps=N, continue_from=CF, diagnostics=True)
        rtol, _ = _pick_rtol([_series(_cat(probe[q], ("meanT", "q_top", "vrms"))) for q in range(Q)], window, N)
        seq, logs, _ = _sweep(ens, T0, PRM9, K, max_steps=N, continue_from=CF, steady=(window, rtol))
        starts = _start_fields(T0, logs, CF)
        ref = []
        for q in range(Q):  # each member alone from its start field, same criterion
            one = EnsembleRollout(net, H, W, [PRM9[q]], DEV)
            one.set_T(starts[q:q + 1])
            one.start_clock(np.inf, save_every=0.0, max_steps=N, steps_per_graph=K, steady=(window, rtol))
            blk = []
            while one.any_active():
                one.run(K, steps_per_graph=K)
                blk.append(one.drain()[0])
            ref.append({**_cat(blk, ("steps", "dt", "meanT", "q_bot", "q_top", "vrms")), "steady": blk[-1]["steady"]})
    taken = [len(r["steps"]) for r in ref]
    assert any(r["steady"] for r in ref) and any(CF[q] >= 0 and ref[CF[q]]["steady"] for q in range(Q)), taken
    assert seq == chain_rule(taken, CF, B)  # the chained rule with the stop steps of the members run alone
    for q in range(Q):
        d = _cat(logs[q], ("steps", "dt", "meanT", "q_bot", "q_top", "vrms"))
        assert list(d["steps"]) == list(ref[q]["steps"]), q
        assert logs[q][-1]["finished"] and logs[q][-1]["steady"] == ref[q]["steady"], q
        # bit for bit on the sweep's own logs: the member's stop follows from the rule replayed on them
        s = first_steady(_series(d), window, rtol)
        assert (s == len(d["steps"]) - 1) if ref[q]["steady"] else (s is None or s >= N - 1), (q, s)
        if CF[q] >= 0:  # handed over at the predecessor's (steady) stop step, T bit for bit
            last_p = [x for b in logs[CF[q]] for x in b["snapshots"]][-1]
            assert last_p["step"] == taken[CF[q]] and np.array_equal(logs[q][0]["start_T"], last_p["T"]), q
        # fp32 differences between a batch of 3 and a member alone grow over the steps: 1e-5 relative after 6 steps
        assert np.all(np.abs(d["dt"] - ref[q]["dt"]) <= 1e-4 * ref[q]["dt"]), q
        assert np.abs(d["meanT"] - ref[q]["meanT"]).max() <= 1e-6, q
        for f in ("q_bot", "q_top", "vrms"):
            assert np.all(np.abs(d[f] - ref[q][f]) <= 1e-4 * np.abs(ref[q][f])), (q, f)


def _raw_run(ens, T0, params, k, **kw):
    """A sweep's raw per-step device rows and drained snapshots, block by block, and the final T."""
    ens.start_sweep(T0, params, np.inf, save_every=0.0, steps_per_graph=k, max_steps=MAX_STEPS, diagnostics=True, **kw)
    rows = {f: [] for f in ("dt", "meanT", "member", "flux", "vrms", "snaps")}
    while ens.any_active():
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k)
        r = slice(par, par + k)
        rows["dt"].append(ens.state.dt_seq[r].cpu().numpy())
        rows["meanT"].append(ens._clk.meanT_seq[r].cpu().numpy())
        rows["member"].append(ens._queue.member_seq[r].cpu().numpy())
        rows["flux"].append(ens._diag.flux_seq[r].cpu().numpy())
        rows["vrms"].append(ens._diag.vrms_seq[r].cpu().numpy())
        rows["snaps"] += [(q, s["step"], s["T"]) for q, d in sorted(ens.drain().items()) for s in d["snapshots"]]
    return rows, ens.T.cpu().numpy().copy()


def test_all_heads_equal_the_sweep_without_chains_and_graphs_are_reused():
    net = _net()
    Q = len(CF)
    T0 = _T0(Q)
    with torch.no_grad():
        ens = EnsembleRollout(net, H, W, PRM9[:B], DEV)
        runs = {"plain": _raw_run(ens, T0, PRM9, K), "heads": _raw_run(ens, T0, PRM9, K, continue_from=[-1] * Q),
                "plain2": _raw_run(ens, T0, PRM9, K)}
        # a chained sweep: no graph re-captured across its blocks, and a second one with the same Q re-uses them
        _, _, g1 = _sweep(ens, T0, PRM9, K, max_steps=MAX_STEPS, continue_from=CF)
        _, _, g2 = _sweep(ens, T0, PRM9, K, max_steps=MAX_STEPS, continue_from=CF)
        assert g1 == [g1[0]] * len(g1) and g2 == [g1[0]] * len(g2)

    def same(a, b):
        (ra, Ta), (rb, Tb) = a, b
        return np.array_equal(Ta, Tb) and all(np.array_equal(x, y) for f in ("dt", "meanT", "member", "flux", "vrms")
                                              for x, y in zip(ra[f], rb[f])) and \
            len(ra["snaps"]) == len(rb["snaps"]) and \
            all(x[:2] == y[:2] and np.array_equal(x[2], y[2]) for x, y in zip(ra["snaps"], rb["snaps"]))

    (rp, Tp), (rh, Th) = runs["plain"], runs["heads"]
    assert all(np.array_equal(x, y) for x, y in zip(rp["member"], rh["member"]))
    assert [x[:2] for x in rp["snaps"]] == [x[:2] for x in rh["snaps"]]
    repeatable = same(runs["plain"], runs["plain2"])
    if repeatable:
        assert same(runs["heads"], runs["plain"])
    else:  # the forward's GroupNorm statistics are atomic sums: within what two runs without chains differ by
        assert np.abs(Th - Tp).max() <= 2e-6
        for a, b in zip(rh["dt"], rp["dt"]):
            assert np.all(np.abs(a - b) <= 1e-6 * np.abs(b))
        for f, tol in (("meanT", 1e-6), ("flux", 1e-3), ("vrms", 1e-4)):
            for a, b in zip(rh[f], rp[f]):
                assert np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), 1e-30)), f
    print(f"two sweeps without chains bit-identical: {repeatable}")


def test_chain_of_the_learned_paper_network(tmp_path):
    h, w = 128, 506  # the fused engine's smallest supported grid for this network's five levels is not 64 x 96
    net = _paper_net()
    cf, max_steps = [-1, 0, -1, 1], [2, 3, 2, 2]
    Q, b, k = len(cf), 2, 3
    T0 = _T0(Q, h, w)
    with torch.no_grad():
        ens = EnsembleRollout(net, h, w, PRM9[:b], DEV)
        seq, logs, _ = _sweep(ens, T0, PRM9[:Q], k, max_steps=max_steps, continue_from=cf)
        assert seq == chain_rule(max_steps, cf, b)
        starts = _start_fields(T0, logs, cf)
        ref = _alone(net, starts, PRM9[:Q], tmp_path, "alone", h, w, t_end=np.inf, save_every=0.0, max_steps=max_steps,
                     check_every=k)
    for q in range(Q):
        d = _cat(logs[q])
        assert list(d["steps"]) == list(range(1, max_steps[q] + 1)) and ref[q][1] == max_steps[q]
        if cf[q] >= 0:
            last_p = [s for blk in logs[cf[q]] for s in blk["snapshots"]][-1]
            assert np.array_equal(logs[q][0]["start_T"], last_p["T"]), q
            assert np.abs(logs[q][0]["start_T"] - ref[cf[q]][3]).max() <= 1e-4, q
        tv_a = np.array(ref[q][2][2]["ML"][1:], dtype=np.float64)
        Tv_a = np.array(ref[q][2][3]["ML"][1:], dtype=np.float64)
        assert np.all(np.abs(d["t"] - tv_a) <= 1e-4 * np.maximum(tv_a, 1e-300)), q
        assert np.isfinite(d["meanT"]).all() and np.abs(d["meanT"] - Tv_a).max() <= 1e-5, q
