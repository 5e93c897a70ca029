"""Per-step wall heat flux, rms velocity and the steady stop on the GPU (pbmc_rollout_diagnosed,
EnsembleRollout.start_clock / start_sweep with diagnostics / steady): the logged values against a float64 recomputation
from every step's snapshot, no effect on T / dt / mean-T, the exact stop step of the steady rule (replayed on the host
from the logged doubles), sweeps refilled at the steady stops, and the graphs."""
import numpy as np
import pytest
import torch

from oracle import ref_numpy as RN
from pbml_mantle_convection_b200.rollout import EnsembleRollout
from tests.test_diag_cpu import first_steady, steady_ratios
from tests.test_gpu_clocked_rollout import _learned_small, _net
from tests.test_gpu_sweep import PRM7, _rule

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
# (network, B, H, W): the primary network at 4 x 64^2 and the learned k = 5 network at 2 x 36x44 (member planes of a
# multiple of 4 cells: the float4 pass), and the primary network at 2 x 35x45 (the scalar pass)
CASES = {"primary_4x64x64": (_net, 4, 64, 64), "learned_k5_2x36x44": (_learned_small, 2, 36, 44),
         "primary_2x35x45": (_net, 2, 35, 45)}
K = 4  # steps per graph


def _T0(B, H, W, seed=21):
    return np.stack([RN.synthetic_T0(H, W, seed=seed + m) for m in range(B)])


def _ens(net, B, H, W, params=None):
    ens = EnsembleRollout(net, H, W, params or PRM7[:B], DEV)
    ens.set_T(_T0(B, H, W))
    return ens


def _run(ens, blocks, **clock):
    """start_clock(inf, snapshot every step, **clock), `blocks` blocks of K steps: the drained logs per member,
    concatenated over the blocks (snapshots listed), and the number of graphs after each block."""
    ens.start_clock(np.inf, save_every=0.0, steps_per_graph=K, **clock)
    logs, graphs = [None] * ens.B, []
    for _ in range(blocks):
        ens.run(K, steps_per_graph=K)
        for m, d in enumerate(ens.drain()):
            if logs[m] is None:
                logs[m] = {f: [] for f in d}
            for f, x in d.items():
                logs[m][f].append(x)
        graphs.append(len(ens._graphs))
    out = []
    for d in logs:
        e = {f: (np.concatenate(x) if f not in ("snapshots", "steady") else x) for f, x in d.items()}
        e["snapshots"] = [s for blk in d["snapshots"] for s in blk]
        if "steady" in d:
            e["steady"] = d["steady"][-1]
        out.append(e)
    return out, graphs


def _series(d):
    """[n, 3] (meanT, q_top, vrms): the series the steady rule watches."""
    return np.stack([d["meanT"], d["q_top"], d["vrms"]], axis=1)


@pytest.mark.parametrize("case", list(CASES))
def test_values_against_float64_recomputation_from_snapshots(case):
    mk, B, H, W = CASES[case]
    with torch.no_grad():
        ens = _ens(mk(), B, H, W)
        logs, _ = _run(ens, 2, diagnostics=True)
    y = ens.grid.y1d64.numpy()
    for m, d in enumerate(logs):
        assert len(d["q_bot"]) == len(d["q_top"]) == len(d["vrms"]) == len(d["dt"]) == 2 * K
        assert d["steady"] is False
        for j, s in enumerate(d["snapshots"]):
            T, u, v = (s[f].astype(np.float64) for f in ("T", "u", "v"))
            prof = T.mean(axis=1)
            ref = {"q_bot": -(prof[1] - prof[0]) / (y[1] - y[0]), "q_top": -(prof[-1] - prof[-2]) / (y[-1] - y[-2]),
                   "vrms": np.sqrt(np.mean(u[1:-1, 1:-1] ** 2 + v[1:-1, 1:-1] ** 2))}
            for f, r in ref.items():
                assert np.isfinite(d[f][j]) and abs(d[f][j] - r) <= 1e-12 * abs(r), (case, m, j, f, d[f][j], r)
            assert abs(d["meanT"][j] - T.mean()) <= 1e-12 * abs(T.mean())


def test_diagnostics_change_nothing_else():
    """T, dt and mean-T of a clocked run with diagnostics (and with a steady criterion that never holds) against the same
    run without: bit-identical whenever two runs without diagnostics are (the forward's GroupNorm statistics are atomic
    sums, so two runs may differ in the last bits), otherwise within what two such runs differ by."""
    mk, B, H, W = CASES["primary_4x64x64"]
    net = mk()
    runs = {}
    with torch.no_grad():
        for name, kw in (("off", {}), ("on", {"diagnostics": True}), ("off2", {}), ("steady_never", {"steady": (4, 0.0)})):
            ens = _ens(net, B, H, W)
            logs, _ = _run(ens, 3, **kw)
            runs[name] = (ens.T.cpu().numpy().copy(), [d["dt"] for d in logs], [d["meanT"] for d in logs])
    same = lambda a, b: np.array_equal(a[0], b[0]) and all(np.array_equal(x, y) for i in (1, 2) for x, y in zip(a[i], b[i]))
    repeatable = same(runs["off"], runs["off2"])
    for name in ("on", "steady_never"):
        if repeatable:
            assert same(runs[name], runs["off"]), name
        else:
            assert np.abs(runs[name][0] - runs["off"][0]).max() <= 2e-6
            for a, b in zip(runs[name][1], runs["off"][1]):
                assert np.all(np.abs(a - b) <= 1e-6 * b)
            for a, b in zip(runs[name][2], runs["off"][2]):
                assert np.abs(a - b).max() <= 1e-6
    print(f"two runs without diagnostics bit-identical: {repeatable}")


def _pick_rtol(series, window, n_steps, margin=1.02):
    """An rtol at least `margin` away (relative) from every ratio the rule compares it with, for which the members'
    first steady steps differ the most (None: never within the logs); (rtol, [first steady step per member])."""
    ratios = np.unique(np.concatenate([steady_ratios(s, window) for s in series]))
    ratios = ratios[np.isfinite(ratios) & (ratios > 0)]
    best = None
    for a, b in zip(ratios[:-1], ratios[1:]):
        if b < a * margin * margin:
            continue
        rtol = float(np.sqrt(a * b))
        first = [first_steady(s, window, rtol) for s in series]
        early = [f for f in first if f is not None and f + 1 < n_steps]
        score = (len(set(early)), len(early))
        if len(early) >= 2 and (best is None or score > best[0]):
            best = (score, rtol, first)
    assert best is not None, "no rtol separates the members' stop steps"
    return best[1], best[2]


@pytest.mark.parametrize("case", ["primary_4x64x64", "learned_k5_2x36x44"])
def test_steady_stop_step_flag_and_frozen_T(case):
    mk, B, H, W = CASES[case]
    net, window, blocks = mk(), 3, 6
    N = blocks * K
    with torch.no_grad():
        probe, _ = _run(_ens(net, B, H, W), blocks, diagnostics=True)
        rtol, first = _pick_rtol([_series(d) for d in probe], window, N)
        ens = _ens(net, B, H, W)
        ens.start_clock(np.inf, save_every=0.0, max_steps=N, steps_per_graph=K, steady=(window, rtol))
        logs, frozen = [[] for _ in range(B)], None
        for blk in range(blocks + 1):  # one block more than any member runs: everyone is frozen in it
            par = ens.n_done % 2
            if blk == blocks:
                frozen = ens.T.clone()
            ens.run(K, steps_per_graph=K)
            for m, d in enumerate(ens.drain()):
                logs[m].append(d)
        assert not ens.any_active()
        assert torch.equal(ens.T, frozen) and (ens.state.dt_seq[par:par + K] == 0).all()
    ck = ens.read_clock()
    stops = []
    for m in range(B):
        d = {f: np.concatenate([b[f] for b in logs[m]]) for f in ("steps", "meanT", "q_top", "vrms")}
        last = int(d["steps"][-1])
        # the first run's first steady step (rtol with a margin: fp32 differences between runs cannot move it)
        want_steady = first[m] is not None and first[m] + 1 < N
        assert last == (first[m] + 1 if want_steady else N), (case, m, first[m], last)
        assert logs[m][-1]["steady"] == want_steady == bool(ck["steady"][m]), (case, m)
        # bit for bit: the rule replayed on this run's own logged doubles first holds after step last - 1 (steady stop),
        # or not before the step limit
        s = first_steady(_series(d), window, rtol)
        assert (s == last - 1) if want_steady else (s is None or s >= N - 1), (case, m, s, last)
        snaps = [x for b in logs[m] for x in b["snapshots"]]
        assert snaps[-1]["step"] == last and torch.equal(frozen[m].cpu(), torch.from_numpy(snaps[-1]["T"]))
        stops.append(last)
    assert len(set(stops)) >= 2, stops


def test_sweep_refills_at_steady_stops_and_matches_members_run_alone():
    mk, _, H, W = CASES["primary_4x64x64"]
    net, Q, B, window, N = mk(), 6, 4, 3, 16
    T0, params = _T0(Q, H, W, seed=31), PRM7[:Q]

    def alone(**kw):
        out = []
        for q in range(Q):
            ens = EnsembleRollout(net, H, W, [params[q]], DEV)
            ens.set_T(T0[q:q + 1])
            ens.start_clock(np.inf, save_every=0.0, max_steps=N, steps_per_graph=K, **kw)
            blk = []
            while ens.any_active():
                ens.run(K, steps_per_graph=K)
                blk.append(ens.drain()[0])
            out.append({f: (np.concatenate([b[f] for b in blk]) if f != "steady" else blk[-1][f])
                        for f in ("steps", "dt", "meanT", "q_bot", "q_top", "vrms", "steady")})
        return out

    with torch.no_grad():
        probe = alone(diagnostics=True)
        rtol, _ = _pick_rtol([_series(d) for d in probe], window, N)
        ref = alone(steady=(window, rtol))
        ens = EnsembleRollout(net, H, W, params[:B], DEV)
        ens.start_sweep(T0, params, np.inf, save_every=0.0, max_steps=N, steps_per_graph=K, steady=(window, rtol))
        seq, logs, n_graphs = [], {q: [] for q in range(Q)}, None
        while ens.any_active():
            par = ens.n_done % 2
            ens.run(K, steps_per_graph=K)
            seq += ens._queue.member_seq[par:par + K].cpu().numpy().tolist()
            for q, d in ens.drain().items():
                logs[q].append(d)
            n_graphs = n_graphs or len(ens._graphs)
            assert len(ens._graphs) == n_graphs  # refills at steady stops re-capture nothing
    taken = [len(r["steps"]) for r in ref]
    assert len(set(taken)) >= 2 and any(r["steady"] for r in ref), taken
    want = _rule(taken, B)  # the refill rank rule, with the stop steps of the members run alone
    assert seq[:len(want)] == want and all(r == [-1] * B for r in seq[len(want):])
    for q in range(Q):
        d = {f: np.concatenate([b[f] for b in logs[q]]) for f in ("steps", "dt", "meanT", "q_bot", "q_top", "vrms")}
        assert list(d["steps"]) == list(ref[q]["steps"]), q
        assert logs[q][-1]["finished"] and logs[q][-1]["steady"] == ref[q]["steady"], q
        assert np.all(np.abs(d["dt"] - ref[q]["dt"]) <= 1e-5 * ref[q]["dt"]), q
        assert np.abs(d["meanT"] - ref[q]["meanT"]).max() <= 1e-6, q
        for f in ("q_bot", "q_top", "vrms"):
            assert np.all(np.abs(d[f] - ref[q][f]) <= 1e-4 * np.abs(ref[q][f])), (q, f)
        # bit for bit on the sweep's own logs: the member's stop follows from the rule replayed on them
        s = first_steady(_series(d), window, rtol)
        assert (s == len(d["steps"]) - 1) if ref[q]["steady"] else (s is None or s >= N - 1), (q, s)


def test_graphs_per_window_and_rtol_and_none_across_blocks():
    mk, B, H, W = CASES["primary_4x64x64"]
    with torch.no_grad():
        ens = _ens(mk(), B, H, W)
        _, g1 = _run(ens, 3, steady=(3, 1e-3))
        assert g1 == [g1[0]] * 3
        _, g2 = _run(ens, 2, steady=(3, 1e-3))  # same (window, rtol): the same buffers and graphs
        assert g2 == [g1[0]] * 2
        _, g3 = _run(ens, 2, steady=(5, 1e-3))  # another window: its own graph
        _, g4 = _run(ens, 2, steady=(3, 2e-3))  # another rtol: its own graph
        assert g3 == [g1[0] + 1] * 2 and g4 == [g1[0] + 2] * 2
        _, g5 = _run(ens, 2, steady=(3, 1e-3))
        assert g5 == [g1[0] + 2] * 2
