"""Sweeps larger than the batch on the GPU (pbmc_rollout_queued, EnsembleRollout.start_sweep, driver.attempt_sweep): the
refill rule's exact step counts and slot sequence, bit-exact refills, agreement with each member run alone and with the
reference's per-step loop, snapshots of slots that switch members inside a block, the empty queue, no re-capture, and
the paper's learned network."""
import numpy as np
import pytest
import torch

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from pbml_mantle_convection_b200 import driver as D
from pbml_mantle_convection_b200 import ops
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_grid
from tests._util import noise
from tests.test_gpu_clocked_rollout import PRM, _net, _save_steps
from tests.test_gpu_net import T_bound, dt_bound

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
H, W = 64, 96
PRM7 = [(PRM[q % 3][0] * (1.0 + 0.05 * q), PRM[q % 3][1], PRM[q % 3][2]) for q in range(8)]  # distinct member rows


def _T0(Q, h=H, w=W):
    return np.stack([RN.synthetic_T0(h, w, seed=11 + q) for q in range(Q)])


def _rule(max_steps, B):
    """Slot occupants (queue entry or -1) of every step under the documented refill rule, all members active from the
    start and stopping on max_steps only: [step][slot]."""
    Q = len(max_steps)
    nxt = min(B, Q)
    slot = [s if s < nxt else -1 for s in range(B)]
    left = [max_steps[q] if q >= 0 else 0 for q in slot]
    seq = []
    while any(x > 0 for x in left) or nxt < Q:
        seq.append([q if x > 0 else -1 for q, x in zip(slot, left)])
        stopped = [s for s in range(B) if left[s] == 1]
        left = [x - 1 if x > 0 else 0 for x in left]
        for s in stopped:
            if nxt < Q:
                slot[s], left[s] = nxt, max_steps[nxt]
                nxt += 1
    return seq


def _alone(net, T0, params, tmp_path, name, h=H, w=W, **kw):
    """Each member run alone (B = 1) through attempt_ensemble: (t, n_step, logs, final T) per member."""
    ens = EnsembleRollout(net, h, w, [params[0]], DEV)
    xc, yc = synthetic_grid(h, w)
    out = []
    for q in range(len(params)):
        ens.members.copy_(ops.make_members([params[q]], DEV))
        ens.set_T(T0[q:q + 1])
        one = {k: (v[q] if isinstance(v, (list, np.ndarray)) else v) for k, v in kw.items()}
        t, n, logs = D.attempt_ensemble(ens, xc, yc, out_dir=str(tmp_path / f"{name}{q}"), **one)
        out.append((t[0], n[0], logs[0], ens.T[0].cpu().numpy().copy()))
    return out


# (max_steps, B, k, refills at block boundaries the case must contain)
#   staggered: one slot stops at a time, several members pass through slot 0 inside block 1
#   simultaneous: all three slots stop after step 2 (the last of block 1) with three members waiting -- ranks 0, 1, 2 take
#   entries 3, 4, 5; slot 1 alone refills mid-block at step 3; slots 0 and 1 stop after step 4 with ONE member waiting --
#   rank 0 (slot 0) takes entry 7, rank 1 (slot 1) finds the queue empty and freezes
SWEEPS = {"staggered": ([1, 2, 3, 5, 6, 9, 11], 3, 4, 0), "simultaneous": ([2, 2, 2, 2, 1, 4, 1, 1], 3, 2, 4)}


@pytest.mark.parametrize("case", list(SWEEPS))
def test_exact_counts_slots_and_agreement_with_members_run_alone(tmp_path, case):
    net = _net()
    max_steps, B, k, min_refills = SWEEPS[case]
    Q = len(max_steps)
    T0 = _T0(Q)
    params = PRM7[:Q]
    want = _rule(max_steps, B)
    ens = EnsembleRollout(net, H, W, params[:B], DEV)
    ens.start_sweep(T0, params, np.inf, save_every=0.0, max_steps=max_steps, steps_per_graph=k)
    seq, logs, refills = [], {q: [] for q in range(Q)}, 0
    while ens.any_active():
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k)
        seq += ens._queue.member_seq[par:par + k].cpu().numpy().tolist()
        for q, d in ens.drain().items():
            logs[q].append(d)
        # a slot refilled after the block's last step i holds the new member's T0 and member row, bit for bit
        i = len(seq)
        for s in range(B):
            if i < len(want) and want[i][s] >= 0 and want[i][s] != want[i - 1][s]:
                q = want[i][s]
                assert ens.read_clock()["slot_member"][s] == q, (case, i, s)
                assert torch.equal(ens.T[s].cpu(), torch.from_numpy(T0[q]).float()), (case, i, s, q)
                assert torch.equal(ens.members[s].cpu(), ops.make_members([params[q]], DEV)[0].cpu()), (case, i, s, q)
                refills += 1
    assert refills >= min_refills
    if case == "simultaneous":  # the member that found the queue empty kept its slot, frozen, with its own member row
        assert want[4] == [7, -1, 5] and torch.equal(ens.members[1].cpu(), ops.make_members([params[6]], DEV)[0].cpu())
    assert seq[:len(want)] == want and all(r == [-1] * B for r in seq[len(want):]) and len(seq) - len(want) < k
    ref = _alone(net, T0, params, tmp_path, "alone", t_end=np.inf, save_every=0.0, max_steps=max_steps, check_every=k)
    bound_dt, bound_T = dt_bound(noise("roll64x96")), T_bound(noise("roll64x96")["step10"]["T_maxabs"])
    for q in range(Q):
        d = {f: np.concatenate([b[f] for b in logs[q]]) for f in ("dt", "t", "meanT", "steps")}
        snaps = [s for b in logs[q] for s in b["snapshots"]]
        assert [b["finished"] for b in logs[q]] == [False] * (len(logs[q]) - 1) + [True]
        assert list(d["steps"]) == list(range(1, max_steps[q] + 1)) and ref[q][1] == max_steps[q]
        _, _, (snap_a, _, tv_a, Tv_a), T_a = ref[q]
        tv_a, Tv_a = np.array(tv_a["ML"][1:], dtype=np.float64), np.array(Tv_a["ML"][1:], dtype=np.float64)
        assert np.all(np.abs(d["t"] - tv_a) <= bound_dt * tv_a), q
        assert d["t"][-1] == np.cumsum(d["dt"])[-1]
        assert np.abs(d["meanT"] - Tv_a).max() <= 1e-6, q
        # a snapshot per step (save_every = 0), every one with its own member, step number and T
        assert [s["step"] for s in snaps] == list(d["steps"]) and [s["t"] for s in snaps] == list(d["t"])
        for s, Ta in zip(snaps, snap_a["ML"]["T"][1:]):
            assert np.abs(s["T"].astype(np.float64).reshape(-1) - Ta).max() <= bound_T, (q, s["step"])
        assert np.abs(snaps[-1]["T"] - T_a).max() <= bound_T


def test_exact_refill_empty_queue_and_no_recapture():
    net = _net()
    Q, B, k = 4, 2, 4
    T0 = _T0(Q)
    max_steps = [4, 6, 5, 3]  # member 0 stops at step 4, the last of block 1: slot 0 is refilled at the block boundary
    ens = EnsembleRollout(net, H, W, PRM7[:B], DEV)
    results = []
    for rep in range(2):
        ens.start_sweep(T0, PRM7[:Q], np.inf, save_every=0.0, max_steps=max_steps, steps_per_graph=k)
        if rep == 1:
            assert len(ens._graphs) == n_graphs  # the same buffers: the first sweep's graphs serve again
        ens.run(k, steps_per_graph=k)
        out = [ens.drain()]
        ck = ens.read_clock()
        assert list(ck["slot_member"]) == [2, 1] and ck["next"] == 3
        assert torch.equal(ens.T[0].cpu(), torch.from_numpy(T0[2]).float())
        assert torch.equal(ens.members[0].cpu(), ops.make_members([PRM7[2]], DEV)[0].cpu())
        assert torch.equal(ens.T[1].cpu(), torch.from_numpy(out[0][1]["snapshots"][-1]["T"]))
        if rep == 0:
            n_graphs = len(ens._graphs)
        while ens.any_active():
            ens.run(k, steps_per_graph=k)
            out.append(ens.drain())
        # block 2: member 1 stops at step 6 and slot 1 takes member 3 (steps 7..9), the queue is then empty; members 2
        # and 3 stop at step 9 and both slots freeze
        assert len(out) == 3 and sorted(out[2]) == [2, 3] and all(d["finished"] for d in out[2].values())
        frozen = ens.T.clone()
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k)  # a block with nothing left to run: slots bit-identical, nothing logged
        assert ens.drain() == {} and not ens.any_active()
        assert torch.equal(ens.T, frozen) and (ens.state.dt_seq[par:par + k] == 0).all()
        assert torch.equal(frozen[0].cpu(), torch.from_numpy(out[2][2]["snapshots"][-1]["T"]))
        assert torch.equal(frozen[1].cpu(), torch.from_numpy(out[2][3]["snapshots"][-1]["T"]))
        assert len(ens._graphs) == n_graphs  # no refill re-captured
        results.append([{q: d["meanT"] for q, d in blk.items()} for blk in out])
    # same inputs, same graphs: the same logs (up to the order of the GroupNorm statistics' atomic sums)
    assert all(a.keys() == b.keys() and all(np.abs(a[q] - b[q]).max() <= 1e-6 for q in a) for a, b in zip(*results))


def test_attempt_sweep_agrees_with_per_step_reference_loop(tmp_path):
    net = _net()
    xc, yc = synthetic_grid(H, W)
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    xcc, ycc = t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W)
    Q, B = 3, 2
    T0 = _T0(Q)
    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=True, net="newfluidnet")

    def per_step(q, out, **kw):
        nd = RN.nondim_params(*PRM[q])
        return D.attempt(ts, t64(T0[q]).view(1, 1, H, W), xcc, ycc, *(t64(x) for x in PRM[q]), *(t64(x) for x in nd),
                         out_dir=str(tmp_path / out), **kw)

    # as in test_attempt_ensemble_agrees_with_per_step_reference_loop: t_end / save_every with a margin >= 1e-4 on every
    # stop and save comparison
    stop = [5, 7, 6]
    t_end, save_every = [], []
    for q in range(Q):
        _, _, (_, _, tv, _) = per_step(q, f"probe{q}", t_end=np.inf, max_steps=stop[q] + 3, save_every=0.0)
        tv = np.array(tv["ML"], dtype=np.float64)
        t_end.append(0.5 * (tv[stop[q]] + tv[stop[q] + 1]))
        assert min(abs(tv[1:] - t_end[q]) / t_end[q]) >= 1e-4
        for f in (2.5, 2.3, 2.7, 2.1, 2.9, 3.3):
            se = f * (tv[stop[q] + 1] - tv[0]) / (stop[q] + 1)
            _, margin = _save_steps(tv[:stop[q] + 2], se)
            if margin >= 1e-4:
                break
        assert margin >= 1e-4, q
        save_every.append(se)
    ref = [per_step(q, f"ref{q}", t_end=t_end[q], save_every=save_every[q]) for q in range(Q)]
    ens = EnsembleRollout(net, H, W, PRM[:B], DEV, xc=xc, yc=yc, cn_max=0.99)
    t_e, n_e, logs = D.attempt_sweep(ens, T0, PRM[:Q], xcc, ycc, t_end=t_end, out_dir=str(tmp_path / "sweep"),
                                     save_every=save_every, check_every=4)
    bound = dt_bound(noise("roll64x96"))
    for q in range(Q):
        t_a, n_a, (snap_a, _, tv_a, Tv_a) = ref[q]
        snap_e, TS_e, tv_e, Tv_e = logs[q]
        assert n_a == n_e[q] == stop[q] + 1
        tv_a, tv_e = np.array(tv_a["ML"], dtype=np.float64), np.array(tv_e["ML"], dtype=np.float64)
        assert tv_a.shape == tv_e.shape and np.all(np.abs(tv_e - tv_a) <= bound * np.maximum(tv_a, 1e-300))
        assert np.abs(np.array(Tv_e["ML"], dtype=np.float64) - np.array(Tv_a["ML"], dtype=np.float64)).max() <= 1e-6
        assert len(TS_e["ML"]) == n_a
        steps, _ = _save_steps(tv_a, save_every[q])
        assert len(snap_a["ML"]["T"]) == len(snap_e["ML"]["T"]) == 1 + len(steps)
        for Te, Ta in zip(snap_e["ML"]["T"][1:], snap_a["ML"]["T"][1:]):
            assert np.abs(Te - Ta).max() <= T_bound(noise("roll64x96")["step10"]["T_maxabs"])
        for name in ("snapshots_ML.pkl", "t_vec_ML.pkl", "T_vec_ML.pkl", "TS_vec_ML.pkl"):
            assert (tmp_path / "sweep" / f"member_{q}" / name).exists()


def _paper_net():
    torch.manual_seed(0)
    net = P.NewFluidNet(5, 7, 16, 1, DEV, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10,
                        repeats=6, f=5, p_pred=False).to(DEV).eval()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, P.BoundaryLearnedConvolution2D):
                m.learnable_bias.normal_(0.0, 0.1)
    return net


def test_sweep_of_the_learned_paper_network(tmp_path):
    h, w = 128, 506
    net = _paper_net()
    xc, yc = synthetic_grid(h, w)
    Q, B, k = 3, 2, 3
    T0 = _T0(Q, h, w)
    max_steps = [2, 4, 3]
    with torch.no_grad():
        ens = EnsembleRollout(net, h, w, PRM7[:B], DEV)
        t_e, n_e, logs = D.attempt_sweep(ens, T0, PRM7[:Q], xc, yc, t_end=np.inf, out_dir=str(tmp_path / "sweep"),
                                         max_steps=max_steps, check_every=k)
        ref = _alone(net, T0, PRM7[:Q], tmp_path, "alone", h, w, t_end=np.inf, max_steps=max_steps, check_every=k)
    for q in range(Q):
        assert n_e[q] == ref[q][1] == max_steps[q]
        tv_a, tv_e = (np.array(x[2]["ML"], dtype=np.float64) for x in (ref[q][2], logs[q]))
        assert np.all(np.abs(tv_e - tv_a) <= 1e-4 * np.maximum(tv_a, 1e-300)), q
        Tv_a, Tv_e = (np.array(x[3]["ML"], dtype=np.float64) for x in (ref[q][2], logs[q]))
        assert np.isfinite(Tv_e).all() and np.abs(Tv_e - Tv_a).max() <= 1e-5, q
