"""Parameter-continuation chains without a GPU: the refusals of pbmc_rollout_chained (checked before any CUDA call) and of
EnsembleRollout.start_sweep(continue_from=...), a host replay of the chained slot rule (include/pbmc.h,
pbmc_member_chain) on hand-built cases, and driver.attempt_sweep's pickles of every member against driver.attempt run
alone from that member's start field, with a stand-in ensemble that follows the documented rule on scripted members."""
import ctypes as C

import numpy as np
import pytest

from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import driver as D
from pbml_mantle_convection_b200.rollout import EnsembleRollout
from tests.test_clock_cpu import _grid
from tests.test_sweep_cpu import FakeSweep, _compare_with_attempt, _T0

H, W = 6, 8


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G

    G.build()
    return L.load()


def _net():
    n = L.Net()
    n.levels, n.repeats, n.c_i, n.c_h, n.c_o, n.ksize = 4, 2, 7, 16, 2, 3
    return n


def test_chained_rollout_refusals(lib):
    n = _net()
    d = C.c_void_p(0x1000)

    def queue(**kw):
        q = L.MemberQueue()
        for name, _ in L.MemberQueue._fields_[:-1]:
            setattr(q, name, 0x1000)
        q.Q = 5
        for k, v in kw.items():
            setattr(q, k, v)
        return q

    def chain(**kw):
        c = L.MemberChain()
        c.heads, c.succ, c.K = 0x1000, 0x1000, 3
        for k, v in kw.items():
            setattr(c, k, v)
        return c

    def diag(**kw):
        g = L.DiagDesc()
        for name in ("flux_seq", "vrms_seq", "hist", "hist_n", "steady", "part"):
            setattr(g, name, 0x1000)
        g.window, g.rtol = 4, 1e-3
        for k, v in kw.items():
            setattr(g, k, v)
        return g

    def call(c, q="ok", g=None, clock=d, slots=4, per_member_dt=1, B=2, H=64):
        q = C.byref(queue()) if q == "ok" else q
        return lib.pbmc_rollout_chained(d, C.byref(n), d, d, d, d, d, d, 0.01, 0.99, per_member_dt, d, 2, 1, 4, d, 8, d, d,
                                        d, d, d, 1 << 30, B, H, 96, clock, d, d, d, slots, q, g, c, None)

    passes = lambda rc: rc not in (-1, -2, -3, -4)  # passes the checks (fails later, on the dummy pointers)
    assert passes(call(C.byref(chain())))             # diag_h may be NULL
    assert call(None) == -3
    assert call(C.byref(chain(heads=None))) == -3 and call(C.byref(chain(succ=None))) == -3
    assert call(C.byref(chain()), q=None) == -3       # a chain needs a queue
    for K in (0, -1, 6):                              # K < 1, K > Q
        assert call(C.byref(chain(K=K))) == -1, K
    assert passes(call(C.byref(chain(K=1)))) and passes(call(C.byref(chain(K=5))))
    # what pbmc_rollout_queued refuses
    for name, _ in L.MemberQueue._fields_[:-1]:
        assert call(C.byref(chain()), q=C.byref(queue(**{name: None}))) == -3, name
    assert call(C.byref(chain()), q=C.byref(queue(Q=0))) == -1
    assert call(C.byref(chain()), q=C.byref(queue(T0=0x1004))) == -4
    # what pbmc_rollout_clocked refuses
    assert call(C.byref(chain()), per_member_dt=0) == -2
    assert call(C.byref(chain()), clock=None) == -3 and call(C.byref(chain()), slots=0) == -1
    # what pbmc_rollout_diagnosed refuses
    assert passes(call(C.byref(chain()), g=C.byref(diag())))
    assert call(C.byref(chain()), g=C.byref(diag(part=None))) == -3
    assert call(C.byref(chain()), g=C.byref(diag(window=-1))) == -1
    assert call(C.byref(chain()), g=C.byref(diag(rtol=float("nan")))) == -1
    assert call(C.byref(chain()), g=C.byref(diag()), H=2) == -1
    assert lib.pbmc_sizeof(b"pbmc_member_chain") == C.sizeof(L.MemberChain)
    for name, st in (("pbmc_member_queue", L.MemberQueue), ("pbmc_diag_desc", L.DiagDesc), ("pbmc_member_clock", L.MemberClock)):
        assert lib.pbmc_sizeof(name.encode()) == C.sizeof(st), name  # unchanged by the chain


BAD = {
    "length": ([-1, 0], {}),
    "float": ([-1, 0.0, -1], {}),
    "bool": ([-1, True, -1], {}),
    "string": ([-1, "0", -1], {}),
    "self": ([-1, 1, -1], {}),
    "later": ([-1, 2, -1], {}),
    "below_minus_one": ([-1, -2, -1], {}),
    "same_predecessor": ([-1, 0, 0], {}),
    "head_takes_no_step": ([-1, 0, -1], {"max_steps": [0, 5, 5]}),
    "successor_takes_no_step": ([-1, 0, -1], {"t_end": [1.0, 0.0, 1.0]}),
    "middle_takes_no_step": ([-1, 0, 1], {"n_step": [0, 7, 0], "max_steps": 7}),
}


@pytest.mark.parametrize("case", list(BAD))
def test_continue_from_refused_before_any_device_work(case):
    cf, kw = BAD[case]
    ens = EnsembleRollout.__new__(EnsembleRollout)  # no device: the arguments are checked first
    with pytest.raises(ValueError):
        ens.start_sweep(np.zeros((3, H, W)), [(1.0, 1.0, 1.0)] * 3, kw.pop("t_end", np.inf), continue_from=cf, **kw)


def test_member_that_takes_no_step_outside_chains_is_not_refused():
    ens = EnsembleRollout.__new__(EnsembleRollout)
    # member 2 takes no step but is in no chain: dropped as without chains, so the checks pass and the call goes on to
    # the device buffers (which this object does not have)
    with pytest.raises(AttributeError):
        ens.start_sweep(np.zeros((3, H, W)), [(1.0, 1.0, 1.0)] * 3, np.inf, max_steps=[3, 3, 0], continue_from=[-1, 0, -1])


# ------------------------------------------------------------------ the slot rule
def chain_rule(max_steps, continue_from, B):
    """Members in each slot at every step (-1: none) under the chain rule of include/pbmc.h, every member able to step
    and stopping on its max_steps only: [step][slot].  After each step the stopping slots, in ascending slot order, hand
    over to their member's successor, or (no successor) take the next chain head while heads remain."""
    Q = len(max_steps)
    succ = {p: q for q, p in enumerate(continue_from) if p >= 0}
    heads = [q for q in range(Q) if continue_from[q] < 0]
    nxt = min(B, len(heads))
    slot = [heads[s] if s < nxt else -1 for s in range(B)]
    left = [max_steps[q] if q >= 0 else 0 for q in slot]
    seq = []
    while any(x > 0 for x in left):
        seq.append([q if x > 0 else -1 for q, x in zip(slot, left)])
        stopped = [s for s in range(B) if left[s] == 1]
        left = [x - 1 if x > 0 else 0 for x in left]
        for s in stopped:
            p = slot[s]
            if p in succ:
                slot[s] = succ[p]
            elif nxt < len(heads):
                slot[s] = heads[nxt]
                nxt += 1
            else:
                continue
            left[s] = max_steps[slot[s]]
    return seq


# (max_steps, continue_from, B, slot occupants of every step)
RULE_CASES = {
    # all three slots stop after step 2: slots 0 and 2 hand over to their successors 3 and 4, slot 1 (no successor) is
    # rank 0 among the head takers and takes head 5; after step 3 slot 0's member 3 has no successor and takes head 6
    "simultaneous": ([2, 2, 2, 1, 3, 2, 1], [-1, -1, -1, 0, 2, -1, -1], 3,
                     [[0, 1, 2], [0, 1, 2], [3, 5, 4], [6, 5, 4], [-1, -1, 4]]),
    # the last head (4) is placed after step 3; the chain 0 -> 2 -> 3 -> 5 goes on in slot 0 after slot 1 froze
    "heads_run_out": ([1, 3, 1, 2, 1, 2], [-1, -1, 0, 2, -1, 3], 2,
                      [[0, 1], [2, 1], [3, 1], [3, 4], [5, -1], [5, -1]]),
    # fewer members than slots: one chain in slot 0, the others stay empty
    "q_below_b": ([1, 2, 1], [-1, 0, 1], 4, [[0, -1, -1, -1], [1, -1, -1, -1], [1, -1, -1, -1], [2, -1, -1, -1]]),
    # two heads for four slots: slot 1 freezes after step 1 with no head left, slot 0 goes on with its successor
    "q_below_b_two_heads": ([2, 1, 2], [-1, -1, 0], 4, [[0, 1, -1, -1], [0, -1, -1, -1], [2, -1, -1, -1], [2, -1, -1, -1]]),
    # without a successor anywhere the rule is the queue's refill rule
    "no_chains": ([1, 2, 3, 1], [-1, -1, -1, -1], 2, [[0, 1], [2, 1], [2, 3], [2, -1]]),
}


@pytest.mark.parametrize("case", list(RULE_CASES))
def test_chain_rule_on_hand_built_cases(case):
    max_steps, cf, B, want = RULE_CASES[case]
    assert chain_rule(max_steps, cf, B) == want
    assert FakeChainSweep.history_of(max_steps, cf, B) == want


# ------------------------------------------------------------------ driver pickles
class FakeChainSweep(FakeSweep):
    """FakeSweep with chains: a stopping slot whose member has a successor hands the member's T over to it (the
    successor's T0 is ignored) and the successor's first drained block carries `start_T`; the other stopping slots, in
    ascending slot order, take the next chain head while heads remain."""

    def start_sweep(self, T0, params, t_end, continue_from=None, **kw):
        super().start_sweep(T0, params, t_end, **kw)
        Q = len(params)
        self.cf = list(continue_from) if continue_from is not None else [-1] * Q
        self.succ = {p: q for q, p in enumerate(self.cf) if p >= 0}
        self.queue = [q for q in self.queue if self.cf[q] < 0]  # the chain heads
        self.next = min(self.B, len(self.queue))
        self.slot = [self.queue[s] if s < self.next else -1 for s in range(self.B)]
        self.history = [list(self.slot)]
        self.starts, self.unreported = {}, set()

    def run(self, n_steps, steps_per_graph, track_time=True):
        assert n_steps == steps_per_graph
        blk, sw = {}, [0] * self.B
        f = lambda c: np.full((H, W), c)
        for _ in range(n_steps):
            stopped = []
            for s, q in enumerate(self.slot):
                if not self._active(q):
                    continue
                d = blk.setdefault(q, {"dt": [], "t": [], "meanT": [], "steps": [], "snapshots": []})
                if q in self.unreported:
                    d["start_T"] = self.starts[q]
                    self.unreported.discard(q)
                self.T[q] = self.T[q] * self.decays[q]
                self.t[q] = self.t[q] + self.dts[q]
                self.steps[q] += 1
                d["dt"].append(self.dts[q])
                d["t"].append(self.t[q])
                d["meanT"].append(self.T[q].reshape(-1).mean())
                d["steps"].append(self.steps[q])
                if self.t[q] > self.save_t[q]:
                    d["snapshots"].append({"step": int(self.steps[q]), "t": float(self.t[q]), "T": self.T[q].copy(),
                                           "u": f(1.0), "v": f(2.0), "p": f(3.0)})
                    self.save_t[q] = self.t[q] + self.save_every[q]
                if not self._active(q):
                    stopped.append(s)
            for s in stopped:  # ascending slot index
                p = self.slot[s]
                if p in self.succ:
                    q = self.succ[p]
                    self.T[q] = self.T[p].copy()
                    self.starts[q] = self.T[p].copy()
                    self.unreported.add(q)
                    self.slot[s] = q
                    sw[s] += 1
                elif self.next < len(self.queue):
                    self.slot[s] = self.queue[self.next]
                    self.next += 1
                    sw[s] += 1
            self.history.append(list(self.slot))
        running = {q for q in self.slot if self._active(q)}
        self._blk = {q: {**{k: (np.asarray(v) if k not in ("snapshots", "start_T") else v) for k, v in d.items()},
                         "finished": q not in running} for q, d in blk.items()}
        self.switches.append(sw)

    @staticmethod
    def history_of(max_steps, cf, B):
        """Slot occupants of every step the fake runs (members with dt = 0 stop on max_steps only)."""
        Q = len(max_steps)
        ens = FakeChainSweep(B, [0.0] * Q, [1.0] * Q)
        ens.start_sweep(np.ones((Q, H, W)), [(1.0, 1.0, 1.0)] * Q, 1.0, max_steps=max_steps, snap_slots=1 << 20,
                        continue_from=cf)
        while ens.any_active():
            ens.run(1, steps_per_graph=1)
        return _occupants(ens, max_steps)


def _occupants(ens, max_steps):
    """[step][slot] members that took each step, from the fake's slot history and the members' step counts."""
    taken = {q: 0 for q in range(len(max_steps))}
    out = []
    for h in ens.history[:-1]:
        row = []
        for q in h:
            if q >= 0 and taken[q] < max_steps[q]:
                taken[q] += 1
                row.append(q)
            else:
                row.append(-1)
        out.append(row)
    while out and out[-1] == [-1] * ens.B:
        out.pop()
    return out


def _run_chained(tmp_path, B, T0, dts, decays, cf, k, **kw):
    xcc, ycc = _grid()
    Q = len(dts)
    ens = FakeChainSweep(B, dts, decays)
    res = D.attempt_sweep(ens, T0, [(1.0, 1.0, 1.0)] * Q, xcc, ycc, out_dir=str(tmp_path / "sweep"), check_every=k,
                          continue_from=cf, **kw)
    starts = np.array([ens.starts[q] if cf[q] >= 0 else T0[q] for q in range(Q)])
    return ens, res, starts


def test_attempt_sweep_chains_equal_attempt_alone_from_the_start_field(tmp_path):
    # two chains and a single member over B = 2 slots; chain 0 -> 2 -> 4 -> 6 stops on t_end (member 2 reaches it after
    # 3 steps, inside block 1), chain 1 -> 3 on max_steps, member 5 is a head that waits for a free slot
    Q, B, k = 7, 2, 4
    T0 = _T0(Q, seed=5)
    dts = [0.25, 0.1, 0.4, 0.3, 0.05, 0.2, 0.5]
    decays = [0.9, 0.97, 0.8, 0.95, 0.99, 0.85, 0.7]
    cf = [-1, -1, 0, 1, 2, -1, 4]
    t_end = [0.5, 9.0, 1.1, 9.0, 0.2, 9.0, 1.0]
    max_steps = [9, 5, 9, 6, 9, 2, 9]
    kw = dict(save_every=0.3, write_every=0.4)
    ens, res, starts = _run_chained(tmp_path, B, T0, dts, decays, cf, k, t_end=t_end, max_steps=max_steps, **kw)
    assert [int(x) for x in res[1]] == [2, 5, 3, 6, 4, 2, 2]
    assert ens.history[0] == [0, 1] and ens.history[2] == [2, 1] and ens.history[5] == [4, 3]
    # a continued member starts from its predecessor's last T (frozen in the fake since), not from its own T0
    for q in (2, 3, 4, 6):
        assert not np.array_equal(starts[q], T0[q]) and np.array_equal(starts[q], ens.T[cf[q]]), q
    _compare_with_attempt(tmp_path, starts, dts, decays, res, lambda q: dict(t_end=t_end[q], max_steps=max_steps[q], **kw))


def test_attempt_sweep_chains_with_restart_arguments_and_simultaneous_stops(tmp_path):
    # slots 0 and 1 stop after the same step: slot 0 hands over to member 2, slot 1 (no successor) takes head 3; t0 and
    # n_step differ per member, and member 4 takes no step outside any chain (dropped, as without chains)
    Q, B, k = 6, 2, 3
    T0 = _T0(Q, seed=9)
    dts, decays = [0.25, 0.25, 0.5, 0.1, 0.2, 0.3], [0.9, 0.8, 0.9, 0.95, 0.85, 0.75]
    t0, n0 = [5.0, 5.0, 1.0, 2.0, 0.0, 0.5], [40, 40, 0, 3, 9, 1]
    max_steps = [42, 42, 3, 100, 9, 5]
    t_end = [100.0, 100.0, 100.0, 2.35, 100.0, 100.0]
    cf = [-1, -1, 0, -1, -1, 2]
    ens, res, starts = _run_chained(tmp_path, B, T0, dts, decays, cf, k, t_end=t_end, t=t0, n_step=n0,
                                    max_steps=max_steps, save_every=0.0)
    assert ens.history[1] == [0, 1] and ens.history[2] == [2, 3]
    assert list(res[1]) == [42, 42, 3, 7, 9, 5]
    _compare_with_attempt(tmp_path, starts, dts, decays, res,
                          lambda q: dict(t_end=t_end[q], t=t0[q], n_step=n0[q], max_steps=max_steps[q], save_every=0.0))


def test_attempt_sweep_without_continue_from_is_unchanged(tmp_path):
    # continue_from=None and all -1 give the same pickles
    Q, B = 5, 2
    T0 = _T0(Q, seed=4)
    dts, decays = [0.25, 0.1, 0.4, 0.3, 0.05], [0.9, 0.97, 0.8, 0.95, 0.99]
    kw = dict(t_end=1.0, max_steps=[2, 3, 4, 1, 5], save_every=0.2)
    xcc, ycc = _grid()
    outs = []
    for name, cf in (("none", None), ("heads", [-1] * Q)):
        ens = FakeChainSweep(B, dts, decays)
        outs.append(D.attempt_sweep(ens, T0, [(1.0, 1.0, 1.0)] * Q, xcc, ycc, out_dir=str(tmp_path / name), check_every=3,
                                    continue_from=cf, **kw))
    (ta, na, la), (tb, nb, lb) = outs
    assert np.array_equal(ta, tb) and np.array_equal(na, nb)
    for a, b in zip(la, lb):
        assert a[2] == b[2] and a[3] == b[3]
        assert all(np.array_equal(x, y) for x, y in zip(a[0]["ML"]["T"], b[0]["ML"]["T"]))
