"""Sweeps larger than the batch without a GPU: the refusals of pbmc_rollout_queued (checked before any CUDA call), its
struct against the ctypes mirror, and driver.attempt_sweep's pickles against driver.attempt's for every member, with a
stand-in ensemble that follows the documented refill rule (include/pbmc.h, pbmc_member_queue) on scripted members."""
import ctypes as C

import numpy as np
import pytest
import torch

from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import driver as D
from tests.test_clock_cpu import _grid, _load, fake_ts_factory

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


def test_queued_rollout_refusals(lib):
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

    def call(q, clock=d, slots=4, per_member_dt=1, B=2):
        return lib.pbmc_rollout_queued(d, C.byref(n), d, d, d, d, d, d, 0.01, 0.99, per_member_dt, d, 2, 1, 4, d, 8, d, d, d,
                                       d, d, 1 << 30, B, 64, 96, clock, d, d, d, slots, q, None)

    assert call(None) == -3
    for name, _ in L.MemberQueue._fields_[:-1]:
        assert call(C.byref(queue(**{name: None}))) == -3, name
    assert call(C.byref(queue(Q=0))) == -1 and call(C.byref(queue(Q=-1))) == -1
    assert call(C.byref(queue(T0=0x1004))) == -4                      # refills copy T0 rows with 16-byte loads
    assert call(C.byref(queue()), per_member_dt=0) == -2             # batch-global dt, as the clocked call
    assert call(C.byref(queue()), clock=None) == -3 and call(C.byref(queue()), slots=0) == -1
    assert call(C.byref(queue()), per_member_dt=0, B=1) not in (-1, -2, -3, -4)  # passes the checks (fails on the dummies)
    assert lib.pbmc_sizeof(b"pbmc_member_queue") == C.sizeof(L.MemberQueue)
    assert lib.pbmc_sizeof(b"pbmc_member_clock") == C.sizeof(L.MemberClock)  # unchanged by the queue


class FakeSweep:
    """EnsembleRollout's sweep interface on scripted members (member q: T *= decay[q], dt = dt[q] every step) with the
    device's rules: a member steps while t < t_end and steps < max_steps; after a step t += dt, steps += 1, mean-T logged,
    a snapshot when t > save_t (then save_t = t + save_every).  After every step the slots whose member stopped, in
    ascending slot order (rank r), take queue entries next + r while the queue lasts; members that would take no step
    never enter the queue."""

    def __init__(self, B, dts, decays):
        self.B, self.H, self.W = B, H, W
        self.dts, self.decays = dts, decays

    def start_sweep(self, T0, params, t_end, save_every=0.0, t0=0.0, max_steps=None, n_step=0, snap_slots=None,
                    steps_per_graph=10):
        Q = len(params)
        bc = lambda x, dt=np.float64: np.broadcast_to(np.asarray(x, dtype=dt), (Q,)).copy()
        self.T = torch.as_tensor(T0).double().numpy().reshape(Q, H, W).copy()
        self.t, self.t_end, self.save_every = bc(t0), bc(t_end), bc(save_every)
        self.steps = bc(n_step, np.int64)
        self.max_steps = bc(1 << 62 if max_steps is None else max_steps, np.int64)
        self.save_t = np.zeros(Q)
        self.queue = [q for q in range(Q) if self._active(q)]
        self.next = min(self.B, len(self.queue))
        self.slot = [self.queue[s] if s < self.next else -1 for s in range(self.B)]
        self.slots = snap_slots
        self.history = [list(self.slot)]  # slot occupants after every step
        self.switches = []                # per block: how many refills each slot saw

    def _active(self, q):
        return q >= 0 and self.t[q] < self.t_end[q] and self.steps[q] < self.max_steps[q]

    def any_active(self):
        return any(self._active(q) for q in self.slot) or self.next < len(self.queue)

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
            for s in stopped:  # ascending slot index: rank r takes entry next + r
                if self.next < len(self.queue):
                    self.slot[s] = self.queue[self.next]
                    self.next += 1
                    sw[s] += 1
            self.history.append(list(self.slot))
        running = {q for q in self.slot if self._active(q)}
        self._blk = {q: {**{k: (np.asarray(v) if k != "snapshots" else v) for k, v in d.items()}, "finished": q not in running}
                     for q, d in blk.items()}
        for d in self._blk.values():
            assert len(d["snapshots"]) <= self.slots
        self.switches.append(sw)

    def drain(self):
        return self._blk

    def stop_clock(self):
        pass


def _compare_with_attempt(tmp_path, T0, dts, decays, res, kw_of):
    """attempt_sweep's results / pickles of every member equal driver.attempt's for that member alone."""
    xcc, ycc = _grid()
    t_e, n_e, _ = res
    one = torch.tensor(1.0, dtype=torch.float64)
    for q in range(len(dts)):
        t_a, n_a, _ = D.attempt(fake_ts_factory(dts[q], decays[q]), torch.tensor(T0[q]).view(1, 1, H, W), xcc, ycc,
                                *([one] * 6), out_dir=str(tmp_path / f"ref{q}"), **kw_of(q))
        assert n_a == n_e[q] and t_a == t_e[q], q
        da, de = tmp_path / f"ref{q}", tmp_path / "sweep" / f"member_{q}"
        for name in ("t_vec_ML.pkl", "T_vec_ML.pkl"):
            a, e = _load(da, name), _load(de, name)
            assert len(a) == len(e) and all(np.array_equal(x, y) for x, y in zip(a, e)), (q, name)
        assert len(_load(da, "TS_vec_ML.pkl")) == len(_load(de, "TS_vec_ML.pkl"))
        a, e = _load(da, "snapshots_ML.pkl"), _load(de, "snapshots_ML.pkl")
        assert sorted(a) == sorted(e)
        assert torch.equal(a["xcc"], e["xcc"]) and torch.equal(a["ycc"], e["ycc"])
        for var in ("T", "v", "P"):
            assert len(a[var]) == len(e[var]) and all(np.array_equal(x, y) for x, y in zip(a[var], e[var])), (q, var)


def _T0(Q, seed=3):
    # float32-representable, so that the device's float32 T0 and attempt's float64 T0 are the same numbers
    return (1.0 + np.random.default_rng(seed).random((Q, H, W))).astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("B", [3, 4, 9])  # 6 queued members: a multiple of B, not a multiple, fewer than B
def test_attempt_sweep_logs_equal_per_member_attempt(tmp_path, B):
    xcc, ycc = _grid()
    Q = 8
    T0 = _T0(Q)
    dts = [0.25, 0.1, 0.4, 0.3, 0.05, 0.2, 0.5, 0.15]
    decays = [0.9, 0.97, 0.8, 0.95, 0.99, 0.85, 0.7, 0.93]
    max_steps = [1, 7, 1, 12, 1, 0, 3, 2]   # member 5 takes no step (n_step = 0 = max_steps)
    t_end = [9.0] * Q
    t_end[2] = 0.0                          # member 2 neither: t0 = 0 is not below t_end
    kw = dict(save_every=0.3, write_every=0.4)
    params = [(1.0, 1.0, 1.0)] * Q
    ens = FakeSweep(B, dts, decays)
    res = D.attempt_sweep(ens, T0, params, xcc, ycc, t_end=t_end, out_dir=str(tmp_path / "sweep"), max_steps=max_steps,
                          check_every=4, **kw)
    assert 2 not in ens.queue and 5 not in ens.queue and len(ens.queue) == Q - 2
    assert [int(x) for x in res[1]] == [1, 7, 0, 12, 1, 0, 3, 2]
    if B == 3:
        # slot 0 runs members 0, then 4 (member 0 stops after step 1), then 6 ...: several members inside block 1
        assert ens.history[0] == [0, 1, 3] and ens.history[1] == [4, 1, 3] and ens.history[2] == [6, 1, 3]
        assert max(ens.switches[0]) >= 2
    if B == 9:
        assert ens.history[0] == [0, 1, 3, 4, 6, 7, -1, -1, -1]
    _compare_with_attempt(tmp_path, T0, dts, decays, res,
                          lambda q: dict(t_end=t_end[q], max_steps=max_steps[q], **kw))


def test_attempt_sweep_restart_arguments_and_simultaneous_stops(tmp_path):
    xcc, ycc = _grid()
    Q, B = 5, 2
    T0 = _T0(Q, seed=7)
    dts, decays = [0.25, 0.25, 0.5, 0.1, 0.2], [0.9, 0.8, 0.9, 0.95, 0.85]
    t0, n0 = [5.0, 5.0, 1.0, 2.0, 0.0], [40, 40, 0, 3, 9]
    max_steps = [42, 42, 3, 100, 10]   # members 0 and 1 stop after the same step: slot 0 takes entry 2, slot 1 entry 3
    t_end = [100.0, 100.0, 100.0, 2.35, 100.0]
    ens = FakeSweep(B, dts, decays)
    res = D.attempt_sweep(ens, T0, [(1.0, 1.0, 1.0)] * Q, xcc, ycc, t_end=t_end, out_dir=str(tmp_path / "sweep"), t=t0,
                          n_step=n0, max_steps=max_steps, check_every=3, save_every=0.0, mode="ML")
    assert ens.history[1] == [0, 1] and ens.history[2] == [2, 3]
    assert list(res[1]) == [42, 42, 3, 7, 10]
    _compare_with_attempt(tmp_path, T0, dts, decays, res,
                          lambda q: dict(t_end=t_end[q], t=t0[q], n_step=n0[q], max_steps=max_steps[q], save_every=0.0))
