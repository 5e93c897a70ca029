"""Run-to-time clock without a GPU: the refusals of pbmc_rollout_clocked (checked before any CUDA call) and the log
assembly of driver.attempt_ensemble against driver.attempt, with a stand-in ensemble that follows the device clock's
rules (include/pbmc.h, pbmc_member_clock) on scripted per-member dynamics."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import driver as D

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


def test_clocked_rollout_refusals(lib):
    n = _net()
    d = C.c_void_p(0x1000)

    def call(clock=d, dt=d, meanT=d, ring=d, meta=d, slots=4, per_member_dt=1, B=2):
        return lib.pbmc_rollout_clocked(d, C.byref(n), d, d, d, d, d, d, 0.01, 0.99, per_member_dt, d, 2, 1, 4, dt, 8, d, d, d,
                                        d, d, 1 << 30, B, 64, 96, clock, meanT, ring, meta, slots, None)

    assert call(clock=None) == -3
    assert call(dt=None) == -3
    assert call(meanT=None) == -3
    assert call(ring=None) == -3 and call(meta=None) == -3
    assert call(slots=0) == -1
    assert call(per_member_dt=0) == -2           # batch-global dt: freezing one member would change the others' dt
    assert call(per_member_dt=0, B=1) != -2      # one member: its dt is its own (fails later, on the dummy pointers)
    assert lib.pbmc_sizeof(b"pbmc_member_clock") == C.sizeof(L.MemberClock)


def fake_ts_factory(dt, decay):
    """TS.forward stand-in (ts=1): T *= decay, constant dt, u = 1, v = 2, p = 3, V = 4."""

    def fake_ts(Tp, *a):
        f = lambda c: torch.full_like(Tp, c)
        return {0: Tp, 1: Tp * decay}, {1: torch.tensor(dt, dtype=torch.float64)}, f(1.0), f(2.0), f(3.0), f(4.0)

    return fake_ts


class FakeEnsemble:
    """EnsembleRollout's clocked interface on scripted members (member m: T *= decay[m], dt = dt[m] every step), with the
    device clock's rules: active = t < t_end and steps < max_steps before a step; after it t += dt, steps += 1, mean-T
    logged, snapshot (T after the step, u, v, p) when t > save_t, then save_t = t + save_every; frozen members log nothing."""

    def __init__(self, T0, dts, decays):
        self.B, self.H, self.W = T0.shape
        self._T = T0.copy()
        self.dts, self.decays = dts, decays

    @property
    def T(self):
        return torch.from_numpy(self._T)

    def start_clock(self, t_end, save_every=0.0, t0=0.0, max_steps=None, n_step=0, snap_slots=None):
        bc = lambda x, dt=np.float64: np.broadcast_to(np.asarray(x, dtype=dt), (self.B,)).copy()
        self.t, self.t_end, self.save_every = bc(t0), bc(t_end), bc(save_every)
        self.save_t = np.zeros(self.B)
        self.steps = bc(n_step, np.int64)
        self.max_steps = bc(1 << 62 if max_steps is None else max_steps, np.int64)
        self.slots = snap_slots
        self.blocks = []
        self.snap_steps = [[] for _ in range(self.B)]

    def _active(self, m):
        return self.t[m] < self.t_end[m] and self.steps[m] < self.max_steps[m]

    def any_active(self):
        return any(self._active(m) for m in range(self.B))

    def run(self, n_steps, steps_per_graph, track_time=True):
        assert n_steps == steps_per_graph
        self._blk = []
        for m in range(self.B):
            d = {"dt": [], "t": [], "meanT": [], "steps": [], "snapshots": []}
            for _ in range(n_steps):
                if not self._active(m):
                    continue
                self._T[m] = self._T[m] * self.decays[m]
                self.t[m] = self.t[m] + self.dts[m]
                self.steps[m] += 1
                d["dt"].append(self.dts[m])
                d["t"].append(self.t[m])
                d["meanT"].append(self._T[m].reshape(-1).mean())
                d["steps"].append(self.steps[m])
                if self.t[m] > self.save_t[m]:
                    f = lambda c: np.full((self.H, self.W), c)
                    d["snapshots"].append({"step": int(self.steps[m]), "t": float(self.t[m]), "T": self._T[m].copy(),
                                           "u": f(1.0), "v": f(2.0), "p": f(3.0)})
                    self.snap_steps[m].append(int(self.steps[m]))
                    self.save_t[m] = self.t[m] + self.save_every[m]
            assert len(d["snapshots"]) <= self.slots
            self._blk.append({k: (np.asarray(v) if k != "snapshots" else v) for k, v in d.items()})
        self.blocks.append([len(d["dt"]) for d in self._blk])

    def drain(self):
        return self._blk

    def stop_clock(self):
        pass


def _grid():
    x = torch.linspace(0, 4, W, dtype=torch.float64).view(1, 1, 1, W).expand(1, 1, H, W).contiguous()
    y = torch.linspace(0, 1, H, dtype=torch.float64).view(1, 1, H, 1).expand(1, 1, H, W).contiguous()
    return x, y


def _load(d, name):
    with open(d / name, "rb") as fh:
        return pickle.load(fh)


def test_attempt_ensemble_logs_equal_per_member_attempt(tmp_path):
    xcc, ycc = _grid()
    rng = np.random.default_rng(3)
    T0 = 1.0 + rng.random((3, H, W))
    dts, decays = [0.25, 0.1, 0.4], [0.9, 0.97, 0.8]
    t_end, save_every, k = 2.0, 0.5, 4
    ens = FakeEnsemble(T0, dts, decays)
    t_e, n_e, logs = D.attempt_ensemble(ens, xcc, ycc, t_end=t_end, out_dir=str(tmp_path / "ens"), save_every=save_every,
                                        write_every=0.3, check_every=k)
    # different dt: the members stop at different step counts, inside a block
    assert [int(x) for x in n_e] == [8, 20, 5]
    per_block = np.array(ens.blocks)
    assert (per_block[:, 0] == [4, 4, 0, 0, 0]).all() and (per_block[:, 2] == [4, 1, 0, 0, 0]).all()
    # member 0 (dt = 0.25): the save_t crossing at t = 1.0 is step 4, the last step of block 1; save_t = 1.5 then applies
    # from the first step of block 2 on (snapshots at steps 1, 4, 7)
    assert ens.snap_steps[0] == [1, 4, 7]
    # member 1 (dt = 0.1): snapshots at t = 0.1, 0.7, 1.3, 1.9, spread over blocks 1, 2, 4, 5
    assert len(_load(tmp_path / "ens" / "member_1", "snapshots_ML.pkl")["T"]) == 1 + 4
    one = torch.tensor(1.0, dtype=torch.float64)
    for m in range(3):
        t_a, n_a, _ = D.attempt(fake_ts_factory(dts[m], decays[m]), torch.tensor(T0[m]).view(1, 1, H, W), xcc, ycc,
                                *([one] * 6), t_end=t_end, out_dir=str(tmp_path / f"ref{m}"), save_every=save_every,
                                write_every=0.3)
        assert n_a == n_e[m] and t_a == t_e[m]
        da, de = tmp_path / f"ref{m}", tmp_path / "ens" / f"member_{m}"
        for name in ("t_vec_ML.pkl", "T_vec_ML.pkl"):
            a, e = _load(da, name), _load(de, name)
            assert len(a) == len(e) and all(np.array_equal(x, y) for x, y in zip(a, e)), (m, name)
        assert len(_load(da, "TS_vec_ML.pkl")) == len(_load(de, "TS_vec_ML.pkl")) == n_a
        a, e = _load(da, "snapshots_ML.pkl"), _load(de, "snapshots_ML.pkl")
        assert sorted(a) == sorted(e)
        assert torch.equal(a["xcc"], e["xcc"]) and torch.equal(a["ycc"], e["ycc"])
        for var in ("T", "v", "P"):
            assert len(a[var]) == len(e[var]) and all(np.array_equal(x, y) for x, y in zip(a[var], e[var])), (m, var)


def test_attempt_ensemble_step_limit_and_restart_arguments(tmp_path):
    xcc, ycc = _grid()
    T0 = np.full((2, H, W), 2.0)
    ens = FakeEnsemble(T0, [0.25, 0.5], [0.9, 0.9])
    t_e, n_e, logs = D.attempt_ensemble(ens, xcc, ycc, t_end=[100.0, 6.0], out_dir=str(tmp_path), t=5.0, n_step=40, max_steps=47,
                                        check_every=3, mode="ML_STOKES")
    assert list(n_e) == [47, 42] and t_e[0] == 5.0 + 7 * 0.25 and t_e[1] == 6.0
    assert len(logs[0][2]["ML_STOKES"]) == 1 + 7 and (tmp_path / "member_1" / "T_vec_ML_STOKES.pkl").exists()
