"""Per-step diagnostics and the steady stop without a GPU: the refusals of pbmc_rollout_diagnosed (checked before any
CUDA call) and of EnsembleRollout's steady argument, a host replay of the steady rule (include/pbmc.h, pbmc_diag_desc)
on hand-built series, and the pickles of driver.attempt_ensemble / attempt_sweep with a stand-in ensemble that logs
scripted fluxes, rms velocities and steady stops."""
import ctypes as C
import math
import pickle

import numpy as np
import pytest
import torch

from pbml_mantle_convection_b200 import _lib as L
from pbml_mantle_convection_b200 import driver as D
from pbml_mantle_convection_b200.rollout import EnsembleRollout

H, W = 6, 8


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G

    G.build()
    return L.load()


# ------------------------------------------------------------------ the steady rule, replayed on logged doubles
def window_steady(win, rtol):
    """The rule on one window [window, 3] of (meanT, q_top, vrms): every value finite and, per series,
    (mx - mn) <= rtol * max(|mx|, |mn|) -- one rounded subtraction and one rounded multiplication, as on the device."""
    win = np.asarray(win, dtype=np.float64)
    if not np.isfinite(win).all():
        return False
    mx, mn = win.max(axis=0), win.min(axis=0)
    return bool(np.all((mx - mn) <= rtol * np.maximum(np.abs(mx), np.abs(mn))))


def first_steady(series, window, rtol):
    """First step s (1-based) after which the member is steady, from its logged series [n, 3]; None if none."""
    for s in range(window, len(series) + 1):
        if window_steady(series[s - window:s], rtol):
            return s
    return None


def steady_ratios(series, window):
    """Per step s >= window: the smallest rtol for which the rule holds after s, as a ratio (what an rtol is compared
    with; inf / nan where no finite rtol makes it hold)."""
    series = np.asarray(series, dtype=np.float64)
    out = []
    for s in range(window, len(series) + 1):
        w = series[s - window:s]
        mx, mn = w.max(axis=0), w.min(axis=0)
        with np.errstate(divide="ignore", invalid="ignore"):
            out.append(np.max((mx - mn) / np.maximum(np.abs(mx), np.abs(mn))) if np.isfinite(w).all() else np.inf)
    return np.array(out)


def test_replay_boundary_cases():
    col = lambda *x: np.array([[v, 1.0, 1.0] for v in x])
    # mx - mn == rtol * max(|mx|, |mn|) exactly (binary fractions): steady; one ulp less rtol: not
    assert window_steady(col(2.0, 1.5), 0.25) and not window_steady(col(2.0, 1.5), np.nextafter(0.25, 0.0))
    # negative means: max(|mx|, |mn|) is |mn|
    assert window_steady(col(-2.0, -1.5), 0.25) and not window_steady(col(-2.0, -1.5), np.nextafter(0.25, 0.0))
    # a sign change: the range is twice the largest magnitude
    assert window_steady(col(-1.0, 1.0), 2.0) and not window_steady(col(-1.0, 1.0), 1.9999999999999998)
    # constant series are steady at rtol = 0, zero ones too; a non-finite value never is
    assert window_steady(col(0.75, 0.75, 0.75), 0.0) and window_steady(np.zeros((3, 3)), 0.0)
    assert not window_steady(col(1.0, np.nan), 1.0) and not window_steady(col(1.0, np.inf), 1e300)
    # every series counts: q_top (column 1) varying alone keeps the member running
    w = np.array([[1.0, 1.0, 1.0], [1.0, 1.25, 1.0]])
    assert not window_steady(w, 0.1) and window_steady(w, 0.2)
    # the first steady step needs `window` values: a constant series is steady after step `window`, not before
    assert first_steady(np.ones((10, 3)), 4, 0.0) == 4
    ser = np.array([[1.0 + 2.0 ** -j, -1.0 - 3.0 ** -j, 3.0] for j in range(12)])
    s = first_steady(ser, 3, 0.05)
    assert s is not None and window_steady(ser[s - 3:s], 0.05) and not any(
        window_steady(ser[t - 3:t], 0.05) for t in range(3, s))
    r = steady_ratios(ser, 3)
    assert first_steady(ser, 3, float(r[s - 3])) == s and np.all(r[:s - 3] > 0.05)


# ------------------------------------------------------------------ refusals
def _net():
    n = L.Net()
    n.levels, n.repeats, n.c_i, n.c_h, n.c_o, n.ksize = 4, 2, 7, 16, 2, 3
    return n


def _desc(**kw):
    g = L.DiagDesc()
    for name in ("flux_seq", "vrms_seq", "hist", "hist_n", "steady", "part"):
        setattr(g, name, 0x1000)
    g.inv_dy_bot = g.inv_dy_top = 100.0
    g.window, g.rtol = 8, 1e-3
    for k, v in kw.items():
        setattr(g, k, v)
    return g


def test_diagnosed_rollout_refusals(lib):
    n = _net()
    d = C.c_void_p(0x1000)

    def call(g, queue=None, clock=d, H=64, B=2):
        return lib.pbmc_rollout_diagnosed(d, C.byref(n), d, d, d, d, d, d, 0.01, 0.99, 1, d, 2, 1, 4, d, 8, d, d, d, d, d,
                                          1 << 30, B, H, 96, clock, d, d, d, 4, queue, g, None)

    passes = lambda rc: rc not in (-1, -2, -3, -4)  # passes the checks (fails later, on the dummy pointers)
    assert call(None) == -3
    for name in ("flux_seq", "vrms_seq", "steady", "part", "hist", "hist_n"):
        assert call(C.byref(_desc(**{name: None}))) == -3, name
    assert passes(call(C.byref(_desc(window=0, hist=None, hist_n=None))))  # no criterion: no history needed
    for w in (-1, 1025):
        assert call(C.byref(_desc(window=w))) == -1, w
    assert passes(call(C.byref(_desc(window=1024)))) and passes(call(C.byref(_desc(rtol=0.0))))
    for r in (-1.0, math.nan, math.inf, -math.inf):
        assert call(C.byref(_desc(rtol=r))) == -1, r
    assert call(C.byref(_desc()), H=2) == -1  # no interior
    assert call(C.byref(_desc()), clock=None) == -3  # what pbmc_rollout_clocked refuses
    q = L.MemberQueue()
    for name, _ in L.MemberQueue._fields_[:-1]:
        setattr(q, name, 0x1000)
    q.Q = 3
    assert passes(call(C.byref(_desc()), queue=C.byref(q)))
    q.next = None
    assert call(C.byref(_desc()), queue=C.byref(q)) == -3  # what pbmc_rollout_queued refuses
    assert lib.pbmc_sizeof(b"pbmc_diag_desc") == C.sizeof(L.DiagDesc)
    assert lib.pbmc_sizeof(b"pbmc_member_clock") == C.sizeof(L.MemberClock)  # unchanged


@pytest.mark.parametrize("steady", [(0, 1e-3), (-3, 1e-3), (1025, 1e-3), (2.5, 1e-3), (4, -1e-3), (4, math.nan),
                                    (4, math.inf)])
def test_steady_argument_refused_before_any_device_work(steady):
    ens = EnsembleRollout.__new__(EnsembleRollout)  # no device: the arguments are checked first
    with pytest.raises(ValueError):
        ens.start_clock(np.inf, steady=steady)
    with pytest.raises(ValueError):
        ens.start_sweep(np.zeros((1, H, W)), [(1.0, 1.0, 1.0)], np.inf, steady=steady)


# ------------------------------------------------------------------ driver pickles
class FakeDiag:
    """EnsembleRollout's clocked (start_clock) and sweep (start_sweep) interfaces with diagnostics on scripted members:
    member q: T *= decay[q] and dt = dt[q] every step; after its j-th step it logs q_bot = 1 + q + j / 8,
    q_top = 2 + q - j / 16, vrms = 3 + q + j / 32.  With `steady`, member q is steady after its step steady_at[q]: it takes
    one more step and stops, reported steady unless t_end / max_steps stop it at that step too.  Clock rules as on the
    device (a step while t < t_end and steps < max_steps; then t += dt, steps += 1, mean-T, a snapshot when t > save_t,
    save_t = t + save_every); a sweep's stopping slots take the next queued members in ascending slot order."""

    def __init__(self, B, dts, decays, steady_at):
        self.B, self.H, self.W = B, H, W
        self.dts, self.decays, self.steady_at = dts, decays, steady_at
        self.calls = []

    @property
    def T(self):
        return torch.from_numpy(self._T[:self.B])

    def set_T(self, T0):
        self._T = np.asarray(T0, dtype=np.float64).copy()

    def _start(self, N, t0, t_end, save_every, max_steps, n_step, snap_slots, kw):
        self.calls.append(kw)
        bc = lambda x, dt=np.float64: np.broadcast_to(np.asarray(x, dtype=dt), (N,)).copy()
        self.t, self.t_end, self.save_every = bc(t0), bc(t_end), bc(save_every)
        self.steps = bc(n_step, np.int64)
        self.max_steps = bc(1 << 62 if max_steps is None else max_steps, np.int64)
        self.save_t, self.taken = np.zeros(N), np.zeros(N, np.int64)
        self.diag = bool(kw.get("diagnostics")) or kw.get("steady") is not None
        self.rule = kw.get("steady") is not None
        self.found, self.done, self.steady = (np.zeros(N, bool) for _ in range(3))
        self.slots = snap_slots

    def start_clock(self, t_end, save_every=0.0, t0=0.0, max_steps=None, n_step=0, snap_slots=None, **kw):
        self._start(self.B, t0, t_end, save_every, max_steps, n_step, snap_slots, kw)
        self.sweep, self.slot, self.queue, self.next = False, list(range(self.B)), list(range(self.B)), self.B

    def start_sweep(self, T0, params, t_end, save_every=0.0, t0=0.0, max_steps=None, n_step=0, snap_slots=None,
                    steps_per_graph=10, **kw):
        Q = len(params)
        self._T = torch.as_tensor(T0).double().numpy().reshape(Q, H, W).copy()
        self._start(Q, t0, t_end, save_every, max_steps, n_step, snap_slots, kw)
        self.sweep, self.queue = True, [q for q in range(Q) if self._active(q)]
        self.next = min(self.B, len(self.queue))
        self.slot = [self.queue[s] if s < self.next else -1 for s in range(self.B)]

    def _active(self, q):
        return q >= 0 and not self.done[q] and self.t[q] < self.t_end[q] and self.steps[q] < self.max_steps[q]

    def any_active(self):
        return any(self._active(q) for q in self.slot) or self.next < len(self.queue)

    def run(self, n_steps, steps_per_graph, track_time=True):
        assert n_steps == steps_per_graph
        keys = ["dt", "t", "meanT", "steps", "snapshots"] + (["q_bot", "q_top", "vrms"] if self.diag else [])
        blk = {} if self.sweep else {q: {k: [] for k in keys} for q in range(self.B)}
        f = lambda c: np.full((H, W), c)
        for _ in range(n_steps):
            stopped = []
            for s, q in enumerate(self.slot):
                if not self._active(q):
                    continue
                d = blk.setdefault(q, {k: [] for k in keys})
                self._T[q] = self._T[q] * self.decays[q]
                self.t[q] = self.t[q] + self.dts[q]
                self.steps[q] += 1
                self.taken[q] += 1
                j = self.taken[q]
                for k, x in (("dt", self.dts[q]), ("t", self.t[q]), ("meanT", self._T[q].mean()), ("steps", self.steps[q])):
                    d[k].append(x)
                if self.diag:
                    d["q_bot"].append(1.0 + q + j / 8)
                    d["q_top"].append(2.0 + q - j / 16)
                    d["vrms"].append(3.0 + q + j / 32)
                if self.t[q] > self.save_t[q]:
                    d["snapshots"].append({"step": int(self.steps[q]), "t": float(self.t[q]), "T": self._T[q].copy(),
                                           "u": f(1.0), "v": f(2.0), "p": f(3.0)})
                    self.save_t[q] = self.t[q] + self.save_every[q]
                if self.found[q]:
                    self.done[q] = True
                    self.steady[q] = self.t[q] < self.t_end[q] and self.steps[q] < self.max_steps[q]
                elif self.rule and j == self.steady_at[q] and self._active(q):
                    self.found[q] = True
                if not self._active(q):
                    stopped.append(s)
            for s in stopped:
                if self.sweep and self.next < len(self.queue):
                    self.slot[s] = self.queue[self.next]
                    self.next += 1
        running = {q for q in self.slot if self._active(q)}
        self._blk = {}
        for q, d in blk.items():
            e = {k: (np.asarray(v) if k != "snapshots" else v) for k, v in d.items()}
            if self.diag:
                e["steady"] = bool(self.steady[q])
            if self.sweep:
                e["finished"] = q not in running
            assert len(e["snapshots"]) <= self.slots
            self._blk[q] = e

    def drain(self):
        return self._blk if self.sweep else [self._blk[m] for m in range(self.B)]

    def stop_clock(self):
        pass


def _grid():
    x = torch.linspace(0, 4, W, dtype=torch.float64).view(1, 1, 1, W).expand(1, 1, H, W).contiguous()
    y = torch.linspace(0, 1, H, dtype=torch.float64).view(1, 1, H, 1).expand(1, 1, H, W).contiguous()
    return x, y


def _load(d, name):
    with open(d / name, "rb") as fh:
        return pickle.load(fh)


def _bytes(d, name):
    return (d / name).read_bytes()


OLD = ("snapshots_ML.pkl", "t_vec_ML.pkl", "T_vec_ML.pkl")  # TS_vec holds wall times: compared by length
NEW = ("Nu_vec_ML.pkl", "vrms_vec_ML.pkl")
DTS, DECAYS, STEADY_AT = [0.25, 0.1, 0.4, 0.2, 0.3], [0.9, 0.97, 0.8, 0.95, 0.85], [3, 6, 100, 2, 7]


def _check_pickles(base, steps, t_vec_expected=None):
    """Nu_vec / vrms_vec of each member directory against the scripted values, one entry per step, aligned with
    t_vec[1:]."""
    for q, n in enumerate(steps):
        d = base / f"member_{q}"
        tv, Nu, vr = _load(d, "t_vec_ML.pkl"), _load(d, "Nu_vec_ML.pkl"), _load(d, "vrms_vec_ML.pkl")
        assert len(tv) == n + 1 and len(Nu) == len(vr) == n == len(_load(d, "TS_vec_ML.pkl")), q
        for j, (a, b) in enumerate(zip(Nu, vr), start=1):
            assert isinstance(a, np.ndarray) and a.shape == (2,) and a.dtype == np.float64
            assert a[0] == 1.0 + q + j / 8 and a[1] == 2.0 + q - j / 16, (q, j)
            assert type(b) is float and b == 3.0 + q + j / 32, (q, j)


@pytest.mark.parametrize("form", ["ensemble", "sweep"])
def test_diagnostics_pickles_and_unchanged_old_pickles(tmp_path, form):
    xcc, ycc = _grid()
    T0 = 1.0 + np.random.default_rng(4).random((5, H, W))
    runs = {}
    for name, kw in (("off", {}), ("on", {"diagnostics": True})):
        if form == "ensemble":
            ens = FakeDiag(5, DTS, DECAYS, STEADY_AT)
            ens.set_T(T0)
            t, n, _ = D.attempt_ensemble(ens, xcc, ycc, t_end=2.0, out_dir=str(tmp_path / name), save_every=0.5,
                                         write_every=0.3, check_every=4, **kw)
        else:
            ens = FakeDiag(2, DTS, DECAYS, STEADY_AT)
            t, n, _ = D.attempt_sweep(ens, T0, [(1.0, 1.0, 1.0)] * 5, xcc, ycc, t_end=2.0, out_dir=str(tmp_path / name),
                                      save_every=0.5, write_every=0.3, check_every=4, **kw)
        runs[name] = (t, n)
        # without diagnostics the ensemble is started exactly as before (no new keyword arguments)
        assert ens.calls == [{"diagnostics": True, "steady": None} if kw else {}]
    assert np.array_equal(runs["on"][1], runs["off"][1]) and np.array_equal(runs["on"][0], runs["off"][0])
    steps = [int(x) for x in runs["on"][1]]
    assert steps == [8, 20, 5, 11, 7]  # t_end = 2.0 only
    _check_pickles(tmp_path / "on", steps)
    for q in range(5):
        off, on = tmp_path / "off" / f"member_{q}", tmp_path / "on" / f"member_{q}"
        assert sorted(p.name for p in off.iterdir()) == sorted(OLD + ("TS_vec_ML.pkl",))
        assert sorted(p.name for p in on.iterdir()) == sorted(OLD + NEW + ("TS_vec_ML.pkl",))
        for name in OLD:
            assert _bytes(off, name) == _bytes(on, name), (q, name)
        assert len(_load(off, "TS_vec_ML.pkl")) == len(_load(on, "TS_vec_ML.pkl"))


@pytest.mark.parametrize("form", ["ensemble", "sweep"])
def test_steady_stops_in_the_pickles(tmp_path, form):
    xcc, ycc = _grid()
    T0 = 1.0 + np.random.default_rng(5).random((5, H, W))
    kw = dict(t_end=2.0, out_dir=str(tmp_path), check_every=3, steady=(4, 1e-3))
    if form == "ensemble":
        ens = FakeDiag(5, DTS, DECAYS, STEADY_AT)
        ens.set_T(T0)
        t, n, logs = D.attempt_ensemble(ens, xcc, ycc, **kw)
    else:
        ens = FakeDiag(2, DTS, DECAYS, STEADY_AT)
        t, n, logs = D.attempt_sweep(ens, T0, [(1.0, 1.0, 1.0)] * 5, xcc, ycc, **kw)
    assert ens.calls == [{"diagnostics": True, "steady": (4, 1e-3)}]
    # steady after step 3 / 6 / 2: one more step (members 0, 1, 3); member 2 never, member 4 (after 7) reaches t_end at
    # step 7 = steady_at, so the criterion is never evaluated as met while it runs
    steps = [int(x) for x in n]
    assert steps == [4, 7, 5, 3, 7]
    assert list(ens.steady) == [True, True, False, True, False]
    _check_pickles(tmp_path, steps)
    for q in range(5):
        tv = _load(tmp_path / f"member_{q}", "t_vec_ML.pkl")
        assert np.isclose(tv[-1], t[q]) and len(logs[q][2]["ML"]) == steps[q] + 1
