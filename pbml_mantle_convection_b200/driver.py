"""GAIA-free form of the reference's rollout driver (SURVEY.md section 8f, N2).

`advect_wi_gaia.py:538-679` (`attempt(t, n_step)`) couples the surrogate to the proprietary GAIA solver: GAIA owns
the state arrays, the surrogate fills `state["v"]`, `state["P"]`, `state["V"]` every step and -- in mode "ML" between
GAIA interventions -- `state["T"]` / `dt` come from `ts_net` (`:632-635`).  GAIA is not available, so this module
provides the same loop for the pure-ML case with a plain dict as the state, and keeps everything the notebooks read
afterwards (`.ipynb_checkpoints/load_advection_results-checkpoint.ipynb:243-326`):

    snapshots_<mode>.pkl   {"v": [ [N,3] ... ], "P": [ [N] ... ], "T": [ [N] ... ], "xcc": tensor, "ycc": tensor}
    t_vec_<mode>.pkl       simulated time after every step (first entry: start time)
    T_vec_<mode>.pkl       mean temperature after every step (first entry: initial mean)     (:547, :647)
    TS_vec_<mode>.pkl      wall-clock seconds of every step                                  (:650-652)

and, with `attempt_ensemble(..., diagnostics=True)` / `attempt_sweep(..., diagnostics=True)` (or `steady=(window,
rtol)`), the per-step quantities of the converged-state analysis, computed on the device:

    Nu_vec_<mode>.pkl      wall heat fluxes np.array([q_bot, q_top]) after every step (include/pbmc.h, pbmc_diag_desc)
    vrms_vec_<mode>.pkl    rms velocity of every step (float)
                           both one entry per step, aligned with t_vec[1:] (no initial entry: vrms needs a step)

with the same cadence rules: a snapshot whenever `t > save_t` (then `save_t = t + save_every`), the pickles rewritten
whenever `t > write_t` and once more at the end (`:654-677`).

Three ways to advance:
  * `attempt(ts_net, ...)`  -- one `ts_net(...)` call per step exactly like `:590-593` (host tensors in, fields read
    back every step); any callable with `TS.forward`'s signature works (the drop-in `TS`, or the reference's own).
  * `attempt_resident(ens, ...)` -- an `EnsembleRollout` advances `check_every` steps per CUDA-graph replay with T, u, v
    and dt on the device; host work (time bookkeeping, cadence checks, snapshots) happens once per block.
  * `attempt_ensemble(ens, ...)` -- every member of an `EnsembleRollout` runs to its own `t_end` on a device-side clock
    (`EnsembleRollout.start_clock`): per-step t / mean-T and snapshots at the exact steps, the four pickles per member,
    read back once per block of `check_every` steps.
  * `attempt_sweep(ens, T0, params, ...)` -- the same for a sweep of Q members run through the B slots of an
    `EnsembleRollout` (`EnsembleRollout.start_sweep`): a slot whose member stops takes the next queued member on the
    device, so Q may exceed B and no slot idles while members wait.  With `continue_from`, a member starts from the
    field its predecessor stopped with (parameter continuation), handed over on the device.

External energy solver (the `ML_STOKES` / `ML_PRE` modes and the `intervene_TS` interventions of mode "ML", `:486-505`,
`:618-630`): the reference calls GAIA's `sim.doTimestep()` with the surrogate's velocities already written into the state
and takes T and dt from it.  `attempt(..., energy_step=f)` is that hook: `f(state) -> dt` advances `state["T"]` in place
(it sees `state["v"]`, `state["P"]`, `state["V"]` of this step) every step for modes other than "ML", and on every
`intervene_TS`-th step in mode "ML"; the driver then applies the reference's wall rows / side columns / clip(0, 2)
(`:624-629`) and feeds the result to the next surrogate call.  With `TS(stokes, None, ...)` (no ADNet, `:488-500`) the
surrogate only supplies (u, v, p, V): `dts` is empty and the time step is the callback's.

One deliberate difference: the reference never feeds `T_new` back into `Tp` between GAIA steps (`Tp` is only
refreshed from GAIA's state, `:618-630`; in pure-ML mode the network would see the initial field forever).  Without
GAIA the state's T *is* the surrogate's T, so `Tp <- T_new[1]` here -- the semantics of `TS(ts=N)`'s own loop (:377).
"""
from __future__ import annotations

import os
import pickle
import time

import numpy as np
import torch


def _new_logs(mode):
    return ({mode: {"v": [], "P": [], "T": []}}, {mode: []}, {mode: []}, {mode: []})


def _snapshot(snap, state):
    for var in ("v", "P", "T"):  # :656-657
        snap[var].append(np.copy(state[var]))


def write_logs(out_dir, mode, snapshots, TS_vec, t_vec, T_vec):
    """The four pickles of `advect_wi_gaia.py:659-677`, same names, same objects."""
    os.makedirs(out_dir, exist_ok=True)
    for name, obj in (("snapshots_", snapshots[mode]), ("TS_vec_", TS_vec[mode]), ("t_vec_", t_vec[mode]), ("T_vec_", T_vec[mode])):
        with open(os.path.join(out_dir, name + mode + ".pkl"), "wb") as fh:
            pickle.dump(obj, fh)


def write_diag_logs(out_dir, mode, Nu_vec, vrms_vec):
    """The two diagnostics pickles next to write_logs' four: Nu_vec_<mode>.pkl, vrms_vec_<mode>.pkl."""
    os.makedirs(out_dir, exist_ok=True)
    for name, obj in (("Nu_vec_", Nu_vec), ("vrms_vec_", vrms_vec)):
        with open(os.path.join(out_dir, name + mode + ".pkl"), "wb") as fh:
            pickle.dump(obj, fh)


def attempt(ts_net, T0, xcc, ycc, raq, fkt, fkp, raq_nd, fkt_nd, fkp_nd, t_end, out_dir, save_every=0.0, write_every=0.0,
            mode="ML", t=0.0, n_step=0, p_pred=True, max_steps=None, sdf=None, sdf2=None, energy_step=None, intervene_TS=0,
            core_cool=False):
    """`attempt(t, n_step)` of advect_wi_gaia.py:538-679 without GAIA: returns (t, n_step, logs) with logs = (snapshots,
    TS_vec, t_vec, T_vec) dicts keyed by mode.  T0, xcc, ycc: [1,1,H,W] float64 host tensors (what `:560-581` builds
    from GAIA's state).  energy_step / intervene_TS / core_cool: the external-energy-solver hook, see the module docstring."""
    if mode != "ML" and energy_step is None and getattr(ts_net, "ad", True) is None:
        raise ValueError(f"mode {mode!r} with a TS that has no ADNet needs energy_step (nothing would advance T)")
    snapshots, TS_vec, t_vec, T_vec = _new_logs(mode)
    H, W = T0.shape[-2:]
    n = H * W
    state = {"T": T0.detach().cpu().numpy().reshape(n).copy(), "v": np.zeros((n, 3)), "P": np.zeros(n), "V": np.zeros(n)}
    T_vec[mode].append(np.copy(state["T"].mean()))
    t_vec[mode].append(np.copy(t))
    save_t = write_t = 0
    _snapshot(snapshots[mode], state)
    snapshots[mode]["xcc"], snapshots[mode]["ycc"] = xcc, ycc
    Tp = T0
    while t < t_end and (max_steps is None or n_step < max_steps):
        n_step += 1
        t0 = time.time()
        with torch.no_grad():
            T_new, dts, u, v, p, V = ts_net(Tp, sdf, sdf2, ycc, raq_nd, fkt_nd, fkp_nd, raq, fkt, fkp, xcc, ycc)  # :590-593
        u = u.detach().cpu().numpy()
        v = v.detach().cpu().numpy()
        V = V.detach().cpu().numpy()
        state["v"][:, :] = np.concatenate((u.reshape(-1, 1), v.reshape(-1, 1), np.zeros_like(u.reshape(-1, 1))), axis=1)  # :602-612
        if p_pred and p is not None:
            state["P"][:] = p.detach().cpu().numpy().flatten()
        state["V"][:] = V.flatten()
        external = energy_step is not None and (mode != "ML" or (intervene_TS and n_step % intervene_TS == 0))
        if external:
            dt = float(energy_step(state))  # sim.doTimestep(): the external solver advances state["T"] with these velocities, :618-620
            Tp = torch.tensor(state["T"], dtype=T0.dtype).view(T0.shape).clone()
            if not core_cool:
                Tp[:, :, 0, :] = 1.0
            Tp[:, :, -1, :] = 0.0
            Tp[:, :, :, 0] = Tp[:, :, :, 1]
            Tp[:, :, :, -1] = Tp[:, :, :, -2]
            Tp = torch.clip(Tp, 0.0, 2.0)  # :621-629
            state["T"][:] = Tp.numpy().flatten()
        else:
            state["T"][:] = T_new[1].clone().detach().cpu().numpy().flatten()  # :633-635
            dt = float(dts[1].clone().detach().cpu().numpy())
            Tp = T_new[1].detach().cpu().reshape(T0.shape)  # see the module docstring
        t += dt
        T_vec[mode].append(np.copy(state["T"].mean()))
        t_vec[mode].append(np.copy(t))
        TS_vec[mode].append(time.time() - t0)
        if t > save_t:
            save_t = t + save_every
            _snapshot(snapshots[mode], state)
        if t > write_t:
            write_t = t + write_every
            write_logs(out_dir, mode, snapshots, TS_vec, t_vec, T_vec)
    write_logs(out_dir, mode, snapshots, TS_vec, t_vec, T_vec)
    return t, n_step, (snapshots, TS_vec, t_vec, T_vec)


def attempt_resident(ens, xcc, ycc, t_end, out_dir, save_every=0.0, write_every=0.0, mode="ML", t=0.0, n_step=0,
                     check_every=10, member=0, max_steps=None):
    """Same outputs from a device-resident `EnsembleRollout` (member `member` is logged): `check_every` time steps per
    CUDA-graph replay, then ONE read of the block's dt values and of mean-T; snapshots / pickles follow the same
    `t > save_t` / `t > write_t` rules, evaluated at block ends (check_every=1 reproduces the per-step cadence)."""
    from . import ops

    snapshots, TS_vec, t_vec, T_vec = _new_logs(mode)
    H, W = ens.H, ens.W
    n = H * W

    def host_state():
        u, v, p, V = ens.fields()
        st = {"T": ens.T[member].double().cpu().numpy().reshape(n)}
        st["v"] = np.concatenate((u[member].double().cpu().numpy().reshape(-1, 1), v[member].double().cpu().numpy().reshape(-1, 1),
                                  np.zeros((n, 1))), axis=1)
        st["P"] = p[member].double().cpu().numpy().reshape(n) if p is not None else np.zeros(n)
        return st

    T_vec[mode].append(np.copy(ens.T[member].double().mean().item()))
    t_vec[mode].append(np.copy(t))
    save_t = write_t = 0
    st0 = {"T": ens.T[member].double().cpu().numpy().reshape(n), "v": np.zeros((n, 3)), "P": np.zeros(n)}
    _snapshot(snapshots[mode], st0)
    snapshots[mode]["xcc"], snapshots[mode]["ycc"] = xcc, ycc
    k = int(check_every)
    while t < t_end and (max_steps is None or n_step < max_steps):
        t0 = time.time()
        par = ens.n_done % 2
        ens.run(k, steps_per_graph=k, track_time=False)
        dts = ens.state.dt_seq[par:par + k, member].cpu().numpy()  # the only per-block host read besides mean-T
        mean_T, _ = ops.diagnostics(ens.T.contiguous())
        mean_T = float(mean_T[member].item())
        wall = (time.time() - t0) / k
        for dt in dts:
            n_step += 1
            t += float(dt)
            t_vec[mode].append(np.copy(t))
            T_vec[mode].append(np.copy(mean_T))  # mean-T is sampled at block ends
            TS_vec[mode].append(wall)
        if t > save_t:
            save_t = t + save_every
            _snapshot(snapshots[mode], host_state())
        if t > write_t:
            write_t = t + write_every
            write_logs(out_dir, mode, snapshots, TS_vec, t_vec, T_vec)
    write_logs(out_dir, mode, snapshots, TS_vec, t_vec, T_vec)
    return t, n_step, (snapshots, TS_vec, t_vec, T_vec)


def attempt_ensemble(ens, xcc, ycc, t_end, out_dir, save_every=0.0, write_every=0.0, mode="ML", t=0.0, n_step=0,
                     check_every=10, max_steps=None, diagnostics=False, steady=None):
    """`attempt` for every member of a device-resident `EnsembleRollout` at once.  Member m runs `while t < t_end[m]` (and
    n_step < max_steps) on its own device-side clock; t_end, save_every, t and n_step are scalars or one value per member.
    Writes the reference's four pickles of member m into `out_dir/member_<m>/` with `attempt`'s cadence: the initial entry
    and snapshot, one t_vec / T_vec entry per step the member took, snapshots at the steps where t > save_t.  Blocks of
    `check_every` steps run as one CUDA-graph replay each, then the block's logs are drained; `t > write_t` is evaluated at
    block ends (it decides when intermediate pickles are written, not their final content).  A TS_vec entry is the block's
    wall time over the steps the member took in it.  Returns (t [B], n_step [B], [logs of member m]) with logs as in
    `attempt`.  diagnostics=True (or steady=(window, rtol), which also stops a member at a statistical steady state:
    `EnsembleRollout.start_clock`) adds Nu_vec_<mode>.pkl and vrms_vec_<mode>.pkl next to the four pickles."""
    B, H, W = ens.B, ens.H, ens.W
    n = H * W
    k = int(check_every)
    logs = [_new_logs(mode) for _ in range(B)]
    dirs = [os.path.join(out_dir, f"member_{m}") for m in range(B)]
    T0 = ens.T.double().cpu().numpy().reshape(B, n)
    t0 = np.broadcast_to(np.asarray(t, dtype=np.float64), (B,)).copy()
    _initial_entries(logs, T0, t0, xcc, ycc, mode, n)
    ens.start_clock(t_end, save_every=save_every, t0=t0, max_steps=max_steps, n_step=n_step, snap_slots=k,
                    **_diag_kwargs(diagnostics, steady))
    return _run_blocks(ens, k, logs, dirs, t0, n_step, write_every, mode, n, _diag_logs(B, diagnostics, steady))


def attempt_sweep(ens, T0, params, xcc, ycc, t_end, out_dir, save_every=0.0, write_every=0.0, mode="ML", t=0.0, n_step=0,
                  check_every=10, max_steps=None, diagnostics=False, steady=None, continue_from=None):
    """`attempt` for each of Q members run through the B slots of a device-resident `EnsembleRollout`
    (`EnsembleRollout.start_sweep`; Q may be larger or smaller than B).  T0: [Q, H, W]; params: Q tuples (RaQ, gamma,
    beta); t_end, save_every, t, n_step, max_steps: scalars or one value per member.  Member q's pickles go to
    `out_dir/member_<q>/`, with `attempt_ensemble`'s cadence and content: the slot a member ran in, and when, make no
    difference.  Returns (t [Q], n_step [Q], [logs of member q]).  diagnostics / steady: as in `attempt_ensemble`.
    continue_from: as in `EnsembleRollout.start_sweep`; a continued member's pickles are those of `attempt` run alone
    from the field its predecessor stopped with (its initial entries are written when it starts)."""
    Q, H, W = len(params), ens.H, ens.W
    n = H * W
    k = int(check_every)
    logs = [_new_logs(mode) for _ in range(Q)]
    dirs = [os.path.join(out_dir, f"member_{q}") for q in range(Q)]
    T0 = torch.as_tensor(T0).to("cpu", torch.float32).reshape(Q, H, W)  # what the device runs from
    t0 = np.broadcast_to(np.asarray(t, dtype=np.float64), (Q,)).copy()
    chain = {} if continue_from is None else {"continue_from": continue_from}
    ens.start_sweep(T0, params, t_end, save_every=save_every, t0=t, max_steps=max_steps, n_step=n_step, snap_slots=k,
                    steps_per_graph=k, **_diag_kwargs(diagnostics, steady), **chain)
    heads = [q for q in range(Q) if continue_from is None or continue_from[q] == -1]
    _initial_entries([logs[q] for q in heads], T0[heads].double().numpy().reshape(len(heads), n), t0[heads], xcc, ycc,
                     mode, n)
    start = lambda m, T: _initial_entries([logs[m]], T.astype(np.float64).reshape(1, n), t0[m:m + 1], xcc, ycc, mode, n)
    return _run_blocks(ens, k, logs, dirs, t, n_step, write_every, mode, n, _diag_logs(Q, diagnostics, steady), start)


def _diag_kwargs(diagnostics, steady):
    """start_clock / start_sweep's diagnostics arguments (none when off, so the call is the one without them)."""
    return {"diagnostics": True, "steady": steady} if diagnostics or steady is not None else {}


def _diag_logs(N, diagnostics, steady):
    """Per member (Nu_vec, vrms_vec) lists, or None without diagnostics."""
    return [([], []) for _ in range(N)] if diagnostics or steady is not None else None


def _initial_entries(logs, T0, t, xcc, ycc, mode, n):
    """`attempt`'s entries before the first step, for every member: mean of T0, the start time, the T0 snapshot."""
    t0 = np.broadcast_to(np.asarray(t, dtype=np.float64), (len(logs),))
    for m, (snapshots, TS_vec, t_vec, T_vec) in enumerate(logs):
        T_vec[mode].append(np.copy(T0[m].mean()))
        t_vec[mode].append(np.copy(t0[m]))
        _snapshot(snapshots[mode], {"T": T0[m].copy(), "v": np.zeros((n, 3)), "P": np.zeros(n)})
        snapshots[mode]["xcc"], snapshots[mode]["ycc"] = xcc, ycc


def _run_blocks(ens, k, logs, dirs, t, n_step, write_every, mode, n, diag=None, start=None):
    """Blocks of k steps (one graph replay each) until no member of the running clock or sweep is left; each drained
    block (a list over the members, or a sweep's dict keyed by member) goes into the logs of its members.  A
    TS_vec entry is the block's wall time over the steps the member took in it; `t > write_t` is evaluated at block
    ends.  Writes every member's pickles at the end; returns (t, n_step, logs) per member.  diag: per member
    (Nu_vec, vrms_vec) lists filled from the blocks' q_bot, q_top, vrms and written with the other pickles.  start:
    start(m, start_T) writes a continued member's initial entries when its first block carries start_T."""

    def write(m):
        write_logs(dirs[m], mode, *logs[m])
        if diag is not None:
            write_diag_logs(dirs[m], mode, *diag[m])

    N = len(logs)
    t_now = np.broadcast_to(np.asarray(t, dtype=np.float64), (N,)).copy()
    n_now = np.broadcast_to(np.asarray(n_step, dtype=np.int64), (N,)).copy()
    write_t = np.zeros(N)
    write_every = np.broadcast_to(np.asarray(write_every, dtype=np.float64), (N,))
    while ens.any_active():
        w0 = time.time()
        ens.run(k, steps_per_graph=k)
        blk = ens.drain()
        wall = time.time() - w0
        for m, d in (blk.items() if isinstance(blk, dict) else enumerate(blk)):
            if "start_T" in d:
                start(m, d["start_T"])
            snapshots, TS_vec, t_vec, T_vec = logs[m]
            taken = len(d["dt"])
            for tm, mt in zip(d["t"], d["meanT"]):
                t_vec[mode].append(np.copy(tm))
                T_vec[mode].append(np.copy(mt))
                TS_vec[mode].append(wall / taken)
            for sn in d["snapshots"]:
                st = {"T": sn["T"].astype(np.float64).reshape(n),
                      "v": np.concatenate((sn["u"].astype(np.float64).reshape(-1, 1), sn["v"].astype(np.float64).reshape(-1, 1),
                                           np.zeros((n, 1))), axis=1),
                      "P": sn["p"].astype(np.float64).reshape(n) if sn["p"] is not None else np.zeros(n)}
                _snapshot(snapshots[mode], st)
            if diag is not None:
                Nu_vec, vrms_vec = diag[m]
                for qb, qt, vr in zip(d["q_bot"], d["q_top"], d["vrms"]):
                    Nu_vec.append(np.array([qb, qt]))
                    vrms_vec.append(float(vr))
            if taken:
                t_now[m], n_now[m] = d["t"][-1], d["steps"][-1]
            if taken and t_now[m] > write_t[m]:
                write_t[m] = t_now[m] + write_every[m]
                write(m)
    for m in range(N):
        write(m)
    ens.stop_clock()
    return t_now, n_now, logs
