"""Throughput of a parameter sweep larger than the batch, run two ways in one process:
  * sequential: `driver.attempt_ensemble` over consecutive batches of B members (a batch lasts as long as its slowest
    member; its finished members keep their slots, frozen, until then);
  * sweep: one `driver.attempt_sweep` of all Q members through B slots (a slot whose member stops takes the next queued
    member on the device, inside the same graph).
Workloads: the primary network (bench.py's) with Q = 64 members of 256^2 through B = 32 slots, and the paper's
learned-boundary network at 128x506 with Q = 16, B = 8.  Member q runs exactly max_steps[q] steps (t_end = inf), drawn
uniformly from [10, 80] with a fixed seed, so the step counts do not depend on dt noise.  Both forms take 10 steps per
graph, a snapshot at the first step (save_every = inf) and write the four pickles per member into a temporary directory.
Per form: wall time of the driver call, the time of its run + drain loop alone (without the pickle writes), member-steps
per second (over the wall time) and slot occupancy (steps members took / slot-steps run).  Each form runs once untimed
first (graph capture, module load).

Then the per-step cost of the queued clock (pbmc_rollout_queued, with a member waiting in the queue and no slot
stopping) against the plain clocked one (pbmc_rollout_clocked), with tools/clock_overhead.py's method: 10-step graphs,
CUDA events, alternating windows in one process, L2 not flushed; 512^2 B = 1 and 32 x 256^2.  The card name and power
limit are read and printed in the same run.

usage: python tools/sweep_throughput.py [--windows N] [--out FILE.json]"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pbml_mantle_convection_b200 import driver as D  # noqa: E402
from pbml_mantle_convection_b200 import ops  # noqa: E402
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_grid, synthetic_T0  # noqa: E402
from tools.clock_overhead import K, PARAMS, primary_net, window_ms  # noqa: E402
from tools.learned_rollout_time import card, paper_net  # noqa: E402

DEV = torch.device("cuda:0")


class LoopTimer:
    """An EnsembleRollout whose run() + drain() time is summed (drain reads the block back, so it ends in a sync)."""

    def __init__(self, ens):
        self.ens, self.seconds = ens, 0.0

    def __getattr__(self, name):
        return getattr(self.ens, name)

    def run(self, *a, **kw):
        t = time.perf_counter()
        self.ens.run(*a, **kw)
        self.seconds += time.perf_counter() - t

    def drain(self):
        t = time.perf_counter()
        out = self.ens.drain()
        self.seconds += time.perf_counter() - t
        return out


def sequential(ens, T0, params, max_steps, xc, yc, out):
    B = ens.B
    for b0 in range(0, len(params), B):
        ens.members.copy_(ops.make_members(params[b0:b0 + B], DEV))
        ens.set_T(T0[b0:b0 + B])
        D.attempt_ensemble(ens, xc, yc, t_end=np.inf, out_dir=os.path.join(out, f"batch{b0}"), save_every=np.inf,
                           write_every=np.inf, check_every=K, max_steps=max_steps[b0:b0 + B])


def sweep(ens, T0, params, max_steps, xc, yc, out):
    D.attempt_sweep(ens, T0, params, xc, yc, t_end=np.inf, out_dir=out, save_every=np.inf, write_every=np.inf,
                    check_every=K, max_steps=max_steps)


def throughput(mk, Q, B, H, W, seed):
    net = mk()
    rng = np.random.default_rng(seed)
    max_steps = rng.integers(10, 81, size=Q)
    params = [(PARAMS[0] * (1.0 + 0.01 * q), PARAMS[1], PARAMS[2]) for q in range(Q)]
    T0 = np.stack([synthetic_T0(H, W, seed=q) for q in range(Q)])
    xc, yc = synthetic_grid(H, W)
    ens = EnsembleRollout(net, H, W, params[:B], DEV, max_steps=64)
    res = {"Q": Q, "B": B, "H": H, "W": W, "max_steps_seed": seed, "member_steps": int(max_steps.sum()),
           "max_steps_mean": float(max_steps.mean()), "steps_per_graph": K}
    tmp = tempfile.mkdtemp(prefix="sweep_throughput_")
    try:
        for name, fn in (("sequential", sequential), ("sweep", sweep)):
            fn(ens, T0, params, np.full(Q, 2), xc, yc, os.path.join(tmp, "warm"))  # capture + module load, same buffers
            timed = LoopTimer(ens)
            n0 = ens.n_done
            torch.cuda.synchronize(DEV)
            t = time.perf_counter()
            fn(timed, T0, params, max_steps, xc, yc, os.path.join(tmp, name))
            torch.cuda.synchronize(DEV)
            wall = time.perf_counter() - t
            slot_steps = (ens.n_done - n0) * B
            res[name] = {"wall_s": wall, "loop_s": timed.seconds, "batch_steps": ens.n_done - n0,
                         "member_steps_per_s": res["member_steps"] / wall,
                         "member_steps_per_s_loop": res["member_steps"] / timed.seconds,
                         "slot_occupancy": res["member_steps"] / slot_steps}
            r = res[name]
            print(f"  {name}: wall {wall:.3f} s (run + drain {r['loop_s']:.3f} s), {r['batch_steps']} batch-steps, "
                  f"{r['member_steps_per_s']:.1f} member-steps/s ({r['member_steps_per_s_loop']:.1f} over run + drain), "
                  f"occupancy {r['slot_occupancy']:.3f}", flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    del ens, net
    torch.cuda.empty_cache()
    return res


def queued_overhead(B, H, W, windows):
    net = primary_net()
    params = [(PARAMS[0] * (1.0 + 0.01 * i), PARAMS[1], PARAMS[2]) for i in range(B + 1)]
    T0 = np.stack([synthetic_T0(H, W, seed=i) for i in range(B + 1)])
    clk = EnsembleRollout(net, H, W, params[:B], DEV, max_steps=64)
    clk.set_T(T0[:B])
    clk.start_clock(np.inf, save_every=np.inf, steps_per_graph=K)
    qd = EnsembleRollout(net, H, W, params[:B], DEV, max_steps=64)
    qd.start_sweep(T0, params, np.inf, save_every=np.inf, steps_per_graph=K)  # one member waits, no slot stops
    g_clk, g_q = clk.graph(K), qd.graph(K)
    for g in (g_clk, g_q):
        for _ in range(3):
            g.replay()
    torch.cuda.synchronize(DEV)
    reps = max(3, int(300.0 / (K * window_ms(g_clk, 3))))
    t_clk, t_q = [], []
    for _ in range(windows):
        t_clk.append(window_ms(g_clk, reps))
        t_q.append(window_ms(g_q, reps))
    ck = qd.read_clock()
    assert ck["active"].all() and ck["next"] == B and bool(torch.isfinite(qd.T).all())
    mc, mq = float(np.median(t_clk)), float(np.median(t_q))
    r = {"B": B, "H": H, "W": W, "replays_per_window": reps, "clocked_ms_per_step": t_clk, "queued_ms_per_step": t_q,
         "clocked_median_ms": mc, "queued_median_ms": mq, "overhead_us_per_step": 1e3 * (mq - mc),
         "overhead_pct": 100.0 * (mq - mc) / mc, "clocked_spread_ms": float(max(t_clk) - min(t_clk)),
         "queued_spread_ms": float(max(t_q) - min(t_q))}
    print(f"  {B} x {H}x{W}: clocked {mc:.4f} ms/step (spread {r['clocked_spread_ms']:.4f}), queued {mq:.4f} ms/step "
          f"(spread {r['queued_spread_ms']:.4f}): {r['overhead_us_per_step']:+.2f} us/step = {r['overhead_pct']:+.2f} %",
          flush=True)
    del clk, qd, g_clk, g_q, net
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=7, help="alternating clocked / queued windows per size")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: these are device timings")
    name, lim = card()
    res = {"card": name, "power_limit_and_max_sm_clock": lim, "l2_flushed": False, "throughput": {}, "queued_vs_clocked": {}}
    print(f"card: {name}; power limit, max SM clock: {lim}", flush=True)
    with torch.no_grad():
        for tag, (mk, Q, B, H, W) in {"primary_Q64_B32_256x256": (primary_net, 64, 32, 256, 256),
                                      "learned_paper_Q16_B8_128x506": (paper_net, 16, 8, 128, 506)}.items():
            print(f"{tag}:", flush=True)
            res["throughput"][tag] = throughput(mk, Q, B, H, W, seed=7)
        print("queued clock vs clocked (10-step graphs, L2 not flushed):", flush=True)
        for tag, (B, H, W) in {"primary_512x512_B1": (1, 512, 512), "primary_32x256x256": (32, 256, 256)}.items():
            res["queued_vs_clocked"][tag] = queued_overhead(B, H, W, a.windows)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
