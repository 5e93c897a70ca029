"""Per-step cost of parameter-continuation chains (pbmc_rollout_chained: the successor test in the clock's apply / commit
launches, no launch added) against the same sweep without chains (pbmc_rollout_queued) and the clocked rollout without a
queue, in ms per step, when no slot stops, at three sizes:
  * 512^2, B = 1, primary network (NewFluidNet(levels=6, c_h=16, c_o=2, k=3, replicate, symmetric, curl), bench.py's);
  * 32 members of 256^2, primary network;
  * 128 x 506, B = 1, the paper's learned-boundary network (levels 5, repeats 6, k 5).
Forms of the same EnsembleRollout configuration as 10-step CUDA graphs, every member with t_end = inf and one snapshot
at its first step: clocked (start_clock); sweep (start_sweep of Q = 2B members, the second B waiting in the queue);
chained (the same sweep with continue_from[q] = q - B: every running member has a successor waiting).
tools/clock_overhead.py's method: CUDA events over back-to-back replays, the forms' windows alternating in one process,
L2 not flushed (a rollout runs its steps back to back).  The card name and power limit are read and printed in the same
run.

usage: python tools/chain_overhead.py [--windows N] [--replays N] [--out FILE.json]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_T0  # noqa: E402
from tools.clock_overhead import K, PARAMS, primary_net, window_ms  # noqa: E402
from tools.learned_rollout_time import card, paper_net  # noqa: E402

DEV = torch.device("cuda:0")
FORMS = ("clocked", "sweep", "chained")


def make(net, B, H, W, form):
    Q = 2 * B
    params = [(PARAMS[0] * (1.0 + 0.01 * i), PARAMS[1], PARAMS[2]) for i in range(Q)]
    T0 = np.stack([synthetic_T0(H, W, seed=i) for i in range(Q)])
    ens = EnsembleRollout(net, H, W, params[:B], DEV, per_member_dt=True, max_steps=64)
    if form == "clocked":
        ens.set_T(T0[:B])
        ens.start_clock(np.inf, save_every=np.inf, steps_per_graph=K)
    else:
        cf = [q - B if q >= B else -1 for q in range(Q)] if form == "chained" else None
        ens.start_sweep(T0, params, np.inf, save_every=np.inf, steps_per_graph=K, continue_from=cf)
    return ens, ens.graph(K)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=7, help="alternating windows per form and size")
    ap.add_argument("--replays", type=int, default=0, help="10-step replays per window (0: about 0.3 s of work)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: these are device timings")
    name, lim = card()
    res = {"card": name, "power_limit_and_max_sm_clock": lim, "l2_flushed": False, "steps_per_graph": K, "sizes": {}}
    print(f"card: {name}; power limit, max SM clock: {lim}; L2 not flushed; {K} steps per graph", flush=True)
    sizes = {"primary_512x512_B1": (primary_net, 1, 512, 512), "primary_32x256x256": (primary_net, 32, 256, 256),
             "learned_paper_128x506_B1": (paper_net, 1, 128, 506)}
    with torch.no_grad():
        for tag, (mk, B, H, W) in sizes.items():
            net = mk()
            runs = {f: make(net, B, H, W, f) for f in FORMS}
            for _, g in runs.values():  # warm-up
                for _ in range(3):
                    g.replay()
            torch.cuda.synchronize(DEV)
            reps = a.replays or max(3, int(300.0 / (K * window_ms(runs["clocked"][1], 3))))
            times = {f: [] for f in FORMS}
            for _ in range(a.windows):
                for f, (_, g) in runs.items():
                    times[f].append(window_ms(g, reps))
            for f, (ens, _) in runs.items():
                assert bool(torch.isfinite(ens.T).all()), f
                ck = ens.read_clock()
                assert ck["active"].all() and (ck["snaps"] == 1).all() and not ck["overflow"].any(), f
                if f != "clocked":
                    assert list(ck["slot_member"]) == list(range(B)) and ck["next"] == B, f  # nobody stopped
            med = {f: float(np.median(t)) for f, t in times.items()}
            spread = {f: float(max(t) - min(t)) for f, t in times.items()}
            r = {"B": B, "H": H, "W": W, "replays_per_window": reps, "ms_per_step": times, "median_ms": med,
                 "spread_ms": spread,
                 "chained_over_sweep_us_per_step": 1e3 * (med["chained"] - med["sweep"]),
                 "chained_over_sweep_pct": 100.0 * (med["chained"] - med["sweep"]) / med["sweep"],
                 "sweep_over_clocked_us_per_step": 1e3 * (med["sweep"] - med["clocked"])}
            res["sizes"][tag] = r
            print(f"{tag}: " + ", ".join(f"{f} {med[f]:.4f} ms/step (spread {spread[f]:.4f})" for f in FORMS) +
                  f"; chained over sweep {r['chained_over_sweep_us_per_step']:+.2f} us/step = "
                  f"{r['chained_over_sweep_pct']:+.2f} %", flush=True)
            del runs, net
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
