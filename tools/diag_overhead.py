"""Cost of the per-step diagnostics (pbmc_rollout_diagnosed: wall fluxes and rms velocity in the clock's apply / commit
launches, no launch added) against the plain and the clocked rollout, in ms per step, at three sizes:
  * 512^2, B = 1, primary network (NewFluidNet(levels=6, c_h=16, c_o=2, k=3, replicate, symmetric, curl), bench.py's);
  * 32 members of 256^2, primary network;
  * 128 x 506, B = 1, the paper's learned-boundary network (levels 5, repeats 6, k 5).
Four forms of the same EnsembleRollout configuration as 10-step CUDA graphs: plain; clocked (t_end = inf, one snapshot
at the first step, then none); clocked + diagnostics (window = 0); clocked + diagnostics + steady criterion
(window = 64, rtol = 0: the window is scanned after every step and never holds).  tools/clock_overhead.py's method:
CUDA events over back-to-back replays, the forms' windows alternating in one process, L2 not flushed (a rollout runs its
steps back to back).  The card name and power limit are read and printed in the same run.

usage: python tools/diag_overhead.py [--windows N] [--replays N] [--out FILE.json]"""
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
FORMS = {"plain": None, "clocked": {}, "diag": {"diagnostics": True}, "diag_steady": {"steady": (64, 0.0)}}


def make(net, B, H, W, clock):
    params = [(PARAMS[0] * (1.0 + 0.01 * i), PARAMS[1], PARAMS[2]) for i in range(B)]
    ens = EnsembleRollout(net, H, W, params, DEV, per_member_dt=True, max_steps=64)
    ens.set_T(np.stack([synthetic_T0(H, W, seed=i) for i in range(B)]))
    if clock is not None:
        ens.start_clock(np.inf, save_every=np.inf, steps_per_graph=K, **clock)
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
            runs = {f: make(net, B, H, W, c) for f, c in FORMS.items()}
            for _, g in runs.values():  # warm-up
                for _ in range(3):
                    g.replay()
            torch.cuda.synchronize(DEV)
            reps = a.replays or max(3, int(300.0 / (K * window_ms(runs["plain"][1], 3))))
            times = {f: [] for f in FORMS}
            for _ in range(a.windows):
                for f, (_, g) in runs.items():
                    times[f].append(window_ms(g, reps))
            for f, (ens, _) in runs.items():
                assert bool(torch.isfinite(ens.T).all()), f
                if FORMS[f] is not None:
                    ck = ens.read_clock()
                    assert ck["active"].all() and (ck["snaps"] == 1).all() and not ck["overflow"].any(), f
                    assert "steady" not in ck or not ck["steady"].any(), f
            med = {f: float(np.median(t)) for f, t in times.items()}
            r = {"B": B, "H": H, "W": W, "replays_per_window": reps, "ms_per_step": times,
                 "median_ms": med, "spread_ms": {f: float(max(t) - min(t)) for f, t in times.items()},
                 "diag_over_clocked_us_per_step": 1e3 * (med["diag"] - med["clocked"]),
                 "diag_steady_over_clocked_us_per_step": 1e3 * (med["diag_steady"] - med["clocked"]),
                 "diag_steady_over_clocked_pct": 100.0 * (med["diag_steady"] - med["clocked"]) / med["clocked"]}
            res["sizes"][tag] = r
            print(f"{tag}: " + ", ".join(f"{f} {med[f]:.4f} ms/step (spread {r['spread_ms'][f]:.4f})" for f in FORMS) +
                  f"; diagnostics +{r['diag_over_clocked_us_per_step']:.2f} us/step, with the window scan "
                  f"+{r['diag_steady_over_clocked_us_per_step']:.2f} us/step = {r['diag_steady_over_clocked_pct']:.2f} % "
                  "over clocked", flush=True)
            del runs, net
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
