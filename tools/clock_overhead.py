"""Cost of the run-to-time clock (pbmc_rollout_clocked: two launches behind every step's stencil) against the plain
rollout, in ms per step, at three sizes:
  * 512^2, B = 1, primary network (NewFluidNet(levels=6, c_h=16, c_o=2, k=3, replicate, symmetric, curl), bench.py's);
  * 32 members of 256^2, primary network;
  * 128 x 506, B = 1, the paper's learned-boundary network (levels 5, repeats 6, k 5).
Both forms run as 10-step CUDA graphs of the same EnsembleRollout configuration (clocked: t_end = inf, one snapshot at
the first step, then none), timed with CUDA events over back-to-back replays, alternating unclocked / clocked windows
in one process.  The L2 is not flushed (a rollout runs its steps back to back).  The card name and power limit are read
and printed in the same run.

usage: python tools/clock_overhead.py [--windows N] [--replays N] [--out FILE.json]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pbml_mantle_convection_b200 as P  # noqa: E402
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_T0  # noqa: E402
from tools.learned_rollout_time import card, paper_net  # noqa: E402

DEV = torch.device("cuda:0")
PARAMS = (6.797, 4.755e8, 2.586)  # (RaQ, gamma, beta)
K = 10


def primary_net():
    torch.manual_seed(0)
    net = P.NewFluidNet(6, 7, 16, 2, DEV, act_fn="gelu", r_p="replicate", loss_type="curl", use_symm=True, dilation=1,
                        a_bound=10, repeats=4, f=3, p_pred=True, factor=2)
    return net.to(DEV).eval()


def make(net, B, H, W, clocked):
    params = [(PARAMS[0] * (1.0 + 0.01 * i), PARAMS[1], PARAMS[2]) for i in range(B)]
    ens = EnsembleRollout(net, H, W, params, DEV, per_member_dt=True, max_steps=64)
    ens.set_T(np.stack([synthetic_T0(H, W, seed=i) for i in range(B)]))
    if clocked:
        ens.start_clock(np.inf, save_every=np.inf, steps_per_graph=K)
    return ens, ens.graph(K)


def window_ms(g, replays):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / (replays * K)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=7, help="alternating unclocked / clocked windows per size")
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
            plain, g_plain = make(net, B, H, W, False)
            clk, g_clk = make(net, B, H, W, True)
            for g in (g_plain, g_clk):  # warm-up
                for _ in range(3):
                    g.replay()
            torch.cuda.synchronize(DEV)
            reps = a.replays or max(3, int(300.0 / (K * window_ms(g_plain, 3))))
            t_plain, t_clk = [], []
            for _ in range(a.windows):
                t_plain.append(window_ms(g_plain, reps))
                t_clk.append(window_ms(g_clk, reps))
            assert bool(torch.isfinite(plain.T).all()) and bool(torch.isfinite(clk.T).all())
            ck = clk.read_clock()
            assert ck["active"].all() and (ck["snaps"] == 1).all() and not ck["overflow"].any()
            mp, mc = float(np.median(t_plain)), float(np.median(t_clk))
            r = {"B": B, "H": H, "W": W, "replays_per_window": reps, "plain_ms_per_step": t_plain, "clocked_ms_per_step": t_clk,
                 "plain_median_ms": mp, "clocked_median_ms": mc, "overhead_us_per_step": 1e3 * (mc - mp),
                 "overhead_pct": 100.0 * (mc - mp) / mp,
                 "plain_spread_ms": float(max(t_plain) - min(t_plain)), "clocked_spread_ms": float(max(t_clk) - min(t_clk))}
            res["sizes"][tag] = r
            print(f"{tag}: plain {mp:.4f} ms/step (spread {r['plain_spread_ms']:.4f}), clocked {mc:.4f} ms/step "
                  f"(spread {r['clocked_spread_ms']:.4f}): overhead {r['overhead_us_per_step']:.2f} us/step = "
                  f"{r['overhead_pct']:.2f} %", flush=True)
            del plain, clk, g_plain, g_clk, net
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
