"""Time step of the paper's learned-boundary network (SURVEY.md section 8f N1: NewFluidNet(levels=5, r_p="learned",
repeats=6, f=5, c_o=1, p_pred=False), 2.13 M parameters) on the fused device-resident rollout, against the per-step
composition TS.forward used for it before (input build, module-level forward replayed as a CUDA graph, uvmax reduction,
stencil -- each issued from Python), plus the ring kernel (pbmc_conv_edge9) alone.

All times are CUDA-event times over many back-to-back steps after a warm-up.  The L2 is NOT flushed between steps: a
rollout runs its steps back to back, and one step's working set (under 60 MB at 128 x 506, B = 1) stays in the 126 MB
L2 as it would in use.  The card name and power limit are read and printed in the same run.

usage: python tools/learned_rollout_time.py [--steps N] [--only fused|all] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pbml_mantle_convection_b200 as P  # noqa: E402
from pbml_mantle_convection_b200 import _lib as L, engine, ops  # noqa: E402
from pbml_mantle_convection_b200.rollout import EnsembleRollout, synthetic_T0, synthetic_grid  # noqa: E402

DEV = torch.device("cuda:0")
PARAMS = (6.797, 4.755e8, 2.586)  # (RaQ, gamma, beta)


def card():
    name = torch.cuda.get_device_name(DEV)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unknown ({e})"
    return name, q


def paper_net():
    torch.manual_seed(0)
    net = P.NewFluidNet(5, 7, 16, 1, DEV, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10,
                        repeats=6, f=5, p_pred=False).to(DEV).eval()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, P.BoundaryLearnedConvolution2D):
                m.learnable_bias.normal_(0.0, 0.1)
    return net


def events_ms(fn, n, warm=3):
    """Mean device time of fn() over n calls (events around the whole window, one sync at the end)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(DEV)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def ensemble_ms_per_step(net, B, H, W, steps):
    params = [(PARAMS[0] * (1.0 + 0.01 * i), PARAMS[1], PARAMS[2]) for i in range(B)]
    ens = EnsembleRollout(net, H, W, params, DEV, per_member_dt=True, max_steps=64)
    ens.set_T(np.stack([synthetic_T0(H, W, seed=i) for i in range(B)]))
    k = 10
    n = max(1, steps // k)
    ms = events_ms(lambda: ens.run(k, steps_per_graph=k, track_time=False), n) / k
    assert bool(torch.isfinite(ens.T).all())
    return ms


def ts_ms_per_step(net, H, W, steps):
    xc, yc = synthetic_grid(H, W)
    T0 = synthetic_T0(H, W)
    from oracle.ref_numpy import nondim_params

    ts = P.TS(net, P.ADNet(DEV, CN_max=0.99), DEV, ts=1, scale=True, p_pred=False, net="newfluidnet")
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    nd = nondim_params(*PARAMS)
    args = (t64(T0).view(1, 1, H, W), None, None, t64(yc).view(1, 1, H, W), t64(nd[0]), t64(nd[1]), t64(nd[2]),
            t64(PARAMS[0]), t64(PARAMS[1]), t64(PARAMS[2]), t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W))
    ms = events_ms(lambda: ts(*args), steps)
    assert ts._plan is not None and ts._plan.graph is not None, "TS did not take the fused rollout"
    return ms


def per_step_composition_ms(net, H, W, steps):
    """What TS.forward ran per step for a learned net before: build_input -> net(...) (module-level forward, CUDA-graph
    replay) -> un-scale -> uvmax -> advect_diffuse, every call issued from Python."""
    xc, yc = synthetic_grid(H, W)
    grid = engine.Grid(torch.tensor(xc), torch.tensor(yc), torch.tensor(yc), DEV)
    members = ops.make_members([PARAMS], DEV)
    state = {"T": torch.tensor(synthetic_T0(H, W), dtype=torch.float32, device=DEV).reshape(1, H, W).contiguous()}

    def step():
        inp, V = ops.build_input(state["T"], grid.xc, grid.yc, grid.ycc, members, want_V=True)
        uu, vv, _ = net(ops.unpack_nchw(inp, 7))
        s = members[:, 6].reshape(1, 1, 1)
        u, v = (uu.float() * s).contiguous(), (vv.float() * s).contiguous()
        uvmax = ops.uvmax_reduce(u, v, batch_global=True)
        state["T"], _, _ = ops.advect_diffuse(state["T"], u, v, grid.xcoef, grid.ycoef, members, uvmax, grid.dx_min, 0.99,
                                              per_member_dt=False)

    return events_ms(step, steps)


def ring_kernel_us(B, H, W, src_channels, cout, k=5, n=200):
    """pbmc_conv_edge9 alone on the ring of one layer's output (sources raw, statistics repaired)."""
    g = torch.Generator(device=DEV).manual_seed(0)
    srcs = [ops.Source(torch.randn(B, ops.nblk(c), H, W, 4, device=DEV, generator=g)) for c in src_channels]
    ws = [torch.randn(cout, sum(src_channels), k, k, device=DEV, generator=g) * 0.05 for _ in range(8)]
    wedge = ops.pack_edge9_weights(ws, src_channels)
    bias = ops.pad_vec(torch.zeros(cout), cout, DEV)
    out = torch.zeros(B, ops.nblk(cout), H, W, 4, device=DEV)
    stats = torch.zeros(B, ops.nblk(cout), 2, dtype=torch.float64, device=DEV)
    return 1e3 * events_ms(lambda: ops.conv_edge9(srcs, wedge, bias, cout, k, L.ACT_NONE, out, stats), n, warm=10)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--only", choices=["fused", "all"], default="all")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: these are device timings")
    name, lim = card()
    res = {"card": name, "power_limit_and_max_sm_clock": lim, "l2_flushed": False, "steps": a.steps,
           "chain_pdl_env": os.environ.get("PBMC_CHAIN_PDL")}
    print(f"card: {name}; power limit, max SM clock: {lim}; L2 not flushed between steps", flush=True)
    net = paper_net()
    H, W = 128, 506
    with torch.no_grad():
        res["fused_ensemble_B1_128x506_ms_per_step"] = ensemble_ms_per_step(net, 1, H, W, a.steps)
        print(f"fused rollout, EnsembleRollout B=1 {H}x{W}, 10 steps per graph: "
              f"{res['fused_ensemble_B1_128x506_ms_per_step']:.4f} ms/step", flush=True)
        if a.only == "all":
            res["fused_ts1_128x506_ms_per_step"] = ts_ms_per_step(net, H, W, a.steps)
            print(f"fused rollout, TS(ts=1).forward with host float64 tensors: {res['fused_ts1_128x506_ms_per_step']:.4f} ms/step",
                  flush=True)
            res["per_step_composition_128x506_ms_per_step"] = per_step_composition_ms(net, H, W, max(20, a.steps // 4))
            print(f"per-step composition (previous TS path): {res['per_step_composition_128x506_ms_per_step']:.4f} ms/step",
                  flush=True)
        res["fused_ensemble_B32_256x256_ms_per_step"] = ensemble_ms_per_step(net, 32, 256, 256, max(20, a.steps // 4))
        print(f"fused rollout, EnsembleRollout 32 x 256^2, 10 steps per graph: "
              f"{res['fused_ensemble_B32_256x256_ms_per_step']:.4f} ms/step (all 32 members)", flush=True)
        if a.only == "all":
            for tag, (b, h, w, src, co) in {"trunk_l0_128x506": (1, 128, 506, [16], 16),
                                            "conv1_128x506": (1, 128, 506, [16] * 5 + [7], 16),
                                            "conv3_128x506": (1, 128, 506, [16], 1),
                                            "trunk_l0_32x256x256": (32, 256, 256, [16], 16)}.items():
                us = ring_kernel_us(b, h, w, src, co)
                res[f"ring_kernel_{tag}_us"] = us
                print(f"ring kernel alone, {tag} (sources {src}, c_out {co}, k 5): {us:.2f} us", flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
