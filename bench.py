#!/usr/bin/env python
"""Benchmark of the surrogate time-stepping hot path (BASELINE.json metric: rollout cell-updates/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

One "step" = one time step of the rollout (7-channel input build -> conv surrogate -> curl/BC/
un-scale head -> advection-diffusion update with the CFL dt) over one batch of synthetic T.
Default workload = BASELINE config 2: 512x512, batch 1, random-init primary network
(`NewFluidNet(levels=6, c_h=16, c_o=2, k=3, replicate, symmetric, curl)`), float32 kernels.
With --gpus N every rank runs its own independent rollout (members differ in Ra and T0):
no data-path collective, weak scaling, value = sum over ranks / max time over ranks.

Prints ONE JSON line (rank 0).  With --dump-outputs DIR, rank 0 also writes what the timed rollout returned after its
last timed step to DIR/<name>.npy (see dump_outputs); the inputs are seeded, so two builds can be compared output for
output.  `--impl reference` times the CPU port of the reference
(`oracle/ref_torch.py`, the reference is PyTorch and cannot travel to the GPU box) on the
host cores, same metric and config.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written there

import numpy as np  # noqa: E402
import torch  # noqa: E402

PARAMS0 = (6.79733173, 475523342.0, 2.58574662)  # load_fluidnet.ipynb:847 (a CV simulation)
FLOP_PER_CELL = 61434  # SURVEY.md section 8a, primary config on 2^n grids
WORKLOADS = {
    "rollout512": dict(H=512, W=512, B=1, desc="512x512 batch-1 surrogate rollout (BASELINE config 2)"),
    "rollout128": dict(H=128, W=128, B=1, desc="128x128 batch-1 surrogate rollout (BASELINE config 1 grid)"),
    "ensemble256": dict(H=256, W=256, B=32, desc="32 members/GPU of 256x256 (BASELINE config 4, weak scaling)"),
    "slab8192": dict(H=8192, W=8192, B=1, desc="one 8192x8192 grid, row slabs over the ranks: stencil + one-row T halo "
                                                "send/recv + dt all-reduce, given u,v (BASELINE config 5, strong scaling)"),
}


def member_params(n, rank=0):
    """Ensemble parameters: member 0 of rank 0 is the reference CV simulation, the others are drawn
    from the ranges of the 130 simulations of the paper (SURVEY.md section 8d)."""
    rng = np.random.default_rng(2024 + rank)
    out = []
    for m in range(n):
        if m == 0 and rank == 0:
            out.append(PARAMS0)
        else:
            out.append((float(rng.uniform(0.126, 9.98)), float(10 ** rng.uniform(6.0035, 9.8888)),
                        float(10 ** rng.uniform(0.00525, 1.9928))))
    return out


def primary_net(device, dtype=torch.float32):
    import pbml_mantle_convection_b200 as P

    torch.manual_seed(0)
    net = P.NewFluidNet(6, 7, 16, 2, device, act_fn="gelu", r_p="replicate", loss_type="curl", use_symm=True, dilation=1,
                        a_bound=10, repeats=4, f=3, p_pred=True, factor=2)
    return net.to(dtype).to(device).eval()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


# ---------------------------------------------------------------------------------------- CPU arm
def cpu_port_rate(H, W, n_steps, warmup=1, dtype=torch.float64):
    """cell-updates/s of the ATen-CPU port of the reference rollout (oracle/ref_torch.py), all host threads."""
    from oracle import ref_numpy as RN
    from oracle import ref_torch as RT

    torch.set_num_threads(os.cpu_count() or 1)
    spec = RN.NetSpec()
    net = primary_net("cpu", torch.float64)
    sd = {k: v.detach().numpy() for k, v in net.state_dict().items()}
    Wt = RT.prepare_weights(sd, spec, dtype)
    xc, yc = RN.synthetic_grid(H, W)
    T = torch.tensor(RN.synthetic_T0(H, W, seed=1), dtype=dtype)[None, None]
    xc, yc = torch.tensor(xc, dtype=dtype), torch.tensor(yc, dtype=dtype)
    with torch.no_grad():
        for _ in range(warmup):
            T = RT.ts_step(Wt, spec, T, xc, yc, *PARAMS0)[0]
        t0 = time.perf_counter()
        for _ in range(n_steps):
            T = RT.ts_step(Wt, spec, T, xc, yc, *PARAMS0)[0]
        dt = time.perf_counter() - t0
    return H * W * n_steps / dt, dt, torch.get_num_threads()


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H, W, B = wl["H"], wl["W"], wl["B"]
    rate, secs, threads = cpu_port_rate(H, W, args.steps, warmup=max(1, min(args.warmup, 3)))
    line = {
        "impl": "reference", "metric": "rollout cell-updates/s", "value": rate, "unit": "cell-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "grid": [H, W], "batch": 1, "note": "one member on the host cores"},
        "cpu_baseline": {"value": rate, "unit": "cell-updates/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} time steps of the {H}x{W} rollout, float64, ATen CPU port of the reference "
                                   f"(oracle/ref_torch.py), {threads} threads"},
        "e2e": {"value": rate, "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------- GPU arm
def time_kernel(fn, iters=20, warm=3, flush=None):
    """Average device time (ms) of fn() with CUDA events on the current stream; optional L2 flush between launches."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        tot += a.elapsed_time(b)
    return tot / iters


def kernel_rooflines(net, H, W, B, dev, flush):
    """Live CUDA-event timing of the dominant kernels on this workload's shapes (DESIGN.md section 5)."""
    from pbml_mantle_convection_b200 import _lib as L
    from pbml_mantle_convection_b200 import ops

    eng = net._engine(dev)
    hbm, tf_burst, tf_sus, which = measured_peaks()
    cells = B * H * W
    g = torch.Generator(device=dev).manual_seed(5)
    act = lambda nb: torch.randn(B, nb, H, W, 4, device=dev, generator=g)
    x16 = act(4)
    stats = torch.stack([x16.double().sum((2, 3, 4)), (x16.double() ** 2).sum((2, 3, 4))], -1).contiguous()
    out = {}
    # (1) trunk layer 16->16 3x3 at level 0, GN+GELU fused on load, stats in the epilogue: 128 B / cell, 4608 FLOP / cell
    lay = eng.trunk[0][1]
    src = ops.Source(x16, L.XFORM_GN_GELU, stats, lay.gamma, lay.beta)
    o16, st16 = torch.empty_like(x16), torch.zeros_like(stats)
    ms = time_kernel(lambda: ops.conv_fwd([src], lay.wpk, lay.bias, 16, 3, "replicate", impl=net.conv_impl,
                                          wpk_umma=lay.wpk_umma, wpk_row=lay.wpk_row, out=o16, stats=st16), flush=flush)
    out["conv16x16_l0"] = {"ms": ms, "bound": "hbm", "achieved": cells * 128 / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                           "tflops": cells * 4608 / (ms * 1e-3) / 1e12}
    # (1b) the R = 4 level-0 trunk layers as ONE persistent launch (csrc/conv_trunk.cu): 4 x 128 B / cell, 4 x 4608 FLOP / cell
    if net.conv_impl in ("auto", "mux_f16x2", "row_f16x2", "mux_bf16", "row_bf16") and getattr(net, "trunk_mode", "auto") == "auto":
        lays = eng.trunk[0]
        ping = [torch.empty_like(x16), torch.empty_like(x16)]
        st_all = torch.empty(len(lays), B, 4, 2, dtype=torch.float64, device=dev)
        sync = torch.empty(B, dtype=torch.int32, device=dev)
        try:
            ms = time_kernel(lambda: ops.trunk_fwd(src, lays, "replicate", impl=net.conv_impl, ping=ping, stats=st_all, sync=sync),
                             flush=flush)
            out["trunk_l0"] = {"ms": ms, "layers": len(lays), "bound": "hbm", "achieved": len(lays) * cells * 128 / (ms * 1e-3) / 1e9,
                               "peak": hbm, "unit": "GB/s", "tflops": len(lays) * cells * 4608 / (ms * 1e-3) / 1e12,
                               "ms_per_layer": ms / len(lays),
                               "note": "one launch = all trunk layers of the level (+ two 4-byte/128-byte memsets of its scratch)"}
        except L.PbmcError:
            pass  # grid cannot be resident at once on this shape: the rollout runs the layers one by one
    # (2) conv[1]: 103 -> 16 over 7 sources: 29664 FLOP / cell (48 % of the forward), (96+8+16)*4 = 480 B / cell
    srcs = [src] + [ops.Source(act(4)) for _ in range(5)] + [ops.Source(act(2))]
    c1 = eng.conv1
    ms = time_kernel(lambda: ops.conv_fwd(srcs, c1.wpk, c1.bias, 16, 3, "replicate", impl=net.conv_impl,
                                          wpk_umma=c1.wpk_umma, wpk_row=c1.wpk_row, out=o16, stats=st16), flush=flush)
    out["conv1_103x16"] = {"ms": ms, "bound": "tensor", "achieved": cells * 29664 / (ms * 1e-3) / 1e12, "peak": tf_burst,
                           "unit": "TFLOP/s", "gbs": cells * 480 / (ms * 1e-3) / 1e9}
    # (3) advection-diffusion stencil + CFL reduce: 16 B / cell
    T = torch.rand(B, H, W, device=dev, generator=g)
    u = torch.randn(B, H, W, device=dev, generator=g) * 1e3
    v = torch.randn(B, H, W, device=dev, generator=g) * 1e3
    grid = eng_grid(H, W, dev)
    members = ops.make_members([PARAMS0] * B, dev)
    uv = ops.uvmax_reduce(u, v)
    To, dto, uvo = torch.empty_like(T), torch.empty(B, dtype=torch.float64, device=dev), torch.zeros_like(uv)
    ms = time_kernel(lambda: ops.advect_diffuse(T, u, v, grid.xcoef, grid.ycoef, members, uv, grid.dx_min, 0.99, T_out=To,
                                                dt_out=dto, uv_out=uvo), flush=flush)
    out["stencil"] = {"ms": ms, "bound": "hbm", "achieved": cells * 16 / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s"}
    for k in out.values():
        k["frac"] = k["achieved"] / k["peak"]
        k["peak_source"] = which
    return out


def stencil_sweep(dev, sizes=(256, 512, 1024, 2048, 4096, 8192), sweeps=50):
    """BASELINE config 3: the advection-diffusion stencil + in-pass CFL reduction alone, ping-pong over `sweeps`
    steps per grid (16 B per cell-update: T, u, v in, T' out; max|u|,|v| comes out of the same pass).  Grids whose
    four fields fit the 126 MB L2 (<= 2048^2) are L2-resident by construction -- the GB/s there is not an HBM number."""
    from pbml_mantle_convection_b200 import ops

    hbm, _, _, which = measured_peaks()
    rows = []
    g = torch.Generator(device=dev).manual_seed(7)
    for n in sizes:
        grid = eng_grid(n, n, dev)
        T = torch.rand(1, n, n, device=dev, generator=g)
        xs = torch.linspace(0, 1, n, device=dev)
        psi = torch.sin(3.14159265 * 3 * xs)[None, :] * torch.sin(3.14159265 * xs)[:, None]
        u = ((psi[2:, :] - psi[:-2, :]) * n * 50).new_zeros(n, n)
        u[1:-1] = (psi[2:, :] - psi[:-2, :]) * n * 50
        v = torch.zeros(n, n, device=dev)
        v[:, 1:-1] = -(psi[:, 2:] - psi[:, :-2]) * n * 50
        u, v = u[None].contiguous(), v[None].contiguous()
        members = ops.make_members([PARAMS0], dev)
        uv = [ops.uvmax_reduce(u, v), torch.zeros(1, dtype=torch.int32, device=dev)]
        Tb = [T, torch.empty_like(T)]
        dto = torch.empty(1, dtype=torch.float64, device=dev)

        def run(k):
            for i in range(k):
                uv[(i + 1) % 2].zero_()
                ops.advect_diffuse(Tb[i % 2], u, v, grid.xcoef, grid.ycoef, members, uv[i % 2], grid.dx_min, 0.99,
                                   T_out=Tb[(i + 1) % 2], dt_out=dto, uv_out=uv[(i + 1) % 2])

        run(4)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()  # the ping-pong loop as one graph: no per-launch host cost in the timing
        with torch.cuda.graph(graph):
            run(sweeps)
        graph.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b) / sweeps
        gbs = n * n * 16 / (ms * 1e-3) / 1e9
        rows.append({"grid": [n, n], "ms_per_sweep": ms, "cell_updates_per_s": n * n / (ms * 1e-3), "achieved_gbs": gbs,
                     "frac_of_hbm_peak": gbs / hbm, "resident": "L2" if 4 * n * n * 4 <= 100e6 else "HBM"})
    return {"bytes_per_cell_update": 16, "peak_gbs": hbm, "peak_source": which, "sweeps": sweeps,
            "note": "CUDA events around one graph replay of the whole ping-pong loop (kernel + 4-byte memset per sweep)", "rows": rows}


def eng_grid(H, W, dev):
    import pbml_mantle_convection_b200 as P
    from pbml_mantle_convection_b200.engine import Grid

    xc, yc = P.synthetic_grid(H, W)
    xc, yc = torch.tensor(xc), torch.tensor(yc)
    return Grid(xc, yc, yc, dev)


def bind_host_to_gpu_numa_node(local, world=1):
    """Multi-rank runs only: pin this process (and the pinned host buffers it first-touches afterwards) to the CPUs NVML
    reports as local to its GPU.  Eight unpinned ranks each moving ~10 MB per 0.45 ms step through host memory measured
    4.5x one rank end to end (profiles/r1_bench_rollout512_8gpu.json).  Best effort: any failure leaves the affinity alone.
    Returns the number of CPUs bound to, or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(local).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        before = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = os.sched_getaffinity(0)
        if len(after) < 4:  # a degenerate mask would serialise the rank's helper threads: undo
            os.sched_setaffinity(0, before)
            return None
        # Several ranks whose GPUs report the SAME CPU set (this pool: all 8 GPUs on NUMA node 0, CPUs 0-31) would
        # still run on top of each other: give each rank its own contiguous slice of that set (>= 2 CPUs).
        cpus = sorted(after)
        per = len(cpus) // max(world, 1)
        if world > 1 and per >= 2:
            mine = cpus[(local % world) * per:(local % world + 1) * per]
            os.sched_setaffinity(0, set(mine))
            return len(mine)
        return len(after)
    except Exception:
        return None


def launches_per_step(L_, R_, persistent_trunk=False):
    # build_input + conv0 + trunk (L*R convs, or L persistent launches) + conv1..3 + (L-1) pools + (L-1) bicubic + head + stencil
    return 1 + 1 + (L_ if persistent_trunk else L_ * R_) + 3 + 2 * (L_ - 1) + 1 + 1


def dump_outputs(path, ens):
    """What a caller of EnsembleRollout holds after the last step: T and that step's u, v, p, V (float32 [B, H, W]) and each
    member's dt (float64 [B]), one DIR/<name>.npy each.  Every rollout workload stays below 64 MB in all
    (ensemble256: 32 members x 5 fields x 256 KiB = 40 MiB)."""
    os.makedirs(path, exist_ok=True)
    u, v, p, V = ens.fields()
    out = {"T": ens.T, "u": u, "v": v, "p": p, "V": V, "dt": ens.last_dt()[(ens.n_done - 1) % 2]}
    for name, t in out.items():
        if t is not None:
            np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def timed_rollout(net, H, W, B, rank, world, local, dev, K, Wm, flush, T0=None, dump=None):
    """Device-resident rollout of B members per rank: one CUDA graph per time step, L2 flushed (untimed) between steps,
    per-step CUDA-event intervals summed.  Returns (device ms over K steps on this rank, wall s, finite, clock sampler).
    With `dump` (a directory) the outputs of the last timed step are written there (dump_outputs)."""
    import torch.distributed as dist

    import pbml_mantle_convection_b200 as P

    prm = member_params(B, rank)
    ens = P.EnsembleRollout(net, H, W, prm, dev, cn_max=0.99, per_member_dt=True)
    if T0 is None:
        T0 = np.stack([P.synthetic_T0(H, W, seed=1 + rank * B + m) for m in range(B)])
    ens.set_T(T0)
    ens.run(Wm + (Wm % 2), steps_per_graph=1)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    evs = []
    with ClockSampler(local) as clk:
        wall0 = time.perf_counter()
        for _ in range(K):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ens.run(1, steps_per_graph=1, track_time=False)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        wall = time.perf_counter() - wall0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    finite = bool(torch.isfinite(ens.T).all().item())
    if dump:
        dump_outputs(dump, ens)
    return dev_ms, wall, finite, clk


def resident_loop_record(net, H, W, B, rank, dev, steps_per_graph=10, replays=10):
    """The rollout as a caller runs it (EnsembleRollout.run(n, steps_per_graph=k)): k time steps per CUDA graph, no L2 flush,
    CUDA events around all replays.  Inside a multi-step graph the next step's input build rides in the stencil launch
    (csrc/stencil.cu BUILD variant), which the one-step-per-graph protocol of the headline number cannot show."""
    import pbml_mantle_convection_b200 as P

    ens = P.EnsembleRollout(net, H, W, member_params(B, rank), dev, cn_max=0.99, per_member_dt=True)
    ens.set_T(np.stack([P.synthetic_T0(H, W, seed=1 + rank * B + m) for m in range(B)]))
    k = int(steps_per_graph)
    ens.run(2 * k, steps_per_graph=k, track_time=False)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ens.run(replays * k, steps_per_graph=k, track_time=False)
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / (replays * k)
    return {"ms_per_step": ms, "cell_updates_per_s": B * H * W / (ms * 1e-3), "steps_per_graph": k, "steps": replays * k,
            "l2": "not flushed (the loop as a caller runs it)", "finite": bool(torch.isfinite(ens.T).all().item()),
            "note": "secondary figure; the headline `value` keeps the one-step-per-graph, L2-flushed protocol"}


def ensemble_record(net, rank, world, local, dev, K, Wm, flush):
    """BASELINE config 4: 32 members of 256x256 per GPU (varied Ra / gamma / beta / initial T), batch-sharded over the
    ranks, per-member dt, no data-path collective -- weak scaling.  Rank 0 returns the record."""
    import torch.distributed as dist

    wl = WORKLOADS["ensemble256"]
    H, W, B = wl["H"], wl["W"], wl["B"]
    dev_ms, wall, finite, clk = timed_rollout(net, H, W, B, rank, world, local, dev, K, Wm, flush)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    fin = torch.tensor([int(finite)], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(fin, op=dist.ReduceOp.MIN)
    ms = t.item()
    return {"metric": "rollout cell-updates/s", "value": world * B * H * W * K / (ms * 1e-3), "unit": "cell-updates/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "dtype": "f32",
            "config": {"workload": "ensemble256", "desc": wl["desc"], "grid": [H, W], "batch_per_gpu": B, "members_total": world * B,
                       "parallelism": f"{world * B} independent members, {B} per GPU, no collective in the loop"},
            "surrogate_steps_per_s": world * B * K / (ms * 1e-3), "finite": bool(fin.item()), "clocks": clk.summary()}


def teardown(code=0):
    """Leave a multi-rank run: barrier, destroy the process group -- under a watchdog.  Round 1's 8-rank slab run printed its
    line and then never exited (process-group teardown with captured NCCL work alive); nothing captures NCCL any more and
    the normal path is taken, but a hung teardown must not turn a finished measurement into a killed run: after 60 s the
    process leaves without running destructors."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return
    dog = threading.Timer(60.0, lambda: (sys.stderr.write("bench.py: teardown watchdog fired\n"), sys.stderr.flush(), os._exit(code)))
    dog.daemon = True
    dog.start()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    dog.cancel()


def run_ours(args, wl):
    import torch.distributed as dist

    import pbml_mantle_convection_b200 as P

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (--impl ours) needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_host_to_gpu_numa_node(local, world) if world > 1 else None  # N = 1 keeps every core for the CPU baseline
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    H, W, B = wl["H"], wl["W"], wl["B"]
    K, Wm = args.steps, max(args.warmup, 3)
    net = primary_net(dev)
    net.conv_impl = args.conv
    net.trunk_mode = args.trunk
    net.up_staged = bool(args.up_staged)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2
    T0 = np.stack([P.synthetic_T0(H, W, seed=1 + rank * B + m) for m in range(B)])
    dev_ms, wall, finite, clk = timed_rollout(net, H, W, B, rank, world, local, dev, K, Wm, flush, T0,
                                              dump=args.dump_outputs if rank == 0 else None)

    # ---- end to end through the drop-in TS call with HOST float64 tensors (advect_wi_gaia.py:590-616)
    ts = P.TS(net, P.ADNet(dev, CN_max=0.99), dev, ts=1, scale=True, p_pred=True, net="newfluidnet")
    xc, yc = P.synthetic_grid(H, W)
    t64 = lambda a_: torch.tensor(a_, dtype=torch.float64)
    xc_t, yc_t = t64(xc).view(1, 1, H, W), t64(yc).view(1, 1, H, W)
    nd = ((PARAMS0[0] - 0.12624371) / (9.70723344 - 0.12624371),
          (np.log10(PARAMS0[1]) - 6.00352841978384) / (9.888820429862925 - 6.00352841978384),
          (np.log10(PARAMS0[2]) - 0.005251646002323797) / (1.9927988938926755 - 0.005251646002323797))
    args_ts = (None, None, yc_t, t64(nd[0]), t64(nd[1]), t64(nd[2]), t64(PARAMS0[0]), t64(PARAMS0[1]), t64(PARAMS0[2]), xc_t,
               yc_t)
    K2 = min(K, 50)

    def e2e_measure(host_dtype):
        """K2 calls of the drop-in TS.forward with a pinned HOST T of `host_dtype` in, and the driver's per-step readback
        (advect_wi_gaia.py:595-616 copies u, v, V and T_new to the host every step) into pinned host buffers.  T_new is
        the next call's (host) input, so it is read back on the main stream and waited for; u, v, V and dt of step k are
        read back on a side stream while step k+1 runs (every TS call returns fresh tensors, double-buffered on the host)
        -- all of it inside the timed region, drained before the clock stops.  TS returns tensors of its input's dtype
        (as the reference does), so a float32 host T halves every PCIe transfer; the kernels compute in fp32 either way."""
        Tp = torch.tensor(T0[:1], dtype=host_dtype).view(1, 1, H, W).pin_memory()
        pin = lambda: torch.empty(1, 1, H, W, dtype=host_dtype).pin_memory()
        hostT = [pin(), pin()]  # ping-pong: step k's T is step k+1's (pinned) input
        hostF = [[pin(), pin(), pin()], [pin(), pin(), pin()]]
        host_dt = [torch.empty(1, dtype=host_dtype).pin_memory() for _ in range(2)]
        calls = [0]
        side = torch.cuda.Stream(dev)
        side_done = [torch.cuda.Event(), torch.cuda.Event()]

        def step(Tp_):
            k = calls[0] % 2
            calls[0] += 1
            x, dts, u, v, p, V = ts(Tp_, *args_ts)
            main = torch.cuda.current_stream(dev)
            Tn_ = hostT[k]
            Tn_.copy_(x[1], non_blocking=True)
            side.wait_stream(main)
            side_done[k].synchronize()  # the host buffers of two steps ago are free again
            with torch.cuda.stream(side):
                for dst, src in zip(hostF[k], (u, v, V)):
                    dst.copy_(src, non_blocking=True)
                    src.record_stream(side)
                host_dt[k].copy_(dts[1].reshape(1), non_blocking=True)
                dts[1].record_stream(side)
                side_done[k].record(side)
            main.synchronize()
            return Tn_, sum(o.numel() * o.element_size() for o in (Tn_, *hostF[k], host_dt[k]))

        for _ in range(10):
            Tn, d2h = step(Tp)
        # The timed region (K2 steps, drained) is repeated three times and the MEDIAN reported: one run in five on a fresh
        # box showed a 2x slower first pass (host side: page-ins / link power state), which says nothing about the code.
        runs = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            Tc = Tp
            for _ in range(K2):
                Tc, d2h = step(Tc)
            torch.cuda.synchronize()  # includes the side stream: the last steps' u, v, V are on the host
            runs.append(time.perf_counter() - t0)
        return statistics.median(runs), runs, int(Tp.numel() * Tp.element_size()), int(d2h)

    e2e64_s, e2e64_runs, h2d64, d2h64 = e2e_measure(torch.float64)  # the reference driver's dtype (round-1 number)
    e2e_s, e2e_runs, h2d, d2h = e2e_measure(torch.float32)          # headline: same API, fp32 host tensors
    e2e_rate = H * W * K2 / e2e_s

    # ---- reduce over ranks: total units / max time
    t_ms = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    e2e_t = torch.tensor([e2e_s, e2e64_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    dev_ms = t_ms.item()
    value = world * B * H * W * K / (dev_ms * 1e-3)
    e2e_rate = world * H * W * K2 / e2e_t[0].item()
    e2e64_rate = world * H * W * K2 / e2e_t[1].item()

    line = None
    if rank == 0:
        roofs = kernel_rooflines(net, H, W, B, dev, flush)
        sweep = stencil_sweep(dev)
        step_ms = dev_ms / K
        # dominant kernel = largest share of the step (conv[1] runs once, the level-0 trunk layer R times)
        share = {"conv1_103x16": roofs["conv1_103x16"]["ms"], "stencil": roofs["stencil"]["ms"]}
        if "trunk_l0" in roofs:
            share["trunk_l0"] = roofs["trunk_l0"]["ms"]  # one persistent launch = the 4 level-0 trunk layers
        else:
            share["conv16x16_l0"] = roofs["conv16x16_l0"]["ms"] * 4
        dom = max(share, key=share.get)
        r = roofs[dom]
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if not os.path.exists(tpath):
            tpath = os.path.join(ROOT, "profiles", "r1_traffic.json")
        if args.workload == "rollout512" and os.path.exists(tpath):  # recorded ncu capture of this kernel at this shape
            rec = json.load(open(tpath)).get(dom)
            if rec:
                traffic, traffic_src = rec["dram_bytes_per_launch"], rec["source"]
        roofline = {"kernel": dom, "bound": r["bound"], "achieved": r["achieved"], "peak": r["peak"], "unit": r["unit"],
                    "frac": r["frac"], "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write, ncu)",
                    "traffic_source": traffic_src, "algorithmic_bytes_per_launch": B * H * W * {"conv16x16_l0": 128, "trunk_l0": 128 * 4, "conv1_103x16": 480}.get(dom, 16),
                    "peak_source": r["peak_source"], "ms_per_launch": r["ms"], "share_of_step": share[dom] / step_ms}
        if traffic is not None and rec.get("tensor_pipe_active_pct_of_active_cycles") is not None:
            # second view of the same kernel: how busy the tensor pipe was in the recorded ncu capture
            roofline["tensor_pipe_active_frac_ncu"] = rec["tensor_pipe_active_pct_of_active_cycles"] / 100.0
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            n_cpu = max(2, min(60, int(15.0 / (1.45e-6 * H * W))))  # ~10-30 s of CPU work (0.38 s per 512^2 step on 16 cores)
            rate, secs, threads = cpu_port_rate(H, W, n_cpu)
            cpu = {"value": rate, "unit": "cell-updates/s", "cores": threads, "kind": "port",
                   "sample": f"{n_cpu} time steps of the same {H}x{W} batch-1 rollout, float64 ATen-CPU port of the "
                             f"reference (oracle/ref_torch.py), {secs:.1f} s"}
        line = {
            "metric": "rollout cell-updates/s", "value": value, "unit": "cell-updates/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "desc": wl["desc"], "grid": [H, W], "batch_per_gpu": B,
                       "net": "NewFluidNet(levels=6,c_i=7,c_h=16,c_o=2,k=3,replicate,symm,curl,repeats=4)", "conv_impl": args.conv, "trunk": args.trunk, "up_staged": bool(args.up_staged),
                       "l2": "flushed (256 MiB write, untimed) between timed steps; per-step CUDA-event intervals summed",
                       "parallelism": f"{world} independent rollouts (no collective)" if world > 1 else "single GPU",
                       "host_affinity": f"each rank bound to its own {numa_cpus} CPUs out of its GPU's NUMA-local set (NVML)" if numa_cpus else "unbound",
                       "graph": "one CUDA graph per time step"},
            "surrogate_steps_per_s": world * K / (dev_ms * 1e-3),
            "gflop_per_step": B * H * W * FLOP_PER_CELL / 1e9,
            "wall_ms_per_step": 1e3 * wall / K,
            "roofline": roofline,
            "kernels": roofs,
            "stencil_sweep": sweep,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_rate, "unit": "cell-updates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": K2, "repeats_ms": [round(t_ * 1e3, 3) for t_ in e2e_runs], "value_is": "median of the repeats",
                    "host_dtype": "float32",
                    "api": "TS.forward(ts=1) with pinned host float32 T in (TS returns its input's dtype, like the reference; the kernels are fp32 either way, so nothing is lost and every PCIe transfer halves); every step T read back and waited for (it is the next input), u,v,V,dt read back on a side stream overlapping the next step; all drained inside the timed region",
                    "float64_host": {"value": e2e64_rate, "h2d_bytes_per_step": h2d64, "d2h_bytes_per_step": d2h64,
                                     "repeats_ms": [round(t_ * 1e3, 3) for t_ in e2e64_runs],
                                     "note": "the same loop with float64 host tensors (the reference driver's dtype, round 1's e2e)"}},
            "resident_loop": resident_loop_record(net, H, W, B, rank, dev),
            "gpu_launches": launches_per_step(6, 4, "trunk_l0" in roofs) * K,
            "clocks": clk.summary(),
            "finite": finite,
        }
    # ---- the two multi-GPU workloads of BASELINE.json as sub-records of the same line (every N, so that the driver's
    # 1/2/4/8 runs carry config 5's strong-scaling curve -- the path WITH a cross-rank exchange -- and config 4's weak one)
    subs = None
    if args.workload == "rollout512" and not args.no_sub_records:
        del ts
        torch.cuda.empty_cache()
        subs = {"ensemble256": ensemble_record(net, rank, world, local, dev, min(K, 20), 4, flush)}
        del flush
        torch.cuda.empty_cache()
        wls = WORKLOADS["slab8192"]
        subs["slab8192"] = slab_record(rank, world, local, dev, wls["H"], wls["W"], 100, 10, "p2p", "flags", wls["desc"])
        if line is not None:
            line["sub_records"] = subs
            line["gpu_launches"] += launches_per_step(6, 4) * subs["ensemble256"]["steps"] + subs["slab8192"]["steps"]
    if line is not None:
        emit(line)
    bad = False
    if subs is not None:
        sl = subs["slab8192"]
        bad = not (sl["finite"] and sl["bounded"] and sl["identical_to_single_gpu"] and subs["ensemble256"]["finite"])
    if world > 1:
        teardown(1 if bad else 0)
    if subs is not None:
        sl = subs["slab8192"]
        if not (sl["finite"] and sl["bounded"] and sl["identical_to_single_gpu"] and subs["ensemble256"]["finite"]):
            raise SystemExit("sub-record check failed: non-finite / unbounded field, or the decomposed slab run differs from the single-domain run")


def slab_velocity(xs, ys, H, W):
    """Smooth cellular flow for the slab workloads, STABLE for the explicit update on this grid (SURVEY.md section 8d
    config 3: "advective dt << diffusive dt, stable in both axes").  The reference takes dt from the x spacing only
    (pytorch_networks_convae.py:555-559), so on an H x W grid over the 4:1 box (dy = dx/4 when H = W) the explicit
    scheme needs  dt (|u|/dx + |v|/dy + 2/dx^2 + 2/dy^2) <= 1  with dt = 0.495 dx / max|u|:
      max|u| = 0.495 dx / (0.1 dy^2)  ->  dt 2/dy^2 = 0.2;   max|v| = 0.05 max|u|  ->  dt |v|/dy <= 0.1 dx/dy <= 0.1 * 4
    (total <= 0.2 + 0.0125 + 0.495 + 0.1 = 0.81 at H = W: a monotone update, T stays inside its initial range).
    Round 1's field (max|u| = 1e3, max|v| = 750 on 8192^2) violated both limits and blew up."""
    dx, dy = 4.0 / (W - 2), 1.0 / (H - 2)
    umax = max(1e3, 0.495 * dx / (0.1 * dy * dy))
    vmax = 0.05 * umax * min(1.0, 4.0 * dy / dx)
    pi = 3.141592653589793
    u = umax * torch.cos(pi * ys)[:, None] * torch.sin(pi * xs / 4 * 3)[None, :]
    v = -vmax * torch.sin(pi * ys)[:, None] * torch.cos(pi * xs / 4 * 3)[None, :]
    return u, v


def _slab_setup(H, W, rank, world, dev, halo, dt_sync):
    import pbml_mantle_convection_b200 as P
    from pbml_mantle_convection_b200 import multigpu as MG

    xc, yc = P.synthetic_grid(H, W)
    st = MG.SlabStencil(H, W, xc[0], yc[:, 0], rank, world, dev, raq=PARAMS0[0], cn_max=0.99, halo=halo, dt_sync=dt_sync)
    s = st.slab
    ys = torch.tensor(yc[s.l0:s.l1, 0], dtype=torch.float32, device=dev)
    xs = torch.tensor(xc[0], dtype=torch.float32, device=dev)
    # the same T0 on every decomposition: the noise is a function of the GLOBAL cell index
    rows = torch.arange(s.l0, s.l1, device=dev, dtype=torch.float32)[:, None]
    cols = torch.arange(W, device=dev, dtype=torch.float32)[None, :]
    T = (1.0 - ys)[:, None] + 0.01 * (0.5 + 0.5 * torch.sin(12.9898 * rows + 78.233 * cols))
    u, v = slab_velocity(xs, ys, H, W)
    st.set_local(T, u, v)
    return st


def slab_identity_check(rank, world, dev, halo, dt_sync, steps=6):
    """Short in-run check of the REAL multi-GPU path (peer stores + flag slots, or NCCL): a 1024-column grid with 64 rows
    per rank, `steps` steps through SlabStencil.step (graph replay included), gathered and compared BIT FOR BIT with the
    single-domain kernel run on rank 0."""
    import torch.distributed as dist

    import pbml_mantle_convection_b200 as P
    from pbml_mantle_convection_b200 import ops
    from pbml_mantle_convection_b200.engine import Grid

    H, W = 64 * world, 1024
    st = _slab_setup(H, W, rank, world, dev, halo, dt_sync)
    st.step(steps)
    got = st.gather()
    dt_last = float(st.last_dt[0])
    st.close()
    ok = torch.ones(1, dtype=torch.int32, device=dev)
    if rank == 0:
        one = _slab_setup(H, W, 0, 1, dev, "nccl", "nccl")  # world 1: the plain single-domain kernel
        one.step(steps)
        ref = one.gather()
        ok[0] = int(torch.equal(ref, got) and float(one.last_dt[0]) == dt_last and bool(torch.isfinite(got).all()))
    if world > 1:
        dist.broadcast(ok, 0)
    return bool(ok.item())


def slab_record(rank, world, local, dev, H, W, K, Wm, halo, dt_sync, desc):
    """BASELINE config 5: a single large grid, slab-decomposed over the ranks (strong scaling: total work fixed)."""
    import torch.distributed as dist

    identical = slab_identity_check(rank, world, dev, halo, dt_sync) if world > 1 else True
    st = _slab_setup(H, W, rank, world, dev, halo, dt_sync)
    s = st.slab
    Wm += Wm % 2
    K += K % 2  # whole ping-pong periods
    # Two ways to issue the steps, both timed (the record's value is the faster one): one kernel launch per step from the
    # host ("eager"), or CUDA graphs of 20 steps.  On two B200s the eager launches were FASTER (0.139 vs 0.150 ms per
    # 8192^2 step): the step is one ~0.1 ms kernel, so launch latency is hidden either way, and consecutive kernel nodes
    # of a graph started later after their predecessor than consecutive stream launches did.
    modes = {}
    with ClockSampler(local) as clk:
        for mode, gs in (("eager", 0), ("graph20", 20)) if world > 1 else (("eager", 0),):
            st.graph_steps = gs
            st.step(max(Wm, 2 * gs), use_graph=gs > 0)  # untimed: warm-up / capture
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            st.step(K, use_graph=gs > 0)
            b.record()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            modes[mode] = a.elapsed_time(b)
    names = sorted(modes)
    t_ms = torch.tensor([modes[m] for m in names], dtype=torch.float64, device=dev)
    fin = torch.tensor([int(torch.isfinite(st.T).all().item()), int(float(st.T.max()) <= 1.02 and float(st.T.min()) >= -0.02)],
                       dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(fin, op=dist.ReduceOp.MIN)
    per_mode = {m: t_ms[i].item() / K for i, m in enumerate(names)}
    best_mode = min(per_mode, key=per_mode.get)
    t_ms = torch.tensor([per_mode[best_mode] * K], dtype=torch.float64)
    ms = t_ms.item()
    st.close()
    hbm, _, _, which = measured_peaks()
    rate = H * W * K / (ms * 1e-3)
    gbs = rate * 16 / world / 1e9  # per rank: T, u, v in, T' out; max|u|,|v| for the next dt comes out of the same pass
    mode = ("halo rows stored into the neighbours' ghost rows by the update kernel (peer memory over NVLink); "
            + ("global max|u|,|v| exchanged through tag|value slots in peer memory INSIDE the kernel: one launch per step, no "
               "collective call" if dt_sync == "flags" else "NCCL all_reduce(MAX) of max|u|,|v| per step")) if (halo == "p2p" and world > 1) else \
           ("NCCL send/recv of one row each way + all_reduce(MAX) per step" if world > 1 else "single domain")
    return {"metric": "stencil cell-updates/s", "value": rate, "unit": "cell-updates/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "slab8192" if H == 8192 else f"slab{H}", "desc": desc, "grid": [H, W], "rows_per_rank": s.hi - s.lo,
                       "l2": "fields (4 x 256 MiB / ranks per rank) exceed L2 up to 8 ranks only marginally: 8192^2 x 4 fields x 4 B = 1 GiB total; no flush",
                       "parallelism": f"{world} row slabs; {mode}"},
            "roofline": {"kernel": "stencil_march_kernel", "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                         "frac": gbs / hbm, "traffic": None, "peak_source": which,
                         "note": "per GPU, 16 algorithmic B/cell; the step is ONE launch holding the dt reduction and the halo exchange"},
            "cpu_baseline": None, "e2e": None, "gpu_launches": K, "clocks": clk.summary(),
            "issue_mode": best_mode, "ms_per_step_by_issue_mode": per_mode,
            "finite": bool(fin[0].item()), "bounded": bool(fin[1].item()), "identical_to_single_gpu": identical}


def run_slab(args, wl):
    import torch.distributed as dist

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rec = slab_record(rank, world, local, dev, wl["H"], wl["W"], args.steps, max(args.warmup, 3), args.halo, args.dt_sync, wl["desc"])
    if rank == 0:
        emit(rec)
    if world > 1:
        teardown(0 if (rec["finite"] and rec["bounded"] and rec["identical_to_single_gpu"]) else 1)
    if not (rec["finite"] and rec["bounded"] and rec["identical_to_single_gpu"]):
        raise SystemExit("slab workload: non-finite / unbounded field or the decomposed run differs from the single-domain run")


_REAL_STDOUT = None


def _own_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner to
    fd 1 when NCCL_DEBUG is set on the box), so fd 1 is pointed at stderr for the whole run and the JSON line goes to
    a private duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _own_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rollout512", choices=sorted(WORKLOADS))
    ap.add_argument("--conv", default="auto", choices=["auto", "ffma", "umma_3xtf32", "umma_bf16", "umma_f16x2", "row_f16x2", "row_bf16", "mux_f16x2", "mux_bf16"])
    ap.add_argument("--trunk", default="auto", choices=["auto", "per_layer", "auto_bulk_loader"],
                    help="auto: the R trunk layers of a pyramid level as one persistent launch where it fits; per_layer: one launch per layer")
    ap.add_argument("--up-staged", dest="up_staged", action="store_true",
                    help="up-sampled pyramid levels written as conv[1]'s fp16 hi|lo operand image and staged by TMA bulk copies")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--halo", default="p2p", choices=["nccl", "p2p"], help="slab workloads: how the one-row T halo moves")
    ap.add_argument("--dt-sync", dest="dt_sync", default="flags", choices=["flags", "nccl"],
                    help="slab workloads with --halo p2p: global dt reduction inside the kernel (flags) or NCCL all_reduce per step")
    ap.add_argument("--no-sub-records", action="store_true", help="default workload: skip the slab8192 / ensemble256 sub-records")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the GPU rollout to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload.startswith("slab")):
        ap.error("--dump-outputs applies to the GPU rollout workloads (--impl ours, not slab)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif args.workload.startswith("slab"):
        run_slab(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
