"""Developer tool: wall time of one forward of the paper's learned-boundary network (SURVEY.md section 8f N1:
levels=5, r_p="learned", repeats=6, f=5, c_o=1; 2.13 M parameters) at the GAIA grid 128x506: `net(x)`, which is the fused
engine's forward, replayed as a CUDA graph and eager; for comparison the module-level composition that FluidNet and the
shapes the engine refuses run (eager).
usage: python tools/learned_time.py [H W]"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pbml_mantle_convection_b200 as P  # noqa: E402
from pbml_mantle_convection_b200.pytorch_networks_convae import _forward_learned_modules  # noqa: E402

dev = torch.device("cuda:0")
H, W = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (128, 506)
torch.manual_seed(0)
net = P.NewFluidNet(5, 7, 16, 1, dev, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10, repeats=6,
                    f=5, p_pred=False).to(dev).eval()
x = torch.randn(1, 7, H, W, device=dev)


def run(label, fwd):
    with torch.no_grad():
        for _ in range(3):
            u, v, p = fwd()
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            u, v, p = fwd()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
    print(f"learned-boundary paper config {H}x{W}, {label}: forward {min(ts) * 1e3:.2f} ms (best of 5, wall), "
          f"{H * W / min(ts):.3e} cells/s, finite={bool(torch.isfinite(u).all())}", flush=True)
    return u


# the fused engine: one stream per pyramid level, every 9-region conv = interior conv + ring kernel
u_g = run("net(x) (fused engine), CUDA-graph replay", lambda: net(x))
net.use_cuda_graph = False
u_e = run("net(x) (fused engine), eager launches", lambda: net(x))
print("graph replay == eager:", bool(torch.equal(u_g, u_e)))
u_m = run("module-level composition, eager launches", lambda: _forward_learned_modules(net, x, 1, True))
print(f"module-level composition vs engine: max|du| / max|u| = {float((u_m - u_e).abs().max() / u_e.abs().max()):.2e}")
