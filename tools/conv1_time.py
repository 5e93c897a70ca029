"""Developer tool: CUDA-event time of the head conv conv[1] alone (103 -> 16, 3x3: five up-sampled levels + the level-0
trunk output with GroupNorm+GELU on load + the 7 raw input channels), L2 flushed between launches.
usage: python tools/conv1_time.py [H W [impl]]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pbml_mantle_convection_b200 import _lib as L  # noqa: E402
from pbml_mantle_convection_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
H, W = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (512, 512)
impl = sys.argv[3] if len(sys.argv) > 3 else "row_f16x2"
g = torch.Generator(device=dev).manual_seed(5)
torch.manual_seed(0)
x = torch.randn(1, 4, H, W, 4, device=dev, generator=g)
stats = torch.stack([x.double().sum((2, 3, 4)), (x.double() ** 2).sum((2, 3, 4))], -1).contiguous()
gam, bet, bias = torch.ones(16, device=dev), torch.zeros(16, device=dev), torch.zeros(16, device=dev)
ch = [16] * 6 + [7]
w = torch.randn(16, sum(ch), 3, 3, device=dev, generator=g) / 30
wpk, wrow = ops.pack_conv_weight(w, ch), ops.pack_conv_weight_row(w, ch)
alias = os.environ.get("CONV1_ALIAS", "0") == "1"   # all five up-sampled sources are ONE tensor: 42 MB of inputs, L2 resident
noflush = os.environ.get("CONV1_NOFLUSH", "0") == "1"
up0 = torch.randn_like(x)
srcs = [ops.Source(up0 if alias else torch.randn_like(x)) for _ in range(5)] + [ops.Source(x, L.XFORM_GN_GELU, stats, gam, bet)] + \
       [ops.Source(torch.randn(1, 2, H, W, 4, device=dev, generator=g))]
o, st = torch.empty_like(x), torch.zeros_like(stats)
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
f = lambda: ops.conv_fwd(srcs, wpk, bias, 16, 3, "replicate", impl=impl, wpk_row=wrow, out=o, stats=st)
for _ in range(5):
    f()
torch.cuda.synchronize()
ts = []
for _ in range(30):
    if not noflush:
        flush.zero_()
    else:
        torch.cuda._sleep(400000)  # keeps the GPU busy while the host enqueues the launch (no host gap between the events)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    f()
    b.record()
    b.synchronize()
    ts.append(a.elapsed_time(b) * 1e3)
ts.sort()
print(f"conv[1] {H}x{W} {impl}: median {ts[len(ts) // 2]:.1f} us, best {ts[0]:.1f} us "
      f"({'no flush' if noflush else 'L2 flushed'}{', aliased sources' if alias else ''}, ), checksum {float(o.double().sum()):.6e}", flush=True)
