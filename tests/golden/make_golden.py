#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ FROM THE REAL REFERENCE.

Runs only in the build container (needs /root/reference, CPU only).  It imports the
reference's own modules (`pytorch_networks_convae`, `symmetric_layers_torch`,
`calculate_profiles`) with a matplotlib stub (SURVEY.md section 8c), runs them in float64 (the
reference's native precision, advect_wi_gaia.py:348,430,468), and stores inputs, weights and
outputs as .npz.  The GPU boxes have no /root/reference: the tests there read only the .npz.

    python tests/golden/make_golden.py            # regenerate everything
    python tests/golden/make_golden.py unet       # only the U-Net vectors
    python tests/golden/make_golden.py learned    # only the whole learned-boundary networks
    python tests/golden/make_golden.py fullsize   # 512^2 (config 2) and 4 x 256^2 (config 4) goldens + their noise floors
    python tests/golden/make_golden.py noise      # ref_fp32_noise.json: the reference's own fp32-vs-fp64 distance per case
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, REPO)


def import_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.lines"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib.lines"].Line2D = object
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, REF)
    import pytorch_networks_convae as P  # noqa

    return P


P = import_reference()
from oracle import ref_numpy as RN  # noqa: E402
from tests._util import at, load_unet_case, sample_index  # noqa: E402

RAQ, FKT, FKP = 6.79733173, 475523342.0, 2.58574662  # a CV simulation, load_fluidnet.ipynb:847


def make_net(spec: RN.NetSpec, seed=0, perturb_affine=True, cls=None):
    torch.manual_seed(seed)
    cls = cls or P.NewFluidNet
    net = cls(spec.levels, spec.c_i, spec.c_h, spec.c_o, torch.device("cpu"), act_fn="gelu", r_p=spec.r_p,
              loss_type=spec.loss_type, use_symm=spec.use_symm, dilation=1, a_bound=spec.a_bound,
              repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred, factor=2).double()
    if perturb_affine:  # default init leaves GroupNorm affine = (1, 0): perturb so it is exercised
        g = torch.Generator().manual_seed(seed + 100)
        with torch.no_grad():
            for n, p_ in net.named_parameters():
                if n.endswith("layers.1.weight") or n.startswith("gn.") and n.endswith("weight"):
                    p_.add_(0.2 * torch.randn(p_.shape, generator=g, dtype=p_.dtype))
                elif n.endswith("layers.1.bias") or n.startswith("gn.") and n.endswith("bias") or n.endswith("learnable_bias"):
                    p_.add_(0.2 * torch.randn(p_.shape, generator=g, dtype=p_.dtype))
    net.eval()
    return net


def f32_if_exact(a):
    """Store an array as float32 when that loses nothing (initial weights are float32 values widened by .double());
    tests/_util.load widens it back."""
    if a.dtype == np.float64 and a.size > 64 and np.array_equal(a.astype(np.float32).astype(np.float64), a):
        return a.astype(np.float32)
    return a


def sample_fields(out, names, H, W, n_interior):
    """Keep the full-size fields `names` of `out` only at sample_index(H, W, n_interior), stored as out["idx"]: every
    golden file stays under 1 MB."""
    out["idx"] = idx = sample_index(H, W, n_interior)
    for k in names:
        out[k] = at(out[k], idx)


def set_grid(net, H, W):
    for m in net.unpool:  # pytorch_networks_convae.py:1227-1229 hard-codes (128, 506)
        m.size = (H, W)


def ref_step(net, ad, T, xc, yc, raq, fkt, fkp):
    """Body of TS.forward's loop (pytorch_networks_convae.py:379-473) around the REFERENCE
    modules, minus the hard-coded view(-1,1,128,506) at :414-417."""
    raq_nd, fkt_nd, fkp_nd = RN.nondim_params(raq, fkt, fkp)
    tt = lambda s: torch.tensor(s, dtype=T.dtype)
    V = P.eta_torch(tt(fkt), tt(fkp), 1.0 - yc, T, 0, 0)
    V = torch.clip(V, 1e-08, 1)
    H, W = T.shape[-2:]
    inp = torch.cat((xc / 4.0, yc / 4.0, torch.log10(V) / 8, tt(raq_nd).expand(1, 1, H, W),
                     tt(fkt_nd).expand(1, 1, H, W), tt(fkp_nd).expand(1, 1, H, W), T), axis=1)
    u, v, p = net(inp)
    s = torch.exp((tt(raq) / 10) * 1.80167667 + torch.log(tt(fkt)) * 0.4330392 + torch.log(tt(fkp)) * -0.46052953) * 5
    u = (u * s).view(-1, 1, H, W)
    v = (v * s).view(-1, 1, H, W)
    inp2 = torch.cat((u, v, T, torch.zeros_like(u) + raq, xc, yc), axis=1)
    Tn, dt = ad(inp2)
    Tn[:, :, 0, :] = 1
    Tn[:, :, -1, :] = 0
    Tn[:, :, :, 0:1] = Tn[:, :, :, 1:2]
    Tn[:, :, :, -1:] = Tn[:, :, :, -2:-1]
    return Tn, dt, u, v, p, V, inp


def sd_numpy(net):
    return {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def set_fp32(net):
    net.float()
    net.dx_center_kernel = net.dx_center_kernel.float()
    net.dy_center_kernel = net.dy_center_kernel.float()


@torch.no_grad()
def golden_rollout(tag, spec, H, W, keep, n_steps, check_numpy_steps=1):
    net = make_net(spec)
    set_grid(net, H, W)
    ad = P.ADNet(torch.device("cpu"), CN_max=0.99).double()
    xc_np, yc_np = RN.synthetic_grid(H, W)
    T0_np = RN.synthetic_T0(H, W, seed=1)
    xc = torch.tensor(xc_np).view(1, 1, H, W)
    yc = torch.tensor(yc_np).view(1, 1, H, W)
    T = torch.tensor(T0_np).view(1, 1, H, W)
    out = {"T0": T0_np, "xc": xc_np, "yc": yc_np, "params": np.array([RAQ, FKT, FKP])}
    dts = []
    for i in range(1, n_steps + 1):
        T, dt, u, v, p, V, inp = ref_step(net, ad, T, xc, yc, RAQ, FKT, FKP)
        dts.append(float(dt))
        if i == 1:
            out.update(u1=u[0, 0].numpy().copy(), v1=v[0, 0].numpy().copy(), p1=p[0].numpy().copy(),
                       V1=V[0, 0].numpy().copy())
        if i in keep:
            out[f"T{i}"] = T[0, 0].numpy().copy()
    out["dts"] = np.asarray(dts)
    mT, Tp, dTp = RN.diagnostics(T[0, 0].numpy(), yc_np[:, 0])
    out.update(meanT=np.float64(mT), Tprof=Tp, dTprof=dTp)
    sd = sd_numpy(net)

    # --- pin the numpy oracle against the reference (fp64)
    Tn, dt_n, un, vn, pn, Vn = RN.ts_step(sd, spec, T0_np[None, None], xc_np, yc_np, RAQ, FKT, FKP)
    print(f"[{tag}] numpy-oracle vs reference, step 1: u {relerr(un[0], out['u1']):.2e} v {relerr(vn[0], out['v1']):.2e} "
          f"p {relerr(pn[0], out['p1']):.2e} T {np.abs(Tn[0,0]-out['T1']).max():.2e} dt {abs(dt_n-dts[0])/dts[0]:.2e}")

    # --- fp32 noise floor of the reference itself (SURVEY.md section 8c "parity metric caveat")
    net32 = make_net(spec)
    set_grid(net32, H, W)
    set_fp32(net32)
    inp32 = RN.build_input(T0_np[None, None], xc_np, yc_np, yc_np, RAQ, FKT, FKP)[0].astype(np.float32)
    u32, v32, p32 = net32(torch.tensor(inp32))
    s = RN.velocity_scaler(RAQ, FKT, FKP)
    noise = np.array([relerr(u32[0].numpy() * s, out["u1"]), relerr(v32[0].numpy() * s, out["v1"]),
                      relerr(p32[0].numpy(), out["p1"])])
    print(f"[{tag}] reference fp32 vs its own fp64 (rel-L2 u,v,p): {noise}")
    out["ref_fp32_noise"] = noise
    np.savez_compressed(os.path.join(HERE, f"{tag}.npz"), **out)
    np.savez_compressed(os.path.join(HERE, f"{tag}_weights.npz"), **sd)
    return out


@torch.no_grad()
def golden_ts_unmodified():
    """128x506 through the UNMODIFIED reference TS(ts=5) (pytorch_networks_convae.py:266-475)."""
    spec = RN.NetSpec()
    H, W = 128, 506
    net = make_net(spec)
    ad = P.ADNet(torch.device("cpu"), CN_max=0.99).double()
    ts = P.TS(net, ad, torch.device("cpu"), ts=5, scale=True, p_pred=True, net="newfluidnet").double()
    xc_np, yc_np = RN.synthetic_grid(H, W)
    T0_np = RN.synthetic_T0(H, W, seed=1)
    t64 = lambda s: torch.tensor(s, dtype=torch.float64)
    raq_nd, fkt_nd, fkp_nd = RN.nondim_params(RAQ, FKT, FKP)
    xc = t64(xc_np).view(1, 1, H, W)
    yc = t64(yc_np).view(1, 1, H, W)
    x, dts, u, v, p, V = ts(t64(T0_np).view(1, 1, H, W), None, None, yc, t64(raq_nd), t64(fkt_nd), t64(fkp_nd),
                            t64(RAQ), t64(FKT), t64(FKP), xc, yc)
    out = {"T0_seed": np.int64(1), "params": np.array([RAQ, FKT, FKP]),
           "T1": x[1][0, 0].numpy().copy(), "T5": x[5][0, 0].numpy().copy(),
           "dts": np.array([float(dts[i]) for i in range(1, 6)]),
           "u5": u[0, 0].numpy().copy(), "v5": v[0, 0].numpy().copy(), "p5": p[0, 0].numpy().copy(),
           "V5": V[0, 0].numpy().copy()}
    sd = sd_numpy(net)
    # numpy oracle, 1 step, vs TS
    Tn, dt_n, *_ = RN.ts_step(sd, spec, T0_np[None, None], xc_np, yc_np, RAQ, FKT, FKP)
    print(f"[ts128x506] numpy-oracle vs unmodified TS: T1 {np.abs(Tn[0,0]-out['T1']).max():.2e} dt {abs(dt_n-out['dts'][0])/out['dts'][0]:.2e}")
    sample_fields(out, ["T1", "T5", "u5", "v5", "p5", "V5"], H, W, 15000)
    np.savez_compressed(os.path.join(HERE, "ts128x506.npz"), **out)
    np.savez_compressed(os.path.join(HERE, "ts128x506_weights.npz"), **sd)


@torch.no_grad()
def golden_variants():
    """Small nets covering the other constructor paths: zeros / reflect padding, no
    symmetry, odd sizes (AvgPool floor, non-integer bicubic ratios), mae head, k=5 trunk."""
    cases = {
        "var_zeros_nosym": (RN.NetSpec(levels=3, c_h=8, c_o=2, r_p="zeros", use_symm=False, repeats=2), 36, 52),
        "var_reflect_sym": (RN.NetSpec(levels=3, c_h=16, c_o=2, r_p="reflect", use_symm=True, repeats=2), 50, 76),
        "var_replicate_odd": (RN.NetSpec(levels=4, c_h=16, c_o=2, r_p="replicate", use_symm=True, repeats=2), 50, 77),
        "var_mae_p": (RN.NetSpec(levels=2, c_h=16, c_o=3, r_p="replicate", use_symm=True, repeats=1, loss_type="mae"), 24, 40),
        "var_k5": (RN.NetSpec(levels=2, c_h=16, c_o=1, r_p="zeros", use_symm=True, repeats=2, f=5, p_pred=False), 32, 48),
    }
    for tag, (spec, H, W) in cases.items():
        net = make_net(spec, seed=3)
        set_grid(net, H, W)
        g = torch.Generator().manual_seed(7)
        inp = torch.randn(2, spec.c_i, H, W, generator=g, dtype=torch.float64)
        u, v, p = net(inp)
        sd = sd_numpy(net)
        un, vn, pn = RN.newfluidnet_forward(sd, spec, inp.numpy())
        print(f"[{tag}] numpy-oracle vs reference: u {relerr(un, u.numpy()):.2e} v {relerr(vn, v.numpy()):.2e}"
              + (f" p {relerr(pn, p.numpy()):.2e}" if p is not None else ""))
        out = {"inp": inp.numpy(), "u": u.numpy(), "v": v.numpy(),
               "spec": np.array([spec.levels, spec.c_i, spec.c_h, spec.c_o, spec.repeats, spec.f, int(spec.use_symm), int(spec.p_pred)]),
               "r_p": np.array(spec.r_p), "loss_type": np.array(spec.loss_type), "a_bound": np.float64(spec.a_bound)}
        if p is not None:
            out["p"] = p.numpy()
        out.update({"w::" + k: v_ for k, v_ in sd.items()})
        np.savez_compressed(os.path.join(HERE, f"{tag}.npz"), **out)


@torch.no_grad()
def golden_ops():
    """Operator-level vectors: ADNet alone, BoundaryLearnedConvolution2D (k=3, k=5, symm),
    a FluidLayer, bicubic/avgpool, plus the calc_mlp_profile known answer."""
    g = torch.Generator().manual_seed(11)
    out = {}
    # ADNet with non-uniform grid and mixed-sign velocities (B=2: batch-global dt, :556)
    H, W = 40, 56
    xc_np, yc_np = RN.synthetic_grid(H, W)
    u = torch.randn(2, 1, H, W, generator=g, dtype=torch.float64) * 50
    v = torch.randn(2, 1, H, W, generator=g, dtype=torch.float64) * 50
    u[0, 0, 5, 5] = 0.0
    T = torch.rand(2, 1, H, W, generator=g, dtype=torch.float64)
    ad = P.ADNet(torch.device("cpu"), CN_max=0.99)
    xc = torch.tensor(xc_np).view(1, 1, H, W).expand(2, 1, H, W)
    yc = torch.tensor(yc_np).view(1, 1, H, W).expand(2, 1, H, W)
    inp = torch.cat((u, v, T, torch.zeros_like(u) + 3.5, xc, yc), 1).clone()
    Tn, dt = ad(inp)
    out.update(ad_u=u.numpy(), ad_v=v.numpy(), ad_T=T.numpy(), ad_xc=xc_np, ad_yc=yc_np, ad_raq=np.float64(3.5),
               ad_Tn=Tn.numpy(), ad_dt=np.float64(float(dt)))
    Tn_np, dt_np = RN.adnet_forward(u.numpy()[:, 0], v.numpy()[:, 0], T.numpy()[:, 0], 3.5, xc_np, yc_np, 0.99)
    print(f"[ops] ADNet numpy-oracle vs reference: max abs {np.abs(Tn_np - Tn.numpy()[:,0]).max():.2e}, dt rel {abs(dt_np-float(dt))/float(dt):.2e}")
    Tn2, _ = ad(inp.clone(), dt=torch.tensor(1e-4, dtype=torch.float64))
    out.update(ad_Tn_fixed_dt=Tn2.numpy())

    # learned boundary conv
    for k, symm, ci, co, tag in ((3, False, 5, 8, "blc3"), (5, False, 4, 8, "blc5"), (3, True, 6, 16, "blc3s")):
        torch.manual_seed(5)
        m = P.BoundaryLearnedConvolution2D(ci, co, k, use_symm=symm).double()
        with torch.no_grad():
            m.learnable_bias.add_(torch.randn(m.learnable_bias.shape, generator=g, dtype=torch.float64))
        x = torch.randn(2, ci, 20, 28, generator=g, dtype=torch.float64)
        y = m(x)
        sd = sd_numpy(m)
        yn = RN.boundary_learned_conv(x.numpy(), sd, "", k, co, use_symm=symm)
        print(f"[ops] {tag} numpy-oracle vs reference: {relerr(yn, y.numpy()):.2e}  out shape {tuple(y.shape)}")
        out.update({f"{tag}_x": x.numpy(), f"{tag}_y": y.numpy()})
        out.update({f"{tag}_w::{kk}": vv for kk, vv in sd.items()})
        if k == 3 and not symm:
            y2 = m(x, bc_x=2, bc_y=2)
            out[f"{tag}_y_bc2"] = y2.numpy()
            yn2 = RN.boundary_learned_conv(x.numpy(), sd, "", k, co, use_symm=symm, bc_x=2, bc_y=2)
            print(f"[ops] {tag} bc=2: {relerr(yn2, y2.numpy()):.2e} out shape {tuple(y2.shape)}")

    # bicubic / avgpool
    x = torch.randn(1, 3, 15, 31, generator=g, dtype=torch.float64)
    up = torch.nn.Upsample(size=(50, 77), mode="bicubic")(x)
    pl = torch.nn.AvgPool2d((2, 2), stride=2)(x)
    out.update(bic_x=x.numpy(), bic_y=up.numpy(), pool_y=pl.numpy())
    print(f"[ops] bicubic numpy-oracle vs torch: {np.abs(RN.bicubic_upsample(x.numpy(), (50, 77)) - up.numpy()).max():.2e}; "
          f"avgpool {np.abs(RN.avg_pool2(x.numpy()) - pl.numpy()).max():.2e}")

    # calc_mlp_profile (calculate_profiles.py:102-134) -- needs cwd = reference dir for the pkl
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        import calculate_profiles as CP

        yp, yprof = CP.calc_mlp_profile([RAQ], [FKT], [FKP])
        out.update(mlp_pred=yp, mlp_yprof=yprof)
        print(f"[ops] calc_mlp_profile: first3 {yp[0,:3]} last3 {yp[0,-3:]} mean {yp.mean():.9f}")
    finally:
        os.chdir(cwd)
    np.savez_compressed(os.path.join(HERE, "ops.npz"), **out)


def save_case(tag, spec, inp_seed, inp, outputs, sd):
    """One network case as tests/golden/<tag>.npz.  The input is stored as its seed and shape (tests/_util.load_unet_case
    redraws it), the weights as float32 where that is exact."""
    out = {"inp_seed": np.int64(inp_seed), "inp_shape": np.array(inp.shape, dtype=np.int64)}
    out.update({n: t.numpy() for n, t in outputs if t is not None})
    out["spec"] = np.array([spec.levels, spec.c_i, spec.c_h, spec.c_o, spec.repeats, spec.f, int(spec.use_symm), int(spec.p_pred)])
    out["r_p"], out["loss_type"] = np.array(spec.r_p), np.array(spec.loss_type)
    out["a_bound"] = np.float64(spec.a_bound)
    out.update({"w::" + k: f32_if_exact(v_) for k, v_ in sd.items()})
    np.savez_compressed(os.path.join(HERE, f"{tag}.npz"), **out)


@torch.no_grad()
def golden_unet():
    """The U-Net time-stepper surrogate (pytorch_networks_convae.py:1700-2068; SURVEY.md section 8f N4), small cases
    covering the curl head with and without p, the mae head, k=3 and k=5, three padding modes, odd sizes."""
    cases = {
        "unet_curl_p": (RN.NetSpec(levels=4, c_i=10, c_h=8, c_o=3, r_p="replicate", use_symm=False, repeats=2, f=3), 36, 50),
        "unet_curl_k5": (RN.NetSpec(levels=3, c_i=10, c_h=16, c_o=2, r_p="reflect", use_symm=False, repeats=2, f=5, p_pred=False), 40, 53),
        "unet_mae": (RN.NetSpec(levels=3, c_i=10, c_h=8, c_o=4, r_p="zeros", use_symm=False, repeats=1, f=3, loss_type="mae"), 24, 30),
        # learned-boundary U-Net: the first conv enlarges the width by 3 columns each side itself (bc_x=4, :1994-1996)
        "unet_learned_k3": (RN.NetSpec(levels=3, c_i=10, c_h=8, c_o=3, r_p="learned", use_symm=False, repeats=2, f=3), 36, 50),
        "unet_learned_k5": (RN.NetSpec(levels=3, c_i=10, c_h=8, c_o=2, r_p="learned", use_symm=False, repeats=1, f=5, p_pred=False), 48, 58),
    }
    for tag, (spec, H, W) in cases.items():
        net = make_net(spec, seed=5, cls=lambda *a, factor=2, **k: P.Unet(*a, **k))
        g = torch.Generator().manual_seed(9)
        inp = torch.randn(2, spec.c_i, H, W, generator=g, dtype=torch.float64)
        u, v, p_, T = net(inp)
        sd = sd_numpy(net)
        res = RN.unet_forward(sd, spec, inp.numpy())
        print(f"[{tag}] numpy-oracle vs reference: " + " ".join(
            f"{n} {relerr(a, b.numpy()):.2e}" for n, a, b in zip("uvpT", res, (u, v, p_, T)) if b is not None))
        save_case(tag, spec, 9, inp, zip("uvpT", (u, v, p_, T)), sd)


@torch.no_grad()
def golden_learned():
    """Whole learned-boundary networks (SURVEY.md section 8f N1): NewFluidNet with the 9-region convs (k=5 and k=3) and
    FluidNet (head conv enlarged by bc_x = bc_y = 2, raw curl)."""
    cases = {
        "learned_k5": (P.NewFluidNet, RN.NetSpec(levels=3, c_h=8, c_o=1, r_p="learned", use_symm=False, repeats=2, f=5, p_pred=False), 40, 56),
        "learned_k3_p": (P.NewFluidNet, RN.NetSpec(levels=2, c_h=16, c_o=2, r_p="learned", use_symm=False, repeats=1, f=3), 36, 44),
        "learned_fluidnet": (P.FluidNet, RN.NetSpec(levels=2, c_h=8, c_o=2, r_p="learned", use_symm=False, repeats=2, f=3), 36, 44),
    }
    for tag, (cls, spec, H, W) in cases.items():
        net = make_net(spec, seed=6, cls=cls)
        set_grid(net, H, W)
        g = torch.Generator().manual_seed(10)
        inp = torch.randn(2, spec.c_i, H, W, generator=g, dtype=torch.float64)
        u, v, p_ = net(inp)
        sd = sd_numpy(net)
        res = RN.learned_net_forward(sd, spec, inp.numpy(), fluidnet=cls is P.FluidNet)
        print(f"[{tag}] numpy-oracle vs reference: " + " ".join(
            f"{n} {relerr(a, b.numpy()):.2e}" for n, a, b in zip("uvp", res, (u, v, p_)) if b is not None))
        save_case(tag, spec, 10, inp, zip("uvp", (u, v, p_)), sd)



# ------------------------------------------------------------------------------------------------------------------
# Noise floors of the reference itself (its float32 run against its float64 run) for EVERY golden case, and the
# full-size goldens of BASELINE configs 2 and 4.  The parity bound of the GPU tests is, per field,
#     rel_L2(new_fp32, ref_fp64) <= max(1e-5, 1.5 * rel_L2(ref_fp32, ref_fp64))          (SURVEY.md section 8c)
# so each case needs its own stored noise: tests/golden/ref_fp32_noise.json.
import contextlib  # noqa: E402
import json  # noqa: E402

_FD_KERNELS = ("dx_right_kernel", "dy_bottom_kernel", "dx_left_kernel", "dy_top_kernel", "dx_center_kernel", "dy_center_kernel")


@contextlib.contextmanager
def reference_fp32():
    """The reference's module-level FD stencils are float64 constants (pytorch_networks_convae.py:183-256): swap them
    for float32 copies while a float32 ADNet runs (SURVEY.md section 8c "fp32 oracle")."""
    saved = {k: getattr(P, k) for k in _FD_KERNELS}
    try:
        for k in _FD_KERNELS:
            setattr(P, k, saved[k].float())
        yield
    finally:
        for k, v in saved.items():
            setattr(P, k, v)


def _rollout_ref(net, T0_np, xc_np, yc_np, params, n_steps, dtype):
    H, W = T0_np.shape
    ad = P.ADNet(torch.device("cpu"), CN_max=0.99)
    xc = torch.tensor(xc_np, dtype=dtype).view(1, 1, H, W)
    yc = torch.tensor(yc_np, dtype=dtype).view(1, 1, H, W)
    T = torch.tensor(T0_np, dtype=dtype).view(1, 1, H, W)
    hist = []
    for _ in range(n_steps):
        T, dt, u, v, p, V, _inp = ref_step(net, ad, T, xc.clone(), yc.clone(), *params)
        hist.append(dict(T=T[0, 0].double().numpy().copy(), dt=float(dt), u=u[0, 0].double().numpy().copy(),
                         v=v[0, 0].double().numpy().copy(), p=None if p is None else p[0].double().numpy().copy(),
                         V=V[0, 0].double().numpy().copy()))
    return hist


def _rollout_noise(spec, H, W, params, n_steps, T0_np, cls=None):
    """(fp64 history, fp32 history) of the reference on one case."""
    xc_np, yc_np = RN.synthetic_grid(H, W)
    net64 = make_net(spec, cls=cls)
    set_grid(net64, H, W)
    h64 = _rollout_ref(net64, T0_np, xc_np, yc_np, params, n_steps, torch.float64)
    net32 = make_net(spec, cls=cls)
    set_grid(net32, H, W)
    set_fp32(net32)
    with reference_fp32():
        h32 = _rollout_ref(net32, T0_np, xc_np, yc_np, params, n_steps, torch.float32)
    return h64, h32, net64


def _field_noise(h64, h32, i):
    a, b = h64[i], h32[i]
    out = {"u": relerr(b["u"], a["u"]), "v": relerr(b["v"], a["v"])}
    if a["p"] is not None:
        out["p"] = relerr(b["p"], a["p"])
    out["T_maxabs"] = float(np.abs(b["T"] - a["T"]).max())
    out["V_maxabs"] = float(np.abs(b["V"] - a["V"]).max())
    out["dt_rel"] = abs(b["dt"] - a["dt"]) / a["dt"]
    return out


@torch.no_grad()
def golden_noise():
    """ref_fp32_noise.json: for every network-level golden case, how far the reference's own float32 run is from its
    float64 run -- rel-L2 per output field, max-abs for T after the stored step counts."""
    noise = {}
    # forward-only cases: variants, learned networks, U-Net
    for tag in ("var_zeros_nosym", "var_reflect_sym", "var_replicate_odd", "var_mae_p", "var_k5"):
        g = dict(np.load(os.path.join(HERE, tag + ".npz")))
        s = g["spec"]
        spec = RN.NetSpec(levels=int(s[0]), c_i=int(s[1]), c_h=int(s[2]), c_o=int(s[3]), repeats=int(s[4]), f=int(s[5]),
                          use_symm=bool(s[6]), p_pred=bool(s[7]), r_p=str(g["r_p"]), loss_type=str(g["loss_type"]),
                          a_bound=float(g["a_bound"]))
        H, W = g["inp"].shape[-2:]
        net = make_net(spec, seed=3)
        set_grid(net, H, W)
        set_fp32(net)
        res = net(torch.tensor(g["inp"], dtype=torch.float32))
        noise[tag] = {n: relerr(r.double().numpy(), g[n]) for n, r in zip("uvp", res) if r is not None}
    for file, cases, seed in (("learned", {"learned_k5": P.NewFluidNet, "learned_k3_p": P.NewFluidNet, "learned_fluidnet": P.FluidNet}, 6),
                              ("unet", {"unet_curl_p": None, "unet_curl_k5": None, "unet_mae": None, "unet_learned_k3": None, "unet_learned_k5": None}, 5)):
        for tag, cls in cases.items():
            spec, inp, d, _w = load_unet_case(tag)
            H, W = inp.shape[-2:]
            if file == "unet":
                net = make_net(spec, seed=seed, cls=lambda *a, factor=2, **k: P.Unet(*a, **k))
                net.float()
                for attr in ("dx_center_kernel", "dy_center_kernel"):
                    if hasattr(net, attr):
                        setattr(net, attr, getattr(net, attr).float())
            else:
                net = make_net(spec, seed=seed, cls=cls)
                set_grid(net, H, W)
                set_fp32(net)
            res = net(torch.tensor(inp, dtype=torch.float32))
            noise[tag] = {n: relerr(r.double().numpy(), d[n]) for n, r in zip("uvpT", res) if r is not None and n in d}
    # rollouts: 128^2 (1 / 10 / 100 steps), 64x96 (1 / 10), 128x506 through the unmodified TS (5 steps)
    for tag, spec, H, W, keep in (("roll128", RN.NetSpec(), 128, 128, (1, 10, 100)), ("roll64x96", RN.NetSpec(levels=4), 64, 96, (1, 10)),
                                  ("ts128x506", RN.NetSpec(), 128, 506, (1, 5))):
        h64, h32, _ = _rollout_noise(spec, H, W, (RAQ, FKT, FKP), max(keep), RN.synthetic_T0(H, W, seed=1))
        g = dict(np.load(os.path.join(HERE, tag + ".npz")))
        T1 = at(h64[0]["T"], g["idx"]) if "idx" in g else h64[0]["T"]
        assert np.abs(T1 - g["T1"]).max() == 0.0, "noise run does not reproduce the stored golden"
        noise[tag] = {f"step{i}": _field_noise(h64, h32, i - 1) for i in keep}
        mT64, Tp64, dTp64 = RN.diagnostics(h64[-1]["T"], RN.synthetic_grid(H, W)[1][:, 0])
        mT32, Tp32, dTp32 = RN.diagnostics(h32[-1]["T"], RN.synthetic_grid(H, W)[1][:, 0])
        noise[tag]["diag_last"] = {"meanT": abs(mT64 - mT32), "Tprof_maxabs": float(np.abs(Tp64 - Tp32).max()),
                                   "dTprof_rel": float(np.abs(dTp64 - dTp32).max() / np.abs(dTp64).max())}
        print(f"[noise] {tag}: {noise[tag]}")
    path = os.path.join(HERE, "ref_fp32_noise.json")
    old = json.load(open(path)) if os.path.exists(path) else {}
    old.update(noise)
    json.dump(old, open(path, "w"), indent=1, sort_keys=True)
    for k, v in noise.items():
        print(k, v)


ENS256_PARAMS = [(RAQ, FKT, FKP), (0.9, 3.0e6, 1.5), (9.1, 5.0e9, 60.0), (4.2, 2.5e8, 12.0)]  # spread over the paper's ranges


@torch.no_grad()
def golden_full_size():
    """BASELINE config 2 (512x512, batch 1): fields of the first forward + T after 3 steps; config 4 (256x256 ensemble):
    4 members with different (RaQ, gamma, beta, T0 seed), each a B = 1 run of the reference (SURVEY.md section 8c
    "Ensembles"), fields and T after 3 steps.  float64, weights = roll128_weights.npz (same spec and seed)."""
    noise = {}
    spec = RN.NetSpec()
    H = W = 512
    T0 = RN.synthetic_T0(H, W, seed=1)
    h64, h32, net = _rollout_noise(spec, H, W, (RAQ, FKT, FKP), 3, T0)
    w128 = dict(np.load(os.path.join(HERE, "roll128_weights.npz")))
    sd = sd_numpy(net)
    assert all(np.array_equal(sd[k], w128[k]) for k in sd), "roll512 must share roll128's weights"
    out = {"params": np.array([RAQ, FKT, FKP]), "T0_seed": np.int64(1), "u1": h64[0]["u"], "v1": h64[0]["v"], "p1": h64[0]["p"],
           "T1": h64[0]["T"], "T3": h64[2]["T"], "dts": np.array([h["dt"] for h in h64])}
    sample_fields(out, ["u1", "v1", "p1", "T1", "T3"], H, W, 18000)
    np.savez_compressed(os.path.join(HERE, "roll512.npz"), **out)
    noise["roll512"] = {"step1": _field_noise(h64, h32, 0), "step3": _field_noise(h64, h32, 2)}
    print("[roll512]", noise["roll512"])
    H = W = 256
    out = {"params": np.array(ENS256_PARAMS), "T0_seeds": np.arange(1, 5)}
    noise["ens256"] = {}
    for m, prm in enumerate(ENS256_PARAMS):
        h64, h32, _ = _rollout_noise(spec, H, W, prm, 3, RN.synthetic_T0(H, W, seed=1 + m))
        out.update({f"m{m}_u3": h64[2]["u"], f"m{m}_v3": h64[2]["v"], f"m{m}_p3": h64[2]["p"], f"m{m}_T3": h64[2]["T"],
                    f"m{m}_dts": np.array([h["dt"] for h in h64])})
        noise["ens256"][f"m{m}"] = _field_noise(h64, h32, 2)
        print(f"[ens256 m{m}]", noise["ens256"][f"m{m}"])
    sample_fields(out, [f"m{m}_{n}3" for m in range(len(ENS256_PARAMS)) for n in "uvpT"], H, W, 5400)
    np.savez_compressed(os.path.join(HERE, "ens256.npz"), **out)
    path = os.path.join(HERE, "ref_fp32_noise.json")
    old = json.load(open(path)) if os.path.exists(path) else {}
    old.update(noise)
    json.dump(old, open(path, "w"), indent=1, sort_keys=True)

if __name__ == "__main__" and sys.argv[1:] == ["noise"]:
    torch.set_num_threads(os.cpu_count())
    golden_noise()
    sys.exit(0)

if __name__ == "__main__" and sys.argv[1:] == ["fullsize"]:
    torch.set_num_threads(os.cpu_count())
    golden_full_size()
    sys.exit(0)

if __name__ == "__main__" and sys.argv[1:] == ["learned"]:
    torch.set_num_threads(os.cpu_count())
    golden_learned()
    sys.exit(0)

if __name__ == "__main__" and sys.argv[1:] == ["unet"]:
    torch.set_num_threads(os.cpu_count())
    golden_unet()
    sys.exit(0)

if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count())
    golden_ops()
    golden_unet()
    golden_learned()
    golden_variants()
    golden_rollout("roll128", RN.NetSpec(), 128, 128, keep=(1, 10, 100), n_steps=100)
    golden_rollout("roll64x96", RN.NetSpec(levels=4), 64, 96, keep=(1, 10), n_steps=10)
    golden_ts_unmodified()
    golden_full_size()
    golden_noise()


def golden_mlp_weights():
    """The reference's MLP asset (numpy arrays only) re-saved as .npz so calc_mlp_profile can be
    checked on machines without /root/reference."""
    import pickle

    mlp = pickle.load(open(os.path.join(REF, "mlp_[128, 128, 128, 128, 128].pkl"), "rb"))
    out = {}
    for i, (W, b) in enumerate(mlp):
        out[f"W{i}"], out[f"b{i}"] = np.asarray(W), np.asarray(b)
    np.savez_compressed(os.path.join(HERE, "mlp_profile_weights.npz"), **out)


if __name__ == "__main__":
    golden_mlp_weights()
