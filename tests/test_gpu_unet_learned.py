"""Network-level parity of the rows SURVEY.md section 8f calls N1 and N4: whole learned-boundary networks and the U-Net
drop-in against the vectors of the real reference (tests/golden/learned_*.npz, unet_*.npz), and the `net="unet"` branch of
TS.  Bound per field: max(1e-5, 1.5 x the reference's own fp32-vs-fp64 distance on the same case)
(tests/golden/ref_fp32_noise.json).  Their host logic is also covered on the CPU (tests/test_host_logic_cpu.py)."""
import numpy as np
import pytest
import torch

import pbml_mantle_convection_b200 as P
from oracle import ref_numpy as RN
from tests._util import LEARNED_CASES, UNET_CASES, field_bound, load_learned_case, load_unet_case, noise, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _net(spec, w):
    net = P.Unet(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p=spec.r_p, loss_type=spec.loss_type,
                 use_symm=False, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({k: torch.tensor(v) for k, v in w.items()})
    return net.to(DEV).eval()


@pytest.mark.parametrize("tag", UNET_CASES)
def test_unet_forward_against_reference_golden(tag):
    spec, inp, outs, w = load_unet_case(tag)
    res = dict(zip("uvpT", _net(spec, w)(torch.tensor(inp, device=DEV))))
    assert (res["p"] is None) == ("p" not in outs)
    nz = noise(tag)
    errs = {n: relerr(res[n].cpu().numpy(), ref) for n, ref in outs.items()}
    print(f"[{tag}] rel-L2 vs reference fp64: {errs}; reference fp32 noise: {nz}")
    for n, ref in outs.items():
        assert tuple(res[n].shape) == ref.shape and res[n].dtype == torch.float64
        # fp32 kernels against the float64 reference; the reference's own fp32 run is 0.6e-6 .. 1.8e-6 away on these
        # (random, non-smooth) inputs, so the curl does not amplify anything here and the bound is north_star's 1e-5
        assert errs[n] <= field_bound(nz[n]), (n, errs[n])


def test_TS_unet_branch():
    spec, _inp, _outs, w = load_unet_case("unet_curl_p")
    net = _net(spec, w)
    H, W = 36, 50
    xc, yc = RN.synthetic_grid(H, W)
    T0 = RN.synthetic_T0(H, W, seed=1)
    raq, fkt, fkp = 6.79733173, 475523342.0, 2.58574662
    nd = RN.nondim_params(raq, fkt, fkp)
    t64 = lambda a: torch.tensor(a, dtype=torch.float64)
    g = torch.Generator().manual_seed(3)
    up, vp = torch.randn(1, 1, H, W, generator=g, dtype=torch.float64), torch.randn(1, 1, H, W, generator=g, dtype=torch.float64)
    dt = torch.full((1, 1, H, W), 1e-3, dtype=torch.float64)
    ts = P.TS(net, None, DEV, ts=2, scale=True, p_pred=True, net="unet")
    grid = lambda a: t64(a).view(1, 1, H, W)
    x, dts, u, v, p, V = ts(grid(T0), None, None, grid(yc), t64(nd[0]), t64(nd[1]), t64(nd[2]), t64(raq), t64(fkt), t64(fkp),
                            grid(xc), grid(yc), u_prev=up, v_prev=vp, dt=dt)
    assert sorted(x) == [0, 1, 2] and dts == {} and p is None
    for i in (1, 2):
        Ti = x[i]
        assert tuple(Ti.shape) == (1, 1, H, W) and Ti.dtype == torch.float64 and torch.isfinite(Ti).all()
        assert (Ti[:, :, 0] == 1).all() and (Ti[:, :, -1] == 0).all()
        assert torch.equal(Ti[..., 0], Ti[..., 1]) and torch.equal(Ti[..., -1], Ti[..., -2])
    # step 1 is the network applied to the reference's 10-channel input (:419-451)
    inp7 = RN.build_input(T0[None, None], xc, yc, yc, raq, fkt, fkp)
    inp7 = inp7[0] if isinstance(inp7, tuple) else inp7
    inp = np.concatenate([inp7[:, 0:2], dt.numpy(), inp7[:, 3:6], inp7[:, 2:3], inp7[:, 6:7], up.numpy(), vp.numpy()], 1)
    u1, v1, _p1, T1 = RN.unet_forward(w, spec, inp)
    T1 = RN.apply_T_bcs(T1[:, None].copy()) if T1.ndim == 3 else T1
    assert np.abs(x[1].cpu().numpy() - T1.reshape(1, 1, H, W)).max() < 1e-5  # T is O(1): north_star's 1e-5
    assert tuple(u.shape) == (1, 1, H, W) and tuple(V.shape) == (1, 1, H, W)


@pytest.mark.parametrize("tag", LEARNED_CASES)
def test_learned_network_against_reference_golden(tag):
    """N1 at network level (until now: runs, finite, first layer == oracle): eager call, then the replayed graph."""
    spec, inp, outs, w = load_learned_case(tag)
    cls = P.FluidNet if tag == "learned_fluidnet" else P.NewFluidNet
    net = cls(spec.levels, spec.c_i, spec.c_h, spec.c_o, DEV, act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False,
              a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).double()
    net.load_state_dict({k: torch.tensor(v) for k, v in w.items()})
    net = net.to(DEV).eval()
    x = torch.tensor(inp, device=DEV)
    nz = noise(tag)
    for call in range(3):  # eager, capture + replay, replay
        res = dict(zip("uvp", net(x)))
        assert (res["p"] is None) == ("p" not in outs)
        errs = {n: relerr(res[n].cpu().numpy(), ref) for n, ref in outs.items()}
        print(f"[{tag} call {call}] rel-L2 vs reference fp64: {errs}; reference fp32 noise: {nz}")
        for n, ref in outs.items():
            assert tuple(res[n].shape) == ref.shape
            assert errs[n] <= field_bound(nz[n]), (call, n, errs[n])  # the reference's own fp32 run: 5e-7 .. 8e-7
