"""`net(x)` of a learned-boundary NewFluidNet (r_p="learned") is the fused engine's forward wherever the engine plans the
shape: the same bits as `net._engine(dev).forward_blocked`, eagerly and replayed as a CUDA graph, with `net.conv_impl`
honoured.  The shapes the engine refuses take the module-level composition, held to the float64 oracle."""
import numpy as np
import pytest
import torch

from oracle import ref_numpy as RN
from pbml_mantle_convection_b200 import engine, ops
from tests._util import field_bound, relerr
from tests.test_gpu_learned_rollout import DEV, _case, _net, _sd

pytestmark = pytest.mark.gpu


def _engine_forward(net, x):
    u, v, p, _ = net._engine(torch.device(DEV)).forward_blocked(ops.pack_nchw(x))
    return u, v, p


def _assert_same_bits(out, ref):
    assert (out[2] is None) == (ref[2] is None)
    for a, b in zip(out, ref):
        if b is not None:
            assert a.dtype == torch.float64 and torch.equal(a.float(), b)


@pytest.mark.parametrize("tag", ["learned_k5", "learned_k3_p", "paper"])
def test_forward_is_the_engine(tag):
    net, inp = _case(tag)[:2]
    x = torch.tensor(inp, device=DEV)
    ref = _engine_forward(net, x)
    for call in range(3):  # eager, capture + replay, replay
        _assert_same_bits(net(x), ref)
    assert net.__dict__["_learned_plan"].graph is not None


def test_forward_honours_conv_impl():
    """A replayed graph of one conv_impl is not reused for another."""
    net, inp = _case("paper")[:2]
    x = torch.tensor(inp, device=DEV)
    auto = [net(x) for _ in range(3)]
    net.conv_impl = "ffma"
    ref = _engine_forward(net, x)
    assert net._engine(torch.device(DEV)).conv_impl == "ffma"
    for call in range(3):
        out = net(x)
        _assert_same_bits(out, ref)
        assert not torch.equal(out[0], auto[call][0])


def test_refused_shape_takes_the_module_composition():
    """32 hidden channels (one ring-kernel tile holds 16 output channels): the module-level composition, against the float64
    oracle under the bound of the oracle's own float32 run on the same case."""
    spec = RN.NetSpec(levels=2, c_i=7, c_h=32, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0,
                      repeats=1, f=5, p_pred=False)
    net = _net(spec, seed=5)
    inp = np.random.default_rng(5).standard_normal((1, 7, 40, 56))
    assert not engine.fused_supported(net, 1, 40, 56)
    sd = _sd(net)
    u64, v64, _ = RN.learned_net_forward(sd, spec, inp)
    u32, v32, _ = RN.learned_net_forward({n: np.asarray(a, np.float32) for n, a in sd.items()}, spec, inp.astype(np.float32))
    noise = {"u": relerr(u32, u64), "v": relerr(v32, v64)}
    x = torch.tensor(inp, device=DEV)
    for call in range(3):
        u, v, p = net(x)
        assert p is None
        errs = {"u": relerr(u.cpu().numpy(), u64), "v": relerr(v.cpu().numpy(), v64)}
        print(f"[c_h = 32 call {call}] rel-L2 {errs}; oracle fp32 noise {noise}")
        for n in errs:
            assert errs[n] <= field_bound(noise[n]), (call, n, errs[n], noise[n])
