"""Host-side planning of the fused engine for learned-boundary networks (pbmc_net.flags & PBMC_NET_LEARNED): which shapes
it takes and how it schedules them.  Dummy (never dereferenced) weight pointers, as in test_capi_cpu.py: no GPU needed."""
import ctypes as C

import pytest

from pbml_mantle_convection_b200 import _lib as L


# pbmc_workspace_bytes of the primary configuration (levels=6, repeats=4, c_h=16, k=3), B = 1, as planned before learned
# networks were added to the engine
WS_PRIMARY_512 = 197445376
WS_PRIMARY_128x506 = 49025536


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G

    G.build()
    return L.load()


def _net(levels=5, repeats=6, c_i=7, c_h=16, c_o=1, k=5, learned=True, wedges=True):
    """pbmc_net of the paper's learned-boundary network (levels=5, repeats=6, f=5, c_o=1) by default."""
    n = L.Net()
    n.levels, n.repeats, n.c_i, n.c_h, n.c_o, n.ksize = levels, repeats, c_i, c_h, c_o, k
    n.pad_mode, n.head_kind, n.p_pred, n.conv_impl = 0, L.HEAD_CURL, 0, L.CONV_IMPL["auto"]
    n.flags = L.NET_LEARNED if learned else 0

    def lay(cin_blks, cout):
        x = L.Layer()
        x.wpk = x.wpk_row = x.bias = x.gamma = x.beta = 16
        x.cin_blks, x.cout, x.ksize = cin_blks, cout, k
        return x

    cib, cb = (c_i + 3) // 4, c_h // 4
    n.conv0 = lay(cib, c_h)
    for l in range(levels):
        for r in range(repeats):
            n.trunk[l * L.MAX_REPEATS + r] = lay(cb, c_h)
            if wedges:
                n.wedge_trunk[l * L.MAX_REPEATS + r] = 32
    n.conv1, n.conv2, n.conv3 = lay(cb * levels + cib, c_h), lay(cb, c_h), lay(cb, c_o)
    if wedges:
        n.wedge_conv0 = n.wedge_conv1 = n.wedge_conv2 = n.wedge_conv3 = 32
    return n


def _budgets(lib, n, B, H, W):
    b = (C.c_int * L.MAX_LEVELS)()
    rc = lib.pbmc_trunk_cta_budgets(C.byref(n), B, H, W, b)
    return rc, list(b)


def test_net_mirror_matches_the_library(lib):
    assert lib.pbmc_sizeof(b"pbmc_net") == C.sizeof(L.Net)
    # the edge-filter pointers come after every field an existing caller sets
    assert L.Net.wedge_conv0.offset == L.Net.conv3.offset + C.sizeof(L.Layer)


def test_paper_network_is_planned_per_layer(lib):
    n = _net()
    assert lib.pbmc_workspace_bytes(C.byref(n), 1, 128, 506) > 0
    rc, bud = _budgets(lib, n, 1, 128, 506)
    assert rc == 0  # never the persistent trunk kernel: it would read GroupNorm sums before the ring kernel repairs them
    assert all(x > 0 for x in bud[:5]) and sum(bud) <= 148, bud
    # k = 3 / c_h = 16 is the persistent kernel's shape: still one launch per layer when the convs are learned
    n3 = _net(levels=6, repeats=4, c_o=2, k=3)
    assert _budgets(lib, n3, 1, 512, 512)[0] == 0
    assert _budgets(lib, _net(levels=6, repeats=4, c_o=2, k=3, learned=False), 1, 512, 512)[0] == 1


def test_unsupported_learned_shapes_are_refused(lib):
    # coarsest level of 64 x 506 over 5 levels: 4 rows, shorter than the k = 5 strip (6 rows)
    assert lib.pbmc_workspace_bytes(C.byref(_net()), 1, 64, 506) == 0
    assert lib.pbmc_trunk_cta_budgets(C.byref(_net()), 1, 64, 506, (C.c_int * L.MAX_LEVELS)()) == -2
    assert lib.pbmc_workspace_bytes(C.byref(_net()), 1, 96, 506) > 0  # coarsest level 6 rows: exactly the strip
    assert lib.pbmc_workspace_bytes(C.byref(_net(k=3)), 1, 48, 506) > 0  # k = 3 strip: 3 rows
    assert lib.pbmc_workspace_bytes(C.byref(_net(k=3)), 1, 32, 506) == 0
    # the same shapes without learned boundaries are fine
    assert lib.pbmc_workspace_bytes(C.byref(_net(learned=False)), 1, 64, 506) > 0
    # the ring kernel's limits: one 16-wide c_out tile, a 4-channel head
    assert lib.pbmc_workspace_bytes(C.byref(_net(c_h=32)), 1, 128, 506) == 0
    assert lib.pbmc_workspace_bytes(C.byref(_net(c_o=5)), 1, 128, 506) == 0


def test_descriptor_without_the_flag_is_planned_as_before(lib):
    """The edge-filter fields are read only with PBMC_NET_LEARNED: a non-learned descriptor plans the same workspace and
    budgets whether they are set or zero (as an existing caller's zero-initialised descriptor has them)."""
    for (levels, repeats, k, B, H, W) in [(6, 4, 3, 1, 512, 512), (5, 6, 5, 1, 128, 506), (6, 4, 3, 32, 256, 256)]:
        a = _net(levels, repeats, k=k, learned=False, wedges=False)
        b = _net(levels, repeats, k=k, learned=False, wedges=True)
        assert lib.pbmc_workspace_bytes(C.byref(a), B, H, W) == lib.pbmc_workspace_bytes(C.byref(b), B, H, W) > 0
        assert _budgets(lib, a, B, H, W) == _budgets(lib, b, B, H, W)
    # values of the planner before learned networks existed (primary configuration, 512^2 and 128x506)
    prim = _net(6, 4, c_o=2, k=3, learned=False, wedges=False)
    assert lib.pbmc_workspace_bytes(C.byref(prim), 1, 512, 512) == WS_PRIMARY_512
    assert lib.pbmc_workspace_bytes(C.byref(prim), 1, 128, 506) == WS_PRIMARY_128x506
    assert _budgets(lib, prim, 1, 512, 512) == (1, [96, 30, 10, 5, 4, 2, 0, 0])


def test_learned_flag_keeps_the_workspace_layout(lib):
    """Learned nets use the same buffers (the ring kernel writes in place into each conv's output)."""
    a, b = _net(learned=False), _net(learned=True)
    assert lib.pbmc_workspace_bytes(C.byref(a), 2, 128, 506) == lib.pbmc_workspace_bytes(C.byref(b), 2, 128, 506)


def test_python_support_query_and_slab_refusal(lib):
    """TS routes a learned NewFluidNet to the fused rollout exactly where the engine plans it; the slab-decomposed
    surrogate refuses learned nets with its own error."""
    import pbml_mantle_convection_b200 as P
    from pbml_mantle_convection_b200 import engine
    from pbml_mantle_convection_b200.slab_surrogate import SlabSurrogate

    net = P.NewFluidNet(5, 7, 16, 1, "cpu", act_fn="gelu", r_p="learned", loss_type="curl", use_symm=False, a_bound=10,
                        repeats=6, f=5, p_pred=False)
    d = engine.shape_desc(net)
    assert d.flags == L.NET_LEARNED and d.ksize == 5 and (d.levels, d.repeats, d.c_h, d.c_o) == (5, 6, 16, 1)
    assert engine.fused_supported(net, 1, 128, 506) and engine.fused_supported(net, 32, 256, 256)
    assert not engine.fused_supported(net, 1, 64, 506)
    with pytest.raises(NotImplementedError, match="learned"):
        SlabSurrogate(net, 128, 506, None, None, (1.0, 1.0, 1.0), None, "cpu")


def test_learned_forward_dispatch(lib, monkeypatch):
    """A learned NewFluidNet's forward runs on the fused engine wherever the engine plans its shape; the shapes it refuses
    and FluidNet (whose enlarged head has no engine form) take the module-level composition.  The engine is stubbed (its
    context needs a GPU); the support query is the library's, asked once per (B, H, W)."""
    import torch

    import pbml_mantle_convection_b200 as P
    from pbml_mantle_convection_b200 import engine, ops
    from pbml_mantle_convection_b200 import pytorch_networks_convae as M
    from tests._util import load_learned_case

    reached, queries = [], []

    class StubEngine:
        def forward_blocked(self, inp):
            reached.append("engine")
            B, _, H, W, _ = inp.shape
            return torch.zeros(B, H, W), torch.zeros(B, H, W), None, None

    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    cpu_device = torch.Tensor.device
    monkeypatch.setattr(torch.Tensor, "device", property(lambda self: torch.device("cuda:0")))
    monkeypatch.setattr(ops, "pack_nchw", lambda x: x[..., None])
    monkeypatch.setattr(M, "_forward_learned_modules",
                        lambda net, x, head_bc, wall_bcs: reached.append(("modules", head_bc, wall_bcs)))
    monkeypatch.setattr(M, "fused_supported", lambda m, B, H, W: queries.append((B, H, W)) or engine.fused_supported(m, B, H, W))

    def mk(spec, cls=P.NewFluidNet):
        net = cls(spec.levels, spec.c_i, spec.c_h, spec.c_o, "cpu", act_fn="gelu", r_p="learned", loss_type="curl",
                  use_symm=False, a_bound=spec.a_bound, repeats=spec.repeats, f=spec.f, p_pred=spec.p_pred).eval()
        monkeypatch.setattr(net, "_engine", lambda dev: StubEngine())
        net.use_cuda_graph = False
        return net

    def route(net, B, H, W):
        reached.clear()
        net(torch.zeros(B, net.c_i, H, W))
        assert len(reached) == 1
        return reached[0]

    from oracle import ref_numpy as RN

    paper = mk(RN.NetSpec(levels=5, c_i=7, c_h=16, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0,
                          repeats=6, f=5, p_pred=False))
    assert route(paper, 1, 128, 506) == "engine" and route(paper, 1, 128, 506) == "engine"
    assert queries == [(1, 128, 506)]
    assert route(paper, 2, 128, 506) == "engine" and queries == [(1, 128, 506), (2, 128, 506)]
    assert route(paper, 1, 64, 506) == ("modules", 1, True)  # coarsest level shorter than the k = 5 strip
    with monkeypatch.context() as mp:  # the engine runs on CUDA devices only
        mp.setattr(torch.Tensor, "device", cpu_device)
        assert route(paper, 1, 128, 506) == ("modules", 1, True)

    k5 = mk(load_learned_case("learned_k5")[0])  # 3 levels, k = 5
    assert route(k5, 2, 40, 56) == "engine"
    assert route(k5, 1, 20, 28) == ("modules", 1, True)  # coarsest level 5 x 7: shorter than the 6-row strip
    wide = mk(RN.NetSpec(levels=2, c_i=7, c_h=32, c_o=1, r_p="learned", loss_type="curl", use_symm=False, a_bound=10.0,
                         repeats=1, f=5, p_pred=False))
    assert route(wide, 1, 40, 56) == ("modules", 1, True)  # one ring-kernel tile holds 16 output channels

    fluid = mk(load_learned_case("learned_fluidnet")[0], P.FluidNet)
    assert engine.fused_supported(fluid, 2, 36, 44)  # the engine would plan the shape ...
    assert route(fluid, 2, 36, 44) == ("modules", 2, False)  # ... but FluidNet's head is enlarged
