"""Drop-in `SymmetricConv2d` (reference: symmetric_layers_torch.py:21-138).

Same constructor, same parameters (`weight` holds only the UNIQUE filters, `bias` has
out_channels entries), hence the same `state_dict` keys/shapes; `forward` runs the sm_100a
conv kernel through the C ABI.  The mirrored filters are materialised when weights are packed,
not on every call as the reference does (`torch.flip` + `cat`, :118-138).
"""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.nn.parameter import Parameter

from . import _lib as L
from . import ops


def _check_conv_supported(m: nn.Conv2d):
    if m.stride != (1, 1) or m.dilation != (1, 1) or m.groups != 1:
        raise NotImplementedError("the B200 conv path implements stride=1, dilation=1, groups=1 (all the rollout uses)")
    k = m.kernel_size
    if k[0] != k[1] or k[0] not in (3, 5):
        raise NotImplementedError("the B200 conv path implements 3x3 and 5x5 kernels")
    if m.padding_mode not in ("zeros", "replicate", "reflect"):
        raise NotImplementedError(f"padding_mode={m.padding_mode!r} is not implemented on the B200 path")


def full_weight(m: nn.Conv2d) -> torch.Tensor:
    """Full [out, in, k, k] filter bank of a conv module (mirrors expanded for SymmetricConv2d)."""
    w = m.weight
    sym = getattr(m, "symmetry", None)
    if sym is None:
        return w
    out = [w]
    ix = 0
    if sym["h"] > 0:
        out.append(torch.flip(w[ix:ix + sym["h"] // 2], (3,)))
        ix += sym["h"] // 2
    if sym["v"] > 0:
        out.append(torch.flip(w[ix:ix + sym["v"] // 2], (2,)))
        ix += sym["v"] // 2
    if sym["hv"] > 0:
        n = sym["hv"] // 4
        out += [torch.flip(w[ix:ix + n], (3,)), torch.flip(w[ix:ix + n], (2,)), torch.flip(w[ix:ix + n], (2, 3))]
    return torch.cat(out, 0)


TENSOR_CORE_MIN_SIDE = 32  # below this a CTA's 128-column strip is mostly padding: the FFMA kernel is used


def _packed_filters(m: nn.Conv2d, dev, want_row: bool):
    """Packed filter images + padded bias of a conv module, cached on the module and rebuilt when the parameters
    change (in-place updates bump `_version`; `.to()` / `load_state_dict(assign=True)` change the storage)."""
    w, b = m.weight, m.bias
    key = (w.data_ptr(), w._version, None if b is None else (b.data_ptr(), b._version), str(dev))
    c = m.__dict__.get("_pbmc_pack")
    if c is None or c["key"] != key:
        c = {"key": key, "wf": full_weight(m).detach().to(dev, torch.float32), "row": None}
        c["wpk"] = ops.pack_conv_weight(c["wf"], [m.in_channels])
        c["bias"] = ops.pad_vec(b, m.out_channels, dev)
        m.__dict__["_pbmc_pack"] = c  # plain attribute: not a parameter, not a buffer, not in the state_dict
    if want_row and c["row"] is None:
        c["row"] = ops.pack_conv_weight_row(c["wf"], [m.in_channels])
    return c["wpk"], (c["row"] if want_row else None), c["bias"]


def conv_module_forward(m: nn.Conv2d, x: torch.Tensor) -> torch.Tensor:
    """Stand-alone forward of an nn.Conv2d-shaped module on an NCHW tensor through libpbmc.
    Images of at least TENSOR_CORE_MIN_SIDE rows and columns with c_in, c_out <= 16 go to the tensor-core kernels (fp16 hi+lo, fp32-grade; the library
    picks the time-multiplexed or the row-streaming one), thin strips (the edge regions of the learned-boundary conv,
    reference :1022-1065) and wide outputs to the FFMA kernel.
    The input may have any magnitude: it is scaled by 2^-s with 2^(s-1) <= max|x| < 2^s (the bias with it) and the output
    by 2^s, exact in float32, so the kernels' fp16 split always sees |x| < 1.  s is computed on the device (no sync)."""
    _check_conv_supported(m)
    if not x.is_cuda:
        raise L.PbmcError("this layer has no CPU implementation; move the module and input to a CUDA device")
    k = m.kernel_size[0]
    pad = m.padding
    if pad == "valid":
        pad = (0, 0)
    elif pad == "same":
        pad = (k // 2, k // 2)
    # (single-group inputs only: the shapes this entry point has been verified with on hardware -- 16->16 and 16->1 at
    # k=5, 7->16 at k=3; wider inputs stay on the FFMA kernel here, the fused network path feeds conv[1] itself)
    tensor_core = m.out_channels <= 16 and m.in_channels <= 16 and min(x.shape[-2:]) >= TENSOR_CORE_MIN_SIDE
    wpk, wrow, bias = _packed_filters(m, x.device, tensor_core)
    mant, s = torch.frexp(x.abs().amax().float())
    s = torch.where(mant > 0, s, torch.zeros_like(s)).clamp(-126, 126)
    xb = ops.pack_nchw(x * ops.pow2(-s).to(x.dtype))
    mode = m.padding_mode if pad != (0, 0) else "zeros"
    yb, _, _ = ops.conv_fwd([ops.Source(xb)], wpk, bias * ops.pow2(-s), m.out_channels, k, mode,
                            impl="auto" if tensor_core else "ffma", wpk_row=wrow)
    y = ops.unpack_nchw(yb, m.out_channels) * ops.pow2(s)
    # 'same' geometry is computed; smaller paddings are a crop of it (exact for zeros / valid)
    cy, cx = k // 2 - pad[0], k // 2 - pad[1]
    if cy < 0 or cx < 0 or ((cy or cx) and mode != "zeros"):
        raise NotImplementedError("padding larger than k//2, or partial non-zero padding, is not implemented")
    if cy or cx:
        y = y[:, :, cy:y.shape[2] - cy, cx:y.shape[3] - cx]
    return y.to(x.dtype)


class SymmetricConv2d(nn.Conv2d):
    def __init__(self, in_channels: int, out_channels: int, kernel_size, stride=1, padding=0, dilation=1, groups: int = 1,
                 bias: bool = True, padding_mode: str = "zeros", symmetry: dict = {}, share_bias: bool = False):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, padding_mode)
        if self.groups > 1:
            raise ValueError(self.__str__() + " does not support groups>1")
        self.share_bias = share_bias if bias else False
        if symmetry is None:
            self.symmetry = None
        else:
            symmetry = dict(symmetry)
            for key in ("h", "v", "hv"):
                symmetry.setdefault(key, 0)
            self.symmetry = symmetry
            if symmetry["h"] % 2 or symmetry["v"] % 2:
                raise ValueError("Number of symmetric h and v filters must be divisible by 2")
            if symmetry["hv"] % 4:
                raise ValueError("Number of symmetric hv filters must be divisible by 4")
            assert sum(symmetry.values()) <= self.out_channels, "Number of symmetric channels exceeds number of out channels"
            self.unique_out_channels = (self.out_channels - symmetry["h"] // 2 - symmetry["v"] // 2 - 3 * symmetry["hv"] // 4)
            # only the unique filters are parameters (same state_dict shape as the reference)
            self.weight = Parameter(torch.empty(self.unique_out_channels, in_channels, *self.kernel_size))
            if bias:
                self.bias = Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def forward(self, input):
        return conv_module_forward(self, input)
