"""ctypes binding of libpbmc.so (the C ABI declared in include/pbmc.h).

There is deliberately no fallback: if the library is missing or a call fails the caller gets
an exception.  PyTorch is used only for device memory and streams; every pointer handed to
the library is `tensor.data_ptr()`.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libpbmc.so")

MAX_SRC, MAX_LEVELS, MAX_REPEATS = 8, 8, 8
PAD = {"zeros": 0, "constant": 0, "replicate": 1, "reflect": 2}
XFORM_NONE, XFORM_GN_GELU, XFORM_GN, XFORM_GELU = 0, 1, 2, 3
LAYOUT_BLOCKED, LAYOUT_STAGED16 = 0, 1
ACT_NONE, ACT_GELU = 0, 1
HEAD_CURL, HEAD_MAE = 0, 1
TRUNK_MODE = {"auto": 0, "per_layer": 1, "auto_bulk_loader": 4}  # pbmc_net.flags bits (PBMC_NET_TRUNK_*)
NET_UP_STAGED = 2
NET_LEARNED = 8
CONV_IMPL = {"auto": 0, "ffma": 1, "umma_3xtf32": 2, "umma_bf16": 3, "umma_f16x2": 4,
             "row_f16x2": 5, "row_bf16": 6, "mux_f16x2": 7, "mux_bf16": 8}


class Member(C.Structure):
    _fields_ = [("raq_nd", C.c_float), ("fkt_nd", C.c_float), ("fkp_nd", C.c_float), ("ln_fkt", C.c_float),
                ("ln_fkp", C.c_float), ("raq", C.c_float), ("scaler", C.c_float), ("reserved", C.c_float)]


class Src(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stats", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("nblk", C.c_int), ("xform", C.c_int), ("inv_count", C.c_double), ("layout", C.c_int), ("reserved", C.c_int)]


class ConvDesc(C.Structure):
    _fields_ = [("src", Src * MAX_SRC), ("nsrc", C.c_int), ("B", C.c_int), ("H", C.c_int), ("W", C.c_int),
                ("cout", C.c_int), ("ksize", C.c_int), ("pad_mode", C.c_int), ("epi_act", C.c_int), ("impl", C.c_int),
                ("max_ctas", C.c_int), ("wpk", C.c_void_p), ("wpk_umma", C.c_void_p), ("wpk_row", C.c_void_p),
                ("bias", C.c_void_p), ("out", C.c_void_p), ("out_stats", C.c_void_p), ("out_chan_sum", C.c_void_p)]


class Layer(C.Structure):
    _fields_ = [("wpk", C.c_void_p), ("wpk_umma", C.c_void_p), ("wpk_row", C.c_void_p), ("bias", C.c_void_p),
                ("gamma", C.c_void_p),
                ("beta", C.c_void_p), ("cin_blks", C.c_int), ("cout", C.c_int), ("ksize", C.c_int), ("reserved", C.c_int)]


class Net(C.Structure):
    _fields_ = [("levels", C.c_int), ("repeats", C.c_int), ("c_i", C.c_int), ("c_h", C.c_int), ("c_o", C.c_int),
                ("ksize", C.c_int), ("pad_mode", C.c_int), ("head_kind", C.c_int), ("p_pred", C.c_int),
                ("conv_impl", C.c_int), ("a_bound", C.c_float), ("flags", C.c_int), ("conv0", Layer),
                ("trunk", Layer * (MAX_LEVELS * MAX_REPEATS)), ("conv1", Layer), ("conv2", Layer), ("conv3", Layer),
                ("wedge_conv0", C.c_void_p), ("wedge_trunk", C.c_void_p * (MAX_LEVELS * MAX_REPEATS)),
                ("wedge_conv1", C.c_void_p), ("wedge_conv2", C.c_void_p), ("wedge_conv3", C.c_void_p)]


MAX_RANKS = 16


class SlabSync(C.Structure):
    _fields_ = [("slot", (C.c_uint64 * MAX_RANKS) * 2), ("steps_done", C.c_uint), ("ctas_done", C.c_uint),
                ("local_max", C.c_uint), ("failed", C.c_uint)]


class Edge9Desc(C.Structure):
    _fields_ = [("src", Src * MAX_SRC), ("nsrc", C.c_int), ("B", C.c_int), ("H", C.c_int), ("W", C.c_int), ("cout", C.c_int),
                ("ksize", C.c_int), ("epi_act", C.c_int), ("reserved", C.c_int), ("wedge", C.c_void_p), ("bias", C.c_void_p),
                ("out", C.c_void_p), ("out_stats", C.c_void_p), ("out_chan_sum", C.c_void_p)]


class TrunkDesc(C.Structure):
    _fields_ = [("src0", Src), ("layers", C.POINTER(Layer)), ("ping", C.c_void_p * 2), ("stats", C.c_void_p),
                ("sync", C.c_void_p), ("R", C.c_int), ("B", C.c_int), ("H", C.c_int), ("W", C.c_int), ("pad_mode", C.c_int),
                ("impl", C.c_int), ("max_ctas", C.c_int), ("pre_zeroed", C.c_int), ("loader", C.c_int), ("reserved", C.c_int)]


_STRUCTS = {"pbmc_edge9_desc": Edge9Desc, "pbmc_trunk_desc": TrunkDesc, "pbmc_slab_sync": SlabSync, "pbmc_member": Member, "pbmc_src": Src, "pbmc_conv_desc": ConvDesc, "pbmc_layer": Layer, "pbmc_net": Net}

# name -> (restype, argtypes); every symbol declared in include/pbmc.h
_vp, _i, _d, _f, _sz = C.c_void_p, C.c_int, C.c_double, C.c_float, C.c_size_t
SIGNATURES = {
    "pbmc_error_string": (C.c_char_p, [_i]),
    "pbmc_version": (_i, []),
    "pbmc_sizeof": (_sz, [C.c_char_p]),
    "pbmc_last_cuda_error": (C.c_char_p, []),
    "pbmc_pack_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "pbmc_unpack_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "pbmc_build_input": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "pbmc_conv_fwd": (_i, [C.POINTER(ConvDesc), _vp]),
    "pbmc_conv_edge9": (_i, [C.POINTER(Edge9Desc), _vp]),
    "pbmc_trunk_fwd": (_i, [C.POINTER(TrunkDesc), _vp]),
    "pbmc_trunk_supported": (_i, [C.POINTER(TrunkDesc)]),
    "pbmc_avgpool2": (_i, [C.POINTER(Src), _vp, _i, _i, _i, _vp]),
    "pbmc_bicubic_up": (_i, [C.POINTER(Src), _vp, _i, _i, _i, _i, _i, _vp]),
    "pbmc_bicubic_up_staged": (_i, [C.POINTER(Src), _vp, _i, _i, _i, _i, _i, _vp]),
    "pbmc_staged_width": (_i, [_i]),
    "pbmc_staged_bytes": (C.c_size_t, [_i, _i, _i]),
    "pbmc_head": (_i, [_vp, _vp, _vp, _f, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "pbmc_advect_diffuse": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _d, _d, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "pbmc_advect_diffuse_slab": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pbmc_slab_sync_publish": (_i, [_vp, _vp, _i, _i, _vp, C.POINTER(C.c_void_p), _i, _i, _vp]),
    "pbmc_advect_diffuse_slab_sync": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp,
                                           C.POINTER(C.c_void_p), _i, _i, _vp]),
    "pbmc_stencil_coefs": (_i, [_vp, _i, _d, _d, _vp, _vp]),
    "pbmc_uvmax": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "pbmc_advect_diffuse_fields": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _i, _vp, _d, _vp, _vp, _vp, _i, _i,
                                        _i, _vp]),
    "pbmc_finalize_nchw": (_i, [C.POINTER(Src), _vp, _i, _i, _i, _i, _vp]),
    "pbmc_clamp_T": (_i, [_vp, _i, _i, _i, _i, _vp]),
    "pbmc_diagnostics": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "pbmc_ctx_create": (_i, [C.POINTER(_vp)]),
    "pbmc_ctx_destroy": (_i, [_vp]),
    "pbmc_workspace_bytes": (_sz, [C.POINTER(Net), _i, _i, _i]),
    "pbmc_trunk_cta_budgets": (_i, [C.POINTER(Net), _i, _i, _i, C.POINTER(C.c_int)]),
    "pbmc_surrogate_forward": (_i, [_vp, C.POINTER(Net), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _i, _i, _vp]),
    "pbmc_rollout": (_i, [_vp, C.POINTER(Net), _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _vp, _i, _i, _i, _vp, _i, _vp, _vp,
                          _vp, _vp, _vp, _sz, _i, _i, _i, _vp]),
}

_lib = None


class PbmcError(RuntimeError):
    pass


def load():
    """Load libpbmc.so (once).  Raises if it has not been built -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PbmcError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a). There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    for name, st in _STRUCTS.items():
        n = lib.pbmc_sizeof(name.encode())
        if n != C.sizeof(st):
            raise PbmcError(f"struct {name}: C size {n} != ctypes size {C.sizeof(st)}")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        lib = load()
        msg = lib.pbmc_error_string(rc).decode()
        cuda = lib.pbmc_last_cuda_error().decode()
        raise PbmcError(f"{what}: {msg}" + (f" [{cuda}]" if rc == -6 and cuda else ""))


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL).  Refuses CPU tensors: no fallback."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PbmcError("libpbmc needs CUDA tensors; this path has no CPU implementation")
    if not t.is_contiguous():
        raise PbmcError("libpbmc needs contiguous tensors")
    return t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def make_src(t, nblk, xform=XFORM_NONE, stats=None, gamma=None, beta=None, inv_count=0.0, layout=LAYOUT_BLOCKED):
    s = Src()
    s.ptr, s.stats, s.gamma, s.beta = ptr(t), ptr(stats), ptr(gamma), ptr(beta)
    s.nblk, s.xform, s.inv_count, s.layout = int(nblk), int(xform), float(inv_count), int(layout)
    return s
