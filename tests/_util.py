"""Shared helpers for the tests: golden loading and error norms."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    """tests/golden/<name>.npz as a dict.  Weights that are exactly float32 values are stored as float32 to keep the files
    small; they come back as the float64 arrays they were written from."""
    d = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    return {k: v.astype(np.float64) if v.dtype == np.float32 else v for k, v in d.items()}


def load_weights(name):
    return load(name + "_weights")


def sample_index(H, W, n_interior, seed=0):
    """Flat indices at which a full-size golden stores an H x W field: every boundary cell (the walls and the padding
    modes act there) and `n_interior` interior cells drawn once with a fixed seed.  Sorted int32."""
    ring = np.zeros((H, W), dtype=bool)
    ring[0], ring[-1], ring[:, 0], ring[:, -1] = True, True, True, True
    flat = np.flatnonzero(ring)
    interior = np.flatnonzero(~ring)
    pick = np.random.default_rng(seed).choice(interior, size=n_interior, replace=False)
    return np.sort(np.concatenate([flat, pick])).astype(np.int32)


def at(a, idx):
    """The values of a 2-D field at the flat indices `idx` (how the full-size goldens store a field)."""
    return np.asarray(a).reshape(-1)[idx]


def split_weights(d, prefix="w::"):
    return {k[len(prefix):]: v for k, v in d.items() if k.startswith(prefix)}


def noise(tag):
    """The reference's OWN float32-vs-float64 distance on golden case `tag` (tests/golden/ref_fp32_noise.json, written by
    make_golden.py from the real reference): rel-L2 per output field, max-abs for T, relative for dt."""
    import json

    return json.load(open(os.path.join(GOLDEN, "ref_fp32_noise.json")))[tag]


def field_bound(ref_noise, floor=1e-5):
    """north_star's 1e-5 relative bound, widened to 1.5 x the reference's own fp32 noise where that is larger
    (SURVEY.md section 8c: no fp32 implementation, PyTorch's included, is closer to the fp64 reference than that)."""
    return max(floor, 1.5 * float(ref_noise))


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def spec_from_variant(d):
    from oracle.ref_numpy import NetSpec

    s = d["spec"]
    return NetSpec(levels=int(s[0]), c_i=int(s[1]), c_h=int(s[2]), c_o=int(s[3]), repeats=int(s[4]), f=int(s[5]),
                   use_symm=bool(s[6]), p_pred=bool(s[7]), r_p=str(d["r_p"]), loss_type=str(d["loss_type"]),
                   a_bound=float(d["a_bound"]))


VARIANTS = ["var_zeros_nosym", "var_reflect_sym", "var_replicate_odd", "var_mae_p", "var_k5"]


UNET_CASES = ["unet_curl_p", "unet_curl_k5", "unet_mae", "unet_learned_k3", "unet_learned_k5"]


LEARNED_CASES = ["learned_k5", "learned_k3_p", "learned_fluidnet"]


def load_learned_case(tag):
    """One whole learned-boundary network case, tests/golden/<tag>.npz: like load_unet_case."""
    return load_unet_case(tag)


def load_unet_case(tag):
    """One network case, tests/golden/<tag>.npz: (spec, input, {name: array for u, v, p, T}, state_dict as numpy).  The
    input is not stored: it is redrawn from its seed exactly as make_golden.py drew it for the reference."""
    import torch

    d = load(tag)
    spec = spec_from_variant(d)
    g = torch.Generator().manual_seed(int(d["inp_seed"]))
    inp = torch.randn(*(int(n) for n in d["inp_shape"]), generator=g, dtype=torch.float64).numpy()
    outs = {n: d[n] for n in "uvpT" if n in d}
    return spec, inp, outs, split_weights(d)
