"""Repository rules that the judge checks mechanically."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _py_files(d):
    for dp, _, fs in os.walk(d):
        for f in fs:
            if f.endswith(".py"):
                yield os.path.join(dp, f)


def test_product_never_imports_oracle():
    pat = re.compile(r"^\s*(from|import)\s+oracle\b", re.M)
    for f in _py_files(os.path.join(ROOT, "pbml_mantle_convection_b200")):
        assert not pat.search(open(f).read()), f"{f} imports the oracle"


def test_product_has_no_reference_or_triton_dependency():
    for f in _py_files(os.path.join(ROOT, "pbml_mantle_convection_b200")):
        src = open(f).read()
        assert ("/root/" + "reference") not in src, f
        assert not re.search(r"^\s*(from|import)\s+triton\b", src, re.M), f
        assert "torch.compile" not in src, f


def test_gpu_side_files_do_not_read_reference():
    for f in list(_py_files(os.path.join(ROOT, "tests"))) + [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]:
        if f.endswith("make_golden.py") or f.endswith("test_layout.py"):
            continue
        assert ("/root/" + "reference") not in open(f).read(), f


def test_library_reads_no_environment_and_keeps_no_launch_switches():
    """What libpbmc runs is decided by its C-ABI arguments alone, and whether a launch is programmatic-dependent by the
    arguments of the function that makes it."""
    csrc = os.path.join(ROOT, "pbml_mantle_convection_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh", ".h")):
            src = open(os.path.join(csrc, f)).read()
            for word in ("getenv", "PBMC_DEV_", "_pdl_next"):
                assert word not in src, f"{f} contains {word}"
