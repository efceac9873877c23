"""CPU checks of the entry points of NTD on the tensor core: declared in include/nnfac_b200.h, bound in nn_fac/_lib.py with the
header's argument count, exported by the library."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "nnfac_b200.h")
LIB = os.path.join(ROOT, "nn-fac_b200", "lib", "libnnfac_b200.so")
ENTRY_POINTS = {"nnfac_nmf_plan_set_operand": 6, "nnfac_nmf_plan_reduce_partials": 6}


def test_ntd_tc_entry_points_are_declared_bound_and_exported():
    from nn_fac import _lib
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    lib = ctypes.CDLL(LIB)
    for name, nargs in ENTRY_POINTS.items():
        m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)", text)
        assert m, f"{name} is not declared"
        assert len(m.group(1).split(",")) == nargs
        assert len(_lib.SIGNATURES[name]) == nargs
        assert hasattr(lib, name), f"{name} is not exported"
