"""CPU tests of pls_bnb_cv_path's host side: the library exports it, and the ctypes binding matches the header."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# C parameter types of include/pls.h and the names of the ctypes types they bind to on LP64 Linux (c_int32 is c_int,
# c_int64 is c_long, c_uint32 is c_uint there)
_CTYPES = {"pls_ctx *": "c_void_p", "const int32_t *": "LP_c_int", "int64_t": "c_long", "const double *": "LP_c_double",
           "uint32_t": "c_uint", "double *": "LP_c_double", "int64_t *": "LP_c_long", "pls_stats *": "LP_PlsStats"}


def _header_params(name):
    with open(os.path.join(ROOT, "include", "pls.h")) as fh:
        text = fh.read()
    m = re.search(r"int\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    params = [" ".join(p.split()) for p in m.group(1).split(",")]
    return [re.sub(r"\s*\w+$", "", p).replace("*", " *").replace("  ", " ").strip() for p in params]


def test_library_exports_bnb_cv_path(pkg):
    assert hasattr(pkg._abi.lib, "pls_bnb_cv_path")
    assert hasattr(pkg._abi.Context, "bnb_cv_path")


def test_ctypes_signature_matches_header(pkg):
    C = pkg._abi.C
    params = _header_params("pls_bnb_cv_path")
    assert len(params) == 13, params
    bound = pkg._abi.lib.pls_bnb_cv_path.argtypes
    assert len(bound) == len(params)
    for p, t in zip(params, bound):
        assert t.__name__ == _CTYPES[p], (p, t.__name__)
    assert pkg._abi.lib.pls_bnb_cv_path.restype is C.c_int
