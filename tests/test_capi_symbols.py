"""The C-ABI library builds, loads, and exports every symbol include/carmpc.h declares (no compute without a GPU)."""
import ctypes
import os
import re

from conftest import ROOT


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "carmpc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(carmpc_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_public_entry_points():
    names = _declared_functions()
    for must in ("carmpc_polytope_create", "carmpc_membership_bitset", "carmpc_membership_grid",
                 "carmpc_membership_bitset_host", "carmpc_rollout_create", "carmpc_rollout_bitset",
                 "carmpc_qp_create", "carmpc_qp_solve", "carmpc_qp_solve_host", "carmpc_closed_loop",
                 "carmpc_destroy", "carmpc_last_error"):
        assert must in names


def test_library_exports_every_declared_symbol():
    from carmpc_b200 import _capi, build
    path = build.build_library()
    assert os.path.isfile(path)
    lib = ctypes.CDLL(path)
    missing = [n for n in _declared_functions() if not hasattr(lib, n)]
    assert not missing, f"declared in carmpc.h but not exported: {missing}"
    assert sorted(_capi.SIGNATURES) == _declared_functions()
    lib.carmpc_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.carmpc_version()


def test_argument_errors_do_not_need_a_gpu():
    from carmpc_b200 import _capi
    lib = _capi.load()
    h = ctypes.c_void_p()
    assert lib.carmpc_polytope_create(None, 3, ctypes.byref(h)) == -1
    assert b"null" in lib.carmpc_last_error()
    assert lib.carmpc_membership_bitset(None, None, None, None, None, 0, None, None, 0, None) == -1
    val = ctypes.c_double()
    assert lib.carmpc_measure_peak(9, ctypes.byref(val)) == -1
