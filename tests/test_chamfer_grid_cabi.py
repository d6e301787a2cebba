"""CPU: the C ABI surface of the grid Chamfer path and of nvsf_eval_points — symbols, argument checks that return
before any launch, workspace sizes, and the "chamfer_grid" option (a host-side switch)."""
import ctypes
import importlib

import pytest


def _lib():
    pkg = importlib.import_module("selfsupervised-nvsf_b200")
    importlib.import_module("selfsupervised-nvsf_b200.build").build()
    return pkg._lib.lib()


def test_new_symbols_are_exported():
    L = _lib()
    for name in ("nvsf_eval_points", "nvsf_eval_points_workspace_bytes", "nvsf_chamfer_forward",
                 "nvsf_chamfer_forward_counted", "nvsf_chamfer_workspace_bytes"):
        assert hasattr(L, name)


@pytest.mark.parametrize("b,n,m", [(1, 1, 1), (1, 4096, 4096), (3, 1000, 777), (1, 67980, 67980), (2, 5, 1 << 20),
                                   (1000, 64, 64)])
def test_chamfer_workspace_is_never_smaller_than_the_keys(b, n, m):
    L = _lib()
    wb = L.nvsf_chamfer_workspace_bytes(b, n, m)
    assert wb >= b * (n + m) * 8
    assert wb <= L.nvsf_chamfer_workspace_bytes(b, n + 1, m) and wb <= L.nvsf_chamfer_workspace_bytes(b, n, m + 1)


def test_eval_points_argument_checks():
    L = _lib()
    fake = ctypes.c_void_p(1 << 20)       # never dereferenced: every check below returns before a launch
    assert L.nvsf_eval_points_workspace_bytes(0, 5) == 0 and L.nvsf_eval_points_workspace_bytes(5, 0) == 0
    assert L.nvsf_eval_points_workspace_bytes(1 << 31, 5) == 0
    wb = L.nvsf_eval_points_workspace_bytes(1000, 2000)
    assert wb >= L.nvsf_chamfer_workspace_bytes(1, 1000, 2000) + 3000 * 8
    args = [fake, 1000, fake, fake, 2000, fake, 0.05, fake, fake, wb, None]
    for i in (0, 2, 3, 5, 7, 8):
        a = list(args)
        a[i] = None
        assert L.nvsf_eval_points(*a) == -1, i
    for i in (1, 4):
        a = list(args)
        a[i] = 0
        assert L.nvsf_eval_points(*a) == -1, i
    a = list(args)
    a[6] = -1.0
    assert L.nvsf_eval_points(*a) == -1
    a = list(args)
    a[8] = ctypes.c_void_p((1 << 20) + 8)   # not 16-byte aligned
    assert L.nvsf_eval_points(*a) == -1
    a = list(args)
    a[9] = wb - 1
    assert L.nvsf_eval_points(*a) == -2


def test_chamfer_grid_option_values():
    L = _lib()
    assert L.nvsf_get_option(b"chamfer_grid") == -1
    try:
        for v in (0, 1, -1):
            assert L.nvsf_set_option(b"chamfer_grid", v) == 0 and L.nvsf_get_option(b"chamfer_grid") == v
        for v in (2, -2, 100):
            assert L.nvsf_set_option(b"chamfer_grid", v) == -1
        assert L.nvsf_get_option(b"chamfer_grid") == -1
    finally:
        L.nvsf_set_option(b"chamfer_grid", -1)
