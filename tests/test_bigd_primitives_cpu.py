"""No-GPU checks of the large-D primitives (csrc/bigd_primitives.cu): the workspace sizes of hmc_start_pts_bigd and
hmc_leap_frog_bigd are non-zero exactly for the configurations the entry points cover, the ctypes declarations match
include/hmc_b200.h, the entry points refuse what they do not cover before touching the device, and the Python mirror's routing
rule."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def _target(L, D):
    t = L.Target()
    t.D, t.D_pad = D, (D + 3) // 4 * 4
    t.Ft = t.mu = t.dt = 0x1000                    # (never dereferenced here)
    return t


@pytest.mark.parametrize("D", [128, 300, 777, 4097, 8192])
@pytest.mark.parametrize("n", [1, 129, 1000, 131072])
def test_workspace_bytes_cover_any_d(D, n):
    L, lib = _lib()
    Dp = (D + 31) // 32 * 32
    Ncp = (n + 511) // 512 * 512
    s = lib.hmc_start_pts_workspace_bytes(n, D)
    assert s >= 3 * Ncp * Dp * 2 + 3 * Dp * Dp * 2 + Ncp * Dp * 4             # split normals, split Lc, product rows
    f = lib.hmc_leap_frog_workspace_bytes(_target(L, D), n, 0)
    assert f >= 2 * 3 * Ncp * Dp * 2 + 3 * Dp * Dp * 2 + 2 * Ncp * Dp * 4     # two operand buffers, split matrix, x and p rows
    assert lib.hmc_leap_frog_workspace_bytes(_target(L, D), n, L.FLAG_TC_FP16X2) == f     # covers both splits
    if D < 8192:
        assert lib.hmc_start_pts_workspace_bytes(n, D + 32) > s
        assert lib.hmc_leap_frog_workspace_bytes(_target(L, D + 32), n, 0) > f


@pytest.mark.parametrize("D,n", [(127, 1000), (8193, 1000), (0, 1000), (1024, 0), (1024, -5), (1024, 2 ** 30 + 1)])
def test_workspace_bytes_zero_outside_coverage(D, n):
    L, lib = _lib()
    assert lib.hmc_start_pts_workspace_bytes(n, D) == 0
    assert lib.hmc_leap_frog_workspace_bytes(_target(L, D), n, 0) == 0


def test_leap_frog_workspace_bytes_without_target():
    _, lib = _lib()
    assert lib.hmc_leap_frog_workspace_bytes(None, 1000, 0) == 0


@pytest.mark.parametrize("dtype,D,why", [(1, 1500, "float32 only"), (0, 127, r"D must be in \[128, 8192\]"),
                                         (0, 8193, r"D must be in \[128, 8192\]")])
def test_entry_points_refuse_what_they_do_not_cover(dtype, D, why):
    """Coverage is checked on the host before anything reaches the device (the pointers are never dereferenced)."""
    L, lib = _lib()
    p = C.c_void_p(0x1000)
    rc = lib.hmc_leap_frog_bigd(dtype, _target(L, D), 256, p, p, p, p, 1, 0, p, 1 << 40, None)
    assert rc == L.HMC_E_UNSUPPORTED
    assert re.search("hmc_leap_frog_bigd does not cover this configuration: " + why, lib.hmc_last_error_string().decode())
    rc = lib.hmc_start_pts_bigd(dtype, 0, 0, 256, D, p, p, None, p, p, 1 << 40, None)
    assert rc == L.HMC_E_UNSUPPORTED
    assert re.search("hmc_start_pts_bigd does not cover this configuration: " + why, lib.hmc_last_error_string().decode())


def test_entry_points_reject_bad_arguments():
    L, lib = _lib()
    p = C.c_void_p(0x1000)
    assert lib.hmc_leap_frog_bigd(0, _target(L, 1500), 0, p, p, p, p, 1, 0, p, 1 << 40, None) == L.HMC_E_BADARG
    assert lib.hmc_leap_frog_bigd(0, _target(L, 1500), 16, p, p, p, p, 0, 0, p, 1 << 40, None) == L.HMC_E_BADARG
    assert lib.hmc_leap_frog_bigd(0, _target(L, 1500), 16, None, p, p, p, 1, 0, p, 1 << 40, None) == L.HMC_E_BADARG
    assert lib.hmc_start_pts_bigd(0, 0, 0, 16, 1500, p, None, None, p, p, 1 << 40, None) == L.HMC_E_BADARG     # no Lc, no sd
    assert lib.hmc_start_pts_bigd(0, 0, 0, 0, 1500, p, p, None, p, p, 1 << 40, None) == L.HMC_E_BADARG


_CTYPES = {"int": C.c_int, "int32_t": C.c_int32, "int64_t": C.c_int64, "uint64_t": C.c_uint64}


def _header_decl(name):
    src = open(os.path.join(ROOT, "include", "hmc_b200.h")).read()
    m = re.search(r"\n(int64_t|int)\s+%s\(([^)]*)\);" % name, src)
    assert m, name
    args = [a.strip() for a in m.group(2).split(",")]
    return m.group(1), args


@pytest.mark.parametrize("name", ["hmc_start_pts_workspace_bytes", "hmc_start_pts_bigd", "hmc_leap_frog_workspace_bytes",
                                  "hmc_leap_frog_bigd"])
def test_ctypes_declarations_match_header(name):
    L, lib = _lib()
    ret, args = _header_decl(name)
    fn = getattr(lib, name)
    assert fn.restype is _CTYPES[ret]
    want = []
    for a in args:
        if a.startswith("const hmc_target*"):
            want.append(C.POINTER(L.Target))
        elif "*" in a:
            want.append(C.c_void_p)
        else:
            want.append(_CTYPES[a.split()[0]])
    assert list(fn.argtypes) == want
    assert name in L.EXPORTS


@pytest.mark.parametrize("D,entry", [(1, "hmc_start_pts"), (128, "hmc_start_pts"), (4096, "hmc_start_pts"),
                                     (4097, "hmc_start_pts_bigd"), (8192, "hmc_start_pts_bigd"), (8193, "hmc_start_pts_bigd")])
def test_start_pts_routing(D, entry):
    import utils as U
    assert U.start_pts_entry(D) == entry


@pytest.mark.parametrize("D,entry", [(2, "hmc_leap_frog"), (128, "hmc_leap_frog"), (1024, "hmc_leap_frog"),
                                     (1025, "hmc_leap_frog_bigd"), (8192, "hmc_leap_frog_bigd"), (8193, "hmc_leap_frog_bigd")])
def test_leap_frog_routing(D, entry):
    import samplers as S
    assert S.leap_frog_entry(D) == entry
