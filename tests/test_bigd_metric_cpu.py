"""No-GPU checks of the large-D Random path with a dense momentum metric (cov_p != I, target.Pt / Mit / Lct): the workspace size is
non-zero exactly for float32, all three matrices and 1024 < D <= 8192; the Python mirror routes exactly those runs there; the
library refuses what the path does not cover before it touches a buffer."""
import os

import pytest


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def _args(L, D, dtype=None, mats="PML", Nchain=1000):
    a = L.RandomArgs()
    a.dtype = L.HMC_F32 if dtype is None else dtype
    a.kernel = L.KERNEL_BIGD
    a.Nchain, a.Niter, a.iter_begin, a.iter_end = Nchain, 10, 0, 10
    a.thin_rate, a.L_low, a.L_high = 1, 1, 2
    a.target.D, a.target.D_pad = D, (D + 3) // 4 * 4
    # the matrices are given by address only (never dereferenced here)
    a.target.Pt = 0x1000 if "P" in mats else None
    a.target.Mit = 0x1000 if "M" in mats else None
    a.target.Lct = 0x1000 if "L" in mats else None
    return a


@pytest.mark.parametrize("D", [1025, 1283, 2048, 8192])
def test_dense_workspace_covers_above_1024(D):
    L, lib = _lib()
    dense = lib.hmc_random_workspace_bytes(_args(L, D))
    ident = lib.hmc_random_workspace_bytes(_args(L, D, mats=""))
    Dp = (D + 31) // 32 * 32
    assert ident > 0
    assert dense >= ident + 9 * Dp * Dp * 2                  # + P, M^-1 and Lc split into three bf16 parts
    assert dense >= ident + 9 * 1024 * Dp * 2 + 3 * 1024 * Dp * 4    # + the products' split rows and float32 results


@pytest.mark.parametrize("D,dtype,mats", [(128, None, "PML"), (300, None, "PML"), (1024, None, "PML"), (2048, 1, "PML"),
                                          (2048, None, "PM"), (2048, None, "L"), (8193, None, "PML")])
def test_dense_workspace_zero_outside_coverage(D, dtype, mats):
    L, lib = _lib()
    assert lib.hmc_random_workspace_bytes(_args(L, D, dtype, mats)) == 0


@pytest.mark.parametrize("D,dtype,mats,why", [(8193, None, "PML", r"D must be in \[128, 8192\]"),
                                              (2048, 1, "PML", "float32 only"),
                                              (2048, None, "PL", "needs target.Pt, Mit and Lct together"),
                                              (1024, None, "PML", "identity momentum metric only for D <= 1024"),
                                              (1024, None, "PL", "identity momentum metric only for D <= 1024"),
                                              (100, None, "PML", "identity momentum metric only for D <= 1024")])
def test_dense_refusals_before_any_buffer_is_touched(D, dtype, mats, why):
    """kernel = bigd with a configuration the path does not cover: HMC_E_UNSUPPORTED from the coverage check, which runs before
    anything is launched (the buffers are addresses only)."""
    import re
    L, lib = _lib()
    a = _args(L, D, dtype, mats)
    a.target.Ft = a.target.mu = a.target.dt = 0x1000
    a.q_start = a.q_chain = a.E_chain = a.dE_chain = a.state_q = a.state_eprev = 0x1000
    assert lib.hmc_random_run(a, None) == L.HMC_E_UNSUPPORTED
    msg = lib.hmc_last_error_string().decode()
    assert msg.startswith("large-D kernel does not cover this configuration: ") and re.search(why, msg), msg


def test_nuts_workspace_stays_identity_only():
    L, lib = _lib()
    a = L.NutsArgs()
    a.dtype, a.kernel, a.Nchain, a.d_max = L.HMC_F32, L.KERNEL_BIGD, 1000, 10
    a.Niter, a.iter_begin, a.iter_end, a.thin_rate = 10, 0, 10, 1
    a.target.D, a.target.D_pad = 2048, 2048
    assert lib.hmc_nuts_workspace_bytes(a) > 0
    a.target.Pt = a.target.Mit = a.target.Lct = 0x1000
    assert lib.hmc_nuts_workspace_bytes(a) == 0


def test_mirror_routing_table():
    import samplers as S
    r = S.random_runs_bigd
    # identity metric: as before
    assert r(1024, "float32", "auto", True) and r(1500, "float32", "auto", True) and r(300, "float32", "bigd", True)
    assert not r(300, "float32", "auto", True) and not r(1500, "float64", "auto", True) and not r(8193, "float32", "bigd", True)
    assert not r(1500, "float32", "generic", True) and not r(127, "float32", "bigd", True)
    # dense metric: float32, 1024 < D <= 8192, auto or bigd
    for D in (1025, 1283, 2048, 8192):
        assert r(D, "float32", "auto", False) and r(D, "float32", "bigd", False)
    assert not r(1024, "float32", "auto", False)             # the generic kernel keeps D <= 1024
    assert not r(1024, "float32", "bigd", False) and not r(300, "float32", "bigd", False)
    assert not r(8193, "float32", "auto", False) and not r(2048, "float64", "auto", False)
    assert not r(2048, "float32", "generic", False) and not r(2048, "float32", "fast", False)
