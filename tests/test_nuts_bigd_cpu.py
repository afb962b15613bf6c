"""No-GPU check of the large-D NUTS path's coverage: hmc_nuts_workspace_bytes is non-zero exactly for the runs the path covers
(float32, identity momentum metric, any 128 <= D <= 8192), 0 otherwise, and grows with the chain count and D.  The size is
computed on the host only."""
import os

import pytest


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def _args(L, D, dtype=None, dense=False, Nchain=1000, d_max=10):
    a = L.NutsArgs()
    a.dtype = L.HMC_F32 if dtype is None else dtype
    a.kernel = L.KERNEL_BIGD
    a.Nchain, a.d_max, a.Niter, a.iter_begin, a.iter_end = Nchain, d_max, 10, 0, 10
    a.thin_rate = 1
    a.target.D, a.target.D_pad = D, (D + 3) // 4 * 4
    if dense:                                       # a dense metric is given by its three matrices (never dereferenced here)
        a.target.Pt = a.target.Mit = a.target.Lct = 0x1000
    return a


@pytest.mark.parametrize("D", [128, 300, 777, 1024, 1500, 8192])
def test_nuts_workspace_bytes_cover_any_d(D):
    L, lib = _lib()
    n = lib.hmc_nuts_workspace_bytes(_args(L, D))
    Dp = (D + 31) // 32 * 32
    # split operand (three parts), split matrix, x / p / gradient rows, all Dp wide over 1,024 padded rows
    assert n >= 3 * 1024 * Dp * 2 + 3 * Dp * Dp * 2 + 3 * 1024 * Dp * 4
    assert lib.hmc_nuts_workspace_bytes(_args(L, D, Nchain=5000)) > n
    if D < 8192:
        assert lib.hmc_nuts_workspace_bytes(_args(L, D + 32)) > n
    assert lib.hmc_nuts_workspace_bytes(_args(L, D, d_max=4)) == n      # the check-point stack lives in the caller's scratch


@pytest.mark.parametrize("D,dtype,dense", [(127, None, False), (100, None, False), (8193, None, False), (1024, 1, False),
                                           (1024, None, True)])
def test_nuts_workspace_bytes_zero_outside_coverage(D, dtype, dense):
    L, lib = _lib()
    assert lib.hmc_nuts_workspace_bytes(_args(L, D, dtype, dense)) == 0


def test_nuts_args_keep_their_offsets():
    """The large-D fields are appended: every field the earlier layout had keeps its offset."""
    import ctypes
    L, _ = _lib()
    assert L.NutsArgs.n_leapfrog.offset + ctypes.sizeof(ctypes.c_void_p) == L.NutsArgs.flags.offset
    assert L.NutsArgs.workspace_bytes.offset + 8 == ctypes.sizeof(L.NutsArgs)
