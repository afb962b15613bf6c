"""No-GPU check of the large-D path's coverage: hmc_random_workspace_bytes is non-zero exactly for the runs the path covers
(float32, identity momentum metric, any 128 <= D <= 8192) and 0 otherwise.  The size is computed on the host only."""
import os

import pytest


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def _args(L, D, dtype=None, dense=False, Nchain=1000):
    a = L.RandomArgs()
    a.dtype = L.HMC_F32 if dtype is None else dtype
    a.kernel = L.KERNEL_BIGD
    a.Nchain, a.Niter, a.iter_begin, a.iter_end = Nchain, 10, 0, 10
    a.thin_rate, a.L_low, a.L_high = 1, 1, 2
    a.target.D, a.target.D_pad = D, (D + 3) // 4 * 4
    if dense:                                       # a dense metric is given by its three matrices (never dereferenced here)
        a.target.Pt = a.target.Mit = a.target.Lct = 0x1000
    return a


@pytest.mark.parametrize("D", [128, 300, 777, 1283, 8192])
def test_workspace_bytes_cover_any_d(D):
    L, lib = _lib()
    n = lib.hmc_random_workspace_bytes(_args(L, D))
    Dp = (D + 31) // 32 * 32
    assert n >= 3 * 2 * 1024 * Dp * 2 + 3 * Dp * Dp * 2 + 3 * 1024 * Dp * 4     # split operands, split matrix, x / x0 / p at Dp


@pytest.mark.parametrize("D,dtype,dense", [(127, None, False), (8193, None, False), (1024, 1, False), (1024, None, True)])
def test_workspace_bytes_zero_outside_coverage(D, dtype, dense):
    L, lib = _lib()
    assert lib.hmc_random_workspace_bytes(_args(L, D, dtype, dense)) == 0
