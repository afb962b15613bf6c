"""No-GPU checks of NUTS with a ring of stored samples (hmc_nuts_args.store_ring, served by the large-D path only): the ctypes field
against include/hmc_b200.h, the rejections hmc_nuts_run makes before anything reaches the device, and the mirror's rule
(samplers.nuts_runs_bigd) with the constructor's acceptance and refusals of stream_stats for NUTS."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def test_store_ring_field_matches_header(tmp_path):
    """NutsArgs.store_ring sits where the header puts it (the former reserved word after flags); the struct keeps its size and the
    fields around it keep their offsets."""
    L, _ = _lib()
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hmc_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                   'sizeof(hmc_nuts_args),offsetof(hmc_nuts_args,store_ring),offsetof(hmc_nuts_args,flags),'
                   'offsetof(hmc_nuts_args,n_leapfrog),offsetof(hmc_nuts_args,workspace_bytes));return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, ring, flags, nleap, wsb = (int(v) for v in subprocess.check_output([str(exe)]).decode().split())
    assert L.NutsArgs.store_ring.offset == ring == flags + 4
    assert L.NutsArgs.flags.offset == flags and L.NutsArgs.n_leapfrog.offset == nleap
    assert L.NutsArgs.workspace.offset == ring + 4
    assert ctypes.sizeof(L.NutsArgs) == size == wsb + 8
    assert "reserved0" not in [f[0] for f in L.NutsArgs._fields_]


def _args(L, D, store_ring, kernel, dtype=None, workspace=True):
    """Arguments that pass every other check of hmc_nuts_run; the device pointers are fake and never dereferenced."""
    p = 1 << 20
    a = L.NutsArgs()
    a.dtype = L.HMC_F32 if dtype is None else dtype
    a.kernel = L.KERNELS[kernel]
    a.Nchain, a.d_max, a.Niter, a.iter_begin, a.iter_end, a.warm_up_num, a.thin_rate = 64, 10, 20, 0, 20, 2, 1
    a.target.D, a.target.D_pad = D, (D + 3) // 4 * 4
    a.target.Ft = a.target.mu = a.target.dt = p
    a.q_start = a.q_chain = a.E_chain = a.dE_chain = a.state_q = a.state_eprev = a.scratch = a.counters = p
    a.store_ring = store_ring
    if workspace:
        a.workspace, a.workspace_bytes = p, 1 << 40
    return a


@pytest.mark.parametrize("kernel", ["auto", "generic", "tc", "bigd"])
def test_negative_store_ring_is_a_bad_argument(kernel):
    L, lib = _lib()
    assert lib.hmc_nuts_run(_args(L, 300, -1, kernel), None) == L.HMC_E_BADARG
    assert "store_ring" in lib.hmc_last_error_string().decode()


@pytest.mark.parametrize("D,kernel,dtype,workspace", [
    (200, "generic", None, True), (300, "generic", None, True), (100, "tc", None, True),   # the kernels that keep the full stream
    (100, "auto", None, True),                                                             # AUTO below the large-D path
    (300, "auto", None, False),                                                            # AUTO without a workspace
    (300, "auto", 1, True)])                                                               # AUTO at float64
def test_store_ring_outside_the_large_d_path_is_unsupported(D, kernel, dtype, workspace):
    """All decided before any CUDA call (this machine needs no device for it)."""
    L, lib = _lib()
    assert lib.hmc_nuts_run(_args(L, D, 8, kernel, dtype, workspace), None) == L.HMC_E_UNSUPPORTED
    msg = lib.hmc_last_error_string().decode()
    assert "store_ring" in msg and "128 <= D <= 8192" in msg, msg


def test_nuts_runs_bigd_rule():
    import samplers as S
    f = S.nuts_runs_bigd
    assert f(300, "float32", "auto", True, False) and f(1500, "float32", "auto", True, False)
    assert not f(200, "float32", "auto", True, False) and f(200, "float32", "auto", True, True)   # auto from D = 128 with a ring
    assert f(128, "float32", "auto", True, True) and not f(127, "float32", "auto", True, True)
    assert f(128, "float32", "bigd", True, False) and f(8192, "float32", "bigd", True, False)
    assert not f(8193, "float32", "bigd", True, True) and not f(100, "float32", "auto", True, True)
    for stream in (False, True):
        assert not f(300, "float64", "auto", True, stream)
        assert not f(300, "float32", "auto", False, stream)
        assert not f(300, "float32", "generic", True, stream) and not f(300, "float32", "tc", True, stream)


def _nuts(D, stream_stats, Niter=100, **kw):
    import samplers as S
    spec = S.MVNSpec(np.zeros(D), np.eye(D), 0.0)
    return S.HMC_sampler(D, None, None, Nchain=4, Niter=Niter, sampler_type="NUTS", dt=0.1, d_max=5, target=spec,
                         stream_stats=stream_stats, **kw)


@pytest.mark.parametrize("D,kw", [(128, {}), (200, {}), (300, {}), (300, dict(kernel="bigd")), (1024, dict(kernel="bigd"))])
def test_constructor_accepts_stream_stats_on_the_large_d_path(D, kw):
    H = _nuts(D, 49, **kw)                                  # n = 50: T up to 49
    assert H.stream_stats == 49


@pytest.mark.parametrize("D,kw", [(100, {}), (200, dict(kernel="generic")), (300, dict(dtype="float64")),
                                  (300, dict(cov_p="dense")), (100, dict(kernel="tc")), (127, {})])
def test_constructor_refuses_stream_stats_off_the_large_d_path(D, kw):
    import samplers as S
    if kw.get("cov_p") == "dense":
        kw = dict(cov_p=S.equicorrelated_cov(D, 0.3))
    with pytest.raises(AssertionError, match="stream_stats") as e:
        _nuts(D, 20, **kw)
    assert "128 <= D <= 8192" in str(e.value)


def test_constructor_bounds_t_for_nuts_as_for_random():
    with pytest.raises(AssertionError, match="stream_stats"):
        _nuts(300, 50)                                      # T > n - 1 = 49
    with pytest.raises(AssertionError, match="stream_stats"):
        _nuts(300, 0)
