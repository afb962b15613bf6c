"""No-GPU checks of the streamed diagnostics (csrc/diag_stream.cu, utils.stream_stats_from_workspace, samplers.stream_blocks):
workspace sizes, the ctypes declarations against include/hmc_b200.h, the argument rejections (made before anything reaches the
device), the host finishing with a maximum lag against a float64 restatement of utils.py:130-157 cut at T, and the iteration-block
plan of a stream_stats run."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import hmc_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FUNCS = ["hmc_diag_stream_workspace_bytes", "hmc_diag_stream_update", "hmc_diag_stream_finish"]


def _lib():
    import hmc_b200_lib as L
    if not os.path.isfile(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return L, L.load()


def test_workspace_bytes_coverage_and_growth():
    L, lib = _lib()
    ws = lib.hmc_diag_stream_workspace_bytes
    assert ws(1, 1, 1) == 8 * 1 * (4 + 1 + 3)
    assert ws(131072, 1024, 64) == 8 * 1024 * (4 + 64 + 3 * 131072)
    for bad in [(0, 100, 10), (-1, 100, 10), (10, 0, 10), (10, 8193, 10), (10, 100, 0), (10, 100, -3), (10, 100, (1 << 20) + 1)]:
        assert ws(*bad) == 0, bad
    assert ws(10, 8192, 1 << 20) > 0
    base = ws(1000, 100, 32)
    assert ws(2000, 100, 32) > base and ws(1000, 200, 32) > base and ws(1000, 100, 64) > base
    assert ws(2000, 100, 32) - base == 8 * 100 * 3 * 1000          # 3 float64 per chain and dimension
    assert ws(1000, 100, 64) - base == 8 * 100 * 32                # one float64 row per lag


_CTYPE = {"int32_t": C.c_int32, "int64_t": C.c_int64, "int": C.c_int}


def test_ctypes_declarations_match_header():
    L, lib = _lib()
    hdr = open(os.path.join(ROOT, "include", "hmc_b200.h")).read()
    for name in FUNCS:
        assert name in L.EXPORTS
        m = re.search(r"^(int64_t|int)\s+%s\s*\(([^;]*)\);" % name, hdr, flags=re.M | re.S)
        assert m, name
        args = [a.strip() for a in m.group(2).replace("\n", " ").split(",")]
        want = [C.c_void_p if "*" in a else _CTYPE[a.split()[0]] for a in args]
        fn = getattr(lib, name)
        assert fn.restype is _CTYPE[m.group(1)], name
        assert list(fn.argtypes) == want, name


def test_update_and_finish_reject_bad_arguments():
    """Every check is made on the host before anything is enqueued: fake device pointers never get dereferenced."""
    L, lib = _lib()
    p = C.c_void_p(1 << 20)
    Nc, D, Lc, T = 8, 10, 41, 5                  # n = 20
    nb = int(lib.hmc_diag_stream_workspace_bytes(Nc, D, T))

    def upd(dtype=L.HMC_F32, ring=p, Nchain=Nc, D_=D, R=T + 4, Lchain=Lc, T_=T, j0=0, j1=4, ws=p, nbytes=nb):
        return lib.hmc_diag_stream_update(dtype, ring, Nchain, D_, R, Lchain, T_, j0, j1, ws, nbytes, None)

    bad = [dict(R=T + 3),                               # R < T + (j1 - j0)
           dict(j0=10, j1=20, R=T + 9),
           dict(T_=0), dict(T_=20, R=40), dict(Lchain=12, T_=5),     # T < 1, T > n - 1
           dict(j0=-1), dict(j0=5, j1=4), dict(j0=38, j1=42, R=20),  # j0 / j1 outside [0, L_chain]
           dict(ws=None), dict(nbytes=nb - 8),          # missing or short workspace
           dict(dtype=7), dict(ring=None), dict(Nchain=0), dict(D_=0), dict(D_=8193)]
    for kw in bad:
        assert upd(**kw) == L.HMC_E_BADARG, kw
    msg = lib.hmc_last_error_string().decode()
    assert "D" in msg
    assert upd(R=T + 3) == L.HMC_E_BADARG and "ring" in lib.hmc_last_error_string().decode()
    assert upd(nbytes=nb - 8) == L.HMC_E_BADARG and "workspace of %d bytes" % nb in lib.hmc_last_error_string().decode()
    out = C.c_void_p(1 << 21)
    fin = lib.hmc_diag_stream_finish
    assert fin(None, nb, D, T, out, out, None) == L.HMC_E_BADARG
    assert fin(p, 8 * D * (4 + T) - 8, D, T, out, out, None) == L.HMC_E_BADARG
    assert fin(p, nb, 0, T, out, out, None) == L.HMC_E_BADARG
    assert fin(p, nb, D, 0, out, out, None) == L.HMC_E_BADARG
    assert fin(p, nb, D, T, None, out, None) == L.HMC_E_BADARG


def _ar1(rng, Nchain, N, D, phi, offset):
    x = np.zeros((Nchain, N, D))
    x[:, 0] = rng.standard_normal((Nchain, D)) / np.sqrt(1 - phi ** 2)
    for t in range(1, N):
        x[:, t] = phi * x[:, t - 1] + rng.standard_normal((Nchain, D))
    return x + offset


def ref_cut_at(x, T):
    """utils.py:107-157 in float64 numpy, with the variogram read only up to lag T: (R, n_eff, truncated)."""
    n, m, std_j, mean_j, halves = O.rhat_moments(x, 1, 0)
    W = std_j.mean(0)
    B = np.sum((mean_j - mean_j.mean(0)) ** 2, 0) * n / float(m - 1)
    var = W * (n - 1) / float(n) + B / float(n)
    R = np.sqrt(var / W)
    D = x.shape[2]
    n_eff, trunc = np.zeros(D), np.zeros(D, dtype=bool)
    for i in range(D):
        def rho(t):
            return 1. - np.sum((halves[:, t:, i] - halves[:, :-t, i]) ** 2) / float(m * (n - t)) / (2 * var[i])
        if rho(1) < 1e-2:
            sum_rho = 0
        else:
            rho_t = [rho(1), rho(2)]
            t = 1
            while t < n - 2:
                if t + 2 > T:
                    trunc[i] = True
                    break
                rho_t.append(rho(t + 2))
                if ((t % 2) == 1) & ((rho_t[t] + rho_t[t + 1]) < 0):
                    break
                t += 1
            sum_rho = max(0.0, np.sum(rho_t[:t]))
        n_eff[i] = m * n / (1 + 2 * sum_rho)
    return R, n_eff, trunc


def _finish_from_numpy(x, T):
    """utils._stats_from_partials fed the partial sums hmc_diag_stream_finish returns (computed here in numpy), lags capped at T."""
    import torch
    import utils as U
    n, m, std_j, mean_j, halves = O.rhat_moments(x, 1, 0)
    D = x.shape[2]
    c = halves[0, 0]
    mom = np.stack([std_j.sum(0), (mean_j - c).sum(0), ((mean_j - c) ** 2).sum(0), c])
    lags = np.stack([np.sum((halves[:, t:] - halves[:, :-t]) ** 2, axis=(0, 1)) for t in range(1, T + 1)])

    def moments_fn(buf):
        buf[:4] = torch.from_numpy(mom)
        nl = min(T, buf.shape[0] - U.ROW_LAGS)
        buf[U.ROW_LAGS:U.ROW_LAGS + nl] = torch.from_numpy(lags[:nl])
        return nl

    def all_lags_fn(buf):
        buf.copy_(torch.from_numpy(lags))

    info = {}
    R, ne = U._stats_from_partials(moments_fn, None, n, D, m, group=False, device=torch.device("cpu"), all_lags_fn=all_lags_fn,
                                   max_lag=T, info=info)
    return R, ne, info["n_eff_truncated"]


@pytest.mark.parametrize("T", [2, 5, 17, 40, 70, 119])
def test_host_finishing_with_max_lag_equals_restatement_cut_at_T(T):
    rng = np.random.RandomState(T)
    parts = [_ar1(rng, 6, 241, 3, phi, off) for phi, off in [(0.5, 0.0), (0.95, 1e3), (0.99, 0.0), (-0.3, 0.0)]]
    x = np.concatenate(parts, axis=2)                                            # n = 120
    R, ne, tr = _finish_from_numpy(x, T)
    R_ref, ne_ref, tr_ref = ref_cut_at(x, T)
    np.testing.assert_array_equal(tr, tr_ref)
    np.testing.assert_allclose(R, R_ref, rtol=1e-12)
    np.testing.assert_allclose(ne, ne_ref, rtol=1e-12)
    R_full, ne_full = O.convergence_stats(x, 1, 0)
    np.testing.assert_allclose(R, R_full, rtol=1e-12)
    np.testing.assert_allclose(ne[~tr], ne_full[~tr], rtol=1e-12)                # closed before T: the full computation
    if T <= 5:
        assert tr[6:9].all()                                                     # phi = 0.99 never closes this early
    if T == 119:
        assert not tr.any()
        np.testing.assert_allclose(ne, ne_full, rtol=1e-12)


def _final_iteration(j, Niter, warm, thin):
    return min(warm + (j + 1) * thin - 1, Niter) if j > 0 or warm + thin - 1 > 0 else 0


@pytest.mark.parametrize("thin", [1, 3])
@pytest.mark.parametrize("warm", [0, 1, 7])
@pytest.mark.parametrize("Niter_extra", [0, 1, 2, 5])
@pytest.mark.parametrize("per_block", [1, 2, 7, 64])
def test_stream_blocks_hand_over_each_sample_once_after_its_window_closes(thin, warm, Niter_extra, per_block):
    import samplers as S
    Niter = warm + 40 * thin + Niter_extra
    Lc = 1 + (Niter - warm) // thin
    blocks = S.stream_blocks(Niter, warm, thin, per_block)
    assert blocks[0][0] == 0 and blocks[-1][1] == Niter
    handed = []
    for k, (b, e, j0, j1) in enumerate(blocks):
        assert b <= e and j0 < j1
        if k:
            assert b == blocks[k - 1][1] and b < e and j0 == blocks[k - 1][3]
        handed += list(range(j0, j1))
        for j in range(j0, j1):                                   # final once iteration e has run ...
            assert _final_iteration(j, Niter, warm, thin) <= e
        # ... and the block writes only its own indices (what the kernels write at iterations (b, e]; index 0 at iteration 0)
        written = {(it - warm) // thin for it in range(b + 1, e + 1) if it >= warm} | ({0} if b == 0 else set())
        assert written <= set(range(j0, j1)), (written, j0, j1)
        if k:
            assert j1 - j0 <= per_block
    assert handed == list(range(Lc))
    assert (Lc - 1) % 2 in (0, 1)


def test_stream_blocks_odd_and_even_used_counts():
    import samplers as S
    for Niter in (40, 41):
        blocks = S.stream_blocks(Niter, 0, 1, 8)
        assert blocks[-1][3] == Niter + 1                         # every stored index, the dropped odd one included
