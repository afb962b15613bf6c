"""Streamed diagnostics on the GPU (csrc/diag_stream.cu): R_q and n_eff_q from a ring of the last stored samples equal the full
stream's, through the C-ABI on synthetic AR(1) streams and end to end through HMC_sampler(stream_stats=T) on every Random kernel.

Tolerances are test_diag_gpu.py's: R_q to rtol 1e-9 (float64) / 1e-6 (float32), n_eff_q to 1e-8 / 2e-4."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import hmc_oracle as O
from test_stream_stats_cpu import ref_cut_at

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"float64": (1e-9, 1e-8), "float32": (1e-6, 2e-4)}


def _ar1_stream(D, Nchain, Lc, seed):
    """AR(1) chains, phi cycling over 0.5 / 0.95 / 0.99 by dimension, an offset of 1e3 on every fourth dimension."""
    rng = np.random.RandomState(seed)
    phi = np.array([0.5, 0.95, 0.99])[np.arange(D) % 3]
    x = np.zeros((Nchain, Lc, D))
    x[:, 0] = rng.standard_normal((Nchain, D)) / np.sqrt(1 - phi ** 2)
    for t in range(1, Lc):
        x[:, t] = phi * x[:, t - 1] + rng.standard_normal((Nchain, D))
    x[:, :, ::4] += 1e3
    return x


def _stream(lib_, x_dev, T, block, R=None):
    """Feed x_dev [Nchain][Lc][D] through a ring of R = T + block rows, `block` stored indices per update; returns the workspace."""
    import torch
    import hmc_b200_lib as L
    Nc, Lc, D = x_dev.shape
    R = T + block if R is None else R
    ring = torch.full((Nc, R, D), float("nan"), dtype=x_dev.dtype, device=x_dev.device)
    nb = int(lib_.hmc_diag_stream_workspace_bytes(Nc, D, T))
    ws = torch.full((nb // 8,), float("nan"), dtype=torch.float64, device=x_dev.device)
    dt = L.HMC_F32 if x_dev.dtype == torch.float32 else L.HMC_F64
    for j0 in range(0, Lc, block):
        j1 = min(j0 + block, Lc)
        for j in range(j0, j1):
            ring[:, j % R] = x_dev[:, j]
        L.check(lib_.hmc_diag_stream_update(dt, L.ptr(ring), Nc, D, R, Lc, T, j0, j1, L.ptr(ws), nb, L.current_stream_ptr()))
    return ws, nb


def _finish(ws, nb, D, T, Lc, Nc):
    import utils as U
    return U.stream_stats_from_workspace(ws.data_ptr(), nb, D, T, Lc, Nc, group=False, device=ws.device)


CABI_CASES = [(1, "float64", 1), (1, "float32", 7), (6, "float64", 7), (6, "float32", 64), (100, "float64", 64),
              (100, "float32", 1), (777, "float32", 7), (777, "float64", 64), (1024, "float32", 64), (1024, "float64", 7)]


@pytest.mark.parametrize("D,dtype,block", CABI_CASES)
def test_cabi_stream_equals_full_stream(D, dtype, block):
    import torch
    import hmc_b200_lib as L
    import utils as U
    Nc, Lc = 24, 2 * 150 + 1 + (D % 2)           # n = 150; odd and even L_chain - 1
    x = _ar1_stream(D, Nc, Lc, seed=D)
    tdt = torch.float64 if dtype == "float64" else torch.float32
    x_dev = torch.from_numpy(x).to("cuda", tdt)
    x_used = x_dev.double().cpu().numpy()[:, 1:]
    n = (Lc - 1) // 2
    R_full, ne_full = U.convergence_stats(x_dev[:, 1:], thin_rate=1, warm_up_num=0, group=False)
    _, t_used = O.finish_from_variogram(*_var_and_table(x_used))
    rt_R, rt_n = TOL[dtype]
    # T at least the truncation lag of every dimension: the full stream's numbers
    T = int(min(n - 1, t_used.max() + 1))
    ws, nb = _stream(L.load(), x_dev, T, block)
    R, ne, tr = _finish(ws, nb, D, T, Lc, Nc)
    assert not tr.any()
    np.testing.assert_allclose(R, R_full, rtol=rt_R)
    np.testing.assert_allclose(ne, ne_full, rtol=rt_n)
    # T below it: the restatement cut at T, with the flag set where the rule had not stopped
    T = 6
    ws, nb = _stream(L.load(), x_dev, T, block)
    R, ne, tr = _finish(ws, nb, D, T, Lc, Nc)
    R_ref, ne_ref, tr_ref = ref_cut_at(x_used, T)
    np.testing.assert_array_equal(tr, tr_ref)
    assert tr[2::3].all()                                         # phi = 0.99 does not close by lag 6
    np.testing.assert_allclose(R, R_ref, rtol=rt_R)
    np.testing.assert_allclose(ne, ne_ref, rtol=rt_n)


def _var_and_table(x):
    n, m, std_j, mean_j, halves = O.rhat_moments(x, 1, 0)
    W = std_j.mean(0)
    B = np.sum((mean_j - mean_j.mean(0)) ** 2, 0) * n / float(m - 1)
    var = W * (n - 1) / float(n) + B / float(n)
    V = np.full((n + 1, x.shape[2]), np.nan)
    for t in range(1, n):
        V[t] = np.sum((halves[:, t:] - halves[:, :-t]) ** 2, axis=(0, 1)) / float(m * (n - t))
    return var, V, m, n


def test_cabi_block_sizes_agree_and_ring_of_exactly_T_plus_block():
    """Different update block sizes give the same sums (to float64 reordering); R = T + (j1 - j0) exactly is enough."""
    import torch
    import hmc_b200_lib as L
    D, Nc, Lc, T = 37, 16, 201, 40
    x_dev = torch.from_numpy(_ar1_stream(D, Nc, Lc, seed=5)).to("cuda", torch.float64)
    outs = []
    for block in (1, 3, 64, Lc):
        ws, nb = _stream(L.load(), x_dev, T, block, R=T + block)
        outs.append(_finish(ws, nb, D, T, Lc, Nc))
    for R, ne, _ in outs[1:]:
        np.testing.assert_allclose(R, outs[0][0], rtol=1e-12)
        np.testing.assert_allclose(ne, outs[0][1], rtol=1e-12)


def _mvn(D, rho, seed):
    import samplers as S
    mu = np.random.RandomState(seed).standard_normal(D)
    return S.MVNSpec.from_cov(mu, O.equicorrelated_cov(D, rho))


def _run(D, kernel, dtype, stream_stats=None, Nchain=256, Niter=250, warm=10, thin=2, cov_p=None, tc_precision=None, iter_block=None,
         chain_id0=0, q_start=None, seed=11):
    import samplers as S
    spec = _mvn(D, 0.6, D)
    if q_start is None:
        q_start = spec.mu + 1.2 * np.random.RandomState(D + 1).standard_normal((Nchain, D))
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=3,
                      L_high=9, dtype=dtype, seed=seed, target=spec, kernel=kernel, cov_p=cov_p, tc_precision=tc_precision,
                      iter_block=iter_block, chain_id0=chain_id0, stream_stats=stream_stats)
    H.gen_sample(q_start, verbose=False, quiet=True)
    H.compute_convergence_stats()
    return H


E2E = [("tc", 100, "float32", None, None), ("fast", 64, "float32", None, None), ("generic", 33, "float64", "dense", None),
       ("generic", 33, "float32", "dense", None), ("bigd", 777, "float32", None, "fp16x2"), ("bigd", 777, "float32", None, "bf16x3"),
       ("bigd", 1024, "float32", None, "fp16x2"), ("bigd", 1024, "float32", None, "bf16x3"), ("bigd", 1283, "float32", "dense", None)]


@pytest.mark.parametrize("kernel,D,dtype,metric,prec", E2E)
def test_sampler_stream_stats_equal_full_run(kernel, D, dtype, metric, prec):
    cov_p = O.equicorrelated_cov(D, 0.3) if metric == "dense" else None
    kw = dict(cov_p=cov_p, tc_precision=prec)
    # warm-up 1, thin 2, 15 stored samples per block: the streamed run's blocks end at iterations 30, 60, ..., as the full run's
    # iter_block=30 launches do, so both runs make the same launches (the tensor-core kernel hands chains over between launches in
    # float32 and is not bit-identical across different launch boundaries)
    F = _run(D, kernel, dtype, warm=1, iter_block=30, **kw)
    n = (F.L_chain - 1) // 2
    H = _run(D, kernel, dtype, stream_stats=n - 1, warm=1, iter_block=30, **kw)
    assert [b[1] for b in H._stream["blocks"]] == [min(e, 250) for e in range(30, 271, 30)]
    assert H._stream["R"] == n - 1 + 15 and H._stream["R"] < F.L_chain
    assert H.accept_R == F.accept_R and H.sum_L == F.sum_L
    rt_R, rt_n = TOL[dtype]
    assert not H.n_eff_truncated.any()
    np.testing.assert_allclose(H.R_q, F.R_q, rtol=rt_R)
    np.testing.assert_allclose(H.n_eff_q, F.n_eff_q, rtol=rt_n)


def test_sampler_iteration_block_sizes_give_the_same_statistics():
    runs = [_run(33, "generic", "float64", stream_stats=40, iter_block=b) for b in (None, 2, 13, 400)]
    for H in runs[1:]:
        np.testing.assert_allclose(H.R_q, runs[0].R_q, rtol=1e-12)
        np.testing.assert_allclose(H.n_eff_q, runs[0].n_eff_q, rtol=1e-12)
        np.testing.assert_array_equal(H.n_eff_truncated, runs[0].n_eff_truncated)


def test_two_shards_combined_on_the_host_equal_one_shard(monkeypatch):
    """chain_id0 = 0 and Nc, each streamed on its own, combined by the host path of a two-rank run (torch.distributed's collectives
    stood in for by the other shard's partial sums) == one shard of 2 Nc chains."""
    import torch
    import torch.distributed as dist
    import hmc_b200_lib as L
    import utils as U
    D, Nc, T = 33, 128, 40
    spec = _mvn(D, 0.6, D)
    qs = spec.mu + 1.2 * np.random.RandomState(3).standard_normal((2 * Nc, D))
    one = _run(D, "generic", "float64", stream_stats=T, Nchain=2 * Nc, q_start=qs)
    A = _run(D, "generic", "float64", stream_stats=T, Nchain=Nc, q_start=qs[:Nc])
    B = _run(D, "generic", "float64", stream_stats=T, Nchain=Nc, q_start=qs[Nc:], chain_id0=Nc)
    mom_B = torch.empty((4, D), dtype=torch.float64, device="cuda")
    lags_B = torch.empty((T, D), dtype=torch.float64, device="cuda")
    L.check(L.load().hmc_diag_stream_finish(C.c_void_p(B._stream["ws_ptr"]), B._stream["ws_bytes"], D, T, L.ptr(mom_B), L.ptr(lags_B),
                                            L.current_stream_ptr()))

    def all_gather_into_tensor(out, buf, group=None):
        rows = buf.shape[0]
        other = torch.zeros_like(buf)
        other[:4] = mom_B
        other[U.ROW_COUNT, 0] = 2 * Nc
        nl = min(T, rows - U.ROW_LAGS)
        other[U.ROW_LAGS:U.ROW_LAGS + nl] = lags_B[:nl]
        out[:rows] = buf
        out[rows:] = other

    def all_reduce(t, group=None):
        assert t.shape == lags_B.shape
        t += lags_B

    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    monkeypatch.setattr(dist, "all_gather_into_tensor", all_gather_into_tensor)
    monkeypatch.setattr(dist, "all_reduce", all_reduce)
    A.distributed = True
    A.compute_convergence_stats()
    np.testing.assert_allclose(A.R_q, one.R_q, rtol=1e-9)
    np.testing.assert_allclose(A.n_eff_q, one.n_eff_q, rtol=1e-8)


def test_stream_mode_refuses_the_full_stream_views_and_nuts():
    import samplers as S
    H = _run(33, "generic", "float32", stream_stats=20, Niter=120)
    for what in ("q_chain", "E_chain", "dE_chain", "q_chain_device"):
        with pytest.raises(RuntimeError, match="stream_stats"):
            getattr(H, what)
    with pytest.raises(RuntimeError, match="stream_stats"):
        H.sample_summary()
    with pytest.raises(AssertionError, match="stream_stats"):
        S.HMC_sampler(10, None, None, Nchain=4, Niter=100, sampler_type="NUTS", dt=0.1, target=_mvn(10, 0.5, 1), stream_stats=10)
    with pytest.raises(AssertionError, match="stream_stats"):
        S.HMC_sampler(10, None, None, Nchain=4, Niter=100, sampler_type="Random", dt=0.1, L_low=3, L_high=5, target=_mvn(10, 0.5, 1),
                      stream_stats=50)                          # T > n - 1 = 49


def test_stream_stats_none_is_the_plain_run():
    """stream_stats=None runs the full-storage path unchanged: its q_chain / E_chain equal a direct C-ABI run of the same arguments in
    one launch, bit for bit, and nothing streamed is allocated."""
    import torch
    import hmc_b200_lib as L
    import samplers as S
    F = _run(100, "tc", "float32", Niter=60)
    assert F._stream is None and F.n_eff_truncated is None
    H = S.HMC_sampler(100, None, None, Nchain=256, Niter=60, thin_rate=2, warm_up_num=10, sampler_type="Random", dt=0.1, L_low=3,
                      L_high=9, dtype="float32", seed=11, target=_mvn(100, 0.6, 100), kernel="tc")
    q_start = H.target.mu + 1.2 * np.random.RandomState(101).standard_normal((256, 100))
    run = H.prepare_random(q_start)
    a = run["args"]
    assert a.store_ring == 0
    a.iter_begin, a.iter_end = 0, 60
    L.check(L.load().hmc_random_run(a, L.current_stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(H.q_chain, F.q_chain)
    np.testing.assert_array_equal(H.E_chain, F.E_chain)


def test_debug_build_bounds_at_the_largest_dimension(tmp_path):
    """The update's ring, window and state indices are checked by device asserts in a build of csrc/diag_stream.cu with
    HMC_DIAG_STREAM_DEBUG; D = 8192, 1,024 chains, a ring of exactly T + 1 rows (one stored index per update), both dtypes, and the
    result equals the release library's."""
    import torch
    import hmc_b200_lib as L
    csrc = os.path.join(ROOT, "understanding-hmc_b200", "csrc")
    stub = tmp_path / "err.cu"
    stub.write_text('#include <cstdio>\n#include <cstdarg>\nstatic char msg[512];\nvoid hmc_set_error(const char* f, ...) '
                    '{ va_list a; va_start(a, f); vsnprintf(msg, sizeof msg, f, a); va_end(a); }\n')
    so = tmp_path / "libdiag_stream_debug.so"
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    subprocess.check_call([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared",
                           "-DHMC_DIAG_STREAM_DEBUG", os.path.join(csrc, "diag_stream.cu"), str(stub), "-o", str(so)])
    dbg = C.CDLL(str(so))
    rel = L.load()
    for f in ("hmc_diag_stream_workspace_bytes", "hmc_diag_stream_update", "hmc_diag_stream_finish"):
        getattr(dbg, f).argtypes, getattr(dbg, f).restype = getattr(rel, f).argtypes, getattr(rel, f).restype
    D, Nc, Lc, T = 8192, 1024, 2 * 24 + 1, 20
    for tdt in (torch.float32, torch.float64):
        x_dev = torch.from_numpy(_ar1_stream(D, Nc, Lc, seed=8)).to("cuda", tdt)
        ws_d, nb = _stream(dbg, x_dev, T, 1)
        torch.cuda.synchronize()
        ws_r, _ = _stream(rel, x_dev, T, 1)
        got, want = _finish(ws_d, nb, D, T, Lc, Nc), _finish(ws_r, nb, D, T, Lc, Nc)
        np.testing.assert_allclose(got[0], want[0], rtol=1e-12)
        np.testing.assert_allclose(got[1], want[1], rtol=1e-12)
        del x_dev, ws_d, ws_r
        torch.cuda.empty_cache()
