"""NUTS on the large-D path with a ring of stored samples (hmc_nuts_args.store_ring = R, csrc/nuts_bigd.cu): through the C-ABI the
ring's rows equal the matching stored indices of a full-storage run bit for bit, and end to end HMC_sampler(sampler_type="NUTS",
stream_stats=T) gives the full run's R_q and n_eff_q.

The C-ABI runs keep L_chain rows per chain of NaN behind the ring, so that a stored index that misses the wrap lands in the buffer
(and fails the comparison) rather than past its end.  Statistics tolerances are test_stream_stats_gpu.py's for float32."""
import numpy as np
import pytest

from test_nuts_bigd_gpu import _dense_target, _spec

pytestmark = pytest.mark.gpu

RT_R, RT_N = 1e-6, 2e-4


def _cabi(tgt, q_start, Niter, warm, thin, R=0, ends=None, prec="bf16x3", chain_id0=0, kernel="bigd", draws=None, seed=5, dt=0.25,
          d_max=10):
    """One hmc_nuts_run per iteration block (block ends `ends`, default one launch); returns the outputs as numpy arrays, the
    stored-sample arrays with R rows per chain (L_chain when R = 0) and the area behind them."""
    import torch
    import hmc_b200_lib as L
    import samplers as S
    lib = L.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    Nc, D = q_start.shape
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="NUTS", dt=dt,
                      d_max=d_max, target=_spec(tgt))
    t, keep, _ = H._build_target(torch, dev)
    Lc = H.L_chain
    rows = R if R else Lc
    nan = float("nan")
    q = torch.full((Nc * Lc * D,), nan, dtype=torch.float32, device=dev)
    E = torch.full((Nc * Lc,), nan, dtype=torch.float64, device=dev)
    dE = torch.full((Nc * Lc,), nan, dtype=torch.float64, device=dev)
    qs = torch.from_numpy(np.ascontiguousarray(q_start, dtype=np.float32)).to(dev)
    state_q = torch.empty((Nc, D), dtype=torch.float32, device=dev)
    state_e = torch.zeros((Nc,), dtype=torch.float64, device=dev)
    counters = torch.zeros((4,), dtype=torch.int64, device=dev)
    status = torch.zeros((Nc,), dtype=torch.int32, device=dev)
    nleap = torch.zeros((Nc,), dtype=torch.int64, device=dev)
    scratch = torch.zeros((Nc + 128, 2 * (d_max + 1) + 7, t.D_pad), dtype=torch.float32, device=dev)
    a = L.NutsArgs()
    a.dtype, a.kernel, a.Nchain, a.d_max, a.chain_id0 = L.HMC_F32, L.KERNELS[kernel], Nc, d_max, chain_id0
    a.Niter, a.warm_up_num, a.thin_rate, a.on_dmax, a.seed = Niter, warm, thin, 1, seed
    a.target = t
    a.q_start = qs.data_ptr()
    if draws is not None:
        keep["tapes"] = [torch.from_numpy(np.ascontiguousarray(draws[k])).to(dev) for k in ("p_tape", "dir_tape", "u_tape")]
        a.p_tape, a.dir_tape, a.u_tape = (x.data_ptr() for x in keep["tapes"])
        a.tape_dir_stride, a.tape_u_stride = draws["dir_tape"].shape[1], draws["u_tape"].shape[1]
    a.q_chain, a.E_chain, a.dE_chain, a.store_ring = q.data_ptr(), E.data_ptr(), dE.data_ptr(), R
    a.state_q, a.state_eprev = state_q.data_ptr(), state_e.data_ptr()
    a.scratch, a.counters, a.status, a.n_leapfrog = scratch.data_ptr(), counters.data_ptr(), status.data_ptr(), nleap.data_ptr()
    a.flags = L.FLAG_TC_FP16X2 if prec == "fp16x2" else 0
    nbytes = int(lib.hmc_nuts_workspace_bytes(a))
    ws, a.workspace = L.aligned_workspace(torch, dev, nbytes)
    a.workspace_bytes = nbytes
    edges = [0] + list(ends or [Niter])
    for b, e in zip(edges[:-1], edges[1:]):
        a.iter_begin, a.iter_end = b, e
        L.check(lib.hmc_nuts_run(a, L.current_stream_ptr()))
    torch.cuda.synchronize()
    qn, En, dEn = q.cpu().numpy(), E.cpu().numpy(), dE.cpu().numpy()
    return dict(q=qn[:Nc * rows * D].reshape(Nc, rows, D), E=En[:Nc * rows].reshape(Nc, rows), dE=dEn[:Nc * rows].reshape(Nc, rows),
                behind=(qn[Nc * rows * D:], En[Nc * rows:], dEn[Nc * rows:]), nleap=nleap.cpu().numpy(), status=status.cpu().numpy(),
                counters=counters.cpu().numpy(), Lc=Lc)


def _assert_ring_equals_full(ring, full, R):
    """Row j % R of the ring == stored index j of the full run for every j in [L_chain - R, L_chain); the area behind the ring is
    untouched; the per-chain records and counters are the full run's."""
    Lc = full["Lc"]
    assert 0 < R < Lc
    for j in range(Lc - R, Lc):
        np.testing.assert_array_equal(ring["q"][:, j % R], full["q"][:, j], err_msg="q, stored index %d" % j)
        np.testing.assert_array_equal(ring["E"][:, j % R], full["E"][:, j], err_msg="E, stored index %d" % j)
        np.testing.assert_array_equal(ring["dE"][:, j % R], full["dE"][:, j], err_msg="dE, stored index %d" % j)
    for x in ring["behind"]:
        assert np.isnan(x).all()
    for k in ("nleap", "status", "counters"):
        np.testing.assert_array_equal(ring[k], full[k])


def _start(tgt, Nc, seed):
    return (tgt.q0 + np.random.RandomState(seed).standard_normal((Nc, tgt.q0.shape[0]))).astype(np.float32)


@pytest.mark.parametrize("thin", [1, 3])
@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("D", [300, 777])
def test_ring_rows_equal_the_full_run(D, prec, thin):
    """D = 300 (Dp = 320) and D = 777 (rows not 16-byte aligned: the scalar store path); warm-up 2, chain ids from 4242, 200 chains
    (padding rows in the last row block); the ring in one launch and in iteration blocks that end inside a thin window."""
    Niter, warm = 14, 2
    tgt = _dense_target(D, 5, 0.5, 10.0)
    qs = _start(tgt, 200, D)
    kw = dict(prec=prec, chain_id0=4242)
    full = _cabi(tgt, qs, Niter, warm, thin, **kw)
    R = 5 if thin == 1 else 3                              # L_chain = 13 / 5
    _assert_ring_equals_full(_cabi(tgt, qs, Niter, warm, thin, R=R, **kw), full, R)
    _assert_ring_equals_full(_cabi(tgt, qs, Niter, warm, thin, R=R, ends=[3, 7, 8, 14], **kw), full, R)


def test_ring_rows_equal_the_full_run_on_injected_tapes():
    D, Nc, Niter, warm = 300, 64, 9, 1
    tgt = _dense_target(D, 5, 0.5, 10.0)
    qs = _start(tgt, Nc, 9)
    rng = np.random.RandomState(9)
    draws = dict(p_tape=rng.standard_normal((Nc, Niter + 1, D)), dir_tape=rng.randint(0, 2, size=(Nc, 10 * Niter)).astype(np.int32),
                 u_tape=rng.random_sample((Nc, 3000)))
    full = _cabi(tgt, qs, Niter, warm, 1, draws=draws)
    _assert_ring_equals_full(_cabi(tgt, qs, Niter, warm, 1, R=4, draws=draws, ends=[2, 5, 9]), full, 4)


def test_ring_of_l_chain_rows_is_the_full_layout_and_auto_takes_the_large_d_path_from_d_128():
    """store_ring = L_chain writes what store_ring = 0 writes; with store_ring > 0 AUTO runs the large-D path at D = 200 (where it
    keeps the generic kernel otherwise), bit for bit as kernel "bigd"."""
    tgt = _dense_target(300, 5, 0.5, 10.0)
    qs = _start(tgt, 130, 1)
    full = _cabi(tgt, qs, 8, 1, 2)
    same = _cabi(tgt, qs, 8, 1, 2, R=full["Lc"])
    for k in ("q", "E", "dE", "nleap", "status", "counters"):
        np.testing.assert_array_equal(same[k], full[k])
    tgt = _dense_target(200, 6, 0.5, 10.0)
    qs = _start(tgt, 130, 2)
    bigd = _cabi(tgt, qs, 10, 1, 1, R=4, kernel="bigd")
    auto = _cabi(tgt, qs, 10, 1, 1, R=4, kernel="auto")
    for k in ("q", "E", "dE", "nleap", "status", "counters"):
        np.testing.assert_array_equal(auto[k], bigd[k])
    assert not np.isnan(auto["q"]).any()


def test_two_shards_equal_one_run_of_both():
    """chain_id0 = 0 and Nc, each with its own ring, equal the matching rows of one run of 2 Nc chains bit for bit."""
    D, Nc = 300, 160
    tgt = _dense_target(D, 5, 0.5, 10.0)
    qs = _start(tgt, 2 * Nc, 4)
    one = _cabi(tgt, qs, 10, 2, 1, R=3)
    for lo in (0, Nc):
        sh = _cabi(tgt, qs[lo:lo + Nc], 10, 2, 1, R=3, chain_id0=lo)
        for k in ("q", "E", "dE", "nleap", "status"):
            np.testing.assert_array_equal(sh[k], one[k][lo:lo + Nc])


def _run(D, stream_stats=None, Nchain=256, Niter=120, warm=10, thin=1, prec=None, iter_block=None, kernel="auto", dt=0.25, d_max=10,
         on_dmax="stop", target=None, q_start=None, seed=3):
    import samplers as S
    tgt = _dense_target(D, 5, 0.5, 10.0) if target is None else target
    qs = _start(tgt, Nchain, D) if q_start is None else q_start
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="NUTS", dt=dt,
                      d_max=d_max, dtype="float32", seed=seed, target=_spec(tgt), kernel=kernel, tc_precision=prec, on_dmax=on_dmax,
                      iter_block=iter_block, stream_stats=stream_stats)
    H.gen_sample(qs, verbose=False)
    H.compute_convergence_stats()
    return H


@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("D", [300, 1024])
def test_sampler_stream_stats_equal_full_run(D, prec):
    F = _run(D, prec=prec)
    n = (F.L_chain - 1) // 2
    H = _run(D, stream_stats=n - 1, prec=prec, iter_block=30)      # blocks of 30 stored samples: a ring of T + 30 < L_chain rows
    assert H.nuts_kernel == "bigd" and F.nuts_kernel == "bigd"
    assert H._stream["R"] < F.L_chain and len(H._stream["blocks"]) > 1
    assert not H.n_eff_truncated.any()
    np.testing.assert_array_equal(H.n_leapfrog, F.n_leapfrog)
    assert H.N_total_steps == F.N_total_steps and H.n_doublings == F.n_doublings
    np.testing.assert_allclose(H.R_q, F.R_q, rtol=RT_R)
    np.testing.assert_allclose(H.n_eff_q, F.n_eff_q, rtol=RT_N)


def test_sampler_iteration_block_sizes_give_the_same_statistics():
    runs = [_run(300, stream_stats=40, Niter=110, iter_block=b) for b in (None, 7, 30)]
    for H in runs[1:]:
        np.testing.assert_array_equal(H.n_leapfrog, runs[0].n_leapfrog)
        np.testing.assert_allclose(H.R_q, runs[0].R_q, rtol=RT_R)
        np.testing.assert_allclose(H.n_eff_q, runs[0].n_eff_q, rtol=RT_N)
        np.testing.assert_array_equal(H.n_eff_truncated, runs[0].n_eff_truncated)


def test_stream_mode_views_raise_and_auto_at_d_200_runs_the_large_d_path():
    H = _run(200, stream_stats=20, Niter=60)
    assert H.nuts_kernel == "bigd"
    for what in ("q_chain", "E_chain", "dE_chain", "q_chain_device"):
        with pytest.raises(RuntimeError, match="stream_stats"):
            getattr(H, what)
    with pytest.raises(RuntimeError, match="stream_stats"):
        H.sample_summary()
    assert np.all(np.isfinite(H.R_q)) and np.all(H.n_eff_q > 0)


def test_dmax_assert_after_a_streamed_run_and_stop_gives_finite_statistics():
    """dt = 1e-3 never turns within d_max = 3: "assert" still raises after the streamed run, "stop" finishes with finite R_q."""
    kw = dict(Nchain=128, Niter=9, warm=0, dt=1e-3, d_max=3)
    with pytest.raises(AssertionError):
        _run(300, stream_stats=2, on_dmax="assert", **kw)
    H = _run(300, stream_stats=2, **kw)
    assert H.n_dmax == 128 * 9 and np.all(H.status == 1)
    assert np.all(np.isfinite(H.R_q))
