"""NUTS on the large-D GEMM path (csrc/nuts_bigd.cu): against the float64 oracle on injected tapes, against the generic NUTS kernel
on the same Philox draws, determinism and iteration blocks, shard invariance at full occupancy, d_max and guards, sampling
statistics at a dimension only this path runs, dispatch and rejections.

Tolerances are those of the tensor-core NUTS kernel's tests (tests/test_nuts_gpu.py): a float32 near-tie in a U-turn test or a
sampling uniform may change a tree, so tree agreement is a fraction of chains and samples are compared where the trees agree."""
import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu


def _dense_target(D, seed, lam_lo, lam_hi):
    """Log-uniform covariance spectrum on [lam_lo, lam_hi] with a random rotation; mean off zero."""
    rng = np.random.RandomState(seed)
    lam = np.exp(rng.uniform(np.log(lam_lo), np.log(lam_hi), D))
    Qm, _ = np.linalg.qr(rng.standard_normal((D, D)))
    cov = (Qm * lam) @ Qm.T
    cov = 0.5 * (cov + cov.T)
    return O.MVNTarget(rng.standard_normal(D) * 0.5, cov)


def _spec(tgt):
    import samplers as S
    return S.MVNSpec(tgt.q0, tgt.inv_cov0, tgt.const)


def _tapes(R, Nchain):
    """The oracle's recorded per-chain draws, padded to [Nchain][stride] (the kernels consume them in order per chain)."""
    nd = max(len(x) for x in R.dir_tape)
    nu = max(len(x) for x in R.u_tape)
    dirs = np.full((Nchain, nd), -1, dtype=np.int32)
    us = np.full((Nchain, nu), np.nan)
    for m in range(Nchain):
        dirs[m, :len(R.dir_tape[m])] = R.dir_tape[m]
        us[m, :len(R.u_tape[m])] = R.u_tape[m]
    return dict(p_tape=R.p_tape, dir_tape=dirs, u_tape=us)


@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("D", [300, 777, 1024])
def test_nuts_bigd_against_oracle_on_tapes(D, prec):
    """Teacher forced on the float64 oracle's own draws: the same trees (leapfrog count per chain) and, where they agree, the
    oracle's samples and energies to float32 accuracy.  D = 300: Dp = 320 (D % 32 != 0); D = 777: the caller's rows are not
    16-byte aligned."""
    import samplers as S
    Nchain, Niter, d_max, dt = 8, 4, 8, 0.25
    tgt = _dense_target(D, 7, 0.5, 10.0)
    rng = np.random.RandomState(D)
    q_start = (tgt.q0 + rng.standard_normal((Nchain, D)) @ np.linalg.cholesky(tgt.cov0).T).astype(np.float32).astype(float)
    np.random.seed(D + 1)
    R = O.gen_sample_NUTS(D, tgt.V, tgt.dVdq, q_start, O.NumpyDraws(D), Nchain, Niter, dt=dt, d_max=d_max, record=True,
                          on_dmax="stop")
    depth = R.depth
    assert depth.min() >= 3 and depth.max() <= 7, (depth.min(), depth.max())
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, sampler_type="NUTS", dt=dt, d_max=d_max, dtype="float32",
                      kernel="bigd", tc_precision=prec, target=_spec(tgt), on_dmax="stop", draws=_tapes(R, Nchain))
    H.gen_sample(q_start, verbose=False)
    assert H.nuts_kernel == "bigd" and H.tc_precision == prec
    want_leap = R.n_leapfrog.sum(axis=1)
    same = H.n_leapfrog == want_leap
    assert same.mean() >= 0.95, (H.n_leapfrog, want_leap)
    qs = np.abs(R.q_chain).max()
    np.testing.assert_allclose(H.q_chain[same], R.q_chain[same], rtol=0, atol=2e-4 * qs)
    np.testing.assert_allclose(H.E_chain[same], R.E_chain[same], rtol=2e-5, atol=2e-3)
    if same.all():
        assert H.N_total_steps == R.N_total_steps
    np.testing.assert_array_equal(H.q_chain[:, 0], q_start)


@pytest.mark.parametrize("D", [128, 200, 256])
def test_nuts_bigd_matches_generic_on_philox_draws(D):
    """Same position-keyed Philox draws as the warp-per-chain kernel (global chain ids from 4242): per chain the same number of
    leapfrog steps on > 97 % of chains, totals within 1 %, the same first stored sample, the same samples where the trees agree."""
    import samplers as S
    Nchain, Niter = 1500, 6
    tgt = _dense_target(D, 3, 0.5, 10.0)
    q_start = (tgt.q0 + np.random.RandomState(3).standard_normal((Nchain, D)) * 1.4).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, thin_rate=1, warm_up_num=0, sampler_type="NUTS", dt=0.25, d_max=10, dtype="float32",
              seed=11, target=_spec(tgt), on_dmax="stop", chain_id0=4242)
    T = S.HMC_sampler(D, None, None, kernel="bigd", **kw)
    T.gen_sample(q_start, verbose=False)
    G = S.HMC_sampler(D, None, None, kernel="generic", **kw)
    G.gen_sample(q_start, verbose=False)
    assert T.nuts_kernel == "bigd" and G.nuts_kernel == "generic"
    same = T.n_leapfrog == G.n_leapfrog
    assert same.mean() > 0.97, same.mean()
    assert abs(T.n_leapfrog_total / float(G.n_leapfrog_total) - 1.0) < 0.01
    assert T.n_doublings > 0 and abs(T.n_doublings / float(G.n_doublings) - 1.0) < 0.01
    np.testing.assert_array_equal(T.q_chain[:, 0], G.q_chain[:, 0])
    amp = np.linalg.norm(G.q_chain[:, -1] - tgt.q0, axis=1)
    rel = np.linalg.norm(T.q_chain[:, -1] - G.q_chain[:, -1], axis=1) / amp
    assert np.quantile(rel[same], 0.9) < 1e-3
    np.testing.assert_allclose(T.E_chain[same][:, 1, 0], G.E_chain[same][:, 1, 0], rtol=2e-5, atol=2e-3)
    assert T.n_instability == 0 and T.n_dmax == 0


def test_nuts_bigd_deterministic_and_iteration_blocks():
    """A repeated run is bit-identical; iteration blocks (resumed from state_q, state_eprev and the stream cursors) reproduce the
    single launch bit for bit, with a target mean off zero, on Philox draws and on injected tapes."""
    import samplers as S
    D, Nchain, Niter = 300, 600, 7
    tgt = _dense_target(D, 5, 0.5, 10.0)
    q_start = (tgt.q0 + np.random.RandomState(4).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, thin_rate=2, warm_up_num=2, sampler_type="NUTS", dt=0.25, d_max=10, dtype="float32",
              seed=5, target=_spec(tgt), kernel="bigd", chain_id0=77)
    A = S.HMC_sampler(D, None, None, **kw)
    A.gen_sample(q_start, verbose=False)
    A2 = S.HMC_sampler(D, None, None, **kw)
    A2.gen_sample(q_start, verbose=False)
    B = S.HMC_sampler(D, None, None, iter_block=3, **kw)
    B.gen_sample(q_start, verbose=False)
    for X in (A2, B):
        np.testing.assert_array_equal(X.q_chain, A.q_chain)
        np.testing.assert_array_equal(X.E_chain, A.E_chain)
        np.testing.assert_array_equal(X.dE_chain, A.dE_chain)
        np.testing.assert_array_equal(X.n_leapfrog, A.n_leapfrog)
        assert X.n_doublings == A.n_doublings
    # injected tapes: the cursors carry the streams over the block boundaries
    Nt = 64
    rng = np.random.RandomState(9)
    draws = dict(p_tape=rng.standard_normal((Nt, Niter + 1, D)), dir_tape=rng.randint(0, 2, size=(Nt, 10 * Niter)).astype(np.int32),
                 u_tape=rng.random_sample((Nt, 2000)))
    kt = dict(kw, Nchain=Nt, chain_id0=0, draws=draws)
    C = S.HMC_sampler(D, None, None, **kt)
    C.gen_sample(q_start[:Nt], verbose=False)
    Cb = S.HMC_sampler(D, None, None, iter_block=2, **kt)
    Cb.gen_sample(q_start[:Nt], verbose=False)
    np.testing.assert_array_equal(Cb.q_chain, C.q_chain)
    np.testing.assert_array_equal(Cb.E_chain, C.E_chain)
    np.testing.assert_array_equal(Cb.n_leapfrog, C.n_leapfrog)


def test_nuts_bigd_full_grid_run_equals_its_own_shards():
    """16,384 chains at D = 512: several rounds of work items per persistent CTA in every pass; each 1,024-chain shard with the
    same global chain ids reproduces its rows bit for bit.  A race in the gradient epilogue or the step kernel would break this."""
    import samplers as S
    D, Nchain, Niter = 512, 16384, 2
    tgt = _dense_target(D, 4, 0.2, 10.0)
    q_start = (tgt.q0 + np.random.RandomState(8).standard_normal((Nchain, D)) * 2.0).astype(np.float32)
    kw = dict(Niter=Niter, thin_rate=1, warm_up_num=0, sampler_type="NUTS", dt=0.2, d_max=8, dtype="float32", seed=4,
              target=_spec(tgt), kernel="bigd", on_dmax="stop")
    F = S.HMC_sampler(D, None, None, Nchain=Nchain, **kw)
    F.gen_sample(q_start, verbose=False)
    assert np.all(np.isfinite(F.q_chain)) and F.n_leapfrog.min() > 0
    for lo in (0, 8192 + 128, Nchain - 1024):
        Sh = S.HMC_sampler(D, None, None, Nchain=1024, chain_id0=lo, **kw)
        Sh.gen_sample(q_start[lo:lo + 1024], verbose=False)
        np.testing.assert_array_equal(Sh.q_chain, F.q_chain[lo:lo + 1024])
        np.testing.assert_array_equal(Sh.E_chain, F.E_chain[lo:lo + 1024])
        np.testing.assert_array_equal(Sh.n_leapfrog, F.n_leapfrog[lo:lo + 1024])


def test_nuts_bigd_dmax_assert_and_stop():
    """samplers.py:596-598: dt = 1e-3 never turns within d_max = 3 doublings: "assert" raises, "stop" keeps the live point after
    1 + 2 + 4 leapfrog steps per iteration; the per-chain counts add up to the total."""
    import samplers as S
    D, Nchain, Niter = 300, 200, 3
    tgt = _dense_target(D, 2, 0.5, 10.0)
    q_start = (tgt.q0 + np.random.RandomState(1).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, sampler_type="NUTS", dt=1e-3, d_max=3, dtype="float32", seed=1, target=_spec(tgt),
              kernel="bigd")
    H = S.HMC_sampler(D, None, None, **kw)
    with pytest.raises(AssertionError):
        H.gen_sample(q_start, verbose=False)
    H2 = S.HMC_sampler(D, None, None, on_dmax="stop", **kw)
    H2.gen_sample(q_start, verbose=False)
    assert H2.n_dmax == Nchain * Niter and np.all(H2.status == 1)
    assert H2.n_leapfrog_total == Nchain * Niter * 7
    assert int(H2.n_leapfrog.sum()) == H2.n_leapfrog_total


def test_nuts_bigd_statistics_at_d_1500():
    """D = 1500 (no other NUTS kernel runs it), a dense target with a log-uniform spectrum and a random rotation, 8,192 chains
    started in the target: per-dimension mean and standard deviation from sample_summary() within Monte-Carlo error (independent
    chains bound it), no instabilities, finite Rhat and n_eff."""
    import samplers as S
    import utils as U
    D, Nchain, Niter, warm = 1500, 8192, 6, 2
    tgt = _dense_target(D, 21, 0.5, 2.0)
    q_start = U.start_pts(tgt.q0, tgt.cov0, Nchain, device="cuda", seed=3)
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, warm_up_num=warm, sampler_type="NUTS", dt=0.3, d_max=10,
                      dtype="float32", seed=17, target=_spec(tgt), kernel="auto", on_dmax="stop")
    H.gen_sample(q_start, verbose=False)
    assert H.nuts_kernel == "bigd" and H.tc_precision == "bf16x3"
    assert H.n_instability == 0 and H.n_dmax == 0
    s = H.sample_summary()
    sd = np.sqrt(np.diag(tgt.cov0))
    z = (s["q_mean"] - tgt.q0) / (sd / np.sqrt(Nchain))
    assert np.abs(z).max() < 5.5, "worst mean deviation %.2f sigma" % np.abs(z).max()
    ratio = np.sqrt(s["q_var"]) / sd
    assert np.abs(ratio - 1).max() < 0.06, "std ratio in [%.4f, %.4f]" % (ratio.min(), ratio.max())
    H.compute_convergence_stats()
    assert np.all(np.isfinite(H.R_q)) and np.all(np.isfinite(H.n_eff_q)) and np.all(H.n_eff_q > 0)


@pytest.mark.parametrize("D,want", [(300, "bigd"), (1500, "bigd"), (100, "tc"), (200, "generic")])
def test_nuts_bigd_auto_dispatch(D, want):
    """AUTO: the tensor-core kernel at D = 100, the generic kernel up to D = 256, the large-D path above; each equals the kernel it
    names, bit for bit."""
    import samplers as S
    Nchain, Niter = 256, 3
    tgt = _dense_target(D, 9, 0.5, 5.0)
    q_start = (tgt.q0 + np.random.RandomState(6).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, sampler_type="NUTS", dt=0.25, d_max=10, dtype="float32", seed=2, target=_spec(tgt),
              on_dmax="stop")
    A = S.HMC_sampler(D, None, None, kernel="auto", **kw)
    A.gen_sample(q_start, verbose=False)
    assert A.nuts_kernel == want
    B = S.HMC_sampler(D, None, None, kernel=want, **kw)
    B.gen_sample(q_start, verbose=False)
    np.testing.assert_array_equal(A.q_chain, B.q_chain)
    np.testing.assert_array_equal(A.n_leapfrog, B.n_leapfrog)


@pytest.mark.parametrize("D,dtype,dense,kernel,why", [
    (300, "float64", False, "auto", "float32 only"),
    (300, "float32", True, "auto", "identity momentum metric only"),
    (8193, "float32", False, "auto", r"D must be in \[128, 8192\]"),
    (300, "float64", False, "bigd", "float32 only"),
    (100, "float32", False, "bigd", r"D must be in \[128, 8192\]")])
def test_nuts_bigd_rejects_what_it_does_not_cover(D, dtype, dense, kernel, why):
    import hmc_b200_lib as L
    import samplers as S
    spec = S.MVNSpec(np.zeros(D), np.eye(D), 0.0)
    cov_p = S.equicorrelated_cov(D, 0.3) if dense else None
    H = S.HMC_sampler(D, None, None, Nchain=4, Niter=1, sampler_type="NUTS", dt=0.1, d_max=3, cov_p=cov_p, dtype=dtype,
                      kernel=kernel, target=spec)
    with pytest.raises(L.HMCError, match=why) as e:
        H.gen_sample(np.zeros((4, D)), verbose=False)
    assert e.value.code == L.HMC_E_UNSUPPORTED
