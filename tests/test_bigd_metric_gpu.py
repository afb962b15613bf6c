"""Large-D Random path with a dense momentum metric (cov_p != I) for 1024 < D <= 8192 (csrc/random_bigd.cu: V, K and p = Lc z as
batched tensor-core products at the trajectory ends): against the float64 oracle on tapes and on the device's own Philox draws,
iteration blocks, determinism, the stored-sample ring, shard invariance, D = 8192, sampling statistics, dispatch and refusals.

The metric is a dense SPD matrix: the identity with a few eigenvalues in [0.7, 1.4] along random directions.  The reference moves
q by p, not by M^-1 p (quirk Q9), so the energy error of a trajectory grows with the metric's distance from I; with this one the
oracle accepts 60-80 % at dt = 0.1-0.2 and D ~ 1500."""
import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu


def _dense_target(D, seed, lam_lo=0.5, lam_hi=20.0):
    rng = np.random.RandomState(seed)
    lam = np.exp(rng.uniform(np.log(lam_lo), np.log(lam_hi), D))           # log-uniform spectrum
    Qm, _ = np.linalg.qr(rng.standard_normal((D, D)))                       # random rotation
    cov = (Qm * lam) @ Qm.T
    cov = 0.5 * (cov + cov.T)
    return O.MVNTarget(rng.standard_normal(D) * 0.5, cov)


def _cov_p(D, seed, k=4, lo=0.7, hi=1.4):
    rng = np.random.RandomState(seed)
    Vk, _ = np.linalg.qr(rng.standard_normal((D, k)))
    lam = np.exp(rng.uniform(np.log(lo), np.log(hi), k))
    c = np.eye(D) + (Vk * (lam - 1.0)) @ Vk.T
    return 0.5 * (c + c.T)


def _spec(tgt):
    import samplers as S
    return S.MVNSpec(tgt.q0, tgt.inv_cov0, tgt.const)


def _energy(tgt, inv_cov_p, q, p):
    d = q - tgt.q0
    return 0.5 * np.einsum("bi,bi->b", d, d @ tgt.inv_cov0.T) + tgt.const + 0.5 * np.einsum("bi,bi->b", p, p @ inv_cov_p.T)


def _philox(seed, chain_id0, Nchain, Niter, D, Llo, Lhi):
    import torch
    import hmc_b200_lib as L
    z = torch.zeros((Nchain, Niter + 1, D), dtype=torch.float64, device="cuda")
    Lt = torch.zeros((Nchain, Niter), dtype=torch.int32, device="cuda")
    u = torch.zeros((Nchain, Niter), dtype=torch.float64, device="cuda")
    L.check(L.load().hmc_philox_draws(seed, chain_id0, Nchain, Niter, D, Llo, Lhi, L.ptr(z), L.ptr(Lt), L.ptr(u), L.current_stream_ptr()))
    torch.cuda.synchronize()
    return z.cpu().numpy(), Lt.cpu().numpy(), u.cpu().numpy()


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3"])
@pytest.mark.parametrize("D,B,vec_dt", [(1283, 200, True), (1283, 200, False), (2048, 256, False), (2048, 256, True)])
def test_dense_metric_teacher_forced_against_oracle(D, B, vec_dt, prec):
    import samplers as S
    tgt = _dense_target(D, 7)
    cov_p = _cov_p(D, 3)
    Lc = np.linalg.cholesky(cov_p)
    rng = np.random.RandomState(11)
    q_init = (tgt.q0 + rng.standard_normal((B, D)) @ np.linalg.cholesky(tgt.cov0).T).astype(np.float32).astype(float)
    p0 = (rng.standard_normal((B, D)) @ Lc.T).astype(np.float32).astype(float)
    p = (rng.standard_normal((B, D)) @ Lc.T).astype(np.float32).astype(float)
    L = rng.randint(5, 20, size=B).astype(np.int32)
    u = rng.random_sample(B)
    dt = (0.1 * rng.uniform(0.8, 1.2, D)) if vec_dt else 0.1
    want = O.one_iteration_batch(tgt, q_init, p, L, u, dt, cov_p=cov_p)
    p_tape = np.stack([p0, p], axis=1)
    H = S.HMC_sampler(D, None, None, Nchain=B, Niter=1, sampler_type="Random", dt=dt, L_low=5, L_high=20, dtype="float32",
                      kernel="bigd", tc_precision=prec, target=_spec(tgt), cov_p=cov_p,
                      draws=dict(p_tape=p_tape, L_tape=L.reshape(B, 1), u_tape=u.reshape(B, 1)))
    H.gen_sample(q_init, verbose=False, quiet=True)
    got = H.q_chain[:, 1, :]
    np.testing.assert_array_equal(H.q_chain[:, 0, :], q_init)
    moved = np.linalg.norm(got - q_init, axis=1) > 1e-6 * np.linalg.norm(q_init - tgt.q0, axis=1)
    E_scale = np.maximum(1.0, np.abs(want["E_init"]))
    near_tie = (want["dE"] >= 0) & (np.abs(np.log(u) + want["dE"]) < 1e-4 * E_scale)
    differ = moved != (want["decision"] == 1)
    assert not np.any(differ & ~near_tie), "%d decision flips away from ties" % int(np.sum(differ & ~near_tie))
    acc = moved & ~differ
    assert acc.sum() > 0.5 * B
    amp = np.maximum(np.linalg.norm(want["q_prop"] - tgt.q0, axis=1), np.linalg.norm(q_init - tgt.q0, axis=1))
    rel = np.linalg.norm(got[acc] - want["q_prop"][acc], axis=1) / amp[acc]
    assert rel.max() < 1e-5, "worst rel-L2 trajectory error %.3g" % rel.max()
    E0 = _energy(tgt, np.linalg.inv(cov_p), q_init, p0)
    np.testing.assert_allclose(H.E_chain[:, 0, 0], E0, rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(H.E_chain[:, 1, 0], want["E_init"], rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(H.dE_chain[:, 1, 0], want["E_init"] - E0, rtol=1e-4, atol=1e-2)
    assert H.sum_L == int(L.sum())
    assert H.N_total_steps == B * 3 + D * int((L.astype(np.int64) ** 2).sum())


def test_dense_metric_free_running_against_oracle_on_device_draws():
    """The device's own Philox z (the oracle gets p = Lc z in float64), D = 1283 (the caller's rows are not 16-byte aligned),
    warm-up, thinning, chain_id0 != 0; then the chain-0 trace of a run that owns chain 0."""
    import samplers as S
    D, Nchain, Niter, warm, thin, Llo, Lhi, seed = 1283, 40, 7, 2, 2, 4, 11, 31
    tgt = _dense_target(D, 5, 0.5, 20.0)
    cov_p = _cov_p(D, 9)
    Lc = np.linalg.cholesky(cov_p)
    q_start = (tgt.q0 + np.random.RandomState(2).standard_normal((Nchain, D)) @ np.linalg.cholesky(tgt.cov0).T).astype(np.float32)
    kw = dict(Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=Llo, L_high=Lhi, dtype="float32",
              seed=seed, target=_spec(tgt), cov_p=cov_p, kernel="bigd", tc_precision="bf16x3")

    def oracle(c0, n, nsave=0):
        z, Lt, ut = _philox(seed, c0, n, Niter, D, Llo, Lhi)
        tape = []
        for m in range(n):
            tape.append(("p", z[m, 0] @ Lc.T))
            for i in range(Niter):
                tape += [("p", z[m, i + 1] @ Lc.T), ("i", int(Lt[m, i])), ("u", float(ut[m, i]))]
        R = O.gen_sample_random(D, tgt.V, tgt.dVdq, q_start[:n].astype(float), O.TapeDraws(tape), n, Niter, thin, warm, 0.1, Llo, Lhi,
                                cov_p=cov_p, N_save_chain0=nsave, record=True)
        R.u = ut
        return R

    F = S.HMC_sampler(D, None, None, Nchain=Nchain, chain_id0=500, **kw)
    F.gen_sample(q_start, verbose=False, quiet=True)
    R = oracle(500, Nchain)
    assert abs(F.accept_R - R.accept_R) < 0.02
    amp = np.linalg.norm(q_start.astype(float) - tgt.q0, axis=1)
    # the first stored sample (iteration warm + thin - 1) within 1e-4 for every chain, unless one of its decisions up to there was
    # a near-tie of the float64 oracle (a float32 energy may then decide the other way)
    rel0 = np.linalg.norm(F.q_chain[:, 0] - R.q_chain[:, 0], axis=1) / amp
    first = warm + thin - 1
    margin = np.abs(np.log(R.u[:, :first]) + R.dE_iter[:, :first])
    tie = np.any((R.dE_iter[:, :first] >= 0) & (margin < 5e-2), axis=1)
    assert np.all((rel0 < 1e-4) | tie), (rel0[~tie].max(), int(tie.sum()))
    assert np.mean(rel0 < 1e-4) > 0.9
    rel_last = np.linalg.norm(F.q_chain[:, -1] - R.q_chain[:, -1], axis=1) / amp
    same = rel_last < 1e-3
    assert np.mean(same) > 0.8
    np.testing.assert_allclose(F.E_chain[same, :, 0], R.E_chain[same, :, 0], rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(F.dE_chain[same, 1:, 0], R.dE_chain[same, 1:, 0], rtol=0, atol=2e-2)

    F0 = S.HMC_sampler(D, None, None, Nchain=4, chain_id0=0, **kw)
    F0.gen_sample(q_start[:4], N_save_chain0=5, verbose=False, quiet=True)
    R0 = oracle(0, 1, nsave=5)
    assert [len(x) for x in F0.phi_q] == [len(x) for x in R0.phi_q]
    np.testing.assert_allclose(np.concatenate(F0.phi_q), np.concatenate(R0.phi_q), rtol=0, atol=2e-4)
    np.testing.assert_array_equal(F0.decision_chain[:5], R0.decision_chain[:5])


@pytest.mark.parametrize("tapes", [False, True])
def test_dense_metric_iteration_blocks_determinism_and_ring(tapes):
    """iter_block launches equal one launch bit for bit (V(x0) is carried within a launch and recomputed on resume: the same x,
    re-derived from the stored float row, gives the same V); a repeat is bit-identical; the store_ring rows equal the full run's
    last R stored samples."""
    import torch
    import hmc_b200_lib as L
    import samplers as S
    D, Nchain, Niter, warm, thin, R = 1283, 300, 9, 2, 1, 3
    tgt = _dense_target(D, 12, 0.5, 20.0)
    cov_p = _cov_p(D, 4)
    q_start = (tgt.q0 + np.random.RandomState(7).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="Random", dt=0.12, L_low=3, L_high=9,
              dtype="float32", seed=41, target=_spec(tgt), cov_p=cov_p, kernel="bigd")
    if tapes:
        rng = np.random.RandomState(3)
        kw["draws"] = dict(p_tape=rng.standard_normal((Nchain, Niter + 1, D)) @ np.linalg.cholesky(cov_p).T,
                           L_tape=rng.randint(3, 9, size=(Nchain, Niter)).astype(np.int32), u_tape=rng.random_sample((Nchain, Niter)))
    runs = []
    for blk in (None, 4, None):
        H = S.HMC_sampler(D, None, None, iter_block=blk, **kw)
        H.gen_sample(q_start, verbose=False, quiet=True)
        runs.append(H)
    assert np.all(np.isfinite(runs[0].q_chain)) and runs[0].accept_R > 0.4
    for H in runs[1:]:
        np.testing.assert_array_equal(H.q_chain, runs[0].q_chain)
        np.testing.assert_array_equal(H.E_chain, runs[0].E_chain)
        np.testing.assert_array_equal(H.dE_chain, runs[0].dE_chain)
        assert H.accept_R == runs[0].accept_R and H.sum_L == runs[0].sum_L
    F = runs[0]
    H = S.HMC_sampler(D, None, None, **kw)
    run = H.prepare_random(q_start)
    a = run["args"]
    qr = torch.zeros((Nchain, R, D), dtype=torch.float32, device="cuda")
    Er = torch.zeros((Nchain, R), dtype=torch.float64, device="cuda")
    dEr = torch.zeros((Nchain, R), dtype=torch.float64, device="cuda")
    a.q_chain, a.E_chain, a.dE_chain, a.store_ring = qr.data_ptr(), Er.data_ptr(), dEr.data_ptr(), R
    a.iter_begin, a.iter_end = 0, Niter
    L.check(L.load().hmc_random_run(a, L.current_stream_ptr()))
    torch.cuda.synchronize()
    qr, Er, dEr = qr.cpu().numpy(), Er.cpu().numpy(), dEr.cpu().numpy()
    for j in range(F.L_chain - R, F.L_chain):
        np.testing.assert_array_equal(qr[:, j % R], F.q_chain[:, j].astype(np.float32))
        np.testing.assert_array_equal(Er[:, j % R], F.E_chain[:, j, 0])
        np.testing.assert_array_equal(dEr[:, j % R], F.dE_chain[:, j, 0])


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3"])
def test_dense_metric_full_grid_equals_its_own_shards(prec):
    """16,384 chains at D = 1100: many listed chains per pass in the product stage; every 1,024-chain shard with the same global
    chain ids reproduces its rows bit for bit.  A race between the product stage and the passes' operand rows would break this."""
    import samplers as S
    D, Nchain, Niter = 1100, 16384, 3
    tgt = _dense_target(D, 4, 0.5, 20.0)
    cov_p = _cov_p(D, 6)
    q_start = (tgt.q0 + np.random.RandomState(8).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Niter=Niter, thin_rate=1, warm_up_num=0, sampler_type="Random", dt=0.1, L_low=3, L_high=25, dtype="float32", seed=4,
              target=_spec(tgt), cov_p=cov_p, kernel="bigd", tc_precision=prec)
    F = S.HMC_sampler(D, None, None, Nchain=Nchain, **kw)
    F.gen_sample(q_start, verbose=False, quiet=True)
    full_q, full_E, full_dE = F.q_chain, F.E_chain, F.dE_chain
    assert np.all(np.isfinite(full_q))
    assert F.accept_R > 0.5
    for lo in (0, 8192 + 128, Nchain - 1024):
        Sh = S.HMC_sampler(D, None, None, Nchain=1024, chain_id0=lo, **kw)
        Sh.gen_sample(q_start[lo:lo + 1024], verbose=False, quiet=True)
        np.testing.assert_array_equal(Sh.q_chain, full_q[lo:lo + 1024])
        np.testing.assert_array_equal(Sh.E_chain, full_E[lo:lo + 1024])
        np.testing.assert_array_equal(Sh.dE_chain, full_dE[lo:lo + 1024])


def test_dense_metric_at_d_8192():
    """D = 8192 on tapes, two iterations: E_chain against V + K of the taped rows in float64 (iteration 2 starts where the first
    stored sample is), finite samples, a bit-identical repeat.  Equicorrelated target: its precision matrix in closed form."""
    import samplers as S
    D, Nchain, Niter, rho = 8192, 256, 2, 0.3
    mu = np.random.RandomState(1).standard_normal(D) * 0.5
    P = (np.eye(D) - rho / (1 - rho + rho * D) * np.ones((D, D))) / (1 - rho)
    const = 0.5 * (D * np.log(2 * np.pi) + (D - 1) * np.log(1 - rho) + np.log(1 - rho + rho * D))
    spec = S.MVNSpec(mu, P, const)
    cov_p = _cov_p(D, 2)
    inv_cov_p = np.linalg.inv(cov_p)
    rng = np.random.RandomState(5)
    p_tape = rng.standard_normal((Nchain, Niter + 1, D)) @ np.linalg.cholesky(cov_p).T
    L_tape = rng.randint(5, 12, size=(Nchain, Niter)).astype(np.int32)
    u_tape = rng.random_sample((Nchain, Niter))
    q_start = (mu + rng.standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, sampler_type="Random", dt=0.1, L_low=5, L_high=12, dtype="float32", target=spec,
              cov_p=cov_p, kernel="auto", draws=dict(p_tape=p_tape, L_tape=L_tape, u_tape=u_tape))
    runs = []
    for _ in range(2):
        H = S.HMC_sampler(D, None, None, **kw)
        H.gen_sample(q_start, verbose=False, quiet=True)
        runs.append(H)
    H = runs[0]
    assert np.all(np.isfinite(H.q_chain))
    np.testing.assert_array_equal(runs[1].q_chain, H.q_chain)
    np.testing.assert_array_equal(runs[1].E_chain, H.E_chain)

    def E(q, p):
        d = q - mu
        return 0.5 * np.einsum("bi,bi->b", d, d @ P) + const + 0.5 * np.einsum("bi,bi->b", p, p @ inv_cov_p)
    q0 = q_start.astype(float)
    np.testing.assert_allclose(H.E_chain[:, 0, 0], E(q0, p_tape[:, 0]), rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(H.E_chain[:, 1, 0], E(q0, p_tape[:, 1]), rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(H.E_chain[:, 2, 0], E(H.q_chain[:, 1], p_tape[:, 2]), rtol=1e-4, atol=1e-2)


def test_dense_metric_statistics_at_d_1500():
    """Chains start in the target, so every stored sample is a draw: per-dimension means within 5 sigma_MC (the run's own n_eff),
    variances within 5 % of the target's diagonal, finite Rhat / n_eff."""
    import torch
    import samplers as S
    import utils as U
    D, Nchain, Niter = 1500, 8192, 21
    tgt = _dense_target(D, 21, 0.5, 2.0)
    cov_p = _cov_p(D, 5)
    q_start = U.start_pts(tgt.q0, tgt.cov0, Nchain, device="cuda", seed=3)
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, sampler_type="Random", dt=0.1, L_low=8, L_high=16,
                      dtype="float32", seed=17, target=_spec(tgt), cov_p=cov_p, kernel="auto")
    H.gen_sample(q_start, verbose=False, quiet=True)
    assert H.tc_precision == "fp16x2"
    assert H.accept_R > 0.5
    H.compute_convergence_stats()
    n_eff = np.asarray(H.n_eff_q, dtype=float)
    assert np.all(np.isfinite(H.R_q)) and np.all(n_eff > 0)
    mean, var = U.device_moments(H.q_chain_device[:, 1:, :])
    torch.cuda.synchronize()
    want_var = np.diag(tgt.cov0)
    z = (mean - tgt.q0) / np.sqrt(want_var / n_eff)
    assert np.abs(z).max() < 5.0, "worst mean deviation %.2f sigma_MC" % np.abs(z).max()
    ratio = var / want_var
    assert np.abs(ratio - 1).max() < 0.05, "variance ratio in [%.4f, %.4f]" % (ratio.min(), ratio.max())


@pytest.mark.parametrize("D,other", [(1500, "bigd"), (1024, "generic")])
def test_dense_metric_auto_dispatch(D, other):
    """AUTO with a dense metric: the large-D path above D = 1024, the generic kernel at D = 1024; bit for bit what it picks."""
    import samplers as S
    Nchain, Niter = 256, 3
    tgt = _dense_target(D, 9, 0.5, 20.0)
    cov_p = _cov_p(D, 1)
    q_start = (tgt.q0 + np.random.RandomState(6).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, sampler_type="Random", dt=0.1, L_low=3, L_high=8, dtype="float32", seed=2, target=_spec(tgt),
              cov_p=cov_p)
    A = S.HMC_sampler(D, None, None, kernel="auto", **kw)
    A.gen_sample(q_start, verbose=False, quiet=True)
    B = S.HMC_sampler(D, None, None, kernel=other, tc_precision=A.tc_precision, **kw)
    B.gen_sample(q_start, verbose=False, quiet=True)
    assert A.tc_precision == ("fp16x2" if other == "bigd" else "bf16x3")
    np.testing.assert_array_equal(A.q_chain, B.q_chain)
    np.testing.assert_array_equal(A.E_chain, B.E_chain)
    assert A.sum_L == B.sum_L and A.accept_R == B.accept_R


def test_dense_metric_refusals():
    import torch
    import hmc_b200_lib as L
    import samplers as S
    D = 1500
    spec = S.MVNSpec(np.zeros(D), np.eye(D), 0.0)
    cov_p = _cov_p(D, 8)
    kw = dict(Nchain=4, Niter=1, sampler_type="Random", dt=0.1, L_low=2, L_high=4, cov_p=cov_p, kernel="bigd")
    # D = 1024 belongs to the generic kernel
    spec1k = S.MVNSpec(np.zeros(1024), np.eye(1024), 0.0)
    H = S.HMC_sampler(1024, None, None, dtype="float32", target=spec1k, **dict(kw, cov_p=_cov_p(1024, 8)))
    with pytest.raises(L.HMCError, match="large-D kernel does not cover this configuration: identity momentum metric only") as e:
        H.gen_sample(np.zeros((4, 1024)), verbose=False, quiet=True)
    assert e.value.code == L.HMC_E_UNSUPPORTED
    # float64
    H = S.HMC_sampler(D, None, None, dtype="float64", target=spec, **kw)
    with pytest.raises(L.HMCError, match="float32 only") as e:
        H.gen_sample(np.zeros((4, D)), verbose=False, quiet=True)
    assert e.value.code == L.HMC_E_UNSUPPORTED
    # a partial matrix set
    H = S.HMC_sampler(D, None, None, dtype="float32", target=spec, **kw)
    run = H.prepare_random(np.zeros((4, D)))
    a = run["args"]
    a.target.Lct = None
    a.iter_begin, a.iter_end = 0, 1
    assert L.load().hmc_random_run(a, L.current_stream_ptr()) == L.HMC_E_UNSUPPORTED
    assert "Pt, Mit and Lct together" in L.load().hmc_last_error_string().decode()
    torch.cuda.synchronize()
    # NUTS keeps the identity metric on the large-D path
    H = S.HMC_sampler(D, None, None, Nchain=4, Niter=1, sampler_type="NUTS", dt=0.1, d_max=4, cov_p=cov_p, dtype="float32",
                      kernel="bigd", target=spec)
    with pytest.raises(L.HMCError, match="large-D NUTS kernel does not cover this configuration: identity momentum metric only") as e:
        H.gen_sample(np.zeros((4, D)), 0, False)
    assert e.value.code == L.HMC_E_UNSUPPORTED
