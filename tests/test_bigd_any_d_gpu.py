"""Large-D path at dimensions that are not multiples of 256 (csrc/random_bigd.cu works on Dp = D rounded up to 32, with a narrow
last column tile when BN does not divide Dp): against the float64 oracle, against the generic kernel on the same Philox draws,
shard invariance, the stored-sample ring, dispatch and sampling statistics.

Column tiles at the D used here (fp16x2: BN = 256, bf16x3: BN = 128; last tile width in brackets):
  D =  300  Dp =  320  fp16x2 2 tiles (64)   bf16x3 3 tiles (64)
  D =  777  Dp =  800  fp16x2 4 tiles (32)   bf16x3 7 tiles (32)    D % 4 != 0: the caller's rows are not 16-byte aligned
  D = 1200  Dp = 1216  fp16x2 5 tiles (192)  bf16x3 10 tiles (64)
  D = 1283  Dp = 1312  fp16x2 6 tiles (32)   bf16x3 11 tiles (32)
Tolerances as in tests/test_bigd_gpu.py: rel-L2 1e-5 for L < 20 on a well-conditioned target, 2e-3 for L in [20, 60) with a
log-uniform spectrum on [0.05, 100]."""
import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu


def _dense_target(D, seed, lam_lo=0.05, lam_hi=100.0):
    rng = np.random.RandomState(seed)
    lam = np.exp(rng.uniform(np.log(lam_lo), np.log(lam_hi), D))           # log-uniform spectrum
    Qm, _ = np.linalg.qr(rng.standard_normal((D, D)))                       # random rotation
    cov = (Qm * lam) @ Qm.T
    cov = 0.5 * (cov + cov.T)
    return O.MVNTarget(rng.standard_normal(D) * 0.5, cov), lam


def _spec(tgt):
    import samplers as S
    return S.MVNSpec(tgt.q0, tgt.inv_cov0, tgt.const)


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3"])
@pytest.mark.parametrize("D,B,Llo,Lhi,lam_lo,lam_hi,tol", [(300, 300, 5, 20, 0.5, 20.0, 1e-5), (777, 300, 5, 20, 0.5, 20.0, 1e-5),
                                                          (1283, 200, 20, 60, 0.05, 100.0, 2e-3)])
def test_bigd_any_d_teacher_forced_against_oracle(D, B, Llo, Lhi, lam_lo, lam_hi, tol, prec):
    import samplers as S
    tgt, _ = _dense_target(D, 7, lam_lo, lam_hi)
    rng = np.random.RandomState(11)
    q_init = (tgt.q0 + rng.standard_normal((B, D)) @ np.linalg.cholesky(tgt.cov0).T).astype(np.float32).astype(float)
    p = rng.standard_normal((B, D)).astype(np.float32).astype(float)
    L = rng.randint(Llo, Lhi, size=B).astype(np.int32)
    u = rng.random_sample(B)
    want = O.one_iteration_batch(tgt, q_init, p, L, u, 0.1)
    p_tape = np.zeros((B, 2, D))
    p_tape[:, 1] = p
    H = S.HMC_sampler(D, None, None, Nchain=B, Niter=1, sampler_type="Random", dt=0.1, L_low=Llo, L_high=Lhi, dtype="float32",
                      kernel="bigd", tc_precision=prec, target=_spec(tgt),
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
    assert rel.max() < tol, "worst rel-L2 trajectory error %.3g" % rel.max()
    np.testing.assert_allclose(H.E_chain[:, 1, 0], want["E_init"], rtol=1e-4, atol=1e-2)
    assert H.sum_L == int(L.sum())
    assert H.N_total_steps == B * 3 + D * int((L.astype(np.int64) ** 2).sum())


@pytest.mark.parametrize("D", [300, 777])
def test_bigd_any_d_free_running_matches_generic_kernel(D):
    """Philox draws (the last slot of a D % 4 != 0 row partly used), warm-up, thinning, iteration blocks (resume through
    state_q), chain_id0 != 0: same draws as the generic float32 kernel => same trajectory lengths, matching stored samples,
    energies and acceptance.  Momentum in a padded dimension would show in the energies."""
    import samplers as S
    Nchain, Niter = 500, 13
    tgt, _ = _dense_target(D, 3, 0.5, 20.0)
    q_start = (tgt.q0 + np.random.RandomState(5).standard_normal((Nchain, D)) * 1.5).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, thin_rate=2, warm_up_num=3, sampler_type="Random", dt=0.12, L_low=4, L_high=11,
              dtype="float32", seed=21, target=_spec(tgt), chain_id0=1000)
    F = S.HMC_sampler(D, None, None, kernel="bigd", iter_block=4, **kw)
    F.gen_sample(q_start, verbose=False, quiet=True)
    G = S.HMC_sampler(D, None, None, kernel="generic", **kw)
    G.gen_sample(q_start, verbose=False, quiet=True)
    assert F.sum_L == G.sum_L and F.N_total_steps == G.N_total_steps
    assert F.q_chain.shape == G.q_chain.shape == (Nchain, 1 + (Niter - 3) // 2, D)
    amp = np.linalg.norm(q_start.astype(float) - tgt.q0, axis=1)
    rel0 = np.linalg.norm(F.q_chain[:, 0] - G.q_chain[:, 0], axis=1) / amp
    assert np.quantile(rel0, 0.98) < 1e-4
    rel_last = np.linalg.norm(F.q_chain[:, -1] - G.q_chain[:, -1], axis=1) / amp
    assert np.mean(rel_last < 1e-3) > 0.9
    assert abs(F.accept_R - G.accept_R) < 2e-2 and abs(F.accept_R_warm_up - G.accept_R_warm_up) < 2e-2
    same = rel_last < 1e-3
    np.testing.assert_allclose(F.E_chain[same, :, 0], G.E_chain[same, :, 0], rtol=2e-4, atol=2e-3)
    np.testing.assert_allclose(F.dE_chain[same, 1:, 0], G.dE_chain[same, 1:, 0], rtol=0, atol=2e-3)

    # chain-0 trace (only the shard that owns chain 0 records it)
    kw0 = dict(kw, Nchain=130, Niter=5, thin_rate=1, warm_up_num=0, chain_id0=0)
    F0 = S.HMC_sampler(D, None, None, kernel="bigd", **kw0)
    F0.gen_sample(q_start[:130], N_save_chain0=4, verbose=False, quiet=True)
    G0 = S.HMC_sampler(D, None, None, kernel="generic", **kw0)
    G0.gen_sample(q_start[:130], N_save_chain0=4, verbose=False, quiet=True)
    assert [len(x) for x in F0.phi_q] == [len(x) for x in G0.phi_q]
    np.testing.assert_allclose(np.concatenate(F0.phi_q), np.concatenate(G0.phi_q), rtol=0, atol=2e-4)
    np.testing.assert_array_equal(F0.decision_chain, G0.decision_chain)
    assert F0.sum_L == G0.sum_L


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3"])
def test_bigd_narrow_last_tile_full_grid_equals_its_own_shards(prec):
    """16,384 chains at D = 1200 (last column tile 192 columns wide for fp16x2, 64 for bf16x3) are several rounds of work items per
    persistent CTA; every 1,024-chain shard with the same global chain ids must reproduce its rows bit for bit.  A race between
    the column tiles of one row block (operand buffers, partial energy sums) would break this."""
    import samplers as S
    D, Nchain, Niter = 1200, 16384, 2
    tgt, _ = _dense_target(D, 4, 0.2, 30.0)
    q_start = (tgt.q0 + np.random.RandomState(8).standard_normal((Nchain, D)) * 2.0).astype(np.float32)
    kw = dict(Niter=Niter, thin_rate=1, warm_up_num=0, sampler_type="Random", dt=0.1, L_low=30, L_high=60, dtype="float32", seed=4,
              target=_spec(tgt), kernel="bigd", tc_precision=prec)
    F = S.HMC_sampler(D, None, None, Nchain=Nchain, **kw)
    F.gen_sample(q_start, verbose=False, quiet=True)
    full_q, full_E = F.q_chain, F.E_chain
    assert np.all(np.isfinite(full_q))
    assert F.accept_R > 0.5
    for lo in (0, 8192 + 128, Nchain - 1024):
        Sh = S.HMC_sampler(D, None, None, Nchain=1024, chain_id0=lo, **kw)
        Sh.gen_sample(q_start[lo:lo + 1024], verbose=False, quiet=True)
        np.testing.assert_array_equal(Sh.q_chain, full_q[lo:lo + 1024])
        np.testing.assert_array_equal(Sh.E_chain, full_E[lo:lo + 1024])


def test_bigd_store_ring_at_d_not_multiple_of_4():
    """store_ring = R at D = 777: the ring rows equal the full run's last R stored samples bit for bit (the stored rows are 777
    floats wide and written without 16-byte accesses)."""
    import torch
    import hmc_b200_lib as L
    import samplers as S
    D, Nchain, Niter, warm, thin, R = 777, 300, 31, 4, 2, 5
    tgt, _ = _dense_target(D, 12, 0.5, 20.0)
    q_start = (tgt.q0 + np.random.RandomState(D).standard_normal((Nchain, D)) * 1.2).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=3, L_high=9,
              dtype="float32", seed=41, target=_spec(tgt), kernel="bigd")
    F = S.HMC_sampler(D, None, None, **kw)
    F.gen_sample(q_start, verbose=False, quiet=True)
    Lc = F.L_chain
    assert Lc > R + 2
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
    for j in range(Lc - R, Lc):
        np.testing.assert_array_equal(qr[:, j % R], F.q_chain[:, j].astype(np.float32))
        np.testing.assert_array_equal(Er[:, j % R], F.E_chain[:, j, 0])
        np.testing.assert_array_equal(dEr[:, j % R], F.dE_chain[:, j, 0])


@pytest.mark.parametrize("D,other", [(1500, "bigd"), (300, "generic")])
def test_bigd_auto_dispatch(D, other):
    """AUTO takes the large-D path for D > 1024 (D = 1500 ran nowhere before) and keeps the generic kernel for 128 < D <= 1024
    when D % 256 != 0: either way it equals the kernel it picks, bit for bit."""
    import samplers as S
    Nchain, Niter = 256, 3
    tgt, _ = _dense_target(D, 9, 0.5, 20.0)
    q_start = (tgt.q0 + np.random.RandomState(6).standard_normal((Nchain, D))).astype(np.float32)
    kw = dict(Nchain=Nchain, Niter=Niter, sampler_type="Random", dt=0.1, L_low=3, L_high=8, dtype="float32", seed=2, target=_spec(tgt))
    A = S.HMC_sampler(D, None, None, kernel="auto", **kw)
    A.gen_sample(q_start, verbose=False, quiet=True)
    B = S.HMC_sampler(D, None, None, kernel=other, tc_precision=A.tc_precision, **kw)
    B.gen_sample(q_start, verbose=False, quiet=True)
    assert A.tc_precision == ("fp16x2" if other == "bigd" else "bf16x3")
    np.testing.assert_array_equal(A.q_chain, B.q_chain)
    np.testing.assert_array_equal(A.E_chain, B.E_chain)
    assert A.sum_L == B.sum_L and A.accept_R == B.accept_R


@pytest.mark.parametrize("D,dtype,dense,why", [(127, "float32", False, r"D must be in \[128, 8192\]"),
                                               (8193, "float32", False, r"D must be in \[128, 8192\]"),
                                               (300, "float64", False, "float32 only"),
                                               (300, "float32", True, "identity momentum metric only")])
def test_bigd_rejects_what_it_does_not_cover(D, dtype, dense, why):
    import hmc_b200_lib as L
    import samplers as S
    spec = S.MVNSpec(np.zeros(D), np.eye(D), 0.0)
    cov_p = S.equicorrelated_cov(D, 0.3) if dense else None
    H = S.HMC_sampler(D, None, None, Nchain=4, Niter=1, sampler_type="Random", dt=0.1, L_low=2, L_high=4, cov_p=cov_p,
                      dtype=dtype, kernel="bigd", target=spec)
    with pytest.raises(L.HMCError, match="large-D kernel does not cover this configuration: " + why) as e:
        H.gen_sample(np.zeros((4, D)), verbose=False, quiet=True)
    assert e.value.code == L.HMC_E_UNSUPPORTED


def test_bigd_statistics_at_d_1500():
    """Sampling statistics at D = 1500 (a dimension only the large-D path runs): chains start in the target, so every stored
    sample is a draw.  Per-dimension means within 5 sigma_MC of the target mean, with sigma_MC^2 = var / n_eff from the run's own
    split-chain ESS; per-dimension variances within 5 % of the target's diagonal (the estimator's own spread at this n_eff is
    below 1 %)."""
    import torch
    import samplers as S
    import utils as U
    D, Nchain, Niter = 1500, 8192, 21
    tgt, _ = _dense_target(D, 21, 0.5, 2.0)
    q_start = U.start_pts(tgt.q0, tgt.cov0, Nchain, device="cuda", seed=3)
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, sampler_type="Random", dt=0.2, L_low=8, L_high=16,
                      dtype="float32", seed=17, target=_spec(tgt), kernel="auto")
    H.gen_sample(q_start, verbose=False, quiet=True)
    assert H.tc_precision == "fp16x2"
    assert H.accept_R > 0.7
    H.compute_convergence_stats()
    n_eff = np.asarray(H.n_eff_q, dtype=float)
    assert np.all(np.isfinite(H.R_q)) and np.all(n_eff > 0)
    assert np.median(n_eff) > 0.1 * Nchain * (Niter)
    mean, var = U.device_moments(H.q_chain_device[:, 1:, :])
    torch.cuda.synchronize()
    want_var = np.diag(tgt.cov0)
    z = (mean - tgt.q0) / np.sqrt(want_var / n_eff)
    assert np.abs(z).max() < 5.0, "worst mean deviation %.2f sigma_MC" % np.abs(z).max()
    ratio = var / want_var
    assert np.abs(ratio - 1).max() < 0.05, "variance ratio in [%.4f, %.4f]" % (ratio.min(), ratio.max())
