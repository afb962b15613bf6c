"""The NUTS kernels against the float64 oracle on the tree builder's rare branches (tests/_nuts_edge_cases.py): instability
rejects, overflowing and mid-range weights, sub-trajectory U-turns, the depth limit, d_max = 12; every case with a target mean
off zero, per-dimension step sizes, warm-up and thinning, on the oracle's recorded draws.  Then the generic kernels with a dense
momentum metric: NUTS on oracle tapes, the random-trajectory sampler on its own Philox draws in every shared-memory staging regime.

Tolerances are the established ones.  float64 generic kernel: the whole stream to 1e-9 of the largest |q| and every counter
exactly (tests/test_nuts_gpu.py::test_f64_nuts_matches_reference).  float32 kernels: the same tree (leapfrog count) on >= 95 % of
chains, and where the trees agree the samples to 2e-4 max|q| and the energies to rtol 2e-5 / atol 2e-3
(tests/test_nuts_bigd_gpu.py::test_nuts_bigd_against_oracle_on_tapes); the two cases whose energy is ill-conditioned in q take
a measured rtol (Case.e_rtol in tests/_nuts_edge_cases.py)."""
import numpy as np
import pytest

import _nuts_edge_cases as C
from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu

TC_REPS = 33        # the tensor-core kernel runs every oracle chain 33 times: 264 chains, three 128-chain CTAs


def _spec(tgt):
    import samplers as S
    return S.MVNSpec(tgt.q0, tgt.inv_cov0, tgt.const)


def _tapes(c, idx):
    """The oracle's recorded per-chain draws for kernel chain i = oracle chain idx[i], padded with -1 / NaN to the most an
    iteration can consume (d_max coins, 2^d_max - 1 uniforms): a kernel that builds a different tree reads padding, never
    another chain's draws or past the buffer."""
    R = c.oracle
    nd, nu = c.Niter * c.d_max, c.Niter * ((1 << c.d_max) - 1)
    dirs = np.full((len(idx), nd), -1, dtype=np.int32)
    us = np.full((len(idx), nu), np.nan)
    for i, m in enumerate(idx):
        dirs[i, :len(R.dir_tape[m])] = R.dir_tape[m]
        us[i, :len(R.u_tape[m])] = R.u_tape[m]
    return dict(p_tape=R.p_tape[idx], dir_tape=dirs, u_tape=us)


def _run(c, dtype, kernel, reps=1, **over):
    import samplers as S
    idx = np.arange(c.Nchain * reps) % c.Nchain
    kw = dict(Nchain=len(idx), Niter=c.Niter, thin_rate=c.thin, warm_up_num=c.warm, sampler_type="NUTS", dt=c.dt, d_max=c.d_max,
              cov_p=c.cov_p, dtype=dtype, kernel=kernel, target=_spec(c.tgt), on_dmax=c.on_dmax, draws=_tapes(c, idx))
    kw.update(over)
    H = S.HMC_sampler(c.D, None, None, **kw)
    H.gen_sample(c.q_start[idx], verbose=False)
    return H, idx


def _check_f64(c, H, idx):
    R = c.oracle
    qs = max(1.0, np.abs(R.q_chain).max())
    es = max(1.0, np.abs(R.E_chain).max())
    np.testing.assert_allclose(H.q_chain, R.q_chain[idx], rtol=0, atol=1e-9 * qs)
    np.testing.assert_allclose(H.E_chain, R.E_chain[idx], rtol=0, atol=1e-9 * es)
    np.testing.assert_allclose(H.dE_chain, R.dE_chain[idx], rtol=0, atol=1e-9 * es)
    np.testing.assert_array_equal(H.n_leapfrog, R.n_leapfrog.sum(axis=1)[idx])
    np.testing.assert_array_equal(H.status, R.dmax_iter.any(axis=1)[idx].astype(np.int32))
    assert (H.N_total_steps, H.n_instability, H.n_dmax) == (R.N_total_steps, R.n_instability, R.n_dmax)


def _check_f32(c, H, idx):
    """The float32 rule; the instability and depth-limit counts equal the oracle's when every tree agrees, and otherwise
    differ by at most one per iteration of the chains whose trees differ."""
    R = c.oracle
    want = R.n_leapfrog.sum(axis=1)[idx]
    same = H.n_leapfrog == want
    assert same.mean() >= 0.95, (H.n_leapfrog, want)
    qs = np.abs(R.q_chain).max()
    np.testing.assert_allclose(H.q_chain[same], R.q_chain[idx][same], rtol=0, atol=2e-4 * qs)
    np.testing.assert_allclose(H.E_chain[same], R.E_chain[idx][same], rtol=c.e_rtol, atol=2e-3)
    n_inst = int(R.n_instab_iter.sum(axis=1)[idx].sum())
    n_dmax = int(R.dmax_iter.sum(axis=1)[idx].sum())
    slack = c.Niter * int((~same).sum())
    assert abs(H.n_instability - n_inst) <= slack and abs(H.n_dmax - n_dmax) <= slack, \
        (H.n_instability, n_inst, H.n_dmax, n_dmax, slack)
    if same.all():
        assert H.N_total_steps == len(idx) * (1 + c.Niter) + (c.D + 1) * int(want.sum())


def _reps_agree(H, c):
    """Replicated chains (same start point, same draws, other CTAs) give bit-identical results."""
    n = c.Nchain
    for r in range(1, len(H.n_leapfrog) // n):
        np.testing.assert_array_equal(H.q_chain[r * n:(r + 1) * n], H.q_chain[:n])
        np.testing.assert_array_equal(H.E_chain[r * n:(r + 1) * n], H.E_chain[:n])
        np.testing.assert_array_equal(H.n_leapfrog[r * n:(r + 1) * n], H.n_leapfrog[:n])


# ---- generic warp-per-chain kernel: D on both sides of its per-lane widths and at its largest D ------------------------------
@pytest.mark.parametrize("D", C.GENERIC_D)
@pytest.mark.parametrize("name", C.EDGE)
def test_generic_f64_edges_match_oracle(name, D):
    c = C.oracle_case(name, D, C.N_ORACLE)
    H, idx = _run(c, "float64", "generic")
    assert H.nuts_kernel == "generic"
    _check_f64(c, H, idx)


@pytest.mark.parametrize("D", C.GENERIC_D)
@pytest.mark.parametrize("name", C.EDGE)
def test_generic_f32_edges_match_oracle(name, D):
    c = C.oracle_case(name, D, C.N_ORACLE)
    H, idx = _run(c, "float32", "generic")
    assert H.nuts_kernel == "generic"
    _check_f32(c, H, idx)


def test_generic_f64_iteration_blocks_after_instability_rejects():
    """Blocks of two iterations resume the tape cursors that instability rejects (no uniform drawn) left behind."""
    c = C.oracle_case("instab", 33, C.N_ORACLE)
    H, idx = _run(c, "float64", "generic", iter_block=2)
    _check_f64(c, H, idx)


# ---- tensor-core kernel, D = 100, bf16x3 and fp16x2 splits ---------------------------------------------------------------
@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("name", C.CASES)
def test_tc_edges_match_oracle(name, prec, monkeypatch):
    """Every oracle chain 33 times over three CTAs; the deep case at d_max = 12, the kernel's deepest check-point stack."""
    if prec == "fp16x2":
        monkeypatch.setenv("HMC_B200_TC_PREC", "fp16x2")
    c = C.oracle_case(name, C.TC_D, C.N_DEEP if name == "deep" else C.N_ORACLE)
    H, idx = _run(c, "float32", "tc", reps=TC_REPS)
    assert H.nuts_kernel == "tc"
    _check_f32(c, H, idx)
    _reps_agree(H, c)


@pytest.mark.parametrize("name", ["instab", "uturn_sub"])
def test_tc_iteration_blocks_on_tapes_match_oracle(name):
    """Injected tapes over iteration blocks (the cursors resume from the per-chain cursor row) with the mean off zero.  Not bit
    equal to the single launch: a block resumes from the stored float32 q, and (x + mu) - mu changes the last bits of x."""
    c = C.oracle_case(name, C.TC_D, C.N_ORACLE)
    H, idx = _run(c, "float32", "tc", reps=TC_REPS, iter_block=2)
    _check_f32(c, H, idx)
    _reps_agree(H, c)


# ---- large-D GEMM path ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("D", C.BIGD_D)
@pytest.mark.parametrize("name", C.EDGE)
def test_bigd_edges_match_oracle(name, D, prec):
    c = C.oracle_case(name, D, C.N_ORACLE)
    H, idx = _run(c, "float32", "bigd", tc_precision=prec)
    assert H.nuts_kernel == "bigd" and H.tc_precision == prec
    _check_f32(c, H, idx)


# ---- dense momentum metric on the generic kernels ------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("name,D", C.METRIC_RUNS)
def test_generic_nuts_dense_metric_matches_oracle(name, D, dtype):
    c = C.oracle_case(name, D, C.N_ORACLE, dense=True)
    H, idx = _run(c, dtype, "generic")
    assert H.nuts_kernel == "generic"
    (_check_f64 if dtype == "float64" else _check_f32)(c, H, idx)


def _philox(seed, chain_id0, Nchain, Niter, D, Llo, Lhi):
    import torch
    import hmc_b200_lib as L
    z = torch.zeros((Nchain, Niter + 1, D), dtype=torch.float64, device="cuda")
    Lt = torch.zeros((Nchain, Niter), dtype=torch.int32, device="cuda")
    u = torch.zeros((Nchain, Niter), dtype=torch.float64, device="cuda")
    L.check(L.load().hmc_philox_draws(seed, chain_id0, Nchain, Niter, D, Llo, Lhi, L.ptr(z), L.ptr(Lt), L.ptr(u), L.current_stream_ptr()))
    torch.cuda.synchronize()
    return z.cpu().numpy(), Lt.cpu().numpy(), u.cpu().numpy()


# D per dtype for each staging regime of random_generic.cu (F, P and M^-1 in shared memory under a 200 KB budget): all three,
# M^-1 read from global memory, only F, none; and the largest D
@pytest.mark.parametrize("dtype,D", [("float32", 128), ("float32", 130), ("float32", 200), ("float32", 300), ("float32", 1024),
                                     ("float64", 64), ("float64", 100), ("float64", 130), ("float64", 200), ("float64", 1024)])
def test_random_generic_dense_metric_on_device_draws(dtype, D):
    """The kernel's own Philox z; the oracle gets p = Lc z in float64 (as tests/test_bigd_metric_gpu.py does for the large-D
    path).  A non-diagonal Lc, so p = Lc^T z would differ.  Per-dimension dt, warm-up, thinning, chain_id0 != 0."""
    import samplers as S
    Nchain, Niter, warm, thin, Llo, Lhi, seed, c0 = 16, 6, 2, 2, 4, 11, 23, 300
    rng = np.random.RandomState(D)
    lam = np.exp(rng.uniform(np.log(0.5), np.log(4.0), D))
    Qm, _ = np.linalg.qr(rng.standard_normal((D, D)))
    cov = (Qm * lam) @ Qm.T
    tgt = O.MVNTarget(rng.standard_normal(D) * 0.5, 0.5 * (cov + cov.T))
    cov_p = C.dense_cov_p(D)
    Lc = np.linalg.cholesky(cov_p)
    dt = 0.12 * rng.uniform(0.8, 1.2, D)
    q_start = tgt.q0 + rng.standard_normal((Nchain, D)) @ np.linalg.cholesky(tgt.cov0).T
    if dtype == "float32":
        q_start = q_start.astype(np.float32).astype(float)
    H = S.HMC_sampler(D, None, None, Nchain=Nchain, Niter=Niter, thin_rate=thin, warm_up_num=warm, sampler_type="Random", dt=dt,
                      L_low=Llo, L_high=Lhi, dtype=dtype, kernel="generic", seed=seed, chain_id0=c0, target=_spec(tgt),
                      cov_p=cov_p)
    H.gen_sample(q_start, verbose=False, quiet=True)
    z, Lt, ut = _philox(seed, c0, Nchain, Niter, D, Llo, Lhi)
    tape = []
    for m in range(Nchain):
        tape.append(("p", Lc @ z[m, 0]))
        for i in range(Niter):
            tape += [("p", Lc @ z[m, i + 1]), ("i", int(Lt[m, i])), ("u", float(ut[m, i]))]
    R = O.gen_sample_random(D, tgt.V, tgt.dVdq, q_start, O.TapeDraws(tape), Nchain, Niter, thin, warm, dt, Llo, Lhi, cov_p=cov_p,
                            record=True)
    assert 0.2 < R.accept_R < 1.0                                      # both decisions occur
    if dtype == "float64":
        qs = max(1.0, np.abs(R.q_chain).max())
        np.testing.assert_allclose(H.q_chain, R.q_chain, rtol=0, atol=1e-9 * qs)
        np.testing.assert_allclose(H.E_chain, R.E_chain, rtol=0, atol=1e-8 * max(1.0, np.abs(R.E_chain).max()))
        assert H.accept_R == R.accept_R
        return
    # float32: the near-tie rule of tests/test_bigd_metric_gpu.py::test_dense_metric_free_running_against_oracle_on_device_draws
    amp = np.linalg.norm(q_start - tgt.q0, axis=1)
    rel0 = np.linalg.norm(H.q_chain[:, 0] - R.q_chain[:, 0], axis=1) / amp
    first = warm + thin - 1
    margin = np.abs(np.log(ut[:, :first]) + R.dE_iter[:, :first])
    tie = np.any((R.dE_iter[:, :first] >= 0) & (margin < 5e-2), axis=1)
    assert np.all((rel0 < 1e-4) | tie), (rel0[~tie].max(), int(tie.sum()))
    assert np.mean(rel0 < 1e-4) > 0.9
    rel_last = np.linalg.norm(H.q_chain[:, -1] - R.q_chain[:, -1], axis=1) / amp
    same = rel_last < 1e-3
    assert np.mean(same) > 0.8
    np.testing.assert_allclose(H.E_chain[same, :, 0], R.E_chain[same, :, 0], rtol=1e-4, atol=1e-2)
    np.testing.assert_allclose(H.dE_chain[same, 1:, 0], R.dE_chain[same, 1:, 0], rtol=0, atol=2e-2)
