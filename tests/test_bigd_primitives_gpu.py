"""Large-D primitives on the tcgen05 GEMM (csrc/bigd_primitives.cu): hmc_start_pts_bigd against hmc_start_pts on the same
draws and against float64 q0 + Lc z, sampling statistics, shard invariance and determinism; hmc_leap_frog_bigd against the
float64 oracle (dense metric, per-dimension dt, both splits), against hmc_leap_frog, shard invariance, merged half kicks and
determinism; the Python mirror's routing; rejections.

Tolerances: float32 results of fp32-grade products (float32 operands split into 16-bit parts, fp32 accumulation): rel-L2 1e-5,
the bound tests/test_bigd_gpu.py holds the large-D sampler to for trajectories of fewer than 20 steps, up to K = D = 5000 and for
single steps.  The accumulation error grows with K: measured on a B200, start points at D = 8192 sit at 1.3e-5 of |q - q0| for
every chain, and ten leapfrog steps at 1.4e-5 (D = 4100) and 2.7e-5 (D = 8192) of the amplitude; those cases are held to 2e-5
and 4e-5."""
import functools

import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu


def _L():
    import hmc_b200_lib as L
    return L, L.load()


def _dev(a, dtype=None):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


def _lower_factor(D, seed):
    """A well-conditioned lower-triangular factor Lc (cov0 = Lc Lc^T), built directly (no D^3 factorisation on the host)."""
    rng = np.random.RandomState(seed)
    Lc = np.tril(rng.standard_normal((D, D))) * (0.5 / np.sqrt(D))
    Lc[np.diag_indices(D)] = 0.5 + rng.random_sample(D)
    return Lc


def _start_bigd(Nchain, D, q0, Lc=None, sd=None, seed=3, chain_id0=0, ws=True):
    import torch
    L, lib = _L()
    out = torch.empty((Nchain, D), dtype=torch.float32, device="cuda")
    nbytes = int(lib.hmc_start_pts_workspace_bytes(Nchain, D))
    buf, wp = L.aligned_workspace(torch, torch.device("cuda"), nbytes) if ws else (None, None)
    q0_d, Lc_d, sd_d = (None if a is None else _dev(a, torch.float64) for a in (q0, Lc, sd))
    L.check(lib.hmc_start_pts_bigd(L.HMC_F32, seed, chain_id0, Nchain, D, L.ptr(q0_d), L.ptr(Lc_d), L.ptr(sd_d), L.ptr(out), wp,
                                   nbytes if ws else 0, L.current_stream_ptr()))
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _start_direct(Nchain, D, q0, Lc=None, sd=None, seed=3, chain_id0=0):
    import torch
    L, lib = _L()
    out = torch.empty((Nchain, D), dtype=torch.float32, device="cuda")
    q0_d, Lc_d, sd_d = (None if a is None else _dev(a, torch.float64) for a in (q0, Lc, sd))
    L.check(lib.hmc_start_pts(L.HMC_F32, seed, chain_id0, Nchain, D, L.ptr(q0_d), L.ptr(Lc_d), L.ptr(sd_d), L.ptr(out),
                              L.current_stream_ptr()))
    torch.cuda.synchronize()
    return out.cpu().numpy()


# ----------------------------------------------------------------------------------------------------------------------------
# start points
# ----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [300, 1024, 4096])
def test_start_pts_bigd_matches_warp_kernel(D):
    Lc = _lower_factor(D, D)
    q0 = np.random.RandomState(1).standard_normal(D)
    got = _start_bigd(256, D, q0, Lc, chain_id0=70001)
    want = _start_direct(256, D, q0, Lc, chain_id0=70001)
    rel = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want.astype(float) - q0, axis=1)
    assert rel.max() < 1e-5, rel.max()


@pytest.mark.parametrize("D", [5000, 8192])
def test_start_pts_bigd_against_float64_product(D):
    Lc = _lower_factor(D, D)
    q0 = np.random.RandomState(2).standard_normal(D)
    z = _start_bigd(64, D, np.zeros(D), sd=np.ones(D), chain_id0=5).astype(float)      # the normals themselves
    want = q0 + z @ Lc.T
    got = _start_bigd(64, D, q0, Lc, chain_id0=5)
    rel = np.linalg.norm(got - want, axis=1) / np.linalg.norm(want - q0, axis=1)
    assert rel.max() < (1e-5 if D <= 5000 else 2e-5), rel.max()


def test_start_pts_bigd_sampling_statistics():
    D, N = 5000, 8192
    Lc = _lower_factor(D, 9)
    q0 = np.random.RandomState(4).standard_normal(D) * 3.0
    q = _start_bigd(N, D, q0, Lc, seed=11).astype(float)
    sd = np.sqrt(np.einsum("ij,ij->i", Lc, Lc))                  # sqrt(diag(cov0))
    assert np.all(np.abs(q.mean(axis=0) - q0) < 5 * sd / np.sqrt(N))
    v = np.random.RandomState(5).standard_normal((16, D))
    want = np.einsum("ij,ij->i", v @ Lc, v @ Lc)                 # v^T cov0 v
    got = ((q - q0) @ v.T).var(axis=0)
    assert np.all(np.abs(got / want - 1) < 0.05), got / want


def test_start_pts_bigd_shards_and_repeats():
    D = 777
    Lc = _lower_factor(D, 6)
    q0 = np.random.RandomState(7).standard_normal(D)
    full = _start_bigd(10000, D, q0, Lc, chain_id0=123)
    for s in range(0, 10000, 1000):
        np.testing.assert_array_equal(_start_bigd(1000, D, q0, Lc, chain_id0=123 + s), full[s:s + 1000])
    np.testing.assert_array_equal(_start_bigd(10000, D, q0, Lc, chain_id0=123), full)


def test_start_pts_diagonal_equals_warp_kernel():
    D = 3001
    q0 = np.random.RandomState(8).standard_normal(D)
    sd = 0.5 + np.random.RandomState(9).random_sample(D)
    np.testing.assert_array_equal(_start_bigd(300, D, q0, sd=sd, chain_id0=9, ws=False), _start_direct(300, D, q0, sd=sd, chain_id0=9))


@pytest.mark.parametrize("D", [300, 4096])
def test_utils_start_pts_below_4097_is_the_warp_kernel(D):
    import utils as U
    Lc = _lower_factor(D, 12)
    q0 = np.random.RandomState(13).standard_normal(D)
    got = U.start_pts(q0, Lc @ Lc.T, 200, device="cuda", seed=3, chain_id0=44).cpu().numpy()
    want = _start_direct(200, D, q0, np.linalg.cholesky(Lc @ Lc.T), chain_id0=44)
    np.testing.assert_array_equal(got, want)


def test_utils_start_pts_above_4096_runs_on_the_gemm():
    import utils as U
    D = 5000
    Lc = _lower_factor(D, 14)
    q0 = np.random.RandomState(15).standard_normal(D)
    cov0 = Lc @ Lc.T
    got = U.start_pts(q0, cov0, 64, device="cuda", seed=3, chain_id0=2).cpu().numpy()
    np.testing.assert_array_equal(got, _start_bigd(64, D, q0, np.linalg.cholesky(cov0), chain_id0=2))
    diag = U.start_pts(q0, np.diag(np.diag(cov0)), 64, device="cuda", seed=3, chain_id0=2).cpu().numpy()
    np.testing.assert_array_equal(diag, _start_bigd(64, D, q0, sd=np.sqrt(np.diag(cov0)), chain_id0=2, ws=False))
    L, _ = _L()
    with pytest.raises(L.HMCError, match="float32 only"):
        U.start_pts(q0, cov0, 64, device="cuda", dtype="float64")


# ----------------------------------------------------------------------------------------------------------------------------
# leap frog
# ----------------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=4)
def _problem(D, seed):
    """Target precision P, dense momentum metric inverse Minv, mean, per-dimension dt."""
    rng = np.random.RandomState(seed)
    S = rng.standard_normal((D, D)) * (0.15 / np.sqrt(D))
    P = np.diag(0.5 + rng.random_sample(D)) + 0.5 * (S + S.T)
    T = rng.standard_normal((D, D)) * (0.1 / np.sqrt(D))
    Minv = np.diag(0.8 + 0.4 * rng.random_sample(D)) + 0.5 * (T + T.T)
    mu = rng.standard_normal(D) * 0.5
    dt = 0.1 + 0.1 * rng.random_sample(D)
    return P, Minv, mu, dt


@functools.lru_cache(maxsize=2)
def _force(D, seed):
    P, Minv, _, _ = _problem(D, seed)
    return Minv @ P                                              # F = M^-1 P (samplers.py:835)


def _target(F, mu, dt, torch_dtype=None):
    import torch
    L, _ = _L()
    D = F.shape[0]
    Dp = (D + 3) // 4 * 4
    ft = np.zeros((D, Dp)); ft[:, :D] = F.T
    vm = np.zeros(Dp); vm[:D] = mu
    vd = np.zeros(Dp); vd[:D] = dt
    tdt = torch_dtype or torch.float32
    keep = [_dev(ft, tdt), _dev(vm, tdt), _dev(vd, tdt)]
    t = L.Target()
    t.D, t.D_pad = D, Dp
    t.Ft, t.mu, t.dt = (k.data_ptr() for k in keep)
    return t, keep


def _lf_bigd(t, p, q, nsteps, flags=0, ws=True, dtype=None):
    import torch
    L, lib = _L()
    pd, qd = _dev(p, torch.float32), _dev(q, torch.float32)
    pn, qn = torch.empty_like(pd), torch.empty_like(qd)
    nbytes = int(lib.hmc_leap_frog_workspace_bytes(t, p.shape[0], flags))
    buf, wp = L.aligned_workspace(torch, torch.device("cuda"), nbytes) if ws else (None, None)
    L.check(lib.hmc_leap_frog_bigd(L.HMC_F32 if dtype is None else dtype, t, p.shape[0], L.ptr(pd), L.ptr(qd), L.ptr(pn), L.ptr(qn),
                                   nsteps, flags, wp, nbytes if ws else 0, L.current_stream_ptr()))
    torch.cuda.synchronize()
    return pn.cpu().numpy(), qn.cpu().numpy()


def _lf_warp(t, p, q, nsteps):
    import torch
    L, lib = _L()
    pd, qd = _dev(p, torch.float32), _dev(q, torch.float32)
    pn, qn = torch.empty_like(pd), torch.empty_like(qd)
    L.check(lib.hmc_leap_frog(L.HMC_F32, t, p.shape[0], L.ptr(pd), L.ptr(qd), L.ptr(pn), L.ptr(qn), nsteps, L.current_stream_ptr()))
    torch.cuda.synchronize()
    return pn.cpu().numpy(), qn.cpu().numpy()


def _state(B, mu, seed):
    rng = np.random.RandomState(seed)
    D = mu.shape[0]
    q = (mu + rng.standard_normal((B, D))).astype(np.float32)
    p = rng.standard_normal((B, D)).astype(np.float32)
    return p, q


def _rel(got, want, old, centre):
    amp = np.maximum(np.linalg.norm(want - centre, axis=1), np.linalg.norm(old - centre, axis=1))
    return (np.linalg.norm(got - want, axis=1) / amp).max()


_ORACLE = {}


@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
@pytest.mark.parametrize("nsteps", [1, 10])
@pytest.mark.parametrize("D", [1500, 4100, 8192])
def test_leap_frog_bigd_against_oracle(D, nsteps, prec):
    L, _ = _L()
    P, Minv, mu, dt = _problem(D, D)
    p, q = _state(256, mu, D + 1)
    key = (D, nsteps)
    if key not in _ORACLE:
        tgt = O.MVNTarget.__new__(O.MVNTarget)
        tgt.q0, tgt.inv_cov0 = mu, P
        pw, qw = p.astype(float), q.astype(float)
        for _ in range(nsteps):
            pw, qw = O.leap_frog_batch(pw, qw, dt, Minv, tgt)
        _ORACLE[key] = (pw, qw)
    pw, qw = _ORACLE[key]
    t, keep = _target(_force(D, D), mu, dt)
    pg, qg = _lf_bigd(t, p, q, nsteps, L.FLAG_TC_FP16X2 if prec == "fp16x2" else 0)
    tol = 1e-5 if nsteps == 1 or D <= 1500 else 4e-5
    assert _rel(qg, qw, q, mu) < tol
    assert _rel(pg, pw, p, 0.0) < tol


@pytest.mark.parametrize("D", [128, 777, 1024])
def test_leap_frog_bigd_matches_warp_kernel(D):
    P, Minv, mu, dt = _problem(D, D + 2)
    p, q = _state(512, mu, D + 3)
    t, keep = _target(Minv @ P, mu, dt)
    for nsteps in (1, 4):
        pg, qg = _lf_bigd(t, p, q, nsteps)
        pw, qw = _lf_warp(t, p, q, nsteps)
        assert _rel(qg, qw, q, mu) < 1e-5 and _rel(pg, pw, p, 0.0) < 1e-5


@pytest.mark.parametrize("prec", ["bf16x3", "fp16x2"])
def test_leap_frog_bigd_shards_and_repeats(prec):
    L, _ = _L()
    D = 1300
    flags = L.FLAG_TC_FP16X2 if prec == "fp16x2" else 0
    P, Minv, mu, dt = _problem(D, 21)
    p, q = _state(40000, mu, 22)
    t, keep = _target(Minv @ P, mu, dt)
    pf, qf = _lf_bigd(t, p, q, 2, flags)
    for s in range(0, 40000, 1000):
        ps, qs = _lf_bigd(t, p[s:s + 1000], q[s:s + 1000], 2, flags)
        np.testing.assert_array_equal(ps, pf[s:s + 1000])
        np.testing.assert_array_equal(qs, qf[s:s + 1000])
    for B in (1, 127, 129):                                      # padding rows in the last row block
        ps, qs = _lf_bigd(t, p[:B], q[:B], 2, flags)
        np.testing.assert_array_equal(ps, pf[:B])
        np.testing.assert_array_equal(qs, qf[:B])
    pr, qr = _lf_bigd(t, p, q, 2, flags)
    np.testing.assert_array_equal(pr, pf)
    np.testing.assert_array_equal(qr, qf)


def test_leap_frog_bigd_merged_half_kicks():
    """nsteps = 3 merges the half kicks between steps: within 1e-6 relative of three single steps."""
    D = 2048
    P, Minv, mu, dt = _problem(D, 31)
    p, q = _state(1024, mu, 32)
    t, keep = _target(Minv @ P, mu, dt)
    p3, q3 = _lf_bigd(t, p, q, 3)
    p1, q1 = p, q
    for _ in range(3):
        p1, q1 = _lf_bigd(t, p1, q1, 1)
    assert _rel(q3, q1, q, mu) < 1e-6 and _rel(p3, p1, p, 0.0) < 1e-6


def _sampler(D, P, Minv, mu, dt, prec=None):
    import samplers as S
    cov_p = np.linalg.inv(Minv)
    return S.HMC_sampler(D, None, None, Nchain=2, Niter=1, sampler_type="Random", dt=dt, L_low=1, L_high=2, dtype="float32",
                         cov_p=cov_p, target=S.MVNSpec(mu, P, 0.0), tc_precision=prec)


@pytest.mark.parametrize("D", [100, 1024])
def test_sampler_leap_frog_up_to_1024_is_the_warp_kernel(D):
    P, Minv, mu, dt = _problem(D, 41)
    p, q = _state(64, mu, 42)
    H = _sampler(D, P, Minv, mu, dt)
    pg, qg = H.leap_frog(p, q, nsteps=2)
    t, keep = _target(H.inv_cov_p @ P, mu, dt)
    pw, qw = _lf_warp(t, p, q, 2)
    np.testing.assert_array_equal(pg, pw.astype(float))
    np.testing.assert_array_equal(qg, qw.astype(float))


@pytest.mark.parametrize("prec", [None, "fp16x2"])
def test_sampler_leap_frog_above_1024_runs_on_the_gemm(prec):
    L, _ = _L()
    D = 1500
    P, Minv, mu, dt = _problem(D, 43)
    p, q = _state(64, mu, 44)
    H = _sampler(D, P, Minv, mu, dt, prec)
    pg, qg = H.leap_frog(p, q, nsteps=2)
    t, keep = _target(H.inv_cov_p @ P, mu, dt)
    pb, qb = _lf_bigd(t, p, q, 2, L.FLAG_TC_FP16X2 if prec == "fp16x2" else 0)
    np.testing.assert_array_equal(pg, pb.astype(float))
    np.testing.assert_array_equal(qg, qb.astype(float))
    H64 = _sampler(D, P, Minv, mu, dt)
    H64.dtype = "float64"
    with pytest.raises(L.HMCError, match="float32 only"):
        H64.leap_frog(p, q)


# ----------------------------------------------------------------------------------------------------------------------------
# rejections
# ----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,dtype,why", [(1500, 1, "float32 only"), (127, 0, r"D must be in \[128, 8192\]"),
                                         (8193, 0, r"D must be in \[128, 8192\]")])
def test_bigd_primitives_reject_what_they_do_not_cover(D, dtype, why):
    import torch
    L, lib = _L()
    tdt = torch.float64 if dtype == L.HMC_F64 else torch.float32
    t, keep = _target(np.eye(D), np.zeros(D), np.full(D, 0.1), tdt)
    p = torch.zeros((4, D), dtype=tdt, device="cuda")
    rc = lib.hmc_leap_frog_bigd(dtype, t, 4, L.ptr(p), L.ptr(p), L.ptr(p), L.ptr(p), 1, 0, None, 0, L.current_stream_ptr())
    assert rc == L.HMC_E_UNSUPPORTED
    assert "hmc_leap_frog_bigd does not cover" in lib.hmc_last_error_string().decode()
    with pytest.raises(L.HMCError, match=why):
        L.check(rc)
    q0 = torch.zeros((D,), dtype=torch.float64, device="cuda")
    Lc = torch.eye(D, dtype=torch.float64, device="cuda")
    rc = lib.hmc_start_pts_bigd(dtype, 0, 0, 4, D, L.ptr(q0), L.ptr(Lc), None, L.ptr(p), None, 0, L.current_stream_ptr())
    assert rc == L.HMC_E_UNSUPPORTED
    with pytest.raises(L.HMCError, match="hmc_start_pts_bigd does not cover this configuration: " + why):
        L.check(rc)
    torch.cuda.synchronize()


def test_bigd_primitives_need_their_workspace():
    import torch
    L, lib = _L()
    D = 1500
    t, keep = _target(np.eye(D), np.zeros(D), np.full(D, 0.1))
    p = torch.zeros((4, D), dtype=torch.float32, device="cuda")
    need = int(lib.hmc_leap_frog_workspace_bytes(t, 4, 0))
    rc = lib.hmc_leap_frog_bigd(L.HMC_F32, t, 4, L.ptr(p), L.ptr(p), L.ptr(p), L.ptr(p), 1, 0, None, 0, L.current_stream_ptr())
    assert rc == L.HMC_E_BADARG and "needs a workspace of %d bytes" % need in lib.hmc_last_error_string().decode()
    buf, wp = L.aligned_workspace(torch, torch.device("cuda"), need)
    rc = lib.hmc_leap_frog_bigd(L.HMC_F32, t, 4, L.ptr(p), L.ptr(p), L.ptr(p), L.ptr(p), 1, 0, wp, need - 1024, L.current_stream_ptr())
    assert rc == L.HMC_E_BADARG
    q0 = torch.zeros((D,), dtype=torch.float64, device="cuda")
    Lc = torch.eye(D, dtype=torch.float64, device="cuda")
    rc = lib.hmc_start_pts_bigd(L.HMC_F32, 0, 0, 4, D, L.ptr(q0), L.ptr(Lc), None, L.ptr(p), None, 0, L.current_stream_ptr())
    assert rc == L.HMC_E_BADARG and "hmc_start_pts_workspace_bytes" in lib.hmc_last_error_string().decode()
    torch.cuda.synchronize()
