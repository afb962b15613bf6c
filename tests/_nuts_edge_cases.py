"""NUTS cases that drive the tree builder into its rare branches, for any dimension D.

Each case is a multivariate normal with a mean off zero, run with a per-dimension step size that is not uniform, warm-up and
thinning.  The stiff cases put one direction v of the target at scale sigma_s and then scale the step-size vector h so that
the leapfrog frequency of that direction, sqrt(lambda_max(h P h)), is a chosen value w: the leapfrog is stable for w < 2
and grows without bound for w > 2.

  instab     w just above 2: some trajectories grow until |E - E_initial| > 1000 (the instability reject), others turn first
  overflow   w just below 2 and start points displaced along v: the energy swings by more than 709 inside a tree without
             reaching the 1000 guard, so the float64 weights exp(E_max - E) overflow
  mid_exp    the same with a smaller displacement: weight arguments in (80, 709), where float32 expf would overflow
  uturn_sub  a plain anisotropic target at a moderate step: sub-trajectory U-turn rejects
  dmax_stop  the same with d_max = 4 and on_dmax="stop": the depth limit ends some trees, U-turns end the others
  deep       d_max = 12 and a step small enough that trees reach depth 11 or 12 (the deepest check-point stack)

tests/test_nuts_oracle_edges_cpu.py runs the float64 oracle on every case and checks that its record shows the branch;
tests/test_nuts_oracle_edges_gpu.py runs the CUDA kernels on the oracle's recorded draws.
"""
import functools

import numpy as np

from oracle import hmc_oracle as O

CASES = ("instab", "overflow", "mid_exp", "uturn_sub", "dmax_stop", "deep")
EDGE = CASES[:-1]                  # run on every kernel; "deep" (d_max = 12) only on the tensor-core kernel

# the dimensions each NUTS kernel runs the cases at: the generic kernel on both sides of its per-lane widths (NJ = 1 | 4 | 8
# switches at D = 32/33 and 128/129) and at its largest D; the tensor-core kernel's only D; the large-D path with D % 32 != 0
# and with rows that are not 16-byte aligned
GENERIC_D = (33, 129, 256)
TC_D = 100
BIGD_D = (300, 777)
N_ORACLE = 8                       # chains the oracle runs (the tensor-core tests replicate them over several CTAs)
N_DEEP = 4
ORACLE_RUNS = [(n, D, N_ORACLE) for n in EDGE for D in GENERIC_D + (TC_D,) + BIGD_D] + [("deep", TC_D, N_DEEP)]
# dense momentum metric on the generic kernel (the stiff cases are tuned for M = I)
METRIC_RUNS = [(n, D) for n in ("uturn_sub", "dmax_stop") for D in (33, 129)]

# name: (seed, d_max, on_dmax, warm-up, thin, Niter)
_RUN = {
    "instab": (1, 10, "stop", 2, 2, 7),
    "overflow": (2, 10, "stop", 1, 2, 5),
    "mid_exp": (3, 10, "stop", 1, 2, 5),
    "uturn_sub": (4, 10, "stop", 2, 2, 6),
    "dmax_stop": (5, 4, "stop", 1, 2, 5),
    "deep": (6, 12, "stop", 1, 2, 3),
}


class Case(object):
    """One run: target, start points, step sizes and sampler settings, plus the oracle's recorded run (``oracle``)."""
    pass


def _stiff_target(D, rng, sigma_s):
    """Unit covariance except along one random direction v, where the scale is sigma_s; mean off zero."""
    v = rng.standard_normal(D)
    v /= np.linalg.norm(v)
    cov = np.eye(D) - (1.0 - sigma_s ** 2) * np.outer(v, v)
    return O.MVNTarget(rng.standard_normal(D) * 0.7, 0.5 * (cov + cov.T)), v


def _scaled_dt(tgt, h, w):
    """h scaled so that the largest leapfrog frequency sqrt(lambda_max(h P h)) equals w."""
    lam = np.linalg.eigvalsh(tgt.inv_cov0 * np.outer(h, h)).max()
    return h * (w / np.sqrt(lam))


def make(name, D, Nchain):
    """The case ``name`` at dimension D with Nchain chains (no oracle run)."""
    seed, d_max, on_dmax, warm, thin, Niter = _RUN[name]
    rng = np.random.RandomState(1000 * seed + D)
    h = rng.uniform(0.7, 1.3, D)                                       # per-dimension step sizes, not uniform
    shift = None
    if name in ("instab", "overflow", "mid_exp"):
        tgt, v = _stiff_target(D, rng, 0.1)
        w, shift = {"instab": (2.001, 0.0), "overflow": (1.95, 4.0), "mid_exp": (1.95, 2.0)}[name]
        dt = _scaled_dt(tgt, h, w)
    elif name in ("uturn_sub", "dmax_stop"):
        tgt = O.MVNTarget(rng.standard_normal(D) * 0.7, np.diag(rng.uniform(0.3, 1.5, D) ** 2))
        dt = 0.25 * h
    else:
        tgt = O.MVNTarget(rng.standard_normal(D) * 0.7, np.eye(D))
        dt = 0.0025 * h
    q_start = tgt.q0 + rng.standard_normal((Nchain, D)) @ np.linalg.cholesky(tgt.cov0).T
    if shift:                                                          # stiff energy about 50 shift^2, +- 20 %
        q_start += np.outer(shift * (1.0 + 0.1 * rng.uniform(-1, 1, Nchain)), v)
    c = Case()
    c.name, c.D, c.Nchain, c.Niter = name, D, Nchain, Niter
    c.tgt, c.dt, c.d_max, c.on_dmax = tgt, dt, d_max, on_dmax
    c.warm, c.thin, c.seed = warm, thin, 100 * seed + D
    # relative tolerance of the float32 kernels' energies.  overflow / mid_exp sit hundreds of units up the stiff direction (curvature
    # 100, |x| ~ 2-4) with the leapfrog at frequency 1.95, where the per-step phase error is ~9x the relative rounding error: after
    # hundreds of steps a float32 sample ~1e-3 off along v (inside the 2e-4 max|q| sample tolerance) moves E by ~400 x 1e-3.  Largest
    # relative energy difference measured where the trees agree: 4.1e-4 (large-D path, bf16x3, D = 300; NVIDIA B200, 1000 W).
    c.e_rtol = 1e-3 if name in ("overflow", "mid_exp") else 2e-5
    c.q_start = q_start.astype(np.float32).astype(float)              # the float32 kernels start from the same points
    return c


class SeededDraws(O.NumpyDraws):
    """np.random draws with momenta p = Lc z from standard normals z: the distribution of NumpyDraws without its
    multivariate_normal factorisation of cov_p at every call (seconds per run at D ~ 800)."""

    def __init__(self, D, cov_p=None):
        O.NumpyDraws.__init__(self, D, cov_p)
        self.Lc = np.linalg.cholesky(self.cov_p)

    def p_sample(self):
        return self.Lc @ np.random.standard_normal(self.D)


def run_oracle(c, cov_p=None):
    """The float64 oracle on np.random draws seeded by the case, recording tapes and the tree builder's branches."""
    np.random.seed(c.seed)
    c.cov_p = cov_p
    with np.errstate(over="ignore", invalid="ignore"):
        c.oracle = O.gen_sample_NUTS(c.D, c.tgt.V, c.tgt.dVdq, c.q_start, SeededDraws(c.D, cov_p), c.Nchain, c.Niter,
                                     thin_rate=c.thin, warm_up_num=c.warm, dt=c.dt, d_max=c.d_max, cov_p=cov_p, record=True,
                                     on_dmax=c.on_dmax)
    return c


def dense_cov_p(D, seed=9, k=4, lo=0.7, hi=1.4):
    """A dense SPD momentum metric: the identity with k eigenvalues in [lo, hi] along random directions (its Cholesky factor
    is not diagonal, so Lc and its transpose differ)."""
    rng = np.random.RandomState(seed)
    Vk, _ = np.linalg.qr(rng.standard_normal((D, k)))
    lam = np.exp(rng.uniform(np.log(lo), np.log(hi), k))
    c = np.eye(D) + (Vk * (lam - 1.0)) @ Vk.T
    return 0.5 * (c + c.T)


@functools.lru_cache(maxsize=None)
def oracle_case(name, D, Nchain, dense=False):
    """The case with its oracle run (cached: the float64 and float32 tests of a kernel share it)."""
    return run_oracle(make(name, D, Nchain), dense_cov_p(D) if dense else None)
