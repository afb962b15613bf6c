"""Shared helpers for the tests: fixture loading and tape reconstruction."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

RANDOM_FIXTURES = ["random_case1a", "random_d10_thin3", "random_case3c_small", "random_case3d_small",
                   "random_case2c_small", "random_vecdt_covp", "random_constL"]
NUTS_FIXTURES = ["nuts_d2", "nuts_d10", "nuts_case3c_small", "nuts_covp"]

# The cases the fixtures were generated from (tests/golden/make_golden.py runs the reference on each).
CASES = [
    # name, sampler, D, rho, Nchain, Niter, warm, thin, dt, extra kwargs, start scale, seed, N_save_chain0
    ("random_case1a", "Random", 2, 0.0, 10, 1000, 200, 1, 0.1, dict(L_low=5, L_high=20), 2.0, 0, 20),
    ("random_d10_thin3", "Random", 10, 0.95, 6, 90, 30, 3, 0.1, dict(L_low=5, L_high=20), 2.0, 1, 0),
    ("random_case3c_small", "Random", 100, 0.95, 4, 60, 20, 1, 0.1, dict(L_low=5, L_high=20), 2.0, 2, 10),
    ("random_case3d_small", "Random", 100, 0.95, 2, 12, 4, 1, 0.1, dict(L_low=50, L_high=200), 2.0, 3, 0),
    ("random_case2c_small", "Random", 100, 0.0, 4, 40, 10, 1, 0.1, dict(L_low=5, L_high=20), 100.0, 4, 0),
    ("random_vecdt_covp", "Random", 6, 0.5, 4, 50, 10, 2, "vec", dict(L_low=3, L_high=9, cov_p="diag"), 2.0, 5, 0),
    # the reference's live sampler with L_low = L, L_high = L + 1: randint(7, 8) is always 7 -- a FIXED trajectory length with
    # the live bookkeeping; pins sampler_type="Fixed" of the B200 build (a silent no-op upstream, SURVEY H8)
    ("random_constL", "Random", 10, 0.9, 5, 40, 10, 1, 0.15, dict(L_low=7, L_high=8), 2.0, 9, 6),
    ("nuts_d2", "NUTS", 2, 0.0, 4, 40, 10, 1, 0.3, dict(d_max=10), 2.0, 6, 0),
    ("nuts_d10", "NUTS", 10, 0.95, 3, 30, 10, 2, 0.1, dict(d_max=12), 2.0, 7, 0),
    ("nuts_case3c_small", "NUTS", 100, 0.95, 2, 8, 2, 1, 0.2, dict(d_max=10), 1.0, 8, 0),
    # NUTS with a non-identity momentum metric (samplers.py:352-356, 811-817, 835-837: force times M^-1, q moved by p, Q9)
    ("nuts_covp", "NUTS", 6, 0.5, 3, 25, 5, 1, 0.15, dict(d_max=10, cov_p="diag"), 2.0, 10, 0),
]


def pin_start(name, q_start):
    """The case's own edits of the drawn start points: case 2c puts chain 0 far out (case2-script.py:58-61)."""
    if name == "random_case2c_small":
        q_start[0, :] = 0
        q_start[0, 0] = 1000
        q_start[0, 1] = -750
    return q_start


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def flat_tape(fx):
    """Structured per-chain tapes of a fixture -> flat ("p"/"i"/"u") tape in the reference's consumption order.

    For NUTS the interleaving of coins and uniforms is data dependent, so the flat order cannot be rebuilt from
    the arrays alone; `ChainTapeDraws` below serves each kind from its own per-chain queue instead."""
    Nchain, Niter = int(fx["Nchain"]), int(fx["Niter"])
    tape = []
    for m in range(Nchain):
        tape.append(("p", fx["p_tape"][m, 0]))
        for i in range(Niter):
            tape.append(("p", fx["p_tape"][m, i + 1]))
            tape.append(("i", int(fx["L_tape"][m, i])))
            tape.append(("u", float(fx["u_tape"][m, i])))
    return tape


class ChainTapeDraws(object):
    """Draw source fed by per-chain queues (p rows, ints, uniforms); chains are consumed one after another.
    A chain is finished once Niter+1 momenta were served, which is how the samplers consume them."""

    def __init__(self, p_tape, i_tape, u_tape):
        self.p_tape, self.i_tape, self.u_tape = p_tape, i_tape, u_tape
        self.m = 0
        self.np = 0
        self.ni = 0
        self.nu = 0
        self.per_chain = p_tape.shape[1]

    def p_sample(self):
        if self.np == self.per_chain:
            self.m += 1
            self.np = self.ni = self.nu = 0
        v = np.array(self.p_tape[self.m, self.np], dtype=float)
        self.np += 1
        return v

    def randint(self, low, high):
        v = int(self.i_tape[self.m, self.ni])
        self.ni += 1
        return v

    def random(self):
        v = float(self.u_tape[self.m, self.nu])
        self.nu += 1
        return v


def sampler_from_fixture(fx, dtype="float64", kernel="generic", with_draws=True, **over):
    """Build the CUDA-backed HMC_sampler (understanding-hmc_b200/samplers.py) for a golden fixture."""
    import samplers as S
    D = int(fx["D"])
    spec = S.MVNSpec.from_cov(fx["q0"], fx["cov0"])
    sampler = str(fx["sampler"])
    dt = fx["dt"] if fx["dt"].ndim else float(fx["dt"])
    cov_p = fx["cov_p"]
    cov_p = None if np.array_equal(cov_p, np.eye(D)) else cov_p
    kw = dict(Nchain=int(fx["Nchain"]), Niter=int(fx["Niter"]), thin_rate=int(fx["thin_rate"]),
              warm_up_num=int(fx["warm_up_num"]), cov_p=cov_p, sampler_type=sampler, dt=dt,
              dtype=dtype, kernel=kernel, target=spec)
    if sampler == "Random":
        kw.update(L_low=int(fx["L_low"]), L_high=int(fx["L_high"]))
        if with_draws:
            kw["draws"] = dict(p_tape=fx["p_tape"], L_tape=fx["L_tape"], u_tape=fx["u_tape"])
    else:
        kw.update(d_max=int(fx["d_max"]))
        if with_draws:
            kw["draws"] = dict(p_tape=fx["p_tape"], dir_tape=fx["dir_tape"], u_tape=fx["u_tape"])
    kw.update(over)
    return S.HMC_sampler(D, None, None, **kw)
