"""The oracle against the reference on the same ``np.random`` stream.

The reference's outputs are the committed fixtures (tests/golden/make_golden.py ran the reference from the seed of each
case).  Here the oracle starts from the same seed, draws the start points with the reference's call, then consumes the
global stream through ``NumpyDraws`` exactly as the reference did, and must land on the reference's numbers."""
import numpy as np
import pytest

from oracle import hmc_oracle as O
from _util import CASES, load, pin_start


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_same_stream_same_numbers(case):
    name, stype, D, rho, Nchain, Niter, warm, thin, dt, kw, sscale, seed, nsave = case
    fx = load(name)
    tgt = O.MVNTarget(fx["q0"], fx["cov0"])
    np.random.seed(seed)
    q_start = np.random.multivariate_normal(tgt.q0, np.diag(np.ones(D)) * sscale, size=Nchain)     # utils.py:204-209
    np.testing.assert_array_equal(pin_start(name, q_start), fx["q_start"])
    dt = fx["dt"] if fx["dt"].ndim else float(fx["dt"])
    draws = O.NumpyDraws(D, fx["cov_p"])
    if stype == "Random":
        R = O.gen_sample_random(D, tgt.V, tgt.dVdq, q_start, draws, Nchain, Niter, thin, warm, dt,
                                kw["L_low"], kw["L_high"], cov_p=fx["cov_p"], N_save_chain0=nsave)
    else:
        R = O.gen_sample_NUTS(D, tgt.V, tgt.dVdq, q_start, draws, Nchain, Niter, thin, warm, dt, kw["d_max"],
                              cov_p=fx["cov_p"])
    np.testing.assert_allclose(R.q_chain, fx["q_chain"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(R.E_chain, fx["E_chain"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(R.dE_chain, fx["dE_chain"], rtol=0, atol=1e-10)
    assert R.N_total_steps == int(fx["N_total_steps"])
    assert R.accept_R == float(fx["accept_R"])
    Rq, neff = O.convergence_stats(R.q_chain[:, 1:, :], 1, 0)
    np.testing.assert_allclose(Rq, fx["R_q"], rtol=1e-12)
    np.testing.assert_allclose(neff, fx["n_eff_q"], rtol=1e-12)
