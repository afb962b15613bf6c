"""The NUTS edge cases of tests/_nuts_edge_cases.py reach the branches they are named for, at every dimension and chain count
tests/test_nuts_oracle_edges_gpu.py runs them with (float64 oracle only: no GPU needed).  A case that stopped reaching its
branch would leave the GPU tests comparing the kernels on ordinary trees."""
import numpy as np
import pytest

import _nuts_edge_cases as C


def _check_branch(c):
    R = c.oracle
    if c.name == "instab":
        frac = (R.n_instab_iter > 0).mean()
        assert 0.2 <= frac <= 0.8, frac                                 # a mix: normal iterations follow rejects
    elif c.name == "overflow":
        assert R.n_instability == 0
        assert (R.max_exp_arg_iter > 709).any() or R.nonfinite_iter.any()
        assert R.nonfinite_iter.any()
    elif c.name == "mid_exp":
        assert ((R.max_exp_arg_iter > 80) & (R.max_exp_arg_iter < 709)).any()
    elif c.name == "uturn_sub":
        assert R.n_uturn_sub_iter.sum() > 0
    elif c.name == "dmax_stop":
        assert c.on_dmax == "stop" and R.dmax_iter.any() and not R.dmax_iter.all()
        assert R.n_dmax == int(R.dmax_iter.sum())
    elif c.name == "deep":
        assert c.d_max == 12 and R.depth.max() >= 11


@pytest.mark.parametrize("name,D,Nchain", C.ORACLE_RUNS)
def test_case_reaches_its_branch(name, D, Nchain):
    c = C.oracle_case(name, D, Nchain)
    assert np.abs(c.tgt.q0).max() > 0.5                                # mean off zero
    assert np.ptp(c.dt) > 0.2 * c.dt.mean()                            # per-dimension step sizes, not uniform
    assert c.warm > 0 and c.thin > 1
    assert c.oracle.n_leapfrog.sum() * (c.D + 1) + c.Nchain * (1 + c.Niter) == c.oracle.N_total_steps
    _check_branch(c)


@pytest.mark.parametrize("name,D", C.METRIC_RUNS)
def test_dense_metric_case_reaches_its_branch(name, D):
    c = C.oracle_case(name, D, C.N_ORACLE, dense=True)
    assert c.cov_p is not None and np.abs(np.linalg.cholesky(c.cov_p) - np.diag(np.diag(np.linalg.cholesky(c.cov_p)))).max() > 1e-3
    _check_branch(c)


def test_recording_changes_nothing():
    """The oracle's record of the tree builder leaves its samples, energies and counters as they are without it."""
    import oracle.hmc_oracle as O
    for name in ("instab", "overflow", "dmax_stop"):
        c = C.make(name, 33, 4)
        out = []
        for record in (False, True):
            np.random.seed(c.seed)
            with np.errstate(over="ignore", invalid="ignore"):
                out.append(O.gen_sample_NUTS(c.D, c.tgt.V, c.tgt.dVdq, c.q_start, C.SeededDraws(c.D), c.Nchain, c.Niter,
                                             thin_rate=c.thin, warm_up_num=c.warm, dt=c.dt, d_max=c.d_max, record=record,
                                             on_dmax=c.on_dmax))
        a, b = out
        np.testing.assert_array_equal(a.q_chain, b.q_chain)
        np.testing.assert_array_equal(a.E_chain, b.E_chain)
        np.testing.assert_array_equal(a.dE_chain, b.dE_chain)
        assert (a.N_total_steps, a.n_instability, a.n_dmax) == (b.N_total_steps, b.n_instability, b.n_dmax)
        assert b.n_instability == int(b.n_instab_iter.sum())
