"""TEST INFRASTRUCTURE ONLY -- float64 numpy restatement of the reference's HMC hot path.

Nothing under ``oracle/`` is part of the product path.  Only ``tests/``, ``tests/golden/make_golden.py``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import it, and
there only as the checker (or as the timed CPU baseline), never as something the product calls.

Parity status: PINNED.  The committed fixtures under ``tests/golden/`` were produced by the reference itself
(``tests/golden/make_golden.py``, through ``oracle/ref_shim.py``).  ``tests/test_oracle_golden.py`` replays their
recorded draws through this restatement, and ``tests/test_oracle_vs_reference.py`` reruns each case from its seed on
the same ``np.random`` stream; both require agreement to 1e-12.  The README known-answer tables (README:332-358) pin
the NUTS index helpers.

Every function cites the reference ``file:line`` it follows (paths relative to /root/reference).
"""
from __future__ import annotations

import math

import numpy as np


# --------------------------------------------------------------------------------------------------
# Targets (what the driver closures compute: case1-script.py:31-49, same in every case script)
# --------------------------------------------------------------------------------------------------
class MVNTarget(object):
    """Multivariate normal target, the only target family the reference's drivers use.

    V(q)    = -scipy.stats.multivariate_normal.logpdf(q, q0, cov0)          (case1-script.py:39-43, utils.py:213-218)
            = 0.5 (q-q0)^T P (q-q0) + 0.5 (D ln 2pi + ln det cov0)          (closed form; SURVEY 8a-3)
    dVdq(q) = np.dot(inv_cov0, q-q0),  inv_cov0 = np.linalg.inv(cov0)       (case1-script.py:36, 45-49)
    """

    def __init__(self, q0, cov0):
        self.q0 = np.asarray(q0, dtype=float)
        self.cov0 = np.asarray(cov0, dtype=float)
        self.D = self.q0.shape[0]
        self.inv_cov0 = np.linalg.inv(self.cov0)
        sign, logdet = np.linalg.slogdet(self.cov0)
        assert sign > 0
        self.const = 0.5 * (self.D * math.log(2.0 * math.pi) + logdet)

    def V(self, q):
        d = q - self.q0
        return 0.5 * np.dot(d, np.dot(self.inv_cov0, d)) + self.const

    def dVdq(self, q):
        return np.dot(self.inv_cov0, (q - self.q0))


def equicorrelated_cov(D, rho):
    """cov0 = (1-rho) I + rho 11^T   (case3-script.py:31-33)."""
    cov0 = np.diag(np.ones(D)) * (1 - rho)
    cov0 += rho
    return cov0


# --------------------------------------------------------------------------------------------------
# Draw sources.  The reference consumes the process-global np.random stream in a fixed order
# (SURVEY 8a-6/7); a draw source reproduces that order and records a structured tape for the GPU.
# --------------------------------------------------------------------------------------------------
class NumpyDraws(object):
    """Draws with the very calls the reference makes, so that equal seeds give equal streams.

    p_sample : np.random.multivariate_normal(np.zeros(D), cov_p, size=1)[0]   (samplers.py:825-829)
    randint  : np.random.randint(low=, high=, size=1)[0]                      (samplers.py:441, 608)
    random   : np.random.random(1) / np.random.random()                       (samplers.py:461, 748, 773)
    """

    def __init__(self, D, cov_p=None):
        self.D = D
        self.cov_p = np.diag(np.ones(D)) if cov_p is None else np.asarray(cov_p, dtype=float)

    def p_sample(self):
        return np.random.multivariate_normal(np.zeros(self.D), self.cov_p, size=1)[0]

    def randint(self, low, high):
        return int(np.random.randint(low=low, high=high, size=1)[0])

    def random(self):
        return float(np.random.random(1)[0])


class TapeDraws(object):
    """Replays a flat tape of ("p", vec) / ("i", int) / ("u", float) entries (oracle/ref_shim.DrawRecorder)."""

    def __init__(self, tape):
        self.tape = tape
        self.pos = 0

    def _next(self, kind):
        k, v = self.tape[self.pos]
        assert k == kind, "tape order mismatch at %d: wanted %s got %s" % (self.pos, kind, k)
        self.pos += 1
        return v

    def p_sample(self):
        return np.array(self._next("p"), dtype=float)

    def randint(self, low, high):
        return int(self._next("i"))

    def random(self):
        return float(self._next("u"))

    def exhausted(self):
        return self.pos == len(self.tape)


class RecordingDraws(object):
    """Wraps another draw source and keeps what it returned, in order."""

    def __init__(self, inner):
        self.inner = inner
        self.tape = []

    def p_sample(self):
        v = self.inner.p_sample()
        self.tape.append(("p", np.array(v, dtype=float)))
        return v

    def randint(self, low, high):
        v = self.inner.randint(low, high)
        self.tape.append(("i", int(v)))
        return v

    def random(self):
        v = self.inner.random()
        self.tape.append(("u", float(v)))
        return v


# --------------------------------------------------------------------------------------------------
# L1 primitives  (samplers.py:811-839)
# --------------------------------------------------------------------------------------------------
def kinetic(p, inv_cov_p):
    """K(p) = p^T M^-1 p / 2   (samplers.py:811-817)."""
    return np.dot(p, np.dot(inv_cov_p, p)) / 2.


def leap_frog(p_old, q_old, dt, inv_cov_p, dVdq):
    """One leapfrog step exactly as written, two gradient calls, force multiplied by M^-1, q moved by p
    (samplers.py:831-839; quirk Q9)."""
    p_half = p_old - dt * np.dot(inv_cov_p, dVdq(q_old)) / 2.
    q_new = q_old + dt * p_half
    p_new = p_half - dt * np.dot(inv_cov_p, dVdq(q_new)) / 2.
    return p_new, q_new


def leap_frog_batch(p_old, q_old, dt, inv_cov_p, tgt):
    """``leap_frog`` (samplers.py:831-839) applied to every row of p_old / q_old at once (same statements, same order;
    rows are independent chains).  ``tgt``: MVNTarget.  Checked against the row-by-row form in tests/test_oracle_golden.py."""
    def dVdq(q):                                                            # case1-script.py:45-49, row-wise
        return np.dot(q - tgt.q0, tgt.inv_cov0.T)
    p_half = p_old - dt * np.dot(dVdq(q_old), inv_cov_p.T) / 2.
    q_new = q_old + dt * p_half
    p_new = p_half - dt * np.dot(dVdq(q_new), inv_cov_p.T) / 2.
    return p_new, q_new


def one_iteration_batch(tgt, q_init, p, L, u, dt, cov_p=None):
    """One iteration of ``gen_sample_random`` (samplers.py:428-472) for B independent (start point, momentum, length,
    uniform) tuples: returns dict(q_prop, p_prop, E_init, dE, decision).  Rows with L[b] < max(L) stop early."""
    q_init = np.asarray(q_init, dtype=float)
    B, D = q_init.shape
    cov_p = np.diag(np.ones(D)) if cov_p is None else np.asarray(cov_p, dtype=float)
    inv_cov_p = np.linalg.inv(cov_p)

    def E(q, pp):                                                           # samplers.py:819-823, row-wise
        d = q - tgt.q0
        return 0.5 * np.einsum("bi,bi->b", d, np.dot(d, tgt.inv_cov0.T)) + tgt.const + \
            0.5 * np.einsum("bi,bi->b", pp, np.dot(pp, inv_cov_p.T))
    q = q_init.copy()
    pp = np.asarray(p, dtype=float).copy()
    L = np.asarray(L).astype(int)
    E_init = E(q, pp)
    for l in range(1, int(L.max()) + 1):                                    # samplers.py:448-449
        on = L >= l
        pn, qn = leap_frog_batch(pp[on], q[on], dt, inv_cov_p, tgt)
        pp[on] = pn
        q[on] = qn
    dE = E(q, pp) - E_init                                                  # samplers.py:455-459
    with np.errstate(divide="ignore"):
        lnu = np.log(np.asarray(u, dtype=float))                            # samplers.py:461
    decision = ((dE < 0) | (lnu < -dE)).astype(np.int32)                    # samplers.py:462
    return dict(q_prop=q, p_prop=pp, E_init=E_init, dE=dE, decision=decision)


class Result(object):
    """Plain attribute bag mirroring the sampler attributes (samplers.py:31-50, 359-360)."""
    pass


# --------------------------------------------------------------------------------------------------
# Random-trajectory-length sampler  (samplers.py:387-491)
# --------------------------------------------------------------------------------------------------
def gen_sample_random(D, V, dVdq, q_start, draws, Nchain, Niter, thin_rate=1, warm_up_num=0,
                      dt=0.1, L_low=5, L_high=20, cov_p=None, N_save_chain0=0, record=False):
    """Restatement of ``HMC_sampler.gen_sample_random`` (samplers.py:387-491).

    Returns a Result with q_chain (Nchain, L_chain, D), E_chain/dE_chain (Nchain, L_chain, 1), accept_R,
    accept_R_warm_up, N_total_steps, phi_q, decision_chain, and -- when ``record`` -- the structured
    per-chain tape (p_tape[Nchain, Niter+1, D], L_tape[Nchain, Niter], u_tape[Nchain, Niter]) plus
    per-iteration teacher-forcing records (q_init, q_prop, dE, decision).
    """
    q_start = np.asarray(q_start, dtype=float)
    assert q_start.shape[0] == Nchain                                       # samplers.py:396
    cov_p = np.diag(np.ones(D)) if cov_p is None else np.asarray(cov_p, dtype=float)
    inv_cov_p = np.linalg.inv(cov_p)                                        # samplers.py:352-356
    L_chain = 1 + ((Niter - warm_up_num) // thin_rate)                      # samplers.py:31
    res = Result()
    res.L_chain = L_chain
    res.q_chain = np.zeros((Nchain, L_chain, D), dtype=float)               # samplers.py:33
    res.E_chain = np.zeros((Nchain, L_chain, 1), dtype=float)               # samplers.py:359
    res.dE_chain = np.zeros((Nchain, L_chain, 1), dtype=float)              # samplers.py:360
    res.N_total_steps = 0
    save_chain = N_save_chain0 > 0
    if save_chain:
        res.decision_chain = np.zeros((N_save_chain0 + 1, 1), dtype=int)    # samplers.py:399
        res.phi_q = []
    if record:
        res.p_tape = np.zeros((Nchain, Niter + 1, D))
        res.L_tape = np.zeros((Nchain, Niter), dtype=np.int32)
        res.u_tape = np.zeros((Nchain, Niter))
        res.q_init = np.zeros((Nchain, Niter, D))
        res.q_prop = np.zeros((Nchain, Niter, D))
        res.p_prop = np.zeros((Nchain, Niter, D))
        res.dE_iter = np.zeros((Nchain, Niter))
        res.E_init_iter = np.zeros((Nchain, Niter))
        res.decision = np.zeros((Nchain, Niter), dtype=np.int32)

    def E(q, p):                                                            # samplers.py:819-823
        return V(q) + kinetic(p, inv_cov_p)

    accept_counter_warm_up = 0
    accept_counter = 0
    for m in range(Nchain):                                                 # samplers.py:410
        res.q_chain[m, 0, :] = q_start[m]
        q_tmp = q_start[m]
        p_tmp = draws.p_sample()                                            # samplers.py:415
        if record:
            res.p_tape[m, 0] = p_tmp
        E_initial = E(q_tmp, p_tmp)
        res.N_total_steps += 1
        res.E_chain[m, 0, 0] = E_initial
        res.dE_chain[m, 0, 0] = 0
        E_previous = E_initial
        for i in range(1, Niter + 1):                                       # samplers.py:428
            q_initial = q_tmp
            p_tmp = draws.p_sample()                                        # samplers.py:431
            E_initial = E(q_tmp, p_tmp)
            res.N_total_steps += 1
            if i >= warm_up_num:                                            # samplers.py:436-438
                res.E_chain[m, (i - warm_up_num) // thin_rate, 0] = E_initial
                res.dE_chain[m, (i - warm_up_num) // thin_rate, 0] = E_initial - E_previous
            L_random = draws.randint(L_low, L_high)                         # samplers.py:441 (high exclusive, Q5)
            if record:
                res.p_tape[m, i] = p_tmp
                res.L_tape[m, i - 1] = L_random
                res.q_init[m, i - 1] = q_initial
                res.E_init_iter[m, i - 1] = E_initial
            if save_chain and (m == 0) and (i < (N_save_chain0 + 1)):
                phi_q_tmp = np.zeros((L_random + 1, 2))
                phi_q_tmp[0, :] = q_tmp[:2]
            for l in range(1, L_random + 1):                                # samplers.py:448-452
                p_tmp, q_tmp = leap_frog(p_tmp, q_tmp, dt, inv_cov_p, dVdq)
                res.N_total_steps += L_random * D                           # Q3
                if save_chain and (m == 0) and (i < (N_save_chain0 + 1)):
                    phi_q_tmp[l, :] = q_tmp[:2]
            E_final = E(q_tmp, p_tmp)                                       # samplers.py:455
            res.N_total_steps += 1
            dE = E_final - E_initial
            E_previous = E_initial                                          # samplers.py:460
            u = draws.random()
            lnu = np.log(u) if u > 0 else -np.inf                           # samplers.py:461
            accepted = (dE < 0) or (lnu < -dE)                              # samplers.py:462
            if record:
                res.u_tape[m, i - 1] = u
                res.q_prop[m, i - 1] = q_tmp
                res.p_prop[m, i - 1] = p_tmp
                res.dE_iter[m, i - 1] = dE
                res.decision[m, i - 1] = 1 if accepted else 0
            if accepted:
                if save_chain and (m == 0) and (i < (N_save_chain0 + 1)):
                    res.decision_chain[i - 1, 0] = 1
                if i >= warm_up_num:
                    res.q_chain[m, (i - warm_up_num) // thin_rate, :] = q_tmp
                    accept_counter += 1
                else:
                    accept_counter_warm_up += 1
            else:
                # Q4: negative index while i < warm_up_num, exactly as written (samplers.py:471)
                res.q_chain[m, (i - warm_up_num) // thin_rate, :] = q_initial
                q_tmp = q_initial
            if save_chain and (m == 0) and (i < (N_save_chain0 + 1)):
                res.phi_q.append(phi_q_tmp)
    res.accept_R_warm_up = None
    if warm_up_num > 0:                                                     # samplers.py:484-488
        res.accept_R_warm_up = accept_counter_warm_up / float(Nchain * warm_up_num)
    res.accept_R = accept_counter / float(Nchain * (Niter - warm_up_num + 1))
    res.accept_counter = accept_counter
    res.accept_counter_warm_up = accept_counter_warm_up
    return res


# --------------------------------------------------------------------------------------------------
# NUTS index helpers: literal restatements (utils.py:222-304, 367-385) and closed forms (SURVEY 8a-7)
# --------------------------------------------------------------------------------------------------
def find_next(table):
    """First empty (-1) slot (utils.py:222-228)."""
    for i, e in enumerate(table):
        if e == -1:
            return i
    return None


def retrieve_save_index(table, l):
    """Slot holding point number l (utils.py:230-237)."""
    for i, m in enumerate(table):
        if m == l:
            return i
    return None


def _power_of_two(r):
    return (r & (r - 1)) == 0                                               # utils.py:239-244, 306-311


def check_points(m):
    """Points against which point m (even) is U-turn checked (utils.py:246-283)."""
    assert (m % 2) == 0
    r = int(m)
    while (not _power_of_two(r)) and r > 2:
        d_last = int(math.floor(math.log2(r)))
        r -= 2 ** d_last
    pow_tmp = int(round(math.log2(r)))
    start = m - r + 1
    pts = [start]
    tmp = start
    while pow_tmp > 1:
        pow_tmp -= 1
        tmp += 2 ** pow_tmp
        pts.append(tmp)
    return np.asarray(pts)


def release(m, l):
    """True if check point l can be freed after the check at m (utils.py:286-304, 367-385)."""
    r_m, r_l = int(m), int(l)
    d_last = int(math.floor(math.log2(r_m)))
    while (not _power_of_two(r_m)) and r_m > 4:
        tmp = 2 ** d_last
        r_m -= tmp
        r_l -= tmp
        d_last = int(math.floor(math.log2(r_m)))
    return (r_m >= 4) and (r_l > 1)


def trailing_zeros(m):
    return (m & -m).bit_length() - 1


def check_points_closed(m):
    """Closed form: {m - 2^j + 1 : j = tz(m) .. 1}  (SURVEY 8a-7; equals check_points(m))."""
    return [m - (1 << j) + 1 for j in range(trailing_zeros(m), 0, -1)]


def release_closed(m, l):
    """Closed form: released unless l == 1 or l is the first (largest sub-tree) check point of m."""
    return (l > 1) and (l != m - (1 << trailing_zeros(m)) + 1)


def slot_closed(l):
    """A collision-free slot for odd point l: popcount((l-1)>>1)  (SURVEY 8a-7)."""
    return bin((l - 1) >> 1).count("1")


# --------------------------------------------------------------------------------------------------
# NUTS sampler  (samplers.py:495-808)
# --------------------------------------------------------------------------------------------------
class DMaxExceeded(AssertionError):
    """samplers.py:596-598 -- `assert False` when d > d_max-1 (quirk Q7)."""
    pass


def gen_sample_NUTS(D, V, dVdq, q_start, draws, Nchain, Niter, thin_rate=1, warm_up_num=0,
                    dt=0.1, d_max=10, cov_p=None, record=False, on_dmax="assert"):
    """Restatement of ``HMC_sampler.gen_sample_NUTS`` (samplers.py:495-808).

    ``on_dmax="stop"`` is this repo's benchmark extension (SURVEY H6): depth overflow ends the doubling
    loop keeping the live point, instead of aborting the whole run.
    With ``record`` the per-chain structured tapes are kept: p_tape[Nchain, Niter+1, D], and per chain the
    flat lists dir_tape / u_tape in consumption order, plus n_leapfrog[Nchain, Niter] and depth[Nchain, Niter], and per
    (chain, iteration) what the tree builder met: n_instab_iter (|E - E_initial| > 1000 rejects), n_uturn_sub_iter
    (sub-trajectory U-turn rejects), dmax_iter (the depth limit was hit), max_exp_arg_iter (largest |argument| of the exp()
    calls of the progressive-sampling and biased-choice weights) and nonfinite_iter (some weight was inf or NaN).  Recording
    changes nothing the sampler computes.
    """
    q_start = np.asarray(q_start, dtype=float)
    assert q_start.shape[0] == Nchain                                       # samplers.py:510
    cov_p = np.diag(np.ones(D)) if cov_p is None else np.asarray(cov_p, dtype=float)
    inv_cov_p = np.linalg.inv(cov_p)
    L_chain = 1 + ((Niter - warm_up_num) // thin_rate)
    res = Result()
    res.L_chain = L_chain
    res.q_chain = np.zeros((Nchain, L_chain, D), dtype=float)
    res.E_chain = np.zeros((Nchain, L_chain, 1), dtype=float)
    res.dE_chain = np.zeros((Nchain, L_chain, 1), dtype=float)
    res.N_total_steps = 0
    res.n_instability = 0
    res.n_dmax = 0
    if record:
        res.p_tape = np.zeros((Nchain, Niter + 1, D))
        res.dir_tape = [[] for _ in range(Nchain)]
        res.u_tape = [[] for _ in range(Nchain)]
        res.n_leapfrog = np.zeros((Nchain, Niter), dtype=np.int64)
        res.depth = np.zeros((Nchain, Niter), dtype=np.int32)
        res.n_instab_iter = np.zeros((Nchain, Niter), dtype=np.int32)
        res.n_uturn_sub_iter = np.zeros((Nchain, Niter), dtype=np.int32)
        res.dmax_iter = np.zeros((Nchain, Niter), dtype=bool)
        res.max_exp_arg_iter = np.zeros((Nchain, Niter))
        res.nonfinite_iter = np.zeros((Nchain, Niter), dtype=bool)

    def note_weights(m, i, args, values):
        """record only: the exp() arguments and the weights of one progressive-sampling or biased-choice step"""
        res.max_exp_arg_iter[m, i - 1] = max(res.max_exp_arg_iter[m, i - 1], max(abs(v) for v in args))
        if not all(np.isfinite(v) for v in values):
            res.nonfinite_iter[m, i - 1] = True

    def E(q, p):
        return V(q) + kinetic(p, inv_cov_p)

    q_save = np.zeros((d_max + 1, D), dtype=float)                          # samplers.py:519-520
    p_save = np.zeros((d_max + 1, D), dtype=float)
    save_index_table = np.ones(d_max + 1, dtype=int) * -1                   # samplers.py:535

    for m in range(Nchain):                                                 # samplers.py:545
        res.q_chain[m, 0, :] = q_start[m]
        q_tmp = q_start[m]
        p_tmp = draws.p_sample()                                            # samplers.py:550
        if record:
            res.p_tape[m, 0] = p_tmp
        E_initial = E(q_tmp, p_tmp)
        res.N_total_steps += 1
        res.E_chain[m, 0, 0] = E_initial
        res.dE_chain[m, 0, 0] = 0
        E_previous = E_initial
        for i in range(1, Niter + 1):                                       # samplers.py:563
            p_tmp = draws.p_sample()                                        # samplers.py:565
            if record:
                res.p_tape[m, i] = p_tmp
            E_initial = E(q_tmp, p_tmp)
            res.N_total_steps += 1
            if i >= warm_up_num:                                            # samplers.py:571-573
                res.E_chain[m, (i - warm_up_num) // thin_rate, 0] = E_initial
                res.dE_chain[m, (i - warm_up_num) // thin_rate, 0] = E_initial - E_previous
            live_point_q_old = q_tmp                                        # samplers.py:577-587
            left_q, left_p = q_tmp, -p_tmp
            right_q, right_p = q_tmp, p_tmp
            E_max_old = E_initial
            pi_old = 1
            left_terminate = False
            right_terminate = False
            d = 0
            nleap = 0
            while (not left_terminate) or (not right_terminate):            # samplers.py:595 (Q6)
                if d > d_max - 1:                                           # samplers.py:596-598 (Q7)
                    res.n_dmax += 1
                    if record:
                        res.dmax_iter[m, i - 1] = True
                    if on_dmax == "assert":
                        raise DMaxExceeded("Doubling number d exceeds d_max = %d" % d_max)
                    break
                save_index_table[:] = -1                                    # samplers.py:601
                L_new_sub = 2 ** d
                u_dir = draws.randint(0, 2)                                 # samplers.py:608
                if record:
                    res.dir_tape[m].append(u_dir)
                if u_dir == 0:                                              # samplers.py:611-614
                    p_tmp, q_tmp = leap_frog(right_p, right_q, dt, inv_cov_p, dVdq)
                else:
                    p_tmp, q_tmp = leap_frog(left_p, left_q, dt, inv_cov_p, dVdq)
                res.N_total_steps += D
                nleap += 1
                live_point_q_new = q_tmp
                E_max_new_now = E(q_tmp, p_tmp)                             # samplers.py:618
                pi_new = 1
                res.N_total_steps += 1
                save_index = find_next(save_index_table)                    # samplers.py:623-626
                q_save[save_index, :] = q_tmp
                p_save[save_index, :] = p_tmp
                save_index_table[save_index] = 1
                trajectory_reject = False
                if L_new_sub > 1:
                    for k in range(1, L_new_sub):                           # samplers.py:637
                        p_tmp, q_tmp = leap_frog(p_tmp, q_tmp, dt, inv_cov_p, dVdq)
                        res.N_total_steps += D
                        nleap += 1
                        E_tmp = E(q_tmp, p_tmp)                             # samplers.py:643
                        res.N_total_steps += 1
                        if np.abs(E_tmp - E_initial) > 1000:                # samplers.py:647-651
                            trajectory_reject = True
                            q_tmp = live_point_q_old
                            res.n_instability += 1
                            if record:
                                res.n_instab_iter[m, i - 1] += 1
                            break
                        if ((k + 1) % 2) == 1:                              # samplers.py:654-658
                            save_index = find_next(save_index_table)
                            q_save[save_index, :] = q_tmp
                            p_save[save_index, :] = p_tmp
                            save_index_table[save_index] = k + 1
                        else:
                            for l in check_points(k + 1):                   # samplers.py:699-736
                                save_index = retrieve_save_index(save_index_table, l)
                                q_check = q_save[save_index, :]
                                p_check = p_save[save_index, :]
                                if u_dir == 0:
                                    left_q_tmp, left_p_tmp = q_check, -p_check
                                    right_q_tmp, right_p_tmp = q_tmp, p_tmp
                                else:
                                    left_q_tmp, left_p_tmp = q_tmp, p_tmp
                                    right_q_tmp, right_p_tmp = q_check, -p_check
                                Dq_tmp = right_q_tmp - left_q_tmp
                                right_terminate_tmp = np.dot(Dq_tmp, right_p_tmp) < 0
                                left_terminate_tmp = np.dot(-Dq_tmp, left_p_tmp) < 0
                                if left_terminate_tmp and right_terminate_tmp:    # Q6: both
                                    trajectory_reject = True
                                    if record:
                                        res.n_uturn_sub_iter[m, i - 1] += 1
                                    q_tmp = live_point_q_old
                                    break
                                if (l > 1) and release(k + 1, l):
                                    save_index_table[save_index] = -1
                        if trajectory_reject:                               # samplers.py:739-740
                            break
                        E_max_new_previous = E_max_new_now                  # samplers.py:743-751
                        E_max_new_now = max(E_max_new_previous, E_tmp)
                        numerator = np.exp(-(E_tmp - E_max_new_now))
                        pi_new = numerator + np.exp(E_max_new_now - E_max_new_previous) * pi_new
                        r = numerator / pi_new
                        u = draws.random()
                        if record:
                            res.u_tape[m].append(u)
                            note_weights(m, i, (E_tmp - E_max_new_now, E_max_new_now - E_max_new_previous),
                                         (numerator, pi_new, r))
                        if u < r:
                            live_point_q_new = q_tmp
                if trajectory_reject:                                       # samplers.py:754-755
                    break
                if u_dir == 0:                                              # samplers.py:758-761
                    right_q, right_p = q_tmp, p_tmp
                else:
                    left_q, left_p = q_tmp, p_tmp
                r = np.exp(-(E_max_new_now - E_max_old)) * pi_old / pi_new  # samplers.py:766 (Q8)
                E_max_old_previous = E_max_old
                E_max_old = max(E_max_old_previous, E_max_new_now)
                pi_old = np.exp(-(E_max_new_now - E_max_old)) * pi_new + \
                    np.exp(-(E_max_old_previous - E_max_old)) * pi_old      # samplers.py:771
                A = min(1, r)
                u = draws.random()                                          # samplers.py:773
                if record:
                    res.u_tape[m].append(u)
                    note_weights(m, i, (E_max_new_now - E_max_old_previous, E_max_new_now - E_max_old,
                                        E_max_old_previous - E_max_old), (r, pi_old))
                if u < A:
                    live_point_q_old = live_point_q_new
                q_tmp = live_point_q_old
                Dq = right_q - left_q                                       # samplers.py:779-781
                right_terminate = np.dot(Dq, right_p) < 0
                left_terminate = np.dot(-Dq, left_p) < 0
                d += 1
            if d > d_max - 1 and on_dmax == "stop":
                q_tmp = live_point_q_old
            E_previous = E_initial                                          # samplers.py:787
            if record:
                res.n_leapfrog[m, i - 1] = nleap
                res.depth[m, i - 1] = d
            if i >= warm_up_num:                                            # samplers.py:790-791
                res.q_chain[m, (i - warm_up_num) // thin_rate, :] = q_tmp
    res.accept_R_warm_up = 1. if warm_up_num > 0 else None                  # samplers.py:800-805
    res.accept_R = 1.
    return res


# --------------------------------------------------------------------------------------------------
# Diagnostics  (utils.py:77-179)
# --------------------------------------------------------------------------------------------------
def variogram(chains, var_num, t_lag):
    """V_t (utils.py:161-179).  chains: list of (n, D) arrays."""
    m = len(chains)
    n = chains[0].shape[0]
    V_t = 0.
    for i in range(m):
        chain_tmp = chains[i][:, var_num]
        V_t += np.sum(np.square(chain_tmp[t_lag:] - chain_tmp[:-t_lag]))
    V_t /= float(m * (n - t_lag))
    return V_t


def _split_chains(q_chain, thin_rate, warm_up_num):
    """utils.py:88-104 (python-2 `/` is integer division at :102)."""
    Nchain = q_chain.shape[0]
    chains = []
    n = None
    for m in range(Nchain):
        c = q_chain[m, warm_up_num:, :][::thin_rate, :]
        L_chain = c.shape[0]
        if (L_chain % 2) != 0:
            c = c[:L_chain - 1]
        n = L_chain // 2
        chains.append(c[:n])
        chains.append(c[n:])
    return chains, n


def convergence_stats(q_chain, thin_rate=5, warm_up_num=0):
    """Literal restatement of utils.convergence_stats (utils.py:77-159), quirks Q1 and Q2 included."""
    Nchain, Niter, D = q_chain.shape
    assert Nchain > 1                                                       # utils.py:85
    chains, n = _split_chains(q_chain, thin_rate, warm_up_num)
    m = len(chains)
    var_within = np.empty((m, D))
    for j in range(m):
        var_within[j, :] = np.std(chains[j], ddof=1, axis=0)                # Q1: std, not var (utils.py:111)
    W = np.mean(var_within, axis=0)
    mean_within = np.empty((m, D))
    for j in range(m):
        mean_within[j, :] = np.mean(chains[j], axis=0)
    mean_all = np.mean(mean_within, axis=0)
    B = np.sum(np.square(mean_within - mean_all), axis=0) * n / float(m - 1)    # utils.py:120
    var = W * (n - 1) / float(n) + B / float(n)                             # utils.py:123
    R = np.sqrt(var / W)                                                    # utils.py:126
    n_eff = np.zeros(D, dtype=float)
    for i in range(D):                                                      # utils.py:130-157
        V_t1 = variogram(chains, i, 1)
        V_t2 = variogram(chains, i, 2)
        rho_t1 = 1. - V_t1 / (2 * var[i])
        rho_t2 = 1. - V_t2 / (2 * var[i])
        if (rho_t1 < 1e-2) or (rho_t1 < 1e-2):                              # Q2 (utils.py:136)
            sum_rho = 0
        else:
            rho_t = [rho_t1, rho_t2]
            t = 1
            while (t < n - 2):
                V_t = variogram(chains, i, t + 2)
                rho_t.append(1 - V_t / (2 * var[i]))
                if ((t % 2) == 1) & ((rho_t[t] + rho_t[t + 1]) < 0):
                    break
                t += 1
            sum_rho = np.sum(rho_t[:t])
            if sum_rho < 0:
                sum_rho = 0
        n_eff[i] = m * n / (1 + 2 * sum_rho)
    return R, n_eff


def rhat_moments(q_chain, thin_rate=1, warm_up_num=0):
    """Vectorised split-chain moments: returns (n, m, std_j[m, D], mean_j[m, D]) (utils.py:88-118)."""
    c = q_chain[:, warm_up_num:, :][:, ::thin_rate, :]
    L_chain = c.shape[1]
    if (L_chain % 2) != 0:
        c = c[:, :L_chain - 1]
    n = L_chain // 2
    halves = c.reshape(c.shape[0] * 2, n, c.shape[2])                       # chain-major, first half then second
    return n, halves.shape[0], np.std(halves, ddof=1, axis=1), np.mean(halves, axis=1), halves


def finish_from_variogram(var, V_by_lag, m, n):
    """The truncation rule of utils.py:130-157 applied to a precomputed table V_by_lag[t] (index t = lag,
    entries for t >= 1; NaN/absent beyond what was computed raises IndexError so callers know to extend)."""
    D = var.shape[0]
    n_eff = np.zeros(D)
    T_used = np.zeros(D, dtype=np.int64)
    for i in range(D):
        rho = lambda t: 1. - V_by_lag[t, i] / (2 * var[i])
        rho_t1 = rho(1)
        if (rho_t1 < 1e-2) or (rho_t1 < 1e-2):
            sum_rho = 0
            T_used[i] = 0
        else:
            rho_t = [rho_t1, rho(2)]
            t = 1
            while (t < n - 2):
                rho_t.append(rho(t + 2))
                if ((t % 2) == 1) & ((rho_t[t] + rho_t[t + 1]) < 0):
                    break
                t += 1
            sum_rho = np.sum(rho_t[:t])
            if sum_rho < 0:
                sum_rho = 0
            T_used[i] = t + 2 if t < n - 2 else t + 1
        n_eff[i] = m * n / (1 + 2 * sum_rho)
    return n_eff, T_used


def convergence_stats_fast(q_chain, thin_rate=5, warm_up_num=0, max_lag=None):
    """Vectorised restatement of utils.convergence_stats; same numbers (tests require 1e-12)."""
    Nchain = q_chain.shape[0]
    assert Nchain > 1
    n, m, std_j, mean_j, halves = rhat_moments(q_chain, thin_rate, warm_up_num)
    W = np.mean(std_j, axis=0)
    mean_all = np.mean(mean_j, axis=0)
    B = np.sum(np.square(mean_j - mean_all), axis=0) * n / float(m - 1)
    var = W * (n - 1) / float(n) + B / float(n)
    R = np.sqrt(var / W)
    D = q_chain.shape[2]
    T = n - 1 if max_lag is None else min(max_lag, n - 1)
    V = np.full((max(T, 2) + 1, D), np.nan)
    for t in range(1, T + 1):
        d = halves[:, t:, :] - halves[:, :-t, :]
        V[t] = np.sum(np.square(d), axis=(0, 1)) / float(m * (n - t))
    n_eff, _ = finish_from_variogram(var, V, m, n)
    return R, n_eff


# --------------------------------------------------------------------------------------------------
# Work accounting closed forms (SURVEY 8a-9; samplers.py:417, 435, 450, 456, 552, 570, 615, 620, 640, 644)
# --------------------------------------------------------------------------------------------------
def n_total_steps_random(Nchain, Niter, D, L_tape):
    return Nchain * (1 + 2 * Niter) + D * int(np.sum(np.asarray(L_tape, dtype=np.int64) ** 2))


def n_total_steps_nuts(Nchain, Niter, D, n_leapfrog_total):
    return Nchain * (1 + Niter) + (D + 1) * int(n_leapfrog_total)
