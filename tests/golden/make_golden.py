"""Generates the committed golden fixtures by running the REAL reference (through oracle/ref_shim.py).

Run in the build container only (needs /root/reference):   python tests/golden/make_golden.py
Each fixture holds the inputs (target, q_start, the reference's own draws as structured tapes) and the
reference's outputs (q_chain, E_chain, dE_chain, acceptance, N_total_steps, R_q, n_eff_q, chain-0 trace).
Draw order per chain (SURVEY 8a-6/7): Random: p0, then per iteration p, L, u.  NUTS: p0, then per iteration
p followed by a data-dependent sequence of direction coins and uniforms.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_shim  # noqa: E402
from _util import CASES, pin_start  # noqa: E402


def split_tape(tape, sampler, Nchain, Niter, D):
    """Flat reference tape -> per-chain structured arrays."""
    p_tape = np.zeros((Nchain, Niter + 1, D))
    if sampler == "Random":
        L_tape = np.zeros((Nchain, Niter), dtype=np.int32)
        u_tape = np.zeros((Nchain, Niter))
        pos = 0
        for m in range(Nchain):
            k, v = tape[pos]; pos += 1
            assert k == "p"
            p_tape[m, 0] = v
            for i in range(Niter):
                (k1, v1), (k2, v2), (k3, v3) = tape[pos:pos + 3]; pos += 3
                assert (k1, k2, k3) == ("p", "i", "u")
                p_tape[m, i + 1] = v1; L_tape[m, i] = v2; u_tape[m, i] = v3
        assert pos == len(tape)
        return dict(p_tape=p_tape, L_tape=L_tape, u_tape=u_tape)
    dirs = [[] for _ in range(Nchain)]
    us = [[] for _ in range(Nchain)]
    np_seen = 0
    for k, v in tape:
        if k == "p":
            m, i = divmod(np_seen, Niter + 1)
            p_tape[m, i] = v
            np_seen += 1
        else:
            m = (np_seen - 1) // (Niter + 1)
            (dirs if k == "i" else us)[m].append(v)
    assert np_seen == Nchain * (Niter + 1)
    nd = max(len(x) for x in dirs); nu = max(len(x) for x in us)
    dir_tape = np.full((Nchain, nd), -1, dtype=np.int32)
    u_tape = np.full((Nchain, nu), np.nan)
    for m in range(Nchain):
        dir_tape[m, :len(dirs[m])] = dirs[m]
        u_tape[m, :len(us[m])] = us[m]
    return dict(p_tape=p_tape, dir_tape=dir_tape, u_tape=u_tape,
                n_dir=np.array([len(x) for x in dirs]), n_u=np.array([len(x) for x in us]))


def main():
    ru, rs = ref_shim.load_reference()
    only = set(sys.argv[1:])
    for (name, sampler, D, rho, Nchain, Niter, warm, thin, dt, extra, sscale, seed, nsave) in CASES:
        if only and name not in only:
            continue
        extra = dict(extra)
        q0 = np.zeros(D)
        cov0 = np.diag(np.ones(D)) * (1 - rho)
        cov0 += rho
        inv_cov0 = np.linalg.inv(cov0)

        def V(q):
            return -ru.normal_lnL(q, q0, cov0)

        def dVdq(q):
            return np.dot(inv_cov0, (q - q0))

        np.random.seed(seed)
        q_start = pin_start(name, ru.start_pts(q0, np.diag(np.ones(D)) * sscale, Nchain))
        dt_val = dt
        if isinstance(dt, str):
            dt_val = 0.05 + 0.1 * np.arange(D) / D
        cov_p = None
        if extra.pop("cov_p", None) == "diag":
            cov_p = np.diag(0.5 + np.arange(D) / float(D))
        H = rs.HMC_sampler(D, V, dVdq, Niter=Niter, Nchain=Nchain, sampler_type=sampler, dt=dt_val,
                           thin_rate=thin, warm_up_num=warm, cov_p=cov_p, **extra)
        with ref_shim.DrawRecorder(rs, H) as rec:
            H.gen_sample(q_start, N_save_chain0=nsave, verbose=False)
        H.compute_convergence_stats()
        out = dict(sampler=sampler, D=D, rho=rho, Nchain=Nchain, Niter=Niter, warm_up_num=warm, thin_rate=thin,
                   dt=np.asarray(dt_val, dtype=float), q0=q0, cov0=cov0, q_start=q_start,
                   cov_p=np.eye(D) if cov_p is None else cov_p,
                   q_chain=H.q_chain, E_chain=H.E_chain, dE_chain=H.dE_chain,
                   accept_R=H.accept_R, accept_R_warm_up=np.nan if H.accept_R_warm_up is None else H.accept_R_warm_up,
                   N_total_steps=H.N_total_steps, R_q=H.R_q, n_eff_q=H.n_eff_q, seed=seed, N_save_chain0=nsave)
        for k, v in extra.items():
            out[k] = v
        out.update(split_tape(rec.tape, sampler, Nchain, Niter, D))
        if nsave > 0:
            out["decision_chain"] = H.decision_chain
            out["phi_len"] = np.array([a.shape[0] for a in H.phi_q])
            out["phi_q"] = np.concatenate(H.phi_q, axis=0)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, os.path.getsize(path), "bytes; accept", H.accept_R, "Rhat med", np.median(H.R_q))

    if only:
        return
    # index-helper known answers straight from the reference functions (README:332-358 tables are their print-outs)
    cp = {m: ru.check_points(m).tolist() for m in range(2, 1025, 2)}
    rel = []
    for m in range(2, 1025, 2):
        for l in cp[m]:
            if l != 1:
                rel.append((m, l, bool(ru.release(m, l)), bool(ru.release_fast(m, l))))
    np.savez_compressed(os.path.join(HERE, "nuts_index_kat.npz"),
                        cp_m=np.array(sorted(cp)), cp_len=np.array([len(cp[m]) for m in sorted(cp)]),
                        cp_flat=np.concatenate([cp[m] for m in sorted(cp)]), release=np.array(rel, dtype=np.int64))
    print("nuts_index_kat ok")


if __name__ == "__main__":
    main()
