"""Large-D Random path with a dense momentum metric against the identity metric: BASELINE config-5 settings (131,072 chains, Niter 2,
dt 0.1, L in [100, 500); target as profiles/bigd_any_d.py) at D = 2048 and 4096, both splits, the two metrics alternating in one
process; plus a short-trajectory row (L in [5, 20)), where the per-trajectory products weigh most.  The dense metric is the identity
with four eigenvalues in [0.7, 1.4] along random directions (rotated: a dense matrix).

Per run: launch time from CUDA events (H.kernel_ms; every instantiation has had a warm-up launch), gradient evaluations per second
(sum L + starts, as profiles/bigd_any_d.py counts them), and hmc_random_workspace_bytes.  Per configuration, one more run with
HMC_B200_BIGD_TIMING=1 gives the per-pass split (CUDA events around the kernels of passes 4..11: main GEMM, events kernel, and the
trajectory end -- with a dense metric the product stage, gather + three GEMMs, and the finish kernel).  Device name and power limit
are read in the same call.

  python profiles/bigd_metric.py [--out FILE.json] [--d 2048,4096] [--chains N]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "understanding-hmc_b200"), os.path.join(ROOT, "profiles")):
    sys.path.insert(0, p)
import numpy as np
import torch
import hmc_b200_lib as L
import samplers as S
import utils as U
from bigd_any_d import target, device_info

PRECS = ("fp16x2", "bf16x3")


def dense_cov_p(D, seed=1, k=4):
    rng = np.random.RandomState(seed)
    Vk, _ = np.linalg.qr(rng.standard_normal((D, k)))
    lam = np.exp(rng.uniform(np.log(0.7), np.log(1.4), k))
    c = np.eye(D) + (Vk * (lam - 1.0)) @ Vk.T
    return 0.5 * (c + c.T)


def workspace_bytes(D, Nc, dense):
    a = L.RandomArgs()
    a.dtype, a.kernel, a.Nchain, a.Niter, a.iter_begin, a.iter_end = L.HMC_F32, L.KERNEL_BIGD, Nc, 2, 0, 2
    a.thin_rate, a.L_low, a.L_high = 1, 1, 2
    a.target.D, a.target.D_pad = D, (D + 3) // 4 * 4
    if dense:                                       # (addresses only: the size does not read the matrices)
        a.target.Pt = a.target.Mit = a.target.Lct = 0x1000
    return int(L.load().hmc_random_workspace_bytes(a))


def run(D, Nc, prec, spec, lam, cov_p, Llo, Lhi, timing=False):
    q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), Nc, device="cuda", seed=1)
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=2, warm_up_num=1, sampler_type="Random", dt=0.1, L_low=Llo, L_high=Lhi,
                      dtype="float32", kernel="bigd", tc_precision=prec, seed=3, target=spec, cov_p=cov_p)
    line = None
    if timing:                                      # the library prints the split on stderr: catch file descriptor 2
        os.environ["HMC_B200_BIGD_TIMING"] = "1"
        sys.stderr.flush()
        saved = os.dup(2)
        with tempfile.TemporaryFile(mode="w+") as f:
            os.dup2(f.fileno(), 2)
            try:
                H.gen_sample(q0, verbose=False, quiet=True)
                torch.cuda.synchronize()
            finally:
                os.dup2(saved, 2)
                os.close(saved)
                del os.environ["HMC_B200_BIGD_TIMING"]
            f.seek(0)
            line = [x for x in f.read().splitlines() if x.startswith("[bigd timing]")]
    else:
        H.gen_sample(q0, verbose=False, quiet=True)
        torch.cuda.synchronize()
    ge = H.sum_L + Nc * 2
    t = H.kernel_ms * 1e-3
    rec = {"D": D, "chains": Nc, "metric": "identity" if cov_p is None else "dense", "L": [Llo, Lhi], "tc_precision": H.tc_precision,
           "kernel_ms": H.kernel_ms, "accept_R": H.accept_R, "grad_evals": ge, "grad_evals_per_s": ge / t,
           "workspace_bytes": workspace_bytes(D, Nc, cov_p is not None)}
    if timing:
        rec = {"D": D, "metric": rec["metric"], "L": [Llo, Lhi], "tc_precision": H.tc_precision, "per_pass": line}
    del H, q0
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results (default: stdout only)")
    ap.add_argument("--d", default="2048,4096")
    ap.add_argument("--chains", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"info": device_info(), "settings": "chains %d, Niter 2 (warm-up 1), dt 0.1; dense cov_p: I with 4 eigenvalues in "
                                              "[0.7, 1.4] along random directions" % args.chains, "runs": [], "per_pass": []}
    Ds = [int(x) for x in args.d.split(",")]
    spec, lam = target(Ds[0])
    cp = dense_cov_p(Ds[0])
    for prec in PRECS:                              # warm-up launch of each instantiation
        for c in (None, cp):
            run(Ds[0], 4096, prec, spec, lam, c, 10, 20)
    rows = [(D, 100, 500) for D in Ds] + [(Ds[0], 5, 20)]
    for D, Llo, Lhi in rows:
        spec, lam = target(D)
        cp = dense_cov_p(D)
        for prec in PRECS:
            for rep in range(args.reps):            # identity and dense alternate
                for c in (None, cp):
                    rec = run(D, args.chains, prec, spec, lam, c, Llo, Lhi)
                    print(json.dumps(rec), flush=True)
                    res["runs"].append(rec)
            for c in (None, cp):
                rec = run(D, args.chains, prec, spec, lam, c, Llo, Lhi, timing=True)
                print(json.dumps(rec), flush=True)
                res["per_pass"].append(rec)
    res["info_after"] = device_info()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
