"""NUTS on the large-D path (csrc/nuts_bigd.cu) at the BASELINE config-5 settings: dense target with a log-uniform spectrum on
[0.05, 100] and a random rotation (profiles/bigd_any_d.py), 131,072 chains, Niter 2, dt 0.1, d_max 10, on_dmax "stop", both
splits, at D = 1024, 1500 and 2048; and the generic NUTS kernel at D = 256 for scale.

Per run: launch time from CUDA events (H.kernel_ms; each instantiation had a warm-up launch), leapfrog steps per second, gradient
rows evaluated per second (the leapfrogs plus the gradient-only passes: chain and iteration starts, a doubling that switches
direction), algorithmic tensor rate (gradient rows x 2 D^2 / time) and executed rate (x Dp^2 x part products: every row of a row
block with a running chain is computed), passes, the mean fraction of running rows per pass, and the GEMM and step-kernel times
per pass (passes 4..11, CUDA events; the HMC_B200_BIGD_TIMING aid, a run of its own).  Device name, power limit and max SM clock
are read in the same call.

  python profiles/nuts_bigd.py [--out FILE.json] [--d 1024,1500,2048] [--chains N]
"""
import argparse
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "understanding-hmc_b200"), os.path.join(ROOT, "profiles")):
    sys.path.insert(0, p)
import numpy as np
import torch
import samplers as S
import utils as U
from bigd_any_d import device_info, target

PRECS = ("bf16x3", "fp16x2")
NPROD = {"fp16x2": 3, "bf16x3": 6}


def _run(D, Nc, prec, kernel, spec, lam, Niter=2, dt=0.1, d_max=10):
    q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), Nc, device="cuda", seed=1)
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, warm_up_num=Niter // 2, sampler_type="NUTS", dt=dt, d_max=d_max,
                      dtype="float32", kernel=kernel, tc_precision=prec, seed=3, target=spec, on_dmax="stop")
    H.gen_sample(q0, verbose=False)
    torch.cuda.synchronize()
    return H


def _captured(fn):
    """fn() with the process's stderr (the library's timing lines) captured."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            out = fn()
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        return out, tmp.read()


def measure(D, Nc, prec, kernel, spec, lam):
    H = _run(D, Nc, prec, kernel, spec, lam)
    t = H.kernel_ms * 1e-3
    Dp = (D + 31) // 32 * 32
    rec = {"D": D, "Dp": Dp, "chains": Nc, "kernel": H.nuts_kernel, "tc_precision": H.tc_precision if kernel == "bigd" else None,
           "kernel_ms": H.kernel_ms, "leapfrogs": H.n_leapfrog_total, "doublings": H.n_doublings, "d_max_hits": H.n_dmax,
           "instabilities": H.n_instability, "leapfrogs_per_s": H.n_leapfrog_total / t}
    del H
    if kernel == "bigd":
        os.environ["HMC_B200_BIGD_TIMING"] = "1"
        try:
            H2, err = _captured(lambda: _run(D, Nc, prec, kernel, spec, lam))
        finally:
            del os.environ["HMC_B200_BIGD_TIMING"]
        m = re.search(r"gemm ([0-9.]+) ms, step ([0-9.]+) ms per pass", err)
        n = re.search(r"passes=(\d+) gradient_rows=(\d+)", err)
        assert m and n, err
        passes, grads = int(n.group(1)), int(n.group(2))
        assert H2.n_leapfrog_total == rec["leapfrogs"]
        rec.update({"passes": passes, "gradient_rows": grads, "gradient_evals_per_s": grads / t,
                    "mean_running_row_fraction": grads / float(passes * Nc),
                    "algorithmic_tflops": grads * 2.0 * D * D / t / 1e12,
                    "tensor_tflops_executed_upper_bound": passes * ((Nc + 511) // 512 * 512) * 2.0 * Dp * Dp * NPROD[prec] / t / 1e12,
                    "gemm_ms_per_pass_4_11": float(m.group(1)), "step_ms_per_pass_4_11": float(m.group(2))})
        del H2
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results (default: stdout only)")
    ap.add_argument("--d", default="1024,1500,2048")
    ap.add_argument("--chains", type=int, default=131072)
    ap.add_argument("--generic-chains", type=int, default=16384)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"info": device_info(),
           "settings": "chains %d, Niter 2 (warm-up 1), dt 0.1, d_max 10, on_dmax stop, config-5 target (log-uniform spectrum on "
                       "[0.05, 100], random rotation)" % args.chains, "runs": []}
    Ds = [int(x) for x in args.d.split(",")]
    spec, lam = target(Ds[0])
    for prec in PRECS:                              # warm-up launch of each instantiation
        _run(Ds[0], 2048, prec, "bigd", spec, lam)
    for D in Ds:
        spec, lam = target(D)
        for prec in PRECS:
            rec = measure(D, args.chains, prec, "bigd", spec, lam)
            print(json.dumps(rec), flush=True)
            res["runs"].append(rec)
    spec, lam = target(256)                         # the generic NUTS kernel (warp per chain, F read from L2) at its largest D
    _run(256, 2048, None, "generic", spec, lam)
    rec = measure(256, args.generic_chains, None, "generic", spec, lam)
    print(json.dumps(rec), flush=True)
    res["generic_D256"] = rec
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
