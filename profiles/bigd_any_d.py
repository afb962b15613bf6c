"""Large-D path at any D: BASELINE config-5 settings (131,072 chains, dt = 0.1, L in [100, 500), 2 iterations, dense target with a
log-uniform spectrum on [0.05, 100] and a random rotation, as profiles/run_bigd_once.py) at D on both sides of multiples of 256,
both splits, plus the generic kernel at D = 1000 on fewer chains for a speedup figure.

Per run: launch time from CUDA events (H.kernel_ms; every kernel instantiation has had a warm-up launch), gradient evaluations
per second with the true D, the algorithmic rate (sum L + starts) 2 D^2 / time, and the tensor FLOP executed with the padded
widths: (sum L + starts) 2 Dp^2 x part products, Dp = D rounded up to 32, the last column tile issued at its own width (rows of
finished chains in a still-live row block are not counted).  Device name and power limit are read in the same call.

  python profiles/bigd_any_d.py [--out FILE.json] [--d 1000,1024,...] [--chains N]
  python profiles/bigd_any_d.py --dump DIR     # q_chain / E_chain of seeded D = 512 and D = 1024 runs (both splits) as .npy,
                                               # to compare two builds output for output
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "understanding-hmc_b200")):
    sys.path.insert(0, p)
import numpy as np
import torch
import samplers as S
import utils as U

PRECS = ("fp16x2", "bf16x3")
NPROD = {"fp16x2": 3, "bf16x3": 6}


def target(D):
    rng = np.random.RandomState(0)
    lam = np.exp(rng.uniform(np.log(0.05), np.log(100.0), D))
    Q, _ = np.linalg.qr(rng.standard_normal((D, D)))
    P = (Q / lam) @ Q.T
    return S.MVNSpec(np.zeros(D), 0.5 * (P + P.T), 0.5 * (D * np.log(2 * np.pi) + np.log(lam).sum())), lam


def run(D, Nc, prec, kernel, spec, lam, Niter=2, Llo=100, Lhi=500):
    q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), Nc, device="cuda", seed=1)
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, warm_up_num=Niter // 2, sampler_type="Random", dt=0.1, L_low=Llo,
                      L_high=Lhi, dtype="float32", kernel=kernel, tc_precision=prec, seed=3, target=spec)
    H.gen_sample(q0, verbose=False, quiet=True)
    torch.cuda.synchronize()
    ge = H.sum_L + Nc * Niter                       # one gradient per leapfrog step plus one per trajectory start
    t = H.kernel_ms * 1e-3
    Dp = (D + 31) // 32 * 32
    rec = {"D": D, "Dp": Dp, "chains": Nc, "kernel": kernel, "tc_precision": H.tc_precision, "kernel_ms": H.kernel_ms,
           "accept_R": H.accept_R, "grad_evals": ge, "grad_evals_per_s": ge / t, "algorithmic_tflops": ge * 2.0 * D * D / t / 1e12}
    if kernel == "bigd":
        rec["tensor_tflops_executed"] = ge * 2.0 * Dp * Dp * NPROD[H.tc_precision] / t / 1e12
    del H, q0
    torch.cuda.empty_cache()
    return rec


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = out.strip()
    except Exception as exc:                        # the numbers stand, but say that the limit could not be read
        info["power_limit_and_max_sm_clock"] = "not read: %r" % exc
    return info


def dump(outdir):
    os.makedirs(outdir, exist_ok=True)
    for D in (512, 1024):
        spec, lam = target(D)
        q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), 2048, device="cuda", seed=5)
        for prec in PRECS:
            H = S.HMC_sampler(D, None, None, Nchain=2048, Niter=4, warm_up_num=1, sampler_type="Random", dt=0.1, L_low=20, L_high=60,
                              dtype="float32", kernel="bigd", tc_precision=prec, seed=9, target=spec)
            H.gen_sample(q0, verbose=False, quiet=True)
            np.save(os.path.join(outdir, "q_chain_D%d_%s.npy" % (D, prec)), H.q_chain_device.cpu().numpy())
            np.save(os.path.join(outdir, "E_chain_D%d_%s.npy" % (D, prec)), H.E_chain[:, :, 0])
            print("dumped D=%d %s sum_L=%d" % (D, prec, H.sum_L), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results (default: stdout only)")
    ap.add_argument("--d", default="1000,1024,1200,1280,1500,1536,2000,2048")
    ap.add_argument("--chains", type=int, default=131072)
    ap.add_argument("--generic-chains", type=int, default=16384)
    ap.add_argument("--dump", metavar="DIR", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    if args.dump:
        dump(args.dump)
        return
    res = {"info": device_info(), "settings": "chains %d, Niter 2 (warm-up 1), dt 0.1, L in [100, 500)" % args.chains, "runs": []}
    Ds = [int(x) for x in args.d.split(",")]
    spec, lam = target(Ds[0])
    for prec in PRECS:                              # warm-up launch of each instantiation
        run(Ds[0], 4096, prec, "bigd", spec, lam, Llo=10, Lhi=20)
    for D in Ds:
        spec, lam = target(D)
        for prec in PRECS:
            rec = run(D, args.chains, prec, "bigd", spec, lam)
            print(json.dumps(rec), flush=True)
            res["runs"].append(rec)
        if D == 1000:                               # the generic kernel (warp per chain, F read from L2) on fewer chains
            run(D, 1024, None, "generic", spec, lam, Llo=10, Lhi=20)
            rec = run(D, args.generic_chains, None, "generic", spec, lam)
            print(json.dumps(rec), flush=True)
            res["generic_D1000"] = rec
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
