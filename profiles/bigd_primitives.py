"""The large-D primitives (csrc/bigd_primitives.cu) timed with CUDA events, after a warm-up call of every shape, in alternating
repeats:

  start points  dense cov0 (a random well-conditioned lower-triangular factor), 8,192 and 131,072 chains: at D = 4096 the
                one-warp-per-chain hmc_start_pts against hmc_start_pts_bigd, at D = 8192 hmc_start_pts_bigd (nothing else runs there).
                Tensor flop of one call: Ncp x Dp^2 x 2 x 6 (bf16x3, every K block multiplied).
  leap_frog     hmc_leap_frog_bigd at D = 2048 and 8192, B = 131,072 rows, nsteps = 10 (11 GEMM passes), both splits: gradient
                rows per second, and the time per pass against the Random sampler's gradient evaluations per second at the same D
                and split from profiles/bigd_any_d.json (the config-5 settings, 131,072 chains; an earlier measurement, not this call).

Device name, power limit and max SM clock are read in the same call.

  python profiles/bigd_primitives.py [--out FILE.json] [--reps 3]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(ROOT), os.path.join(os.path.dirname(ROOT), "understanding-hmc_b200"), ROOT):
    sys.path.insert(0, p)
import numpy as np
import torch
import hmc_b200_lib as L
from bigd_any_d import device_info


def _lower_factor(D, seed=0):
    rng = np.random.RandomState(seed)
    Lc = np.tril(rng.standard_normal((D, D)).astype(np.float32)).astype(float) * (0.5 / np.sqrt(D))
    Lc[np.diag_indices(D)] = 0.5 + rng.random_sample(D)
    return torch.from_numpy(Lc).cuda()


def _timed(fn, reps):
    """Milliseconds of each of `reps` calls of fn, CUDA events around each."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def start_points(reps):
    lib = L.load()
    st = L.current_stream_ptr()
    runs = []
    for D in (4096, 8192):
        Lc = _lower_factor(D)
        q0 = torch.zeros((D,), dtype=torch.float64, device="cuda")
        for N in (8192, 131072):
            out = torch.empty((N, D), dtype=torch.float32, device="cuda")
            nbytes = int(lib.hmc_start_pts_workspace_bytes(N, D))
            ws, wp = L.aligned_workspace(torch, torch.device("cuda"), nbytes)
            calls = {"hmc_start_pts_bigd": lambda: L.check(lib.hmc_start_pts_bigd(L.HMC_F32, 1, 0, N, D, L.ptr(q0), L.ptr(Lc), None,
                                                                                  L.ptr(out), wp, nbytes, st))}
            if D <= 4096:
                calls["hmc_start_pts"] = lambda: L.check(lib.hmc_start_pts(L.HMC_F32, 1, 0, N, D, L.ptr(q0), L.ptr(Lc), None, L.ptr(out), st))
            for fn in calls.values():                       # warm-up
                fn()
            torch.cuda.synchronize()
            times = {k: [] for k in calls}
            for _ in range(reps):                           # alternating
                for k, fn in calls.items():
                    times[k] += _timed(fn, 1)
            Dp, Ncp = (D + 31) // 32 * 32, (N + 511) // 512 * 512
            rec = {"D": D, "chains": N, "ms": times, "best_ms": {k: min(v) for k, v in times.items()},
                   "bigd_tensor_tflops_executed": Ncp * Dp * Dp * 2.0 * 6 / (min(times["hmc_start_pts_bigd"]) * 1e-3) / 1e12}
            if "hmc_start_pts" in times:
                rec["speedup_bigd_over_warp"] = min(times["hmc_start_pts"]) / min(times["hmc_start_pts_bigd"])
            print(json.dumps(rec), flush=True)
            runs.append(rec)
            del out, ws
            torch.cuda.empty_cache()
    return runs


def leap_frog(reps, B=131072, nsteps=10):
    lib = L.load()
    st = L.current_stream_ptr()
    ref = {}
    try:
        with open(os.path.join(ROOT, "bigd_any_d.json")) as f:
            for r in json.load(f)["runs"]:
                ref[(r["D"], r["tc_precision"])] = r["grad_evals_per_s"]
    except (OSError, KeyError, ValueError):
        pass
    runs = []
    for D in (2048, 8192):
        rng = np.random.RandomState(D)
        Ft = torch.from_numpy((np.eye(D) + rng.standard_normal((D, D)) * (0.1 / np.sqrt(D))).astype(np.float32)).cuda()
        mu = torch.zeros((D,), dtype=torch.float32, device="cuda")
        dt = torch.full((D,), 0.1, dtype=torch.float32, device="cuda")
        t = L.Target()
        t.D, t.D_pad, t.Ft, t.mu, t.dt = D, D, Ft.data_ptr(), mu.data_ptr(), dt.data_ptr()
        p = torch.randn((B, D), dtype=torch.float32, device="cuda")
        q = torch.randn((B, D), dtype=torch.float32, device="cuda")
        pn, qn = torch.empty_like(p), torch.empty_like(q)
        nbytes = int(lib.hmc_leap_frog_workspace_bytes(t, B, 0))
        ws, wp = L.aligned_workspace(torch, torch.device("cuda"), nbytes)
        calls = {prec: (lambda fl: lambda: L.check(lib.hmc_leap_frog_bigd(L.HMC_F32, t, B, L.ptr(p), L.ptr(q), L.ptr(pn), L.ptr(qn),
                                                                           nsteps, fl, wp, nbytes, st)))(fl)
                 for prec, fl in (("bf16x3", 0), ("fp16x2", L.FLAG_TC_FP16X2))}
        for fn in calls.values():
            fn()
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        for _ in range(reps):
            for k, fn in calls.items():
                times[k] += _timed(fn, 1)
        for prec, v in times.items():
            best = min(v) * 1e-3
            rec = {"D": D, "rows": B, "nsteps": nsteps, "tc_precision": prec, "ms": v, "best_ms": min(v),
                   "gemm_passes": nsteps + 1, "ms_per_pass": min(v) / (nsteps + 1),
                   "gradient_rows_per_s": B * (nsteps + 1) / best,
                   "sampler_grad_evals_per_s_bigd_any_d_json": ref.get((D, prec))}
            if rec["sampler_grad_evals_per_s_bigd_any_d_json"]:
                rec["rows_per_s_over_sampler"] = rec["gradient_rows_per_s"] / rec["sampler_grad_evals_per_s_bigd_any_d_json"]
            print(json.dumps(rec), flush=True)
            runs.append(rec)
        del p, q, pn, qn, ws, Ft
        torch.cuda.empty_cache()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results (default: stdout only)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"info": device_info(), "start_points": start_points(args.reps), "leap_frog": leap_frog(args.reps)}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
