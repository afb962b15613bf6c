"""Streamed convergence statistics for NUTS on the large-D path (HMC_sampler(sampler_type="NUTS", stream_stats=T), store_ring in
csrc/nuts_bigd.cu): the config-5 NUTS shape of profiles/nuts_bigd.py -- its target (log-uniform spectrum on [0.05, 100], random
rotation), 131,072 chains, D = 1024, dt 0.1, d_max 10, on_dmax "stop", bf16x3 -- for 120 iterations with 24 warm-up (97 stored
samples), T = 32 and 32 stored samples per block (a ring of 64 rows per chain).

Recorded: CUDA-event times of each block's sampler launch and of the hmc_diag_stream_update after it; the peak of allocated device
memory against the bytes the full stream of this run and of a 1,000-iteration run (warm-up 200, 801 stored samples) would need
(computed); R_q / n_eff_q summaries.  With --parent-lib, profiles/nuts_bigd.py's D = 1024 case (both splits, store_ring = 0) is run
three times with that library (loaded through HMC_B200_LIB) and three times with this tree's, alternating, each in a process of its
own.  Device name and power limit are read in the same call.

  python profiles/nuts_stream_stats.py [--out FILE.json] [--parts stream,compare] [--parent-lib PATH] [--chains N] [--niter N]

(--parts runs either half alone, with its own device read, and --merge FILE.json ... joins such halves into --out.)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(ROOT), os.path.join(os.path.dirname(ROOT), "understanding-hmc_b200"), ROOT):
    sys.path.insert(0, p)
import numpy as np
import torch
import hmc_b200_lib as L
import samplers as S
import utils as U
from bigd_any_d import target, device_info


def streamed_nuts(D, Nc, Niter, warm, spec, q0, T, per_block, prec="bf16x3"):
    """One streamed NUTS run through the mirror, its block loop timed with CUDA events around each launch and each update."""
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, warm_up_num=warm, sampler_type="NUTS", dt=0.1, d_max=10, dtype="float32",
                      kernel="auto", tc_precision=prec, seed=3, target=spec, on_dmax="stop", stream_stats=T, iter_block=per_block)
    lib = L.load()
    times = []

    def timed_blocks(run, a, stream):                  # HMC_sampler._run_blocks in stream mode, with events around each call
        st = H._stream
        for (b, e, j0, j1) in st["blocks"]:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            a.iter_begin, a.iter_end = b, e
            ev[0].record()
            L.check(run(a, stream))
            ev[1].record()
            L.check(lib.hmc_diag_stream_update(a.dtype, L.C.c_void_p(a.q_chain), Nc, D, st["R"], H.L_chain, T, j0, j1,
                                               L.C.c_void_p(st["ws_ptr"]), st["ws_bytes"], stream))
            ev[2].record()
            times.append(((b, e, j0, j1), ev))

    H._run_blocks = timed_blocks
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    H.gen_sample(q0, verbose=False)
    torch.cuda.synchronize()
    blocks = [{"iterations": [b, e], "stored_indices": [j0, j1], "sampler_ms": ev[0].elapsed_time(ev[1]),
               "update_ms": ev[1].elapsed_time(ev[2])} for (b, e, j0, j1), ev in times]
    H.compute_convergence_stats()
    peak = torch.cuda.max_memory_allocated()
    return H, blocks, peak


def full_stream_bytes(Nc, D, Lc):
    return Nc * Lc * (D * 4 + 2 * 8)                   # q_chain (float32) + E_chain + dE_chain (float64)


def compare_libs(parent_lib, reps=3):
    """profiles/nuts_bigd.py --d 1024 with the parent library and this tree's, alternating, one process per run."""
    here = os.environ.get("HMC_B200_LIB") or os.path.join(os.path.dirname(ROOT), "understanding-hmc_b200", "libhmc_b200.so")
    out = {"parent_lib": "the parent commit's build (--parent-lib)", "this_lib": os.path.relpath(here, os.path.dirname(ROOT)), "runs": []}
    for r in range(reps):
        for name, lib in (("parent", parent_lib), ("this", here)):
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "r.json")
                env = dict(os.environ, HMC_B200_LIB=lib)
                subprocess.check_call([sys.executable, os.path.join(ROOT, "nuts_bigd.py"), "--d", "1024", "--out", path], env=env,
                                      stdout=subprocess.DEVNULL)
                res = json.load(open(path))
            rec = {"lib": name, "rep": r}
            for x in res["runs"]:
                rec[x["tc_precision"]] = {k: x[k] for k in ("kernel_ms", "leapfrogs", "passes", "gemm_ms_per_pass_4_11",
                                                            "step_ms_per_pass_4_11")}
            print(json.dumps(rec), flush=True)
            out["runs"].append(rec)
    for prec in ("bf16x3", "fp16x2"):
        for name in ("parent", "this"):
            ms = [x[prec]["kernel_ms"] for x in out["runs"] if x["lib"] == name]
            out["%s_%s_kernel_ms" % (name, prec)] = {"min": min(ms), "median": float(np.median(ms)), "max": max(ms)}
        same = {x[prec]["leapfrogs"] for x in out["runs"]}
        out["%s_same_leapfrogs_every_run" % prec] = len(same) == 1
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "nuts_stream_stats.json"))
    ap.add_argument("--parent-lib", default=None, help="libhmc_b200.so of the parent commit (store_ring = 0 timing comparison)")
    ap.add_argument("--chains", type=int, default=131072)
    ap.add_argument("--niter", type=int, default=120)
    ap.add_argument("--warm", type=int, default=24)
    ap.add_argument("--T", type=int, default=32)
    ap.add_argument("--per-block", type=int, default=32)
    ap.add_argument("--parts", default="stream,compare")
    ap.add_argument("--merge", nargs="*", default=None, help="join the JSON files of separate --parts runs into --out")
    args = ap.parse_args()
    if args.merge:
        res = {}
        for path in args.merge:
            part = json.load(open(path))
            if "store_ring_0_timing" in part and "device_info" in part and "blocks" not in part:
                part["store_ring_0_timing"]["device_info"] = part.pop("device_info")
            res.update(part)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        return
    assert torch.cuda.is_available(), "profiles/nuts_stream_stats.py measures on the GPU"
    parts = args.parts.split(",")
    if "stream" not in parts:
        assert args.parent_lib, "--parts compare needs --parent-lib"
        res = {"device_info": device_info(), "store_ring_0_timing": compare_libs(args.parent_lib)}
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        return
    D, Nc = 1024, args.chains
    spec, lam = target(D)
    q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), Nc, device="cuda", seed=1)
    streamed_nuts(D, 2048, 40, 8, spec, q0[:2048], 8, 8)          # warm-up of every kernel shape
    torch.cuda.empty_cache()
    H, blocks, peak = streamed_nuts(D, Nc, args.niter, args.warm, spec, q0, args.T, args.per_block)
    total = torch.cuda.get_device_properties(0).total_memory
    full = full_stream_bytes(Nc, D, H.L_chain)
    full_1000 = full_stream_bytes(Nc, D, 1 + (1000 - 200))
    res = {"device_info": device_info(),
           "settings": "config-5 NUTS shape: %d chains, D = %d, Niter %d, warm-up %d, dt 0.1, d_max 10, on_dmax stop, bf16x3, kernel "
                       "auto (large-D path), stream_stats T = %d, %d stored samples per block" % (Nc, D, args.niter, args.warm, args.T,
                                                                                                args.per_block),
           "nuts_kernel": H.nuts_kernel, "L_chain": H.L_chain, "ring_rows": H._stream["R"], "blocks": blocks,
           "sampler_ms_total": sum(b["sampler_ms"] for b in blocks), "update_ms_total": sum(b["update_ms"] for b in blocks),
           "leapfrogs": H.n_leapfrog_total, "d_max_hits": H.n_dmax, "instabilities": H.n_instability,
           "peak_device_bytes_allocated": peak, "device_total_bytes": total,
           "full_stream_bytes_this_run": full, "full_stream_bytes_1000_iterations_warm_up_200": full_1000,
           "R_q": {"min": float(H.R_q.min()), "median": float(np.median(H.R_q)), "max": float(H.R_q.max())},
           "n_eff_q": {"min": float(H.n_eff_q.min()), "median": float(np.median(H.n_eff_q)), "max": float(H.n_eff_q.max())},
           "n_eff_truncated_dims": int(H.n_eff_truncated.sum())}
    res["update_over_sampler"] = res["update_ms_total"] / res["sampler_ms_total"]
    print(json.dumps({k: v for k, v in res.items() if k != "blocks"}), flush=True)
    del H
    torch.cuda.empty_cache()
    if args.parent_lib and "compare" in parts:
        res["store_ring_0_timing"] = compare_libs(args.parent_lib)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
