"""Streamed convergence statistics (csrc/diag_stream.cu, HMC_sampler(stream_stats=T)): cost of the updates against the sampler's
own kernel time and against the windowed full-stream pass at the same T, and the memory a streamed run needs.

  case3c : 65,536 chains x D = 100 (rho = 0.95), 1,000 iterations, warm-up 200, L in [5, 20), dt 0.1, T = 320, 64 stored samples per
           block.  Windowed reference: a full-storage run of the same seed, then hmc_diag_moments + hmc_diag_variogram for lags 1..T
           (the kernels convergence_stats uses under HMC_B200_DIAG_NO_FFT=1), timed with CUDA events.
  config5: 131,072 chains x D = 1024 (the config-5 target of profiles/bigd_any_d.py, large-D path, fp16x2), 440 iterations, warm-up
           40 (401 stored samples), L in [5, 20) (config 5 itself draws L in [100, 500): only the sampler time changes), T = 64.  The
           full stream (215 GB) does not fit on the card; the windowed reference is timed on the first 32,768 chains of a full-storage
           run and scaled by 4.
Per workload: the sampler's launches and the updates are timed separately with CUDA events around each call of the block loop;
achieved FLOP/s of the pair arithmetic (3 per pair: subtract, multiply, add) and bytes read by the lag kernels' window loads (the new
rows and the rows they pair with, per chain and lag launch) over the update time, against the measured FP32 FFMA peak and 7.7 TB/s.
Device name and power limit are read in the same call.

  python profiles/stream_stats.py [--out FILE.json] [--only case3c,config5]
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
import samplers as S
import utils as U
from bigd_any_d import target, device_info

HBM_TBPS = 7.7


def pair_and_byte_counts(Lc, T, blocks, Nc, D, esize):
    """Pairs formed and bytes the lag kernels load, replaying the host loop of stream_update (pieces of <= 64 inside one split chain,
    lags in launches of 128)."""
    n = (Lc - 1) // 2
    pairs = 0
    rows = 0
    for (_, _, j0, j1) in blocks:
        ilo, ihi = max(j0, 1), min(j1, 2 * n + 1)
        lo = ilo
        while lo < ihi:
            s0, send = (1, n + 1) if lo <= n else (n + 1, 2 * n + 1)
            hi = min(lo + 64, send, ihi)
            for i in range(lo, hi):
                pairs += min(T, i - s0)
            tl = 1
            while tl <= T:
                th = min(tl + 128, T + 1)
                if hi - 1 - tl < s0:
                    break
                elo = max(s0, lo - th + 1)
                rows += (hi - lo) + max(0, hi - tl - elo)
                tl += 128
            lo = hi
    return pairs * Nc * D, rows * Nc * D * esize


def streamed_run(D, Nc, Niter, warm, spec, q0, T, per_block, kernel, prec=None):
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=5, L_high=20,
                      dtype="float32", kernel=kernel, tc_precision=prec, seed=3, target=spec, stream_stats=T, iter_block=per_block)
    torch.cuda.reset_peak_memory_stats()
    lib = L.load()
    run = H.prepare_random(q0)
    a, st = run["args"], H._stream
    stream = L.current_stream_ptr()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in st["blocks"]]
    for (b, e, j0, j1), (e0, e1, e2) in zip(st["blocks"], ev):
        a.iter_begin, a.iter_end = b, e
        e0.record()
        L.check(lib.hmc_random_run(a, stream))
        e1.record()
        L.check(lib.hmc_diag_stream_update(a.dtype, L.C.c_void_p(a.q_chain), Nc, D, st["R"], H.L_chain, T, j0, j1,
                                           L.C.c_void_p(st["ws_ptr"]), st["ws_bytes"], stream))
        e2.record()
    torch.cuda.synchronize()
    sampler_ms = sum(e0.elapsed_time(e1) for e0, e1, _ in ev)
    update_ms = sum(e1.elapsed_time(e2) for _, e1, e2 in ev)
    H._stream = st
    R, ne, tr = U.stream_stats_from_workspace(st["ws_ptr"], st["ws_bytes"], D, T, H.L_chain, Nc, group=False, device=st["device"])
    peak = torch.cuda.max_memory_allocated()
    return dict(H=H, sampler_ms=sampler_ms, update_ms=update_ms, R=R, n_eff=ne, truncated=tr, peak_bytes=peak, ring_rows=st["R"],
                workspace_bytes=st["ws_bytes"], blocks=st["blocks"], updates=len(st["blocks"]))


def windowed_ms(x, T, reps=3):
    """hmc_diag_moments + hmc_diag_variogram over lags 1..T (32 per call) on a full stream x [Nc][>= 2n][D], float32; best of reps."""
    lib = L.load()
    Nc, _, D = x.shape
    n = x.shape[1] // 2
    mom = torch.empty((4, D), dtype=torch.float64, device=x.device)
    lags = torch.empty((T, D), dtype=torch.float64, device=x.device)
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.hmc_diag_moments(L.HMC_F32, L.ptr(x), Nc, n, D, x.stride(0), L.ptr(mom), L.current_stream_ptr()))
        for l0 in range(1, T + 1, 32):
            nl = min(32, T - l0 + 1)
            L.check(lib.hmc_diag_variogram(L.HMC_F32, L.ptr(x), Nc, n, D, x.stride(0), l0, nl, L.ptr(lags[l0 - 1:]), L.current_stream_ptr()))
        e1.record()
        e1.synchronize()
        t = e0.elapsed_time(e1)
        best = t if best is None else min(best, t)
    return best


def record(name, res, T, Nc, D, win_ms, win_note, ffma_peak, extra=None):
    pairs, nbytes = pair_and_byte_counts(res["H"].L_chain, T, res["blocks"], Nc, D, 4)
    upd_s = res["update_ms"] * 1e-3
    flops = 3.0 * pairs
    t_fl, t_by = flops / ffma_peak, nbytes / (HBM_TBPS * 1e12)
    out = {"name": name, "chains": Nc, "D": D, "Niter": res["H"].Niter, "warm_up_num": res["H"].warm_up_num, "L_chain": res["H"].L_chain,
           "T": T, "ring_rows": res["ring_rows"], "updates": res["updates"], "sampler_kernel_ms": res["sampler_ms"],
           "update_ms_total": res["update_ms"], "update_over_sampler": res["update_ms"] / res["sampler_ms"],
           "windowed_full_stream_ms": win_ms, "windowed_note": win_note, "update_over_windowed": res["update_ms"] / win_ms,
           "pairs": pairs, "pair_gflops_achieved": flops / upd_s / 1e9, "window_bytes": nbytes, "window_gbps_achieved": nbytes / upd_s / 1e9,
           "roofline": {"fp32_peak_tflops_measured": ffma_peak / 1e12, "hbm_tbps": HBM_TBPS, "bound": "flops" if t_fl > t_by else "bytes",
                        "frac_of_bound": max(t_fl, t_by) / upd_s},
           "stream_workspace_bytes": res["workspace_bytes"], "peak_device_bytes_allocated": res["peak_bytes"],
           "n_eff_truncated_dims": int(res["truncated"].sum())}
    if extra:
        out.update(extra)
    return out


def case3c(ffma_peak):
    D, Nc, Niter, warm, T = 100, 65536, 1000, 200, 320
    spec = S.MVNSpec.from_cov(np.zeros(D), S.equicorrelated_cov(D, 0.95))
    q0 = U.start_pts(np.zeros(D), S.equicorrelated_cov(D, 0.95), Nc, device="cuda", seed=1)
    streamed_run(D, 1024, 60, 10, spec, q0[:1024], 20, 64, "auto")             # warm-up of every kernel shape
    res = streamed_run(D, Nc, Niter, warm, spec, q0, T, 64, "auto")
    F = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=5, L_high=20,
                      dtype="float32", kernel="auto", seed=3, target=spec)
    F.gen_sample(q0, verbose=False, quiet=True)
    x = F.q_chain_device[:, 1:]
    win = windowed_ms(x, T)
    R_full, ne_full = U.convergence_stats(x, thin_rate=1, warm_up_num=0, group=False)
    ok = ~res["truncated"]
    extra = {"full_stream_bytes": x.numel() * 4, "max_rel_diff_R_vs_full": float(np.max(np.abs(res["R"] / R_full - 1))),
             "max_rel_diff_n_eff_vs_full_untruncated": float(np.max(np.abs(res["n_eff"][ok] / ne_full[ok] - 1))) if ok.any() else None}
    del F, x
    torch.cuda.empty_cache()
    return record("case3c", res, T, Nc, D, win, "full-storage run of the same seed; moments + windowed variogram lags 1..T, best of 3",
                  ffma_peak, extra)


def config5(ffma_peak):
    D, Nc, Niter, warm, T = 1024, 131072, 440, 40, 64
    spec, lam = target(D)
    q0 = U.start_pts(np.zeros(D), np.diag(lam.mean() * np.ones(D)), Nc, device="cuda", seed=1)
    streamed_run(D, 2048, 60, 10, spec, q0[:2048], 20, 64, "bigd", "fp16x2")
    res = streamed_run(D, Nc, Niter, warm, spec, q0, T, 64, "bigd", "fp16x2")
    Lc = res["H"].L_chain
    full_bytes = Nc * Lc * D * 4
    total = torch.cuda.get_device_properties(0).total_memory
    res["H"]._q_dev = res["H"]._E_dev = res["H"]._dE_dev = res["H"]._stream = None
    torch.cuda.empty_cache()
    sub = 32768
    F = S.HMC_sampler(D, None, None, Nchain=sub, Niter=Niter, warm_up_num=warm, sampler_type="Random", dt=0.1, L_low=5, L_high=20,
                      dtype="float32", kernel="bigd", tc_precision="fp16x2", seed=3, target=spec)
    F.gen_sample(q0[:sub], verbose=False, quiet=True)
    win = windowed_ms(F.q_chain_device[:, 1:], T) * (Nc / sub)
    del F
    torch.cuda.empty_cache()
    extra = {"full_stream_bytes": full_bytes, "device_total_bytes": total, "full_stream_fits": bool(full_bytes < total),
             "statement": "the full q_chain of this run (%.0f GB) exceeds the card's %.0f GB; the streamed run peaked at %.1f GB allocated"
                          % (full_bytes / 1e9, total / 1e9, res["peak_bytes"] / 1e9)}
    return record("config5", res, T, Nc, D, win, "windowed pass timed on the first %d chains of a full-storage run, scaled by %d"
                  % (sub, Nc // sub), ffma_peak, extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "stream_stats.json"))
    ap.add_argument("--only", default="case3c,config5")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "profiles/stream_stats.py measures on the GPU"
    import ctypes
    peak = ctypes.c_double()
    L.check(L.load().hmc_ffma_peak(ctypes.byref(peak), 1, L.current_stream_ptr()))
    pk = peak.value
    out = {"device_info": device_info(), "fp32_ffma_peak_flops_measured": pk, "results": []}
    for name in args.only.split(","):
        rec = {"case3c": case3c, "config5": config5}[name](pk)
        print(json.dumps(rec), flush=True)
        out["results"].append(rec)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
