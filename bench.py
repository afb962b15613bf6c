#!/usr/bin/env python
"""bench.py -- leapfrog gradient-evals/sec (and ESS/sec) of the fused HMC trajectory kernel (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload = "case3c_65536"): Case 3c of the reference (case3-script.py:136-181, README:40-45): MVN D=100,
rho=0.95, random trajectory length L in {5..19}, dt=0.1, 1000 iterations of which 200 are warm-up, scaled to 65,536
chains PER GPU (weak scaling: chains are independent units, no data-path collective; SURVEY 8e).  A "step" is ONE SUCH
RUN: one launch of the fused kernel over all 1000 iterations of every chain (~12 leapfrog steps each; the 801 stored
samples and energies per chain, 21.8 GB, are the only HBM traffic).  Definitions printed with the number (SURVEY 8d):
  gradient-eval = one full grad U = P (q - mu) for one chain = 2 D^2 = 20,000 flop; value counts the
  leapfrog gradient evaluations sum(L) only (the extra evaluation at the first point of every trajectory is
  NOT counted, but is included in roofline.achieved since the kernel does execute it).

value      : device-timed (CUDA events on the launching stream, barrier + synchronize on both sides, max over
             ranks), start points resident in HBM, every step a fresh run (new Philox seed) into the same output slab.
e2e        : the same run through the public API (samplers.HMC_sampler.gen_sample + compute_convergence_stats)
             with q_start in pinned HOST memory (H2D inside the timed region) and the diagnostics' result (Rhat, n_eff per
             dimension) read back to the host (D2H inside); at N>1 the Rhat/ESS partial sums go through NCCL.  q_chain stays
             on the device (SURVEY H10: 21 GB per GPU; the host gets it lazily, on attribute access).
roofline   : tensor bound: the gradient runs on tcgen05 as an FP32-grade split product (fp16x2: 3 MMA passes; bf16x3: 6);
             achieved = executed gradient evals * 2 D^2 / kernel time against the measured dense bf16 (= fp16) peak, with
             the executed tensor flop and the FP32 FFMA peak measured in this run reported beside it.
secondary  : measured in the same run (rank 0 reports; all ranks take part): Case 3d ESS/sec, Case 2c burn-in (262,144 chains
             over all ranks, Rhat over early windows), NUTS config 4, and the diagnostics kernels' own HBM rooflines.
cpu_baseline / --impl reference : the oracle port of the reference sampler (oracle/hmc_oracle.py) with the
             reference's own library calls (scipy logpdf for V, np.random.multivariate_normal for p), one
             process per host core, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "understanding-hmc_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

if "reference" in sys.argv:
    # the CPU arm runs one single-threaded process per core: BLAS/OpenMP pools must be pinned to 1 thread
    # BEFORE numpy/scipy load (the reference's 100x100 factorizations are 7.6x slower when oversubscribed, SURVEY 3.4)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_v] = "1"

import numpy as np  # noqa: E402

D, RHO, DT, L_LOW, L_HIGH = 100, 0.95, 0.1, 5, 20
CHAINS_PER_GPU = 65536
NITER, WARM = 1000, 200            # README:40-45 (Case 3c as listed; case3-script.py runs 2000 / 1000)
METRIC = "leapfrog grad-evals/sec, D=100 rho=0.95 MVN (Case 3c), 65536 chains per B200"
UNIT = "grad-evals/s"
DUMP_CHAINS = 128                  # --dump-outputs: 128 chains x 801 samples x 100 dims of float32 is 41 MB


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port), also used for cpu_baseline
# ------------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, nchain, niter = args
    os.environ["OMP_NUM_THREADS"] = "1"
    from oracle import hmc_oracle as O
    from scipy.stats import multivariate_normal
    q0 = np.zeros(D)
    cov0 = O.equicorrelated_cov(D, RHO)
    inv_cov0 = np.linalg.inv(cov0)

    def V(q):                                   # case3-script.py:39-43 -> utils.py:213-218 (scipy logpdf)
        return -multivariate_normal.logpdf(q, mean=q0, cov=cov0)

    def dVdq(q):                                # case3-script.py:45-49
        return np.dot(inv_cov0, (q - q0))

    np.random.seed(seed)
    q_start = np.random.multivariate_normal(q0, np.diag(np.ones(D)) * 2, size=nchain)
    t0 = time.time()
    R = O.gen_sample_random(D, V, dVdq, q_start, O.NumpyDraws(D), nchain, niter, 1, 0, DT, L_LOW, L_HIGH, record=True)
    O.convergence_stats(R.q_chain[:, 1:, :], 1, 0)      # the e2e leg of the GPU arm includes the diagnostics: so does this one
    dt = time.time() - t0
    return int(R.L_tape.sum()), dt


def cpu_reference(nchain_per_proc=8, niter=60, cores=None):
    """Returns (leapfrog grad-evals/s over all processes, cores, description).  Counts one gradient-eval per
    leapfrog step, like `value` (the reference itself spends two dVdq calls per step, samplers.py:835-837)."""
    import multiprocessing as mp
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cores = cores or max(1, min(avail, 64))
    ctx = mp.get_context("fork")
    t0 = time.time()
    with ctx.Pool(cores) as pool:
        out = pool.map(_cpu_worker, [(1000 + i, nchain_per_proc, niter) for i in range(cores)])
    wall = time.time() - t0
    total_L = sum(o[0] for o in out)
    busy = max(o[1] for o in out)
    sample = "%d procs x %d chains x %d iterations of Case 3c (D=100, rho=0.95), OMP_NUM_THREADS=1" % (cores, nchain_per_proc, niter)
    return total_L / busy, cores, sample, wall


# ------------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """Samples SM clocks / clock-event (throttle) reasons DURING the timed region: an NVML polling thread (5 ms period;
    the timed region of the default run is a few hundred ms, too short for `nvidia-smi -lms`), with the profiling
    recipe's `nvidia-smi` line as the fallback when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.rows = []          # [sm_mhz, max_mhz, hw_slowdown, hw_thermal, sw_thermal, sw_power_cap]
        self.thread = None
        self.stop_flag = False
        self.source = None

    def _nvml_loop(self, nv, h):
        bits = [(getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), 2), (getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), 3),
                (getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), 4), (getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4), 5)]
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                row = [str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx), "", "", "", ""]
                r = int(get_reasons(h))
                for mask, col in bits:
                    row[col] = "Active" if (r & mask) else "Not Active"
                self.rows.append(row)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.source = "nvml, 5 ms period"
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi -lms 100"
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = b""
        for line in out.decode(errors="ignore").splitlines():
            self.rows.append([x.strip() for x in line.split(",")])

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": self.source}


def _hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 7700.0, "fallback: nominal 7.7 TB/s (B200_PROFILING.md)"


def secondary_measurements(torch, dist, S, U, L, lib, rank, world, dev, log):
    """Measured in the same run as the headline (VERDICT r1 item 4): every entry says what it is and how it was timed."""
    out = []
    hbm, hbm_src = _hbm_peak()

    def timed(fn):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return r, float(t.item())

    cov = S.equicorrelated_cov(D, RHO)
    spec = S.MVNSpec.from_cov(np.zeros(D), cov)
    Nc = CHAINS_PER_GPU
    # ---- Case 3d (case3-script-2.py:6-68): L in [50,200): the configuration whose ESS means something --------------------
    try:
        def run3d():
            q0 = U.start_pts(np.zeros(D), 2.0 * np.eye(D), Nc, device=dev, seed=91, chain_id0=rank * Nc)
            H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=300, thin_rate=1, warm_up_num=100, sampler_type="Random", dt=DT,
                              L_low=50, L_high=200, dtype="float32", kernel="auto", seed=5, chain_id0=rank * Nc, target=spec,
                              distributed=(world > 1))
            H.gen_sample(q0, verbose=False, quiet=True)
            H.compute_convergence_stats()
            return H
        run3d()
        H, t = timed(run3d)
        out.append({"name": "case3d_ess", "what": "Case 3d (D=100 rho=0.95, L in [50,200), dt=0.1), %d chains/GPU, 300 iterations, 100 warm-up; "
                    "start points generated on the device; wall time of gen_sample + compute_convergence_stats" % Nc,
                    "seconds": t, "kernel_ms": H.kernel_ms, "accept_R": H.accept_R, "grad_evals_per_sec": H.sum_L / t,
                    "rhat_median": float(np.median(H.R_q)), "rhat_max": float(np.max(H.R_q)),
                    "n_eff_median": float(np.median(H.n_eff_q)), "n_eff_min": float(np.min(H.n_eff_q)),
                    "stored_samples": int(world * Nc * 200), "ess_per_stored_sample": float(np.median(H.n_eff_q)) / (world * Nc * 200.0),
                    "ess_per_sec_median": float(np.median(H.n_eff_q)) / t, "ess_per_sec_min": float(np.min(H.n_eff_q)) / t})
        del H
        log("secondary: case3d done")
    except Exception as exc:
        out.append({"name": "case3d_ess", "failed": repr(exc)})
    torch.cuda.empty_cache()
    # ---- Case 2c (case2-script.py:57-61, 136-195): unit MVN, start ~N(0, 100 I), chain 0 pinned; 262,144 chains over all ranks ----
    try:
        tot = 262144
        Ncl = tot // world
        spec2 = S.MVNSpec.from_cov(np.zeros(D), np.eye(D))

        def run2c():
            q0 = U.start_pts(np.zeros(D), 100.0 * np.eye(D), Ncl, device=dev, seed=92, chain_id0=rank * Ncl)
            if rank == 0:
                q0[0, :] = 0.0
                q0[0, 0], q0[0, 1] = 1000.0, -750.0
            H = S.HMC_sampler(D, None, None, Nchain=Ncl, Niter=200, thin_rate=1, warm_up_num=0, sampler_type="Random", dt=DT,
                              L_low=L_LOW, L_high=L_HIGH, dtype="float32", kernel="auto", seed=6, chain_id0=rank * Ncl,
                              target=spec2, distributed=(world > 1))
            H.gen_sample(q0, verbose=False, quiet=True)
            grp = None if world > 1 else False
            wins = {}
            for (lo, hi) in ((1, 21), (21, 51), (51, 101), (101, 201)):      # burn-in: Rhat over early windows of stored samples
                R, _ = U.convergence_stats(H.q_chain_device[:, lo:hi, :], thin_rate=1, warm_up_num=0, group=grp)
                wins["%d-%d" % (lo, hi - 1)] = {"rhat_median": float(np.median(R)), "rhat_max": float(np.max(R))}
            return H, wins
        run2c()
        (H, wins), t = timed(run2c)
        out.append({"name": "case2c_burn_in", "what": "Case 2c (unit MVN D=100, start ~N(0,100 I), chain 0 at (1000,-750,0,...)), %d chains over %d GPU(s), "
                    "200 iterations, L in [5,20); Rhat of windows of stored samples through the all-gather of chain moments" % (tot, world),
                    "seconds": t, "kernel_ms": H.kernel_ms, "tc_precision": H.tc_precision, "accept_R": H.accept_R,
                    "grad_evals_per_sec_kernel": H.sum_L / (H.kernel_ms * 1e-3), "rhat_windows": wins})
        del H
        log("secondary: case2c done")
    except Exception as exc:
        out.append({"name": "case2c_burn_in", "failed": repr(exc)})
    torch.cuda.empty_cache()
    # ---- NUTS (BASELINE config 4): D=100 rho=0.95, dt=0.1, d_max=10 ------------------------------------------------------------
    try:
        Nn = int(os.environ.get("HMC_BENCH_NUTS_CHAINS", str(Nc)))

        def runnuts():
            q0 = U.start_pts(np.zeros(D), 2.0 * np.eye(D), Nn, device=dev, seed=93, chain_id0=rank * Nn)
            H = S.HMC_sampler(D, None, None, Nchain=Nn, Niter=4, sampler_type="NUTS", dt=DT, d_max=10, dtype="float32", seed=7,
                              chain_id0=rank * Nn, target=spec, on_dmax="stop", distributed=(world > 1))
            H.gen_sample(q0, verbose=False)
            return H
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            H, t = timed(runnuts)
        out.append({"name": "nuts_config4", "what": "NUTS, D=100 rho=0.95, dt=0.1, d_max=10, on_dmax=stop (a chain at depth 10 keeps its live point; "
                    "the reference would abort the whole run, SURVEY H6), %d chains/GPU, 4 iterations" % Nn,
                    "seconds": t, "kernel_ms": H.kernel_ms, "leapfrogs": int(H.n_leapfrog_total), "dmax_hits": int(H.n_dmax),
                    "leapfrogs_per_iteration": H.n_leapfrog_total / float(world * Nn * 4),
                    "leapfrogs_per_sec": H.n_leapfrog_total / (H.kernel_ms * 1e-3), "kernel": getattr(H, "nuts_kernel", "generic")})
        del H
        log("secondary: nuts done")
    except Exception as exc:
        out.append({"name": "nuts_config4", "failed": repr(exc)})
    torch.cuda.empty_cache()
    # ---- BASELINE config 5: dense-covariance MVN D = 1024, 131,072 chains per GPU (1M over 8), L in [100, 500) ----------------------
    try:
        Db, Nb = 1024, int(os.environ.get("HMC_BENCH_BIGD_CHAINS", "131072"))
        rs = np.random.RandomState(0)
        lam = np.exp(rs.uniform(np.log(0.05), np.log(100.0), Db))              # SURVEY 8d-5: log-uniform spectrum, random rotation
        Qr, _ = np.linalg.qr(rs.standard_normal((Db, Db)))
        Pb = (Qr / lam) @ Qr.T
        specb = S.MVNSpec(np.zeros(Db), 0.5 * (Pb + Pb.T), 0.5 * (Db * np.log(2 * np.pi) + np.log(lam).sum()))

        def runbig():
            q0 = U.start_pts(np.zeros(Db), np.diag(lam.mean() * np.ones(Db)), Nb, device=dev, seed=94, chain_id0=rank * Nb)
            H = S.HMC_sampler(Db, None, None, Nchain=Nb, Niter=2, warm_up_num=1, sampler_type="Random", dt=DT, L_low=100, L_high=500,
                              dtype="float32", kernel="auto", seed=8, chain_id0=rank * Nb, target=specb, distributed=(world > 1))
            H.gen_sample(q0, verbose=False, quiet=True)
            return H
        H, t = timed(runbig)
        ge = H.sum_L + world * Nb * 2
        alg = ge * 2.0 * Db * Db / (H.kernel_ms * 1e-3) / 1e12
        try:
            pk = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]) * world
        except Exception:
            pk = 2250.0 * world
        out.append({"name": "bigd_config5", "what": "dense-covariance MVN D=1024 (log-uniform spectrum on [0.05,100], random rotation), %d chains/GPU, "
                    "2 iterations, L in [100,500), dt=0.1: one tcgen05 GEMM over all chains per leapfrog step (TMA operands with the B tile multicast "
                    "to clusters of two, fp16x2 split, leapfrog fused into a TMA-fed epilogue); all ranks' work over the slowest rank's kernel time" % Nb,
                    "seconds": t, "kernel_ms": H.kernel_ms, "accept_R": H.accept_R, "tc_precision": H.tc_precision,
                    "leapfrog_grad_evals_per_sec": H.sum_L / (H.kernel_ms * 1e-3),
                    "roofline": {"bound": "tensor", "achieved": alg, "peak": pk, "unit": "TFLOP/s", "frac": alg / pk,
                                 "tensor_tflops_executed": 3.0 * alg, "frac_executed": 3.0 * alg / pk,
                                 "note": "algorithmic 2 D^2 per gradient evaluation; three fp16 part products executed; rows are chains sorted by "
                                         "planned passes, so finished row blocks drop out of the GEMM; the run still ends with a thinning tail of passes "
                                         "(a full pass runs at ~990 TFLOP/s executed)"}})
        del H
        log("secondary: config 5 done")
    except Exception as exc:
        out.append({"name": "bigd_config5", "failed": repr(exc)})
    torch.cuda.empty_cache()
    # ---- diagnostics kernels on a 6.55 GB float32 stream: algorithmic bytes / kernel time against the measured HBM bandwidth ----
    if rank == 0:
        try:
            x = torch.empty((Nc, 250, D), dtype=torch.float32, device=dev).normal_()
            xs = torch.empty((Nc, 50, D), dtype=torch.float32, device=dev).normal_()
            buf = torch.empty((40, D), dtype=torch.float64, device=dev)
            st = L.current_stream_ptr()
            cases = [("diag_moments", x, lambda: lib.hmc_diag_moments(L.HMC_F32, L.ptr(x), Nc, 125, D, 250 * D, L.ptr(buf), st), 1.0),
                     ("diag_variogram_32lags", x, lambda: lib.hmc_diag_variogram(L.HMC_F32, L.ptr(x), Nc, 125, D, 250 * D, 33, 32, L.ptr(buf), st), 2.0),
                     ("diag_variogram_16lags", x, lambda: lib.hmc_diag_variogram(L.HMC_F32, L.ptr(x), Nc, 125, D, 250 * D, 33, 16, L.ptr(buf), st), 1.0),
                     ("diag_short_series", xs, lambda: lib.hmc_diag_short_series(L.HMC_F32, L.ptr(xs), Nc, 25, D, 50 * D, 24, L.ptr(buf), L.ptr(buf[5:]), st), 1.0)]
            for name, arr, fn, passes in cases:
                for _ in range(2):
                    L.check(fn())
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(5):
                    L.check(fn())
                e1.record()
                e1.synchronize()
                ms = e0.elapsed_time(e1) / 5
                nbytes = arr.numel() * 4
                out.append({"name": name, "roofline": {"bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                                       "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "peak_source": hbm_src,
                                                       "algorithmic_bytes": nbytes, "launch_ms": ms, "passes_over_the_stream": passes,
                                                       "traffic": None}})
            del x, xs
            torch.cuda.empty_cache()
            # the all-lags FFT pass on the headline run's own stream shape (400-sample split chains, 21 GB): its cost is per (chain,
            # dimension) transform, not per byte -- bound by instruction issue / shared-memory latency (DESIGN 4.4); reported against
            # the HBM bandwidth like the other diagnostics and against the FP32 peak (~60 kflop per 1024-point complex transform)
            xl = torch.empty((Nc, 800, D), dtype=torch.float32, device=dev).normal_()
            abuf = torch.empty((399, D), dtype=torch.float64, device=dev)
            ws = torch.empty((int(lib.hmc_diag_variogram_all_workspace_bytes(400, D)) // 8,), dtype=torch.float64, device=dev)
            fn = lambda: lib.hmc_diag_variogram_all(L.HMC_F32, L.ptr(xl), Nc, 400, D, 800 * D, 399, L.ptr(abuf), L.ptr(ws), ws.numel() * 8, st)
            for _ in range(2):
                L.check(fn())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                L.check(fn())
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / 5
            nbytes = xl.numel() * 4
            flop = float(Nc) * D * 60.0e3
            ffma = None
            try:
                pk = L.C.c_double(0.0)
                L.check(lib.hmc_ffma_peak(L.C.byref(pk), 0, st))
                ffma = pk.value / 1e12
            except Exception:
                pass
            out.append({"name": "diag_variogram_all_lags_fft",
                        "what": "every variogram lag (399) of %d x 100 series of 2 x 400 samples in one pass: one 1024-point complex FFT per (chain, "
                                "dimension); the windowed kernel needs 4.4 ms per 16 lags on this stream" % Nc,
                        "roofline": {"bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                     "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "peak_source": hbm_src, "algorithmic_bytes": nbytes,
                                     "launch_ms": ms, "passes_over_the_stream": 1.0, "traffic": None,
                                     "fp32_tflops": flop / (ms * 1e-3) / 1e12, "fp32_ffma_peak": ffma,
                                     "frac_of_fp32_ffma_peak": (flop / (ms * 1e-3) / 1e12 / ffma) if ffma else None,
                                     "note": "not an HBM-bound kernel: ~60 kflop per transform, issue / shared-memory-latency bound at 12 warps per SM"}})
            del xl
            log("secondary: diagnostics kernels done")
        except Exception as exc:
            out.append({"name": "diag_kernels", "failed": repr(exc)})
    torch.cuda.empty_cache()
    return out


def dump_last_step(out_dir, torch, H, step_counters, log):
    """What a caller of the timed path receives from its last step, for comparing two builds output for output: stored
    samples and energies of a fixed seeded sample of chains, and that step's counters (warm-up accepts, accepts, sum L,
    sum L^2)."""
    Nc, Lc, D = H._q_dev.shape
    n = min(Nc, DUMP_CHAINS, max(1, (48 << 20) // (Lc * (D * 4 + 16))))
    idx = np.sort(np.random.RandomState(0).choice(Nc, n, replace=False))
    idx_d = torch.from_numpy(idx).to(H._q_dev.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"q_chain": H._q_dev.index_select(0, idx_d), "E_chain": H._E_dev.index_select(0, idx_d),
              "dE_chain": H._dE_dev.index_select(0, idx_d), "counters": step_counters[:4].to(torch.float64)}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
    log("outputs of the last step (%d of %d chains) written to %s" % (n, Nc, out_dir))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU, help="chains per GPU")
    ap.add_argument("--niter", type=int, default=NITER)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0: a fixed sample of %d chains) as DIR/<name>.npy"
                         % DUMP_CHAINS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")
    T0 = time.time()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    W = args.warmup
    K = args.steps
    Niter = args.niter
    warm = min(WARM, Niter // 5)
    Lc = 1 + (Niter - warm)
    config = {"workload": "case3c_65536", "D": D, "rho": RHO, "dt": DT, "L": "[%d,%d)" % (L_LOW, L_HIGH),
              "chains_per_gpu": args.chains, "iterations_per_step": Niter, "warm_up": warm, "sampler": "Random",
              "step": "one Case 3c run: one fused-kernel launch over all iterations of all chains",
              "parallelism": "chains sharded, %d rank(s)" % world,
              "l2": "state is on-chip; each step streams a %.2f GB output slab per GPU (> 126 MB L2)" %
                    (args.chains * Lc * (D * 4 + 16) / 1e9)}

    if args.impl == "reference":
        if rank != 0:
            return
        vals = []
        cores = sample = None
        # bounded sample per step, sized so that the whole --steps/--warmup run stays within a couple of minutes
        niter = max(12, min(60, int(60 * 23 / float(W + K))))
        for i in range(W + K):
            v, cores, sample, _ = cpu_reference(niter=niter)
            if i >= W:
                vals.append(v)
        value = float(np.mean(vals))
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
                "warmup": W, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import hmc_b200_lib as L
    import samplers as S
    import utils as U

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()

    def log(msg):
        if rank == 0:
            sys.stderr.write("[bench %.1fs] %s\n" % (time.time() - T0, msg))
            sys.stderr.flush()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cov0 = S.equicorrelated_cov(D, RHO)
    spec = S.MVNSpec.from_cov(np.zeros(D), cov0)
    Nc = args.chains
    id0 = rank * Nc
    rng = np.random.RandomState(1234 + rank)
    q_start = (rng.standard_normal((Nc, D)) * np.sqrt(2.0)).astype(np.float32)      # case3-script.py:57-58

    # ---- device-resident leg: every step = one run (one launch) from the resident start points, new seed, same output slab ----
    H = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, thin_rate=1, warm_up_num=warm, sampler_type="Random",
                      dt=DT, L_low=L_LOW, L_high=L_HIGH, dtype="float32", kernel="auto", seed=2026, chain_id0=id0,
                      target=spec)
    run = H.prepare_random(q_start)               # allocates outputs/state, builds the C-ABI argument block, H2D of q_start
    counters = run["counters"]
    a = run["args"]
    a.iter_begin, a.iter_end = 0, Niter
    stream = L.current_stream_ptr()
    log("buffers ready (%d chains, %d iterations per step)" % (Nc, Niter))
    sampler_thread = ClockSampler(local_rank) if rank == 0 else None      # samples through warm-up + timed region
    if sampler_thread:
        sampler_thread.start()
    for i in range(W):
        a.seed = 2026 + i
        L.check(lib.hmc_random_run(a, stream))
    barrier()
    log("warm-up done")
    c0 = counters.clone()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(W, W + K):
        a.seed = 2026 + i
        if args.dump_outputs and i == W + K - 1:
            # the counters accumulate over launches: snapshot them before the last step to get its own.  With --steps
            # above 1 this one 64-byte device copy falls inside the timed window (microseconds against a ~120 ms step)
            c_last = counters.clone() if i > W else c0
        L.check(lib.hmc_random_run(a, stream))
    ev1.record()
    barrier()
    if sampler_thread:
        sampler_thread.stop()
    ms = ev0.elapsed_time(ev1)
    log("timed region done: %.1f ms for %d steps" % (ms, K))
    if args.dump_outputs and rank == 0:
        dump_last_step(args.dump_outputs, torch, H, counters - c_last, log)
    dc = (counters - c0).cpu().numpy().astype(np.int64)
    acc_post, sumL = int(dc[1]), int(dc[2])
    n_traj = Nc * K * Niter
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    # the tensor-core kernel evaluates the gradient at the first point of every trajectory too: L + 1 per iteration
    tot = torch.tensor([float(sumL), float(sumL + n_traj)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot)
    ms_max = float(t.item())
    value = float(tot[0].item()) / (ms_max * 1e-3)
    executed_local = float(sumL + n_traj)
    env_prec = os.environ.get("HMC_B200_TC_PREC", "")[:1]
    fp16 = env_prec == "f" or (bool(a.flags & L.FLAG_TC_FP16X2) and env_prec != "b")

    # ---- roofline of the fused kernel (rank 0's kernel, its own events) ----------------------------------------
    # The gradient runs on the tensor pipe as NP part products (fp16x2 split: 3, bf16x3 split: 6; both FP32-grade) of a
    # 128 x 112 x 112 tile per 128 chain-evaluations: executed tensor flop = NP * (112/100)^2 x the algorithmic 2 D^2.
    peak = L.C.c_double(0.0)
    L.check(lib.hmc_ffma_peak(L.C.byref(peak), 0, stream))
    flop = executed_local * 2.0 * D * D
    achieved = flop / (ms * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bf16_peak = float(peaks.get("bf16_tflops_sustained", 0.0)) or 2250.0
    nprod = 3.0 if fp16 else 6.0
    tensor_exec = achieved * nprod * (112.0 / D) ** 2
    traffic, traffic_src = None, None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "tc_kernel_traffic.json")))
        if tr.get("chains") == Nc and tr.get("niter") == Niter and tr.get("split") == ("fp16x2" if fp16 else "bf16x3"):
            traffic, traffic_src = float(tr["dram_bytes_per_launch"]), tr.get("source")
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "hmc_random_tc_kernel<UDT=true, %s> (tcgen05, 128 chains per CTA)" % ("fp16x2" if fp16 else "bf16x3"),
                "achieved": achieved, "peak": bf16_peak, "unit": "TFLOP/s", "frac": achieved / bf16_peak,
                "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step; the dense fp16 rate equals the bf16 rate)" if peaks
                                else "fallback: nominal dense bf16 2250"),
                "traffic": traffic, "traffic_source": traffic_src or "not captured for this configuration",
                "algorithmic_bytes": float(Nc) * Lc * (D * 4 + 16), "launch_ms": ms / K,
                "tensor_tflops_executed": tensor_exec, "frac_executed": tensor_exec / bf16_peak,
                "fp32_ffma_peak": peak.value / 1e12, "frac_of_fp32_ffma_peak": achieved / (peak.value / 1e12),
                "note": "achieved = algorithmic flop (executed gradient evals: sum L + one per trajectory start) * 2*D^2 / kernel time; "
                        "an FP32-grade gradient costs %.2f 16-bit tensor flop per algorithmic flop (tensor_tflops_executed); "
                        "fp32_ffma_peak is the FFMA microbenchmark of this run (what a CUDA-core kernel is bounded by)" % (nprod * 1.2544)}

    # ---- end-to-end leg through the public API, host buffers ----------------------------------------------------
    q_pinned = torch.from_numpy(q_start).pin_memory()
    del H, run, a
    torch.cuda.empty_cache()
    e2e_ms = []
    e2e_L = []
    ess = None
    for i in range(1 + K):
        H2 = S.HMC_sampler(D, None, None, Nchain=Nc, Niter=Niter, thin_rate=1, warm_up_num=warm, sampler_type="Random",
                           dt=DT, L_low=L_LOW, L_high=L_HIGH, dtype="float32", kernel="auto", seed=77 + i,
                           chain_id0=id0, target=spec, distributed=(world > 1))
        barrier()
        U.D2H_BYTES[0] = 0
        t0 = time.perf_counter()
        H2.gen_sample(q_pinned, verbose=False, quiet=True)       # H2D of q_start inside
        H2.compute_convergence_stats()                           # GPU reductions (+ NCCL), D2H of the partial sums
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t0
        tt = torch.tensor([dt_s], dtype=torch.float64, device=dev)
        ll = torch.tensor([float(H2.sum_L_local)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(ll)
        if i >= 1:
            e2e_d2h = int(U.D2H_BYTES[0])                        # counted where the mirror reads results back (utils._host)
            e2e_ms.append(float(tt.item()) * 1e3)
            e2e_L.append(float(ll.item()))
            ess = {"what": "reference-formula n_eff (utils.py:77-159) of the stored samples of one step's run, over its wall time incl. diagnostics",
                   "n_eff_median": float(np.median(H2.n_eff_q)), "n_eff_min": float(np.min(H2.n_eff_q)),
                   "rhat_median": float(np.median(H2.R_q)), "stored_samples": int(world * Nc * (Lc - 1)),
                   "ess_per_sec_median": float(np.median(H2.n_eff_q)) / float(tt.item()),
                   "ess_per_sec_min": float(np.min(H2.n_eff_q)) / float(tt.item()), "accept_R": H2.accept_R,
                   "kernel_ms": H2.kernel_ms}
        del H2
    log("e2e done")
    e2e_value = float(np.sum(e2e_L) / (np.sum(e2e_ms) * 1e-3))
    h2d = Nc * D * 4
    d2h = e2e_d2h                                     # packed statistics buffer, counters, the all-lags variogram buffer

    secondary = None
    if not args.no_secondary:
        secondary = secondary_measurements(torch, dist, S, U, L, lib, rank, world, dev, log)

    cpu = None
    if rank == 0 and not args.no_cpu:
        # separate process: forking a pool out of a CUDA/NCCL-initialised parent is not safe
        try:
            out = subprocess.check_output([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                           "--warmup", "0"], timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
            cpu = json.loads(out.decode().strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:   # the baseline is reported, never required
            cpu = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "failed: %r" % (exc,)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "clocks": sampler_thread.summary() if sampler_thread else None,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": float(np.mean(e2e_ms)),
                        "note": "gen_sample + compute_convergence_stats per step; q_chain (%.1f GB per GPU) stays device-resident and is "
                                "never copied to the host inside the timed region" % (Nc * Lc * D * 4 / 1e9)},
                "gpu_launches": K,
                "roofline": roofline, "cpu_baseline": cpu, "ess": ess, "secondary": secondary,
                "grad_evals_executed_per_sec": float(tot[1].item()) / (ms_max * 1e-3),
                "reference_unit_steps_per_sec": value * D,
                "accept_rate": (acc_post + int(dc[0])) / float(n_traj)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
