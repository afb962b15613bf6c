"""Host-side mirror of the reference's ``samplers.py`` sampler classes, backed by hand-written sm_100a CUDA.

Same constructor, ``gen_sample`` / ``compute_convergence_stats`` API and result attributes as
/root/reference/samplers.py:4-65, 297-384 so that the ``case*-script.py`` drivers run against it; the hot loops
(``gen_sample_random`` :387-491, ``gen_sample_NUTS`` :495-808, ``K/E/p_sample/leap_frog`` :811-839) and the
diagnostics (utils.py:77-179) run in libhmc_b200.so through the C-ABI of include/hmc_b200.h.  There is no CPU
fallback: a target that is not a multivariate normal, or a missing CUDA library, raises.

Extra keyword-only constructor arguments (defaults keep the reference behaviour):
  dtype="float32"|"float64", seed=0 (Philox key), kernel="auto"|"generic"|"fast"|"tc"|"bigd", draws=None (the reference's
  own draws as structured tapes, see tests/golden/make_golden.py), on_dmax="assert"|"stop" (NUTS, SURVEY H6),
  chain_id0=0 / distributed=False (chains sharded over ranks; counters and moments are all-reduced),
  iter_block=None (iterations per kernel launch), target=None (explicit ``MVNSpec`` instead of probing V/dVdq),
  tc_precision="bf16x3"|"fp16x2" (split of the tensor-core gradient product: three bf16 parts / six tensor passes -- the
  default of the D = 100 kernel and of NUTS on the large-D path -- or two fp16 parts / three passes -- the default of the
  large-D GEMM path of the random-trajectory sampler; at D = 100, rho = 0.95 fp16x2 is 10 % faster at 3x the trajectory error,
  see DESIGN 4.0; a D = 100 run whose start points leave the fp16 range repeats itself with bf16x3).
"""
import os

from utils import *  # noqa: F401,F403  (samplers.py:1)
import utils as _utils

import hmc_b200_lib as _L


class MVNSpec(object):
    """The multivariate-normal target behind the driver closures V / dVdq (case1-script.py:39-49):
    dVdq(q) = P (q - mu),  V(q) = 0.5 (q-mu)^T P (q-mu) + const."""

    def __init__(self, mu, P, const):
        self.mu = np.asarray(mu, dtype=float)
        self.P = np.asarray(P, dtype=float)
        self.const = float(const)
        self.D = self.mu.shape[0]

    @classmethod
    def from_cov(cls, q0, cov0):
        cov0 = np.asarray(cov0, dtype=float)
        D = cov0.shape[0]
        sign, logdet = np.linalg.slogdet(cov0)
        return cls(q0, np.linalg.inv(cov0), 0.5 * (D * np.log(2 * np.pi) + logdet))


def leap_frog_entry(D):
    """The library entry point ``HMC_sampler.leap_frog`` calls for dimension D: ``hmc_leap_frog`` (one warp per pair) up to
    D = 1024, ``hmc_leap_frog_bigd`` (the large-D tensor-core GEMM, float32, D <= 8192) above."""
    return "hmc_leap_frog" if D <= 1024 else "hmc_leap_frog_bigd"


def random_runs_bigd(D, dtype, kernel, cov_p_identity):
    """Whether the random-trajectory sampler runs on the large-D GEMM path (csrc/api.cu's AUTO rule and the path's coverage):
    float32 and 128 <= D <= 8192 with the identity metric, under kernel="bigd", or under "auto" for D % 256 == 0 and D > 1024;
    a dense ``cov_p`` for 1024 < D <= 8192 under "bigd" or "auto" (up to D = 1024 the generic kernel runs a dense metric)."""
    if dtype != "float32" or kernel not in ("auto", "bigd") or not 128 <= D <= 8192:
        return False
    if not cov_p_identity:
        return D > 1024
    return kernel == "bigd" or D % 256 == 0 or D > 1024


def equicorrelated_cov(D, rho):
    """cov0 of the reference's drivers: (1 - rho) I + rho 1 1^T (case3-script.py:31-33)."""
    return (1.0 - rho) * np.eye(D) + rho * np.ones((D, D))


def extract_mvn_target(D, V, dVdq, rtol=1e-8):
    """Recover (mu, P, const) from the opaque callables by probing (SURVEY H1): g0 = dVdq(0), column i of P is
    dVdq(e_i) - g0, mu solves P mu = -g0, const = V(mu).  Verified at random points; anything that is not an
    exact quadratic form raises NotImplementedError -- a CUDA kernel cannot call Python and there is no CPU path."""
    zero = np.zeros(D)
    g0 = np.asarray(dVdq(zero), dtype=float).reshape(D)
    P = np.empty((D, D))
    for i in range(D):
        e = np.zeros(D)
        e[i] = 1.0
        P[:, i] = np.asarray(dVdq(e), dtype=float).reshape(D) - g0
    mu = np.linalg.solve(P, -g0)
    const = float(V(mu))
    rng = np.random.RandomState(12345)
    scale = max(1.0, float(np.abs(mu).max()))
    for _ in range(3):
        x = mu + scale * rng.standard_normal(D)
        g = np.asarray(dVdq(x), dtype=float).reshape(D)
        g_fit = np.dot(P, x - mu)
        v = float(V(x))
        v_fit = 0.5 * np.dot(x - mu, g_fit) + const
        if (not np.allclose(g, g_fit, rtol=rtol, atol=rtol * max(1.0, np.abs(g).max()))) or \
                abs(v - v_fit) > 1e-6 * max(1.0, abs(v)):
            raise NotImplementedError("V/dVdq are not a multivariate-normal potential; the B200 build only "
                                      "implements MVN targets in CUDA and has no CPU fallback")
    if not np.allclose(P, P.T, rtol=1e-6, atol=1e-9 * np.abs(P).max()):
        raise NotImplementedError("gradient is not that of a symmetric quadratic form")
    return MVNSpec(mu, P, const)


class sampler(object):
    """Parent class holding the chain bookkeeping (samplers.py:4-65)."""

    def __init__(self, D, target_lnL, Nchain=2, Niter=1000, thin_rate=1, warm_up_num=0):
        self.D = D
        self.target_lnL = target_lnL
        self.Nchain = Nchain
        self.Niter = Niter
        self.thin_rate = thin_rate
        self.warm_up_num = warm_up_num
        self.L_chain = 1 + ((self.Niter - self.warm_up_num) // self.thin_rate)       # samplers.py:31
        # Results live on the device (chain-major, compute dtype); the float64 host arrays of the reference
        # layout (Nchain, L_chain, D) are materialised on first access.
        self._q_dev = None
        self._q_host = None
        self._lnL_host = None
        self.R_q = None
        self.R_lnL = None
        self.n_eff_q = None
        self.accept_R_warm_up = None
        self.accept_R = None
        self.dt_total = 0
        self.N_total_steps = 0

    @property
    def q_chain(self):
        if self._q_host is None:
            if self._q_dev is None:
                self._q_host = np.zeros((self.Nchain, self.L_chain, self.D), dtype=float)   # samplers.py:33
            else:
                self._q_host = self._q_dev.double().cpu().numpy()
        return self._q_host

    @q_chain.setter
    def q_chain(self, value):
        self._q_host = value
        self._q_dev = None

    @property
    def q_chain_device(self):
        """(Nchain, L_chain, D) CUDA tensor in the compute dtype (no host copy)."""
        return self._q_dev

    def compute_convergence_stats(self):
        """R_q, n_eff_q over stored samples 1.. (samplers.py:53-64), on the GPU."""
        src = self._q_dev if self._q_dev is not None else self.q_chain
        group = None if getattr(self, "distributed", False) else False
        self.R_q, self.n_eff_q = _utils.convergence_stats(src[:, 1:, :], warm_up_num=0, thin_rate=1, group=group)
        return

    def sample_summary(self, xmax=None, dx=None):
        """Everything ``plot_samples`` derives from the samples (samplers.py:84-113, 160-186, 209-250), computed by GPU
        reductions over the device-resident outputs (csrc/summary.cu): per-dimension mean / variance over stored samples
        1.., 2.5 / 97.5 percentiles, plot ranges and histograms of q1, q2 (all stored samples) and of the centred energies
        E and the energy differences dE (stored samples 1..).  Sharded runs all-reduce the counts."""
        q = self._q_dev
        assert q is not None, "sample_summary needs a finished gen_sample"
        group = None if getattr(self, "distributed", False) else False
        out = {}
        out["q_mean"], out["q_var"] = _utils.device_moments(q[:, 1:, :], group=group)         # samplers.py:209-216, 244-250

        def rng_of(x, N):
            lo, hi = _utils.device_percentile(x, [2.5, 97.5], group=group)                     # samplers.py:97-103
            c, r = (hi + lo) / 2., (hi - lo) * 2.5
            return c - r / 2., c + r / 2., r

        for name, col in (("q1", 0), ("q2", 1)):
            if col >= self.D:
                continue
            x = q[:, :, col]
            if xmax is None:
                lo, hi, r = rng_of(x, None)
            else:
                lo, hi, r = -xmax, xmax, 2. * xmax                                             # samplers.py:117-121
            w = r / 100. if dx is None else dx                                                 # samplers.py:124-128
            edges = np.arange(lo, hi, w)
            out[name + "_range"] = (lo, hi)
            out[name + "_edges"] = edges
            out[name + "_hist"] = _utils.device_histogram(x, edges, group=group)[0]             # samplers.py:160-175
        E, dE = getattr(self, "_E_dev", None), getattr(self, "_dE_dev", None)
        if E is not None and E.shape[1] > 1:
            Em, _ = _utils.device_moments(E[:, 1:, None], group=group)                         # samplers.py:86-87
            out["E_mean"] = float(Em[0])
            lo, hi = _utils.device_percentile(E[:, 1:], [2.5, 97.5], group=group) - out["E_mean"]   # samplers.py:177-183
            c, r = (lo + hi) / 2., (hi - lo) * 2.5
            edges = np.arange(c - r / 2., c + r / 2., r / 100.)
            out["E_range"] = (c - r / 2., c + r / 2.)
            out["E_edges"] = edges
            out["E_hist"] = _utils.device_histogram(E[:, 1:], edges, shift=out["E_mean"], group=group)[0]
            out["dE_hist"] = _utils.device_histogram(dE[:, 1:], edges, group=group)[0]         # samplers.py:184-186
        return out

    def plot_samples(self, title_prefix, show=False, savefig=False, xmax=None, dx=None, plot_normal=True,
                     plot_cov=True, q0=None, cov0=None):
        """3x3 summary figure (samplers.py:67-291).  Drawing is presentation and outside the B200 hot-path build; the
        numbers the figure shows are computed on the GPU (``sample_summary``) and printed instead."""
        if self._q_dev is None:
            print("plot_samples: no device samples; skipped for %s" % title_prefix)
            return
        s = self.sample_summary(xmax=xmax, dx=dx)
        self.summary = s
        print("plot_samples[%s]: D/Nchain/Niter/Warm-up/Thin = %d/%d/%d/%d/%d (figure not drawn: plotting is outside the hot path)"
              % (title_prefix, self.D, self.Nchain, self.Niter, self.warm_up_num, self.thin_rate))
        if q0 is not None:
            print("  bias(mean) min/max: %.3e / %.3e" % (np.min(s["q_mean"] - q0), np.max(s["q_mean"] - q0)))
        if cov0 is not None:
            ratio = s["q_var"] / np.diag(np.asarray(cov0))
            print("  estimated/true variance min/max: %.4f / %.4f" % (ratio.min(), ratio.max()))
        if self.R_q is not None:
            print("  R med/std: %.3f / %.3f" % (np.median(self.R_q), np.std(self.R_q)))
            print("  Ntot/eff med: %.1E/%.1E" % (self.L_chain * self.Nchain, np.median(self.n_eff_q)))
            print("  #steps/ES med: %.2E" % (self.N_total_steps / np.median(self.n_eff_q)))
        if self.accept_R is not None:
            print("  RA after warm-up: %.3f" % self.accept_R)
        return


class HMC_sampler(sampler):
    """HMC sampler for multivariate-normal targets (samplers.py:297-384), CUDA backed.

    ``kernel`` of the random-trajectory sampler (float32, ``cov_p = I`` unless noted; "auto" picks as csrc/api.cu does,
    ``random_runs_bigd`` is the large-D rule):
      "tc"       tensor-core kernel, D % 4 == 0, D <= 100 (zero-padded 100-wide tile); auto for 52 <= D <= 100
      "bigd"     large-D GEMM path, any 128 <= D <= 8192 (padded to D rounded up to 32); auto for D % 256 == 0 and D > 1024.
                 A dense ``cov_p`` for 1024 < D <= 8192 (auto there too): its V, K and p = Lc z are batched tensor-core products
                 at the trajectory ends
      "fast"     FFMA2 kernel, 20 < D <= 128; auto where neither of the above applies
      "generic"  warp-per-chain kernel, D <= 1024, float64 and dense ``cov_p`` too; auto for the rest

    ``kernel`` of the NUTS sampler (reported as ``nuts_kernel``):
      "tc"       tensor-core kernel, D = 100, float32, ``cov_p = I``, d_max <= 12; auto there
      "bigd"     large-D GEMM path, any 128 <= D <= 8192, float32, ``cov_p = I`` (bf16x3 split unless tc_precision="fp16x2");
                 auto for D > 256
      "generic"  warp-per-chain kernel, D <= 256, float64 and dense ``cov_p`` too; auto for the rest
    """

    def __init__(self, D, V, dVdq, Nchain=2, Niter=1000, thin_rate=1, warm_up_num=0,
                 cov_p=None, sampler_type="Fixed", L=None, global_dt=True, dt=None,
                 L_low=None, L_high=None, log2L=None, d_max=10, *,
                 dtype="float32", seed=0, kernel="auto", draws=None, on_dmax="assert", chain_id0=0,
                 distributed=False, iter_block=None, target=None, tc_precision=None):
        sampler.__init__(self, D=D, target_lnL=None, Nchain=Nchain, Niter=Niter, thin_rate=thin_rate,
                         warm_up_num=warm_up_num)
        self.V = V
        self.dVdq = dVdq
        assert (sampler_type == "Fixed") or (sampler_type == "Random") or (sampler_type == "NUTS") or \
            (sampler_type == "Static")                                               # samplers.py:331
        assert (dt is not None)                                                      # samplers.py:332
        self.dt = dt
        self.global_dt = global_dt
        self.sampler_type = sampler_type
        if self.sampler_type == "Fixed":
            assert (L is not None)
            self.L = L
        elif self.sampler_type == "Random":
            assert (L_low is not None) and (L_high is not None)
            self.L_low = L_low
            self.L_high = L_high
        elif self.sampler_type == "Static":
            assert (log2L is not None)
            self.log2L = log2L
        elif self.sampler_type == "NUTS":
            assert d_max is not None
            self.d_max = d_max
        self._cov_p_identity = cov_p is None
        if cov_p is None:                                                            # samplers.py:352-356
            self.cov_p = np.diag(np.ones(self.D))
        else:
            self.cov_p = np.asarray(cov_p, dtype=float)
            self._cov_p_identity = bool(np.array_equal(self.cov_p, np.eye(self.D)))
        self.inv_cov_p = np.linalg.inv(self.cov_p)
        self._E_dev = None
        self._dE_dev = None
        self._E_host = None
        self._dE_host = None
        # B200 extras
        assert dtype in ("float32", "float64")
        assert kernel in _L.KERNELS
        assert on_dmax in ("assert", "stop")
        assert tc_precision in (None, "fp16x2", "bf16x3")
        self.tc_precision = tc_precision
        self.dtype = dtype
        self.seed = int(seed)
        self.kernel = kernel
        self.draws = draws
        self.on_dmax = on_dmax
        self.chain_id0 = int(chain_id0)
        self.distributed = bool(distributed)
        self.iter_block = iter_block
        self.target = target
        self.kernel_ms = 0.0
        self.sum_L = 0
        self.n_leapfrog = None
        self.status = None

    # ---- reference-layout host views of the energy streams (samplers.py:359-360) ----
    @property
    def E_chain(self):
        if self._E_host is None:
            self._E_host = np.zeros((self.Nchain, self.L_chain, 1)) if self._E_dev is None else \
                self._E_dev.cpu().numpy()[:, :, None]
        return self._E_host

    @property
    def lnL_chain(self):
        """(Nchain, L_chain, 1) zeros, as the reference allocates it (samplers.py:34; its live samplers never fill it)."""
        if self._lnL_host is None:
            self._lnL_host = np.zeros((self.Nchain, self.L_chain, 1))
        return self._lnL_host

    @property
    def dE_chain(self):
        if self._dE_host is None:
            self._dE_host = np.zeros((self.Nchain, self.L_chain, 1)) if self._dE_dev is None else \
                self._dE_dev.cpu().numpy()[:, :, None]
        return self._dE_host

    # ---- device-side target ----
    def _build_target(self, torch, dev):
        spec = self.target if self.target is not None else extract_mvn_target(self.D, self.V, self.dVdq)
        self.target = spec
        tdt = torch.float32 if self.dtype == "float32" else torch.float64
        D = self.D
        D_pad = (D + 3) // 4 * 4

        def dev_mat_t(M):
            out = np.zeros((D, D_pad))
            out[:, :D] = np.asarray(M, dtype=float).T
            return torch.from_numpy(out).to(device=dev, dtype=tdt).contiguous()

        def dev_vec(v):
            out = np.zeros(D_pad)
            out[:D] = v
            return torch.from_numpy(out).to(device=dev, dtype=tdt).contiguous()

        keep = {}
        F = spec.P if self._cov_p_identity else np.dot(self.inv_cov_p, spec.P)      # samplers.py:835
        keep["Ft"] = dev_mat_t(F)
        if not self._cov_p_identity:
            keep["Pt"] = dev_mat_t(spec.P)
            keep["Mit"] = dev_mat_t(self.inv_cov_p)
            keep["Lct"] = dev_mat_t(np.linalg.cholesky(self.cov_p))
        keep["mu"] = dev_vec(spec.mu)
        dt_vec = np.broadcast_to(np.asarray(self.dt, dtype=float), (D,))             # scalar or (D,) (samplers.py:333)
        keep["dt"] = dev_vec(dt_vec)
        t = _L.Target()
        t.D, t.D_pad = D, D_pad
        t.Ft = keep["Ft"].data_ptr()
        t.Pt = keep["Pt"].data_ptr() if "Pt" in keep else None
        t.Mit = keep["Mit"].data_ptr() if "Mit" in keep else None
        t.Lct = keep["Lct"].data_ptr() if "Lct" in keep else None
        t.mu = keep["mu"].data_ptr()
        t.dt = keep["dt"].data_ptr()
        t.v_const = spec.const
        return t, keep, tdt

    def _blocks(self):
        nb = self.Niter if not self.iter_block else int(self.iter_block)
        nb = max(1, nb)
        edges = list(range(0, self.Niter, nb)) + [self.Niter]
        if self.Niter == 0:
            edges = [0, 0]
        return list(zip(edges[:-1], edges[1:]))

    def _all_reduce(self, torch, t):
        if self.distributed:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.all_reduce(t)
        return t

    def gen_sample(self, q_start, N_save_chain0=0, verbose=True, quiet=False):
        """Dispatch on sampler type (samplers.py:363-383).  "Fixed" runs the random-length loop with a constant
        L (SURVEY H8); "Static" stays the no-op it is in the reference (Q11)."""
        if (self.sampler_type == "Random"):
            self.gen_sample_random(q_start, N_save_chain0, verbose, quiet)
        elif (self.sampler_type == "NUTS"):
            self.gen_sample_NUTS(q_start, N_save_chain0, verbose)
        elif (self.sampler_type == "Fixed"):
            self.L_low, self.L_high = int(self.L), int(self.L) + 1
            self.gen_sample_random(q_start, N_save_chain0, verbose, quiet)
        return

    def _to_device(self, torch, q_start, dev, tdt):
        """q_start: numpy array or (pinned) host torch tensor, shape (Nchain, D)."""
        if isinstance(q_start, torch.Tensor):
            return q_start.to(device=dev, dtype=tdt, non_blocking=True).contiguous()
        return torch.from_numpy(np.ascontiguousarray(np.asarray(q_start), dtype=float)).to(device=dev, dtype=tdt).contiguous()

    def _fp16x2_flag(self):
        """FLAG_TC_FP16X2 when tc_precision asks for the two-part fp16 split of the tensor-core gradient product and the target
        allows it, else 0.  The split needs a target whose scale is not far below 1 (fp16 subnormals); otherwise tc_precision
        falls back to bf16x3."""
        if self.tc_precision != "fp16x2":
            return 0
        if float(np.min(1.0 / np.sqrt(np.abs(np.diag(self.target.P))))) < 2.0 ** -10:
            self.tc_precision = "bf16x3"
            return 0
        return _L.FLAG_TC_FP16X2

    @staticmethod
    def _set_workspace(torch, dev, a, nbytes):
        """Point the launch arguments a at a new 1024-byte aligned device workspace of nbytes; returns the tensor that owns it."""
        buf, a.workspace = _L.aligned_workspace(torch, dev, nbytes)
        a.workspace_bytes = nbytes
        return buf

    def prepare_random(self, q_start, N_save_chain0=0):
        """Allocate the device-resident outputs/state and build the C-ABI argument block (hmc_random_args) of
        the random-trajectory sampler; the caller launches iteration blocks with hmc_random_run."""
        import torch
        assert q_start.shape[0] == self.Nchain                                       # samplers.py:396
        dev = torch.device("cuda", torch.cuda.current_device())
        tgt, keep, tdt = self._build_target(torch, dev)
        Nc, D, Lc = self.Nchain, self.D, self.L_chain
        f64 = torch.float64
        owns0 = self.chain_id0 == 0
        save_chain = N_save_chain0 > 0
        self._q_dev = torch.empty((Nc, Lc, D), dtype=tdt, device=dev)     # every stored sample / energy is written by the kernel
        self._E_dev = torch.empty((Nc, Lc), dtype=f64, device=dev)
        self._dE_dev = torch.empty((Nc, Lc), dtype=f64, device=dev)
        self._q_host = self._E_host = self._dE_host = None
        keep["qs"] = self._to_device(torch, q_start, dev, tdt)
        keep["state_q"] = torch.empty((Nc, D), dtype=tdt, device=dev)
        # scratch: work-queue head, per-chain progress words, range flag (cleared by the launches themselves)
        keep["state_g"] = torch.empty((Nc + 64,), dtype=torch.float64, device=dev)
        keep["state_e"] = torch.empty((Nc,), dtype=f64, device=dev)
        counters = torch.zeros((8,), dtype=torch.int64, device=dev)      # [0..4) kernel counters, [4] chains of this rank
        a = _L.RandomArgs()
        a.dtype = _L.HMC_F32 if self.dtype == "float32" else _L.HMC_F64
        a.kernel = _L.KERNELS[self.kernel]
        a.Nchain, a.chain_id0 = Nc, self.chain_id0
        a.Niter, a.warm_up_num, a.thin_rate = self.Niter, self.warm_up_num, self.thin_rate
        a.L_low, a.L_high = int(self.L_low), int(self.L_high)
        a.N_save_chain0 = int(N_save_chain0) if owns0 else 0
        a.seed = self.seed
        a.target = tgt
        a.flags = _L.FLAG_UNIFORM_DT if np.ndim(self.dt) == 0 or np.all(np.asarray(self.dt) == np.asarray(self.dt).flat[0]) else 0
        bigd = random_runs_bigd(D, self.dtype, self.kernel, self._cov_p_identity)
        if self.tc_precision is None:
            self.tc_precision = "fp16x2" if bigd else "bf16x3"
        # (the fp16 split also needs |q - mu| < 16384: the tensor-core kernel checks it, word 16 + Nchain of state_g)
        a.flags |= self._fp16x2_flag()
        a.flags |= (int(os.environ.get("HMC_B200_TILE_VARIANT", "0")) & 0xff) << 8      # tuning knob
        a.q_start = keep["qs"].data_ptr()
        if self.draws is not None:
            keep["p_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["p_tape"], dtype=float)).to(dev)
            keep["L_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["L_tape"], dtype=np.int32)).to(dev)
            keep["u_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["u_tape"], dtype=float)).to(dev)
            assert keep["p_tape"].shape == (Nc, self.Niter + 1, D)
            assert keep["L_tape"].shape == (Nc, self.Niter) and keep["u_tape"].shape == (Nc, self.Niter)
            a.p_tape, a.L_tape, a.u_tape = (keep[k].data_ptr() for k in ("p_tape", "L_tape", "u_tape"))
        a.q_chain, a.E_chain, a.dE_chain = self._q_dev.data_ptr(), self._E_dev.data_ptr(), self._dE_dev.data_ptr()
        a.state_q, a.state_g, a.state_eprev = keep["state_q"].data_ptr(), keep["state_g"].data_ptr(), \
            keep["state_e"].data_ptr()
        a.counters = counters.data_ptr()
        if bigd:                                  # large-D GEMM path: its scratch (split operands, state, per-chain scalars)
            keep["workspace"] = self._set_workspace(torch, dev, a, int(_L.load().hmc_random_workspace_bytes(a)))
        if save_chain and owns0:
            keep["phi"] = torch.zeros((N_save_chain0, int(self.L_high), 2), dtype=f64, device=dev)
            keep["phi_len"] = torch.zeros((N_save_chain0,), dtype=torch.int32, device=dev)
            keep["dec"] = torch.zeros((N_save_chain0 + 1,), dtype=torch.int32, device=dev)
            a.phi_q, a.phi_len, a.decision_chain = (keep[k].data_ptr() for k in ("phi", "phi_len", "dec"))
        return dict(args=a, keep=keep, counters=counters, device=dev)

    def gen_sample_random(self, q_start, N_save_chain0, verbose, quiet=False):
        """Random trajectory length sampler (samplers.py:387-491) on the GPU."""
        import torch
        lib = _L.load()
        say = (lambda *x: None) if quiet else print
        run = self.prepare_random(q_start, N_save_chain0)
        a, keep, counters, dev = run["args"], run["keep"], run["counters"], run["device"]
        Nc, D = self.Nchain, self.D
        owns0 = self.chain_id0 == 0
        save_chain = N_save_chain0 > 0
        stream = _L.current_stream_ptr()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if verbose:
            say("Running %d chains x %d iterations on %s (%s, kernel=%s)" %
                (Nc, self.Niter, torch.cuda.get_device_name(dev), self.dtype, self.kernel))
        ev0.record()
        for (b, e) in self._blocks():
            a.iter_begin, a.iter_end = b, e
            _L.check(lib.hmc_random_run(a, stream))
        ev1.record()
        ev1.synchronize()
        self.kernel_ms = ev0.elapsed_time(ev1)
        tc_ran = self.dtype == "float32" and self._cov_p_identity and D % 4 == 0 and \
            ((self.kernel == "tc" and 4 <= D <= 100) or (self.kernel == "auto" and 52 <= D <= 100))       # csrc/api.cu AUTO rule
        if (a.flags & _L.FLAG_TC_FP16X2) and tc_ran and int(keep["state_g"].view(torch.int32)[16 + Nc].item()) != 0:
            # a start point left the range of the fp16 split (tensor-core kernel only): repeat with the bf16x3 split
            self.tc_precision = "bf16x3"
            return self.gen_sample_random(q_start, N_save_chain0, verbose, quiet)
        if verbose:                                                                  # samplers.py:478-481 (Q10)
            self.dt_total += self.kernel_ms * 1e-3
            say("Time taken: %.2f\n" % (self.kernel_ms * 1e-3))
        # one packed buffer: local counters and chain count, all-reduced copy behind them -> one collective, one D2H
        counters[4] = Nc
        if self.distributed:
            both = _utils._host(torch.cat([counters, self._all_reduce(torch, counters.clone())]))
        else:
            both = _utils._host(torch.cat([counters, counters]))
        self.sum_L_local = int(both[2])
        acc_warm, acc_post, sumL, sumL2, nchain_all = (int(v) for v in both[8:13])
        self.sum_L = sumL
        self.N_total_steps = nchain_all * (1 + 2 * self.Niter) + D * sumL2          # samplers.py:417,435,450,456 (Q3)
        say("Compute acceptance rate")
        if self.warm_up_num > 0:                                                     # samplers.py:484-488
            self.accept_R_warm_up = acc_warm / float(nchain_all * self.warm_up_num)
            say("During warm up: %.3f" % self.accept_R_warm_up)
        self.accept_R = acc_post / float(nchain_all * (self.Niter - self.warm_up_num + 1))
        say("After warm up: %.3f" % self.accept_R)
        say("Completed.")
        if save_chain and owns0:                                                     # samplers.py:397-400, 442-475
            nrec = min(N_save_chain0, self.Niter)
            lens = keep["phi_len"].cpu().numpy()
            phi = keep["phi"].cpu().numpy()
            self.phi_q = [phi[i, :lens[i], :].copy() for i in range(nrec)]
            self.decision_chain = keep["dec"].cpu().numpy().astype(int)[:, None]
        return

    def gen_sample_NUTS(self, q_start, N_save_chain0, verbose):
        """NUTS sampler (samplers.py:495-808) on the GPU."""
        import torch
        lib = _L.load()
        assert q_start.shape[0] == self.Nchain                                       # samplers.py:510
        if N_save_chain0 > 0:
            self.phi_q = []                                                          # samplers.py:514 (never filled)
        dev = torch.device("cuda", torch.cuda.current_device())
        tgt, keep, tdt = self._build_target(torch, dev)
        Nc, D, Lc = self.Nchain, self.D, self.L_chain
        f64 = torch.float64
        self._q_dev = torch.zeros((Nc, Lc, D), dtype=tdt, device=dev)
        self._E_dev = torch.zeros((Nc, Lc), dtype=f64, device=dev)
        self._dE_dev = torch.zeros((Nc, Lc), dtype=f64, device=dev)
        self._q_host = self._E_host = self._dE_host = None
        qs = self._to_device(torch, q_start, dev, tdt)
        state_q = torch.empty((Nc, D), dtype=tdt, device=dev)
        state_e = torch.zeros((Nc,), dtype=f64, device=dev)
        counters = torch.zeros((4,), dtype=torch.int64, device=dev)
        status = torch.zeros((Nc,), dtype=torch.int32, device=dev)
        nleap = torch.zeros((Nc,), dtype=torch.int64, device=dev)
        # (+128 row blocks: the tensor-core kernel indexes the stack rows by resident slot, 128 per CTA, not by chain)
        scratch = torch.zeros((Nc + 128, 2 * (self.d_max + 1) + 7, tgt.D_pad), dtype=tdt, device=dev)
        a = _L.NutsArgs()
        a.dtype = _L.HMC_F32 if self.dtype == "float32" else _L.HMC_F64
        a.kernel = _L.KERNELS[self.kernel]
        # (mirror of the library's AUTO rule, for reports: csrc/api.cu hmc_nuts_run)
        bigd_ok = self.dtype == "float32" and self._cov_p_identity and 128 <= D <= 8192
        if self.kernel in ("auto", "tc") and self.dtype == "float32" and D == 100 and self.d_max <= 12:
            self.nuts_kernel = "tc"
        elif bigd_ok and (self.kernel == "bigd" or (self.kernel == "auto" and D > 256)):
            self.nuts_kernel = "bigd"
        else:
            self.nuts_kernel = "generic"
        a.Nchain, a.d_max, a.chain_id0 = Nc, int(self.d_max), self.chain_id0
        a.Niter, a.warm_up_num, a.thin_rate = self.Niter, self.warm_up_num, self.thin_rate
        a.on_dmax = 0 if self.on_dmax == "assert" else 1
        a.seed = self.seed
        a.target = tgt
        a.q_start = qs.data_ptr()
        if self.draws is not None:
            keep["p_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["p_tape"], dtype=float)).to(dev)
            keep["dir_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["dir_tape"], dtype=np.int32)).to(dev)
            keep["u_tape"] = torch.from_numpy(np.ascontiguousarray(self.draws["u_tape"], dtype=float)).to(dev)
            assert keep["p_tape"].shape == (Nc, self.Niter + 1, D)
            a.p_tape, a.dir_tape, a.u_tape = (keep[k].data_ptr() for k in ("p_tape", "dir_tape", "u_tape"))
            a.tape_dir_stride, a.tape_u_stride = keep["dir_tape"].shape[1], keep["u_tape"].shape[1]
        a.q_chain, a.E_chain, a.dE_chain = self._q_dev.data_ptr(), self._E_dev.data_ptr(), self._dE_dev.data_ptr()
        a.state_q, a.state_eprev = state_q.data_ptr(), state_e.data_ptr()
        a.scratch, a.counters, a.status, a.n_leapfrog = scratch.data_ptr(), counters.data_ptr(), status.data_ptr(), \
            nleap.data_ptr()
        if self.nuts_kernel == "bigd":            # large-D GEMM path: its scratch (split operands, x / p / gradient rows, chain states)
            if self.tc_precision is None:
                self.tc_precision = "bf16x3"      # tree decisions are sign tests and near-ties: the split without fp16's V bias
            a.flags |= self._fp16x2_flag()
            keep["workspace"] = self._set_workspace(torch, dev, a, int(lib.hmc_nuts_workspace_bytes(a)))
        stream = _L.current_stream_ptr()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if verbose:
            print("Running %d NUTS chains x %d iterations on %s (%s, kernel=%s)" %
                  (Nc, self.Niter, torch.cuda.get_device_name(dev), self.dtype, self.nuts_kernel))
        ev0.record()
        for (b, e) in self._blocks():
            a.iter_begin, a.iter_end = b, e
            _L.check(lib.hmc_nuts_run(a, stream))
        ev1.record()
        ev1.synchronize()
        self.kernel_ms = ev0.elapsed_time(ev1)
        if verbose:
            self.dt_total += self.kernel_ms * 1e-3
            print("Time taken: %.2f\n" % (self.kernel_ms * 1e-3))
        c = self._all_reduce(torch, counters.clone()).cpu().numpy()
        nchain_all = self._all_reduce(torch, torch.tensor([Nc], dtype=torch.int64, device=dev)).item()
        n_leap, n_doubling, n_instab, n_dmax = (int(v) for v in c)
        self.n_leapfrog_total, self.n_doublings, self.n_instability, self.n_dmax = n_leap, n_doubling, n_instab, n_dmax
        self.n_leapfrog = nleap.cpu().numpy()
        self.status = status.cpu().numpy()
        for _ in range(n_instab):
            if _ < 10:
                print("Large energy difference instability.")                      # samplers.py:650
        if n_dmax > 0 and self.on_dmax == "assert":                                  # samplers.py:596-598 (Q7)
            print("Doubling number d exceeds d_max = %d" % self.d_max)
            assert False
        self.N_total_steps = nchain_all * (1 + self.Niter) + (D + 1) * n_leap       # samplers.py:552,570,615,620,640,644
        print("Compute acceptance rate: By default equal to 1.")                    # samplers.py:800-805
        if self.warm_up_num > 0:
            self.accept_R_warm_up = 1.
            print("During warm up: %.3f" % self.accept_R_warm_up)
        self.accept_R = 1.
        print("After warm up: %.3f" % self.accept_R)
        print("Completed.")
        return

    # ---- host mirrors of the primitives (samplers.py:811-839), for API completeness / small checks ----
    def K(self, p):
        return np.dot(p, np.dot(self.inv_cov_p, p)) / 2.

    def E(self, q, p):
        return self.V(q) + self.K(p)

    def p_sample(self):
        return np.random.multivariate_normal(np.zeros(self.D), self.cov_p, size=1)

    def leap_frog(self, p_old, q_old, nsteps=1):
        """One leapfrog step (samplers.py:831-839) -- on the GPU, for a single (p, q) pair or a batch of rows:
        p' = p - dt M^-1 dVdq(q) / 2, q' = q + dt p', p'' = p' - dt M^-1 dVdq(q') / 2, as the reference writes it (force times
        M^-1, q moved by p: Q9).  Returns (p_new, q_new) as float64 numpy arrays of the input's shape.  ``nsteps`` > 1 repeats the
        step (this repo's extension).  D <= 1024 runs ``hmc_leap_frog``; above, float32 runs ``hmc_leap_frog_bigd`` on the large-D
        GEMM (up to D = 8192, bf16x3 split unless tc_precision="fp16x2"; there nsteps > 1 merges the half kicks between steps, which
        changes the last bits)."""
        import torch
        lib = _L.load()
        dev = torch.device("cuda", torch.cuda.current_device())
        t, keep, tdt = self._build_target(torch, dev)
        p = np.asarray(p_old, dtype=float)
        q = np.asarray(q_old, dtype=float)
        shape = q.shape
        p2, q2 = p.reshape(-1, self.D), q.reshape(-1, self.D)
        assert p2.shape == q2.shape
        pd = torch.from_numpy(np.ascontiguousarray(p2)).to(device=dev, dtype=tdt)
        qd = torch.from_numpy(np.ascontiguousarray(q2)).to(device=dev, dtype=tdt)
        pn, qn = torch.empty_like(pd), torch.empty_like(qd)
        dtype = _L.HMC_F32 if self.dtype == "float32" else _L.HMC_F64
        if leap_frog_entry(self.D) == "hmc_leap_frog":
            _L.check(lib.hmc_leap_frog(dtype, t, q2.shape[0], _L.ptr(pd), _L.ptr(qd), _L.ptr(pn), _L.ptr(qn), int(nsteps),
                                       _L.current_stream_ptr()))
        else:
            flags = self._fp16x2_flag()
            nbytes = int(lib.hmc_leap_frog_workspace_bytes(t, q2.shape[0], flags)) if self.dtype == "float32" else 0
            ws, ws_ptr = _L.aligned_workspace(torch, dev, nbytes) if nbytes else (None, None)
            _L.check(lib.hmc_leap_frog_bigd(dtype, t, q2.shape[0], _L.ptr(pd), _L.ptr(qd), _L.ptr(pn), _L.ptr(qn), int(nsteps), flags,
                                            ws_ptr, nbytes, _L.current_stream_ptr()))
        return pn.double().cpu().numpy().reshape(shape), qn.double().cpu().numpy().reshape(shape)

    def make_movie(self, title_prefix, q0=None, cov0=None, plot_cov=True, qmin=-3, qmax=3):
        """Slide deck of chain-0 trajectories (samplers.py:843-871): presentation, out of scope; the captured
        inputs ``phi_q`` / ``decision_chain`` are produced by the kernel."""
        assert self.sampler_type == "Random"                                         # samplers.py:850
        print("make_movie: rendering is outside the B200 hot-path build; %d trajectories captured in phi_q" %
              len(getattr(self, "phi_q", [])))
        return
