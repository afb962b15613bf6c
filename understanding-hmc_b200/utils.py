"""Host-side mirror of the reference's ``utils.py`` for the HMC hot path (B200 build).

Same public names as /root/reference/utils.py so that ``from utils import *`` in the case scripts resolves:
``np`` (with the removed aliases ``np.float`` / ``np.int`` restored, case1-script.py:28), ``time``,
``convergence_stats``, ``variogram``, ``acceptance_rate``, ``start_pts``, ``normal_lnL``, the NUTS index helpers
and -- when the optional libraries are installed -- ``plt``, ``mpl``, ``Ellipse``, ``multivariate_normal``,
``norm``, ``chi2`` (utils.py:1-19).  matplotlib is optional (plotting is out of scope, SURVEY section 2).

``convergence_stats`` runs on the GPU (csrc/diag.cu through the C-ABI) -- there is no CPU implementation here.
"""
import os as _os
import time  # noqa: F401  (re-exported, utils.py:3)

import numpy as np

# Python-2-era numpy aliases the drivers use (case1-script.py:28 `dtype=np.float`).
if not hasattr(np, "float"):
    np.float = float
if not hasattr(np, "int"):
    np.int = int

try:  # utils.py:2, 12, 19 -- optional here
    import matplotlib as mpl
    mpl.use("Agg")
    import matplotlib.pyplot as plt
    from matplotlib.patches import Ellipse
    HAVE_MPL = True
except Exception:  # pragma: no cover - image has no matplotlib
    mpl = None
    plt = None
    Ellipse = None
    HAVE_MPL = False

from scipy.stats import multivariate_normal, norm, chi2  # noqa: E402,F401  (utils.py:5-7)

import hmc_b200_lib as _L  # noqa: E402


# ----------------------------------------------------------------------------------------------------------
# Plot helpers (utils.py:21-71) are presentation code outside the hot path (SURVEY section 2): the names stay
# importable for `from utils import *`, the drawing itself is not part of this build.
# ----------------------------------------------------------------------------------------------------------
def cov_ellipse(cov, q=None, nsig=None, **kwargs):
    raise NotImplementedError("cov_ellipse: plotting geometry is outside the B200 hot-path build (SURVEY section 2)")


def plot_cov_ellipse(ax, mus, covs, var_num1, var_num2, MoG_color="Blue", lw=2):
    print("plot_cov_ellipse: plotting is outside the B200 hot-path build (SURVEY section 2); skipped")
    return


# ----------------------------------------------------------------------------------------------------------
# Convergence statistics on the GPU (utils.py:77-179)
# ----------------------------------------------------------------------------------------------------------
class _NeffState(object):
    """Per-dimension state of the sequential truncation rule (vectorised over dimensions)."""

    def __init__(self, D):
        self.rho = np.zeros((0, D))             # rho[k] = autocorrelation at lag k + 1, for the lags received so far
        self.t = 1                              # common loop index of the dimensions still running (utils.py:141)
        self.started = False
        self.done = np.zeros(D, dtype=bool)
        self.t_stop = np.zeros(D, dtype=int)    # number of leading rho terms summed (utils.py:154)
        self.sum_rho = np.zeros(D)

    def close(self, mask, t_stop):
        """Finish the dimensions in ``mask``: sum_rho = max(0, sum(rho[:t_stop])) (utils.py:154-156)."""
        if not np.any(mask):
            return
        t_stop = np.broadcast_to(t_stop, mask.shape)
        csum = np.vstack([np.zeros((1, self.rho.shape[1])), np.cumsum(self.rho, axis=0)])
        idx = np.nonzero(mask)[0]
        s = csum[np.minimum(t_stop[idx], self.rho.shape[0]), idx]
        self.sum_rho[idx] = np.where(s < 0, 0.0, s)
        self.t_stop[idx] = t_stop[idx]
        self.done[idx] = True


def _finish_n_eff(var, V_rows, m, n, state):
    """The sequential truncation rule of utils.py:130-157 applied to the lags received so far, all dimensions at once.

    ``state``: a _NeffState.  Returns True when every dimension is done."""
    st = state
    rho_new = 1. - np.asarray(V_rows, dtype=float).reshape(len(V_rows), -1) / (2 * var)      # utils.py:134-135, 144
    st.rho = np.vstack([st.rho, rho_new])
    have = st.rho.shape[0]
    if not st.started and have >= 2:
        st.started = True
        early = (~st.done) & ((st.rho[0] < 1e-2) | (st.rho[0] < 1e-2))       # Q2: rho_t1 tested twice (utils.py:136)
        st.sum_rho[early] = 0
        st.done |= early
    if not st.started:
        return False
    hi = min(n - 2, have - 1)                                               # the loop needs rho[t + 1] (utils.py:141-152)
    if hi > st.t:
        ts = np.arange(st.t, hi)
        cond = ((ts % 2) == 1)[:, None] & ((st.rho[ts] + st.rho[ts + 1]) < 0)
        hit = cond.any(axis=0) & ~st.done
        st.close(hit, ts[cond.argmax(axis=0)])
        st.t = hi
    if st.t >= n - 2:
        st.close(~st.done, np.full(st.done.shape, st.t))
    return bool(np.all(st.done))


ROW_SHIFT, ROW_COUNT, ROW_LAGS = 3, 4, 5        # layout of the packed statistics buffer [5 + lag_chunk][D]


FFT_MIN_N = 192        # split chains at least this long take the all-lags FFT pass straight away (see _stats_from_partials)


def _stats_from_partials(moments_fn, variogram_fn, n, D, m_local, group=None, lag_chunk=32, device=None, all_lags_fn=None):
    """Rhat / n_eff from per-rank partial sums (utils.py:107-157).

    ``moments_fn(buf)`` fills the float64 buffer ``buf`` [5 + lag_chunk][D]: rows 0..2 = sum_j std_j, sum_j (mean_j - c),
    sum_j (mean_j - c)^2 over the LOCAL split chains, row 3 = the rank's shift c (the first sample of its first chain, so
    that nothing cancels when the chains sit far from zero); it may also fill rows 5.. with the variogram numerators of
    lags 1..lag_chunk (short series: everything comes out of one kernel) and returns how many lag rows it filled.
    ``variogram_fn(lag0, nl, buf)`` fills ``buf`` [lag_chunk][D].  Row 4 carries the local split-chain count.

    When torch.distributed is initialised (and ``group is not False``) the packed buffer is all-gathered -- ONE collective
    and one D2H copy per call for short series, plus one all-reduce per further lag chunk; the only exchange step on the
    whole path (SURVEY 8e).  Ranks are combined on the host: counts and lag sums add up; the between-chain sum of squares
    uses the pairwise update  M2 = sum_r M2_r + sum_r m_r (mean_r - mean)^2  (the two-round form of SURVEY 8e without a
    second round).  Everything after that is O(lags * D) host arithmetic.

    ``all_lags_fn(buf)`` (optional) fills ``buf`` [n - 1][D] with the numerators of EVERY lag in one pass over the samples
    (csrc/diag_fft.cu: one FFT per chain and dimension, a fixed cost per chain).  Long split chains (n >= FFT_MIN_N) use it
    straight away; shorter ones try one windowed chunk first (a well-mixed chain ends within it) and switch when the
    truncation rule has not fired.  Sharded runs all-reduce that one buffer."""
    import torch
    import torch.distributed as dist
    distributed = dist.is_available() and dist.is_initialized() and (group is not False)
    grp = None if group in (None, False) else group
    buf = _scratch("stats", (ROW_LAGS + lag_chunk, D), torch.float64, device)
    nfilled = moments_fn(buf)
    buf[ROW_COUNT, 0] = float(m_local)
    if distributed:
        world = dist.get_world_size(group=grp)
        allbuf = _scratch("stats_all", (world, ROW_LAGS + lag_chunk, D), torch.float64, device)
        dist.all_gather_into_tensor(allbuf.view(world * (ROW_LAGS + lag_chunk), D), buf, group=grp)
        host = _host(allbuf)
    else:
        host = _host(buf)[None]
    m_r = np.rint(host[:, ROW_COUNT, 0])                            # split chains per rank
    m = int(m_r.sum())
    W = host[:, 0].sum(axis=0) / m                                  # utils.py:112 (mean of std, Q1)
    mean_r = host[:, ROW_SHIFT] + host[:, 1] / m_r[:, None]         # per-rank mean of the chain means
    M2_r = host[:, 2] - host[:, 1] ** 2 / m_r[:, None]              # per-rank sum_j (mean_j - mean_r)^2
    mean_all = (m_r[:, None] * mean_r).sum(axis=0) / m              # utils.py:119
    M2 = M2_r.sum(axis=0) + (m_r[:, None] * (mean_r - mean_all) ** 2).sum(axis=0)
    B = M2 * n / float(m - 1)                                       # utils.py:120
    var = W * (n - 1) / float(n) + B / float(n)                     # utils.py:123
    R = np.sqrt(var / W)                                            # utils.py:126

    state = _NeffState(D)
    lag0 = 1
    max_lag = n - 1
    vbuf = None
    while lag0 <= max_lag:
        nl = min(lag_chunk, max_lag - lag0 + 1)
        if lag0 == 1 and nfilled:
            rows = host[:, ROW_LAGS:ROW_LAGS + nl].sum(axis=0)
        elif all_lags_fn is not None and (lag0 > 1 or n >= FFT_MIN_N):
            abuf = _scratch("all_lags", (max_lag, D), torch.float64, device)
            all_lags_fn(abuf)
            if distributed:
                dist.all_reduce(abuf, group=grp)
            rows = _host(abuf[lag0 - 1:])
            nl = max_lag - lag0 + 1
        else:
            if vbuf is None:
                vbuf = _scratch("lags", (lag_chunk, D), torch.float64, device)
            variogram_fn(lag0, nl, vbuf)
            if distributed:
                dist.all_reduce(vbuf, group=grp)
            rows = _host(vbuf[:nl])
        V_rows = [rows[k] / float(m * (n - (lag0 + k))) for k in range(nl)]      # utils.py:177
        if _finish_n_eff(var, V_rows, m, n, state):
            break
        lag0 += nl
    state.close(~state.done, np.full(D, state.t))        # chains too short to ever start (n < 3): use what exists
    n_eff = m * n / (1 + 2 * state.sum_rho)                                             # utils.py:157
    return R, n_eff


_SCRATCH = {}
D2H_BYTES = [0]          # bytes read back from the device by the diagnostics / counters (bench.py reports them per step)


def _host(t):
    """Device tensor -> numpy (one D2H copy, counted)."""
    D2H_BYTES[0] += t.numel() * t.element_size()
    return t.cpu().numpy()


def _scratch(name, shape, dtype, device=None):
    """Per-device scratch tensors reused across calls (no allocation / fill on the diagnostics path)."""
    import torch
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    key = (name, str(device), tuple(shape), dtype)
    t = _SCRATCH.get(key)
    if t is None:
        t = torch.zeros(shape, dtype=dtype, device=device)
        _SCRATCH[key] = t
    return t


def _device_stats(x, n, group=None, lag_chunk=32):
    """x: CUDA tensor (Nchain_local, >=2n, D), float32/float64, last dim contiguous.  Returns (R, n_eff) numpy.
    The per-device partial sums come from csrc/diag.cu through the C-ABI."""
    import torch
    lib = _L.load()
    assert x.is_cuda and x.dim() == 3 and x.stride(2) == 1 and x.stride(1) == x.shape[2]
    Nchain, _, D = x.shape
    dtype = _L.HMC_F32 if x.dtype == torch.float32 else _L.HMC_F64
    stride_chain = x.stride(0)

    def moments_fn(buf):
        if 2 <= n <= 32 and lag_chunk == 32:    # short series: moments and every lag in one pass over the samples
            _L.check(lib.hmc_diag_short_series(dtype, _L.ptr(x), Nchain, n, D, stride_chain, max(1, n - 1), _L.ptr(buf),
                                               _L.ptr(buf[ROW_LAGS:]), _L.current_stream_ptr()))
            return max(1, n - 1)
        _L.check(lib.hmc_diag_moments(dtype, _L.ptr(x), Nchain, n, D, stride_chain, _L.ptr(buf), _L.current_stream_ptr()))
        return 0

    def variogram_fn(lag0, nl, buf):
        _L.check(lib.hmc_diag_variogram(dtype, _L.ptr(x), Nchain, n, D, stride_chain, lag0, nl, _L.ptr(buf),
                                        _L.current_stream_ptr()))

    all_lags_fn = None
    if (x.dtype == torch.float32 and 32 < n <= 512 and D % 4 == 0 and stride_chain % 4 == 0 and x.data_ptr() % 16 == 0
            and _os.environ.get("HMC_B200_DIAG_NO_FFT") is None):
        def all_lags_fn(buf):
            ws = _scratch("fft_ws", (int(lib.hmc_diag_variogram_all_workspace_bytes(n, D)) // 8,), torch.float64, x.device)
            _L.check(lib.hmc_diag_variogram_all(dtype, _L.ptr(x), Nchain, n, D, stride_chain, n - 1, _L.ptr(buf), _L.ptr(ws),
                                                ws.numel() * 8, _L.current_stream_ptr()))

    return _stats_from_partials(moments_fn, variogram_fn, n, D, 2 * Nchain, group=group, lag_chunk=lag_chunk, device=x.device,
                                all_lags_fn=all_lags_fn)


def convergence_stats(q_chain, thin_rate=5, warm_up_num=0, group=None):
    """Split-chain Rhat and variogram ESS per dimension (utils.py:77-159), computed on the GPU.

    ``q_chain``: (Nchain, Niter, D) numpy array or CUDA torch tensor.  Reference quirks kept: W is a mean of
    standard deviations (Q1), ``rho_t1`` is tested twice (Q2)."""
    import torch
    if isinstance(q_chain, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(q_chain)).cuda()
    else:
        x = q_chain
    Nchain, Niter, D = x.shape
    assert Nchain > 1                                               # utils.py:85
    x = x[:, warm_up_num:, :][:, ::thin_rate, :]                    # utils.py:91-94
    L_chain = x.shape[1]
    if (L_chain % 2) != 0:                                          # utils.py:96-99
        x = x[:, :L_chain - 1]
    n = L_chain // 2                                                # utils.py:102
    if not (x.stride(2) == 1 and x.stride(1) == D):
        x = x.contiguous()
    return _device_stats(x, n, group=group)


def variogram(chains, var_num, t_lag):
    """V_t of BDA3 (11.7) for one variable and one lag (utils.py:161-179), on the GPU."""
    import torch
    lib = _L.load()
    m = len(chains)
    n = chains[0].shape[0]
    x = torch.from_numpy(np.ascontiguousarray(np.stack([np.asarray(c)[:, var_num] for c in chains])[:, :, None])).cuda()
    # each "chain" of length n is treated as one split chain: use n_half = n with a dummy second half of stride 0
    x2 = torch.cat([x, x], dim=1).contiguous()                      # halves [0,n) and [n,2n) are the same series
    out = torch.empty((1, 1), dtype=torch.float64, device=x.device)
    _L.check(lib.hmc_diag_variogram(_L.HMC_F64, _L.ptr(x2), m, n, 1, 2 * n, t_lag, 1, _L.ptr(out),
                                    _L.current_stream_ptr()))
    return float(out.item()) / 2.0 / float(m * (n - t_lag))


def acceptance_rate(decision_chain, start=None, end=None):
    """utils.py:183-200 is never called by the samplers or the drivers (SURVEY section 2); the samplers report
    ``accept_R`` / ``accept_R_warm_up`` from the device counters instead."""
    raise NotImplementedError("acceptance_rate is not part of the B200 hot-path build; use HMC_sampler.accept_R")


def start_pts_entry(D):
    """The library entry point ``start_pts(device=...)`` calls for dimension D: ``hmc_start_pts`` (one warp per chain) up to
    D = 4096, ``hmc_start_pts_bigd`` (the large-D tensor-core GEMM, float32, D <= 8192) above."""
    return "hmc_start_pts" if D <= 4096 else "hmc_start_pts_bigd"


def start_pts(q0, cov0, size, device=None, seed=0, chain_id0=0, dtype="float32"):
    """Starting points ~ N(q0, cov0) (utils.py:204-209).

    Default (``device=None``): the reference's own call on the host, consuming the global ``np.random`` stream, so the
    drivers reproduce their start points.  ``device="cuda"``: generated on the GPU (Philox keyed by (seed, global chain id):
    independent of how chains are sharded) and returned as a CUDA tensor that ``HMC_sampler.gen_sample`` takes as is -- no
    host draws, no H2D copy of Nchain x D values.  Up to D = 4096 ``hmc_start_pts`` (csrc/summary.cu) makes them; above, up to
    D = 8192 and in float32 only, ``hmc_start_pts_bigd`` (csrc/bigd_primitives.cu) from the same normals (start_pts_entry)."""
    if device is None:
        return np.random.multivariate_normal(q0, cov0, size=size)
    import torch
    lib = _L.load()
    dev = torch.device(device)
    q0 = np.asarray(q0, dtype=float)
    cov0 = np.asarray(cov0, dtype=float)
    D = q0.shape[0]
    q0_d = torch.from_numpy(np.ascontiguousarray(q0)).to(dev)
    if np.array_equal(cov0, np.diag(np.diag(cov0))):
        fac, Lc_d = torch.from_numpy(np.sqrt(np.diag(cov0)).copy()).to(dev), None
    else:
        Lc_d, fac = torch.from_numpy(np.ascontiguousarray(np.linalg.cholesky(cov0))).to(dev), None
    tdt = torch.float32 if dtype == "float32" else torch.float64
    out = torch.empty((int(size), D), dtype=tdt, device=dev)
    dt_id = _L.HMC_F32 if tdt == torch.float32 else _L.HMC_F64
    with torch.cuda.device(dev):
        if start_pts_entry(D) == "hmc_start_pts":
            _L.check(lib.hmc_start_pts(dt_id, int(seed), int(chain_id0), int(size), D, _L.ptr(q0_d), _L.ptr(Lc_d), _L.ptr(fac),
                                       _L.ptr(out), _L.current_stream_ptr()))
        else:                                      # (the workspace holds the GEMM operands: dense cov0 in float32 only)
            nbytes = int(lib.hmc_start_pts_workspace_bytes(int(size), D)) if Lc_d is not None and tdt == torch.float32 else 0
            ws, ws_ptr = _L.aligned_workspace(torch, dev, nbytes) if nbytes else (None, None)
            _L.check(lib.hmc_start_pts_bigd(dt_id, int(seed), int(chain_id0), int(size), D, _L.ptr(q0_d), _L.ptr(Lc_d), _L.ptr(fac),
                                            _L.ptr(out), ws_ptr, nbytes, _L.current_stream_ptr()))
    return out


# ----------------------------------------------------------------------------------------------------------
# Sample summaries on the GPU: the inputs of sampler.plot_samples (samplers.py:84-113, 160-186, 209-250)
# ----------------------------------------------------------------------------------------------------------
def _series_args(x):
    """(ptr, dtype, Nchain, nsamp, stride_sample, stride_chain) of a 2-D view [chain][sample] of a CUDA tensor."""
    import torch
    assert x.is_cuda and x.dim() == 2 and x.dtype in (torch.float32, torch.float64)
    return _L.ptr(x), (_L.HMC_F32 if x.dtype == torch.float32 else _L.HMC_F64), x.shape[0], x.shape[1], x.stride(1), x.stride(0)


def _reduce(t, group):
    import torch.distributed as dist
    if group is not False and dist.is_available() and dist.is_initialized():
        dist.all_reduce(t, group=None if group is None else group)
    return t


def device_order_statistic(x, ks, group=False):
    """The ks-th smallest values (0-based ranks over all elements, all ranks of ``group``) of the 2-D CUDA view ``x``
    [chain][sample], by radix select on the device (hmc_summary_select: one HBM pass per 11-bit digit)."""
    import torch
    lib = _L.load()
    ptr, dt, nc, ns, ss, sc = _series_args(x)
    bits = 32 if dt == _L.HMC_F32 else 64
    hist = torch.empty((2048,), dtype=torch.int64, device=x.device)
    out = []
    for k in ks:
        prefix, done, rem = 0, 0, int(k)
        while done < bits:
            nb = min(11, bits - done)
            sh = bits - done - nb
            _L.check(lib.hmc_summary_select(dt, ptr, nc, ns, ss, sc, prefix, (bits - done) if done else 64, sh, nb, _L.ptr(hist),
                                            _L.current_stream_ptr()))
            h = _reduce(hist, group).cpu().numpy()[:1 << nb]
            cum = np.cumsum(h)
            d = int(np.searchsorted(cum, rem, side="right"))
            if d > 0:
                rem -= int(cum[d - 1])
            prefix = (prefix << nb) | d
            done += nb
        if bits == 32:
            u = np.uint32(prefix)
            u = np.uint32(~u) if not (u & np.uint32(0x80000000)) else np.uint32(u & np.uint32(0x7fffffff))
            out.append(float(u.view(np.float32)))
        else:
            u = np.uint64(prefix)
            u = np.uint64(~u) if not (u & np.uint64(0x8000000000000000)) else np.uint64(u & np.uint64(0x7fffffffffffffff))
            out.append(float(u.view(np.float64)))
    return out


def device_percentile(x, qs, n_total=None, group=False):
    """np.percentile(x.flatten(), qs) (linear interpolation between order statistics) without leaving the device."""
    N = int(n_total if n_total is not None else x.shape[0] * x.shape[1])
    pos = [q / 100.0 * (N - 1) for q in qs]
    ranks = sorted({int(np.floor(p)) for p in pos} | {min(int(np.floor(p)) + 1, N - 1) for p in pos})
    vals = dict(zip(ranks, device_order_statistic(x, ranks, group=group)))
    out = []
    for p in pos:
        lo = int(np.floor(p))
        hi = min(lo + 1, N - 1)
        f = p - lo
        out.append(vals[lo] + (vals[hi] - vals[lo]) * f)
    return np.asarray(out)


def device_histogram(x, edges, shift=0.0, group=False):
    """np.histogram(x.flatten() - shift, bins=edges)[0] on the device; also returns (#below, #above)."""
    import torch
    lib = _L.load()
    ptr, dt, nc, ns, ss, sc = _series_args(x)
    edges = np.ascontiguousarray(edges, dtype=float)
    nb = edges.shape[0] - 1
    e_d = torch.from_numpy(edges).to(x.device)
    cnt = torch.empty((nb + 2,), dtype=torch.int64, device=x.device)
    _L.check(lib.hmc_summary_hist(dt, ptr, nc, ns, ss, sc, float(shift), _L.ptr(e_d), nb, _L.ptr(cnt), _L.current_stream_ptr()))
    c = _reduce(cnt, group).cpu().numpy()
    return c[:nb].copy(), int(c[nb]), int(c[nb + 1])


def device_moments(x3, group=False, count=None):
    """Per-dimension mean and (population) variance over all chains and samples of a CUDA tensor [chain][sample][D]
    (np.mean / np.std(...)**2 of samplers.py:209-216, 244-250)."""
    import torch
    lib = _L.load()
    assert x3.is_cuda and x3.dim() == 3 and x3.stride(2) == 1
    nc, ns, D = x3.shape
    dt = _L.HMC_F32 if x3.dtype == torch.float32 else _L.HMC_F64
    out = torch.empty((2, D), dtype=torch.float64, device=x3.device)
    _L.check(lib.hmc_summary_moments(dt, _L.ptr(x3), nc, ns, D, x3.stride(1), x3.stride(0), _L.ptr(out), _L.current_stream_ptr()))
    n = torch.tensor([float(nc * ns)], dtype=torch.float64, device=x3.device)
    o = _reduce(out, group).cpu().numpy()
    N = float(_reduce(n, group).item())
    mean = o[0] / N
    return mean, o[1] / N - mean ** 2


def normal_lnL(q, q0, cov0):
    """Multivariate-normal log-density (utils.py:213-218)."""
    return multivariate_normal.logpdf(q, mean=q0, cov=cov0)


# ----------------------------------------------------------------------------------------------------------
# NUTS index helpers (utils.py:222-311, 367-385) in closed form; the CUDA kernel uses the same formulas.
# ----------------------------------------------------------------------------------------------------------
def find_next(table):
    for i, e in enumerate(table):
        if e == -1:
            return i


def retrieve_save_index(table, l):
    for i, m in enumerate(table):
        if m == l:
            return i


def power_of_two(r):
    assert type(r) == int
    return (r & (r - 1)) == 0


def power_of_two_fast(r):
    r = int(r)
    return (r & (r - 1)) == 0


def _tz(m):
    m = int(m)
    return (m & -m).bit_length() - 1


def check_points(m):
    """Points against which even point m is U-turn checked: m - 2^j + 1 for j = tz(m) .. 1 (utils.py:246-283)."""
    assert (m % 2) == 0
    return np.asarray([int(m) - (1 << j) + 1 for j in range(_tz(m), 0, -1)])


def release(m, l):
    """True if check point l is no longer needed after the check at m (utils.py:286-304)."""
    assert (l != 1) and (m % 2) == 0
    return release_fast(m, l)


def release_fast(m, l):
    m, l = int(m), int(l)
    return (l > 1) and (l != m - (1 << _tz(m)) + 1)


def rvs(dim=3):
    """Haar-distributed random rotation matrix (same role as utils.py:424-441; QR of a Gaussian matrix with the
    sign convention fixed, determinant forced to +1)."""
    A = np.random.normal(size=(dim, dim))
    Q, Rm = np.linalg.qr(A)
    Q = Q * np.sign(np.diag(Rm))
    if np.linalg.det(Q) < 0:
        Q[:, 0] = -Q[:, 0]
    return Q
