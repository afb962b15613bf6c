"""ctypes binding of libhmc_b200.so (C-ABI declared in include/hmc_b200.h).

There is no CPU fallback: if the CUDA library is missing, importing a sampler that needs it raises.
torch is used for device memory and streams only (tensors' ``data_ptr()`` are the plain pointers of the ABI).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HMC_B200_LIB") or os.path.join(_HERE, "libhmc_b200.so")      # (HMC_B200_LIB: a profiling / variant build)

HMC_F32, HMC_F64 = 0, 1
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_FAST, KERNEL_TC, KERNEL_BIGD = 0, 1, 2, 3, 4
KERNELS = {"auto": KERNEL_AUTO, "generic": KERNEL_GENERIC, "fast": KERNEL_FAST, "tc": KERNEL_TC, "bigd": KERNEL_BIGD}
FLAG_UNIFORM_DT, FLAG_TC_FP16X2 = 1, 2
HMC_OK, HMC_E_BADARG, HMC_E_UNSUPPORTED, HMC_E_CUDA, HMC_E_DMAX = 0, 1, 2, 3, 4

EXPORTS = ["hmc_random_run", "hmc_nuts_run", "hmc_diag_moments", "hmc_diag_variogram", "hmc_diag_short_series", "hmc_philox_draws",
           "hmc_ffma_peak", "hmc_version", "hmc_last_error_string", "hmc_start_pts", "hmc_summary_moments", "hmc_summary_hist",
           "hmc_summary_select", "hmc_random_workspace_bytes", "hmc_diag_variogram_all", "hmc_diag_variogram_all_workspace_bytes", "hmc_leap_frog",
           "hmc_nuts_workspace_bytes", "hmc_start_pts_workspace_bytes", "hmc_start_pts_bigd", "hmc_leap_frog_workspace_bytes",
           "hmc_leap_frog_bigd"]


class Target(C.Structure):
    _fields_ = [("D", C.c_int32), ("D_pad", C.c_int32), ("Ft", C.c_void_p), ("Pt", C.c_void_p),
                ("Mit", C.c_void_p), ("Lct", C.c_void_p), ("mu", C.c_void_p), ("dt", C.c_void_p),
                ("v_const", C.c_double)]


class RandomArgs(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("kernel", C.c_int32), ("Nchain", C.c_int32), ("flags", C.c_int32),
                ("chain_id0", C.c_int64), ("Niter", C.c_int32), ("iter_begin", C.c_int32), ("iter_end", C.c_int32),
                ("warm_up_num", C.c_int32), ("thin_rate", C.c_int32), ("L_low", C.c_int32), ("L_high", C.c_int32),
                ("N_save_chain0", C.c_int32), ("seed", C.c_uint64), ("target", Target), ("q_start", C.c_void_p),
                ("p_tape", C.c_void_p), ("L_tape", C.c_void_p), ("u_tape", C.c_void_p), ("q_chain", C.c_void_p),
                ("E_chain", C.c_void_p), ("dE_chain", C.c_void_p), ("state_q", C.c_void_p), ("state_g", C.c_void_p),
                ("state_eprev", C.c_void_p), ("counters", C.c_void_p), ("phi_q", C.c_void_p), ("phi_len", C.c_void_p),
                ("decision_chain", C.c_void_p), ("store_ring", C.c_int32), ("reserved0", C.c_int32),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64)]


class NutsArgs(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("kernel", C.c_int32), ("Nchain", C.c_int32), ("d_max", C.c_int32),
                ("chain_id0", C.c_int64), ("Niter", C.c_int32), ("iter_begin", C.c_int32), ("iter_end", C.c_int32),
                ("warm_up_num", C.c_int32), ("thin_rate", C.c_int32), ("on_dmax", C.c_int32), ("seed", C.c_uint64),
                ("target", Target), ("q_start", C.c_void_p), ("p_tape", C.c_void_p), ("dir_tape", C.c_void_p),
                ("u_tape", C.c_void_p), ("tape_dir_stride", C.c_int32), ("tape_u_stride", C.c_int32),
                ("q_chain", C.c_void_p), ("E_chain", C.c_void_p), ("dE_chain", C.c_void_p), ("state_q", C.c_void_p),
                ("state_eprev", C.c_void_p), ("scratch", C.c_void_p), ("counters", C.c_void_p), ("status", C.c_void_p),
                ("n_leapfrog", C.c_void_p), ("flags", C.c_int32), ("reserved0", C.c_int32), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_int64)]


_lib = None


def load():
    """Load the CUDA library or fail loudly (the product path has no CPU implementation)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError("CUDA extension %s is missing: build it with `python -c \"import __graft_entry__ as g; "
                           "g.build()\"` (or `make -C understanding-hmc_b200/csrc`). There is no CPU fallback."
                           % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.hmc_random_run.argtypes = [C.POINTER(RandomArgs), C.c_void_p]
    lib.hmc_random_run.restype = C.c_int
    lib.hmc_random_workspace_bytes.argtypes = [C.POINTER(RandomArgs)]
    lib.hmc_random_workspace_bytes.restype = C.c_int64
    lib.hmc_nuts_run.argtypes = [C.POINTER(NutsArgs), C.c_void_p]
    lib.hmc_nuts_run.restype = C.c_int
    lib.hmc_nuts_workspace_bytes.argtypes = [C.POINTER(NutsArgs)]
    lib.hmc_nuts_workspace_bytes.restype = C.c_int64
    lib.hmc_diag_moments.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_void_p,
                                     C.c_void_p]
    lib.hmc_diag_moments.restype = C.c_int
    lib.hmc_diag_short_series.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmc_diag_short_series.restype = C.c_int
    lib.hmc_diag_variogram.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32,
                                       C.c_int32, C.c_void_p, C.c_void_p]
    lib.hmc_diag_variogram.restype = C.c_int
    lib.hmc_diag_variogram_all.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.hmc_diag_variogram_all.restype = C.c_int
    lib.hmc_diag_variogram_all_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
    lib.hmc_diag_variogram_all_workspace_bytes.restype = C.c_int64
    lib.hmc_leap_frog.argtypes = [C.c_int32, C.POINTER(Target), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_void_p]
    lib.hmc_leap_frog.restype = C.c_int
    lib.hmc_leap_frog_workspace_bytes.argtypes = [C.POINTER(Target), C.c_int64, C.c_int32]
    lib.hmc_leap_frog_workspace_bytes.restype = C.c_int64
    lib.hmc_leap_frog_bigd.argtypes = [C.c_int32, C.POINTER(Target), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.hmc_leap_frog_bigd.restype = C.c_int
    lib.hmc_philox_draws.argtypes = [C.c_uint64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hmc_philox_draws.restype = C.c_int
    lib.hmc_start_pts.argtypes = [C.c_int32, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
    lib.hmc_start_pts.restype = C.c_int
    lib.hmc_start_pts_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
    lib.hmc_start_pts_workspace_bytes.restype = C.c_int64
    lib.hmc_start_pts_bigd.argtypes = [C.c_int32, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.hmc_start_pts_bigd.restype = C.c_int
    lib.hmc_summary_moments.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int64,
                                        C.c_void_p, C.c_void_p]
    lib.hmc_summary_moments.restype = C.c_int
    lib.hmc_summary_hist.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_double,
                                     C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    lib.hmc_summary_hist.restype = C.c_int
    lib.hmc_summary_select.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_uint64,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.hmc_summary_select.restype = C.c_int
    lib.hmc_ffma_peak.argtypes = [C.POINTER(C.c_double), C.c_int32, C.c_void_p]
    lib.hmc_ffma_peak.restype = C.c_int
    lib.hmc_version.argtypes = []
    lib.hmc_version.restype = C.c_int
    lib.hmc_last_error_string.argtypes = []
    lib.hmc_last_error_string.restype = C.c_char_p
    _lib = lib
    return lib


class HMCError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libhmc_b200 error %d: %s" % (code, msg))
        self.code = code


def check(rc):
    if rc != HMC_OK:
        msg = load().hmc_last_error_string()
        raise HMCError(rc, msg.decode() if msg else "")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def aligned_workspace(torch, dev, nbytes):
    """A new device workspace of nbytes, 1024-byte aligned (as the large-D entry points want it): (tensor that owns it, address)."""
    buf = torch.empty((nbytes + 1024,), dtype=torch.uint8, device=dev)
    return buf, (buf.data_ptr() + 1023) // 1024 * 1024


def current_stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
