"""ctypes binding of libstellar_rhmc.so (include/stellar_rhmc.h).

This is the whole Python<->CUDA boundary: plain pointers and sizes, no torch types.  The library is built
in-tree by `__graft_entry__.build()` / `python -m hmc_stellar_toy_model_b200.build`; importing the package
without it, or calling into it without a CUDA device, raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SRHMC_LIB") or os.path.join(_HERE, "libstellar_rhmc.so")  # SRHMC_LIB: experimental builds
ABI_VERSION = 3

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_uint8_p = C.POINTER(C.c_uint8)


class SrhmcError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libstellar_rhmc error %d: %s" % (code, message))
        self.code = code


class Config(C.Structure):
    """struct srhmc_config"""

    _fields_ = [
        ("abi_version", C.c_int32),
        ("device", C.c_int32),
        ("precision", C.c_int32),
        ("n_fields", C.c_int32),
        ("num_rows", C.c_int32),
        ("num_cols", C.c_int32),
        ("max_stars", C.c_int32),
        ("patch_radius", C.c_int32),
        ("shared_data", C.c_int32),
        ("fixed_point_mode", C.c_int32),
        ("use_prior", C.c_int32),
        ("use_Vc", C.c_int32),
        ("psf_fwhm_pix", C.c_double),
        ("B_count", C.c_double),
        ("f_lim", C.c_double),
        ("f_low", C.c_double),
        ("g0", C.c_double),
        ("g1", C.c_double),
        ("g2", C.c_double),
        ("g_xx", C.c_double),
        ("g_ff", C.c_double),
        ("alpha", C.c_double),
        ("V_prior_const", C.c_double),
        ("Vc_r_pow", C.c_double),
        ("enable_hessian", C.c_int32),
        ("reserved0", C.c_int32),
    ]


class LsArgs(C.Structure):
    """struct srhmc_ls_args"""

    _fields_ = [
        ("variant", C.c_int32),
        ("niter", C.c_int32),
        ("q0", c_double_p),
        ("nstars", c_int32_p),
        ("dt", c_double_p),
        ("n_dt", C.c_int32),
        ("zero_xy_momentum", C.c_int32),
        ("f_lim", C.c_double),
        ("factor1", C.c_double),
        ("normals", c_double_p),
        ("steps", c_int32_p),
        ("lnu", c_double_p),
        ("background", c_double_p),
        ("q_chain", c_double_p),
        ("E_chain", c_double_p),
        ("dE_chain", c_double_p),
        ("A_chain", c_uint8_p),
        ("q_final", c_double_p),
        ("accept_count", c_double_p),
    ]


class RunArgs(C.Structure):
    """struct srhmc_run_args"""

    _fields_ = [
        ("q0", c_double_p),
        ("nstars", c_int32_p),
        ("niter", C.c_int32),
        ("nsteps", C.c_int32),
        ("dt", C.c_double),
        ("delta", C.c_double),
        ("counter_max", C.c_int32),
        ("f_pos", C.c_int32),
        ("g_ff2", C.c_double),
        ("beta", C.c_double),
        ("g_ff2_schedule", c_double_p),
        ("n_g_ff2", C.c_int32),
        ("beta_schedule", c_double_p),
        ("n_beta", C.c_int32),
        ("normals", c_double_p),
        ("lnu", c_double_p),
        ("seed", C.c_uint64),
        ("chain_stride", C.c_int32),
        ("reserved", C.c_int32),
        ("q_chain", c_double_p),
        ("p_chain", c_double_p),
        ("E_chain", c_double_p),
        ("V_chain", c_double_p),
        ("T_chain", c_double_p),
        ("A_chain", c_uint8_p),
        ("q_final", c_double_p),
        ("accept_rate", c_double_p),
        ("field_id_base", C.c_int32),
        ("field_id_stride", C.c_int32),
        ("field_ids", c_int32_p),
    ]


class BigConfig(C.Structure):
    """struct srhmc_big_config"""

    _fields_ = [(n, C.c_int32) for n in ("abi_version", "device", "rows_global", "cols", "own_lo", "own_hi", "row0",
                                         "nrows", "nrows_halo", "max_stars", "max_ghosts", "patch_radius", "use_prior",
                                         "world_size", "rank")] + \
               [(n, C.c_double) for n in ("psf_fwhm_pix", "B_count", "f_lim", "f_low", "g0", "g1", "g2", "g_xx", "g_ff",
                                          "alpha", "V_prior_const")]


class BigStep(C.Structure):
    """struct srhmc_big_step"""

    _fields_ = [("dt", C.c_double), ("delta", C.c_double), ("g_ff2", C.c_double), ("counter_max", C.c_int32),
                ("f_pos", C.c_int32), ("iteration", C.c_int32), ("fixed_point_mode", C.c_int32), ("seed", C.c_uint64)]


class BigBuffers(C.Structure):
    """struct srhmc_big_buffers_t"""

    _fields_ = [("ghost_send", C.c_void_p), ("ghost_send_doubles", C.c_int64), ("ghost_recv", C.c_void_p),
                ("ghost_recv_doubles", C.c_int64), ("scalars", C.c_void_p), ("global_scalars", C.c_void_p),
                ("n_scalars", C.c_int64), ("counters", C.c_void_p), ("n_counters", C.c_int64)]


# name -> (restype, argtypes); every symbol declared in include/stellar_rhmc.h
SIGNATURES = {
    "srhmc_abi_version": (C.c_int, []),
    "srhmc_last_error": (C.c_char_p, []),
    "srhmc_device_count": (C.c_int, []),
    "srhmc_chain_group_size": (C.c_int, []),
    "srhmc_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "srhmc_destroy": (C.c_int, [C.c_void_p]),
    "srhmc_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "srhmc_synchronize": (C.c_int, [C.c_void_p]),
    "srhmc_last_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "srhmc_launch_count": (C.c_int64, [C.c_void_p]),
    "srhmc_host_alloc": (C.c_void_p, [C.c_uint64]),
    "srhmc_host_free": (C.c_int, [C.c_void_p]),
    "srhmc_set_data": (C.c_int, [C.c_void_p, c_double_p, C.c_int64]),
    "srhmc_gen_model": (C.c_int, [C.c_void_p, c_double_p, c_int32_p, c_double_p]),
    "srhmc_gen_mock_data": (C.c_int, [C.c_void_p, c_double_p, c_int32_p, C.c_uint64, C.c_int64, c_double_p]),
    "srhmc_convergence_stats": (C.c_int, [C.c_int32, c_double_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, c_double_p, c_double_p]),
    "srhmc_find_peaks_descend": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                           c_uint8_p, c_int32_p]),
    "srhmc_run_stats": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, c_double_p, c_double_p]),
    "srhmc_eval": (C.c_int, [C.c_void_p, c_double_p, c_int32_p, C.c_int32, C.c_double, C.c_double,
                             c_double_p, c_double_p, c_double_p, c_double_p]),
    "srhmc_metric": (C.c_int, [C.c_void_p, c_double_p, C.c_int64, C.c_double, c_double_p, c_double_p]),
    "srhmc_kinetic": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_int32_p, C.c_double,
                                c_double_p, c_double_p, c_double_p]),
    "srhmc_kinetic_diag": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_int64, c_double_p]),
    "srhmc_step": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_int32_p, C.c_int32, C.c_double, C.c_double,
                             C.c_int32, C.c_double, C.c_double, c_int32_p]),
    "srhmc_run": (C.c_int, [C.c_void_p, C.POINTER(RunArgs)]),
    "srhmc_run_upload": (C.c_int, [C.c_void_p, C.POINTER(RunArgs)]),
    "srhmc_run_launch": (C.c_int, [C.c_void_p, C.POINTER(RunArgs)]),
    "srhmc_run_download": (C.c_int, [C.c_void_p, C.POINTER(RunArgs)]),
    "srhmc_run_single": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_int32_p, C.c_int32, C.c_double, C.c_double,
                                   C.c_int32, C.c_int32, C.c_double, C.c_double,
                                   c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "srhmc_ls_run": (C.c_int, [C.c_void_p, C.POINTER(LsArgs)]),
    "srhmc_eval_background": (C.c_int, [C.c_void_p, c_double_p, c_int32_p, c_double_p, c_double_p, c_double_p]),
    "srhmc_hessian": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_int32_p, C.c_double, C.c_int32,
                                c_double_p, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
    "srhmc_philox_draws": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int32, c_double_p, c_double_p]),
    "srhmc_philox_draws_ids": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, c_double_p,
                                         c_double_p]),
    "srhmc_plan_chunks": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "srhmc_test_device_math": (C.c_int, [C.c_void_p, C.c_int32, c_double_p, c_double_p, C.c_int32]),
    "srhmc_measure_fma_peak": (C.c_int, [C.c_int32, C.c_int32, c_double_p, C.POINTER(C.c_float)]),
    "srhmc_big_last_error": (C.c_char_p, []),
    "srhmc_big_create": (C.c_int, [C.POINTER(BigConfig), C.POINTER(C.c_void_p)]),
    "srhmc_big_destroy": (C.c_int, [C.c_void_p]),
    "srhmc_big_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "srhmc_big_adopt_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "srhmc_big_synchronize": (C.c_int, [C.c_void_p]),
    "srhmc_big_launch_count": (C.c_int64, [C.c_void_p]),
    "srhmc_big_set_data": (C.c_int, [C.c_void_p, c_double_p]),
    "srhmc_big_set_precision": (C.c_int, [C.c_void_p, C.c_int32]),
    "srhmc_big_mock_data": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_uint64, c_double_p]),
    "srhmc_big_set_stars": (C.c_int, [C.c_void_p, c_double_p, C.POINTER(C.c_int64), C.c_int32]),
    "srhmc_big_get_stars": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_double_p]),
    "srhmc_big_set_momenta": (C.c_int, [C.c_void_p, c_double_p]),
    "srhmc_big_buffers": (C.c_int, [C.c_void_p, C.POINTER(BigBuffers)]),
    "srhmc_big_comm_export": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "srhmc_big_comm_import": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "srhmc_big_set_draws": (C.c_int, [C.c_void_p, c_double_p, c_double_p, C.c_int32]),
    "srhmc_big_alloc_chains": (C.c_int, [C.c_void_p, C.c_int32]),
    "srhmc_big_read_chains": (C.c_int, [C.c_void_p, C.c_int32, c_double_p, c_double_p, c_double_p, c_uint8_p,
                                        C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "srhmc_big_read_scalars": (C.c_int, [C.c_void_p, c_double_p]),
    "srhmc_big_phase": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(BigStep)]),
    "srhmc_big_set_recording": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "srhmc_big_read_samples": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_double_p, c_double_p]),
    "srhmc_big_convergence_stats": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, c_double_p, c_double_p]),
}


def measure_fma_peak(device=0, precision=64):
    """(TFLOP/s, ms) of the register-resident FMA-chain microbenchmark on `device`."""
    lib = load_library()
    tf = C.c_double()
    ms = C.c_float()
    check(lib.srhmc_measure_fma_peak(int(device), int(precision), C.byref(tf), C.byref(ms)))
    return float(tf.value), float(ms.value)

_lib = None


def load_library(path: str | None = None):
    """dlopen the in-tree shared library and attach prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.isfile(path):
        raise ImportError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the RHMC path)" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    got = lib.srhmc_abi_version()
    if got != ABI_VERSION:
        raise ImportError("libstellar_rhmc ABI %d != binding ABI %d" % (got, ABI_VERSION))
    _lib = lib
    return lib


def check(code):
    if code != 0:
        raise SrhmcError(code, load_library().srhmc_last_error().decode("utf-8", "replace"))


def check_big(code):
    if code != 0:
        raise SrhmcError(code, load_library().srhmc_big_last_error().decode("utf-8", "replace"))


def dptr(a):
    return None if a is None else a.ctypes.data_as(c_double_p)


def iptr(a):
    return None if a is None else a.ctypes.data_as(c_int32_p)


def bptr(a):
    return None if a is None else a.ctypes.data_as(c_uint8_p)


def as_f64(a, shape=None):
    out = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        out = out.reshape(shape)
    return out


class PinnedBuffer:
    """A page-locked host array (cudaMallocHost) exposed as a numpy view."""

    def __init__(self, shape, dtype=np.float64):
        lib = load_library()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = lib.srhmc_host_alloc(max(self.nbytes, 8))
        if not self._ptr:
            raise SrhmcError(-2, lib.srhmc_last_error().decode())
        buf = (C.c_byte * max(self.nbytes, 8)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            load_library().srhmc_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
