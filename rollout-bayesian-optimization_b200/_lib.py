"""ctypes binding of csrc/librbo.so (include/rbo.h). Fails loudly when the CUDA library is missing: there is
no CPU fallback on the product path."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RBO_LIB_PATH", os.path.join(_HERE, "csrc", "librbo.so"))  # override = development aid (timer build)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class SolverOpts(C.Structure):
    _fields_ = [("maxit", C.c_int32), ("maxtry", C.c_int32), ("gtol", C.c_double), ("xtol", C.c_double),
                ("pred_tol", C.c_double), ("eta", C.c_double), ("delta0_box", C.c_double), ("delta0_ell", C.c_double),
                ("stol", C.c_double)]


class Summary(C.Structure):
    _fields_ = [("mean", C.c_double), ("std", C.c_double), ("n_traj", C.c_int32), ("n_failed", C.c_int32),
                ("kernel_ms", C.c_double), ("flops", C.c_double), ("flops_executed", C.c_double),
                ("n_evals", C.c_int64), ("gpu_launches", C.c_int32), ("tail_ms", C.c_double)]


class SgaOpts(C.Structure):
    _fields_ = [("optimizer", C.c_int32), ("max_iterations", C.c_int32), ("use_eswavs", C.c_int32), ("project", C.c_int32),
                ("eta", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double)]


# every symbol include/rbo.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "rbo_abi_version": (C.c_int, []),
    "rbo_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "rbo_destroy": (C.c_int, [C.c_void_p]),
    "rbo_last_error": (C.c_char_p, [C.c_void_p]),
    "rbo_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rbo_default_solver_opts": (None, [C.POINTER(SolverOpts)]),
    "rbo_set_solver_opts": (C.c_int, [C.c_void_p, C.POINTER(SolverOpts)]),
    "rbo_set_htol": (C.c_int, [C.c_void_p, C.c_double]),
    "rbo_set_tuning": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "rbo_set_surrogate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, _dp, C.c_double, C.c_int,
                                    _dp, C.c_int, C.c_int, C.c_double]),
    "rbo_condition": (C.c_int, [C.c_void_p, _dp, C.c_double]),
    "rbo_get_surrogate": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), _dp, C.c_int, _dp, _dp]),
    "rbo_set_normals": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "rbo_generate_normals": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "rbo_get_normals": (C.c_int, [C.c_void_p, _dp]),
    "rbo_set_quadrature": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int, C.c_int]),
    "rbo_set_starts": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "rbo_rollout": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_int, C.c_int, _dp, _dp,
                              _dp, _dp, _dp, _ip, _ip, _ip, C.POINTER(Summary)]),
    "rbo_rollout_device": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_int, C.c_int,
                                     C.c_void_p, C.c_void_p, C.POINTER(Summary)]),
    "rbo_rollout_batch": (C.c_int, [C.c_void_p, _dp, C.c_int, _dp, C.c_int, _dp, _dp, C.c_int, C.c_double, C.c_int, _dp, _dp, _dp, _dp, _ip,
                                    C.POINTER(Summary)]),
    "rbo_default_sga_opts": (None, [C.POINTER(SgaOpts)]),
    "rbo_stochastic_solve_batch": (C.c_int, [C.c_void_p, C.POINTER(SgaOpts), _dp, C.c_int, _dp, C.c_int, _dp, _dp, C.c_int, C.c_double, _dp,
                                             _dp, _ip, _ip, _ip, _dp, _dp, _dp, _dp, _dp, C.POINTER(Summary)]),
    "rbo_partial_sums_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "rbo_partial_sums_host": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "rbo_get_results": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _ip, _ip, _ip]),
    "rbo_finalize_sums": (C.c_int, [_dp, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp]),
    "rbo_get_tape": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _dp, _ip, _ip, _ip]),
    "rbo_get_tape_ex": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _dp, _dp]),
    "rbo_sobol_uniform": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp]),
    "rbo_sobol_uint32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_uint32)]),
    "rbo_generate_initial_guesses": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp]),
    "rbo_multistart_base_solve": (C.c_int, [C.c_void_p, _dp, C.c_int, _dp, _dp, _dp, _dp, C.POINTER(Summary)]),
    "rbo_fp64_peak": (C.c_int, [C.c_void_p, _dp]),
    "rbo_tr_step_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _ip]),
    "rbo_num_sms": (C.c_int, [C.c_void_p]),
}

_lib = None


class RboError(RuntimeError):
    pass


def load():
    """Loads librbo.so. Raises (never falls back) if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RboError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def dptr(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and (a.flags["F_CONTIGUOUS"] or a.flags["C_CONTIGUOUS"])
    return a.ctypes.data_as(_dp)


def iptr(a):
    if a is None:
        return None
    assert a.dtype == np.int32
    return a.ctypes.data_as(_ip)


class Handle:
    """Owns one rbo_handle (one CUDA device + stream). Raises RboError with rbo_last_error() on failure."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.rbo_create(C.byref(h), int(device))
        if rc != 0:
            raise RboError(f"rbo_create failed ({rc}): {self.lib.rbo_last_error(None).decode()}")
        self.h = h
        self.device = device

    def check(self, rc):
        if rc != 0:
            raise RboError(f"librbo error {rc}: {self.lib.rbo_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.rbo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
