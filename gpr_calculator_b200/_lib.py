"""ctypes binding of libgpr_b200.so (C ABI declared in include/gpr_b200.h).

There is no CPU fallback: if the library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GPRB_LIB: another build of the same library (kernel A/B experiments, tools/build_variant.sh); the default is the in-tree build
LIB_PATH = os.environ.get("GPRB_LIB") or os.path.join(_HERE, "libgpr_b200.so")

c_int, c_ll, c_dbl, c_vp = ctypes.c_int, ctypes.c_longlong, ctypes.c_double, ctypes.c_void_p
c_int_p = ctypes.POINTER(ctypes.c_int)

RBF, DOT = 0, 1
FF_FULL, FF_SYMMETRIC, FF_DIAG, FF_UPPER = 0, 1, 2, 3
MAX_DST = 8          # GPRB_MAX_DST: matrices one gprb_k*_multi call stores into
OK, ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_LINALG = 0, 1, 2, 3, 4

# name -> (restype, argtypes); every symbol declared in include/gpr_b200.h
SIGNATURES = {
    "gprb_version": (c_int, []),
    "gprb_last_error": (ctypes.c_char_p, []),
    "gprb_launch_count": (c_ll, []),
    "gprb_device_info": (c_int, [c_int_p, c_int_p, c_int_p]),
    "gprb_pack_create": (c_int, [ctypes.POINTER(c_vp), c_int, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_dbl, c_vp]),
    "gprb_pack_destroy": (None, [c_vp]),
    "gprb_pack_info": (c_int, [c_vp, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p]),
    "gprb_pack_pair_count": (c_ll, [c_vp, c_int, c_int, c_vp]),
    "gprb_atom_plan_host": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gprb_atom_plan_cost": (c_int, [c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "gprb_kff": (c_int, [c_int, c_vp, c_vp, c_dbl, c_dbl, c_dbl, c_int, c_dbl, c_int, c_int, c_int,
                         c_vp, c_ll, c_vp, c_ll, c_vp]),
    "gprb_kef": (c_int, [c_int, c_vp, c_vp, c_dbl, c_dbl, c_dbl, c_int, c_int,
                         c_vp, c_ll, c_vp, c_ll, c_vp, c_ll, c_vp, c_ll, c_vp]),
    "gprb_kff_multi": (c_int, [c_int, c_vp, c_vp, c_dbl, c_dbl, c_dbl, c_int, c_dbl, c_int, c_int, c_int,
                               c_int, ctypes.POINTER(c_vp), c_ll, c_vp, c_ll, c_vp]),
    "gprb_kfe_multi": (c_int, [c_int, c_vp, c_vp, c_dbl, c_dbl, c_dbl, c_int, c_int,
                               c_int, ctypes.POINTER(c_vp), c_ll, c_vp, c_ll, c_vp]),
    "gprb_peer_alloc": (c_int, [ctypes.POINTER(c_vp), ctypes.c_ulonglong]),
    "gprb_peer_free": (c_int, [c_vp]),
    "gprb_peer_export": (c_int, [c_vp, ctypes.c_char_p]),
    "gprb_peer_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "gprb_peer_close": (c_int, [c_vp]),
    "gprb_kee": (c_int, [c_int, c_vp, c_vp, c_dbl, c_dbl, c_dbl, c_int, c_int, c_vp, c_ll, c_vp, c_ll, c_vp]),
    "gprb_kee_diag": (c_int, [c_int, c_vp, c_dbl, c_dbl, c_dbl, c_vp, c_vp]),
    "gprb_add_noise": (c_int, [c_vp, c_ll, c_int, c_int, c_dbl, c_dbl, c_vp]),
    "gprb_chol_factor": (c_int, [c_vp, c_ll, c_int, c_vp]),
    "gprb_chol_inverse_rows": (c_int, [c_vp, c_ll, c_int, c_int, c_int, c_int, c_vp, c_ll, c_vp]),
    "gprb_symmetrize": (c_int, [c_vp, c_ll, c_int, c_vp]),
    "gprb_transpose_copy": (c_int, [c_vp, c_ll, c_vp, c_ll, c_int, c_int, c_vp]),
    "gprb_fp64_dmma_peak": (c_int, [c_vp, c_vp]),
    "gprb_lml_eval": (c_int, [c_vp, c_ll, c_int, c_int, c_vp, c_dbl, c_dbl, c_vp, c_ll, c_int, c_vp, c_int, c_int, c_int, c_int,
                             c_vp, c_vp, c_ll, c_vp, c_vp]),
    "gprb_chol_panel": (c_int, [c_vp, c_ll, c_int, c_int, c_int, c_vp, c_vp]),
    "gprb_chol_trailing": (c_int, [c_vp, c_ll, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "gprb_lml_eval_work": (c_ll, [c_int, c_int, c_int, c_int]),
    "gprb_predict": (c_int, [c_int, c_int, c_vp, c_ll, c_vp, c_vp, c_ll, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gprb_predict_chol": (c_int, [c_int, c_int, c_vp, c_ll, c_vp, c_vp, c_ll, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gprb_predict_cov": (c_int, [c_int, c_int, c_vp, c_ll, c_vp, c_ll, c_vp, c_ll, c_vp, c_vp]),
    "gprb_cur_scores": (c_int, [c_vp, c_ll, c_int, c_dbl, c_vp, c_vp, c_int_p, c_vp]),
    "gprb_so3_neighbors": (c_int, [c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_dbl, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gprb_so3_radial": (c_int, [c_int, c_vp, c_int, c_int, c_int, c_dbl, c_dbl, c_vp, c_vp, c_vp, c_vp]),
    "gprb_so3_power": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_dbl, c_dbl, c_vp,
                               c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
}


class GprB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libgpr_b200 error %d: %s" % (code, msg))
        self.code = code


class NotPositiveDefinite(GprB200Error):
    pass


_lib = None


def load():
    """Load the shared library (raises if it has not been built: no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C gpr_calculator_b200/csrc`. gpr_calculator_b200 has no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code):
    if code != OK:
        msg = load().gprb_last_error().decode("utf-8", "replace")
        if code == ERR_LINALG:
            raise NotPositiveDefinite(code, msg)
        raise GprB200Error(code, msg)


# Optional per-call device timing (bench.py): set PROFILE to a list and every call() appends
# (name, start_event, end_event, host_seconds_inside_the_call), CUDA events recorded on the current torch
# stream around the call.
PROFILE = None


def call(name, *args):
    if PROFILE is None:
        check(getattr(load(), name)(*args))
        return
    import time
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    check(getattr(load(), name)(*args))
    t1 = time.perf_counter()
    e1.record()
    PROFILE.append((name, e0, e1, t1 - t0))
