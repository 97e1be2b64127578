"""ctypes loader for libfpsb200.so (the C ABI declared in include/fpsb.h).

There is NO fallback: if the shared library is missing, or no CUDA device is visible when a
handle is created, the call raises.  This module never imports anything from oracle/.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("FPSB200_LIB", os.path.join(_HERE, "libfpsb200.so"))

FPSB_HOST, FPSB_DEVICE = 0, 1

ERRORS = {0: "FPSB_OK", -1: "FPSB_EINVAL", -2: "FPSB_ECUDA", -3: "FPSB_ESTATE", -4: "FPSB_ENOMEM",
          -5: "FPSB_ENCCL"}


class KrylovStats(C.Structure):
    """fpsb_krylov_stats — mirrors Krylov.jl's stats fields read by the reference."""
    _fields_ = [("niter", C.c_int64), ("solved", C.c_int32), ("inconsistent", C.c_int32),
                ("status", C.c_int32), ("pad_", C.c_int32), ("rnorm", C.c_double),
                ("arnorm", C.c_double), ("anorm", C.c_double), ("acond", C.c_double),
                ("xnorm", C.c_double)]

    def as_dict(self):
        return dict(niter=int(self.niter), solved=bool(self.solved),
                    inconsistent=bool(self.inconsistent), status=int(self.status),
                    rnorm=self.rnorm, arnorm=self.arnorm, anorm=self.anorm, acond=self.acond,
                    xnorm=self.xnorm)


class IterOpts(C.Structure):
    _fields_ = [("ls_atol", C.c_double), ("ls_rtol", C.c_double), ("ls_itmax", C.c_int64),
                ("ln_atol", C.c_double), ("ln_rtol", C.c_double), ("ln_btol", C.c_double),
                ("ln_conlim", C.c_double), ("ln_itmax", C.c_int64),
                ("ne_atol", C.c_double), ("ne_rtol", C.c_double), ("ne_etol", C.c_double),
                ("ne_conlim", C.c_double), ("ne_itmax", C.c_int64)]


class LdltOpts(C.Structure):
    _fields_ = [("ldlt_tol", C.c_double), ("ldlt_r1", C.c_double), ("ldlt_r2", C.c_double)]


class ExtrasOpts(C.Structure):
    """fpsb_extras_opts — tolerances of the batched LDLt solve_two_extras (itmax 0 = Krylov.jl's default)."""
    _fields_ = [("cg_atol", C.c_double), ("cg_rtol", C.c_double), ("cg_itmax", C.c_int64),
                ("mr_atol", C.c_double), ("mr_rtol", C.c_double), ("mr_etol", C.c_double),
                ("mr_conlim", C.c_double), ("mr_itmax", C.c_int64)]


# every symbol include/fpsb.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "fpsb_version", "fpsb_last_error", "fpsb_device_count", "fpsb_create", "fpsb_destroy",
    "fpsb_dims", "fpsb_pin_host", "fpsb_unpin_host", "fpsb_stream", "fpsb_set_caller_stream", "fpsb_synchronize", "fpsb_timer_start", "fpsb_timer_stop",
    "fpsb_launch_count", "fpsb_pipeline_gate", "fpsb_tile_stats", "fpsb_set_jac_values", "fpsb_jprod", "fpsb_jtprod", "fpsb_jprod2",
    "fpsb_jtprod2", "fpsb_iter_default_opts", "fpsb_iter_setup", "fpsb_iter_solve_two_mixed",
    "fpsb_iter_solve_two_least_squares", "fpsb_iter_solve_two_extras", "fpsb_iter_last_profile", "fpsb_iter_loop_info", "fpsb_ldlt_default_opts",
    "fpsb_ldlt_analyze", "fpsb_ldlt_symbolic_sizes", "fpsb_ldlt_get_symbolic",
    "fpsb_ldlt_plan_info", "fpsb_ldlt_factorize", "fpsb_ldlt_get_factor",
    "fpsb_ldlt_solve_two_mixed", "fpsb_ldlt_solve_two_least_squares", "fpsb_ldlt_solve_two_extras",
    "fpsb_ldlt_batch_solve_two_mixed", "fpsb_ldlt_batch_solve_two_least_squares", "fpsb_ldlt_batch_solve_two_extras",
    "fpsb_symbolic_create", "fpsb_symbolic_destroy", "fpsb_symbolic_sizes", "fpsb_symbolic_get",
    "fpsb_symbolic_plan_info", "fpsb_order_dissection", "fpsb_batch_solve_two",
    "fpsb_dist_unique_id", "fpsb_dist_attach", "fpsb_dist_jprod", "fpsb_dist_jtprod",
    "fpsb_dist_solve_two_mixed", "fpsb_dist_solve_two_least_squares", "fpsb_dist_solve_two_extras", "fpsb_dist_profile", "fpsb_dist_last_profile",
    "fpsb_dist_peer_blob_bytes", "fpsb_dist_peer_export", "fpsb_dist_peer_attach", "fpsb_dist_peer_active",
    "fpsb_fp_ys_gs", "fpsb_fp_hash", "fpsb_fp_obj", "fpsb_fp_grad", "fpsb_fp_ptv", "fpsb_fp_hprod2", "fpsb_fp_hprod1", "fpsb_trcg_init", "fpsb_trcg_step",
    "fpsb_fp_batch_ys_gs", "fpsb_fp_batch_hash", "fpsb_fp_batch_obj", "fpsb_fp_batch_grad", "fpsb_fp_batch_ptv",
    "fpsb_fp_batch_hprod2", "fpsb_fp_batch_hprod1", "fpsb_batch_jprod", "fpsb_batch_jtprod", "fpsb_trcg_batch_init",
    "fpsb_trcg_batch_step",
]

_lib = None


def build():
    """Compile libfpsb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    subprocess.check_call(["bash", os.path.join(_HERE, "csrc", "build.sh")])
    return SO_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (nvcc, sm_100a). There is no CPU fallback for this path.")
        L = C.CDLL(SO_PATH)
        L.fpsb_last_error.restype = C.c_char_p
        L.fpsb_stream.restype = C.c_void_p
        L.fpsb_launch_count.restype = C.c_int64
        _lib = L
    return _lib


class FpsbError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = lib().fpsb_last_error().decode("utf-8", "replace")
        raise FpsbError(f"{what} failed: {ERRORS.get(rc, rc)}: {msg}")
