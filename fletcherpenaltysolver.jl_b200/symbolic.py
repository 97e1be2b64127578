"""Host-only symbolic analysis of K = [I A'; A -dI] (binding of fpsb_symbolic_* in include/fpsb.h).

Mirrors the `ldl_analyze` step of the LDLtSolver constructor
(/root/reference/src/solve_two_systems_struct.jl:343-344).  Runs without a GPU.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check


class SymbolicAnalysis:
    def __init__(self, nvar, ncon, jrow, jcol, P=None, index_base=0):
        L = _lib.lib()
        jrow = np.ascontiguousarray(jrow, dtype=np.int64)
        jcol = np.ascontiguousarray(jcol, dtype=np.int64)
        Pa = np.ascontiguousarray(P, dtype=np.int64) if P is not None else None
        self.h = C.c_void_p()
        check(L.fpsb_symbolic_create(C.c_int64(nvar), C.c_int64(ncon), C.c_int64(len(jrow)),
                                     jrow.ctypes.data_as(C.c_void_p), jcol.ctypes.data_as(C.c_void_p),
                                     C.c_int(index_base),
                                     Pa.ctypes.data_as(C.c_void_p) if Pa is not None else None,
                                     C.byref(self.h)), "fpsb_symbolic_create")
        N, lnz = C.c_int64(), C.c_int64()
        check(L.fpsb_symbolic_sizes(self.h, C.byref(N), C.byref(lnz)), "fpsb_symbolic_sizes")
        self.N, self.lnz = N.value, lnz.value

    def get(self):
        N, lnz = self.N, self.lnz
        P = np.zeros(N, np.int64); parent = np.zeros(N, np.int64); Lnz = np.zeros(N, np.int64)
        Lp = np.zeros(N + 1, np.int64); Li = np.zeros(max(lnz, 1), np.int64)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        check(_lib.lib().fpsb_symbolic_get(self.h, p(P), p(parent), p(Lnz), p(Lp), p(Li)),
              "fpsb_symbolic_get")
        return dict(P=P, parent=parent, Lnz=Lnz, Lp=Lp, Li=Li[:lnz])

    def plan_info(self):
        ns, pn, npairs, fl, nl, nf = C.c_int64(), C.c_int64(), C.c_int64(), C.c_double(), C.c_int64(), C.c_int64()
        check(_lib.lib().fpsb_symbolic_plan_info(self.h, C.byref(ns), C.byref(pn), C.byref(npairs),
                                                 C.byref(fl), C.byref(nl), C.byref(nf)), "fpsb_symbolic_plan_info")
        return dict(nsuper=ns.value, panel_nnz=pn.value, npairs=npairs.value, flops=fl.value,
                    nlevels=nl.value, nleaf=nf.value)

    def routes(self):
        """Which LDLt routines and staging passes the plan of this analysis goes through (fpsb_symbolic_ldlt_routes;
        keys: _lib.LDLT_ROUTE_KEYS)."""
        return _lib.ldlt_routes(_lib.lib().fpsb_symbolic_ldlt_routes, self.h, "fpsb_symbolic_ldlt_routes")

    def __del__(self):
        try:
            if self.h:
                _lib.lib().fpsb_symbolic_destroy(self.h)
                self.h = None
        except Exception:
            pass


def order_dissection(nvar, ncon, jrow, jcol, nparts=0, index_base=0):
    """BFS level-set dissection ordering of K (binding of fpsb_order_dissection); returns P."""
    jrow = np.ascontiguousarray(jrow, dtype=np.int64)
    jcol = np.ascontiguousarray(jcol, dtype=np.int64)
    P = np.zeros(nvar + ncon, np.int64)
    check(_lib.lib().fpsb_order_dissection(C.c_int64(nvar), C.c_int64(ncon), C.c_int64(len(jrow)),
                                           jrow.ctypes.data_as(C.c_void_p), jcol.ctypes.data_as(C.c_void_p),
                                           C.c_int(index_base), C.c_int(nparts),
                                           P.ctypes.data_as(C.c_void_p)), "fpsb_order_dissection")
    return P
