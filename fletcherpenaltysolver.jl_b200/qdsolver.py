"""Host-side mirror of the reference's QD linear-algebra plugin surface, backed by libfpsb200.so.

Reference (all paths under /root/reference):
    abstract type QDSolver                         src/solve_two_systems_struct.jl:16
    IterativeSolver(nlp, ::T; kwargs...)           src/solve_two_systems_struct.jl:23-160
    LDLtSolver(nlp, ::T; kwargs...)                src/solve_two_systems_struct.jl:299-353
    solve_two_extras / _least_squares / _mixed     src/solve_linear_system.jl:1-252
    qdsolver_correspondence                        src/parameters.jl:197

Same names, argument meaning and error behaviour: numerical failure only warns
(`warnings.warn`, the analogue of `@warn`) and returns the last iterate / the untouched
right-hand sides.  All arithmetic happens in hand-written CUDA behind the C ABI
(include/fpsb.h); nothing here computes on the CPU and there is no CPU fallback.
"""
import ctypes as C
import warnings

import numpy as np

from . import _lib
from ._lib import FPSB_DEVICE, FPSB_HOST, ExtrasOpts, IterOpts, KrylovStats, LdltOpts, check

SQRT_EPS = float(np.sqrt(np.finfo(np.float64).eps))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class B200Handle:
    """Owns one fpsb_handle: the device-resident Jacobian (CSR of A and A') and workspaces."""

    def __init__(self, nvar, ncon, jrow, jcol, index_base=0, device=0):
        L = _lib.lib()
        self.nvar, self.ncon = int(nvar), int(ncon)
        jrow = np.ascontiguousarray(jrow, dtype=np.int64)
        jcol = np.ascontiguousarray(jcol, dtype=np.int64)
        self.nnzj = int(jrow.shape[0])
        self.h = C.c_void_p()
        check(L.fpsb_create(C.c_int64(self.nvar), C.c_int64(self.ncon), C.c_int64(self.nnzj),
                            _ptr(jrow), _ptr(jcol), C.c_int(index_base), C.c_int(device),
                            C.byref(self.h)), "fpsb_create")
        self.device = device

    # -- lifetime ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            _lib.lib().fpsb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers -------------------------------------------------------------------------------
    def _arg(self, a):
        """numpy array -> (pointer, FPSB_HOST); torch CUDA tensor / raw int -> (pointer, FPSB_DEVICE)."""
        if isinstance(a, np.ndarray):
            return _ptr(a), FPSB_HOST
        if hasattr(a, "data_ptr"):
            if a.is_cuda:
                self._follow_torch_stream(a)
            return C.c_void_p(a.data_ptr()), (FPSB_DEVICE if a.is_cuda else FPSB_HOST)
        raise TypeError("expected a numpy array or a torch tensor")

    def _follow_torch_stream(self, t):
        """Device tensors are produced / consumed on torch's current stream: tell the library, which orders
        its own (non-blocking) stream against it on the way in and out of every FPSB_DEVICE call."""
        import torch
        s = int(torch.cuda.current_stream(t.device).cuda_stream)
        if s != getattr(self, "_caller_stream", 0):
            check(_lib.lib().fpsb_set_caller_stream(self.h, C.c_void_p(s)), "fpsb_set_caller_stream")
            self._caller_stream = s

    @staticmethod
    def pin_host(a):
        """Page-lock a long-lived numpy array so FPSB_HOST calls DMA directly from / into it."""
        check(_lib.lib().fpsb_pin_host(_ptr(a), C.c_int64(a.nbytes)), "fpsb_pin_host")

    @staticmethod
    def unpin_host(a):
        _lib.lib().fpsb_unpin_host(_ptr(a))

    def stream(self):
        return _lib.lib().fpsb_stream(self.h)

    def synchronize(self):
        check(_lib.lib().fpsb_synchronize(self.h), "fpsb_synchronize")

    def timer_start(self):
        check(_lib.lib().fpsb_timer_start(self.h), "fpsb_timer_start")

    def timer_stop(self):
        ms = C.c_double()
        check(_lib.lib().fpsb_timer_stop(self.h, C.byref(ms)), "fpsb_timer_stop")
        return ms.value

    def launch_count(self):
        return int(_lib.lib().fpsb_launch_count(self.h))

    def tile_stats(self):
        """{tiles, windowed, multi-segment} of A and of A' (fpsb_tile_stats)."""
        out = (C.c_int64 * 6)()
        check(_lib.lib().fpsb_tile_stats(self.h, out), "fpsb_tile_stats")
        v = [int(x) for x in out]
        return {"A": dict(tiles=v[0], windowed=v[1], multi_segment=v[2]),
                "At": dict(tiles=v[3], windowed=v[4], multi_segment=v[5])}

    # -- Jacobian ------------------------------------------------------------------------------
    def set_jac_values(self, vals):
        if isinstance(vals, np.ndarray):
            vals = _f64(vals)
        p, loc = self._arg(vals)
        check(_lib.lib().fpsb_set_jac_values(self.h, p, C.c_int(loc)), "fpsb_set_jac_values")

    def _spmv(self, fn, x, nout, ncols=1):
        if isinstance(x, np.ndarray):
            x = _f64(x)
            y = np.empty(nout * ncols)
            check(fn(self.h, _ptr(x), _ptr(y), C.c_int(FPSB_HOST)), fn.__name__)
            return y
        import torch
        y = torch.empty(nout * ncols, dtype=torch.float64, device=x.device)
        self._follow_torch_stream(x)
        check(fn(self.h, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), C.c_int(FPSB_DEVICE)),
              fn.__name__)
        return y

    def jprod(self, v):
        return self._spmv(_lib.lib().fpsb_jprod, v, self.ncon)

    def jtprod(self, u):
        return self._spmv(_lib.lib().fpsb_jtprod, u, self.nvar)

    def _batch_spmv(self, fn, name, jvals, X, nin, nout):
        import torch
        if not (hasattr(X, "is_cuda") and X.is_cuda):
            raise TypeError(f"{name}: expects CUDA tensors")
        X = X.to(torch.float64).contiguous()
        jvals = torch.as_tensor(jvals, dtype=torch.float64, device=X.device).contiguous()
        if X.ndim != 2 or X.shape[1] != nin:
            raise ValueError(f"{name}: the vectors must be (ninst, {nin})")
        ninst = int(X.shape[0])
        if tuple(jvals.shape) == (self.nnzj,):
            stride = 0
        elif tuple(jvals.shape) == (ninst, self.nnzj):
            stride = self.nnzj
        else:
            raise ValueError(f"{name}: jvals must be ({self.nnzj},) or (ninst, {self.nnzj})")
        out = torch.empty((ninst, nout), dtype=torch.float64, device=X.device)
        if ninst == 0:
            return out
        self._follow_torch_stream(X)
        check(fn(self.h, C.c_int64(ninst), C.c_void_p(jvals.data_ptr()), C.c_int64(stride), C.c_void_p(X.data_ptr()),
                 C.c_void_p(out.data_ptr())), name)
        return out

    def batch_jprod(self, jvals, V):
        """A_i v_i for every row of V (ninst, nvar) -> (ninst, ncon), A_i with the values jvals[i] (COO order of this
        handle's pattern); jvals (nnzj,) is one set of values for every instance (fpsb_batch_jprod).  CUDA tensors."""
        return self._batch_spmv(_lib.lib().fpsb_batch_jprod, "fpsb_batch_jprod", jvals, V, self.nvar, self.ncon)

    def batch_jtprod(self, jvals, U):
        """A_i' u_i for every row of U (ninst, ncon) -> (ninst, nvar) (fpsb_batch_jtprod); jvals as in batch_jprod."""
        return self._batch_spmv(_lib.lib().fpsb_batch_jtprod, "fpsb_batch_jtprod", jvals, U, self.ncon, self.nvar)

    def jprod2(self, v):
        return self._spmv(_lib.lib().fpsb_jprod2, v, self.ncon, 2)

    def jtprod2(self, u):
        return self._spmv(_lib.lib().fpsb_jtprod2, u, self.nvar, 2)

    # -- raw 2-RHS solves (numpy in -> numpy out, or torch CUDA in -> torch CUDA out) -----------
    def _outs(self, like, sizes):
        if isinstance(like, np.ndarray):
            return [np.empty(s) for s in sizes]
        import torch
        return [torch.empty(s, dtype=torch.float64, device=like.device) for s in sizes]

    def _two(self, fn, name, pre, rhs1, rhs2, with_stats, out=None):
        if isinstance(rhs1, np.ndarray):
            rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        n, m = self.nvar, self.ncon
        p1, q1, p2, q2 = out if out is not None else self._outs(rhs1, [n, m, n, m])
        a1, loc = self._arg(rhs1)
        a2, _ = self._arg(rhs2)
        tail = (KrylovStats * 2)() if with_stats else C.c_int(0)
        rc = fn(self.h, *pre, a1, a2, self._arg(p1)[0], self._arg(q1)[0], self._arg(p2)[0],
                self._arg(q2)[0], C.c_int(loc), tail if with_stats else C.byref(tail))
        check(rc, name)
        extra = [tail[0].as_dict(), tail[1].as_dict()] if with_stats else bool(tail.value)
        return p1, q1, p2, q2, extra

    def iter_setup(self, opts=None):
        check(_lib.lib().fpsb_iter_setup(self.h, C.byref(opts) if opts is not None else None),
              "fpsb_iter_setup")

    def iter_last_profile(self):
        ms, nl = C.c_double(), C.c_int64()
        check(_lib.lib().fpsb_iter_last_profile(self.h, C.byref(ms), C.byref(nl)), "fpsb_iter_last_profile")
        return ms.value, nl.value

    def loop_info(self):
        """Persistent-loop geometry of the last iter_solve_two_* call (fpsb_iter_loop_info)."""
        out = (C.c_int64 * 8)()
        check(_lib.lib().fpsb_iter_loop_info(self.h, out), "fpsb_iter_loop_info")
        keys = ("persistent", "early", "nstage", "grid", "stage_bytes", "inflight", "nspec", "chunk")
        return {k: int(v) for k, v in zip(keys, out)}

    def iter_solve_two_mixed(self, delta, rhs1, rhs2, out=None):
        return self._two(_lib.lib().fpsb_iter_solve_two_mixed, "fpsb_iter_solve_two_mixed",
                         (C.c_double(delta),), rhs1, rhs2, True, out)

    def iter_solve_two_least_squares(self, delta, rhs1, rhs2):
        return self._two(_lib.lib().fpsb_iter_solve_two_least_squares,
                         "fpsb_iter_solve_two_least_squares", (C.c_double(delta),), rhs1, rhs2, True)

    def _extras(self, fn, name, delta, rhs1, rhs2):
        if isinstance(rhs1, np.ndarray):
            rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        u1, u2 = self._outs(rhs1, [self.ncon, self.ncon])
        a1, loc = self._arg(rhs1)
        st = (KrylovStats * 2)()
        check(fn(self.h, C.c_double(delta), a1, self._arg(rhs2)[0], self._arg(u1)[0],
                 self._arg(u2)[0], C.c_int(loc), st), name)
        return u1, u2, [st[0].as_dict(), st[1].as_dict()]

    def iter_solve_two_extras(self, delta, rhs1, rhs2):
        return self._extras(_lib.lib().fpsb_iter_solve_two_extras, "fpsb_iter_solve_two_extras",
                            delta, rhs1, rhs2)

    def ldlt_solve_two_extras(self, delta, rhs1, rhs2):
        return self._extras(_lib.lib().fpsb_ldlt_solve_two_extras, "fpsb_ldlt_solve_two_extras",
                            delta, rhs1, rhs2)

    def ldlt_analyze(self, P=None, index_base=0, opts=None):
        Pa = np.ascontiguousarray(P, dtype=np.int64) if P is not None else None
        check(_lib.lib().fpsb_ldlt_analyze(self.h, _ptr(Pa) if Pa is not None else None,
                                           C.c_int(index_base),
                                           C.byref(opts) if opts is not None else None),
              "fpsb_ldlt_analyze")

    def ldlt_symbolic(self):
        L = _lib.lib()
        N, lnz = C.c_int64(), C.c_int64()
        check(L.fpsb_ldlt_symbolic_sizes(self.h, C.byref(N), C.byref(lnz)), "fpsb_ldlt_symbolic_sizes")
        N, lnz = N.value, lnz.value
        P = np.zeros(N, np.int64); parent = np.zeros(N, np.int64); Lnz = np.zeros(N, np.int64)
        Lp = np.zeros(N + 1, np.int64); Li = np.zeros(max(lnz, 1), np.int64)
        check(L.fpsb_ldlt_get_symbolic(self.h, _ptr(P), _ptr(parent), _ptr(Lnz), _ptr(Lp), _ptr(Li)),
              "fpsb_ldlt_get_symbolic")
        return dict(P=P, parent=parent, Lnz=Lnz, Lp=Lp, Li=Li[:lnz])

    def ldlt_plan_info(self):
        ns, pn, npairs, fl, nl, nf = C.c_int64(), C.c_int64(), C.c_int64(), C.c_double(), C.c_int64(), C.c_int64()
        check(_lib.lib().fpsb_ldlt_plan_info(self.h, C.byref(ns), C.byref(pn), C.byref(npairs),
                                             C.byref(fl), C.byref(nl), C.byref(nf)), "fpsb_ldlt_plan_info")
        return dict(nsuper=ns.value, panel_nnz=pn.value, npairs=npairs.value, flops=fl.value,
                    nlevels=nl.value, nleaf=nf.value)

    def ldlt_factorize(self, delta):
        ok = C.c_int(0)
        check(_lib.lib().fpsb_ldlt_factorize(self.h, C.c_double(delta), C.byref(ok)),
              "fpsb_ldlt_factorize")
        return bool(ok.value)

    def ldlt_get_factor(self):
        s = self.ldlt_symbolic()
        Lx = np.zeros(max(len(s["Li"]), 1)); D = np.zeros(len(s["P"]))
        check(_lib.lib().fpsb_ldlt_get_factor(self.h, _ptr(Lx), _ptr(D)), "fpsb_ldlt_get_factor")
        return Lx[:len(s["Li"])], D

    def ldlt_solve_two_mixed(self, delta, rhs1, rhs2):
        return self._two(_lib.lib().fpsb_ldlt_solve_two_mixed, "fpsb_ldlt_solve_two_mixed",
                         (C.c_double(delta),), rhs1, rhs2, False)

    def ldlt_solve_two_least_squares(self, rhs1, rhs2):
        return self._two(_lib.lib().fpsb_ldlt_solve_two_least_squares,
                         "fpsb_ldlt_solve_two_least_squares", (), rhs1, rhs2, False)

    # -- batched LDLt path: many instances of this handle's pattern in one call ------------------
    def _batch(self, fn, name, pre, rhs1, rhs2, n2):
        host = isinstance(rhs1, np.ndarray)
        if host:
            rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        else:
            import torch
            rhs1, rhs2 = rhs1.to(torch.float64).contiguous(), rhs2.to(torch.float64).contiguous()
        n, m = self.nvar, self.ncon
        ninst = int(rhs1.shape[0])
        if tuple(rhs1.shape) != (ninst, n) or tuple(rhs2.shape) != (ninst, n2):
            raise ValueError(f"{name}: rhs1 must be (ninst, {n}) and rhs2 (ninst, {n2})")
        p1, q1, p2, q2 = self._outs(rhs1, [(ninst, n), (ninst, m), (ninst, n), (ninst, m)])
        if host:
            fac = np.zeros(ninst, dtype=np.int32)
        else:
            import torch
            fac = torch.zeros(ninst, dtype=torch.int32, device=rhs1.device)
        a1, loc = self._arg(rhs1)
        ptrs = [self._arg(a)[0] for a in (*pre, rhs2, p1, q1, p2, q2, fac)]
        check(fn(self.h, C.c_int64(ninst), *ptrs[:len(pre)], a1, *ptrs[len(pre):], C.c_int(loc)), name)
        return p1, q1, p2, q2, (fac.astype(bool) if host else fac.bool())

    def ldlt_batch_solve_two_mixed(self, delta, jvals, rhs1, rhs2):
        """Refactor + solve of `ninst` instances of this handle's pattern (fpsb_ldlt_batch_solve_two_mixed).
        jvals (ninst, nnzj), rhs1 (ninst, nvar), rhs2 (ninst, ncon): numpy arrays, or CUDA tensors (device path);
        delta: a scalar or one value per instance.  Returns p1, q1, p2, q2 as (ninst, .) arrays and `factorized`
        (bool, per instance).  The factors stay on the device for ldlt_batch_solve_two_least_squares."""
        ninst = int(rhs1.shape[0])
        if isinstance(rhs1, np.ndarray):
            jvals = _f64(jvals)
            d = _f64(np.broadcast_to(np.asarray(delta, dtype=np.float64), (ninst,)))
        else:
            import torch
            jvals = torch.as_tensor(jvals, dtype=torch.float64, device=rhs1.device).contiguous()
            d = torch.as_tensor(delta, dtype=torch.float64, device=rhs1.device).expand(ninst).contiguous()
        if tuple(jvals.shape) != (ninst, self.nnzj):
            raise ValueError(f"ldlt_batch_solve_two_mixed: jvals must be (ninst, {self.nnzj})")
        return self._batch(_lib.lib().fpsb_ldlt_batch_solve_two_mixed, "fpsb_ldlt_batch_solve_two_mixed",
                           (jvals, d), rhs1, rhs2, self.ncon)

    def ldlt_batch_solve_two_least_squares(self, rhs1, rhs2):
        """Least-squares solves of the instances of the last ldlt_batch_solve_two_mixed call (same ninst) with their
        stored factors; rhs1, rhs2 (ninst, nvar)."""
        return self._batch(_lib.lib().fpsb_ldlt_batch_solve_two_least_squares,
                           "fpsb_ldlt_batch_solve_two_least_squares", (), rhs1, rhs2, self.nvar)

    def ldlt_batch_solve_two_extras(self, delta, jvals, rhs1, rhs2, opts=None):
        """solve_two_extras of the LDLt path for `ninst` instances of this handle's pattern
        (fpsb_ldlt_batch_solve_two_extras): u1 = cgls(A', rhs1, lambda = tau), u2 = minres(A A', rhs2, lambda = tau),
        tau = max(delta, 1e-14), with each instance's own Jacobian values.  jvals (ninst, nnzj), rhs1 (ninst, nvar),
        rhs2 (ninst, ncon): numpy arrays, or CUDA tensors (device path); delta: a scalar or one value per instance;
        opts: an ExtrasOpts (None: the tolerances of ldlt_solve_two_extras).  Needs neither ldlt_analyze nor
        set_jac_values and changes neither.  Returns u1, u2 as (ninst, ncon) arrays and the stats as a dict of
        (ninst, 2) arrays (column 0 CGLS, column 1 MINRES) keyed like KrylovStats.as_dict()."""
        host = isinstance(rhs1, np.ndarray)
        n, m, name = self.nvar, self.ncon, "ldlt_batch_solve_two_extras"
        if host:
            rhs1, rhs2, jvals = _f64(rhs1), _f64(rhs2), _f64(jvals)
            d = np.asarray(delta, dtype=np.float64)
        else:
            import torch
            dev = rhs1.device
            rhs1, rhs2 = rhs1.to(torch.float64).contiguous(), rhs2.to(torch.float64).contiguous()
            jvals = torch.as_tensor(jvals, dtype=torch.float64, device=dev).contiguous()
            d = torch.as_tensor(delta, dtype=torch.float64, device=dev)
        ninst = int(rhs1.shape[0]) if rhs1.ndim == 2 else -1
        if (ninst < 0 or tuple(rhs1.shape) != (ninst, n) or tuple(rhs2.shape) != (ninst, m)
                or tuple(jvals.shape) != (ninst, self.nnzj)):
            raise ValueError(f"{name}: jvals must be (ninst, {self.nnzj}), rhs1 (ninst, {n}) and rhs2 (ninst, {m})")
        if d.ndim == 0:
            d = np.full(ninst, float(d)) if host else d.expand(ninst).contiguous()
        elif tuple(d.shape) != (ninst,):
            raise ValueError(f"{name}: delta must be a scalar or have one value per instance")
        else:
            d = _f64(d) if host else d.contiguous()
        u1, u2 = self._outs(rhs1, [(ninst, m), (ninst, m)])
        # fpsb_krylov_stats [ninst][2] is 8 doubles per entry
        if host:
            st = np.zeros((ninst, 2, 8))
        else:
            import torch
            st = torch.zeros((ninst, 2, 8), dtype=torch.float64, device=rhs1.device)
        a1, loc = self._arg(rhs1)
        ptrs = [self._arg(a)[0] for a in (jvals, d, rhs2, u1, u2, st)]
        check(_lib.lib().fpsb_ldlt_batch_solve_two_extras(
            self.h, C.c_int64(ninst), ptrs[0], ptrs[1], a1, *ptrs[2:],
            C.byref(opts) if opts is not None else None, C.c_int(loc)), "fpsb_ldlt_batch_solve_two_extras")
        return u1, u2, _stats_arrays(st, host)


def _stats_arrays(st, host):
    """(ninst, 2, 8) float64 view of fpsb_krylov_stats [ninst][2] -> dict of (ninst, 2) arrays (KrylovStats layout:
    niter int64 | solved, inconsistent, status, pad int32 | rnorm, arnorm, anorm, acond, xnorm)."""
    if host:
        i64, i32, cp = st.view(np.int64), st.view(np.int32), np.copy
    else:
        import torch
        i64, i32, cp = st.view(torch.int64), st.view(torch.int32), torch.clone
    out = dict(niter=cp(i64[..., 0]), solved=i32[..., 2] != 0, inconsistent=i32[..., 3] != 0, status=cp(i32[..., 4]))
    for k, name in enumerate(("rnorm", "arnorm", "anorm", "acond", "xnorm")):
        out[name] = cp(st[..., 3 + k])
    return out


# --------------------------------------------------------------------------------------------------
# plugin surface
# --------------------------------------------------------------------------------------------------
class QDSolver:
    """abstract type QDSolver (src/solve_two_systems_struct.jl:16)."""


def _npen(nlp, explicit_linear_constraints):
    return nlp.meta.nnln if explicit_linear_constraints else nlp.meta.ncon


def _structure(nlp, explicit_linear_constraints):
    if explicit_linear_constraints:
        return nlp.jac_nln_structure()
    return nlp.jac_structure()


class IterativeSolver(QDSolver):
    """IterativeSolver(nlp, ::T; kwargs...) <: QDSolver — Krylov path on the GPU.

    Keyword names and defaults are the reference's (src/solve_two_systems_struct.jl:94-131);
    unknown keywords are swallowed like the reference's `kwargs...`.
    """

    def __init__(self, nlp, _zero=0.0, *, explicit_linear_constraints=False, ls_atol=SQRT_EPS,
                 ls_rtol=SQRT_EPS, ls_itmax=None, ln_atol=SQRT_EPS, ln_rtol=SQRT_EPS,
                 ln_btol=SQRT_EPS, ln_conlim=1 / SQRT_EPS, ln_itmax=None, ne_atol=SQRT_EPS,
                 ne_rtol=SQRT_EPS, ne_etol=SQRT_EPS, ne_itmax=0, ne_conlim=1 / SQRT_EPS, device=0,
                 **kwargs):
        ncon = _npen(nlp, explicit_linear_constraints)
        nvar = nlp.meta.nvar
        self.explicit_linear_constraints = explicit_linear_constraints
        o = IterOpts()
        o.ls_atol, o.ls_rtol = ls_atol, ls_rtol
        o.ls_itmax = 5 * (ncon + nvar) if ls_itmax is None else ls_itmax
        o.ln_atol, o.ln_rtol, o.ln_btol, o.ln_conlim = ln_atol, ln_rtol, ln_btol, ln_conlim
        o.ln_itmax = 5 * (ncon + nvar) if ln_itmax is None else ln_itmax
        o.ne_atol, o.ne_rtol, o.ne_etol, o.ne_conlim, o.ne_itmax = ne_atol, ne_rtol, ne_etol, ne_conlim, ne_itmax
        self.opts = o
        rows, cols = _structure(nlp, explicit_linear_constraints)
        self.handle = B200Handle(nvar, ncon, rows, cols, index_base=0, device=device)
        self.handle.iter_setup(o)
        self.last_stats = None


class LDLtSolver(QDSolver):
    """LDLtSolver(nlp, ::T; ldlt_tol, ldlt_r1, ldlt_r2, kwargs...) <: QDSolver — direct path.

    The constructor performs the reference's `ldl_analyze` (src/solve_two_systems_struct.jl:343-348):
    host-side ordering + symbolic analysis, uploaded to the GPU; `P` may supply the permutation
    (LDLFactorizations' `ldl_analyze(A, P)`), otherwise `ordering` picks the built-in one: "amd" (minimum
    degree, what the reference does), "dissection" (B200-oriented, shallow elimination tree) or "auto"
    (minimum degree below AUTO_DISSECTION_FROM unknowns, dissection from there on).
    """
    AUTO_DISSECTION_FROM = 20000

    def __init__(self, nlp, _zero=0.0, *, explicit_linear_constraints=False, ldlt_tol=SQRT_EPS,
                 ldlt_r1=SQRT_EPS, ldlt_r2=-SQRT_EPS, P=None, ordering="auto", device=0, **kwargs):
        ncon = _npen(nlp, explicit_linear_constraints)
        nvar = nlp.meta.nvar
        self.explicit_linear_constraints = explicit_linear_constraints
        rows, cols = _structure(nlp, explicit_linear_constraints)
        self.nnz = nvar + len(rows) + ncon
        self.handle = B200Handle(nvar, ncon, rows, cols, index_base=0, device=device)
        o = LdltOpts()
        o.ldlt_tol, o.ldlt_r1, o.ldlt_r2 = ldlt_tol, ldlt_r1, ldlt_r2
        self.opts = o
        if ordering not in ("auto", "amd", "dissection"):
            raise ValueError("ordering must be 'auto', 'amd' or 'dissection'")
        if ordering == "auto":
            # minimum degree (what the reference's ldl_analyze does) for small systems; from 20 000 unknowns on the
            # dissection ordering, whose elimination tree is O(log N) deep instead of chain-like (C2: 14 ms vs 168 ms)
            ordering = "dissection" if nvar + ncon >= LDLtSolver.AUTO_DISSECTION_FROM else "amd"
        self.ordering = ordering
        if P is None and ordering == "dissection":
            # B200-oriented ordering: same fill class as minimum degree on band-like structure but a
            # dependency depth of O(log) instead of O(N) (see fpsb_order_dissection in include/fpsb.h)
            from .symbolic import order_dissection
            P = order_dissection(nvar, ncon, rows, cols)
        self.handle.ldlt_analyze(P, 0, o)
        self.factorized = False
        self.last_stats = None
        self.last_batch_stats = None


qdsolver_correspondence = {"iterative": IterativeSolver, "ldlt": LDLtSolver}


def _jac_values(fpnlp, x):
    if fpnlp.explicit_linear_constraints:
        return fpnlp.nlp.jac_nln_coord(x)
    return fpnlp.nlp.jac_coord(x)


def solve_two_mixed(fpnlp, x, rhs1, rhs2):
    """p1, q1, p2, q2 = solve_two_mixed(nlp, x, rhs1, rhs2)   (src/solve_linear_system.jl:29-43)

    rhs1 has size nvar, rhs2 size ncon.  Refreshes the Jacobian at x (jac_coord! / jac_op!),
    then solves K [p1 p2; q1 q2] = [rhs1 0; 0 rhs2]."""
    qds = fpnlp.qdsolver
    if hasattr(qds, "solve_two_mixed"):          # user-defined QDSolver subtype (dispatch on type)
        return qds.solve_two_mixed(fpnlp, x, rhs1, rhs2)
    H = qds.handle
    H.set_jac_values(_jac_values(fpnlp, x))
    if isinstance(qds, IterativeSolver):
        p1, q1, p2, q2, st = H.iter_solve_two_mixed(float(fpnlp.delta), rhs1, rhs2)
        qds.last_stats = st
        if not st[0]["solved"]:
            warnings.warn("Failed solving 1st linear system lsqr in mixed.")
        if not st[1]["solved"]:
            warnings.warn("Failed solving 2nd linear system craig in mixed.")
        return p1, q1, p2, q2
    if isinstance(qds, LDLtSolver):
        p1, q1, p2, q2, ok = H.ldlt_solve_two_mixed(float(fpnlp.delta), rhs1, rhs2)
        qds.factorized = ok
        if not ok:
            warnings.warn("_solve_ldlt_factorization: failed _factorization")
        return p1, q1, p2, q2
    raise TypeError(f"solve_two_mixed: no method for {type(qds).__name__}")


def solve_two_least_squares(fpnlp, x, rhs1, rhs2):
    """p1, q1, p2, q2 = solve_two_least_squares(nlp, x, rhs1, rhs2)  (src/solve_linear_system.jl:12-27)

    Both right-hand sides have size nvar.  The Jacobian / factorisation of the last
    solve_two_mixed call is trusted (reference comments at :86 and :178)."""
    qds = fpnlp.qdsolver
    if hasattr(qds, "solve_two_least_squares"):
        return qds.solve_two_least_squares(fpnlp, x, rhs1, rhs2)
    H = qds.handle
    if isinstance(qds, IterativeSolver):
        p1, q1, p2, q2, st = H.iter_solve_two_least_squares(float(fpnlp.delta), rhs1, rhs2)
        qds.last_stats = st
        if not st[0]["solved"]:
            warnings.warn("Failed solving 1st linear system lsqr.")
        if not st[1]["solved"]:
            warnings.warn("Failed solving 2nd linear system lsqr.")
        return p1, q1, p2, q2
    if isinstance(qds, LDLtSolver):
        p1, q1, p2, q2, ok = H.ldlt_solve_two_least_squares(rhs1, rhs2)
        if not ok:
            warnings.warn("_solve_ldlt_factorization: failed _factorization")
        return p1, q1, p2, q2
    raise TypeError(f"solve_two_least_squares: no method for {type(qds).__name__}")


def solve_two_extras(fpnlp, x, rhs1, rhs2):
    """invJtJJv, invJtJSsv = solve_two_extras(nlp, x, rhs1, rhs2)  (src/solve_linear_system.jl:1-10)"""
    qds = fpnlp.qdsolver
    if hasattr(qds, "solve_two_extras"):
        return qds.solve_two_extras(fpnlp, x, rhs1, rhs2)
    H = qds.handle
    if isinstance(qds, IterativeSolver):
        u1, u2, st = H.iter_solve_two_extras(float(fpnlp.delta), rhs1, rhs2)
        qds.last_stats = st
        if not st[0]["solved"]:
            warnings.warn("Failed solving 1st linear system lsqr in extra.")
        if not st[1]["solved"]:
            warnings.warn("Failed solving 2nd linear system minres in extra.")
        return u1, u2
    if isinstance(qds, LDLtSolver):
        # the reference re-evaluates jac_op at x here (src/solve_linear_system.jl:149-153)
        H.set_jac_values(_jac_values(fpnlp, x))
        u1, u2, st = H.ldlt_solve_two_extras(float(fpnlp.delta), rhs1, rhs2)
        qds.last_stats = st
        return u1, u2
    raise TypeError(f"solve_two_extras: no method for {type(qds).__name__}")


def solve_two_mixed_batch(fpnlp, X, rhs1, rhs2, delta=None):
    """solve_two_mixed at every row of X in one batched call (LDLtSolver only): instance i is
    solve_two_mixed(fpnlp, X[i], rhs1[i], rhs2[i]) with delta[i] (default fpnlp.delta for all), the Jacobian values
    evaluated at X[i] (jac_coord / jac_nln_coord, as solve_two_mixed does).  Returns p1, q1, p2, q2 as (ninst, .)
    arrays; warns once per instance whose factorisation failed.  The factors are kept for
    solve_two_least_squares_batch."""
    qds = fpnlp.qdsolver
    if not isinstance(qds, LDLtSolver):
        raise TypeError(f"solve_two_mixed_batch: no method for {type(qds).__name__}")
    H = qds.handle
    X = np.asarray(X, dtype=np.float64)
    J = np.empty((X.shape[0], H.nnzj))
    for i, x in enumerate(X):
        J[i] = _jac_values(fpnlp, x)
    if not isinstance(rhs1, np.ndarray):
        import torch
        J = torch.as_tensor(J, device=rhs1.device)
    p1, q1, p2, q2, ok = H.ldlt_batch_solve_two_mixed(float(fpnlp.delta) if delta is None else delta, J, rhs1, rhs2)
    _warn_failed(ok)
    return p1, q1, p2, q2


def solve_two_least_squares_batch(fpnlp, X, rhs1, rhs2):
    """solve_two_least_squares for the instances of the last solve_two_mixed_batch call (same number of rows): the
    factorisations of that call are trusted, as the single-instance function trusts the last solve_two_mixed."""
    qds = fpnlp.qdsolver
    if not isinstance(qds, LDLtSolver):
        raise TypeError(f"solve_two_least_squares_batch: no method for {type(qds).__name__}")
    p1, q1, p2, q2, ok = qds.handle.ldlt_batch_solve_two_least_squares(rhs1, rhs2)
    _warn_failed(ok)
    return p1, q1, p2, q2


def solve_two_extras_batch(fpnlp, X, rhs1, rhs2, delta=None):
    """solve_two_extras at every row of X in one batched call (LDLtSolver only): instance i is
    solve_two_extras(fpnlp, X[i], rhs1[i], rhs2[i]) with delta[i] (default fpnlp.delta for all), the Jacobian values
    evaluated at X[i] (jac_coord / jac_nln_coord, as solve_two_extras does).  rhs1 (ninst, nvar), rhs2 (ninst, npen).
    Returns u1, u2 as (ninst, npen) arrays; the per-instance Krylov stats go to qdsolver.last_batch_stats.  Like the
    single LDLt solve_two_extras it does not warn.  Leaves the factors of solve_two_mixed_batch alone."""
    qds = fpnlp.qdsolver
    if not isinstance(qds, LDLtSolver):
        raise TypeError(f"solve_two_extras_batch: no method for {type(qds).__name__}")
    H = qds.handle
    X = np.asarray(X, dtype=np.float64)
    J = np.empty((X.shape[0], H.nnzj))
    for i, x in enumerate(X):
        J[i] = _jac_values(fpnlp, x)
    if not isinstance(rhs1, np.ndarray):
        import torch
        J = torch.as_tensor(J, device=rhs1.device)
    u1, u2, st = H.ldlt_batch_solve_two_extras(float(fpnlp.delta) if delta is None else delta, J, rhs1, rhs2)
    qds.last_batch_stats = st
    return u1, u2


def _warn_failed(ok):
    failed = int((~ok).sum()) if isinstance(ok, np.ndarray) else int((~ok).sum().item())
    for _ in range(failed):
        warnings.warn("_solve_ldlt_factorization: failed _factorization")


def batch_solve_two(A, delta, rhs1, rhs2, kind="mixed", opts=None, device=0):
    """Throughput mode (BASELINE config C5): `ninst` independent small instances sharing
    (nvar, ncon).  A: (ninst, ncon, nvar); rhs1: (ninst, nvar); rhs2: (ninst, ncon) for
    kind="mixed" or (ninst, nvar) for kind="least_squares".  numpy in -> numpy out.
    Returns p1, q1, p2, q2, factorized (bool array)."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    ninst, m, n = A.shape
    rhs1 = np.ascontiguousarray(rhs1, dtype=np.float64)
    rhs2 = np.ascontiguousarray(rhs2, dtype=np.float64)
    k = 0 if kind == "mixed" else 1
    assert rhs1.shape == (ninst, n) and rhs2.shape == (ninst, m if k == 0 else n)
    p1 = np.empty((ninst, n)); q1 = np.empty((ninst, m)); p2 = np.empty((ninst, n)); q2 = np.empty((ninst, m))
    fac = np.zeros(ninst, dtype=np.int32)
    check(_lib.lib().fpsb_batch_solve_two(C.c_int64(ninst), C.c_int(n), C.c_int(m), C.c_int(k), _ptr(A),
                                          C.c_double(delta), _ptr(rhs1), _ptr(rhs2), _ptr(p1), _ptr(q1),
                                          _ptr(p2), _ptr(q2), _ptr(fac),
                                          C.byref(opts) if opts is not None else None, C.c_int(FPSB_HOST),
                                          C.c_int(device)), "fpsb_batch_solve_two")
    return p1, q1, p2, q2, fac.astype(bool)
