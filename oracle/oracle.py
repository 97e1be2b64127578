"""ctypes binding of oracle/libfps_oracle.so — the CPU restatement of the reference hot path.

TEST INFRASTRUCTURE ONLY (see oracle/fps_oracle.c header).  Functions mirror the reference's
plugin surface for the path:

    IterativeOracle.solve_two_mixed / solve_two_least_squares / solve_two_extras
        -> /root/reference/src/solve_linear_system.jl:45-140
    LDLtOracle.solve_two_mixed / solve_two_least_squares / solve_two_extras
        -> /root/reference/src/solve_linear_system.jl:142-252
    ldl_analyze / ldl_factorize / ldl_solve2  -> LDLFactorizations.jl (SURVEY App. B1-B3)
    lsqr / craig / minres_normal / cgls       -> Krylov.jl 0.10      (SURVEY App. B5)

Parity status: pinned on the reference's own known-answer tests (tests/golden/), not on the real
Julia packages (no Julia in this image) — "parity unpinned" at the bit level.
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfps_oracle.so")

SQRT_EPS = float(np.sqrt(np.finfo(np.float64).eps))

STATUS = {0: "unknown", 1: "x = 0 is a zero-residual solution", 2: "solved", 3: "zero residual",
          4: "forward error small", 5: "maximum number of iterations exceeded",
          6: "ill-conditioned (machine)", 7: "ill-conditioned (conlim)", 8: "inconsistent",
          9: "x = 0 is a minimum least-squares solution"}


def build(force=False):
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(
            os.path.join(_HERE, "fps_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libfps_oracle.so"],
                              stdout=subprocess.DEVNULL)
    return _SO


class Stats(C.Structure):
    _fields_ = [("niter", C.c_int64), ("solved", C.c_int32), ("inconsistent", C.c_int32),
                ("status", C.c_int32), ("pad", C.c_int32), ("rnorm", C.c_double),
                ("arnorm", C.c_double), ("anorm", C.c_double), ("acond", C.c_double),
                ("xnorm", C.c_double)]

    def as_dict(self):
        return dict(niter=int(self.niter), solved=bool(self.solved),
                    inconsistent=bool(self.inconsistent), status=int(self.status),
                    rnorm=self.rnorm, arnorm=self.arnorm, anorm=self.anorm, acond=self.acond,
                    xnorm=self.xnorm)


class IterTol(C.Structure):
    _fields_ = [("ls_atol", C.c_double), ("ls_rtol", C.c_double), ("ls_itmax", C.c_int64),
                ("ln_atol", C.c_double), ("ln_rtol", C.c_double), ("ln_btol", C.c_double),
                ("ln_conlim", C.c_double), ("ln_itmax", C.c_int64),
                ("ne_atol", C.c_double), ("ne_rtol", C.c_double), ("ne_etol", C.c_double),
                ("ne_conlim", C.c_double), ("ne_itmax", C.c_int64)]


_lib = None


def _threaded_so():
    """libfps_oracle_omp.so (-fopenmp -DFO_OMP): only bench.py's reference arm asks for it (FPS_ORACLE_OMP=1);
    falls back to the sequential build when OpenMP is not available."""
    so = os.path.join(_HERE, "libfps_oracle_omp.so")
    src = os.path.join(_HERE, "fps_oracle.c")
    try:
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", _HERE, "-B", "libfps_oracle_omp.so"], stdout=subprocess.DEVNULL,
                                  stderr=subprocess.DEVNULL)
        C.CDLL(so)
        return so
    except (OSError, subprocess.CalledProcessError):
        return None


THREADED = False


def lib():
    global _lib, THREADED
    if _lib is None:
        build()
        so = _SO
        if os.environ.get("FPS_ORACLE_OMP", "0") not in ("", "0"):
            t = _threaded_so()
            if t is not None:
                so, THREADED = t, True
        _lib = C.CDLL(so)
        _lib.fo_ldl_analyze.restype = C.c_void_p
        _lib.fo_ldlt_create.restype = C.c_void_p
        _lib.fo_ldlt_str.restype = C.c_void_p
        _lib.fo_ldl_n.restype = C.c_int64
        _lib.fo_ldl_lnz.restype = C.c_int64
        _lib.fo_coo_to_csc.restype = C.c_int64
        _lib.fo_ldlt_check_factor.restype = C.c_double
        _lib.fo_ldlt_check_solve.restype = C.c_double
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def coo_to_csc(N, I, J, V):
    """sparse(I, J, V, N, N) — 0-based."""
    I, J, V = _i64(I), _i64(J), _f64(V)
    nz = len(I)
    Cp = np.zeros(N + 1, np.int64)
    Ci = np.zeros(max(nz, 1), np.int64)
    Cx = np.zeros(max(nz, 1), np.float64)
    slot = np.zeros(max(nz, 1), np.int64)
    nnz = lib().fo_coo_to_csc(C.c_int64(N), C.c_int64(nz), _p(I), _p(J), _p(V), _p(Cp), _p(Ci),
                              _p(Cx), _p(slot))
    return Cp, Ci[:nnz].copy(), Cx[:nnz].copy(), slot[:nz].copy()


class LDL:
    """LDLFactorization object: ldl_analyze + ldl_factorize! + ldiv!."""

    def __init__(self, n, Ap, Ai, P=None):
        self.n = n
        self.Ap, self.Ai = _i64(Ap), _i64(Ai)
        Pa = _i64(P) if P is not None else None
        self.h = C.c_void_p(lib().fo_ldl_analyze(C.c_int64(n), _p(self.Ap), _p(self.Ai), _p(Pa)))
        self.own = True

    def set_reg(self, n_d, tol, r1, r2):
        lib().fo_ldl_set_reg(self.h, C.c_int64(n_d), C.c_double(tol), C.c_double(r1), C.c_double(r2))

    def factorize(self, Ax):
        Ax = _f64(Ax)
        return bool(lib().fo_ldl_factorize(self.h, _p(self.Ap), _p(self.Ai), _p(Ax)))

    def solve2(self, B):
        """B: (n, 2) array; returns solution (n, 2)."""
        Bf = np.asfortranarray(B, dtype=np.float64).copy(order="F")
        lib().fo_ldl_solve2(self.h, _p(Bf))
        return Bf

    def symbolic(self):
        n = self.n
        lnz = lib().fo_ldl_lnz(self.h)
        P = np.zeros(n, np.int64); parent = np.zeros(n, np.int64); Lnz = np.zeros(n, np.int64)
        Lp = np.zeros(n + 1, np.int64); Li = np.zeros(max(lnz, 1), np.int64)
        lib().fo_ldl_get_symbolic(self.h, _p(P), _p(parent), _p(Lnz), _p(Lp), _p(Li))
        return dict(P=P, parent=parent, Lnz=Lnz, Lp=Lp, Li=Li[:lnz])

    def numeric(self):
        lnz = lib().fo_ldl_lnz(self.h)
        Lx = np.zeros(max(lnz, 1)); D = np.zeros(self.n)
        lib().fo_ldl_get_numeric(self.h, _p(Lx), _p(D))
        return Lx[:lnz], D

    def regularised(self):
        """Boolean mask (permuted order) of the pivots the last factorisation regularised."""
        reg = np.zeros(self.n, np.int8)
        lib().fo_ldl_get_regularised(self.h, _p(reg))
        return reg.astype(bool)

    def __del__(self):
        try:
            if self.own and self.h:
                lib().fo_ldl_free(self.h)
        except Exception:
            pass


class _Mat:
    """A (m x n) as CSR plus CSR of A' (both int64 / float64)."""

    def __init__(self, A):
        import scipy.sparse as sp
        A = sp.csr_matrix(A, dtype=np.float64)
        A.sort_indices()
        At = sp.csr_matrix(A.T)
        At.sort_indices()
        self.m, self.n = A.shape
        self.rp, self.ci, self.vx = _i64(A.indptr), _i64(A.indices), _f64(A.data)
        self.trp, self.tci, self.tvx = _i64(At.indptr), _i64(At.indices), _f64(At.data)

    def args(self):
        return (C.c_int64(self.m), C.c_int64(self.n), _p(self.rp), _p(self.ci), _p(self.vx),
                _p(self.trp), _p(self.tci), _p(self.tvx))


def lsqr(A, b, lam=0.0, atol=SQRT_EPS, rtol=SQRT_EPS, itmax=0, transpose=False, axtol=SQRT_EPS,
         btol=SQRT_EPS, etol=SQRT_EPS, conlim=1 / SQRT_EPS):
    """Krylov.lsqr on A (transpose=False) or A' (True); the defaults are the reference's call-site kwargs
    (axtol, btol, etol and conlim are Krylov.jl's defaults, which that call site does not override)."""
    M = _Mat(A); b = _f64(b)
    x = np.zeros(M.m if transpose else M.n); st = Stats()
    lib().fo_lsqr_full_csr(*M.args(), C.c_int(1 if transpose else 0), _p(b), C.c_double(lam),
                           C.c_double(atol), C.c_double(rtol), C.c_double(axtol), C.c_double(btol),
                           C.c_double(etol), C.c_double(conlim), C.c_int64(itmax), _p(x), C.byref(st))
    return x, st.as_dict()


def craig(A, b, delta=0.0, atol=SQRT_EPS, rtol=SQRT_EPS, btol=SQRT_EPS, conlim=1 / SQRT_EPS, itmax=0):
    """Krylov.craig! as called by solve_least_norm (M = (1/delta) I, sqd = true when delta != 0)."""
    M = _Mat(A); b = _f64(b)
    x = np.zeros(M.n); y = np.zeros(M.m); st = Stats()
    sqd = 1 if delta != 0 else 0
    ms = 1.0 / delta if delta != 0 else 1.0
    lib().fo_craig_csr(*M.args(), C.c_int(0), _p(b), C.c_int(sqd), C.c_double(ms), C.c_double(atol),
                       C.c_double(rtol), C.c_double(btol), C.c_double(conlim), C.c_int64(itmax),
                       _p(x), _p(y), C.byref(st))
    return x, y, st.as_dict()


def minres_normal(A, b, lam, atol=SQRT_EPS / 100, rtol=SQRT_EPS / 100, etol=SQRT_EPS,
                  conlim=1 / SQRT_EPS, itmax=0):
    """Krylov.minres on the operator A*A' with shift lam."""
    M = _Mat(A); b = _f64(b)
    x = np.zeros(M.m); st = Stats()
    lib().fo_minres_normal_csr(*M.args(), _p(b), C.c_double(lam), C.c_double(atol), C.c_double(rtol),
                               C.c_double(etol), C.c_double(conlim), C.c_int64(itmax), _p(x),
                               C.byref(st))
    return x, st.as_dict()


def cgls(A, b, lam=0.0, atol=SQRT_EPS, rtol=SQRT_EPS, itmax=0, transpose=False):
    M = _Mat(A); b = _f64(b)
    x = np.zeros(M.m if transpose else M.n); st = Stats()
    lib().fo_cgls_csr(*M.args(), C.c_int(1 if transpose else 0), _p(b), C.c_double(lam),
                      C.c_double(atol), C.c_double(rtol), C.c_int64(itmax), _p(x), C.byref(st))
    return x, st.as_dict()


class IterativeOracle:
    """IterativeSolver + its three solve_two_* methods (reference defaults)."""

    def __init__(self, A, **kw):
        self.M = _Mat(A)
        self.tol = IterTol()
        lib().fo_itertol_defaults(C.byref(self.tol), C.c_int64(self.M.n), C.c_int64(self.M.m))
        for k, v in kw.items():
            setattr(self.tol, k, v)

    def solve_two_mixed(self, delta, rhs1, rhs2):
        M = self.M; rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        p1 = np.zeros(M.n); q1 = np.zeros(M.m); p2 = np.zeros(M.n); q2 = np.zeros(M.m)
        st = (Stats * 2)()
        lib().fo_iter_solve_two_mixed(*M.args(), C.byref(self.tol), C.c_double(delta), _p(rhs1),
                                      _p(rhs2), _p(p1), _p(q1), _p(p2), _p(q2), st)
        return p1, q1, p2, q2, [st[0].as_dict(), st[1].as_dict()]

    def solve_two_least_squares(self, delta, rhs1, rhs2):
        M = self.M; rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        p1 = np.zeros(M.n); q1 = np.zeros(M.m); p2 = np.zeros(M.n); q2 = np.zeros(M.m)
        st = (Stats * 2)()
        lib().fo_iter_solve_two_least_squares(*M.args(), C.byref(self.tol), C.c_double(delta),
                                              _p(rhs1), _p(rhs2), _p(p1), _p(q1), _p(p2), _p(q2), st)
        return p1, q1, p2, q2, [st[0].as_dict(), st[1].as_dict()]

    def solve_two_extras(self, delta, rhs1, rhs2):
        M = self.M; rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        u1 = np.zeros(M.m); u2 = np.zeros(M.m)
        st = (Stats * 2)()
        lib().fo_iter_solve_two_extras(*M.args(), C.byref(self.tol), C.c_double(delta), _p(rhs1),
                                       _p(rhs2), _p(u1), _p(u2), st)
        return u1, u2, [st[0].as_dict(), st[1].as_dict()]


class LDLtOracle:
    """LDLtSolver + its three solve_two_* methods.

    jrow/jcol: 0-based COO structure of the Jacobian (what jac_structure! returns, minus 1).
    P: permutation (0-based, P[k] = index eliminated k-th) — ldl_analyze(A, P); the reference's
    default P = amd(K) comes from SuiteSparse, absent here, so P is always supplied explicitly.
    """

    def __init__(self, nvar, ncon, jrow, jcol, P, ldlt_tol=SQRT_EPS, ldlt_r1=SQRT_EPS,
                 ldlt_r2=-SQRT_EPS):
        self.nvar, self.ncon = nvar, ncon
        self.jrow, self.jcol = _i64(jrow), _i64(jcol)
        self.nnzj = len(self.jrow)
        P = _i64(P)
        self.h = C.c_void_p(lib().fo_ldlt_create(
            C.c_int64(nvar), C.c_int64(ncon), C.c_int64(self.nnzj), _p(self.jrow), _p(self.jcol),
            _p(P), C.c_double(ldlt_tol), C.c_double(ldlt_r1), C.c_double(ldlt_r2)))
        self.jvals = None

    def _str(self):
        s = LDL.__new__(LDL)
        s.n = self.nvar + self.ncon
        s.h = C.c_void_p(lib().fo_ldlt_str(self.h))
        s.own = False
        return s

    def symbolic(self):
        return self._str().symbolic()

    def numeric(self):
        return self._str().numeric()

    def regularised(self):
        return self._str().regularised()

    def check_factor(self, Lx, D, reg=None):
        """Per-entry error-model check of a factor L^, D^ in this oracle's CSC layout against K as the last
        solve_two_mixed assembled it, in long double: max over the pattern of L (diagonal included, the diagonals of
        the `reg` pivots skipped) of |(P K P' - L^ D^ L^')_ij| / ((c_ij + 4) 2^-53 (|L^| |D^| |L^'|)_ij), c_ij the
        number of k < j with L(i,k) L(j,k) structurally nonzero.  Returns dict(ratio, where, bound, dpre): `where`
        indexes [Lx | D], `bound` holds every denominator, `dpre` the pivots before regularisation."""
        Lx, D = _f64(Lx), _f64(D)
        N = self.nvar + self.ncon
        reg = None if reg is None else np.ascontiguousarray(reg, dtype=np.int8)
        bound = np.zeros(len(Lx) + N); dpre = np.zeros(N); where = C.c_int64(-1)
        r = lib().fo_ldlt_check_factor(self.h, _p(Lx), _p(D), _p(reg), C.byref(where), _p(bound), _p(dpre))
        return dict(ratio=r, where=where.value, bound=bound, dpre=dpre)

    def check_solve(self, Lx, D, x, b, reg=None):
        """Error-model check of a solution x^ = [p; q] of K x = b computed with L^, D^, in long double: max over i of
        |b - K~ x^|_i / ((3c + 10) 2^-53 (P' |L^| |D^| |L^'| P |x^|)_i), c the largest row or column count of L,
        K~ = K plus the pivot changes of the `reg` pivots.  Returns (ratio, i)."""
        Lx, D, x, b = _f64(Lx), _f64(D), _f64(x), _f64(b)
        reg = None if reg is None else np.ascontiguousarray(reg, dtype=np.int8)
        where = C.c_int64(-1)
        r = lib().fo_ldlt_check_solve(self.h, _p(Lx), _p(D), _p(reg), _p(x), _p(b), C.byref(where))
        return r, where.value

    def solve_two_mixed(self, jvals, delta, rhs1, rhs2):
        jvals, rhs1, rhs2 = _f64(jvals), _f64(rhs1), _f64(rhs2)
        self.jvals = jvals
        n, m = self.nvar, self.ncon
        p1 = np.zeros(n); q1 = np.zeros(m); p2 = np.zeros(n); q2 = np.zeros(m)
        ok = lib().fo_ldlt_solve_two_mixed(self.h, _p(jvals), C.c_double(delta), _p(rhs1), _p(rhs2),
                                           _p(p1), _p(q1), _p(p2), _p(q2))
        return p1, q1, p2, q2, bool(ok)

    def solve_two_least_squares(self, rhs1, rhs2):
        rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        n, m = self.nvar, self.ncon
        p1 = np.zeros(n); q1 = np.zeros(m); p2 = np.zeros(n); q2 = np.zeros(m)
        ok = lib().fo_ldlt_solve_two_least_squares(self.h, _p(rhs1), _p(rhs2), _p(p1), _p(q1),
                                                   _p(p2), _p(q2))
        return p1, q1, p2, q2, bool(ok)

    def solve_two_extras(self, delta, rhs1, rhs2):
        import scipy.sparse as sp
        A = sp.csr_matrix((self.jvals, (self.jrow, self.jcol)), shape=(self.ncon, self.nvar))
        M = _Mat(A); rhs1, rhs2 = _f64(rhs1), _f64(rhs2)
        u1 = np.zeros(M.m); u2 = np.zeros(M.m)
        st = (Stats * 2)()
        lib().fo_ldlt_solve_two_extras(*M.args(), C.c_double(delta), _p(rhs1), _p(rhs2), _p(u1),
                                       _p(u2), st)
        return u1, u2, [st[0].as_dict(), st[1].as_dict()]

    def __del__(self):
        try:
            lib().fo_ldlt_destroy(self.h)
        except Exception:
            pass
