"""fps_solve — the user entry of the reference, around the 2-RHS solves (SURVEY §8 a14, a17, f3, f4).

Mirror of `fps_solve` (src/FletcherPenaltySolver.jl:127-207), `AlgoData` / `GNSolver` / `FPSSSolver`
(src/parameters.jl:35-345), the outer penalty loop `SolverCore.solve!` (src/algo.jl:26-288) with its
parameter updates (:295-395) and the feasibility restoration `feasibility_step` / `TR_lsmr`
(src/feasibility.jl:21-235).  The surface is the reference's (same keyword names — the Greek ones are
accepted next to their ASCII spellings —, same defaults, same status symbols); none of it is
accelerated: every flop of weight happens in `solve_two_*` -> libfpsb200.so, which this loop drives
through `FletcherPenaltyNLP` (host buffers) or `DeviceFletcherPenaltyNLP` (vectors resident in HBM).

Two pieces of the reference are third-party programs that cannot be restated here:
  * Stopping.jl's `NLPStopping` — `_Stopping` below keeps the part `algo.jl` reads (start!/stop!, the
    optimal / suboptimal / unbounded / tired / iteration_limit / stalled / fail_sub_pb flags, nb_of_stop,
    `status_stopping_to_stats`);
  * the subproblem solver (`ipopt` by default, `tron`/`trunk`/`lbfgs`/`R2`/`knitro` by keyword,
    src/parameters.jl:199-206).  Here it is `trunk`: a matrix-free trust-region Newton method with a
    Steihaug–Toint CG (the method of JSOSolvers' TrunkSolver), written on `obj/grad/hprod` only so that it
    runs unchanged on numpy arrays and on device tensors (SURVEY §8 f3); with bounds it works on the free
    variables and projects (the role `tron` plays in the reference).
All vector arithmetic goes through the small `_V` helpers, which accept numpy arrays and torch tensors.
"""
import math
import os
import time
import warnings

import numpy as np

from .fletcher_nlp import FletcherPenaltyNLP
from .qdsolver import QDSolver, qdsolver_correspondence

EPS = float(np.finfo(np.float64).eps)
SQRT_EPS = math.sqrt(EPS)


# --------------------------------------------------------------------------------------------------
# array helpers (numpy arrays or torch tensors)
# --------------------------------------------------------------------------------------------------
class _V:
    @staticmethod
    def dot(a, b):
        return float(a @ b) if len(a) else 0.0

    @staticmethod
    def norm(a):
        return math.sqrt(max(_V.dot(a, a), 0.0))

    @staticmethod
    def ninf(a):
        return float(abs(a).max()) if len(a) else 0.0

    @staticmethod
    def copy(a):
        return a.clone() if hasattr(a, "clone") else np.array(a, dtype=np.float64, copy=True)

    @staticmethod
    def host(a):
        return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a, dtype=np.float64)

    @staticmethod
    def like(a, values):
        """`values` (host array) in the container type of `a`."""
        if hasattr(a, "detach"):
            import torch
            return torch.as_tensor(np.asarray(values, dtype=np.float64), device=a.device)
        return np.asarray(values, dtype=np.float64)

    @staticmethod
    def zeros_like(a):
        return a * 0.0

    @staticmethod
    def equal(a, b):
        return bool((a == b).all())

    @staticmethod
    def maximum(a, b):
        if hasattr(a, "detach"):
            import torch
            return torch.maximum(a, b)
        return np.maximum(a, b)

    @staticmethod
    def clip(a, lo, hi):
        if hasattr(a, "detach"):
            import torch
            return torch.maximum(torch.minimum(a, hi), lo)
        return np.maximum(np.minimum(a, hi), lo)


# --------------------------------------------------------------------------------------------------
# parameters (src/parameters.jl)
# --------------------------------------------------------------------------------------------------
_GREEK = {"σ_0": "sigma_0", "σ_max": "sigma_max", "σ_update": "sigma_update", "ρ_0": "rho_0",
          "ρ_max": "rho_max", "ρ_update": "rho_update", "δ_0": "delta_0", "δ_max": "delta_max",
          "δ_update": "delta_update", "η_1": "eta_1", "η_update": "eta_update", "Δ": "Delta"}


def _ascii_kwargs(kw):
    return {_GREEK.get(k, k): v for k, v in kw.items()}


class AlgoData:
    """AlgoData(; kwargs...)  (src/parameters.jl:35-121) — defaults for T = Float64."""

    def __init__(self, *, sigma_0=1e3, sigma_max=1 / SQRT_EPS, sigma_update=2.0, rho_0=1.0,
                 rho_max=1 / SQRT_EPS, rho_update=2.0, delta_0=SQRT_EPS, delta_max=1 / SQRT_EPS,
                 delta_update=10.0, eta_1=0.0, eta_update=1.0, yM=float("inf"), Delta=0.95,
                 subproblem_solver="trunk", subpb_unbounded_threshold=1 / SQRT_EPS,
                 subsolver_max_iter=20000, atol_sub=lambda atol: atol, rtol_sub=lambda rtol: rtol,
                 hessian_approx=2, explicit_linear_constraints=False, convex_subproblem=False,
                 lagrange_bound=1 / SQRT_EPS, refresh_memo_on_update=False, **kwargs):
        self.sigma_0, self.sigma_max, self.sigma_update = sigma_0, sigma_max, sigma_update
        self.rho_0, self.rho_max, self.rho_update = rho_0, rho_max, rho_update
        self.delta_0, self.delta_max, self.delta_update = delta_0, delta_max, delta_update
        self.eta_1, self.eta_update, self.yM, self.Delta = eta_1, eta_update, yM, Delta
        self.subproblem_solver = subproblem_solver
        self.subpb_unbounded_threshold = subpb_unbounded_threshold
        self.subsolver_max_iter = subsolver_max_iter
        self.atol_sub, self.rtol_sub = atol_sub, rtol_sub
        self.hessian_approx = hessian_approx
        self.explicit_linear_constraints = explicit_linear_constraints
        self.convex_subproblem = convex_subproblem
        self.lagrange_bound = lagrange_bound
        # Not a reference option.  False (default) = the reference: the memo of FletcherPenaltyNLP is keyed on hash(x)
        # only (SURVEY App. D-1), so right after a sigma / rho / delta update the first evaluation at the unchanged x
        # still returns ys / gs of the OLD parameters.  True drops the memo when the parameters change.
        self.refresh_memo_on_update = refresh_memo_on_update


class GNSolver:
    """GNSolver(x, y; kwargs...)  (src/parameters.jl:143-195): parameters of the feasibility step."""

    def __init__(self, x0=None, y0=None, *, eta1=1e-3, eta2=0.66, sigma1=0.25, sigma2=2.0, Delta0=1.0,
                 bad_steps_lim=3, feas_expected_decrease=0.95, fused=False):
        self.eta1, self.eta2, self.sigma1, self.sigma2, self.Delta0 = eta1, eta2, sigma1, sigma2, Delta0
        self.bad_steps_lim = bad_steps_lim
        self.feas_expected_decrease = feas_expected_decrease
        # not a reference option: compute the normal steps with the QDSolver's fused kernels (TR_fused) instead of the
        # host-loop LSMR (TR_lsmr).  Off by default: LSMR's truncated iterate and the scaled minimum-norm step are both
        # valid trust-region steps but not the same vector, and the reference's is LSMR's.
        self.fused = fused


class GenericExecutionStats:
    """The fields of SolverCore's GenericExecutionStats that src/algo.jl:269-282 sets."""

    def __init__(self, nlp=None):
        self.reset()

    def reset(self):
        self.status = "unknown"
        self.solution = None
        self.objective = float("inf")
        self.primal_feas = float("inf")
        self.dual_feas = float("inf")
        self.multipliers = None
        self.multipliers_L = None
        self.multipliers_U = None
        self.iter = -1
        self.elapsed_time = float("inf")
        self.solver_specific = {}

    def __repr__(self):
        return f"Execution stats: {self.status} (iter={self.iter}, f={self.objective:.6e}, " \
               f"primal={self.primal_feas:.2e}, dual={self.dual_feas:.2e})"


# --------------------------------------------------------------------------------------------------
# what algo.jl reads of Stopping.jl
# --------------------------------------------------------------------------------------------------
_STATUS_ORDER = (("optimal", "first_order"), ("fail_sub_pb", "unknown"), ("suboptimal", "acceptable"),
                 ("unbounded", "unbounded"), ("unbounded_pb", "unbounded"), ("stalled", "stalled"),
                 ("iteration_limit", "max_iter"), ("tired", "max_time"), ("resources", "max_eval"),
                 ("infeasible", "infeasible"), ("stopbyuser", "user"), ("domainerror", "exception"))


class _Meta:
    FLAGS = tuple(f for f, _ in _STATUS_ORDER)

    def __init__(self, atol, rtol, max_iter=5000, max_time=300.0, max_eval=20000,
                 unbounded_threshold=1e50, unbounded_x=1e50):
        self.atol, self.rtol = atol, rtol
        self.max_iter, self.max_time, self.max_eval = max_iter, max_time, max_eval
        self.unbounded_threshold, self.unbounded_x = unbounded_threshold, unbounded_x
        self.nb_of_stop = 0
        self.start_time = float("nan")
        self.optimality0 = 1.0
        self.clear()

    def clear(self):
        for f in self.FLAGS:
            setattr(self, f, False)


class _State:
    def __init__(self, x, ncon):
        self.x = x
        self.fx = float("nan")
        self.gx = None
        self.cx = None
        self.res = None
        self.lam = None          # `lambda` in the reference
        self.mu = None
        self.current_score = None
        self.current_time = float("nan")


class _Stopping:
    """NLPStopping of the main problem with `Fletcher_penalty_optimality_check`
    (src/FletcherPenaltySolver.jl:28-50) and the tolerance vector `Fptc` (src/parameters.jl:267-268)."""

    def __init__(self, pb, x0, cx0, gx0, atol=1e-7, rtol=1e-7, **kw):
        self.pb = pb
        allowed = {k: v for k, v in kw.items() if k in ("max_iter", "max_time", "max_eval",
                                                        "unbounded_threshold", "unbounded_x")}
        self.meta = _Meta(atol, rtol, **allowed)
        st = _State(_V.copy(x0), pb.meta.ncon)
        st.cx, st.gx, st.res = cx0, gx0, gx0
        st.lam = _V.zeros_like(cx0)
        self.current_state = st
        self._c0, self._g0 = _V.ninf(cx0), _V.ninf(gx0)
        lv, uv = np.asarray(pb.meta.lvar), np.asarray(pb.meta.uvar)
        self.has_bounds = bool(np.any(lv > -np.inf) or np.any(uv < np.inf))
        self._lcon, self._ucon = _V.like(cx0, pb.meta.lcon), _V.like(cx0, pb.meta.ucon)
        if self.has_bounds:
            self._lvar, self._uvar = _V.like(x0, lv), _V.like(x0, uv)

    def tol_check(self):
        return self.meta.rtol * (1.0 + self._c0), self.meta.rtol * (1.0 + self._g0)

    def score(self):
        st = self.current_state
        nxk = max(_V.norm(st.x), 1.0)
        nlk = 1.0 if st.lam is None else max(_V.norm(st.lam), 1.0)
        c = st.cx
        # max.(cx .- ucon, lcon .- cx, 0) ./ max(‖x‖, 1)
        cpart = _V.maximum(_V.maximum(c - self._ucon, self._lcon - c), c * 0.0) / nxk if len(c) else c
        if self.has_bounds:
            rpart = st.x - _V.clip(st.x - st.res, self._lvar, self._uvar)
        else:
            rpart = st.res / nlk
        st.current_score = (cpart, rpart)
        return st.current_score

    def _check(self):
        st, m = self.current_state, self.meta
        cpart, rpart = self.score()
        sc, sr = _V.ninf(cpart), _V.ninf(rpart)
        tc, tr = self.tol_check()
        if math.isnan(sc) or math.isnan(sr):
            m.domainerror = True
        m.optimal = (sc <= tc) and (sr <= tr)
        st.current_time = time.time()
        if st.current_time - m.start_time > m.max_time:
            m.tired = True
        if m.nb_of_stop > m.max_iter:
            m.iteration_limit = True
        if not math.isnan(st.fx) and st.fx <= -m.unbounded_threshold:
            m.unbounded_pb = True
        if _V.norm(st.x) >= m.unbounded_x:
            m.unbounded = True
        c = getattr(self.pb, "counters", None)
        if c is not None and (c.neval_obj > m.max_eval or c.neval_cons > m.max_eval):
            m.resources = True
        return any(getattr(m, f) for f in m.FLAGS)

    def start(self):
        self.meta.start_time = time.time()
        self.meta.nb_of_stop = 0
        self.meta.clear()
        cpart, rpart = self.score()
        self.meta.optimality0 = max(_V.ninf(cpart), _V.ninf(rpart))
        return self._check()

    def stop(self):
        self.meta.nb_of_stop += 1
        return self._check()

    def status(self):
        for flag, sym in _STATUS_ORDER:
            if getattr(self.meta, flag):
                return sym
        return "unknown"


# --------------------------------------------------------------------------------------------------
# subproblem solver: trust-region Newton-CG on obj / grad / hprod
# --------------------------------------------------------------------------------------------------
class SubStats:
    """What `sub_stp` tells the outer loop (src/algo.jl:118-165)."""

    def __init__(self):
        self.optimal = self.suboptimal = self.unbounded = self.unbounded_pb = False
        self.tired = self.resources = self.iteration_limit = self.stalled = False
        self.x = None
        self.fx = float("nan")
        self.gx = None
        self.lam = self.res = None       # explicit linear constraints: their multipliers and g + A'lam
        self.current_score = float("inf")
        self.iter = 0
        self.cg_iter = 0

    def status(self):
        for f in ("optimal", "suboptimal", "unbounded", "unbounded_pb", "stalled", "iteration_limit",
                  "tired", "resources"):
            if getattr(self, f):
                return f
        return "unknown"


def _steihaug(hv, g, radius, tol, itmax, free=None):
    """Steihaug–Toint truncated CG for  min g's + s'Hs/2, ‖s‖ ≤ radius  (on the `free` variables).
    Returns s, the model decrease −q(s) and the number of Hessian products."""
    s = _V.zeros_like(g)
    r = -g if free is None else -g * free
    d = _V.copy(r)
    rr = _V.dot(r, r)
    q = 0.0
    nprod = 0
    if math.sqrt(rr) <= tol:
        return s, 0.0, 0
    for _ in range(itmax):
        Hd = hv(d)
        if free is not None:
            Hd = Hd * free
        nprod += 1
        dHd = _V.dot(d, Hd)
        ss, sd, dd = _V.dot(s, s), _V.dot(s, d), _V.dot(d, d)
        # positive step to the boundary along d
        disc = max(sd * sd + dd * (radius * radius - ss), 0.0)
        to_boundary = (-sd + math.sqrt(disc)) / dd if dd > 0 else 0.0
        if dHd <= EPS * dd:                                   # negative / zero curvature
            q += to_boundary * (-_V.dot(r, d)) + 0.5 * to_boundary * to_boundary * dHd
            return s + to_boundary * d, -q, nprod
        alpha = rr / dHd
        if alpha >= to_boundary:
            q += to_boundary * (-_V.dot(r, d)) + 0.5 * to_boundary * to_boundary * dHd
            return s + to_boundary * d, -q, nprod
        q += alpha * (-_V.dot(r, d)) + 0.5 * alpha * alpha * dHd
        s = s + alpha * d
        r = r - alpha * Hd
        rr_new = _V.dot(r, r)
        if math.sqrt(rr_new) <= tol:
            return s, -q, nprod
        d = r + (rr_new / rr) * d
        rr = rr_new
    return s, -q, nprod


class _LinearRows:
    """The linear rows of `nlp` as a model of their own (what a QDSolver constructor reads: meta, jac_structure, jac_coord)."""

    def __init__(self, nlp):
        from .models import NLPModelMeta
        self.parent = nlp
        lin = list(nlp.meta.lin)
        self.meta = NLPModelMeta(nlp.meta.nvar, len(lin), x0=nlp.meta.x0, lcon=np.asarray(nlp.meta.lcon)[lin],
                                 ucon=np.asarray(nlp.meta.ucon)[lin], name=nlp.meta.name + "-linear-rows")
        self._rows, self._cols = nlp.jac_lin_structure()
        self.meta.nnzj = len(self._rows)

    def jac_structure(self):
        return self._rows, self._cols

    def jac_coord(self, x):
        return self.parent.jac_lin_coord(x)


class LinearConstraintProjector:
    """Null-space projections for the explicit linear constraints `A x = b` of the subproblem
    (`explicit_linear_constraints = true`, src/parameters.jl:290-309; in the reference the constraints are simply handed
    to ipopt / knitro).  Both operations are 2-RHS solves of the SAME kernel family as the penalty's own — a QDSolver
    on `[I A'; A 0]` with the constant linear rows:
        project(v)  = (I - A'(AA')^-1 A) v  and  (AA')^-1 A v          <- p1, q1 of solve_two_least_squares(v, v)
        correct(r)  = A'(AA')^-1 r   (minimum-norm d with A d = r)      <- p2 of solve_two_mixed(0, r)"""

    def __init__(self, nlp, qds_factory):
        self.rows = _LinearRows(nlp)
        self.nlp = self.rows                    # what solve_two_* read through `fpnlp.nlp`
        self.explicit_linear_constraints = False
        self.delta = 0.0
        self.qdsolver = qds_factory(self.rows)
        self.b = np.asarray(self.rows.meta.lcon, dtype=np.float64)
        self._ready = False
        self._x0 = np.asarray(nlp.meta.x0, dtype=np.float64)

    def _setup(self):
        if not self._ready:                     # values / factorisation of the constant rows: once
            from .qdsolver import solve_two_mixed
            n, m = self.rows.meta.nvar, self.rows.meta.ncon
            solve_two_mixed(self, self._x0, np.zeros(n), np.zeros(m))
            self._ready = True

    def residual(self, x):
        return self.rows.parent.cons_lin(x) - self.b

    def project(self, v):
        from .qdsolver import solve_two_least_squares
        self._setup()
        p1, q1, _, _ = solve_two_least_squares(self, self._x0, v, v)
        return np.array(p1, copy=True), np.array(q1, copy=True)

    def correct(self, r):
        from .qdsolver import solve_two_mixed
        n = self.rows.meta.nvar
        _, _, p2, _ = solve_two_mixed(self, self._x0, np.zeros(n), np.asarray(r, dtype=np.float64))
        self._ready = True
        return np.array(p2, copy=True)


def _steihaug_device(handle, hv, g, radius, tol, itmax, free=None):
    """`_steihaug` with the CG state resident in HBM (SURVEY §8 f3): s, r, d are device vectors, the five inner products
    of an iteration, the step to the boundary, alpha, beta, the model decrease and the exit decision are computed by the
    fused kernels behind fpsb_trcg_init / fpsb_trcg_step; the host reads five doubles per iteration (one synchronisation
    instead of six) and only supplies Hd = hv(d), i.e. the model's 2-RHS solves."""
    import ctypes as C
    import torch
    from . import _lib
    L = _lib.lib()
    handle._follow_torch_stream(g)
    s, r, d = torch.empty_like(g), torch.empty_like(g), torch.empty_like(g)
    out = (C.c_double * 5)()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    fr = None if free is None else free.to(torch.float64).contiguous()
    _lib.check(L.fpsb_trcg_init(handle.h, p(g), p(fr), p(s), p(r), p(d), out), "fpsb_trcg_init")
    if math.sqrt(max(out[0], 0.0)) <= tol:
        return s, 0.0, 0
    nprod = 0
    for _ in range(itmax):
        Hd = hv(d)
        nprod += 1
        handle._follow_torch_stream(Hd)
        _lib.check(L.fpsb_trcg_step(handle.h, p(Hd), p(fr), p(s), p(r), p(d), C.c_double(radius), C.c_double(tol), out),
                   "fpsb_trcg_step")
        if out[4] != 0.0:
            break
    return s, -out[1], nprod


def _steihaug_batch(handle, hv, G, radius, tol, itmax, free=None):
    """`_steihaug_device` for K subproblems in lock-step: instance i is  min G[i]'s + s'H_i s/2, ‖s‖ ≤ radius[i], and
    `hv(D)` returns the K products H_i D[i] as one (K, n) tensor (one batched `hprod`).  radius and tol are scalars or
    (K,); free is None or (K, n).  Each instance runs inside one CTA of fpsb_trcg_batch_step; an instance that has left
    (boundary, negative curvature, converged) is frozen while the others keep going, and its rows of the later products
    are computed with the batch and discarded, so `hv` always sees the full batch.  The host reads one 4-byte count of
    active instances per iteration.  Returns S (K, n), pred (K,) (the model decrease −q), nprod (K,) int32 and the exit
    flags (K,): 0 itmax reached, 1 left through the boundary or met non-positive curvature, 2 converged (also for a
    gradient with ‖g‖ ≤ tol, with no product)."""
    import ctypes as C
    import torch
    from . import _lib
    L = _lib.lib()
    if G.ndim != 2 or G.shape[1] != handle.nvar:
        raise ValueError(f"_steihaug_batch: G must be (K, {handle.nvar})")
    K = int(G.shape[0])
    G = G.to(torch.float64).contiguous()
    f64 = dict(dtype=torch.float64, device=G.device)
    per = lambda a: torch.as_tensor(a, **f64).expand(K).contiguous()
    rad, tl = per(radius), per(tol)
    fr = None if free is None else free.to(torch.float64).contiguous()
    if fr is not None and tuple(fr.shape) != tuple(G.shape):
        raise ValueError("_steihaug_batch: free must have the shape of G")
    S, R, D = torch.empty_like(G), torch.empty_like(G), torch.empty_like(G)
    st = torch.zeros((K, 5), **f64)
    nprod = torch.zeros(K, dtype=torch.int32, device=G.device)
    if K == 0:
        return S, st[:, 1], nprod, st[:, 4]
    handle._follow_torch_stream(G)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    nact = C.c_int32()
    _lib.check(L.fpsb_trcg_batch_init(handle.h, C.c_int64(K), p(G), p(fr), p(tl), p(S), p(R), p(D), p(st), p(nprod),
                                      C.byref(nact)), "fpsb_trcg_batch_init")
    it = 0
    while nact.value > 0 and it < itmax:
        Hd = hv(D).to(torch.float64).contiguous()
        it += 1
        handle._follow_torch_stream(Hd)
        _lib.check(L.fpsb_trcg_batch_step(handle.h, C.c_int64(K), p(Hd), p(fr), p(rad), p(tl), p(S), p(R), p(D), p(st),
                                          p(nprod), C.byref(nact)), "fpsb_trcg_batch_step")
    return S, -st[:, 1], nprod, st[:, 4].clone()


def _cg_solver_for(model, g):
    """The device-resident CG when the iterate lives on the GPU and the model owns a libfpsb200 handle, else the host loop."""
    h = getattr(model, "handle", None)
    if h is not None and hasattr(g, "is_cuda") and g.is_cuda and os.environ.get("FPSB_TRCG_HOST", "0") != "1":
        return lambda hv, g_, radius, tol, itmax, free: _steihaug_device(h, hv, g_, radius, tol, itmax, free)
    return _steihaug


def trunk(model, x0, *, atol=1e-7, rtol=1e-7, max_iter=20000, max_time=300.0, unbounded_threshold=1 / SQRT_EPS,
          lvar=None, uvar=None, verbose=0, stop_callback=None, lin=None):
    """Trust-region Newton-CG for  min φσ(x)  [l ≤ x ≤ u].  Optimality as Stopping's
    `unconstrained_check` / `optim_check_bounded`: ‖∇φσ‖∞ (projected) ≤ max(atol, rtol·score(x0)).
    `stop_callback(model, x)` may name a SubStats flag to leave with (the outer loop uses it to stop a
    subproblem whose multiplier estimate has blown up — the outer loop discards such a subproblem anyway,
    :118, :151 — once its steps have shrunk below 1e-6·‖x‖)."""
    t0 = time.time()
    out = SubStats()
    bounded = lvar is not None
    x = _V.copy(x0)
    if bounded:
        x = _V.clip(x, lvar, uvar)
    # `lin` (LinearConstraintProjector): linear equality constraints A x = b kept explicit in the subproblem.  The
    # iterates stay on the manifold (minimum-norm correction of the start, steps in the null space of A), the CG runs on
    # the projected Hessian P H P, optimality is the reduced gradient P g = g + A'lam with lam = -(AA')^-1 A g.
    lam = None
    if lin is not None:
        if bounded:
            raise NotImplementedError("explicit linear constraints together with bounds")
        x = x - lin.correct(lin.residual(x))
    f, g = model.objgrad(x)
    n = len(x)

    def pgrad(x, g):
        nonlocal lam
        if lin is not None:
            gp, q = lin.project(g)
            lam = -q
            return gp
        return x - _V.clip(x - g, lvar, uvar) if bounded else g

    gred = pgrad(x, g)                                        # the gradient the steps are computed from
    score = _V.ninf(gred)
    tol = max(atol, rtol * score)
    radius = min(max(0.1 * _V.norm(g), 1.0), 100.0)
    it = 0
    small_steps = noise_steps = 0
    tiny_step = False
    while True:
        out.current_score = score
        if math.isnan(score) or math.isnan(f):
            out.stalled = True
            break
        if score <= tol:
            out.optimal = True
            break
        if f <= -unbounded_threshold:
            out.unbounded_pb = True
            break
        # consulted only once the iteration has degenerated into tiny steps
        flag = stop_callback(model, x) if (stop_callback is not None and tiny_step) else None
        if flag:
            setattr(out, flag, True)
            break
        if it >= max_iter:
            out.iteration_limit = True
            break
        if time.time() - t0 > max_time:
            out.tired = True
            break
        free = None
        if bounded:
            act = ((x <= lvar) & (g > 0)) | ((x >= uvar) & (g < 0))
            free = (~act) * 1.0
        gcg = gred if lin is not None else g
        gn = _V.norm(gcg if free is None else gcg * free)
        cgtol = max(EPS, min(0.1, math.sqrt(gn)) * gn)
        hv = (lambda v: lin.project(model.hprod(x, v))[0]) if lin is not None else (lambda v: model.hprod(x, v))
        s, pred, nprod = _cg_solver_for(model, gcg)(hv, gcg, radius, cgtol, max(2 * n, 10), free)
        if lin is not None:
            s = lin.project(s)[0]                             # rounding drift out of the null space
        out.cg_iter += nprod
        if bounded:
            xt = _V.clip(x + s, lvar, uvar)
            if not _V.equal(xt, x + s):                       # the projection changed the step
                s = xt - x
                pred = -(_V.dot(g, s) + 0.5 * _V.dot(s, model.hprod(x, s)))
                if pred <= 0.0:                               # projected Cauchy step instead
                    s = _V.clip(x - (radius / max(_V.norm(g), EPS)) * g, lvar, uvar) - x
                    pred = -(_V.dot(g, s) + 0.5 * _V.dot(s, model.hprod(x, s)))
        else:
            xt = x + s
        snorm = _V.norm(s)
        tiny_step = snorm <= 1e-6 * max(1.0, _V.norm(x))
        # a model decrease below the rounding error of φσ itself cannot be verified: three in a row = stalled
        in_noise = pred <= 10 * EPS * max(1.0, abs(f))
        if not in_noise:
            noise_steps = 0
        ft = model.obj(xt)
        ared = f - ft
        gt = None
        # rounding guard of trust-region codes: tiny reductions are measured against the model
        if abs(ared) <= 10 * EPS * max(1.0, abs(f)) and abs(pred) <= 10 * EPS * max(1.0, abs(f)):
            rho = 1.0
        elif math.isnan(ft) or pred <= 0.0:
            rho = -1.0
        else:
            rho = ared / pred
        if rho < 1e-4 and pred > 0.0 and pred <= 1e3 * EPS * max(1.0, abs(f)) and not math.isnan(ft):
            # the function values are noise at this scale: measure the reduction with the slopes at both
            # ends, -(g + g⁺)'s / 2 (Conn, Gould & Toint §17.4.2); φσ(xt) is memoised, the gradient costs no solve
            gt = model.grad(xt)
            ared_g = -0.5 * _V.dot(g + gt, s)
            if not math.isnan(ared_g) and ared_g / pred >= 1e-4:
                rho = ared_g / pred
        if verbose:
            print(f"  trunk {it:4d} f={f: .6e} |g|={score:.2e} Δ={radius:.2e} |s|={snorm:.2e} ρ={rho: .2e} cg={nprod}")
        if rho >= 1e-4:
            x, f = xt, ft
            g = gt if gt is not None else model.grad(x)
            gred = pgrad(x, g)
            new_score = _V.ninf(gred)
            if in_noise:                                      # unverifiable step: a stall unless the gradient still drops
                noise_steps = 0 if new_score <= 0.9 * score else noise_steps + 1
            score = new_score
            if rho >= 0.99 and snorm >= 0.99 * radius:
                radius = min(3.0 * radius, 1e20)
            small_steps = small_steps + 1 if snorm <= EPS * max(1.0, _V.norm(x)) else 0
        else:
            radius = min(radius, snorm) / 3.0
            small_steps += 1 if radius <= EPS * max(1.0, _V.norm(x)) else 0
            noise_steps += 1 if in_noise else 0
        it += 1
        if small_steps >= 3 or noise_steps >= 3 or radius < 1e-300:
            out.stalled = True
            break
    # leave the model's memo (fx, cx, gx, ys — read by the outer loop, src/algo.jl:118-145) at x
    out.fx = model.obj(x)
    out.x, out.gx, out.iter = x, g, it
    out.lam, out.res = lam, (gred if lin is not None else g)  # multipliers of the explicit linear constraints, g + A'lam
    return out


subproblem_solver_correspondence = {"trunk": trunk, "tron": trunk}


# --------------------------------------------------------------------------------------------------
# feasibility restoration (src/feasibility.jl)
# --------------------------------------------------------------------------------------------------
def _lsmr_radius(Aprod, Atprod, b, n, radius, atol=SQRT_EPS, btol=SQRT_EPS, itmax=None):
    """LSMR (Fong & Saunders) for min ‖Ax − b‖ with the trust-region exit Krylov.jl's `radius` keyword adds:
    once ‖x‖ would leave the ball the last step is cut on the boundary.  Returns x, solved."""
    m = len(b)
    itmax = itmax or 2 * (m + n)
    u = _V.copy(b)
    beta = _V.norm(u)
    x = None
    if beta == 0.0:
        return _V.zeros_like(Atprod(u)), True
    u = u / beta
    v = Atprod(u)
    alpha = _V.norm(v)
    x = _V.zeros_like(v)
    if alpha == 0.0:
        return x, True
    v = v / alpha
    zetabar, alphabar, rho, rhobar, cbar, sbar = alpha * beta, alpha, 1.0, 1.0, 1.0, 0.0
    h, hbar = _V.copy(v), _V.zeros_like(v)
    normA2, normb = alpha * alpha, beta
    betadd, betad, rhodold, tautildeold, thetatilde, zeta, d = beta, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0
    for _ in range(itmax):
        u = Aprod(v) - alpha * u
        beta = _V.norm(u)
        if beta > 0.0:
            u = u / beta
            v = Atprod(u) - beta * v
            alpha = _V.norm(v)
            if alpha > 0.0:
                v = v / alpha
        rhoold = rho
        rho = math.hypot(alphabar, 0.0) if beta == 0.0 else math.hypot(alphabar, beta)
        c, s = alphabar / rho, beta / rho
        thetanew, alphabar = s * alpha, c * alpha
        rhobarold, zetaold = rhobar, zeta
        thetabar = sbar * rho
        rhotemp = cbar * rho
        rhobar = math.hypot(cbar * rho, thetanew)
        cbar, sbar = cbar * rho / rhobar, thetanew / rhobar
        zeta, zetabar = cbar * zetabar, -sbar * zetabar
        hbar = h - (thetabar * rho / (rhoold * rhobarold)) * hbar
        step = (zeta / (rho * rhobar)) * hbar
        xn = x + step
        if radius > 0.0 and _V.norm(xn) > radius:
            # cut on the boundary: largest t in [0, 1] with ‖x + t·step‖ = radius
            xx, xs, ss = _V.dot(x, x), _V.dot(x, step), _V.dot(step, step)
            t = (-xs + math.sqrt(max(xs * xs + ss * (radius * radius - xx), 0.0))) / ss if ss > 0 else 0.0
            return x + t * step, True
        x = xn
        h = v - (thetanew / rho) * h
        # residual estimates (for the stopping tests)
        betaacute, betacheck = c * betadd, -s * betadd
        betahat, betadd = c * betaacute, -s * betaacute
        thetatildeold = thetatilde
        rhotildeold = math.hypot(rhodold, thetabar)
        ctildeold, stildeold = rhodold / rhotildeold, thetabar / rhotildeold
        thetatilde, rhodold = stildeold * rhobar, ctildeold * rhobar
        betad = -stildeold * betad + ctildeold * betahat
        tautildeold = (zetaold - thetatildeold * tautildeold) / rhotildeold
        taud = (zeta - thetatilde * tautildeold) / rhodold
        d = d + betacheck * betacheck
        normr = math.sqrt(d + (betad - taud) ** 2 + betadd * betadd)
        normA2 += beta * beta
        normA = math.sqrt(normA2)
        normA2 += alpha * alpha
        normAr = abs(zetabar)
        normx = _V.norm(x)
        test1 = normr / normb
        test2 = normAr / (normA * normr) if normA * normr > 0 else float("inf")
        if test2 <= atol or test1 <= btol + atol * normA * normx / normb or 1 + test2 <= 1 or 1 + test1 <= 1:
            return x, True
    return x, False


def _cg(Hprod, b, rtol=SQRT_EPS, atol=SQRT_EPS, itmax=None):
    x = _V.zeros_like(b)
    r = _V.copy(b)
    p = _V.copy(r)
    rr = _V.dot(r, r)
    tol = atol + rtol * math.sqrt(rr)
    for _ in range(itmax or 2 * len(b)):
        if math.sqrt(rr) <= tol:
            return x, True
        Hp = Hprod(p)
        pHp = _V.dot(p, Hp)
        if pHp <= 0.0:
            return (x if _V.dot(x, x) > 0 else p), False
        a = rr / pHp
        x = x + a * p
        r = r - a * Hp
        rr_new = _V.dot(r, r)
        p = r + (rr_new / rr) * p
        rr = rr_new
    return x, math.sqrt(rr) <= tol


def TR_lsmr(nlp, z, cz, ctol, Delta, normcz):
    """d = argmin ‖c + J d‖, ‖d‖ ≤ Δ   (src/feasibility.jl:208-235)."""
    d, solved = _lsmr_radius(lambda v: nlp.jprod(z, v), lambda u: nlp.jtprod(z, u), -cz, nlp.meta.nvar, Delta)
    infeasible = _V.norm(d) < ctol * min(normcz, 1.0)
    if not solved:
        warnings.warn("Fail lsmr in TR_lsmr")
    return d, nlp.jprod(z, d), infeasible, solved


def TR_fused(qds, nlp, z, cz, ctol, Delta, normcz):
    """TR_lsmr's job on the fused Krylov kernels of libfpsb200 (SURVEY §8 f4): the Jacobian values at z go into the QDSolver's
    tiled operator, u = (JJ')⁻¹ c comes from the MINRES slot of `solve_two_extras` (Krylov path: the device-resident
    recurrences over the fused 2-column SpMM; LDLt path: one refactorisation), d = −J'u is the minimum-norm Gauss–Newton
    step, cut back to the trust-region boundary when it leaves the ball.  z, cz may be numpy arrays or device tensors."""
    from .qdsolver import IterativeSolver
    H = qds.handle
    H.set_jac_values(nlp.jac_coord(z))
    zero = _V.zeros_like(z)
    if isinstance(qds, IterativeSolver):
        _, u, st = H.iter_solve_two_extras(0.0, zero, cz)
        solved = bool(st[1]["solved"])
    else:
        _, u, _ = H.ldlt_solve_two_extras(0.0, zero, cz)
        solved = True
    d = -H.jtprod(u)
    nd = _V.norm(d)
    if Delta > 0.0 and nd > Delta:
        d = (Delta / nd) * d
        nd = Delta
    infeasible = nd < ctol * min(normcz, 1.0)
    if not solved:
        warnings.warn("Fail minres in TR_fused")
    return d, H.jprod(d), infeasible, solved


def feasibility_step(fs, nlp, x, cx, normcx, rho, ctol, verbose=0, *, max_eval=1000, max_time=60.0,
                     max_feas_iter=2 ** 62, qds=None):
    """Trust-region Levenberg–Marquardt on ‖c(x) − l‖   (src/feasibility.jl:21-189).
    `nlp` supplies cons / jprod / jtprod / hprod (the products run on whatever the model runs on)."""
    lcon = nlp.meta.lcon
    cons_norhs = lambda z: nlp.cons(z) - lcon
    z, cz, normcz = x, cx, normcx
    Delta = fs.Delta0
    feas_iter = consecutive_bad = 0
    failed_step_comp = infeasible = False
    nev = lambda: nlp.counters.neval_obj + nlp.counters.neval_cons
    t0 = time.time()
    tired = nev() > max_eval
    while not (normcz <= rho or tired or infeasible):
        if qds is not None and getattr(fs, "fused", False):
            d, Jd, infeasible, _ = TR_fused(qds, nlp, z, cz, ctol, Delta, normcz)
        else:
            d, Jd, infeasible, _ = TR_lsmr(nlp, z, cz, ctol, Delta, normcz)
        if infeasible:
            failed_step_comp = True
        else:
            zp = z + d
            czp = cons_norhs(zp)
            normczp = _V.norm(czp)
            Pred = 0.5 * (normcz ** 2 - _V.norm(Jd + cz) ** 2)
            Ared = 0.5 * (normcz ** 2 - normczp ** 2)
            if Pred <= 0.0 or Ared / Pred < fs.eta1:
                Delta = max(1e-8, Delta * fs.sigma1)
            else:
                consecutive_bad = consecutive_bad + 1 if normczp / normcz > fs.feas_expected_decrease else 0
                z, cz = zp, czp
                if Ared / Pred > fs.eta2 and _V.norm(d) >= 0.99 * Delta:
                    Delta *= fs.sigma2
                normcz = normczp
        if normcz > rho and (consecutive_bad >= fs.bad_steps_lim or failed_step_comp):
            # aggressive normal step: (H_c + J'J) d = J'c   (:117-144)
            Hop = lambda v: nlp.hprod(z, cz, v, obj_weight=0.0) + nlp.jtprod(z, nlp.jprod(z, v))
            d, solved = _cg(Hop, nlp.jtprod(z, cz))
            if not solved:
                warnings.warn("Fail cg in feasibility_step")
            zp = z - d
            czp = cons_norhs(zp)
            nczp = _V.norm(czp)
            if nczp < normcz:
                infeasible = failed_step_comp = False
                z, cz, normcz = zp, czp, nczp
            elif _V.norm(d) < ctol * min(nczp, 1.0):
                infeasible = True
        feas_iter += 1
        tired = nev() > max_eval or time.time() - t0 > max_time or feas_iter > max_feas_iter
    if normcz <= rho:
        status = "success"
    elif tired:
        status = "max_eval" if nev() > max_eval else ("max_time" if time.time() - t0 > max_time else "max_iter")
    elif infeasible:
        status = "infeasible"
    else:
        status = "unknown"
    return z, cz, normcz, status


# --------------------------------------------------------------------------------------------------
# FPSSSolver / fps_solve  (src/parameters.jl:231-345, src/FletcherPenaltySolver.jl:127-207)
# --------------------------------------------------------------------------------------------------
class FPSSSolver:
    """FPSSSolver(nlp [, x0]; qds_solver = :ldlt, kwargs...): every structure of one `fps_solve` call.

    `qds_solver` is a key of `qdsolver_correspondence` ("ldlt" | "iterative"), a QDSolver subtype or an
    instance; `model_factory(nlp, sigma, rho, delta, hessian_approx, qds=...)` builds the penalty model
    (`FletcherPenaltyNLP` by default, `DeviceFletcherPenaltyNLP` for the device-resident loop)."""

    def __init__(self, nlp, x0=None, *, qds_solver="ldlt", model_factory=None, **kwargs):
        kwargs = _ascii_kwargs(kwargs)
        self.kwargs = kwargs
        x0 = nlp.meta.x0 if x0 is None else x0
        self.meta = AlgoData(**kwargs)
        explicit = bool(self.meta.explicit_linear_constraints)
        if isinstance(qds_solver, QDSolver):
            self.qdsolver = qds_solver
            qds_cls = type(qds_solver)
        elif isinstance(qds_solver, type) or callable(qds_solver):
            self.qdsolver = qds_solver(nlp, 0.0, **kwargs)
            qds_cls = qds_solver
        else:
            qds_cls = qdsolver_correspondence[str(qds_solver).lstrip(":")]
            self.qdsolver = qds_cls(nlp, 0.0, **kwargs)
        self.feasibility_solver = GNSolver(fused=bool(kwargs.get("feas_fused", False)))
        factory = model_factory or FletcherPenaltyNLP
        model_kw = dict(qds=self.qdsolver, consistent_gradient=bool(kwargs.get("consistent_gradient", False)))
        if explicit:
            # the linear rows stay constraints of the subproblem (src/parameters.jl:300-309); here they are kept by
            # null-space projections that run on a second QDSolver of the same type (LinearConstraintProjector)
            if model_factory is not None:
                raise NotImplementedError("explicit_linear_constraints with a custom / device-resident model factory")
            model_kw["explicit_linear_constraints"] = True
        self.model = factory(nlp, self.meta.sigma_0, self.meta.rho_0, 0.0, self.meta.hessian_approx, **model_kw)
        self.lin_projector = None
        if explicit and nlp.meta.nlin > 0:
            if np.any(np.asarray(nlp.meta.lcon)[list(nlp.meta.lin)] != np.asarray(nlp.meta.ucon)[list(nlp.meta.lin)]):
                raise NotImplementedError("explicit linear constraints: equalities only (SlackModel turns the others into "
                                          "equalities with bounded slacks, which the projected subsolver does not handle)")
            lin_kw = {k: v for k, v in kwargs.items() if k != "explicit_linear_constraints"}
            self.lin_projector = LinearConstraintProjector(nlp, lambda rows: qds_cls(rows, 0.0, **lin_kw))
        self.subproblem_solver = self.meta.subproblem_solver if callable(self.meta.subproblem_solver) \
            else subproblem_solver_correspondence[str(self.meta.subproblem_solver)]
        self.sub_stats = None
        self._set_problem(nlp, x0)

    def _set_problem(self, nlp, x0):
        self.nlp = nlp
        x0 = _V.copy(x0)
        cx0, gx0 = nlp.cons(x0) if nlp.meta.ncon > 0 else _V.zeros_like(x0)[:0], nlp.grad(x0)
        stop_kw = {k: v for k, v in self.kwargs.items() if k in ("atol", "rtol", "max_iter", "max_time", "max_eval",
                                                                 "unbounded_threshold", "unbounded_x")}
        self.stp = _Stopping(nlp, x0, cx0, gx0, **stop_kw)

    def reset(self, nlp=None):
        """SolverCore.reset!(solver[, nlp])   (src/parameters.jl:347-362)."""
        if nlp is not None:
            assert nlp.meta.nvar == self.nlp.meta.nvar and nlp.meta.ncon == self.nlp.meta.ncon
            self.model.nlp = nlp
        self.model.shahx = 0
        self._set_problem(nlp or self.nlp, (nlp or self.nlp).meta.x0)
        return self


def _has_inequalities(nlp):
    return bool(np.any(np.asarray(nlp.meta.lcon) < np.asarray(nlp.meta.ucon)))


def fps_solve(nlp, x0=None, *, verbose=0, subsolver_verbose=0, callback=None, **kwargs):
    """stats = fps_solve(nlp, x0 = nlp.meta.x0; kwargs...)   (src/FletcherPenaltySolver.jl:127-186).

    Inequalities are turned into equalities + bounded slacks first (NLPModelsModifiers.SlackModel in the
    reference, `models.SlackModel` here) and the statistics are cut back to the original variables."""
    if not nlp.meta.minimize:
        raise ValueError("fps_solve only works for minimization problem")
    x0 = nlp.meta.x0 if x0 is None else x0
    ineq = _has_inequalities(nlp)
    orig = nlp
    if ineq:
        from .models import SlackModel
        nlp = SlackModel(nlp)
        x0 = np.concatenate([_V.host(x0), np.zeros(nlp.meta.nvar - orig.meta.nvar)])
    solver = FPSSSolver(nlp, x0, **kwargs)
    stats = solve(solver, verbose=verbose, subsolver_verbose=subsolver_verbose, callback=callback)
    if ineq:
        stats.solution = stats.solution[:orig.meta.nvar]
    stats.solver_specific["solver"] = solver
    return stats


def _go_log(stp, sub, model, fx, ncx, mess, verbose):
    it = stp.meta.nb_of_stop
    if verbose > 0 and it % verbose == 0:
        print(f"{it:5d} {mess:8s} f={fx: .6e} ‖c‖={ncx:.2e} ‖∇φ‖={sub.current_score:.2e} σ={model.sigma:.1e} "
              f"ρ={model.rho:.1e} δ={model.delta:.1e} {sub.status():>15s} ‖λ‖={_V.ninf(model.ys):.2e}")


def _update_parameters(meta, model, feas):
    """src/algo.jl:366-381"""
    model.sigma *= meta.sigma_update
    if not feas:
        model.rho *= meta.rho_update
    # The penalty changed.  The reference keeps its memo here (it is keyed on hash(x) only, SURVEY App. D-1), so its
    # first evaluation at the unchanged x still sees ys / gs of the OLD sigma: that is the default.  The option
    # refresh_memo_on_update (not a reference option) drops the memo instead.
    if getattr(meta, "refresh_memo_on_update", False):
        model.shahx = 0


def _update_parameters_unbdd(meta, model, feas):
    """src/algo.jl:388-395"""
    if model.delta == 0:
        model.delta = meta.delta_0
    else:
        model.delta *= meta.delta_update
    _update_parameters(meta, model, feas)


def _random_restoration(stp, model, rng):
    """src/algo.jl:340-359"""
    radius = min(max(stp.meta.atol, 1 / model.sigma, 1e-3), 1.0)
    st = stp.current_state
    st.x = st.x + radius * _V.like(st.x, rng.random(len(st.x)))


def _restoration_feasibility(fs, stp, model, feas_tol, ncx, verbose, rng):
    """src/algo.jl:295-333"""
    st = stp.current_state
    host = stp.pb
    qds = getattr(model, "qdsolver", None) if getattr(fs, "fused", False) else None
    if qds is not None and (not hasattr(qds, "handle") or getattr(model, "explicit_linear_constraints", False)):
        qds = None                                   # a user-defined QDSolver, or a handle on the nonlinear rows only
    z, cz, _, status = feasibility_step(fs, host, st.x, st.cx - stp._lcon, ncx, feas_tol, feas_tol, verbose, qds=qds)
    if status == "success":
        st.x, st.cx = z, cz + stp._lcon
    else:
        _random_restoration(stp, model, rng)


def solve(fpssolver, *, verbose=0, subsolver_verbose=0, callback=None, seed=1234):
    """SolverCore.solve!(fpssolver, stp, stats)   (src/algo.jl:26-288); same branch structure."""
    stats = GenericExecutionStats()
    stp, meta, model = fpssolver.stp, fpssolver.meta, fpssolver.model
    st = stp.current_state
    rng = np.random.default_rng(seed)
    if _has_inequalities(stp.pb):
        raise ValueError("Error: consider only problem with equalities and bounds. Use `SlackModel`.")
    model.sigma, model.rho, model.delta = meta.sigma_0, meta.rho_0, 0.0
    model.shahx = 0
    OK = stp.start()
    sub_atol, sub_rtol = meta.atol_sub(stp.meta.atol), meta.rtol_sub(stp.meta.rtol)
    feas_tol = stp.meta.atol
    unsuccessful_subpb = unbounded_subpb = stalling = 0
    feasibility_phase = restoration_phase = False
    sub_x = _V.copy(st.x)
    bounds = dict(lvar=stp._lvar, uvar=stp._uvar) if stp.has_bounds else {}
    lin_proj = getattr(fpssolver, "lin_projector", None)
    lin_kw = dict(lin=lin_proj) if lin_proj is not None else {}
    sub = SubStats()
    ys_blown_up = lambda mdl, x: "unbounded" if _V.ninf(mdl.ys) >= meta.lagrange_bound else None
    if callback:
        callback(model, fpssolver, stats)
    while not OK and stats.status != "user":
        max_time = max(stp.meta.max_time - (time.time() - stp.meta.start_time), 0.0)
        sub = fpssolver.subproblem_solver(model, sub_x, atol=sub_atol, rtol=sub_rtol,
                                          max_iter=meta.subsolver_max_iter, max_time=max_time,
                                          unbounded_threshold=meta.subpb_unbounded_threshold,
                                          verbose=subsolver_verbose, stop_callback=ys_blown_up, **bounds, **lin_kw)
        fpssolver.sub_stats = sub
        unbounded_lagrange_multiplier = _V.ninf(model.ys) >= meta.lagrange_bound
        sub_ok = sub.optimal or sub.suboptimal
        sub_unbdd = sub.unbounded or sub.unbounded_pb or unbounded_lagrange_multiplier
        sub_tired = sub.tired or sub.resources or sub.iteration_limit or sub.stalled
        if sub_ok:
            if _V.equal(sub.x, st.x):
                stalling += 1
            unsuccessful_subpb = unbounded_subpb = 0
            if lin_proj is not None:
                # src/algo.jl:127-137: multipliers and constraint values of the linear rows come from the subproblem,
                # those of the nonlinear rows from the penalty model; the residual is the subproblem's g + J_lin' lambda.
                # Sign: sub.lam = -(AA')^-1 A g, the convention of the penalised rows (lambda = -ys, ys = (JJ')^-1 J g),
                # so that both modes report the same multipliers for a linear row.
                lin_i, nln_i = list(stp.pb.meta.lin), list(stp.pb.meta.nln)
                lam = np.zeros(stp.pb.meta.ncon)
                lam[lin_i] = sub.lam
                lam[nln_i] = -model.ys
                cx = np.zeros(stp.pb.meta.ncon)
                cx[lin_i] = stp.pb.cons_lin(sub.x)
                cx[nln_i] = model.cx + np.asarray(stp.pb.meta.lcon)[nln_i]
                st.lam, st.cx, st.res = lam, cx, sub.res
            else:
                st.lam = -model.ys
                st.cx = model.cx + stp._lcon
                st.res = sub.gx
            st.x, st.fx, st.gx = _V.copy(sub.x), model.fx, model.gx
            _go_log(stp, sub, model, st.fx, _V.norm(model.cx), "Optml", verbose)
        elif sub_unbdd:
            stalling = unsuccessful_subpb = 0
            unbounded_subpb += 1
            ncx = _V.ninf(model.cx)
            if ncx < feas_tol:
                stp.meta.unbounded_pb = True
            _go_log(stp, sub, model, sub.fx, ncx, "Unbdd", verbose)
        elif sub_tired:
            stalling = unbounded_subpb = 0
            unsuccessful_subpb += 1
            _go_log(stp, sub, model, sub.fx, _V.norm(model.cx), "Tired" if (sub.tired or sub.resources) else "Stlld",
                    verbose)
        else:
            stp.meta.fail_sub_pb = True
            warnings.warn(f"Exception of unexpected failure: {sub.status()}")
        stp.meta.fail_sub_pb = stp.meta.fail_sub_pb or (model.sigma > meta.sigma_max or model.rho > meta.rho_max
                                                        or model.delta > meta.delta_max)
        OK = stp.stop()
        if not OK:
            ncx = _V.norm(model.cx)
            feas = ncx < feas_tol
            restart_x = None
            if sub_ok:
                if feas:                                       # tighten the tolerances (:194-200)
                    sub_atol = max(sub_atol / 10, EPS)
                    sub_rtol = max(sub_rtol / 10, EPS)
                    model.eta = max(meta.eta_1, model.eta * meta.eta_update)
                    model.xk = _V.copy(st.x)
                    _go_log(stp, sub, model, st.fx, ncx, "D-ϵ", verbose)
                elif not feasibility_phase and (stalling >= 3 or sub_atol < EPS):
                    feasibility_phase = True
                    unbounded_subpb = 0
                    _restoration_feasibility(fpssolver.feasibility_solver, stp, model, feas_tol, ncx, verbose, rng)
                    restart_x = st.x
                    stalling = unsuccessful_subpb = 0
                    _go_log(stp, sub, model, st.fx, _V.norm(st.cx - stp._lcon), "R", verbose)
                elif stalling >= 3 or sub_atol < EPS:          # infeasible stationary point
                    stp.meta.suboptimal = True
                    OK = True
                else:
                    _update_parameters(meta, model, feas)
                    _go_log(stp, sub, model, st.fx, ncx, "D", verbose)
            elif sub_unbdd:
                if not feasibility_phase and unbounded_subpb >= 3 and not feas:
                    feasibility_phase = True
                    unbounded_subpb = 0
                    _restoration_feasibility(fpssolver.feasibility_solver, stp, model, feas_tol, ncx, verbose, rng)
                    restart_x = st.x
                    stalling = unsuccessful_subpb = 0
                    _go_log(stp, sub, model, st.fx, _V.norm(st.cx - stp._lcon), "R", verbose)
                elif not restoration_phase and unbounded_subpb >= 3:
                    restoration_phase = True
                    unbounded_subpb = 0
                    _random_restoration(stp, model, rng)
                    restart_x = st.x
                    _go_log(stp, sub, model, st.fx, _V.norm(st.cx - stp._lcon), "R-Unbdd", verbose)
                else:
                    _update_parameters_unbdd(meta, model, feas)
                    _go_log(stp, sub, model, st.fx, ncx, "D", verbose)
            elif sub_tired:
                if not restoration_phase and unsuccessful_subpb >= 3 and feas:
                    restoration_phase = True
                    unsuccessful_subpb = 0
                    _random_restoration(stp, model, rng)
                    restart_x = st.x
                    _go_log(stp, sub, model, st.fx, _V.norm(st.cx - stp._lcon), "R-Unscc", verbose)
                elif not feasibility_phase and unsuccessful_subpb >= 3 and not feas:
                    feasibility_phase = True
                    unsuccessful_subpb = 0
                    _restoration_feasibility(fpssolver.feasibility_solver, stp, model, feas_tol, ncx, verbose, rng)
                    restart_x = st.x
                    stalling = unsuccessful_subpb = 0
                    _go_log(stp, sub, model, st.fx, _V.norm(st.cx - stp._lcon), "R", verbose)
                else:
                    _update_parameters(meta, model, feas)
                    _go_log(stp, sub, model, st.fx, ncx, "D", verbose)
            # the next subproblem starts where the sub-state is: the restoration point if there was one,
            # otherwise the subsolver's last iterate (the reference keeps x in `reinit!`, :374-380)
            if restart_x is not None:
                model.shahx = 0
                sub_x = _V.copy(restart_x)
            else:
                sub_x = _V.copy(sub.x)
        stats.status = stp.status()
        stats.solution = _V.host(st.x).copy()
        stats.objective = float(st.fx)
        stats.primal_feas = _V.ninf(st.cx - stp._lcon)
        stats.dual_feas = float(sub.current_score)
        stats.multipliers = _V.host(st.lam).copy()
        stats.iter = stp.meta.nb_of_stop
        stats.elapsed_time = st.current_time - stp.meta.start_time
        if callback:
            callback(model, fpssolver, stats)
    if stats.solution is None:                                  # optimal at the start (:55-59)
        stats.status = stp.status()
        stats.solution = _V.host(st.x).copy()
        stats.objective = float(st.fx) if not math.isnan(st.fx) else float(stp.pb.obj(st.x))
        stats.primal_feas = _V.ninf(st.cx - stp._lcon)
        stats.dual_feas = _V.ninf(st.res)
        stats.multipliers = _V.host(st.lam).copy()
        stats.iter = 0
        stats.elapsed_time = 0.0
    stats.solver_specific.update(sigma=model.sigma, rho=model.rho, delta=model.delta,
                                 restoration=restoration_phase, feasibility=feasibility_phase)
    return stats
