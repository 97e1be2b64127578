"""Device-resident FletcherPenaltyNLP (SURVEY §8 f1): the same evaluation as fletcher_nlp.py
(src/model-Fletcherpenaltynlp.jl:234-252, 352-437, 521-570) with x, g, c, ys, gs, v, w and every
intermediate living in HBM.  The 2-RHS solves are called with device pointers (FPSB_DEVICE), the
vector combinations either side of them are the fused fpsb_fp_* kernels of libfpsb200, and the memo
key is computed on the device (fpsb_fp_hash) instead of hash(x) on the host.

The user model must evaluate on the device: `obj(x) -> float`, `grad(x)`, `cons(x)`, `jac_coord(x)`,
`hprod(x, y, v, obj_weight)` taking / returning torch CUDA float64 tensors (DeviceSparseQP below is
the synthetic model of BASELINE configs C2 / C4, DeviceCurvedQP its variant with curved constraints).  Both Hessian
variants are device-resident: Val(2), and Val(1) (round 2) which adds `ghjvprod(x, g, v)` on the device model and the
`solve_two_extras` pair with device pointers (src/model-Fletcherpenaltynlp.jl:572-634).

BatchFletcherPenaltyNLP evaluates K points of one model in lock-step (LDLt path): the batched solves, the
fpsb_fp_batch_* combinations and the batched Jacobian products of libfpsb200.
"""
import ctypes as C

import numpy as np

from . import _lib
from .models import AbstractNLPModel, NLPModelMeta
from .qdsolver import LDLtSolver, _warn_failed, solve_two_extras, solve_two_least_squares, solve_two_mixed


def _dp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _rowsum(A):
    """Sum of every row of A (K, n) by a fixed pairwise tree of element-wise additions: torch's reduction kernels pick
    their split from the tensor's shape, so a row's sum could round differently with the number of rows."""
    import torch
    K, n = A.shape
    if n == 0:
        return torch.zeros(K, dtype=A.dtype, device=A.device)
    p = 1 << (n - 1).bit_length()
    if p != n:
        A = torch.nn.functional.pad(A, (0, p - n))
    while A.shape[1] > 1:
        h = A.shape[1] // 2
        A = A[:, :h] + A[:, h:]
    return A[:, 0]


class DeviceSparseQP(AbstractNLPModel):
    """min 1/2 x' diag(Q) x + q'x  s.t.  A x = b  with all data on the GPU (the model side is user code:
    it uses torch for its own arithmetic)."""

    def __init__(self, host_qp, device="cuda"):
        import torch
        super().__init__()
        self.host = host_qp
        A = host_qp.A
        self.meta = NLPModelMeta(A.shape[1], A.shape[0], x0=np.zeros(A.shape[1]), nnzj=A.nnz, name=host_qp.meta.name + "-device")
        self._rows, self._cols = host_qp.jac_structure()
        f64 = dict(dtype=torch.float64, device=device)
        self.Q = torch.tensor(host_qp.Q, **f64)
        self.q = torch.tensor(host_qp.q, **f64)
        self.b = torch.tensor(host_qp.b, **f64)
        self._vals = torch.tensor(host_qp._vals, **f64)          # the values of A in the COO order of jac_structure
        self._device = device
        self._H = None          # the model's own operator handle for c(x) = A x - b (hand-written SpMV, no cuSPARSE)

    def _op(self):
        if self._H is None:
            import torch
            from .qdsolver import B200Handle
            d = torch.device(self._device)
            idx = d.index if d.index is not None else torch.cuda.current_device()
            self._H = B200Handle(self.meta.nvar, self.meta.ncon, self._rows, self._cols, device=idx)
            self._H.set_jac_values(self._vals)
        return self._H

    def obj(self, x):
        return float(0.5 * (x * self.Q * x).sum() + self.q @ x)

    def grad(self, x):
        return self.Q * x + self.q

    def cons(self, x):
        return self._op().jprod(x) - self.b

    def jac_structure(self):
        return self._rows, self._cols

    def jac_coord(self, x):
        return self._vals

    def hprod(self, x, y, v, obj_weight=1.0):
        return obj_weight * self.Q * v

    # -- the batched model protocol of BatchFletcherPenaltyNLP: one point per row of X (K, nvar) -------------------
    def obj_batch(self, X):
        return 0.5 * _rowsum(X * self.Q * X) + _rowsum(self.q * X)

    def grad_batch(self, X):
        return self.Q * X + self.q

    def cons_batch(self, X):
        return self._op().batch_jprod(self._vals, X) - self.b

    def jac_coord_batch(self, X):
        return self._vals.expand(X.shape[0], -1)

    def hprod_batch(self, X, Y, V, obj_weight=1.0):
        return obj_weight * self.Q * V


class DeviceCurvedQP(DeviceSparseQP):
    """models.CurvedQPModel with all data on the GPU: curved constraints, so `hprod` depends on y and `ghjvprod` is not
    zero (the model side is user code: torch for its own arithmetic, the repo's SpMV for A x)."""

    def __init__(self, host_model, device="cuda"):
        import torch
        super().__init__(host_model, device=device)
        f64 = dict(dtype=torch.float64, device=device)
        self.d = torch.tensor(host_model.d, **f64)
        self._k = torch.tensor(host_model._k, dtype=torch.int64, device=device)
        self._first = torch.tensor(host_model._first, dtype=torch.int64, device=device)

    def cons(self, x):
        return self._op().jprod(x) + 0.5 * self.d * x[self._k] ** 2 - self.b

    def jac_coord(self, x):
        vals = self._vals.clone()
        vals[self._first] += self.d * x[self._k]
        return vals

    def hprod(self, x, y, v, obj_weight=1.0):
        out = obj_weight * self.Q * v
        out.index_add_(0, self._k, y * self.d * v[self._k])
        return out

    def ghjvprod(self, x, g, v):
        return g[self._k] * self.d * v[self._k]

    def cons_batch(self, X):
        return self._op().batch_jprod(self._vals, X) + 0.5 * self.d * X[:, self._k] ** 2 - self.b

    def jac_coord_batch(self, X):
        vals = self._vals.repeat(X.shape[0], 1)
        vals[:, self._first] += self.d * X[:, self._k]
        return vals

    def hprod_batch(self, X, Y, V, obj_weight=1.0):
        # the constraint-Hessian terms of every variable are added in a fixed order (the single hprod's index_add_ adds
        # repeated indices in no fixed order on CUDA), so a row's product does not depend on the rest of the batch
        import torch
        out = obj_weight * self.Q * V
        terms = torch.nn.functional.pad(Y * self.d * V[:, self._k], (0, 1))     # column ncon: zero
        rov = self._rows_of_var()
        for t in range(rov.shape[1]):
            out = out + terms[:, rov[:, t]]
        return out

    def _rows_of_var(self):
        """(nvar, maxdeg): the rows i with k_i = j for every variable j, in row order, padded with ncon."""
        if getattr(self, "_rov", None) is None:
            import torch
            k = np.asarray(self.host._k, dtype=np.int64)
            m, n = len(k), self.meta.nvar
            deg = np.bincount(k, minlength=n)
            order = np.argsort(k, kind="stable")
            start = np.concatenate([[0], np.cumsum(deg)[:-1]])
            rov = np.full((n, int(deg.max()) if m else 0), m, dtype=np.int64)
            rov[k[order], np.arange(m) - start[k[order]]] = order
            self._rov = torch.tensor(rov, dtype=torch.int64, device=self._k.device)
        return self._rov

    def ghjvprod_batch(self, X, G, V):
        return G[:, self._k] * self.d * V[:, self._k]


class DeviceFletcherPenaltyNLP:
    """FletcherPenaltyNLP(nlp, sigma, rho, delta, Val(1) | Val(2); qds = ...) with device-resident state."""

    def __init__(self, nlp, sigma=1.0, rho=0.0, delta=0.0, hessian_approx=2, *, qds=None, device="cuda",
                 consistent_gradient=False):
        import torch
        assert hessian_approx in (1, 2), "hessian_approx is Val(1) or Val(2)"
        self.consistent_gradient = consistent_gradient      # see FletcherPenaltyNLP
        self.torch = torch
        self.nlp = nlp
        self.explicit_linear_constraints = False
        self.nvar, self.npen = nlp.meta.nvar, nlp.meta.ncon
        self.sigma, self.rho, self.delta, self.eta = sigma, rho, delta, 0.0
        self.qdsolver = qds if qds is not None else LDLtSolver(nlp, 0.0)
        self.handle = self.qdsolver.handle
        self.hessian_approx = int(hessian_approx)
        f64 = dict(dtype=torch.float64, device=device)
        n, m = self.nvar, self.npen
        self.key = None
        self.fx = float("nan")
        self.gx = self.cx = None
        self.gs, self.v, self.xk = (torch.empty(n, **f64) for _ in range(3))
        self.xk.zero_()
        self.ys, self.w = (torch.empty(m, **f64) for _ in range(2))
        self.neval = dict(obj=0, grad=0, hprod=0)
        self._lib = _lib.lib()

    @property
    def shahx(self):
        return self.key

    @shahx.setter
    def shahx(self, value):          # `shahx = 0` drops the memo (what reinit! does to the sub-state)
        self.key = None if not value else value

    def _hash(self, x):
        self.handle._follow_torch_stream(x)      # every fpsb_fp_* call is ordered against torch's current stream
        k = C.c_uint64()
        _lib.check(self._lib.fpsb_fp_hash(self.handle.h, _dp(x), C.byref(k)), "fpsb_fp_hash")
        return k.value

    def _compute_ys_gs(self, x):
        key = self._hash(x)
        if key != self.key:
            self.key = key
            self.fx = self.nlp.obj(x)
            self.gx = self.nlp.grad(x)
            self.cx = self.nlp.cons(x)          # lcon = 0 for the equality models handled here
            p1, q1, p2, q2 = solve_two_mixed(self, x, self.gx, self.cx)
            _lib.check(self._lib.fpsb_fp_ys_gs(self.handle.h, C.c_double(self.sigma), _dp(p1), _dp(q1), _dp(p2), _dp(q2),
                                               _dp(self.gs), _dp(self.ys), _dp(self.v), _dp(self.w)), "fpsb_fp_ys_gs")
        return self.gs, self.ys, self.v, self.w

    def obj(self, x):
        self.neval["obj"] += 1
        self._compute_ys_gs(x)
        phi = C.c_double()
        _lib.check(self._lib.fpsb_fp_obj(self.handle.h, C.c_double(self.fx), C.c_double(self.rho), C.c_double(self.eta),
                                         _dp(self.cx), _dp(self.ys), _dp(x), _dp(self.xk), C.byref(phi)), "fpsb_fp_obj")
        return phi.value

    def grad(self, x):
        self.neval["grad"] += 1
        gs, ys, v, w = self._compute_ys_gs(x)
        Hsv = self.nlp.hprod(x, -ys if self.consistent_gradient else ys, v, obj_weight=1.0)
        Sstw = self.nlp.hprod(x, w, gs, obj_weight=0.0)
        Jtc = self.handle.jtprod(self.cx) if self.rho > 0.0 else None
        g = self.torch.empty_like(x)
        _lib.check(self._lib.fpsb_fp_grad(self.handle.h, C.c_double(self.sigma), C.c_double(self.rho), C.c_double(self.eta),
                                          _dp(gs), _dp(Hsv), _dp(v), _dp(Sstw), _dp(Jtc), _dp(x), _dp(self.xk), _dp(g)),
                   "fpsb_fp_grad")
        return g

    def objgrad(self, x):
        g = self.grad(x)
        return self.obj(x), g

    def hprod(self, x, v, obj_weight=1.0):
        self.neval["hprod"] += 1
        gs, ys, _, _ = self._compute_ys_gs(x)
        mys = -ys
        Hsv = self.nlp.hprod(x, mys, v, obj_weight=1.0)
        p1, _, p2, _ = solve_two_least_squares(self, x, v, Hsv)
        Ptv = self.torch.empty_like(v)
        _lib.check(self._lib.fpsb_fp_ptv(self.handle.h, _dp(v), _dp(p1), _dp(Ptv)), "fpsb_fp_ptv")
        HsPtv = self.nlp.hprod(x, mys, Ptv, obj_weight=1.0)
        Hcv = JtJv = None
        if self.rho > 0.0:
            JtJv = self.handle.jtprod(self.handle.jprod(v))
            Hcv = self.nlp.hprod(x, self.cx, v, obj_weight=0.0)
        Hv = self.torch.empty_like(v)
        if self.hessian_approx == 1:
            # the exact Hessian's two extra terms (src/model-Fletcherpenaltynlp.jl:603-634): ghjvprod on the device model,
            # the MINRES / LSQR (or LDLt) pair of solve_two_extras with device pointers, one product with A'
            Ssv = self.nlp.ghjvprod(x, gs, v)
            invJtJJv, invJtJSsv = solve_two_extras(self, x, v, Ssv)
            JtinvJtJSsv = self.handle.jtprod(invJtJSsv)
            SsinvJtJJv = self.nlp.hprod(x, invJtJJv, gs, obj_weight=0.0)
            _lib.check(self._lib.fpsb_fp_hprod1(self.handle.h, C.c_double(self.sigma), C.c_double(self.rho), C.c_double(self.eta),
                                                C.c_double(obj_weight), _dp(p2), _dp(HsPtv), _dp(Ptv), _dp(JtinvJtJSsv),
                                                _dp(SsinvJtJJv), _dp(Hcv), _dp(JtJv), _dp(v), _dp(Hv)), "fpsb_fp_hprod1")
            return Hv
        _lib.check(self._lib.fpsb_fp_hprod2(self.handle.h, C.c_double(self.sigma), C.c_double(self.rho), C.c_double(self.eta),
                                            C.c_double(obj_weight), _dp(p2), _dp(HsPtv), _dp(Ptv), _dp(Hcv), _dp(JtJv), _dp(v),
                                            _dp(Hv)), "fpsb_fp_hprod2")
        return Hv


def _rows(nlp, name, X, *args, **kw):
    """The batched model protocol: nlp.<name>_batch(X, ...) when the model has it, else the single method looped over
    the rows (X and the tensor arguments row by row) and stacked; obj returns a (K,) tensor."""
    import torch
    f = getattr(nlp, name + "_batch", None)
    if f is not None:
        return f(X, *args, **kw)
    g = getattr(nlp, name)
    out = [g(X[i], *(a[i] for a in args), **kw) for i in range(X.shape[0])]
    if name == "obj":
        return torch.tensor(out, dtype=torch.float64, device=X.device)
    if not out:
        return None
    return torch.stack([torch.as_tensor(o, dtype=torch.float64, device=X.device) for o in out])


class BatchFletcherPenaltyNLP:
    """K instances of FletcherPenaltyNLP(nlp, sigma, rho, delta, Val(1) | Val(2)) evaluated in lock-step on the device:
    one model, one LDLtSolver handle, and per instance its own point X[i] and its own sigma, rho, delta, eta, xk (each
    a scalar or one value per instance; xk None, (nvar,) or (K, nvar)).  Every method takes X (K, nvar) as a CUDA
    float64 tensor and returns (K,) / (K, .) tensors; instance i gives what DeviceFletcherPenaltyNLP gives at X[i]
    (the combinations are bitwise the single kernels', the Jacobian products differ from the single SELL-32 products
    in the last bits).  The solves are the batched LDLt ones (ldlt_batch_solve_two_mixed / _least_squares / _extras).

    The model is evaluated through obj_batch / grad_batch / cons_batch / jac_coord_batch / hprod_batch /
    ghjvprod_batch when it has them, else through its single methods row by row.

    Memo: one key per row (fpsb_fp_batch_hash).  When K changes, or any row's key changes, the model and the batched
    mixed solve are evaluated again for the whole batch, because the batched least-squares solve of `hprod` needs the
    factors of all K instances.  Every per-instance computation is deterministic and independent of the rest of the
    batch, so re-solving an unchanged row gives the same bits: an instance's results do not depend on which neighbours
    moved.  The factors live on the handle: another batched mixed solve on the same handle between `obj` / `grad` and
    `hprod` replaces them."""

    def __init__(self, nlp, sigma=1.0, rho=0.0, delta=0.0, hessian_approx=2, *, qds=None, device="cuda",
                 consistent_gradient=False, explicit_linear_constraints=False):
        import torch
        if hessian_approx not in (1, 2):
            raise ValueError("hessian_approx is Val(1) or Val(2)")
        if explicit_linear_constraints or getattr(qds, "explicit_linear_constraints", False):
            raise NotImplementedError("BatchFletcherPenaltyNLP: explicit_linear_constraints is not supported")
        if qds is not None and not isinstance(qds, LDLtSolver):
            raise TypeError(f"BatchFletcherPenaltyNLP: no batched path for {type(qds).__name__} (LDLtSolver only)")
        self.torch = torch
        self.nlp = nlp
        self.consistent_gradient = consistent_gradient      # see FletcherPenaltyNLP
        self.explicit_linear_constraints = False
        self.nvar, self.npen = nlp.meta.nvar, nlp.meta.ncon
        self.sigma, self.rho, self.delta, self.eta = sigma, rho, delta, 0.0
        self.xk = None
        self.qdsolver = qds if qds is not None else LDLtSolver(nlp, 0.0)
        self.handle = self.qdsolver.handle
        self.hessian_approx = int(hessian_approx)
        self.device = torch.device(device)
        self.keys = None
        self.fx = self.gx = self.cx = self.jvals = None
        self.gs = self.ys = self.v = self.w = None
        self.neval = dict(obj=0, grad=0, hprod=0)
        self._lib = _lib.lib()
        self._scal_cache = (None, None)

    # -- per-instance parameters ---------------------------------------------------------------------------------
    def _per(self, val, K, name):
        a = val.detach().cpu().numpy() if hasattr(val, "detach") else np.asarray(val, dtype=np.float64)
        a = np.asarray(a, dtype=np.float64)
        if a.ndim == 0:
            return np.full(K, float(a))
        if a.shape != (K,):
            raise ValueError(f"BatchFletcherPenaltyNLP: {name} must be a scalar or have one value per instance ({K})")
        return a

    def _scalars(self, K):
        """sigma, rho, delta, eta as (K,) device tensors (cached while the values hold); rho / eta are None when every
        instance has 0, which is what the single evaluator's `rho > 0` / `eta > 0` branches see."""
        host = [self._per(getattr(self, k), K, k) for k in ("sigma", "rho", "delta", "eta")]
        key = (K, b"".join(h.tobytes() for h in host))
        if self._scal_cache[0] != key:
            dev = [self.torch.tensor(h, dtype=self.torch.float64, device=self.device) for h in host]
            sigma, rho, delta, eta = dev
            self._scal_cache = (key, dict(sigma=sigma, rho=rho if (host[1] > 0).any() else None, delta=delta,
                                          eta=eta if (host[3] > 0).any() else None))
        return self._scal_cache[1]

    def _xk(self, K):
        t = self.torch
        if self.xk is None:
            return t.zeros((K, self.nvar), dtype=t.float64, device=self.device)
        xk = t.as_tensor(self.xk, dtype=t.float64, device=self.device)
        if xk.ndim == 1 and xk.shape[0] == self.nvar:
            return xk.expand(K, -1).contiguous()
        if tuple(xk.shape) != (K, self.nvar):
            raise ValueError(f"BatchFletcherPenaltyNLP: xk must be ({self.nvar},) or (K, {self.nvar})")
        return xk.contiguous()

    def _check(self, X, name="X", like=None):
        t = self.torch
        if not (hasattr(X, "is_cuda") and X.is_cuda):
            raise TypeError(f"BatchFletcherPenaltyNLP: {name} must be a CUDA tensor")
        if X.ndim != 2 or X.shape[1] != self.nvar or (like is not None and X.shape[0] != like.shape[0]):
            raise ValueError(f"BatchFletcherPenaltyNLP: {name} must be (K, {self.nvar})"
                             + ("" if like is None else f" with K = {like.shape[0]}"))
        return X.to(t.float64).contiguous()

    # -- memo --------------------------------------------------------------------------------------------------
    def _hash(self, X):
        t = self.torch
        keys = t.empty(X.shape[0], dtype=t.int64, device=X.device)
        self.handle._follow_torch_stream(X)
        _lib.check(self._lib.fpsb_fp_batch_hash(self.handle.h, C.c_int64(X.shape[0]), _dp(X), _dp(keys)),
                   "fpsb_fp_batch_hash")
        return keys

    def _compute_ys_gs(self, X):
        t = self.torch
        K = X.shape[0]
        keys = self._hash(X)
        if self.keys is not None and self.keys.shape[0] == K and t.equal(keys, self.keys):
            return self.gs, self.ys, self.v, self.w
        sc = self._scalars(K)
        nlp, H = self.nlp, self.handle
        self.keys = None                        # a failure below must not leave a memo of half-updated state
        self.fx = _rows(nlp, "obj", X)
        self.gx = _rows(nlp, "grad", X)
        self.cx = _rows(nlp, "cons", X)         # lcon = 0 for the equality models handled here
        J = _rows(nlp, "jac_coord", X)
        # one set of values shared by every row (a linear model's expand()) stays shared for the products (stride 0)
        self.jvals = J[0] if K > 0 and J.stride(0) == 0 else J.contiguous()
        p1, q1, p2, q2, ok = H.ldlt_batch_solve_two_mixed(sc["delta"], J, self.gx, self.cx)
        _warn_failed(ok)
        f64 = dict(dtype=t.float64, device=X.device)
        self.gs, self.v = t.empty((K, self.nvar), **f64), t.empty((K, self.nvar), **f64)
        self.ys, self.w = t.empty((K, self.npen), **f64), t.empty((K, self.npen), **f64)
        _lib.check(self._lib.fpsb_fp_batch_ys_gs(H.h, C.c_int64(K), _dp(sc["sigma"]), _dp(p1), _dp(q1), _dp(p2), _dp(q2),
                                                 _dp(self.gs), _dp(self.ys), _dp(self.v), _dp(self.w)),
                   "fpsb_fp_batch_ys_gs")
        self.keys = keys
        return self.gs, self.ys, self.v, self.w

    # -- FletcherPenaltyNLP surface, one row per instance ------------------------------------------------------------
    def obj(self, X):
        """phi_sigma at every row of X -> (K,) device tensor."""
        X = self._check(X)
        K = X.shape[0]
        self.neval["obj"] += 1
        phi = self.torch.empty(K, dtype=self.torch.float64, device=X.device)
        if K == 0:
            return phi
        self._compute_ys_gs(X)
        sc = self._scalars(K)
        xk = self._xk(K) if sc["eta"] is not None else None
        _lib.check(self._lib.fpsb_fp_batch_obj(self.handle.h, C.c_int64(K), _dp(self.fx), _dp(sc["rho"]), _dp(sc["eta"]),
                                               _dp(self.cx), _dp(self.ys), _dp(X if xk is not None else None), _dp(xk),
                                               _dp(phi)), "fpsb_fp_batch_obj")
        return phi

    def grad(self, X):
        X = self._check(X)
        K = X.shape[0]
        self.neval["grad"] += 1
        g = self.torch.empty_like(X)
        if K == 0:
            return g
        gs, ys, v, w = self._compute_ys_gs(X)
        sc = self._scalars(K)
        Hsv = _rows(self.nlp, "hprod", X, -ys if self.consistent_gradient else ys, v, obj_weight=1.0)
        Sstw = _rows(self.nlp, "hprod", X, w, gs, obj_weight=0.0)
        Jtc = self.handle.batch_jtprod(self.jvals, self.cx) if sc["rho"] is not None else None
        xk = self._xk(K) if sc["eta"] is not None else None
        _lib.check(self._lib.fpsb_fp_batch_grad(self.handle.h, C.c_int64(K), _dp(sc["sigma"]), _dp(sc["rho"]),
                                                _dp(sc["eta"]), _dp(gs), _dp(Hsv), _dp(v), _dp(Sstw), _dp(Jtc),
                                                _dp(X if xk is not None else None), _dp(xk), _dp(g)), "fpsb_fp_batch_grad")
        return g

    def objgrad(self, X):
        g = self.grad(X)
        return self.obj(X), g

    def hprod(self, X, V, obj_weight=1.0):
        """∇²phi_sigma(X[i]) V[i] for every row (Val(2), or Val(1) with the exact Hessian's two extra terms);
        obj_weight a scalar or (K,)."""
        t = self.torch
        X = self._check(X)
        V = self._check(V, "V", like=X)
        K = X.shape[0]
        self.neval["hprod"] += 1
        Hv = t.empty_like(V)
        if K == 0:
            return Hv
        ow = t.tensor(self._per(obj_weight, K, "obj_weight"), dtype=t.float64, device=X.device)
        gs, ys, _, _ = self._compute_ys_gs(X)
        sc = self._scalars(K)
        H, nlp = self.handle, self.nlp
        mys = -ys
        Hsv = _rows(nlp, "hprod", X, mys, V, obj_weight=1.0)
        p1, _, p2, _, ok = H.ldlt_batch_solve_two_least_squares(V, Hsv)
        _warn_failed(ok)
        Ptv = t.empty_like(V)
        _lib.check(self._lib.fpsb_fp_batch_ptv(H.h, C.c_int64(K), _dp(V), _dp(p1), _dp(Ptv)), "fpsb_fp_batch_ptv")
        HsPtv = _rows(nlp, "hprod", X, mys, Ptv, obj_weight=1.0)
        Hcv = JtJv = None
        if sc["rho"] is not None:
            JtJv = H.batch_jtprod(self.jvals, H.batch_jprod(self.jvals, V))
            Hcv = _rows(nlp, "hprod", X, self.cx, V, obj_weight=0.0)
        if self.hessian_approx == 1:
            # the exact Hessian's two extra terms (src/model-Fletcherpenaltynlp.jl:603-634)
            Ssv = _rows(nlp, "ghjvprod", X, gs, V)
            invJtJJv, invJtJSsv, st = H.ldlt_batch_solve_two_extras(sc["delta"], self.jvals.expand(K, -1), V, Ssv)
            self.qdsolver.last_batch_stats = st
            JtinvJtJSsv = H.batch_jtprod(self.jvals, invJtJSsv)
            SsinvJtJJv = _rows(nlp, "hprod", X, invJtJJv, gs, obj_weight=0.0)
            _lib.check(self._lib.fpsb_fp_batch_hprod1(H.h, C.c_int64(K), _dp(sc["sigma"]), _dp(sc["rho"]), _dp(sc["eta"]),
                                                      _dp(ow), _dp(p2), _dp(HsPtv), _dp(Ptv), _dp(JtinvJtJSsv),
                                                      _dp(SsinvJtJJv), _dp(Hcv), _dp(JtJv), _dp(V), _dp(Hv)),
                       "fpsb_fp_batch_hprod1")
            return Hv
        _lib.check(self._lib.fpsb_fp_batch_hprod2(H.h, C.c_int64(K), _dp(sc["sigma"]), _dp(sc["rho"]), _dp(sc["eta"]),
                                                  _dp(ow), _dp(p2), _dp(HsPtv), _dp(Ptv), _dp(Hcv), _dp(JtJv), _dp(V),
                                                  _dp(Hv)), "fpsb_fp_batch_hprod2")
        return Hv
