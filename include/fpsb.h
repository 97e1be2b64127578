/*
 * fpsb.h — C ABI of libfpsb200.so: B200-native (sm_100a) 2-right-hand-side quasi-definite solves
 *
 *        K = [ I   A' ]      A = J(x) in R^{ncon x nvar}  (the user model's Jacobian)
 *            [ A  -dI ]
 *
 * This is the drop-in boundary for FletcherPenaltySolver.jl's hot path.  Every entry point
 * replaces one piece of the reference's plugin surface; the Julia shim that binds them with
 * `ccall` is fletcherpenaltysolver.jl_b200/julia/B200Solver.jl (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ / torch types cross this boundary;
 *   - every function returns an int: FPSB_OK (0) or a negative FPSB_E* code; numerical failure is
 *     NEVER an error return: it is reported through `factorized` / `stats[].solved`, exactly like
 *     the reference (`@warn`, never throw: src/solve_linear_system.jl:54,73,92,101,128,136,197,245);
 *   - `loc` says where the caller's vectors live: FPSB_HOST (pageable or pinned host memory, the
 *     copies happen inside the call) or FPSB_DEVICE (device pointers on the handle's GPU; the call
 *     is stream-ordered on the handle's stream and synchronises before returning stats);
 *   - vectors are float64; index arrays are int64 (Julia `Int`);
 *   - a handle is not thread-safe (the reference is single-threaded and non re-entrant);
 *   - there is no CPU fallback: without a CUDA device every entry point fails with FPSB_ECUDA.
 */
#ifndef FPSB_H
#define FPSB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FPSB_VERSION 100

typedef struct fpsb_handle_s *fpsb_handle;

enum { FPSB_HOST = 0, FPSB_DEVICE = 1 };

enum {
    FPSB_OK = 0,
    FPSB_EINVAL = -1,   /* bad argument (NULL, negative size, index out of range) */
    FPSB_ECUDA = -2,    /* CUDA runtime error (see fpsb_last_error) */
    FPSB_ESTATE = -3,   /* call order violated (e.g. solve before analyze / set_jac_values) */
    FPSB_ENOMEM = -4,
    FPSB_ENCCL = -5
};

/* Krylov termination status (mirrors Krylov.jl's status strings; same codes as the oracle) */
enum {
    FPSB_ST_UNKNOWN = 0, FPSB_ST_ZERO_RHS = 1, FPSB_ST_SOLVED = 2, FPSB_ST_ZERO_RESID = 3,
    FPSB_ST_FWD_ERR = 4, FPSB_ST_TIRED = 5, FPSB_ST_ILLCOND_MACH = 6, FPSB_ST_ILLCOND_LIM = 7,
    FPSB_ST_INCONSISTENT = 8, FPSB_ST_ZERO_ATB = 9
};

/* Krylov.jl `stats` fields the reference reads (`.solved`, src/solve_linear_system.jl:53,72,...) */
typedef struct {
    int64_t niter;
    int32_t solved;
    int32_t inconsistent;
    int32_t status;
    int32_t pad_;
    double rnorm, arnorm, anorm, acond, xnorm;
} fpsb_krylov_stats;

/* IterativeSolver fields (src/solve_two_systems_struct.jl:23-73, defaults :99-115).
   itmax == 0 means "Krylov.jl default" as in the reference. */
typedef struct {
    double ls_atol, ls_rtol; int64_t ls_itmax;
    double ln_atol, ln_rtol, ln_btol, ln_conlim; int64_t ln_itmax;
    double ne_atol, ne_rtol, ne_etol, ne_conlim; int64_t ne_itmax;
} fpsb_iter_opts;

/* LDLtSolver keyword arguments (src/solve_two_systems_struct.jl:312-314) */
typedef struct {
    double ldlt_tol, ldlt_r1, ldlt_r2;
} fpsb_ldlt_opts;

/* ---------------------------------------------------------------------------------------------
 * Library / handle
 * ------------------------------------------------------------------------------------------- */
int fpsb_version(void);
/* last error message of the calling thread ("" when none) */
const char *fpsb_last_error(void);
/* number of CUDA devices visible; <= 0 means the library cannot run */
int fpsb_device_count(void);

/* Replaces the structural part of both QDSolver constructors
 *   LDLtSolver(nlp, ::T; ...)      src/solve_two_systems_struct.jl:308-353 (jac_structure!, :333-337)
 *   IterativeSolver(nlp, ::T; ...) src/solve_two_systems_struct.jl:94-160
 * jrow/jcol: the COO structure returned by jac_structure!(nlp, rows, cols) (length nnzj),
 * `index_base` 1 for Julia, 0 for C/Python.  Builds on the device: CSR of A and of A' (for
 * jprod / jtprod without atomics) and the COO->CSR value maps. `device` is the CUDA ordinal. */
int fpsb_create(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow, const int64_t *jcol,
                int index_base, int device, fpsb_handle *out);
int fpsb_destroy(fpsb_handle h);
int fpsb_dims(fpsb_handle h, int64_t *nvar, int64_t *ncon, int64_t *nnzj);
/* Optional: page-lock a caller-owned host buffer (cudaHostRegister) so that FPSB_HOST calls DMA
 * straight from / into it instead of staging through the handle's pinned area. Meant for the
 * solver-owned, long-lived vectors of the Julia shim (jvals, p1, q1, p2, q2). Unpin before freeing. */
int fpsb_pin_host(void *ptr, int64_t bytes);
int fpsb_unpin_host(void *ptr);
/* the handle's CUDA stream (cudaStream_t) so callers can order their own work / events on it */
void *fpsb_stream(fpsb_handle h);
/* FPSB_DEVICE callers: the stream (cudaStream_t) the caller's own kernels run on; default NULL = the
 * legacy default stream (what PyTorch / CUDA.jl's default task stream use).  The handle's stream is
 * non-blocking, so every entry that takes device pointers waits for this stream on the way in and
 * makes it wait for the handle's stream on the way out: inputs written by caller kernels are seen,
 * results are complete before the caller's next kernel reads them. */
int fpsb_set_caller_stream(fpsb_handle h, void *stream);
int fpsb_synchronize(fpsb_handle h);
/* CUDA-event stopwatch on the handle's stream (used by bench.py for device-side timing) */
int fpsb_timer_start(fpsb_handle h);
int fpsb_timer_stop(fpsb_handle h, double *elapsed_ms);
/* Pipelined throughput mode for host buffers (not in the reference, whose caller is one thread): with the gate on, the
 * fpsb_iter_solve_two_* calls of different handles / host threads of this process take turns for the compute part on a
 * device, while their host<->device copies overlap the solve that is running (process-wide switch, default off). */
int fpsb_pipeline_gate(int on);
/* number of kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t fpsb_launch_count(fpsb_handle h);
/* Layout of the tiled operators behind jprod / jtprod and the Krylov loops (the storage that replaces the reference's
 * LinearOperator `jac_op!`, src/solve_linear_system.jl:119-121): out = {tiles of A, of those with a shared-memory gather
 * window, of those with a multi-segment window (stencil operators), the same three for A'}. */
int fpsb_tile_stats(fpsb_handle h, int64_t out[6]);
/* Finer layout of the same operators, out[0..7] for A and out[8..15] for A': {tiles, tiles with a window, tiles with a
 * multi-segment window, tiles without a window (global int32 column indices), tiles with an odd window length, rows
 * longer than the SELL limit (long-row kernel), tiles without any slice (every row long), tiles holding long rows
 * next to their slices}.  Host only: touches nothing on the device. */
int fpsb_tile_layout(fpsb_handle h, int64_t out[16]);
/* The gather-window segments of one tile of A (transpose = 0) or A' (transpose = 1) on an operator that has
 * multi-segment tiles: out = {start column, length} of up to four column runs copied back to back, unused ones zero.
 * A single-window tile reports its one run, a tile without a window zeros; all zero when the operator has no
 * multi-segment tile.  Host only. */
int fpsb_tile_segments(fpsb_handle h, int transpose, int64_t tile, int64_t out[8]);

/* Replaces jac_coord!(nlp, x, vals[nvar+1 : nvar+nnzj]) feeding both paths
 *   src/solve_linear_system.jl:224-228 (LDLt)  and  jac_op! at :119-121 (Iterative).
 * vals: nnzj values in the COO order given to fpsb_create. */
int fpsb_set_jac_values(fpsb_handle h, const double *vals, int loc);

/* jprod! / jtprod! of the Jacobian operator (NLPModels jac_op!, SURVEY App. B6): out = A v, A' u.
 * Also used by the caller side for the rho-terms (src/model-Fletcherpenaltynlp.jl:388-395,552-563).
 * With loc = FPSB_DEVICE the four products are asynchronous: the work is ordered after the caller's stream
 * (fpsb_set_caller_stream) on entry and the caller's stream after it on exit; nothing waits on the host. */
int fpsb_jprod(fpsb_handle h, const double *v, double *Av, int loc);
int fpsb_jtprod(fpsb_handle h, const double *u, double *Atu, int loc);
/* two-column variants (columns contiguous: v is [v1 | v2], each of the natural length) */
int fpsb_jprod2(fpsb_handle h, const double *v, double *Av, int loc);
int fpsb_jtprod2(fpsb_handle h, const double *u, double *Atu, int loc);

/* ---------------------------------------------------------------------------------------------
 * Iterative path — IterativeSolver (LSQR / CRAIG / MINRES fused iterations)
 * ------------------------------------------------------------------------------------------- */
/* defaults of src/solve_two_systems_struct.jl:99-115 for given (nvar, ncon) */
int fpsb_iter_default_opts(int64_t nvar, int64_t ncon, fpsb_iter_opts *opts);
/* allocates the Krylov workspaces (LsqrWorkspace/CraigWorkspace/MinresWorkspace equivalents) */
int fpsb_iter_setup(fpsb_handle h, const fpsb_iter_opts *opts);

/* solve_two_mixed [Iterative]  src/solve_linear_system.jl:107-140
 *   q1 = LSQR(A', rhs1, lambda = sqrt(delta)), p1 = rhs1 - A' q1
 *   (x, y) = CRAIG(A, -rhs2 [, M = I/delta, sqd]), p2 = -x, q2 = y
 * rhs1: nvar, rhs2: ncon; p1, p2: nvar; q1, q2: ncon. stats[0] = LSQR, stats[1] = CRAIG. */
int fpsb_iter_solve_two_mixed(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                              double *p1, double *q1, double *p2, double *q2, int loc,
                              fpsb_krylov_stats stats[2]);
/* solve_two_least_squares [Iterative]  src/solve_linear_system.jl:79-105 (two LSQR on A');
 * rhs1, rhs2: nvar. (The reference returns q1 aliased to q2; here both are returned.) */
int fpsb_iter_solve_two_least_squares(fpsb_handle h, double delta, const double *rhs1,
                                      const double *rhs2, double *p1, double *q1, double *p2,
                                      double *q2, int loc, fpsb_krylov_stats stats[2]);
/* CUDA-event time (ms) of the Krylov loop region of the last solve_two_mixed/_least_squares call
 * on this handle and the number of fused SpMM step kernels launched in it (bench.py roofline). */
int fpsb_iter_last_profile(fpsb_handle h, double *loop_ms, int64_t *step_launches);
/* Geometry of the persistent Krylov loop kernel in the last iter_solve_two_* call on this handle, as launched:
 * out = {persistent kernel used (0/1), early row sums (0/1), ring stages, grid (CTAs), bytes per ring stage, tiles a
 * step-kernel producer may have in flight, tiles requested before a phase is decided, iterations per launch}.
 * All zero when that solve ran one launch per half iteration.  Host only: touches nothing on the device. */
int fpsb_iter_loop_info(fpsb_handle h, int64_t out[8]);
/* solve_two_extras [Iterative]  src/solve_linear_system.jl:45-77
 *   u1 = LSQR(A', rhs1, lambda = sqrt(tau)); u2 = MINRES(A A', rhs2, lambda = tau), tau = max(delta,1e-14) */
int fpsb_iter_solve_two_extras(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                               double *u1, double *u2, int loc, fpsb_krylov_stats stats[2]);

/* ---------------------------------------------------------------------------------------------
 * Host-only symbolic analysis (no CUDA device needed) — the `ldl_analyze` half of the LDLtSolver
 * constructor, src/solve_two_systems_struct.jl:343-344. fpsb_ldlt_analyze runs exactly this and
 * uploads the plan; exposing it lets the bit-exact symbolic check run on a CPU-only machine.
 * ------------------------------------------------------------------------------------------- */
typedef struct fpsb_symbolic_s *fpsb_symbolic;
int fpsb_symbolic_create(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow,
                         const int64_t *jcol, int index_base, const int64_t *P, fpsb_symbolic *out);
int fpsb_symbolic_destroy(fpsb_symbolic s);
/* B200-oriented alternative ordering (host only): BFS level-set dissection of the KKT graph into
 * `nparts` pieces (<= 0: automatic) with cyclic-reduction order of the separators. It trades some
 * fill for a dependency depth of O(piece depth + log2 nparts) instead of the O(N / 64) chain that
 * minimum degree produces on band-like structure. Pass the result as P to fpsb_ldlt_analyze /
 * fpsb_symbolic_create (the `ldl_analyze(A, P)` form of LDLFactorizations). */
int fpsb_order_dissection(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow,
                          const int64_t *jcol, int index_base, int nparts, int64_t *P_out);
int fpsb_symbolic_sizes(fpsb_symbolic s, int64_t *N, int64_t *lnz);
int fpsb_symbolic_get(fpsb_symbolic s, int64_t *P, int64_t *parent, int64_t *Lnz, int64_t *Lp,
                      int64_t *Li);
int fpsb_symbolic_plan_info(fpsb_symbolic s, int64_t *nsuper, int64_t *panel_nnz, int64_t *npairs,
                            double *flops, int64_t *nlevels, int64_t *nleaf);
/* Routes of the supernodal plan through the LDLt kernels, from the predicates the launches use.  Host only.
 *   [0] supernodes  [1] one-wide leaves (flat leaf kernels)  [2] leaves wider than one column (scalar CTA routines)
 *   [3] warp-level supernodes (w <= 8 and w (w + nr) <= 512; one-wide leaves excluded)  [4] of those, above the leaves
 *   [5] warp bundles (tasks of 1..8 warp-level supernodes)  [6] full bundles (8)
 *   [7] CTA-level supernodes above the leaves (the staged block routines in modes 1 and 2)  [8] of those with w = 64
 *   [9] of those with 33 <= w <= 63  [10] largest nr (rows below a supernode's diagonal block)
 *   [11] CTA-level panels (as [7]) with nr > 128 (more than one TRSM pass)  [12] with nr > 1024 (more than one
 *        backward-solve staging pass)
 *   update pairs into the supernodes of [7] (Schur update passes), nrow = rows of the source from the pair's first row,
 *   ncol = its columns in the target, wd = width of the source:
 *   [13] nrow > 64 (more than one pass)  [14] nrow % 8 != 0  [15] ncol % 8 != 0  [16] wd % 4 != 0
 *   [17] leaf contributions (leaf_update / leaf_fwd_update entries)  [18] explicit zero slots that relaxed
 *        amalgamation stores in the lower part of the panels  [19] panel slots assembled from more than one entry
 *   [20] dependency levels
 *   last staging pass one row short of full, exactly full, holding one row after a full one: [21..23] TRSM passes of the panels of [7]
 *   (128 rows), [24..26] backward-solve passes of the same panels (1024 rows), [27..29] Schur update passes of the
 *   pairs of [13] (64 rows) */
#define FPSB_LDLT_ROUTES 30
int fpsb_symbolic_ldlt_routes(fpsb_symbolic s, int64_t out[FPSB_LDLT_ROUTES]);

/* ---------------------------------------------------------------------------------------------
 * LDLt path — LDLtSolver (host symbolic analysis + device numeric refactorisation + 2-RHS solves)
 * ------------------------------------------------------------------------------------------- */
int fpsb_ldlt_default_opts(fpsb_ldlt_opts *opts);
/* ldl_analyze(Symmetric(sparse(rows, cols, vals), :U))  src/solve_two_systems_struct.jl:343-348.
 * P: permutation of size nvar+ncon, P[k] = (index_base-based) index eliminated k-th, or NULL for
 * the built-in approximate-minimum-degree ordering (LDLFactorizations' default is amd()).
 * Sets n_d = nvar, tol, r1, r2 from opts. Host work: ordering, elimination tree, column counts,
 * fill pattern, supernodes, dependency lists; uploads the device plan. */
int fpsb_ldlt_analyze(fpsb_handle h, const int64_t *P, int index_base, const fpsb_ldlt_opts *opts);
/* sizes of the symbolic factor: N = nvar + ncon and nnz(L) (strict lower part, like LDLFactorizations) */
int fpsb_ldlt_symbolic_sizes(fpsb_handle h, int64_t *N, int64_t *lnz);
/* bit-exact check surface: 0-based P, parent (-1 = root), Lnz, Lp (N+1), Li (lnz). Any may be NULL. */
int fpsb_ldlt_get_symbolic(fpsb_handle h, int64_t *P, int64_t *parent, int64_t *Lnz, int64_t *Lp,
                           int64_t *Li);
/* summary of the supernodal plan: nsuper, nnz stored in panels (incl. relaxed zeros), number of
 * (descendant -> target) update pairs, flops of the numeric factorisation, height of the supernodal
 * dependency DAG (critical path, in supernodes) and number of leaf supernodes */
int fpsb_ldlt_plan_info(fpsb_handle h, int64_t *nsuper, int64_t *panel_nnz, int64_t *npairs,
                        double *flops, int64_t *nlevels, int64_t *nleaf);
/* fpsb_symbolic_ldlt_routes of the plan fpsb_ldlt_analyze built (host only) */
int fpsb_ldlt_routes(fpsb_handle h, int64_t out[FPSB_LDLT_ROUTES]);
/* ldl_factorize!(M, str) with vals = [1..1 | jac values | -delta..-delta]
 *   src/solve_linear_system.jl:231-234. Uses the values last given to fpsb_set_jac_values.
 * *factorized mirrors LDLFactorizations.factorized(str). */
int fpsb_ldlt_factorize(fpsb_handle h, double delta, int *factorized);
/* numeric factor in LDLFactorizations' layout (Lx aligned with Li above, D of size N), host copies */
int fpsb_ldlt_get_factor(fpsb_handle h, double *Lx, double *D);

/* solve_two_mixed [LDLt]  src/solve_linear_system.jl:206-252 : refactor + K [p1 p2; q1 q2] = [rhs1 0; 0 rhs2].
 * On a failed factorisation the outputs hold the right-hand sides (reference behaviour, :242-251). */
int fpsb_ldlt_solve_two_mixed(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                              double *p1, double *q1, double *p2, double *q2, int loc,
                              int *factorized);
/* solve_two_least_squares [LDLt]  src/solve_linear_system.jl:161-204 : no refactor,
 * K [p1 p2; q1 q2] = [rhs1 rhs2; 0 0] */
int fpsb_ldlt_solve_two_least_squares(fpsb_handle h, const double *rhs1, const double *rhs2,
                                      double *p1, double *q1, double *p2, double *q2, int loc,
                                      int *factorized);
/* solve_two_extras [LDLt]  src/solve_linear_system.jl:142-159 : cgls(A', rhs1, lambda = tau),
 * minres(A A', rhs2, lambda = tau) with Krylov.jl default tolerances */
int fpsb_ldlt_solve_two_extras(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                               double *u1, double *u2, int loc, fpsb_krylov_stats stats[2]);

/* Batched LDLt path: `ninst` instances that share this handle's Jacobian pattern and its symbolic analysis
 * (fpsb_ldlt_analyze must have run), each with its own Jacobian values, delta and right-hand sides; one kernel launch
 * per call, one CTA per instance at a time.  Per-entry results are those of the single-instance entries above run on
 * each instance alone (same routines, same operation order).
 *   jvals [ninst][nnzj] (COO order given to fpsb_create), delta [ninst],
 *   rhs1 [ninst][nvar], rhs2 [ninst][ncon] (mixed) or [ninst][nvar] (least squares),
 *   p1, p2 [ninst][nvar], q1, q2 [ninst][ncon], factorized [ninst] (where `loc` says, like the outputs).
 * mixed = refactor + solve of every instance (src/solve_linear_system.jl:206-252); the factors stay on the device
 * (ninst x (panel_nnz + nvar + ncon) doubles, grown and never shrunk) and
 * fpsb_ldlt_batch_solve_two_least_squares (:161-204) reuses them (same ninst required, FPSB_ESTATE otherwise).
 * An instance whose factorisation fails gets factorized[i] = 0 and its right-hand sides as outputs (:242-251).
 * ninst == 0 is a no-op.  The single-instance factor, values and state of the handle are left alone.  With
 * loc = FPSB_DEVICE the call is asynchronous, ordered against the caller's stream (fpsb_set_caller_stream). */
int fpsb_ldlt_batch_solve_two_mixed(fpsb_handle h, int64_t ninst, const double *jvals, const double *delta,
                                    const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2,
                                    double *q2, int *factorized, int loc);
int fpsb_ldlt_batch_solve_two_least_squares(fpsb_handle h, int64_t ninst, const double *rhs1, const double *rhs2,
                                            double *p1, double *q1, double *p2, double *q2, int *factorized, int loc);

/* Tolerances of fpsb_ldlt_batch_solve_two_extras; NULL = what the reference's LDLt call uses, i.e. exactly what
 * fpsb_ldlt_solve_two_extras runs (Krylov.jl defaults: cgls atol = rtol = sqrt(eps), itmax = nvar + ncon; minres
 * atol = rtol = sqrt(eps)/100, etol = sqrt(eps), conlim = 1/sqrt(eps), itmax = 2 ncon).  itmax == 0 means that
 * default; a negative itmax is FPSB_EINVAL. */
typedef struct {
    double cg_atol, cg_rtol; int64_t cg_itmax;
    double mr_atol, mr_rtol, mr_etol, mr_conlim; int64_t mr_itmax;
} fpsb_extras_opts;
/* Batched solve_two_extras [LDLt]  src/solve_linear_system.jl:142-159: for each of `ninst` instances of this handle's
 * Jacobian pattern, u1 = cgls(A', rhs1, lambda = tau) and u2 = minres(A A', rhs2, lambda = tau), tau = max(delta, 1e-14),
 * with the instance's own Jacobian values.  One kernel launch per call: every (instance, method) pair runs inside one
 * CTA, with fixed-order reductions, so results are bitwise reproducible and do not depend on the batch (size, position)
 * or on `loc`; they agree with fpsb_ldlt_solve_two_extras on the same instance to the Krylov tolerances (its reductions
 * span many CTAs and round differently).
 *   jvals [ninst][nnzj] (COO order given to fpsb_create), delta [ninst], rhs1 [ninst][nvar], rhs2 [ninst][ncon],
 *   u1, u2 [ninst][ncon], stats [ninst][2] (CGLS, MINRES; where `loc` says, like the outputs).
 * Runs on any handle: it needs neither fpsb_ldlt_analyze nor fpsb_set_jac_values, and leaves the handle's
 * single-instance values, Krylov workspaces and the factors of fpsb_ldlt_batch_solve_two_mixed alone (mixed -> least
 * squares -> extras is the Val(1) hprod order).  ninst == 0 is a no-op.  With loc = FPSB_DEVICE the call is
 * asynchronous, ordered against the caller's stream (fpsb_set_caller_stream). */
int fpsb_ldlt_batch_solve_two_extras(fpsb_handle h, int64_t ninst, const double *jvals, const double *delta,
                                     const double *rhs1, const double *rhs2, double *u1, double *u2,
                                     fpsb_krylov_stats *stats, const fpsb_extras_opts *opts, int loc);

/* ---------------------------------------------------------------------------------------------
 * Throughput mode — many independent SMALL instances (BASELINE config C5): the LDLt path of
 * solve_two_mixed (kind 0, src/solve_linear_system.jl:206-252) or solve_two_least_squares (kind 1,
 * :161-204) for `ninst` instances that share (nvar, ncon), nvar + ncon <= 32, natural ordering.
 * A: [ninst][ncon][nvar] dense row-major Jacobians; rhs / outputs instance-major; factorized[i]
 * mirrors LDLFactorizations.factorized (outputs hold the right-hand sides when it is 0).
 * Multi-GPU: shard the instances across ranks (one call per rank, `device` = local GPU); no
 * communication is involved. */
int fpsb_batch_solve_two(int64_t ninst, int nvar, int ncon, int kind, const double *A, double delta,
                         const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2,
                         double *q2, int *factorized, const fpsb_ldlt_opts *opts, int loc, int device);

/* ---------------------------------------------------------------------------------------------
 * Row-partitioned Krylov path over several GPUs (one process per GPU, NCCL over NVLink) — what the
 * reference would reach by giving every Julia process a row block of the Jacobian (SURVEY 8e; the
 * reference itself is single-process, src/solve_linear_system.jl:79-140).
 *
 * Rank r creates its handle with fpsb_create on its LOCAL operator A_loc (ncon = owned constraint
 * rows, nvar = n_ext "extended" columns = owned variables + the halo columns its rows touch, in
 * global column order) and then attaches the exchange pattern:
 *   own_off, n_own        the owned variables are the extended columns [own_off, own_off + n_own)
 *   recv_start/recv_cnt   [nranks] my halo slots owned by peer p: extended columns [start, start+cnt)
 *   send_ptr/send_idx     [nranks+1] / [send_ptr[nranks]] owned extended columns peer p keeps as halo
 * jprod needs a gather of halo values (ncclSend/ncclRecv), jtprod a scatter-add of halo partial sums,
 * the Krylov inner products one ncclAllReduce of 4 doubles per half iteration.
 * Vectors: n-space arguments are the OWNED slices (n_own), m-space arguments the local rows (ncon).
 * fpsb_dist_unique_id: rank 0 makes the 128-byte ncclUniqueId the host program broadcasts. */
int fpsb_dist_unique_id(void *out128);
int fpsb_dist_attach(fpsb_handle h, int nranks, int rank, const void *nccl_id128, int64_t own_off,
                     int64_t n_own, const int64_t *recv_start, const int64_t *recv_cnt,
                     const int64_t *send_ptr, const int64_t *send_idx);
/* Peer-memory transport (NVLink / NVSwitch, up to 8 ranks of one node): every rank owns a mailbox in
 * HBM that its peers map through CUDA IPC; one small kernel per half iteration then does the halo
 * scatter-add, the boundary rows' epilogue, the halo gather and the all-reduction of the Krylov inner
 * products by writing into the peers' mailboxes and spinning on sequence flags — no NCCL call on the
 * iteration path (4 launches per Krylov iteration instead of 8 kernels + 4 NCCL operations).
 *   1. every rank: fpsb_dist_peer_export(h, blob)      blob = fpsb_dist_peer_blob_bytes() bytes
 *   2. the host program all-gathers the blobs (rank order)
 *   3. every rank: fpsb_dist_peer_attach(h, blobs)
 * Without these calls (or with FPSB_DIST_NCCL=1) the exchanges go through NCCL. */
int64_t fpsb_dist_peer_blob_bytes(void);
int fpsb_dist_peer_export(fpsb_handle h, void *blob_out);
int fpsb_dist_peer_attach(fpsb_handle h, const void *blobs);
int fpsb_dist_peer_active(fpsb_handle h);
/* Measurement only: fpsb_dist_profile(1) records a CUDA event after every launch of the row-partitioned
 * Krylov loop; fpsb_dist_last_profile returns, for the last profiled solve of this process, the mean
 * microseconds and the number of launches of {n-space step, exchange after it, m-space step, exchange
 * after it} (the exchange share of an iteration that bench.py reports). */
int fpsb_dist_profile(int on);
int fpsb_dist_last_profile(double mean_us[4], int64_t count[4]);
int fpsb_dist_jprod(fpsb_handle h, const double *x_own, double *y_loc, int loc);
int fpsb_dist_jtprod(fpsb_handle h, const double *u_loc, double *y_own, int loc);
int fpsb_dist_solve_two_mixed(fpsb_handle h, double delta, int64_t nvar_global, int64_t ncon_global,
                              const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2,
                              double *q2, int loc, fpsb_krylov_stats stats[2]);
int fpsb_dist_solve_two_least_squares(fpsb_handle h, double delta, int64_t nvar_global,
                                      int64_t ncon_global, const double *rhs1, const double *rhs2,
                                      double *p1, double *q1, double *p2, double *q2, int loc,
                                      fpsb_krylov_stats stats[2]);
/* solve_two_extras of IterativeSolver (src/solve_linear_system.jl:45-77) on the row-partitioned operator:
 * u1 = LSQR(A', rhs1, lambda = sqrt(tau)), u2 = MINRES(A A' + tau I, rhs2), tau = max(delta, 1e-14).
 * rhs1: the OWNED n-space slice; rhs2, u1, u2: the local m-space slices. */
int fpsb_dist_solve_two_extras(fpsb_handle h, double delta, int64_t nvar_global, int64_t ncon_global,
                               const double *rhs1, const double *rhs2, double *u1, double *u2, int loc,
                               fpsb_krylov_stats stats[2]);

/* ---------------------------------------------------------------------------------------------
 * Device-resident FletcherPenaltyNLP glue (SURVEY 8 f1): the vector combinations either side of the
 * 2-RHS solves, fused, on the handle's stream.  ALL vector arguments are DEVICE pointers (n = nvar,
 * m = ncon of the handle); together with loc = FPSB_DEVICE solves this keeps x, g, c, y(x) and the
 * penalty gradient in HBM across the outer loop of src/algo.jl.
 *   fpsb_fp_ys_gs   gs = p1 + sigma p2, ys = q1 + sigma q2, v = p2, w = q2   src/model-Fletcherpenaltynlp.jl:244-248
 *   fpsb_fp_hash    memo key of x computed on the device (replaces hash(x), :235)
 *   fpsb_fp_obj     phi = fx - c'ys + rho/2 |c|^2 (+ eta/2 |x - xk|^2)       :364-367   (x, xk may be NULL when eta = 0)
 *   fpsb_fp_grad    g = gs - Hsv + sigma v + Sstw (+ rho Jtc) (+ eta (x - xk))   :382-398
 *   fpsb_fp_ptv     Ptv = v - p1                                              :544
 *   fpsb_fp_hprod2  Hv = obj_weight (p2 - HsPtv + 2 sigma Ptv (+ Hcv + rho JtJv) (+ eta v))   :546-568 (Val(2))
 *   fpsb_fp_hprod1  Hv = obj_weight (p2 - HsPtv + 2 sigma Ptv - J'(JJ')^-1 Ss v - Ss'(JJ')^-1 J v (+ rho (Hcv + JtJv)) (+ eta v))
 *                   :572-634 (Val(1): the two extra terms come from ghjvprod + fpsb_*_solve_two_extras) */
int fpsb_fp_ys_gs(fpsb_handle h, double sigma, const double *p1, const double *q1, const double *p2,
                  const double *q2, double *gs, double *ys, double *v, double *w);
int fpsb_fp_hash(fpsb_handle h, const double *x, uint64_t *key);
int fpsb_fp_obj(fpsb_handle h, double fx, double rho, double eta, const double *c, const double *ys,
                const double *x, const double *xk, double *phi);
int fpsb_fp_grad(fpsb_handle h, double sigma, double rho, double eta, const double *gs, const double *Hsv,
                 const double *v, const double *Sstw, const double *Jtc, const double *x, const double *xk,
                 double *g);
int fpsb_fp_ptv(fpsb_handle h, const double *v, const double *p1, double *Ptv);
int fpsb_fp_hprod2(fpsb_handle h, double sigma, double rho, double eta, double obj_weight, const double *p2,
                   const double *HsPtv, const double *Ptv, const double *Hcv, const double *JtJv,
                   const double *v, double *Hv);
/* Steihaug-Toint truncated CG of the trust-region subproblem  min g's + s'Hs/2, |s| <= radius  (SURVEY 8 f3; in the
 * reference this is the third-party subproblem solver that calls obj / grad! / hprod! of FletcherPenaltyNLP,
 * src/parameters.jl:199-206, src/algo.jl:113-116).  All vectors are DEVICE pointers of length nvar; the caller supplies
 * Hd = H d between the calls (the 2-RHS solves).  free_mask (nullable): 1.0 on free variables, 0.0 on active bounds.
 * out = {rr, q (model value at s), tau (step taken along d), beta, flag}: flag 0 go on, 1 left through the boundary or
 * non-positive curvature (s is final), 2 converged (sqrt(rr) <= tol).  The five inner products, alpha, beta, the step
 * to the boundary and the exit decision are computed on the device; one 40-byte read-back per iteration.
 *   fpsb_trcg_init  s = 0, r = d = -g (masked), rr = r'r
 *   fpsb_trcg_step  one iteration given Hd: updates s, r, d in place */
int fpsb_trcg_init(fpsb_handle h, const double *g, const double *free_mask, double *s, double *r, double *d,
                   double out[5]);
int fpsb_trcg_step(fpsb_handle h, const double *Hd, const double *free_mask, double *s, double *r, double *d,
                   double radius, double tol, double out[5]);
int fpsb_fp_hprod1(fpsb_handle h, double sigma, double rho, double eta, double obj_weight, const double *p2,
                   const double *HsPtv, const double *Ptv, const double *JtinvJtJSsv, const double *SsinvJtJJv,
                   const double *Hcv, const double *JtJv, const double *v, double *Hv);

/* ---------------------------------------------------------------------------------------------
 * Batched FletcherPenaltyNLP glue: the entries above for `ninst` instances of ONE model (one handle), each at its own
 * point with its own sigma, rho, eta, xk and Jacobian values.  ALL arguments are DEVICE pointers; vectors are
 * instance-major, [ninst][nvar] or [ninst][ncon]; per-instance scalars are arrays [ninst].  rho, eta and obj_weight may
 * be NULL, which reads as 0 (obj_weight: 1) for every instance; a non-NULL rho needs its J'c / Hcv and J'Jv arguments
 * and a non-NULL eta needs x and xk, else FPSB_EINVAL (the checks of the single entries, made on the host without
 * reading the arrays).  The element-wise entries evaluate the single kernel's expression in its operation order, so
 * every entry is bitwise what the single entry gives on the same inputs; per-instance sums run inside one CTA, so
 * results do not depend on ninst or on an instance's position in the batch.  ninst == 0 is a no-op, a negative ninst
 * FPSB_EINVAL.  Asynchronous and ordered against the caller's stream (fpsb_set_caller_stream), except the CG entries,
 * which return after one 4-byte read-back.  None of them touches the handle's single-instance Jacobian values, Krylov
 * workspaces or the factors of fpsb_ldlt_batch_solve_two_mixed (Val(1): mixed -> least squares -> extras -> products).
 *   fpsb_fp_batch_ys_gs   fpsb_fp_ys_gs per instance                                  src/model-Fletcherpenaltynlp.jl:244-248
 *   fpsb_fp_batch_hash    keys [ninst] (device): key i is bit for bit fpsb_fp_hash of row i                     :235
 *   fpsb_fp_batch_obj     phi [ninst] (device) = fx - c'ys + rho/2 |c|^2 (+ eta/2 |x - xk|^2), fx [ninst]  :364-367
 *   fpsb_fp_batch_grad    fpsb_fp_grad per instance                                                     :382-398
 *   fpsb_fp_batch_ptv     fpsb_fp_ptv per instance                                                          :544
 *   fpsb_fp_batch_hprod2  fpsb_fp_hprod2 per instance, obj_weight [ninst]                               :546-568
 *   fpsb_fp_batch_hprod1  fpsb_fp_hprod1 per instance, obj_weight [ninst]                               :572-634
 *   fpsb_batch_jprod      out_i = A_i v_i  [ninst][ncon]  (jprod! of the rho-terms, :560-566; cons of linear models)
 *   fpsb_batch_jtprod     out_i = A_i' u_i [ninst][nvar]  (jtprod! of J'c :390, J'Jv :566, Val(1) :612)
 *                         jvals + i * jstride holds instance i's values in the COO order given to fpsb_create;
 *                         jstride is nnzj, or 0 when every instance shares one set of values.  One thread per output
 *                         row sums in plain CSR order, so results differ from fpsb_jprod / fpsb_jtprod (tiled SELL-32)
 *                         in the last bits. */
int fpsb_fp_batch_ys_gs(fpsb_handle h, int64_t ninst, const double *sigma, const double *p1, const double *q1,
                        const double *p2, const double *q2, double *gs, double *ys, double *v, double *w);
int fpsb_fp_batch_hash(fpsb_handle h, int64_t ninst, const double *x, uint64_t *keys);
int fpsb_fp_batch_obj(fpsb_handle h, int64_t ninst, const double *fx, const double *rho, const double *eta, const double *c,
                      const double *ys, const double *x, const double *xk, double *phi);
int fpsb_fp_batch_grad(fpsb_handle h, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                       const double *gs, const double *Hsv, const double *v, const double *Sstw, const double *Jtc,
                       const double *x, const double *xk, double *g);
int fpsb_fp_batch_ptv(fpsb_handle h, int64_t ninst, const double *v, const double *p1, double *Ptv);
int fpsb_fp_batch_hprod2(fpsb_handle h, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                         const double *obj_weight, const double *p2, const double *HsPtv, const double *Ptv, const double *Hcv,
                         const double *JtJv, const double *v, double *Hv);
int fpsb_fp_batch_hprod1(fpsb_handle h, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                         const double *obj_weight, const double *p2, const double *HsPtv, const double *Ptv,
                         const double *JtinvJtJSsv, const double *SsinvJtJJv, const double *Hcv, const double *JtJv,
                         const double *v, double *Hv);
int fpsb_batch_jprod(fpsb_handle h, int64_t ninst, const double *jvals, int64_t jstride, const double *v, double *out);
int fpsb_batch_jtprod(fpsb_handle h, int64_t ninst, const double *jvals, int64_t jstride, const double *u, double *out);
/* Batched Steihaug-Toint CG (fpsb_trcg_init / fpsb_trcg_step per instance, one CTA per instance, one kernel per
 * iteration).  g, free_mask (nullable), s, r, d, Hd [ninst][nvar]; radius, tol [ninst]; st [ninst][5] = {rr, q, tau,
 * beta, flag} as `out` of the single entry, except that init already sets flag 2 when sqrt(rr) <= tol (zero step, no
 * product); nprod [ninst] (int32) counts the products each instance consumed.  An instance whose flag is non-zero is
 * frozen: its s, r, d, st and nprod are not touched again, so the caller keeps computing Hd for the whole batch and
 * ignores the frozen rows.  *nactive (host) receives the number of instances still going: the one host
 * synchronisation per iteration of the whole batch. */
int fpsb_trcg_batch_init(fpsb_handle h, int64_t ninst, const double *g, const double *free_mask, const double *tol,
                         double *s, double *r, double *d, double *st, int32_t *nprod, int32_t *nactive);
int fpsb_trcg_batch_step(fpsb_handle h, int64_t ninst, const double *Hd, const double *free_mask, const double *radius,
                         const double *tol, double *s, double *r, double *d, double *st, int32_t *nprod, int32_t *nactive);

#ifdef __cplusplus
}
#endif
#endif /* FPSB_H */
