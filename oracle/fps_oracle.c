/*
 * fps_oracle.c — CPU ORACLE (TEST INFRASTRUCTURE ONLY; never on the product path).
 *
 * A plain-C restatement of the arithmetic behind FletcherPenaltySolver.jl's hot path:
 * the two-right-hand-side quasi-definite solves K = [I A'; A -delta*I].
 *
 *   reference call sites restated here
 *     src/solve_two_systems_struct.jl:308-353   LDLtSolver ctor: COO of triu(K), ldl_analyze, n_d/tol/r1/r2
 *     src/solve_linear_system.jl:206-252        solve_two_mixed [LDLt]
 *     src/solve_linear_system.jl:161-204        solve_two_least_squares [LDLt]
 *     src/solve_linear_system.jl:142-159        solve_two_extras [LDLt]  (cgls + minres, default tolerances)
 *     src/solve_linear_system.jl:107-140        solve_two_mixed [Iterative] (lsqr + craig)
 *     src/solve_linear_system.jl:79-105         solve_two_least_squares [Iterative] (lsqr, lsqr)
 *     src/solve_linear_system.jl:45-77          solve_two_extras [Iterative] (lsqr + minres)
 *     src/solve_two_systems_struct.jl:167-185   solve_least_square (lsqr call-site tolerances)
 *     src/solve_two_systems_struct.jl:210-244   solve_least_norm  (craig!, M=(1/delta) I, sqd=true)
 *
 * The arithmetic itself lives in un-vendored third-party Julia packages that are ABSENT from
 * /root/reference (Project.toml:25-38, no Manifest): LDLFactorizations.jl (compat 0.8/0.9/0.10),
 * Krylov.jl (0.10), SparseArrays (stdlib).  Their published algorithms are restated from
 * SURVEY.md Appendix B:
 *     B1  ldl_analyze      (Davis' LDL symbolic, upper-triangle variant, given a permutation P)
 *     B2  ldl_factorize!   (up-looking numeric LDL' + dynamic regularisation (n_d, tol, r1, r2))
 *     B3  ldiv!            (2-column permuted L, D, L' sweeps)
 *     B4  sparse(I,J,V)    (COO -> CSC, duplicates summed, explicit zeros kept, rows ascending)
 *     B5  lsqr / craig / minres / cgls with Krylov.jl's stopping rules
 *
 * PARITY PINNING: there is no Julia in this image, so the oracle cannot be checked against the
 * real packages.  It IS pinned against every golden vector the reference's own tests hold for this
 * path (test/unit-test.jl known answers, SURVEY Appendix C G1-G4 -> tests/golden/) and against an
 * independent dense numpy.linalg.solve on K.  Bit-level agreement with LDLFactorizations/Krylov
 * (pivot order of roundoff, iteration counts) is "parity unpinned" — see DESIGN.md.
 *
 * Indices are 0-based int64 here (the reference uses 1-based Int64).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <float.h>

typedef int64_t i64;

/* ------------------------------------------------------------------------------------------ */
/* B4: sparse(I, J, V, N, N)  — COO -> CSC, duplicates summed in order of appearance,          */
/* explicit zeros kept, row indices ascending within each column.                             */
/* Returns nnz of the CSC. Cp has N+1 entries; Ci/Cx need capacity nz.                        */
/* src_of (optional, capacity nz): for every COO entry, the CSC slot it was summed into.      */
/* ------------------------------------------------------------------------------------------ */
i64 fo_coo_to_csc(i64 N, i64 nz, const i64 *I, const i64 *J, const double *V,
                  i64 *Cp, i64 *Ci, double *Cx, i64 *slot_of)
{
    i64 *cnt = (i64 *)calloc((size_t)N + 1, sizeof(i64));
    i64 *ord = (i64 *)malloc((size_t)(nz > 0 ? nz : 1) * sizeof(i64));
    i64 *tmp = (i64 *)malloc((size_t)(nz > 0 ? nz : 1) * sizeof(i64));
    /* stable counting sort by row, then stable counting sort by column => (col,row) order,
       ties in order of appearance */
    i64 *rc = (i64 *)calloc((size_t)N + 1, sizeof(i64));
    for (i64 k = 0; k < nz; k++) rc[I[k] + 1]++;
    for (i64 i = 0; i < N; i++) rc[i + 1] += rc[i];
    for (i64 k = 0; k < nz; k++) tmp[rc[I[k]]++] = k;
    for (i64 k = 0; k < nz; k++) cnt[J[k] + 1]++;
    for (i64 j = 0; j < N; j++) cnt[j + 1] += cnt[j];
    i64 *pos = (i64 *)malloc((size_t)(N + 1) * sizeof(i64));
    memcpy(pos, cnt, (size_t)(N + 1) * sizeof(i64));
    for (i64 t = 0; t < nz; t++) { i64 k = tmp[t]; ord[pos[J[k]]++] = k; }
    /* compress duplicates */
    i64 out = 0;
    for (i64 j = 0; j < N; j++) {
        i64 start = out;
        (void)start;
        i64 p0 = cnt[j], p1 = cnt[j + 1];
        Cp[j] = out;
        i64 last_row = -1;
        for (i64 p = p0; p < p1; p++) {
            i64 k = ord[p];
            if (I[k] == last_row) {
                Cx[out - 1] += V ? V[k] : 0.0;
            } else {
                Ci[out] = I[k];
                Cx[out] = V ? V[k] : 0.0;
                last_row = I[k];
                out++;
            }
            if (slot_of) slot_of[k] = out - 1;
        }
    }
    Cp[N] = out;
    free(cnt); free(ord); free(tmp); free(rc); free(pos);
    return out;
}

/* ------------------------------------------------------------------------------------------ */
/* B1-B3: LDL' (LDLFactorizations.jl restated)                                                 */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    i64 n;
    i64 *P, *pinv;
    i64 *Cp, *Ci, *Cpos;      /* row form of the strict upper triangle (+ position of the value) */
    i64 *parent, *Lnz, *Lp, *Li;
    double *Lx, *D, *Y;
    i64 *pattern, *flag;
    signed char *reg;         /* reg[k] = 1: pivot k was replaced by the dynamic regularisation */
    double r1, r2, tol;
    i64 n_d;
    int factorized;
} fo_ldl;

void fo_ldl_free(fo_ldl *S)
{
    if (!S) return;
    free(S->P); free(S->pinv); free(S->Cp); free(S->Ci); free(S->Cpos);
    free(S->parent); free(S->Lnz); free(S->Lp); free(S->Li);
    free(S->Lx); free(S->D); free(S->Y); free(S->pattern); free(S->flag); free(S->reg);
    free(S);
}

/* ldl_analyze(A::Symmetric{:U}, P): A given as CSC (Ap, Ai) holding the upper triangle
   (entries with row > col are ignored).  P[k] = original index eliminated k-th. */
fo_ldl *fo_ldl_analyze(i64 n, const i64 *Ap, const i64 *Ai, const i64 *P)
{
    fo_ldl *S = (fo_ldl *)calloc(1, sizeof(fo_ldl));
    S->n = n;
    S->P = (i64 *)malloc((size_t)n * sizeof(i64));
    S->pinv = (i64 *)malloc((size_t)n * sizeof(i64));
    for (i64 k = 0; k < n; k++) { S->P[k] = P ? P[k] : k; S->pinv[S->P[k]] = k; }
    /* row form of the strict upper triangle: row r -> columns c > r */
    S->Cp = (i64 *)calloc((size_t)n + 1, sizeof(i64));
    for (i64 j = 0; j < n; j++)
        for (i64 p = Ap[j]; p < Ap[j + 1]; p++)
            if (Ai[p] < j) S->Cp[Ai[p] + 1]++;
    for (i64 i = 0; i < n; i++) S->Cp[i + 1] += S->Cp[i];
    i64 cn = S->Cp[n];
    S->Ci = (i64 *)malloc((size_t)(cn > 0 ? cn : 1) * sizeof(i64));
    S->Cpos = (i64 *)malloc((size_t)(cn > 0 ? cn : 1) * sizeof(i64));
    {
        i64 *w = (i64 *)malloc((size_t)(n + 1) * sizeof(i64));
        memcpy(w, S->Cp, (size_t)(n + 1) * sizeof(i64));
        for (i64 j = 0; j < n; j++)
            for (i64 p = Ap[j]; p < Ap[j + 1]; p++)
                if (Ai[p] < j) { i64 q = w[Ai[p]]++; S->Ci[q] = j; S->Cpos[q] = p; }
        free(w);
    }
    S->parent = (i64 *)malloc((size_t)n * sizeof(i64));
    S->Lnz = (i64 *)malloc((size_t)n * sizeof(i64));
    S->Lp = (i64 *)malloc((size_t)(n + 1) * sizeof(i64));
    S->flag = (i64 *)malloc((size_t)n * sizeof(i64));
    S->pattern = (i64 *)malloc((size_t)n * sizeof(i64));
    i64 *parent = S->parent, *Lnz = S->Lnz, *flag = S->flag, *pinv = S->pinv;
    /* ldl_symbolic_upper!: etree + column counts by row-subtree walks */
    for (i64 k = 0; k < n; k++) {
        parent[k] = -1; flag[k] = k; Lnz[k] = 0;
        i64 pk = S->P[k];
        for (i64 p = Ap[pk]; p < Ap[pk + 1]; p++) {
            if (Ai[p] > pk) continue;               /* not in the upper triangle */
            i64 i = pinv[Ai[p]];
            if (i >= k) continue;
            for (; flag[i] != k; i = parent[i]) {
                if (parent[i] == -1) parent[i] = k;
                Lnz[i]++; flag[i] = k;
            }
        }
        for (i64 q = S->Cp[pk]; q < S->Cp[pk + 1]; q++) {
            i64 i = pinv[S->Ci[q]];
            if (i >= k) continue;
            for (; flag[i] != k; i = parent[i]) {
                if (parent[i] == -1) parent[i] = k;
                Lnz[i]++; flag[i] = k;
            }
        }
    }
    S->Lp[0] = 0;
    for (i64 k = 0; k < n; k++) S->Lp[k + 1] = S->Lp[k] + Lnz[k];
    i64 lnz = S->Lp[n];
    S->Li = (i64 *)malloc((size_t)(lnz > 0 ? lnz : 1) * sizeof(i64));
    S->Lx = (double *)malloc((size_t)(lnz > 0 ? lnz : 1) * sizeof(double));
    S->D = (double *)calloc((size_t)n, sizeof(double));
    S->Y = (double *)calloc((size_t)n, sizeof(double));
    S->reg = (signed char *)calloc((size_t)(n > 0 ? n : 1), 1);
    S->factorized = 0;
    return S;
}

void fo_ldl_set_reg(fo_ldl *S, i64 n_d, double tol, double r1, double r2)
{ S->n_d = n_d; S->tol = tol; S->r1 = r1; S->r2 = r2; }

i64 fo_ldl_n(const fo_ldl *S) { return S->n; }
i64 fo_ldl_lnz(const fo_ldl *S) { return S->Lp[S->n]; }
int fo_ldl_factorized(const fo_ldl *S) { return S->factorized; }
/* copy-out for the bit-exact symbolic comparison. After a numeric factorisation Lnz/Li are those
   of the numeric pass (identical to the symbolic ones by construction). */
void fo_ldl_get_symbolic(const fo_ldl *S, i64 *P, i64 *parent, i64 *Lnz, i64 *Lp, i64 *Li)
{
    i64 n = S->n;
    if (P) memcpy(P, S->P, (size_t)n * sizeof(i64));
    if (parent) memcpy(parent, S->parent, (size_t)n * sizeof(i64));
    if (Lnz) for (i64 k = 0; k < n; k++) Lnz[k] = S->Lp[k + 1] - S->Lp[k];
    if (Lp) memcpy(Lp, S->Lp, (size_t)(n + 1) * sizeof(i64));
    if (Li) memcpy(Li, S->Li, (size_t)S->Lp[n] * sizeof(i64));
}
void fo_ldl_get_numeric(const fo_ldl *S, double *Lx, double *D)
{
    if (Lx) memcpy(Lx, S->Lx, (size_t)S->Lp[S->n] * sizeof(double));
    if (D) memcpy(D, S->D, (size_t)S->n * sizeof(double));
}

/* reg[k] = 1 where the last factorisation regularised pivot k (permuted order) */
void fo_ldl_get_regularised(const fo_ldl *S, signed char *reg) { memcpy(reg, S->reg, (size_t)S->n); }

/* ldl_factorize!(A, S): up-looking LDL' on the permuted matrix; dynamic regularisation.
   Returns 1 when factorised, 0 when a zero pivot was met (S->factorized mirrors it). */
int fo_ldl_factorize(fo_ldl *S, const i64 *Ap, const i64 *Ai, const double *Ax)
{
    i64 n = S->n;
    i64 *parent = S->parent, *Lnz = S->Lnz, *Lp = S->Lp, *Li = S->Li, *flag = S->flag,
        *pattern = S->pattern, *pinv = S->pinv;
    double *Lx = S->Lx, *D = S->D, *Y = S->Y;
    int dynamic_reg = (S->r1 != 0.0) || (S->r2 != 0.0);
    S->factorized = 0;
    for (i64 k = 0; k < n; k++) {
        Y[k] = 0.0;
        i64 top = n;
        flag[k] = k;
        Lnz[k] = 0;
        i64 pk = S->P[k];
        for (i64 p = Ap[pk]; p < Ap[pk + 1]; p++) {
            if (Ai[p] > pk) continue;
            i64 i = pinv[Ai[p]];
            if (i > k) continue;
            Y[i] += Ax[p];
            i64 len = 0;
            for (; flag[i] != k; i = parent[i]) { pattern[len++] = i; flag[i] = k; }
            while (len > 0) pattern[--top] = pattern[--len];
        }
        for (i64 q = S->Cp[pk]; q < S->Cp[pk + 1]; q++) {
            i64 i = pinv[S->Ci[q]];
            if (i > k) continue;
            Y[i] += Ax[S->Cpos[q]];
            i64 len = 0;
            for (; flag[i] != k; i = parent[i]) { pattern[len++] = i; flag[i] = k; }
            while (len > 0) pattern[--top] = pattern[--len];
        }
        D[k] = Y[k];
        Y[k] = 0.0;
        for (; top < n; top++) {
            i64 i = pattern[top];
            double yi = Y[i];
            Y[i] = 0.0;
            i64 p2 = Lp[i] + Lnz[i];
            i64 p;
            for (p = Lp[i]; p < p2; p++) Y[Li[p]] -= Lx[p] * yi;
            double l_ki = yi / D[i];
            D[k] -= l_ki * yi;
            Li[p] = k;
            Lx[p] = l_ki;
            Lnz[i]++;
        }
        S->reg[k] = dynamic_reg && fabs(D[k]) < S->tol;
        if (S->reg[k]) {
            double r = (S->P[k] < S->n_d) ? S->r1 : S->r2;
            double sgn = (r > 0) - (r < 0);
            double a = fabs(D[k] + r), b = fabs(r);
            D[k] = sgn * (a > b ? a : b);
        }
        if (D[k] == 0.0) return 0;
    }
    S->factorized = 1;
    return 1;
}

/* ldiv!(S, B): B is n x 2 column-major; overwritten by the solution of K x = b. */
void fo_ldl_solve2(fo_ldl *S, double *B)
{
    i64 n = S->n;
    const i64 *Lp = S->Lp, *Li = S->Li, *P = S->P;
    const double *Lx = S->Lx, *D = S->D;
    double *y = (double *)malloc((size_t)n * 2 * sizeof(double));
    for (i64 k = 0; k < n; k++) { y[2 * k] = B[P[k]]; y[2 * k + 1] = B[n + P[k]]; }
    for (i64 j = 0; j < n; j++) {
        double a = y[2 * j], b = y[2 * j + 1];
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) {
            i64 i = Li[p];
            y[2 * i] -= Lx[p] * a;
            y[2 * i + 1] -= Lx[p] * b;
        }
    }
    for (i64 j = 0; j < n; j++) { y[2 * j] /= D[j]; y[2 * j + 1] /= D[j]; }
    for (i64 j = n - 1; j >= 0; j--) {
        double a = y[2 * j], b = y[2 * j + 1];
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) {
            i64 i = Li[p];
            a -= Lx[p] * y[2 * i];
            b -= Lx[p] * y[2 * i + 1];
        }
        y[2 * j] = a; y[2 * j + 1] = b;
    }
    for (i64 k = 0; k < n; k++) { B[P[k]] = y[2 * k]; B[n + P[k]] = y[2 * k + 1]; }
    free(y);
}

/* ------------------------------------------------------------------------------------------ */
/* Operators: A (m x n) stored twice as CSR (A and A').  jprod = A*v, jtprod = A'*u.           */
/* B6: jac_op! products.                                                                      */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    i64 m, n;
    const i64 *rp, *ci; const double *vx;      /* CSR of A  */
    const i64 *trp, *tci; const double *tvx;   /* CSR of A' */
} fo_mat;

/* -DFO_OMP (oracle/Makefile: libfps_oracle_omp.so) threads the row loops and the element-wise loops of the
 * Krylov methods for bench.py's reference arm ("all the host threads it can use").  The checker used by the
 * tests is always the sequential build: its sums have one fixed order. */
#ifdef FO_OMP
#define FO_PAR _Pragma("omp parallel for schedule(static)")
#define FO_PAR_SUM _Pragma("omp parallel for schedule(static) reduction(+:s)")
#else
#define FO_PAR
#define FO_PAR_SUM
#endif
static void csr_mv(i64 nr, const i64 *rp, const i64 *ci, const double *vx, const double *x, double *y)
{
    FO_PAR for (i64 i = 0; i < nr; i++) {
        double s = 0.0;
        for (i64 p = rp[i]; p < rp[i + 1]; p++) s += vx[p] * x[ci[p]];
        y[i] = s;
    }
}
/* op kinds: 0: A (m x n)   1: A' (n x m)   2: A*A' (m x m, symmetric; tmp needed) */
typedef struct { const fo_mat *M; int kind; double *tmp; } fo_op;
static i64 op_rows(const fo_op *o) { return o->kind == 1 ? o->M->n : o->M->m; }
static i64 op_cols(const fo_op *o) { return o->kind == 0 ? o->M->n : o->M->m; }
static void op_mul(const fo_op *o, const double *x, double *y)
{
    const fo_mat *M = o->M;
    if (o->kind == 0) csr_mv(M->m, M->rp, M->ci, M->vx, x, y);
    else if (o->kind == 1) csr_mv(M->n, M->trp, M->tci, M->tvx, x, y);
    else { csr_mv(M->n, M->trp, M->tci, M->tvx, x, o->tmp); csr_mv(M->m, M->rp, M->ci, M->vx, o->tmp, y); }
}
static void op_tmul(const fo_op *o, const double *x, double *y)
{
    const fo_mat *M = o->M;
    if (o->kind == 0) csr_mv(M->n, M->trp, M->tci, M->tvx, x, y);
    else if (o->kind == 1) csr_mv(M->m, M->rp, M->ci, M->vx, x, y);
    else op_mul(o, x, y);
}

static double dotr(i64 n, const double *a, const double *b)
{ double s = 0.0; FO_PAR_SUM for (i64 i = 0; i < n; i++) s += a[i] * b[i]; return s; }
static double nrm2(i64 n, const double *a) { return sqrt(dotr(n, a, a)); }

/* Krylov.jl sym_givens */
static void sym_givens(double a, double b, double *c, double *s, double *rho)
{
    if (b == 0.0) {
        *c = (a == 0.0) ? 1.0 : (double)((a > 0) - (a < 0));
        *s = 0.0; *rho = fabs(a);
    } else if (a == 0.0) {
        *c = 0.0; *s = (double)((b > 0) - (b < 0)); *rho = fabs(b);
    } else if (fabs(b) > fabs(a)) {
        double t = a / b;
        *s = (double)((b > 0) - (b < 0)) / sqrt(1.0 + t * t);
        *c = *s * t; *rho = b / *s;
    } else {
        double t = b / a;
        *c = (double)((a > 0) - (a < 0)) / sqrt(1.0 + t * t);
        *s = *c * t; *rho = a / *c;
    }
}

/* status codes shared with include/fpsb.h */
enum {
    FO_ST_UNKNOWN = 0, FO_ST_ZERO_RHS = 1, FO_ST_SOLVED = 2, FO_ST_ZERO_RESID = 3, FO_ST_FWD_ERR = 4,
    FO_ST_TIRED = 5, FO_ST_ILLCOND_MACH = 6, FO_ST_ILLCOND_LIM = 7, FO_ST_INCONSISTENT = 8,
    FO_ST_ZERO_ATB = 9
};
typedef struct {
    i64 niter; int32_t solved; int32_t inconsistent; int32_t status; int32_t pad;
    double rnorm; double arnorm; double anorm; double acond; double xnorm;
} fo_stats;

#define WINDOW 5

/* ---- LSQR (Krylov.jl lsqr!, M = N = I, radius = 0) ---------------------------------------- */
/* min ||b - Op x||^2 + lambda^2 ||x||^2.  x has op_cols entries.                             */
void fo_lsqr(const fo_op *Op, const double *b, double lambda, double atol, double rtol,
             double axtol, double btol, double etol, double conlim, i64 itmax,
             double *x, fo_stats *st)
{
    i64 m = op_rows(Op), n = op_cols(Op);
    double *u = (double *)malloc((size_t)m * sizeof(double));
    double *v = (double *)malloc((size_t)n * sizeof(double));
    double *w = (double *)malloc((size_t)n * sizeof(double));
    double *Av = (double *)malloc((size_t)m * sizeof(double));
    double *Atu = (double *)malloc((size_t)n * sizeof(double));
    memset(st, 0, sizeof(*st));
    double lambda2 = lambda * lambda;
    double ctol = conlim > 0 ? 1.0 / conlim : 0.0;
    FO_PAR for (i64 i = 0; i < n; i++) x[i] = 0.0;
    memcpy(u, b, (size_t)m * sizeof(double));
    double beta1 = nrm2(m, u);
    if (beta1 == 0.0) {
        st->niter = 0; st->solved = 1; st->inconsistent = 0; st->status = FO_ST_ZERO_RHS;
        goto done;
    }
    {
    double beta = beta1;
    FO_PAR for (i64 i = 0; i < m; i++) u[i] /= beta1;
    op_tmul(Op, u, Atu);
    memcpy(v, Atu, (size_t)n * sizeof(double));
    double Anorm2 = dotr(n, v, v);
    double Anorm = sqrt(Anorm2);
    double alpha = Anorm;
    double Acond = 0.0, xNorm = 0.0, xNorm2 = 0.0, dNorm2 = 0.0;
    double c2 = -1.0, s2 = 0.0, z = 0.0;
    double xENorm2 = 0.0, err_lbnd = 0.0;
    double err_vec[WINDOW] = {0, 0, 0, 0, 0};
    i64 iter = 0;
    if (itmax == 0) itmax = m + n;
    double rNorm = beta1, res2 = 0.0;
    double ArNorm = alpha * beta, ArNorm0 = ArNorm;
    if (alpha == 0.0) {
        st->niter = 0; st->solved = 1; st->inconsistent = 0; st->status = FO_ST_ZERO_ATB;
        st->rnorm = rNorm; goto done;
    }
    FO_PAR for (i64 i = 0; i < n; i++) v[i] /= alpha;
    memcpy(w, v, (size_t)n * sizeof(double));
    double phibar = beta1, rhobar = alpha;
    int solved_lim = ArNorm / (Anorm * rNorm) <= axtol;
    int solved_mach = 1.0 + ArNorm / (Anorm * rNorm) <= 1.0;
    int solved = solved_mach | solved_lim;
    int tired = iter >= itmax;
    int ill_cond = 0, ill_cond_mach = 0, ill_cond_lim = 0;
    int zero_resid_lim = rNorm / beta1 <= axtol;
    int zero_resid_mach = 1.0 + rNorm / beta1 <= 1.0;
    int zero_resid = zero_resid_mach | zero_resid_lim;
    int fwd_err = 0;
    while (!(solved || tired || ill_cond)) {
        iter++;
        /* beta_{k+1} u_{k+1} = A v_k - alpha_k u_k */
        op_mul(Op, v, Av);
        FO_PAR for (i64 i = 0; i < m; i++) u[i] = Av[i] - alpha * u[i];
        beta = nrm2(m, u);
        if (beta != 0.0) {
            FO_PAR for (i64 i = 0; i < m; i++) u[i] /= beta;
            Anorm2 = Anorm2 + alpha * alpha + beta * beta;
            if (lambda > 0) Anorm2 += lambda2;
            /* alpha_{k+1} v_{k+1} = A' u_{k+1} - beta_{k+1} v_k */
            op_tmul(Op, u, Atu);
            FO_PAR for (i64 i = 0; i < n; i++) v[i] = Atu[i] - beta * v[i];
            alpha = nrm2(n, v);
            if (alpha != 0.0) FO_PAR for (i64 i = 0; i < n; i++) v[i] /= alpha;
        }
        double c1, s1, rhobar1;
        sym_givens(rhobar, lambda, &c1, &s1, &rhobar1);
        double psi = s1 * phibar;
        phibar = c1 * phibar;
        double c, s, rho;
        sym_givens(rhobar1, beta, &c, &s, &rho);
        double phi = c * phibar;
        phibar = s * phibar;
        xENorm2 += phi * phi;
        err_vec[iter % WINDOW] = phi;
        if (iter >= WINDOW) err_lbnd = nrm2(WINDOW, err_vec);
        double tau = s * phi;
        double theta = s * alpha;
        rhobar = -c * alpha;
        dNorm2 += dotr(n, w, w) / (rho * rho);
        double sigma = phi / rho;
        FO_PAR for (i64 i = 0; i < n; i++) x[i] += sigma * w[i];
        double tr = theta / rho;
        FO_PAR for (i64 i = 0; i < n; i++) w[i] = v[i] - tr * w[i];
        double delta = s2 * rho;
        double gammabar = -c2 * rho;
        double rhs = phi - delta * z;
        double zbar = rhs / gammabar;
        xNorm = sqrt(xNorm2 + zbar * zbar);
        double gamma;
        sym_givens(gammabar, theta, &c2, &s2, &gamma);
        z = rhs / gamma;
        xNorm2 += z * z;
        Anorm = sqrt(Anorm2);
        Acond = Anorm * sqrt(dNorm2);
        double res1 = phibar * phibar;
        res2 += psi * psi;
        rNorm = sqrt(res1 + res2);
        ArNorm = alpha * fabs(tau);
        double test1 = rNorm / beta1;
        double test2 = ArNorm / (Anorm * rNorm);
        double test3 = 1.0 / Acond;
        double t1 = test1 / (1.0 + Anorm * xNorm / beta1);
        double rNormtol = btol + axtol * Anorm * xNorm / beta1;
        ill_cond_mach = (1.0 + test3 <= 1.0);
        solved_mach = (1.0 + test2 <= 1.0);
        zero_resid_mach = (1.0 + t1 <= 1.0);
        tired = iter >= itmax;
        ill_cond_lim = (test3 <= ctol);
        solved_lim = (test2 <= axtol);
        int solved_opt = ArNorm <= atol + rtol * ArNorm0;
        zero_resid_lim = (test1 <= rNormtol);
        if (iter >= WINDOW) fwd_err = err_lbnd <= etol * sqrt(xENorm2);
        ill_cond = ill_cond_mach || ill_cond_lim;
        zero_resid = zero_resid_mach || zero_resid_lim;
        solved = solved_mach || solved_lim || solved_opt || zero_resid || fwd_err;
    }
    int status = FO_ST_UNKNOWN;
    if (tired) status = FO_ST_TIRED;
    if (ill_cond_mach) status = FO_ST_ILLCOND_MACH;
    if (ill_cond_lim) status = FO_ST_ILLCOND_LIM;
    if (solved) status = FO_ST_SOLVED;
    if (zero_resid) status = FO_ST_ZERO_RESID;
    if (fwd_err) status = FO_ST_FWD_ERR;
    st->niter = iter; st->solved = solved; st->inconsistent = !zero_resid; st->status = status;
    st->rnorm = rNorm; st->arnorm = ArNorm; st->anorm = Anorm; st->acond = Acond; st->xnorm = xNorm;
    }
done:
    free(u); free(v); free(w); free(Av); free(Atu);
}

/* ---- CRAIG (Krylov.jl craig!, N = I, M = mscale * I (mscale = 1 when unused)) -------------- */
/* sqd != 0 forces lambda = 1.  Solves  A x + (lambda^2/mscale) y = b, x = A' y  (sqd form)    */
/* x has op_cols (n) entries, y has op_rows (m) entries.                                       */
void fo_craig(const fo_op *Op, const double *b, int sqd, double mscale, double lambda,
              double atol, double rtol, double btol, double conlim, i64 itmax,
              double *x, double *y, fo_stats *st)
{
    i64 m = op_rows(Op), n = op_cols(Op);
    double *Mu = (double *)malloc((size_t)m * sizeof(double));
    double *u = (double *)malloc((size_t)m * sizeof(double));
    double *v = (double *)calloc((size_t)n, sizeof(double));
    double *w = (double *)calloc((size_t)m, sizeof(double));
    double *w2 = (double *)calloc((size_t)n, sizeof(double));
    double *Av = (double *)malloc((size_t)m * sizeof(double));
    double *Atu = (double *)malloc((size_t)n * sizeof(double));
    memset(st, 0, sizeof(*st));
    if (sqd) lambda = 1.0;
    FO_PAR for (i64 i = 0; i < n; i++) x[i] = 0.0;
    FO_PAR for (i64 i = 0; i < m; i++) y[i] = 0.0;
    memcpy(Mu, b, (size_t)m * sizeof(double));
    FO_PAR for (i64 i = 0; i < m; i++) u[i] = mscale * Mu[i];
    double beta1 = sqrt(dotr(m, u, Mu));
    double rNorm = beta1;
    if (beta1 == 0.0) {
        st->niter = 0; st->solved = 1; st->inconsistent = 0; st->status = FO_ST_ZERO_RHS;
        goto done;
    }
    {
    double beta1sq = beta1 * beta1;
    double beta = beta1, theta = beta1, xi = -1.0, delta = lambda, rho_prev = 1.0;
    FO_PAR for (i64 i = 0; i < m; i++) { u[i] /= beta1; Mu[i] /= beta1; }
    double Anorm2 = 0.0, Anorm = 0.0, Dnorm2 = 0.0, Acond = 0.0, xNorm2 = 0.0;
    i64 iter = 0;
    if (itmax == 0) itmax = m + n;
    double eps_c = atol + rtol * rNorm;
    double ctol = conlim > 0 ? 1.0 / conlim : 0.0;
    double bkwerr = 1.0;
    int solved_lim = bkwerr <= btol;
    int solved_mach = 1.0 + bkwerr <= 1.0;
    int solved_resid_tol = rNorm <= eps_c;
    int solved_resid_lim = rNorm <= btol + atol * Anorm * sqrt(xNorm2) / beta1;
    int solved = solved_mach | solved_lim | solved_resid_tol | solved_resid_lim;
    int ill_cond = 0, ill_cond_mach = 0, ill_cond_lim = 0, inconsistent = 0;
    int tired = iter >= itmax;
    double c1 = 1.0, s1 = 0.0, rho;
    while (!(solved || inconsistent || ill_cond || tired)) {
        /* alpha_{k+1} v_{k+1} = A' u_{k+1} - beta_{k+1} v_k */
        op_tmul(Op, u, Atu);
        FO_PAR for (i64 i = 0; i < n; i++) v[i] = Atu[i] - beta * v[i];
        double alpha = nrm2(n, v);
        if (alpha == 0.0) { inconsistent = 1; continue; }
        FO_PAR for (i64 i = 0; i < n; i++) v[i] /= alpha;
        Anorm2 += alpha * alpha;
        if (lambda > 0) sym_givens(alpha, delta, &c1, &s1, &rho);
        else rho = alpha;
        xi = -theta / rho * xi;
        if (lambda > 0) {
            FO_PAR for (i64 i = 0; i < n; i++) x[i] += xi * c1 * v[i];
            FO_PAR for (i64 i = 0; i < n; i++) x[i] += xi * s1 * w2[i];
            FO_PAR for (i64 i = 0; i < n; i++) w2[i] = s1 * v[i] - c1 * w2[i];
        } else {
            FO_PAR for (i64 i = 0; i < n; i++) x[i] += xi * v[i];
        }
        double tr = theta / rho_prev, xr = xi / rho;
        FO_PAR for (i64 i = 0; i < m; i++) w[i] = u[i] - tr * w[i];
        FO_PAR for (i64 i = 0; i < m; i++) y[i] += xr * w[i];
        /* Krylov.jl craig.jl accumulates the 2-norm (not its square) here; kept as upstream. */
        Dnorm2 += nrm2(m, w);
        /* beta_{k+1} M u_{k+1} = A v_k - alpha_k M u_k */
        op_mul(Op, v, Av);
        FO_PAR for (i64 i = 0; i < m; i++) Mu[i] = Av[i] - alpha * Mu[i];
        FO_PAR for (i64 i = 0; i < m; i++) u[i] = mscale * Mu[i];
        beta = sqrt(dotr(m, u, Mu));
        if (beta != 0.0) FO_PAR for (i64 i = 0; i < m; i++) { u[i] /= beta; Mu[i] /= beta; }
        double gamma = 0.0;
        if (lambda > 0) { theta = c1 * beta; gamma = s1 * beta; }
        else theta = beta;
        if (lambda > 0) {
            double c2, s2;
            sym_givens(lambda, gamma, &c2, &s2, &delta);
            FO_PAR for (i64 i = 0; i < n; i++) w2[i] *= s2;
        }
        Anorm2 += beta * beta;
        Anorm = sqrt(Anorm2);
        Acond = Anorm * sqrt(Dnorm2);
        xNorm2 += xi * xi;
        rNorm = beta * fabs(xi);
        if (lambda > 0) rNorm *= fabs(c1);
        iter++;
        bkwerr = rNorm / sqrt(beta1sq + Anorm2 * xNorm2);
        rho_prev = rho;
        solved_lim = bkwerr <= btol;
        solved_mach = 1.0 + bkwerr <= 1.0;
        solved_resid_tol = rNorm <= eps_c;
        solved_resid_lim = rNorm <= btol + atol * Anorm * sqrt(xNorm2) / beta1;
        solved = solved_mach | solved_lim | solved_resid_tol | solved_resid_lim;
        ill_cond_mach = 1.0 + 1.0 / Acond <= 1.0;
        ill_cond_lim = 1.0 / Acond <= ctol;
        ill_cond = ill_cond_mach | ill_cond_lim;
        inconsistent = 0;
        tired = iter >= itmax;
    }
    int status = FO_ST_UNKNOWN;
    if (tired) status = FO_ST_TIRED;
    if (solved) status = FO_ST_SOLVED;
    if (ill_cond_mach) status = FO_ST_ILLCOND_MACH;
    if (ill_cond_lim) status = FO_ST_ILLCOND_LIM;
    if (inconsistent) status = FO_ST_INCONSISTENT;
    st->niter = iter; st->solved = solved; st->inconsistent = inconsistent; st->status = status;
    st->rnorm = rNorm; st->anorm = Anorm; st->acond = Acond; st->xnorm = sqrt(xNorm2);
    }
done:
    free(Mu); free(u); free(v); free(w); free(w2); free(Av); free(Atu);
}

/* ---- MINRES (Krylov.jl minres!, M = I, no warm start): (Op + lambda I) x = b -------------- */
void fo_minres(const fo_op *Op, const double *b, double lambda, double atol, double rtol,
               double etol, double conlim, i64 itmax, double *x, fo_stats *st)
{
    i64 n = op_rows(Op);
    double *r1 = (double *)malloc((size_t)n * sizeof(double));
    double *r2 = (double *)malloc((size_t)n * sizeof(double));
    double *w1 = (double *)calloc((size_t)n, sizeof(double));
    double *w2 = (double *)calloc((size_t)n, sizeof(double));
    double *y = (double *)malloc((size_t)n * sizeof(double));
    memset(st, 0, sizeof(*st));
    const double epsM = DBL_EPSILON;
    double ctol = conlim > 0 ? 1.0 / conlim : 0.0;
    FO_PAR for (i64 i = 0; i < n; i++) x[i] = 0.0;
    memcpy(r1, b, (size_t)n * sizeof(double));
    memcpy(r2, r1, (size_t)n * sizeof(double));
    double *v = r2;
    double beta1 = dotr(n, r1, v);
    if (beta1 == 0.0) {
        st->niter = 0; st->solved = 1; st->inconsistent = 0; st->status = FO_ST_ZERO_RHS;
        goto done;
    }
    {
    beta1 = sqrt(beta1);
    double beta = beta1, oldbeta = 0.0, deltabar = 0.0, eps_ = 0.0;
    double rNorm = beta1, phibar = beta1, rhs1 = beta1, rhs2 = 0.0;
    double gmax = 0.0, gmin = INFINITY, cs = -1.0, sn = 0.0;
    double ANorm2 = 0.0, ANorm = 0.0, Acond = 0.0, ArNorm = 0.0, xNorm = 0.0;
    double xENorm2 = 0.0, err_lbnd = 0.0;
    double err_vec[WINDOW] = {0, 0, 0, 0, 0};
    i64 iter = 0;
    if (itmax == 0) itmax = 2 * n;
    double tol = atol + rtol * beta1;
    int solved = (rNorm <= rtol), solved_mach = solved, solved_lim = solved;
    int tired = iter >= itmax;
    int ill_cond = 0, ill_cond_mach = 0, ill_cond_lim = 0;
    int zero_resid = (rNorm <= tol), zero_resid_mach = zero_resid, zero_resid_lim = zero_resid;
    int fwd_err = 0, resid_decrease = 0;
    int early_ls = 0;
    (void)solved_mach; (void)solved_lim; (void)zero_resid_mach; (void)zero_resid_lim;
    while (!(solved || tired || ill_cond)) {
        iter++;
        op_mul(Op, v, y);
        if (lambda != 0.0) FO_PAR for (i64 i = 0; i < n; i++) y[i] += lambda * v[i];
        FO_PAR for (i64 i = 0; i < n; i++) y[i] /= beta;
        if (iter >= 2) { double c = beta / oldbeta; FO_PAR for (i64 i = 0; i < n; i++) y[i] -= c * r1[i]; }
        double alpha = dotr(n, v, y) / beta;
        { double c = alpha / beta; FO_PAR for (i64 i = 0; i < n; i++) y[i] -= c * r2[i]; }
        double delta = cs * deltabar + sn * alpha;
        double *w;
        if (iter == 1) w = w2;
        else {
            if (iter >= 3) FO_PAR for (i64 i = 0; i < n; i++) w1[i] *= -eps_;
            w = w1;
            FO_PAR for (i64 i = 0; i < n; i++) w[i] -= delta * w2[i];
        }
        { double c = 1.0 / beta; FO_PAR for (i64 i = 0; i < n; i++) w[i] += c * v[i]; }
        memcpy(r1, r2, (size_t)n * sizeof(double));
        memcpy(r2, y, (size_t)n * sizeof(double));
        oldbeta = beta;
        beta = dotr(n, r2, v);
        beta = sqrt(beta);
        ANorm2 = ANorm2 + alpha * alpha + oldbeta * oldbeta + beta * beta;
        double gammabar = sn * deltabar - cs * alpha;
        eps_ = sn * beta;
        deltabar = -cs * beta;
        double root = sqrt(gammabar * gammabar + deltabar * deltabar);
        ArNorm = phibar * root;
        double gamma = sqrt(gammabar * gammabar + beta * beta);
        gamma = gamma > epsM ? gamma : epsM;
        cs = gammabar / gamma;
        sn = beta / gamma;
        double phi = cs * phibar;
        phibar = sn * phibar;
        { double c = 1.0 / gamma; FO_PAR for (i64 i = 0; i < n; i++) w[i] *= c; }
        FO_PAR for (i64 i = 0; i < n; i++) x[i] += phi * w[i];
        xENorm2 += phi * phi;
        if (iter >= 2) { double *t = w1; w1 = w2; w2 = t; }
        err_vec[iter % WINDOW] = phi;
        if (iter >= WINDOW) err_lbnd = nrm2(WINDOW, err_vec);
        gmax = gmax > gamma ? gmax : gamma;
        gmin = gmin < gamma ? gmin : gamma;
        double zeta = rhs1 / gamma;
        rhs1 = rhs2 - delta * zeta;
        rhs2 = -eps_ * zeta;
        ANorm = sqrt(ANorm2);
        xNorm = nrm2(n, x);
        rNorm = phibar;
        double test1 = rNorm / (ANorm * xNorm);
        double test2 = root / ANorm;
        Acond = gmax / gmin;
        if (iter == 1 && beta / beta1 <= 10 * epsM) { early_ls = 1; break; }
        ill_cond_mach = (1.0 + 1.0 / Acond <= 1.0);
        solved_mach = (1.0 + test2 <= 1.0);
        zero_resid_mach = (1.0 + test1 <= 1.0);
        int resid_decrease_mach = (rNorm + 1.0 <= 1.0);
        tired = iter >= itmax;
        ill_cond_lim = (1.0 / Acond <= ctol);
        solved_lim = (test2 <= tol);
        zero_resid_lim = (test1 <= tol);
        int resid_decrease_lim = (rNorm <= tol);
        if (iter >= WINDOW) fwd_err = err_lbnd <= etol * sqrt(xENorm2);
        zero_resid = zero_resid_mach | zero_resid_lim;
        resid_decrease = resid_decrease_mach | resid_decrease_lim;
        ill_cond = ill_cond_mach | ill_cond_lim;
        solved = solved_mach | solved_lim | zero_resid | fwd_err | resid_decrease;
    }
    int status = FO_ST_UNKNOWN;
    if (early_ls) { st->niter = 1; st->solved = 1; st->inconsistent = 1; st->status = FO_ST_ZERO_ATB; }
    else {
        if (tired) status = FO_ST_TIRED;
        if (ill_cond_mach) status = FO_ST_ILLCOND_MACH;
        if (ill_cond_lim) status = FO_ST_ILLCOND_LIM;
        if (solved) status = FO_ST_SOLVED;
        if (zero_resid) status = FO_ST_ZERO_RESID;
        if (fwd_err) status = FO_ST_FWD_ERR;
        if (resid_decrease) status = FO_ST_SOLVED;
        st->niter = iter; st->solved = solved; st->inconsistent = !zero_resid; st->status = status;
    }
    st->rnorm = rNorm; st->arnorm = ArNorm; st->anorm = ANorm; st->acond = Acond; st->xnorm = xNorm;
    }
done:
    /* w1/w2 may have been swapped; free both (order irrelevant) */
    free(r1); free(r2); free(w1); free(w2); free(y);
}

/* ---- CGLS (Krylov.jl cgls!, M = I, radius = 0): min ||b - Op x||^2 + lambda ||x||^2 -------- */
void fo_cgls(const fo_op *Op, const double *b, double lambda, double atol, double rtol, i64 itmax,
             double *x, fo_stats *st)
{
    i64 m = op_rows(Op), n = op_cols(Op);
    double *r = (double *)malloc((size_t)m * sizeof(double));
    double *q = (double *)malloc((size_t)m * sizeof(double));
    double *s = (double *)malloc((size_t)n * sizeof(double));
    double *p = (double *)malloc((size_t)n * sizeof(double));
    memset(st, 0, sizeof(*st));
    FO_PAR for (i64 i = 0; i < n; i++) x[i] = 0.0;
    memcpy(r, b, (size_t)m * sizeof(double));
    double bNorm = nrm2(m, r);
    if (bNorm == 0.0) { st->niter = 0; st->solved = 1; st->status = FO_ST_ZERO_RHS; goto done; }
    {
    op_tmul(Op, r, s);
    memcpy(p, s, (size_t)n * sizeof(double));
    double gamma = dotr(n, s, s);
    i64 iter = 0;
    if (itmax == 0) itmax = m + n;
    double rNorm = bNorm, ArNorm = sqrt(gamma);
    double eps_ = atol + rtol * ArNorm;
    int solved = ArNorm <= eps_;
    int tired = iter >= itmax;
    while (!(solved || tired)) {
        op_mul(Op, p, q);
        double delta = dotr(m, q, q);
        if (lambda > 0) delta += lambda * dotr(n, p, p);
        double alpha = gamma / delta;
        FO_PAR for (i64 i = 0; i < n; i++) x[i] += alpha * p[i];
        FO_PAR for (i64 i = 0; i < m; i++) r[i] -= alpha * q[i];
        op_tmul(Op, r, s);
        if (lambda > 0) FO_PAR for (i64 i = 0; i < n; i++) s[i] -= lambda * x[i];
        double gamma_next = dotr(n, s, s);
        double beta = gamma_next / gamma;
        FO_PAR for (i64 i = 0; i < n; i++) p[i] = s[i] + beta * p[i];
        gamma = gamma_next;
        rNorm = nrm2(m, r);
        ArNorm = sqrt(gamma);
        iter++;
        solved = ArNorm <= eps_;
        tired = iter >= itmax;
    }
    st->niter = iter; st->solved = solved; st->inconsistent = 0;
    st->status = solved ? FO_ST_SOLVED : FO_ST_TIRED;
    st->rnorm = rNorm; st->arnorm = ArNorm;
    }
done:
    free(r); free(q); free(s); free(p);
}

/* ------------------------------------------------------------------------------------------ */
/* ctypes-friendly wrappers                                                                   */
/* ------------------------------------------------------------------------------------------ */
static void mk_mat(fo_mat *M, i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                   const i64 *trp, const i64 *tci, const double *tvx)
{ M->m = m; M->n = n; M->rp = rp; M->ci = ci; M->vx = vx; M->trp = trp; M->tci = tci; M->tvx = tvx; }

/* tolerances block (IterativeSolver fields, src/solve_two_systems_struct.jl:99-115) */
typedef struct {
    double ls_atol, ls_rtol; i64 ls_itmax;
    double ln_atol, ln_rtol, ln_btol, ln_conlim; i64 ln_itmax;
    double ne_atol, ne_rtol, ne_etol, ne_conlim; i64 ne_itmax;
} fo_itertol;

static const double SQRT_EPS = 1.4901161193847656e-08;   /* sqrt(eps(Float64)) */

void fo_itertol_defaults(fo_itertol *t, i64 nvar, i64 ncon)
{
    t->ls_atol = t->ls_rtol = SQRT_EPS; t->ls_itmax = 5 * (ncon + nvar);
    t->ln_atol = t->ln_rtol = t->ln_btol = SQRT_EPS; t->ln_conlim = 1.0 / SQRT_EPS;
    t->ln_itmax = 5 * (ncon + nvar);
    t->ne_atol = t->ne_rtol = t->ne_etol = SQRT_EPS; t->ne_conlim = 1.0 / SQRT_EPS; t->ne_itmax = 0;
}

/* solve_least_square (src/solve_two_systems_struct.jl:167-185): LSQR on Aop' (n x m) */
static void solve_least_square(const fo_mat *M, const fo_itertol *t, const double *b, double lambda,
                               double *q, fo_stats *st)
{
    fo_op op = { M, 1, NULL };
    fo_lsqr(&op, b, lambda, t->ls_atol, t->ls_rtol, SQRT_EPS, SQRT_EPS, SQRT_EPS, 1.0 / SQRT_EPS,
            t->ls_itmax, q, st);
}

/* solve_two_mixed [Iterative] (src/solve_linear_system.jl:107-140) */
void fo_iter_solve_two_mixed(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                             const i64 *trp, const i64 *tci, const double *tvx,
                             const fo_itertol *t, double delta,
                             const double *rhs1, const double *rhs2,
                             double *p1, double *q1, double *p2, double *q2, fo_stats *st /*[2]*/)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    solve_least_square(&M, t, rhs1, sqrt(delta), q1, &st[0]);
    csr_mv(n, trp, tci, tvx, q1, p1);
    for (i64 i = 0; i < n; i++) p1[i] = rhs1[i] - p1[i];
    double *nb = (double *)malloc((size_t)m * sizeof(double));
    for (i64 i = 0; i < m; i++) nb[i] = -rhs2[i];
    fo_op op = { &M, 0, NULL };
    if (delta != 0.0)
        fo_craig(&op, nb, 1, 1.0 / delta, 0.0, t->ln_atol, t->ln_rtol, t->ln_btol, t->ln_conlim,
                 t->ln_itmax, p2, q2, &st[1]);
    else
        fo_craig(&op, nb, 0, 1.0, 0.0, t->ln_atol, t->ln_rtol, t->ln_btol, t->ln_conlim,
                 t->ln_itmax, p2, q2, &st[1]);
    for (i64 i = 0; i < n; i++) p2[i] = -p2[i];
    free(nb);
}

/* solve_two_least_squares [Iterative] (src/solve_linear_system.jl:79-105).
   The reference returns q1 and q2 aliased to the same workspace vector (q1 == q2 on return);
   here both are returned separately, callers only use p1/p2. */
void fo_iter_solve_two_least_squares(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                                     const i64 *trp, const i64 *tci, const double *tvx,
                                     const fo_itertol *t, double delta,
                                     const double *rhs1, const double *rhs2,
                                     double *p1, double *q1, double *p2, double *q2, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    solve_least_square(&M, t, rhs1, sqrt(delta), q1, &st[0]);
    csr_mv(n, trp, tci, tvx, q1, p1);
    for (i64 i = 0; i < n; i++) p1[i] = rhs1[i] - p1[i];
    solve_least_square(&M, t, rhs2, sqrt(delta), q2, &st[1]);
    csr_mv(n, trp, tci, tvx, q2, p2);
    for (i64 i = 0; i < n; i++) p2[i] = rhs2[i] - p2[i];
}

/* solve_two_extras [Iterative] (src/solve_linear_system.jl:45-77) */
void fo_iter_solve_two_extras(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                              const i64 *trp, const i64 *tci, const double *tvx,
                              const fo_itertol *t, double delta,
                              const double *rhs1, const double *rhs2,
                              double *u1, double *u2, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    double tau = delta > 1e-14 ? delta : 1e-14;
    solve_least_square(&M, t, rhs1, sqrt(tau), u1, &st[0]);
    double *tmp = (double *)malloc((size_t)n * sizeof(double));
    fo_op op = { &M, 2, tmp };
    fo_minres(&op, rhs2, tau, t->ne_atol, t->ne_rtol, t->ne_etol, t->ne_conlim, t->ne_itmax, u2, &st[1]);
    free(tmp);
}

/* solve_two_extras [LDLt] (src/solve_linear_system.jl:142-159): cgls + minres, Krylov defaults */
void fo_ldlt_solve_two_extras(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                              const i64 *trp, const i64 *tci, const double *tvx, double delta,
                              const double *rhs1, const double *rhs2,
                              double *u1, double *u2, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    double tau = delta > 1e-14 ? delta : 1e-14;
    fo_op opt = { &M, 1, NULL };
    fo_cgls(&opt, rhs1, tau, SQRT_EPS, SQRT_EPS, 0, u1, &st[0]);
    double *tmp = (double *)malloc((size_t)n * sizeof(double));
    fo_op op = { &M, 2, tmp };
    fo_minres(&op, rhs2, tau, SQRT_EPS / 100, SQRT_EPS / 100, SQRT_EPS, 1.0 / SQRT_EPS, 0, u2, &st[1]);
    free(tmp);
}

/* raw single-solver entry points (used by tests to pin each Krylov method separately) */
void fo_lsqr_csr(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                 const i64 *trp, const i64 *tci, const double *tvx, int kind,
                 const double *b, double lambda, double atol, double rtol, i64 itmax,
                 double *x, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    fo_op op = { &M, kind, NULL };
    fo_lsqr(&op, b, lambda, atol, rtol, SQRT_EPS, SQRT_EPS, SQRT_EPS, 1.0 / SQRT_EPS, itmax, x, st);
}
/* LSQR with every threshold settable (fo_lsqr_csr fixes axtol = btol = etol = sqrt(eps) and conlim = 1/sqrt(eps),
   as the reference's call site does); tests scale them to show that a stopping decision is not a near tie */
void fo_lsqr_full_csr(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                      const i64 *trp, const i64 *tci, const double *tvx, int kind,
                      const double *b, double lambda, double atol, double rtol, double axtol, double btol,
                      double etol, double conlim, i64 itmax, double *x, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    fo_op op = { &M, kind, NULL };
    fo_lsqr(&op, b, lambda, atol, rtol, axtol, btol, etol, conlim, itmax, x, st);
}
void fo_craig_csr(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                  const i64 *trp, const i64 *tci, const double *tvx, int kind,
                  const double *b, int sqd, double mscale, double atol, double rtol, double btol,
                  double conlim, i64 itmax, double *x, double *y, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    fo_op op = { &M, kind, NULL };
    fo_craig(&op, b, sqd, mscale, 0.0, atol, rtol, btol, conlim, itmax, x, y, st);
}
void fo_minres_normal_csr(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                          const i64 *trp, const i64 *tci, const double *tvx,
                          const double *b, double lambda, double atol, double rtol, double etol,
                          double conlim, i64 itmax, double *x, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    double *tmp = (double *)malloc((size_t)n * sizeof(double));
    fo_op op = { &M, 2, tmp };
    fo_minres(&op, b, lambda, atol, rtol, etol, conlim, itmax, x, st);
    free(tmp);
}
void fo_cgls_csr(i64 m, i64 n, const i64 *rp, const i64 *ci, const double *vx,
                 const i64 *trp, const i64 *tci, const double *tvx, int kind,
                 const double *b, double lambda, double atol, double rtol, i64 itmax,
                 double *x, fo_stats *st)
{
    fo_mat M; mk_mat(&M, m, n, rp, ci, vx, trp, tci, tvx);
    fo_op op = { &M, kind, NULL };
    fo_cgls(&op, b, lambda, atol, rtol, itmax, x, st);
}
void fo_csr_mv(i64 nr, const i64 *rp, const i64 *ci, const double *vx, const double *x, double *y)
{ csr_mv(nr, rp, ci, vx, x, y); }

/* ------------------------------------------------------------------------------------------ */
/* LDLtSolver restated (src/solve_two_systems_struct.jl:299-353)                               */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    i64 nvar, ncon, nnzj, nnz, N;
    i64 *rows, *cols; double *vals;     /* COO of triu(K), layout [I | J' | -delta I] */
    i64 *Kp, *Ki; double *Kx;           /* sparse() scratch (rebuilt every refactor like the reference) */
    fo_ldl *str;
    double *sol;                        /* N x 2 column-major */
} fo_ldlt_solver;

/* jrow/jcol: 0-based COO structure of the Jacobian (jac_structure!), P: permutation of size N. */
fo_ldlt_solver *fo_ldlt_create(i64 nvar, i64 ncon, i64 nnzj, const i64 *jrow, const i64 *jcol,
                               const i64 *P, double tol, double r1, double r2)
{
    fo_ldlt_solver *S = (fo_ldlt_solver *)calloc(1, sizeof(*S));
    S->nvar = nvar; S->ncon = ncon; S->nnzj = nnzj; S->nnz = nvar + nnzj + ncon; S->N = nvar + ncon;
    i64 nnz = S->nnz, N = S->N;
    S->rows = (i64 *)malloc((size_t)nnz * sizeof(i64));
    S->cols = (i64 *)malloc((size_t)nnz * sizeof(i64));
    S->vals = (double *)calloc((size_t)nnz, sizeof(double));
    for (i64 k = 0; k < nvar; k++) { S->rows[k] = k; S->cols[k] = k; S->vals[k] = 1.0; }
    for (i64 k = 0; k < nnzj; k++) { S->rows[nvar + k] = jcol[k]; S->cols[nvar + k] = nvar + jrow[k]; }
    for (i64 k = 0; k < ncon; k++) { S->rows[nvar + nnzj + k] = nvar + k; S->cols[nvar + nnzj + k] = nvar + k; }
    S->Kp = (i64 *)malloc((size_t)(N + 1) * sizeof(i64));
    S->Ki = (i64 *)malloc((size_t)nnz * sizeof(i64));
    S->Kx = (double *)malloc((size_t)nnz * sizeof(double));
    fo_coo_to_csc(N, nnz, S->rows, S->cols, S->vals, S->Kp, S->Ki, S->Kx, NULL);
    S->str = fo_ldl_analyze(N, S->Kp, S->Ki, P);
    fo_ldl_set_reg(S->str, nvar, tol, r1, r2);
    S->sol = (double *)calloc((size_t)N * 2, sizeof(double));
    return S;
}
void fo_ldlt_destroy(fo_ldlt_solver *S)
{
    if (!S) return;
    free(S->rows); free(S->cols); free(S->vals); free(S->Kp); free(S->Ki); free(S->Kx);
    fo_ldl_free(S->str); free(S->sol); free(S);
}
fo_ldl *fo_ldlt_str(fo_ldlt_solver *S) { return S->str; }

/* solve_two_mixed [LDLt]: jvals = jac_coord!(x) (length nnzj). returns factorized flag. */
int fo_ldlt_solve_two_mixed(fo_ldlt_solver *S, const double *jvals, double delta,
                            const double *rhs1, const double *rhs2,
                            double *p1, double *q1, double *p2, double *q2)
{
    i64 nvar = S->nvar, ncon = S->ncon, nnzj = S->nnzj, N = S->N;
    memcpy(S->vals + nvar, jvals, (size_t)nnzj * sizeof(double));
    for (i64 k = 0; k < ncon; k++) S->vals[nvar + nnzj + k] = -delta;
    fo_coo_to_csc(N, S->nnz, S->rows, S->cols, S->vals, S->Kp, S->Ki, S->Kx, NULL);
    fo_ldl_factorize(S->str, S->Kp, S->Ki, S->Kx);
    double *sol = S->sol;
    for (i64 i = 0; i < nvar; i++) { sol[i] = rhs1[i]; sol[N + i] = 0.0; }
    for (i64 i = 0; i < ncon; i++) { sol[nvar + i] = 0.0; sol[N + nvar + i] = rhs2[i]; }
    int ok = S->str->factorized;
    if (ok) fo_ldl_solve2(S->str, sol);
    memcpy(p1, sol, (size_t)nvar * sizeof(double));
    memcpy(q1, sol + nvar, (size_t)ncon * sizeof(double));
    memcpy(p2, sol + N, (size_t)nvar * sizeof(double));
    memcpy(q2, sol + N + nvar, (size_t)ncon * sizeof(double));
    return ok;
}
/* solve_two_least_squares [LDLt]: no refactor; rhs = [rhs1;0], [rhs2;0] */
int fo_ldlt_solve_two_least_squares(fo_ldlt_solver *S, const double *rhs1, const double *rhs2,
                                    double *p1, double *q1, double *p2, double *q2)
{
    i64 nvar = S->nvar, ncon = S->ncon, N = S->N;
    double *sol = S->sol;
    for (i64 i = 0; i < nvar; i++) { sol[i] = rhs1[i]; sol[N + i] = rhs2[i]; }
    for (i64 i = 0; i < ncon; i++) { sol[nvar + i] = 0.0; sol[N + nvar + i] = 0.0; }
    int ok = S->str->factorized;
    if (ok) fo_ldl_solve2(S->str, sol);
    memcpy(p1, sol, (size_t)nvar * sizeof(double));
    memcpy(q1, sol + nvar, (size_t)ncon * sizeof(double));
    memcpy(p2, sol + N, (size_t)nvar * sizeof(double));
    memcpy(q2, sol + N + nvar, (size_t)ncon * sizeof(double));
    return ok;
}

/* ------------------------------------------------------------------------------------------ */
/* Error-model checks of a given factor L^, D^ (LDLFactorizations' CSC layout: the Lp / Li of S->str) and of solutions */
/* computed with it, in long double, against K as the last fo_ldlt_solve_two_mixed assembled it (S->Kp/Ki/Kx).       */
/* u = 2^-53.  reg (permuted order, may be NULL): pivots replaced by the dynamic regularisation.                      */
/* ------------------------------------------------------------------------------------------ */
/* row structure of L: for row i, the columns k < i with L(i, k) structurally nonzero and the position of the value */
static void ldl_rows(const fo_ldl *L, i64 **Rp_out, i64 **Rpos_out)
{
    i64 n = L->n, lnz = L->Lp[n];
    i64 *Rp = (i64 *)calloc((size_t)n + 1, sizeof(i64));
    i64 *Rpos = (i64 *)malloc((size_t)(lnz > 0 ? lnz : 1) * sizeof(i64));
    for (i64 p = 0; p < lnz; p++) Rp[L->Li[p] + 1]++;
    for (i64 i = 0; i < n; i++) Rp[i + 1] += Rp[i];
    i64 *w = (i64 *)malloc((size_t)(n + 1) * sizeof(i64));
    memcpy(w, Rp, (size_t)(n + 1) * sizeof(i64));
    for (i64 j = 0; j < n; j++)
        for (i64 p = L->Lp[j]; p < L->Lp[j + 1]; p++) Rpos[w[L->Li[p]]++] = p;   /* ascending column within a row */
    free(w);
    *Rp_out = Rp; *Rpos_out = Rpos;
}

/* diagonal of P K P' (permuted order) */
static void perm_diag(const fo_ldlt_solver *S, long double *kd)
{
    const fo_ldl *L = S->str;
    for (i64 k = 0; k < S->N; k++) kd[k] = 0.0L;
    for (i64 c = 0; c < S->N; c++)
        for (i64 p = S->Kp[c]; p < S->Kp[c + 1]; p++)
            if (S->Ki[p] == c) kd[L->pinv[c]] += (long double)S->Kx[p];
}

/* Factor check: for every (i, j) of the pattern of L (diagonal included),
 *   |(P K P' - L^ D^ L^')_ij| / ((c_ij + 4) u (|L^| |D^| |L^'|)_ij),
 * c_ij = #{k < j : L(i,k) L(j,k) structurally nonzero}; the diagonal positions of regularised pivots are skipped.
 * Returns the worst ratio; *where = its position (p < lnz: Lx[p], lnz + j: the diagonal j).  bound (optional, lnz + N):
 * the denominator of every position.  dpre (optional, N): d_k = (P K P')_kk - sum_{j<k} L^_kj^2 D^_j, the pivot before
 * any regularisation. */
double fo_ldlt_check_factor(const fo_ldlt_solver *S, const double *Lx, const double *D, const signed char *reg,
                            i64 *where, double *bound, double *dpre)
{
    const fo_ldl *L = S->str;
    const i64 n = L->n, lnz = L->Lp[n];
    const i64 *Lp = L->Lp, *Li = L->Li;
    const long double u = ldexpl(1.0L, -53);
    i64 *Rp, *Rpos;
    ldl_rows(L, &Rp, &Rpos);
    /* lower triangle of P K P' by permuted columns: (row, value) lists */
    i64 *Cp = (i64 *)calloc((size_t)n + 1, sizeof(i64));
    for (i64 c = 0; c < n; c++)
        for (i64 p = S->Kp[c]; p < S->Kp[c + 1]; p++) {
            i64 a = L->pinv[S->Ki[p]], b = L->pinv[c];
            Cp[(a < b ? a : b) + 1]++;
        }
    for (i64 j = 0; j < n; j++) Cp[j + 1] += Cp[j];
    i64 *Ci = (i64 *)malloc((size_t)(Cp[n] > 0 ? Cp[n] : 1) * sizeof(i64));
    long double *Cx = (long double *)malloc((size_t)(Cp[n] > 0 ? Cp[n] : 1) * sizeof(long double));
    {
        i64 *w = (i64 *)malloc((size_t)(n + 1) * sizeof(i64));
        memcpy(w, Cp, (size_t)(n + 1) * sizeof(i64));
        for (i64 c = 0; c < n; c++)
            for (i64 p = S->Kp[c]; p < S->Kp[c + 1]; p++) {
                i64 a = L->pinv[S->Ki[p]], b = L->pinv[c];
                i64 q = w[a < b ? a : b]++;
                Ci[q] = a > b ? a : b; Cx[q] = (long double)S->Kx[p];
            }
        free(w);
    }
    i64 *col = (i64 *)malloc((size_t)(lnz > 0 ? lnz : 1) * sizeof(i64));
    for (i64 k = 0; k < n; k++) for (i64 p = Lp[k]; p < Lp[k + 1]; p++) col[p] = k;
    long double *acc = (long double *)calloc((size_t)(n > 0 ? n : 1), sizeof(long double));
    long double *mag = (long double *)calloc((size_t)(n > 0 ? n : 1), sizeof(long double));
    i64 *cnt = (i64 *)calloc((size_t)(n > 0 ? n : 1), sizeof(i64));
    double worst = 0.0;
    i64 wpos = -1;
    for (i64 j = 0; j < n; j++) {
        /* acc[i] = (L^ D^ L^' - P K P')_ij for i = j and the rows i of column j: the columns k < j of row j contribute
           their rows from j down (the elimination tree puts them in the pattern of column j) */
        for (i64 q = Rp[j]; q < Rp[j + 1]; q++) {
            const i64 pj = Rpos[q], k = col[pj];
            const long double ljd = (long double)Lx[pj] * (long double)D[k];
            for (i64 p = pj; p < Lp[k + 1]; p++) {
                const long double t = (long double)Lx[p] * ljd;
                acc[Li[p]] += t; mag[Li[p]] += fabsl(t); cnt[Li[p]]++;
            }
        }
        acc[j] += (long double)D[j]; mag[j] += fabsl((long double)D[j]);      /* k = j, L(j, j) = 1 */
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) {
            const long double t = (long double)Lx[p] * (long double)D[j];
            acc[Li[p]] += t; mag[Li[p]] += fabsl(t);
        }
        for (i64 p = Cp[j]; p < Cp[j + 1]; p++) acc[Ci[p]] -= Cx[p];
        if (dpre) dpre[j] = (double)((long double)D[j] - acc[j]);
        for (i64 e = -1; e < Lp[j + 1] - Lp[j]; e++) {
            const i64 i = e < 0 ? j : Li[Lp[j] + e];
            const i64 pos = e < 0 ? lnz + j : Lp[j] + e;
            const long double b = (long double)(cnt[i] + 4) * u * mag[i];
            if (bound) bound[pos] = (double)b;
            if (!(e < 0 && reg && reg[j])) {
                const long double err = fabsl(acc[i]);
                const double r = err == 0.0L ? 0.0 : (b > 0.0L ? (double)(err / b) : INFINITY);
                if (wpos < 0 || r > worst) { worst = r; wpos = pos; }
            }
            acc[i] = 0.0L; mag[i] = 0.0L; cnt[i] = 0;
        }
    }
    if (where) *where = wpos;
    free(Rp); free(Rpos); free(Cp); free(Ci); free(Cx); free(acc); free(mag); free(cnt); free(col);
    return worst;
}

/* Solve check of one solution x^ (original order, N) of K x = b: for every i,
 *   |b - K~ x^|_i / ((3c + 10) u (P' |L^| |D^| |L^'| P |x^|)_i),
 * c = the largest row or column count of L, K~ = K with the pivot change D^_k - d_k (fo_ldlt_check_factor's dpre) added
 * at the regularised positions k, whose factor is the one L^ D^ L^' stands for.  Returns the worst ratio, *where = i. */
double fo_ldlt_check_solve(const fo_ldlt_solver *S, const double *Lx, const double *D, const signed char *reg,
                           const double *x, const double *b, i64 *where)
{
    const fo_ldl *L = S->str;
    const i64 n = L->n;
    const i64 *Lp = L->Lp, *Li = L->Li, *P = L->P;
    const long double u = ldexpl(1.0L, -53);
    long double *y = (long double *)calloc((size_t)(n > 0 ? n : 1), sizeof(long double));
    long double *t = (long double *)calloc((size_t)(n > 0 ? n : 1), sizeof(long double));
    long double *t3 = (long double *)calloc((size_t)(n > 0 ? n : 1), sizeof(long double));
    i64 *rc = (i64 *)calloc((size_t)(n > 0 ? n : 1), sizeof(i64));
    i64 c = 0;
    for (i64 j = 0; j < n; j++) {
        i64 cc = Lp[j + 1] - Lp[j];
        if (cc > c) c = cc;
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) rc[Li[p]]++;
    }
    for (i64 i = 0; i < n; i++) if (rc[i] > c) c = rc[i];
    /* K x (K holds the upper triangle) */
    for (i64 col = 0; col < n; col++)
        for (i64 p = S->Kp[col]; p < S->Kp[col + 1]; p++) {
            const i64 r = S->Ki[p];
            const long double v = (long double)S->Kx[p];
            y[r] += v * (long double)x[col];
            if (r != col) y[col] += v * (long double)x[r];
        }
    if (reg) {
        /* d_k = (P K P')_kk - sum_j L^_kj^2 D^_j */
        perm_diag(S, t);
        for (i64 j = 0; j < n; j++)
            for (i64 p = Lp[j]; p < Lp[j + 1]; p++) t[Li[p]] -= (long double)Lx[p] * (long double)Lx[p] * (long double)D[j];
        for (i64 k = 0; k < n; k++)
            if (reg[k]) y[P[k]] += ((long double)D[k] - t[k]) * (long double)x[P[k]];
    }
    /* P' |L^| |D^| |L^'| P |x^|: t = |L^'| z, t *= |D^|, t3 = |L^| t */
    for (i64 k = 0; k < n; k++) t[k] = fabsl((long double)x[P[k]]);
    for (i64 j = 0; j < n; j++)
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) t[j] += fabsl((long double)Lx[p]) * fabsl((long double)x[P[Li[p]]]);
    for (i64 k = 0; k < n; k++) { t[k] *= fabsl((long double)D[k]); t3[k] = t[k]; }
    for (i64 j = 0; j < n; j++)
        for (i64 p = Lp[j]; p < Lp[j + 1]; p++) t3[Li[p]] += fabsl((long double)Lx[p]) * t[j];
    double worst = 0.0;
    i64 wi = -1;
    for (i64 k = 0; k < n; k++) {
        const i64 i = P[k];
        const long double err = fabsl((long double)b[i] - y[i]);
        const long double bd = (long double)(3 * c + 10) * u * t3[k];
        const double r = err == 0.0L ? 0.0 : (bd > 0.0L ? (double)(err / bd) : INFINITY);
        if (wi < 0 || r > worst) { worst = r; wi = i; }
    }
    if (where) *where = wi;
    free(y); free(t); free(t3); free(rc);
    return worst;
}
