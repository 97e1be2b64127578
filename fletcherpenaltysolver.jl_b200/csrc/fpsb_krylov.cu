// fpsb_krylov.cu — SpMV / fused two-column SpMM and the fused LSQR / CRAIG / MINRES / CGLS
// iterations of the IterativeSolver path.
//
// Reference surface replaced (file:line under /root/reference):
//   jac_op! products                         NLPModels (SURVEY App. B6), used at src/solve_linear_system.jl:119-121
//   solve_least_square  (LSQR on A')         src/solve_two_systems_struct.jl:167-185
//   solve_least_norm    (CRAIG, M=I/delta)   src/solve_two_systems_struct.jl:210-244
//   solve_two_mixed / least_squares / extras src/solve_linear_system.jl:45-140 (Iterative), :142-159 (LDLt extras)
//
// Design (B200): the Jacobian lives in HBM twice, as A and as A' (both products are gather-type row
// products: no atomics, deterministic), each as a tiled SELL-32 operator whose tiles are single
// contiguous blocks [values | 16-bit window-relative indices | row map].  Persistent CTAs (one per
// SM) stream the tiles through a shared-memory ring with TMA bulk copies (cp.async.bulk + mbarrier,
// four producer warps), three consumer groups reduce every row against BOTH right-hand-side columns
// with one 16-byte shared-memory gather per nonzero (the two Golub-Kahan vectors are interleaved),
// and the row epilogue applies the axpby / norm / delayed x,w updates of the Krylov method so that
// every vector is read and written once per iteration.  Norms use fixed-order reductions; the
// scalar recurrences (Givens rotations, stopping tests) run on the device — inside the LSQR / CRAIG
// loops deferred into the prologue of the next launch — and the host only polls a done flag every
// few iterations.  See the comment above gk_step_kernel and DESIGN.md §4.
#include "fpsb_internal.h"
#include "fpsb_device.cuh"
#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <cstdlib>

// NCCL types for fpsb_dist.inl (bound at run time with dlopen; the header is optional)
#include <dlfcn.h>
#if __has_include(<nccl.h>)
#include <nccl.h>
#else
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
typedef int ncclDataType_t;
typedef int ncclRedOp_t;
#define ncclSuccess 0
#define ncclDouble 8
#define ncclSum 0
#endif


#ifndef FPSB_EXP
#define FPSB_EXP 0     /* > 0: timing experiments that deliberately break the numerics (never shipped) */
#endif

namespace fpsb {

static const double kSqrtEps = 1.4901161193847656e-08;

enum Mode {
    MD_NONE = 0,
    MD_PLAIN,
    MD_LSQR_INIT_M,   // v1 = A' u1 : first half step (row space of the LSQR solution)
    MD_LSQR_U,        // u <- Op v - alpha u          (row space of the LSQR right-hand side)
    MD_LSQR_V,        // w,x updates; v <- Op' u - beta v
    MD_CRAIG_V,       // delayed x,w2 updates; v <- Op' u - beta v
    MD_CRAIG_U,       // w,y updates; Mu <- Op v - alpha Mu
    MD_MINRES_M,
    MD_CGLS_INIT_M,
    MD_CGLS_N,
    MD_CGLS_M
};

enum EwOp {
    EW_COPY = 0,          // out = c0 * in
    EW_INIT_LSQR,         // self = b ; acc ||b||^2
    EW_INIT_CRAIG,        // self = c0 * b ; w = y = 0 ; acc
    EW_CRAIG_FLUSH,       // out = -(x + pending update)
    EW_MINRES_INIT,
    EW_MINRES_E1,
    EW_MINRES_E2,
    EW_CGLS_INIT,
    EW_CGLS_EN,
    EW_CGLS_EM
};

struct SlotIO {
    int mode;
    int pad;
    const double *gin;   // gather source (non-pair kernels)
    double *self;        // recurred vector of this row space (non-pair kernels)
    double *a0, *a1, *a2;
    double c0, c1;
};

struct TileMeta;

// Row-partitioned runs with the peer-memory transport (fpsb_dist.inl): what the last CTA of an m-space
// step needs to all-reduce its four norm sums through the peers' mailboxes and run the recurrences itself
constexpr int kMboxMaxRanks = 8;
constexpr size_t kMboxOffTot = 8 * sizeof(uint64_t);        // mailbox: flags u64[8] | tot double[2][8][4] | ...
struct PeerTail {
    int nranks, rank;
    unsigned char *mine;
    unsigned char *peer[kMboxMaxRanks];
    int *err;
};
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

struct StepParams {
    // tiled SELL-32 operator (see the kernel comment)
    const TileMeta *tiles;
    int ntiles;
    int win_cap;           // capacity of the shared-memory gather window (16-byte entries)
    int stage_bytes, nstage;   // ring geometry
    int inflight;          // tiles a producer may have in flight (bounds the HBM queueing delay of every other load)
    int nlong;
    const unsigned char *tbuf;   // the tiles' blocks, back to back
    int blk_cap;           // capacity of the block part of a ring stage (bytes)
    const int2 *wsegs;     // multi-segment windows (stencil operators): per tile 4 x {source start, window offset | length << 16};
                           // nullptr: every window is the one segment [cmin, cmin + ccnt)
    const unsigned char *rowflag;   // nrows : 1 long row (own kernel), 2 raw row (row sums go to raw_out, no epilogue); nullptr: all 0
    double2 *raw_out;               // row-partitioned runs: raw sums of the halo / boundary rows (see fpsb_dist.inl)
    // long rows (CSR)
    const int *long_row;
    const int *long_rp;
    const int *long_col;
    const double *long_val;
    int nrows;
    const double2 *gin2;   // interleaved gather pair (PAIR kernels)
    double2 *self2;        // interleaved recurred pair of this row space (PAIR kernels)
    SlotIO io[2];
    SlotState *st;
    double *partials;      // [grid][4]
    unsigned *counter;
    int *done_flag;        // set to 1 when no slot remains active
    double *tot_out;       // row-partitioned runs: the last CTA leaves the four local sums here instead of
                           // running the scalar recurrences (an all-reduce and finish_kernel follow)
    // deferred recurrences (LSQR / CRAIG loops): this launch leaves only its per-CTA partials; the NEXT
    // launch reduces them in its prologue (every CTA, same fixed order), runs the recurrences on its
    // shared-memory state copy, and CTA 0 publishes the state to st_out (the other state buffer)
    SlotState *st_out;             // non-null: deferred mode
    const double *pend_partials;   // partials of the previous launch (null: nothing pending)
    int pend_nparts, pend_m0, pend_m1;
    // peer-memory tail (with tot_out): the last CTA exchanges the sums and finishes the step itself
    const PeerTail *ptail;
    unsigned long long pt_sig;     // signals issued before this launch
    int pt_par;                    // half of the peers' tot inbox this exchange uses
};

// ------------------------------------------------------------------------------------------------
// scalar recurrences (one thread, last CTA) — line-by-line the reference algorithms
// ------------------------------------------------------------------------------------------------
// experiment: the scalar recurrences as one out-of-line function (4 inlined copies make the step kernel
// 16.5 K instructions; see profiles/README.md on instruction-fetch cost)
#ifdef FPSB_FINISH_NOINLINE
#define FPSB_FINISH_INLINE __noinline__
#else
#define FPSB_FINISH_INLINE
#endif
__device__ void slot_stop(SlotState &S) { S.active = 0; }

__device__ void lsqr_status(SlotState &S) {
    int st = FPSB_ST_UNKNOWN;
    if (S.tired) st = FPSB_ST_TIRED;
    if (S.ill_mach) st = FPSB_ST_ILLCOND_MACH;
    if (S.ill_lim) st = FPSB_ST_ILLCOND_LIM;
    if (S.solved) st = FPSB_ST_SOLVED;
    if (S.zero_resid) st = FPSB_ST_ZERO_RESID;
    if (S.fwd_err) st = FPSB_ST_FWD_ERR;
    S.status = st;
    S.inconsistent = !S.zero_resid;
}

__device__ void fin_init_lsqr(SlotState &S, double bb) {
    double beta1 = sqrt(bb);
    S.beta1 = beta1;
    S.iter = 0;
    if (beta1 == 0.0) {
        S.active = 0; S.solved = 1; S.inconsistent = 0; S.status = FPSB_ST_ZERO_RHS;
        return;
    }
    S.beta = beta1;
    S.su = 1.0 / beta1;
}

__device__ void fin_lsqr_init_m(SlotState &S, double vv) {
    S.Anorm2 = vv;
    S.Anorm = sqrt(vv);
    S.alpha = S.Anorm;
    S.Acond = 0; S.xNorm = 0; S.xNorm2 = 0; S.dNorm2 = 0;
    S.c2 = -1.0; S.s2 = 0.0; S.z = 0.0;
    S.xENorm2 = 0; S.err_lbnd = 0;
    for (int i = 0; i < 5; ++i) S.err_vec[i] = 0;
    S.rNorm = S.beta1; S.res2 = 0;
    S.ArNorm = S.ArNorm0 = S.alpha * S.beta;
    if (S.alpha == 0.0) {
        S.active = 0; S.solved = 1; S.inconsistent = 0; S.status = FPSB_ST_ZERO_ATB;
        return;
    }
    S.sv = 1.0 / S.alpha;
    S.phibar = S.beta1;
    S.rhobar = S.alpha;
    S.first = 1;
    int solved_lim = S.ArNorm / (S.Anorm * S.rNorm) <= S.axtol;
    int solved_mach = 1.0 + S.ArNorm / (S.Anorm * S.rNorm) <= 1.0;
    S.solved = solved_mach | solved_lim;
    S.tired = S.iter >= S.itmax;
    S.zero_resid = (S.rNorm / S.beta1 <= S.axtol) | (1.0 + S.rNorm / S.beta1 <= 1.0);
    S.ill_mach = S.ill_lim = S.fwd_err = 0;
    if (S.solved || S.tired) { lsqr_status(S); S.active = 0; }
}

// after u <- Op v - alpha u
__device__ void fin_lsqr_u(SlotState &S, double uu) {
    S.iter += 1;
    double beta = sqrt(uu);
    S.beta = beta;
    if (beta != 0.0) {
        S.su = 1.0 / beta;
        S.beta_zero = 0;
        S.Anorm2 = S.Anorm2 + S.alpha * S.alpha + beta * beta;
        if (S.lambda > 0) S.Anorm2 += S.lambda * S.lambda;
    } else {
        S.su = 0.0;
        S.beta_zero = 1;
    }
    double c1, s1, rhobar1;
    sym_givens(S.rhobar, S.lambda, c1, s1, rhobar1);
    S.psi = s1 * S.phibar;
    S.phibar = c1 * S.phibar;
    sym_givens(rhobar1, beta, S.c, S.s, S.rho);
    S.phi = S.c * S.phibar;
    S.phibar = S.s * S.phibar;
    S.xENorm2 += S.phi * S.phi;
    S.err_vec[S.iter % 5] = S.phi;
    if (S.iter >= 5) {
        double e = 0;
        for (int i = 0; i < 5; ++i) e += S.err_vec[i] * S.err_vec[i];
        S.err_lbnd = sqrt(e);
    }
    S.tau = S.s * S.phi;
    S.sigma = S.phi / S.rho;
}

// after v <- Op' u - beta v (and the x, w updates)
__device__ void fin_lsqr_v(SlotState &S, double vv, double ww) {
    if (!S.beta_zero) {
        S.alpha = sqrt(vv);
        S.sv = (S.alpha != 0.0) ? 1.0 / S.alpha : 0.0;
    }
    double theta = S.s * S.alpha;
    S.rhobar = -S.c * S.alpha;
    S.dNorm2 += ww / (S.rho * S.rho);
    S.tr_prev = theta / S.rho;
    S.first = 0;
    double delta = S.s2 * S.rho;
    double gammabar = -S.c2 * S.rho;
    double rhs = S.phi - delta * S.z;
    double zbar = rhs / gammabar;
    S.xNorm = sqrt(S.xNorm2 + zbar * zbar);
    double gamma;
    sym_givens(gammabar, theta, S.c2, S.s2, gamma);
    S.z = rhs / gamma;
    S.xNorm2 += S.z * S.z;
    S.Anorm = sqrt(S.Anorm2);
    S.Acond = S.Anorm * sqrt(S.dNorm2);
    double res1 = S.phibar * S.phibar;
    S.res2 += S.psi * S.psi;
    S.rNorm = sqrt(res1 + S.res2);
    S.ArNorm = S.alpha * fabs(S.tau);
    double test1 = S.rNorm / S.beta1;
    double test2 = S.ArNorm / (S.Anorm * S.rNorm);
    double test3 = 1.0 / S.Acond;
    double t1 = test1 / (1.0 + S.Anorm * S.xNorm / S.beta1);
    double rNormtol = S.btol + S.axtol * S.Anorm * S.xNorm / S.beta1;
    S.ill_mach = (1.0 + test3 <= 1.0);
    int solved_mach = (1.0 + test2 <= 1.0);
    int zero_resid_mach = (1.0 + t1 <= 1.0);
    S.tired = S.iter >= S.itmax;
    S.ill_lim = (test3 <= S.ctol);
    int solved_lim = (test2 <= S.axtol);
    int solved_opt = S.ArNorm <= S.atol + S.rtol * S.ArNorm0;
    int zero_resid_lim = (test1 <= rNormtol);
    if (S.iter >= 5) S.fwd_err = S.err_lbnd <= S.etol * sqrt(S.xENorm2);
    int ill_cond = S.ill_mach || S.ill_lim;
    S.zero_resid = zero_resid_mach || zero_resid_lim;
    S.solved = solved_mach || solved_lim || solved_opt || S.zero_resid || S.fwd_err;
    if (S.solved || S.tired || ill_cond) { lsqr_status(S); S.active = 0; }
}

__device__ void craig_status(SlotState &S) {
    int st = FPSB_ST_UNKNOWN;
    if (S.tired) st = FPSB_ST_TIRED;
    if (S.solved) st = FPSB_ST_SOLVED;
    if (S.ill_mach) st = FPSB_ST_ILLCOND_MACH;
    if (S.ill_lim) st = FPSB_ST_ILLCOND_LIM;
    if (S.inconsistent) st = FPSB_ST_INCONSISTENT;
    S.status = st;
}

__device__ void fin_init_craig(SlotState &S, double bb) {
    double beta1 = sqrt(S.mscale * bb);   // sqrt(u'Mu), u = mscale * Mu
    S.beta1 = beta1;
    S.rNorm = beta1;
    S.iter = 0;
    if (beta1 == 0.0) {
        S.active = 0; S.solved = 1; S.inconsistent = 0; S.status = FPSB_ST_ZERO_RHS;
        return;
    }
    S.beta1sq = beta1 * beta1;
    S.beta = beta1;
    S.theta = beta1;
    S.xi = -1.0;
    S.deltag = S.lambda;
    S.rho_prev = 1.0;
    S.su = 1.0 / beta1;
    S.sv = 0.0;
    S.pend = 0;
    S.c1 = 1.0; S.s1 = 0.0; S.s2g = 1.0;
    S.Anorm2 = 0; S.Anorm = 0; S.dNorm2 = 0; S.Acond = 0; S.xNorm2 = 0;
    S.eps_c = S.atol + S.rtol * S.rNorm;
    double bkwerr = 1.0;
    int solved_lim = bkwerr <= S.btol;
    int solved_mach = 1.0 + bkwerr <= 1.0;
    int solved_resid_tol = S.rNorm <= S.eps_c;
    int solved_resid_lim = S.rNorm <= S.btol + S.atol * S.Anorm * sqrt(S.xNorm2) / beta1;
    S.solved = solved_mach | solved_lim | solved_resid_tol | solved_resid_lim;
    S.tired = S.iter >= S.itmax;
    S.ill_mach = S.ill_lim = 0;
    S.inconsistent = 0;
    if (S.solved || S.tired) { craig_status(S); S.active = 0; }
}

// after v <- Op' u - beta v
__device__ void fin_craig_v(SlotState &S, double vv) {
    S.pend = 0;   // the previous iteration's x update was applied by this kernel
    double alpha = sqrt(vv);
    if (alpha == 0.0) {
        S.inconsistent = 1;
        craig_status(S);
        S.active = 0;
        return;
    }
    S.alpha = alpha;
    S.sv = 1.0 / alpha;
    S.Anorm2 += alpha * alpha;
    if (S.lambda > 0) sym_givens(alpha, S.deltag, S.c1, S.s1, S.rho);
    else S.rho = alpha;
    S.xi = -S.theta / S.rho * S.xi;
    S.trw = S.theta / S.rho_prev;
    S.xr = S.xi / S.rho;
    S.pend = 1;
}

// after Mu <- Op v - alpha Mu (and the w, y updates)
__device__ void fin_craig_u(SlotState &S, double uu, double ww) {
    double beta = sqrt(S.mscale * uu);
    S.beta = beta;
    S.su = (beta != 0.0) ? 1.0 / beta : 0.0;
    if (S.lambda > 0) {
        S.theta = S.c1 * beta;
        double gamma = S.s1 * beta;
        double c2;
        sym_givens(S.lambda, gamma, c2, S.s2g, S.deltag);
    } else {
        S.theta = beta;
    }
    S.Anorm2 += beta * beta;
    S.Anorm = sqrt(S.Anorm2);
    S.dNorm2 += sqrt(ww);   // upstream craig.jl accumulates the 2-norm here (kept)
    S.Acond = S.Anorm * sqrt(S.dNorm2);
    S.xNorm2 += S.xi * S.xi;
    S.rNorm = beta * fabs(S.xi);
    if (S.lambda > 0) S.rNorm *= fabs(S.c1);
    S.iter += 1;
    double bkwerr = S.rNorm / sqrt(S.beta1sq + S.Anorm2 * S.xNorm2);
    S.rho_prev = S.rho;
    int solved_lim = bkwerr <= S.btol;
    int solved_mach = 1.0 + bkwerr <= 1.0;
    int solved_resid_tol = S.rNorm <= S.eps_c;
    int solved_resid_lim = S.rNorm <= S.btol + S.atol * S.Anorm * sqrt(S.xNorm2) / S.beta1;
    S.solved = solved_mach | solved_lim | solved_resid_tol | solved_resid_lim;
    S.ill_mach = 1.0 + 1.0 / S.Acond <= 1.0;
    S.ill_lim = 1.0 / S.Acond <= S.ctol;
    S.inconsistent = 0;
    S.tired = S.iter >= S.itmax;
    S.xNorm = sqrt(S.xNorm2);
    if (S.solved || S.ill_mach || S.ill_lim || S.tired) { craig_status(S); S.active = 0; }
}

// ---- MINRES ------------------------------------------------------------------------------------
__device__ void fin_minres_init(SlotState &S, double bb) {
    S.iter = 0;
    if (bb == 0.0) {
        S.active = 0; S.solved = 1; S.inconsistent = 0; S.status = FPSB_ST_ZERO_RHS;
        S.beta1 = 0;
        return;
    }
    double beta1 = sqrt(bb);
    S.beta1 = beta1; S.beta = beta1; S.oldbeta = 0; S.deltabar = 0; S.eps_ = 0;
    S.rNorm = beta1; S.phibar = beta1; S.rhs1 = beta1; S.rhs2 = 0;
    S.gmax = 0; S.gmin = INFINITY; S.cs = -1.0; S.sn = 0;
    S.Anorm2 = 0; S.Anorm = 0; S.Acond = 0; S.ArNorm = 0; S.xNorm = 0; S.xENorm2 = 0; S.err_lbnd = 0;
    for (int i = 0; i < 5; ++i) S.err_vec[i] = 0;
    S.tol = S.atol + S.rtol * beta1;
    S.solved = (S.rNorm <= S.rtol);
    S.tired = S.iter >= S.itmax;
    S.zero_resid = (S.rNorm <= S.tol);
    S.ill_mach = S.ill_lim = S.fwd_err = 0;
    if (S.solved || S.tired) {
        S.status = S.solved ? FPSB_ST_SOLVED : FPSB_ST_TIRED;
        S.inconsistent = !S.zero_resid;
        S.active = 0;
    }
}
__device__ void fin_minres_m(SlotState &S, double vy) {
    S.iter += 1;
    S.alpha = vy / S.beta;
    S.delta = S.cs * S.deltabar + S.sn * S.alpha;
}
__device__ void fin_minres_e1(SlotState &S, double yy) {
    S.oldbeta = S.beta;
    S.beta = sqrt(yy);
    double alpha = S.alpha, beta = S.beta;
    S.Anorm2 = S.Anorm2 + alpha * alpha + S.oldbeta * S.oldbeta + beta * beta;
    S.gammabar = S.sn * S.deltabar - S.cs * alpha;
    S.eps_ = S.sn * beta;
    S.deltabar = -S.cs * beta;
    S.root = sqrt(S.gammabar * S.gammabar + S.deltabar * S.deltabar);
    S.ArNorm = S.phibar * S.root;
    double gamma = sqrt(S.gammabar * S.gammabar + beta * beta);
    gamma = fmax(gamma, 2.220446049250313e-16);
    S.gamma = gamma;
    S.cs = S.gammabar / gamma;
    S.sn = beta / gamma;
    S.phi = S.cs * S.phibar;
    S.phibar = S.sn * S.phibar;
}
__device__ void fin_minres_e2(SlotState &S, double xx) {
    const double epsM = 2.220446049250313e-16;
    S.xENorm2 += S.phi * S.phi;
    S.err_vec[S.iter % 5] = S.phi;
    if (S.iter >= 5) {
        double e = 0;
        for (int i = 0; i < 5; ++i) e += S.err_vec[i] * S.err_vec[i];
        S.err_lbnd = sqrt(e);
    }
    S.gmax = fmax(S.gmax, S.gamma);
    S.gmin = fmin(S.gmin, S.gamma);
    double zeta = S.rhs1 / S.gamma;
    S.rhs1 = S.rhs2 - S.delta * zeta;
    S.rhs2 = -S.eps_ * zeta;
    S.Anorm = sqrt(S.Anorm2);
    S.xNorm = sqrt(xx);
    S.rNorm = S.phibar;
    double test1 = S.rNorm / (S.Anorm * S.xNorm);
    double test2 = S.root / S.Anorm;
    S.Acond = S.gmax / S.gmin;
    if (S.iter == 1 && S.beta / S.beta1 <= 10 * epsM) {
        S.solved = 1; S.inconsistent = 1; S.status = FPSB_ST_ZERO_ATB; S.active = 0;
        return;
    }
    S.ill_mach = (1.0 + 1.0 / S.Acond <= 1.0);
    int solved_mach = (1.0 + test2 <= 1.0);
    int zero_resid_mach = (1.0 + test1 <= 1.0);
    int resid_decrease_mach = (S.rNorm + 1.0 <= 1.0);
    S.tired = S.iter >= S.itmax;
    S.ill_lim = (1.0 / S.Acond <= S.ctol);
    int solved_lim = (test2 <= S.tol);
    int zero_resid_lim = (test1 <= S.tol);
    int resid_decrease_lim = (S.rNorm <= S.tol);
    if (S.iter >= 5) S.fwd_err = S.err_lbnd <= S.etol * sqrt(S.xENorm2);
    S.zero_resid = zero_resid_mach | zero_resid_lim;
    int resid_decrease = resid_decrease_mach | resid_decrease_lim;
    int ill_cond = S.ill_mach | S.ill_lim;
    S.solved = solved_mach | solved_lim | S.zero_resid | S.fwd_err | resid_decrease;
    if (S.solved || S.tired || ill_cond) {
        int st = FPSB_ST_UNKNOWN;
        if (S.tired) st = FPSB_ST_TIRED;
        if (S.ill_mach) st = FPSB_ST_ILLCOND_MACH;
        if (S.ill_lim) st = FPSB_ST_ILLCOND_LIM;
        if (S.solved) st = FPSB_ST_SOLVED;
        if (S.zero_resid) st = FPSB_ST_ZERO_RESID;
        if (S.fwd_err) st = FPSB_ST_FWD_ERR;
        if (resid_decrease) st = FPSB_ST_SOLVED;
        S.status = st;
        S.inconsistent = !S.zero_resid;
        S.active = 0;
    }
}

// ---- CGLS --------------------------------------------------------------------------------------
__device__ void fin_cgls_init(SlotState &S, double bb) {
    S.iter = 0;
    S.bnorm = sqrt(bb);
    S.rNorm = S.bnorm;
    if (S.bnorm == 0.0) { S.active = 0; S.solved = 1; S.status = FPSB_ST_ZERO_RHS; }
}
__device__ void fin_cgls_init_m(SlotState &S, double ss) {
    S.gamma_c = ss;
    S.pp = ss;
    S.ArNorm = sqrt(ss);
    S.tol = S.atol + S.rtol * S.ArNorm;
    S.solved = S.ArNorm <= S.tol;
    S.tired = S.iter >= S.itmax;
    if (S.solved || S.tired) { S.status = S.solved ? FPSB_ST_SOLVED : FPSB_ST_TIRED; S.active = 0; }
}
__device__ void fin_cgls_n(SlotState &S, double qq) {
    double delta = qq;
    if (S.lambda > 0) delta += S.lambda * S.pp;
    S.alpha = S.gamma_c / delta;
}
__device__ void fin_cgls_en(SlotState &S, double rr) { S.rNorm = sqrt(rr); }
__device__ void fin_cgls_m(SlotState &S, double ss) {
    S.beta_c = ss / S.gamma_c;
    S.gamma_c = ss;
}
__device__ void fin_cgls_em(SlotState &S, double pp) {
    S.pp = pp;
    S.ArNorm = sqrt(S.gamma_c);
    S.iter += 1;
    S.solved = S.ArNorm <= S.tol;
    S.tired = S.iter >= S.itmax;
    if (S.solved || S.tired) { S.status = S.solved ? FPSB_ST_SOLVED : FPSB_ST_TIRED; S.active = 0; }
}

__device__ FPSB_FINISH_INLINE void finish_step(SlotState &S, int mode, double a0, double a1) {
    switch (mode) {
        case MD_LSQR_INIT_M: fin_lsqr_init_m(S, a0); break;
        case MD_LSQR_U: fin_lsqr_u(S, a0); break;
        case MD_LSQR_V: fin_lsqr_v(S, a0, a1); break;
        case MD_CRAIG_V: fin_craig_v(S, a0); break;
        case MD_CRAIG_U: fin_craig_u(S, a0, a1); break;
        case MD_MINRES_M: fin_minres_m(S, a0); break;
        case MD_CGLS_INIT_M: fin_cgls_init_m(S, a0); break;
        case MD_CGLS_N: fin_cgls_n(S, a0); break;
        case MD_CGLS_M: fin_cgls_m(S, a0); break;
        default: break;
    }
#if defined(FPSB_EXP) && FPSB_EXP > 0
    // experiments that break the numerics still run a fixed number of iterations
    if (S.algo != ALGO_NONE) { if (S.iter < S.itmax) S.active = 1; else S.active = 0; }
#endif
}
__device__ void finish_ew(SlotState &S, int op, double a0) {
    switch (op) {
        case EW_INIT_LSQR: fin_init_lsqr(S, a0); break;
        case EW_INIT_CRAIG: fin_init_craig(S, a0); break;
        case EW_MINRES_INIT: fin_minres_init(S, a0); break;
        case EW_MINRES_E1: fin_minres_e1(S, a0); break;
        case EW_MINRES_E2: fin_minres_e2(S, a0); break;
        case EW_CGLS_INIT: fin_cgls_init(S, a0); break;
        case EW_CGLS_EN: fin_cgls_en(S, a0); break;
        case EW_CGLS_EM: fin_cgls_em(S, a0); break;
        default: break;
    }
}

// ------------------------------------------------------------------------------------------------
// per-slot coefficients loaded once per CTA
// ------------------------------------------------------------------------------------------------
struct Coef {
    int mode;
    int first, pend, lampos;     // LSQR first iteration / CRAIG pending x update / lambda > 0 (MINRES: != 0)
    int rd0, rd1, wr0, wr1;      // which aux vectors (a0 / a1) the row epilogue reads / writes
    int rdself;
    int pad_;
    double k[7];                 // mode-specific scalars, see load_coef
};

// compact form kept in registers by the step kernel's epilogue threads
struct CoefR {
    int mode, flags;             // flags: bit0 first, bit1 pend, bit2 lampos, bit3 rd0, bit4 rd1, bit5 wr0, bit6 wr1, bit7 rdself
    double k[7];
    __device__ __forceinline__ bool first() const { return flags & 1; }
    __device__ __forceinline__ bool pend() const { return flags & 2; }
    __device__ __forceinline__ bool lampos() const { return flags & 4; }
    __device__ __forceinline__ bool rd0() const { return flags & 8; }
    __device__ __forceinline__ bool rd1() const { return flags & 16; }
    __device__ __forceinline__ bool wr0() const { return flags & 32; }
    __device__ __forceinline__ bool wr1() const { return flags & 64; }
    __device__ __forceinline__ bool rdself() const { return flags & 128; }
};
__device__ __forceinline__ CoefR to_regs(const Coef &C) {
    CoefR R;
    R.mode = C.mode;
    R.flags = (C.first ? 1 : 0) | (C.pend ? 2 : 0) | (C.lampos ? 4 : 0) | (C.rd0 ? 8 : 0) | (C.rd1 ? 16 : 0) |
              (C.wr0 ? 32 : 0) | (C.wr1 ? 64 : 0) | (C.rdself ? 128 : 0);
#pragma unroll
    for (int i = 0; i < 7; ++i) R.k[i] = C.k[i];
    return R;
}

// the read / write flags only (what the operand loads of a row need): k[] stays dead, i.e. costs no registers
__device__ __forceinline__ CoefR coef_flags(const Coef &C) {
    CoefR R;
    R.mode = C.mode;
    R.flags = (C.first ? 1 : 0) | (C.pend ? 2 : 0) | (C.lampos ? 4 : 0) | (C.rd0 ? 8 : 0) | (C.rd1 ? 16 : 0) |
              (C.wr0 ? 32 : 0) | (C.wr1 ? 64 : 0) | (C.rdself ? 128 : 0);
#pragma unroll
    for (int i = 0; i < 7; ++i) R.k[i] = 0.0;
    return R;
}
// the scalars of a mode, re-read from shared memory where they are used (16 registers per slot that need not
// live through the row sums)
__device__ __forceinline__ void coef_scalars(CoefR &R, const Coef &C) {
    const volatile double *k = C.k;
#pragma unroll
    for (int i = 0; i < 7; ++i) R.k[i] = k[i];
}

// k[] per mode:
//   PLAIN        c0, c1h
//   LSQR_INIT_M  gsc
//   LSQR_U       gsc, alpha, ssc
//   LSQR_V       gsc, beta, ssc, tr_prev, sigma
//   CRAIG_V      gsc, beta, ssc, xi, c1, s1, s2g
//   CRAIG_U      gsc, alpha, ssc, mscale, trw, xr
//   MINRES_M     lambda, beta, oldbeta
//   CGLS_M       alpha, lambda
__device__ __forceinline__ void load_coef(Coef &C, const SlotIO &io, const SlotState *st, bool use_state) {
    C.mode = io.mode;
    C.rd0 = C.rd1 = C.wr0 = C.wr1 = C.rdself = 0;
    C.first = 0; C.pend = 0; C.lampos = 0; C.pad_ = 0;
    for (int i = 0; i < 7; ++i) C.k[i] = 0.0;
    if (io.mode == MD_NONE) return;
    if (io.mode == MD_PLAIN) { C.k[0] = io.c0; C.k[1] = io.c1; C.rd0 = io.a0 != nullptr; return; }
    if (!use_state) return;
    switch (io.mode) {
        case MD_LSQR_INIT_M: C.k[0] = st->su; break;
        case MD_LSQR_U:
            C.k[0] = st->sv; C.k[1] = st->alpha; C.k[2] = st->su; C.rdself = 1;
            break;
        case MD_LSQR_V:
            C.first = st->first;
            C.k[0] = st->su; C.k[1] = st->beta; C.k[2] = st->sv; C.k[3] = st->tr_prev; C.k[4] = st->sigma;
            C.rdself = 1;
            C.rd0 = C.rd1 = !C.first; C.wr0 = C.wr1 = 1;
            break;
        case MD_CRAIG_V:
            C.pend = st->pend; C.lampos = st->lambda > 0;
            C.k[0] = st->mscale * st->su; C.k[1] = st->beta; C.k[2] = st->sv; C.k[3] = st->xi;
            C.k[4] = st->c1; C.k[5] = st->s1; C.k[6] = st->s2g;
            C.rdself = 1;
            C.rd0 = C.wr0 = C.pend;
            C.rd1 = C.wr1 = C.pend && C.lampos;
            break;
        case MD_CRAIG_U:
            C.k[0] = st->sv; C.k[1] = st->alpha; C.k[2] = st->su; C.k[3] = st->mscale; C.k[4] = st->trw; C.k[5] = st->xr;
            C.rdself = 1;
            C.rd0 = C.rd1 = C.wr0 = C.wr1 = 1;
            break;
        case MD_MINRES_M:
            C.k[0] = st->lambda; C.k[1] = st->beta; C.k[2] = st->oldbeta; C.lampos = st->lambda != 0.0;
            C.rd0 = 1; C.rd1 = (st->iter + 1 >= 2);
            break;
        case MD_CGLS_M:
            C.k[0] = st->alpha; C.k[1] = st->lambda; C.lampos = st->lambda > 0;
            C.rd0 = C.rd1 = 1; C.wr0 = 1;
            break;
        default: break;
    }
}

// row epilogue on values: (sraw, selfold, a0, a1) -> returns new self; a0 / a1 updated in place
template <class CT>
__device__ __forceinline__ double row_epilogue_t(const CT &C, int mode, bool first, bool pend, bool lampos, bool rd0, bool rd1,
                                                 double sraw, double selfold, double &a0, double &a1, double &acc0, double &acc1) {
    double out = 0.0;
    switch (mode) {
        case MD_PLAIN: {
            out = C.k[0] * sraw;
            if (rd0) out += C.k[1] * a0;
            acc0 += out * out;
        } break;
        case MD_LSQR_INIT_M: {
            out = C.k[0] * sraw;
            acc0 += out * out;
        } break;
        case MD_LSQR_U: {
            out = C.k[0] * sraw - C.k[1] * (selfold * C.k[2]);
            acc0 += out * out;
        } break;
        case MD_LSQR_V: {
            const double vj = selfold * C.k[2];
            const double wj = first ? vj : (vj - C.k[3] * a0);
            acc1 += wj * wj;
            a0 = wj;
            a1 = (first ? 0.0 : a1) + C.k[4] * wj;
            out = C.k[0] * sraw - C.k[1] * vj;
            acc0 += out * out;
        } break;
        case MD_CRAIG_V: {
            const double vp = selfold * C.k[2];
            if (pend) {
                if (lampos) {
                    const double w2 = a1;
                    double x = a0 + (C.k[3] * C.k[4]) * vp;
                    x = x + (C.k[3] * C.k[5]) * w2;
                    a0 = x;
                    a1 = C.k[6] * (C.k[5] * vp - C.k[4] * w2);
                } else {
                    a0 += C.k[3] * vp;
                }
            }
            out = C.k[0] * sraw - C.k[1] * vp;
            acc0 += out * out;
        } break;
        case MD_CRAIG_U: {
            const double mu = selfold * C.k[2];
            const double uj = C.k[3] * mu;
            const double wj = uj - C.k[4] * a0;
            a0 = wj;
            a1 += C.k[5] * wj;
            acc1 += wj * wj;
            out = C.k[0] * sraw - C.k[1] * mu;
            acc0 += out * out;
        } break;
        case MD_MINRES_M: {
            // a0 = r2 (= v), a1 = r1 ; self = y
            const double r2 = a0;
            double y = sraw;
            if (lampos) y += C.k[0] * r2;
            y *= (1.0 / C.k[1]);
            if (rd1) y -= (C.k[1] / C.k[2]) * a1;
            out = y;
            acc0 += r2 * y;
        } break;
        case MD_CGLS_INIT_M: {
            out = sraw;           // p = s
            acc0 += out * out;
        } break;
        case MD_CGLS_N: {
            out = sraw;           // q
            acc0 += out * out;
        } break;
        case MD_CGLS_M: {
            // a0 = x, a1 = p ; self = s
            const double x = a0 + C.k[0] * a1;
            a0 = x;
            double sv = sraw;
            if (lampos) sv -= C.k[1] * x;
            out = sv;
            acc0 += sv * sv;
        } break;
        default: break;
    }
    return out;
}
__device__ __forceinline__ double row_epilogue(const Coef &C, double sraw, double selfold, double &a0, double &a1,
                                               double &acc0, double &acc1) {
    return row_epilogue_t(C, C.mode, C.first != 0, C.pend != 0, C.lampos != 0, C.rd0 != 0, C.rd1 != 0, sraw, selfold, a0, a1, acc0, acc1);
}
__device__ __forceinline__ double row_epilogue(const CoefR &C, double sraw, double selfold, double &a0, double &a1,
                                               double &acc0, double &acc1) {
    return row_epilogue_t(C, C.mode, C.first(), C.pend(), C.lampos(), C.rd0(), C.rd1(), sraw, selfold, a0, a1, acc0, acc1);
}

// ------------------------------------------------------------------------------------------------
// the fused SpMM step kernel — tiled SELL-32 streamed through a TMA ring by persistent CTAs.
//
// Layout: the rows of the operator are cut into tiles of up to kTileRows (256) consecutive rows — as
// many as fit a ring stage, so that a tile block is 25-30 KB whether rows are long or short; inside
// a tile the rows are sorted by length and packed into up to 8 slices of 32 (lane == row).  A slice
// stores its entries as "pair rows": entries 2p and 2p+1 of the 32 lanes are interleaved, so one
// 16-byte access brings two values and one 8-byte access two column indices per lane (an odd last
// entry is stored as a plain 32-entry row).  Everything a tile needs from the operator —
// [values | column indices | lane -> row map] — is ONE contiguous block in HBM.
//
// One persistent CTA per SM walks the tiles b, b + grid, b + 2 grid, ... :
//   producers (warps 0-3, one lane each) keep the ring full with cp.async.bulk (TMA) + mbarrier:
//             warps 0/1 copy the blocks of the CTA's even / odd tiles, warps 2/3 the slice of the
//             gathered vector(s) the tile can touch — columns [cmin, cmin + ccnt) — into the same
//             ring stage.  Measured on B200 (tools/micro/tma_bw.cu): a bulk copy costs its issuing
//             thread ~0.35 us whatever its size and an SM sustains one per ~0.17 us, so full HBM
//             bandwidth needs >= 16 KB per copy: hence one big block per tile and two issuing warps.
//   consumers kGroups groups of 4 warps; group g takes the CTA's tiles g, g + kGroups, ...
//     phase 1  warp w reduces slices w and ns-1-w (the widest with the narrowest: balanced): values /
//              indices are read conflict-free from the stage, the gathers cost shared-memory bank
//              cycles instead of one L1 wavefront per distinct 128-byte line; the two row sums of
//              every row go to a small per-group buffer indexed by the row's position in the tile,
//              and the stage is handed back to the producers.
//     phase 2  the Krylov row epilogue runs over the tile's rows in natural order (thread t: rows t
//              and t + 128), so every vector it reads and writes is accessed fully coalesced even
//              though SELL permuted the rows; the operands of the first row were requested before
//              phase 1, those of the second while the first is finished.
//   Groups are in different phases at any time, so the shared-memory pipe, the HBM stream and the
//   epilogue traffic overlap inside one SM.  Measured (tools/loop_timers.py): a group needs ~1.8 us
//   per tile almost independently of the tile's size (a latency chain, not a throughput limit),
//   which is why short-row operators get 256-row tiles.
// Tiles whose column span exceeds the window capacity gather from global memory instead.
// Rows longer than kLongRow are handled by a small separate kernel (one CTA per row) launched
// before this one; its per-row norm partials join the fixed-order reduction below.
// Norms: per-thread partial sums over the CTA's tiles (fixed order) -> fixed-tree CTA sum -> the
// grid's last CTA adds the per-CTA partials in index order and runs the scalar recurrences.  The
// result does not depend on the order in which CTAs finish.
// ------------------------------------------------------------------------------------------------
constexpr int kTileRows = 256;
constexpr int kTileSlices = kTileRows / 32;
constexpr int kGroups = 3;
constexpr int kGroupThreads = 128;                             // phase 1: a warp per slice pair ; phase 2: a thread per row pair
constexpr int kGroupWarps = kGroupThreads / 32;
constexpr int kProducerThreads = 128;                          // warps 0,1: tile blocks (even / odd tiles), warps 2,3: gather windows
constexpr int kStepThreads = kProducerThreads + kGroups * kGroupThreads;
constexpr int kStageBytesMax = 40 * 1024;                      // tile block + window
constexpr int kMaxStages = 8;
#ifndef FPSB_RING_KB
#define FPSB_RING_KB 188
#endif
constexpr int kRingBudget = FPSB_RING_KB * 1024;
constexpr int kWinCapMax = 1536;          // window capacity (entries of 16 bytes) a tile may ask for
constexpr int kSegCapMax = 1664;          // ... when the window is multi-segment (three 2 x 256 + 4 runs of an interleaved 5-point stencil: 1 548)
constexpr int kSegStageBytesMax = 44 * 1024;   // tile block + multi-segment window (still four ring stages)
constexpr int kLongThreads = 256;

struct __align__(16) TileMeta {
    long long boff;      // byte offset of the tile's block [values elems*8 | indices elems*2 (window-relative u16) or elems*4 (global) | row map ns*32 (u8)]
    int elems;           // stored entries (multiple of 32)
    int ns;              // slices in the tile, ns <= kTileSlices
    int cmin, ccnt;      // gather window (ccnt == 0: gather from global memory, indices are global columns)
    int row0, nrows;     // rows [row0, row0 + nrows) of the operator
    unsigned char width[kTileSlices];   // entries per row of each slice (rows sorted by length: widths descend)
    int nsell;           // rows stored in the slices (nrows minus the long rows): lane l of slice s is a row iff 32 s + l < nsell
    int pad_;
};
static_assert(sizeof(TileMeta) == 48 && kTileSlices == 8, "TileMeta is loaded as three int4");
static_assert(kTileRows == 2 * kGroupThreads, "phase 2 maps a thread to rows t and t + 128");
static_assert(kTileRows <= 256, "the lane -> row map is stored as bytes");

__host__ __device__ __forceinline__ unsigned tile_block_bytes(int elems, int ns, int ccnt) {
    return (unsigned)elems * (ccnt > 0 ? 10u : 12u) + (unsigned)ns * 32u;
}

__device__ __forceinline__ TileMeta load_tile(const TileMeta *tiles, int t) {
    const int4 *tp = reinterpret_cast<const int4 *>(tiles + t);
    const int4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
    TileMeta T;
    T.boff = (long long)(((unsigned long long)(unsigned)a.y << 32) | (unsigned)a.x);
    T.elems = a.z; T.ns = a.w;
    T.cmin = b.x; T.ccnt = b.y; T.row0 = b.z; T.nrows = b.w;
    *reinterpret_cast<int *>(&T.width[0]) = c.x; *reinterpret_cast<int *>(&T.width[4]) = c.y;
    T.nsell = c.z; T.pad_ = 0;
    return T;
}
// what a block producer needs of a descriptor
struct PTile { long long boff; int elems, ns, cmin, ccnt; };
__device__ __forceinline__ PTile load_ptile(const TileMeta *tiles, int t) {
    const int4 *tp = reinterpret_cast<const int4 *>(tiles + t);
    const int4 a = __ldg(tp);
    const int2 b = __ldg(reinterpret_cast<const int2 *>(tp + 1));
    PTile T;
    T.boff = (long long)(((unsigned long long)(unsigned)a.y << 32) | (unsigned)a.x);
    T.elems = a.z; T.ns = a.w; T.cmin = b.x; T.ccnt = b.y;
    return T;
}

// what a consumer keeps of a tile descriptor (registers): everything but the block offset
struct CTile {
    int elems, cmin, ccnt, row0;
    int pk;              // ns | nrows << 4 | nsell << 14
    unsigned w0, w1;     // the eight slice widths, one byte each (widths <= kLongRow < 256)
    __device__ __forceinline__ int ns() const { return pk & 0xf; }
    __device__ __forceinline__ int nrows() const { return (pk >> 4) & 0x3ff; }
    __device__ __forceinline__ int nsell() const { return pk >> 14; }
    __device__ __forceinline__ int width(int i) const {
        return (int)((((unsigned long long)w1 << 32 | (unsigned long long)w0) >> (8 * i)) & 0xffull);
    }
};
__device__ __forceinline__ CTile load_ctile(const TileMeta *tiles, int t) {
    const int4 *tp = reinterpret_cast<const int4 *>(tiles + t);
    const int4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
    CTile T;
    T.elems = a.z; T.cmin = b.x; T.ccnt = b.y; T.row0 = b.z;
    T.pk = a.w | (b.w << 4) | (c.z << 14);
    T.w0 = (unsigned)c.x; T.w1 = (unsigned)c.y;
    return T;
}

__device__ __forceinline__ void group_bar(int g) {
    asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(kGroupThreads) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void *p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
// all consumer threads of the CTA (the producer warps never join: they run on 40 registers and leave early)
__device__ __forceinline__ void consumers_bar() {
    asm volatile("bar.sync %0, %1;" ::"n"(1 + kGroups), "n"(kGroups * kGroupThreads) : "memory");
}
// fixed-tree sum of 4 values per consumer thread; result valid in every lane of consumer warp 0
__device__ __forceinline__ void consumers_sum4(double (&v)[4], double *scratch /* 4*32 */, int cw, int lane) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const double x = warp_sum(v[q]);
        if (lane == 0) scratch[q * 32 + cw] = x;
    }
    consumers_bar();
    if (cw == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = warp_sum(lane < kGroups * kGroupWarps ? scratch[q * 32 + lane] : 0.0);
    }
    consumers_bar();
}
// warp-group register reallocation (sm_90+): the four producer warps need ~40 registers, which frees
// 24 more for every consumer thread (128 -> 152) out of the same 64 K register file
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
constexpr int kProducerRegs = 40, kConsumerRegs = 152;
static_assert(kProducerThreads * kProducerRegs + kGroups * kGroupThreads * kConsumerRegs <= 65536, "register file");

// ---- consumer building blocks shared by gk_step_kernel and gk_loop_kernel ----------------------------
// operands of one row of the Krylov row epilogue
struct RowOps { double2 old2; double a00, a01, a10, a11; };

template <bool PAIR>
__device__ __forceinline__ void load_row_ops(const StepParams &P, const CoefR &C0, const CoefR &C1, int row, RowOps &R) {
    if (PAIR) R.old2 = P.self2[row];
    else {
        R.old2 = make_double2(0.0, 0.0);
        if (C0.rdself()) R.old2.x = P.io[0].self[row];
        if (C1.rdself()) R.old2.y = P.io[1].self[row];
    }
    R.a00 = R.a01 = R.a10 = R.a11 = 0.0;
    if (C0.rd0()) R.a00 = __ldcs(P.io[0].a0 + row);
    if (C0.rd1()) R.a01 = __ldcs(P.io[0].a1 + row);
    if (C1.rd0()) R.a10 = __ldcs(P.io[1].a0 + row);
    if (C1.rd1()) R.a11 = __ldcs(P.io[1].a1 + row);
}
// pull the epilogue operands of the group's next tile into L2 (no registers held)
template <bool PAIR>
__device__ __forceinline__ void prefetch_row_ops(const StepParams &P, const CoefR &C0, const CoefR &C1, int r2, int t) {
    if (PAIR) { if ((t & 7) == 0) prefetch_l2(P.self2 + r2); }
    else if ((t & 15) == 0) {
        if (C0.rdself()) prefetch_l2(P.io[0].self + r2);
        if (C1.rdself()) prefetch_l2(P.io[1].self + r2);
    }
    if ((t & 15) == 0) {
        if (C0.rd0()) prefetch_l2(P.io[0].a0 + r2);
        if (C0.rd1()) prefetch_l2(P.io[0].a1 + r2);
        if (C1.rd0()) prefetch_l2(P.io[1].a0 + r2);
        if (C1.rd1()) prefetch_l2(P.io[1].a1 + r2);
    }
}
// the Krylov row epilogue of one row (phase 2) ; raw rows of a row-partitioned run only leave their sums
template <bool PAIR>
__device__ __forceinline__ void finish_row(const StepParams &P, const CoefR &C0, const CoefR &C1, bool act0, bool act1, int row,
                                           int rflag, const double2 sm, RowOps &R, double (&acc)[4]) {
    if (rflag == 2 && P.raw_out == nullptr) rflag = 0;     // raw rows only matter to launches that ask for them
    if (rflag == 2) P.raw_out[row] = sm;                   // halo / boundary row of a row-partitioned run
    if (rflag != 0) return;
    double n0 = R.old2.x, n1 = R.old2.y;
    if (act0) n0 = row_epilogue(C0, sm.x, R.old2.x, R.a00, R.a01, acc[0], acc[1]);
    if (act1) n1 = row_epilogue(C1, sm.y, R.old2.y, R.a10, R.a11, acc[2], acc[3]);
    if (PAIR) P.self2[row] = make_double2(n0, n1);
    else {
        if (act0) P.io[0].self[row] = n0;
        if (act1) P.io[1].self[row] = n1;
    }
    if (C0.wr0()) __stcs(P.io[0].a0 + row, R.a00);
    if (C0.wr1()) __stcs(P.io[0].a1 + row, R.a01);
    if (C1.wr0()) __stcs(P.io[1].a0 + row, R.a10);
    if (C1.wr1()) __stcs(P.io[1].a1 + row, R.a11);
}
// row sums of one slice against both columns (phase 1).  VOLATILE_GATHER: the gathered vector changes
// during the kernel's life time (persistent loop), so global gathers must not use the read-only path
template <bool PAIR, bool VOLATILE_GATHER>
__device__ __forceinline__ double2 slice_sums(const StepParams &P, const unsigned char *st, int elems, bool windowed, int off, int width,
                                              const unsigned char *s_win, bool act0, bool act1, int lane) {
    const double *s_val = reinterpret_cast<const double *>(st);
    const int *s_col = reinterpret_cast<const int *>(st + (size_t)elems * 8);                        // global columns
    const unsigned short *s_c16 = reinterpret_cast<const unsigned short *>(st + (size_t)elems * 8);   // window-relative
    const int npair = width >> 1;
    const bool tail = (width & 1) != 0;
    double s0 = 0.0, s1 = 0.0, u0 = 0.0, u1 = 0.0;     // two accumulator pairs: shorter DFMA chains
    const double2 *sv = reinterpret_cast<const double2 *>(s_val + off) + lane;
    const int2 *sc = reinterpret_cast<const int2 *>(s_col + off) + lane;
    const ushort2 *sc16 = reinterpret_cast<const ushort2 *>(s_c16 + off) + lane;
    if (PAIR) {
        if (windowed) {
            const double2 *win2 = reinterpret_cast<const double2 *>(s_win);
#pragma unroll 5
            for (int p = 0; p < npair; ++p) {
                const double2 v = sv[p * 32];
                const ushort2 c = sc16[p * 32];
                const double2 x0 = win2[c.x], x1 = win2[c.y];
                s0 = fma(v.x, x0.x, s0); s1 = fma(v.x, x0.y, s1);
                u0 = fma(v.y, x1.x, u0); u1 = fma(v.y, x1.y, u1);
            }
            if (tail) {
                const double v = s_val[off + npair * 64 + lane];
                const double2 x = win2[s_c16[off + npair * 64 + lane]];
                s0 = fma(v, x.x, s0); s1 = fma(v, x.y, s1);
            }
        } else {
            const double2 *gin2 = P.gin2;
            auto ld = [&](int c) { return VOLATILE_GATHER ? __ldcg(gin2 + c) : __ldg(gin2 + c); };
#pragma unroll 5
            for (int p = 0; p < npair; ++p) {
                const double2 v = sv[p * 32];
                const int2 c = sc[p * 32];
                const double2 x0 = ld(c.x), x1 = ld(c.y);
                s0 = fma(v.x, x0.x, s0); s1 = fma(v.x, x0.y, s1);
                u0 = fma(v.y, x1.x, u0); u1 = fma(v.y, x1.y, u1);
            }
            if (tail) {
                const double v = s_val[off + npair * 64 + lane];
                const double2 x = ld(s_col[off + npair * 64 + lane]);
                s0 = fma(v, x.x, s0); s1 = fma(v, x.y, s1);
            }
        }
    } else {
        const double *win0 = reinterpret_cast<const double *>(s_win);
        const double *win1 = win0 + P.win_cap;
        auto gather_fma = [&](double v, int c, double &r0, double &r1) {
            if (act0) r0 = fma(v, windowed ? win0[c] : __ldg(P.io[0].gin + c), r0);
            if (act1) r1 = fma(v, windowed ? win1[c] : __ldg(P.io[1].gin + c), r1);
        };
#pragma unroll 5
        for (int p = 0; p < npair; ++p) {
            const double2 v = sv[p * 32];
            int cx, cy;
            if (windowed) { const ushort2 c = sc16[p * 32]; cx = c.x; cy = c.y; }
            else { const int2 c = sc[p * 32]; cx = c.x; cy = c.y; }
            gather_fma(v.x, cx, s0, s1);
            gather_fma(v.y, cy, u0, u1);
        }
        if (tail) gather_fma(s_val[off + npair * 64 + lane],
                             windowed ? (int)s_c16[off + npair * 64 + lane] : s_col[off + npair * 64 + lane], s0, s1);
    }
    return make_double2(s0 + u0, s1 + u1);
}
// phase 1 of a tile: warp `wid` of the group reduces slices wid and ns - 1 - wid
template <bool PAIR, bool VOLATILE_GATHER>
__device__ __forceinline__ void tile_row_sums(const StepParams &P, const CTile &T, const unsigned char *st, const unsigned char *s_win,
                                              bool act0, bool act1, int wid, int lane, double2 *sum) {
    const int ns = T.ns();
    const bool windowed = T.ccnt > 0;
    const unsigned char *s_map = st + (size_t)T.elems * (windowed ? 10 : 12);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int sl = h == 0 ? wid : ns - 1 - wid;
        if (h == 0 ? (sl >= ns) : (sl < kGroupWarps)) continue;
        int off = 0;
#pragma unroll
        for (int i = 0; i < kTileSlices - 1; ++i) if (i < sl) off += T.width(i) * 32;
        const double2 r = slice_sums<PAIR, VOLATILE_GATHER>(P, st, T.elems, windowed, off, T.width(sl), s_win, act0, act1, lane);
        const int idx = sl * 32 + lane;
        if (idx < T.nsell()) sum[s_map[idx]] = r;
    }
}

#ifdef FPSB_PHASE_TIMERS
__device__ unsigned long long g_phase_cycles[16];
#endif

template <bool PAIR>
__global__ void __launch_bounds__(kStepThreads, 1) gk_step_kernel(const __grid_constant__ StepParams P, int use_state) {
    extern __shared__ __align__(128) unsigned char s_dyn[];
    __shared__ double2 s_sum[kGroups][2][kTileRows];        // [group][double buffer][row]
    __shared__ double s_red[4 * 32];
    __shared__ alignas(8) uint64_t full_bar[kMaxStages];
    __shared__ alignas(8) uint64_t empty_bar[kMaxStages];
    __shared__ int s_rel[kMaxStages];                       // rounds seen filled, per stage (see stage_turn_wait)
    __shared__ SlotState sS[2];
    __shared__ Coef sC[2];
    __shared__ int s_last;

    const int tid = threadIdx.x;
    const int cta = blockIdx.x, nstage = P.nstage, gsz = (int)gridDim.x;
    // Programmatic dependent launch: this grid may be scheduled while the previous kernel of the
    // stream drains (its CTAs free their SMs one by one).  Everything above the wait touches only
    // this CTA's own shared memory; everything below may read what the previous kernel wrote.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid == 0) {
        for (int s = 0; s < nstage; ++s) { mbar_init(&full_bar[s], 2); mbar_init(&empty_bar[s], kGroupWarps); s_rel[s] = 0; }
        mbar_fence_init();
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // ---- prologue: one round trip brings both slot states (and the previous launch's partials) in ----
    __shared__ double s_tot[4];
    if (use_state) {
        const double *g = reinterpret_cast<const double *>(P.st);
        double *d = reinterpret_cast<double *>(sS);
        for (int i = tid; i < (int)(2 * sizeof(SlotState) / sizeof(double)); i += kStepThreads) d[i] = __ldcg(g + i);
    }
    if (P.pend_partials != nullptr) {
        // deferred recurrences of the previous step: fixed-order sum of its per-CTA partials ...
        double tot[4] = {0.0, 0.0, 0.0, 0.0};
        for (int i = tid; i < P.pend_nparts; i += kStepThreads) {
            const double *pp = P.pend_partials + (size_t)i * 4;
            tot[0] += __ldcg(pp + 0); tot[1] += __ldcg(pp + 1);
            tot[2] += __ldcg(pp + 2); tot[3] += __ldcg(pp + 3);
        }
        block_sum<4>(tot, s_red);
        if (tid == 0) { s_tot[0] = tot[0]; s_tot[1] = tot[1]; s_tot[2] = tot[2]; s_tot[3] = tot[3]; }
        __syncthreads();
        // ... then the two slots' scalar recurrences side by side (thread 0 and thread 32)
        if (tid == 0 && P.pend_m0 != MD_NONE && sS[0].active) finish_step(sS[0], P.pend_m0, s_tot[0], s_tot[1]);
        if (tid == 32 && P.pend_m1 != MD_NONE && sS[1].active) finish_step(sS[1], P.pend_m1, s_tot[2], s_tot[3]);
    }
    __syncthreads();
    if (P.st_out != nullptr && cta == 0) {
        if (tid == 0 && !sS[0].active && !sS[1].active) *P.done_flag = 1;
        const double *src = reinterpret_cast<const double *>(sS);
        double *dst = reinterpret_cast<double *>(P.st_out);
        for (int i = tid; i < (int)(2 * sizeof(SlotState) / sizeof(double)); i += kStepThreads) dst[i] = src[i];
    }
    const bool act0 = P.io[0].mode != MD_NONE && (!use_state || sS[0].active);
    const bool act1 = P.io[1].mode != MD_NONE && (!use_state || sS[1].active);
    if (!act0 && !act1) return;
    if (tid == 0) {
        load_coef(sC[0], P.io[0], &sS[0], use_state);
        load_coef(sC[1], P.io[1], &sS[1], use_state);
        if (!act0) { sC[0].mode = MD_NONE; sC[0].rd0 = sC[0].rd1 = sC[0].wr0 = sC[0].wr1 = sC[0].rdself = 0; }
        if (!act1) { sC[1].mode = MD_NONE; sC[1].rd0 = sC[1].rd1 = sC[1].wr0 = sC[1].wr1 = sC[1].rdself = 0; }
    }
    __syncthreads();
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    // stage layout: [tile block, blk_cap bytes | window win_cap*16 bytes]
    const size_t stage_bytes = (size_t)P.stage_bytes;
    // vectors of doubles need 16-byte aligned sources for the TMA path (the pairs always are)
    const bool win_tma = PAIR || ((((uintptr_t)P.io[0].gin | (uintptr_t)P.io[1].gin) & 15) == 0);
    bool ok = true;

    if (tid < kProducerThreads) {
        // ------------------------------- producers -------------------------------
        reg_dec<kProducerRegs>();
        // multi-segment windows: lanes 0..3 of a window producer warp own one segment each (they issue their bulk copies
        // side by side); everything else is lane 0's
        const int seg_lane = tid & 31;
        if (seg_lane == 0 || (seg_lane < 4 && (tid >> 5) >= 2 && P.wsegs != nullptr)) {
            // a bulk copy costs its issuing thread a few hundred ns whatever its size: two warps share
            // the tile blocks (even / odd tiles of this CTA), two more the gather windows
            const int role = tid >> 5;
            const bool blocks = role < 2;
            const int par = role & 1;
            const bool segd = !blocks && P.wsegs != nullptr;
            const unsigned seg_mask = segd ? 0xfu : 0x1u;
            int2 G = make_int2(0, 0), G1 = make_int2(0, 0);        // this lane's segment of tiles T / T1
            // tile descriptors are fetched one of this producer's tiles ahead of their use
            int k = par, tile = cta + par * gsz;
            PTile T{}, T1{};
            if (tile < P.ntiles) { T = load_ptile(P.tiles, tile); if (segd) G = __ldg(P.wsegs + (size_t)tile * 4 + seg_lane); }
            for (; tile < P.ntiles; k += 2) {
                const int t1 = tile + 2 * gsz;
                if (t1 < P.ntiles) { T1 = load_ptile(P.tiles, t1); if (segd) G1 = __ldg(P.wsegs + (size_t)t1 * 4 + seg_lane); }
                const int s = k % nstage;
                if (k >= nstage) ok = mbar_wait(&empty_bar[s], (uint32_t)((k / nstage - 1) & 1)) && ok;
                // bounded run-ahead: tile k - inflight must have landed.  Everything an SM requests is
                // served in order, so a deep TMA backlog is pure latency for the epilogue's own loads
                if (k >= P.inflight) {
                    const int kb = k - P.inflight;
                    ok = mbar_wait(&full_bar[kb % nstage], (uint32_t)((kb / nstage) & 1)) && ok;
                }
                unsigned char *st = s_dyn + (size_t)s * stage_bytes;
                if (blocks) {
                    const uint32_t bytes = tile_block_bytes(T.elems, T.ns, T.ccnt);
                    mbar_expect_tx(&full_bar[s], bytes);
                    if (bytes) tma_bulk_g2s(st, P.tbuf + T.boff, bytes, &full_bar[s]);
                } else {
                    unsigned char *s_win = st + (size_t)P.blk_cap;
                    uint32_t wbytes = 0, tot = 0;
                    if (T.ccnt > 0) {
                        if (PAIR) { wbytes = (uint32_t)T.ccnt * 16u; tot = wbytes; }
                        else if (win_tma && !(T.ccnt & 1)) { wbytes = (uint32_t)T.ccnt * 8u; tot = wbytes * ((act0 ? 1u : 0u) + (act1 ? 1u : 0u)); }
                    }
                    if (seg_lane == 0) mbar_expect_tx(&full_bar[s], tot);
                    if (segd) {
                        // the expectation is posted before any of the four lanes' copies can complete
                        __syncwarp(seg_mask);
                        const int glen = G.y >> 16, goff = G.y & 0xffff;
                        if (wbytes && glen > 0) {
                            if (PAIR) tma_bulk_g2s(s_win + (size_t)goff * 16, P.gin2 + G.x, (uint32_t)glen * 16u, &full_bar[s]);
                            else {
                                double *w0 = reinterpret_cast<double *>(s_win);
                                if (act0) tma_bulk_g2s(w0 + goff, P.io[0].gin + G.x, (uint32_t)glen * 8u, &full_bar[s]);
                                if (act1) tma_bulk_g2s(w0 + P.win_cap + goff, P.io[1].gin + G.x, (uint32_t)glen * 8u, &full_bar[s]);
                            }
                        }
                    } else if (wbytes) {
                        if (PAIR) tma_bulk_g2s(s_win, P.gin2 + T.cmin, wbytes, &full_bar[s]);
                        else {
                            double *w0 = reinterpret_cast<double *>(s_win);
                            if (act0) tma_bulk_g2s(w0, P.io[0].gin + T.cmin, wbytes, &full_bar[s]);
                            if (act1) tma_bulk_g2s(w0 + P.win_cap, P.io[1].gin + T.cmin, wbytes, &full_bar[s]);
                        }
                    }
                }
                T = T1; G = G1; tile = t1;
            }
            if (!ok) atomicExch(P.done_flag, -1);
        }
        return;          // the reductions and recurrences below belong to the consumer warps
    }
    // ------------------------------- consumers -------------------------------
    const int ct = tid - kProducerThreads;
    const int cw = ct >> 5, clane = ct & 31;
    {
        // (1 CTA per SM with a 215 KB ring leaves almost no L1: a register spill costs an L2 round
        //  trip, so this kernel must stay spill-free)
        reg_inc<kConsumerRegs>();
        const int g = ct / kGroupThreads, t = ct % kGroupThreads;
        const int lane = t & 31, wid = t >> 5;
        const CoefR C0 = to_regs(sC[0]), C1 = to_regs(sC[1]);
        int k = g;
        int tile = cta + k * gsz;
        // tile descriptors are fetched two tiles ahead of their use; the row-epilogue operands of the
        // group's next tile are pulled into L2 one tile ahead (no registers held)
        CTile T{}, Tn{}, Tnn{};
        if (tile < P.ntiles) T = load_ctile(P.tiles, tile);
        if (tile + kGroups * gsz < P.ntiles) Tn = load_ctile(P.tiles, tile + kGroups * gsz);
        for (; tile < P.ntiles; k += kGroups) {
            const int s = k % nstage;
            const int ntile = cta + (k + kGroups) * gsz, nntile = cta + (k + 2 * kGroups) * gsz;
            if (nntile < P.ntiles) Tnn = load_ctile(P.tiles, nntile);
            // row-epilogue operands of this thread's first row: in flight during the wait and phase 1.
            // The row flags are only consumed in phase 2: the operand loads do not wait for them (they are
            // in bounds for flagged rows too), so the flags cost no extra round trip per tile
            const int rowA = T.row0 + t, rowB = rowA + kGroupThreads;
            const bool inA = t < T.nrows(), inB = t + kGroupThreads < T.nrows();
            const int flagA = (P.rowflag != nullptr && inA) ? (int)P.rowflag[rowA] : 0;
            const int flagB = (P.rowflag != nullptr && inB) ? (int)P.rowflag[rowB] : 0;
            RowOps RA{};
            if (inA) load_row_ops<PAIR>(P, C0, C1, rowA, RA);
            if (ntile < P.ntiles) {
                if (t < Tn.nrows()) prefetch_row_ops<PAIR>(P, C0, C1, Tn.row0 + t, t);
                if (t + kGroupThreads < Tn.nrows()) prefetch_row_ops<PAIR>(P, C0, C1, Tn.row0 + kGroupThreads + t, t);
            }
            const unsigned char *st = s_dyn + (size_t)s * stage_bytes;
            unsigned char *s_win = const_cast<unsigned char *>(st) + (size_t)P.blk_cap;
            stage_turn_wait(&s_rel[s], k / nstage);
            ok = mbar_wait(&full_bar[s], (uint32_t)((k / nstage) & 1)) && ok;
            if (t == 0) stage_seen(&s_rel[s], k / nstage);
            if (!PAIR && T.ccnt > 0 && !(win_tma && !(T.ccnt & 1))) {
                // unaligned / odd-sized caller vectors: the group stages the window itself
                double *win0 = reinterpret_cast<double *>(s_win);
                double *win1 = win0 + P.win_cap;
                if (P.wsegs != nullptr) {
                    for (int sgi = 0; sgi < 4; ++sgi) {
                        const int2 G = __ldg(P.wsegs + (size_t)tile * 4 + sgi);
                        const int glen = G.y >> 16, goff = G.y & 0xffff;
                        for (int i = t; i < glen; i += kGroupThreads) {
                            if (act0) win0[goff + i] = P.io[0].gin[G.x + i];
                            if (act1) win1[goff + i] = P.io[1].gin[G.x + i];
                        }
                    }
                } else
                for (int i = t; i < T.ccnt; i += kGroupThreads) {
                    if (act0) win0[i] = P.io[0].gin[T.cmin + i];
                    if (act1) win1[i] = P.io[1].gin[T.cmin + i];
                }
                group_bar(g);
            }
            // ---------------- phase 1: row sums ----------------
            double2 *sum = s_sum[g][(k / kGroups) & 1];
            tile_row_sums<PAIR, false>(P, T, st, s_win, act0, act1, wid, lane, sum);
            // the stage is consumed: hand it back to the producers (one arrival per warp)
            if (!PAIR) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // group-staged windows
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[s]);
            group_bar(g);
            // ---------------- phase 2: row epilogue in natural row order ----------------
            RowOps RB{};
            if (inB) load_row_ops<PAIR>(P, C0, C1, rowB, RB);
            if (inA) finish_row<PAIR>(P, C0, C1, act0, act1, rowA, flagA, sum[t], RA, acc);
            if (inB) finish_row<PAIR>(P, C0, C1, act0, act1, rowB, flagB, sum[t + kGroupThreads], RB, acc);
            T = Tn; Tn = Tnn;
            tile = ntile;
        }
    }
    if (!ok) atomicExch(P.done_flag, -1);
    if (!use_state) return;

    // deterministic norms: one partial per CTA, reduced in a fixed order — by the next launch's
    // prologue (deferred mode) or by this grid's last CTA
    constexpr int kCons = kGroups * kGroupThreads;
    consumers_sum4(acc, s_red, cw, clane);
    if (P.st_out != nullptr) {
        if (ct == 0) {
            double *pp = P.partials + (size_t)cta * 4;
            pp[0] = acc[0]; pp[1] = acc[1]; pp[2] = acc[2]; pp[3] = acc[3];
        }
        return;
    }
    if (ct == 0) {
        double *pp = P.partials + (size_t)cta * 4;
        pp[0] = acc[0]; pp[1] = acc[1]; pp[2] = acc[2]; pp[3] = acc[3];
        __threadfence();
        unsigned tk = atomicAdd(P.counter, 1u);
        s_last = (tk == gridDim.x - 1);
    }
    consumers_bar();
    if (!s_last) return;
    __threadfence();
    double tot[4] = {0.0, 0.0, 0.0, 0.0};
    const int nparts = (int)gridDim.x + P.nlong;       // long-row partials follow the CTA partials
    for (int i = ct; i < nparts; i += kCons) {
        const double *pp = P.partials + (size_t)i * 4;
        tot[0] += __ldcg(pp + 0); tot[1] += __ldcg(pp + 1);
        tot[2] += __ldcg(pp + 2); tot[3] += __ldcg(pp + 3);
    }
    consumers_sum4(tot, s_red, cw, clane);
    if (P.tot_out != nullptr && P.ptail == nullptr) {
        if (ct == 0) {
            P.tot_out[0] = tot[0]; P.tot_out[1] = tot[1]; P.tot_out[2] = tot[2]; P.tot_out[3] = tot[3];
            *P.counter = 0;
        }
        return;
    }
    if (P.ptail != nullptr) {
        // all-reduce over the ranks through the mailboxes: put, signal, wait, sum in rank order
        const PeerTail &X = *P.ptail;
        const int R = X.nranks;
        const unsigned long long seq = P.pt_sig + 1;
        if (ct == 0) {
            for (int p = 0; p < R; ++p) {
                if (p == X.rank) continue;
                double *dst = reinterpret_cast<double *>(X.peer[p] + kMboxOffTot) + ((size_t)P.pt_par * kMboxMaxRanks + X.rank) * 4;
                dst[0] = tot[0]; dst[1] = tot[1]; dst[2] = tot[2]; dst[3] = tot[3];
            }
            __threadfence_system();
        }
        consumers_bar();
        if (ct < R && ct != X.rank) {
            st_release_sys(reinterpret_cast<unsigned long long *>(X.peer[ct]) + X.rank, seq);
            const unsigned long long *f = reinterpret_cast<const unsigned long long *>(X.mine) + ct;
            const unsigned long long t0 = global_ns();
            while (ld_acquire_sys(f) < seq) {
                if (global_ns() - t0 > 4000000000ull) { atomicExch(X.err, 1); break; }
            }
        }
        consumers_bar();
        if (ct == 0) {
            const double *in = reinterpret_cast<const double *>(X.mine + kMboxOffTot) + (size_t)P.pt_par * kMboxMaxRanks * 4;
            double all[4] = {0.0, 0.0, 0.0, 0.0};
            for (int r = 0; r < R; ++r)
                for (int q = 0; q < 4; ++q) all[q] += (r == X.rank) ? tot[q] : __ldcg(in + r * 4 + q);
            tot[0] = all[0]; tot[1] = all[1]; tot[2] = all[2]; tot[3] = all[3];
            P.tot_out[0] = tot[0]; P.tot_out[1] = tot[1]; P.tot_out[2] = tot[2]; P.tot_out[3] = tot[3];
        }
    }
    // scalar recurrences on the shared-memory copy of the slot states (global memory would cost one
    // L2 round trip per field): the two slots side by side on two warps, then one coalesced write-back
    // (the totals live in consumer warp 0: slot 1's pair is handed over through shared memory)
    if (ct == 0) { s_tot[2] = tot[2]; s_tot[3] = tot[3]; }
    consumers_bar();
    if (ct == 0 && act0) finish_step(sS[0], P.io[0].mode, tot[0], tot[1]);
    if (ct == 32 && act1) finish_step(sS[1], P.io[1].mode, s_tot[2], s_tot[3]);
    consumers_bar();
    if (ct == 0) {
        if (!sS[0].active && !sS[1].active) *P.done_flag = 1;
        *P.counter = 0;
    }
    {
        const double *src = reinterpret_cast<const double *>(sS);
        double *dst = reinterpret_cast<double *>(P.st);
        for (int i = ct; i < (int)(2 * sizeof(SlotState) / sizeof(double)); i += kCons) dst[i] = src[i];
    }
}

// recurrences of a deferred step whose successor is not a step launch (end of a chunk / of the loop)
__global__ void __launch_bounds__(256) flush_finish_kernel(SlotState *st, const double *partials, int nparts, int m0, int m1,
                                                           int *done_flag) {
    __shared__ double s_red[4 * 32];
    __shared__ SlotState sS[2];
    __shared__ double s_tot[4];
    const int tid = threadIdx.x;
    for (int i = tid; i < (int)(2 * sizeof(SlotState) / sizeof(double)); i += 256)
        reinterpret_cast<double *>(sS)[i] = reinterpret_cast<const double *>(st)[i];
    double tot[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = tid; i < nparts; i += 256) {
        const double *pp = partials + (size_t)i * 4;
        tot[0] += pp[0]; tot[1] += pp[1]; tot[2] += pp[2]; tot[3] += pp[3];
    }
    block_sum<4>(tot, s_red);
    if (tid == 0) { s_tot[0] = tot[0]; s_tot[1] = tot[1]; s_tot[2] = tot[2]; s_tot[3] = tot[3]; }
    __syncthreads();
    if (tid == 0 && m0 != MD_NONE && sS[0].active) finish_step(sS[0], m0, s_tot[0], s_tot[1]);
    if (tid == 32 && m1 != MD_NONE && sS[1].active) finish_step(sS[1], m1, s_tot[2], s_tot[3]);
    __syncthreads();
    if (tid == 0 && !sS[0].active && !sS[1].active) *done_flag = 1;
    for (int i = tid; i < (int)(2 * sizeof(SlotState) / sizeof(double)); i += 256)
        reinterpret_cast<double *>(st)[i] = reinterpret_cast<const double *>(sS)[i];
}

#include "fpsb_loop.inl"

// rows longer than kLongRow: one CTA per row, strided over the row, fixed-tree block reduction.
// Launched before gk_step_kernel of the same step; leaves its norm partials at partials[pbase + row#].
template <bool PAIR>
__global__ void __launch_bounds__(kLongThreads) long_rows_kernel(StepParams P, int use_state, int pbase) {
    __shared__ double s_red[4 * 32];
    __shared__ Coef sC[2];
    const int tid = threadIdx.x;
    const bool act0 = P.io[0].mode != MD_NONE && (!use_state || P.st[0].active);
    const bool act1 = P.io[1].mode != MD_NONE && (!use_state || P.st[1].active);
    if (!act0 && !act1) return;
    if (tid == 0) {
        load_coef(sC[0], P.io[0], &P.st[0], use_state);
        load_coef(sC[1], P.io[1], &P.st[1], use_state);
        if (!act0) { sC[0].mode = MD_NONE; sC[0].rd0 = sC[0].rd1 = sC[0].wr0 = sC[0].wr1 = sC[0].rdself = 0; }
        if (!act1) { sC[1].mode = MD_NONE; sC[1].rd0 = sC[1].rd1 = sC[1].wr0 = sC[1].wr1 = sC[1].rdself = 0; }
    }
    __syncthreads();
    const Coef &C0 = sC[0];
    const Coef &C1 = sC[1];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const int lr = blockIdx.x;
    const int row = P.long_row[lr];
    const int e0 = P.long_rp[lr], e1 = P.long_rp[lr + 1];
    double a[2] = {0.0, 0.0};
    for (int k = e0 + tid; k < e1; k += kLongThreads) {
        const double v = P.long_val[k];
        const int c = P.long_col[k];
        if (PAIR) {
            const double2 x = __ldg(P.gin2 + c);
            a[0] += v * x.x; a[1] += v * x.y;
        } else {
            if (act0) a[0] += v * __ldg(P.io[0].gin + c);
            if (act1) a[1] += v * __ldg(P.io[1].gin + c);
        }
    }
    block_sum<2>(a, s_red);
    if (tid == 0) {
        double a00 = 0.0, a01 = 0.0, a10 = 0.0, a11 = 0.0;
        if (C0.rd0) a00 = P.io[0].a0[row];
        if (C0.rd1) a01 = P.io[0].a1[row];
        if (C1.rd0) a10 = P.io[1].a0[row];
        if (C1.rd1) a11 = P.io[1].a1[row];
        if (PAIR) {
            const double2 old2 = P.self2[row];
            double2 nw = old2;
            if (act0) nw.x = row_epilogue(C0, a[0], old2.x, a00, a01, acc[0], acc[1]);
            if (act1) nw.y = row_epilogue(C1, a[1], old2.y, a10, a11, acc[2], acc[3]);
            P.self2[row] = nw;
        } else {
            if (act0) {
                const double so = C0.rdself ? P.io[0].self[row] : 0.0;
                P.io[0].self[row] = row_epilogue(C0, a[0], so, a00, a01, acc[0], acc[1]);
            }
            if (act1) {
                const double so = C1.rdself ? P.io[1].self[row] : 0.0;
                P.io[1].self[row] = row_epilogue(C1, a[1], so, a10, a11, acc[2], acc[3]);
            }
        }
        if (C0.wr0) P.io[0].a0[row] = a00;
        if (C0.wr1) P.io[0].a1[row] = a01;
        if (C1.wr0) P.io[1].a0[row] = a10;
        if (C1.wr1) P.io[1].a1[row] = a11;
        if (use_state) {
            double *pp = P.partials + (size_t)(pbase + lr) * 4;
            pp[0] = acc[0]; pp[1] = acc[1]; pp[2] = acc[2]; pp[3] = acc[3];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// element-wise fused kernels (initialisation, MINRES / CGLS vector updates, output flush)
// ------------------------------------------------------------------------------------------------
struct EwParams {
    int op, slot, n, pair_slot;      // pair_slot: -1 plain, else column of the interleaved pair
    const double *in0;
    double *v0, *v1, *v2, *v3, *v4;
    double2 *pair;
    double c0;
    SlotState *st;
    double *partials;
    unsigned *counter;
    int *done_flag;
    int use_state;
    double *tot_out;       // row-partitioned runs: local sum left here, finish_kernel follows the all-reduce
};

__global__ void __launch_bounds__(kBlock) ew_kernel(EwParams P) {
    __shared__ double s_red[32];
    __shared__ int s_last;
    SlotState *S = P.st ? &P.st[P.slot] : nullptr;
    const bool is_init = (P.op == EW_INIT_LSQR || P.op == EW_INIT_CRAIG || P.op == EW_MINRES_INIT ||
                          P.op == EW_CGLS_INIT);
    const bool is_out = (P.op == EW_COPY || P.op == EW_CRAIG_FLUSH);
    if (P.use_state && !is_init && !is_out && !S->active) return;
    double acc[1] = {0.0};
    const int stride = gridDim.x * blockDim.x;
    // coefficients
    double alpha = 0, beta = 0, delta = 0, eps_ = 0, gamma = 1, phi = 0, xi = 0, c1 = 0,
           s1 = 0, sv = 0, lambda = 0, beta_c = 0;
    int iter = 0, pend = 0;
    if (S && !is_init) {
        alpha = S->alpha; beta = S->beta; delta = S->delta; eps_ = S->eps_;
        gamma = S->gamma; phi = S->phi; xi = S->xi; c1 = S->c1; s1 = S->s1; sv = S->sv;
        lambda = S->lambda; beta_c = S->beta_c; iter = S->iter; pend = S->pend;
    }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += stride) {
        switch (P.op) {
            case EW_COPY: P.v0[i] = P.c0 * P.in0[i]; break;
            case EW_INIT_LSQR: {
                double b = P.in0[i];
                double *dst = reinterpret_cast<double *>(P.pair + i) + P.pair_slot;
                *dst = b;
                acc[0] += b * b;
            } break;
            case EW_INIT_CRAIG: {
                double b = P.c0 * P.in0[i];
                double *dst = reinterpret_cast<double *>(P.pair + i) + P.pair_slot;
                *dst = b;
                P.v0[i] = 0.0;   // w
                P.v1[i] = 0.0;   // y
                acc[0] += b * b;
            } break;
            case EW_CRAIG_FLUSH: {
                // v0 = x, v1 = w2, pair = vhat ; out v2 = -(x + pending)
                double x = P.v0[i];
                if (pend) {
                    double vp = (reinterpret_cast<const double *>(P.pair + i))[P.pair_slot] * sv;
                    if (lambda > 0) { x = x + (xi * c1) * vp; x = x + (xi * s1) * P.v1[i]; }
                    else x += xi * vp;
                }
                P.v2[i] = -x;
            } break;
            case EW_MINRES_INIT: {
                double b = P.in0[i];
                P.v0[i] = b;     // r1
                P.v1[i] = b;     // r2
                P.v2[i] = 0.0;   // w1
                P.v3[i] = 0.0;   // w2
                P.v4[i] = 0.0;   // x
                acc[0] += b * b;
            } break;
            case EW_MINRES_E1: {
                // in0 = y(pre) ; v0 = r1, v1 = r2, v2 = w1-role, v3 = w2-role ; iter already incremented
                double r2 = P.v1[i];
                double y = P.in0[i] - (alpha / beta) * r2;
                double w;
                if (iter == 1) {
                    w = P.v3[i] + (1.0 / beta) * r2;
                    P.v3[i] = w;
                } else {
                    double w1 = P.v2[i];
                    if (iter >= 3) w1 *= -eps_;
                    w1 -= delta * P.v3[i];
                    w = w1 + (1.0 / beta) * r2;
                    P.v2[i] = w;
                }
                P.v0[i] = r2;
                P.v1[i] = y;
                acc[0] += y * y;
            } break;
            case EW_MINRES_E2: {
                // v2 = the w just written (role resolved by the host), v4 = x
                double w = P.v2[i] * (1.0 / gamma);
                P.v2[i] = w;
                double x = P.v4[i] + phi * w;
                P.v4[i] = x;
                acc[0] += x * x;
            } break;
            case EW_CGLS_INIT: {
                double b = P.in0[i];
                P.v0[i] = b;     // r
                acc[0] += b * b;
            } break;
            case EW_CGLS_EN: {   // r -= alpha q
                double r = P.v0[i] - alpha * P.v1[i];
                P.v0[i] = r;
                acc[0] += r * r;
            } break;
            case EW_CGLS_EM: {   // p = s + beta p
                double p = P.v0[i] + beta_c * P.v1[i];
                P.v1[i] = p;
                acc[0] += p * p;
            } break;
            default: break;
        }
    }
    if (!P.use_state || is_out) return;
    block_sum<1>(acc, s_red);
    if (threadIdx.x == 0) {
        P.partials[blockIdx.x] = acc[0];
        __threadfence();
        unsigned t = atomicAdd(P.counter, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double tot[1] = {0.0};
    for (int i = threadIdx.x; i < (int)gridDim.x; i += kBlock) tot[0] += __ldcg(P.partials + i);
    block_sum<1>(tot, s_red);
    if (threadIdx.x == 0 && P.tot_out != nullptr) {
        P.tot_out[0] = tot[0]; P.tot_out[1] = 0.0; P.tot_out[2] = 0.0; P.tot_out[3] = 0.0;
        *P.counter = 0;
        return;
    }
    if (threadIdx.x == 0) {
        finish_ew(*S, P.op, tot[0]);
        if (!P.st[0].active && !P.st[1].active) *P.done_flag = 1;
        *P.counter = 0;
        __threadfence();
    }
}

// Jacobian value refresh of the tiled operator: one CTA per tile, values land in the tile's block
__global__ void refresh_tiles_kernel(const TileMeta *tiles, const int *tperm0, const int *perm, const double *coo,
                                     unsigned char *tbuf) {
    const TileMeta T = load_tile(tiles, blockIdx.x);
    const int p0 = tperm0[blockIdx.x];
    double *v = reinterpret_cast<double *>(tbuf + T.boff);
    for (int e = threadIdx.x; e < T.elems; e += blockDim.x) {
        const int p = perm[p0 + e];
        v[e] = (p >= 0) ? coo[p] : 0.0;
    }
}

__global__ void gather_vals_kernel(int nnz, const int *perm, const double *coo, double *vx) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) { const int p = perm[i]; vx[i] = (p >= 0) ? coo[p] : 0.0; }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct IterWs {
    DevBuf<double2> Gnm;                 // one allocation: [Gn | Gm] so a single L2 persisting window covers both
    struct View { double2 *p = nullptr; size_t n = 0;
                  void zero(cudaStream_t s) { if (p) FPSB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(double2), s)); } };
    View Gn, Gm;                         // interleaved Golub-Kahan pairs (n-space, m-space)
    DevBuf<double> an[2][2];             // n-space aux per slot (CRAIG x, w2 ; CGLS r, q ; MINRES t)
    DevBuf<double> am[2][5];             // m-space aux per slot
    DevBuf<double> ym;                   // MINRES y / CGLS s
    DevBuf<SlotState> st;
    DevBuf<double> partials;
    DevBuf<unsigned> counter;
    DevBuf<int> done;
    int *h_done = nullptr;               // pinned
    SlotState *h_st = nullptr;           // pinned [2]
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaEvent_t pev[2] = {nullptr, nullptr};   // profile: Krylov loop region
    int64_t prof_launch0 = 0, prof_launch1 = 0;
    bool prof_armed = false;
    int ew_grid = 0;
    size_t partials_stride = 0;          // two partials buffers (deferred recurrences)
    // persistent loop kernel (fpsb_loop.inl)
    DevBuf<double> loop_parts;           // [2][grid][4]
    DevBuf<unsigned long long> gbar;     // grid-barrier arrivals (zeroed before every launch)
    int *h_fin = nullptr;                // pinned [4]: done | phases run | error | -
    int64_t prof_loop_launches = 0;      // chunk launches inside the profiled region
};

static void build_csr_host(int nrows, int ncols, int64_t nnz, const int64_t *ri, const int64_t *cj,
                           std::vector<int> &rp, std::vector<int> &ci, std::vector<int> &perm) {
    rp.assign((size_t)nrows + 1, 0);
    for (int64_t k = 0; k < nnz; ++k) rp[(size_t)ri[k] + 1]++;
    for (int i = 0; i < nrows; ++i) rp[i + 1] += rp[i];
    ci.resize((size_t)nnz);
    perm.resize((size_t)nnz);
    // stable counting sort by column first, then by row => rows hold ascending columns
    std::vector<int> cp((size_t)ncols + 1, 0);
    for (int64_t k = 0; k < nnz; ++k) cp[(size_t)cj[k] + 1]++;
    for (int j = 0; j < ncols; ++j) cp[j + 1] += cp[j];
    std::vector<int> bycol((size_t)nnz);
    for (int64_t k = 0; k < nnz; ++k) bycol[(size_t)cp[(size_t)cj[k]]++] = (int)k;
    std::vector<int> pos(rp.begin(), rp.end() - 1);
    for (int64_t t = 0; t < nnz; ++t) {
        int k = bycol[(size_t)t];
        int q = pos[(size_t)ri[k]]++;
        ci[(size_t)q] = (int)cj[k];
        perm[(size_t)q] = k;
    }
}

constexpr int kLongRow = 96;     // rows longer than this leave the SELL part (a 32-row slice must fit a stage)

// CSR -> tiled SELL-32 (+ CSR of the long rows) and upload
static void upload_sell(Handle *h, CsrDev &M, int nrows, int ncols, const std::vector<int> &rp,
                        const std::vector<int> &ci, const std::vector<int> &perm) {
    M.nrows = nrows; M.ncols = ncols; M.nnz = (int64_t)ci.size();
    M.nseg_tiles = M.nwin_tiles = 0;
    M.nglob_tiles = M.nodd_tiles = M.nns0_tiles = M.nmixed_tiles = 0;
    M.wsegs_host.clear();
    std::vector<int> long_row, long_rp(1, 0), long_col, long_perm;
    std::vector<unsigned char> rowflag((size_t)nrows + 8, 0);
    std::vector<TileMeta> tiles;
    std::vector<int> tperm0;              // first entry of every tile in sperm
    std::vector<std::vector<int>> tile_rows;   // rows per lane of every tile's slices (host only)
    std::vector<int> order, widths;
    int win_cap = 0;
    size_t blk_cap = 128, total_bytes = 0, total_elems = 0;
    auto rlen = [&](int r) { return rp[(size_t)r + 1] - rp[(size_t)r]; };
    for (int r = 0; r < nrows; ++r) {
        if (rlen(r) > kLongRow) {
            long_row.push_back(r);
            rowflag[(size_t)r] = 1;
            for (int p = rp[(size_t)r]; p < rp[(size_t)r + 1]; ++p) { long_col.push_back(ci[(size_t)p]); long_perm.push_back(perm[(size_t)p]); }
            long_rp.push_back((int)long_col.size());
        }
    }
    // Multi-segment windows (stencil operators, BASELINE config C3: a 5-point stencil row touches columns a grid line apart,
    // so the column SPAN of a tile never fits a window while the columns it actually touches are a few short runs): when
    // the span exceeds the capacity the distinct columns of the tile are cut at their (up to kMaxSeg - 1) largest gaps
    // into segments; the window in shared memory is the segments back to back (one bulk copy each) and the 16-bit
    // indices are relative to that concatenation, so the consumers do not know the difference.  Starts are even and all
    // lengths but possibly the last are even (16-byte units of plain vectors); the segments are sorted and may overlap.
    constexpr int kMaxSeg = 4, kMinGap = 32;
    static const bool no_segs = getenv("FPSB_NO_SEGS") != nullptr;
    std::vector<int> ucols, gapidx;
    struct Seg { int start, len; };
    std::vector<Seg> segs;                // of the tile fit_tile looked at last (empty: one segment or no window)
    std::vector<std::array<Seg, kMaxSeg>> tile_segs;
    auto find_segments = [&](int w0, int R) {      // -> total window entries (0: does not fit)
        segs.clear();
        if (no_segs) return 0;
        ucols.clear();
        for (int r = w0; r < w0 + R; ++r) {
            if (rowflag[(size_t)r]) continue;
            for (int p = rp[(size_t)r]; p < rp[(size_t)r + 1]; ++p) ucols.push_back(ci[(size_t)p]);
        }
        std::sort(ucols.begin(), ucols.end());
        ucols.erase(std::unique(ucols.begin(), ucols.end()), ucols.end());
        if (ucols.empty()) return 0;
        // the kMaxSeg - 1 largest gaps (ties: the leftmost), at least kMinGap wide
        gapidx.clear();
        for (size_t i = 0; i + 1 < ucols.size(); ++i) if (ucols[i + 1] - ucols[i] >= kMinGap) gapidx.push_back((int)i);
        if (gapidx.size() > (size_t)(kMaxSeg - 1)) {
            std::stable_sort(gapidx.begin(), gapidx.end(), [&](int a, int b) { return ucols[(size_t)a + 1] - ucols[(size_t)a] > ucols[(size_t)b + 1] - ucols[(size_t)b]; });
            gapidx.resize((size_t)(kMaxSeg - 1));
            std::sort(gapidx.begin(), gapidx.end());
        }
        int total = 0;
        size_t a = 0;
        for (size_t g = 0; g <= gapidx.size(); ++g) {
            const size_t b = g < gapidx.size() ? (size_t)gapidx[g] : ucols.size() - 1;     // last column of this segment
            Seg sg;
            sg.start = ucols[a] & ~1;
            sg.len = ucols[b] - sg.start + 1;
            if ((sg.len & 1) && sg.start + sg.len + 1 <= ncols) ++sg.len;                  // never past the vector's end
            segs.push_back(sg);
            total += sg.len;
            a = b + 1;
        }
        if (total > kSegCapMax || segs.size() < 2) { segs.clear(); return 0; }
        for (size_t g = 0; g + 1 < segs.size(); ++g) if (segs[g].len & 1) { segs.clear(); return 0; }   // (cannot happen: only the last may be odd)
        return total;
    };
    // largest tile starting at row w0 with at most `want` rows whose block + window fit a stage (halving)
    int cnt = 0, c0 = 0, elems = 0;
    auto fit_tile = [&](int w0, int want) {
        int R = std::min(want, nrows - w0);
        for (;;) {
            order.clear();
            int cmin = ncols, cmax = -1;
            for (int r = w0; r < w0 + R; ++r) {
                if (rowflag[(size_t)r]) continue;
                order.push_back(r);
                if (rlen(r) > 0) {      // columns ascend within a row
                    cmin = std::min(cmin, ci[(size_t)rp[(size_t)r]]);
                    cmax = std::max(cmax, ci[(size_t)rp[(size_t)r + 1] - 1]);
                }
            }
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rlen(a) > rlen(b); });
            widths.clear();
            elems = 0;
            for (size_t i = 0; i < order.size(); i += 32) { widths.push_back(rlen(order[i])); elems += widths.back() * 32; }
            c0 = 0; cnt = 0;
            if (cmax >= 0) {
                c0 = cmin & ~1;               // 16-byte aligned start for vectors of doubles
                cnt = cmax - c0 + 1;
                // even length: plain (8-byte) vectors are then bulk-copied in whole 16-byte units; an odd window would
                // send the tile down the group-staged path of the one-column products.  Never past the vector's end.
                if ((cnt & 1) && c0 + cnt + 1 <= ncols) ++cnt;
                segs.clear();
                if (cnt > kWinCapMax) {
                    cnt = find_segments(w0, R);
                    if (cnt > 0) c0 = segs[0].start;
                }
            } else segs.clear();
            if ((size_t)tile_block_bytes(elems, (int)widths.size(), cnt) + (size_t)cnt * 16 <= (size_t)(segs.empty() ? kStageBytesMax : kSegStageBytesMax)) break;
            if (R > 32) { R = std::max(32, ((R / 2) + 31) & ~31); continue; }
            cnt = 0;     // a single slice (at most kLongRow wide, 36 KB): drop the window
            segs.clear();
            break;
        }
        return R;
    };
    // Tile boundaries.  The persistent CTAs take tiles b, b + grid, ...: a tile count that is not a multiple
    // of the grid leaves most SMs idle for one tile at the end of every pass (3.7 % at the headline size),
    // so when there are enough tiles the rows are cut into a multiple of the grid of (slightly smaller) tiles
    std::vector<int> cuts;                 // desired tile starts ; a tile that does not fit is split further
    {
        int ntl = 0;
        for (int w0 = 0; w0 < nrows; ++ntl) w0 += fit_tile(w0, kTileRows);
        const int G = std::max(1, h->num_sms);
        static const bool no_cuts = getenv("FPSB_NO_CUTS") != nullptr;
        if (ntl >= 4 * G && !no_cuts) {
            const int64_t target = (int64_t)((ntl + G - 1) / G) * G;
            for (int64_t i = 0; i < target; ++i) cuts.push_back((int)((i * (int64_t)nrows) / target));
        }
    }
    size_t icut = 0;
    for (int w0 = 0; w0 < nrows;) {
        int want = kTileRows;
        if (!cuts.empty()) {
            while (icut < cuts.size() && cuts[icut] <= w0) ++icut;
            const int next = icut < cuts.size() ? cuts[icut] : nrows;
            want = std::min(kTileRows, next - w0);
        }
        const int R = fit_tile(w0, want);
        TileMeta T{};
        T.boff = (long long)total_bytes;
        T.row0 = w0; T.nrows = R;
        T.cmin = cnt > 0 ? c0 : 0; T.ccnt = cnt;
        T.elems = elems;
        T.ns = (int)widths.size();
        T.nsell = (int)order.size();
        for (int i = 0; i < kTileSlices; ++i) T.width[i] = (unsigned char)(i < T.ns ? widths[(size_t)i] : 0);
        const size_t bytes = (((size_t)tile_block_bytes(elems, T.ns, cnt)) + 127) & ~(size_t)127;    // blocks start 128-byte aligned
        win_cap = std::max(win_cap, cnt);
        blk_cap = std::max(blk_cap, bytes);
        {
            std::array<Seg, kMaxSeg> sg{};
            if (!segs.empty()) { for (size_t g = 0; g < segs.size(); ++g) sg[g] = segs[g]; ++M.nseg_tiles; }
            else if (cnt > 0) sg[0] = Seg{c0, cnt};
            if (cnt > 0) ++M.nwin_tiles; else ++M.nglob_tiles;
            if (cnt & 1) ++M.nodd_tiles;
            if (T.ns == 0) ++M.nns0_tiles;
            if (T.nsell < T.nrows) ++M.nmixed_tiles;
            tile_segs.push_back(sg);
        }
        tperm0.push_back((int)total_elems);
        total_bytes += bytes;
        total_elems += (size_t)elems;
        std::vector<int> lanes;
        for (size_t i = 0; i < order.size(); i += 32)
            for (size_t l = 0; l < 32; ++l) lanes.push_back((i + l < order.size()) ? order[i + l] : -1);
        tile_rows.push_back(std::move(lanes));
        tiles.push_back(T);
        w0 += R;
    }
    // Order of the entries inside every row: the gather of step j reads, for the 8 lanes of a
    // quarter warp, 8 window entries of 16 bytes — conflict-free iff their columns differ mod 8.
    // Greedy: at every step each lane takes, among its remaining entries, the one whose bank group
    // is least used by the lanes of its quarter so far (ties: smallest column).  `eorder` holds, per
    // lane, the permutation of the row's CSR entries.
    // fill the blocks: [values (refreshed on the device) | indices | lane -> row map]
    std::vector<unsigned char> tbuf(total_bytes + 128, 0);
    std::vector<int> sperm(total_elems + 8, -1);
    for (size_t ti = 0; ti < tiles.size(); ++ti) {
        const TileMeta &T = tiles[ti];
        const bool win = T.ccnt > 0;
        const std::array<Seg, kMaxSeg> &sg = tile_segs[ti];
        int sg_off[kMaxSeg];
        { int o = 0; for (int g = 0; g < kMaxSeg; ++g) { sg_off[g] = o; o += sg[g].len; } }
        // window-relative index of column c: its position in the concatenated segments (the last segment that starts at or before c)
        auto wrel = [&](int c) {
            if (!win) return c;
            int g = kMaxSeg - 1;
            while (g > 0 && (sg[g].len == 0 || sg[g].start > c)) --g;
            return sg_off[g] + (c - sg[g].start);
        };
        int *cols = reinterpret_cast<int *>(tbuf.data() + T.boff + (size_t)T.elems * 8);
        unsigned short *cols16 = reinterpret_cast<unsigned short *>(tbuf.data() + T.boff + (size_t)T.elems * 8);
        unsigned char *rmap = tbuf.data() + T.boff + (size_t)T.elems * (win ? 10 : 12);
        int *tp = sperm.data() + tperm0[ti];
        int off = 0;
        std::vector<int> eorder, used;
        for (int sl = 0; sl < T.ns; ++sl) {
            const int width = T.width[sl], npair = width / 2;
            eorder.assign((size_t)32 * std::max(width, 1), -1);
            used.assign((size_t)32 * std::max(width, 1), 0);
            for (int q0 = 0; q0 < 32; q0 += 8) {
                for (int j = 0; j < width; ++j) {
                    int cnt8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                    for (int l = q0; l < q0 + 8; ++l) {
                        const int r = tile_rows[ti][(size_t)sl * 32 + l];
                        if (r < 0) continue;
                        const int base = rp[(size_t)r], len = rp[(size_t)r + 1] - base;
                        if (j >= len) continue;
                        int best = -1, bestc = 1 << 30;
                        for (int e = 0; e < len; ++e) {
                            if (used[(size_t)l * width + e]) continue;
                            const int bg = win ? (wrel(ci[(size_t)(base + e)]) & 7) : 0;
                            if (cnt8[bg] < bestc) { bestc = cnt8[bg]; best = e; }
                        }
                        used[(size_t)l * width + best] = 1;
                        eorder[(size_t)l * width + j] = best;
                        if (win) cnt8[wrel(ci[(size_t)(base + best)]) & 7]++;
                    }
                }
            }
            for (int l = 0; l < 32; ++l) {
                const int r = tile_rows[ti][(size_t)sl * 32 + l];
                rmap[sl * 32 + l] = (unsigned char)(r >= 0 ? r - T.row0 : 0);      // lanes >= nsell are padding (never stored)
                int len = 0, base = 0;
                if (r >= 0) { base = rp[(size_t)r]; len = rp[(size_t)r + 1] - base; }
                for (int j = 0; j < width; ++j) {
                    // pair rows: entries 2p, 2p+1 of a lane are adjacent; an odd last entry is a plain row
                    const int q = (j < 2 * npair) ? off + ((j >> 1) * 32 + l) * 2 + (j & 1) : off + npair * 64 + l;
                    int cval = 0;
                    if (j < len) {
                        const int e = eorder[(size_t)l * width + j];
                        cval = wrel(ci[(size_t)(base + e)]); tp[q] = perm[(size_t)(base + e)];
                    } else tp[q] = -1;                       // padding: value 0, valid column
                    if (win) cols16[q] = (unsigned short)cval; else cols[q] = cval;
                }
            }
            off += width * 32;
        }
    }
    M.padded = (int64_t)total_elems;
    M.nlong = (int)long_row.size();
    M.ntiles = (int)tiles.size();
    M.win_cap = (win_cap + 7) & ~7;
    M.blk_cap = (int)((blk_cap + 127) & ~(size_t)127);
    M.stage_bytes = (int)((((size_t)M.blk_cap + (size_t)M.win_cap * 16) + 127) & ~(size_t)127);
    M.nstage = std::max(2, std::min(kMaxStages, kRingBudget / M.stage_bytes));
    M.tbuf.from(tbuf, h->stream);
    M.sperm.from(sperm, h->stream);
    M.tperm0.from(tperm0, h->stream);
    M.tiles.alloc((tiles.size() + 1) * sizeof(TileMeta));
    if (!tiles.empty()) FPSB_CUDA(cudaMemcpyAsync(M.tiles.p, tiles.data(), tiles.size() * sizeof(TileMeta), cudaMemcpyHostToDevice, h->stream));
    M.rowflag.from(rowflag, h->stream);
    if (M.nseg_tiles > 0) {
        std::vector<int> ws(tiles.size() * 2 * kMaxSeg + 8, 0);
        for (size_t ti = 0; ti < tiles.size(); ++ti) {
            int o = 0;
            for (int g = 0; g < kMaxSeg; ++g) {
                ws[(ti * kMaxSeg + g) * 2] = tile_segs[ti][g].start;
                ws[(ti * kMaxSeg + g) * 2 + 1] = o | (tile_segs[ti][g].len << 16);
                o += tile_segs[ti][g].len;
            }
        }
        M.wsegs.from(ws, h->stream);
        M.wsegs_host.swap(ws);
    }
    M.long_row.from(long_row, h->stream);
    M.long_rp.from(long_rp, h->stream);
    M.long_col.from(long_col, h->stream);
    M.long_perm.from(long_perm, h->stream);
    M.long_val.alloc(long_col.size() + 8);
    M.long_val.zero(h->stream);
    M.grid = nrows > 0 ? std::max(1, std::min(h->num_sms, M.ntiles)) : 0;
    FPSB_CUDA(cudaStreamSynchronize(h->stream));     // the host vectors above die with this scope
}

// one step of the fused operator: the long rows first (their norm partials are picked up by the
// last CTA of the main kernel), then the persistent tile kernel
static void launch_step(Handle *h, const CsrDev &M, const StepParams &P, bool pair, int use_state) {
    if (M.grid == 0) return;
    if (M.nlong > 0) {
        if (pair) long_rows_kernel<true><<<M.nlong, kLongThreads, 0, h->stream>>>(P, use_state, M.grid);
        else long_rows_kernel<false><<<M.nlong, kLongThreads, 0, h->stream>>>(P, use_state, M.grid);
        h->launches += 1;
    }
    const size_t smem = (size_t)M.nstage * (size_t)M.stage_bytes;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)M.grid); cfg.blockDim = dim3(kStepThreads);
    cfg.dynamicSmemBytes = smem; cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    static const bool no_pdl = getenv("FPSB_NO_PDL") != nullptr;
    cfg.attrs = attr; cfg.numAttrs = no_pdl ? 0 : 1;
    if (pair) FPSB_CUDA(cudaLaunchKernelEx(&cfg, gk_step_kernel<true>, P, use_state));
    else FPSB_CUDA(cudaLaunchKernelEx(&cfg, gk_step_kernel<false>, P, use_state));
    h->launches += 1;
}

// debug builds (-DFPSB_XCHG_TIMERS): read and reset the exchange segment timers, [2][16]
void xchg_timers(unsigned long long *out) {
    cudaMemcpyFromSymbol(out, g_xchg_t, sizeof(unsigned long long) * 32);
    unsigned long long z[32] = {};
    cudaMemcpyToSymbol(g_xchg_t, z, sizeof(z));
}

// debug builds (-DFPSB_LOOP_TIMERS): the stamps of the last persistent-loop launch, [64][160][8]
void loop_timers(unsigned long long *out) {
#ifdef FPSB_LOOP_TIMERS
    cudaMemcpyFromSymbol(out, g_loop_t, sizeof(unsigned long long) * 64 * 160 * 16);
    cudaMemcpyFromSymbol(out + 64 * 160 * 16, g_loop_seg, sizeof(unsigned long long) * 160 * 2 * kGroups * 8);
    unsigned long long *z = new unsigned long long[160 * 2 * kGroups * 8]();
    cudaMemcpyToSymbol(g_loop_seg, z, sizeof(unsigned long long) * 160 * 2 * kGroups * 8);
    delete[] z;
#else
    (void)out;
#endif
}

void phase_timers(unsigned long long *out, int reset) {
#ifdef FPSB_PHASE_TIMERS
    if (out) cudaMemcpyFromSymbol(out, g_phase_cycles, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z)); }
#else
    if (out) for (int i = 0; i < 16; ++i) out[i] = 0;
    (void)reset;
#endif
}

void csr_build(Handle *h) {
    const int m = (int)h->ncon, n = (int)h->nvar;
    {
        int dev = 0, sms = 148;
        FPSB_CUDA(cudaGetDevice(&dev));
        FPSB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        h->num_sms = sms;
        FPSB_CUDA(cudaFuncSetAttribute(gk_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingBudget + 8 * 1024));
        FPSB_CUDA(cudaFuncSetAttribute(gk_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingBudget + 8 * 1024));
        FPSB_CUDA(cudaFuncSetAttribute(gk_loop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingBudget + 8 * 1024));
        FPSB_CUDA(cudaFuncSetAttribute(gk_loop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingBudget + 8 * 1024));
    }
    std::vector<int> rp, ci, perm;
    build_csr_host(m, n, h->nnzj, h->jrow.data(), h->jcol.data(), rp, ci, perm);
    upload_sell(h, h->A, m, n, rp, ci, perm);
    build_csr_host(n, m, h->nnzj, h->jcol.data(), h->jrow.data(), rp, ci, perm);
    upload_sell(h, h->At, n, m, rp, ci, perm);
    h->coo_vals.alloc((size_t)h->nnzj + 8);
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
}

void csr_refresh_values(Handle *h) {
    for (CsrDev *M : {&h->A, &h->At}) {
        if (M->ntiles > 0) {
            refresh_tiles_kernel<<<M->ntiles, 256, 0, h->stream>>>(reinterpret_cast<const TileMeta *>(M->tiles.p), M->tperm0.p,
                                                                   M->sperm.p, h->coo_vals.p, M->tbuf.p);
            h->launches += 1;
        }
        const int nl = (int)(M->long_col.n > 8 ? M->long_col.n - 8 : 0);
        if (M->nlong > 0 && nl > 0) {
            gather_vals_kernel<<<(nl + 255) / 256, 256, 0, h->stream>>>(nl, M->long_perm.p, h->coo_vals.p, M->long_val.p);
            h->launches += 1;
        }
    }
    FPSB_CUDA(cudaGetLastError());
}

static void fill_csr(StepParams &P, const CsrDev &M) {
    P.tiles = reinterpret_cast<const TileMeta *>(M.tiles.p); P.ntiles = M.ntiles; P.win_cap = M.win_cap; P.blk_cap = M.blk_cap;
    P.tbuf = M.tbuf.p;
    P.stage_bytes = M.stage_bytes; P.nstage = M.nstage; P.nlong = M.nlong;
    {
        static const int env_inflight = [] { const char *e = getenv("FPSB_INFLIGHT"); return e ? atoi(e) : 0; }();
        P.inflight = env_inflight > 0 ? env_inflight : 2;
        if (P.inflight > M.nstage - 1) P.inflight = std::max(1, M.nstage - 1);      // a tile must not wait for the stage it is about to refill
    }
    P.rowflag = (M.nlong > 0 || M.has_raw_rows) ? M.rowflag.p : nullptr;
    P.wsegs = M.nseg_tiles > 0 ? reinterpret_cast<const int2 *>(M.wsegs.p) : nullptr;
    P.long_row = M.long_row.p; P.long_rp = M.long_rp.p; P.long_col = M.long_col.p; P.long_val = M.long_val.p;
    P.nrows = M.nrows;
}

// y = Op x for 1 or 2 plain columns (columns contiguous in memory)
void spmv_plain(Handle *h, bool transpose, const double *x, double *y, int ncols_rhs) {
    const CsrDev &M = transpose ? h->At : h->A;
    if (M.nrows == 0 || M.grid == 0) return;
    StepParams P{};
    fill_csr(P, M);
    for (int s = 0; s < 2; ++s) {
        P.io[s].mode = (s < ncols_rhs) ? MD_PLAIN : MD_NONE;
        P.io[s].gin = x + (size_t)s * M.ncols;
        P.io[s].self = y + (size_t)s * M.nrows;
        P.io[s].a0 = nullptr;
        P.io[s].c0 = 1.0; P.io[s].c1 = 0.0;
    }
    launch_step(h, M, P, false, 0);
    FPSB_CUDA(cudaGetLastError());
}

void iter_setup(Handle *h) {
    if (h->iter) return;
    IterWs *W = new IterWs();
    h->iter = W;
    const size_t n = (size_t)h->nvar, m = (size_t)h->ncon;
    {
        const size_t gn = (n + 4 + 7) & ~(size_t)7, gm = (m + 4 + 7) & ~(size_t)7;
        W->Gnm.alloc(gn + gm);
        W->Gn.p = W->Gnm.p; W->Gn.n = gn;
        W->Gm.p = W->Gnm.p + gn; W->Gm.n = gm;
        // keep the gathered vectors resident in L2 across the 240 MB matrix stream of every iteration
        int dev = 0, maxp = 0, maxw = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&maxp, cudaDevAttrMaxPersistingL2CacheSize, dev);
        cudaDeviceGetAttribute(&maxw, cudaDevAttrMaxAccessPolicyWindowSize, dev);
        const size_t bytes = (gn + gm) * sizeof(double2);
        if (maxp > 0 && maxw > 0) {
            const size_t want = std::min(bytes, (size_t)maxp);
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
            cudaStreamAttrValue attr;
            memset(&attr, 0, sizeof(attr));
            attr.accessPolicyWindow.base_ptr = (void *)W->Gnm.p;
            attr.accessPolicyWindow.num_bytes = std::min(bytes, (size_t)maxw);
            attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)want / (double)std::max<size_t>(bytes, 1));
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            if (cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
        }
        cudaGetLastError();
    }
    for (int s = 0; s < 2; ++s) {
        for (int k = 0; k < 2; ++k) W->an[s][k].alloc(n + 4);
        for (int k = 0; k < 5; ++k) W->am[s][k].alloc(m + 4);
    }
    W->ym.alloc(m + 4);
    W->st.alloc(4);          // two state buffers (deferred recurrences ping-pong between them)
    int maxblk = std::max(h->A.grid + h->A.nlong, h->At.grid + h->At.nlong);
    W->ew_grid = 148 * 4;
    W->partials_stride = (size_t)std::max(maxblk, W->ew_grid) * 4 + 16;
    W->partials.alloc(2 * W->partials_stride);
    W->counter.alloc(4);
    W->done.alloc(4);
    W->counter.zero(h->stream);
    W->done.zero(h->stream);
    W->loop_parts.alloc((size_t)2 * 4 * (size_t)std::max(h->num_sms, 1) + 16);
    W->gbar.alloc(4);       // grid-barrier arrivals | exchanges | scatter-complete | boundary-slice arrivals (fpsb_loop.inl)
    W->gbar.zero(h->stream);
    FPSB_CUDA(cudaMallocHost((void **)&W->h_fin, 4 * sizeof(int)));
    FPSB_CUDA(cudaMallocHost((void **)&W->h_done, 2 * sizeof(int)));
    FPSB_CUDA(cudaMallocHost((void **)&W->h_st, 2 * sizeof(SlotState)));
    FPSB_CUDA(cudaEventCreateWithFlags(&W->ev[0], cudaEventDisableTiming));
    FPSB_CUDA(cudaEventCreateWithFlags(&W->ev[1], cudaEventDisableTiming));
    FPSB_CUDA(cudaEventCreate(&W->pev[0]));
    FPSB_CUDA(cudaEventCreate(&W->pev[1]));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
}

void iter_free(Handle *h) {
    if (!h->iter) return;
    IterWs *W = h->iter;
    if (W->h_done) cudaFreeHost(W->h_done);
    if (W->h_fin) cudaFreeHost(W->h_fin);
    if (W->h_st) cudaFreeHost(W->h_st);
    if (W->ev[0]) cudaEventDestroy(W->ev[0]);
    if (W->ev[1]) cudaEventDestroy(W->ev[1]);
    if (W->pev[0]) cudaEventDestroy(W->pev[0]);
    if (W->pev[1]) cudaEventDestroy(W->pev[1]);
    delete W;
    h->iter = nullptr;
    // the gathered vectors of this handle were marked persisting in L2 (iter_setup): give the lines back
    if (cudaCtxResetPersistingL2Cache() != cudaSuccess) cudaGetLastError();
}

// ---- slot configuration (host fills a SlotState, uploaded before the solve) ---------------------
static SlotState make_lsqr(double lambda, double atol, double rtol, int64_t itmax, int64_t m_op, int64_t n_op) {
    SlotState S;
    memset(&S, 0, sizeof(S));
    S.algo = ALGO_LSQR;
    S.lambda = lambda; S.atol = atol; S.rtol = rtol;
    S.axtol = kSqrtEps; S.btol = kSqrtEps; S.etol = kSqrtEps; S.ctol = kSqrtEps;   // conlim = 1/sqrt(eps)
    int64_t im = itmax == 0 ? m_op + n_op : itmax;
    S.itmax = (int)std::min<int64_t>(im, 2000000000);
    S.active = 1;
    S.mscale = 1.0;
    return S;
}
static SlotState make_craig(double delta, double atol, double rtol, double btol, double conlim,
                            int64_t itmax, int64_t m_op, int64_t n_op) {
    SlotState S;
    memset(&S, 0, sizeof(S));
    S.algo = ALGO_CRAIG;
    S.sqd = delta != 0.0;
    S.lambda = S.sqd ? 1.0 : 0.0;
    S.mscale = S.sqd ? 1.0 / delta : 1.0;
    S.atol = atol; S.rtol = rtol; S.btol = btol;
    S.ctol = conlim > 0 ? 1.0 / conlim : 0.0;
    int64_t im = itmax == 0 ? m_op + n_op : itmax;
    S.itmax = (int)std::min<int64_t>(im, 2000000000);
    S.active = 1;
    return S;
}
// make_minres / make_cgls also run on the device: the batched extras kernel (fpsb_extras_batch.inl) sets up every
// instance's state from its own delta with them
static __host__ __device__ SlotState make_minres(double lambda, double atol, double rtol, double etol, double conlim,
                                                 int64_t itmax, int64_t n_op) {
    SlotState S;
    memset(&S, 0, sizeof(S));
    S.algo = ALGO_MINRES;
    S.lambda = lambda; S.atol = atol; S.rtol = rtol; S.etol = etol;
    S.ctol = conlim > 0 ? 1.0 / conlim : 0.0;
    int64_t im = itmax == 0 ? 2 * n_op : itmax;
    S.itmax = (int)(im < 2000000000 ? im : 2000000000);
    S.active = 1;
    S.mscale = 1.0;
    return S;
}
static __host__ __device__ SlotState make_cgls(double lambda, double atol, double rtol, int64_t itmax, int64_t m_op,
                                               int64_t n_op) {
    SlotState S;
    memset(&S, 0, sizeof(S));
    S.algo = ALGO_CGLS;
    S.lambda = lambda; S.atol = atol; S.rtol = rtol;
    int64_t im = itmax == 0 ? m_op + n_op : itmax;
    S.itmax = (int)(im < 2000000000 ? im : 2000000000);
    S.active = 1;
    S.mscale = 1.0;
    return S;
}
static SlotState make_none() {
    SlotState S;
    memset(&S, 0, sizeof(S));
    S.algo = ALGO_NONE;
    S.active = 0;
    S.solved = 1;
    return S;
}

static __host__ __device__ void stats_from(const SlotState &S, fpsb_krylov_stats &o) {
    o.niter = S.iter; o.solved = S.solved; o.inconsistent = S.inconsistent; o.status = S.status;
    o.pad_ = 0;
    o.rnorm = S.rNorm; o.arnorm = S.ArNorm; o.anorm = S.Anorm; o.acond = S.Acond; o.xnorm = S.xNorm;
}

struct Engine {
    Handle *h;
    IterWs *W;
    StepParams base_m, base_n;   // M: rows of A (m-space rows), N: rows of A' (n-space rows)
    double *tot_out = nullptr;   // non-null: row-partitioned run (see fpsb_dist.inl)
    const PeerTail *ptail = nullptr;          // set around a step whose last CTA does the peer exchange itself
    unsigned long long pt_sig = 0;
    int pt_par = 0;
    Engine(Handle *hh) : h(hh), W(hh->iter) {
        memset(h->loop_info, 0, sizeof(h->loop_info));      // run_loop fills it in if this solve runs the persistent loop
        memset(&base_m, 0, sizeof(base_m));
        memset(&base_n, 0, sizeof(base_n));
        fill_csr(base_m, h->A);
        fill_csr(base_n, h->At);
        for (StepParams *P : {&base_m, &base_n}) {
            P->st = W->st.p; P->partials = W->partials.p; P->counter = W->counter.p; P->done_flag = W->done.p;
        }
        base_m.gin2 = W->Gn.p; base_m.self2 = W->Gm.p;
        base_n.gin2 = W->Gm.p; base_n.self2 = W->Gn.p;
    }
    // deferred recurrences (see StepParams): host-side bookkeeping
    int64_t max_it = 0;          // largest itmax of the two slots (bounds the host loop)
    bool defer = false;          // set by the LSQR / CRAIG drivers around their loops
    int cur = 0;                 // state buffer holding the current slot states
    int pbuf = 0;                // partials buffer the next deferred launch writes
    struct Pending { bool valid = false; int m0 = 0, m1 = 0, nparts = 0, buf = 0; } pend;
    SlotState *st_cur() const { return W->st.p + 2 * cur; }
    double *partials_buf(int b) const { return W->partials.p + (size_t)b * W->partials_stride; }
    void flush_pending() {
        if (!pend.valid) return;
        flush_finish_kernel<<<1, 256, 0, h->stream>>>(st_cur(), partials_buf(pend.buf), pend.nparts, pend.m0, pend.m1, W->done.p);
        h->launches += 1;
        pend.valid = false;
    }
    void begin(const SlotState &s0, const SlotState &s1) {
        SlotState hs[2] = {s0, s1};
        memcpy(W->h_st, hs, sizeof(hs));
        cur = 0; pbuf = 0; pend.valid = false; defer = false;
        max_it = std::max<int64_t>(s0.algo != ALGO_NONE ? s0.itmax : 0, s1.algo != ALGO_NONE ? s1.itmax : 0);
        FPSB_CUDA(cudaMemcpyAsync(W->st.p, W->h_st, sizeof(hs), cudaMemcpyHostToDevice, h->stream));
        FPSB_CUDA(cudaMemsetAsync(W->done.p, 0, 4 * sizeof(int), h->stream));
        W->counter.zero(h->stream);
        loop_phases_pending = false;
    }
    void step(bool mspace, bool pair, const SlotIO &io0, const SlotIO &io1) {
        StepParams P = mspace ? base_m : base_n;
        P.io[0] = io0; P.io[1] = io1;
        P.tot_out = tot_out;
        P.ptail = ptail; P.pt_sig = pt_sig; P.pt_par = pt_par;
        const CsrDev &M = mspace ? h->A : h->At;
        if (M.grid == 0) return;
        if (defer && tot_out == nullptr && M.nlong == 0) {
            P.st = st_cur();
            P.st_out = W->st.p + 2 * (cur ^ 1);
            P.partials = partials_buf(pbuf);
            if (pend.valid) { P.pend_partials = partials_buf(pend.buf); P.pend_nparts = pend.nparts; P.pend_m0 = pend.m0; P.pend_m1 = pend.m1; }
            launch_step(h, M, P, pair, 1);
            cur ^= 1;
            pend.valid = true; pend.m0 = io0.mode; pend.m1 = io1.mode; pend.nparts = M.grid; pend.buf = pbuf;
            pbuf ^= 1;
            return;
        }
        flush_pending();
        P.st = st_cur();
        P.partials = partials_buf(0);
        launch_step(h, M, P, pair, 1);
    }
    void ew(int op, int slot, int n, const double *in0, double *v0, double *v1, double *v2, double *v3,
            double *v4, double2 *pair, int pair_slot, double c0, int use_state = 1) {
        if (n == 0 && !(use_state)) return;
        if (use_state) flush_pending();
        EwParams P{};
        P.op = op; P.slot = slot; P.n = n; P.pair_slot = pair_slot; P.in0 = in0;
        P.v0 = v0; P.v1 = v1; P.v2 = v2; P.v3 = v3; P.v4 = v4; P.pair = pair; P.c0 = c0;
        P.st = st_cur(); P.partials = partials_buf(0); P.counter = W->counter.p; P.done_flag = W->done.p;
        P.use_state = use_state;
        P.tot_out = tot_out;
        int grid = std::max(1, std::min(W->ew_grid, (n + kBlock - 1) / kBlock));
        ew_kernel<<<grid, kBlock, 0, h->stream>>>(P);
        h->launches += 1;
    }
    // run `body(k)` (k = 1, 2, ...) until the device reports every slot stopped
    template <class F>
    void loop(F body, int chunk, int its_per_body = 1) {
        int k = 0, pending = 0, slot = 0;
        // every method stops at its itmax at the latest; the cap only guards against a step that cannot
        // run its recurrences at all (degenerate operator) — it must never be what ends a healthy solve
        int64_t hard_cap = max_it / its_per_body + 4 * (int64_t)chunk + 8;
#if FPSB_EXP > 0
        if (const char *e = getenv("FPSB_MAXLOOP")) hard_cap = atoll(e);     // timing experiments only
#endif
        bool done = false;
        while (!done && k < hard_cap) {
            for (int c = 0; c < chunk; ++c) body(++k);
            FPSB_CUDA(cudaMemcpyAsync(&W->h_done[slot], W->done.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
            FPSB_CUDA(cudaEventRecord(W->ev[slot], h->stream));
            pending++;
            if (pending == 2) {
                int prev = slot ^ 1;
                FPSB_CUDA(cudaEventSynchronize(W->ev[prev]));
                if (W->h_done[prev] != 0) done = true;
                pending--;
            }
            slot ^= 1;
        }
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
        FPSB_CUDA(cudaGetLastError());
        if (W->h_done[0] < 0 || W->h_done[1] < 0) {
            set_error("TMA/mbarrier wait timed out inside gk_step_kernel");
            throw CudaFail{FPSB_ECUDA};
        }
    }
    // ---- persistent loop kernel (fpsb_loop.inl): a whole chunk of Krylov iterations per launch ----
    bool loop_phases_pending = false;
    const DistLoop *loop_dx = nullptr;       // row-partitioned run: device copy of the exchange description (fpsb_dist.inl)
    double2 *loop_raw = nullptr;             // ... and where the raw sums of the halo / boundary rows go
    static int env_int(const char *name, int dflt) { const char *e = getenv(name); return (e && *e) ? atoi(e) : dflt; }
    // one ring geometry for both operators; false when the persistent kernel cannot run this handle
    bool loop_geometry(int &blk_cap, int &win_cap, int &stage_bytes, int &nstage, int &grid) const {
        static const int mode = env_int("FPSB_LOOP", 2);
        if (mode == 0 || (tot_out != nullptr && loop_dx == nullptr)) return false;
        const CsrDev &A = h->A, &At = h->At;
        if (A.nlong > 0 || At.nlong > 0 || A.ntiles == 0 || At.ntiles == 0) return false;
        blk_cap = std::max(A.blk_cap, At.blk_cap);
        win_cap = std::max(A.win_cap, At.win_cap);
        stage_bytes = (int)((((size_t)blk_cap + (size_t)win_cap * 16) + 127) & ~(size_t)127);
        nstage = std::min(kMaxStages, kRingBudget / stage_bytes);
        if (nstage < 2) return false;
        { static const int cap = env_int("FPSB_LOOP_NSTAGE", 0); if (cap >= 2) nstage = std::min(nstage, cap); }
        if (!getenv("FPSB_LOOP_ODD")) nstage &= ~1;              // even: every stage is always served by the same producer warp (fpsb_loop.inl)
        grid = std::max(1, std::min(std::min(h->num_sms, kLoopMaxGrid), std::min(A.ntiles, At.ntiles)));
        return true;
    }
    bool can_persist() const { int a, b, c, d, e; return loop_geometry(a, b, c, d, e); }
    // LSQR / CRAIG loop: phases alternate n-space (rows of A') and m-space (rows of A), n-space first
    void run_loop(const SlotIO &n0, const SlotIO &n1, const SlotIO &m0, const SlotIO &m1) {
        flush_pending();
        defer = false;
        static const int mode = env_int("FPSB_LOOP", 2);
        static const int chunk_it = std::max(1, env_int("FPSB_LOOP_CHUNK", 24));
        LoopParams L;
        memset(&L, 0, sizeof(L));
        int blk_cap, win_cap, stage_bytes, nstage, grid;
        if (!loop_geometry(blk_cap, win_cap, stage_bytes, nstage, grid)) { set_error("persistent loop: unsupported operator"); throw CudaFail{FPSB_ESTATE}; }
        L.op[0] = base_n; L.op[0].io[0] = n0; L.op[0].io[1] = n1;
        L.op[1] = base_m; L.op[1].io[0] = m0; L.op[1].io[1] = m1;
        for (int i = 0; i < 2; ++i) {
            L.op[i].blk_cap = blk_cap; L.op[i].win_cap = win_cap; L.op[i].stage_bytes = stage_bytes; L.op[i].nstage = nstage;
            L.op[i].inflight = std::min(L.op[i].inflight, nstage);
            L.op[i].st = st_cur();
        }
        L.dx = loop_dx;
        if (loop_dx != nullptr) L.op[0].raw_out = loop_raw;
        L.first = 0;
        L.nphase = 2 * chunk_it;
        L.nspec = std::max(0, std::min(env_int("FPSB_LOOP_NSPEC", kGroups), nstage - 1));
        L.early = mode >= 2 ? 1 : 0;
        // (FPSB_DIST_EARLY=0: row-partitioned runs without the early row sums, for A/B timing)
        if (loop_dx != nullptr && env_int("FPSB_DIST_EARLY", 1) == 0) L.early = 0;
        L.st = st_cur();
        L.parts = W->loop_parts.p;
        L.gbar = W->gbar.p;
        L.done_flag = W->done.p;
        {
            const int64_t info[8] = {1, L.early, nstage, grid, stage_bytes, std::max(L.op[0].inflight, L.op[1].inflight),
                                     L.nspec, chunk_it};
            memcpy(h->loop_info, info, sizeof(info));
        }
        const size_t smem = (size_t)nstage * (size_t)stage_bytes;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kStepThreads);
        cfg.dynamicSmemBytes = smem; cfg.stream = h->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        loop([&](int) {
            FPSB_CUDA(cudaMemsetAsync(W->gbar.p, 0, 4 * sizeof(unsigned long long), h->stream));      // arrivals | exchanges | ...
            if (loop_dx != nullptr) FPSB_CUDA(cudaLaunchKernelEx(&cfg, gk_loop_kernel<true>, L));
            else FPSB_CUDA(cudaLaunchKernelEx(&cfg, gk_loop_kernel<false>, L));
            h->launches += 1;
            W->prof_loop_launches += 1;
        }, 1, chunk_it);
        loop_phases_pending = true;
    }
    // CUDA-event bracket around the Krylov loop (first step kernel .. last chunk), for the roofline
    void mark_begin() {
        FPSB_CUDA(cudaEventRecord(W->pev[0], h->stream));
        W->prof_launch0 = h->launches;
        W->prof_loop_launches = 0;
        W->prof_armed = true;
    }
    void mark_end() {
        flush_pending();
        defer = false;
        FPSB_CUDA(cudaEventRecord(W->pev[1], h->stream));
        W->prof_launch1 = h->launches;
    }
    void fetch(fpsb_krylov_stats *st) {
        flush_pending();
        defer = false;
        FPSB_CUDA(cudaMemcpyAsync(W->h_st, st_cur(), 2 * sizeof(SlotState), cudaMemcpyDeviceToHost, h->stream));
        FPSB_CUDA(cudaMemcpyAsync(W->h_fin, W->done.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
        if (W->h_fin[2] != 0) {
            set_error("persistent Krylov loop kernel failed (code %d: 1 = TMA/mbarrier wait, 2 = grid barrier timed out)", W->h_fin[2]);
            throw CudaFail{FPSB_ECUDA};
        }
        stats_from(W->h_st[0], st[0]);
        stats_from(W->h_st[1], st[1]);
        if (W->prof_armed) {
            float ms = 0.f;
            FPSB_CUDA(cudaEventElapsedTime(&ms, W->pev[0], W->pev[1]));
            h->prof_loop_ms = ms;
            // half iterations executed: step launches + the phases the persistent kernel ran
            h->prof_step_launches = W->prof_launch1 - W->prof_launch0;
            if (loop_phases_pending) h->prof_step_launches += (int64_t)W->h_fin[1] - W->prof_loop_launches;
            W->prof_armed = false;
        }
    }
};

static SlotIO io_none() { SlotIO io{}; io.mode = MD_NONE; return io; }
static SlotIO io_mode(int mode, double *a0 = nullptr, double *a1 = nullptr, double *a2 = nullptr) {
    SlotIO io{};
    io.mode = mode; io.a0 = a0; io.a1 = a1; io.a2 = a2; io.c0 = 1.0; io.c1 = 0.0;
    return io;
}

// p = rhs - A' q  (n-space), plain kernel
static void residual_p(Engine &E, const double *rhs, const double *q, double *p) {
    Handle *h = E.h;
    if (h->At.grid == 0) return;
    StepParams P = E.base_n;
    P.io[0] = io_mode(MD_PLAIN, const_cast<double *>(rhs));
    P.io[0].gin = q; P.io[0].self = p; P.io[0].c0 = -1.0; P.io[0].c1 = 1.0;
    P.io[1] = io_none();
    launch_step(h, h->At, P, false, 0);
}

static const int kChunk = 4;

// LSQR on A' occupies: Gn[:,slot] = u, Gm[:,slot] = v, am[slot][0] = w, am[slot][1] = x
static void lsqr_init(Engine &E, int slot, const double *rhs) {
    E.ew(EW_INIT_LSQR, slot, (int)E.h->nvar, rhs, nullptr, nullptr, nullptr, nullptr, nullptr, E.W->Gn.p, slot, 1.0);
}

// K = [I A'; A -delta I] with no constraints or no variables: closed forms (nothing to iterate on).
// Returns true when it handled the call.
__global__ void fill_kernel(int n, double *dst, const double *src, double c) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src ? c * src[i] : 0.0;
}
static bool degenerate_two(Handle *h, int kind, double delta, const double *rhs1, const double *rhs2, double *p1, double *q1,
                           double *p2, double *q2, fpsb_krylov_stats *st) {
    const int64_t n = h->nvar, m = h->ncon;
    if (n > 0 && m > 0) return false;
    memset(h->loop_info, 0, sizeof(h->loop_info));
    auto fill = [&](int64_t cnt, double *dst, const double *src, double c) {
        if (cnt > 0) { fill_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, h->stream>>>((int)cnt, dst, src, c); h->launches += 1; }
    };
    // no constraints: K = I            -> p = rhs (n-space right-hand sides), nothing else
    // no variables:   K = -delta I     -> q2 = -rhs2 / delta for the mixed system (0 when delta = 0)
    fill(n, p1, rhs1, 1.0);
    fill(n, p2, kind == 1 ? rhs2 : nullptr, 1.0);
    fill(m, q1, nullptr, 0.0);
    fill(m, q2, (kind == 0 && delta != 0.0) ? rhs2 : nullptr, delta != 0.0 ? -1.0 / delta : 0.0);
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    for (int s = 0; s < 2; ++s) {
        memset(&st[s], 0, sizeof(st[s]));
        st[s].solved = 1; st[s].status = FPSB_ST_SOLVED;
    }
    return true;
}

void iter_solve_two_mixed(Handle *h, double delta, const double *rhs1, const double *rhs2, double *p1,
                          double *q1, double *p2, double *q2, fpsb_krylov_stats *st) {
    iter_setup(h);
    if (degenerate_two(h, 0, delta, rhs1, rhs2, p1, q1, p2, q2, st)) return;
    Engine E(h);
    IterWs *W = h->iter;
    const fpsb_iter_opts &o = h->iopts;
    const int64_t n = h->nvar, m = h->ncon;
    E.begin(make_lsqr(sqrt(delta), o.ls_atol, o.ls_rtol, o.ls_itmax, n, m),
            make_craig(delta, o.ln_atol, o.ln_rtol, o.ln_btol, o.ln_conlim, o.ln_itmax, m, n));
    W->Gn.zero(h->stream); W->Gm.zero(h->stream);
    W->an[1][0].zero(h->stream); W->an[1][1].zero(h->stream);   // CRAIG x, w2
    W->am[0][1].zero(h->stream);                                // LSQR x
    lsqr_init(E, 0, rhs1);
    E.ew(EW_INIT_CRAIG, 1, (int)m, rhs2, W->am[1][0].p, W->am[1][1].p, nullptr, nullptr, nullptr, W->Gm.p, 1, -1.0);
    SlotIO l_init = io_mode(MD_LSQR_INIT_M);
    SlotIO l_u = io_mode(MD_LSQR_U);
    SlotIO l_v = io_mode(MD_LSQR_V, W->am[0][0].p, W->am[0][1].p);
    SlotIO c_v = io_mode(MD_CRAIG_V, W->an[1][0].p, W->an[1][1].p);
    SlotIO c_u = io_mode(MD_CRAIG_U, W->am[1][0].p, W->am[1][1].p);
    E.mark_begin();
    E.defer = true;
    E.step(true, true, l_init, io_none());
    if (E.can_persist()) E.run_loop(l_u, c_v, l_v, c_u);
    else E.loop([&](int) {
        E.step(false, true, l_u, c_v);
        E.step(true, true, l_v, c_u);
    }, kChunk);
    E.mark_end();
    // outputs
    E.ew(EW_COPY, 0, (int)m, W->am[0][1].p, q1, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
    residual_p(E, rhs1, q1, p1);
    E.ew(EW_CRAIG_FLUSH, 1, (int)n, nullptr, W->an[1][0].p, W->an[1][1].p, p2, nullptr, nullptr, W->Gn.p, 1, 1.0, 1);
    E.ew(EW_COPY, 1, (int)m, W->am[1][1].p, q2, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
    E.fetch(st);
}

void iter_solve_two_least_squares(Handle *h, double delta, const double *rhs1, const double *rhs2,
                                  double *p1, double *q1, double *p2, double *q2,
                                  fpsb_krylov_stats *st) {
    iter_setup(h);
    if (degenerate_two(h, 1, delta, rhs1, rhs2, p1, q1, p2, q2, st)) return;
    Engine E(h);
    IterWs *W = h->iter;
    const fpsb_iter_opts &o = h->iopts;
    const int64_t n = h->nvar, m = h->ncon;
    SlotState s = make_lsqr(sqrt(delta), o.ls_atol, o.ls_rtol, o.ls_itmax, n, m);
    E.begin(s, s);
    W->Gn.zero(h->stream); W->Gm.zero(h->stream);
    W->am[0][1].zero(h->stream); W->am[1][1].zero(h->stream);
    lsqr_init(E, 0, rhs1);
    lsqr_init(E, 1, rhs2);
    SlotIO init0 = io_mode(MD_LSQR_INIT_M), init1 = io_mode(MD_LSQR_INIT_M);
    SlotIO u0 = io_mode(MD_LSQR_U), u1 = io_mode(MD_LSQR_U);
    SlotIO v0 = io_mode(MD_LSQR_V, W->am[0][0].p, W->am[0][1].p);
    SlotIO v1 = io_mode(MD_LSQR_V, W->am[1][0].p, W->am[1][1].p);
    E.mark_begin();
    E.defer = true;
    E.step(true, true, init0, init1);
    if (E.can_persist()) E.run_loop(u0, u1, v0, v1);
    else E.loop([&](int) {
        E.step(false, true, u0, u1);
        E.step(true, true, v0, v1);
    }, kChunk);
    E.mark_end();
    E.ew(EW_COPY, 0, (int)m, W->am[0][1].p, q1, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
    E.ew(EW_COPY, 1, (int)m, W->am[1][1].p, q2, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
    // p_i = rhs_i - A' q_i : one two-column SpMM
    if (h->At.grid) {
        StepParams P = E.base_n;
        P.io[0] = io_mode(MD_PLAIN, const_cast<double *>(rhs1));
        P.io[0].gin = q1; P.io[0].self = p1; P.io[0].c0 = -1.0; P.io[0].c1 = 1.0;
        P.io[1] = io_mode(MD_PLAIN, const_cast<double *>(rhs2));
        P.io[1].gin = q2; P.io[1].self = p2; P.io[1].c0 = -1.0; P.io[1].c1 = 1.0;
        launch_step(h, h->At, P, false, 0);
    }
    E.fetch(st);
}

// MINRES on (A A' + lambda I) in slot `slot` (non-pair kernels), result copied to `out`
static void run_minres(Engine &E, int slot, const double *rhs, double *out) {
    Handle *h = E.h;
    IterWs *W = E.W;
    const int m = (int)h->ncon;
    double *r1 = W->am[slot][0].p, *r2 = W->am[slot][1].p, *wa = W->am[slot][2].p, *wb = W->am[slot][3].p,
           *x = W->am[slot][4].p, *y = W->ym.p, *t = W->an[slot][0].p;
    E.ew(EW_MINRES_INIT, slot, m, rhs, r1, r2, wa, wb, x, nullptr, -1, 1.0);
    double *w1 = wa, *w2 = wb;
    SlotIO none = io_none();
    E.loop([&](int k) {
        // t = A' r2 ; y = (A t + lambda r2)/beta - (beta/oldbeta) r1 ; alpha = r2'y / beta
        SlotIO n_io = io_mode(MD_PLAIN);
        n_io.gin = r2; n_io.self = t; n_io.c0 = 1.0;
        SlotIO m_io = io_mode(MD_MINRES_M, r2, r1);
        m_io.gin = t; m_io.self = y;
        if (slot == 0) { E.step(false, false, n_io, none); E.step(true, false, m_io, none); }
        else { E.step(false, false, none, n_io); E.step(true, false, none, m_io); }
        E.ew(EW_MINRES_E1, slot, m, y, r1, r2, w1, w2, nullptr, nullptr, -1, 1.0);
        double *wcur = (k == 1) ? w2 : w1;
        E.ew(EW_MINRES_E2, slot, m, nullptr, nullptr, nullptr, wcur, nullptr, x, nullptr, -1, 1.0);
        if (k >= 2) std::swap(w1, w2);
    }, 2);
    E.ew(EW_COPY, slot, m, x, out, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
}

// CGLS on A' (min ||b - A' x||^2 + lambda ||x||^2) in slot `slot`, result copied to `out`
static void run_cgls(Engine &E, int slot, const double *rhs, double *out) {
    Handle *h = E.h;
    IterWs *W = E.W;
    const int m = (int)h->ncon, n = (int)h->nvar;
    double *r = W->an[slot][0].p, *q = W->an[slot][1].p;
    double *x = W->am[slot][0].p, *p = W->am[slot][1].p, *s = W->am[slot][2].p;
    W->am[slot][0].zero(h->stream);
    E.ew(EW_CGLS_INIT, slot, n, rhs, r, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0);
    SlotIO none = io_none();
    {
        SlotIO io = io_mode(MD_CGLS_INIT_M);
        io.gin = r; io.self = p;
        if (slot == 0) E.step(true, false, io, none); else E.step(true, false, none, io);
    }
    E.loop([&](int) {
        SlotIO n_io = io_mode(MD_CGLS_N);
        n_io.gin = p; n_io.self = q;
        if (slot == 0) E.step(false, false, n_io, none); else E.step(false, false, none, n_io);
        E.ew(EW_CGLS_EN, slot, n, nullptr, r, q, nullptr, nullptr, nullptr, nullptr, -1, 1.0);
        SlotIO m_io = io_mode(MD_CGLS_M, x, p);
        m_io.gin = r; m_io.self = s;
        if (slot == 0) E.step(true, false, m_io, none); else E.step(true, false, none, m_io);
        E.ew(EW_CGLS_EM, slot, m, nullptr, s, p, nullptr, nullptr, nullptr, nullptr, -1, 1.0);
    }, 2);
    E.ew(EW_COPY, slot, m, x, out, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
}

void iter_solve_two_extras(Handle *h, double delta, const double *rhs1, const double *rhs2, double *u1,
                           double *u2, fpsb_krylov_stats *st, bool ldlt_variant) {
    iter_setup(h);
    if (h->nvar == 0 || h->ncon == 0) {
        // (A A' + tau I) u = rhs with no variables: u1 = 0 (A rhs1 is empty), u2 = rhs2 / tau ; no constraints: nothing
        const double tau = std::max(delta, 1e-14);
        memset(h->loop_info, 0, sizeof(h->loop_info));
        if (h->ncon > 0) {
            fill_kernel<<<(unsigned)((h->ncon + 255) / 256), 256, 0, h->stream>>>((int)h->ncon, u1, nullptr, 0.0);
            fill_kernel<<<(unsigned)((h->ncon + 255) / 256), 256, 0, h->stream>>>((int)h->ncon, u2, rhs2, 1.0 / tau);
            h->launches += 2;
        }
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
        for (int s = 0; s < 2; ++s) { memset(&st[s], 0, sizeof(st[s])); st[s].solved = 1; st[s].status = FPSB_ST_SOLVED; }
        return;
    }
    Engine E(h);
    IterWs *W = h->iter;
    const fpsb_iter_opts &o = h->iopts;
    const int64_t n = h->nvar, m = h->ncon;
    const double tau = std::max(delta, 1e-14);
    fpsb_krylov_stats tmp[2];
    if (!ldlt_variant) {
        // LSQR(A', rhs1, lambda = sqrt(tau))   src/solve_linear_system.jl:53
        E.begin(make_lsqr(sqrt(tau), o.ls_atol, o.ls_rtol, o.ls_itmax, n, m), make_none());
        W->Gn.zero(h->stream); W->Gm.zero(h->stream);
        W->am[0][1].zero(h->stream);
        lsqr_init(E, 0, rhs1);
        SlotIO l_init = io_mode(MD_LSQR_INIT_M), l_u = io_mode(MD_LSQR_U);
        SlotIO l_v = io_mode(MD_LSQR_V, W->am[0][0].p, W->am[0][1].p);
        E.defer = true;
        E.step(true, true, l_init, io_none());
        if (E.can_persist()) E.run_loop(l_u, io_none(), l_v, io_none());
        else E.loop([&](int) {
            E.step(false, true, l_u, io_none());
            E.step(true, true, l_v, io_none());
        }, kChunk);
        E.ew(EW_COPY, 0, (int)m, W->am[0][1].p, u1, nullptr, nullptr, nullptr, nullptr, nullptr, -1, 1.0, 0);
        E.fetch(tmp);
        st[0] = tmp[0];
        // MINRES(A A', rhs2, lambda = tau, ne_*)   src/solve_linear_system.jl:60-70
        E.begin(make_none(), make_minres(tau, o.ne_atol, o.ne_rtol, o.ne_etol, o.ne_conlim, o.ne_itmax, m));
        run_minres(E, 1, rhs2, u2);
        E.fetch(tmp);
        st[1] = tmp[1];
    } else {
        // cgls(A', rhs1, lambda = tau) ; minres(A A', rhs2, lambda = tau) — Krylov.jl defaults
        E.begin(make_cgls(tau, kSqrtEps, kSqrtEps, 0, n, m), make_none());
        run_cgls(E, 0, rhs1, u1);
        E.fetch(tmp);
        st[0] = tmp[0];
        E.begin(make_none(), make_minres(tau, kSqrtEps / 100, kSqrtEps / 100, kSqrtEps, 1.0 / kSqrtEps, 0, m));
        run_minres(E, 1, rhs2, u2);
        E.fetch(tmp);
        st[1] = tmp[1];
    }
}

#include "fpsb_extras_batch.inl"

#include "fpsb_dist.inl"

}  // namespace fpsb
