// fpsb_ldlt.cu — numeric LDL' refactorisation and 2-RHS triangular solves on the GPU.
//
// Reference surface replaced (file:line under /root/reference):
//   sparse(rows, cols, vals) + ldl_factorize!(M, str)   src/solve_linear_system.jl:231-234
//   ldiv!(str, sol) on the N x 2 `sol`                  src/solve_linear_system.jl:242-243, :194-195
//   LDLFactorizations' up-looking numeric LDL' with dynamic regularisation (SURVEY App. B2/B3)
//
// Design (B200): the fill pattern is known from the host analysis (fpsb_symbolic.cpp), so L is
// stored as dense supernodal panels in HBM.  One persistent kernel factorises everything:
// CTAs (or single warps for tiny supernodes) take supernodes from a level-ordered ticket queue and
// pull the updates of their descendants (left-looking, no floating-point atomics => bitwise
// reproducible), waiting on per-supernode release/acquire flags instead of level barriers.
// The diagonal block is factorised in shared memory with the reference's pivot rule
//   |D[k]| < tol  =>  D[k] = sign(r) * max(|D[k] + r|, |r|),  r = (P[k] < n_d ? r1 : r2),
// and the triangular solves run the same dependency-driven schedule on an interleaved N x 2
// right-hand side (both columns share every load of L).
#include "fpsb_internal.h"
#include "fpsb_symbolic.h"
#include "fpsb_device.cuh"
#include <algorithm>
#include <cstring>
#include <stdexcept>

namespace fpsb {

constexpr int kMaxW = 64;               // == kMaxSuperWidth in fpsb_symbolic.cpp
constexpr int kLdltBlock = 256;
constexpr int kWarpsPerBlock = kLdltBlock / 32;
constexpr int kSmallW = 8;              // warp-level supernodes: w <= kSmallW and w*(w+nr) <= 512
constexpr int kShDoubles = (kMaxW + 1) * kMaxW + 4 * kMaxW;
// CTA-level supernodes (fpsb_ldlt.cu "block" routines): shared-memory staging of the fronts
constexpr int kBS = kMaxW + 1;                         // row stride of the diagonal block in shared memory
constexpr int kUpdRows = 64;                            // rows of a descendant panel staged per pass of the Schur update
constexpr int kTrsmRows = 2 * kUpdRows;                 // rows of L21 staged per pass (reuses the two update buffers)
constexpr int kFacDoubles = kBS * kMaxW + 2 * kMaxW + 2 * kUpdRows * kMaxW;      // B | dd | rk | S | C
constexpr int kSolveRows = 1024;                        // rows of a panel whose x[R[r]] are staged per pass of the backward solve
constexpr int kSolDoubles = kBS * kMaxW + 2 * kMaxW + 2 * kSolveRows + 2 * kWarpsPerBlock * kMaxW;   // L11 | ys | xr | per-warp partials
constexpr int kWarpShDoubles = (kSmallW + 1) * kSmallW + 4 * kSmallW;   // per warp-level supernode
static_assert(kWarpShDoubles <= kFacDoubles / kWarpsPerBlock, "warp-level supernodes share the block's buffer");
static_assert(kWarpShDoubles <= kSolDoubles / kWarpsPerBlock, "warp-level supernodes share the block's buffer");

struct PlanDev {
    int N, nsuper, ntasks;
    const int *sfirst;
    const int64_t *rptr;
    const int *rows;
    const int64_t *poff;
    const int *order;
    const int *task_start, *task_cnt;
    const int64_t *uptr;
    const int64_t *umid;      // pairs [uptr[t], umid[t]) come from non-leaf sources
    const int *usrc, *ua, *ub;
    const int64_t *urel;
    const int *rel;
    const int64_t *tptr;
    const int *ttgt;
    const int *P;
    const int *sn_of;
    // leaf contributions grouped by target column
    const int64_t *lcptr, *lc_src, *lc_rel;
    const int *lc_cnt, *lc_ldd, *lc_wd, *lc_fd;
    int ntasks_leaf;          // tasks [0, ntasks_leaf) are leaf supernodes (no incoming update)
    double *panels;
    double *D;
    double2 *Y;
    int *done_f, *done_s, *done_b;
    int *ticket;        // [3]
    int *fail;          // 0 ok ; >0 (index+1) zero pivot ; -2 dependency wait timed out
    int n_d;
    double tol, r1, r2;
    int dynamic_reg;
    unsigned long long *tstamp;   // debug builds (-DFPSB_LDLT_TIMERS): [3][nsuper] completion times (globaltimer ns)
};
// The storage one numeric factorisation works on: the handle's own (single instance, SYNC routines: flags and
// tickets order the supernodes across CTAs) or one instance's slice of the batched factor store (one CTA owns the
// instance and walks the plan level by level: no flags, __syncthreads between dependent steps).
struct LdltWork {
    double *panels;
    double *D;
    double2 *Y;
    int *fail;
};
__host__ __device__ __forceinline__ LdltWork work_of(const PlanDev &P) { return LdltWork{P.panels, P.D, P.Y, P.fail}; }

#ifdef FPSB_LDLT_TIMERS
#define LDLT_STAMP(P, phase, t) do { unsigned long long now_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now_)); \
        (P).tstamp[(size_t)(phase) * (P).nsuper + (t)] = now_; } while (0)
#else
#define LDLT_STAMP(P, phase, t) do { } while (0)
#endif

struct LdltPlan {
    Symbolic S;
    fpsb_ldlt_opts opts{};
    DevBuf<int> sfirst, rows, order, task_start, task_cnt, usrc, ua, ub, rel, ttgt, P, pinv, asrc, sn_of;
    DevBuf<int> lc_cnt, lc_ldd, lc_wd, lc_fd;
    DevBuf<int64_t> rptr, poff, uptr, umid, urel, tptr, aslot, aptr, lcptr, lc_src, lc_rel;
    int ntasks_leaf = 0;
    DevBuf<double> panels, D;
    DevBuf<double2> Y;
    DevBuf<int> done_f, done_s, done_b, ticket, fail;
    DevBuf<unsigned long long> tstamp;
    // batched path: supernodes grouped into steps of mutually independent ones (bsn; bstep: {first, first warp-level,
    // end} per step, step 0 = the leaves wider than one column, step l = dependency level l), the factor store
    // (ninst x bstride doubles: panels | D), per-CTA right-hand sides, per-instance factorisation status
    DevBuf<int> bsn, bstep;
    int nbstep = 0;
    int64_t bstride = 0;
    DevBuf<double> bstore;
    DevBuf<double2> bY;
    DevBuf<int> bok;
    int64_t bstore_inst = 0, bY_rows = 0, bok_inst = 0;
    int64_t bninst = -1;        // ninst of the last batched mixed call (-1: none), whose factors bstore holds
    int ntasks = 0;
    int epoch = 0;
    int64_t naslot = 0;
    bool factorized = false;
    bool have_factor = false;
    PlanDev dev{};
};

__device__ __forceinline__ int ld_acquire(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <bool WARP>
__device__ __forceinline__ void gsync() {
    if (WARP) __syncwarp();
    else __syncthreads();
}

// one thread spins (bounded), the group then synchronises
template <bool WARP>
__device__ __forceinline__ void wait_done(const int *flag, int epoch, int tid, int *fail) {
    if (tid == 0) {
        // A CTA that took an early ticket may legitimately wait for almost the whole factorisation: the
        // bound is wall time (60 s: a scheduling bug, not a long factorisation), polled rarely
        int it = 0;
        unsigned long long t0 = 0;
        while (ld_acquire(flag) != epoch) {
            __nanosleep(40);
            ++it;
            if ((it & 1023) == 0) {
                if (ld_acquire(fail) == -2) break;                      // someone already gave up
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > 60000000000ull) { atomicExch(fail, -2); break; }
            }
        }
        __threadfence();
    }
    gsync<WARP>();
}

// ------------------------------------------------------------------------------------------------
// assembly: panels <- [1..1 | jac values | -delta..]  through the precomputed slot map
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void assemble_slot(int64_t i, const int64_t *aslot, const int64_t *aptr, const int *asrc,
                                              const double *jvals, int nvar, int64_t nnzj, double delta, double *panels) {
    double s = 0.0;
    for (int64_t p = aptr[i]; p < aptr[i + 1]; ++p) {
        int id = asrc[p];
        double v = (id < nvar) ? 1.0 : ((int64_t)id < nvar + nnzj ? jvals[id - nvar] : -delta);
        s += v;
    }
    panels[aslot[i]] = s;
}
__global__ void assemble_kernel(int64_t nslot, const int64_t *aslot, const int64_t *aptr, const int *asrc,
                                const double *jvals, int nvar, int64_t nnzj, double delta, double *panels) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nslot) return;
    assemble_slot(i, aslot, aptr, asrc, jvals, nvar, nnzj, delta, panels);
}

// ------------------------------------------------------------------------------------------------
// numeric factorisation of one supernode (left-looking)
// ------------------------------------------------------------------------------------------------
template <bool WARP, bool SYNC = true>
__device__ void factor_supernode(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid, int nt) {
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    double *panel = W.panels + P.poff[t];

    // 1. pull the updates of every non-leaf descendant supernode (leaf contributions were applied
    //    by leaf_update_kernel before this launch)
    for (int64_t q = P.uptr[t]; q < P.umid[t]; ++q) {
        const int d = P.usrc[q];
        if (SYNC) wait_done<WARP>(&P.done_f[d], epoch, tid, P.fail);
        const int fd = P.sfirst[d];
        const int wd = P.sfirst[d + 1] - fd;
        const int nrd = (int)(P.rptr[d + 1] - P.rptr[d]);
        const int ldd = wd + nrd;
        const double *pd = W.panels + P.poff[d] + wd;     // rows below d's block
        const double *Dd = W.D + fd;
        const int a = P.ua[q], b = P.ub[q];
        const int *relq = P.rel + P.urel[q];
        const int nrow = nrd - a, ncol = b - a;
        const int total = nrow * ncol;
        for (int e = tid; e < total; e += nt) {
            const int j = e / nrow;
            const int i = e - j * nrow;
            if (i < j) continue;
            double s = 0.0;
            for (int k = 0; k < wd; ++k) {
                const double lj = __ldcg(pd + (size_t)k * ldd + a + j);
                const double li = __ldcg(pd + (size_t)k * ldd + a + i);
                s += li * (lj * __ldcg(Dd + k));
            }
            panel[(size_t)relq[j] * ld + relq[i]] -= s;
        }
        gsync<WARP>();
    }

    // 2. dense LDL' of the w x w diagonal block in shared memory (row-major, stride w+1)
    const int ws = w + 1;
    double *B = sh;
    double *yk = sh + (size_t)ws * w;
    double *dd = yk + w;
    for (int e = tid; e < w * w; e += nt) {
        const int j = e / w, i = e - j * w;      // column j, row i
        if (i >= j) B[i * ws + j] = panel[(size_t)j * ld + i];
    }
    gsync<WARP>();
    for (int k = 0; k < w; ++k) {
        if (tid == 0) {
            double dk = B[k * ws + k];
            if (P.dynamic_reg && fabs(dk) < P.tol) {
                const double r = (P.P[f + k] < P.n_d) ? P.r1 : P.r2;
                const double sg = (double)((r > 0.0) - (r < 0.0));
                dk = sg * fmax(fabs(dk + r), fabs(r));
            }
            if (dk == 0.0) { atomicCAS(W.fail, 0, f + k + 1); dk = 1.0; }
            dd[k] = dk;
            W.D[f + k] = dk;
        }
        gsync<WARP>();
        const double dk = dd[k];
        for (int i = k + 1 + tid; i < w; i += nt) {
            const double y = B[i * ws + k];
            yk[i] = y;
            B[i * ws + k] = y / dk;
        }
        gsync<WARP>();
        const int rem = w - k - 1;
        for (int e = tid; e < rem * rem; e += nt) {
            const int jj = e / rem, ii = e - jj * rem;
            if (ii < jj) continue;
            const int i = k + 1 + ii, j = k + 1 + jj;
            B[i * ws + j] -= B[i * ws + k] * yk[j];
        }
        gsync<WARP>();
    }
    for (int e = tid; e < w * w; e += nt) {
        const int j = e / w, i = e - j * w;
        if (i > j) panel[(size_t)j * ld + i] = B[i * ws + j];
    }

    // 3. sub-diagonal block: y_k = a_k - sum_{j<k} y_j L11[k][j] ; L21[i][k] = y_k / d_k
    for (int i = tid; i < nr; i += nt) {
        double y[kMaxW];
        double *row = panel + w + i;
        for (int k = 0; k < w; ++k) {
            double s = row[(size_t)k * ld];
            for (int j = 0; j < k; ++j) s -= y[j] * B[k * ws + j];
            y[k] = s;
            row[(size_t)k * ld] = s / dd[k];
        }
    }
    if (SYNC) __threadfence();
    gsync<WARP>();
    if (SYNC && tid == 0) { st_release(&P.done_f[t], epoch); LDLT_STAMP(P, 0, t); }
}

template <bool WARP, bool SYNC = true>
__device__ void fwd_supernode(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid, int nt) {
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    const double *panel = W.panels + P.poff[t];
    double2 *ys = reinterpret_cast<double2 *>(sh);     // w entries
    for (int k = tid; k < w; k += nt) ys[k] = W.Y[f + k];
    gsync<WARP>();
    for (int64_t q = P.uptr[t]; q < P.umid[t]; ++q) {
        const int d = P.usrc[q];
        if (SYNC) wait_done<WARP>(&P.done_s[d], epoch, tid, P.fail);
        const int fd = P.sfirst[d];
        const int wd = P.sfirst[d + 1] - fd;
        const int nrd = (int)(P.rptr[d + 1] - P.rptr[d]);
        const int ldd = wd + nrd;
        const double *pd = W.panels + P.poff[d] + wd;
        const int a = P.ua[q], b = P.ub[q];
        const int *relq = P.rel + P.urel[q];
        for (int j = a + tid; j < b; j += nt) {
            double s0 = 0.0, s1 = 0.0;
            for (int k = 0; k < wd; ++k) {
                const double l = __ldcg(pd + (size_t)k * ldd + j);
                const double2 yv = __ldcg(W.Y + fd + k);
                s0 += l * yv.x; s1 += l * yv.y;
            }
            const int lc = relq[j - a];
            ys[lc].x -= s0; ys[lc].y -= s1;
        }
        gsync<WARP>();
    }
    // unit lower triangular solve with L11
    for (int k = 0; k < w; ++k) {
        const double2 yk = ys[k];
        for (int i = k + 1 + tid; i < w; i += nt) {
            const double l = panel[(size_t)k * ld + i];
            ys[i].x -= l * yk.x; ys[i].y -= l * yk.y;
        }
        gsync<WARP>();
    }
    for (int k = tid; k < w; k += nt) W.Y[f + k] = ys[k];
    if (SYNC) __threadfence();
    gsync<WARP>();
    if (SYNC && tid == 0) { st_release(&P.done_s[t], epoch); LDLT_STAMP(P, 1, t); }
}

template <bool WARP, bool SYNC = true>
__device__ void bwd_supernode(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid, int nt, bool nowait) {
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    const double *panel = W.panels + P.poff[t];
    const int *R = P.rows + P.rptr[t];
    if (SYNC && !nowait)
        for (int64_t q = P.tptr[t]; q < P.tptr[t + 1]; ++q)
            wait_done<WARP>(&P.done_b[P.ttgt[q]], epoch, tid, P.fail);
    double2 *xs = reinterpret_cast<double2 *>(sh);     // w entries
    // xs[k] = y_k / d_k - sum_r L21[r][k] x[R[r]]
    const int lane = tid & 31, wid = tid >> 5, nwarp = WARP ? 1 : (nt >> 5);
    for (int k = wid; k < w; k += nwarp) {
        double s0 = 0.0, s1 = 0.0;
        const double *col = panel + (size_t)k * ld + w;
        for (int r = lane; r < nr; r += 32) {
            const double l = col[r];
            const double2 xv = __ldcg(W.Y + R[r]);
            s0 += l * xv.x; s1 += l * xv.y;
        }
        s0 = warp_sum(s0); s1 = warp_sum(s1);
        if (lane == 0) {
            const double2 yv = W.Y[f + k];
            const double dk = W.D[f + k];
            xs[k] = make_double2(yv.x / dk - s0, yv.y / dk - s1);
        }
    }
    gsync<WARP>();
    for (int i = w - 1; i > 0; --i) {
        const double2 xi = xs[i];
        for (int k = tid; k < i; k += nt) {
            const double l = panel[(size_t)k * ld + i];
            xs[k].x -= l * xi.x; xs[k].y -= l * xi.y;
        }
        gsync<WARP>();
    }
    for (int k = tid; k < w; k += nt) W.Y[f + k] = xs[k];
    if (SYNC) __threadfence();
    gsync<WARP>();
    if (SYNC && tid == 0) { st_release(&P.done_b[t], epoch); LDLT_STAMP(P, 2, t); }
}


// ================================================================================================
// CTA-level supernodes with the fronts staged in shared memory
// ================================================================================================
__device__ __forceinline__ void prefetch_l2_range(const double *p, size_t count, int tid, int nt) {
    const char *c = reinterpret_cast<const char *>(p);
    const size_t bytes = count * sizeof(double);
    for (size_t o = (size_t)tid * 128; o < bytes; o += (size_t)nt * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(c + o));
}

// FP64 tensor-core tile (DMMA, m8n8k4): D(8x8) += A(8x4, row) * B(4x8, col); lane l holds A[l/4][l%4], B[l%4][l/4],
// C[l/4][2*(l%4) .. +1]
__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Schur update of the target panel by one descendant d: panel(rel[i], rel[j]) -= sum_k L_d(a+i, k) D_d(k) L_d(a+j, k)
// for 0 <= j < b - a, j <= i < nr_d - a.  The descendant's rows are staged k-major in shared memory (S: 64 rows per
// pass, C: the b - a "column rows" scaled by D), each thread owns a 4 x 4 register tile (rows ti + 16 ii, columns
// 4 tj + jj), or, with DMMA, each warp owns 8 x 64 strips of 8 x 8 tensor-core tiles.
template <bool DMMA>
__device__ __forceinline__ void schur_update_block(const PlanDev &P, const LdltWork &W, int64_t q, double *panel, int ld,
                                                   double *S, double *Cc, int tid) {
    const int d = P.usrc[q];
    const int fd = P.sfirst[d];
    const int wd = P.sfirst[d + 1] - fd;
    const int nrd = (int)(P.rptr[d + 1] - P.rptr[d]);
    const int ldd = wd + nrd;
    const int a = P.ua[q], b = P.ub[q];
    const double *pd = W.panels + P.poff[d] + wd + a;     // row a of the rows below d's block
    const double *Dd = W.D + fd;
    const int *relq = P.rel + P.urel[q];
    const int nrow = nrd - a, ncol = b - a;
    for (int e = tid; e < wd * kUpdRows; e += kLdltBlock) {
        const int k = e / kUpdRows, j = e - k * kUpdRows;
        Cc[e] = (j < ncol) ? __ldcg(pd + (size_t)k * ldd + j) * __ldcg(Dd + k) : 0.0;
    }
    for (int r0 = 0; r0 < nrow; r0 += kUpdRows) {
        for (int e = tid; e < wd * kUpdRows; e += kLdltBlock) {
            const int k = e / kUpdRows, r = e - k * kUpdRows;
            S[e] = (r0 + r < nrow) ? __ldcg(pd + (size_t)k * ldd + r0 + r) : 0.0;
        }
        __syncthreads();
        if (!DMMA) {
            const int ti = tid & 15, j0 = (tid >> 4) * 4;
            if (j0 < ncol && r0 + ti < nrow && r0 + ti + 48 >= j0) {
                double acc[4][4];
#pragma unroll
                for (int ii = 0; ii < 4; ++ii)
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) acc[ii][jj] = 0.0;
                for (int k = 0; k < wd; ++k) {
                    const double *sk = S + k * kUpdRows + ti;
                    const double r_0 = sk[0], r_1 = sk[16], r_2 = sk[32], r_3 = sk[48];
                    const double2 ca = *reinterpret_cast<const double2 *>(Cc + k * kUpdRows + j0);
                    const double2 cb = *reinterpret_cast<const double2 *>(Cc + k * kUpdRows + j0 + 2);
                    acc[0][0] += r_0 * ca.x; acc[0][1] += r_0 * ca.y; acc[0][2] += r_0 * cb.x; acc[0][3] += r_0 * cb.y;
                    acc[1][0] += r_1 * ca.x; acc[1][1] += r_1 * ca.y; acc[1][2] += r_1 * cb.x; acc[1][3] += r_1 * cb.y;
                    acc[2][0] += r_2 * ca.x; acc[2][1] += r_2 * ca.y; acc[2][2] += r_2 * cb.x; acc[2][3] += r_2 * cb.y;
                    acc[3][0] += r_3 * ca.x; acc[3][1] += r_3 * ca.y; acc[3][2] += r_3 * cb.x; acc[3][3] += r_3 * cb.y;
                }
#pragma unroll
                for (int ii = 0; ii < 4; ++ii) {
                    const int gi = r0 + ti + 16 * ii;
                    if (gi >= nrow) continue;
                    const int ri = relq[gi];
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int gj = j0 + jj;
                        if (gj < ncol && gi >= gj) panel[(size_t)relq[gj] * ld + ri] -= acc[ii][jj];
                    }
                }
            }
        } else {
            // warp wi owns the 8-row strip wi of this pass; 8 column tiles of 8; k in steps of 4
            const int lane = tid & 31, wi = tid >> 5;
            const int rl = lane >> 2, kl = lane & 3;
            if (r0 + wi * 8 < nrow) {
                double c[8][2];
#pragma unroll
                for (int t = 0; t < 8; ++t) { c[t][0] = 0.0; c[t][1] = 0.0; }
                const int ntile = (ncol + 7) >> 3;
                for (int k = 0; k < wd; k += 4) {
                    const bool kin = k + kl < wd;
                    const double av = kin ? S[(k + kl) * kUpdRows + wi * 8 + rl] : 0.0;
#pragma unroll
                    for (int t = 0; t < 8; ++t) {
                        if (t < ntile) {
                            const double bv = kin ? Cc[(k + kl) * kUpdRows + t * 8 + rl] : 0.0;
                            dmma_m8n8k4(c[t][0], c[t][1], av, bv);
                        }
                    }
                }
                const int gi = r0 + wi * 8 + rl;
                if (gi < nrow) {
                    const int ri = relq[gi];
#pragma unroll
                    for (int t = 0; t < 8; ++t) {
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int gj = t * 8 + 2 * kl + u;
                            if (gj < ncol && gi >= gj) panel[(size_t)relq[gj] * ld + ri] -= c[t][u];
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
}

template <bool DMMA, bool SYNC = true>
__device__ void factor_supernode_block(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid) {
    constexpr int nt = kLdltBlock;
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    double *panel = W.panels + P.poff[t];
    double *B = sh;                          // [w][kBS] lower triangle, row-major
    double *dd = B + kBS * kMaxW;            // pivots
    double *rk = dd + kMaxW;                 // regularisation value of each pivot
    double *S = rk + kMaxW;                  // staging: descendant rows / L21 rows
    double *Cc = S + kUpdRows * kMaxW;       // staging: D-scaled column rows of the descendant

    // 1. updates of every non-leaf descendant (leaf contributions were applied by leaf_update_kernel before)
    for (int64_t q = P.uptr[t]; q < P.umid[t]; ++q) {
        if (SYNC) wait_done<false>(&P.done_f[P.usrc[q]], epoch, tid, P.fail);
        schur_update_block<DMMA>(P, W, q, panel, ld, S, Cc, tid);
    }
    __syncthreads();

    // 2. dense LDL' of the w x w diagonal block in shared memory: right-looking, one barrier per column; column k
    //    stays un-scaled (y_ik = l_ik d_k) until the end, every thread derives the pivot itself
    for (int e = tid; e < w * w; e += nt) {
        const int j = e / w, i = e - j * w;
        if (i >= j) B[i * kBS + j] = panel[(size_t)j * ld + i];
    }
    if (tid < w) rk[tid] = (P.P[f + tid] < P.n_d) ? P.r1 : P.r2;
    __syncthreads();
    for (int k = 0; k < w; ++k) {
        double dk = B[k * kBS + k];
        if (P.dynamic_reg && fabs(dk) < P.tol) {
            const double r = rk[k];
            const double sg = (double)((r > 0.0) - (r < 0.0));
            dk = sg * fmax(fabs(dk + r), fabs(r));
        }
        const bool zero = (dk == 0.0);
        if (zero) dk = 1.0;
        if (tid == 0) { dd[k] = dk; if (zero) atomicCAS(W.fail, 0, f + k + 1); }
        const int i = k + 1 + (tid >> 2);
        if (i < w) {
            const double lik = B[i * kBS + k] / dk;
            for (int j = k + 1 + (tid & 3); j <= i; j += 4) B[i * kBS + j] -= lik * B[j * kBS + k];
        }
        __syncthreads();
    }
    if (tid < w) W.D[f + tid] = dd[tid];
    for (int e = tid; e < w * w; e += nt) {
        const int j = e / w, i = e - j * w;
        if (i > j) {
            const double l = B[i * kBS + j] / dd[j];
            B[i * kBS + j] = l;
            panel[(size_t)j * ld + i] = l;
        }
    }
    __syncthreads();

    // 3. rows below the block, 128 at a time through shared memory (k-major, one thread per row):
    //    y_k = a_k - sum_{j<k} y_j L11[k][j] ; L21[i][k] = y_k / d_k
    double *T = S;                           // [w][kTrsmRows]
    for (int r0 = 0; r0 < nr; r0 += kTrsmRows) {
        const int rows = min(kTrsmRows, nr - r0);
        for (int e = tid; e < w * kTrsmRows; e += nt) {
            const int k = e / kTrsmRows, r = e - k * kTrsmRows;
            if (r < rows) T[e] = panel[(size_t)k * ld + w + r0 + r];
        }
        __syncthreads();
        // a thread per row, the sums in the reference's order (j ascending: the factor is then bit-identical to the
        // scalar routine and to the CPU oracle, which the regularised-pivot tests rely on); the un-scaled y_j stay in
        // T until the write-back
        if (tid < rows) {
            for (int k = 1; k < w; ++k) {
                double sv = T[k * kTrsmRows + tid];
                const double *bk = B + k * kBS;
                for (int j = 0; j < k; ++j) sv -= T[j * kTrsmRows + tid] * bk[j];
                T[k * kTrsmRows + tid] = sv;
            }
        }
        __syncthreads();
        for (int e = tid; e < w * kTrsmRows; e += nt) {
            const int k = e / kTrsmRows, r = e - k * kTrsmRows;
            if (r < rows) panel[(size_t)k * ld + w + r0 + r] = T[e] / dd[k];
        }
        __syncthreads();
    }
    if (SYNC) {
        __threadfence();
        __syncthreads();
        if (tid == 0) { st_release(&P.done_f[t], epoch); LDLT_STAMP(P, 0, t); }
    }
}

// 2-column forward / backward substitution with the w x w unit triangle held in shared memory (forward: k-major,
// Ls[k*64 + i] = L(i,k); backward: row-major with stride kBS, Ls[i*kBS + k] = L(i,k) — both conflict-free),
// done by ONE warp with the two right-hand sides in registers (lane owns rows lane and lane + 32)
__device__ __forceinline__ void tri_solve_warp(const double *Ls, double2 *ys, int w, int lane, bool backward) {
    double2 y0 = lane < w ? ys[lane] : make_double2(0.0, 0.0);
    double2 y1 = lane + 32 < w ? ys[lane + 32] : make_double2(0.0, 0.0);
    if (!backward) {
        for (int k = 0; k < w; ++k) {
            const double2 src = (k < 32) ? y0 : y1;
            const double bx = __shfl_sync(0xffffffffu, src.x, k & 31), by = __shfl_sync(0xffffffffu, src.y, k & 31);
            const double *col = Ls + k * kMaxW;
            if (lane > k && lane < w) { const double l = col[lane]; y0.x -= l * bx; y0.y -= l * by; }
            if (lane + 32 > k && lane + 32 < w) { const double l = col[lane + 32]; y1.x -= l * bx; y1.y -= l * by; }
        }
    } else {
        // x_k -= sum_{i>k} L[i][k] x_i : column i of the transposed triangle is row i of L
        for (int i = w - 1; i > 0; --i) {
            const double2 src = (i < 32) ? y0 : y1;
            const double bx = __shfl_sync(0xffffffffu, src.x, i & 31), by = __shfl_sync(0xffffffffu, src.y, i & 31);
            if (lane < i) { const double l = Ls[i * kBS + lane]; y0.x -= l * bx; y0.y -= l * by; }
            if (lane + 32 < i) { const double l = Ls[i * kBS + lane + 32]; y1.x -= l * bx; y1.y -= l * by; }
        }
    }
    if (lane < w) ys[lane] = y0;
    if (lane + 32 < w) ys[lane + 32] = y1;
}

template <bool SYNC = true>
__device__ void fwd_supernode_block(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid) {
    constexpr int nt = kLdltBlock;
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    const double *panel = W.panels + P.poff[t];
    double *Ls = sh;                                                    // [w][64] k-major strict lower triangle
    double2 *ys = reinterpret_cast<double2 *>(sh + kBS * kMaxW);      // w entries
    double2 *part = ys + kMaxW + kSolveRows;                            // [8 warps][w] partial pulls
    const int lane = tid & 31, wid = tid >> 5;
    // the factor is read-only here: the triangle is staged before the dependencies are waited for
    for (int e = tid; e < w * w; e += nt) {
        const int k = e / w, i = e - k * w;
        if (i > k) Ls[k * kMaxW + i] = panel[(size_t)k * ld + i];
    }
    for (int k = tid; k < kWarpsPerBlock * kMaxW; k += nt) part[k] = make_double2(0.0, 0.0);
    __syncthreads();
    // pulls: warp wid takes the pairs q = uptr + wid, + 8, ... (fixed assignment and a fixed final order of the eight
    // partial sums keep the result reproducible); lanes over the target rows
    double2 *mine = part + wid * kMaxW;
    for (int64_t q = P.uptr[t] + wid; q < P.umid[t]; q += kWarpsPerBlock) {
        const int d = P.usrc[q];
        if (SYNC) wait_done<true>(&P.done_s[d], epoch, lane, P.fail);
        const int fd = P.sfirst[d];
        const int wd = P.sfirst[d + 1] - fd;
        const int nrd = (int)(P.rptr[d + 1] - P.rptr[d]);
        const int ldd = wd + nrd;
        const double *pd = W.panels + P.poff[d] + wd;
        const int a = P.ua[q], b = P.ub[q];
        const int *relq = P.rel + P.urel[q];
        for (int j = a + lane; j < b; j += 32) {
            double s0 = 0.0, s1 = 0.0;
            for (int k = 0; k < wd; ++k) {
                const double l = __ldcg(pd + (size_t)k * ldd + j);
                const double2 yv = __ldcg(W.Y + fd + k);
                s0 += l * yv.x; s1 += l * yv.y;
            }
            const int lc = relq[j - a];
            mine[lc].x += s0; mine[lc].y += s1;
        }
        __syncwarp();
    }
    __syncthreads();
    for (int k = tid; k < w; k += nt) {
        double2 y = W.Y[f + k];
#pragma unroll
        for (int u = 0; u < kWarpsPerBlock; ++u) { const double2 pp = part[u * kMaxW + k]; y.x -= pp.x; y.y -= pp.y; }
        ys[k] = y;
    }
    __syncthreads();
    if (wid == 0) {
        tri_solve_warp(Ls, ys, w, lane, false);
        __syncwarp();
        for (int k = lane; k < w; k += 32) W.Y[f + k] = ys[k];
        if (SYNC) {
            __threadfence();
            __syncwarp();
            if (lane == 0) { st_release(&P.done_s[t], epoch); LDLT_STAMP(P, 1, t); }
        }
    }
}

template <bool SYNC = true>
__device__ void bwd_supernode_block(const PlanDev &P, const LdltWork &W, int t, double *sh, int epoch, int tid, bool nowait) {
    constexpr int nt = kLdltBlock;
    const int f = P.sfirst[t];
    const int w = P.sfirst[t + 1] - f;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    const int ld = w + nr;
    const double *panel = W.panels + P.poff[t];
    const int *R = P.rows + P.rptr[t];
    double *Ls = sh;                                                    // [i][kBS] row-major: Ls[i*kBS + k] = L(i, k)
    double2 *xs = reinterpret_cast<double2 *>(sh + kBS * kMaxW);      // w entries
    double2 *xr = xs + kMaxW;                                           // kSolveRows staged x[R[r]]
    const int lane = tid & 31, wid = tid >> 5;
    for (int e = tid; e < w * w; e += nt) {
        const int k = e / w, i = e - k * w;
        if (i > k) Ls[i * kBS + k] = panel[(size_t)k * ld + i];
    }
    prefetch_l2_range(panel, (size_t)ld * w, tid, nt);
    if (SYNC && !nowait)
        for (int64_t q = P.tptr[t]; q < P.tptr[t + 1]; ++q)
            wait_done<false>(&P.done_b[P.ttgt[q]], epoch, tid, P.fail);
    // xs[k] = y_k / d_k - sum_r L21[r][k] x[R[r]] : the gathered x are staged once, a warp per column
    for (int k = tid; k < w; k += nt) {
        const double2 yv = W.Y[f + k];
        const double dk = W.D[f + k];
        xs[k] = make_double2(yv.x / dk, yv.y / dk);
    }
    for (int r0 = 0; r0 < nr; r0 += kSolveRows) {
        const int rows = min(kSolveRows, nr - r0);
        __syncthreads();
        for (int r = tid; r < rows; r += nt) xr[r] = __ldcg(W.Y + R[r0 + r]);
        __syncthreads();
        for (int k = wid; k < w; k += kWarpsPerBlock) {
            double s0 = 0.0, s1 = 0.0;
            const double *col = panel + (size_t)k * ld + w + r0;
            for (int r = lane; r < rows; r += 32) {
                const double l = col[r];
                const double2 xv = xr[r];
                s0 += l * xv.x; s1 += l * xv.y;
            }
            s0 = warp_sum(s0); s1 = warp_sum(s1);
            if (lane == 0) { xs[k].x -= s0; xs[k].y -= s1; }
        }
    }
    __syncthreads();
    if (wid == 0) {
        tri_solve_warp(Ls, xs, w, lane, true);
        __syncwarp();
        for (int k = lane; k < w; k += 32) W.Y[f + k] = xs[k];
        if (SYNC) {
            __threadfence();
            __syncwarp();
            if (lane == 0) { st_release(&P.done_b[t], epoch); LDLT_STAMP(P, 2, t); }
        }
    }
}

// phase: 0 factor, 1 forward, 2 backward (tasks taken in reverse)
// tasks [task_lo, task_hi) are taken through ticket counter `tk`; `nowait`: every dependency is
// known to be complete (an earlier launch), so the backward phase skips its flag waits
// MODE 0: scalar CTA routines (global-memory operands); 1: fronts staged in shared memory, register-tiled Schur
// update; 2: as 1 with the Schur update on the FP64 tensor cores (DMMA m8n8k4).  Dynamic shared memory: phase_smem().
template <int PHASE, int MODE>
__global__ void __launch_bounds__(kLdltBlock, MODE == 0 ? 4 : 2) ldlt_phase_kernel(PlanDev P, int epoch, int task_lo, int task_hi,
                                                                int tk, int nowait) {
    extern __shared__ __align__(16) double sh[];
    __shared__ int s_task;
    const int tid = threadIdx.x;
    const LdltWork W = work_of(P);
    for (;;) {
        if (tid == 0) s_task = atomicAdd(&P.ticket[tk], 1);
        __syncthreads();
        int task = task_lo + s_task;
        __syncthreads();
        if (task >= task_hi) break;
        if (PHASE == 2) task = task_hi - 1 - (task - task_lo);
        const int t0 = P.task_start[task], cnt = P.task_cnt[task];
        if (cnt == 0) {
            const int t = P.order[t0];
            if (MODE == 0) {
                if (PHASE == 0) factor_supernode<false>(P, W, t, sh, epoch, tid, kLdltBlock);
                else if (PHASE == 1) fwd_supernode<false>(P, W, t, sh, epoch, tid, kLdltBlock);
                else bwd_supernode<false>(P, W, t, sh, epoch, tid, kLdltBlock, nowait != 0);
            } else {
                if (PHASE == 0) factor_supernode_block<MODE == 2>(P, W, t, sh, epoch, tid);
                else if (PHASE == 1) fwd_supernode_block(P, W, t, sh, epoch, tid);
                else bwd_supernode_block(P, W, t, sh, epoch, tid, nowait != 0);
            }
        } else {
            const int wid = tid >> 5, lane = tid & 31;
            if (wid < cnt) {
                // in the backward phase the bundle is walked in reverse as well
                const int t = P.order[PHASE == 2 ? t0 + cnt - 1 - wid : t0 + wid];
                double *wsh = sh + wid * kWarpShDoubles;
                if (PHASE == 0) factor_supernode<true>(P, W, t, wsh, epoch, lane, 32);
                else if (PHASE == 1) fwd_supernode<true>(P, W, t, wsh, epoch, lane, 32);
                else bwd_supernode<true>(P, W, t, wsh, epoch, lane, 32, nowait != 0);
            }
        }
        __syncthreads();
    }
}
static size_t phase_smem(int phase, int mode) {
    if (mode == 0) return (size_t)kShDoubles * sizeof(double);
    return (size_t)(phase == 0 ? kFacDoubles : kSolDoubles) * sizeof(double);
}
// FPSB_LDLT_MODE: 0 scalar, 1 staged fronts (default), 2 staged fronts + DMMA Schur update
static int ldlt_mode() {
    static const int mode = [] { const char *e = getenv("FPSB_LDLT_MODE"); const int v = (e && *e) ? atoi(e) : 1; return v < 0 || v > 2 ? 1 : v; }();
    return mode;
}
template <int PHASE>
static void launch_phase(Handle *h, const PlanDev &P, int ntasks, int epoch, int lo, int hi, int tk, int nowait, bool leaves = false) {
    // the leaf launches are all warp-level bundles on the headline shapes: small shared memory, many resident CTAs
    const int mode = leaves ? 0 : ldlt_mode();
    const size_t smem = phase_smem(PHASE, mode);
    const int grid = std::max(1, std::min(ntasks, h->num_sms * (mode == 0 ? 4 : 2)));
    static bool attr_done = false;
    if (!attr_done) {
        attr_done = true;
        for (int m = 1; m <= 2; ++m) {
            const int b0 = (int)phase_smem(0, m), b1 = (int)phase_smem(1, m);
            if (m == 1) {
                FPSB_CUDA(cudaFuncSetAttribute(ldlt_phase_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, b0));
                FPSB_CUDA(cudaFuncSetAttribute(ldlt_phase_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, b1));
                FPSB_CUDA(cudaFuncSetAttribute(ldlt_phase_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, b1));
            } else {
                FPSB_CUDA(cudaFuncSetAttribute(ldlt_phase_kernel<0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, b0));
            }
        }
    }
    if (mode == 0) ldlt_phase_kernel<PHASE, 0><<<grid, kLdltBlock, smem, h->stream>>>(P, epoch, lo, hi, tk, nowait);
    else if (mode == 2 && PHASE == 0) ldlt_phase_kernel<0, 2><<<grid, kLdltBlock, smem, h->stream>>>(P, epoch, lo, hi, tk, nowait);
    else ldlt_phase_kernel<PHASE, 1><<<grid, kLdltBlock, smem, h->stream>>>(P, epoch, lo, hi, tk, nowait);
    h->launches += 1;
}

// ------------------------------------------------------------------------------------------------
// leaf contributions: embarrassingly parallel over TARGET columns (each column is owned by one
// 8-lane group, sources applied in ascending order => deterministic, no floating-point atomics)
// ------------------------------------------------------------------------------------------------
// column j, lane l8 of the 8-lane group that owns it
__device__ __forceinline__ void leaf_update_column(const PlanDev &P, const LdltWork &W, int j, int l8) {
    if (j >= P.N) return;
    const int64_t e0 = P.lcptr[j], e1 = P.lcptr[j + 1];
    if (e0 == e1) return;
    const unsigned gmask = 0xFFu << ((threadIdx.x & 31) & ~7);
    const int t = P.sn_of[j];
    const int ft = P.sfirst[t];
    const int ldt = P.sfirst[t + 1] - ft + (int)(P.rptr[t + 1] - P.rptr[t]);
    double *col = W.panels + P.poff[t] + (size_t)(j - ft) * ldt;
    for (int64_t e = e0; e < e1; ++e) {
        const double *src = W.panels + P.lc_src[e];
        const int cnt = P.lc_cnt[e], ldd = P.lc_ldd[e], wd = P.lc_wd[e];
        const double *Dd = W.D + P.lc_fd[e];
        const int *relp = P.rel + P.lc_rel[e];
        for (int i = l8; i < cnt; i += 8) {
            double s = 0.0;
            for (int k = 0; k < wd; ++k) s += src[(size_t)k * ldd + i] * (src[(size_t)k * ldd] * Dd[k]);
            col[relp[i]] -= s;
        }
        __syncwarp(gmask);
    }
}
__global__ void __launch_bounds__(256) leaf_update_kernel(PlanDev P) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    leaf_update_column(P, work_of(P), gt >> 3, gt & 7);
}

// ------------------------------------------------------------------------------------------------
// one-wide leaf supernodes (a variable nobody was eliminated before: ~2/3 of all columns of a KKT matrix under a
// dissection ordering).  No dependencies, no triangle: flat kernels, 8 lanes per leaf, instead of tickets and bundles.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void leaf1_factor(const PlanDev &P, const LdltWork &W, int i, int l8, int nleaf) {
    if (i >= nleaf) return;
    const int t = P.order[i];
    const int f = P.sfirst[t];
    if (P.sfirst[t + 1] - f != 1) return;
    const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
    double *panel = W.panels + P.poff[t];
    double dk = panel[0];
    if (P.dynamic_reg && fabs(dk) < P.tol) {
        const double r = (P.P[f] < P.n_d) ? P.r1 : P.r2;
        const double sg = (double)((r > 0.0) - (r < 0.0));
        dk = sg * fmax(fabs(dk + r), fabs(r));
    }
    if (dk == 0.0) { if (l8 == 0) atomicCAS(W.fail, 0, f + 1); dk = 1.0; }
    if (l8 == 0) W.D[f] = dk;
    for (int r = l8; r < nr; r += 8) panel[1 + r] = panel[1 + r] / dk;
}
__global__ void __launch_bounds__(256) leaf1_factor_kernel(PlanDev P, int nleaf) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    leaf1_factor(P, work_of(P), gt >> 3, gt & 7, nleaf);
}
// backward: x_f = y_f / d_f - sum_r L21[r] x[R[r]]  (the rows R are ancestors: already final).  All 32 lanes of the
// warp call it (8-lane shuffle reduction).
__device__ __forceinline__ void leaf1_bwd(const PlanDev &P, const LdltWork &W, int i, int l8, int nleaf) {
    const int t = i < nleaf ? P.order[i] : -1;
    const int f = t >= 0 ? P.sfirst[t] : 0;
    const bool on = t >= 0 && P.sfirst[t + 1] - f == 1;
    double s0 = 0.0, s1 = 0.0;
    if (on) {
        const int nr = (int)(P.rptr[t + 1] - P.rptr[t]);
        const double *col = W.panels + P.poff[t] + 1;
        const int *R = P.rows + P.rptr[t];
        for (int r = l8; r < nr; r += 8) {
            const double l = col[r];
            const double2 xv = W.Y[R[r]];
            s0 += l * xv.x; s1 += l * xv.y;
        }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
    if (on && l8 == 0) {
        const double2 yv = W.Y[f];
        const double dk = W.D[f];
        W.Y[f] = make_double2(yv.x / dk - s0, yv.y / dk - s1);
    }
}
__global__ void __launch_bounds__(256) leaf1_bwd_kernel(PlanDev P, int nleaf) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    leaf1_bwd(P, work_of(P), gt >> 3, gt & 7, nleaf);
}

// forward solve: y[j] -= sum over leaf sources d containing row j of L_d(j, :) . y_d
__device__ __forceinline__ void leaf_fwd_update_row(const PlanDev &P, const LdltWork &W, int j) {
    if (j >= P.N) return;
    const int64_t e0 = P.lcptr[j], e1 = P.lcptr[j + 1];
    if (e0 == e1) return;
    double s0 = 0.0, s1 = 0.0;
    for (int64_t e = e0; e < e1; ++e) {
        const double *src = W.panels + P.lc_src[e];
        const int ldd = P.lc_ldd[e], wd = P.lc_wd[e], fd = P.lc_fd[e];
        for (int k = 0; k < wd; ++k) {
            const double l = src[(size_t)k * ldd];
            const double2 yv = W.Y[fd + k];
            s0 += l * yv.x; s1 += l * yv.y;
        }
    }
    double2 y = W.Y[j];
    y.x -= s0; y.y -= s1;
    W.Y[j] = y;
}
__global__ void __launch_bounds__(256) leaf_fwd_update_kernel(PlanDev P) {
    leaf_fwd_update_row(P, work_of(P), blockIdx.x * blockDim.x + threadIdx.x);
}

// Y[k] = (B0[P[k]], B1[P[k]]) with B0 = [rhs1; 0], B1 = kind == 0 ? [0; rhs2] : [rhs2; 0]
__device__ __forceinline__ double2 rhs_entry(int k, int nvar, int kind, const int *P, const double *rhs1, const double *rhs2) {
    const int i = P[k];
    double2 v;
    v.x = (i < nvar) ? rhs1[i] : 0.0;
    if (kind == 0) v.y = (i < nvar) ? 0.0 : rhs2[i - nvar];
    else v.y = (i < nvar) ? rhs2[i] : 0.0;
    return v;
}
__global__ void load_rhs_kernel(int N, int nvar, int kind, const int *P, const double *rhs1,
                                const double *rhs2, double2 *Y) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    Y[k] = rhs_entry(k, nvar, kind, P, rhs1, rhs2);
}
__device__ __forceinline__ void store_sol_entry(int i, int nvar, const int *pinv, const double2 *Y, double *p1, double *q1,
                                                double *p2, double *q2) {
    const double2 v = Y[pinv[i]];
    if (i < nvar) { p1[i] = v.x; p2[i] = v.y; }
    else { q1[i - nvar] = v.x; q2[i - nvar] = v.y; }
}
__global__ void store_sol_kernel(int N, int nvar, const int *pinv, const double2 *Y, double *p1, double *q1,
                                 double *p2, double *q2) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    store_sol_entry(i, nvar, pinv, Y, p1, q1, p2, q2);
}
// reference behaviour on a failed factorisation: `sol` still holds the right-hand sides
__device__ __forceinline__ void passthrough_entry(int i, int nvar, int ncon, int kind, const double *rhs1, const double *rhs2,
                                                  double *p1, double *q1, double *p2, double *q2) {
    if (i < nvar) { p1[i] = rhs1[i]; p2[i] = (kind == 0) ? 0.0 : rhs2[i]; }
    if (i < ncon) { q1[i] = 0.0; q2[i] = (kind == 0) ? rhs2[i] : 0.0; }
}
__global__ void passthrough_kernel(int nvar, int ncon, int kind, const double *rhs1, const double *rhs2,
                                   double *p1, double *q1, double *p2, double *q2) {
    passthrough_entry(blockIdx.x * blockDim.x + threadIdx.x, nvar, ncon, kind, rhs1, rhs2, p1, q1, p2, q2);
}

// ================================================================================================
// batched path: many instances of one plan (same pattern and symbolic analysis, their own values, delta and
// right-hand sides) in one launch.  One CTA owns one instance at a time (i = blockIdx.x, += gridDim.x) and walks the
// plan in steps of mutually independent supernodes (LdltPlan::bstep) with the routine the single-instance launches
// pick for each supernode, so every entry goes through the same operations in the same order as there; a
// __syncthreads between dependent steps is the only synchronisation (no tickets, no flags, no waits).
// ================================================================================================
struct BatchDev {
    const int *sn, *step;       // LdltPlan::bsn / bstep
    int nstep, nleaf;
    int64_t ninst, stride, psize;
    const int64_t *aslot, *aptr;
    const int *asrc;
    int64_t naslot, nnzj;
    const int *pinv;
    double *store;              // [ninst][stride]: panels | D
    double2 *Y;                 // [gridDim.x][N]
    int *ok;                    // [ninst]: factorisation status, kept for the least-squares call
    const double *jvals, *delta, *rhs1, *rhs2;
    double *p1, *q1, *p2, *q2;
    int *factorized;
    int kind;                   // 0 mixed: refactor + solve ; 1 least squares: solve with the stored factors
};

// one step: its CTA-level supernodes one after the other, then its warp-level ones spread over the warps.  M: the
// routines of that part of the plan (0 for the leaves, as their launches; ldlt_mode() for the rest); PHASE 0 factor,
// 1 forward, 2 backward
template <int M, int PHASE>
__device__ __forceinline__ void batch_step(const PlanDev &P, const LdltWork &W, const BatchDev &B, int s, double *sh, int tid) {
    const int s0 = B.step[3 * s], s1 = B.step[3 * s + 1], s2 = B.step[3 * s + 2];
    for (int k = s0; k < s1; ++k) {
        const int t = B.sn[k];
        if (M == 0) {
            if (PHASE == 0) factor_supernode<false, false>(P, W, t, sh, 0, tid, kLdltBlock);
            else if (PHASE == 1) fwd_supernode<false, false>(P, W, t, sh, 0, tid, kLdltBlock);
            else bwd_supernode<false, false>(P, W, t, sh, 0, tid, kLdltBlock, true);
        } else {
            if (PHASE == 0) factor_supernode_block<M == 2, false>(P, W, t, sh, 0, tid);
            else if (PHASE == 1) fwd_supernode_block<false>(P, W, t, sh, 0, tid);
            else bwd_supernode_block<false>(P, W, t, sh, 0, tid, true);
        }
        __syncthreads();
    }
    const int wid = tid >> 5, lane = tid & 31;
    double *wsh = sh + wid * kWarpShDoubles;
    for (int k = s1 + wid; k < s2; k += kWarpsPerBlock) {
        const int t = B.sn[k];
        if (PHASE == 0) factor_supernode<true, false>(P, W, t, wsh, 0, lane, 32);
        else if (PHASE == 1) fwd_supernode<true, false>(P, W, t, wsh, 0, lane, 32);
        else bwd_supernode<true, false>(P, W, t, wsh, 0, lane, 32, true);
    }
    __syncthreads();
}

constexpr int kBatchDoubles = kFacDoubles;     // dynamic shared memory of the batch kernel: the largest routine's
static_assert(kBatchDoubles >= kSolDoubles && kBatchDoubles >= kShDoubles && kBatchDoubles >= kWarpsPerBlock * kWarpShDoubles,
              "the batch kernel runs every routine in one buffer");

// MODE: ldlt_mode() (the routines of the non-leaf supernodes); the sequence per instance is that of ldlt_factorize /
// ldlt_solve2: assemble, one-wide leaves, other leaves, leaf contributions, levels 1.. ; forward, backward, store
template <int MODE>
__global__ void __launch_bounds__(kLdltBlock, 2) ldlt_batch_kernel(PlanDev P, BatchDev B) {
    extern __shared__ __align__(16) double sh[];
    __shared__ int s_fail;
    const int tid = threadIdx.x;
    const int N = P.N, nvar = P.n_d, ncon = P.N - P.n_d;
    const int n2 = B.kind == 0 ? ncon : nvar;
    constexpr int kGroups = kLdltBlock / 8;      // 8-lane groups of the leaf routines
    LdltWork W;
    W.Y = B.Y + (size_t)blockIdx.x * N;
    W.fail = &s_fail;
    for (int64_t i = blockIdx.x; i < B.ninst; i += gridDim.x) {
        W.panels = B.store + i * B.stride;
        W.D = W.panels + B.psize;
        int ok;
        if (B.kind == 0) {
            if (tid == 0) s_fail = 0;
            for (int64_t e = tid; e < B.psize; e += kLdltBlock) W.panels[e] = 0.0;
            __syncthreads();
            const double *jv = B.jvals + i * B.nnzj;
            const double delta = B.delta[i];
            for (int64_t e = tid; e < B.naslot; e += kLdltBlock)
                assemble_slot(e, B.aslot, B.aptr, B.asrc, jv, nvar, B.nnzj, delta, W.panels);
            __syncthreads();
            for (int l0 = 0; l0 < B.nleaf; l0 += kGroups) leaf1_factor(P, W, l0 + (tid >> 3), tid & 7, B.nleaf);
            __syncthreads();
            if (B.nstep > 0) batch_step<0, 0>(P, W, B, 0, sh, tid);
            if (B.nstep > 1) {
                for (int j0 = 0; j0 < N; j0 += kGroups) leaf_update_column(P, W, j0 + (tid >> 3), tid & 7);
                __syncthreads();
                for (int s = 1; s < B.nstep; ++s) batch_step<MODE, 0>(P, W, B, s, sh, tid);
            }
            ok = s_fail == 0;
            if (tid == 0) B.ok[i] = ok;
        } else {
            ok = B.ok[i];
        }
        if (tid == 0) B.factorized[i] = ok;
        const double *r1 = B.rhs1 + i * nvar, *r2 = B.rhs2 + i * n2;
        double *p1 = B.p1 + i * nvar, *q1 = B.q1 + i * ncon, *p2 = B.p2 + i * nvar, *q2 = B.q2 + i * ncon;
        if (ok) {
            for (int k = tid; k < N; k += kLdltBlock) W.Y[k] = rhs_entry(k, nvar, B.kind, P.P, r1, r2);
            __syncthreads();
            if (B.nstep > 0) batch_step<0, 1>(P, W, B, 0, sh, tid);
            if (B.nstep > 1) {
                for (int j = tid; j < N; j += kLdltBlock) leaf_fwd_update_row(P, W, j);
                __syncthreads();
                for (int s = 1; s < B.nstep; ++s) batch_step<MODE, 1>(P, W, B, s, sh, tid);
                for (int s = B.nstep - 1; s >= 1; --s) batch_step<MODE, 2>(P, W, B, s, sh, tid);
            }
            if (B.nstep > 0) batch_step<0, 2>(P, W, B, 0, sh, tid);
            for (int l0 = 0; l0 < B.nleaf; l0 += kGroups) leaf1_bwd(P, W, l0 + (tid >> 3), tid & 7, B.nleaf);
            __syncthreads();
            for (int k = tid; k < N; k += kLdltBlock) store_sol_entry(k, nvar, B.pinv, W.Y, p1, q1, p2, q2);
        } else {
            for (int k = tid; k < max(nvar, ncon); k += kLdltBlock) passthrough_entry(k, nvar, ncon, B.kind, r1, r2, p1, q1, p2, q2);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
template <class T>
static void up(DevBuf<T> &b, const std::vector<T> &v, cudaStream_t s) { b.from(v, s); }

void ldlt_analyze(Handle *h, const int64_t *Puser, const fpsb_ldlt_opts *opts) {
    ldlt_free(h);
    LdltPlan *L = new LdltPlan();
    h->ldlt = L;
    if (opts) L->opts = *opts;
    else fpsb_ldlt_default_opts(&L->opts);
    try {
        analyze((int)h->nvar, (int)h->ncon, h->nnzj, h->jrow.data(), h->jcol.data(), Puser, L->S);
    } catch (const std::invalid_argument &e) {
        set_error("fpsb_ldlt_analyze: %s", e.what());
        throw CudaFail{FPSB_EINVAL};
    } catch (const std::exception &e) {
        set_error("fpsb_ldlt_analyze: %s", e.what());
        throw CudaFail{FPSB_ESTATE};
    }
    Symbolic &S = L->S;
    // tasks: big supernodes alone, small ones bundled one per warp
    std::vector<int> tstart, tcnt;
    {
        auto small = [&](int s) {
            int w = S.sfirst[(size_t)s + 1] - S.sfirst[(size_t)s];
            int nr = (int)(S.rptr[(size_t)s + 1] - S.rptr[(size_t)s]);
            return w <= kSmallW && (int64_t)w * (w + nr) <= 512;
        };
        // `order` is sorted by level: the first nleaf entries are the leaf supernodes; bundles never
        // straddle the leaf / non-leaf boundary (they are processed by different launches)
        for (int part = 0; part < 2; part++) {
            int i = part == 0 ? 0 : S.nleaf;
            const int end = part == 0 ? S.nleaf : S.nsuper;
            auto leaf1 = [&](int s) { return part == 0 && S.sfirst[(size_t)s + 1] - S.sfirst[(size_t)s] == 1; };
            while (i < end) {
                if (leaf1(S.order[(size_t)i])) { i++; continue; }      // leaf1_*_kernel
                if (small(S.order[(size_t)i])) {
                    int j = i;
                    while (j < end && j - i < kWarpsPerBlock && small(S.order[(size_t)j]) && !leaf1(S.order[(size_t)j])) j++;
                    tstart.push_back(i); tcnt.push_back(j - i);
                    i = j;
                } else {
                    tstart.push_back(i); tcnt.push_back(0);
                    i++;
                }
            }
            if (part == 0) L->ntasks_leaf = (int)tstart.size();      // tasks of the leaves wider than one column
        }
    }
    L->ntasks = (int)tstart.size();
    // batched path: one step per dependency level (supernodes of one level do not depend on each other), the CTA-level
    // supernodes of a step first; the one-wide leaves are left to leaf1_factor / leaf1_bwd as in the launches above
    std::vector<int> bsn, bstep;
    {
        auto warp_level = [&](int t) {
            const int w = S.sfirst[(size_t)t + 1] - S.sfirst[(size_t)t];
            const int nr = (int)(S.rptr[(size_t)t + 1] - S.rptr[(size_t)t]);
            return w <= kSmallW && (int64_t)w * (w + nr) <= 512;
        };
        int i = 0;
        for (int lv = 0; lv < S.nlevels; ++lv) {
            int j = i;
            while (j < S.nsuper && S.level[(size_t)S.order[(size_t)j]] == lv) j++;
            bstep.push_back((int)bsn.size());
            for (int pass = 0; pass < 2; ++pass) {
                if (pass == 1) bstep.push_back((int)bsn.size());
                for (int k = i; k < j; ++k) {
                    const int t = S.order[(size_t)k];
                    if (lv == 0 && S.sfirst[(size_t)t + 1] - S.sfirst[(size_t)t] == 1) continue;
                    if (warp_level(t) == (pass == 1)) bsn.push_back(t);
                }
            }
            bstep.push_back((int)bsn.size());
            i = j;
        }
        L->nbstep = S.nlevels;
        L->bstride = (S.panel_size + S.N + 15) / 16 * 16;
    }
    cudaStream_t s = h->stream;
    up(L->bsn, bsn, s); up(L->bstep, bstep, s);
    up(L->sfirst, S.sfirst, s); up(L->rows, S.rows, s); up(L->order, S.order, s);
    up(L->task_start, tstart, s); up(L->task_cnt, tcnt, s);
    up(L->usrc, S.usrc, s); up(L->ua, S.ua, s); up(L->ub, S.ub, s); up(L->rel, S.rel, s);
    up(L->ttgt, S.ttgt, s); up(L->P, S.P, s); up(L->pinv, S.pinv, s); up(L->asrc, S.asrc, s);
    up(L->rptr, S.rptr, s); up(L->poff, S.poff, s); up(L->uptr, S.uptr, s); up(L->urel, S.urel, s);
    up(L->tptr, S.tptr, s); up(L->aslot, S.aslot, s); up(L->aptr, S.aptr, s);
    up(L->umid, S.umid, s); up(L->sn_of, S.sn_of, s);
    up(L->lcptr, S.lcptr, s); up(L->lc_src, S.lc_src, s); up(L->lc_rel, S.lc_rel, s);
    up(L->lc_cnt, S.lc_cnt, s); up(L->lc_ldd, S.lc_ldd, s); up(L->lc_wd, S.lc_wd, s); up(L->lc_fd, S.lc_fd, s);
    L->naslot = (int64_t)S.aslot.size();
    L->panels.alloc((size_t)S.panel_size + 8);
    L->D.alloc((size_t)S.N + 8);
    L->Y.alloc((size_t)S.N + 8);
    L->done_f.alloc((size_t)S.nsuper + 8); L->done_s.alloc((size_t)S.nsuper + 8); L->done_b.alloc((size_t)S.nsuper + 8);
    L->done_f.zero(s); L->done_s.zero(s); L->done_b.zero(s);
    L->ticket.alloc(8); L->fail.alloc(8);
#ifdef FPSB_LDLT_TIMERS
    L->tstamp.alloc((size_t)3 * S.nsuper + 8);
    L->tstamp.zero(s);
#endif
    L->ticket.zero(s); L->fail.zero(s);
    FPSB_CUDA(cudaStreamSynchronize(s));
    PlanDev &D = L->dev;
    D.N = S.N; D.nsuper = S.nsuper; D.ntasks = L->ntasks;
    D.sfirst = L->sfirst.p; D.rptr = L->rptr.p; D.rows = L->rows.p; D.poff = L->poff.p; D.order = L->order.p;
    D.task_start = L->task_start.p; D.task_cnt = L->task_cnt.p;
    D.uptr = L->uptr.p; D.usrc = L->usrc.p; D.ua = L->ua.p; D.ub = L->ub.p; D.urel = L->urel.p; D.rel = L->rel.p;
    D.tptr = L->tptr.p; D.ttgt = L->ttgt.p; D.P = L->P.p;
    D.umid = L->umid.p; D.sn_of = L->sn_of.p;
    D.lcptr = L->lcptr.p; D.lc_src = L->lc_src.p; D.lc_rel = L->lc_rel.p;
    D.lc_cnt = L->lc_cnt.p; D.lc_ldd = L->lc_ldd.p; D.lc_wd = L->lc_wd.p; D.lc_fd = L->lc_fd.p;
    D.ntasks_leaf = L->ntasks_leaf;
    D.panels = L->panels.p; D.D = L->D.p; D.Y = L->Y.p;
    D.done_f = L->done_f.p; D.done_s = L->done_s.p; D.done_b = L->done_b.p;
    D.ticket = L->ticket.p; D.fail = L->fail.p;
    D.tstamp = L->tstamp.p;
    D.n_d = (int)h->nvar;
    D.tol = L->opts.ldlt_tol; D.r1 = L->opts.ldlt_r1; D.r2 = L->opts.ldlt_r2;
    D.dynamic_reg = (D.r1 != 0.0) || (D.r2 != 0.0);
}

void ldlt_free(Handle *h) {
    if (h->ldlt) { delete h->ldlt; h->ldlt = nullptr; }
}

void ldlt_factorize(Handle *h, double delta, int *factorized) {
    LdltPlan *L = h->ldlt;
    cudaStream_t s = h->stream;
    L->factorized = false;
    L->have_factor = false;
    L->epoch += 1;
    FPSB_CUDA(cudaMemsetAsync(L->panels.p, 0, (size_t)(L->S.panel_size + 8) * sizeof(double), s));
    FPSB_CUDA(cudaMemsetAsync(L->ticket.p, 0, 8 * sizeof(int), s));
    FPSB_CUDA(cudaMemsetAsync(L->fail.p, 0, sizeof(int), s));
    if (L->naslot) {
        int grid = (int)((L->naslot + 255) / 256);
        assemble_kernel<<<grid, 256, 0, s>>>(L->naslot, L->aslot.p, L->aptr.p, L->asrc.p, h->coo_vals.p,
                                             (int)h->nvar, h->nnzj, delta, L->panels.p);
        h->launches += 1;
    }
    const int nl = L->ntasks_leaf, nn = L->ntasks - L->ntasks_leaf, N = L->S.N;
    const int nleaf = L->S.nleaf;
    if (nleaf) {  // leaves: no dependencies at all
        leaf1_factor_kernel<<<(int)(((int64_t)nleaf * 8 + 255) / 256), 256, 0, s>>>(L->dev, nleaf);
        h->launches += 1;
    }
    if (nl) launch_phase<0>(h, L->dev, nl, L->epoch, 0, nl, 0, 1, true);
    if (nn) {
        if (nleaf) {
            leaf_update_kernel<<<(int)(((int64_t)N * 8 + 255) / 256), 256, 0, s>>>(L->dev);
            h->launches += 1;
        }
        launch_phase<0>(h, L->dev, nn, L->epoch, nl, L->ntasks, 1, 0);
    }
    int fail = 0;
    FPSB_CUDA(cudaMemcpyAsync(&fail, L->fail.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    FPSB_CUDA(cudaStreamSynchronize(s));
    FPSB_CUDA(cudaGetLastError());
    if (fail == -2) {
        set_error("ldlt_factorize: dependency wait timed out (internal scheduling error)");
        throw CudaFail{FPSB_ECUDA};
    }
    L->have_factor = true;
    L->factorized = (fail == 0);
    if (factorized) *factorized = L->factorized ? 1 : 0;
}

// kind 0: mixed right-hand sides, 1: least squares
void ldlt_solve2(Handle *h, int kind, const double *rhs1, const double *rhs2, double *p1, double *q1,
                 double *p2, double *q2, int *factorized) {
    LdltPlan *L = h->ldlt;
    cudaStream_t s = h->stream;
    const int N = L->S.N, nvar = (int)h->nvar, ncon = (int)h->ncon;
    if (factorized) *factorized = L->factorized ? 1 : 0;
    if (N == 0) return;
    const int grid = (N + 255) / 256;
    if (!L->factorized) {
        passthrough_kernel<<<(std::max(nvar, ncon) + 255) / 256, 256, 0, s>>>(nvar, ncon, kind, rhs1, rhs2, p1, q1, p2, q2);
        h->launches += 1;
        return;
    }
    L->epoch += 1;
    FPSB_CUDA(cudaMemsetAsync(L->ticket.p, 0, 8 * sizeof(int), s));
    load_rhs_kernel<<<grid, 256, 0, s>>>(N, nvar, kind, L->P.p, rhs1, rhs2, L->Y.p);
    const int nl = L->ntasks_leaf, nn = L->ntasks - L->ntasks_leaf;
    // forward: leaves (independent) -> leaf contributions by target row -> the rest (dependency driven)
    if (nl) launch_phase<1>(h, L->dev, nl, L->epoch, 0, nl, 0, 1, true);
    if (nn) {
        if (L->S.nleaf) { leaf_fwd_update_kernel<<<grid, 256, 0, s>>>(L->dev); h->launches += 1; }
        launch_phase<1>(h, L->dev, nn, L->epoch, nl, L->ntasks, 1, 0);
        // backward: the non-leaf part in reverse dependency order, then all leaves at once
        launch_phase<2>(h, L->dev, nn, L->epoch, nl, L->ntasks, 2, 0);
    }
    if (nl) launch_phase<2>(h, L->dev, nl, L->epoch, 0, nl, 3, 1, true);
    if (L->S.nleaf) { leaf1_bwd_kernel<<<(int)(((int64_t)L->S.nleaf * 8 + 255) / 256), 256, 0, s>>>(L->dev, L->S.nleaf); h->launches += 1; }
    store_sol_kernel<<<grid, 256, 0, s>>>(N, nvar, L->pinv.p, L->Y.p, p1, q1, p2, q2);
    h->launches += 2;
    FPSB_CUDA(cudaGetLastError());
}

template <int MODE>
static void launch_batch(Handle *h, const PlanDev &P, BatchDev &B) {
    LdltPlan *L = h->ldlt;
    const size_t smem = (size_t)kBatchDoubles * sizeof(double);
    FPSB_CUDA(cudaFuncSetAttribute(ldlt_batch_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    FPSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ldlt_batch_kernel<MODE>, kLdltBlock, smem));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(B.ninst, (int64_t)h->num_sms * std::max(per_sm, 1)));
    const int64_t yrows = (int64_t)grid * P.N;
    if (L->bY_rows < yrows) { L->bY.alloc((size_t)yrows + 8); L->bY_rows = yrows; }
    B.Y = L->bY.p;
    ldlt_batch_kernel<MODE><<<grid, kLdltBlock, smem, h->stream>>>(P, B);
    h->launches += 1;
    FPSB_CUDA(cudaGetLastError());
}

// kind 0: refactor every instance and solve (the factors stay in the factor store), 1: least squares with the factors of
// the last kind-0 call.  Device pointers; factorized == NULL: the status is left in L->bok only.
static void ldlt_batch(Handle *h, int kind, int64_t ninst, const double *jvals, const double *delta, const double *rhs1,
                       const double *rhs2, double *p1, double *q1, double *p2, double *q2, int *factorized) {
    LdltPlan *L = h->ldlt;
    if (kind == 0) {
        L->bninst = -1;
        // grown, never shrunk; the old contents are not kept (this call refactors every instance)
        if (L->bstore_inst < ninst) {
            L->bstore.release(); L->bstore_inst = 0;
            L->bstore.alloc((size_t)ninst * (size_t)L->bstride + 8);
            L->bstore_inst = ninst;
        }
        if (L->bok_inst < ninst) {
            L->bok.release(); L->bok_inst = 0;
            L->bok.alloc((size_t)ninst + 8);
            L->bok_inst = ninst;
        }
    }
    if (!factorized) factorized = L->bok.p;
    BatchDev B{};
    B.sn = L->bsn.p; B.step = L->bstep.p; B.nstep = L->nbstep; B.nleaf = L->S.nleaf;
    B.ninst = ninst; B.stride = L->bstride; B.psize = L->S.panel_size;
    B.aslot = L->aslot.p; B.aptr = L->aptr.p; B.asrc = L->asrc.p; B.naslot = L->naslot; B.nnzj = h->nnzj;
    B.pinv = L->pinv.p;
    B.store = L->bstore.p; B.ok = L->bok.p;
    B.jvals = jvals; B.delta = delta; B.rhs1 = rhs1; B.rhs2 = rhs2;
    B.p1 = p1; B.q1 = q1; B.p2 = p2; B.q2 = q2; B.factorized = factorized;
    B.kind = kind;
    const int mode = ldlt_mode();
    if (mode == 0) launch_batch<0>(h, L->dev, B);
    else if (mode == 2) launch_batch<2>(h, L->dev, B);
    else launch_batch<1>(h, L->dev, B);
    if (kind == 0) L->bninst = ninst;
}

}  // namespace fpsb

// ------------------------------------------------------------------------------------------------
// C ABI: LDLt entry points
// ------------------------------------------------------------------------------------------------
using namespace fpsb;

#define REQ(cond, code, msg) do { if (!(cond)) { fpsb::set_error(msg); return code; } } while (0)
#define TRY_ try {
#define CATCH_ } catch (const fpsb::CudaFail &f) { return f.code; } \
    catch (const std::bad_alloc &) { fpsb::set_error("out of memory"); return FPSB_ENOMEM; } \
    catch (const std::exception &e) { fpsb::set_error("%s", e.what()); return FPSB_ECUDA; } \
    catch (...) { fpsb::set_error("unexpected C++ exception"); return FPSB_ECUDA; }

struct fpsb_symbolic_s { Symbolic S; };

extern "C" {

int fpsb_ldlt_default_opts(fpsb_ldlt_opts *o) {
    REQ(o, FPSB_EINVAL, "NULL opts");
    const double se = 1.4901161193847656e-08;
    o->ldlt_tol = se; o->ldlt_r1 = se; o->ldlt_r2 = -se;
    return FPSB_OK;
}

// host-only symbolic analysis (no CUDA needed): used by fpsb_ldlt_analyze and by the CPU tests
int fpsb_symbolic_create(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow, const int64_t *jcol,
                         int index_base, const int64_t *P, fpsb_symbolic *out) {
    REQ(out, FPSB_EINVAL, "NULL out");
    *out = nullptr;
    REQ(nvar >= 0 && ncon >= 0 && nnzj >= 0 && (nnzj == 0 || (jrow && jcol)), FPSB_EINVAL, "bad arguments");
    TRY_
    std::vector<int64_t> r((size_t)nnzj), c((size_t)nnzj), Pz;
    for (int64_t k = 0; k < nnzj; ++k) {
        r[(size_t)k] = jrow[k] - index_base; c[(size_t)k] = jcol[k] - index_base;
        REQ(r[(size_t)k] >= 0 && r[(size_t)k] < ncon && c[(size_t)k] >= 0 && c[(size_t)k] < nvar, FPSB_EINVAL,
            "Jacobian index out of range");
    }
    if (P) { Pz.resize((size_t)(nvar + ncon)); for (int64_t k = 0; k < nvar + ncon; ++k) Pz[(size_t)k] = P[k] - index_base; }
    fpsb_symbolic_s *S = new fpsb_symbolic_s();
    try {
        analyze((int)nvar, (int)ncon, nnzj, r.data(), c.data(), P ? Pz.data() : nullptr, S->S);
    } catch (const std::invalid_argument &e) {
        delete S;
        fpsb::set_error("fpsb_symbolic_create: %s", e.what());
        return FPSB_EINVAL;
    } catch (...) { delete S; throw; }
    *out = S;
    return FPSB_OK;
    CATCH_
}
int fpsb_symbolic_destroy(fpsb_symbolic s) { delete s; return FPSB_OK; }

// host-only: dissection ordering of K (P_out: nvar+ncon entries, index_base-based)
int fpsb_order_dissection(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow, const int64_t *jcol,
                          int index_base, int nparts, int64_t *P_out) {
    REQ(P_out && nvar >= 0 && ncon >= 0 && nnzj >= 0 && (nnzj == 0 || (jrow && jcol)), FPSB_EINVAL, "bad arguments");
    TRY_
    std::vector<int64_t> r((size_t)nnzj), c((size_t)nnzj);
    for (int64_t k = 0; k < nnzj; ++k) {
        r[(size_t)k] = jrow[k] - index_base; c[(size_t)k] = jcol[k] - index_base;
        REQ(r[(size_t)k] >= 0 && r[(size_t)k] < ncon && c[(size_t)k] >= 0 && c[(size_t)k] < nvar, FPSB_EINVAL,
            "Jacobian index out of range");
    }
    std::vector<int64_t> Gp;
    std::vector<int> Gi, P;
    build_kkt_graph((int)nvar, (int)ncon, nnzj, r.data(), c.data(), Gp, Gi);
    dissection_order((int)(nvar + ncon), Gp, Gi, nparts, P);
    for (size_t k = 0; k < P.size(); ++k) P_out[k] = P[k] + index_base;
    return FPSB_OK;
    CATCH_
}

static void sym_sizes(const Symbolic &S, int64_t *N, int64_t *lnz) {
    if (N) *N = S.N;
    if (lnz) *lnz = S.Lp.empty() ? 0 : S.Lp[(size_t)S.N];
}
static void sym_get(const Symbolic &S, int64_t *P, int64_t *parent, int64_t *Lnz, int64_t *Lp, int64_t *Li) {
    const int N = S.N;
    for (int k = 0; k < N; ++k) {
        if (P) P[k] = S.P[(size_t)k];
        if (parent) parent[k] = S.parent[(size_t)k];
        if (Lnz) Lnz[k] = S.Lp[(size_t)k + 1] - S.Lp[(size_t)k];
    }
    if (Lp) for (int k = 0; k <= N; ++k) Lp[k] = S.Lp[(size_t)k];
    if (Li) for (size_t p = 0; p < S.Li.size(); ++p) Li[p] = S.Li[p];
}
static void sym_plan(const Symbolic &S, int64_t *nsuper, int64_t *panel_nnz, int64_t *npairs, double *flops,
                     int64_t *nlevels, int64_t *nleaf) {
    if (nlevels) *nlevels = S.nlevels;
    if (nleaf) *nleaf = S.nleaf;
    if (nsuper) *nsuper = S.nsuper;
    if (panel_nnz) *panel_nnz = S.panel_size;
    if (npairs) *npairs = (int64_t)S.usrc.size();
    if (flops) *flops = S.flops;
}
int fpsb_symbolic_sizes(fpsb_symbolic s, int64_t *N, int64_t *lnz) {
    REQ(s, FPSB_EINVAL, "NULL symbolic");
    sym_sizes(s->S, N, lnz);
    return FPSB_OK;
}
int fpsb_symbolic_get(fpsb_symbolic s, int64_t *P, int64_t *parent, int64_t *Lnz, int64_t *Lp, int64_t *Li) {
    REQ(s, FPSB_EINVAL, "NULL symbolic");
    sym_get(s->S, P, parent, Lnz, Lp, Li);
    return FPSB_OK;
}
int fpsb_symbolic_plan_info(fpsb_symbolic s, int64_t *nsuper, int64_t *panel_nnz, int64_t *npairs, double *flops,
                            int64_t *nlevels, int64_t *nleaf) {
    REQ(s, FPSB_EINVAL, "NULL symbolic");
    sym_plan(s->S, nsuper, panel_nnz, npairs, flops, nlevels, nleaf);
    return FPSB_OK;
}



/* debug builds (-DFPSB_LDLT_TIMERS; not in fpsb.h): per dependency level, the latest completion time (us after the
 * earliest stamp of the phase) of the last factorisation / forward / backward sweep */
int fpsb_debug_ldlt_level_times(fpsb_handle hh, int phase, double *out_us, int cap) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h || !h->ldlt || !h->ldlt->tstamp.p || phase < 0 || phase > 2) return -1;
    const Symbolic &S = h->ldlt->S;
    std::vector<unsigned long long> ts((size_t)S.nsuper);
    cudaMemcpy(ts.data(), h->ldlt->tstamp.p + (size_t)phase * S.nsuper, ts.size() * 8, cudaMemcpyDeviceToHost);
    unsigned long long t0 = ~0ull;
    for (int t = 0; t < S.nsuper; ++t) if (ts[(size_t)t] && S.level[(size_t)t] > 0) t0 = std::min(t0, ts[(size_t)t]);
    std::vector<unsigned long long> mx((size_t)S.nlevels + 1, 0);
    for (int t = 0; t < S.nsuper; ++t) mx[(size_t)S.level[(size_t)t]] = std::max(mx[(size_t)S.level[(size_t)t]], ts[(size_t)t]);
    int nl = 0;
    for (int l = 0; l <= S.nlevels && l < cap; ++l, ++nl) out_us[l] = mx[(size_t)l] >= t0 ? 1e-3 * (double)(mx[(size_t)l] - t0) : 0.0;
    return nl;
}

/* debug (not in fpsb.h): per-level statistics of the supernodal plan on stderr */
void fpsb_debug_plan_dump(fpsb_symbolic sy) {
    if (!sy) return;
    const Symbolic &S = sy->S;
    struct Lv { long long cnt = 0, sw = 0, snr = 0, pairs = 0; int maxw = 0, maxnr = 0, maxpairs = 0; double upd = 0, self = 0; };
    std::vector<Lv> lv((size_t)S.nlevels + 1);
    for (int t = 0; t < S.nsuper; ++t) {
        Lv &l = lv[(size_t)S.level[(size_t)t]];
        const int w = S.sfirst[(size_t)t + 1] - S.sfirst[(size_t)t];
        const int nr = (int)(S.rptr[(size_t)t + 1] - S.rptr[(size_t)t]);
        l.cnt++; l.sw += w; l.snr += nr; l.maxw = std::max(l.maxw, w); l.maxnr = std::max(l.maxnr, nr);
        const int np = (int)(S.umid[(size_t)t] - S.uptr[(size_t)t]);
        l.pairs += np; l.maxpairs = std::max(l.maxpairs, np);
        for (int64_t q = S.uptr[(size_t)t]; q < S.umid[(size_t)t]; ++q) {
            const int d = S.usrc[(size_t)q];
            const int wd = S.sfirst[(size_t)d + 1] - S.sfirst[(size_t)d];
            const int nrd = (int)(S.rptr[(size_t)d + 1] - S.rptr[(size_t)d]);
            l.upd += 2.0 * (double)(nrd - S.ua[(size_t)q]) * (double)(S.ub[(size_t)q] - S.ua[(size_t)q]) * wd;
        }
        l.self += (double)w * w * w / 3.0 + (double)nr * w * w;
    }
    fprintf(stderr, "level count sum_w max_w sum_nr max_nr pairs maxpairs upd_MFLOP self_MFLOP\n");
    for (size_t i = 0; i < lv.size(); ++i) {
        const Lv &l = lv[i];
        if (!l.cnt) continue;
        fprintf(stderr, "%3zu %8lld %8lld %3d %9lld %5d %7lld %4d %10.2f %10.2f\n", i, l.cnt, l.sw, l.maxw, l.snr, l.maxnr, l.pairs, l.maxpairs,
                l.upd * 1e-6, l.self * 1e-6);
    }
}

int fpsb_ldlt_analyze(fpsb_handle hh, const int64_t *P, int index_base, const fpsb_ldlt_opts *opts) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h, FPSB_EINVAL, "NULL handle");
    REQ(index_base == 0 || index_base == 1, FPSB_EINVAL, "index_base must be 0 or 1");
    TRY_
    FPSB_CUDA(cudaSetDevice(h->device));
    std::vector<int64_t> Pz;
    if (P) { Pz.resize((size_t)(h->nvar + h->ncon)); for (size_t k = 0; k < Pz.size(); ++k) Pz[k] = P[k] - index_base; }
    ldlt_analyze(h, P ? Pz.data() : nullptr, opts);
    return FPSB_OK;
    CATCH_
}
int fpsb_ldlt_symbolic_sizes(fpsb_handle hh, int64_t *N, int64_t *lnz) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    sym_sizes(h->ldlt->S, N, lnz);
    return FPSB_OK;
}
int fpsb_ldlt_get_symbolic(fpsb_handle hh, int64_t *P, int64_t *parent, int64_t *Lnz, int64_t *Lp, int64_t *Li) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    sym_get(h->ldlt->S, P, parent, Lnz, Lp, Li);
    return FPSB_OK;
}
int fpsb_ldlt_plan_info(fpsb_handle hh, int64_t *nsuper, int64_t *panel_nnz, int64_t *npairs, double *flops,
                        int64_t *nlevels, int64_t *nleaf) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    sym_plan(h->ldlt->S, nsuper, panel_nnz, npairs, flops, nlevels, nleaf);
    return FPSB_OK;
}
int fpsb_ldlt_factorize(fpsb_handle hh, double delta, int *factorized) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    REQ(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    TRY_
    FPSB_CUDA(cudaSetDevice(h->device));
    ldlt_factorize(h, delta, factorized);
    return FPSB_OK;
    CATCH_
}
int fpsb_ldlt_get_factor(fpsb_handle hh, double *Lx, double *D) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    REQ(h->ldlt->have_factor, FPSB_ESTATE, "no numeric factorisation available");
    TRY_
    FPSB_CUDA(cudaSetDevice(h->device));
    LdltPlan *L = h->ldlt;
    const Symbolic &S = L->S;
    std::vector<double> panels((size_t)S.panel_size + 1), Dh((size_t)S.N + 1);
    FPSB_CUDA(cudaMemcpy(panels.data(), L->panels.p, (size_t)S.panel_size * sizeof(double), cudaMemcpyDeviceToHost));
    FPSB_CUDA(cudaMemcpy(Dh.data(), L->D.p, (size_t)S.N * sizeof(double), cudaMemcpyDeviceToHost));
    if (D) memcpy(D, Dh.data(), (size_t)S.N * sizeof(double));
    if (Lx) {
        for (int s = 0; s < S.nsuper; ++s) {
            const int f = S.sfirst[(size_t)s], l = S.sfirst[(size_t)s + 1] - 1, w = l - f + 1;
            const int nr = (int)(S.rptr[(size_t)s + 1] - S.rptr[(size_t)s]);
            const int ld = w + nr;
            const int *R = S.rows.data() + S.rptr[(size_t)s];
            const double *pan = panels.data() + S.poff[(size_t)s];
            for (int j = f; j <= l; ++j) {
                for (int64_t p = S.Lp[(size_t)j]; p < S.Lp[(size_t)j + 1]; ++p) {
                    const int r = S.Li[(size_t)p];
                    int lr;
                    if (r <= l) lr = r - f;
                    else lr = w + (int)(std::lower_bound(R, R + nr, r) - R);
                    Lx[p] = pan[(size_t)(j - f) * ld + lr];
                }
            }
        }
    }
    return FPSB_OK;
    CATCH_
}

static int ldlt_solve_api(fpsb_handle hh, int kind, bool refactor, double delta, const double *rhs1,
                          const double *rhs2, double *p1, double *q1, double *p2, double *q2, int loc,
                          int *factorized) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    REQ(rhs1 && rhs2 && p1 && q1 && p2 && q2, FPSB_EINVAL, "NULL argument");
    REQ(!refactor || h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    TRY_
    FPSB_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)h->nvar, m = (size_t)h->ncon;
    const size_t n2 = kind == 0 ? m : n;
    int ok = 0;
    if (loc == FPSB_DEVICE) caller_order_in(h);      // the caller's kernels wrote the right-hand sides on its own stream
    if (refactor) ldlt_factorize(h, delta, &ok);
    // host staging (same scheme as the iterative path)
    double *d_in = nullptr, *d_out = nullptr, *pinned = nullptr;
    const double *d1 = rhs1, *d2 = rhs2;
    double *o1 = p1, *o2 = q1, *o3 = p2, *o4 = q2;
    if (loc == FPSB_HOST) {
        if (h->stage_in.n < n + n2 + 8) h->stage_in.alloc(n + n2 + 8);
        if (h->stage_out.n < 2 * (n + m) + 8) h->stage_out.alloc(2 * (n + m) + 8);
        const size_t need = n + n2 + 2 * (n + m) + 8;
        if (h->pin_count < need) {
            if (h->pin) cudaFreeHost(h->pin);
            h->pin = nullptr; h->pin_count = 0;
            FPSB_CUDA(cudaMallocHost((void **)&h->pin, need * sizeof(double)));
            h->pin_count = need;
        }
        pinned = h->pin;
        memcpy(pinned, rhs1, n * sizeof(double));
        memcpy(pinned + n, rhs2, n2 * sizeof(double));
        d_in = h->stage_in.p; d_out = h->stage_out.p;
        FPSB_CUDA(cudaMemcpyAsync(d_in, pinned, (n + n2) * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d1 = d_in; d2 = d_in + n;
        o1 = d_out; o2 = d_out + n; o3 = d_out + n + m; o4 = d_out + 2 * n + m;
    }
    ldlt_solve2(h, kind, d1, d2, o1, o2, o3, o4, &ok);
    if (loc == FPSB_HOST) {
        double *res = pinned + n + n2;
        FPSB_CUDA(cudaMemcpyAsync(res, d_out, 2 * (n + m) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
        memcpy(p1, res, n * sizeof(double));
        memcpy(q1, res + n, m * sizeof(double));
        memcpy(p2, res + n + m, n * sizeof(double));
        memcpy(q2, res + 2 * n + m, m * sizeof(double));
    } else {
        caller_order_out(h);
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
    }
    FPSB_CUDA(cudaGetLastError());
    int fail = 0;
    FPSB_CUDA(cudaMemcpy(&fail, h->ldlt->fail.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (fail == -2) { fpsb::set_error("ldlt solve: dependency wait timed out"); return FPSB_ECUDA; }
    if (factorized) *factorized = ok;
    return FPSB_OK;
    CATCH_
}

int fpsb_ldlt_solve_two_mixed(fpsb_handle h, double delta, const double *rhs1, const double *rhs2, double *p1,
                              double *q1, double *p2, double *q2, int loc, int *factorized) {
    return ldlt_solve_api(h, 0, true, delta, rhs1, rhs2, p1, q1, p2, q2, loc, factorized);
}
int fpsb_ldlt_solve_two_least_squares(fpsb_handle h, const double *rhs1, const double *rhs2, double *p1,
                                      double *q1, double *p2, double *q2, int loc, int *factorized) {
    return ldlt_solve_api(h, 1, false, 0.0, rhs1, rhs2, p1, q1, p2, q2, loc, factorized);
}

static int ldlt_batch_api(fpsb_handle hh, int kind, int64_t ninst, const double *jvals, const double *delta,
                          const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2, double *q2,
                          int *factorized, int loc) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQ(h && h->ldlt, FPSB_ESTATE, "fpsb_ldlt_analyze has not been called");
    REQ(ninst >= 0, FPSB_EINVAL, "negative ninst");
    REQ(loc == FPSB_HOST || loc == FPSB_DEVICE, FPSB_EINVAL, "loc must be FPSB_HOST or FPSB_DEVICE");
    if (ninst == 0) return FPSB_OK;
    REQ(rhs1 && rhs2 && p1 && q1 && p2 && q2 && factorized && (kind == 1 || (jvals && delta)), FPSB_EINVAL, "NULL argument");
    REQ(kind == 0 || h->ldlt->bninst == ninst, FPSB_ESTATE,
        "no batched factorisation of this many instances (call fpsb_ldlt_batch_solve_two_mixed first)");
    TRY_
    FPSB_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)h->nvar, m = (size_t)h->ncon, ni = (size_t)ninst, nz = (size_t)h->nnzj;
    const size_t n2 = kind == 0 ? m : n;
    if (loc == FPSB_DEVICE) {
        caller_order_in(h);      // the caller's kernels wrote the inputs on its own stream
        ldlt_batch(h, kind, ninst, jvals, delta, rhs1, rhs2, p1, q1, p2, q2, factorized);
        caller_order_out(h);
        return FPSB_OK;
    }
    // host buffers: staged through the handle's pinned area and device staging buffers (grown, never shrunk)
    const size_t nin = (kind == 0 ? ni * nz + ni : 0) + ni * n + ni * n2;
    const size_t nout = ni * 2 * (n + m);
    const size_t nfac = (ni + 1) / 2;           // the int status after the doubles
    if (h->stage_in.n < nin + 8) h->stage_in.alloc(nin + 8);
    if (h->stage_out.n < nout + 8) h->stage_out.alloc(nout + 8);
    const size_t need = nin + nout + nfac + 8;
    if (h->pin_count < need) {
        if (h->pin) cudaFreeHost(h->pin);
        h->pin = nullptr; h->pin_count = 0;
        FPSB_CUDA(cudaMallocHost((void **)&h->pin, need * sizeof(double)));
        h->pin_count = need;
    }
    double *pin = h->pin, *din = h->stage_in.p, *dout = h->stage_out.p;
    size_t off = 0;
    const double *dj = nullptr, *dd = nullptr;
    if (kind == 0) {
        memcpy(pin, jvals, ni * nz * sizeof(double)); dj = din; off = ni * nz;
        memcpy(pin + off, delta, ni * sizeof(double)); dd = din + off; off += ni;
    }
    memcpy(pin + off, rhs1, ni * n * sizeof(double));
    const double *d1 = din + off; off += ni * n;
    memcpy(pin + off, rhs2, ni * n2 * sizeof(double));
    const double *d2 = din + off;
    FPSB_CUDA(cudaMemcpyAsync(din, pin, nin * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    double *o1 = dout, *o2 = o1 + ni * n, *o3 = o2 + ni * m, *o4 = o3 + ni * n;
    ldlt_batch(h, kind, ninst, dj, dd, d1, d2, o1, o2, o3, o4, nullptr);
    double *res = pin + nin;
    int *fres = reinterpret_cast<int *>(res + nout);
    FPSB_CUDA(cudaMemcpyAsync(res, dout, nout * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    FPSB_CUDA(cudaMemcpyAsync(fres, h->ldlt->bok.p, ni * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(p1, res, ni * n * sizeof(double));
    memcpy(q1, res + ni * n, ni * m * sizeof(double));
    memcpy(p2, res + ni * (n + m), ni * n * sizeof(double));
    memcpy(q2, res + ni * (2 * n + m), ni * m * sizeof(double));
    memcpy(factorized, fres, ni * sizeof(int));
    return FPSB_OK;
    CATCH_
}

int fpsb_ldlt_batch_solve_two_mixed(fpsb_handle h, int64_t ninst, const double *jvals, const double *delta,
                                    const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2,
                                    double *q2, int *factorized, int loc) {
    return ldlt_batch_api(h, 0, ninst, jvals, delta, rhs1, rhs2, p1, q1, p2, q2, factorized, loc);
}
int fpsb_ldlt_batch_solve_two_least_squares(fpsb_handle h, int64_t ninst, const double *rhs1, const double *rhs2,
                                            double *p1, double *q1, double *p2, double *q2, int *factorized, int loc) {
    return ldlt_batch_api(h, 1, ninst, nullptr, nullptr, rhs1, rhs2, p1, q1, p2, q2, factorized, loc);
}

}  // extern "C"
