// fpsb_internal.h — shared declarations of libfpsb200 (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/fpsb.h"

namespace fpsb {

// ------------------------------------------------------------------------------------------------
// error plumbing: no exceptions cross the C ABI
// ------------------------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
struct CudaFail { int code; };

#define FPSB_CUDA(call)                                                                  \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            fpsb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                \
                            cudaGetErrorString(e__));                                    \
            throw fpsb::CudaFail{FPSB_ECUDA};                                            \
        }                                                                                \
    } while (0)

template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    void alloc(size_t count) {
        release();
        const cudaError_t e = cudaMalloc((void **)&p, (count ? count : 1) * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr; n = 0;
            cudaGetLastError();
            fpsb::set_error("cudaMalloc of %zu bytes failed: %s", (count ? count : 1) * sizeof(T), cudaGetErrorString(e));
            throw fpsb::CudaFail{e == cudaErrorMemoryAllocation ? FPSB_ENOMEM : FPSB_ECUDA};
        }
        n = count;
    }
    void zero(cudaStream_t s) { if (p) FPSB_CUDA(cudaMemsetAsync(p, 0, (n ? n : 1) * sizeof(T), s)); }
    void upload(const T *h, size_t count, cudaStream_t s) {
        if (count) FPSB_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void from(const std::vector<T> &h, cudaStream_t s) { alloc(h.size() + 8); upload(h.data(), h.size(), s); }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
};

// ------------------------------------------------------------------------------------------------
// CSR operator on the device with its row-block tiling (one CTA per row block)
// ------------------------------------------------------------------------------------------------
constexpr int kBlock = 256;       // threads per CTA (8 warps, one SELL slice per warp at a time)

// Operator stored as tiled SELL-32 (+ CSR of the few long rows)
struct CsrDev {
    int nrows = 0, ncols = 0;
    int64_t nnz = 0;
    int64_t padded = 0;           // stored entries including padding
    int nlong = 0;
    DevBuf<int> sperm, tperm0;                 // sperm: stored entry -> COO index (-1 = padding); first entry per tile
    DevBuf<unsigned char> tbuf;                // tile blocks [values | indices | lane -> row map], back to back
    DevBuf<unsigned char> tiles;               // TileMeta[ntiles] (fpsb_krylov.cu)
    DevBuf<unsigned char> rowflag;             // 1 = long row, 2 = raw row (row-partitioned runs)
    bool has_raw_rows = false;
    DevBuf<int> wsegs;                         // multi-segment gather windows: 4 x {start, offset | length << 16} per tile
    int nseg_tiles = 0, nwin_tiles = 0;        // tiles whose window has more than one segment / tiles with a window at all
    int ntiles = 0, win_cap = 0, blk_cap = 0, stage_bytes = 0, nstage = 0;
    DevBuf<int> long_row, long_rp, long_col, long_perm;
    DevBuf<double> long_val;
    int grid = 0;                 // persistent CTAs of the tile kernel (long rows: nlong extra CTAs of their own kernel)
};

// ------------------------------------------------------------------------------------------------
// Krylov engine state (device-resident scalars; one per "slot" = one right-hand side)
// ------------------------------------------------------------------------------------------------
enum Algo { ALGO_NONE = 0, ALGO_LSQR = 1, ALGO_CRAIG = 2, ALGO_MINRES = 3, ALGO_CGLS = 4 };

struct SlotState {
    // configuration
    int algo, itmax, sqd, pad0;
    double lambda, atol, rtol, axtol, btol, etol, ctol, mscale;
    // control
    int active, iter, solved, inconsistent, status, first, pend, beta_zero;
    int tired, ill_mach, ill_lim, zero_resid, fwd_err, pad1, pad2, pad3;
    // shared scalars
    double beta1, alpha, beta, Anorm2, Anorm, Acond, xNorm, xNorm2, dNorm2;
    double rNorm, ArNorm, ArNorm0, phibar, rhobar, res2, xENorm2, err_lbnd, err_vec[5];
    double c, s, rho, phi, psi, tau, c2, s2, z;
    // coefficients consumed by the vector kernels
    double su, sv, sigma, tr_prev;
    // CRAIG
    double theta, xi, deltag, rho_prev, c1, s1, s2g, trw, xr, beta1sq, eps_c;
    // MINRES
    double oldbeta, deltabar, eps_, rhs1, rhs2, gmax, gmin, cs, sn, delta, gamma, gammabar, root, tol;
    // CGLS
    double gamma_c, pp, delta_c, beta_c, bnorm;
};

struct IterWs;     // defined in fpsb_krylov.cu
struct LdltPlan;   // defined in fpsb_ldlt.cu
struct DistCtx;    // defined in fpsb_dist.inl (row-partitioned multi-GPU runs)
struct FpWs;       // defined in fpsb_fpnlp.cu
struct ExtrasWs;   // defined in fpsb_extras_batch.inl

struct Handle {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // FPSB_DEVICE callers: the stream their own kernels run on (default: the legacy default stream, what
    // PyTorch uses).  Every entry that takes device pointers orders h->stream after it on the way in and
    // it after h->stream on the way out (the handle's stream is non-blocking: nothing is implicit).
    cudaStream_t caller_stream = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    int64_t nvar = 0, ncon = 0, nnzj = 0;
    std::vector<int64_t> jrow, jcol;          // 0-based COO structure (host copy)
    CsrDev A, At;                             // A (ncon x nvar) and A' (nvar x ncon)
    DevBuf<double> coo_vals;                  // jac_coord values in COO order
    bool have_vals = false;
    int64_t launches = 0;
    // host staging (pinned)
    double *pin = nullptr;
    size_t pin_count = 0;
    DevBuf<double> stage_in, stage_out;
    IterWs *iter = nullptr;
    LdltPlan *ldlt = nullptr;
    DistCtx *dist = nullptr;
    FpWs *fp = nullptr;
    ExtrasWs *extras = nullptr;               // batched solve_two_extras: CSR patterns + workspace (built at first use)
    fpsb_iter_opts iopts{};
    bool iopts_set = false;
    double prof_loop_ms = 0.0;          // CUDA-event time of the last Krylov loop region
    int64_t prof_step_launches = 0;     // fused SpMM step kernels launched in that region
    // geometry the persistent loop of the last Krylov solve ran with (fpsb_iter_loop_info): persistent, early,
    // nstage, grid, stage_bytes, inflight, nspec, chunk iterations; all zero when that solve took the step path
    int64_t loop_info[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

// api.cu: stream ordering against the caller of FPSB_DEVICE entries
void caller_order_in(Handle *h);
void caller_order_out(Handle *h);

// krylov.cu
void csr_build(Handle *h);
void csr_refresh_values(Handle *h);
void spmv_plain(Handle *h, bool transpose, const double *x, double *y, int ncols_rhs);
void phase_timers(unsigned long long *out, int reset);   // debug builds (-DFPSB_PHASE_TIMERS)
void loop_timers(unsigned long long *out);
void xchg_timers(unsigned long long *out);                // debug builds (-DFPSB_LOOP_TIMERS)
void iter_setup(Handle *h);
void iter_free(Handle *h);
void iter_solve_two_mixed(Handle *h, double delta, const double *rhs1, const double *rhs2, double *p1,
                          double *q1, double *p2, double *q2, fpsb_krylov_stats *st);
void iter_solve_two_least_squares(Handle *h, double delta, const double *rhs1, const double *rhs2,
                                  double *p1, double *q1, double *p2, double *q2,
                                  fpsb_krylov_stats *st);
void iter_solve_two_extras(Handle *h, double delta, const double *rhs1, const double *rhs2, double *u1,
                           double *u2, fpsb_krylov_stats *st, bool ldlt_variant);
// fpsb_extras_batch.inl: solve_two_extras of the LDLt path for ninst instances of the handle's pattern (device
// buffers, stream-ordered on h->stream); opts == nullptr: the single-instance entry's tolerances
void extras_batch(Handle *h, int64_t ninst, const double *jvals, const double *delta, const double *rhs1,
                  const double *rhs2, double *u1, double *u2, fpsb_krylov_stats *stats, const fpsb_extras_opts *opts);
void extras_free(Handle *h);
// the plain CSR patterns of A and A' with the COO index of every slot, built at the first call (device, int):
// rpA [m+1] | ciA [nnz] | pmA [nnz] | rpT [n+1] | ciT [nnz] | pmT [nnz]; used by extras_batch and fpb_spmv
const int *jac_csr(Handle *h);

// fpsb_dist.inl (row-partitioned Krylov over NCCL)
void dist_unique_id(void *out128);
void dist_attach(Handle *h, int nranks, int rank, const void *id128, int64_t own_off, int64_t n_own,
                 const int64_t *recv_start, const int64_t *recv_cnt, const int64_t *send_ptr, const int64_t *send_idx);
void dist_free(Handle *h);
int64_t dist_peer_blob_bytes();
void dist_peer_export(Handle *h, void *blob_out);
void dist_peer_attach(Handle *h, const void *blobs);
bool dist_peer_active(Handle *h);
int64_t dist_n_own(Handle *h);
void dist_profile(bool on);
void dist_last_profile(double *us4, long long *cnt4);
void dist_jprod(Handle *h, const double *x_own, double *y_loc);
void dist_jtprod(Handle *h, const double *u_loc, double *y_own);
void dist_solve_two_mixed(Handle *h, double delta, const double *rhs1, const double *rhs2, double *p1, double *q1,
                          double *p2, double *q2, fpsb_krylov_stats *st, int64_t nvar_global, int64_t ncon_global);
void dist_solve_two_least_squares(Handle *h, double delta, const double *rhs1, const double *rhs2, double *p1, double *q1,
                                  double *p2, double *q2, fpsb_krylov_stats *st, int64_t nvar_global, int64_t ncon_global);

void dist_solve_two_extras(Handle *h, double delta, const double *rhs1, const double *rhs2, double *u1, double *u2,
                           fpsb_krylov_stats *st, int64_t nvar_global, int64_t ncon_global);

// fpsb_fpnlp.cu (device-resident FletcherPenaltyNLP glue)
void fp_free(Handle *h);
void fp_ys_gs(Handle *h, int64_t n, int64_t m, double sigma, const double *p1, const double *q1, const double *p2,
              const double *q2, double *gs, double *ys, double *v, double *w);
double fp_obj(Handle *h, int64_t n, int64_t m, double fx, double rho, double eta, const double *c, const double *ys,
              const double *x, const double *xk);
void fp_grad(Handle *h, int64_t n, double sigma, double rho, double eta, const double *gs, const double *Hsv, const double *v,
             const double *Sstw, const double *Jtc, const double *x, const double *xk, double *g);
void fp_ptv(Handle *h, int64_t n, const double *v, const double *p1, double *Ptv);
void fp_hprod2(Handle *h, int64_t n, double sigma, double rho, double eta, double obj_weight, const double *p2, const double *HsPtv,
               const double *Ptv, const double *Hcv, const double *JtJv, const double *v, double *Hv);
void fp_hprod1(Handle *h, int64_t n, double sigma, double rho, double eta, double obj_weight, const double *p2, const double *HsPtv,
               const double *Ptv, const double *JtinvJtJSsv, const double *SsinvJtJJv, const double *Hcv, const double *JtJv,
               const double *v, double *Hv);
void trcg_init(Handle *h, int64_t n, const double *g, const double *fr, double *s, double *r, double *d, double *out5);
void trcg_step(Handle *h, int64_t n, const double *Hd, const double *fr, double *s, double *r, double *d, double radius, double tol,
               double *out5);
uint64_t fp_hash(Handle *h, int64_t n, const double *x);
// fpsb_fpnlp_batch.inl: the same for `ninst` instances ([ninst][n] / [ninst][m] vectors, [ninst] scalar arrays)
void fpb_ys_gs(Handle *h, int64_t ninst, const double *sigma, const double *p1, const double *q1, const double *p2,
               const double *q2, double *gs, double *ys, double *v, double *w);
void fpb_hash(Handle *h, int64_t ninst, const double *x, uint64_t *keys);
void fpb_obj(Handle *h, int64_t ninst, const double *fx, const double *rho, const double *eta, const double *c,
             const double *ys, const double *x, const double *xk, double *phi);
void fpb_grad(Handle *h, int64_t ninst, const double *sigma, const double *rho, const double *eta, const double *gs,
              const double *Hsv, const double *v, const double *Sstw, const double *Jtc, const double *x, const double *xk,
              double *g);
void fpb_ptv(Handle *h, int64_t ninst, const double *v, const double *p1, double *Ptv);
void fpb_hprod2(Handle *h, int64_t ninst, const double *sigma, const double *rho, const double *eta, const double *obj_weight,
                const double *p2, const double *HsPtv, const double *Ptv, const double *Hcv, const double *JtJv,
                const double *v, double *Hv);
void fpb_hprod1(Handle *h, int64_t ninst, const double *sigma, const double *rho, const double *eta, const double *obj_weight,
                const double *p2, const double *HsPtv, const double *Ptv, const double *JtinvJtJSsv,
                const double *SsinvJtJJv, const double *Hcv, const double *JtJv, const double *v, double *Hv);
void fpb_spmv(Handle *h, bool transpose, int64_t ninst, const double *jvals, int64_t jstride, const double *x, double *out);
int32_t trcg_batch_init(Handle *h, int64_t ninst, const double *g, const double *fr, const double *tol, double *s, double *r,
                        double *d, double *st, int *nprod);
int32_t trcg_batch_step(Handle *h, int64_t ninst, const double *Hd, const double *fr, const double *radius, const double *tol,
                        double *s, double *r, double *d, double *st, int *nprod);

// symbolic.cpp / ldlt.cu
void ldlt_analyze(Handle *h, const int64_t *P, const fpsb_ldlt_opts *opts);
void ldlt_free(Handle *h);
void ldlt_factorize(Handle *h, double delta, int *factorized);
void ldlt_solve2(Handle *h, int kind, const double *rhs1, const double *rhs2, double *p1, double *q1,
                 double *p2, double *q2, int *factorized);

}  // namespace fpsb
