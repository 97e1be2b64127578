// fpsb_api.cu — the C ABI of libfpsb200.so (include/fpsb.h): handle management, host<->device
// staging for FPSB_HOST callers, argument checking, exception firewall.
#include "fpsb_internal.h"
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <new>
#include <atomic>
#include <mutex>

namespace fpsb {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void caller_order_in(Handle *h) {
    FPSB_CUDA(cudaEventRecord(h->ev_in, h->caller_stream));
    FPSB_CUDA(cudaStreamWaitEvent(h->stream, h->ev_in, 0));
}
void caller_order_out(Handle *h) {
    FPSB_CUDA(cudaEventRecord(h->ev_out, h->stream));
    FPSB_CUDA(cudaStreamWaitEvent(h->caller_stream, h->ev_out, 0));
}

// pinned staging area large enough for `count` doubles
static double *pin(Handle *h, size_t count) {
    if (count > h->pin_count) {
        if (h->pin) cudaFreeHost(h->pin);
        h->pin = nullptr;
        h->pin_count = 0;
        FPSB_CUDA(cudaMallocHost((void **)&h->pin, count * sizeof(double)));
        h->pin_count = count;
    }
    return h->pin;
}

// true when `p` is page-locked host memory (cudaHostRegister / cudaMallocHost): DMA straight from it
static bool is_pinned_host(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

struct Staged {
    // device views of the caller's vectors; for FPSB_HOST they live in the handle's stage buffers
    Handle *h;
    int loc;
    size_t in_off = 0, out_off = 0;
    std::vector<std::pair<double *, std::pair<size_t, size_t>>> outs;   // (host dst, (offset, count))
    Staged(Handle *hh, int l, size_t in_total, size_t out_total) : h(hh), loc(l) {
        if (loc == FPSB_DEVICE) caller_order_in(h);      // the caller's kernels wrote the inputs on its own stream
        if (loc == FPSB_HOST) {
            if (h->stage_in.n < in_total + 8) h->stage_in.alloc(in_total + 8);
            if (h->stage_out.n < out_total + 8) h->stage_out.alloc(out_total + 8);
            pin(h, in_total + out_total + 8);
        }
    }
    const double *in(const double *p, size_t count) {
        if (loc == FPSB_DEVICE) return p;
        double *d = h->stage_in.p + in_off;
        if (is_pinned_host(p)) {
            FPSB_CUDA(cudaMemcpyAsync(d, p, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        } else {
            double *hp = h->pin + in_off;
            memcpy(hp, p, count * sizeof(double));
            FPSB_CUDA(cudaMemcpyAsync(d, hp, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        }
        in_off += count;
        return d;
    }
    double *out(double *p, size_t count) {
        if (loc == FPSB_DEVICE) return p;
        double *d = h->stage_out.p + out_off;
        outs.push_back({p, {out_off, count}});
        out_off += count;
        return d;
    }
    // device_sync = false: FPSB_DEVICE calls that return nothing to the host stay asynchronous (stream-ordered
    // after the caller's stream on entry and before it on exit, like a library kernel launch)
    void finish(bool device_sync = true) {
        if (loc == FPSB_DEVICE) { caller_order_out(h); if (device_sync) FPSB_CUDA(cudaStreamSynchronize(h->stream)); return; }
        double *hp = h->pin + in_off;   // staged results go after the inputs in the pinned area
        std::vector<char> direct(outs.size(), 0);
        for (size_t i = 0; i < outs.size(); ++i) {
            auto &o = outs[i];
            const size_t bytes = o.second.second * sizeof(double);
            if (is_pinned_host(o.first)) {
                direct[i] = 1;
                FPSB_CUDA(cudaMemcpyAsync(o.first, h->stage_out.p + o.second.first, bytes, cudaMemcpyDeviceToHost, h->stream));
            } else {
                FPSB_CUDA(cudaMemcpyAsync(hp + o.second.first, h->stage_out.p + o.second.first, bytes, cudaMemcpyDeviceToHost, h->stream));
            }
        }
        FPSB_CUDA(cudaStreamSynchronize(h->stream));
        for (size_t i = 0; i < outs.size(); ++i)
            if (!direct[i]) memcpy(outs[i].first, hp + outs[i].second.first, outs[i].second.second * sizeof(double));
    }
};

}  // namespace fpsb

using namespace fpsb;

#define FPSB_TRY try {
#define FPSB_CATCH                                                        \
    }                                                                     \
    catch (const fpsb::CudaFail &f) { return f.code; }                    \
    catch (const std::bad_alloc &) { fpsb::set_error("out of host memory"); return FPSB_ENOMEM; } \
    catch (...) { fpsb::set_error("unexpected C++ exception"); return FPSB_ECUDA; }

#define REQUIRE(cond, code, msg)                       \
    do { if (!(cond)) { fpsb::set_error(msg); return code; } } while (0)

extern "C" {

int fpsb_version(void) { return FPSB_VERSION; }
const char *fpsb_last_error(void) { return g_err; }
int fpsb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int fpsb_create(int64_t nvar, int64_t ncon, int64_t nnzj, const int64_t *jrow, const int64_t *jcol,
                int index_base, int device, fpsb_handle *out) {
    REQUIRE(out, FPSB_EINVAL, "fpsb_create: out is NULL");
    *out = nullptr;
    REQUIRE(nvar >= 0 && ncon >= 0 && nnzj >= 0, FPSB_EINVAL, "fpsb_create: negative size");
    REQUIRE(nnzj == 0 || (jrow && jcol), FPSB_EINVAL, "fpsb_create: NULL structure");
    REQUIRE(nvar + ncon < 2000000000LL && nnzj < 2000000000LL, FPSB_EINVAL, "fpsb_create: sizes exceed int32 device indices");
    REQUIRE(index_base == 0 || index_base == 1, FPSB_EINVAL, "fpsb_create: index_base must be 0 or 1");
    for (int64_t k = 0; k < nnzj; ++k) {
        int64_t r = jrow[k] - index_base, c = jcol[k] - index_base;
        REQUIRE(r >= 0 && r < ncon && c >= 0 && c < nvar, FPSB_EINVAL, "fpsb_create: Jacobian index out of range");
    }
    int ndev = fpsb_device_count();
    REQUIRE(ndev > 0, FPSB_ECUDA, "fpsb_create: no CUDA device available (libfpsb200 has no CPU fallback)");
    REQUIRE(device >= 0 && device < ndev, FPSB_EINVAL, "fpsb_create: bad device ordinal");
    Handle *h = nullptr;
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(device));
    h = new Handle();
    h->device = device;
    h->nvar = nvar; h->ncon = ncon; h->nnzj = nnzj;
    h->jrow.resize((size_t)nnzj); h->jcol.resize((size_t)nnzj);
    for (int64_t k = 0; k < nnzj; ++k) { h->jrow[(size_t)k] = jrow[k] - index_base; h->jcol[(size_t)k] = jcol[k] - index_base; }
    FPSB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    FPSB_CUDA(cudaEventCreate(&h->ev0));
    FPSB_CUDA(cudaEventCreate(&h->ev1));
    FPSB_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
    FPSB_CUDA(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
    csr_build(h);
    fpsb_iter_default_opts(nvar, ncon, &h->iopts);
    *out = reinterpret_cast<fpsb_handle>(h);
    return FPSB_OK;
    }
    catch (const fpsb::CudaFail &f) { if (h) fpsb_destroy(reinterpret_cast<fpsb_handle>(h)); return f.code; }
    catch (const std::bad_alloc &) { fpsb::set_error("out of host memory"); return FPSB_ENOMEM; }
    catch (...) { fpsb::set_error("unexpected C++ exception"); return FPSB_ECUDA; }
}

int fpsb_destroy(fpsb_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    if (!h) return FPSB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    dist_free(h);
    fp_free(h);
    iter_free(h);
    extras_free(h);
    ldlt_free(h);
    if (h->pin) cudaFreeHost(h->pin);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_out) cudaEventDestroy(h->ev_out);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return FPSB_OK;
}

// page-lock / unlock a caller-owned host buffer so FPSB_HOST calls DMA directly from / into it
int fpsb_pin_host(void *ptr, int64_t bytes) {
    REQUIRE(ptr && bytes > 0, FPSB_EINVAL, "fpsb_pin_host: bad arguments");
    cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return FPSB_OK; }
    if (e != cudaSuccess) { fpsb::set_error("cudaHostRegister: %s", cudaGetErrorString(e)); cudaGetLastError(); return FPSB_ECUDA; }
    return FPSB_OK;
}
int fpsb_unpin_host(void *ptr) {
    REQUIRE(ptr, FPSB_EINVAL, "fpsb_unpin_host: NULL");
    cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); }
    return FPSB_OK;
}

int fpsb_dims(fpsb_handle hh, int64_t *nvar, int64_t *ncon, int64_t *nnzj) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    if (nvar) *nvar = h->nvar;
    if (ncon) *ncon = h->ncon;
    if (nnzj) *nnzj = h->nnzj;
    return FPSB_OK;
}
void *fpsb_stream(fpsb_handle hh) { return hh ? (void *)reinterpret_cast<Handle *>(hh)->stream : nullptr; }
int fpsb_set_caller_stream(fpsb_handle hh, void *stream) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    h->caller_stream = reinterpret_cast<cudaStream_t>(stream);
    return FPSB_OK;
}
int fpsb_synchronize(fpsb_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_timer_start(fpsb_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    FPSB_CUDA(cudaEventRecord(h->ev0, h->stream));
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_timer_stop(fpsb_handle hh, double *ms) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && ms, FPSB_EINVAL, "NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    FPSB_CUDA(cudaEventRecord(h->ev1, h->stream));
    FPSB_CUDA(cudaEventSynchronize(h->ev1));
    float f = 0;
    FPSB_CUDA(cudaEventElapsedTime(&f, h->ev0, h->ev1));
    *ms = f;
    return FPSB_OK;
    FPSB_CATCH
}
int64_t fpsb_launch_count(fpsb_handle hh) { return hh ? reinterpret_cast<Handle *>(hh)->launches : 0; }
int fpsb_tile_stats(fpsb_handle hh, int64_t out[6]) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && out, FPSB_EINVAL, "fpsb_tile_stats: NULL argument");
    out[0] = h->A.ntiles;  out[1] = h->A.nwin_tiles;  out[2] = h->A.nseg_tiles;
    out[3] = h->At.ntiles; out[4] = h->At.nwin_tiles; out[5] = h->At.nseg_tiles;
    return FPSB_OK;
}

int fpsb_set_jac_values(fpsb_handle hh, const double *vals, int loc) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    REQUIRE(vals || h->nnzj == 0, FPSB_EINVAL, "fpsb_set_jac_values: NULL vals");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    size_t nz = (size_t)h->nnzj;
    if (nz) {
        if (loc == FPSB_HOST && is_pinned_host(vals)) {
            FPSB_CUDA(cudaMemcpyAsync(h->coo_vals.p, vals, nz * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        } else if (loc == FPSB_HOST) {
            double *hp = pin(h, nz);
            memcpy(hp, vals, nz * sizeof(double));
            FPSB_CUDA(cudaMemcpyAsync(h->coo_vals.p, hp, nz * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        } else {
            caller_order_in(h);
            FPSB_CUDA(cudaMemcpyAsync(h->coo_vals.p, vals, nz * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        }
    }
    csr_refresh_values(h);
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    h->have_vals = true;
    return FPSB_OK;
    FPSB_CATCH
}

static int do_spmv(fpsb_handle hh, bool transpose, const double *x, double *y, int loc, int ncols) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && x && y, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    size_t nin = (size_t)(transpose ? h->ncon : h->nvar) * ncols, nout = (size_t)(transpose ? h->nvar : h->ncon) * ncols;
    Staged S(h, loc, nin, nout);
    const double *dx = S.in(x, nin);
    double *dy = S.out(y, nout);
    if (nout) {
        if ((transpose ? h->At.grid : h->A.grid) == 0) FPSB_CUDA(cudaMemsetAsync(dy, 0, nout * sizeof(double), h->stream));
        spmv_plain(h, transpose, dx, dy, ncols);
    }
    S.finish(false);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_jprod(fpsb_handle h, const double *v, double *Av, int loc) { return do_spmv(h, false, v, Av, loc, 1); }
int fpsb_jtprod(fpsb_handle h, const double *u, double *Atu, int loc) { return do_spmv(h, true, u, Atu, loc, 1); }
int fpsb_jprod2(fpsb_handle h, const double *v, double *Av, int loc) { return do_spmv(h, false, v, Av, loc, 2); }
int fpsb_jtprod2(fpsb_handle h, const double *u, double *Atu, int loc) { return do_spmv(h, true, u, Atu, loc, 2); }

int fpsb_iter_default_opts(int64_t nvar, int64_t ncon, fpsb_iter_opts *o) {
    REQUIRE(o, FPSB_EINVAL, "NULL opts");
    const double se = 1.4901161193847656e-08;
    o->ls_atol = o->ls_rtol = se; o->ls_itmax = 5 * (ncon + nvar);
    o->ln_atol = o->ln_rtol = o->ln_btol = se; o->ln_conlim = 1.0 / se; o->ln_itmax = 5 * (ncon + nvar);
    o->ne_atol = o->ne_rtol = o->ne_etol = se; o->ne_conlim = 1.0 / se; o->ne_itmax = 0;
    return FPSB_OK;
}
int fpsb_iter_setup(fpsb_handle hh, const fpsb_iter_opts *opts) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    if (opts) h->iopts = *opts;
    h->iopts_set = true;
    iter_setup(h);
    return FPSB_OK;
    FPSB_CATCH
}

/* debug builds only (-DFPSB_PHASE_TIMERS): accumulated clock64 cycles per kernel phase; not in fpsb.h */
void fpsb_debug_phase_timers(unsigned long long *out, int reset) { fpsb::phase_timers(out, reset); }
void fpsb_debug_loop_timers(unsigned long long *out) { fpsb::loop_timers(out); }
void fpsb_debug_xchg_timers(unsigned long long *out) { fpsb::xchg_timers(out); }

int fpsb_iter_last_profile(fpsb_handle hh, double *loop_ms, int64_t *step_launches) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    if (loop_ms) *loop_ms = h->prof_loop_ms;
    if (step_launches) *step_launches = h->prof_step_launches;
    return FPSB_OK;
}
int fpsb_iter_loop_info(fpsb_handle hh, int64_t out[8]) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && out, FPSB_EINVAL, "fpsb_iter_loop_info: NULL argument");
    for (int i = 0; i < 8; ++i) out[i] = h->loop_info[i];
    return FPSB_OK;
}

// Pipelined throughput mode (several handles of one process driven by their own host threads): one solve COMPUTES at
// a time per device.  The H2D copies of a waiting handle are already enqueued on its stream and the D2H of a finished
// one happens after it leaves the gate, so they ride on the copy engines under the running Krylov loop; without the
// gate two persistent loops interleave chunk by chunk, finish together and copy together.
static std::atomic<int> g_gate_on{0};
static std::mutex g_gate[16];
struct ComputeGate {
    std::mutex *m = nullptr;
    explicit ComputeGate(int device) { if (g_gate_on.load(std::memory_order_relaxed)) { m = &g_gate[device & 15]; m->lock(); } }
    ~ComputeGate() { if (m) m->unlock(); }
};
int fpsb_pipeline_gate(int on) { g_gate_on.store(on ? 1 : 0); return FPSB_OK; }

static int iter_solve(fpsb_handle hh, int kind, double delta, const double *rhs1, const double *rhs2,
                      double *p1, double *q1, double *p2, double *q2, int loc, fpsb_krylov_stats *stats) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && rhs1 && rhs2 && p1 && q1 && p2 && q2 && stats, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    REQUIRE(delta >= 0.0, FPSB_EINVAL, "delta must be >= 0");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    size_t n = (size_t)h->nvar, m = (size_t)h->ncon;
    size_t n2 = (kind == 0) ? m : n;
    Staged S(h, loc, n + n2, 2 * n + 2 * m);
    const double *d1 = S.in(rhs1, n), *d2 = S.in(rhs2, n2);
    double *dp1 = S.out(p1, n), *dq1 = S.out(q1, m), *dp2 = S.out(p2, n), *dq2 = S.out(q2, m);
    {
        ComputeGate gate(h->device);
        if (kind == 0) iter_solve_two_mixed(h, delta, d1, d2, dp1, dq1, dp2, dq2, stats);
        else iter_solve_two_least_squares(h, delta, d1, d2, dp1, dq1, dp2, dq2, stats);
    }
    S.finish();
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_iter_solve_two_mixed(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                              double *p1, double *q1, double *p2, double *q2, int loc,
                              fpsb_krylov_stats stats[2]) {
    return iter_solve(h, 0, delta, rhs1, rhs2, p1, q1, p2, q2, loc, stats);
}
int fpsb_iter_solve_two_least_squares(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                                      double *p1, double *q1, double *p2, double *q2, int loc,
                                      fpsb_krylov_stats stats[2]) {
    return iter_solve(h, 1, delta, rhs1, rhs2, p1, q1, p2, q2, loc, stats);
}

static int extras(fpsb_handle hh, bool ldlt_variant, double delta, const double *rhs1, const double *rhs2,
                  double *u1, double *u2, int loc, fpsb_krylov_stats *stats) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && rhs1 && rhs2 && u1 && u2 && stats, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    size_t n = (size_t)h->nvar, m = (size_t)h->ncon;
    Staged S(h, loc, n + m, 2 * m);
    const double *d1 = S.in(rhs1, n), *d2 = S.in(rhs2, m);
    double *du1 = S.out(u1, m), *du2 = S.out(u2, m);
    iter_solve_two_extras(h, delta, d1, d2, du1, du2, stats, ldlt_variant);
    S.finish();
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_iter_solve_two_extras(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                               double *u1, double *u2, int loc, fpsb_krylov_stats stats[2]) {
    return extras(h, false, delta, rhs1, rhs2, u1, u2, loc, stats);
}
int fpsb_ldlt_solve_two_extras(fpsb_handle h, double delta, const double *rhs1, const double *rhs2,
                               double *u1, double *u2, int loc, fpsb_krylov_stats stats[2]) {
    return extras(h, true, delta, rhs1, rhs2, u1, u2, loc, stats);
}

// batched LDLt solve_two_extras: host buffers go through the handle's pinned area and stage buffers (Staged); device
// buffers are stream-ordered against the caller and the call returns without waiting for the result
int fpsb_ldlt_batch_solve_two_extras(fpsb_handle hh, int64_t ninst, const double *jvals, const double *delta,
                                     const double *rhs1, const double *rhs2, double *u1, double *u2,
                                     fpsb_krylov_stats *stats, const fpsb_extras_opts *opts, int loc) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h, FPSB_EINVAL, "NULL handle");
    REQUIRE(ninst >= 0, FPSB_EINVAL, "negative ninst");
    REQUIRE(loc == FPSB_HOST || loc == FPSB_DEVICE, FPSB_EINVAL, "loc must be FPSB_HOST or FPSB_DEVICE");
    if (ninst == 0) return FPSB_OK;
    REQUIRE(jvals && delta && rhs1 && rhs2 && u1 && u2 && stats, FPSB_EINVAL, "NULL argument");
    REQUIRE(!opts || (opts->cg_itmax >= 0 && opts->mr_itmax >= 0), FPSB_EINVAL, "negative itmax");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)h->nvar, m = (size_t)h->ncon, ni = (size_t)ninst, nz = (size_t)h->nnzj;
    const size_t sw = sizeof(fpsb_krylov_stats) / sizeof(double);     // the stats travel as doubles
    Staged S(h, loc, ni * nz + ni + ni * n + ni * m, 2 * ni * m + 2 * ni * sw);
    const double *dj = S.in(jvals, ni * nz), *dd = S.in(delta, ni), *d1 = S.in(rhs1, ni * n), *d2 = S.in(rhs2, ni * m);
    double *o1 = S.out(u1, ni * m), *o2 = S.out(u2, ni * m);
    fpsb_krylov_stats *ost = reinterpret_cast<fpsb_krylov_stats *>(S.out(reinterpret_cast<double *>(stats), 2 * ni * sw));
    extras_batch(h, ninst, dj, dd, d1, d2, o1, o2, ost, opts);
    S.finish(false);
    return FPSB_OK;
    FPSB_CATCH
}

/* ---- row-partitioned Krylov over NCCL (SURVEY 8e) ------------------------------------------------ */
int fpsb_dist_unique_id(void *out128) {
    REQUIRE(out128, FPSB_EINVAL, "fpsb_dist_unique_id: NULL");
    FPSB_TRY
    dist_unique_id(out128);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_dist_attach(fpsb_handle hh, int nranks, int rank, const void *nccl_id128, int64_t own_off, int64_t n_own,
                     const int64_t *recv_start, const int64_t *recv_cnt, const int64_t *send_ptr, const int64_t *send_idx) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && nccl_id128 && recv_start && recv_cnt && send_ptr, FPSB_EINVAL, "fpsb_dist_attach: NULL argument");
    REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, FPSB_EINVAL, "fpsb_dist_attach: bad rank / nranks");
    REQUIRE(own_off >= 0 && n_own >= 0 && own_off + n_own <= h->nvar, FPSB_EINVAL, "fpsb_dist_attach: owned block outside the extended space");
    REQUIRE(send_ptr[0] == 0 && (send_ptr[nranks] == 0 || send_idx), FPSB_EINVAL, "fpsb_dist_attach: bad send lists");
    for (int p = 0; p < nranks; ++p) {
        REQUIRE(send_ptr[p + 1] >= send_ptr[p], FPSB_EINVAL, "fpsb_dist_attach: send_ptr must be non-decreasing");
        REQUIRE(recv_cnt[p] >= 0 && recv_start[p] >= 0 && recv_start[p] + recv_cnt[p] <= h->nvar, FPSB_EINVAL, "fpsb_dist_attach: halo block outside the extended space");
    }
    for (int64_t i = 0; i < send_ptr[nranks]; ++i)
        REQUIRE(send_idx[i] >= own_off && send_idx[i] < own_off + n_own, FPSB_EINVAL, "fpsb_dist_attach: send index is not an owned column");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    dist_attach(h, nranks, rank, nccl_id128, own_off, n_own, recv_start, recv_cnt, send_ptr, send_idx);
    return FPSB_OK;
    FPSB_CATCH
}
int64_t fpsb_dist_peer_blob_bytes(void) { return dist_peer_blob_bytes(); }
int fpsb_dist_peer_export(fpsb_handle hh, void *blob_out) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && blob_out, FPSB_EINVAL, "fpsb_dist_peer_export: NULL argument");
    REQUIRE(h->dist, FPSB_ESTATE, "not a row-partitioned handle (call fpsb_dist_attach first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    dist_peer_export(h, blob_out);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_dist_peer_attach(fpsb_handle hh, const void *blobs) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && blobs, FPSB_EINVAL, "fpsb_dist_peer_attach: NULL argument");
    REQUIRE(h->dist, FPSB_ESTATE, "not a row-partitioned handle (call fpsb_dist_attach first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    dist_peer_attach(h, blobs);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_dist_peer_active(fpsb_handle hh) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    return (h && dist_peer_active(h)) ? 1 : 0;
}
int fpsb_dist_profile(int on) { dist_profile(on != 0); return FPSB_OK; }
int fpsb_dist_last_profile(double mean_us[4], int64_t count[4]) {
    REQUIRE(mean_us && count, FPSB_EINVAL, "fpsb_dist_last_profile: NULL argument");
    long long c[4];
    dist_last_profile(mean_us, c);
    for (int i = 0; i < 4; ++i) count[i] = c[i];
    return FPSB_OK;
}
static int dist_spmv(fpsb_handle hh, bool transpose, const double *x, double *y, int loc) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && x && y, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->dist, FPSB_ESTATE, "not a row-partitioned handle (call fpsb_dist_attach first)");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    const int64_t nown = dist_n_own(h);
    const size_t nin = transpose ? (size_t)h->ncon : (size_t)nown, nout = transpose ? (size_t)nown : (size_t)h->ncon;
    Staged S(h, loc, nin, nout);
    const double *dx = S.in(x, nin);
    double *dy = S.out(y, nout);
    if (transpose) dist_jtprod(h, dx, dy); else dist_jprod(h, dx, dy);
    S.finish();
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_dist_jprod(fpsb_handle h, const double *x_own, double *y_loc, int loc) { return dist_spmv(h, false, x_own, y_loc, loc); }
int fpsb_dist_jtprod(fpsb_handle h, const double *u_loc, double *y_own, int loc) { return dist_spmv(h, true, u_loc, y_own, loc); }

static int dist_solve(fpsb_handle hh, int kind, double delta, int64_t nvar_global, int64_t ncon_global, const double *rhs1,
                      const double *rhs2, double *p1, double *q1, double *p2, double *q2, int loc, fpsb_krylov_stats *stats) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && rhs1 && rhs2 && p1 && q1 && p2 && q2 && stats, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->dist, FPSB_ESTATE, "not a row-partitioned handle (call fpsb_dist_attach first)");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)dist_n_own(h), m = (size_t)h->ncon;
    const size_t n2 = kind == 0 ? m : n;
    Staged S(h, loc, n + n2, 2 * n + 2 * m);
    const double *d1 = S.in(rhs1, n), *d2 = S.in(rhs2, n2);
    double *dp1 = S.out(p1, n), *dq1 = S.out(q1, m), *dp2 = S.out(p2, n), *dq2 = S.out(q2, m);
    if (kind == 0) dist_solve_two_mixed(h, delta, d1, d2, dp1, dq1, dp2, dq2, stats, nvar_global, ncon_global);
    else dist_solve_two_least_squares(h, delta, d1, d2, dp1, dq1, dp2, dq2, stats, nvar_global, ncon_global);
    S.finish();
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_dist_solve_two_mixed(fpsb_handle h, double delta, int64_t nvar_global, int64_t ncon_global, const double *rhs1,
                              const double *rhs2, double *p1, double *q1, double *p2, double *q2, int loc,
                              fpsb_krylov_stats stats[2]) {
    return dist_solve(h, 0, delta, nvar_global, ncon_global, rhs1, rhs2, p1, q1, p2, q2, loc, stats);
}
int fpsb_dist_solve_two_least_squares(fpsb_handle h, double delta, int64_t nvar_global, int64_t ncon_global,
                                      const double *rhs1, const double *rhs2, double *p1, double *q1, double *p2,
                                      double *q2, int loc, fpsb_krylov_stats stats[2]) {
    return dist_solve(h, 1, delta, nvar_global, ncon_global, rhs1, rhs2, p1, q1, p2, q2, loc, stats);
}

int fpsb_dist_solve_two_extras(fpsb_handle hh, double delta, int64_t nvar_global, int64_t ncon_global, const double *rhs1,
                               const double *rhs2, double *u1, double *u2, int loc, fpsb_krylov_stats stats[2]) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && rhs1 && rhs2 && u1 && u2 && stats, FPSB_EINVAL, "NULL argument");
    REQUIRE(h->dist, FPSB_ESTATE, "not a row-partitioned handle (call fpsb_dist_attach first)");
    REQUIRE(h->have_vals, FPSB_ESTATE, "Jacobian values not set (call fpsb_set_jac_values first)");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)dist_n_own(h), m = (size_t)h->ncon;
    Staged S(h, loc, n + m, 2 * m);
    const double *d1 = S.in(rhs1, n), *d2 = S.in(rhs2, m);
    double *du1 = S.out(u1, m), *du2 = S.out(u2, m);
    dist_solve_two_extras(h, delta, d1, d2, du1, du2, stats, nvar_global, ncon_global);
    S.finish();
    return FPSB_OK;
    FPSB_CATCH
}

/* ---- device-resident FletcherPenaltyNLP glue (SURVEY 8 f1); all vector arguments are DEVICE pointers ---- */
int fpsb_fp_ys_gs(fpsb_handle hh, double sigma, const double *p1, const double *q1, const double *p2, const double *q2,
                  double *gs, double *ys, double *v, double *w) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && p1 && q1 && p2 && q2 && gs && ys && v && w, FPSB_EINVAL, "fpsb_fp_ys_gs: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    fp_ys_gs(h, h->nvar, h->ncon, sigma, p1, q1, p2, q2, gs, ys, v, w);
    caller_order_out(h);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_obj(fpsb_handle hh, double fx, double rho, double eta, const double *c, const double *ys, const double *x,
                const double *xk, double *phi) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && c && ys && phi, FPSB_EINVAL, "fpsb_fp_obj: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    *phi = fp_obj(h, h->nvar, h->ncon, fx, rho, eta, c, ys, x, xk);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_grad(fpsb_handle hh, double sigma, double rho, double eta, const double *gs, const double *Hsv, const double *v,
                 const double *Sstw, const double *Jtc, const double *x, const double *xk, double *g) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && gs && Hsv && v && Sstw && g, FPSB_EINVAL, "fpsb_fp_grad: NULL argument");
    REQUIRE(!(rho > 0.0) || Jtc, FPSB_EINVAL, "fpsb_fp_grad: rho > 0 needs J'c");
    REQUIRE(!(eta > 0.0) || (x && xk), FPSB_EINVAL, "fpsb_fp_grad: eta > 0 needs x and xk");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    fp_grad(h, h->nvar, sigma, rho, eta, gs, Hsv, v, Sstw, Jtc, x, xk, g);
    caller_order_out(h);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_ptv(fpsb_handle hh, const double *v, const double *p1, double *Ptv) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && v && p1 && Ptv, FPSB_EINVAL, "fpsb_fp_ptv: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    fp_ptv(h, h->nvar, v, p1, Ptv);
    caller_order_out(h);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_hprod2(fpsb_handle hh, double sigma, double rho, double eta, double obj_weight, const double *p2,
                   const double *HsPtv, const double *Ptv, const double *Hcv, const double *JtJv, const double *v, double *Hv) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && p2 && HsPtv && Ptv && v && Hv, FPSB_EINVAL, "fpsb_fp_hprod2: NULL argument");
    REQUIRE(!(rho > 0.0) || (Hcv && JtJv), FPSB_EINVAL, "fpsb_fp_hprod2: rho > 0 needs Hcv and J'Jv");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    fp_hprod2(h, h->nvar, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, Hcv, JtJv, v, Hv);
    caller_order_out(h);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_hprod1(fpsb_handle hh, double sigma, double rho, double eta, double obj_weight, const double *p2,
                   const double *HsPtv, const double *Ptv, const double *JtinvJtJSsv, const double *SsinvJtJJv,
                   const double *Hcv, const double *JtJv, const double *v, double *Hv) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && p2 && HsPtv && Ptv && JtinvJtJSsv && SsinvJtJJv && v && Hv, FPSB_EINVAL, "fpsb_fp_hprod1: NULL argument");
    REQUIRE(!(rho > 0.0) || (Hcv && JtJv), FPSB_EINVAL, "fpsb_fp_hprod1: rho > 0 needs Hcv and J'Jv");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    fp_hprod1(h, h->nvar, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, JtinvJtJSsv, SsinvJtJJv, Hcv, JtJv, v, Hv);
    caller_order_out(h);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_trcg_init(fpsb_handle hh, const double *g, const double *free_mask, double *s, double *r, double *d, double out[5]) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && out && ((g && s && r && d) || h->nvar == 0), FPSB_EINVAL, "fpsb_trcg_init: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    trcg_init(h, h->nvar, g, free_mask, s, r, d, out);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_trcg_step(fpsb_handle hh, const double *Hd, const double *free_mask, double *s, double *r, double *d, double radius,
                   double tol, double out[5]) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && out && ((Hd && s && r && d) || h->nvar == 0), FPSB_EINVAL, "fpsb_trcg_step: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    trcg_step(h, h->nvar, Hd, free_mask, s, r, d, radius, tol, out);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_fp_hash(fpsb_handle hh, const double *x, uint64_t *key) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && key && (x || h->nvar == 0), FPSB_EINVAL, "fpsb_fp_hash: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    *key = fp_hash(h, h->nvar, x);
    return FPSB_OK;
    FPSB_CATCH
}

/* ---- the same glue for many instances of one model; all arguments are DEVICE pointers, instance-major ---- */
#define FPB_BEGIN(name)                                                       \
    Handle *h = reinterpret_cast<Handle *>(hh);                               \
    REQUIRE(h, FPSB_EINVAL, name ": NULL handle");                            \
    REQUIRE(ninst >= 0, FPSB_EINVAL, name ": negative ninst");                \
    if (ninst == 0) return FPSB_OK;
#define FPB_RUN(call)                                                         \
    FPSB_TRY                                                                  \
    FPSB_CUDA(cudaSetDevice(h->device));                                      \
    caller_order_in(h);                                                       \
    call;                                                                     \
    caller_order_out(h);                                                      \
    return FPSB_OK;                                                           \
    FPSB_CATCH

int fpsb_fp_batch_ys_gs(fpsb_handle hh, int64_t ninst, const double *sigma, const double *p1, const double *q1,
                        const double *p2, const double *q2, double *gs, double *ys, double *v, double *w) {
    FPB_BEGIN("fpsb_fp_batch_ys_gs")
    REQUIRE(sigma && p1 && q1 && p2 && q2 && gs && ys && v && w, FPSB_EINVAL, "fpsb_fp_batch_ys_gs: NULL argument");
    FPB_RUN(fpb_ys_gs(h, ninst, sigma, p1, q1, p2, q2, gs, ys, v, w))
}
int fpsb_fp_batch_hash(fpsb_handle hh, int64_t ninst, const double *x, uint64_t *keys) {
    FPB_BEGIN("fpsb_fp_batch_hash")
    REQUIRE(keys && (x || h->nvar == 0), FPSB_EINVAL, "fpsb_fp_batch_hash: NULL argument");
    FPB_RUN(fpb_hash(h, ninst, x, keys))
}
int fpsb_fp_batch_obj(fpsb_handle hh, int64_t ninst, const double *fx, const double *rho, const double *eta, const double *c,
                      const double *ys, const double *x, const double *xk, double *phi) {
    FPB_BEGIN("fpsb_fp_batch_obj")
    REQUIRE(fx && phi && ((c && ys) || h->ncon == 0), FPSB_EINVAL, "fpsb_fp_batch_obj: NULL argument");
    REQUIRE(!eta || ((x && xk) || h->nvar == 0), FPSB_EINVAL, "fpsb_fp_batch_obj: eta needs x and xk");
    FPB_RUN(fpb_obj(h, ninst, fx, rho, eta, c, ys, x, xk, phi))
}
int fpsb_fp_batch_grad(fpsb_handle hh, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                       const double *gs, const double *Hsv, const double *v, const double *Sstw, const double *Jtc,
                       const double *x, const double *xk, double *g) {
    FPB_BEGIN("fpsb_fp_batch_grad")
    REQUIRE(sigma && gs && Hsv && v && Sstw && g, FPSB_EINVAL, "fpsb_fp_batch_grad: NULL argument");
    REQUIRE(!rho || Jtc, FPSB_EINVAL, "fpsb_fp_batch_grad: rho needs J'c");
    REQUIRE(!eta || (x && xk), FPSB_EINVAL, "fpsb_fp_batch_grad: eta needs x and xk");
    FPB_RUN(fpb_grad(h, ninst, sigma, rho, eta, gs, Hsv, v, Sstw, Jtc, x, xk, g))
}
int fpsb_fp_batch_ptv(fpsb_handle hh, int64_t ninst, const double *v, const double *p1, double *Ptv) {
    FPB_BEGIN("fpsb_fp_batch_ptv")
    REQUIRE(v && p1 && Ptv, FPSB_EINVAL, "fpsb_fp_batch_ptv: NULL argument");
    FPB_RUN(fpb_ptv(h, ninst, v, p1, Ptv))
}
int fpsb_fp_batch_hprod2(fpsb_handle hh, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                         const double *obj_weight, const double *p2, const double *HsPtv, const double *Ptv, const double *Hcv,
                         const double *JtJv, const double *v, double *Hv) {
    FPB_BEGIN("fpsb_fp_batch_hprod2")
    REQUIRE(sigma && p2 && HsPtv && Ptv && v && Hv, FPSB_EINVAL, "fpsb_fp_batch_hprod2: NULL argument");
    REQUIRE(!rho || (Hcv && JtJv), FPSB_EINVAL, "fpsb_fp_batch_hprod2: rho needs Hcv and J'Jv");
    FPB_RUN(fpb_hprod2(h, ninst, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, Hcv, JtJv, v, Hv))
}
int fpsb_fp_batch_hprod1(fpsb_handle hh, int64_t ninst, const double *sigma, const double *rho, const double *eta,
                         const double *obj_weight, const double *p2, const double *HsPtv, const double *Ptv,
                         const double *JtinvJtJSsv, const double *SsinvJtJJv, const double *Hcv, const double *JtJv,
                         const double *v, double *Hv) {
    FPB_BEGIN("fpsb_fp_batch_hprod1")
    REQUIRE(sigma && p2 && HsPtv && Ptv && JtinvJtJSsv && SsinvJtJJv && v && Hv, FPSB_EINVAL,
            "fpsb_fp_batch_hprod1: NULL argument");
    REQUIRE(!rho || (Hcv && JtJv), FPSB_EINVAL, "fpsb_fp_batch_hprod1: rho needs Hcv and J'Jv");
    FPB_RUN(fpb_hprod1(h, ninst, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, JtinvJtJSsv, SsinvJtJJv, Hcv, JtJv, v, Hv))
}
int fpsb_batch_jprod(fpsb_handle hh, int64_t ninst, const double *jvals, int64_t jstride, const double *v, double *out) {
    FPB_BEGIN("fpsb_batch_jprod")
    REQUIRE(jstride == 0 || jstride == h->nnzj, FPSB_EINVAL, "fpsb_batch_jprod: jstride must be 0 or nnzj");
    REQUIRE((jvals || h->nnzj == 0) && (v || h->nvar == 0) && (out || h->ncon == 0), FPSB_EINVAL,
            "fpsb_batch_jprod: NULL argument");
    FPB_RUN(fpb_spmv(h, false, ninst, jvals, jstride, v, out))
}
int fpsb_batch_jtprod(fpsb_handle hh, int64_t ninst, const double *jvals, int64_t jstride, const double *u, double *out) {
    FPB_BEGIN("fpsb_batch_jtprod")
    REQUIRE(jstride == 0 || jstride == h->nnzj, FPSB_EINVAL, "fpsb_batch_jtprod: jstride must be 0 or nnzj");
    REQUIRE((jvals || h->nnzj == 0) && (u || h->ncon == 0) && (out || h->nvar == 0), FPSB_EINVAL,
            "fpsb_batch_jtprod: NULL argument");
    FPB_RUN(fpb_spmv(h, true, ninst, jvals, jstride, u, out))
}
int fpsb_trcg_batch_init(fpsb_handle hh, int64_t ninst, const double *g, const double *free_mask, const double *tol,
                         double *s, double *r, double *d, double *st, int32_t *nprod, int32_t *nactive) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && nactive, FPSB_EINVAL, "fpsb_trcg_batch_init: NULL argument");
    REQUIRE(ninst >= 0, FPSB_EINVAL, "fpsb_trcg_batch_init: negative ninst");
    *nactive = 0;
    if (ninst == 0) return FPSB_OK;
    REQUIRE(tol && st && nprod && ((g && s && r && d) || h->nvar == 0), FPSB_EINVAL, "fpsb_trcg_batch_init: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    *nactive = trcg_batch_init(h, ninst, g, free_mask, tol, s, r, d, st, nprod);
    return FPSB_OK;
    FPSB_CATCH
}
int fpsb_trcg_batch_step(fpsb_handle hh, int64_t ninst, const double *Hd, const double *free_mask, const double *radius,
                         const double *tol, double *s, double *r, double *d, double *st, int32_t *nprod, int32_t *nactive) {
    Handle *h = reinterpret_cast<Handle *>(hh);
    REQUIRE(h && nactive, FPSB_EINVAL, "fpsb_trcg_batch_step: NULL argument");
    REQUIRE(ninst >= 0, FPSB_EINVAL, "fpsb_trcg_batch_step: negative ninst");
    *nactive = 0;
    if (ninst == 0) return FPSB_OK;
    REQUIRE(radius && tol && st && nprod && ((Hd && s && r && d) || h->nvar == 0), FPSB_EINVAL,
            "fpsb_trcg_batch_step: NULL argument");
    FPSB_TRY
    FPSB_CUDA(cudaSetDevice(h->device));
    caller_order_in(h);
    *nactive = trcg_batch_step(h, ninst, Hd, free_mask, radius, tol, s, r, d, st, nprod);
    return FPSB_OK;
    FPSB_CATCH
}

}  // extern "C"
