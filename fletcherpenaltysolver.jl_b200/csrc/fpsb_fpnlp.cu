// fpsb_fpnlp.cu — device-resident evaluation glue of FletcherPenaltyNLP (SURVEY §8 f1): the vector
// combinations either side of the 2-RHS solves as fused kernels on the handle's stream, so that x, g,
// c, the multipliers and the penalty gradient never leave HBM across the outer algo.jl loop.
//
// Reference code replaced (file:line under /root/reference):
//   _compute_ys_gs!   gs = p1 + sigma p2, ys = q1 + sigma q2, v = p2, w = q2   src/model-Fletcherpenaltynlp.jl:244-248
//                     memo key hash(x)                                          :235
//   obj               f - c'ys + rho/2 |c|^2 (+ eta/2 |x - xk|^2)               :364-367
//   grad!             gs - Hsv + sigma v + Sstw (+ rho J'c) (+ eta (x - xk))    :382-398
//   hprod! (Val 2)    Ptv = v - p1 ; Hv = p2 - HsPtv + 2 sigma Ptv (+ Hcv + rho J'Jv) (+ eta v), times obj_weight   :543-568
// All pointers are DEVICE pointers; scalar results come back through a pinned host slot.
// The batched forms (many instances of one model, fpsb_fp_batch_*, fpsb_batch_j*prod, fpsb_trcg_batch_*) are in
// fpsb_fpnlp_batch.inl, included at the end.
#include "fpsb_internal.h"
#include "fpsb_device.cuh"

namespace fpsb {

__global__ void fp_ys_gs_kernel(int n, int m, double sigma, const double *p1, const double *q1, const double *p2,
                                const double *q2, double *gs, double *ys, double *v, double *w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const double b = p2[i]; gs[i] = p1[i] + sigma * b; v[i] = b; }
    if (i < m) { const double b = q2[i]; ys[i] = q1[i] + sigma * b; w[i] = b; }
}

// fixed-order two-level reduction of up to 3 sums: out[0..2] (device) ; the last CTA finishes
__global__ void __launch_bounds__(256) fp_obj_kernel(int m, int n, const double *c, const double *ys, const double *x,
                                                      const double *xk, double *partials, unsigned *counter, double *out) {
    __shared__ double s_red[3 * 32];
    __shared__ int s_last;
    double acc[3] = {0.0, 0.0, 0.0};
    const int stride = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) { const double ci = c[i]; acc[0] += ci * ys[i]; acc[1] += ci * ci; }
    if (xk != nullptr)
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) { const double d = x[i] - xk[i]; acc[2] += d * d; }
    block_sum<3>(acc, s_red);
    if (threadIdx.x == 0) {
        double *pp = partials + (size_t)blockIdx.x * 3;
        pp[0] = acc[0]; pp[1] = acc[1]; pp[2] = acc[2];
        __threadfence();
        s_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double tot[3] = {0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < (int)gridDim.x; i += 256) {
        tot[0] += __ldcg(partials + (size_t)i * 3); tot[1] += __ldcg(partials + (size_t)i * 3 + 1); tot[2] += __ldcg(partials + (size_t)i * 3 + 2);
    }
    block_sum<3>(tot, s_red);
    if (threadIdx.x == 0) { out[0] = tot[0]; out[1] = tot[1]; out[2] = tot[2]; *counter = 0; }
}

__global__ void fp_grad_kernel(int n, double sigma, double rho, double eta, const double *gs, const double *Hsv,
                               const double *v, const double *Sstw, const double *Jtc, const double *x, const double *xk,
                               double *g) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r = gs[i] - Hsv[i] + sigma * v[i] + Sstw[i];
    if (rho > 0.0 && Jtc != nullptr) r = r + rho * Jtc[i];
    if (eta > 0.0 && xk != nullptr) r = r + eta * (x[i] - xk[i]);
    g[i] = r;
}

__global__ void fp_ptv_kernel(int n, const double *v, const double *p1, double *Ptv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) Ptv[i] = v[i] - p1[i];
}

__global__ void fp_hprod2_kernel(int n, double sigma, double rho, double eta, double obj_weight, const double *p2,
                                 const double *HsPtv, const double *Ptv, const double *Hcv, const double *JtJv,
                                 const double *v, double *Hv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r = p2[i] - HsPtv[i] + 2.0 * sigma * Ptv[i];
    if (rho > 0.0 && Hcv != nullptr && JtJv != nullptr) r = r + Hcv[i] + rho * JtJv[i];
    if (eta > 0.0) r = r + eta * v[i];
    Hv[i] = obj_weight * r;
}

// Val(1): the two extra terms of the exact Hessian (src/model-Fletcherpenaltynlp.jl:572-634), same operation order as the host mirror
__global__ void fp_hprod1_kernel(int n, double sigma, double rho, double eta, double obj_weight, const double *p2,
                                 const double *HsPtv, const double *Ptv, const double *JtinvJtJSsv, const double *SsinvJtJJv,
                                 const double *Hcv, const double *JtJv, const double *v, double *Hv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r = p2[i] - HsPtv[i] + 2.0 * sigma * Ptv[i] - JtinvJtJSsv[i];
    r = r - SsinvJtJJv[i];
    if (rho > 0.0 && Hcv != nullptr && JtJv != nullptr) r = r + rho * (Hcv[i] + JtJv[i]);
    if (eta > 0.0) r = r + eta * v[i];
    Hv[i] = obj_weight * r;
}

// memo key of x: order-independent sum of per-element mixes of (bit pattern, index) — any 64-bit key
// that changes when x changes serves the reference's purpose (it memoises on hash(x) alone)
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z ^= z >> 33; z *= 0xff51afd7ed558ccdULL; z ^= z >> 33; z *= 0xc4ceb9fe1a85ec53ULL; z ^= z >> 33;
    return z;
}
__global__ void __launch_bounds__(256) fp_hash_kernel(int n, const double *x, unsigned long long *out) {
    unsigned long long acc = 0;
    const int stride = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        acc += mix64((unsigned long long)__double_as_longlong(x[i]) ^ (0x9e3779b97f4a7c15ULL * (unsigned long long)(i + 1)));
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);      // integer addition: order-independent, exact
}

// ------------------------------------------------------------------------------------------------
// Steihaug–Toint truncated CG of the trust-region subproblem (SURVEY §8 f3: the matrix-free subsolver that drives the
// penalty model, `trunk` in fps_solve.py).  One CG iteration = the model's Hessian product (the 2-RHS solves) + the three
// kernels below; every inner product, the step to the boundary, alpha, beta, the model decrease q and the exit decision
// stay on the device (state st[]), the host reads five doubles once per iteration.
//   st: [0] rr  [1] q  [2] tau (step taken along d)  [3] beta  [4] flag (0 go on, 1 left through the boundary /
//       non-positive curvature, 2 converged)
// Reductions: per-thread over a fixed stride -> block_sum -> the last block adds the per-block partials in index order.
// ------------------------------------------------------------------------------------------------
template <int K>
__device__ __forceinline__ bool trcg_last_block(double (&acc)[K], double *s_red, int *s_last, double *partials, unsigned *counter) {
    block_sum<K>(acc, s_red);
    if (threadIdx.x == 0) {
        double *pp = partials + (size_t)blockIdx.x * K;
#pragma unroll
        for (int k = 0; k < K; ++k) pp[k] = acc[k];
        __threadfence();
        *s_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!*s_last) return false;
    __threadfence();
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += 256)
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] += __ldcg(partials + (size_t)i * K + k);
    block_sum<K>(acc, s_red);
    if (threadIdx.x == 0) *counter = 0;
    return true;
}

__global__ void __launch_bounds__(256) trcg_init_kernel(int n, const double *g, const double *fr, double *s, double *r, double *d,
                                                         double *partials, unsigned *counter, double *st) {
    __shared__ double s_red[32];
    __shared__ int s_last;
    double acc[1] = {0.0};
    const int stride = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double ri = fr != nullptr ? -g[i] * fr[i] : -g[i];
        s[i] = 0.0; r[i] = ri; d[i] = ri;
        acc[0] += ri * ri;
    }
    if (!trcg_last_block<1>(acc, s_red, &s_last, partials, counter)) return;
    if (threadIdx.x == 0) { st[0] = acc[0]; st[1] = 0.0; st[2] = 0.0; st[3] = 0.0; st[4] = 0.0; }
}

// the five inner products of an iteration and every scalar decision that follows from them
__global__ void __launch_bounds__(256) trcg_dots_kernel(int n, const double *d, const double *Hd, const double *s, const double *r,
                                                         const double *fr, double radius, double *partials, unsigned *counter,
                                                         double *st) {
    __shared__ double s_red[5 * 32];
    __shared__ int s_last;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int stride = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double di = d[i], si = s[i];
        const double hd = fr != nullptr ? Hd[i] * fr[i] : Hd[i];
        acc[0] += di * hd; acc[1] += si * si; acc[2] += si * di; acc[3] += di * di; acc[4] += r[i] * di;
    }
    if (!trcg_last_block<5>(acc, s_red, &s_last, partials, counter)) return;
    if (threadIdx.x == 0) {
        const double dHd = acc[0], ss = acc[1], sd = acc[2], dd = acc[3], rd = acc[4];
        const double rr = st[0];
        const double disc = fmax(sd * sd + dd * (radius * radius - ss), 0.0);
        const double to_boundary = dd > 0.0 ? (-sd + sqrt(disc)) / dd : 0.0;      // positive step to the boundary along d
        double tau, flag;
        if (dHd <= 2.220446049250313e-16 * dd) { tau = to_boundary; flag = 1.0; }   // negative / zero curvature
        else {
            const double alpha = rr / dHd;
            if (alpha >= to_boundary) { tau = to_boundary; flag = 1.0; } else { tau = alpha; flag = 0.0; }
        }
        st[1] = st[1] + (tau * (-rd) + 0.5 * tau * tau * dHd);
        st[2] = tau; st[4] = flag;
    }
}

// s += tau d ; inside the ball also r -= tau Hd, rr_new, beta and the convergence test
__global__ void __launch_bounds__(256) trcg_update_kernel(int n, const double *d, const double *Hd, double *s, double *r,
                                                           const double *fr, double tol, double *partials, unsigned *counter,
                                                           double *st) {
    __shared__ double s_red[32];
    __shared__ int s_last;
    const double tau = __ldcg(st + 2);
    const bool inside = __ldcg(st + 4) == 0.0;
    double acc[1] = {0.0};
    const int stride = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        s[i] = s[i] + tau * d[i];
        if (inside) {
            const double hd = fr != nullptr ? Hd[i] * fr[i] : Hd[i];
            const double ri = r[i] - tau * hd;
            r[i] = ri;
            acc[0] += ri * ri;
        }
    }
    if (!trcg_last_block<1>(acc, s_red, &s_last, partials, counter)) return;
    if (threadIdx.x == 0 && inside) {
        const double rr = st[0], rr_new = acc[0];
        st[3] = rr_new / rr;
        st[0] = rr_new;
        if (sqrt(rr_new) <= tol) st[4] = 2.0;
    }
}

__global__ void trcg_dir_kernel(int n, const double *r, double *d, const double *st) {
    if (__ldcg(st + 4) != 0.0) return;
    const double beta = __ldcg(st + 3);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = r[i] + beta * d[i];
}

struct FpWs {
    DevBuf<double> partials, out, trcg;
    DevBuf<unsigned> counter;
    DevBuf<unsigned long long> key;
    DevBuf<unsigned> bcount;               // batched CG: instances still going
    double *h_out = nullptr;               // pinned: 3 doubles + 1 u64 + 1 u32 (batched CG count, at double 6)
};

static FpWs *fp_ws(Handle *h) {
    if (!h->fp) {
        FpWs *W = new FpWs();
        W->partials.alloc(5 * 1024 + 8);
        W->trcg.alloc(8);
        W->trcg.zero(h->stream);
        W->out.alloc(8);
        W->counter.alloc(4);
        W->key.alloc(2);
        W->counter.zero(h->stream);
        W->bcount.alloc(1);
        FPSB_CUDA(cudaMallocHost((void **)&W->h_out, 8 * sizeof(double)));
        h->fp = W;
    }
    return h->fp;
}
void fp_free(Handle *h) {
    if (!h->fp) return;
    if (h->fp->h_out) cudaFreeHost(h->fp->h_out);
    delete h->fp;
    h->fp = nullptr;
}

void fp_ys_gs(Handle *h, int64_t n, int64_t m, double sigma, const double *p1, const double *q1, const double *p2,
              const double *q2, double *gs, double *ys, double *v, double *w) {
    const int64_t N = n > m ? n : m;
    if (N == 0) return;
    fp_ys_gs_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>((int)n, (int)m, sigma, p1, q1, p2, q2, gs, ys, v, w);
    h->launches += 1;
    FPSB_CUDA(cudaGetLastError());
}
double fp_obj(Handle *h, int64_t n, int64_t m, double fx, double rho, double eta, const double *c, const double *ys,
              const double *x, const double *xk) {
    FpWs *W = fp_ws(h);
    const bool prox = eta > 0.0 && x && xk;
    const int64_t N = (prox && n > m) ? n : m;
    int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, (N + 255) / 256));
    fp_obj_kernel<<<grid, 256, 0, h->stream>>>((int)m, (int)n, c, ys, x, prox ? xk : nullptr, W->partials.p, W->counter.p, W->out.p);
    h->launches += 1;
    FPSB_CUDA(cudaMemcpyAsync(W->h_out, W->out.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    double phi = fx - W->h_out[0] + rho / 2 * W->h_out[1];
    if (prox) phi += eta / 2 * W->h_out[2];
    return phi;
}
void fp_grad(Handle *h, int64_t n, double sigma, double rho, double eta, const double *gs, const double *Hsv, const double *v,
             const double *Sstw, const double *Jtc, const double *x, const double *xk, double *g) {
    if (n == 0) return;
    fp_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int)n, sigma, rho, eta, gs, Hsv, v, Sstw, Jtc, x, xk, g);
    h->launches += 1;
    FPSB_CUDA(cudaGetLastError());
}
void fp_ptv(Handle *h, int64_t n, const double *v, const double *p1, double *Ptv) {
    if (n == 0) return;
    fp_ptv_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int)n, v, p1, Ptv);
    h->launches += 1;
}
void fp_hprod2(Handle *h, int64_t n, double sigma, double rho, double eta, double obj_weight, const double *p2, const double *HsPtv,
               const double *Ptv, const double *Hcv, const double *JtJv, const double *v, double *Hv) {
    if (n == 0) return;
    fp_hprod2_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int)n, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, Hcv, JtJv, v, Hv);
    h->launches += 1;
}
void fp_hprod1(Handle *h, int64_t n, double sigma, double rho, double eta, double obj_weight, const double *p2, const double *HsPtv,
               const double *Ptv, const double *JtinvJtJSsv, const double *SsinvJtJJv, const double *Hcv, const double *JtJv,
               const double *v, double *Hv) {
    if (n == 0) return;
    fp_hprod1_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int)n, sigma, rho, eta, obj_weight, p2, HsPtv, Ptv, JtinvJtJSsv,
                                                                        SsinvJtJJv, Hcv, JtJv, v, Hv);
    h->launches += 1;
}
static void trcg_read(Handle *h, FpWs *W, double *out5) {
    FPSB_CUDA(cudaMemcpyAsync(W->h_out, W->trcg.p, 5 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    for (int k = 0; k < 5; ++k) out5[k] = W->h_out[k];
}
void trcg_init(Handle *h, int64_t n, const double *g, const double *fr, double *s, double *r, double *d, double *out5) {
    FpWs *W = fp_ws(h);
    const int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, (n + 255) / 256));
    trcg_init_kernel<<<grid, 256, 0, h->stream>>>((int)n, g, fr, s, r, d, W->partials.p, W->counter.p, W->trcg.p);
    h->launches += 1;
    FPSB_CUDA(cudaGetLastError());
    trcg_read(h, W, out5);
}
void trcg_step(Handle *h, int64_t n, const double *Hd, const double *fr, double *s, double *r, double *d, double radius, double tol,
               double *out5) {
    FpWs *W = fp_ws(h);
    const int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, (n + 255) / 256));
    trcg_dots_kernel<<<grid, 256, 0, h->stream>>>((int)n, d, Hd, s, r, fr, radius, W->partials.p, W->counter.p, W->trcg.p);
    trcg_update_kernel<<<grid, 256, 0, h->stream>>>((int)n, d, Hd, s, r, fr, tol, W->partials.p, W->counter.p, W->trcg.p);
    if (n > 0) trcg_dir_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int)n, r, d, W->trcg.p);
    h->launches += 3;
    FPSB_CUDA(cudaGetLastError());
    trcg_read(h, W, out5);
}
uint64_t fp_hash(Handle *h, int64_t n, const double *x) {
    FpWs *W = fp_ws(h);
    FPSB_CUDA(cudaMemsetAsync(W->key.p, 0, sizeof(unsigned long long), h->stream));
    if (n > 0) {
        int grid = (int)std::min<int64_t>(1024, (n + 255) / 256);
        fp_hash_kernel<<<grid, 256, 0, h->stream>>>((int)n, x, W->key.p);
        h->launches += 1;
    }
    unsigned long long *hk = reinterpret_cast<unsigned long long *>(W->h_out + 4);
    FPSB_CUDA(cudaMemcpyAsync(hk, W->key.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    FPSB_CUDA(cudaStreamSynchronize(h->stream));
    return (uint64_t)*hk;
}

#include "fpsb_fpnlp_batch.inl"

}  // namespace fpsb
