// enl_large.cu -- large-Jacobian regime of the B200 ENLSIP engine (BASELINE.json config 4: one problem,
// m = 4M residuals, n = 256, row-sharded over the GPUs of one box; config 5: n = 4096, m = 16384 on one GPU).
//
// Per Gauss-Newton iteration (reference: one pass of the `while exit_code == 0` loop, EF:2776-2878):
//   li_build_kernel      r = tanh(Wx) - y, J = diag(1 - tanh^2) W         -> [J | r] in HBM   (new_point!, EF:34-52)
//   tsqr_factor          [J | r] -> R (n+1 x n+1)   (enl_tsqr.cuh: Householder panels + DMMA trailing updates)
//   NCCL all-gather      of the per-GPU R factors, stacked and re-factored identically on every GPU
//   r_to_colmajor        R -> column-major [J~ | r~], device resident
//   small stage          the ENLSIP iteration on the compressed problem: every matrix (A, C.A, J~, J~ Q1, the three
//                        pivoted QR factorisations, triangular solves, multiplier and direction products) lives in HBM
//                        and is worked on by the kernels of enl_small.cuh; the host (enl_large_host.h, replicated per
//                        rank) keeps the scalar decision logic, the working set and O(n) vectors
//   li_dir_kernel        v = W p, Jp = s .* v, {r.r, r.Jp, Jp.Jp}                              (EF:2222-2224)
//   li_ls_kernel         per trial step: ||r(x + a p)||^2 and the linesearch model dots        (EF:1307-1340, 1665-1689)
//   NCCL all-reduce      of those few doubles
// General row families (enl_large_generic.cuh) take the same TSQR path when created with ENLSIPB200_LARGE_FACTOR_TSQR
// (lg_build_rows_kernel -> tsqr_factor on n rounded up to 32 columns -> rows_unpad_kernel); without it their column-major
// [J | r] goes through the plain-Householder mode of qrcp_device.
// sm_100a only; no CPU fallback (every entry point fails with ENLSIPB200_ENOGPU without a device).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <string>
#include <map>
#include <vector>

#include "../../include/enlsip_b200.h"
#include "enl_base.h"
#include "enl_large_family.h"
#include "enl_large_host.h"
#include "enl_tsqr.cuh"
#include "enl_small.cuh"
#include "enl_large_generic.cuh"
#if defined(ENL_LARGE_USER_FAMILY)
#include "enl_large_user.h"
#endif

using namespace enl_large;

namespace {

thread_local std::string g_lerr;
int lfail(int code, const std::string& msg) { g_lerr = msg; return code; }
#define LCU(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return lfail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? ENLSIPB200_ENOGPU \
                                                                                      : ENLSIPB200_ECUDA, \
                         std::string(#call) + ": " + cudaGetErrorString(e_));                            \
    } while (0)

// ---- NCCL, bound at run time (the torch-bundled libnccl.so.2 is already mapped in a torch process) ----
struct NcclApi {
    typedef struct { char internal[128]; } UniqueId;
    typedef void* Comm;
    int (*GetUniqueId)(UniqueId*) = nullptr;
    int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, Comm, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
    std::string err;
    bool load() {
        if (ok) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        void* h = nullptr;
        for (const char* nm : names) {
            h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) { err = std::string("dlopen libnccl: ") + dlerror(); return false; }
        auto sym = [&](const char* s) { return dlsym(h, s); };
        GetUniqueId = (int (*)(UniqueId*))sym("ncclGetUniqueId");
        CommInitRank = (int (*)(Comm*, int, UniqueId, int))sym("ncclCommInitRank");
        CommDestroy = (int (*)(Comm))sym("ncclCommDestroy");
        AllReduce = (int (*)(const void*, void*, size_t, int, int, Comm, cudaStream_t))sym("ncclAllReduce");
        AllGather = (int (*)(const void*, void*, size_t, int, Comm, cudaStream_t))sym("ncclAllGather");
        GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
        ok = GetUniqueId && CommInitRank && CommDestroy && AllReduce && AllGather && GetErrorString;
        if (!ok) err = "libnccl is missing a required symbol";
        return ok;
    }
};
NcclApi g_nccl;
constexpr int NCCL_FLOAT64 = 8, NCCL_SUM = 0;

// ---------------------------------------------------------------------------------------------
// elementwise kernels of the single-index family
// ---------------------------------------------------------------------------------------------
constexpr int LI_PARTS = 592;   // 148 SMs x 4 CTAs; fixed so that reductions are deterministic

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// one warp per row: u = w_i . x, r = det_tanh(u) - y, s = 1 - tanh^2; row i of [s W | r | 0..] into A.
// NC > 0: the warp also accumulates its share of J'r (lane owns columns 2 lane + 64 k, +1; NC = ceil(n / 64) register
// pairs) and of r'r; the CTA folds its 8 warps in a fixed order into gpart[blockIdx][0..n] ([n] = r'r).  The gradient is
// what the termination test of the new point reads (EF:2838, 2411), so that the factorisation can wait until the
// iteration is known to continue.  NC == 0 (n > 64 * 8): no gradient here, li_grad_kernel does it.
// FD: the Jacobian row by forward differences (jac_forward_diff, cnls_model.jl:65-82) instead of s * w_i: entry j is
// (r_i(x + delta_j e_j) - r_i(x)) / delta_j with delta_j = max(|x_j|, 1) sqrt(eps); for this family
// w_i . (x + delta_j e_j) = u_i + delta_j w_ij, so the perturbed residual costs one det_tanh and no second pass over W.
__device__ __forceinline__ double li_fd_entry(double uu, double wij, double dj, double yi, double rr) {
    const double rj = __dsub_rn(enl::det_tanh(fma(dj, wij, uu)), yi);
    return __ddiv_rn(__dsub_rn(rj, rr), dj);
}
template <int NC, bool FD = false>
__global__ void __launch_bounds__(256) li_build_kernel(const double* __restrict__ W, const double* __restrict__ y,
                                                       const double* __restrict__ x, long long m, int n, int ld,
                                                       double* __restrict__ A, double* __restrict__ u,
                                                       double* __restrict__ r, double* __restrict__ s,
                                                       double* __restrict__ gpart) {
    extern __shared__ double xs[];   // x [n]; then, NC > 0: 8 x (n + 1) partial gradients; FD: then delta [n]
    double* dls = xs + n + (NC > 0 ? 8 * (n + 1) : 0);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        xs[j] = x[j];
        if (FD) dls[j] = __dmul_rn(fmax(fabs(x[j]), 1.0), 1.4901161193847656e-08);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    double ga[NC > 0 ? 2 * NC : 1];
    double rsq = 0.0;
#pragma unroll
    for (int k = 0; k < (NC > 0 ? 2 * NC : 1); ++k) ga[k] = 0.0;
    for (long long i = warp0; i < m; i += nwarps) {
        const double* wr = W + i * n;
        double acc = 0.0;
        for (int c = 2 * lane; c < n; c += 64) {
            double2 wv = *reinterpret_cast<const double2*>(wr + c);
            acc = fma(wv.x, xs[c], acc);
            acc = fma(wv.y, xs[c + 1], acc);
        }
        const double uu = warp_sum(acc);
        const double th = enl::det_tanh(uu);
        const double rr = __dsub_rn(th, y[i]);
        const double ss = __dsub_rn(1.0, __dmul_rn(th, th));
        double* ar = A + i * ld;
        if (NC > 0) {
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const int c = 2 * lane + 64 * k;
                if (c < n) {
                    double2 wv = *reinterpret_cast<const double2*>(wr + c);
                    const double j0 = FD ? li_fd_entry(uu, wv.x, dls[c], y[i], rr) : __dmul_rn(ss, wv.x);
                    const double j1 = FD ? li_fd_entry(uu, wv.y, dls[c + 1], y[i], rr) : __dmul_rn(ss, wv.y);
                    *reinterpret_cast<double2*>(ar + c) = make_double2(j0, j1);
                    ga[2 * k] = fma(j0, rr, ga[2 * k]);
                    ga[2 * k + 1] = fma(j1, rr, ga[2 * k + 1]);
                }
            }
            rsq = fma(rr, rr, rsq);
        } else {
            for (int c = 2 * lane; c < n; c += 64) {
                double2 wv = *reinterpret_cast<const double2*>(wr + c);
                const double j0 = FD ? li_fd_entry(uu, wv.x, dls[c], y[i], rr) : __dmul_rn(ss, wv.x);
                const double j1 = FD ? li_fd_entry(uu, wv.y, dls[c + 1], y[i], rr) : __dmul_rn(ss, wv.y);
                *reinterpret_cast<double2*>(ar + c) = make_double2(j0, j1);
            }
        }
        if (lane < ld - n) ar[n + lane] = (lane == 0) ? rr : 0.0;
        if (lane == 0) { u[i] = uu; r[i] = rr; s[i] = ss; }
    }
    if (NC > 0) {
        double* gs = xs + n;
        const int w = threadIdx.x >> 5;
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            const int c = 2 * lane + 64 * k;
            if (c < n) { gs[w * (n + 1) + c] = ga[2 * k]; gs[w * (n + 1) + c + 1] = ga[2 * k + 1]; }
        }
        if (lane == 0) gs[w * (n + 1) + n] = rsq;
        __syncthreads();
        for (int j = threadIdx.x; j <= n; j += blockDim.x) {
            double t = 0.0;
            for (int ww = 0; ww < 8; ++ww) t += gs[ww * (n + 1) + j];
            gpart[(size_t)blockIdx.x * (n + 1) + j] = t;
        }
    }
}

// generic J'r for wide problems (n > 512): gpart[b][j] = sum over the rows of CTA b of A[i][j] * A[i][n]  (A = [J | r]),
// [n] = r'r; thread = column
__global__ void __launch_bounds__(256) li_grad_kernel(const double* __restrict__ A, int ld, long long m, int n,
                                                      double* __restrict__ gpart) {
    const long long per = (m + gridDim.x - 1) / gridDim.x;
    const long long i0 = per * blockIdx.x, i1 = (i0 + per < m) ? i0 + per : m;
    for (int j = threadIdx.x; j <= n; j += blockDim.x) {
        double t = 0.0;
        for (long long i = i0; i < i1; ++i) t = fma(A[i * ld + j], A[i * ld + n], t);
        gpart[(size_t)blockIdx.x * (n + 1) + j] = t;
    }
}

// out[j] = sum_b gpart[b][j] in a fixed order: one warp per column (lane l sums b = l, l + 32, ...; then a butterfly)
__global__ void __launch_bounds__(256) li_grad_finish_kernel(const double* __restrict__ gpart, int nparts, int n,
                                                             double* __restrict__ out) {
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j > n) return;
    double t = 0.0;
    for (int b = lane; b < nparts; b += 32) t += gpart[(size_t)b * (n + 1) + j];
    t = warp_sum(t);
    if (lane == 0) out[j] = t;
}

__device__ __forceinline__ void block_reduce4(double (&v)[4], double* part) {
    __shared__ double sh[8][4];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = warp_sum(v[k]);
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 4; ++k) sh[w][k] = v[k];
    __syncthreads();
    if (threadIdx.x < 4) {
        double t = 0.0;
        for (int ww = 0; ww < (int)(blockDim.x >> 5); ++ww) t += sh[ww][threadIdx.x];
        part[blockIdx.x * 4 + threadIdx.x] = t;
    }
}

// v = W p (one warp per row), Jp = s .* v; partial sums {r.r, r.Jp, Jp.Jp, 0}
// fd != 0: Jp is the product with the forward-difference Jacobian of li_build_kernel<., true> (entries recomputed on the fly
// from u, y, r and the point xcur), so that the linesearch model sees the Jacobian the iteration was built on
__global__ void __launch_bounds__(256) li_dir_kernel(const double* __restrict__ W, const double* __restrict__ p,
                                                     const double* __restrict__ r, const double* __restrict__ s,
                                                     long long m, int n, double* __restrict__ v,
                                                     double* __restrict__ Jp, double* __restrict__ part, int fd,
                                                     const double* __restrict__ xcur, const double* __restrict__ u,
                                                     const double* __restrict__ y) {
    extern __shared__ double xs[];      // p [n]; fd: then delta [n]
    double* dls = xs + n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        xs[j] = p[j];
        if (fd) dls[j] = __dmul_rn(fmax(fabs(xcur[j]), 1.0), 1.4901161193847656e-08);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long i = warp0; i < m; i += nwarps) {
        const double* wr = W + i * n;
        double acc = 0.0, accj = 0.0;
        const double ui = fd ? u[i] : 0.0, yi = fd ? y[i] : 0.0, rri = fd ? r[i] : 0.0;
        for (int c = 2 * lane; c < n; c += 64) {
            double2 wv = *reinterpret_cast<const double2*>(wr + c);
            acc = fma(wv.x, xs[c], acc);
            acc = fma(wv.y, xs[c + 1], acc);
            if (fd) {
                accj = fma(li_fd_entry(ui, wv.x, dls[c], yi, rri), xs[c], accj);
                accj = fma(li_fd_entry(ui, wv.y, dls[c + 1], yi, rri), xs[c + 1], accj);
            }
        }
        const double vv = warp_sum(acc);
        const double jfd = fd ? warp_sum(accj) : 0.0;
        if (lane == 0) {
            const double jp = fd ? jfd : s[i] * vv, ri = r[i];
            v[i] = vv; Jp[i] = jp;
            sums[0] = fma(ri, ri, sums[0]); sums[1] = fma(ri, jp, sums[1]); sums[2] = fma(jp, jp, sums[2]);
        }
    }
    block_reduce4(sums, part);
}

// trial point x + alpha p: r_a = det_tanh(u + alpha v) - y;  partial sums {r_a.r_a, r.v2, Jp.v2, v2.v2}
// with v2 = ((r_a - r)/alpha - Jp)/alpha  (coefficients_linesearch!, EF:1687)
__global__ void __launch_bounds__(256) li_ls_kernel(const double* __restrict__ u, const double* __restrict__ v,
                                                    const double* __restrict__ y, const double* __restrict__ r,
                                                    const double* __restrict__ Jp, long long m, double alpha,
                                                    int with_coeffs, double* __restrict__ part) {
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        const double ra = __dsub_rn(enl::det_tanh(fma(alpha, v[i], u[i])), y[i]);
        sums[0] = fma(ra, ra, sums[0]);
        if (with_coeffs) {
            const double ri = r[i], jp = Jp[i];
            const double v2 = (__ddiv_rn(__dsub_rn(ra, ri), alpha) - jp) / alpha;
            sums[1] = fma(ri, v2, sums[1]); sums[2] = fma(jp, v2, sums[2]); sums[3] = fma(v2, v2, sums[3]);
        }
    }
    block_reduce4(sums, part);
}

__global__ void li_finish_kernel(const double* __restrict__ part, int nparts, double* __restrict__ out) {
    const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;   // 4 warps, one per quantity
    double t = 0.0;
    for (int i = lane; i < nparts; i += 32) t += part[i * 4 + k];
    t = warp_sum(t);
    if (lane == 0) out[k] = t;
}

// R (row major, leading dimension ld, upper triangle valid) -> column-major nc x nc with explicit zeros below the
// diagonal: the layout of the compressed problem [J~ | r~] the host driver and enl_dense.cuh work on
__global__ void r_to_colmajor_kernel(const double* __restrict__ R, int ld, int nc, double* __restrict__ out) {
    __shared__ double tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < nc && c < nc && r <= c) ? R[(size_t)r * ld + c] : 0.0;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (r < nc && c < nc) out[(size_t)c * nc + r] = tile[threadIdx.x][i];
    }
}

// TSQR path of the row families: R of [J | 0 | r] (row major, leading dimension ld; nt = n rounded up to 32, r in column
// nt) -> the column-major (n+1) x (n+1) [R_J | z ; 0 | rho] of the compressed problem.  The zero columns n..nt-1 got
// identity reflectors (tau = 0), so rows n..nt-1 of the r column hold entries of r that no reflector reduced, and R[nt][nt]
// is the norm of what the panels left in the r column below the extracted rows.  rho counts each of them once:
// rho = sqrt(R[nt][nt]^2 + sum_{k=n}^{nt-1} R[k][nt]^2) (= R[n][n] itself when nt = n).
__global__ void rows_unpad_kernel(const double* __restrict__ R, int ld, int n, int nt, double* __restrict__ out) {
    const int nc = n + 1;
    const long long ne = (long long)nc * nc;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e / nc), r = (int)(e % nc);
        double v;
        if (c < n) {
            v = (r <= c) ? R[(size_t)r * ld + c] : 0.0;
        } else if (r < n) {
            v = R[(size_t)r * ld + nt];
        } else if (nt == n) {
            v = R[(size_t)nt * ld + nt];
        } else {
            double sq = 0.0;
            for (int k = n; k < nt; ++k) sq = fma(R[(size_t)k * ld + nt], R[(size_t)k * ld + nt], sq);
            const double d = R[(size_t)nt * ld + nt];
            v = sqrt(fma(d, d, sq));
        }
        out[e] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// device implementation of LargeOps
// ---------------------------------------------------------------------------------------------
// structural non-zeros of the single-index constraint Jacobian (row-major l x n, zero elsewhere): block rows
__global__ void si_jac_blocks_kernel(const double* __restrict__ x, int nb, int ineq, int n, double* __restrict__ Arow) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 4 * nb) return;
    const int k = e >> 2;
    const double v = 2.0 * x[e];
    Arow[(size_t)k * n + e] = ineq ? -v : v;
}
// ... and the constant bound rows [+e_j ; -e_j] (cnls_model.jl:402-403), written once
__global__ void si_jac_bounds_kernel(const int* __restrict__ idx, int nlo, int nup, int row0, int n, double* __restrict__ Arow) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nlo + nup) return;
    Arow[(size_t)(row0 + e) * n + idx[e]] = (e < nlo) ? 1.0 : -1.0;
}

struct LargeHandle : LargeOps, SmallBackend {
    int device = 0;
    // ---- SmallBackend state: the small stage's matrices, all column major in HBM ----
    int tcap = 0, lv = 0;             // the working-set buffers hold tcap + 1 rows (min(l, n) + 1 at first, grown on
                                      // demand up to l); length of the scratch vectors
    double* dArow = nullptr;          // A, row major l x n  (= column-major n x l)
    double *dCA = nullptr, *dCA2 = nullptr;   // C.A, row major t x n (= C.A' column major n x t); spare for row removal
    double *dFA = nullptr, *dtauA = nullptr;  // factors of qr(C.A')   n x t
    double *dFL = nullptr, *dtauL = nullptr;  // factors of qr(R_A')   t x min(n, t)
    double *dJQ1 = nullptr;                    // J~ Q1                 (n+1) x n
    double *dF2 = nullptr, *dtau2 = nullptr;   // factors of qr(J2)     (n+1) x (n - rankA)
    int *dpA = nullptr, *dipA = nullptr, *dpL = nullptr, *dipL = nullptr, *dp2 = nullptr, *dip2 = nullptr, *dact = nullptr, *dbidx = nullptr;
    double* dvec[8] = {nullptr};      // scratch vectors
    double* dscal = nullptr;
    // compact-WY T factors of the three factorisations (all panels; built on first use after a factorisation) and the
    // scratch of the cooperative vector kernels
    double *dTA = nullptr, *dTL = nullptr, *dT2 = nullptr, *dwpart = nullptr;
    bool ta_valid = false, tl_valid = false, t2_valid = false;
    double* hst = nullptr;            // pinned staging, 4 * lv doubles
    int* hsti = nullptr;              // pinned staging for permutations
    enl_small::QrWork qw;
    enl_small::WyWork ww;
    int fa_rows = 0, fa_cols = 0, fa_k = 0, fl_rows = 0, fl_cols = 0, fl_k = 0, f2_rows = 0, f2_cols = 0, f2_k = 0;
    bool jq1_valid = false;
    int ca_rows = 0;
    long long n_dev_qrcp = 0, n_dev_mulq = 0, n_ws_grow = 0;
    double ms_small = 0;              // host wall clock inside the small-stage calls (kernels + waits)

    // general row families (enl_large_generic.cuh): gv != nullptr; [J | r] column major in dQ, factored without pivoting
    const GenericVt* gv = nullptr;
    int ncu = 0;                      // the family's own constraints (equalities + inequalities); bounds follow
    double *dQ = nullptr, *dJkeep = nullptr, *dtauQ = nullptr, *dcu = nullptr;
    int* dpQ = nullptr;
    const double* gd[2] = {nullptr, nullptr};     // family data slots
    double* gown[2] = {nullptr, nullptr};
    int jac_fd = 0;                   // forward-difference Jacobians requested (cnls_model.jl:65-82)
    // ENLSIPB200_LARGE_FACTOR_TSQR: [J | 0 | r] row major in dA (nt columns for J, nt = n rounded up to 32), factored by
    // tsqr_factor like the single-index family; a row-major copy of J (dJrow) serves J p.  This rank holds the global rows
    // row0 .. row0 + m_local - 1; rows_joined: the shards are known to cover m (always so when m_local = m).
    bool tsqr_rows = false, rows_joined = true;
    long long row0 = 0;
    double* dJrow = nullptr;
    int nt = 0;                       // columns the TSQR factors: n rounded up to 32 on that path, n otherwise
    std::vector<double> hxcur;        // the point of the last eval (linesearch trial points are x + alpha p)
    long long m_local = 0, rows_pad = 0, dT_subtiles = 0;
    int ld = 0, rr_rows = 0;
    SingleIndexConstraints sc;
    cudaStream_t st = nullptr;
    // device data
    const double* dW = nullptr;
    const double* dy = nullptr;
    double *ownW = nullptr, *owny = nullptr;
    long long own_count[2] = {0, 0};
    double *dA = nullptr, *du = nullptr, *dr = nullptr, *ds = nullptr, *dv = nullptr, *dJp = nullptr;
    double *dx = nullptr, *dp = nullptr, *dT = nullptr, *dpart = nullptr, *dout = nullptr;
    double *dR = nullptr, *dStack = nullptr, *dR2 = nullptr;
    double* dP = nullptr;            // cross-rank level of the TSQR tree: max(nranks, 8) * 32 rows x ld (enl_tsqr.cuh, TsqrDist)
    double* dPscal = nullptr;
    bool tree_dist = false;          // every rank has at least 32 rows and ENLSIP_TSQR_DIST != stack
    double* dJc = nullptr;          // [J~ | r~] column major (n+1) x (n+1): stays resident for enl_dense.cuh
    std::vector<double> hR;         // host copy of dJc
    // comm
    NcclApi::Comm comm = nullptr;
    int rank = 0, nranks = 1;
    // stats
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    double ms_build = 0, ms_tsqr = 0, ms_ls = 0, ms_host = 0, ms_total = 0;
    long long n_newpoint = 0, n_ls = 0, launches = 0;
    float last_tsqr_ms = 0, last_build_ms = 0;

    ~LargeHandle() override { release(); }
    void release() {
        cudaSetDevice(device);
        if (small_prof_on() && !small_prof.empty()) {
            for (const auto& kv : small_prof)
                fprintf(stderr, "[small stage] %-24s %6lld calls %10.3f ms\n", kv.first.c_str(), kv.second.second, kv.second.first);
            small_prof.clear();
        }
        for (double* p : {ownW, owny, dA, du, dr, ds, dv, dJp, dx, dp, dT, dpart, dout, dR, dStack, dR2, dJc, dArow, dCA, dCA2, dFA,
                          dtauA, dFL, dtauL, dJQ1, dF2, dtau2, dscal, qw.vn1, qw.vn2, qw.F, qw.auxv, qw.pbest, qw.psum, ww.Vb, ww.T, ww.W, ww.W2, ww.part})
            if (p) cudaFree(p);
        for (double*& p : dvec) { if (p) cudaFree(p); p = nullptr; }
        for (double** p : {&dTA, &dTL, &dT2, &dwpart, &dP, &dPscal}) { if (*p) cudaFree(*p); *p = nullptr; }
        tree_dist = false;
        ta_valid = tl_valid = t2_valid = false;
        for (double* p : {dQ, dJkeep, dtauQ, dcu, dJrow, gown[0], gown[1]})
            if (p) cudaFree(p);
        if (dpQ) cudaFree(dpQ);
        dQ = dJkeep = dtauQ = dcu = dJrow = nullptr; dpQ = nullptr; gown[0] = gown[1] = nullptr;
        for (int* p : {dpA, dipA, dpL, dipL, dp2, dip2, dact, dbidx, qw.flags, qw.pidx})
            if (p) cudaFree(p);
        qw.drop_graphs();
        if (qw.state) cudaFree(qw.state);
        if (qw.ticket) cudaFree(qw.ticket);
        qw = enl_small::QrWork();
        ww = enl_small::WyWork();
        dArow = dCA = dCA2 = dFA = dtauA = dFL = dtauL = dJQ1 = dF2 = dtau2 = dscal = nullptr;
        dpA = dipA = dpL = dipL = dp2 = dip2 = dact = dbidx = nullptr;
        if (hst) cudaFreeHost(hst);
        if (hsti) cudaFreeHost(hsti);
        hst = nullptr; hsti = nullptr;
        if (hpin) cudaFreeHost(hpin);
        hpin = nullptr;
        if (hgrad) cudaFreeHost(hgrad);
        hgrad = nullptr;
        if (dgpart) cudaFree(dgpart);
        if (dgrad) cudaFree(dgrad);
        dgpart = dgrad = nullptr;
        dJc = nullptr;
        ownW = owny = dA = du = dr = ds = dv = dJp = dx = dp = dT = dpart = dout = dR = dStack = dR2 = nullptr;
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (e2) cudaEventDestroy(e2);
        e0 = e1 = e2 = nullptr;
        if (comm && g_nccl.ok) g_nccl.CommDestroy(comm);
        comm = nullptr;
        if (st) cudaStreamDestroy(st);
        st = nullptr;
    }
    int alloc() {
        LCU(cudaSetDevice(device));
        LCU(cudaStreamCreate(&st));
        LCU(cudaEventCreate(&e0)); LCU(cudaEventCreate(&e1)); LCU(cudaEventCreate(&e2));
        nt = tsqr_rows ? (n + TS_B - 1) / TS_B * TS_B : n;
        ld = nt + 8;
        rows_pad = ((m_local + TS_B - 1) / TS_B) * TS_B;
        if (rows_pad < TS_B) rows_pad = TS_B;
        rr_rows = nt + TS_B;   // rows of an R factor padded to a multiple of 32
        if (gv) {
            const size_t mm = (size_t)(m_local > 0 ? m_local : 1);
            if (tsqr_rows) {
                LCU(cudaMalloc(&dJrow, sizeof(double) * mm * n));
            } else {
                LCU(cudaMalloc(&dQ, sizeof(double) * mm * (n + 1)));
                LCU(cudaMalloc(&dJkeep, sizeof(double) * mm * n));
                LCU(cudaMalloc(&dtauQ, sizeof(double) * (n + 1)));
                LCU(cudaMalloc(&dpQ, sizeof(int) * (n + 1)));
                rows_pad = TS_B;      // no TSQR work matrix
            }
            LCU(cudaMalloc(&dcu, sizeof(double) * (ncu > 0 ? ncu : 1)));
        }
        LCU(cudaMalloc(&dA, sizeof(double) * rows_pad * ld));
        LCU(cudaMemsetAsync(dA, 0, sizeof(double) * rows_pad * ld, st));
        for (double** p : {&du, &dr, &ds, &dv, &dJp}) LCU(cudaMalloc(p, sizeof(double) * (m_local > 0 ? m_local : 1)));
        LCU(cudaMalloc(&dx, sizeof(double) * n));
        LCU(cudaMalloc(&dp, sizeof(double) * n));
        long long nblk = rows_pad / TS_B;
        long long nsub = (nblk + TS_FAN - 1) / TS_FAN;
        dT_subtiles = nsub > 64 ? nsub : 64;
        LCU(cudaMalloc(&dT, sizeof(double) * dT_subtiles * TS_B * TS_B));
        LCU(cudaMalloc(&dpart, sizeof(double) * LI_PARTS * 4));
        LCU(cudaMalloc(&dout, sizeof(double) * 8));
        LCU(cudaHostAlloc(&hpin, sizeof(double) * 8, cudaHostAllocDefault));
        LCU(cudaMalloc(&dgpart, sizeof(double) * LI_PARTS * (size_t)(nt + 1)));
        LCU(cudaMalloc(&dgrad, sizeof(double) * (nt + 1)));
        LCU(cudaHostAlloc(&hgrad, sizeof(double) * (n + 1), cudaHostAllocDefault));
        LCU(cudaMalloc(&dR, sizeof(double) * rr_rows * ld));
        LCU(cudaMalloc(&dJc, sizeof(double) * (size_t)(n + 1) * (n + 1)));
        hR.resize((size_t)(n + 1) * (n + 1));
        return alloc_small();
    }
    // the small stage's matrices and scratch (sizes from n, l)
    int alloc_small() {
        const size_t mt = (size_t)n + 1;
        tcap = l < n ? l : n;
        lv = (int)(mt > (size_t)l ? mt : (size_t)l) + 32;
        LCU(cudaMalloc(&dArow, sizeof(double) * (size_t)l * n));
        LCU(cudaMemsetAsync(dArow, 0, sizeof(double) * (size_t)l * n, st));
        LCU(cudaMalloc(&dCA, sizeof(double) * (size_t)(tcap + 1) * n));
        LCU(cudaMalloc(&dFA, sizeof(double) * (size_t)n * (tcap + 1)));
        LCU(cudaMalloc(&dtauA, sizeof(double) * (tcap + 1)));
        LCU(cudaMalloc(&dFL, sizeof(double) * (size_t)(tcap + 1) * (tcap + 1)));
        LCU(cudaMalloc(&dtauL, sizeof(double) * (tcap + 1)));
        LCU(cudaMalloc(&dJQ1, sizeof(double) * mt * n));
        LCU(cudaMalloc(&dF2, sizeof(double) * mt * n));
        LCU(cudaMalloc(&dtau2, sizeof(double) * mt));
        for (int** p : {&dpA, &dipA, &dpL, &dipL}) LCU(cudaMalloc(p, sizeof(int) * (tcap + 1)));
        for (int** p : {&dp2, &dip2}) LCU(cudaMalloc(p, sizeof(int) * (n + 1)));
        LCU(cudaMalloc(&dact, sizeof(int) * (l + 1)));
        for (double*& p : dvec) LCU(cudaMalloc(&p, sizeof(double) * lv));
        LCU(cudaMalloc(&dscal, sizeof(double) * 8));
        LCU(cudaHostAlloc(&hst, sizeof(double) * 4 * (size_t)lv, cudaHostAllocDefault));
        LCU(cudaHostAlloc(&hsti, sizeof(int) * 2 * (size_t)lv, cudaHostAllocDefault));
        // per-column QR scratch: n + 1 columns ([J | r], J2, and qr(C.A') while t <= n + 1); ensure_ws_capacity grows it
        if (alloc_qr_cols((int)mt) != 0) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
        LCU(cudaMalloc(&qw.auxv, sizeof(double) * enl_small::QR_NB));
        LCU(cudaMalloc(&qw.pbest, sizeof(double) * enl_small::QR_MAXPART));
        LCU(cudaMalloc(&qw.psum, sizeof(double) * enl_small::QR_PSUM_LEN));
        LCU(cudaMalloc(&qw.pidx, sizeof(int) * enl_small::QR_PIDX_LEN));
        LCU(cudaMalloc(&qw.state, sizeof(enl_small::QrState)));
        LCU(cudaMalloc(&qw.ticket, sizeof(unsigned int) * enl_small::QR_TICKET_LEN));
        LCU(cudaMemsetAsync(qw.ticket, 0, sizeof(unsigned int) * enl_small::QR_TICKET_LEN, st));
        {
            const size_t tlen = ((size_t)mt / 32 + 2) * 1024;
            for (double** p : {&dTA, &dTL, &dT2}) LCU(cudaMalloc(p, sizeof(double) * tlen));
            LCU(cudaMalloc(&dwpart, sizeof(double) * enl_small::RW_WPART_LEN));
        }
        LCU(cudaMalloc(&ww.Vb, sizeof(double) * mt * 32));
        LCU(cudaMalloc(&ww.T, sizeof(double) * 32 * 32));
        LCU(cudaMalloc(&ww.W, sizeof(double) * mt * 32));
        LCU(cudaMalloc(&ww.W2, sizeof(double) * mt * 32));
        LCU(cudaMalloc(&ww.part, sizeof(double) * mt * 32 * enl_small::GEMM_MAX_SPLITS));
        // constant bound rows of A
        const int nlo = (int)sc.lo_idx.size(), nup = (int)sc.up_idx.size();
        if (nlo + nup > 0) {
            std::vector<int> idx(sc.lo_idx);
            idx.insert(idx.end(), sc.up_idx.begin(), sc.up_idx.end());
            LCU(cudaMalloc(&dbidx, sizeof(int) * idx.size()));
            LCU(cudaMemcpyAsync(dbidx, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice, st));
            si_jac_bounds_kernel<<<(nlo + nup + 255) / 256, 256, 0, st>>>(dbidx, nlo, nup, gv ? ncu : sc.nb, n, dArow);
            LCU(cudaStreamSynchronize(st));
        }
        LCU(cudaGetLastError());
        return 0;
    }
    // QrWork's per-column arrays for `cols` columns (the contents are scratch of one factorisation)
    int alloc_qr_cols(int cols) {
        for (double* p : {qw.vn1, qw.vn2, qw.F}) if (p) cudaFree(p);
        if (qw.flags) cudaFree(qw.flags);
        qw.vn1 = qw.vn2 = qw.F = nullptr; qw.flags = nullptr; qw.cap_cols = 0;
        if (cudaMalloc(&qw.vn1, sizeof(double) * cols) != cudaSuccess || cudaMalloc(&qw.vn2, sizeof(double) * cols) != cudaSuccess ||
            cudaMalloc(&qw.F, sizeof(double) * (size_t)cols * enl_small::QR_NB) != cudaSuccess ||
            cudaMalloc(&qw.flags, sizeof(int) * cols) != cudaSuccess)
            return -1;
        qw.cap_cols = cols;
        return 0;
    }
    // Nothing bounds the working set by n: init_working_set takes every violated row, so t can reach l.  The buffers
    // sized by t are (re)allocated here, before t rows enter C.A; their contents are rebuilt by gather_active and the
    // factorisations that follow, so nothing is copied.  The small stage runs identically on every rank, so every rank
    // grows at the same call.  Starts whose working set stays within min(l, n) + 1 rows never come here.
    void ensure_ws_capacity(int t) {
        if (t <= tcap + 1) return;
        // rows of C.A the new buffers hold (never fewer than alloc_small's min(l, n) + 1, also after a failed growth)
        const int rows = std::min(l, std::max({t, 2 * (tcap + 1), std::min(l, n) + 1}));
        sm_sync();
        // until every new buffer exists the handle holds no working set: a cudaMalloc failure below throws with tcap = -1,
        // so need_ws refuses every later call and the next gather_active allocates afresh
        tcap = -1;
        for (double** p : {&dCA, &dCA2, &dFA, &dtauA, &dFL, &dtauL}) { if (*p) cudaFree(*p); *p = nullptr; }
        for (int** p : {&dpA, &dipA, &dpL, &dipL}) { if (*p) cudaFree(*p); *p = nullptr; }
        qw.drop_graphs();                 // captured QR graphs hold the old factor and scratch pointers
        sm_check(cudaMalloc(&dCA, sizeof(double) * (size_t)rows * n), "cudaMalloc");
        sm_check(cudaMalloc(&dFA, sizeof(double) * (size_t)n * rows), "cudaMalloc");
        sm_check(cudaMalloc(&dtauA, sizeof(double) * rows), "cudaMalloc");
        sm_check(cudaMalloc(&dFL, sizeof(double) * (size_t)rows * std::min(rows, n)), "cudaMalloc");   // t x min(n, t)
        sm_check(cudaMalloc(&dtauL, sizeof(double) * rows), "cudaMalloc");
        for (int** p : {&dpA, &dipA, &dpL, &dipL}) sm_check(cudaMalloc(p, sizeof(int) * rows), "cudaMalloc");
        const int qcols = std::max(rows, n + 1);       // [J | r] and J2 need n + 1 columns whatever t is
        if (qcols > qw.cap_cols && alloc_qr_cols(qcols) != 0) sm_check(cudaErrorMemoryAllocation, "cudaMalloc");
        ta_valid = tl_valid = jq1_valid = false;
        tcap = rows - 1;
        ++n_ws_grow;
    }
    // every small-stage entry point that takes t: refuse a working set the buffers do not hold
    void need_ws(int t) const {
        if (t > tcap + 1)
            throw std::runtime_error("device small stage: working set of " + std::to_string(t) + " rows exceeds the " +
                                     std::to_string(tcap + 1) + " rows of its buffers");
    }
    void qrcp(double* f, int rows, int cols, double* tau, int* jpvt) {
        const int rc = enl_small::qrcp_device(f, rows, cols, tau, jpvt, qw, st);
        if (rc < 0) throw std::runtime_error("device small stage: pivoted QR with more columns than its scratch holds");
        launches += rc;
        ++n_dev_qrcp;
    }
    int grid_rows() const {   // CTAs for the warp-per-row kernels
        long long want = (m_local + 7) / 8;
        return (int)(want < LI_PARTS ? (want > 0 ? want : 1) : LI_PARTS);
    }
    // sum-reduce dout[0..3] over the ranks, bring to the host
    int finish4(double out[4]) {
        li_finish_kernel<<<1, 128, 0, st>>>(dpart, cur_parts, dout);
        ++launches;
        if (nranks > 1) {
            int rc = g_nccl.AllReduce(dout, dout, 4, NCCL_FLOAT64, NCCL_SUM, comm, st);
            if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
        }
        // pinned landing buffer: a pageable destination costs a staging copy and an extra synchronisation per call
        LCU(cudaMemcpyAsync(hpin, dout, sizeof(double) * 4, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        for (int k = 0; k < 4; ++k) out[k] = hpin[k];
        return 0;
    }
    int cur_parts = LI_PARTS;
    double* hpin = nullptr;
    double *dgpart = nullptr, *dgrad = nullptr, *hgrad = nullptr;   // J'r partials [LI_PARTS][n+1], result [n+1], pinned copy
    bool point_factored = true;
    long long n_factor = 0;

    // row families on the TSQR path: [J | 0 | r] and the copy of J at x, J'r and r'r over CTAs and ranks -> hgrad
    int eval_at_rows(const double* x) {
        hxcur.assign(x, x + n);
        LCU(cudaMemcpyAsync(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        jq1_valid = false;
        LCU(cudaEventRecord(e0, st));
        const int parts = grid_rows();
        gv->build_rows(parts, st, n, m_local, rows_pad, row0, dx, gd[0], gd[1], jac_fd, nt, ld, dA, dJrow, dr);
        // [J'r | 0 | r'r]: the zero columns give zero sums
        li_grad_kernel<<<parts, 256, 0, st>>>(dA, ld, m_local, nt, dgpart);
        li_grad_finish_kernel<<<(nt + 8) / 8, 256, 0, st>>>(dgpart, parts, nt, dgrad);
        launches += 3;
        if (nranks > 1) {
            int rc = g_nccl.AllReduce(dgrad, dgrad, (size_t)nt + 1, NCCL_FLOAT64, NCCL_SUM, comm, st);
            if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
        }
        gv->cons(st, n, ncu, dx, gd[0], gd[1], dcu);
        gv->jac_cons(st, n, ncu, dx, gd[0], gd[1], jac_fd, dcu, dArow);
        launches += 2;
        LCU(cudaEventRecord(e1, st));
        LCU(cudaMemcpyAsync(hgrad, dgrad, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
        LCU(cudaMemcpyAsync(hgrad + n, dgrad + nt, sizeof(double), cudaMemcpyDeviceToHost, st));
        if (ncu > 0) LCU(cudaMemcpyAsync(hst, dcu, sizeof(double) * ncu, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_build_ms, e0, e1));
        ms_build += last_build_ms;
        ++n_newpoint;
        point_factored = false;
        return 0;
    }
    // r, s, u and [J | r] at x (li_build_kernel), gradient J'r and r'r reduced over CTAs and ranks -> hgrad (pinned)
    int eval_at_generic(const double* x) {
        if (tsqr_rows) return eval_at_rows(x);
        hxcur.assign(x, x + n);
        LCU(cudaMemcpyAsync(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        jq1_valid = false;
        LCU(cudaEventRecord(e0, st));
        gv->build(grid_rows(), st, n, m_local, dx, gd[0], gd[1], jac_fd, dQ, dr);
        LCU(cudaMemcpyAsync(dJkeep, dQ, sizeof(double) * (size_t)m_local * n, cudaMemcpyDeviceToDevice, st));
        // [J'r ; r'r] = [J | r]' r
        launches += 1 + enl_small::gemv_t(dQ, (int)m_local, (int)m_local, n + 1, dQ + (size_t)n * m_local, dgrad, st);
        // constraints and their Jacobian rows (bound rows of A are constant)
        gv->cons(st, n, ncu, dx, gd[0], gd[1], dcu);
        gv->jac_cons(st, n, ncu, dx, gd[0], gd[1], jac_fd, dcu, dArow);
        launches += 2;
        LCU(cudaEventRecord(e1, st));
        LCU(cudaMemcpyAsync(hgrad, dgrad, sizeof(double) * (n + 1), cudaMemcpyDeviceToHost, st));
        if (ncu > 0) LCU(cudaMemcpyAsync(hst, dcu, sizeof(double) * ncu, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_build_ms, e0, e1));
        ms_build += last_build_ms;
        ++n_newpoint;
        point_factored = false;
        return 0;
    }
    // c (l) from the family's constraints (already in hst[0..ncu)) followed by the bound rows
    void finish_cons(const double* x, double* cx) {
        for (int k = 0; k < ncu; ++k) cx[k] = hst[k];
        sc.cons(x, cx + ncu);          // sc.nb == 0 for general families: only [x - x_low ; x_upp - x]
    }
    int eval_at(const double* x) {
        LCU(cudaSetDevice(device));
        if (gv) return eval_at_generic(x);
        LCU(cudaMemcpyAsync(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        if (sc.nb > 0) {   // constraint Jacobian A(x): only the block rows depend on x
            si_jac_blocks_kernel<<<(4 * sc.nb + 255) / 256, 256, 0, st>>>(dx, sc.nb, sc.ineq ? 1 : 0, n, dArow);
            ++launches;
        }
        jq1_valid = false;
        LCU(cudaEventRecord(e0, st));
        int parts = grid_rows();
        if (m_local > 0) {
            const int nc = (n + 63) / 64;
            const size_t sh = sizeof(double) * (2 * (size_t)n + 8 * (size_t)(n + 1));
            if (jac_fd) {
                if (nc <= 1) li_build_kernel<1, true><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
                else if (nc <= 2) li_build_kernel<2, true><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
                else if (nc <= 4) li_build_kernel<4, true><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
                else if (nc <= 8) li_build_kernel<8, true><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
                else {
                    li_build_kernel<0, true><<<parts, 256, sizeof(double) * 2 * n, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);   // (n <= 3072: 48 KB)
                    li_grad_kernel<<<parts, 256, 0, st>>>(dA, ld, m_local, n, dgpart);
                    ++launches;
                }
            } else if (nc <= 1) li_build_kernel<1><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
            else if (nc <= 2) li_build_kernel<2><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
            else if (nc <= 4) li_build_kernel<4><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
            else if (nc <= 8) li_build_kernel<8><<<parts, 256, sh, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
            else {
                li_build_kernel<0><<<parts, 256, sizeof(double) * n, st>>>(dW, dy, dx, m_local, n, ld, dA, du, dr, ds, dgpart);
                li_grad_kernel<<<parts, 256, 0, st>>>(dA, ld, m_local, n, dgpart);
                ++launches;
            }
            li_grad_finish_kernel<<<(n + 8) / 8, 256, 0, st>>>(dgpart, parts, n, dgrad);
            launches += 2;
        } else {
            LCU(cudaMemsetAsync(dgrad, 0, sizeof(double) * (n + 1), st));
        }
        if (nranks > 1) {
            int rc = g_nccl.AllReduce(dgrad, dgrad, (size_t)n + 1, NCCL_FLOAT64, NCCL_SUM, comm, st);
            if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
        }
        LCU(cudaEventRecord(e1, st));
        LCU(cudaMemcpyAsync(hgrad, dgrad, sizeof(double) * (n + 1), cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_build_ms, e0, e1));
        ms_build += last_build_ms;
        ++n_newpoint;
        point_factored = false;
        return 0;
    }

    // factor the [J | r] of the last eval_at: dJc = column-major [J~ | r~] (identical on every rank), optionally
    // copied to hR.  Destroys [J | r] (in-place Householder), so it runs at most once per point.
    int factor_point(bool want_host_R = true) {
        if (point_factored) return lfail(ENLSIPB200_EINVAL, "point already factored");
        LCU(cudaSetDevice(device));
        if (gv && !tsqr_rows) {      // plain Householder QR of the column-major [J | r] (dgeqrf order), R -> [J~ | r~]
            LCU(cudaEventRecord(e1, st));
            const int rc = enl_small::qrcp_device(dQ, (int)m_local, n + 1, dtauQ, dpQ, qw, st, 1);
            if (rc < 0) return lfail(ENLSIPB200_ECUDA, "QR of [J | r]: more columns than the QR scratch holds");
            launches += rc;
            const long long ne = (long long)(n + 1) * (n + 1);
            enl_small::upper_to_square_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dQ, (int)m_local, n + 1, dJc);
            ++launches;
            jq1_valid = false;
            point_factored = true;
            LCU(cudaEventRecord(e2, st));
            if (want_host_R) LCU(cudaMemcpyAsync(hR.data(), dJc, sizeof(double) * (size_t)(n + 1) * (n + 1), cudaMemcpyDeviceToHost, st));
            LCU(cudaStreamSynchronize(st));
            LCU(cudaGetLastError());
            LCU(cudaEventElapsedTime(&last_tsqr_ms, e1, e2));
            ms_tsqr += last_tsqr_ms;
            ++n_factor;
            return 0;
        }
        LCU(cudaEventRecord(e1, st));
        LCU(cudaMemsetAsync(dR, 0, sizeof(double) * rr_rows * ld, st));
        double* dfinal = dR;
        if (nranks > 1 && tree_dist) {
            TsqrDist td;
            td.nranks = nranks; td.rank = rank; td.P = dP; td.scal = dPscal; td.ctx = this;
            td.allgather = [](void* c, const double* send, double* recv, size_t count, cudaStream_t s) {
                LargeHandle* h = static_cast<LargeHandle*>(c);
                return g_nccl.AllGather(send, recv, count, NCCL_FLOAT64, h->comm, s);
            };
            td.allreduce_sum = [](void* c, double* buf, size_t count, cudaStream_t s) {
                LargeHandle* h = static_cast<LargeHandle*>(c);
                return g_nccl.AllReduce(buf, buf, count, NCCL_FLOAT64, NCCL_SUM, h->comm, s);
            };
            const int rc = tsqr_factor(dA, ld, rows_pad, nt, dR, ld, dT, dpart, st, &td);
            if (rc < 0) return lfail(ENLSIPB200_ECUDA, "NCCL collective inside the row-sharded TSQR failed");
            launches += rc;
        } else {
            launches += tsqr_factor(dA, ld, rows_pad, nt, dR, ld, dT, dpart, st);
        }
        if (nranks > 1 && !tree_dist) {
            int rc = g_nccl.AllGather(dR, dStack, (size_t)rr_rows * ld, NCCL_FLOAT64, comm, st);
            if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllGather: ") + g_nccl.GetErrorString(rc));
            LCU(cudaMemsetAsync(dR2, 0, sizeof(double) * rr_rows * ld, st));
            launches += tsqr_factor(dStack, ld, (long long)nranks * rr_rows, nt, dR2, ld, dT, dpart, st);
            dfinal = dR2;
        }
        if (tsqr_rows) {
            const long long ne = (long long)(n + 1) * (n + 1);
            rows_unpad_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dfinal, ld, n, nt, dJc);
            ++launches;
        } else {
            const int nc = n + 1;
            dim3 grid((nc + 31) / 32, (nc + 31) / 32), block(32, 8);
            r_to_colmajor_kernel<<<grid, block, 0, st>>>(dfinal, ld, nc, dJc);
            ++launches;
        }
        jq1_valid = false;
        point_factored = true;
        LCU(cudaEventRecord(e2, st));
        if (want_host_R) LCU(cudaMemcpyAsync(hR.data(), dJc, sizeof(double) * (size_t)(n + 1) * (n + 1), cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_tsqr_ms, e1, e2));
        ms_tsqr += last_tsqr_ms;
        ++n_factor;
        return 0;
    }
    int factor_at(const double* x, bool want_host_R = true) {
        int rc = eval_at(x);
        return rc != 0 ? rc : factor_point(want_host_R);
    }

    // =========================================================================================
    // SmallBackend on the device (kernels: enl_small.cuh).  Vectors travel host <-> device per call (a few KB);
    // matrices never leave HBM.
    // =========================================================================================
    std::vector<int> hpA, hpL, hp2;     // host copies of the three permutations
    // ENLSIP_SMALL_PROF=1: per-call breakdown of the small stage (each call is followed by a stream synchronisation, so
    // the figures include what the call left in flight), printed when the handle is released
    std::map<std::string, std::pair<double, long long>> small_prof;
    static bool small_prof_on() {
        static const bool v = [] { const char* e = getenv("ENLSIP_SMALL_PROF"); return e && e[0] == '1'; }();
        return v;
    }
    struct SmallScope {
        LargeHandle* h; std::chrono::steady_clock::time_point t0; const char* name;
        explicit SmallScope(LargeHandle* hh, const char* nm = __builtin_FUNCTION())
            : h(hh), t0(std::chrono::steady_clock::now()), name(nm) { cudaSetDevice(hh->device); }
        ~SmallScope() {
            if (small_prof_on()) cudaStreamSynchronize(h->st);
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            h->ms_small += ms;
            if (small_prof_on()) { auto& e = h->small_prof[name]; e.first += ms; e.second += 1; }
        }
    };
    void sm_check(cudaError_t e, const char* what) {
        if (e != cudaSuccess) throw std::runtime_error(std::string("device small stage: ") + what + ": " + cudaGetErrorString(e));
    }
    void up(double* d, const double* src, int cnt) {   // pageable source: staged by the runtime before the call returns
        if (cnt > 0) sm_check(cudaMemcpyAsync(d, src, sizeof(double) * cnt, cudaMemcpyHostToDevice, st), "H2D");
    }
    void up_i(int* d, const int* src, int cnt) {
        if (cnt > 0) sm_check(cudaMemcpyAsync(d, src, sizeof(int) * cnt, cudaMemcpyHostToDevice, st), "H2D");
    }
    void down(int slot_off, const double* d, int cnt) {  // into the pinned staging area at hst + slot_off
        if (cnt > 0) sm_check(cudaMemcpyAsync(hst + slot_off, d, sizeof(double) * cnt, cudaMemcpyDeviceToHost, st), "D2H");
    }
    void sm_sync() {
        sm_check(cudaStreamSynchronize(st), "synchronize");
        sm_check(cudaGetLastError(), "kernel");
    }
    // T factors of a factorisation (dFA / dFL / dF2), built once per factorisation
    double* wy_t_of(const double* f, int frows, int k, const double* tau) {
        double* T = nullptr; bool* valid = nullptr;
        if (f == dFA) { T = dTA; valid = &ta_valid; }
        else if (f == dFL) { T = dTL; valid = &tl_valid; }
        else if (f == dF2) { T = dT2; valid = &t2_valid; }
        if (!T) return nullptr;
        if (!*valid) {
            const int rc = enl_small::wy_build_t_all(f, frows, k, tau, T, ww.part, (size_t)(n + 1) * 32 * enl_small::GEMM_MAX_SPLITS, st);
            if (rc < 0) return nullptr;
            launches += rc;
            *valid = true;
        }
        return T;
    }
    void k_reflect(const double* f, int frows, int k, const double* tau, double* v, int transpose) {
        launches += enl_small::reflect_vec(f, frows, k, tau, v, transpose, [&] { return wy_t_of(f, frows, k, tau); }, dwpart,
                                           qw.ticket + 1, st);
    }
    void k_trsv_upper(const double* f, int ldf, int k, double* x) {
        launches += enl_small::trsv_upper(f, ldf, k, x, false, qw.ticket + 1, st);
    }
    void k_trsv_upperT(const double* f, int ldf, int k, double* x) {
        launches += enl_small::trsv_upper(f, ldf, k, x, true, qw.ticket + 1, st);
    }
    void k_copy_pad(double* dst, const double* src, int k, int len) {
        if (len <= 0) return;
        enl_small::copy_pad_kernel<<<(len + 255) / 256, 256, 0, st>>>(dst, src, k, len);
        ++launches;
    }
    // diag(R), inverse permutation and the permutation itself of a finished factorisation -> FactorInfo
    void finish_factor(const double* f, int rows, int cols, const int* dperm, int* diperm, FactorInfo& F, std::vector<int>& hperm) {
        const int k = rows < cols ? rows : cols;
        F.rows = rows; F.cols = cols; F.k = k;
        F.diagv.assign(k, 0.0);
        F.p.assign(cols, 0);
        if (cols > 0) {
            enl_small::qr_finish_kernel<<<(cols + 255) / 256, 256, 0, st>>>(f, rows, cols, dperm, dvec[7], diperm);
            ++launches;
            down(0, dvec[7], k);
            sm_check(cudaMemcpyAsync(hsti, dperm, sizeof(int) * cols, cudaMemcpyDeviceToHost, st), "D2H");
            sm_sync();
            for (int i = 0; i < k; ++i) F.diagv[i] = hst[i];
            for (int i = 0; i < cols; ++i) F.p[i] = hsti[i];
        }
        hperm = F.p;
    }

    int new_point_eval(const double* x, double* gradf, double* rr, double* cx) override {
        int rc = eval_at(x);
        if (rc != 0) return rc;
        for (int j = 0; j < n; ++j) gradf[j] = hgrad[j];
        *rr = hgrad[n];
        if (gv) finish_cons(x, cx);
        else sc.cons(x, cx);
        return 0;
    }
    int new_point_compress(double* rt, double* gradf) override {
        int rc = factor_point(false);
        if (rc != 0) return rc;
        SmallScope sc_(this);
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        launches += enl_small::gemv_t(dJc, mt, mt, n, rtd, dvec[0], st);     // J~' r~
        down(0, rtd, mt);
        down(lv, dvec[0], n);
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        for (int r = 0; r < mt; ++r) rt[r] = hst[r];
        for (int j = 0; j < n; ++j) gradf[j] = hst[lv + j];
        return 0;
    }
    void gather_active(const int* active, int t) override {
        SmallScope sc_(this);
        ensure_ws_capacity(t);
        ca_rows = t;
        if (t <= 0) return;
        up_i(dact, active, t);
        enl_small::gather_rows_kernel<<<t, 256, 0, st>>>(dArow, n, dact, dCA);
        ++launches;
    }
    void evaluate_scaling(int t, bool scaling, double* rown) override {
        SmallScope sc_(this);
        need_ws(t);
        if (t <= 0) return;
        enl_small::row_norm_scale_kernel<<<t, 256, 0, st>>>(dCA, n, scaling ? 1 : 0, dvec[0]);
        ++launches;
        down(0, dvec[0], t);
        sm_sync();
        for (int i = 0; i < t; ++i) rown[i] = hst[i];
    }
    void rebuild_scaled_rows(const int* active, int t, const double* diag_scale) override {
        SmallScope sc_(this);
        need_ws(t);
        if (t <= 0) return;
        up_i(dact, active, t);
        up(dvec[0], diag_scale, t);
        enl_small::rebuild_scaled_rows_kernel<<<t, 256, 0, st>>>(dArow, n, dact, dvec[0], dCA);
        ++launches;
    }
    void remove_active_row(int s0) override {
        SmallScope sc_(this);
        need_ws(ca_rows);
        const int below = ca_rows - 1 - s0;
        if (below > 0) {
            if (!dCA2) sm_check(cudaMalloc(&dCA2, sizeof(double) * (size_t)(tcap + 1) * n), "cudaMalloc");
            const size_t bytes = sizeof(double) * (size_t)below * n;
            sm_check(cudaMemcpyAsync(dCA2, dCA + (size_t)(s0 + 1) * n, bytes, cudaMemcpyDeviceToDevice, st), "D2D");
            sm_check(cudaMemcpyAsync(dCA + (size_t)s0 * n, dCA2, bytes, cudaMemcpyDeviceToDevice, st), "D2D");
        }
        ca_rows -= 1;
    }
    void factor_A(int t, FactorInfo& F) override {
        SmallScope sc_(this);
        need_ws(t);
        fa_rows = n; fa_cols = t; fa_k = n < t ? n : t;
        jq1_valid = false;
        if (t > 0) {
            sm_check(cudaMemcpyAsync(dFA, dCA, sizeof(double) * (size_t)n * t, cudaMemcpyDeviceToDevice, st), "D2D");
            qrcp(dFA, n, t, dtauA, dpA);
            ta_valid = false;
        }
        finish_factor(dFA, n, t, dpA, dipA, F, hpA);
    }
    void factor_L11(FactorInfo& F) override {    // qr(F_A.R', ColumnNorm()); F_A.R is min(n, t) x t
        SmallScope sc_(this);
        const int kr = fa_k, t = fa_cols;
        need_ws(t);
        fl_rows = t; fl_cols = kr; fl_k = t < kr ? t : kr;
        if (t > 0 && kr > 0) {
            const long long ne = (long long)t * kr;
            enl_small::build_rt_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dFA, n, t, kr, dFL);
            ++launches;
            qrcp(dFL, t, kr, dtauL, dpL);
            tl_valid = false;
        }
        finish_factor(dFL, t, kr, dpL, dipL, F, hpL);
    }
    void ensure_jq1() {
        if (jq1_valid) return;
        const int mt = n + 1;
        sm_check(cudaMemcpyAsync(dJQ1, dJc, sizeof(double) * (size_t)mt * n, cudaMemcpyDeviceToDevice, st), "D2D");
        if (fa_k > 0) {
            double* TA = wy_t_of(dFA, n, fa_k, dtauA);        // all T factors of qr(C.A') at once; nullptr: per panel inside mulq_device
            launches += enl_small::mulq_device(dJQ1, mt, n, dFA, n, fa_k, dtauA, ww, st, TA, false);
            ++n_dev_mulq;
        }
        jq1_valid = true;
    }
    void factor_J2(int rankA, FactorInfo& F) override {
        SmallScope sc_(this);
        ensure_jq1();
        const int mt = n + 1, cols2 = n - rankA;
        f2_rows = mt; f2_cols = cols2; f2_k = mt < cols2 ? mt : cols2;
        if (cols2 > 0) {
            sm_check(cudaMemcpyAsync(dF2, dJQ1 + (size_t)rankA * mt, sizeof(double) * (size_t)mt * cols2, cudaMemcpyDeviceToDevice, st), "D2D");
            qrcp(dF2, mt, cols2, dtau2, dp2);
            t2_valid = false;
        }
        finish_factor(dF2, mt, cols2, dp2, dip2, F, hp2);
    }
    void first_lagrange(int prankA, int t, const Vec& gradf, const Vec& Ccx, Vec& v, Vec& u, double& grad_res) override {
        SmallScope sc_(this);
        need_ws(t);
        Vec y0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < prankA; ++i) y0[i] = -Ccx[hpA[i]];
        up(dvec[0], gradf.data(), n);
        up(dvec[1], y0.data(), t);
        k_reflect(dFA, n, fa_k, dtauA, dvec[0], 1);                      // b = Q1' gradf
        k_copy_pad(dvec[2], dvec[0], prankA, t);
        k_trsv_upper(dFA, n, prankA, dvec[2]);                           // v = R^-1 b[1:r]
        enl_small::norm_range_kernel<<<1, 1024, 0, st>>>(dvec[0], prankA, n, dscal);
        ++launches;
        k_trsv_upperT(dFA, n, prankA, dvec[1]);                          // u = R^-1 R^-T (-c[P])[1:r]
        k_trsv_upper(dFA, n, prankA, dvec[1]);
        down(0, dvec[2], t);
        down(lv, dvec[1], t);
        down(2 * lv, dscal, 1);
        sm_sync();
        v.assign(hst, hst + t);
        u.assign(hst + lv, hst + lv + t);
        grad_res = (n > prankA) ? hst[2 * lv] : 0.0;
    }
    void second_lagrange(int prankA, int t, const Vec& p_gn, Vec& v) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        up(dvec[0], p_gn.data(), n);
        launches += enl_small::gemv_n(dJc, mt, mt, n, dvec[0], 1.0, rtd, 1.0, dvec[1], st);    // s = r + J p_gn
        if (t > 0) sm_check(cudaMemsetAsync(dvec[2], 0, sizeof(double) * t, st), "memset");
        launches += enl_small::gemv_t(dJQ1, mt, mt, prankA, dvec[1], dvec[2], st);             // J1' s
        k_trsv_upper(dFA, n, prankA, dvec[2]);
        down(0, dvec[2], t);
        sm_sync();
        v.assign(hst, hst + t);
    }
    void sub_search_direction(int t, int rankA, int dimA, int dimJ2, int code, const Vec& Ccx, Vec& p, Vec& b, Vec& d) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        Vec b0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < t; ++i) b0[i] = -Ccx[hpA[i]];
        up(dvec[0], b0.data(), t);
        const double* p1;
        if (code == 1) {
            k_trsv_upperT(dFA, n, t, dvec[0]);                          // L11 p1 = -P'c
            p1 = dvec[0];
        } else {
            k_reflect(dFL, fl_rows, fl_k, dtauL, dvec[0], 1);           // b = Q2'(-P'c)
            k_copy_pad(dvec[1], dvec[0], dimA, t);
            k_trsv_upper(dFL, fl_rows, dimA, dvec[1]);                  // [R11[1:dimA] \ b[1:dimA]; 0]
            if (rankA > 0) {
                enl_small::gather_pad_kernel<<<(rankA + 255) / 256, 256, 0, st>>>(dvec[2], dvec[1], dipL, t, rankA);
                ++launches;
            }
            p1 = dvec[2];
        }
        launches += enl_small::gemv_n(dJQ1, mt, mt, rankA, p1, -1.0, rtd, -1.0, dvec[3], st);   // -J1 p1 - r
        k_reflect(dF2, mt, f2_k, dtau2, dvec[3], 1);                    // d = Q3'(...)
        const int dj = dimJ2 > 0 ? dimJ2 : 0;
        k_copy_pad(dvec[4], dvec[3], dj, dj);
        k_trsv_upper(dF2, mt, dj, dvec[4]);
        if (rankA > 0) sm_check(cudaMemcpyAsync(dvec[5], p1, sizeof(double) * rankA, cudaMemcpyDeviceToDevice, st), "D2D");
        if (f2_cols > 0) {
            enl_small::gather_pad_kernel<<<(f2_cols + 255) / 256, 256, 0, st>>>(dvec[5] + rankA, dvec[4], dip2, dj, f2_cols);
            ++launches;
        }
        k_reflect(dFA, n, fa_k, dtauA, dvec[5], 0);                     // p = Q1 [p1; p2]
        down(0, dvec[5], n);
        down(lv, dvec[3], mt);
        if (code != 1) down(2 * lv, dvec[0], t);
        sm_sync();
        p.assign(hst, hst + n);
        d.assign(hst + lv, hst + lv + mt);
        if (code == 1) b.assign(b0.begin(), b0.begin() + t);
        else b.assign(hst + 2 * lv, hst + 2 * lv + t);
    }
    void subspace_rhs(int t, const Vec& Ccx, Vec& b) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        Vec b0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < t; ++i) b0[i] = -Ccx[hpA[i]];
        up(dvec[0], b0.data(), t);
        k_reflect(dFL, fl_rows, fl_k, dtauL, dvec[0], 1);
        down(0, dvec[0], t);
        sm_sync();
        b.assign(hst, hst + t);
    }
    void subspace_d(int rankA, int dimA, int rankJ2, const Vec& b, Vec& d) override {
        SmallScope sc_(this);
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        int ra = rankA > 0 ? rankA : 0;
        if (ra > 0) {
            const int da = dimA > 0 ? dimA : 0;
            up(dvec[0], b.data(), (int)b.size());
            k_copy_pad(dvec[1], dvec[0], da, da);
            k_trsv_upper(dFL, fl_rows, da, dvec[1]);
            sm_check(cudaMemsetAsync(dvec[2], 0, sizeof(double) * ra, st), "memset");
            if (da > 0) {
                enl_small::scatter_perm_kernel<<<(da + 255) / 256, 256, 0, st>>>(dvec[2], dvec[1], dpL, da, ra);
                ++launches;
            }
        }
        launches += enl_small::gemv_n(dJQ1, mt, mt, ra, dvec[2], -1.0, rtd, -1.0, dvec[3], st);   // -(r + J1 p1)
        if (rankJ2 > 0) k_reflect(dF2, mt, f2_k, dtau2, dvec[3], 1);
        down(0, dvec[3], mt);
        sm_sync();
        d.assign(hst, hst + mt);
    }
    void products(const Vec& p, int t, Vec& Jp, Vec& Ap, Vec& active_Ap) override {
        SmallScope sc_(this);
        need_ws(t);
        const int mt = n + 1;
        up(dvec[0], p.data(), n);
        launches += enl_small::gemv_n(dJc, mt, mt, n, dvec[0], 1.0, nullptr, 0.0, dvec[1], st);
        launches += enl_small::gemv_t(dArow, n, n, l, dvec[0], dvec[2], st);
        launches += enl_small::gemv_t(dCA, n, n, t, dvec[0], dvec[3], st);
        down(0, dvec[1], mt);
        down(lv, dvec[2], l);
        down(2 * lv, dvec[3], t);
        sm_sync();
        Jp.assign(hst, hst + mt);
        Ap.assign(hst + lv, hst + lv + l);
        active_Ap.assign(hst + 2 * lv, hst + 2 * lv + t);
    }
    double At_c_norm(int t, const Vec& Ccx) override {
        SmallScope sc_(this);
        need_ws(t);
        if (ca_rows <= 0 || t <= 0) return 0.0;
        up(dvec[0], Ccx.data(), t);
        launches += enl_small::gemv_n(dCA, n, n, t, dvec[0], 1.0, nullptr, 0.0, dvec[1], st);
        enl_small::norm_range_kernel<<<1, 1024, 0, st>>>(dvec[1], 0, n, dscal);
        ++launches;
        down(0, dscal, 1);
        sm_sync();
        return hst[0];
    }

    // ---- LargeOps ----
    // the host-matrix forms of new_point! belong to the CPU test backend; the product keeps A and J~ in HBM
    // (new_point_eval / new_point_compress above) and has no host path to fall back to
    int eval_point(const double*, double*, double*, double*, double*) override {
        return lfail(ENLSIPB200_EINVAL, "host-matrix eval_point is not part of the product path");
    }
    int compress(double*, double*) override {
        return lfail(ENLSIPB200_EINVAL, "host-matrix compress is not part of the product path");
    }
    double agreed_elapsed(double local_elapsed) override {
        if (nranks <= 1) return local_elapsed;
        cudaSetDevice(device);
        hst[0] = local_elapsed / nranks;
        if (cudaMemcpyAsync(dscal, hst, sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess ||
            g_nccl.AllReduce(dscal, dscal, 1, NCCL_FLOAT64, NCCL_SUM, comm, st) != 0 ||
            cudaMemcpyAsync(hst, dscal, sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            throw std::runtime_error("agreed_elapsed: all-reduce of the wall clock failed");
        return hst[0];
    }
    int set_direction(const double*, const double* p, double sums[3]) override {
        LCU(cudaSetDevice(device));
        auto t0 = std::chrono::steady_clock::now();
        LCU(cudaMemcpyAsync(dp, p, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        cur_parts = grid_rows();
        if (gv && tsqr_rows) {
            lg_dir_rows_kernel<<<cur_parts, 256, 0, st>>>(dJrow, n, m_local, dp, dr, dJp, dpart);
        } else if (gv) {
            launches += enl_small::gemv_n(dJkeep, (int)m_local, (int)m_local, n, dp, 1.0, nullptr, 0.0, dJp, st);
            lg_dir_sums_kernel<<<cur_parts, 256, 0, st>>>(dr, dJp, m_local, dpart);
        } else {
            li_dir_kernel<<<cur_parts, 256, sizeof(double) * (jac_fd ? 2 : 1) * n, st>>>(dW, dp, dr, ds, m_local, n, dv, dJp, dpart, jac_fd, dx, du, dy);
        }
        ++launches;
        double o[4];
        int rc = finish4(o);
        if (rc != 0) return rc;
        ms_ls += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        sums[0] = o[0]; sums[1] = o[1]; sums[2] = o[2];
        return 0;
    }
    int ls_eval(double alpha, int with_coeffs, double o[4]) {
        LCU(cudaSetDevice(device));
        auto t0 = std::chrono::steady_clock::now();
        long long want = (m_local + 255) / 256;
        cur_parts = (int)(want < LI_PARTS ? (want > 0 ? want : 1) : LI_PARTS);
        if (gv) gv->ls(cur_parts, st, n, m_local, row0, dx, dp, alpha, gd[0], gd[1], dr, dJp, with_coeffs, dpart);
        else li_ls_kernel<<<cur_parts, 256, 0, st>>>(du, dv, dy, dr, dJp, m_local, alpha, with_coeffs, dpart);
        ++launches;
        int rc = finish4(o);
        if (rc != 0) return rc;
        ms_ls += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        ++n_ls;
        return 0;
    }
    int res_sq(double alpha, double* out) override {
        double o[4];
        int rc = ls_eval(alpha, 0, o);
        *out = o[0];
        return rc;
    }
    int ls_coeffs(double alpha, double out[4]) override { return ls_eval(alpha, 1, out); }
    int cons(const double* x, double* cx) override {
        if (!gv) { sc.cons(x, cx); return 0; }
        LCU(cudaSetDevice(device));
        LCU(cudaMemcpyAsync(dvec[6], x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        gv->cons(st, n, ncu, dvec[6], gd[0], gd[1], dcu);
        ++launches;
        if (ncu > 0) LCU(cudaMemcpyAsync(hst, dcu, sizeof(double) * ncu, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        finish_cons(x, cx);
        return 0;
    }
};

LargeHandle* LH(enlsipb200_large h) { return reinterpret_cast<LargeHandle*>(h); }

}  // namespace

// scratch of the known-answer hooks (enlsipb200_dense_*)
namespace {
float g_dense_ms = 0.0f;     // device time (CUDA events) of the last hook call
struct DenseScratch {
    enl_small::QrWork qw;
    enl_small::WyWork ww;
    std::vector<void*> owned;
    template <class T>
    bool get(T** p, size_t count) {
        if (cudaMalloc(p, sizeof(T) * (count > 0 ? count : 1)) != cudaSuccess) return false;
        owned.push_back(*p);
        return true;
    }
    ~DenseScratch() { for (void* p : owned) cudaFree(p); }
};
}  // namespace


// =============================================================================================
// C ABI (include/enlsip_b200.h, large-Jacobian section)
// =============================================================================================
extern "C" {

const char* enlsipb200_large_last_error(void) { return g_lerr.c_str(); }

int enlsipb200_large_create(int family, int n, long long m_local, long long m_global, int nb, int ineq,
                            const double* rho, const double* x_low, const double* x_upp, int device,
                            enlsipb200_large* out) {
    if (!out) return lfail(ENLSIPB200_EINVAL, "out is NULL");
    *out = nullptr;
    const bool want_tsqr = (family & ENLSIPB200_LARGE_FACTOR_TSQR) != 0;
    family &= ~ENLSIPB200_LARGE_FACTOR_TSQR;
    const GenericVt* gv = nullptr;
#if defined(ENL_LARGE_USER_FAMILY)
    if (family == ENLSIPB200_FAMILY_USER) gv = generic_vt<LFamUser>();
    else return lfail(ENLSIPB200_EINVAL, "this library was compiled for ENLSIPB200_FAMILY_USER only");
#else
    if (family == ENLSIPB200_FAMILY_LARGE_CHAINED_ROSENBROCK) gv = generic_vt<LFamChainedRosenbrock>();
    else if (family != ENLSIPB200_FAMILY_SINGLE_INDEX) return lfail(ENLSIPB200_EINVAL, "unknown large-regime family");
#endif
    if (gv) {
        if (n < 3) return lfail(ENLSIPB200_EINVAL, "n >= 3 required");
        if (want_tsqr) {
            if (m_global != gv->m_of(n) || m_local < 0 || m_local > m_global)
                return lfail(ENLSIPB200_EINVAL, "row families with ENLSIPB200_LARGE_FACTOR_TSQR: 0 <= m_local <= m_global = the family's m(n)");
        } else if (m_local != gv->m_of(n) || m_global != m_local) {
            return lfail(ENLSIPB200_EINVAL, "general families are not row-sharded: m_local = m_global = the family's m(n)");
        }
        nb = 0; ineq = 0; rho = nullptr;
    } else if (n < TS_B || n % TS_B != 0) {
        return lfail(ENLSIPB200_EINVAL, "n must be a positive multiple of 32");
    } else if (n > enl_small::VEC_STAGE_MAX) {
        return lfail(ENLSIPB200_EINVAL, "single-index family: n <= 6144 (x is staged in 48 KB of shared memory)");
    }
    if (m_local < 0 || m_global < m_local || nb < 0 || 4 * nb > n) return lfail(ENLSIPB200_EINVAL, "bad sizes");
    if ((long long)n + m_global < 1000)
        return lfail(ENLSIPB200_EINVAL, "n + m < 1000: second derivatives stay on in the reference (EF:2658); use the batched engine");
    if (nb > 0 && !rho) return lfail(ENLSIPB200_EINVAL, "rho is NULL");
    int ndev = 0;
    LCU(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    if (device >= ndev) return lfail(ENLSIPB200_EINVAL, "device out of range");
    LargeHandle* h = new LargeHandle();
    h->device = device;
    h->n = n; h->m = m_global; h->m_local = m_local;
    h->sc.n = n; h->sc.nb = nb; h->sc.ineq = ineq != 0;
    if (nb > 0) h->sc.rho.assign(rho, rho + nb);
    h->sc.set_bounds(x_low, x_upp);
    h->l = h->sc.l(); h->q = h->sc.q();
    h->gv = gv;
    h->tsqr_rows = gv && want_tsqr;
    h->rows_joined = !h->tsqr_rows || m_local == m_global;
    if (gv) {
        h->q = gv->q_of(n);
        h->ncu = h->q + gv->ni_of(n);
        h->l = h->ncu + h->sc.l();
    }
    if (h->l == 0) { delete h; return lfail(ENLSIPB200_EINVAL, "There must be at least one constraint (cnls_model.jl:367)"); }
    int rc = h->alloc();
    if (rc != 0) { delete h; return rc; }
    *out = reinterpret_cast<enlsipb200_large>(h);
    return 0;
}

int enlsipb200_large_destroy(enlsipb200_large hh) {
    if (!hh) return 0;
    delete LH(hh);
    return 0;
}

int enlsipb200_large_set_data(enlsipb200_large hh, int slot, const double* ptr, long long count, int on_device) {
    LargeHandle* h = LH(hh);
    if (!h || !ptr) return lfail(ENLSIPB200_EINVAL, "NULL argument");
    LCU(cudaSetDevice(h->device));
    if (h->gv) {     // general families: two free-form data slots handed to the family's functions
        if (slot < 0 || slot > 1 || count < 0) return lfail(ENLSIPB200_EINVAL, "bad slot / count");
        if (on_device) { h->gd[slot] = ptr; return 0; }
        if (h->gown[slot]) { cudaFree(h->gown[slot]); h->gown[slot] = nullptr; }
        LCU(cudaMalloc(&h->gown[slot], sizeof(double) * (count > 0 ? count : 1)));
        LCU(cudaMemcpy(h->gown[slot], ptr, sizeof(double) * count, cudaMemcpyHostToDevice));
        h->gd[slot] = h->gown[slot];
        return 0;
    }
    long long want = slot == 0 ? h->m_local * h->n : h->m_local;
    if (slot < 0 || slot > 1 || count != want) return lfail(ENLSIPB200_EINVAL, "bad slot / count");
    const double** dst = slot == 0 ? &h->dW : &h->dy;
    double** own = slot == 0 ? &h->ownW : &h->owny;
    if (on_device) { *dst = ptr; return 0; }
    if (*own && h->own_count[slot] != count) { cudaFree(*own); *own = nullptr; }
    if (!*own) LCU(cudaMalloc(own, sizeof(double) * (count > 0 ? count : 1)));
    h->own_count[slot] = count;
    LCU(cudaMemcpy(*own, ptr, sizeof(double) * count, cudaMemcpyHostToDevice));
    *dst = *own;
    return 0;
}

int enlsipb200_large_comm_id(void* id128) {
    if (!g_nccl.load()) return lfail(ENLSIPB200_ECUDA, g_nccl.err);
    NcclApi::UniqueId id;
    int rc = g_nccl.GetUniqueId(&id);
    if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(rc));
    memcpy(id128, &id, 128);
    return 0;
}

int enlsipb200_large_comm_init(enlsipb200_large hh, const void* id128, int rank, int nranks) {
    LargeHandle* h = LH(hh);
    if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return lfail(ENLSIPB200_EINVAL, "bad comm arguments");
    if (nranks == 1) {
        if (h->tsqr_rows && h->m_local != h->m) return lfail(ENLSIPB200_EINVAL, "row shards: one rank must hold all m_global rows");
        h->rank = 0; h->nranks = 1; h->rows_joined = true;
        return 0;
    }
    if (!g_nccl.load()) return lfail(ENLSIPB200_ECUDA, g_nccl.err);
    LCU(cudaSetDevice(h->device));
    NcclApi::UniqueId id;
    memcpy(&id, id128, 128);
    int rc = g_nccl.CommInitRank(&h->comm, nranks, id, rank);
    if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(rc));
    h->rank = rank; h->nranks = nranks;
    if (h->tsqr_rows) {   // row shards of a row family: every rank learns every m_local, takes its row0 and checks the total
        double* dm = nullptr;
        LCU(cudaMalloc(&dm, sizeof(double) * (nranks + 1)));
        const double mine = (double)h->m_local;
        std::vector<double> all(nranks, 0.0);
        cudaError_t ce = cudaMemcpy(dm + nranks, &mine, sizeof(double), cudaMemcpyHostToDevice);
        rc = ce == cudaSuccess ? g_nccl.AllGather(dm + nranks, dm, 1, NCCL_FLOAT64, h->comm, nullptr) : 0;
        if (ce == cudaSuccess && rc == 0) ce = cudaMemcpy(all.data(), dm, sizeof(double) * nranks, cudaMemcpyDeviceToHost);
        cudaFree(dm);
        LCU(ce);
        if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllGather: ") + g_nccl.GetErrorString(rc));
        long long below = 0, total = 0;
        for (int k = 0; k < nranks; ++k) {
            total += (long long)all[k];
            if (k < rank) below += (long long)all[k];
        }
        // every rank sees the same counts, so every rank refuses together and none waits in a later collective
        if (total != h->m)
            return lfail(ENLSIPB200_EINVAL, "row shards: the ranks hold " + std::to_string(total) + " rows, m_global is " +
                                                std::to_string(h->m));
        h->row0 = below;
        h->rows_joined = true;
    }
    LCU(cudaMalloc(&h->dStack, sizeof(double) * (size_t)nranks * h->rr_rows * h->ld));
    LCU(cudaMalloc(&h->dR2, sizeof(double) * (size_t)h->rr_rows * h->ld));
    {   // the cross-rank stage as one more level of every panel's tree (TsqrDist) needs a 32-row block on every rank
        const size_t prow = (size_t)(nranks > 8 ? nranks : 8) * TS_B;
        LCU(cudaMalloc(&h->dP, sizeof(double) * prow * h->ld));
        LCU(cudaMemset(h->dP, 0, sizeof(double) * prow * h->ld));
        LCU(cudaMalloc(&h->dPscal, sizeof(double) * 2));
        const double mine = (h->rows_pad < TS_B || (h->gv && !h->tsqr_rows)) ? 1.0 : 0.0;
        LCU(cudaMemcpy(h->dPscal, &mine, sizeof(double), cudaMemcpyHostToDevice));
        rc = g_nccl.AllReduce(h->dPscal, h->dPscal, 1, NCCL_FLOAT64, NCCL_SUM, h->comm, nullptr);
        if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
        double short_ranks = 0.0;
        LCU(cudaMemcpy(&short_ranks, h->dPscal, sizeof(double), cudaMemcpyDeviceToHost));
        const char* e = getenv("ENLSIP_TSQR_DIST");
        h->tree_dist = short_ranks == 0.0 && !(e && e[0] == 's');
    }
    {   // the T-factor buffer also serves the second-stage TSQR of the nranks stacked R factors: one 32 x 32 per subtile
        const long long nsub2 = ((long long)nranks * h->rr_rows / TS_B + TS_FAN - 1) / TS_FAN;
        if (nsub2 > h->dT_subtiles) {
            LCU(cudaFree(h->dT));
            h->dT = nullptr;
            LCU(cudaMalloc(&h->dT, sizeof(double) * nsub2 * TS_B * TS_B));
            h->dT_subtiles = nsub2;
        }
    }
    return 0;
}

int enlsipb200_large_solve(enlsipb200_large hh, const double* x0, const enlsipb200_options* o, double* x, double* f,
                           int* exit_code, int* status, int* iters, int* nact, int* active, double* trace,
                           int trace_cap) {
    LargeHandle* h = LH(hh);
    if (!h || !x0 || !o || !x || !f) return lfail(ENLSIPB200_EINVAL, "NULL argument");
    if (!h->gv && (!h->dW || !h->dy)) return lfail(ENLSIPB200_EINVAL, "family data (W, y) not set");
    if (!h->rows_joined) return lfail(ENLSIPB200_EINVAL, "row shard (m_local < m_global) not joined: enlsipb200_large_comm_init first");
    h->jac_fd = (o->jac_mode == ENLSIPB200_JAC_FORWARD_DIFF) ? 1 : 0;
    if (h->jac_fd && !h->gv && h->n > 3072)
        return lfail(ENLSIPB200_EINVAL, "forward-difference Jacobians of the single-index family: n <= 3072 (x and the steps are staged in 48 KB of shared memory)");
    LargeOptions opt;
    opt.max_iter = o->max_iter;
    opt.scaling = o->scaling;
    opt.time_limit = o->time_limit;
    double abs_tol = (o->abs_tol == o->abs_tol) ? o->abs_tol : EPS;
    double rel_tol = (o->rel_tol == o->rel_tol) ? o->rel_tol : sqrt(abs_tol);
    opt.eps_rel = rel_tol;
    opt.eps_c = (o->c_tol == o->c_tol) ? o->c_tol : rel_tol;
    opt.eps_x = (o->x_tol == o->x_tol) ? o->x_tol : rel_tol;
    auto t0 = std::chrono::steady_clock::now();
    LargeResult R;
    try {
        LargeSolver S(*h, opt, h);      // h is the SmallBackend: the small stage runs on the device
        R = S.solve(x0, trace != nullptr && trace_cap > 0);
    } catch (const std::exception& e) {
        g_lerr = e.what();
        return ENLSIPB200_ECUDA;
    }
    double total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    h->ms_total += total;
    memcpy(x, R.x.data(), sizeof(double) * h->n);
    *f = R.f;
    if (exit_code) *exit_code = R.exit_code;
    if (status) *status = R.status;
    if (iters) *iters = R.iterations;
    if (nact) *nact = R.nact;
    if (active)
        for (int i = 0; i < h->l; ++i) active[i] = i < R.nact ? R.active[i] : 0;
    if (trace && trace_cap > 0) {
        int rows = (int)R.trace.size();
        const int n = h->n;
        for (int k = 0; k < rows && k < trace_cap; ++k) {
            double* tr = trace + (size_t)k * (ENLSIPB200_TRACE_HDR + n);
            const IterTraceL& t = R.trace[k];
            tr[0] = t.f_new; tr[1] = t.t; tr[2] = t.rankA; tr[3] = t.rankJ2; tr[4] = t.dimA; tr[5] = t.dimJ2;
            tr[6] = t.code; tr[7] = t.alpha; tr[8] = t.p_norm; tr[9] = t.index_del; tr[10] = t.exit_code;
            tr[11] = t.active_cx_sum; tr[12] = t.progress; tr[13] = t.k; tr[14] = 0; tr[15] = 0;
            memcpy(tr + ENLSIPB200_TRACE_HDR, R.trace_x.data() + (size_t)k * n, sizeof(double) * n);
        }
    }
    return 0;
}

int enlsipb200_large_factor(enlsipb200_large hh, const double* x, double* R, float* build_ms, float* tsqr_ms) {
    LargeHandle* h = LH(hh);
    if (!h || !x) return lfail(ENLSIPB200_EINVAL, "NULL argument");
    if (!h->gv && (!h->dW || !h->dy)) return lfail(ENLSIPB200_EINVAL, "family data (W, y) not set");
    if (!h->rows_joined) return lfail(ENLSIPB200_EINVAL, "row shard (m_local < m_global) not joined: enlsipb200_large_comm_init first");
    int rc = h->factor_at(x);
    if (rc != 0) return rc;
    const int nc = h->n + 1;
    if (R)
        for (int r = 0; r < nc; ++r)
            for (int c = 0; c < nc; ++c) R[(size_t)r * nc + c] = h->hR[(size_t)c * nc + r];
    if (build_ms) *build_ms = h->last_build_ms;
    if (tsqr_ms) *tsqr_ms = h->last_tsqr_ms;
    return 0;
}

int enlsipb200_large_stats(enlsipb200_large hh, double* out, int count) {
    LargeHandle* h = LH(hh);
    if (!h || !out) return lfail(ENLSIPB200_EINVAL, "NULL argument");
    double v[13] = {(double)h->n_newpoint, h->ms_build, h->ms_tsqr, h->ms_ls, h->ms_total, (double)h->n_ls,
                    (double)h->launches, (double)h->rows_pad, (double)h->n_dev_qrcp, (double)h->n_dev_mulq, h->ms_small,
                    (double)h->n_factor, (double)h->n_ws_grow};
    for (int i = 0; i < count && i < 13; ++i) out[i] = v[i];
    return 0;
}

// ---- known-answer hooks of enl_small.cuh (tests/test_gpu_kat.py, tests/test_gpu_dense_dispatch.py) ----
// qrcp_device on a copy of f: dgeqp3 (nopivot = 0, jpvt returned) or dgeqrf (nopivot = 1, jpvt may be NULL)
static int dense_qr_run(int rows, int cols, double* f, double* tau, int* jpvt, int device, int nopivot) {
    if (rows < 1 || cols < 1 || !f || !tau || (!jpvt && !nopivot)) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    LCU(cudaSetDevice(device));
    DenseScratch S;
    double *df = nullptr, *dtau = nullptr;
    int* dp = nullptr;
    const int k = rows < cols ? rows : cols;
    bool ok = S.get(&df, (size_t)rows * cols) && S.get(&dtau, k) && S.get(&dp, cols) && S.get(&S.qw.vn1, cols) &&
              S.get(&S.qw.vn2, cols) && S.get(&S.qw.F, (size_t)cols * enl_small::QR_NB) && S.get(&S.qw.auxv, enl_small::QR_NB) &&
              S.get(&S.qw.flags, cols) && S.get(&S.qw.state, 1) && S.get(&S.qw.ticket, enl_small::QR_TICKET_LEN) &&
              S.get(&S.qw.pbest, enl_small::QR_MAXPART) && S.get(&S.qw.psum, enl_small::QR_PSUM_LEN) &&
              S.get(&S.qw.pidx, enl_small::QR_PIDX_LEN);
    if (!ok) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    S.qw.cap_cols = cols;
    LCU(cudaMemcpy(df, f, sizeof(double) * (size_t)rows * cols, cudaMemcpyHostToDevice));
    LCU(cudaMemset(dtau, 0, sizeof(double) * k));
    cudaStream_t hs = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    LCU(cudaStreamCreate(&hs));
    LCU(cudaEventCreate(&ev0)); LCU(cudaEventCreate(&ev1));
    LCU(cudaEventRecord(ev0, hs));
    enl_small::qrcp_device(df, rows, cols, dtau, dp, S.qw, hs, nopivot);
    LCU(cudaEventRecord(ev1, hs));
    cudaError_t es = cudaStreamSynchronize(hs);
    if (es == cudaSuccess) es = cudaGetLastError();
    cudaEventElapsedTime(&g_dense_ms, ev0, ev1);
    S.qw.drop_graphs();
    cudaEventDestroy(ev0); cudaEventDestroy(ev1); cudaStreamDestroy(hs);
    LCU(es);
    LCU(cudaMemcpy(f, df, sizeof(double) * (size_t)rows * cols, cudaMemcpyDeviceToHost));
    LCU(cudaMemcpy(tau, dtau, sizeof(double) * k, cudaMemcpyDeviceToHost));
    if (jpvt) LCU(cudaMemcpy(jpvt, dp, sizeof(int) * cols, cudaMemcpyDeviceToHost));
    return 0;
}

int enlsipb200_dense_qrcp(int rows, int cols, double* f, double* tau, int* jpvt, int device) {
    return dense_qr_run(rows, cols, f, tau, jpvt, device, 0);
}

int enlsipb200_dense_qr(int rows, int cols, double* f, double* tau, int device) {
    return dense_qr_run(rows, cols, f, tau, nullptr, device, 1);
}

float enlsipb200_dense_last_ms(void) { return g_dense_ms; }

int enlsipb200_dense_mulq(int mr, int nq, int k, const double* f, const double* tau, double* M, int device) {
    if (mr < 1 || nq < 1 || k < 0 || k > nq || !f || !tau || !M) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    LCU(cudaSetDevice(device));
    DenseScratch S;
    double *df = nullptr, *dtau = nullptr, *dM = nullptr, *dTall = nullptr;
    bool ok = S.get(&df, (size_t)nq * (k > 0 ? k : 1)) && S.get(&dtau, k) && S.get(&dM, (size_t)mr * nq) &&
              S.get(&dTall, ((size_t)nq / 32 + 2) * 1024) &&
              S.get(&S.ww.Vb, (size_t)nq * 32) && S.get(&S.ww.T, 32 * 32) && S.get(&S.ww.W, (size_t)mr * 32) &&
              S.get(&S.ww.W2, (size_t)mr * 32) && S.get(&S.ww.part, (size_t)mr * 32 * enl_small::GEMM_MAX_SPLITS);
    if (!ok) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(df, f, sizeof(double) * (size_t)nq * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dtau, tau, sizeof(double) * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dM, M, sizeof(double) * (size_t)mr * nq, cudaMemcpyHostToDevice));
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    LCU(cudaEventCreate(&ev0)); LCU(cudaEventCreate(&ev1));
    LCU(cudaEventRecord(ev0, nullptr));
    enl_small::mulq_device(dM, mr, nq, df, nq, k, dtau, S.ww, nullptr, dTall, true);
    LCU(cudaEventRecord(ev1, nullptr));
    cudaError_t es = cudaDeviceSynchronize();
    if (es == cudaSuccess) es = cudaGetLastError();
    cudaEventElapsedTime(&g_dense_ms, ev0, ev1);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    LCU(es);
    LCU(cudaMemcpy(M, dM, sizeof(double) * (size_t)mr * nq, cudaMemcpyDeviceToHost));
    return 0;
}

// Known-answer hook for the vector kernels of the small stage (tests/test_gpu_kat.py).  kind 0: v <- Q' v, 1: v <- Q v
// (f: frows x k reflectors in dgeqrf layout, tau [k], v [frows]; compact-WY cooperative kernel);
// kind 2: v <- UpperTriangular(f[0:k, 0:k]) \ v, 3: v <- UpperTriangular(f[0:k, 0:k])' \ v (f: frows x k, v [k];
// multi-CTA cooperative kernels).  Kinds 4-7: the operations of kinds 0-3 with the kernel chosen by size as the solver
// chooses it (enl_small::reflect_vec / trsv_upper).
int enlsipb200_dense_vecop(int kind, int frows, int k, const double* f, const double* tau, double* v, int device) {
    if (kind < 0 || kind > 7 || frows < 1 || k < 1 || k > frows || !f || !v || ((kind & 3) < 2 && !tau)) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    const bool dispatched = kind >= 4;
    kind &= 3;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    LCU(cudaSetDevice(device));
    DenseScratch S;
    const int vlen = kind < 2 ? frows : k;
    double *df = nullptr, *dtau = nullptr, *dv = nullptr, *dTall = nullptr, *dscr = nullptr, *dwp = nullptr;
    unsigned int* dbar = nullptr;
    const size_t scr = (size_t)1024 * ((frows + enl_small::WY_SLAB - 1) / enl_small::WY_SLAB) * 8;
    bool ok = S.get(&df, (size_t)frows * k) && S.get(&dtau, k) && S.get(&dv, vlen) && S.get(&dTall, ((size_t)k / 32 + 2) * 1024) &&
              S.get(&dscr, scr) && S.get(&dwp, enl_small::RW_WPART_LEN) && S.get(&dbar, 16);
    if (!ok) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(df, f, sizeof(double) * (size_t)frows * k, cudaMemcpyHostToDevice));
    if (kind < 2) LCU(cudaMemcpy(dtau, tau, sizeof(double) * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dv, v, sizeof(double) * vlen, cudaMemcpyHostToDevice));
    LCU(cudaMemset(dbar, 0, sizeof(unsigned int) * 16));
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    LCU(cudaEventCreate(&ev0)); LCU(cudaEventCreate(&ev1));
    int rc = 0;
    if (dispatched) {
        LCU(cudaEventRecord(ev0, nullptr));
        if (kind < 2) {
            auto t_of = [&]() -> const double* {
                return enl_small::wy_build_t_all(df, frows, k, dtau, dTall, dscr, scr, nullptr) >= 0 ? dTall : nullptr;
            };
            rc = enl_small::reflect_vec(df, frows, k, dtau, dv, kind == 0 ? 1 : 0, t_of, dwp, dbar, nullptr);
        } else {
            rc = enl_small::trsv_upper(df, frows, k, dv, kind == 3, dbar, nullptr);
        }
    } else if (kind < 2) {
        rc = enl_small::wy_build_t_all(df, frows, k, dtau, dTall, dscr, scr, nullptr);
        LCU(cudaEventRecord(ev0, nullptr));
        if (rc >= 0) rc = enl_small::reflect_vec_wy(df, frows, k, dTall, dv, kind == 0 ? 1 : 0, dwp, dbar, nullptr);
    } else {
        LCU(cudaEventRecord(ev0, nullptr));
        rc = enl_small::trsv_coop(df, frows, k, dv, kind == 3, dbar, nullptr);
    }
    LCU(cudaEventRecord(ev1, nullptr));
    cudaError_t es = cudaDeviceSynchronize();
    if (es == cudaSuccess) es = cudaGetLastError();
    cudaEventElapsedTime(&g_dense_ms, ev0, ev1);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    LCU(es);
    if (rc < 0) return lfail(ENLSIPB200_EINVAL, "shape not supported by the cooperative kernel");
    LCU(cudaMemcpy(v, dv, sizeof(double) * vlen, cudaMemcpyDeviceToHost));
    return 0;
}

// Known-answer hook for the small stage's gemv (enl_small::gemv_n / gemv_t).  A: rows x cols, column major, lda >= rows.
// trans 0: y [rows] = alpha A x + beta y0 (x [cols]; y0 [rows] or NULL = 0); trans 1: y [cols] = A' x (x [rows]; alpha,
// y0 and beta unused: gemv_t forms the plain product).
int enlsipb200_dense_gemv(int trans, int rows, int cols, const double* A, int lda, const double* x, double alpha,
                          const double* y0, double beta, double* y, int device) {
    if ((trans != 0 && trans != 1) || rows < 1 || cols < 1 || lda < rows || !A || !x || !y) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    LCU(cudaSetDevice(device));
    DenseScratch S;
    const int xlen = trans ? rows : cols, ylen = trans ? cols : rows;
    const bool with_y0 = !trans && y0;
    double *dA = nullptr, *dx = nullptr, *dy0 = nullptr, *dy = nullptr;
    bool ok = S.get(&dA, (size_t)lda * cols) && S.get(&dx, xlen) && S.get(&dy, ylen) && (!with_y0 || S.get(&dy0, ylen));
    if (!ok) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(dA, A, sizeof(double) * (size_t)lda * cols, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dx, x, sizeof(double) * xlen, cudaMemcpyHostToDevice));
    if (with_y0) LCU(cudaMemcpy(dy0, y0, sizeof(double) * ylen, cudaMemcpyHostToDevice));
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    LCU(cudaEventCreate(&ev0)); LCU(cudaEventCreate(&ev1));
    LCU(cudaEventRecord(ev0, nullptr));
    if (trans) enl_small::gemv_t(dA, lda, rows, cols, dx, dy, nullptr);
    else enl_small::gemv_n(dA, lda, rows, cols, dx, alpha, dy0, beta, dy, nullptr);
    LCU(cudaEventRecord(ev1, nullptr));
    cudaError_t es = cudaDeviceSynchronize();
    if (es == cudaSuccess) es = cudaGetLastError();
    cudaEventElapsedTime(&g_dense_ms, ev0, ev1);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    LCU(es);
    LCU(cudaMemcpy(y, dy, sizeof(double) * ylen, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
