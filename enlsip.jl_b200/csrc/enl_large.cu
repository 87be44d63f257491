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
#include "enl_small_device.cuh"
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
        if (FD) dls[j] = __dmul_rn(fmax(fabs(x[j]), 1.0), SQRT_EPS);
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
        if (fd) dls[j] = __dmul_rn(fmax(fabs(xcur[j]), 1.0), SQRT_EPS);
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
// the m-sized backend: LargeOps and the DevicePoint of the small stage
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

using enl_small::DevBuf;
using enl_small::PinnedBuf;
using enl_small::dev_alloc;
using enl_small::pinned_alloc;

struct LargeHandle : LargeOps, DevicePoint {
    int device = 0;
    DeviceSmall small{*this};         // the small stage on the compressed problem (enl_small_device.cuh)

    // general row families (enl_large_generic.cuh): gv != nullptr; [J | r] column major in dQ, factored without pivoting
    const GenericVt* gv = nullptr;
    int ncu = 0;                      // the family's own constraints (equalities + inequalities); bounds follow
    DevBuf<double> dQ, dJkeep, dtauQ, dcu;
    DevBuf<int> dpQ;
    const double* gd[2] = {nullptr, nullptr};     // family data slots
    DevBuf<double> gown[2];
    int jac_fd = 0;                   // forward-difference Jacobians requested (cnls_model.jl:65-82)
    // ENLSIPB200_LARGE_FACTOR_TSQR: [J | 0 | r] row major in dA (nt columns for J, nt = n rounded up to 32), factored by
    // tsqr_factor like the single-index family; a row-major copy of J (dJrow) serves J p.  This rank holds the global rows
    // row0 .. row0 + m_local - 1; rows_joined: the shards are known to cover m (always so when m_local = m).
    bool tsqr_rows = false, rows_joined = true;
    long long row0 = 0;
    DevBuf<double> dJrow;
    int nt = 0;                       // columns the TSQR factors: n rounded up to 32 on that path, n otherwise
    // ENLSIPB200_LARGE_MIDSIZE: second derivatives on (Newton steps, EF:348-423).  The Hessian's inputs: r at x; x / lam /
    // active; the bound values (x_low then x_upp, in the order of dbidx).  Allocated with the handle, midsize handles only.
    bool midsize = false;
    DevBuf<double> dhr, dxn, dlamn, dbval;
    DevBuf<int> dactn, dbidx;
    cudaEvent_t eh0 = nullptr, eh1 = nullptr;
    double ms_hess = 0;
    long long m_local = 0, rows_pad = 0, dT_subtiles = 0;
    int ld = 0, rr_rows = 0;
    SingleIndexConstraints sc;
    cudaStream_t st = nullptr;
    // device data
    const double* dW = nullptr;
    const double* dy = nullptr;
    DevBuf<double> ownW, owny;
    long long own_count[2] = {0, 0};
    DevBuf<double> dA, du, dr, ds, dv, dJp, dx, dp, dT, dpart, dout, dR, dStack, dR2;
    DevBuf<double> dP;               // cross-rank level of the TSQR tree: max(nranks, 8) * 32 rows x ld (enl_tsqr.cuh, TsqrDist)
    DevBuf<double> dPscal;
    bool tree_dist = false;          // every rank has at least 32 rows and ENLSIP_TSQR_DIST != stack
    DevBuf<double> dJc;              // [J~ | r~] column major (n+1) x (n+1): stays resident for the small stage
    std::vector<double> hR;          // host copy of dJc
    int cur_parts = LI_PARTS;
    PinnedBuf<double> hpin;          // pinned landing buffer of finish4
    DevBuf<double> dgpart, dgrad;    // J'r partials [LI_PARTS][n+1], result [n+1]
    PinnedBuf<double> hgrad;         // pinned copy of dgrad
    bool point_factored = true;
    // comm
    NcclApi::Comm comm = nullptr;
    int rank = 0, nranks = 1;
    // stats
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    double ms_build = 0, ms_tsqr = 0, ms_ls = 0, ms_host = 0, ms_total = 0;
    long long n_newpoint = 0, n_ls = 0, n_factor = 0, launches = 0;
    float last_tsqr_ms = 0, last_build_ms = 0;

    // the buffers free themselves after this, on this device
    ~LargeHandle() override {
        cudaSetDevice(device);
        for (cudaEvent_t e : {e0, e1, e2, eh0, eh1})
            if (e) cudaEventDestroy(e);
        if (comm && g_nccl.ok) g_nccl.CommDestroy(comm);
        if (st) cudaStreamDestroy(st);
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
        const size_t mm = (size_t)(m_local > 0 ? m_local : 1);
        if (gv) {
            if (tsqr_rows) {
                LCU(dev_alloc(dJrow, mm * n));
            } else {
                LCU(dev_alloc(dQ, mm * (n + 1)));
                LCU(dev_alloc(dJkeep, mm * n));
                LCU(dev_alloc(dtauQ, n + 1));
                LCU(dev_alloc(dpQ, n + 1));
                rows_pad = TS_B;      // no TSQR work matrix
            }
            LCU(dev_alloc(dcu, ncu > 0 ? ncu : 1));
        }
        LCU(dev_alloc(dA, rows_pad * ld));
        LCU(cudaMemsetAsync(dA.get(), 0, sizeof(double) * rows_pad * ld, st));
        for (DevBuf<double>* p : {&du, &dr, &ds, &dv, &dJp}) LCU(dev_alloc(*p, mm));
        LCU(dev_alloc(dx, n));
        LCU(dev_alloc(dp, n));
        long long nblk = rows_pad / TS_B;
        long long nsub = (nblk + TS_FAN - 1) / TS_FAN;
        dT_subtiles = nsub > 64 ? nsub : 64;
        LCU(dev_alloc(dT, dT_subtiles * TS_B * TS_B));
        LCU(dev_alloc(dpart, LI_PARTS * 4));
        LCU(dev_alloc(dout, 8));
        LCU(pinned_alloc(hpin, 8));
        LCU(dev_alloc(dgpart, LI_PARTS * (size_t)(nt + 1)));
        LCU(dev_alloc(dgrad, nt + 1));
        LCU(pinned_alloc(hgrad, n + 1));
        LCU(dev_alloc(dR, rr_rows * ld));
        LCU(dev_alloc(dJc, (size_t)(n + 1) * (n + 1)));
        hR.resize((size_t)(n + 1) * (n + 1));
        LCU(small.alloc(device, n, l, midsize, st, dJc.get()));
        // constant bound rows of A
        const int nlo = (int)sc.lo_idx.size(), nup = (int)sc.up_idx.size();
        if (nlo + nup > 0) {
            std::vector<int> idx(sc.lo_idx);
            idx.insert(idx.end(), sc.up_idx.begin(), sc.up_idx.end());
            LCU(dev_alloc(dbidx, idx.size()));
            LCU(cudaMemcpyAsync(dbidx.get(), idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice, st));
            si_jac_bounds_kernel<<<(nlo + nup + 255) / 256, 256, 0, st>>>(dbidx.get(), nlo, nup, gv ? ncu : sc.nb, n, small.dArow.get());
            if (midsize) {
                std::vector<double> val(sc.lo_val);
                val.insert(val.end(), sc.up_val.begin(), sc.up_val.end());
                LCU(dev_alloc(dbval, val.size()));
                LCU(cudaMemcpyAsync(dbval.get(), val.data(), sizeof(double) * val.size(), cudaMemcpyHostToDevice, st));
            }
            LCU(cudaStreamSynchronize(st));
        }
        if (midsize) {
            LCU(dev_alloc(dhr, (size_t)m_local));
            LCU(dev_alloc(dxn, n));
            LCU(dev_alloc(dlamn, l + 1));
            LCU(dev_alloc(dactn, l + 1));
            LCU(cudaEventCreate(&eh0)); LCU(cudaEventCreate(&eh1));
        }
        LCU(cudaGetLastError());
        return 0;
    }
    int grid_rows() const {   // CTAs for the warp-per-row kernels
        long long want = (m_local + 7) / 8;
        return (int)(want < LI_PARTS ? (want > 0 ? want : 1) : LI_PARTS);
    }
    int all_reduce_sum(double* buf, size_t count) {
        if (nranks <= 1) return 0;
        const int rc = g_nccl.AllReduce(buf, buf, count, NCCL_FLOAT64, NCCL_SUM, comm, st);
        return rc != 0 ? lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc)) : 0;
    }
    // sum-reduce dout[0..3] over the ranks, bring to the host
    int finish4(double out[4]) {
        li_finish_kernel<<<1, 128, 0, st>>>(dpart.get(), cur_parts, dout.get());
        ++launches;
        if (int rc = all_reduce_sum(dout.get(), 4)) return rc;
        // pinned landing buffer: a pageable destination costs a staging copy and an extra synchronisation per call
        LCU(cudaMemcpyAsync(hpin.get(), dout.get(), sizeof(double) * 4, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        for (int k = 0; k < 4; ++k) out[k] = hpin[k];
        return 0;
    }

    // single-index family: r, s, u and [J | r] at x (li_build_kernel), J'r and r'r over CTAs and ranks -> dgrad
    int build_single_index(int parts) {
        if (m_local > 0) {
            // NC register pairs of J'r per lane (n <= 64 NC); 0: n > 512, J'r by li_grad_kernel
            static const decltype(&li_build_kernel<0>) kern[2][5] = {
                {li_build_kernel<0>, li_build_kernel<1>, li_build_kernel<2>, li_build_kernel<4>, li_build_kernel<8>},
                {li_build_kernel<0, true>, li_build_kernel<1, true>, li_build_kernel<2, true>, li_build_kernel<4, true>,
                 li_build_kernel<8, true>}};
            const int nc = (n + 63) / 64, k = nc <= 1 ? 1 : nc <= 2 ? 2 : nc <= 4 ? 3 : nc <= 8 ? 4 : 0;
            // k == 0 with forward differences: n <= 3072 (48 KB)
            const size_t sh = sizeof(double) * (k ? 2 * (size_t)n + 8 * (size_t)(n + 1) : (jac_fd ? 2 : 1) * (size_t)n);
            kern[jac_fd][k]<<<parts, 256, sh, st>>>(dW, dy, dx.get(), m_local, n, ld, dA.get(), du.get(), dr.get(), ds.get(), dgpart.get());
            if (k == 0) {
                li_grad_kernel<<<parts, 256, 0, st>>>(dA.get(), ld, m_local, n, dgpart.get());
                ++launches;
            }
            li_grad_finish_kernel<<<(n + 8) / 8, 256, 0, st>>>(dgpart.get(), parts, n, dgrad.get());
            launches += 2;
        } else {
            LCU(cudaMemsetAsync(dgrad.get(), 0, sizeof(double) * (n + 1), st));
        }
        return all_reduce_sum(dgrad.get(), (size_t)n + 1);
    }
    // row families on the TSQR path: [J | 0 | r] and the copy of J at x, [J'r | 0 | r'r] over CTAs and ranks -> dgrad
    int build_rows(int parts) {
        gv->build_rows(parts, st, n, m_local, rows_pad, row0, dx.get(), gd[0], gd[1], jac_fd, nt, ld, dA.get(), dJrow.get(), dr.get());
        // the zero columns give zero sums
        li_grad_kernel<<<parts, 256, 0, st>>>(dA.get(), ld, m_local, nt, dgpart.get());
        li_grad_finish_kernel<<<(nt + 8) / 8, 256, 0, st>>>(dgpart.get(), parts, nt, dgrad.get());
        launches += 3;
        return all_reduce_sum(dgrad.get(), (size_t)nt + 1);
    }
    // other row families: column-major [J | r] at x and a copy of J, [J'r ; r'r] = [J | r]' r -> dgrad
    int build_generic(int parts) {
        gv->build(parts, st, n, m_local, dx.get(), gd[0], gd[1], jac_fd, dQ.get(), dr.get());
        LCU(cudaMemcpyAsync(dJkeep.get(), dQ.get(), sizeof(double) * (size_t)m_local * n, cudaMemcpyDeviceToDevice, st));
        launches += 1 + enl_small::gemv_t(dQ.get(), (int)m_local, (int)m_local, n + 1, dQ.get() + (size_t)n * m_local, dgrad.get(), st);
        return 0;
    }
    // new_point! at x: the family's build and reduce step, then (row families) the constraints and their Jacobian rows
    // (the bound rows of A are constant); J'r and r'r -> hgrad (pinned), the family's constraints -> small.hst
    int eval_at(const double* x) {
        LCU(cudaSetDevice(device));
        LCU(cudaMemcpyAsync(dx.get(), x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        if (!gv && sc.nb > 0) {   // constraint Jacobian A(x): only the block rows depend on x
            si_jac_blocks_kernel<<<(4 * sc.nb + 255) / 256, 256, 0, st>>>(dx.get(), sc.nb, sc.ineq ? 1 : 0, n, small.dArow.get());
            ++launches;
        }
        LCU(cudaEventRecord(e0, st));
        const int parts = grid_rows();
        const int rc = !gv ? build_single_index(parts) : tsqr_rows ? build_rows(parts) : build_generic(parts);
        if (rc != 0) return rc;
        if (gv) {
            gv->cons(st, n, ncu, dx.get(), gd[0], gd[1], dcu.get());
            gv->jac_cons(st, n, ncu, dx.get(), gd[0], gd[1], jac_fd, dcu.get(), small.dArow.get());
            launches += 2;
        }
        LCU(cudaEventRecord(e1, st));
        if (tsqr_rows) {
            LCU(cudaMemcpyAsync(hgrad.get(), dgrad.get(), sizeof(double) * n, cudaMemcpyDeviceToHost, st));
            LCU(cudaMemcpyAsync(hgrad.get() + n, dgrad.get() + nt, sizeof(double), cudaMemcpyDeviceToHost, st));
        } else {
            LCU(cudaMemcpyAsync(hgrad.get(), dgrad.get(), sizeof(double) * (n + 1), cudaMemcpyDeviceToHost, st));
        }
        if (gv && ncu > 0) LCU(cudaMemcpyAsync(small.hst.get(), dcu.get(), sizeof(double) * ncu, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_build_ms, e0, e1));
        ms_build += last_build_ms;
        ++n_newpoint;
        point_factored = false;
        return 0;
    }
    // c (l) from the family's constraints (already in small.hst[0..ncu)) followed by the bound rows
    void finish_cons(const double* x, double* cx) {
        for (int k = 0; k < ncu; ++k) cx[k] = small.hst[k];
        sc.cons(x, cx + ncu);          // sc.nb == 0 for general families: only [x - x_low ; x_upp - x]
    }

    // ---- DevicePoint ----
    int eval_point(const double* x, double* gradf, double* rr, double* cx) override {
        int rc = eval_at(x);
        if (rc != 0) return rc;
        for (int j = 0; j < n; ++j) gradf[j] = hgrad[j];
        *rr = hgrad[n];
        if (gv) finish_cons(x, cx);
        else sc.cons(x, cx);
        return 0;
    }
    // factor the [J | r] of the last eval_at: dJc = column-major [J~ | r~] (identical on every rank), optionally
    // copied to hR.  Destroys [J | r] (in-place Householder), so it runs at most once per point.
    int factor_point(bool want_host_R) override {
        if (point_factored) return lfail(ENLSIPB200_EINVAL, "point already factored");
        LCU(cudaSetDevice(device));
        LCU(cudaEventRecord(e1, st));
        if (gv && !tsqr_rows) {      // plain Householder QR of the column-major [J | r] (dgeqrf order), R -> [J~ | r~]
            const int rc = enl_small::qrcp_device(dQ.get(), (int)m_local, n + 1, dtauQ.get(), dpQ.get(), small.qw, st, 1);
            if (rc < 0) return lfail(ENLSIPB200_ECUDA, "QR of [J | r]: more columns than the QR scratch holds");
            launches += rc;
            const long long ne = (long long)(n + 1) * (n + 1);
            enl_small::upper_to_square_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dQ.get(), (int)m_local, n + 1, dJc.get());
            ++launches;
        } else {
            LCU(cudaMemsetAsync(dR.get(), 0, sizeof(double) * rr_rows * ld, st));
            double* dfinal = dR.get();
            if (nranks > 1 && tree_dist) {
                TsqrDist td;
                td.nranks = nranks; td.rank = rank; td.P = dP.get(); td.scal = dPscal.get(); td.ctx = this;
                td.allgather = [](void* c, const double* send, double* recv, size_t count, cudaStream_t s) {
                    LargeHandle* h = static_cast<LargeHandle*>(c);
                    return g_nccl.AllGather(send, recv, count, NCCL_FLOAT64, h->comm, s);
                };
                td.allreduce_sum = [](void* c, double* buf, size_t count, cudaStream_t s) {
                    LargeHandle* h = static_cast<LargeHandle*>(c);
                    return g_nccl.AllReduce(buf, buf, count, NCCL_FLOAT64, NCCL_SUM, h->comm, s);
                };
                const int rc = tsqr_factor(dA.get(), ld, rows_pad, nt, dR.get(), ld, dT.get(), dpart.get(), st, &td);
                if (rc < 0) return lfail(ENLSIPB200_ECUDA, "NCCL collective inside the row-sharded TSQR failed");
                launches += rc;
            } else {
                launches += tsqr_factor(dA.get(), ld, rows_pad, nt, dR.get(), ld, dT.get(), dpart.get(), st);
            }
            if (nranks > 1 && !tree_dist) {
                int rc = g_nccl.AllGather(dR.get(), dStack.get(), (size_t)rr_rows * ld, NCCL_FLOAT64, comm, st);
                if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllGather: ") + g_nccl.GetErrorString(rc));
                LCU(cudaMemsetAsync(dR2.get(), 0, sizeof(double) * rr_rows * ld, st));
                launches += tsqr_factor(dStack.get(), ld, (long long)nranks * rr_rows, nt, dR2.get(), ld, dT.get(), dpart.get(), st);
                dfinal = dR2.get();
            }
            if (tsqr_rows) {
                const long long ne = (long long)(n + 1) * (n + 1);
                rows_unpad_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dfinal, ld, n, nt, dJc.get());
            } else {
                const int nc = n + 1;
                dim3 grid((nc + 31) / 32, (nc + 31) / 32), block(32, 8);
                r_to_colmajor_kernel<<<grid, block, 0, st>>>(dfinal, ld, nc, dJc.get());
            }
            ++launches;
        }
        point_factored = true;
        LCU(cudaEventRecord(e2, st));
        if (want_host_R) LCU(cudaMemcpyAsync(hR.data(), dJc.get(), sizeof(double) * (size_t)(n + 1) * (n + 1), cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        LCU(cudaEventElapsedTime(&last_tsqr_ms, e1, e2));
        ms_tsqr += last_tsqr_ms;
        ++n_factor;
        return 0;
    }
    // G (device, n x n) at x by lg_hessian_kernel over the family's rows and the active constraints; its device time
    // (CUDA events) adds to the Hessian ms of enlsipb200_large_stats
    int hessian(const double* x, const double* lam, const int* active, int t, double* G) override {
        if (!midsize || !gv) return lfail(ENLSIPB200_EINVAL, "second derivatives: row families created with ENLSIPB200_LARGE_MIDSIZE only");
        LCU(cudaMemcpyAsync(dxn.get(), x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        if (t > 0) {
            LCU(cudaMemcpyAsync(dlamn.get(), lam, sizeof(double) * t, cudaMemcpyHostToDevice, st));
            LCU(cudaMemcpyAsync(dactn.get(), active, sizeof(int) * t, cudaMemcpyHostToDevice, st));
        }
        LCU(cudaEventRecord(eh0, st));
        gv->hessian(st, n, m_local, dxn.get(), gd[0], gd[1], dhr.get(), ncu, (int)sc.lo_idx.size(), dbidx.get(), dbval.get(), t,
                    dactn.get(), dlamn.get(), G);
        launches += 2;
        LCU(cudaEventRecord(eh1, st));
        LCU(cudaStreamSynchronize(st));
        LCU(cudaGetLastError());
        float ms = 0.0f;
        LCU(cudaEventElapsedTime(&ms, eh0, eh1));
        ms_hess += ms;
        return 0;
    }
    const char* last_error() const override { return g_lerr.c_str(); }

    // ---- LargeOps ----
    double agreed_elapsed(double local_elapsed) override {
        if (nranks <= 1) return local_elapsed;
        cudaSetDevice(device);
        double* hs = small.hst.get();
        hs[0] = local_elapsed / nranks;
        if (cudaMemcpyAsync(small.dscal.get(), hs, sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess ||
            g_nccl.AllReduce(small.dscal.get(), small.dscal.get(), 1, NCCL_FLOAT64, NCCL_SUM, comm, st) != 0 ||
            cudaMemcpyAsync(hs, small.dscal.get(), sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            throw std::runtime_error("agreed_elapsed: all-reduce of the wall clock failed");
        return hs[0];
    }
    int set_direction(const double*, const double* p, double sums[3]) override {
        LCU(cudaSetDevice(device));
        auto t0 = std::chrono::steady_clock::now();
        LCU(cudaMemcpyAsync(dp.get(), p, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        cur_parts = grid_rows();
        if (gv && tsqr_rows) {
            lg_dir_rows_kernel<<<cur_parts, 256, 0, st>>>(dJrow.get(), n, m_local, dp.get(), dr.get(), dJp.get(), dpart.get());
        } else if (gv) {
            launches += enl_small::gemv_n(dJkeep.get(), (int)m_local, (int)m_local, n, dp.get(), 1.0, nullptr, 0.0, dJp.get(), st);
            lg_dir_sums_kernel<<<cur_parts, 256, 0, st>>>(dr.get(), dJp.get(), m_local, dpart.get());
        } else {
            li_dir_kernel<<<cur_parts, 256, sizeof(double) * (jac_fd ? 2 : 1) * n, st>>>(
                dW, dp.get(), dr.get(), ds.get(), m_local, n, dv.get(), dJp.get(), dpart.get(), jac_fd, dx.get(), du.get(), dy);
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
        if (gv) gv->ls(cur_parts, st, n, m_local, row0, dx.get(), dp.get(), alpha, gd[0], gd[1], dr.get(), dJp.get(), with_coeffs, dpart.get());
        else li_ls_kernel<<<cur_parts, 256, 0, st>>>(du.get(), dv.get(), dy, dr.get(), dJp.get(), m_local, alpha, with_coeffs, dpart.get());
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
        double* dxc = small.dvec[6].get();
        LCU(cudaMemcpyAsync(dxc, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
        gv->cons(st, n, ncu, dxc, gd[0], gd[1], dcu.get());
        ++launches;
        if (ncu > 0) LCU(cudaMemcpyAsync(small.hst.get(), dcu.get(), sizeof(double) * ncu, cudaMemcpyDeviceToHost, st));
        LCU(cudaStreamSynchronize(st));
        finish_cons(x, cx);
        return 0;
    }
};

LargeHandle* LH(enlsipb200_large h) { return reinterpret_cast<LargeHandle*>(h); }

// ---- frame of the known-answer hooks (enlsipb200_dense_*) ----
float g_dense_ms = 0.0f;     // device time (CUDA events) of the last hook call

// a hook's device scratch: at least one element
template <class T> bool dense_get(DevBuf<T>& b, size_t count) { return dev_alloc(b, count > 0 ? count : 1) == cudaSuccess; }

int dense_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(ENLSIPB200_ENOGPU, "no CUDA device");
    if (device < 0) LCU(cudaGetDevice(&device));
    LCU(cudaSetDevice(device));
    return 0;
}

// work(stream) between two CUDA events, then a synchronisation; its device time goes to g_dense_ms.  own_stream: on a
// stream created here (qrcp_device captures its panels as graphs only on a non-null stream), else on the legacy default
// stream.  What is created here is released on every return.
template <class Work> int dense_timed(bool own_stream, Work&& work) {
    cudaStream_t st = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaError_t e = own_stream ? cudaStreamCreate(&st) : cudaSuccess;
    if (e == cudaSuccess) e = cudaEventCreate(&ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&ev1);
    if (e == cudaSuccess) e = cudaEventRecord(ev0, st);
    if (e == cudaSuccess) {
        work(st);
        e = cudaEventRecord(ev1, st);
        cudaError_t es = own_stream ? cudaStreamSynchronize(st) : cudaDeviceSynchronize();
        if (es == cudaSuccess) es = cudaGetLastError();
        cudaEventElapsedTime(&g_dense_ms, ev0, ev1);
        if (e == cudaSuccess) e = es;
    }
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (st) cudaStreamDestroy(st);
    LCU(e);
    return 0;
}

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
    const bool midsize = (family & ENLSIPB200_LARGE_MIDSIZE) != 0;
    family &= ~(ENLSIPB200_LARGE_FACTOR_TSQR | ENLSIPB200_LARGE_MIDSIZE);
    const GenericVt* gv = nullptr;
#if defined(ENL_LARGE_USER_FAMILY)
    if (family == ENLSIPB200_FAMILY_USER) gv = generic_vt<LFamUser>();
    else return lfail(ENLSIPB200_EINVAL, "this library was compiled for ENLSIPB200_FAMILY_USER only");
#else
    if (family == ENLSIPB200_FAMILY_LARGE_CHAINED_ROSENBROCK) gv = generic_vt<LFamChainedRosenbrock>();
    else if (family != ENLSIPB200_FAMILY_SINGLE_INDEX) return lfail(ENLSIPB200_EINVAL, "unknown large-regime family");
#endif
    if (midsize) {
        if (!gv)
            return lfail(ENLSIPB200_EINVAL, "ENLSIPB200_LARGE_MIDSIZE: row families only (the single-index family has no Newton step)");
        if (want_tsqr)
            return lfail(ENLSIPB200_EINVAL, "ENLSIPB200_LARGE_MIDSIZE and ENLSIPB200_LARGE_FACTOR_TSQR do not combine (mid-size problems are not sharded)");
        if ((long long)n + m_global >= 1000)
            return lfail(ENLSIPB200_EINVAL, "ENLSIPB200_LARGE_MIDSIZE: n + m < 1000 required (larger problems run without second derivatives, EF:2658)");
        if (m_global < (long long)n + 1)
            return lfail(ENLSIPB200_EINVAL, "ENLSIPB200_LARGE_MIDSIZE: m >= n + 1 required ([J | r] is compressed by a QR of at least n + 1 rows)");
    }
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
    if ((long long)n + m_global < 1000 && !midsize)
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
    h->midsize = midsize;
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
        LCU(dev_alloc(h->gown[slot], count > 0 ? count : 1));
        LCU(cudaMemcpy(h->gown[slot].get(), ptr, sizeof(double) * count, cudaMemcpyHostToDevice));
        h->gd[slot] = h->gown[slot].get();
        return 0;
    }
    long long want = slot == 0 ? h->m_local * h->n : h->m_local;
    if (slot < 0 || slot > 1 || count != want) return lfail(ENLSIPB200_EINVAL, "bad slot / count");
    const double** dst = slot == 0 ? &h->dW : &h->dy;
    DevBuf<double>& own = slot == 0 ? h->ownW : h->owny;
    if (on_device) { *dst = ptr; return 0; }
    if (!own || h->own_count[slot] != count) LCU(dev_alloc(own, count > 0 ? count : 1));
    h->own_count[slot] = count;
    LCU(cudaMemcpy(own.get(), ptr, sizeof(double) * count, cudaMemcpyHostToDevice));
    *dst = own.get();
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
    if (h->comm) {   // a second call replaces the communicator and the cross-rank buffers of the first
        g_nccl.CommDestroy(h->comm);
        h->comm = nullptr;
    }
    NcclApi::UniqueId id;
    memcpy(&id, id128, 128);
    int rc = g_nccl.CommInitRank(&h->comm, nranks, id, rank);
    if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(rc));
    h->rank = rank; h->nranks = nranks;
    if (h->tsqr_rows) {   // row shards of a row family: every rank learns every m_local, takes its row0 and checks the total
        DevBuf<double> dm;
        LCU(dev_alloc(dm, nranks + 1));
        const double mine = (double)h->m_local;
        std::vector<double> all(nranks, 0.0);
        LCU(cudaMemcpy(dm.get() + nranks, &mine, sizeof(double), cudaMemcpyHostToDevice));
        rc = g_nccl.AllGather(dm.get() + nranks, dm.get(), 1, NCCL_FLOAT64, h->comm, nullptr);
        if (rc == 0) LCU(cudaMemcpy(all.data(), dm.get(), sizeof(double) * nranks, cudaMemcpyDeviceToHost));
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
    LCU(dev_alloc(h->dStack, (size_t)nranks * h->rr_rows * h->ld));
    LCU(dev_alloc(h->dR2, (size_t)h->rr_rows * h->ld));
    {   // the cross-rank stage as one more level of every panel's tree (TsqrDist) needs a 32-row block on every rank
        const size_t prow = (size_t)(nranks > 8 ? nranks : 8) * TS_B;
        LCU(dev_alloc(h->dP, prow * h->ld));
        LCU(cudaMemset(h->dP.get(), 0, sizeof(double) * prow * h->ld));
        LCU(dev_alloc(h->dPscal, 2));
        const double mine = (h->rows_pad < TS_B || (h->gv && !h->tsqr_rows)) ? 1.0 : 0.0;
        LCU(cudaMemcpy(h->dPscal.get(), &mine, sizeof(double), cudaMemcpyHostToDevice));
        rc = g_nccl.AllReduce(h->dPscal.get(), h->dPscal.get(), 1, NCCL_FLOAT64, NCCL_SUM, h->comm, nullptr);
        if (rc != 0) return lfail(ENLSIPB200_ECUDA, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
        double short_ranks = 0.0;
        LCU(cudaMemcpy(&short_ranks, h->dPscal.get(), sizeof(double), cudaMemcpyDeviceToHost));
        const char* e = getenv("ENLSIP_TSQR_DIST");
        h->tree_dist = short_ranks == 0.0 && !(e && e[0] == 's');
    }
    {   // the T-factor buffer also serves the second-stage TSQR of the nranks stacked R factors: one 32 x 32 per subtile
        const long long nsub2 = ((long long)nranks * h->rr_rows / TS_B + TS_FAN - 1) / TS_FAN;
        if (nsub2 > h->dT_subtiles) {
            LCU(dev_alloc(h->dT, nsub2 * TS_B * TS_B));
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
    opt.second_derivatives = h->midsize;
    double abs_tol = (o->abs_tol == o->abs_tol) ? o->abs_tol : EPS;
    double rel_tol = (o->rel_tol == o->rel_tol) ? o->rel_tol : sqrt(abs_tol);
    opt.eps_rel = rel_tol;
    opt.eps_c = (o->c_tol == o->c_tol) ? o->c_tol : rel_tol;
    opt.eps_x = (o->x_tol == o->x_tol) ? o->x_tol : rel_tol;
    auto t0 = std::chrono::steady_clock::now();
    LargeResult R;
    try {
        LargeSolver S(*h, opt, h->small);
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
    int rc = h->eval_at(x);
    if (rc == 0) rc = h->factor_point(true);
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
    const DeviceSmall& s = h->small;
    double v[15] = {(double)h->n_newpoint, h->ms_build, h->ms_tsqr, h->ms_ls, h->ms_total, (double)h->n_ls,
                    (double)(h->launches + s.launches), (double)h->rows_pad, (double)s.n_dev_qrcp, (double)s.n_dev_mulq,
                    s.ms_small, (double)h->n_factor, (double)s.n_ws_grow, (double)s.n_newton, h->ms_hess};
    for (int i = 0; i < count && i < 15; ++i) out[i] = v[i];
    return 0;
}

// ---- known-answer hooks of enl_small.cuh (tests/test_gpu_kat.py, tests/test_gpu_dense_dispatch.py) ----
// qrcp_device on a copy of f: dgeqp3 (nopivot = 0, jpvt returned) or dgeqrf (nopivot = 1, jpvt may be NULL)
static int dense_qr_run(int rows, int cols, double* f, double* tau, int* jpvt, int device, int nopivot) {
    if (rows < 1 || cols < 1 || !f || !tau || (!jpvt && !nopivot)) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    if (int rc = dense_device(device)) return rc;
    DevBuf<double> df, dtau;
    DevBuf<int> dp;
    enl_small::QrWork qw;
    const int k = rows < cols ? rows : cols;
    if (!dense_get(df, (size_t)rows * cols) || !dense_get(dtau, k) || !dense_get(dp, cols) || qw.alloc(cols) != cudaSuccess)
        return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(df.get(), f, sizeof(double) * (size_t)rows * cols, cudaMemcpyHostToDevice));
    LCU(cudaMemset(dtau.get(), 0, sizeof(double) * k));
    if (int rc = dense_timed(true, [&](cudaStream_t st) { enl_small::qrcp_device(df.get(), rows, cols, dtau.get(), dp.get(), qw, st, nopivot); }))
        return rc;
    LCU(cudaMemcpy(f, df.get(), sizeof(double) * (size_t)rows * cols, cudaMemcpyDeviceToHost));
    LCU(cudaMemcpy(tau, dtau.get(), sizeof(double) * k, cudaMemcpyDeviceToHost));
    if (jpvt) LCU(cudaMemcpy(jpvt, dp.get(), sizeof(int) * cols, cudaMemcpyDeviceToHost));
    return 0;
}

int enlsipb200_dense_qrcp(int rows, int cols, double* f, double* tau, int* jpvt, int device) {
    return dense_qr_run(rows, cols, f, tau, jpvt, device, 0);
}

int enlsipb200_dense_qr(int rows, int cols, double* f, double* tau, int device) {
    return dense_qr_run(rows, cols, f, tau, nullptr, device, 1);
}

float enlsipb200_dense_last_ms(void) { return g_dense_ms; }

// Known-answer hook of the Newton step's Cholesky factorisation (enl_small::potrf_upper): a [n x n] column major, upper
// triangle in, U out (dpotrf('U')); info as dpotrf's
int enlsipb200_dense_potrf(int n, double* a, int* info, int device) {
    if (n < 1 || n > enl_small::VEC_STAGE_MAX || !a || !info) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    if (int rc = dense_device(device)) return rc;
    DevBuf<double> da;
    DevBuf<int> dinfo;
    if (!dense_get(da, (size_t)n * n) || !dense_get(dinfo, 1)) return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(da.get(), a, sizeof(double) * (size_t)n * n, cudaMemcpyHostToDevice));
    if (int rc = dense_timed(false, [&](cudaStream_t st) { enl_small::potrf_upper(da.get(), n, n, dinfo.get(), st); })) return rc;
    LCU(cudaMemcpy(a, da.get(), sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToHost));
    LCU(cudaMemcpy(info, dinfo.get(), sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

int enlsipb200_dense_mulq(int mr, int nq, int k, const double* f, const double* tau, double* M, int device) {
    if (mr < 1 || nq < 1 || k < 0 || k > nq || !f || !tau || !M) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    if (int rc = dense_device(device)) return rc;
    DevBuf<double> df, dtau, dM, dTall;
    enl_small::WyWork ww;
    if (!dense_get(df, (size_t)nq * (k > 0 ? k : 1)) || !dense_get(dtau, k) || !dense_get(dM, (size_t)mr * nq) ||
        !dense_get(dTall, ((size_t)nq / 32 + 2) * 1024) || ww.alloc(nq, mr) != cudaSuccess)
        return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(df.get(), f, sizeof(double) * (size_t)nq * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dtau.get(), tau, sizeof(double) * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dM.get(), M, sizeof(double) * (size_t)mr * nq, cudaMemcpyHostToDevice));
    if (int rc = dense_timed(false, [&](cudaStream_t st) {
            enl_small::mulq_device(dM.get(), mr, nq, df.get(), nq, k, dtau.get(), ww, st, dTall.get(), true);
        }))
        return rc;
    LCU(cudaMemcpy(M, dM.get(), sizeof(double) * (size_t)mr * nq, cudaMemcpyDeviceToHost));
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
    if (int rc = dense_device(device)) return rc;
    const int vlen = kind < 2 ? frows : k;
    DevBuf<double> df, dtau, dv, dTall, dscr, dwp;
    DevBuf<unsigned int> dbar;
    const size_t scr = (size_t)1024 * ((frows + enl_small::WY_SLAB - 1) / enl_small::WY_SLAB) * 8;
    if (!dense_get(df, (size_t)frows * k) || !dense_get(dtau, k) || !dense_get(dv, vlen) || !dense_get(dTall, ((size_t)k / 32 + 2) * 1024) ||
        !dense_get(dscr, scr) || !dense_get(dwp, enl_small::RW_WPART_LEN) || !dense_get(dbar, 16))
        return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(df.get(), f, sizeof(double) * (size_t)frows * k, cudaMemcpyHostToDevice));
    if (kind < 2) LCU(cudaMemcpy(dtau.get(), tau, sizeof(double) * k, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dv.get(), v, sizeof(double) * vlen, cudaMemcpyHostToDevice));
    LCU(cudaMemset(dbar.get(), 0, sizeof(unsigned int) * 16));
    int rc = 0;
    // the direct compact-WY kernel is timed without the T factors it reads
    if (!dispatched && kind < 2) rc = enl_small::wy_build_t_all(df.get(), frows, k, dtau.get(), dTall.get(), dscr.get(), scr, nullptr);
    if (int trc = dense_timed(false, [&](cudaStream_t st) {
            if (dispatched && kind < 2) {
                auto t_of = [&]() -> const double* {
                    return enl_small::wy_build_t_all(df.get(), frows, k, dtau.get(), dTall.get(), dscr.get(), scr, st) >= 0 ? dTall.get() : nullptr;
                };
                rc = enl_small::reflect_vec(df.get(), frows, k, dtau.get(), dv.get(), kind == 0 ? 1 : 0, t_of, dwp.get(), dbar.get(), st);
            } else if (dispatched) {
                rc = enl_small::trsv_upper(df.get(), frows, k, dv.get(), kind == 3, dbar.get(), st);
            } else if (kind < 2) {
                if (rc >= 0) rc = enl_small::reflect_vec_wy(df.get(), frows, k, dTall.get(), dv.get(), kind == 0 ? 1 : 0, dwp.get(), dbar.get(), st);
            } else {
                rc = enl_small::trsv_coop(df.get(), frows, k, dv.get(), kind == 3, dbar.get(), st);
            }
        }))
        return trc;
    if (rc < 0) return lfail(ENLSIPB200_EINVAL, "shape not supported by the cooperative kernel");
    LCU(cudaMemcpy(v, dv.get(), sizeof(double) * vlen, cudaMemcpyDeviceToHost));
    return 0;
}

// Known-answer hook for the small stage's gemv (enl_small::gemv_n / gemv_t).  A: rows x cols, column major, lda >= rows.
// trans 0: y [rows] = alpha A x + beta y0 (x [cols]; y0 [rows] or NULL = 0); trans 1: y [cols] = A' x (x [rows]; alpha,
// y0 and beta unused: gemv_t forms the plain product).
int enlsipb200_dense_gemv(int trans, int rows, int cols, const double* A, int lda, const double* x, double alpha,
                          const double* y0, double beta, double* y, int device) {
    if ((trans != 0 && trans != 1) || rows < 1 || cols < 1 || lda < rows || !A || !x || !y) return lfail(ENLSIPB200_EINVAL, "bad arguments");
    if (int rc = dense_device(device)) return rc;
    const int xlen = trans ? rows : cols, ylen = trans ? cols : rows;
    const bool with_y0 = !trans && y0;
    DevBuf<double> dA, dx, dy0, dy;
    if (!dense_get(dA, (size_t)lda * cols) || !dense_get(dx, xlen) || !dense_get(dy, ylen) || (with_y0 && !dense_get(dy0, ylen)))
        return lfail(ENLSIPB200_ENOMEM, "cudaMalloc");
    LCU(cudaMemcpy(dA.get(), A, sizeof(double) * (size_t)lda * cols, cudaMemcpyHostToDevice));
    LCU(cudaMemcpy(dx.get(), x, sizeof(double) * xlen, cudaMemcpyHostToDevice));
    if (with_y0) LCU(cudaMemcpy(dy0.get(), y0, sizeof(double) * ylen, cudaMemcpyHostToDevice));
    if (int rc = dense_timed(false, [&](cudaStream_t st) {
            if (trans) enl_small::gemv_t(dA.get(), lda, rows, cols, dx.get(), dy.get(), st);
            else enl_small::gemv_n(dA.get(), lda, rows, cols, dx.get(), alpha, dy0.get(), beta, dy.get(), st);
        }))
        return rc;
    LCU(cudaMemcpy(y, dy.get(), sizeof(double) * ylen, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
