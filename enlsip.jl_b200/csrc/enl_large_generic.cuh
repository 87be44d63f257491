// enl_large_generic.cuh -- the m-sized kernels of the large regime for GENERAL problem families (row families of
// enl_large_family.h), i.e. the replacement of the reference's evaluation wrappers res_eval! / jacres_eval! /
// cons_eval! / jaccons_eval! (src/cnls_model.jl:40-62) and of jac_forward_diff (src/cnls_model.jl:65-82) when the
// problem is not the single-index family with its specialised kernels (enl_large.cu).  [J | r] is built column major
// (m x (n+1)) and factored by the plain-Householder mode of qrcp_device (enl_small.cuh); a copy of J serves J p.
// With ENLSIPB200_LARGE_FACTOR_TSQR the family builds the TSQR's row-major work matrix instead (lg_build_rows_kernel:
// [J | 0 | r], n padded to a multiple of 32) and J p comes from a row-major copy of J (lg_dir_rows_kernel).
#pragma once
#include <cuda_runtime.h>

#include "enl_large_family.h"

namespace enl_large {

constexpr double G_SQRT_EPS = 1.4901161193847656e-08;

__device__ __forceinline__ double g_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// four sums over the CTA -> part[blockIdx * 4 + k] (fixed order)
__device__ __forceinline__ void g_block_reduce4(double (&v)[4], double* part) {
    __shared__ double sh[8][4];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = g_warp_sum(v[k]);
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

// new_point!: one warp per residual row: r_i and row i of J (analytic or forward differences) into Q = [J | r]
template <class F>
__global__ void __launch_bounds__(256) lg_build_kernel(int n, long long m, const double* __restrict__ x,
                                                       const double* __restrict__ d0, const double* __restrict__ d1, int fd,
                                                       double* __restrict__ Q, double* __restrict__ r_out) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp0; i < m; i += nwarps) {
        const double ri = F::residual(i, n, XPlain{x}, d0, d1);
        for (int j = lane; j < n; j += 32) {
            double v;
            if (fd || !F::HAS_JAC) {
                const double dj = __dmul_rn(fmax(fabs(x[j]), 1.0), G_SQRT_EPS);
                v = __ddiv_rn(__dsub_rn(F::residual(i, n, XPert{x, j, dj}, d0, d1), ri), dj);
            } else {
                v = F::jac_residual(i, j, n, x, d0, d1);
            }
            Q[(size_t)j * m + i] = v;
        }
        if (lane == 0) { Q[(size_t)n * m + i] = ri; r_out[i] = ri; }
    }
}

// TSQR work matrix (rows_pad x ld, row major): one warp per row, lanes over the columns (coalesced stores).  Row i holds
// [J_i | 0 | r_i | 0]: J in columns 0..n-1, zeros up to column nt - 1 (nt = n rounded up to 32), r in column nt, zeros up
// to ld - 1; rows m..rows_pad-1 are all zero.  Every entry of the row is rewritten at each point, so nothing the previous
// factorisation left in the matrix survives.  Entries of J by the arithmetic of lg_build_kernel; the family sees the
// global row row0 + i.  Jrow: row-major m x n copy of J for the direction products.
template <class F>
__global__ void __launch_bounds__(256) lg_build_rows_kernel(int n, long long m, long long rows_pad, long long row0,
                                                            const double* __restrict__ x, const double* __restrict__ d0,
                                                            const double* __restrict__ d1, int fd, int nt, int ld,
                                                            double* __restrict__ A, double* __restrict__ Jrow,
                                                            double* __restrict__ r_out) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp0; i < rows_pad; i += nwarps) {
        double* ar = A + i * ld;
        if (i >= m) {
            for (int j = lane; j < ld; j += 32) ar[j] = 0.0;
            continue;
        }
        const long long gi = row0 + i;
        const double ri = F::residual(gi, n, XPlain{x}, d0, d1);
        double* jr = Jrow + i * n;
        for (int j = lane; j < ld; j += 32) {
            double v = 0.0;
            if (j < n) {
                if (fd || !F::HAS_JAC) {
                    const double dj = __dmul_rn(fmax(fabs(x[j]), 1.0), G_SQRT_EPS);
                    v = __ddiv_rn(__dsub_rn(F::residual(gi, n, XPert{x, j, dj}, d0, d1), ri), dj);
                } else {
                    v = F::jac_residual(gi, j, n, x, d0, d1);
                }
                jr[j] = v;
            } else if (j == nt) {
                v = ri;
            }
            ar[j] = v;
        }
        if (lane == 0) r_out[i] = ri;
    }
}

// Jp = J p from the row-major copy of J (one warp per row) and the sums {r.r, r.Jp, Jp.Jp, 0}
__global__ void __launch_bounds__(256) lg_dir_rows_kernel(const double* __restrict__ J, int n, long long m,
                                                          const double* __restrict__ p, const double* __restrict__ r,
                                                          double* __restrict__ Jp, double* __restrict__ part) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long i = warp0; i < m; i += nwarps) {
        const double* jr = J + i * n;
        double acc = 0.0;
        for (int j = lane; j < n; j += 32) acc = fma(jr[j], p[j], acc);
        const double jp = g_warp_sum(acc);
        if (lane == 0) {
            const double ri = r[i];
            Jp[i] = jp;
            sums[0] = fma(ri, ri, sums[0]); sums[1] = fma(ri, jp, sums[1]); sums[2] = fma(jp, jp, sums[2]);
        }
    }
    g_block_reduce4(sums, part);
}

// sums {r.r, r.Jp, Jp.Jp, 0} for the direction just set
__global__ void __launch_bounds__(256) lg_dir_sums_kernel(const double* __restrict__ r, const double* __restrict__ Jp, long long m,
                                                          double* __restrict__ part) {
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        const double ri = r[i], jp = Jp[i];
        sums[0] = fma(ri, ri, sums[0]); sums[1] = fma(ri, jp, sums[1]); sums[2] = fma(jp, jp, sums[2]);
    }
    g_block_reduce4(sums, part);
}

// trial point x + alpha p: partial sums {r_a.r_a, r.v2, Jp.v2, v2.v2}, v2 = ((r_a - r)/alpha - Jp)/alpha  (EF:1687)
template <class F>
__global__ void __launch_bounds__(256) lg_ls_kernel(int n, long long m, long long row0, const double* __restrict__ x, const double* __restrict__ p,
                                                    double alpha, const double* __restrict__ d0, const double* __restrict__ d1,
                                                    const double* __restrict__ r, const double* __restrict__ Jp, int with_coeffs,
                                                    double* __restrict__ part) {
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    const XStep xs{x, p, alpha};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        const double ra = F::residual(row0 + i, n, xs, d0, d1);
        sums[0] = fma(ra, ra, sums[0]);
        if (with_coeffs) {
            const double ri = r[i], jp = Jp[i];
            const double v2 = (__ddiv_rn(__dsub_rn(ra, ri), alpha) - jp) / alpha;
            sums[1] = fma(ri, v2, sums[1]); sums[2] = fma(jp, v2, sums[2]); sums[3] = fma(v2, v2, sums[3]);
        }
    }
    g_block_reduce4(sums, part);
}

// the family's own constraints (equalities then inequalities) at x
template <class F>
__global__ void lg_cons_kernel(int n, int nc, const double* __restrict__ x, const double* __restrict__ d0,
                               const double* __restrict__ d1, double* __restrict__ c) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nc) c[k] = F::constraint(k, n, XPlain{x}, d0, d1);
}
// their Jacobian rows into A (row major l x n); c0 = constraints at x (forward differences)
template <class F>
__global__ void lg_jac_cons_kernel(int n, int nc, const double* __restrict__ x, const double* __restrict__ d0,
                                   const double* __restrict__ d1, int fd, const double* __restrict__ c0,
                                   double* __restrict__ Arow) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)nc * n) return;
    const int k = (int)(e / n), j = (int)(e % n);
    double v;
    if (fd || !F::HAS_JAC) {
        const double dj = __dmul_rn(fmax(fabs(x[j]), 1.0), G_SQRT_EPS);
        v = __ddiv_rn(__dsub_rn(F::constraint(k, n, XPert{x, j, dj}, d0, d1), c0[k]), dj);
    } else {
        v = F::jac_constraint(k, j, n, x, d0, d1);
    }
    Arow[e] = v;
}

// host-side dispatch table of one family
struct GenericVt {
    long long (*m_of)(int);
    int (*q_of)(int);
    int (*ni_of)(int);
    void (*build)(int grid, cudaStream_t st, int n, long long m, const double* x, const double* d0, const double* d1, int fd, double* Q, double* r);
    void (*build_rows)(int grid, cudaStream_t st, int n, long long m, long long rows_pad, long long row0, const double* x,
                       const double* d0, const double* d1, int fd, int nt, int ld, double* A, double* Jrow, double* r);
    void (*ls)(int grid, cudaStream_t st, int n, long long m, long long row0, const double* x, const double* p, double alpha,
               const double* d0, const double* d1, const double* r, const double* Jp, int with_coeffs, double* part);
    void (*cons)(cudaStream_t st, int n, int nc, const double* x, const double* d0, const double* d1, double* c);
    void (*jac_cons)(cudaStream_t st, int n, int nc, const double* x, const double* d0, const double* d1, int fd, const double* c0, double* Arow);
};
template <class F>
const GenericVt* generic_vt() {
    static const GenericVt vt = {
        [](int n) { return F::m_of(n); }, [](int n) { return F::q_of(n); }, [](int n) { return F::ni_of(n); },
        [](int grid, cudaStream_t st, int n, long long m, const double* x, const double* d0, const double* d1, int fd, double* Q, double* r) {
            lg_build_kernel<F><<<grid, 256, 0, st>>>(n, m, x, d0, d1, fd, Q, r);
        },
        [](int grid, cudaStream_t st, int n, long long m, long long rows_pad, long long row0, const double* x, const double* d0,
           const double* d1, int fd, int nt, int ld, double* A, double* Jrow, double* r) {
            lg_build_rows_kernel<F><<<grid, 256, 0, st>>>(n, m, rows_pad, row0, x, d0, d1, fd, nt, ld, A, Jrow, r);
        },
        [](int grid, cudaStream_t st, int n, long long m, long long row0, const double* x, const double* p, double alpha,
           const double* d0, const double* d1, const double* r, const double* Jp, int with_coeffs, double* part) {
            lg_ls_kernel<F><<<grid, 256, 0, st>>>(n, m, row0, x, p, alpha, d0, d1, r, Jp, with_coeffs, part);
        },
        [](cudaStream_t st, int n, int nc, const double* x, const double* d0, const double* d1, double* c) {
            if (nc > 0) lg_cons_kernel<F><<<(nc + 127) / 128, 128, 0, st>>>(n, nc, x, d0, d1, c);
        },
        [](cudaStream_t st, int n, int nc, const double* x, const double* d0, const double* d1, int fd, const double* c0, double* Arow) {
            const long long ne = (long long)nc * n;
            if (ne > 0) lg_jac_cons_kernel<F><<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(n, nc, x, d0, d1, fd, c0, Arow);
        }};
    return &vt;
}

}  // namespace enl_large
