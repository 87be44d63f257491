// enl_small.cuh -- the matrix-sized half of the large regime's small stage as CUDA kernels (sm_100a).
//
// The ENLSIP iteration on the compressed problem [J~ | r~] ((n+1) x (n+1), enl_large.cu) needs, per iteration
// (reference: src/enlsip_functions.jl = EF):
//   * qr(C.A', ColumnNorm())  (EF:700), qr(F_A.R', ColumnNorm()) (EF:769), qr(J2, ColumnNorm()) (EF:223)
//         -> qrcp_device(): LAPACK dgeqp3 restated for the GPU -- blocked dlaqps panels (nb = 32) for the leading
//            min(m,n) - 128 columns, each panel ONE persistent cooperative kernel (qr_panel_persist_kernel: two grid
//            barriers per pivoted column) followed by the rank-nb trailing update; unblocked dlaqp2 steps for the rest
//            (dgeqp3's crossover nx = 128); matrices that fit the shared memory of a thread-block cluster are factored
//            by one cluster kernel (qr_cluster_kernel).  First-max pivot, dlarfg with beta = -sign(alpha) dlapy2,
//            partial-norm downdate with the tol3z recompute rule (deferred to the end of a panel in the blocked part
//            exactly like dlaqps' lsticc list);
//   * J * F_A.Q                (EF:219)  -> mulq_device(): compact-WY panels (dlarft T factors of all panels in two
//            launches, wy_build_t_all), three DMMA GEMMs (mma.sync.m8n8k4.f64) per panel;
//   * F.Q' v, F.Q v            (EF:137, 143, 152, 484)  -> reflect_vec_wy_kernel (long vectors: the compact-WY panels in
//            one cooperative kernel, one grid barrier per 32 reflectors) / reflect_vec_warp_kernel (short vectors);
//   * R \ v, R' \ v            (EF:133-147, 486-500)    -> trsv_upper(T)_coop_kernel (one warp per diagonal block of 32
//            spread over the SMs, solved blocks announced through a release/acquire counter) / the one-warp kernels;
//   * J p, A p, J1 p1, J1' s, C.A' c (EF:2222-2224, 526, 2497) -> gemv_n_kernel / gemv_t_kernel.
// Column-major storage everywhere (a row-major l x n matrix is the column-major n x l matrix of its transpose).
// Everything is enqueued on one stream; indices that depend on the data (where a dlaqps panel stops) live in a device
// state block, so the host never synchronises inside a factorisation.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>

namespace enl_small {

constexpr double S_TOL3Z = 1.0536712127723509e-08;   // sqrt(dlamch('Epsilon')) = sqrt(2^-53)
constexpr int QR_NB = 32;                             // dgeqp3 block size (ilaenv(1, 'DGEQRF') = 32)
constexpr int QR_NX = 128;                            // dgeqp3 crossover (ilaenv(3, 'DGEQRF') = 128)

__device__ __forceinline__ double s_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// sum over the CTA, identical in every thread (fixed order); sh: 32 doubles
__device__ __forceinline__ double s_block_sum(double v, double* sh) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = s_warp_sum(v);
    __syncthreads();
    if (lane == 0) sh[w] = v;
    __syncthreads();
    double t = 0.0;
    for (int i = 0; i < nw; ++i) t += sh[i];
    return t;
}
__device__ __forceinline__ double s_lapy2(double x, double y) {
    const double xa = fabs(x), ya = fabs(y), w = fmax(xa, ya), z = fmin(xa, ya);
    if (z == 0.0) return w;
    const double q = z / w;
    return w * sqrt(1.0 + q * q);
}
__device__ __forceinline__ void s_dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// =============================================================================================
// GEMM on FP64 tensor cores:  C (M x N, ldc) = alpha * A (M x K, lda) * op(B) + beta * C
//   op(B) = B (K x N, ldb)            TRANSB = false
//   op(B) = B' with B (N x K, ldb)    TRANSB = true
// CTA tile 64 x 64, K in slabs of 32 staged through shared memory, 8 warps, each warp owns a 16 x 32 sub-tile
// (2 x 4 m8n8 accumulators).  Grid-stride over the tiles.
// =============================================================================================
inline int imin_host(int a, int b) { return a < b ? a : b; }

template <bool TRANSB>
__device__ __forceinline__ void gemm_tile(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb,
                                          double* __restrict__ C, int ldc, int M, int N, int K, double alpha, double beta,
                                          int tm, int tn, double (*As)[65], double (*Bs)[65]) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wm = (w & 3) * 16, wn = (w >> 2) * 32;      // warp sub-tile origin inside the 64 x 64 tile
    const int gr = lane >> 2, gc = lane & 3;               // fragment coordinates
    double acc[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int m0 = tm * 64, n0 = tn * 64;
    for (int k0 = 0; k0 < K; k0 += 32) {
        __syncthreads();
        // As[k][m] = A(m0 + m, k0 + k): threads walk m fastest (coalesced, column major)
        for (int e = tid; e < 32 * 64; e += 256) {
            const int mm = e & 63, kk = e >> 6;
            const int gm = m0 + mm, gk = k0 + kk;
            As[kk][mm] = (gm < M && gk < K) ? A[(size_t)gk * lda + gm] : 0.0;
        }
        if (TRANSB) {   // Bs[k][n] = B(n0 + n, k0 + k)
            for (int e = tid; e < 32 * 64; e += 256) {
                const int nn = e & 63, kk = e >> 6;
                const int gn = n0 + nn, gk = k0 + kk;
                Bs[kk][nn] = (gn < N && gk < K) ? B[(size_t)gk * ldb + gn] : 0.0;
            }
        } else {        // Bs[k][n] = B(k0 + k, n0 + n)
            for (int e = tid; e < 32 * 64; e += 256) {
                const int kk = e & 31, nn = e >> 5;
                const int gn = n0 + nn, gk = k0 + kk;
                Bs[kk][nn] = (gn < N && gk < K) ? B[(size_t)gn * ldb + gk] : 0.0;
            }
        }
        __syncthreads();
#pragma unroll
        for (int ks = 0; ks < 32; ks += 4) {
            double af[2], bf[4];
#pragma unroll
            for (int i = 0; i < 2; ++i) af[i] = As[ks + gc][wm + 8 * i + gr];      // A fragment: row = lane/4, k = lane%4
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = Bs[ks + gc][wn + 8 * j + gr];      // B fragment: k = lane%4, col = lane/4
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) s_dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
    }
    // D fragment: row = lane/4, cols = 2 (lane%4), 2 (lane%4) + 1
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int gm = m0 + wm + 8 * i + gr, gn = n0 + wn + 8 * j + 2 * gc + h;
                if (gm < M && gn < N) {
                    double* cp = C + (size_t)gn * ldc + gm;
                    const double v = alpha * acc[i][j][h];
                    *cp = (beta == 0.0) ? v : fma(beta, *cp, v);
                }
            }
}

template <bool TRANSB>
__global__ void __launch_bounds__(256) gemm_dmma_kernel(const double* __restrict__ A, int lda, const double* __restrict__ B,
                                                        int ldb, double* __restrict__ C, int ldc, int M, int N, int K,
                                                        double alpha, double beta) {
    __shared__ double As[32][65];
    __shared__ double Bs[32][65];
    const int tmn = (M + 63) / 64, tnn = (N + 63) / 64;
    for (int t = blockIdx.x; t < tmn * tnn; t += gridDim.x)
        gemm_tile<TRANSB>(A, lda, B, ldb, C, ldc, M, N, K, alpha, beta, t % tmn, t / tmn, As, Bs);
}

inline int gemm_grid(int M, int N) {
    long long t = (long long)((M + 63) / 64) * ((N + 63) / 64);
    return (int)(t < 1 ? 1 : (t > 148 * 8 ? 148 * 8 : t));
}
// C = alpha A op(B) + beta C on the stream; returns the number of launches
template <bool TRANSB>
inline int gemm(const double* A, int lda, const double* B, int ldb, double* C, int ldc, int M, int N, int K, double alpha,
                double beta, cudaStream_t st) {
    if (M <= 0 || N <= 0) return 0;
    gemm_dmma_kernel<TRANSB><<<gemm_grid(M, N), 256, 0, st>>>(A, lda, B, ldb, C, ldc, M, N, K, alpha, beta);
    return 1;
}

// Skinny products (N <= 64, long K: W = M V of the compact-WY update): the K range is cut into `splits` slabs, one CTA per
// (tile, slab) writes its partial product, a second kernel adds the partials in slab order (deterministic).
template <bool TRANSB>
__global__ void __launch_bounds__(256) gemm_dmma_splitk_kernel(const double* __restrict__ A, int lda, const double* __restrict__ B,
                                                               int ldb, double* __restrict__ part, int M, int N, int K, int kc) {
    __shared__ double As[32][65];
    __shared__ double Bs[32][65];
    const int tmn = (M + 63) / 64, tnn = (N + 63) / 64;
    const int ks = blockIdx.y, k0 = ks * kc;
    const int kl = (K - k0) < kc ? (K - k0) : kc;
    if (kl <= 0) return;
    const double* Ak = A + (size_t)k0 * lda;
    const double* Bk = TRANSB ? (B + (size_t)k0 * ldb) : (B + k0);
    double* Cp = part + (size_t)ks * M * N;
    for (int t = blockIdx.x; t < tmn * tnn; t += gridDim.x)
        gemm_tile<TRANSB>(Ak, lda, Bk, ldb, Cp, M, M, N, kl, 1.0, 0.0, t % tmn, t / tmn, As, Bs);
}
__global__ void splitk_reduce_kernel(const double* __restrict__ part, int splits, long long mn, double alpha, double beta,
                                     double* __restrict__ C, int M, int ldc) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= mn) return;
    double t = 0.0;
    for (int q = 0; q < splits; ++q) t += part[(size_t)q * mn + e];
    double* cp = C + (size_t)(e / M) * ldc + (e % M);
    *cp = (beta == 0.0) ? alpha * t : fma(beta, *cp, alpha * t);
}
constexpr int GEMM_MAX_SPLITS = 16;

// =============================================================================================
// QRCP (LAPACK dgeqp3 semantics)
// =============================================================================================
// Device state of one factorisation.
struct QrState {
    int j0;        // first column of the current dlaqps panel (= number of finished columns)
    int k;         // columns of the current panel already factored (valid when the panel ends)
    int stop;      // a norm has to be recomputed: the panel ends after k columns (dlaqps: lsticc != 0)
    int jb;        // columns this panel may take (min(nb, topbmn - j0))
    int active;    // the blocked phase still has work
    int pvt;       // pivot column chosen for the panel column in flight
    int anyflag;   // some column was flagged by the norm downdate of the column just finished
    int nopivot;   // plain Householder QR (dgeqrf order): columns stay where they are
    unsigned int ticket1, ticket2;
    double tau_k, sc_k, beta_k;   // dlarfg scalars of the panel column in flight (the column itself is stored unscaled
                                  // until the next finish kernel scales it in place)
};
constexpr int QR_MAXPART = 1024;   // partial results of the multi-CTA reductions

__global__ void qr_init_kernel(const double* __restrict__ f, int rows, int cols, double* vn1, double* vn2, int* jpvt,
                               QrState* stt, int topbmn, int nopivot) {
    __shared__ double sh[32];
    const int c = blockIdx.x;
    const double* cc = f + (size_t)c * rows;
    double s = 0.0;
    for (int r = threadIdx.x; r < rows; r += blockDim.x) s = fma(cc[r], cc[r], s);
    s = s_block_sum(s, sh);
    if (threadIdx.x == 0) {
        vn1[c] = vn2[c] = sqrt(s);
        jpvt[c] = c;
        if (c == 0) {
            stt->j0 = 0; stt->k = 0; stt->stop = 0;
            stt->jb = topbmn < QR_NB ? topbmn : QR_NB;
            stt->active = topbmn > 0 ? 1 : 0;
            stt->pvt = 0; stt->anyflag = 0; stt->ticket1 = 0; stt->ticket2 = 0; stt->nopivot = nopivot;
            stt->tau_k = 0.0; stt->sc_k = 1.0; stt->beta_k = 0.0;
        }
    }
}

// F is stored row-major here: F(j, i) at F[j * QR_NB + i] (one 256-byte line per column j of the matrix).
// Panel column kk, kernel 1 of 3 (grid over the trailing columns, one WARP per column, lane = panel index; kk = 0 .. jb):
//   finish column kk-1 (dlaqps, after the F column): F(j, kk-1) += F(j, 0:kk-1) auxv; pivot row of A updated;
//   partial-norm downdate, a column under the tol3z rule is flagged and ends the panel;
//   CTA 0 also scales the finished column in place (it was kept unscaled for the gemv) and stores beta;
//   then the pivot search for column kk: first maximum of vn1 over the trailing columns, per-CTA candidates combined
//   in index order by the last CTA (atomic ticket), which also swaps jpvt / vn1 / vn2 / the rows of F.
__global__ void __launch_bounds__(256) qr_panel_finish_pivot_kernel(double* __restrict__ f, int rows, int cols, double* vn1,
                                                                    double* vn2, int* jpvt, double* __restrict__ F,
                                                                    const double* __restrict__ auxv, int* flags,
                                                                    QrState* stt, double* pbest, int* pidx, int kk) {
    __shared__ double s_best[32];
    __shared__ int s_idx[32];
    __shared__ int s_last;
    if (!stt->active || stt->stop) return;
    const int j0 = stt->j0, k = kk, jb = stt->jb;
    if (k > jb) return;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
    const int jc = j0 + k;                       // the column about to be factored; trailing set = [jc, cols)
    const int kp = k - 1, rkp = j0 + kp;
    double aux_l = 0.0, frow_l = 0.0;            // lane i: auxv(i) for i < kp; A(rkp, j0 + i) for i < kp, 1 for i == kp
    if (k > 0) {
        aux_l = (lane < kp) ? auxv[lane] : 0.0;
        frow_l = (lane < kp) ? f[(size_t)(j0 + lane) * rows + rkp] : (lane == kp ? 1.0 : 0.0);
        if (blockIdx.x == 0) {                   // column jcp: v = [1; x * sc], R(rkp, jcp) = beta
            const double sc = stt->sc_k;
            double* cj = f + (size_t)rkp * rows;
            if (sc != 1.0)
                for (int r = rkp + 1 + tid; r < rows; r += blockDim.x) cj[r] *= sc;
            if (tid == 0) cj[rkp] = stt->beta_k;
        }
    }
    double best = -1.0; int idx = cols;          // per warp (identical in its lanes)
    int any = 0;
    for (int j = jc + blockIdx.x * nw + w; j < cols; j += gridDim.x * nw) {
        double v = 0.0;
        if (k > 0) {
            double fl = (lane <= kp) ? F[(size_t)j * QR_NB + lane] : 0.0;   // F(j, lane); beyond kp: stale, never read
            const double s = s_warp_sum(fl * aux_l);                 // lanes >= kp contribute 0
            const double fjk = __shfl_sync(0xffffffffu, fl, kp) + s;
            if (lane == kp) { fl = fjk; if (kp > 0) F[(size_t)j * QR_NB + kp] = fjk; }
            const double ru = s_warp_sum(frow_l * fl);               // sum_{i <= kp} A(rkp, j0 + i) F(j, i)
            double* ap = f + (size_t)j * rows + rkp;
            const double a = __shfl_sync(0xffffffffu, (lane == 0) ? *ap : 0.0, 0) - ru;
            double v1 = vn1[j];
            if (v1 != 0.0) {
                double temp = fabs(a) / v1;
                temp = fmax(0.0, (1.0 + temp) * (1.0 - temp));
                const double rq = v1 / vn2[j];
                if (temp * (rq * rq) <= S_TOL3Z && !stt->nopivot) { any = 1; if (lane == 0) flags[j] = 1; }
                else { v1 = v1 * sqrt(temp); if (lane == 0) vn1[j] = v1; }
            }
            if (lane == 0) *ap = a;
            v = v1;
        } else {
            v = vn1[j];
        }
        if (v > best) { best = v; idx = j; }
    }
    __threadfence();                     // this thread's F / A / vn1 / flags writes before the ticket below
    any = __syncthreads_or(any);
    if (lane == 0) { s_best[w] = best; s_idx[w] = idx; }
    __syncthreads();
    if (tid == 0) {
        double b = s_best[0]; int bi = s_idx[0];
        for (int q = 1; q < nw; ++q)
            if (s_best[q] > b || (s_best[q] == b && s_idx[q] < bi)) { b = s_best[q]; bi = s_idx[q]; }
        pbest[blockIdx.x] = b; pidx[blockIdx.x] = bi;
        if (any) atomicOr(&stt->anyflag, 1);
        __threadfence();
        s_last = (atomicAdd(&stt->ticket1, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // last CTA: combine the per-CTA candidates (parallel loads past L1, first maximum), bookkeeping by thread 0
    double b = -1.0; int bi = cols;
    for (int q = tid; q < (int)gridDim.x; q += blockDim.x) {
        const double pb = __ldcg(pbest + q); const int pi = __ldcg(pidx + q);
        if (pb > b || (pb == b && pi < bi)) { b = pb; bi = pi; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, b, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > b || (ob == b && oi < bi)) { b = ob; bi = oi; }
    }
    __syncthreads();
    if (lane == 0) { s_best[w] = b; s_idx[w] = bi; }
    __syncthreads();
    if (w == 0) {
        // warp 0 finishes: lanes hold the per-warp results
        b = (lane < nw) ? s_best[lane] : -1.0; bi = (lane < nw) ? s_idx[lane] : cols;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, b, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ob > b || (ob == b && oi < bi)) { b = ob; bi = oi; }
        }
        const int flagged = __ldcg(&stt->anyflag);
        if (bi >= cols || stt->nopivot) bi = jc;
        const bool pivoting = !flagged && k < jb;
        if (pivoting && bi != jc && lane < k) {          // swap the rows of F (k <= 32 entries)
            const double t = __ldcg(F + (size_t)bi * QR_NB + lane);
            F[(size_t)bi * QR_NB + lane] = __ldcg(F + (size_t)jc * QR_NB + lane);
            F[(size_t)jc * QR_NB + lane] = t;
        }
        if (lane == 0) {
            stt->ticket1 = 0;
            stt->anyflag = 0;
            stt->k = k;
            if (flagged) stt->stop = 1;
            else if (k < jb) {
                stt->pvt = bi;
                if (bi != jc) {              // other CTAs wrote these: read past L1
                    const int tp = __ldcg(jpvt + bi); jpvt[bi] = __ldcg(jpvt + jc); jpvt[jc] = tp;
                    vn1[bi] = __ldcg(vn1 + jc); vn2[bi] = __ldcg(vn2 + jc);
                }
            }
        }
    }
}

// kernel 2 of 3 (grid over row slices of 256): swap the pivot column in, A(rk:, jc) -= A(rk:, j0:jc) F(jc, 0:k)',
// partial sums of squares below the diagonal; the last CTA (ticket) computes the dlarfg scalars.
__global__ void __launch_bounds__(256) qr_panel_column_kernel(double* __restrict__ f, int rows, int cols, double* tau,
                                                              const double* __restrict__ F, QrState* stt, double* psum, int kk) {
    __shared__ double frow[QR_NB];
    __shared__ double sh[32];
    __shared__ int s_last;
    if (!stt->active || stt->stop) return;
    const int j0 = stt->j0, k = kk;
    if (k >= stt->jb) return;
    const int jc = j0 + k, rk = jc, pvt = stt->pvt;
    const int tid = threadIdx.x;
    if (tid < QR_NB) frow[tid] = (tid < k) ? F[(size_t)jc * QR_NB + tid] : 0.0;
    __syncthreads();
    double* cj = f + (size_t)jc * rows;
    double* cp = f + (size_t)pvt * rows;
    double part = 0.0;
    for (int r = blockIdx.x * blockDim.x + tid; r < rows; r += gridDim.x * blockDim.x) {
        double a = cp[r];
        if (pvt != jc) cp[r] = cj[r];
        if (r >= rk) {
            double s = 0.0;
            for (int i = 0; i < k; ++i) s = fma(f[(size_t)(j0 + i) * rows + r], frow[i], s);
            a -= s;
            if (r > rk) part = fma(a, a, part);
        }
        cj[r] = a;
    }
    __threadfence();
    part = s_block_sum(part, sh);
    if (tid == 0) {
        psum[blockIdx.x] = part;
        __threadfence();
        s_last = (atomicAdd(&stt->ticket2, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // last CTA: the partial sums in CTA order (loads in parallel, fixed-order adds by thread 0 through shared memory)
    __shared__ double ps[QR_MAXPART];
    for (int q = tid; q < (int)gridDim.x; q += blockDim.x) ps[q] = __ldcg(psum + q);
    __syncthreads();
    if (tid != 0) return;
    stt->ticket2 = 0;
    double tot = 0.0;
    for (int q = 0; q < (int)gridDim.x; ++q) tot += ps[q];
    double tau_k = 0.0, sc = 1.0;
    const double alpha = ((volatile double*)cj)[rk];
    double beta = alpha;
    if (rk < rows - 1) {
        const double xn = sqrt(tot);
        if (xn != 0.0) {
            beta = -copysign(s_lapy2(alpha, xn), alpha);
            tau_k = (beta - alpha) / beta;
            sc = 1.0 / (alpha - beta);
        }
    }
    tau[jc] = tau_k;
    stt->tau_k = tau_k; stt->sc_k = sc; stt->beta_k = beta;
}

// kernel 3 of 3 (grid, 8 columns per CTA, threads walk the rows): with v = [1; sc * x] (x = the unscaled column jc below
// the diagonal)  F(j, k) = tau * A(rk:, j)' v for the trailing columns j > jc,  F(j0..jc, k) = 0,
// auxv(i) = -tau * A(rk:, j0 + i)' v for the panel columns i < k.
constexpr int QR_GCOLS = 8;
__global__ void __launch_bounds__(256) qr_panel_gemv_kernel(const double* __restrict__ f, int rows, int cols,
                                                            double* __restrict__ F, double* auxv, const QrState* stt, int kk) {
    __shared__ double red[8][QR_GCOLS];
    if (!stt->active || stt->stop) return;
    const int j0 = stt->j0, k = kk;
    if (k >= stt->jb) return;
    const int jc = j0 + k, rk = jc;
    const double tau_k = stt->tau_k, sc = stt->sc_k;
    const int ntrail = cols - jc - 1, nitems = ntrail + k;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const double* x = f + (size_t)jc * rows;
    for (int it0 = blockIdx.x * QR_GCOLS; it0 < nitems; it0 += gridDim.x * QR_GCOLS) {
        const double* cptr[QR_GCOLS];
#pragma unroll
        for (int c = 0; c < QR_GCOLS; ++c) {
            int it = it0 + c;
            if (it >= nitems) it = nitems - 1;
            const int col = (it < ntrail) ? (jc + 1 + it) : (j0 + (it - ntrail));
            cptr[c] = f + (size_t)col * rows;
        }
        double acc[QR_GCOLS];
#pragma unroll
        for (int c = 0; c < QR_GCOLS; ++c) acc[c] = 0.0;
        for (int r = rk + 1 + tid; r < rows; r += 256) {
            const double xv = x[r];
#pragma unroll
            for (int c = 0; c < QR_GCOLS; ++c) acc[c] = fma(cptr[c][r], xv, acc[c]);
        }
#pragma unroll
        for (int c = 0; c < QR_GCOLS; ++c) acc[c] = s_warp_sum(acc[c]);
        __syncthreads();
        if (lane == 0)
#pragma unroll
            for (int c = 0; c < QR_GCOLS; ++c) red[w][c] = acc[c];
        __syncthreads();
        if (tid < QR_GCOLS && it0 + tid < nitems) {
            double t = 0.0;
            for (int q = 0; q < 8; ++q) t += red[q][tid];
            const int it = it0 + tid;
            const int col = (it < ntrail) ? (jc + 1 + it) : (j0 + (it - ntrail));
            const double dotv = f[(size_t)col * rows + rk] + sc * t;          // head of v is 1
            if (it < ntrail) F[(size_t)col * QR_NB + k] = tau_k * dotv;
            else auxv[it - ntrail] = -tau_k * dotv;
        }
    }
    if (blockIdx.x == 0)
        for (int j = j0 + tid; j <= jc; j += blockDim.x) F[(size_t)j * QR_NB + k] = 0.0;
}

// Trailing update of a finished panel (kb = stt->k columns): A(j0+kb:, j0+kb:) -= A(j0+kb:, j0:j0+kb) F(j0+kb:, 0:kb)',
// on the FP64 FMA pipe with coalesced accesses to the trailing matrix.  At K = 32 the update is bound by reading and
// writing C (2 x 8 bytes against 64 flops per element), not by the tensor pipe, and a DMMA tile form touches C in 8 x 8
// patches (half-used sectors; measured 1.0 TB/s, profiles/r2_qr_panel_trail_ncu.txt).
// Here a thread owns one row of a 128 x 32 tile (its 32 panel entries in registers) and 16 of its columns; the lanes of
// a warp are 32 consecutive rows of one column (256-byte segments), F is read from shared memory as 16-byte broadcasts.
constexpr int QT_ROWS = 128, QT_COLS = 32;
__global__ void __launch_bounds__(256) qr_panel_trail_fma_kernel(double* __restrict__ f, int rows, int cols,
                                                                 const double* __restrict__ F, const QrState* stt) {
    __shared__ __align__(16) double Bs[QT_COLS][QR_NB + 2];
    if (!stt->active) return;
    const int j0 = stt->j0, kb = stt->k;
    if (kb <= 0) return;
    const int r0 = j0 + kb, c0 = j0 + kb;
    const int M = rows - r0, N = cols - c0;
    if (M <= 0 || N <= 0) return;
    const int tm = (M + QT_ROWS - 1) / QT_ROWS, tn = (N + QT_COLS - 1) / QT_COLS;
    const int tid = threadIdx.x, rl = tid & (QT_ROWS - 1), cg = tid >> 7;          // cg: columns [16 cg, 16 cg + 16) of the tile
    for (int t = blockIdx.x; t < tm * tn; t += gridDim.x) {
        const int ti = t % tm, tj = t / tm;
        const int r = r0 + ti * QT_ROWS + rl, cbase = c0 + tj * QT_COLS;
        const bool rok = r < rows;
        __syncthreads();
        for (int e = tid; e < QT_COLS * QR_NB; e += 256) {
            const int cc = e >> 5, kk = e & 31;
            Bs[cc][kk] = (cbase + cc < cols && kk < kb) ? F[(size_t)(cbase + cc) * QR_NB + kk] : 0.0;
        }
        double a[QR_NB];
#pragma unroll
        for (int kk = 0; kk < QR_NB; ++kk) a[kk] = (rok && kk < kb) ? f[(size_t)(j0 + kk) * rows + r] : 0.0;
        double acc[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int cc = cbase + cg * 16 + q;
            acc[q] = (rok && cc < cols) ? f[(size_t)cc * rows + r] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const double2* bp = reinterpret_cast<const double2*>(&Bs[cg * 16 + q][0]);
            double c = acc[q];
#pragma unroll
            for (int kk = 0; kk < QR_NB / 2; ++kk) {
                const double2 b = bp[kk];
                c = fma(-a[2 * kk], b.x, c);
                c = fma(-a[2 * kk + 1], b.y, c);
            }
            acc[q] = c;
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int cc = cbase + cg * 16 + q;
            if (rok && cc < cols) f[(size_t)cc * rows + r] = acc[q];
        }
    }
}

// After the trailing update: recompute the flagged norms (dlaqps: the lsticc list), one CTA per candidate column;
// the last CTA to finish (atomic ticket) opens the next panel.
__global__ void __launch_bounds__(256) qr_panel_close_kernel(const double* __restrict__ f, int rows, int cols, double* vn1,
                                                             double* vn2, int* flags, QrState* stt, int topbmn,
                                                             unsigned int* ticket) {
    __shared__ double sh[32];
    __shared__ int s_last;
    if (!stt->active) return;
    const int j0 = stt->j0, kb = stt->k;
    const int rnext = j0 + kb;          // first row of the trailing matrix
    for (int j = rnext + blockIdx.x; j < cols; j += gridDim.x) {
        if (!flags[j]) continue;          // uniform per CTA
        const double* cc = f + (size_t)j * rows;
        double s = 0.0;
        for (int r = rnext + threadIdx.x; r < rows; r += blockDim.x) s = fma(cc[r], cc[r], s);
        s = s_block_sum(s, sh);
        __syncthreads();
        if (threadIdx.x == 0) { vn1[j] = vn2[j] = sqrt(s); flags[j] = 0; }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        *ticket = 0;
        const int nj = j0 + kb;
        stt->j0 = nj; stt->k = 0; stt->stop = 0;
        const int left = topbmn - nj;
        stt->jb = left < QR_NB ? left : QR_NB;
        stt->active = left > 0 ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// One dlaqps panel as ONE persistent cooperative kernel (default; the three-kernels-per-column form above stays selectable
// with ENLSIP_QR_PANEL=graph).  A pivoted column step is a chain of grid-wide dependencies (pivot -> column -> norm ->
// F column -> row / norm downdate -> next pivot); as separate kernels that chain costs three launches and three
// last-CTA tails per column.  Here it is two grid barriers per column:
//   phase P  every CTA combines the per-CTA pivot candidates (same result everywhere); the CTAs that own a slice of rows
//            (slices are fixed for the whole panel, the panel columns of a slice stay in shared memory) bring the pivot
//            column in, scale the previous reflector in place, apply the panel's reflectors to the new column and leave
//            partial sums of squares and partial dot products of the panel columns with it (for auxv);
//   phase Q  every CTA adds the partials in a fixed order and forms the dlarfg scalars and auxv (same bits everywhere);
//            then, on its own chunk of the trailing columns, 16 at a time: the dots with the new reflector (streaming
//            pass over the trailing matrix), and straight away -- one warp per column -- the F entry, the correction of
//            the F column, the pivot-row entry, the partial-norm downdate with its tol3z flag and the pivot candidate
//            of the next column.
// The F row of the column that a pivot exchange moves away from position jc is dead after phase P (only rows behind the
// panel are read later), so the exchange of F rows is a one-way move done by the warp that finishes column `pvt`.
constexpr int QP_THREADS = 512, QP_NW = QP_THREADS / 32, QP_GC = 16, QP_MAXG = 160, QP_MAXRW = 512, QP_MINRW = 128, QP_MAXSLICES = 64;

__device__ __forceinline__ unsigned int qp_ld_acquire(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Barrier over all CTAs of the (co-resident) grid.  bar[0]: epoch reached by the previous launches, bar[1]: exit ticket,
// bar[4 + 8 c]: arrival flag of CTA c (one 32-byte sector each).  A CTA publishes its epoch with a release store to
// its own flag and warp 0 polls all flags.  Measured on B200 (tools/qp_probe.cu, 148 CTAs): SLOWER than one counter
// that every CTA increments and polls (QP_BARRIER_FLAGS=0: bar[2]) -- 5.4 k / 9.5 k cycles for the two barriers of a
// column against 2.7 k / 5.0 k (arrival skew included); the counter is the default.
#ifndef QP_BARRIER_FLAGS
#define QP_BARRIER_FLAGS 0
#endif
__device__ __forceinline__ void qp_grid_barrier(unsigned int* bar, unsigned int& epoch) {
    __syncthreads();
#if QP_BARRIER_FLAGS
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x, G = gridDim.x;
        ++epoch;
        if (lane == 0) {
            __threadfence();
            asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(bar + 4 + 8 * blockIdx.x), "r"(epoch) : "memory");
        }
        bool ok;
        do {
            ok = true;
            for (int q = lane; q < G; q += 32) ok = ok && ((int)(qp_ld_acquire(bar + 4 + 8 * q) - epoch) >= 0);
        } while (!__all_sync(0xffffffffu, ok));
        __threadfence();
    }
#else
    if (threadIdx.x == 0) {
        epoch += gridDim.x;
        __threadfence();
        atomicAdd(bar + 2, 1u);
        while (qp_ld_acquire(bar + 2) < epoch) { }
        __threadfence();
    }
#endif
    __syncthreads();
}
__device__ __forceinline__ void qp_first_max(double& b, int& bi, double ob, int oi) {
    if (ob > b || (ob == b && oi < bi)) { b = ob; bi = oi; }
}
__host__ __device__ inline int qp_rows_per_slice(int rows, int G) {          // at most QP_MAXSLICES slices
    const int ns = G < QP_MAXSLICES ? G : QP_MAXSLICES;
    const int rw = (rows + ns - 1) / ns;
    return rw < QP_MINRW ? QP_MINRW : rw;
}
inline size_t qp_smem_bytes(int rows, int G) {
    return sizeof(double) * ((size_t)qp_rows_per_slice(rows, G) * (QR_NB + 2) + (size_t)QP_GC * QP_THREADS);
}

#ifdef QP_PROF
__device__ unsigned long long qp_prof[8];      // cycles of CTA 0 per phase, summed over the columns (tools/qp_probe.cu)
#define QP_STAMP(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { const long long t_ = clock64(); qp_prof[i] += (unsigned long long)(t_ - qp_t); qp_t = t_; } } while (0)
#else
#define QP_STAMP(i) do { } while (0)
#endif
__global__ void __launch_bounds__(QP_THREADS, 1)
qr_panel_persist_kernel(double* f, int rows, int cols, double* vn1, double* vn2, int* jpvt, double* tau, double* F,
                        int* flags, QrState* stt, double* pbest, int* pidx, int* pany, double* ppart, unsigned int* bar) {
    extern __shared__ double qp_dyn[];
    __shared__ double s_tot[QR_NB + 1];
    __shared__ double s_aux[QR_NB], s_frow[QR_NB], s_prow[QR_NB];
    __shared__ double s_best[QP_NW];
    __shared__ int s_idx[QP_NW], s_any[QP_NW];
    __shared__ double s_scal[3];
    __shared__ int s_pv[2];
    if (!stt->active) return;
    const int j0 = stt->j0, jb = stt->jb, nopivot = stt->nopivot;
    const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int rw = qp_rows_per_slice(rows, G), Gp = (rows + rw - 1) / rw;
    const int r0 = c * rw, nr = (c < Gp) ? ((rows - r0 < rw) ? rows - r0 : rw) : 0;
    double* Vs = qp_dyn;                          // [rw][QR_NB + 1]: this slice of the panel columns
    double* s_a = qp_dyn + (size_t)rw * (QR_NB + 1);   // [rw]: the new column
    double* s_acc = s_a + rw;                          // [QP_GC][QP_THREADS]: partial dot products of a column group
    constexpr int VL = QR_NB + 1;
#if QP_BARRIER_FLAGS
    unsigned int epoch = __ldcg(bar);             // continues where the previous launch stopped (flags are never reset)
#else
    unsigned int epoch = 0;
#endif
    int kb = jb;

    // pivot candidates of the first column: first maximum of vn1 over this CTA's chunk of [j0, cols)
    {
        const int nt = cols - j0, cw = (nt + G - 1) / G;
        const int jbeg = j0 + c * cw, jend = (jbeg + cw < cols) ? jbeg + cw : cols;
        double b = -1.0; int bi = cols;
        for (int j = jbeg + tid; j < jend; j += QP_THREADS) qp_first_max(b, bi, __ldcg(vn1 + j), j);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            qp_first_max(b, bi, __shfl_xor_sync(0xffffffffu, b, o), __shfl_xor_sync(0xffffffffu, bi, o));
        if (lane == 0) { s_best[w] = b; s_idx[w] = bi; }
        __syncthreads();
        if (tid == 0) {
            for (int q = 1; q < QP_NW; ++q) qp_first_max(b, bi, s_best[q], s_idx[q]);
            pbest[c] = b; pidx[c] = bi; pany[c] = 0;
        }
        qp_grid_barrier(bar, epoch);
    }

#ifdef QP_PROF
    long long qp_t = clock64();
#endif
    for (int k = 0; k < jb; ++k) {
        const int jc = j0 + k, rk = jc;
        // ---------------- phase P ----------------
        QP_STAMP(7);
        if (w == 0) {
            double b = -1.0; int bi = cols, any = 0;
            {
                constexpr int NU = (QP_MAXG + 31) / 32;
                double cb[NU]; int ci[NU], ca[NU];
#pragma unroll
                for (int u = 0; u < NU; ++u) {            // all loads in flight together
                    const int q = lane + 32 * u;
                    cb[u] = (q < G) ? __ldcg(pbest + q) : -1.0;
                    ci[u] = (q < G) ? __ldcg(pidx + q) : cols;
                    ca[u] = (q < G) ? __ldcg(pany + q) : 0;
                }
#pragma unroll
                for (int u = 0; u < NU; ++u) { qp_first_max(b, bi, cb[u], ci[u]); any |= ca[u]; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
                qp_first_max(b, bi, __shfl_xor_sync(0xffffffffu, b, o), __shfl_xor_sync(0xffffffffu, bi, o));
            any = __any_sync(0xffffffffu, any);
            if (bi >= cols || nopivot) bi = jc;
            if (lane == 0) { s_pv[0] = bi; s_pv[1] = any; }
        }
        __syncthreads();
        const int pvt = s_pv[0];
        if (s_pv[1]) { kb = k; break; }               // a norm has to be recomputed: the panel ends (dlaqps lsticc)
        QP_STAMP(0);
        {
            // every load that depends on the pivot only goes out before the block barrier (QP_MAXRW == QP_THREADS:
            // a thread owns at most one row of the slice)
            const bool has_row = tid < nr;
            const int r = r0 + tid;
            double* cj = f + (size_t)jc * rows;
            double* cp = f + (size_t)pvt * rows;
            double a = 0.0, oldj = 0.0;
            if (has_row) { a = __ldcg(cp + r); if (pvt != jc) oldj = __ldcg(cj + r); }
            if (tid < QR_NB) s_frow[tid] = (tid < k) ? __ldcg(F + (size_t)pvt * QR_NB + tid) : 0.0;
            if (c == 0 && tid == 0 && pvt != jc) {
                const int tp = __ldcg(jpvt + pvt); jpvt[pvt] = __ldcg(jpvt + jc); jpvt[jc] = tp;
                vn1[pvt] = __ldcg(vn1 + jc); vn2[pvt] = __ldcg(vn2 + jc);
            }
            __syncthreads();
            if (nr > 0) {
                const double sc_prev = s_scal[1], beta_prev = s_scal[2];
                if (has_row) {
                    double* vrow = Vs + (size_t)tid * VL;
                    if (pvt != jc) cp[r] = oldj;
                    if (k > 0) {                          // the previous reflector: v = [1; x * sc], R(rk-1, jc-1) = beta
                        double* cq = f + (size_t)(jc - 1) * rows;
                        if (r > rk - 1) {
                            if (sc_prev != 1.0) { const double v = vrow[k - 1] * sc_prev; cq[r] = v; vrow[k - 1] = v; }
                        } else if (r == rk - 1) {
                            cq[r] = beta_prev;
                        }
                    }
                    if (r >= rk) {
                        double s = 0.0;
#pragma unroll 8
                        for (int i = 0; i < k; ++i) s = fma(vrow[i], s_frow[i], s);
                        a -= s;
                        vrow[k] = a;
                    }
                    s_a[tid] = (r > rk) ? a : 0.0;
                    cj[r] = a;
                }
                __syncthreads();
                // partial sums over this slice: warp per quantity (i < k: panel column i . a ; i == k: a . a), fixed order
                for (int i = w; i <= k; i += QP_NW) {
                    double t = 0.0;
                    if (i < k) { for (int rl = lane; rl < nr; rl += 32) if (r0 + rl > rk) t = fma(Vs[rl * VL + i], s_a[rl], t); }
                    else { for (int rl = lane; rl < nr; rl += 32) t = fma(s_a[rl], s_a[rl], t); }
                    t = s_warp_sum(t);
                    if (lane == 0) ppart[(size_t)c * VL + (i < k ? i : QR_NB)] = t;
                }
            }
        }
        QP_STAMP(1);
        qp_grid_barrier(bar, epoch);
        QP_STAMP(2);

        // ---------------- phase Q ----------------
        // (Deferring this block behind the first streaming pass -- the dots need none of the dlarfg scalars -- was
        // measured: no gain, the values held across the pass cost the streaming loop its registers.)
        double alpha = 0.0, prow = 0.0;
        if (w == 0) {
            alpha = __ldcg(f + (size_t)jc * rows + rk);
            if (lane < k) prow = __ldcg(f + (size_t)(j0 + lane) * rows + rk);
            else if (lane == k) prow = 1.0;
        }
        // 16 threads per quantity (i < k: dot of panel column i with the new column; i == k: its sum of squares)
        constexpr int NPU = QP_MAXSLICES / 16;
        const int qi = tid >> 4, qsub = tid & 15;
        const int qslot = (qi < k) ? qi : QR_NB;
        double part[NPU];
#pragma unroll
        for (int u = 0; u < NPU; ++u) {
            const int q = qsub + 16 * u;
            part[u] = (qi <= k && q < Gp) ? __ldcg(ppart + (size_t)q * VL + qslot) : 0.0;
        }
        auto scalars = [&]() {                       // all threads; fixed summation order, the same bits in every CTA
            double t = 0.0;
#pragma unroll
            for (int u = 0; u < NPU; ++u) t += part[u];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (qsub == 0 && qi <= k) s_tot[qslot] = t;
            __syncthreads();
            if (w == 0) {
                double beta = alpha, tau_k = 0.0, sc = 1.0;
                if (rk < rows - 1) {
                    const double xn = sqrt(s_tot[QR_NB]);
                    if (xn != 0.0) {
                        beta = -copysign(s_lapy2(alpha, xn), alpha);
                        tau_k = (beta - alpha) / beta;
                        sc = 1.0 / (alpha - beta);
                    }
                }
                if (lane == 0) {
                    s_scal[0] = tau_k; s_scal[1] = sc; s_scal[2] = beta;
                    if (c == 0) tau[jc] = tau_k;
                }
                s_prow[lane] = prow;
                s_aux[lane] = (lane < k) ? -tau_k * (prow + sc * s_tot[lane]) : 0.0;
            }
            __syncthreads();
        };
        scalars();
        QP_STAMP(3);
        {
            const double tau_k = s_scal[0], sc = s_scal[1], aux_l = s_aux[lane], prow_l = s_prow[lane];
            const int ntrail = cols - jc - 1, cw = (ntrail + G - 1) / G;
            const int jbeg = jc + 1 + c * cw, jend = (jbeg + cw < cols) ? jbeg + cw : cols;
            const int ncol = jend > jbeg ? jend - jbeg : 0;
            const int ngrp = (ncol + QP_GC - 1) / QP_GC, gsz = ngrp ? (ncol + ngrp - 1) / ngrp : 0;   // even groups of <= 16
            const double* x = f + (size_t)jc * rows;
            double best = -1.0; int bidx = cols, any = 0;
            for (int g0 = jbeg; g0 < jend; g0 += gsz) {
                const int nc = (jend - g0 < gsz) ? jend - g0 : gsz;
                // what the finishing warp of column g0 + w needs, in flight during the streaming pass
                const int j = g0 + w;
                const bool fin = w < nc;
                const bool moved = fin && (j == pvt && pvt != jc);
                double fl = 0.0, arkj = 0.0, v1 = 0.0, v2 = 1.0;
                if (fin) {
                    if (lane < k) fl = __ldcg(F + (size_t)(moved ? jc : j) * QR_NB + lane);
                    if (lane == 0) { arkj = __ldcg(f + (size_t)j * rows + rk); v1 = __ldcg(vn1 + j); v2 = __ldcg(vn2 + j); }
                }
                double acc[QP_GC];
#pragma unroll
                for (int q = 0; q < QP_GC; ++q) acc[q] = 0.0;
                const double* base = f + (size_t)g0 * rows;
                if (nc == QP_GC) {
#pragma unroll 2
                    for (int r = rk + 1 + tid; r < rows; r += QP_THREADS) {
                        const double xv = __ldcg(x + r);
#pragma unroll
                        for (int q = 0; q < QP_GC; ++q) acc[q] = fma(__ldcg(base + (size_t)q * rows + r), xv, acc[q]);
                    }
                } else if (nc <= QP_GC / 2) {        // few columns per CTA: latency bound, deeper unrolling
#pragma unroll 4
                    for (int r = rk + 1 + tid; r < rows; r += QP_THREADS) {
                        const double xv = __ldcg(x + r);
#pragma unroll
                        for (int q = 0; q < QP_GC / 2; ++q)
                            if (q < nc) acc[q] = fma(__ldcg(base + (size_t)q * rows + r), xv, acc[q]);
                    }
                } else {
#pragma unroll 2
                    for (int r = rk + 1 + tid; r < rows; r += QP_THREADS) {
                        const double xv = __ldcg(x + r);
#pragma unroll
                        for (int q = 0; q < QP_GC; ++q)
                            if (q < nc) acc[q] = fma(__ldcg(base + (size_t)q * rows + r), xv, acc[q]);
                    }
                }
                // the per-thread partial sums go through shared memory; the finishing warp of a column adds the 512 partials
                // of its column (16 per lane in a fixed order, then the lane tree): 10 shuffles per warp instead of 62
#pragma unroll
                for (int q = 0; q < QP_GC; ++q)
                    if (q < nc) s_acc[q * QP_THREADS + tid] = acc[q];
                __syncthreads();
                if (fin) {                          // finish column j: one warp, lane = panel index
                    double t = 0.0;
#pragma unroll
                    for (int u = 0; u < QP_NW; ++u) t += s_acc[w * QP_THREADS + lane + 32 * u];
                    t = s_warp_sum(t);
                    arkj = __shfl_sync(0xffffffffu, arkj, 0);
                    v1 = __shfl_sync(0xffffffffu, v1, 0);
                    v2 = __shfl_sync(0xffffffffu, v2, 0);
                    const double dotv = arkj + sc * t;                       // head of v is 1
                    const double s = s_warp_sum(fl * aux_l);
                    const double fjk = tau_k * dotv + s;
                    if (lane == k) fl = fjk;
                    if (moved ? (lane <= k) : (lane == k)) F[(size_t)j * QR_NB + lane] = fl;
                    const double ru = s_warp_sum(prow_l * fl);            // sum_{i <= k} A(rk, j0 + i) F(j, i)
                    const double a = arkj - ru;
                    if (v1 != 0.0) {
                        double temp = fabs(a) / v1;
                        temp = fmax(0.0, (1.0 + temp) * (1.0 - temp));
                        const double rq = v1 / v2;
                        if (temp * (rq * rq) <= S_TOL3Z && !nopivot) { any = 1; if (lane == 0) flags[j] = 1; }
                        else { v1 = v1 * sqrt(temp); if (lane == 0) vn1[j] = v1; }
                    }
                    if (lane == 0) f[(size_t)j * rows + rk] = a;
                    if (v1 > best) { best = v1; bidx = j; }
                }
                __syncthreads();
            }
            if (lane == 0) { s_best[w] = best; s_idx[w] = bidx; s_any[w] = any; }
            __syncthreads();
            if (w == 0) {
                double b = (lane < QP_NW) ? s_best[lane] : -1.0;
                int bi = (lane < QP_NW) ? s_idx[lane] : cols;
                const int an = __any_sync(0xffffffffu, (lane < QP_NW) ? s_any[lane] : 0);
#pragma unroll
                for (int o = QP_NW / 2; o > 0; o >>= 1)
                    qp_first_max(b, bi, __shfl_xor_sync(0xffffffffu, b, o), __shfl_xor_sync(0xffffffffu, bi, o));
                if (lane == 0) { pbest[c] = b; pidx[c] = bi; pany[c] = an; }
            }
        }
        QP_STAMP(4);
        qp_grid_barrier(bar, epoch);
        QP_STAMP(5);
    }
    // the last reflector of the panel: scale in place, store beta
    if (kb > 0 && nr > 0) {
        const int kl = kb - 1, rkl = j0 + kl;
        const double sc = s_scal[1], beta = s_scal[2];
        double* cq = f + (size_t)rkl * rows;
        for (int rl = tid; rl < nr; rl += QP_THREADS) {
            const int r = r0 + rl;
            if (r > rkl) { if (sc != 1.0) cq[r] = Vs[rl * VL + kl] * sc; }
            else if (r == rkl) cq[r] = beta;
        }
    }
    if (tid == 0) {
        if (c == 0) { stt->k = kb; stt->stop = 0; }
        __threadfence();
        if (atomicAdd(bar + 1, 1u) == (unsigned int)G - 1) {     // last CTA out: nobody polls any more
#if QP_BARRIER_FLAGS
            bar[0] = epoch;
#else
            bar[2] = 0;
#endif
            bar[1] = 0;
            __threadfence();
        }
    }
}

// ---- unblocked dlaqp2 steps (the last min(m,n) - topbmn columns; host-driven column index i) ----
__global__ void __launch_bounds__(1024) qr_p2_pivot_house_kernel(double* __restrict__ f, int rows, int cols, int i,
                                                                  double* vn1, double* vn2, int* jpvt, double* tau, int nopivot) {
    __shared__ double sh[32];
    __shared__ double s_best[32];
    __shared__ int s_idx[32];
    __shared__ int s_pvt;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
    double best = -1.0; int idx = cols;
    for (int j = i + tid; j < cols; j += blockDim.x) {
        const double v = vn1[j];
        if (v > best) { best = v; idx = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ob > best || (ob == best && oi < idx)) { best = ob; idx = oi; }
    }
    if (lane == 0) { s_best[w] = best; s_idx[w] = idx; }
    __syncthreads();
    if (tid == 0) {
        double b = s_best[0]; int bi = s_idx[0];
        for (int q = 1; q < nw; ++q)
            if (s_best[q] > b || (s_best[q] == b && s_idx[q] < bi)) { b = s_best[q]; bi = s_idx[q]; }
        if (bi >= cols || nopivot) bi = i;
        s_pvt = bi;
        if (bi != i) {
            const int tp = jpvt[bi]; jpvt[bi] = jpvt[i]; jpvt[i] = tp;
            vn1[bi] = vn1[i]; vn2[bi] = vn2[i];
        }
    }
    __syncthreads();
    const int pvt = s_pvt;
    double* ci = f + (size_t)i * rows;
    if (pvt != i) {
        double* cp = f + (size_t)pvt * rows;
        for (int r = tid; r < rows; r += blockDim.x) { const double a = ci[r]; ci[r] = cp[r]; cp[r] = a; }
    }
    __syncthreads();
    double tau_i = 0.0;
    if (i < rows - 1) {
        double s = 0.0;
        for (int r = i + 1 + tid; r < rows; r += blockDim.x) s = fma(ci[r], ci[r], s);
        s = s_block_sum(s, sh);
        const double xn = sqrt(s);
        if (xn != 0.0) {
            const double alpha = ci[i];
            const double beta = -copysign(s_lapy2(alpha, xn), alpha);
            tau_i = (beta - alpha) / beta;
            const double sc = 1.0 / (alpha - beta);
            __syncthreads();
            for (int r = i + 1 + tid; r < rows; r += blockDim.x) ci[r] *= sc;
            if (tid == 0) ci[i] = beta;
        }
    }
    if (tid == 0) tau[i] = tau_i;
}

// apply H_i to the trailing columns (one warp per column) + dlaqp2 partial-norm downdate of that column.  STAGED: the
// reflector is first copied to shared memory (len <= VEC_STAGE_MAX); otherwise it is read from column i of f, which this
// launch does not write.  Both forms add in the same order, so they give the same bits.
constexpr int VEC_STAGE_MAX = 6144;   // doubles in the 48 KB of dynamic shared memory a launch gets without an opt-in
template <bool STAGED>
__global__ void __launch_bounds__(256) qr_p2_apply_kernel(double* __restrict__ f, int rows, int cols, int i, double* vn1,
                                                          double* vn2, const double* __restrict__ tau) {
    extern __shared__ double vsm[];
    const int len = rows - i - 1;
    const double* v = f + (size_t)i * rows + i + 1;
    if (STAGED) {
        for (int r = threadIdx.x; r < len; r += blockDim.x) vsm[r] = v[r];
        __syncthreads();
    }
    const double* vs = STAGED ? vsm : v;
    const double tau_i = tau[i];
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int c = i + 1 + gw; c < cols; c += nwarps) {
        double* cc = f + (size_t)c * rows + i;
        double ci = cc[0];
        if (tau_i != 0.0) {
            double s = 0.0;
            for (int r = lane; r < len; r += 32) s = fma(vs[r], cc[1 + r], s);
            s = s_warp_sum(s);
            const double wv = (ci + s) * tau_i;
            for (int r = lane; r < len; r += 32) cc[1 + r] = fma(-wv, vs[r], cc[1 + r]);
            ci -= wv;
            if (lane == 0) cc[0] = ci;
        }
        __syncwarp();
        const double v1 = vn1[c];
        if (v1 != 0.0) {
            const double tq = fabs(ci) / v1;
            const double temp = fmax(1.0 - tq * tq, 0.0);
            const double rq = v1 / vn2[c];
            const double temp2 = temp * (rq * rq);
            if (temp2 <= S_TOL3Z) {
                double s = 0.0;
                if (i < rows - 1) {
                    for (int r = lane; r < len; r += 32) s = fma(cc[1 + r], cc[1 + r], s);
                    s = s_warp_sum(s);
                }
                if (lane == 0) vn1[c] = vn2[c] = sqrt(s);
            } else if (lane == 0) {
                vn1[c] = v1 * sqrt(temp);
            }
        }
    }
}

// ---- the whole factorisation in ONE THREAD-BLOCK CLUSTER (dlaqp2 semantics), the matrix resident in shared memory ----
// Column c of the matrix lives in the shared memory of CTA c % 8 (slot c / 8).  Per column step: every CTA proposes its
// best remaining column (first maximum of the partial norms by current position), the proposals are exchanged through
// distributed shared memory, the owner of the winner runs dlarfg and stores the reflector into every CTA's shared
// memory, then each CTA applies it to its own columns (one warp per column) and downdates their norms.  Two cluster
// barriers per step and no L2 round trip: a 257 x 192 factorisation (config 4's J2) takes 1.04 ms (5 us per column).
// (A variant with ONE barrier per step -- every CTA ships its candidate column with the proposal and runs dlarfg
// redundantly -- was measured slower: 1.33 ms; the 8-fold column traffic through distributed shared memory costs more
// than the barrier it saves.)
// Columns are never moved: `pos` tracks the position dlaqp2's swaps would have given them.
constexpr int QC_MAXCTAS = 8, QC_THREADS = 512;   // (1024 threads: 0.43 / 0.38 / 1.34 ms instead of 0.30 / 0.26 / 1.05: wider barriers cost more than the second round of column updates)
constexpr size_t QC_MAX_SMEM = 200 * 1024;
inline size_t qc_smem_bytes(int rows, int cols, int nctas) {
    const int ncl = (cols + nctas - 1) / nctas;
    return sizeof(double) * ((size_t)ncl * rows + rows + 2 + 2 * (size_t)ncl + QC_MAXCTAS) + sizeof(int) * ((size_t)ncl + cols + 2 * QC_MAXCTAS + 2);
}
template <int QC_CTAS>
__global__ void __cluster_dims__(QC_CTAS, 1, 1) __launch_bounds__(QC_THREADS)
qr_cluster_kernel(double* __restrict__ f, int rows, int cols, double* __restrict__ tau, int* __restrict__ jpvt, int nopivot) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    extern __shared__ double sm[];
    __shared__ double sh[32];
    __shared__ double s_rb[32];
    __shared__ int s_rp[32], s_rs[32];
    __shared__ int s_wphys;
    const int ncl = (cols + QC_CTAS - 1) / QC_CTAS;
    double* Al = sm;                                // [ncl][rows]
    double* vbuf = Al + (size_t)ncl * rows;         // [rows] reflector (entries i+1..), [rows] = tau
    double* vn1 = vbuf + rows + 2;                  // [ncl]
    double* vn2 = vn1 + ncl;                        // [ncl]
    double* cval = vn2 + ncl;                       // [QC_CTAS] proposals: value
    int* pos = reinterpret_cast<int*>(cval + QC_MAXCTAS);   // [ncl] current position of the local column
    int* l2p = pos + ncl;                           // [cols] position -> column (replicated in every CTA)
    int* cpos = l2p + cols;                         // [QC_CTAS] proposals: position
    int* cphys = cpos + QC_MAXCTAS;                    // [QC_CTAS] proposals: column
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = QC_THREADS / 32;
    const int nloc = (cols > rank) ? (cols - rank + QC_CTAS - 1) / QC_CTAS : 0;     // my columns: rank, rank + 8, ...
    const int k = rows < cols ? rows : cols;
    for (int s = w; s < nloc; s += nw) {
        const double* src = f + (size_t)(rank + s * QC_CTAS) * rows;
        double* dst = Al + (size_t)s * rows;
        double acc = 0.0;
        for (int r = lane; r < rows; r += 32) { const double x = src[r]; dst[r] = x; acc = fma(x, x, acc); }
        acc = s_warp_sum(acc);
        if (lane == 0) { vn1[s] = vn2[s] = sqrt(acc); pos[s] = rank + s * QC_CTAS; }
    }
    for (int c = tid; c < cols; c += QC_THREADS) l2p[c] = c;
    cluster.sync();        // every CTA has read its input: the output may overwrite f at the end
    for (int i = 0; i < k; ++i) {
        // ---- 1. local proposal: largest vn1 among my columns still to the right of i, ties -> smallest position
        double best = -1.0; int bpos = 0x7fffffff, bslot = -1;
        for (int s = tid; s < nloc; s += QC_THREADS) {
            const int p = pos[s];
            if (p >= i) {
                const double x = vn1[s];
                if (x > best || (x == best && p < bpos)) { best = x; bpos = p; bslot = s; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int op = __shfl_xor_sync(0xffffffffu, bpos, o);
            const int os = __shfl_xor_sync(0xffffffffu, bslot, o);
            if (ob > best || (ob == best && op < bpos)) { best = ob; bpos = op; bslot = os; }
        }
        if (lane == 0) { s_rb[w] = best; s_rp[w] = bpos; s_rs[w] = bslot; }
        __syncthreads();
        if (tid < QC_CTAS) {
            double b = s_rb[0]; int bp = s_rp[0], bs = s_rs[0];
            for (int q = 1; q < nw; ++q)
                if (s_rb[q] > b || (s_rb[q] == b && s_rp[q] < bp)) { b = s_rb[q]; bp = s_rp[q]; bs = s_rs[q]; }
            // thread t delivers this CTA's proposal to CTA t
            double* rv = cluster.map_shared_rank(cval, tid);
            int* rp = cluster.map_shared_rank(cpos, tid);
            int* rph = cluster.map_shared_rank(cphys, tid);
            rv[rank] = b; rp[rank] = bp; rph[rank] = (bs >= 0) ? (rank + bs * QC_CTAS) : -1;
        }
        cluster.sync();
        // ---- 2. the winner, identically in every CTA; position bookkeeping of dlaqp2's column swap
        if (tid == 0) {
            double b = -1.0; int bp = 0x7fffffff, bph = -1;
            for (int q = 0; q < QC_CTAS; ++q)
                if (cphys[q] >= 0 && (cval[q] > b || (cval[q] == b && cpos[q] < bp))) { b = cval[q]; bp = cpos[q]; bph = cphys[q]; }
            if (bph < 0 || nopivot) { bp = i; bph = l2p[i]; }   // nothing comparable (NaN norms) / plain QR: the column stays
            const int q = l2p[i];                           // the column sitting at position i moves to the winner's place
            l2p[bp] = q; l2p[i] = bph;
            if (q % QC_CTAS == rank) pos[q / QC_CTAS] = bp;
            if (bph % QC_CTAS == rank) pos[bph / QC_CTAS] = i;
            s_wphys = bph;
        }
        __syncthreads();
        const int wphys = s_wphys;
        // ---- 3. owner: dlarfg, reflector into every CTA
        if (wphys % QC_CTAS == rank) {
            double* col = Al + (size_t)(wphys / QC_CTAS) * rows;
            double tau_i = 0.0;
            if (i < rows - 1) {
                double part = 0.0;
                for (int r = i + 1 + tid; r < rows; r += QC_THREADS) part = fma(col[r], col[r], part);
                const double xn = sqrt(s_block_sum(part, sh));
                if (xn != 0.0) {
                    const double alpha = col[i];
                    const double beta = -copysign(s_lapy2(alpha, xn), alpha);
                    tau_i = (beta - alpha) / beta;
                    const double sc = 1.0 / (alpha - beta);
                    __syncthreads();
                    for (int r = i + 1 + tid; r < rows; r += QC_THREADS) col[r] *= sc;
                    if (tid == 0) col[i] = beta;
                    __syncthreads();
                }
            }
            const int len = rows - i - 1;
            for (int e = tid; e < (len + 1) * QC_CTAS; e += QC_THREADS) {
                const int dstr = e % QC_CTAS, r = e / QC_CTAS;       // r == len: the tau slot
                double* rv = cluster.map_shared_rank(vbuf, dstr);
                if (r < len) rv[i + 1 + r] = col[i + 1 + r];
                else rv[rows] = tau_i;
            }
            if (tid == 0) tau[i] = tau_i;
        }
        cluster.sync();
        // ---- 4. H_i on my remaining columns + dlaqp2 norm downdate, one warp per column
        const double tau_i = vbuf[rows];
        const int len = rows - i - 1;
        for (int s = w; s < nloc; s += nw) {
            if (pos[s] <= i) continue;
            double* cc = Al + (size_t)s * rows + i;
            double c0 = cc[0];
            if (tau_i != 0.0) {
                double acc = 0.0;
                for (int r = lane; r < len; r += 32) acc = fma(vbuf[i + 1 + r], cc[1 + r], acc);
                acc = s_warp_sum(acc);
                const double wv = (c0 + acc) * tau_i;
                for (int r = lane; r < len; r += 32) cc[1 + r] = fma(-wv, vbuf[i + 1 + r], cc[1 + r]);
                c0 -= wv;
                __syncwarp();
                if (lane == 0) cc[0] = c0;
            }
            const double v1 = vn1[s];
            if (v1 != 0.0) {
                const double tq = fabs(c0) / v1;
                const double temp = fmax(1.0 - tq * tq, 0.0);
                const double rq = v1 / vn2[s];
                if (temp * (rq * rq) <= S_TOL3Z) {
                    double acc = 0.0;
                    if (i < rows - 1) {
                        for (int r = lane; r < len; r += 32) acc = fma(cc[1 + r], cc[1 + r], acc);
                        acc = s_warp_sum(acc);
                    }
                    __syncwarp();
                    if (lane == 0) vn1[s] = vn2[s] = sqrt(acc);
                } else {
                    __syncwarp();
                    if (lane == 0) vn1[s] = v1 * sqrt(temp);
                }
            }
        }
        __syncthreads();
    }
    cluster.sync();
    // output in dgeqp3 layout: the column now at position p goes to column p of f
    for (int s = w; s < nloc; s += nw) {
        const int p = pos[s];
        const double* src = Al + (size_t)s * rows;
        double* dst = f + (size_t)p * rows;
        for (int r = lane; r < rows; r += 32) dst[r] = src[r];
        if (lane == 0) jpvt[p] = rank + s * QC_CTAS;
    }
}

// R of a factored rows x nc matrix (dgeqrf layout, column major) -> out (nc x nc column major), zeros below the diagonal
// and in rows >= rows
__global__ void upper_to_square_kernel(const double* __restrict__ f, int rows, int nc, double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)nc * nc) return;
    const int r = (int)(e % nc), c = (int)(e / nc);
    out[e] = (r <= c && r < rows) ? f[(size_t)c * rows + r] : 0.0;
}

// diag(R) and the inverse permutation of a finished factorisation
__global__ void qr_finish_kernel(const double* __restrict__ f, int rows, int cols, const int* __restrict__ jpvt,
                                 double* diag, int* ipvt) {
    const int k = rows < cols ? rows : cols;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < k) diag[i] = f[(size_t)i * rows + i];
    if (i < cols) ipvt[jpvt[i]] = i;
}

struct QrGraph {          // one dlaqps panel (3 x 32 + 3 kernels) captured as a CUDA graph; indices come from the device state
    cudaGraphExec_t exec = nullptr;
    const void* f = nullptr; int rows = 0, cols = 0; const void* tau = nullptr; const void* jpvt = nullptr; int topbmn = 0;
};
constexpr int QR_PSUM_LEN = QP_MAXG * (QR_NB + 1) > QR_MAXPART ? QP_MAXG * (QR_NB + 1) : QR_MAXPART;   // doubles in QrWork::psum
constexpr int QR_PIDX_LEN = QR_MAXPART + QP_MAXG;                                                    // ints in QrWork::pidx
constexpr int QR_TICKET_LEN = 8 + 8 * QP_MAXG;   // [0] close ticket; from [1]: the grid barrier of the persistent panel (qp_grid_barrier)
struct QrWork {          // scratch of one factorisation (sized for the largest matrix of the solve)
    double *vn1 = nullptr, *vn2 = nullptr, *F = nullptr, *auxv = nullptr, *pbest = nullptr, *psum = nullptr;   // psum: QR_PSUM_LEN
    int *flags = nullptr, *pidx = nullptr;                                                                     // pidx: QR_PIDX_LEN
    QrState* state = nullptr;
    unsigned int* ticket = nullptr;                                                                            // QR_TICKET_LEN
    int cap_cols = 0;
    QrGraph graphs[6];
    int next_graph = 0;
    bool use_graphs = true;
    void drop_graphs() {
        for (QrGraph& g : graphs) { if (g.exec) cudaGraphExecDestroy(g.exec); g = QrGraph(); }
    }
};

// grid of the persistent panel kernel (one CTA per SM, co-resident: cooperative launch); 0 = not available
inline int qp_grid() {
    static const int g = [] {
        const char* e = getenv("ENLSIP_QR_PANEL");
        if (e && e[0] == 'g') return 0;                        // "graph": the three-kernels-per-column form
        int dev = 0, sms = 0, coop = 0, per_sm = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (!coop || sms <= 0) return 0;
        const int max_dyn = (int)(sizeof(double) * (QP_MAXRW * (QR_NB + 2) + QP_GC * QP_THREADS));
        if (cudaFuncSetAttribute(qr_panel_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, qr_panel_persist_kernel, QP_THREADS, max_dyn) != cudaSuccess ||
            per_sm < 1) {
            cudaGetLastError();
            return 0;
        }
        return sms < QP_MAXG ? sms : QP_MAXG;
    }();
    return g;
}
inline int qr_enqueue_panel_persist(double* f, int rows, int cols, double* tau, int* jpvt, QrWork& wk, int topbmn, int G,
                                    cudaStream_t st) {
    double *vn1 = wk.vn1, *vn2 = wk.vn2, *F = wk.F, *pbest = wk.pbest, *ppart = wk.psum;
    int *flags = wk.flags, *pidx = wk.pidx, *pany = wk.pidx + QR_MAXPART;
    QrState* stt = wk.state;
    unsigned int* bar = wk.ticket + 1;
    void* args[] = {&f, &rows, &cols, &vn1, &vn2, &jpvt, &tau, &F, &flags, &stt, &pbest, &pidx, &pany, &ppart, &bar};
    cudaLaunchCooperativeKernel((const void*)qr_panel_persist_kernel, dim3(G), dim3(QP_THREADS), args, qp_smem_bytes(rows, G), st);
    qr_panel_trail_fma_kernel<<<148 * 4, 256, 0, st>>>(f, rows, cols, wk.F, wk.state);
    qr_panel_close_kernel<<<148, 256, 0, st>>>(f, rows, cols, wk.vn1, wk.vn2, wk.flags, wk.state, topbmn, wk.ticket);
    return 3;
}

inline int qr_enqueue_panel(double* f, int rows, int cols, double* tau, int* jpvt, QrWork& wk, int topbmn, cudaStream_t st) {
    const int g_fin = imin_host((cols + 7) / 8, QR_MAXPART), g_col = imin_host((rows + 255) / 256, QR_MAXPART);
    const int g_gemv = imin_host((cols + QR_GCOLS - 1) / QR_GCOLS + 4, 148 * 8);
    int launches = 0;
    for (int k = 0; k < QR_NB; ++k) {
        qr_panel_finish_pivot_kernel<<<g_fin, 256, 0, st>>>(f, rows, cols, wk.vn1, wk.vn2, jpvt, wk.F, wk.auxv, wk.flags, wk.state, wk.pbest, wk.pidx, k);
        qr_panel_column_kernel<<<g_col, 256, 0, st>>>(f, rows, cols, tau, wk.F, wk.state, wk.psum, k);
        qr_panel_gemv_kernel<<<g_gemv, 256, 0, st>>>(f, rows, cols, wk.F, wk.auxv, wk.state, k);
        launches += 3;
    }
    qr_panel_finish_pivot_kernel<<<g_fin, 256, 0, st>>>(f, rows, cols, wk.vn1, wk.vn2, jpvt, wk.F, wk.auxv, wk.flags, wk.state, wk.pbest, wk.pidx, QR_NB);
    qr_panel_trail_fma_kernel<<<148 * 4, 256, 0, st>>>(f, rows, cols, wk.F, wk.state);
    qr_panel_close_kernel<<<148, 256, 0, st>>>(f, rows, cols, wk.vn1, wk.vn2, wk.flags, wk.state, topbmn, wk.ticket);
    return launches + 3;
}

// f: rows x cols column major on the device, factored in place (dgeqp3 layout); tau [min(rows, cols)]; jpvt [cols]
// (0-based).  Returns the number of kernels launched, or -1 (nothing launched) when `cols` exceeds the per-column scratch
// of `wk` (wk.cap_cols).  At most one host synchronisation (blocked phase only).
inline int qrcp_device(double* f, int rows, int cols, double* tau, int* jpvt, QrWork& wk, cudaStream_t st, int nopivot = 0) {
    const int minmn = rows < cols ? rows : cols;
    if (minmn <= 0) return 0;
    if (cols > wk.cap_cols) return -1;
    // cluster size: the smallest of 2 / 4 / 8 CTAs whose shared memory holds the matrix with at most one column per warp
    // (a single round of the warp-per-column update), else 8; ENLSIP_QC_NC overrides it.  Measured (B200, 512 threads):
    // 256 x 64: 0.43 / 0.34 / 0.30 / 0.34 ms with 1 / 2 / 4 / 8 CTAs, 64 x 64: 0.34 / 0.29 / 0.26 / 0.27 ms -- a column step
    // costs 4-5 us whatever the cluster size: the dependent chain inside a step (reductions, IEEE divisions and square
    // roots of dlarfg and of the norm downdate), not the cluster barrier, sets the pace
    {
        static const int forced = [] { const char* e = getenv("ENLSIP_QC_NC"); return e ? atoi(e) : 0; }();
        int nc = 0;
        for (int c : {2, 4, 8})
            if (!nc && qc_smem_bytes(rows, cols, c) <= QC_MAX_SMEM && (cols + c - 1) / c <= QC_THREADS / 32) nc = c;
        if (!nc && qc_smem_bytes(rows, cols, 8) <= QC_MAX_SMEM) nc = 8;
        if (forced && qc_smem_bytes(rows, cols, forced) <= QC_MAX_SMEM) nc = forced;
        if (nc) {
            static bool attr_set = false;
            if (!attr_set) {
                cudaFuncSetAttribute(qr_cluster_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QC_MAX_SMEM);
                cudaFuncSetAttribute(qr_cluster_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QC_MAX_SMEM);
                cudaFuncSetAttribute(qr_cluster_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QC_MAX_SMEM);
                cudaFuncSetAttribute(qr_cluster_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QC_MAX_SMEM);
                attr_set = true;
            }
            const size_t shb = qc_smem_bytes(rows, cols, nc);
            if (nc == 1) qr_cluster_kernel<1><<<1, QC_THREADS, shb, st>>>(f, rows, cols, tau, jpvt, nopivot);
            else if (nc == 2) qr_cluster_kernel<2><<<2, QC_THREADS, shb, st>>>(f, rows, cols, tau, jpvt, nopivot);
            else if (nc == 4) qr_cluster_kernel<4><<<4, QC_THREADS, shb, st>>>(f, rows, cols, tau, jpvt, nopivot);
            else qr_cluster_kernel<8><<<8, QC_THREADS, shb, st>>>(f, rows, cols, tau, jpvt, nopivot);
            return 1;
        }
    }
    // dgeqp3: blocked (dlaqps) while j <= topbmn = minmn - nx, if nb < minmn and nx < minmn
    int topbmn = (QR_NB < minmn && QR_NX < minmn) ? (minmn - QR_NX) : 0;
    int launches = 0;
    cudaMemsetAsync(wk.flags, 0, sizeof(int) * cols, st);
    cudaMemsetAsync(wk.ticket, 0, sizeof(unsigned int) * QR_TICKET_LEN, st);
    qr_init_kernel<<<cols, 256, 0, st>>>(f, rows, cols, wk.vn1, wk.vn2, jpvt, wk.state, topbmn, nopivot);
    ++launches;
    if (topbmn > 0) {
        // A panel that stops early (a norm to recompute) re-opens at its next column, so more than ceil(topbmn / nb)
        // panels may be needed; each stopped panel still retires at least one column.  Enqueue the regular count plus a
        // margin, then (rarely) top up after looking at the state.
        const int per_panel = 3 * QR_NB + 3;
        cudaGraphExec_t exec = nullptr;
        const int G = qp_grid();
        const bool persist = G > 0 && qp_rows_per_slice(rows, G) <= QP_MAXRW;
        if (!persist && wk.use_graphs && st != nullptr) {
            for (QrGraph& g : wk.graphs)
                if (g.exec && g.f == f && g.rows == rows && g.cols == cols && g.tau == tau && g.jpvt == jpvt && g.topbmn == topbmn) exec = g.exec;
            if (!exec) {
                cudaGraph_t graph = nullptr;
                if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                    qr_enqueue_panel(f, rows, cols, tau, jpvt, wk, topbmn, st);
                    if (cudaStreamEndCapture(st, &graph) == cudaSuccess && graph &&
                        cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
                        QrGraph& slot = wk.graphs[wk.next_graph];
                        wk.next_graph = (wk.next_graph + 1) % 6;
                        if (slot.exec) cudaGraphExecDestroy(slot.exec);
                        slot.exec = exec; slot.f = f; slot.rows = rows; slot.cols = cols; slot.tau = tau; slot.jpvt = jpvt; slot.topbmn = topbmn;
                    } else {
                        exec = nullptr;
                    }
                    if (graph) cudaGraphDestroy(graph);
                }
                if (!exec) { cudaGetLastError(); wk.use_graphs = false; }
            }
        }
        int budget = (topbmn + QR_NB - 1) / QR_NB + 2;
        for (;;) {
            for (int pnl = 0; pnl < budget; ++pnl) {
                if (persist) launches += qr_enqueue_panel_persist(f, rows, cols, tau, jpvt, wk, topbmn, G, st);
                else if (exec) { cudaGraphLaunch(exec, st); launches += per_panel; }
                else launches += qr_enqueue_panel(f, rows, cols, tau, jpvt, wk, topbmn, st);
            }
            QrState h;
            cudaMemcpyAsync(&h, wk.state, sizeof(QrState), cudaMemcpyDeviceToHost, st);
            cudaStreamSynchronize(st);
            if (!h.active) break;
            budget = (topbmn - h.j0 + QR_NB - 1) / QR_NB + 2;
        }
    }
    for (int i = topbmn; i < minmn; ++i) {
        qr_p2_pivot_house_kernel<<<1, 1024, 0, st>>>(f, rows, cols, i, wk.vn1, wk.vn2, jpvt, tau, nopivot);
        ++launches;
        if (i < cols - 1) {
            const int len = rows - i - 1;
            int ncol = cols - i - 1;
            int grid = (ncol + 7) / 8;
            if (grid > 148 * 4) grid = 148 * 4;
            if (len <= VEC_STAGE_MAX)
                qr_p2_apply_kernel<true><<<grid, 256, sizeof(double) * (size_t)(len > 0 ? len : 1), st>>>(f, rows, cols, i, wk.vn1, wk.vn2, tau);
            else
                qr_p2_apply_kernel<false><<<grid, 256, 0, st>>>(f, rows, cols, i, wk.vn1, wk.vn2, tau);
            ++launches;
        }
    }
    return launches;
}

// =============================================================================================
// M <- M * Q,  Q = H(0) ... H(k-1) stored in f (frows x k, dgeqp3 layout) / tau : compact-WY panels of 32
// =============================================================================================
// explicit V of a panel: Vb (len x pw, ld = len) = rows j0.. of the columns j0..j0+pw of f with unit diagonal, zeros above
__global__ void wy_build_v_kernel(const double* __restrict__ f, int frows, int j0, int pw, double* __restrict__ Vb) {
    const int len = frows - j0;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)len * pw) return;
    const int r = (int)(e % len), c = (int)(e / len);
    Vb[e] = (r < c) ? 0.0 : (r == c ? 1.0 : f[(size_t)(j0 + c) * frows + j0 + r]);
}
// dlarft (forward, columnwise): T (pw x pw upper, ld = 32) from Vb and tau; one CTA.  The Gram matrix V'V is accumulated
// from 64-row slabs of Vb staged in shared memory (coalesced loads), thread (a, b) owns G(a, b).
__global__ void __launch_bounds__(1024) wy_build_t_kernel(const double* __restrict__ Vb, int len, int pw,
                                                          const double* __restrict__ tau, double* __restrict__ T) {
    __shared__ double Vs[64][33];
    __shared__ double G[32][33];
    __shared__ double Ts[32][33];
    __shared__ double tmp[32];
    const int a = threadIdx.x & 31, b = threadIdx.x >> 5;     // G(a, b) = V(:, a)' V(:, b), a < b
    double s = 0.0;
    for (int r0 = 0; r0 < len; r0 += 64) {
        __syncthreads();
        for (int e = threadIdx.x; e < 64 * 32; e += 1024) {
            const int rr = e & 63, c = e >> 6;
            Vs[rr][c] = (r0 + rr < len && c < pw) ? Vb[(size_t)c * len + r0 + rr] : 0.0;
        }
        __syncthreads();
        if (a < b)
#pragma unroll 8
            for (int rr = 0; rr < 64; ++rr) s = fma(Vs[rr][a], Vs[rr][b], s);
    }
    G[a][b] = s;
    Ts[a][b] = 0.0;
    __syncthreads();
    for (int i = 0; i < pw; ++i) {
        const double ti = tau[i];
        // T(0:i, i) = -tau_i * T(0:i, 0:i) * G(0:i, i)
        if (threadIdx.x < 32) {
            double acc = 0.0;
            if ((int)threadIdx.x < i)
                for (int c = threadIdx.x; c < i; ++c) acc = fma(Ts[threadIdx.x][c], G[c][i], acc);
            tmp[threadIdx.x] = -ti * acc;
        }
        __syncthreads();
        if ((int)threadIdx.x < i) Ts[threadIdx.x][i] = tmp[threadIdx.x];
        if (threadIdx.x == 0) Ts[i][i] = ti;
        __syncthreads();
    }
    T[b * 32 + a] = (a < pw && b < pw) ? Ts[a][b] : 0.0;    // column major, ld = 32
}

// ---- the T factors of ALL panels of a factorisation in two launches (dlarft, forward columnwise) ----
// wy_gram_kernel: grid (slabs of 256 rows, panels); gpart[(panel * nslab + slab) * 1024 + b * 32 + a] = the slab's share of
// V(:, a)' V(:, b) (a < b), V = the panel's reflectors read from f (unit diagonal, zeros above).
constexpr int WY_SLAB = 256;
__global__ void __launch_bounds__(1024) wy_gram_kernel(const double* __restrict__ f, int frows, int k, int p0,
                                                       double* __restrict__ gpart, int nslab) {
    __shared__ double Vs[128][33];
    const int panel = p0 + blockIdx.y, j0 = panel * 32;
    const int pw = (k - j0) < 32 ? (k - j0) : 32, len = frows - j0;
    const int a = threadIdx.x & 31, b = threadIdx.x >> 5;
    double s = 0.0;
    for (int half = 0; half < WY_SLAB / 128; ++half) {
        const int r0 = blockIdx.x * WY_SLAB + half * 128;
        __syncthreads();
        for (int e = threadIdx.x; e < 128 * 32; e += 1024) {
            const int rr = e & 127, c = e >> 7, r = r0 + rr;
            double v = 0.0;
            if (r < len && c < pw) v = (r < c) ? 0.0 : (r == c ? 1.0 : f[(size_t)(j0 + c) * frows + j0 + r]);
            Vs[rr][c] = v;
        }
        __syncthreads();
        if (a < b && r0 < len)
#pragma unroll 8
            for (int rr = 0; rr < 128; ++rr) s = fma(Vs[rr][a], Vs[rr][b], s);
    }
    gpart[((size_t)blockIdx.y * nslab + blockIdx.x) * 1024 + threadIdx.x] = s;
}
// wy_t_kernel: one CTA per panel; adds the slab shares in slab order, then T(0:i, i) = -tau_i T(0:i, 0:i) G(0:i, i)
__global__ void __launch_bounds__(1024) wy_t_kernel(const double* __restrict__ gpart, int nslab, int frows, int k, int p0,
                                                    const double* __restrict__ tau, double* __restrict__ Tall) {
    __shared__ double G[32][33];
    __shared__ double Ts[32][33];
    __shared__ double tmp[32];
    const int panel = p0 + blockIdx.x, j0 = panel * 32;
    const int pw = (k - j0) < 32 ? (k - j0) : 32, len = frows - j0;
    const int a = threadIdx.x & 31, b = threadIdx.x >> 5;
    const int ns = (len + WY_SLAB - 1) / WY_SLAB;
    double s = 0.0;
    const double* gp = gpart + (size_t)blockIdx.x * nslab * 1024 + threadIdx.x;
#pragma unroll 4
    for (int q = 0; q < ns; ++q) s += gp[(size_t)q * 1024];
    G[a][b] = s;
    Ts[a][b] = 0.0;
    __syncthreads();
    for (int i = 0; i < pw; ++i) {
        const double ti = tau[j0 + i];
        if (threadIdx.x < 32) {
            double acc = 0.0;
            if ((int)threadIdx.x < i)
                for (int c = threadIdx.x; c < i; ++c) acc = fma(Ts[threadIdx.x][c], G[c][i], acc);
            tmp[threadIdx.x] = -ti * acc;
        }
        __syncthreads();
        if ((int)threadIdx.x < i) Ts[threadIdx.x][i] = tmp[threadIdx.x];
        if (threadIdx.x == 0) Ts[i][i] = ti;
        __syncthreads();
    }
    Tall[(size_t)panel * 1024 + b * 32 + a] = (a < pw && b < pw) ? Ts[a][b] : 0.0;    // column major, ld = 32
}
// Tall: ceil(k / 32) x 1024 doubles; scratch: cap doubles (>= 1024 * ceil(frows / 256))
inline int wy_build_t_all(const double* f, int frows, int k, const double* tau, double* Tall, double* scratch, size_t cap,
                          cudaStream_t st) {
    const int np = (k + 31) / 32, nslab = (frows + WY_SLAB - 1) / WY_SLAB;
    int per = (int)(cap / ((size_t)nslab * 1024));
    if (per < 1) return -1;
    int launches = 0;
    for (int p0 = 0; p0 < np; p0 += per) {
        const int cnt = (np - p0) < per ? (np - p0) : per;
        wy_gram_kernel<<<dim3(nslab, cnt), 1024, 0, st>>>(f, frows, k, p0, scratch, nslab);
        wy_t_kernel<<<cnt, 1024, 0, st>>>(scratch, nslab, frows, k, p0, tau, Tall);
        launches += 2;
    }
    return launches;
}

struct WyWork { double *Vb = nullptr, *T = nullptr, *W = nullptr, *W2 = nullptr, *part = nullptr; };   // Vb: frows x 32, T: 32 x 32, W/W2: mr x 32, part: GEMM_MAX_SPLITS x mr x 32

// M: mr x nq column major (ld = mr); f: frows (= nq) x k
// Tall (optional): the T factors of all panels (wy_build_t_all) -- built here if `build_t`, reusable by reflect_vec_wy
inline int mulq_device(double* M, int mr, int nq, const double* f, int frows, int k, const double* tau, WyWork& wk,
                       cudaStream_t st, double* Tall = nullptr, bool build_t = true) {
    int launches = 0;
    if (Tall && build_t) {
        const int rc = wk.part ? wy_build_t_all(f, frows, k, tau, Tall, wk.part, (size_t)mr * 32 * GEMM_MAX_SPLITS, st) : -1;
        if (rc < 0) Tall = nullptr; else launches += rc;
    }
    for (int j0 = 0; j0 < k; j0 += 32) {
        const int pw = (k - j0) < 32 ? (k - j0) : 32;
        const int len = frows - j0;
        if (len <= 0) break;
        const long long ne = (long long)len * pw;
        wy_build_v_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(f, frows, j0, pw, wk.Vb);
        const double* Tp = wk.T;
        if (Tall) Tp = Tall + (size_t)(j0 / 32) * 1024;
        else { wy_build_t_kernel<<<1, 1024, 0, st>>>(wk.Vb, len, pw, tau + j0, wk.T); ++launches; }
        ++launches;
        // W = M(:, j0:) Vb ; W2 = W T ; M(:, j0:) -= W2 Vb'
        int splits = len / 256;                                   // W = M V: N = 32, K = len
        if (splits > GEMM_MAX_SPLITS) splits = GEMM_MAX_SPLITS;
        if (splits >= 2 && wk.part) {
            const int kc = ((len + splits - 1) / splits + 31) / 32 * 32;
            splits = (len + kc - 1) / kc;
            dim3 grid((mr + 63) / 64, splits);
            gemm_dmma_splitk_kernel<false><<<grid, 256, 0, st>>>(M + (size_t)j0 * mr, mr, wk.Vb, len, wk.part, mr, pw, len, kc);
            const long long mn = (long long)mr * pw;
            splitk_reduce_kernel<<<(unsigned)((mn + 255) / 256), 256, 0, st>>>(wk.part, splits, mn, 1.0, 0.0, wk.W, mr, mr);
            launches += 2;
        } else {
            launches += gemm<false>(M + (size_t)j0 * mr, mr, wk.Vb, len, wk.W, mr, mr, pw, len, 1.0, 0.0, st);
        }
        launches += gemm<false>(wk.W, mr, Tp, 32, wk.W2, mr, mr, pw, pw, 1.0, 0.0, st);
        launches += gemm<true>(wk.W2, mr, wk.Vb, len, M + (size_t)j0 * mr, mr, mr, len, pw, -1.0, 1.0, st);
    }
    return launches;
}

// =============================================================================================
// vectors: F.Q' v / F.Q v (reflector sweep), triangular solves, gemv, small glue
// =============================================================================================
// v (frows entries) <- Q' v (forward sweep, transpose = 1) or Q v (backward sweep); one CTA, v kept in shared memory
__global__ void __launch_bounds__(1024) reflect_vec_kernel(const double* __restrict__ f, int frows, int k,
                                                           const double* __restrict__ tau, double* __restrict__ v,
                                                           int transpose) {
    extern __shared__ double vsm[];
    __shared__ double sh[32];
    for (int r = threadIdx.x; r < frows; r += blockDim.x) vsm[r] = v[r];
    __syncthreads();
    for (int s = 0; s < k; ++s) {
        const int i = transpose ? s : (k - 1 - s);
        const double ti = tau[i];
        if (ti == 0.0) continue;
        const double* ci = f + (size_t)i * frows;
        double acc = 0.0;
        for (int r = i + 1 + threadIdx.x; r < frows; r += blockDim.x) acc = fma(ci[r], vsm[r], acc);
        acc = s_block_sum(acc, sh);
        const double w = (vsm[i] + acc) * ti;
        __syncthreads();
        for (int r = i + 1 + threadIdx.x; r < frows; r += blockDim.x) vsm[r] = fma(-w, ci[r], vsm[r]);
        if (threadIdx.x == 0) vsm[i] -= w;
        __syncthreads();
    }
    for (int r = threadIdx.x; r < frows; r += blockDim.x) v[r] = vsm[r];
}

// the same sweep by ONE warp (no block barrier): vectors of a few hundred entries, where 32 warps only wait for each other
__global__ void __launch_bounds__(32) reflect_vec_warp_kernel(const double* __restrict__ f, int frows, int k,
                                                              const double* __restrict__ tau, double* __restrict__ v,
                                                              int transpose) {
    extern __shared__ double vsm[];
    const int lane = threadIdx.x;
    for (int r = lane; r < frows; r += 32) vsm[r] = v[r];
    __syncwarp();
    for (int s = 0; s < k; ++s) {
        const int i = transpose ? s : (k - 1 - s);
        const double ti = tau[i];
        if (ti == 0.0) continue;
        const double* ci = f + (size_t)i * frows;
        double acc = 0.0;
        for (int r = i + 1 + lane; r < frows; r += 32) acc = fma(ci[r], vsm[r], acc);
        acc = s_warp_sum(acc);
        const double w = (vsm[i] + acc) * ti;
        __syncwarp();
        for (int r = i + 1 + lane; r < frows; r += 32) vsm[r] = fma(-w, ci[r], vsm[r]);
        if (lane == 0) vsm[i] -= w;
        __syncwarp();
    }
    for (int r = lane; r < frows; r += 32) v[r] = vsm[r];
}
// triangular solves by one warp, column oriented (k of a few hundred): x_i = x_i / R_ii, then the remaining entries
__global__ void __launch_bounds__(32) trsv_upper_warp_kernel(const double* __restrict__ f, int ldf, int k, double* __restrict__ x) {
    extern __shared__ double xs[];
    const int lane = threadIdx.x;
    for (int r = lane; r < k; r += 32) xs[r] = x[r];
    __syncwarp();
    for (int i = k - 1; i >= 0; --i) {
        const double* ci = f + (size_t)i * ldf;
        const double xi = xs[i] / ci[i];
        __syncwarp();
        for (int r = lane; r < i; r += 32) xs[r] = fma(-ci[r], xi, xs[r]);
        if (lane == 0) xs[i] = xi;
        __syncwarp();
    }
    for (int r = lane; r < k; r += 32) x[r] = xs[r];
}
__global__ void __launch_bounds__(32) trsv_upperT_warp_kernel(const double* __restrict__ f, int ldf, int k, double* __restrict__ x) {
    extern __shared__ double xs[];
    const int lane = threadIdx.x;
    for (int r = lane; r < k; r += 32) xs[r] = x[r];
    __syncwarp();
    for (int i = 0; i < k; ++i) {
        const double* ci = f + (size_t)i * ldf;
        double s = 0.0;
        for (int r = lane; r < i; r += 32) s = fma(ci[r], xs[r], s);
        s = s_warp_sum(s);
        __syncwarp();
        if (lane == 0) xs[i] = (xs[i] - s) / ci[i];
        __syncwarp();
    }
    for (int r = lane; r < k; r += 32) x[r] = xs[r];
}
// ---- v <- Q' v / Q v with the compact-WY panels (dormqr's blocked form), ONE cooperative kernel ----
// CTA c keeps rows [c rw, (c+1) rw) of v in shared memory for the whole sweep.  Per panel (32 reflectors): the slice
// of V goes to shared memory, the CTA leaves its share of w = V' v (32 numbers), ONE grid barrier, every CTA adds the
// shares in CTA order, forms z = T' w (Q') or T w (Q) and updates its rows v -= V z.  T comes from wy_build_t_all.
constexpr int RW_THREADS = 256, RW_ROWS = 128, RW_MAXG = 148;
constexpr int RW_WPART_LEN = 2 * RW_MAXG * 32;      // doubles of the wpart scratch
__global__ void __launch_bounds__(RW_THREADS, 1)
reflect_vec_wy_kernel(const double* __restrict__ f, int frows, int k, const double* __restrict__ Tall, double* v,
                      int transpose, double* wpart, unsigned int* bar) {
    extern __shared__ double rw_dyn[];
    __shared__ double Ts[32][33];
    __shared__ double s_w[32], s_z[32];
    const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int rw = ((frows + G - 1) / G + 31) / 32 * 32;
    const int r0 = c * rw, nr = (frows - r0) < rw ? (frows - r0 > 0 ? frows - r0 : 0) : rw;
    double* vs = rw_dyn;                         // [rw]
    double* Vs = rw_dyn + rw;                    // [rw][33]
    for (int rl = tid; rl < nr; rl += RW_THREADS) vs[rl] = v[r0 + rl];
    const int np = (k + 31) / 32;
    unsigned int epoch = 0;
    for (int sp = 0; sp < np; ++sp) {
        const int p = transpose ? sp : (np - 1 - sp), j0 = p * 32;
        const int pw = (k - j0) < 32 ? (k - j0) : 32;
        // the shares are double-buffered: a CTA can be at most one barrier ahead of the slowest reader
        double* wbuf = wpart + (size_t)(sp & 1) * RW_MAXG * 32;
        __syncthreads();
        // slice of V (unit diagonal, zeros above) and T of the panel
        for (int e = tid; e < rw * 32; e += RW_THREADS) {
            const int rl = e % rw, cc = e / rw, r = r0 + rl, d = j0 + cc;
            double x = 0.0;
            if (rl < nr && cc < pw) x = (r < d) ? 0.0 : (r == d ? 1.0 : f[(size_t)d * frows + r]);
            Vs[rl * 33 + cc] = x;
        }
        for (int e = tid; e < 1024; e += RW_THREADS) Ts[e & 31][e >> 5] = Tall[(size_t)p * 1024 + e];   // Ts[a][b] = T(a, b)
        __syncthreads();
        // share of w_cc = sum_r V(r, cc) v(r): warp per 4 columns, lanes over the rows
        for (int cc = w; cc < 32; cc += RW_THREADS / 32) {
            double t = 0.0;
            for (int rl = lane; rl < nr; rl += 32) t = fma(Vs[rl * 33 + cc], vs[rl], t);
            t = s_warp_sum(t);
            if (lane == 0) wbuf[(size_t)c * 32 + cc] = t;
        }
        qp_grid_barrier(bar, epoch);
        {
            // 8 threads per column; all loads of a thread in flight together, sums in a fixed order
            constexpr int NU = (RW_MAXG + 7) / 8;
            const int cc = tid >> 3, sub = tid & 7;
            double part[NU];
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                const int q = sub + 8 * u;
                part[u] = (q < G) ? __ldcg(wbuf + (size_t)q * 32 + cc) : 0.0;
            }
            double t = 0.0;
#pragma unroll
            for (int u = 0; u < NU; ++u) t += part[u];
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (sub == 0) s_w[cc] = t;
        }
        __syncthreads();
        if (tid < 32) {
            double z = 0.0;
            if (transpose) { for (int j = 0; j <= tid; ++j) z = fma(Ts[j][tid], s_w[j], z); }      // (T' w)_c
            else { for (int j = tid; j < 32; ++j) z = fma(Ts[tid][j], s_w[j], z); }                // (T w)_c
            s_z[tid] = z;
        }
        __syncthreads();
        for (int rl = tid; rl < nr; rl += RW_THREADS) {
            double t = 0.0;
#pragma unroll 8
            for (int cc = 0; cc < 32; ++cc) t = fma(Vs[rl * 33 + cc], s_z[cc], t);
            vs[rl] -= t;
        }
    }
    __syncthreads();
    for (int rl = tid; rl < nr; rl += RW_THREADS) v[r0 + rl] = vs[rl];
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(bar + 1, 1u) == (unsigned int)G - 1) { bar[2] = 0; bar[1] = 0; __threadfence(); }
    }
}
inline int rw_grid(int frows) {
    int g = (frows + RW_ROWS - 1) / RW_ROWS;
    return g < 1 ? 1 : (g > RW_MAXG ? RW_MAXG : g);
}
inline size_t rw_smem_bytes(int frows, int G) {
    const int rw = ((frows + G - 1) / G + 31) / 32 * 32;
    return sizeof(double) * (size_t)rw * 34;
}
// returns the number of launches, or -1 when the shape does not fit (caller falls back to the reflector sweep)
inline int reflect_vec_wy(const double* f, int frows, int k, const double* Tall, double* v, int transpose, double* wpart,
                          unsigned int* bar, cudaStream_t st) {
    const int G = rw_grid(frows);
    const size_t shb = rw_smem_bytes(frows, G);
    if (shb > 200 * 1024) return -1;
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(reflect_vec_wy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    void* args[] = {&f, &frows, &k, &Tall, &v, &transpose, &wpart, &bar};
    if (cudaLaunchCooperativeKernel((const void*)reflect_vec_wy_kernel, dim3(G), dim3(RW_THREADS), args, shb, st) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return 1;
}

// ---- triangular solves over many CTAs: one WARP per diagonal block of 32, blocks solved in sequence, a solved block is
// announced through a counter (release / acquire) and every warp folds it into its own rows while the next block is
// being solved.  The arithmetic (order of every sum) is that of trsv_upper_kernel / trsv_upperT_kernel below. ----
__device__ __forceinline__ void ts_wait(const unsigned int* flag, unsigned int need, int lane) {
    if (lane == 0) while (qp_ld_acquire(flag) < need) { }
    __syncwarp();
}
__device__ __forceinline__ void ts_post(unsigned int* flag, unsigned int val, int lane) {
    __threadfence();
    __syncwarp();
    if (lane == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(flag), "r"(val) : "memory");
}
// x <- UpperTriangular(f[0:k, 0:k]) \ x.  Blocks are aligned to the bottom (block t = rows [k - 32 (t+1), k - 32 t)).
__global__ void trsv_upper_coop_kernel(const double* __restrict__ f, int ldf, int k, double* x, int bpc, unsigned int* bar) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nblk = (k + 31) / 32, t = blockIdx.x * bpc + w;
    unsigned int* solved = bar + 3;
    if (t < nblk && w < bpc) {
        const int b1 = k - 32 * t, b0 = (b1 - 32 > 0) ? b1 - 32 : 0, nb = b1 - b0;
        const int r = b0 + lane;
        const bool live = lane < nb;
        double xr = live ? x[r] : 0.0;
        double Rv[32];
        for (int s = 0; s < t; ++s) {                   // fold in the blocks below, in the order they are solved
            const int cb0 = k - 32 * (s + 1);
#pragma unroll
            for (int cc = 0; cc < 32; ++cc) Rv[cc] = live ? f[(size_t)(cb0 + cc) * ldf + r] : 0.0;   // in flight while waiting
            ts_wait(solved, (unsigned int)(s + 1), lane);
            const double xb = __ldcg(x + cb0 + lane);
            double sum = 0.0;
#pragma unroll
            for (int cc = 0; cc < 32; ++cc) sum = fma(Rv[cc], __shfl_sync(0xffffffffu, xb, cc), sum);
            xr -= sum;
        }
        // back substitution inside the block: lane = row, Rv[cc] = R(b0 + lane, b0 + cc)
#pragma unroll
        for (int cc = 0; cc < 32; ++cc) Rv[cc] = (live && cc < nb) ? f[(size_t)(b0 + cc) * ldf + r] : 1.0;
#pragma unroll
        for (int i = 31; i >= 0; --i) {
            if (i < nb) {
                const double xi = __shfl_sync(0xffffffffu, xr / Rv[i], i);      // lane i: x_i / R(i, i)
                if (lane == i) xr = xi;
                else if (lane < i) xr = fma(-Rv[i], xi, xr);
            }
        }
        if (live) x[r] = xr;
        ts_post(solved, (unsigned int)(t + 1), lane);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(bar + 1, 1u) == gridDim.x - 1) { bar[3] = 0; bar[1] = 0; __threadfence(); }
    }
}
// x <- LowerTriangular(f[0:k, 0:k]') \ x (forward).  Blocks from the top (block t = [32 t, min(32 t + 32, k))).
__global__ void trsv_upperT_coop_kernel(const double* __restrict__ f, int ldf, int k, double* x, int bpc, unsigned int* bar) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nblk = (k + 31) / 32, t = blockIdx.x * bpc + w;
    unsigned int* solved = bar + 3;
    if (t < nblk && w < bpc) {
        const int b0 = 32 * t, b1 = (b0 + 32 < k) ? b0 + 32 : k, nb = b1 - b0;
        double acc[32], Rv[32];
#pragma unroll
        for (int cc = 0; cc < 32; ++cc) acc[cc] = 0.0;
        for (int s = 0; s < t; ++s) {                   // rows of block s: lane = row, one accumulator per column of this block
            const int rr = 32 * s + lane;
#pragma unroll
            for (int cc = 0; cc < 32; ++cc) Rv[cc] = (cc < nb) ? f[(size_t)(b0 + cc) * ldf + rr] : 0.0;
            ts_wait(solved, (unsigned int)(s + 1), lane);
            const double xr = __ldcg(x + rr);
#pragma unroll
            for (int cc = 0; cc < 32; ++cc) acc[cc] = fma(Rv[cc], xr, acc[cc]);
        }
        // column sums over the lanes (the pairing of s_warp_sum), lane cc ends with the sum of column cc
#pragma unroll
        for (int h = 16; h > 0; h >>= 1) {
            const bool up = (lane & h) != 0;
#pragma unroll
            for (int q = 0; q < h; ++q) {
                const double keep = up ? acc[q + h] : acc[q];
                const double send = up ? acc[q] : acc[q + h];
                acc[q] = keep + __shfl_xor_sync(0xffffffffu, send, h);
            }
        }
        const bool live = lane < nb;
        double xc = live ? (x[b0 + lane] - acc[0]) : 0.0;
        // forward recurrence inside the block: lane = column c, Rv[ii] = R(b0 + ii, b0 + c)
#pragma unroll
        for (int ii = 0; ii < 32; ++ii) Rv[ii] = (live && ii < nb) ? f[(size_t)(b0 + lane) * ldf + b0 + ii] : 1.0;
#pragma unroll
        for (int ii = 0; ii < 32; ++ii) {
            if (ii < nb) {
                const double xi = __shfl_sync(0xffffffffu, xc / Rv[ii], ii);    // lane ii: x_ii / R(ii, ii)
                if (lane == ii) xc = xi;
                else if (lane > ii) xc = fma(-Rv[ii], xi, xc);
            }
        }
        if (live) x[b0 + lane] = xc;
        ts_post(solved, (unsigned int)(t + 1), lane);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(bar + 1, 1u) == gridDim.x - 1) { bar[3] = 0; bar[1] = 0; __threadfence(); }
    }
}
// returns 1 (launched) or -1 (shape does not fit / launch refused: caller falls back)
inline int trsv_coop(const double* f, int ldf, int k, double* x, bool transposed, unsigned int* bar, cudaStream_t st) {
    const int nblk = (k + 31) / 32;
    int G = nblk < 148 ? nblk : 148;
    int bpc = (nblk + G - 1) / G;
    if (bpc > 8) return -1;                    // k > 37888
    G = (nblk + bpc - 1) / bpc;
    void* args[] = {&f, &ldf, &k, &x, &bpc, &bar};
    const void* fn = transposed ? (const void*)trsv_upperT_coop_kernel : (const void*)trsv_upper_coop_kernel;
    if (cudaLaunchCooperativeKernel(fn, dim3(G), dim3(32 * bpc), args, 0, st) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return 1;
}

constexpr int VEC_WARP_MAX = 640;     // up to this many entries the one-warp kernels are used

// x (k entries) <- UpperTriangular(f[0:k, 0:k]) \ x ; one CTA of 1024 threads, blocks of 32 from the bottom
__global__ void __launch_bounds__(1024) trsv_upper_kernel(const double* __restrict__ f, int ldf, int k, double* __restrict__ x) {
    extern __shared__ double xs[];
    for (int r = threadIdx.x; r < k; r += blockDim.x) xs[r] = x[r];
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int b1 = k; b1 > 0; b1 -= 32) {
        const int b0 = b1 - 32 > 0 ? b1 - 32 : 0;
        if (w == 0) {                                  // back substitution inside the diagonal block (one warp)
            for (int i = b1 - 1; i >= b0; --i) {
                const double xi = xs[i] / f[(size_t)i * ldf + i];
                __syncwarp();
                if (lane == 0) xs[i] = xi;
                const int r = b0 + lane;
                if (r < i) xs[r] = fma(-f[(size_t)i * ldf + r], xi, xs[r]);
                __syncwarp();
            }
        }
        __syncthreads();
        // rows above the block: x_r -= sum_{c in block} R(r, c) x_c
        for (int r = threadIdx.x; r < b0; r += blockDim.x) {
            double s = 0.0;
            for (int c = b0; c < b1; ++c) s = fma(f[(size_t)c * ldf + r], xs[c], s);
            xs[r] -= s;
        }
        __syncthreads();
    }
    for (int r = threadIdx.x; r < k; r += blockDim.x) x[r] = xs[r];
}

// x (k entries) <- LowerTriangular(f[0:k, 0:k]') \ x ; forward, blocks of 32: one warp per column of the block for the
// part of the dot product that lies above the block, one warp for the in-block recurrence
__global__ void __launch_bounds__(1024) trsv_upperT_kernel(const double* __restrict__ f, int ldf, int k, double* __restrict__ x) {
    extern __shared__ double xs[];
    for (int r = threadIdx.x; r < k; r += blockDim.x) xs[r] = x[r];
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int b0 = 0; b0 < k; b0 += 32) {
        const int b1 = b0 + 32 < k ? b0 + 32 : k;
        const int i = b0 + w;
        if (i < b1) {
            const double* ci = f + (size_t)i * ldf;
            double s = 0.0;
            for (int r = lane; r < b0; r += 32) s = fma(ci[r], xs[r], s);
            s = s_warp_sum(s);
            if (lane == 0) xs[i] -= s;
        }
        __syncthreads();
        if (w == 0) {
            for (int ii = b0; ii < b1; ++ii) {
                const double xi = xs[ii] / f[(size_t)ii * ldf + ii];
                __syncwarp();
                if (lane == 0) xs[ii] = xi;
                const int c = ii + 1 + lane;           // later columns of the block: x_c -= R(ii, c) x_ii
                if (c < b1) xs[c] = fma(-f[(size_t)c * ldf + ii], xi, xs[c]);
                __syncwarp();
            }
        }
        __syncthreads();
    }
    for (int r = threadIdx.x; r < k; r += blockDim.x) x[r] = xs[r];
}

// ---- the size selection of the vector operations (the solver's small stage and the known-answer hook use these) ----
// v (frows entries) <- Q' v (transpose = 1) / Q v: one warp up to VEC_WARP_MAX entries, else the compact-WY cooperative
// kernel with the T factors t_of() returns (nullptr: none), else one CTA.  Returns the launches (t_of()'s not included).
template <class TOf>
inline int reflect_vec(const double* f, int frows, int k, const double* tau, double* v, int transpose, TOf&& t_of,
                       double* wpart, unsigned int* bar, cudaStream_t st) {
    if (frows <= 0 || k <= 0) return 0;
    if (frows <= VEC_WARP_MAX) {
        reflect_vec_warp_kernel<<<1, 32, sizeof(double) * (size_t)frows, st>>>(f, frows, k, tau, v, transpose);
        return 1;
    }
    if (const double* T = t_of()) {
        const int rc = reflect_vec_wy(f, frows, k, T, v, transpose, wpart, bar, st);
        if (rc > 0) return rc;
    }
    reflect_vec_kernel<<<1, 1024, sizeof(double) * (size_t)frows, st>>>(f, frows, k, tau, v, transpose);
    return 1;
}
inline int trsv_coop_min() {     // smallest triangle solved by the multi-CTA kernels (ENLSIP_TRSV_COOP_MIN overrides)
    static const int v = [] { const char* e = getenv("ENLSIP_TRSV_COOP_MIN"); return e ? atoi(e) : 320; }();
    return v;
}
// x (k entries) <- R \ x (transposed: R' \ x), R = UpperTriangular(f[0:k, 0:k]): the cooperative kernels from
// trsv_coop_min() entries, else one warp up to VEC_WARP_MAX, else one CTA.  Returns the number of launches.
inline int trsv_upper(const double* f, int ldf, int k, double* x, bool transposed, unsigned int* bar, cudaStream_t st) {
    if (k <= 0) return 0;
    if (k >= trsv_coop_min() && trsv_coop(f, ldf, k, x, transposed, bar, st) > 0) return 1;
    const size_t shb = sizeof(double) * (size_t)k;
    if (k <= VEC_WARP_MAX) {
        if (transposed) trsv_upperT_warp_kernel<<<1, 32, shb, st>>>(f, ldf, k, x);
        else trsv_upper_warp_kernel<<<1, 32, shb, st>>>(f, ldf, k, x);
    } else if (transposed) {
        trsv_upperT_kernel<<<1, 1024, shb, st>>>(f, ldf, k, x);
    } else {
        trsv_upper_kernel<<<1, 1024, shb, st>>>(f, ldf, k, x);
    }
    return 1;
}

// y (rows) = alpha * A (rows x cols, lda) x + beta * y0   (y0 may be nullptr = 0); thread per row, columns streamed.
// STAGED: x is first copied to shared memory (cols <= VEC_STAGE_MAX), otherwise read from global memory; same sums.
template <bool STAGED>
__global__ void __launch_bounds__(256) gemv_n_kernel(const double* __restrict__ A, int lda, int rows, int cols,
                                                     const double* __restrict__ x, double alpha, const double* __restrict__ y0,
                                                     double beta, double* __restrict__ y) {
    extern __shared__ double xsm[];
    if (STAGED) {
        for (int c = threadIdx.x; c < cols; c += blockDim.x) xsm[c] = x[c];
        __syncthreads();
    }
    const double* xs = STAGED ? xsm : x;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int c = 0;
    for (; c + 4 <= cols; c += 4) {
        s0 = fma(A[(size_t)c * lda + r], xs[c], s0);
        s1 = fma(A[(size_t)(c + 1) * lda + r], xs[c + 1], s1);
        s2 = fma(A[(size_t)(c + 2) * lda + r], xs[c + 2], s2);
        s3 = fma(A[(size_t)(c + 3) * lda + r], xs[c + 3], s3);
    }
    for (; c < cols; ++c) s0 = fma(A[(size_t)c * lda + r], xs[c], s0);
    const double s = (s0 + s1) + (s2 + s3);
    y[r] = alpha * s + (y0 ? beta * y0[r] : 0.0);
}
// the same for short matrices (rows of a few hundred): CTA = 32 rows (lane = row), its 8 warps split the columns and
// their partial sums are added in warp order -- 8x the parallelism of a thread per row
__global__ void __launch_bounds__(256) gemv_n_split_kernel(const double* __restrict__ A, int lda, int rows, int cols,
                                                           const double* __restrict__ x, double alpha,
                                                           const double* __restrict__ y0, double beta, double* __restrict__ y) {
    __shared__ double part[8][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int r = blockIdx.x * 32 + lane;
    const int per = (cols + 7) / 8, c0 = w * per, c1 = (c0 + per < cols) ? c0 + per : cols;
    double s0 = 0.0, s1 = 0.0;
    if (r < rows) {
        int c = c0;
        for (; c + 2 <= c1; c += 2) {
            s0 = fma(A[(size_t)c * lda + r], x[c], s0);
            s1 = fma(A[(size_t)(c + 1) * lda + r], x[c + 1], s1);
        }
        if (c < c1) s0 = fma(A[(size_t)c * lda + r], x[c], s0);
    }
    part[w][lane] = s0 + s1;
    __syncthreads();
    if (w == 0 && r < rows) {
        double s = 0.0;
        for (int q = 0; q < 8; ++q) s += part[q][lane];
        y[r] = alpha * s + (y0 ? beta * y0[r] : 0.0);
    }
}
// y (cols) = A' x : one warp per column
__global__ void __launch_bounds__(256) gemv_t_kernel(const double* __restrict__ A, int lda, int rows, int cols,
                                                     const double* __restrict__ x, double* __restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int c = gw; c < cols; c += nwarps) {
        const double* cc = A + (size_t)c * lda;
        double s = 0.0;
        for (int r = lane; r < rows; r += 32) s = fma(cc[r], x[r], s);
        s = s_warp_sum(s);
        if (lane == 0) y[c] = s;
    }
}
inline int gemv_n(const double* A, int lda, int rows, int cols, const double* x, double alpha, const double* y0, double beta,
                  double* y, cudaStream_t st) {
    if (rows <= 0) return 0;
    if (rows <= 2048) gemv_n_split_kernel<<<(rows + 31) / 32, 256, 0, st>>>(A, lda, rows, cols, x, alpha, y0, beta, y);
    else if (cols <= VEC_STAGE_MAX)
        gemv_n_kernel<true><<<(rows + 255) / 256, 256, sizeof(double) * (size_t)(cols > 0 ? cols : 1), st>>>(A, lda, rows, cols, x, alpha, y0, beta, y);
    else gemv_n_kernel<false><<<(rows + 255) / 256, 256, 0, st>>>(A, lda, rows, cols, x, alpha, y0, beta, y);
    return 1;
}
inline int gemv_t(const double* A, int lda, int rows, int cols, const double* x, double* y, cudaStream_t st) {
    if (cols <= 0) return 0;
    int grid = (cols + 7) / 8;
    if (grid > 148 * 8) grid = 148 * 8;
    gemv_t_kernel<<<grid, 256, 0, st>>>(A, lda, rows, cols, x, y);
    return 1;
}

// out[0] = ||v[lo:hi)||  (one CTA)
__global__ void __launch_bounds__(1024) norm_range_kernel(const double* __restrict__ v, int lo, int hi, double* out) {
    __shared__ double sh[32];
    double s = 0.0;
    for (int r = lo + threadIdx.x; r < hi; r += blockDim.x) s = fma(v[r], v[r], s);
    s = s_block_sum(s, sh);
    if (threadIdx.x == 0) out[0] = sqrt(s);
}
// dst[i] = i < k ? src[i] : 0,  i < len
__global__ void copy_pad_kernel(double* dst, const double* src, int k, int len) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) dst[i] = (i < k) ? src[i] : 0.0;
}
// dst[i] = (idx[i] < k) ? src[idx[i]] : 0,  i < len      (x[invperm][..] of a zero-padded vector)
__global__ void gather_pad_kernel(double* dst, const double* src, const int* idx, int k, int len) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) { const int j = idx[i]; dst[i] = (j < k) ? src[j] : 0.0; }
}
// p1 = P[0:ra, 0:ra] * [dp1 (k entries); 0] : p1[perm[j]] = dp1[j] for j < k, perm[j] < ra   (dst pre-zeroed)
__global__ void scatter_perm_kernel(double* dst, const double* src, const int* perm, int k, int ra) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < k && j < ra) { const int r = perm[j]; if (r < ra) dst[r] = src[j]; }
}
// ---- rows of A (row-major l x n = column-major n x l) ----
__global__ void __launch_bounds__(256) gather_rows_kernel(const double* __restrict__ Arow, int n, const int* __restrict__ active,
                                                          double* __restrict__ CA) {
    const double* src = Arow + (size_t)(active[blockIdx.x] - 1) * n;
    double* dst = CA + (size_t)blockIdx.x * n;
    for (int c = threadIdx.x; c < n; c += blockDim.x) dst[c] = src[c];
}
__global__ void __launch_bounds__(256) row_norm_scale_kernel(double* __restrict__ CA, int n, int scaling, double* __restrict__ rown) {
    __shared__ double sh[32];
    double* row = CA + (size_t)blockIdx.x * n;
    double s = 0.0;
    for (int c = threadIdx.x; c < n; c += blockDim.x) s = fma(row[c], row[c], s);
    s = s_block_sum(s, sh);
    double nr = sqrt(s);
    if (threadIdx.x == 0) rown[blockIdx.x] = nr;
    if (scaling) {
        if (fabs(nr) < 2.220446049250313e-16) nr = 1.0;
        for (int c = threadIdx.x; c < n; c += blockDim.x) row[c] = row[c] / nr;
    }
}
__global__ void __launch_bounds__(256) rebuild_scaled_rows_kernel(const double* __restrict__ Arow, int n,
                                                                  const int* __restrict__ active, const double* __restrict__ ds,
                                                                  double* __restrict__ CA) {
    const double* src = Arow + (size_t)(active[blockIdx.x] - 1) * n;
    double* dst = CA + (size_t)blockIdx.x * n;
    const double d = ds[blockIdx.x];
    for (int c = threadIdx.x; c < n; c += blockDim.x) dst[c] = src[c] * d;
}
// Rt (t x kr, ld = t): Rt(c, r) = R_A(r, c), R_A = upper triangle of FA (ld = n)
__global__ void build_rt_kernel(const double* __restrict__ FA, int n, int t, int kr, double* __restrict__ Rt) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)t * kr) return;
    const int c = (int)(e % t), r = (int)(e / t);
    Rt[e] = (r <= c) ? FA[(size_t)c * n + r] : 0.0;
}

}  // namespace enl_small
