// enl_tsqr.cuh -- tall-skinny Householder QR (R factor only) of a row-major FP64 matrix on sm_100a.
//
// Replaces, for the large-Jacobian regime, the reference's `qr(J2, ColumnNorm())` + `F.Q' * v` on the
// m x n residual Jacobian (src/enlsip_functions.jl:219-223, 135-151): the engine reduces the augmented
// matrix [J | r] (m x (n+1), m ~ 4e6) to its (n+1) x (n+1) triangular factor and runs the pivoted
// small-matrix stage on that (pivot choices are invariant under the left orthogonal transform).
//
// Algorithm: communication-avoiding blocked Householder QR, panel width 32.
//   for each 32-column panel j:
//     level 0, 1, 2, ...: the rows are cut into blocks of 32; a "subtile" is 8 blocks (stride 8^level
//       blocks apart, i.e. at level >= 1 the top blocks of the subtiles of the level below).
//       tsqr_panel_cg_kernel     : one CTA per subtile; Householder QR of its 256 x 32 panel held in
//                                  registers (warp w = columns 4w..4w+3 of all 256 rows), ONE block barrier per
//                                  column; compact-WY T = (striu(V'V) + diag(1/tau))^-1; V is stored in place, T
//                                  in a side buffer; the residual column of [J | r] is updated here as well
//                                  (b <- (I - V T' V') b with the reflectors still in registers)
//       tsqr_trail_staged_kernel : one CTA per (subtile, chunk of 32-column blocks of the trailing matrix):
//                                  B <- (I - V T' V')B with three FP64 tensor-core products
//                                  (mma.sync.m8n8k4.f64 = DMMA.8x8x4): G = V'B, W = -T'G, B += V W
//     the top 32 rows of the last level are the finished rows 32j..32j+31 of R: copied out, then
//     zeroed in place so later panels see them as empty rows.
//   after the last panel the residual column only needs its norm (R[n][n]).
// Every subtile is independent inside a level, so each kernel is a plain grid over subtiles; the
// price is 1/7 more flops than a flat tree (each level re-factors 1/8 of the rows).
// Algorithmic flops: 2 m n^2 (n = number of columns).  See DESIGN.md for the roofline accounting.
#pragma once
#include <cuda_runtime.h>

namespace enl_large {

constexpr int TS_B = 32;     // block rows = panel width
constexpr int TS_FAN = 8;    // blocks per subtile

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------
// panel factorisation of one subtile: warp w owns columns 4w..4w+3 of all 256 rows of the subtile
// ---------------------------------------------------------------------------------------------
// Lane l of warp w holds columns 4w..4w+3 of the rows 32 r + l (r = 0..7: one row of every 32-row block of the subtile).
// One block barrier per column i:
//   * the scalar chain of the column (norm, rsqrt, reciprocal -- dlarfg) runs in ONE warp, the owner of the column,
//     which publishes the raw column u_i (the entries below the pivot) together with tau and scale;
//   * every warp then takes ONE pass of dot products g_c = u_i . a_c with its columns.  The reflector
//     v_i = e_i + scale * u_i is linear in the raw column, so v_i . a_c = a_c[i] + scale * g_c: live columns (c > i)
//     are updated with it, finished ones (c < i) give v_c . v_i, the Gram matrix of V that the T factor needs;
//   * a finished column group costs its warp only those 32 dot products: no update, and none of the scalar chain;
//   * every dot product is reduced inside a warp (shuffles), there is no cross-warp reduction; the pivot-row entry of
//     a column is fetched from the owning lane by one shuffle.
// Finished columns keep their reflector UNSCALED in registers (u_c, v_c = e_c + scale_c u_c): scaling happens once, when
// the panel is stored.  Top block: rows <= i are masked out of the published column, so the finished rows of R simply
// stay where they are.  The residual column of [J | r] (column rcol) is updated at the end with the block reflector of
// the panel, so the trailing-update kernel only sees full 32-column blocks.
__device__ __forceinline__ double warp_allsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// sums over the warp of 4 values per lane; every lane receives the 4 totals (fixed order: 10 shuffles instead of 20)
__device__ __forceinline__ void warp_allsum4(const double (&d)[4], double (&g)[4], int lane) {
    const bool hi = (lane & 16) != 0, h8 = (lane & 8) != 0;
    const double x = (hi ? d[2] : d[0]) + __shfl_xor_sync(0xffffffffu, hi ? d[0] : d[2], 16);
    const double y = (hi ? d[3] : d[1]) + __shfl_xor_sync(0xffffffffu, hi ? d[1] : d[3], 16);
    double z = (h8 ? y : x) + __shfl_xor_sync(0xffffffffu, h8 ? x : y, 8);   // column 2 hi + h8
    z += __shfl_xor_sync(0xffffffffu, z, 4);
    z += __shfl_xor_sync(0xffffffffu, z, 2);
    z += __shfl_xor_sync(0xffffffffu, z, 1);
#pragma unroll
    for (int c = 0; c < 4; ++c) g[c] = __shfl_sync(0xffffffffu, z, 16 * (c >> 1) + 8 * (c & 1));
}

__global__ void __launch_bounds__(256, 2)
tsqr_panel_cg_kernel(double* __restrict__ A, int ld, long long nblk, long long stride, int col0, int upper_only,
                     int rcol, double* __restrict__ Tbuf) {
    __shared__ double vbuf[2][TS_FAN][TS_B];   // published raw pivot column (rows <= i of the top block masked)
    __shared__ double sc[2][2];                // tau, scale of the published column
    __shared__ double Gs[TS_B][TS_B + 1];      // Gs[c][i] = v_c . v_i, c < i
    __shared__ double taus[TS_B];
    __shared__ double bsh[TS_FAN][TS_B];       // residual column of the subtile
    __shared__ double gb[TS_B], wb[TS_B];
    __shared__ double part[TS_FAN][TS_FAN][TS_B];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long sub = blockIdx.x;
    double a[4][TS_FAN];
    double ms[4] = {0.0, 0.0, 0.0, 0.0};
    // residual column: thread (w, lane) <-> row lane of block w
    const long long bblk = (sub * TS_FAN + w) * stride;
    double* bptr = A + (bblk * TS_B + lane) * (long long)ld + rcol;
    const bool bvalid = bblk < nblk;
    const double bval = (bvalid && rcol >= 0) ? *bptr : 0.0;
#pragma unroll
    for (int r = 0; r < TS_FAN; ++r) {
        const long long blk = (sub * TS_FAN + r) * stride;
        double2 v01 = make_double2(0.0, 0.0), v23 = make_double2(0.0, 0.0);
        if (blk < nblk) {
            const double* src = A + (blk * TS_B + lane) * (long long)ld + col0 + 4 * w;
            v01 = *reinterpret_cast<const double2*>(src);
            v23 = *reinterpret_cast<const double2*>(src + 2);
        }
        a[0][r] = v01.x; a[1][r] = v01.y; a[2][r] = v23.x; a[3][r] = v23.y;
        if (upper_only) {   // level >= 1: every block is the R block of a subtile below; under its diagonal lie stale reflectors
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (lane > 4 * w + j) a[j][r] = 0.0;
        }
    }
#pragma unroll 1
    for (int ib = 0; ib < TS_B / 4; ++ib) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = ib * 4 + k;
            const int buf = k & 1;
            if (w == ib) {
                // ---- owner of column i: norm of the column below the pivot, dlarfg scalars, publication ----
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int r = 0; r < TS_FAN; r += 2) {
                    double x0 = a[k][r], x1 = a[k][r + 1];
                    if (r == 0 && lane <= i) x0 = 0.0;      // top block: the pivot row and the rows above it
                    vbuf[buf][r][lane] = x0;
                    vbuf[buf][r + 1][lane] = x1;
                    s0 = fma(x0, x0, s0);
                    s1 = fma(x1, x1, s1);
                }
                const double sigma = warp_allsum(s0 + s1);
                const double alpha = __shfl_sync(0xffffffffu, a[k][0], i);
                double tau = 0.0, scale = 0.0, beta = alpha;
                if (sigma != 0.0) {   // dlarfg: beta = -sign(alpha) * ||(alpha, x)||, tau = (beta - alpha) / beta
                    // one rsqrt and one reciprocal instead of sqrt + two divisions (the scalar chain is on the critical
                    // path of every column): ||.|| = s * rsqrt(s), 1/beta = -sign(alpha) * rsqrt(s); each within ~1 ulp,
                    // which perturbs H by O(eps) exactly like the rounding of tau itself
                    const double s2 = fma(alpha, alpha, sigma);
                    const double rs = rsqrt(s2);
                    beta = -copysign(s2 * rs, alpha);
                    const double dab = alpha - beta;
                    scale = __drcp_rn(dab);
                    tau = dab * copysign(rs, alpha);
                }
                if (lane == 0) { sc[buf][0] = tau; sc[buf][1] = scale; taus[i] = tau; }
                if (lane == i) a[k][0] = beta;
                ms[k] = scale;
            }
            __syncthreads();
            {
                // ---- every warp: u_i . (own columns); live columns (> i) are updated, finished ones feed T ----
                double v[TS_FAN];
#pragma unroll
                for (int r = 0; r < TS_FAN; ++r) v[r] = vbuf[buf][r][lane];
                const double tau = sc[buf][0], scale = sc[buf][1];
                double d[4], g[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    double e0 = v[0] * a[j][0], e1 = v[1] * a[j][1];
#pragma unroll
                    for (int r = 2; r < TS_FAN; r += 2) { e0 = fma(v[r], a[j][r], e0); e1 = fma(v[r + 1], a[j][r + 1], e1); }
                    d[j] = e0 + e1;
                }
                warp_allsum4(d, g, lane);
                if (w >= ib) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const bool later = (w > ib) || (j > k);              // column 4w + j > i
                        const double pr = __shfl_sync(0xffffffffu, a[j][0], i);   // its entry in the pivot row
                        const double gv = fma(scale, g[j], pr);
                        const double wc = later ? tau * gv : 0.0;
                        if (w == ib && j < k && lane == 0) Gs[4 * w + j][i] = ms[j] * gv;   // v_c . v_i, c < i in the owner's group
                        if (lane == i) a[j][0] -= wc;
                        const double cs = wc * scale;
#pragma unroll
                        for (int r = 0; r < TS_FAN; ++r) a[j][r] = fma(-cs, v[r], a[j][r]);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const double pr = __shfl_sync(0xffffffffu, a[j][0], i);
                        if (lane == 0) Gs[4 * w + j][i] = ms[j] * fma(scale, g[j], pr);
                    }
                }
            }
        }
    }
    // ---- store: R on and above the diagonal of the top block, scaled reflectors everywhere else ----
#pragma unroll
    for (int r = 0; r < TS_FAN; ++r) {
        const long long blk = (sub * TS_FAN + r) * stride;
        double o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool is_r = (r == 0) && (lane <= 4 * w + j);
            o[j] = is_r ? a[j][r] : a[j][r] * ms[j];
            // keep V (unit lower trapezoid, scaled) for the residual-column update below
            a[j][r] = (r == 0 && lane < 4 * w + j) ? 0.0 : ((r == 0 && lane == 4 * w + j) ? 1.0 : o[j]);
        }
        if (blk < nblk) {
            double* dst = A + (blk * TS_B + lane) * (long long)ld + col0 + 4 * w;
            *reinterpret_cast<double2*>(dst) = make_double2(o[0], o[1]);
            *reinterpret_cast<double2*>(dst + 2) = make_double2(o[2], o[3]);
        }
    }
    bsh[w][lane] = bval;
    __syncthreads();
    // compact-WY factor: T = U^-1 with U = striu(V'V) + diag(1/tau); column `lane` by back substitution.
    // tau_r = 0 (H_r = I) gives a zero row/column r, as in dlarft.
    if (w == 0) {
        double t[TS_B];
#pragma unroll
        for (int r = TS_B - 1; r >= 0; --r) {
            double sa = (r == lane) ? 1.0 : 0.0, sb = 0.0;
#pragma unroll
            for (int kk = r + 1; kk < TS_B; kk += 2) {
                sa = fma(-Gs[r][kk], t[kk], sa);
                if (kk + 1 < TS_B) sb = fma(-Gs[r][kk + 1], t[kk + 1], sb);
            }
            t[r] = (r <= lane) ? (sa + sb) * taus[r] : 0.0;
        }
        double* Tg = Tbuf + sub * (TS_B * TS_B);
#pragma unroll
        for (int r = 0; r < TS_B; ++r) Tg[r * TS_B + lane] = t[r];
    }
    if (rcol < 0) return;
    // ---- residual column: b <- (I - V T' V') b ----
    {
        double d[4] = {0.0, 0.0, 0.0, 0.0}, g[4];
#pragma unroll
        for (int r = 0; r < TS_FAN; ++r) {
            const double br = bsh[r][lane];
#pragma unroll
            for (int j = 0; j < 4; ++j) d[j] = fma(br, a[j][r], d[j]);
        }
        warp_allsum4(d, g, lane);
        if (lane < 4) gb[4 * w + lane] = (lane == 0) ? g[0] : ((lane == 1) ? g[1] : ((lane == 2) ? g[2] : g[3]));
    }
    __syncthreads();
    if (w == 0) {
        const double* Tg = Tbuf + sub * (TS_B * TS_B);          // column `lane` of T: this lane's own stores
        double w0 = 0.0, w1 = 0.0;
#pragma unroll
        for (int kk = 0; kk < TS_B; kk += 2) {
            w0 = fma(Tg[kk * TS_B + lane], gb[kk], w0);
            w1 = fma(Tg[(kk + 1) * TS_B + lane], gb[kk + 1], w1);
        }
        wb[lane] = -(w0 + w1);                                   // W = -T' (V'b)
    }
    __syncthreads();
    {
        const double w4[4] = {wb[4 * w], wb[4 * w + 1], wb[4 * w + 2], wb[4 * w + 3]};
#pragma unroll
        for (int r = 0; r < TS_FAN; ++r) {
            double e = a[0][r] * w4[0];
#pragma unroll
            for (int j = 1; j < 4; ++j) e = fma(a[j][r], w4[j], e);
            part[w][r][lane] = e;                                // this column group's share of (V W)[row 32 r + lane]
        }
    }
    __syncthreads();
    if (bvalid) {
        const double t = ((part[0][w][lane] + part[1][w][lane]) + (part[2][w][lane] + part[3][w][lane])) +
                         ((part[4][w][lane] + part[5][w][lane]) + (part[6][w][lane] + part[7][w][lane]));
        *bptr = bval + t;
    }
}

// ---------------------------------------------------------------------------------------------
// trailing update, staged form: one CTA per (subtile, chunk of 32-column blocks)
// ---------------------------------------------------------------------------------------------
// The reflector block V (256 x 32) and T are brought into shared memory ONCE per CTA with cp.async and serve every
// column block of the chunk; the 256 x 32 block of B is staged by cp.async as well, and the copy of the NEXT block is
// in flight while the W stage and the second product of the current one run.  All DMMA operands then come from
// shared memory (leading dimension 36 doubles: conflict-free m8n8k4 fragment loads for both products), so no warp
// waits on a global load in front of the tensor pipe.
//   pass 1  G = V'B : warps 0-3 take rows 0..127, warps 4-7 rows 128..255; inside a half each warp owns one 16 x 16
//           quadrant of G (2 x 2 tiles, 4 independent accumulator chains); the two half sums land in G0 / G1 and are
//           added, in that fixed order, where they are consumed -- no reduction tree, one barrier
//   W stage W = -T'(G0 + G1), 2 tiles per warp
//   pass 2  B_w += V_w W : warp w owns rows 32w..32w+31 (4 x 4 tiles), accumulators preloaded from the staged block
// B is read from HBM once and written once; V once per chunk.
constexpr int TR_LD = 36;
constexpr int TR_ROWS = TS_B * TS_FAN;   // 256
constexpr int TR_NW = 8;                 // warps per CTA
constexpr int TR_KS = TR_NW / 4;         // row splits of pass 1 (each split: 4 warps = the 4 quadrants of G)
constexpr int TR_SMEM = (2 * TR_ROWS * TR_LD + (2 + TR_KS) * TS_B * TR_LD) * (int)sizeof(double);   // V, B | T, W, G[KS]

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc, bool pred) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = pred ? 16 : 0;   // src-size 0: the 16 bytes are zero-filled, nothing is read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int NW>
__global__ void __launch_bounds__(32 * NW, 1)
tsqr_trail_staged_kernel(double* __restrict__ A, int ld, long long nblk, long long stride, int col0, int ncb, int cbpc,
                         const double* __restrict__ Tbuf) {
    constexpr int NTH = 32 * NW;
    constexpr int KS = NW / 4;            // row splits in pass 1
    constexpr int KROWS = TR_ROWS / KS;   // rows per split
    constexpr int RW = TR_ROWS / NW;      // rows per warp in pass 2
    constexpr int RT = RW / 8;            // 8-row tiles per warp in pass 2
    extern __shared__ __align__(16) double smem[];
    double* Vs = smem;
    double* Bs = Vs + TR_ROWS * TR_LD;
    double* Ts = Bs + TR_ROWS * TR_LD;
    double* Ws = Ts + TS_B * TR_LD;
    double* Gs = Ws + TS_B * TR_LD;       // KS partial sums of G, one per row split
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int nchunks = (ncb + cbpc - 1) / cbpc;
    const long long sub = blockIdx.x / (unsigned)nchunks;
    const int chunk = (int)(blockIdx.x % (unsigned)nchunks);
    const int cb_begin = chunk * cbpc;
    const int cb_end = (cb_begin + cbpc < ncb) ? cb_begin + cbpc : ncb;
    // 256 x 32 tile at column c0 of this subtile -> dst (16-byte chunks; 16 consecutive threads cover one row)
    auto stage = [&](double* dst, int c0) {
#pragma unroll
        for (int q = 0; q < 4096 / NTH; ++q) {
            const int id = tid + NTH * q;
            const int row = id >> 4, c16 = id & 15;
            const long long blk = (sub * TS_FAN + (row >> 5)) * stride;
            const bool ok = blk < nblk;
            const double* src = ok ? A + (blk * TS_B + (row & 31)) * (long long)ld + c0 + 2 * c16 : A;
            cp_async16(dst + row * TR_LD + 2 * c16, src, ok);
        }
    };
    stage(Vs, col0);
    stage(Bs, col0 + TS_B * (cb_begin + 1));
    cp_async_commit();
    {
        const double* Tg = Tbuf + sub * (TS_B * TS_B);
#pragma unroll
        for (int q = 0; q < 1024 / NTH; ++q) {
            const int idx = tid + NTH * q;
            Ts[(idx >> 5) * TR_LD + (idx & 31)] = Tg[idx];
        }
    }
    cp_async_wait_all();
    __syncthreads();
    // the top block of V is a unit lower trapezoid (R of the panel sits on and above its diagonal)
#pragma unroll
    for (int q = 0; q < 1024 / NTH; ++q) {
        const int idx = tid + NTH * q;
        const int r = idx >> 5, c = idx & 31;
        if (r <= c) Vs[r * TR_LD + c] = (r == c) ? 1.0 : 0.0;
    }
    __syncthreads();
    const long long myblk = (sub * TS_FAN + ((w * RW) >> 5)) * stride;   // block holding this warp's rows of pass 2
    const bool valid = myblk < nblk;
    const int kh = w >> 2, qd = w & 3;
    const int ti0 = (qd >> 1) * 2, tj0 = (qd & 1) * 2;
    double* Gk = Gs + kh * (TS_B * TR_LD);
    for (int cb = cb_begin; cb < cb_end; ++cb) {
        if (cb > cb_begin) {
            cp_async_wait_all();
            __syncthreads();
        }
        // ---- pass 1: this warp's quadrant of G over its share of the rows ----
        double acc[2][2][2];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        {
            const double* vp = Vs + (kh * KROWS + t) * TR_LD + ti0 * 8 + g;
            const double* bp = Bs + (kh * KROWS + t) * TR_LD + tj0 * 8 + g;
#pragma unroll 8
            for (int kk = 0; kk < KROWS / 4; ++kk) {
                const double a0 = vp[kk * 4 * TR_LD], a1 = vp[kk * 4 * TR_LD + 8];
                const double b0 = bp[kk * 4 * TR_LD], b1 = bp[kk * 4 * TR_LD + 8];
                dmma884(acc[0][0][0], acc[0][0][1], a0, b0);
                dmma884(acc[0][1][0], acc[0][1][1], a0, b1);
                dmma884(acc[1][0][0], acc[1][0][1], a1, b0);
                dmma884(acc[1][1][0], acc[1][1][1], a1, b1);
            }
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
                *reinterpret_cast<double2*>(Gk + ((ti0 + i) * 8 + g) * TR_LD + (tj0 + j) * 8 + 2 * t) =
                    make_double2(acc[i][j][0], acc[i][j][1]);
        // accumulators of pass 2: this warp's rows of the staged block
        double b2[RT][4][2];
#pragma unroll
        for (int ri = 0; ri < RT; ++ri)
#pragma unroll
            for (int cj = 0; cj < 4; ++cj) {
                const double2 v = *reinterpret_cast<const double2*>(Bs + (w * RW + ri * 8 + g) * TR_LD + cj * 8 + 2 * t);
                b2[ri][cj][0] = v.x; b2[ri][cj][1] = v.y;
            }
        __syncthreads();
        if (cb + 1 < cb_end) {   // Bs is free: the next block streams in during the W stage and pass 2
            stage(Bs, col0 + TS_B * (cb + 2));
            cp_async_commit();
        }
        // ---- W = -T' G, G = the row-split partial sums added in a fixed order: 16 tiles over the warps ----
#pragma unroll
        for (int id = w; id < 16; id += NW) {
            const int ti = id >> 2, tj = id & 3;
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
                const int o = (kk * 4 + t) * TR_LD + tj * 8 + g;
                double gv;
                if (KS == 2) gv = Gs[o] + Gs[TS_B * TR_LD + o];
                else gv = (Gs[o] + Gs[TS_B * TR_LD + o]) + (Gs[2 * TS_B * TR_LD + o] + Gs[3 * TS_B * TR_LD + o]);
                dmma884(c0, c1, Ts[(kk * 4 + t) * TR_LD + ti * 8 + g], gv);
            }
            *reinterpret_cast<double2*>(Ws + (ti * 8 + g) * TR_LD + tj * 8 + 2 * t) = make_double2(-c0, -c1);
        }
        __syncthreads();
        // ---- pass 2: B_w += V_w W ----
        {
            const double* vp = Vs + (w * RW + g) * TR_LD + t;
            const double* wp = Ws + t * TR_LD + g;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
                double av[RT], bw[4];
#pragma unroll
                for (int ri = 0; ri < RT; ++ri) av[ri] = vp[ri * 8 * TR_LD + kk * 4];
#pragma unroll
                for (int cj = 0; cj < 4; ++cj) bw[cj] = wp[kk * 4 * TR_LD + cj * 8];
#pragma unroll
                for (int ri = 0; ri < RT; ++ri)
#pragma unroll
                    for (int cj = 0; cj < 4; ++cj) dmma884(b2[ri][cj][0], b2[ri][cj][1], av[ri], bw[cj]);
            }
        }
        if (valid) {
            double* Bb = A + (myblk * TS_B + ((w * RW) & 31)) * (long long)ld + col0 + TS_B * (cb + 1);
#pragma unroll
            for (int ri = 0; ri < RT; ++ri)
#pragma unroll
                for (int cj = 0; cj < 4; ++cj)
                    *reinterpret_cast<double2*>(Bb + (long long)(ri * 8 + g) * ld + cj * 8 + 2 * t) =
                        make_double2(b2[ri][cj][0], b2[ri][cj][1]);
        }
    }
}

// rows 0..31 of the matrix now hold rows col0..col0+31 of R: copy them out and clear them in place
// (one CTA per row: at n = 4096 a single CTA needed 140 us per panel)
__global__ void tsqr_extract_kernel(double* __restrict__ A, int ld, int col0, int ncols, double* __restrict__ Rout,
                                    int ldr) {
    const int r = blockIdx.x;
    for (int c = col0 + threadIdx.x; c < ld; c += blockDim.x) {
        double v = A[(long long)r * ld + c];
        if (c < col0 + TS_B && c - col0 < r) v = 0.0;
        if (c < ncols) Rout[(long long)(col0 + r) * ldr + c] = v;
        A[(long long)r * ld + c] = 0.0;
    }
}

// sum of squares of one column: stage 1 (fixed grid, fixed tree) and stage 2
__global__ void __launch_bounds__(256) tsqr_colsq_kernel(const double* __restrict__ A, int ld, long long rows, int col,
                                                          double* __restrict__ part) {
    __shared__ double sh[256];
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < rows; i += (long long)gridDim.x * 256) {
        double v = A[i * ld + col];
        s = fma(v, v, s);
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}
__global__ void tsqr_colsq_finish_kernel(const double* __restrict__ part, int nparts, double* __restrict__ Rout,
                                         int ldr, int col) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < nparts; ++i) s += part[i];
        Rout[(long long)col * ldr + col] = sqrt(s);
    }
}

// distributed variant of the last column: local sum of squares -> out[0] (all-reduced by the caller) -> sqrt into R
__global__ void tsqr_colsq_partial_kernel(const double* __restrict__ part, int nparts, double* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < nparts; ++i) s += part[i];
        out[0] = s;
    }
}
__global__ void tsqr_sqrt_store_kernel(const double* __restrict__ in, double* __restrict__ Rout, int ldr, int col) {
    if (threadIdx.x == 0 && blockIdx.x == 0) Rout[(long long)col * ldr + col] = sqrt(in[0]);
}
// rows 0..31 of the local matrix <- this rank's 32 rows of the cross-rank stage (columns left of c_from hold reflector
// data there: they are zero in the matrix)
__global__ void tsqr_copyback_kernel(double* __restrict__ A, const double* __restrict__ P, int ld, int c_from) {
    const int r = blockIdx.x;
    for (int c = threadIdx.x; c < ld; c += blockDim.x) A[(long long)r * ld + c] = (c >= c_from) ? P[(long long)r * ld + c] : 0.0;
}

// Row-sharded factorisation (one process per GPU): the cross-rank stage is ONE MORE LEVEL of every panel's tree.  After
// the local levels of panel j each rank holds a 32-row R block (rows 0..31 of its matrix); the blocks are all-gathered
// (32 x ld doubles per rank), every rank factors the stacked nranks x 32 rows (one subtile for up to 8 ranks) and
// updates their trailing columns -- replicated, identical bits everywhere; rows 0..31 of the result are rows
// 32 j .. 32 j + 31 of the global R, the other blocks are fill that goes back to rows 0..31 of their owners and takes part
// in the next panel.  Against factoring locally, gathering the whole R factors and factoring the (nranks (n + 32)) x (n + 1)
// stack again (~100 launches of latency-bound single-wave kernels): 8 small all-gathers + 8 x (one panel + one trailing
// launch) at n = 256.
struct TsqrDist {
    int nranks = 1, rank = 0;
    double* P = nullptr;         // max(nranks, 8) * 32 rows x ld, zero-initialised
    double* scal = nullptr;      // one double
    void* ctx = nullptr;
    int (*allgather)(void* ctx, const double* send, double* recv, size_t count, cudaStream_t st) = nullptr;
    int (*allreduce_sum)(void* ctx, double* buf, size_t count, cudaStream_t st) = nullptr;
};

// Chunking of the trailing launches: twice the prologue of a chunk (V and T staged), in units of one column block.
// Measured on B200 at n = 4096, m = 16384: 48.7 / 49.1 / 49.5 / 50.4 ms per factorisation with 1 / 2 / 4 / 8.
constexpr int TS_CHUNK_PROLOGUE2 = 1;

// Host-side launcher.  A: rows_pad x ld row major, rows_pad a multiple of 32, pad rows zero.
// ncols = n + 1 with n a multiple of 32 (columns n+1 .. ld-1 must be zero; ld = n + 8).
// Rout: (n + 1) x ldr row major, zero-initialised by the caller.  Tbuf: ceil(nblk / 8) * 1024 doubles.
// part: >= 512 doubles.  Returns the number of kernels launched.
// dist (optional): row-sharded factorisation, see TsqrDist; returns -1 when a collective fails.
inline int tsqr_factor(double* A, int ld, long long rows_pad, int n, double* Rout, int ldr, double* Tbuf, double* part,
                       cudaStream_t st, const TsqrDist* dist = nullptr) {
    const long long nblk = rows_pad / TS_B;
    const int npanels = n / TS_B;
    int launches = 0;
    // > 48 KB of dynamic shared memory needs the opt-in (per device, so it is simply set on every call)
    cudaFuncSetAttribute(tsqr_trail_staged_kernel<TR_NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, TR_SMEM);
    // all tree levels of panel j on the matrix M (nblk_m blocks of 32 rows)
    auto panel_levels = [&](double* M, long long nblk_m, int j) {
        const long long nblk = nblk_m;
        double* A = M;
        const int col0 = j * TS_B;
        const int ncb32 = npanels - 1 - j;
        long long stride = 1;
        for (int level = 0;; ++level) {
            long long nb_level = (nblk + stride - 1) / stride;
            if (level > 0 && nb_level <= 1) break;
            long long nsub = (nb_level + TS_FAN - 1) / TS_FAN;
            tsqr_panel_cg_kernel<<<(unsigned)nsub, 256, 0, st>>>(A, ld, nblk, stride, col0, level > 0, n, Tbuf);
            ++launches;
            if (ncb32 > 0) {
                // Column blocks per CTA (chunk).  One CTA per SM is resident (registers, shared memory), so the launch runs
                // in waves of 148 CTAs; a CTA costs a prologue (V and T staged once per chunk, about half a block's worth) plus
                // its column blocks.  Pick the chunking with the fewest wave-units: with thousands of subtiles that is one
                // chunk per subtile, with a few dozen subtiles (m = 4 n, upper tree levels) it avoids a mostly empty last
                // wave.  The arithmetic of a column block does not depend on the chunk it is in.
                int cbpc = ncb32;
                long long best_cost = -1;
                for (int c = ncb32; c >= 1; --c) {
                    const long long chunks = (ncb32 + c - 1) / c;
                    if (c < ncb32 && (ncb32 + c) / (c + 1) == chunks) continue;      // same chunk count as c + 1: larger CTAs for nothing
                    const long long waves = (nsub * chunks + 147) / 148;
                    const long long cost = waves * (TS_CHUNK_PROLOGUE2 + 2 * c);
                    if (best_cost < 0 || cost < best_cost) { best_cost = cost; cbpc = c; }
                }
                const int nchunks = (ncb32 + cbpc - 1) / cbpc;
                tsqr_trail_staged_kernel<TR_NW><<<(unsigned)(nsub * nchunks), 32 * TR_NW, TR_SMEM, st>>>(A, ld, nblk, stride, col0, ncb32,
                                                                                          cbpc, Tbuf);
                ++launches;
            }
            stride *= TS_FAN;
        }
    };
    const bool sharded = dist && dist->nranks > 1;
    for (int j = 0; j < npanels; ++j) {
        const int col0 = j * TS_B;
        panel_levels(A, nblk, j);
        if (sharded) {
            if (dist->allgather(dist->ctx, A, dist->P, (size_t)TS_B * ld, st) != 0) return -1;
            panel_levels(dist->P, dist->nranks, j);
            tsqr_extract_kernel<<<TS_B, 256, 0, st>>>(dist->P, ld, col0, n + 1, Rout, ldr);
            tsqr_copyback_kernel<<<TS_B, 256, 0, st>>>(A, dist->P + (size_t)TS_B * dist->rank * ld, ld, col0 + TS_B);
            launches += 2;
        } else {
            tsqr_extract_kernel<<<TS_B, 256, 0, st>>>(A, ld, col0, n + 1, Rout, ldr);
            ++launches;
        }
    }
    const int nparts = 296;
    tsqr_colsq_kernel<<<nparts, 256, 0, st>>>(A, ld, rows_pad, n, part);
    if (sharded) {
        tsqr_colsq_partial_kernel<<<1, 32, 0, st>>>(part, nparts, dist->scal);
        if (dist->allreduce_sum(dist->ctx, dist->scal, 1, st) != 0) return -1;
        tsqr_sqrt_store_kernel<<<1, 32, 0, st>>>(dist->scal, Rout, ldr, n);
        return launches + 3;
    }
    tsqr_colsq_finish_kernel<<<1, 32, 0, st>>>(part, nparts, Rout, ldr, n);
    return launches + 2;
}

}  // namespace enl_large
