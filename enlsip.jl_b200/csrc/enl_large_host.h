// enl_large_host.h -- ENLSIP iteration driver of the LARGE-JACOBIAN regime (BASELINE.json configs 4/5).
//
// The reference iteration (`enlsip`, src/enlsip_functions.jl = EF, EF:2638-2880 and everything it
// calls) touches the m x n residual Jacobian J and the m-vector r only through
//   (i)   orthogonally invariant quantities: J'r, J*Q1, QRCP(J2), Q3'(-J1 p1 - r), norms, dots;
//   (ii)  evaluations of r at trial points of the linesearch (EF:1307-1340, 1665-1689).
// The engine therefore factors the augmented matrix [J r] = Q [R_J z; 0 rho] ONCE per iterate
// with a tall-skinny QR on the GPU (enl_tsqr.cuh) and runs (i) on the compressed problem
//     J~ = [R_J; 0]  ((n+1) x n),   r~ = [z; rho]  (n+1),
// which has exactly the same search direction, multipliers, ranks, pivots and norms as (J, r);
// (ii) is served by elementwise kernels over the device-resident m-vectors (LargeOps below).
//
// This header is pure C++ (no CUDA): the product compiles it into libenlsip_b200.so with the CUDA
// implementation of LargeOps (enl_large.cu); tests compile it with a plain CPU LargeOps to check the
// driver logic against the oracle without a GPU (oracle/hostport, test infrastructure only).
//
// Semantics restated from the reference, with the same quirks as the batched core (enl_solver.h):
//   * the always-reverted first-order deletion (EF:706-765, SURVEY.md T3) is skipped, keeping its
//     surviving side effects;  J*F_A.Q is formed once per factorisation (EF:219, 526, 1249);
//   * aliasing schedule of Iteration.rx / .cx (SURVEY.md T1) modelled by snapshot-or-live scalars;
//   * where Julia would throw / loop forever the solve ends with exit code -99 / -98.
// Newton steps (EF:348-423) do not exist in this regime: `second_derivatives` is forced off when
// n + m >= 1000 (EF:2658), and the entry point rejects smaller problems (they belong to the batched engine).
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <stdexcept>
#include <string>
#include <vector>

namespace enl_large {

constexpr double EPS = 2.220446049250313e-16;
constexpr double SQRT_EPS = 1.4901161193847656e-08;
constexpr double TOL3Z = 1.0536712127723509e-08;   // dlaqp2: sqrt(dlamch('Epsilon')) = sqrt(2^-53) (same constant as enl_base.h)

struct WouldThrow { const char* what; };
struct WouldHang { const char* what; };

using Vec = std::vector<double>;

struct Mat {   // column major
    int rows = 0, cols = 0;
    Vec a;
    Mat() {}
    Mat(int r, int c) : rows(r), cols(c), a((size_t)r * c, 0.0) {}
    double& operator()(int r, int c) { return a[(size_t)c * rows + r]; }
    double operator()(int r, int c) const { return a[(size_t)c * rows + r]; }
    double* col(int c) { return a.data() + (size_t)c * rows; }
    const double* col(int c) const { return a.data() + (size_t)c * rows; }
};

inline double dot_n(const double* a, const double* b, int n) {
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    int i = 0;
    for (; i + 4 <= n; i += 4) {
        s0 += a[i] * b[i]; s1 += a[i + 1] * b[i + 1]; s2 += a[i + 2] * b[i + 2]; s3 += a[i + 3] * b[i + 3];
    }
    for (; i < n; ++i) s0 += a[i] * b[i];
    return (s0 + s1) + (s2 + s3);
}
inline double norm_n(const double* a, int n) { return sqrt(dot_n(a, a, n)); }
// dnrm2 as dgeqp3 / dlaqp2 / dlarfg call it (OpenBLAS' x86-64 kernel sums the squares in x87 extended precision, then
// rounds the square root to double).  With row scaling every column of C.A' has norm 1 up to an ulp, and the pivot
// order is decided by how that last bit rounds: a plain double sum picks other pivots than the reference.
// Where long double is not the x87 format (aarch64: IEEE quad) the sum stays in double.
inline double nrm2_ext(const double* a, int n) {
#if LDBL_MANT_DIG == 64
    long double s = 0.0L;
    for (int i = 0; i < n; ++i) s += (long double)a[i] * a[i];
    return (double)sqrtl(s);
#else
    return norm_n(a, n);
#endif
}
inline double dotv(const Vec& a, const Vec& b) { return dot_n(a.data(), b.data(), (int)a.size()); }
inline double normv(const Vec& a) { return norm_n(a.data(), (int)a.size()); }
inline double lapy2(double x, double y) {
    double xa = fabs(x), ya = fabs(y), w = fmax(xa, ya), z = fmin(xa, ya);
    if (z == 0.0) return w;
    double q = z / w;
    return w * sqrt(1.0 + q * q);
}

// norm(v[1:k]) with Julia range semantics: empty if k <= 0, BoundsError if k > length
inline double norm_range(const Vec& v, int k) {
    if (k <= 0) return 0.0;
    if (k > (int)v.size()) throw WouldThrow{"BoundsError v[1:k]"};
    return norm_n(v.data(), k);
}

// ------------------------------------------------------------------------------------------
// Wall-clock profile of the host driver (development aid, printed when ENLSIP_PROF is set)
struct HostProf {
    static constexpr int N = 16;
    double ms[N] = {0};
    long long calls[N] = {0};
    const char* names[N] = {"new_point", "gather_active", "factor_A", "factor_L11", "ensure_JQ1", "gn_search_direction",
                            "first_lagrange", "second_lagrange", "update_working_set", "search_direction_analys",
                            "compute_steplength", "upper_bound_steplength", "evaluate_violated", "termination", "compute_gradf", "other"};
    void dump() const {
        for (int i = 0; i < N; ++i)
            if (calls[i]) fprintf(stderr, "  [enlsip host prof] %-26s %6lld calls %10.2f ms\n", names[i], calls[i], ms[i]);
    }
};
inline HostProf& host_prof() { static thread_local HostProf p; return p; }
struct ProfScope {
    int id;
    std::chrono::steady_clock::time_point t0;
    explicit ProfScope(int i) : id(i), t0(std::chrono::steady_clock::now()) {}
    ~ProfScope() {
        host_prof().ms[id] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        host_prof().calls[id]++;
    }
};

// ------------------------------------------------------------------------------------------
// qr(M, ColumnNorm()) = LAPACK dgeqp3 (restated as the unblocked dlaqp2: first-max pivot, dlarfg
// with beta = -sign(alpha)*dlapy2, partial-norm downdate with the tol3z recompute rule; SURVEY.md 10)
// ------------------------------------------------------------------------------------------
struct QRP {
    int rows = 0, cols = 0, k = 0;
    Mat f;            // factors
    Vec tau;
    std::vector<int> p;   // jpvt, 0-based

    void factor(const Mat& M) {
        f = M;
        rows = M.rows; cols = M.cols; k = std::min(rows, cols);
        tau.assign(k, 0.0);
        p.resize(cols);
        Vec vn1(cols), vn2(cols);
        for (int j = 0; j < cols; ++j) {
            p[j] = j;
            vn1[j] = vn2[j] = nrm2_ext(f.col(j), rows);
        }
        Vec wv(cols);
        for (int i = 0; i < k; ++i) {
            int pvt = i;
            double best = vn1[i];
            for (int j = i + 1; j < cols; ++j)
                if (vn1[j] > best) { best = vn1[j]; pvt = j; }
            if (pvt != i) {
                std::swap_ranges(f.col(pvt), f.col(pvt) + rows, f.col(i));
                std::swap(p[pvt], p[i]);
                vn1[pvt] = vn1[i];
                vn2[pvt] = vn2[i];
            }
            double* ci = f.col(i);
            double tau_i = 0.0;
            if (i < rows - 1) {
                double alpha = ci[i];
                double xn = nrm2_ext(ci + i + 1, rows - i - 1);
                if (xn != 0.0) {
                    double beta = -copysign(lapy2(alpha, xn), alpha);
                    tau_i = (beta - alpha) / beta;
                    double sc = 1.0 / (alpha - beta);
                    for (int r = i + 1; r < rows; ++r) ci[r] *= sc;
                    ci[i] = beta;
                }
            }
            tau[i] = tau_i;
            if (i < cols - 1 && tau_i != 0.0) {
                const int len = rows - i - 1;
#pragma omp parallel for schedule(static) if ((long long)len * (cols - i) > 200000)
                for (int c = i + 1; c < cols; ++c) {
                    double* cc = f.col(c);
                    double w = (cc[i] + dot_n(ci + i + 1, cc + i + 1, len)) * tau_i;
                    cc[i] -= w;
                    for (int r = i + 1; r < rows; ++r) cc[r] -= w * ci[r];
                }
            }
            for (int j = i + 1; j < cols; ++j) {
                double v1 = vn1[j];
                if (v1 != 0.0) {
                    double tq = fabs(f(i, j)) / v1;
                    double temp = fmax(1.0 - tq * tq, 0.0);
                    double rq = v1 / vn2[j];
                    double temp2 = temp * (rq * rq);
                    if (temp2 <= TOL3Z) {
                        if (i < rows - 1) {
                            vn1[j] = vn2[j] = nrm2_ext(f.col(j) + i + 1, rows - i - 1);
                        } else {
                            vn1[j] = vn2[j] = 0.0;
                        }
                    } else {
                        vn1[j] = v1 * sqrt(temp);
                    }
                }
            }
        }
    }
    double R(int r, int c) const { return (r <= c) ? f(r, c) : 0.0; }
    double diag(int i) const { return f(i, i); }
    std::vector<int> invperm() const {
        std::vector<int> ip(cols);
        for (int j = 0; j < cols; ++j) ip[p[j]] = j;
        return ip;
    }
    // v <- Q' v   (v has `rows` entries)
    void Qt_mul(double* v) const {
        for (int i = 0; i < k; ++i) {
            double ti = tau[i];
            if (ti == 0.0) continue;
            const double* ci = f.col(i);
            double w = (v[i] + dot_n(ci + i + 1, v + i + 1, rows - i - 1)) * ti;
            v[i] -= w;
            for (int r = i + 1; r < rows; ++r) v[r] -= w * ci[r];
        }
    }
    // v <- Q v
    void Q_mul(double* v) const {
        for (int i = k - 1; i >= 0; --i) {
            double ti = tau[i];
            if (ti == 0.0) continue;
            const double* ci = f.col(i);
            double w = (v[i] + dot_n(ci + i + 1, v + i + 1, rows - i - 1)) * ti;
            v[i] -= w;
            for (int r = i + 1; r < rows; ++r) v[r] -= w * ci[r];
        }
    }
    // M <- M * Q   (M is mr x rows): apply H(0), H(1), ... from the right; column major M so each
    // reflector is a rank-one update of the columns i.. of M
    void mul_Q(Mat& M) const {
        const int mr = M.rows;
        Vec w(mr);
        for (int i = 0; i < k; ++i) {
            double ti = tau[i];
            if (ti == 0.0) continue;
            const double* ci = f.col(i);
            // w = M[:, i:] * v
            std::copy(M.col(i), M.col(i) + mr, w.begin());
            for (int c = i + 1; c < rows; ++c) {
                double vc = ci[c];
                if (vc == 0.0) continue;
                const double* mc = M.col(c);
                for (int r = 0; r < mr; ++r) w[r] += vc * mc[r];
            }
            for (int r = 0; r < mr; ++r) w[r] *= ti;
            double* mi = M.col(i);
            for (int r = 0; r < mr; ++r) mi[r] -= w[r];
#pragma omp parallel for schedule(static) if ((long long)mr * (rows - i) > 200000)
            for (int c = i + 1; c < rows; ++c) {
                double vc = ci[c];
                if (vc == 0.0) continue;
                double* mc = M.col(c);
                for (int r = 0; r < mr; ++r) mc[r] -= w[r] * vc;
            }
        }
    }
};

// UpperTriangular(R[1:k,1:k]) \ b  where R = upper triangle of the factor f (LAPACK trtrs: throws on zero diagonal)
inline void solve_upper(const QRP& F, int k, double* x) {
    for (int i = k - 1; i >= 0; --i) {
        double s = x[i];
        for (int j = i + 1; j < k; ++j) s -= F.f(i, j) * x[j];
        double d = F.f(i, i);
        if (d == 0.0) throw WouldThrow{"SingularException (upper)"};
        x[i] = s / d;
    }
}
// LowerTriangular(R[1:k,1:k]') \ b
inline void solve_upperT(const QRP& F, int k, double* x) {
    for (int i = 0; i < k; ++i) {
        double s = x[i];
        for (int j = 0; j < i; ++j) s -= F.f(j, i) * x[j];
        double d = F.f(i, i);
        if (d == 0.0) throw WouldThrow{"SingularException (lower)"};
        x[i] = s / d;
    }
}

// EF:17-31 on the diagonal of a factor
inline int pseudo_rank(const QRP& F, double eps_rank) {
    int len = F.k;
    if (len <= 0 || fabs(F.diag(0)) < eps_rank) return 0;
    double tol = fabs(F.diag(0)) * sqrt((double)len) * eps_rank;
    int r = 1;
    while (r < len && fabs(F.diag(r - 1)) > tol) ++r;
    return r - ((r == len && fabs(F.diag(r - 1)) > tol) ? 0 : 1);
}

// What the iteration logic reads of a pivoted QR factorisation: sizes, diag(R), the permutation.  The factors
// themselves (reflectors, R) stay with the SmallBackend that produced them (host memory or HBM).
struct FactorInfo {
    int rows = 0, cols = 0, k = 0;
    Vec diagv;               // diag(R), k entries
    std::vector<int> p;      // jpvt, 0-based
    double diag(int i) const { return diagv[i]; }
    std::vector<int> invperm() const {
        std::vector<int> ip(cols);
        for (int j = 0; j < cols; ++j) ip[p[j]] = j;
        return ip;
    }
    void take(const QRP& F) {
        rows = F.rows; cols = F.cols; k = F.k; p = F.p;
        diagv.resize(k);
        for (int i = 0; i < k; ++i) diagv[i] = F.f(i, i);
    }
};
inline int pseudo_rank(const FactorInfo& F, double eps_rank) {   // EF:17-31
    int len = F.k;
    if (len <= 0 || fabs(F.diag(0)) < eps_rank) return 0;
    double tol = fabs(F.diag(0)) * sqrt((double)len) * eps_rank;
    int r = 1;
    while (r < len && fabs(F.diag(r - 1)) > tol) ++r;
    return r - ((r == len && fabs(F.diag(r - 1)) > tol) ? 0 : 1);
}

// ------------------------------------------------------------------------------------------
// what the driver needs from the m-sized world (device resident in the product)
// ------------------------------------------------------------------------------------------
struct LargeOps {
    int n = 0, l = 0, q = 0;
    long long m = 0;         // true number of residuals (all shards)
    virtual ~LargeOps() {}
    // evaluate r, J, c, A at x (new_point!, EF:34-52): the m-sized part stays with the backend; returned are
    // gradf = J'r (n), *rr = r'r, cx (l), A (l x n, column major).  Returns 0 or an API error.
    // This is all the termination test of the point needs (EF:2838 reads ||J'r||, ||r||^2 and c), so the
    // factorisation below is only paid for points from which the iteration goes on.
    virtual int eval_point(const double* x, double* gradf, double* rr, double* cx, double* A) = 0;
    // compress the point of the last eval_point: Jt ((n+1) x n, column major) = [R_J; 0], rt (n+1) = [z; rho]
    virtual int compress(double* Jt, double* rt) = 0;
    // fix the direction of the linesearch at the current point: sums = {r.r, r.Jp, Jp.Jp}
    virtual int set_direction(const double* x, const double* p, double sums[3]) = 0;
    // ||r(x + alpha p)||^2
    virtual int res_sq(double alpha, double* out) = 0;
    // out = {||r_a||^2, r.v2, Jp.v2, v2.v2} with r_a = r(x + alpha p), v2 = ((r_a - r)/alpha - Jp)/alpha  (EF:1687)
    virtual int ls_coeffs(double alpha, double out[4]) = 0;
    // constraints only (host or device, tiny)
    virtual int cons(const double* x, double* cx) = 0;
    // Wall-clock seconds since the start of the solve as every rank must see them: the time-limit test (EF:2509) is the
    // only termination input that is not bit-replicated across the ranks of a row-sharded solve, and ranks that disagree
    // on it leave each other alone in the next collective.  Sharded backends return the mean over the ranks (one sum
    // all-reduce of elapsed / nranks).
    virtual double agreed_elapsed(double local_elapsed) { return local_elapsed; }
};

struct LargeOptions {
    int max_iter = 100;
    int scaling = 0;
    double time_limit = 1e3;
    double eps_abs = 1e-10, eps_rel = SQRT_EPS, eps_x = SQRT_EPS, eps_c = SQRT_EPS, eps_rank = SQRT_EPS;
};

struct IterTraceL {   // one record per executed iteration (mirrors oracle IterTrace)
    int k, t, rankA, rankJ2, dimA, dimJ2, code, index_del, exit_code;
    double f_new, alpha, p_norm, active_cx_sum, progress;
};

struct LargeResult {
    int exit_code = 0, status = 0, iterations = 0, nact = 0;
    double f = 0.0;
    Vec x;
    std::vector<int> active;
    std::vector<IterTraceL> trace;
    Vec trace_x;          // [iterations executed][n]
    int n_new_point = 0, n_res_eval = 0;
};

struct IterL {   // structures.jl:63-98 (vectors the algorithm really reads + scalars)
    Vec x, p, lam, w, b_gn, d_gn;
    int t = 0, index_alpha_upp = 0, rankA = 0, rankJ2 = 0, dimA = 0, dimJ2 = 0, index_del = 0, code = 1,
        nb_newton_steps = 0;
    double alpha = 1.0, predicted_reduction = 0, progress = 0, grad_res = 0, speed = 0, beta = 0;
    bool restart = false, first = true, add = false, dele = false;
    // rx / cx of the reference are only ever read through dot(rx,rx) / dot(cx,cx) of the PREVIOUS
    // iteration (EF:1141, 1159); `alias` reproduces `iter.rx = rx` (SURVEY.md T1): the value is
    // the live buffer's at copy time
    double rx_sum = 0, cx_sum = 0;
    bool alias = false;
};

struct WorkingSetL {   // structures.jl:209-267, 1-based ids, 0 = empty
    int q = 0, l = 0, t = 0;
    std::vector<int> active, inactive;
    void remove_constraint(int s) {
        inactive[l - t] = active[s - 1];
        std::sort(inactive.begin(), inactive.begin() + (l - t + 1));
        for (int i = s; i < t; ++i) active[i - 1] = active[i];
        active[t - 1] = 0;
        t -= 1;
    }
    void add_constraint(int s) {
        active[t] = inactive[s - 1];
        std::sort(active.begin(), active.begin() + (t + 1));
        for (int i = s; i < l - t; ++i) inactive[i - 1] = inactive[i];
        inactive[l - t - 1] = 0;
        t += 1;
    }
};

struct ConstraintL {   // structures.jl:145-150 ; the t x n matrix A (row i = gradient of active constraint i) lives in the SmallBackend
    Vec cx;
    bool scaling = false;
    Vec diag_scale;
};

// ------------------------------------------------------------------------------------------
// The matrix-sized half of the small stage: everything of the iteration that touches A (l x n), the active
// block C.A (t x n), the compressed Jacobian J~ ((n+1) x n), J~*Q1 and the three pivoted QR factorisations
// (EF:700 F_A, EF:769 F_L11, EF:223 F_J2).  The driver below keeps the scalar logic, the working set and the
// O(n) vectors; it hands vectors in and gets vectors / diagonals / permutations back.
//   HostSmall    (this header): host memory, the CPU test backend;
//   DeviceSmall  (enl_small.cuh, product): everything resident in HBM, CUDA kernels only.
// Size-dependent error situations of the reference (BoundsError, DimensionMismatch, SingularException) are
// decided by the driver from FactorInfo BEFORE a backend call, so a backend never has to throw.
// ------------------------------------------------------------------------------------------
struct SmallBackend {
    virtual ~SmallBackend() {}
    // new_point! (EF:34-52), first half: r, c, A at x; returns J'r (n), ||r||^2 and c (l).  A stays with the backend.
    virtual int new_point_eval(const double* x, double* gradf, double* rr, double* cx) = 0;
    // second half: compress [J | r] of that point; returns r~ (n+1) and J~' r~ (n)
    virtual int new_point_compress(double* rt, double* gradf) = 0;
    // C.A = A[active, :]
    virtual void gather_active(const int* active, int t) = 0;
    // structures.jl:160-178: rown[i] = ||C.A[i, :]||; scaling: C.A[i, :] /= (|rown[i]| < eps ? 1 : rown[i])
    virtual void evaluate_scaling(int t, bool scaling, double* rown) = 0;
    // surviving side effect of the reverted first-order deletion with scaling (EF:742-745):
    // C.A[i, :] = A[active[i], :] * diag_scale[i]
    virtual void rebuild_scaled_rows(const int* active, int t, const double* diag_scale) = 0;
    virtual void remove_active_row(int s0) = 0;                  // 0-based row of C.A
    virtual void factor_A(int t, FactorInfo& F) = 0;             // qr(C.A', ColumnNorm())          EF:700
    virtual void factor_L11(FactorInfo& F) = 0;                  // qr(F_A.R', ColumnNorm())        EF:769
    virtual void factor_J2(int rankA, FactorInfo& F) = 0;        // J*Q1 (once per F_A); qr(J2, ColumnNorm())   EF:219-223
    // EF:461-508: v = R^-1 (Q1' gradf)[1:r] (zero padded to t), grad_res = ||(Q1' gradf)[r+1:n]||,
    //             u = R^-1 R^-T (-c[P])[1:r] (zero padded to t)
    virtual void first_lagrange(int prankA, int t, const Vec& gradf, const Vec& Ccx, Vec& v, Vec& u, double& grad_res) = 0;
    // EF:514-537: v = R^-1 (J1' (r + J p_gn))[1:r] (zero padded to t)
    virtual void second_lagrange(int prankA, int t, const Vec& p_gn, Vec& v) = 0;
    // EF:116-153 (sizes already validated by the driver)
    virtual void sub_search_direction(int t, int rankA, int dimA, int dimJ2, int code, const Vec& Ccx, Vec& p, Vec& b,
                                      Vec& d) = 0;
    // EF:1249-1251: b = F_L11.Q' (-c[P])
    virtual void subspace_rhs(int t, const Vec& Ccx, Vec& b) = 0;
    // EF:1131-1147: d = F_J2.Q' (-(r + J1 p1)), p1 = P_L11[1:rankA,1:rankA] [R11[1:dimA,1:dimA] \ b[1:dimA]; 0]  (rankA > 0)
    //               d = F_J2.Q' (-r)                                                                     (rankA <= 0)
    virtual void subspace_d(int rankA, int dimA, int rankJ2, const Vec& b, Vec& d) = 0;
    // EF:2222-2224: Jp = J~ p (n+1), Ap = A p (l), active_Ap = C.A p (t)
    virtual void products(const Vec& p, int t, Vec& Jp, Vec& Ap, Vec& active_Ap) = 0;
    // EF:2497: ||C.A' C.cx||
    virtual double At_c_norm(int t, const Vec& Ccx) = 0;
};

// Host-memory backend: the CPU test path (oracle/hostport/largeport.cpp).  The product never instantiates it.
struct HostSmall : SmallBackend {
    LargeOps& ops;
    int n, l, mt;
    Mat J;      // mt x n
    Vec rx;     // mt
    Mat A;      // l x n
    Mat CA;     // t x n
    QRP F_A, F_L11, F_J2;
    Mat JQ1;          // J * F_A.Q, formed once per F_A (EF:219, 526, 1249 recompute it)
    bool jq1_valid = false;

    explicit HostSmall(LargeOps& o) : ops(o), n(o.n), l(o.l), mt(o.n + 1) {
        J = Mat(mt, n);
        rx.assign(mt, 0.0);
        A = Mat(l, n);
    }
    int new_point_eval(const double* x, double* gradf, double* rr, double* cx) override {
        jq1_valid = false;
        return ops.eval_point(x, gradf, rr, cx, A.a.data());
    }
    int new_point_compress(double* rt, double* gradf) override {
        int rc = ops.compress(J.a.data(), rx.data());
        if (rc != 0) return rc;
        for (int r = 0; r < mt; ++r) rt[r] = rx[r];
        for (int j = 0; j < n; ++j) gradf[j] = dot_n(J.col(j), rx.data(), mt);
        return 0;
    }
    void gather_active(const int* active, int t) override { ProfScope prof_(1);
        CA = Mat(t, n);
        for (int j = 0; j < n; ++j) {
            const double* aj = A.col(j);
            double* cj = CA.col(j);
            for (int i = 0; i < t; ++i) cj[i] = aj[active[i] - 1];
        }
    }
    void evaluate_scaling(int t, bool scaling, double* rown) override {
        Vec row(n);
        for (int i = 0; i < t; ++i) {
            for (int j = 0; j < n; ++j) row[j] = CA(i, j);
            double row_i = normv(row);
            rown[i] = row_i;
            if (scaling) {
                if (fabs(row_i) < EPS) row_i = 1.0;
                for (int j = 0; j < n; ++j) CA(i, j) = CA(i, j) / row_i;
            }
        }
    }
    void rebuild_scaled_rows(const int* active, int t, const double* diag_scale) override {
        for (int i = 0; i < t; ++i) {
            int k = active[i] - 1;
            for (int j = 0; j < n; ++j) CA(i, j) = A(k, j) * diag_scale[i];
        }
    }
    void remove_active_row(int s0) override {
        Mat A2(CA.rows - 1, n);
        for (int i = 0, o = 0; i < CA.rows; ++i) {
            if (i == s0) continue;
            for (int j = 0; j < n; ++j) A2(o, j) = CA(i, j);
            ++o;
        }
        CA = A2;
    }
    void factor_A(int t, FactorInfo& F) override { ProfScope prof_(2);
        Mat At(n, t);
        for (int i = 0; i < t; ++i)
            for (int j = 0; j < n; ++j) At(j, i) = CA(i, j);
        F_A.factor(At);
        jq1_valid = false;
        F.take(F_A);
    }
    void factor_L11(FactorInfo& F) override { ProfScope prof_(3);   // F_A.R is min(n,t) x t
        int kr = F_A.k, t = F_A.cols;
        Mat Rt(t, kr);
        for (int r = 0; r < kr; ++r)
            for (int c = 0; c < t; ++c) Rt(c, r) = F_A.R(r, c);
        F_L11.factor(Rt);
        F.take(F_L11);
    }
    void ensure_JQ1() { ProfScope prof_(4);
        if (!jq1_valid) {
            JQ1 = J;
            F_A.mul_Q(JQ1);
            jq1_valid = true;
        }
    }
    void factor_J2(int rankA, FactorInfo& F) override {
        ensure_JQ1();
        Mat J2(mt, n - rankA);
        for (int c = rankA; c < n; ++c) std::copy(JQ1.col(c), JQ1.col(c) + mt, J2.col(c - rankA));
        F_J2.factor(J2);
        F.take(F_J2);
    }
    void first_lagrange(int prankA, int t, const Vec& gradf, const Vec& Ccx, Vec& v, Vec& u, double& grad_res) override {
        Vec b = gradf;
        F_A.Qt_mul(b.data());
        v.assign(t, 0.0);
        for (int i = 0; i < prankA; ++i) v[i] = b[i];
        solve_upper(F_A, prankA, v.data());
        grad_res = (n > prankA) ? norm_n(b.data() + prankA, n - prankA) : 0.0;
        Vec y(t, 0.0);
        u.assign(t, 0.0);
        for (int i = 0; i < prankA; ++i) y[i] = -Ccx[F_A.p[i]];
        solve_upperT(F_A, prankA, y.data());
        for (int i = 0; i < prankA; ++i) u[i] = y[i];
        solve_upper(F_A, prankA, u.data());
    }
    void second_lagrange(int prankA, int t, const Vec& p_gn, Vec& v) override {
        ensure_JQ1();
        // b = J1' (rx + J p_gn), J1 = JQ1[:, 0:t]
        Vec s(rx);
        for (int c = 0; c < n; ++c) {
            const double* jc = J.col(c);
            double pc = p_gn[c];
            for (int r = 0; r < mt; ++r) s[r] += jc[r] * pc;
        }
        v.assign(t, 0.0);
        for (int i = 0; i < prankA; ++i) v[i] = dot_n(JQ1.col(i), s.data(), mt);
        solve_upper(F_A, prankA, v.data());
    }
    void sub_search_direction(int t, int rankA, int dimA, int dimJ2, int code, const Vec& Ccx, Vec& p, Vec& b,
                              Vec& d) override {
        Vec p1;
        if (code == 1) {
            b.resize(t);
            for (int i = 0; i < t; ++i) b[i] = -Ccx[F_A.p[i]];
            p1 = b;
            solve_upperT(F_A, t, p1.data());
        } else {
            b.resize(t);
            for (int i = 0; i < t; ++i) b[i] = -Ccx[F_A.p[i]];
            F_L11.Qt_mul(b.data());
            Vec dp1(std::max(dimA, 0));
            for (int i = 0; i < dimA; ++i) dp1[i] = b[i];
            solve_upper(F_L11, std::max(dimA, 0), dp1.data());
            // [dp1; zeros(t-dimA)][invperm(F_L11.p)][1:rankA]
            Vec full(t, 0.0);
            for (int i = 0; i < dimA; ++i) full[i] = dp1[i];
            std::vector<int> ip = F_L11.invperm();
            p1.resize(rankA);
            for (int i = 0; i < rankA; ++i) p1[i] = full[ip[i]];
        }
        int np1 = (int)p1.size();
        // d_temp = -J1*p1 - rx   (J1 has rankA columns; code 1: p1 has t == rankA entries)
        d.assign(mt, 0.0);
        for (int c = 0; c < rankA; ++c) {
            const double* jc = JQ1.col(c);
            double pc = p1[c];
            for (int r = 0; r < mt; ++r) d[r] += jc[r] * pc;
        }
        for (int r = 0; r < mt; ++r) d[r] = -d[r] - rx[r];
        F_J2.Qt_mul(d.data());
        int dj = std::max(dimJ2, 0);
        Vec dp2(dj);
        for (int i = 0; i < dj; ++i) dp2[i] = d[i];
        solve_upper(F_J2, dj, dp2.data());
        std::vector<int> ip2 = F_J2.invperm();
        Vec y(np1 + (int)ip2.size());
        for (int i = 0; i < np1; ++i) y[i] = p1[i];
        for (size_t i = 0; i < ip2.size(); ++i) y[np1 + i] = (ip2[i] < dj) ? dp2[ip2[i]] : 0.0;
        F_A.Q_mul(y.data());
        p = y;
    }
    void subspace_rhs(int t, const Vec& Ccx, Vec& b) override {
        ensure_JQ1();
        b.resize(t);
        for (int i = 0; i < t; ++i) b[i] = -Ccx[F_A.p[i]];
        F_L11.Qt_mul(b.data());
    }
    void subspace_d(int rankA, int dimA, int rankJ2, const Vec& b, Vec& d) override {
        d.assign(mt, 0.0);
        if (rankA <= 0) {
            for (int r = 0; r < mt; ++r) d[r] = -rx[r];
        } else {
            Vec dp1(std::max(dimA, 0));
            for (int i = 0; i < dimA; ++i) dp1[i] = b[i];
            solve_upper(F_L11, std::max(dimA, 0), dp1.data());
            // p1 = P[1:rankA,1:rankA] * [dp1; zeros] : P[p[j], j] = 1
            Vec p1(rankA, 0.0);
            for (int j = 0; j < rankA; ++j) {
                int r = F_L11.p[j];
                if (r < rankA) p1[r] += (j < dimA) ? dp1[j] : 0.0;
            }
            for (int c = 0; c < rankA; ++c) {
                const double* jc = JQ1.col(c);
                double pc = p1[c];
                for (int r = 0; r < mt; ++r) d[r] += jc[r] * pc;
            }
            for (int r = 0; r < mt; ++r) d[r] = -(rx[r] + d[r]);
        }
        if (rankJ2 > 0) F_J2.Qt_mul(d.data());
    }
    void products(const Vec& p, int t, Vec& Jp, Vec& Ap, Vec& active_Ap) override {
        Jp.assign(mt, 0.0);
        for (int c = 0; c < n; ++c) {
            const double* jc = J.col(c);
            double pc = p[c];
            if (pc == 0.0) continue;
            for (int r = 0; r < mt; ++r) Jp[r] += jc[r] * pc;
        }
        // A * p for every row, columns outermost (A is column major): per row the same summation order
        // c = 0..n-1 as the row-wise dot product of the reference
        Ap.assign(l, 0.0);
        for (int c = 0; c < n; ++c) {
            double pc = p[c];
            for (int r = 0; r < l; ++r) Ap[r] += A(r, c) * pc;
        }
        active_Ap.assign(t, 0.0);
        for (int c = 0; c < n; ++c) {
            double pc = p[c];
            for (int r = 0; r < t; ++r) active_Ap[r] += CA(r, c) * pc;
        }
    }
    double At_c_norm(int t, const Vec& Ccx) override {
        if (!CA.rows) return 0.0;
        Vec v(n, 0.0);
        for (int j = 0; j < n; ++j)
            for (int i = 0; i < CA.rows; ++i) v[j] += CA(i, j) * Ccx[i];
        (void)t;
        return normv(v);
    }
};

class LargeSolver {
public:
    LargeOps& ops;
    LargeOptions opt;
    int n, l, q, mt;
    long long m;

    // the matrix-sized state lives in the backend; here: vectors and scalars
    HostSmall* own_small = nullptr;
    SmallBackend* sb = nullptr;
    Vec rx;     // r~ (mt)
    Vec cx;     // l
    Vec gradf;
    Vec K[4];
    WorkingSetL W;
    ConstraintL C;
    FactorInfo F_A, F_L11, F_J2;
    int n_new_point = 0, n_res_eval = 0;

    // backend == nullptr: host memory (CPU tests); the product passes its device backend
    LargeSolver(LargeOps& o, const LargeOptions& op, SmallBackend* backend = nullptr) : ops(o), opt(op) {
        n = o.n; l = o.l; q = o.q; m = o.m; mt = n + 1;
        if (backend) sb = backend;
        else { own_small = new HostSmall(o); sb = own_small; }
    }
    ~LargeSolver() { delete own_small; }
    LargeSolver(const LargeSolver&) = delete;
    LargeSolver& operator=(const LargeSolver&) = delete;

    // ---- small helpers ------------------------------------------------------------------
    void check(int rc) { if (rc != 0) throw std::runtime_error("LargeOps failure"); }

    // EF:34-52 in two halves.  do_eval_point: r, c, A at x and the two m-sized quantities of the termination test
    // (gradf = J'r, returned ||r||^2).  do_factor: the compressed problem [J~ | r~] of that point -- called only when
    // the iteration continues from it, after which gradf / ||r||^2 are re-derived from the compressed problem so that
    // every quantity of an iteration comes from one and the same factorisation.
    double do_eval_point(const Vec& x) { ProfScope prof_(0);
        double rr = 0.0;
        check(sb->new_point_eval(x.data(), gradf.data(), &rr, cx.data()));
        ++n_new_point;
        cur_rr = rr;
        return rr;
    }
    double do_factor() { ProfScope prof_(0);
        check(sb->new_point_compress(rx.data(), gradf.data()));
        cur_rr = dotv(rx, rx);
        return cur_rr;
    }
    double cur_rr = 0.0;   // ||r||^2 at the point of the last do_eval_point
    void gather_active() {   // C.cx = cx[active], C.A = A[active, :]
        int t = W.t;
        C.cx.resize(t);
        for (int i = 0; i < t; ++i) C.cx[i] = cx[W.active[i] - 1];
        sb->gather_active(W.active.data(), t);
    }
    void evaluate_scaling() {   // structures.jl:160-178
        int t = W.t;
        C.diag_scale.assign(t, 0.0);
        Vec rown(t, 0.0);
        sb->evaluate_scaling(t, C.scaling, rown.data());
        for (int i = 0; i < t; ++i) {
            double row_i = rown[i];
            C.diag_scale[i] = row_i;
            if (C.scaling) {
                if (fabs(row_i) < EPS) row_i = 1.0;
                C.cx[i] = C.cx[i] / row_i;
                C.diag_scale[i] = 1.0 / row_i;
            }
        }
    }
    void factor_A() { sb->factor_A(W.t, F_A); }          // F_A = qr(C.A', ColumnNorm())
    void factor_L11() { sb->factor_L11(F_L11); }          // F_L11 = qr(F_A.R', ColumnNorm())

    static void need_nonzero_diag(const FactorInfo& F, int k, const char* what) {   // LAPACK trtrs: SingularException
        for (int i = 0; i < k; ++i)
            if (F.diag(i) == 0.0) throw WouldThrow{what};
    }

    // EF:116-153.  The reference's BoundsError / DimensionMismatch / SingularException situations depend on sizes and
    // on diag(R) only: decided here, the backend then runs the arithmetic.
    void sub_search_direction(int t, int rankA, int dimA, int dimJ2, int code, Vec& p, Vec& b, Vec& d) {
        int np1;
        if (code == 1) {
            // LowerTriangular(F_A.R') \ b : R' is t x min(n,t); the reference solve needs it square
            if (F_A.k < t) throw WouldThrow{"DimensionMismatch in L11 solve"};
            need_nonzero_diag(F_A, t, "SingularException (lower)");
            np1 = t;
        } else if (code == -1) {
            if (dimA > t || dimA > F_L11.k) throw WouldThrow{"BoundsError R11[1:dimA,1:dimA]"};
            need_nonzero_diag(F_L11, std::max(dimA, 0), "SingularException (upper)");
            if (t - dimA < 0) throw WouldThrow{"negative zeros() length"};
            // [dp1; zeros(t - dimA)][invperm(F_L11)] indexes a t-vector with a permutation of length min(n, t):
            // legal in Julia unless the permutation is the longer one
            if (F_L11.cols > t) throw WouldThrow{"BoundsError in invperm indexing"};
            if (rankA > t) throw WouldThrow{"BoundsError [1:rankA]"};
            np1 = rankA;
        } else {
            throw WouldThrow{"sub_search_direction: code"};
        }
        // d_temp = -J1*p1 - rx   (J1 has rankA columns; code 1: p1 has t == rankA entries)
        if (np1 != rankA) throw WouldThrow{"DimensionMismatch J1*p1"};
        if (dimJ2 > F_J2.k) throw WouldThrow{"BoundsError R22[1:dimJ2,1:dimJ2]"};
        if (dimJ2 > mt) throw WouldThrow{"BoundsError d[1:dimJ2]"};
        int dj = std::max(dimJ2, 0);
        need_nonzero_diag(F_J2, dj, "SingularException (upper)");
        int tail = (code == 1) ? (n - t - dimJ2) : (n - rankA - dimJ2);
        if (tail < 0) throw WouldThrow{"negative zeros() length"};
        int k2 = dj + tail;   // length of [dp2; zeros]
        if (F_J2.cols != k2) {
            // indexing a k2-vector with a permutation of another length: BoundsError unless shorter and in range
            for (int j = 0; j < F_J2.cols; ++j) if (j >= k2) throw WouldThrow{"BoundsError p2 permutation"};
        }
        if (np1 + F_J2.cols != n) throw WouldThrow{"DimensionMismatch in Q1*[p1;p2]"};
        sb->sub_search_direction(t, rankA, dimA, dimJ2, code, C.cx, p, b, d);
    }

    // EF:206-234
    void gn_search_direction(int rankA, int t, IterL& it, Vec& p_gn) { ProfScope prof_(5);
        int code = (rankA == t) ? 1 : -1;
        sb->factor_J2(rankA, F_J2);
        int rankJ2 = pseudo_rank(F_J2, opt.eps_rank);
        Vec b, d;
        sub_search_direction(t, rankA, rankA, rankJ2, code, p_gn, b, d);
        it.rankA = rankA;
        it.rankJ2 = rankJ2;
        it.dimA = rankA;
        it.dimJ2 = rankJ2;
        it.b_gn = b;
        it.d_gn = d;
    }

    // EF:461-508
    void first_lagrange_mult_estimate(Vec& lam, IterL& it) { ProfScope prof_(6);
        int t = W.t;
        std::vector<int> inv_p = F_A.invperm();
        int prankA = pseudo_rank(F_A, opt.eps_rank);
        need_nonzero_diag(F_A, prankA, "SingularException (upper)");
        Vec v, u;
        sb->first_lagrange(prankA, t, gradf, C.cx, v, u, it.grad_res);
        lam.resize(t);
        for (int i = 0; i < t; ++i) lam[i] = v[inv_p[i]] + u[inv_p[i]];
        if (C.scaling)
            for (int i = 0; i < t; ++i) lam[i] = lam[i] * C.diag_scale[i];
    }

    // EF:514-537
    void second_lagrange_mult_estimate(Vec& lam, const Vec& p_gn, int t) { ProfScope prof_(7);
        int prankA = pseudo_rank(F_A, SQRT_EPS);
        if (prankA > t) throw WouldThrow{"BoundsError b[1:prankA]"};
        need_nonzero_diag(F_A, prankA, "SingularException (upper)");
        Vec v;
        sb->second_lagrange(prankA, t, p_gn, v);
        std::vector<int> ip = F_A.invperm();
        lam.resize(t);
        for (int i = 0; i < t; ++i) lam[i] = v[ip[i]];
        if (C.scaling)
            for (int i = 0; i < t; ++i) lam[i] = lam[i] * C.diag_scale[i];
    }

    // EF:540-564
    void minmax_lagrangian_mult(const Vec& lam, double& sigmin, double& lam_abs_max) {
        sigmin = INFINITY;
        lam_abs_max = 0.0;
        if (W.t > W.q) {
            for (double v : lam) lam_abs_max = fmax(lam_abs_max, fabs(v));
            for (int i = W.q; i < W.t; ++i) {
                double row = C.scaling ? (1.0 / C.diag_scale[i]) : C.diag_scale[i];
                double li = lam[i];
                if (li * row <= -SQRT_EPS && li < sigmin) sigmin = li;
            }
        }
    }

    // EF:574-603 : returns a 1-based position (0 = none)
    int check_constraint_deletion(const Vec& lam, double grad_res) {
        int t = W.t;
        double lam_max = 1.0;
        if (!lam.empty()) {
            lam_max = 0.0;
            for (double v : lam) lam_max = fmax(lam_max, fabs(v));
        }
        double sq_rel = SQRT_EPS * lam_max;
        int s = 0;
        if (t > W.q) {
            double e = sq_rel;
            for (int i = W.q + 1; i <= t; ++i) {
                double row_i = C.scaling ? (1.0 / C.diag_scale[i - 1]) : C.diag_scale[i - 1];
                double v = row_i * lam[i - 1];
                if (v <= sq_rel && v <= e) { e = v; s = i; }
            }
            if (grad_res > -e * 10.0) s = 0;
        }
        return s;
    }

    // EF:608-650
    bool evaluate_violated_constraints(int index_alpha_upp) { ProfScope prof_(12);
        const double eps_ = SQRT_EPS, delta = 0.1;
        int bnd = std::min(W.l, n);
        bool added = false;
        int swaps = 0;
        if (W.l > W.t) {
            int i = 1;
            while (i <= W.l - W.t) {
                int k = W.inactive[i - 1];
                if (cx[k - 1] < eps_ || (k == index_alpha_upp && cx[k - 1] < delta)) {
                    if (W.t >= bnd) {
                        int worst_k = 0;
                        double worst_val = -INFINITY;
                        for (int j = W.q + 1; j <= W.t; ++j) {
                            int jj = W.active[j - 1];
                            if (cx[jj - 1] > worst_val) { worst_val = cx[jj - 1]; worst_k = j; }
                        }
                        if (worst_k > 0 && worst_val > cx[k - 1]) {
                            if (++swaps > 4 * W.l + 16) throw WouldHang{"evaluate_violated_constraints swap cycle"};
                            W.remove_constraint(worst_k);
                        } else {
                            ++i;
                            continue;
                        }
                    }
                    W.add_constraint(i);
                    added = true;
                } else {
                    ++i;
                }
            }
        }
        return added;
    }

    // EF:686-795 (first-order deletion detour skipped: it is always reverted, SURVEY.md T3)
    void update_working_set(IterL& it, Vec& p_gn) { ProfScope prof_(8);
        Vec lam;
        factor_A();
        first_lagrange_mult_estimate(lam, it);
        int s = check_constraint_deletion(lam, it.grad_res);
        if (s != 0) {
            // surviving side effects of the reverted branch (EF:742-745)
            it.index_del = 0;
            it.dele = false;
            if (C.scaling) {
                sb->rebuild_scaled_rows(W.active.data(), W.t, C.diag_scale.data());
                factor_A();
            }
        }
        int rankA = pseudo_rank(F_A, opt.eps_rank);
        factor_L11();
        gn_search_direction(rankA, W.t, it, p_gn);
        // second-order branch (EF:767-791)
        long long mn = std::min<long long>(m, (long long)(n - rankA));
        if (!(W.t != rankA || (long long)it.rankJ2 != mn)) {
            second_lagrange_mult_estimate(lam, p_gn, W.t);
            int s2 = check_constraint_deletion(lam, 0.0);
            if (s2 != 0) {
                int index_s2 = W.active[s2 - 1];
                lam.erase(lam.begin() + (s2 - 1));
                C.diag_scale.erase(C.diag_scale.begin() + (s2 - 1));
                C.cx.erase(C.cx.begin() + (s2 - 1));
                W.remove_constraint(s2);
                it.dele = true;
                it.index_del = index_s2;
                sb->remove_active_row(s2 - 1);
                factor_A();
                rankA = pseudo_rank(F_A, opt.eps_rank);
                factor_L11();
                gn_search_direction(rankA, W.t, it, p_gn);
            }
        }
        it.lam = lam;
    }

    // EF:826-859
    void init_working_set(IterL& step) {
        const double delta = 0.1, eps_ = 0.01;
        for (int i = 0; i < 4; ++i) K[i].assign(l, delta);
        step.w.assign(l, 0.0);
        for (int i = 0; i < l; ++i) step.w[i] = fmin(fabs(cx[i]) + eps_, delta);
        W.q = q; W.l = l;
        W.active.assign(l, 0);
        W.inactive.assign(std::max(l - q, 0), 0);
        int t = q, lmt = 0;
        for (int i = 0; i < q; ++i) W.active[i] = i + 1;
        for (int i = q + 1; i <= l; ++i) {
            if (cx[i - 1] <= 0.0) { ++t; W.active[t - 1] = i; }
            else { ++lmt; W.inactive[lmt - 1] = i; }
        }
        W.t = t;
        step.t = t;
    }

    // ---- EF:864-1176 subspace dimension heuristics ---------------------------------------
    static double g1(const Vec& v, int i) {
        if (i < 1 || i > (int)v.size()) throw WouldThrow{"BoundsError in subspace heuristics"};
        return v[i - 1];
    }
    int subspace_min_previous_step(const Vec& tau, const Vec& rho, double rho_prk, double c1, int pseudo_rk,
                                   int previous_dimR, double progress, double predicted_linear_progress,
                                   double prelin_previous_dim, double previous_alpha) {
        const double stepb = 2e-1, pgb1 = 3e-1, pgb2 = 1e-1, predb = 7e-1, rlenb = 2.0, c2 = 1e2;
        if (previous_alpha < stepb && progress <= pgb1 * predicted_linear_progress * predicted_linear_progress &&
            progress <= pgb2 * prelin_previous_dim * prelin_previous_dim) {
            int dim = std::max(1, previous_dimR - 1);
            if (previous_dimR > 1 && g1(rho, dim) > c1 * rho_prk) return dim;
        }
        int dim = previous_dimR;
        int suggested;
        if (previous_dimR < (int)tau.size() &&
            ((g1(rho, dim) > predb * rho_prk && rlenb * g1(tau, dim) < g1(tau, dim + 1)) ||
             (c2 * g1(tau, dim) < g1(tau, dim + 1)))) {
            suggested = dim;
        } else {
            int i1 = previous_dimR - 1;
            if (i1 <= 0) {
                suggested = pseudo_rk;
            } else {
                suggested = pseudo_rk;
                bool found = false;
                for (int i = i1; i <= previous_dimR; ++i)
                    if (g1(rho, i) > predb * rho_prk) {
                        if (!found || i < suggested) suggested = i;
                        found = true;
                    }
            }
        }
        return suggested;
    }
    static int gn_previous_step(const Vec& tau, double tau_prk, int mindim, const Vec& rho, double rho_prk, int prank) {
        const double tau_max = 2e-1, rho_min = 5e-1;
        int pm1 = prank - 1;
        if (mindim > pm1) return mindim;
        int k = pm1;
        while ((tau[k - 1] >= tau_max * tau_prk || rho[k - 1] <= rho_min * rho_prk) && k > mindim) --k;
        return (k > mindim) ? k : std::max(mindim, pm1);
    }
    // EF:1041-1113 ; R = factor whose diagonal is used, y = right-hand side
    int determine_solving_dim(int previous_dimR, int rankR, double predicted_linear_progress, double obj_progress,
                              double prelin_previous_dim, const FactorInfo& Rf, const Vec& y, double previous_alpha,
                              bool restart) {
        const double c1 = 0.1;
        int newdim = rankR, mindim = 1;
        if (rankR > 0) {
            if (rankR > (int)y.size()) throw WouldThrow{"BoundsError in determine_solving_dim"};
            Vec sd(rankR), rh(rankR);
            sd[0] = fabs(y[0]);
            rh[0] = fabs(y[0] / Rf.diag(0));
            for (int i = 1; i < rankR; ++i) {
                sd[i] = y[i];
                rh[i] = y[i] / Rf.diag(i);
                rh[i] = sqrt(rh[i - 1] * rh[i - 1] + rh[i] * rh[i]);
                sd[i] = sqrt(sd[i - 1] * sd[i - 1] + sd[i] * sd[i]);
            }
            double nrm_sd = sd[rankR - 1], nrm_rh = rh[rankR - 1];
            double dsum = 0.0, psimax = 0.0;
            for (int i = 0; i < rankR; ++i) {
                dsum += sd[i] * sd[i];
                double psi_ = sqrt(dsum) * fabs(Rf.diag(i));
                if (psi_ > psimax) { psimax = psi_; mindim = i + 1; }
            }
            if (!restart) {
                int suggested;
                if (previous_dimR == rankR || previous_dimR <= 0)
                    suggested = gn_previous_step(sd, nrm_sd, mindim, rh, nrm_rh, rankR);
                else
                    suggested = subspace_min_previous_step(sd, rh, nrm_rh, c1, rankR, previous_dimR, obj_progress,
                                                           predicted_linear_progress, prelin_previous_dim,
                                                           previous_alpha);
                newdim = std::max(mindim, suggested);
            } else {
                newdim = std::max(0, std::min(rankR, previous_dimR));
            }
        }
        return newdim;
    }
    // EF:1118-1176
    void choose_subspace_dimensions(double rx_sum, double active_cx_sum, int t, int rankJ2, int rankA, const Vec& b,
                                    const IterL& prev, bool restart, int& dimA, int& dimJ2) {
        const double alpha_low = 0.2;
        double previous_alpha = prev.alpha;
        int previous_dimA;
        Vec d;
        if (rankA <= 0) {
            dimA = 0;
            previous_dimA = 0;
        } else {
            previous_dimA = abs(prev.dimA) + t - prev.t;
            double nrm_b_asprev = norm_range(b, previous_dimA);
            double nrm_b = normv(b);
            double constraint_progress = prev.cx_sum - active_cx_sum;
            dimA = determine_solving_dim(previous_dimA, rankA, nrm_b, constraint_progress, nrm_b_asprev, F_L11, b,
                                         previous_alpha, restart);
            if (dimA > F_L11.k || dimA > (int)b.size()) throw WouldThrow{"BoundsError R11[1:dimA]"};
            need_nonzero_diag(F_L11, std::max(dimA, 0), "SingularException (upper)");
            if (rankA - dimA < 0) throw WouldThrow{"negative zeros() length"};
            if (rankA > F_L11.cols) throw WouldThrow{"BoundsError in F_L11.P[1:rankA,1:rankA]"};
        }
        sb->subspace_d(rankA, dimA, rankJ2, b, d);
        int previous_dimJ2 = abs(prev.dimJ2) + prev.t - t;
        double nrm_d_asprev = norm_range(d, previous_dimJ2);
        double nrm_d = normv(d);
        double residual_progress = prev.rx_sum - rx_sum;
        dimJ2 = determine_solving_dim(previous_dimJ2, rankJ2, nrm_d, residual_progress, nrm_d_asprev, F_J2, d,
                                      previous_alpha, restart);
        if (!restart && previous_alpha >= alpha_low) {
            dimA = std::max(dimA, previous_dimA);
            dimJ2 = std::max(dimJ2, previous_dimJ2);
        }
    }

    // EF:943-1030
    int check_gn_direction(double b1nrm, double d1nrm, double d1nrm_as_km1, double dnrm, double active_c_sum,
                           int iter_number, int rankA, bool restart, bool constraint_added, bool constraint_deleted,
                           const Vec& lam, const IterL& km1, double& beta_k) {
        const double delta = 1e-1, c1 = 0.5, c2 = 0.1, c3 = 4.0, c4 = 10.0, c5 = 0.05;
        beta_k = sqrt(d1nrm * d1nrm + b1nrm * b1nrm);
        int method_code = 1;
        bool newton_or_restart = km1.code == 2 || restart;
        bool first_iter = iter_number == 0;
        bool submin_prev = km1.code == -1;
        bool add_or_del = constraint_added || constraint_deleted;
        bool conv_lower = beta_k < c1 * km1.beta;
        bool progress_not_close = (km1.progress > c2 * km1.predicted_reduction) && (dnrm <= c3 * beta_k);
        if (newton_or_restart || (!first_iter && (submin_prev || !(add_or_del || conv_lower || progress_not_close)))) {
            method_code = -1;
            double nonlin_k = sqrt(d1nrm * d1nrm + active_c_sum);
            double nonlin_km1 = sqrt(d1nrm_as_km1 * d1nrm_as_km1 + active_c_sum);
            bool to_reduce = false;
            if (W.q < W.t) {
                bool any1 = false, any2 = false;
                for (int i = W.q; i < W.t; ++i) {
                    double row = C.scaling ? (1.0 / C.diag_scale[i]) : C.diag_scale[i];
                    if (lam[i] * row >= -SQRT_EPS) any1 = true;
                    if (lam[i] < 0) any2 = true;
                }
                to_reduce = to_reduce || (any1 && any2);
            }
            if (W.l - W.t > 0) {
                for (int i = 0; i < W.l - W.t; ++i)
                    if (cx[W.inactive[i] - 1] < delta) to_reduce = true;
            }
            bool newton_previously = km1.code == 2 && !constraint_deleted;
            bool cond4 = active_c_sum > c2;
            bool cond5 = constraint_deleted || constraint_added || to_reduce || (W.t == n && W.t == rankA);
            double eps_ = fmax(1e-2, 10.0 * EPS);
            bool cond6 = (!((W.l == W.q) || (rankA <= W.t))) &&
                         (!((beta_k < eps_ * dnrm) || (b1nrm < eps_ && m == (long long)(n - W.t))));
            if (newton_previously || !(cond4 || cond5 || cond6)) {
                bool cond7 = (km1.alpha < c5 && nonlin_km1 < c2 * nonlin_k) || m == (long long)(n - W.t);
                bool cond8 = !(dnrm <= c4 * beta_k);
                if (newton_previously || cond7 || cond8) method_code = 2;
            }
        }
        return method_code;
    }

    // EF:1191-1291
    int search_direction_analys(const IterL& prev, IterL& cur, int iter_number, double active_cx_sum, const Vec& p_gn) { ProfScope prof_(9);
        double rx_sum = dotv(rx, rx);
        double nrm_b1_gn = norm_range(cur.b_gn, cur.dimA);
        int rankA = cur.rankA;
        double nrm_d_gn = normv(cur.d_gn);
        double nrm_d1_gn = norm_range(cur.d_gn, cur.dimJ2);
        int rankJ2 = cur.rankJ2;
        int prev_dimJ2m1 = prev.dimJ2 + prev.t - W.t - 1;
        double nrm_d1_asprev = norm_range(cur.d_gn, prev_dimJ2m1);
        bool restart = cur.restart;
        int error_code = 0;
        double beta;
        int method_code = check_gn_direction(nrm_b1_gn, nrm_d1_gn, nrm_d1_asprev, nrm_d_gn, active_cx_sum, iter_number,
                                             rankA, restart, cur.add, cur.dele, cur.lam, prev, beta);
        int dimA, dimJ2;
        Vec p, b, d;
        if (method_code == 1) {
            dimA = rankA; dimJ2 = rankJ2;
            p = p_gn; b = cur.b_gn; d = cur.d_gn;
        } else if (method_code == -1) {
            sb->subspace_rhs(W.t, C.cx, b);
            choose_subspace_dimensions(rx_sum, active_cx_sum, W.t, rankJ2, rankA, b, prev, restart, dimA, dimJ2);
            sub_search_direction(W.t, rankA, dimA, dimJ2, method_code, p, b, d);
            if (dimA == rankA && dimJ2 == rankJ2) method_code = 1;
        } else {   // 2: Newton requested, but second derivatives are off in this regime (EF:2658) -> EF:1272-1276
            p = p_gn; b = cur.b_gn; d = cur.d_gn;
            dimA = rankA; dimJ2 = rankJ2;
            error_code = -4;
        }
        cur.b_gn = b;
        cur.d_gn = d;
        cur.dimA = dimA;
        cur.dimJ2 = dimJ2;
        cur.code = method_code;
        cur.speed = beta / prev.beta;
        cur.beta = beta;
        cur.p = p;
        return error_code;
    }

    // ---- merit function, penalty weights (EF:1307-1629) -----------------------------------
    double penalty_part(const Vec& c, const Vec& w) const {
        double pen = 0.0;
        for (int i = 0; i < W.t; ++i) {
            int j = W.active[i] - 1;
            pen += w[j] * c[j] * c[j];
        }
        for (int i = 0; i < W.l - W.t; ++i) {
            int j = W.inactive[i] - 1;
            if (c[j] < 0.0) pen += w[j] * c[j] * c[j];
        }
        return pen;
    }
    // ||r(x + alpha p)||^2 of the trial points of the current direction: the reference evaluates the same point several
    // times (EF:2000 vs 2005, the accepted step again at EF:2281); every evaluation is an m-sized kernel (+ an all-reduce
    // when row-sharded), so the values are kept for the life of the direction.  The kernels compute this sum with the
    // same arithmetic whether or not the model coefficients are requested, so a cached value is the value.
    double ls_alpha[8], ls_rs[8];
    int ls_cached = 0, ls_next = 0;
    void ls_cache_reset() { ls_cached = 0; ls_next = 0; }
    bool ls_cache_get(double alpha, double& rs) const {
        for (int i = 0; i < ls_cached; ++i)
            if (ls_alpha[i] == alpha) { rs = ls_rs[i]; return true; }
        return false;
    }
    void ls_cache_put(double alpha, double rs) {
        double dummy;
        if (ls_cache_get(alpha, dummy)) return;
        ls_alpha[ls_next] = alpha; ls_rs[ls_next] = rs;
        ls_next = (ls_next + 1) % 8;
        if (ls_cached < 8) ++ls_cached;
    }
    double res_sq_cached(double alpha) {
        double rs;
        ++n_res_eval;
        if (ls_cache_get(alpha, rs)) return rs;
        check(ops.res_sq(alpha, &rs));
        ls_cache_put(alpha, rs);
        return rs;
    }
    // psi(x + alpha p) with the direction fixed by ops.set_direction (EF:1307-1340)
    double psi(const Vec& x, double alpha, const Vec& p, const Vec& w, Vec& cbuf) {
        Vec xn(n);
        for (int j = 0; j < n; ++j) xn[j] = x[j] + alpha * p[j];
        double rs = res_sq_cached(alpha);
        check(ops.cons(xn.data(), cbuf.data()));
        return 0.5 * (rs + penalty_part(cbuf, w));
    }
    void assort(const Vec& w, int t) {   // EF:1344-1360
        for (int i = 0; i < t; ++i)
            for (int ii = 0; ii < 4; ++ii) {
                int k = W.active[i] - 1;
                if (w[k] > K[ii][k]) {
                    for (int j = 3; j > ii; --j) K[j][k] = K[j - 1][k];
                    K[ii][k] = w[k];
                }
            }
    }
    // EF:1374-1423
    static void min_norm_w(int ctrl, Vec& w, const Vec& w_old, Vec y, double tau, std::vector<int>& pos_index,
                           int nb_pos) {
        w = w_old;
        if (nb_pos > 0) {
            double y_sum = 0.0;
            for (double v : y) y_sum += v * v;
            double y_norm = sqrt(y_sum);
            if (y_norm != 0.0)
                for (double& v : y) v /= y_norm;
            double tau_new = tau, s = 0.0;
            int n_runch = nb_pos;
            bool terminated = false;
            while (!terminated) {
                tau_new -= s;
                double ymax = 0.0;
                for (double v : y) ymax = fmax(ymax, fabs(v));
                double c = (ymax <= EPS) ? 1.0 : tau_new / y_sum;
                y_sum = 0.0; s = 0.0;
                int i_stop = n_runch;
                int k = 1;
                while (k <= n_runch) {
                    int i = pos_index[k - 1] - 1;
                    double buff = c * y[k - 1] * y_norm;
                    if (buff >= w_old[i]) {
                        w[i] = buff;
                        y_sum += y[k - 1] * y[k - 1];
                        ++k;
                    } else {
                        s += w_old[i] * y[k - 1] * y_norm;
                        --n_runch;
                        for (int j = k; j <= n_runch; ++j) {
                            pos_index[j - 1] = pos_index[j];
                            y[j - 1] = y[j];
                        }
                    }
                }
                y_sum *= y_norm * y_norm;
                terminated = (n_runch <= 0) || (ctrl == 2) || (i_stop == n_runch);
            }
        }
    }
    // EF:1429-1497
    Vec euclidean_norm_weight_update(const Vec& vA, const Vec& cxs, int t, double mu, int dimA, const Vec& previous_w) {
        Vec w = previous_w;
        if (t != 0) {
            Vec z(t);
            for (int i = 0; i < t; ++i) z[i] = vA[i] * vA[i];
            Vec w_old = K[3];
            double ztw = 0.0;
            for (int i = 0; i < t; ++i) ztw += z[i] * w_old[W.active[i] - 1];
            std::vector<int> pos_index(t, 0);
            if (ztw >= mu && dimA < t) {
                Vec y(t, 0.0);
                int nb_pos = 0;
                double gamma = 0.0;
                for (int i = 0; i < t; ++i) {
                    int k = W.active[i];
                    double y_elem = vA[i] * (vA[i] + cxs[k - 1]);
                    if (y_elem > 0) { ++nb_pos; pos_index[nb_pos - 1] = k; y[nb_pos - 1] = y_elem; }
                    else gamma -= y_elem * w_old[k - 1];
                }
                min_norm_w(2, w, w_old, y, gamma, pos_index, nb_pos);
            } else if (ztw < mu && dimA < t) {
                Vec e(t, 0.0);
                int nb_pos = 0;
                double tau = mu;
                for (int i = 0; i < t; ++i) {
                    int k = W.active[i];
                    double e_elem = -vA[i] * cxs[k - 1];
                    if (e_elem > 0) { ++nb_pos; pos_index[nb_pos - 1] = k; e[nb_pos - 1] = e_elem; }
                    else tau -= e_elem * w_old[k - 1];
                }
                min_norm_w(2, w, w_old, e, tau, pos_index, nb_pos);
            } else if (ztw < mu && dimA == t) {
                for (int i = 0; i < t; ++i) pos_index[i] = W.active[i];
                min_norm_w(1, w, w_old, z, mu, pos_index, t);
            }
            assort(w, t);
        }
        return w;
    }
    // EF:1545-1629 ; Jp / rx enter only through norms and one dot (compressed vectors)
    Vec penalty_weight_update(const Vec& w_old, const Vec& Jp, Vec Ap, const Vec& rxv, Vec cxs, int dimA,
                              double& dpsi0) {
        const double delta = 0.25;
        int t = W.t;
        if (dimA < 0 || dimA > W.l) throw WouldThrow{"active[1:dimA] out of range"};
        double nrm_Ap = sqrt(dotv(Ap, Ap));
        double nrm_cx = 0.0;
        for (int i = 0; i < dimA; ++i) {
            if (W.active[i] == 0) throw WouldThrow{"cx[0]"};
            nrm_cx = fmax(nrm_cx, fabs(cxs[W.active[i] - 1]));
        }
        double nrm_Jp = sqrt(dotv(Jp, Jp));
        double nrm_rx = sqrt(dotv(rxv, rxv));
        double jr = 0.0;   // dot(Jp/nrm_Jp, rx/nrm_rx)
        {
            double sj = (nrm_Jp != 0) ? nrm_Jp : 1.0, sr = (nrm_rx != 0) ? nrm_rx : 1.0;
            for (int r = 0; r < (int)Jp.size(); ++r) jr += (Jp[r] / sj) * (rxv[r] / sr);
        }
        if (nrm_Ap != 0)
            for (double& v : Ap) v /= nrm_Ap;
        if (nrm_cx != 0)
            for (double& v : cxs) v /= nrm_cx;
        double Jp_rx = jr * nrm_Jp * nrm_rx;
        double AtwA = 0.0, BtwA = 0.0;
        for (int i = 0; i < dimA; ++i) {
            int k = W.active[i] - 1;
            AtwA += w_old[k] * Ap[i] * Ap[i];
            BtwA += w_old[k] * Ap[i] * cxs[k];
        }
        AtwA *= nrm_Ap * nrm_Ap;
        BtwA *= nrm_Ap * nrm_cx;
        double rmy = (fabs(Jp_rx + nrm_Jp * nrm_Jp) / delta) - nrm_Jp * nrm_Jp;
        Vec vA(Ap), cs(cxs);
        for (double& v : vA) v *= nrm_Ap;
        for (double& v : cs) v *= nrm_cx;
        Vec w = euclidean_norm_weight_update(vA, cs, t, rmy, dimA, w_old);
        BtwA = 0.0; AtwA = 0.0;
        for (int i = 0; i < t; ++i) {
            int k = W.active[i] - 1;
            AtwA += w[k] * Ap[i] * Ap[i];
            BtwA += w[k] * Ap[i] * cxs[k];
        }
        BtwA *= nrm_Ap * nrm_cx;
        dpsi0 = BtwA + Jp_rx;
        return w;
    }

    // ---- linesearch (EF:1635-2143) --------------------------------------------------------
    // constraint part of `concatenate` (EF:1635-1659): entries m+1..m+l of v
    void concat_c(Vec& v, const Vec& c, const Vec& w) const {
        std::fill(v.begin(), v.end(), 0.0);
        for (int i = 0; i < W.t; ++i) {
            int k = W.active[i] - 1;
            v[k] = sqrt(w[k]) * c[k];
        }
        for (int j = 0; j < W.l - W.t; ++j) {
            int k = W.inactive[j] - 1;
            v[k] = (c[k] > 0) ? 0.0 : sqrt(w[k]) * c[k];
        }
    }
    static double minimize_quadratic(double x1, double y1, double x2, double y2, double x3, double y3) {
        double d1 = y2 - y1, d2 = y3 - y1;
        double s = (x3 - x1) * (x3 - x1) * d1 - (x2 - x1) * (x2 - x1) * d2;
        double qq = 2 * ((x2 - x1) * d2 - (x3 - x1) * d1);
        return x1 - s / qq;
    }
    static double clampd(double u, double lo, double hi) { return (u > hi) ? hi : ((u < lo) ? lo : u); }
    static void minrn(double x1, double y1, double x2, double y2, double x3, double y3, double alpha_min,
                      double alpha_max, double p_max, double& a, double& pa) {
        double eps_ = SQRT_EPS / p_max;
        if (fabs(x1 - x2) < eps_ || fabs(x3 - x1) < eps_ || fabs(x3 - x2) < eps_) { a = 0.0; pa = 0.0; return; }
        double u = minimize_quadratic(x1, y1, x2, y2, x3, y3);
        a = clampd(u, alpha_min, alpha_max);
        double t1 = (a - x1) * (a - x2) * y3 / ((x3 - x1) * (x3 - x2));
        double t2 = (a - x3) * (a - x2) * y1 / ((x1 - x3) * (x1 - x2));
        double t3 = (a - x3) * (a - x2) * y2 / ((x2 - x1) * (x2 - x3));
        pa = t1 + t2 + t3;
    }
    struct Poly {   // Polynomials.jl: trailing zeros chopped, Horner with fma (evalpoly -> muladd)
        std::vector<double> c;
        explicit Poly(std::vector<double> cc) : c(std::move(cc)) {
            while (c.size() > 1 && c.back() == 0.0) c.pop_back();
        }
        double operator()(double x) const {
            double acc = c.back();
            for (int i = (int)c.size() - 2; i >= 0; --i) acc = acc * x + c[i];
            return acc;
        }
        Poly derivative() const {
            if (c.size() <= 1) return Poly({0.0});
            std::vector<double> d(c.size() - 1);
            for (size_t i = 1; i < c.size(); ++i) d[i - 1] = (double)i * c[i];
            return Poly(d);
        }
    };
    static double newton_raphson(double x_min, double Dm, const Poly& ds, const Poly& dds) {
        double alpha = x_min;
        int it = 0;
        double eps_ = 1e-4, error = 1.0;
        while ((error > eps_ || it < 3) && it < 50) {
            double c = dds(alpha);
            if (fabs(c) < EPS) break;
            double h = -ds(alpha) / c;
            alpha += h;
            error = (2 * Dm * h * h) / fabs(c);
            ++it;
        }
        return alpha;
    }
    static double one_root(double c, double d, double a) {
        double arg1 = -c / 2 + sqrt(d), arg2 = -c / 2 - sqrt(d);
        return cbrt(arg1) + cbrt(arg2) - a / 3;
    }
    static void two_roots(double b, double c, double a, double x_min, double& r1, double& r2) {
        double phi = acos(fabs(c / 2) / pow(-b / 3, 1.5));
        if (phi != phi) throw WouldThrow{"DomainError in acos"};
        double t = (c <= 0) ? 2 * sqrt(-b / 3) : -2 * sqrt(-b / 3);
        double b1 = t * cos(phi / 3) - a / 3;
        double b2 = t * cos((phi + 2 * M_PI) / 3) - a / 3;
        double b3 = t * cos((phi + 4 * M_PI) / 3) - a / 3;
        double s[3] = {b1, b2, b3};
        std::sort(s, s + 3);
        if (x_min <= s[1]) { r1 = s[0]; r2 = s[2]; } else { r1 = s[2]; r2 = s[0]; }
    }
    // EF:1739-1783 ; dots: v1v2, v2v2
    static void parameters_rm(double v1v2, double normv2, double x_min, const Poly& ds, const Poly& dds,
                              double& alpha_hat, double& beta_hat) {
        double dds_best = dds(x_min);
        const double eta = 0.1;
        double d = 1.0;
        double h0 = fabs(ds(x_min) / dds_best);
        double Dm = fabs(6 * v1v2 + 12 * x_min * normv2) + 24 * h0 * normv2;
        double hm = fmax(h0, 1.0);
        bool have_beta = false;
        if (dds_best * eta < 2 * Dm * hm) {
            const std::vector<double>& cf = ds.c;
            if (cf.size() < 3) throw WouldThrow{"BoundsError destructuring coeffs(ds)"};
            double a3 = cf[0] / (2 * normv2), a2 = cf[1] / (2 * normv2), a1 = cf[2] / (2 * normv2);
            double b = a2 - (a1 * a1) / 3;
            double c = a3 - a1 * a2 / 3 + 2 * (a1 / 3) * (a1 / 3) * (a1 / 3);
            d = (c / 2) * (c / 2) + (b / 3) * (b / 3) * (b / 3);
            if (d < 0) {
                two_roots(b, c, a1, x_min, alpha_hat, beta_hat);
                have_beta = true;
            } else {
                if (d != d) throw WouldThrow{"NaN discriminant"};
                alpha_hat = one_root(c, d, a1);
            }
        } else {
            alpha_hat = newton_raphson(x_min, Dm, ds, dds);
        }
        if (d >= 0) { beta_hat = alpha_hat; have_beta = true; }
        if (!have_beta) throw WouldThrow{"UndefVarError beta_hat"};
    }
    static void bounds_rm(double alpha_min, double alpha_max, double& alpha, double& sval, const Poly& s) {
        if (alpha != alpha) { sval = s(alpha); return; }
        alpha = fmin(alpha, alpha_max);
        alpha = fmax(alpha, alpha_min);
        sval = s(alpha);
    }
    // EF:1841-1862 with the six dot products given
    static void minrm(const double dd[6] /* v0v0, v0v1, v0v2, v1v1, v1v2, v2v2 */, double x_min, double alpha_min,
                      double alpha_max, double& alpha_hat, double& s_a, double& beta_hat, double& s_b) {
        Poly s({0.5 * dd[0], dd[1], dd[2] + 0.5 * dd[3], dd[4], 0.5 * dd[5]});
        Poly ds = s.derivative();
        Poly dds = ds.derivative();
        parameters_rm(dd[4], dd[5], x_min, ds, dds, alpha_hat, beta_hat);
        s_a = s(alpha_hat);
        s_b = s(beta_hat);
        double alpha_old = alpha_hat;
        bounds_rm(alpha_min, alpha_max, alpha_hat, s_a, s);
        if (alpha_old == beta_hat) {
            beta_hat = alpha_hat;
            s_b = s(alpha_hat);
        } else {
            bounds_rm(alpha_min, alpha_max, beta_hat, s_b, s);
        }
    }
    static bool check_reduction(double psi_alpha, double psi_k, double approx_k, double eta, double diff_psi) {
        const double delta = 0.2;
        if (psi_alpha - approx_k >= eta * diff_psi)
            return !((psi_alpha - psi_k < eta * diff_psi) && (psi_k > delta * psi_alpha));
        return false;
    }

    // the six dot products of coefficients_linesearch + minrm at trial step alpha_k (EF:1665-1689, 1849-1851)
    void ls_dots(const Vec& x, const Vec& p, double alpha_k, const Vec& v1c, const Vec& w, const double sums[3],
                 double dd[6]) {
        double o[4];
        check(ops.ls_coeffs(alpha_k, o));
        ++n_res_eval;
        ls_cache_put(alpha_k, o[0]);
        Vec xn(n), cn(l), v0c(l), vbc(l);
        for (int j = 0; j < n; ++j) xn[j] = x[j] + alpha_k * p[j];
        check(ops.cons(xn.data(), cn.data()));
        concat_c(v0c, cx, w);
        concat_c(vbc, cn, w);
        double c00 = 0, c01 = 0, c02 = 0, c11 = 0, c12 = 0, c22 = 0;
        for (int k = 0; k < l; ++k) {
            double v2 = ((vbc[k] - v0c[k]) / alpha_k - v1c[k]) / alpha_k;
            c00 += v0c[k] * v0c[k]; c01 += v0c[k] * v1c[k]; c02 += v0c[k] * v2;
            c11 += v1c[k] * v1c[k]; c12 += v1c[k] * v2; c22 += v2 * v2;
        }
        dd[0] = sums[0] + c00;
        dd[1] = sums[1] + c01;
        dd[2] = o[1] + c02;
        dd[3] = sums[2] + c11;
        dd[4] = o[2] + c12;
        dd[5] = o[3] + c22;
    }

    // EF:1940-2143
    double linesearch_constrained(const Vec& x, double alpha0, const Vec& p, const Vec& Ap, const Vec& w,
                                  double psi0, double dpsi0, double alpha_low, double alpha_upp, const double sums[3],
                                  bool& gac_error) {
        const double eta = 0.3, tau = 0.25, gamma = 0.4;
        double alpha_min = alpha_low, alpha_max = alpha_upp;
        double alpha_k = fmin(alpha0, alpha_max);
        double alpha_km1 = 0.0, psi_km1 = psi0;
        double p_max = 0.0;
        for (double v : p) p_max = fmax(p_max, fabs(v));
        gac_error = false;
        Vec v1c(l, 0.0), cbuf(l);
        for (int i = 0; i < W.t; ++i) {
            int k = W.active[i] - 1;
            v1c[k] = sqrt(w[k]) * Ap[k];
        }
        for (int j = 0; j < W.l - W.t; ++j) {
            int k = W.inactive[j] - 1;
            v1c[k] = (cx[k] > 0) ? 0.0 : sqrt(w[k]) * Ap[k];
        }
        auto PSI = [&](double a) { return psi(x, a, p, w, cbuf); };
        double dd[6];
        ls_dots(x, p, alpha_k, v1c, w, sums, dd);      // (before psi(alpha_k): its residual sum serves both, EF:2000 / 2005)
        double psi_k = PSI(alpha_k);
        double diff_psi = psi0 - psi_k;
        double x_min = (diff_psi >= 0) ? alpha_k : 0.0;
        double alpha_kp1, pk, beta, pbeta;
        minrm(dd, x_min, alpha_min, alpha_max, alpha_kp1, pk, beta, pbeta);
        if (alpha_kp1 != beta && pbeta < pk && beta <= alpha_k) { alpha_kp1 = beta; pk = pbeta; }
        double alpha_km2 = alpha_km1, psi_km2 = psi_km1;
        alpha_km1 = alpha_k; psi_km1 = psi_k;
        alpha_k = alpha_kp1;
        psi_k = PSI(alpha_k);
        auto shift = [&](double a_new) {
            alpha_km2 = alpha_km1; psi_km2 = psi_km1;
            alpha_km1 = alpha_k; psi_km1 = psi_k;
            alpha_k = a_new;
            psi_k = PSI(alpha_k);
        };
        if ((-diff_psi <= tau * dpsi0 * alpha_km1) || (psi_km1 < gamma * psi0)) {
            diff_psi = psi0 - psi_k;
            bool reduction_likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
            while (reduction_likely) {
                minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, alpha_min, alpha_max, p_max, alpha_kp1, pk);
                shift(alpha_kp1);
                diff_psi = psi0 - psi_k;
                reduction_likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
            }
            if ((psi_km1 - pk >= eta * diff_psi) && (psi_k < psi_km1)) { alpha_km1 = alpha_k; psi_km1 = psi_k; }
        } else {
            diff_psi = psi0 - psi_k;
            if ((-diff_psi <= tau * dpsi0 * alpha_k) || (psi_k < gamma * psi0)) {
                if (psi0 <= psi_km1) {
                    x_min = alpha_k;
                    ls_dots(x, p, alpha_k, v1c, w, sums, dd);
                    minrm(dd, x_min, alpha_min, alpha_max, alpha_kp1, pk, beta, pbeta);
                    if (alpha_kp1 != beta && pbeta < pk && beta <= alpha_k) { alpha_kp1 = beta; pk = pbeta; }
                    alpha_km1 = 0.0;
                    psi_km1 = psi0;
                } else {
                    minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, alpha_min, alpha_max, p_max, alpha_kp1, pk);
                }
                shift(alpha_kp1);
                bool reduction_likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
                while (reduction_likely) {
                    minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, alpha_min, alpha_max, p_max, alpha_kp1, pk);
                    shift(alpha_kp1);
                    reduction_likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
                }
                if ((psi_km1 - pk >= eta * diff_psi) && (psi_k < psi_km1)) { alpha_km1 = alpha_k; psi_km1 = psi_k; }
            } else {
                // goldstein_armijo_step (EF:1893-1923)
                double u = alpha_k;
                bool ex = (p_max * u < SQRT_EPS) || (u <= alpha_min);
                double psi_u = PSI(u);
                while (!ex && (psi_u > psi0 + tau * u * dpsi0)) {
                    u *= 0.5;
                    psi_u = PSI(u);
                    ex = (p_max * u < SQRT_EPS) || (u <= alpha_min);
                }
                alpha_km1 = u;
                gac_error = ex;
            }
        }
        return alpha_km1;
    }

    // EF:2149-2178
    double upper_bound_steplength(const Vec& Ap, int index_del, int& index_alpha_upp) { ProfScope prof_(11);
        double alpha_upper = INFINITY;
        index_alpha_upp = 0;
        int mx = 0;
        for (int v : W.inactive) mx = std::max(mx, abs(v));
        if (!W.inactive.empty() && mx > 0) {
            // g = A * p for every row: the Ap of compute_steplength (same summation order c = 0..n-1 as the row-wise
            // dot product of the reference)
            for (int i = 0; i < W.l - W.t; ++i) {
                int j = W.inactive[i];
                if (j != index_del) {
                    const double g = Ap[j - 1];
                    double a_j = -cx[j - 1] / g;
                    if (cx[j - 1] > 0 && g < 0 && a_j < alpha_upper) { alpha_upper = a_j; index_alpha_upp = j; }
                }
            }
        }
        return fmin(3.0, alpha_upper);
    }

    // EF:2197-2293
    double compute_steplength(IterL& it, const IterL& prev, const Vec& x, Vec& w_out, int& Psi_error) { ProfScope prof_(10);
        const Vec& p = it.p;
        int dimA = it.dimA;
        // Jp (compressed), Ap, active_Ap
        Vec Jp, Ap, active_Ap;
        sb->products(p, W.t, Jp, Ap, active_Ap);
        if (C.scaling)
            for (int r = 0; r < W.t; ++r) active_Ap[r] = active_Ap[r] / C.diag_scale[r];
        Psi_error = 0;
        double alpha;
        if (it.code != 2) {
            double dpsi0;
            Vec w = penalty_weight_update(prev.w, Jp, active_Ap, rx, cx, dimA, dpsi0);
            double rr = dotv(rx, rx);
            double wc = 0.0;
            for (int i = 0; i < W.t; ++i) {
                int k = W.active[i] - 1;
                wc += w[k] * (cx[k] * cx[k]);
            }
            double psi0 = 0.5 * (rr + wc);
            if (dpsi0 >= 0) {
                alpha = 1.0;
                Psi_error = -1;
                it.index_alpha_upp = 0;
            } else {
                int index_alpha_upp;
                double alpha_upp = upper_bound_steplength(Ap, it.index_del, index_alpha_upp);
                double alpha_low = alpha_upp / 3000.0;
                double magfy = (it.rankJ2 < prev.rankJ2) ? 6.0 : 3.0;
                double alpha0 = fmin(fmin(1.0, magfy * prev.alpha), alpha_upp);
                double sums[3];
                check(ops.set_direction(x.data(), p.data(), sums));
                ls_cache_reset();
                bool gac_error;
                alpha = linesearch_constrained(x, alpha0, p, Ap, w, psi0, dpsi0, alpha_low, alpha_upp, sums, gac_error);
                Vec cbuf(l);
                if (gac_error) {
                    double psi_k = psi(x, alpha, p, w, cbuf);
                    // check_derivatives (EF:2295-2322)
                    double psi_ma = psi(x, -alpha, p, w, cbuf);
                    double f = (psi_k - psi0) / alpha, b = (psi0 - psi_ma) / alpha, c = (psi_k - psi_ma) / (2 * alpha);
                    double max_diff = fmax(fmax(fabs(f - c), fabs(f - b)), fabs(b - c));
                    bool inconsistency = fabs(f - dpsi0) > max_diff && fabs(c - dpsi0) > max_diff;
                    Psi_error = inconsistency ? -1 : 0;
                }
                double uppbound = fmin(1.0, alpha_upp);
                double atwa = 0.0;
                for (int i = 0; i < W.t; ++i) atwa += w[W.active[i] - 1] * (active_Ap[i] * active_Ap[i]);
                it.predicted_reduction = uppbound * (-2.0 * dotv(Jp, rx) - uppbound * dotv(Jp, Jp) +
                                                     (2.0 - uppbound * uppbound) * atwa);
                // progress at the accepted step (EF:2281-2287)
                Vec xn(n), cn(l);
                for (int j = 0; j < n; ++j) xn[j] = x[j] + alpha * p[j];
                double rs = res_sq_cached(alpha);
                check(ops.cons(xn.data(), cn.data()));
                double whsum = 0.0;
                for (int i = 0; i < W.t; ++i) {
                    int k = W.active[i] - 1;
                    whsum += w[k] * (cn[k] * cn[k]);
                }
                it.progress = 2 * psi0 - rs - whsum;
                it.index_alpha_upp = (index_alpha_upp != 0 && fabs(alpha - alpha_upp) > 0.1) ? 0 : index_alpha_upp;
            }
            w_out = w;
        } else {
            w_out = prev.w;
            it.index_alpha_upp = 0;
            alpha = 1.0;
        }
        return alpha;
    }

    // EF:2399-2517
    int check_termination_criteria(const IterL& it, const IterL& prev, const Vec& x, double rx_sum, int nb_iter,
                                   int error_code, double delta_time, double sigma_min, double lam_abs_max,
                                   int Psi_error) {
        int exit_code = 0;
        double alfnoi = EPS / (normv(it.p) + EPS);
        bool preliminary = !(it.restart || (it.code == -1 && alfnoi <= 0.25));
        if (preliminary) {
            bool necessary = (!it.dele) && (normv(C.cx) < opt.eps_c) &&
                             (it.grad_res < sqrt(opt.eps_rel) * (1 + normv(gradf)));
            if (W.l - W.t > 0)
                for (int i = 0; i < W.l - W.t; ++i) necessary = necessary && (cx[W.inactive[i] - 1] > 0);
            if (W.t > W.q) {
                double factor = (W.t == 1) ? (1 + rx_sum) : lam_abs_max;
                necessary = necessary && (sigma_min >= opt.eps_rel * factor);
            }
            if (necessary) {
                if (it.dimJ2 > (int)it.d_gn.size()) throw WouldThrow{"BoundsError d_gn[1:dimJ2]"};
                double d1 = 0.0;
                for (int i = 0; i < it.dimJ2; ++i) d1 += it.d_gn[i] * it.d_gn[i];
                double xd = 0.0;
                for (int j = 0; j < n; ++j) xd += (prev.x[j] - x[j]) * (prev.x[j] - x[j]);
                double x_diff = sqrt(xd);
                if (d1 <= rx_sum * opt.eps_rel * opt.eps_rel) exit_code += 10000;
                if (rx_sum <= opt.eps_abs * opt.eps_abs) exit_code += 2000;
                if (x_diff < opt.eps_x * normv(x)) exit_code += 300;
                if (alfnoi > 0.25) exit_code += 40;
                if (exit_code > 0 && W.l - W.t > 0) {
                    int feas = 1;
                    for (int ii = 0; ii < W.l - W.t; ++ii)
                        if (cx[W.inactive[ii] - 1] <= 0.0) { feas = -1; break; }
                    exit_code *= feas;
                }
            }
        }
        if (exit_code == 0) {
            double xd = 0.0;
            for (int j = 0; j < n; ++j) xd += (prev.x[j] - x[j]) * (prev.x[j] - x[j]);
            double x_diff = sqrt(xd);
            double Atcx_nrm = sb->At_c_norm(W.t, C.cx);
            double aps = 0.0;
            for (int i = 0; i < W.t; ++i) { double wv = it.w[W.active[i] - 1]; aps += wv * wv; }
            if (nb_iter >= opt.max_iter) exit_code = -2;
            else if (error_code >= -5 && error_code <= -3) exit_code = error_code;
            else if (it.nb_newton_steps > 5) exit_code = -9;
            else if (Psi_error == -1) exit_code = -6;
            else if (x_diff <= 10.0 * opt.eps_x && Atcx_nrm <= 10.0 * opt.eps_c && aps >= 1.0) exit_code = -10;
            else if (delta_time > 0) exit_code = -11;
        }
        return exit_code;
    }

    static int convert_exit_code(int code) {   // cnls_model.jl:166-178
        if (code > 0) return 1;
        if (code == -2 || code == -11) return code;
        return -1;
    }

    // snapshot copy of an iteration (structures.jl:93-98) given the live sums (T1)
    IterL copy_iter(const IterL& s, double live_rx_sum, double live_cx_sum) const {
        IterL c = s;
        if (s.alias) { c.rx_sum = live_rx_sum; c.cx_sum = live_cx_sum; }
        c.alias = false;
        return c;
    }

    // EF:2638-2880
    LargeResult solve(const double* x0, bool want_trace) {
        LargeResult res;
        rx.assign(mt, 0.0);
        cx.assign(l, 0.0);
        gradf.assign(n, 0.0);
        C.scaling = opt.scaling != 0;
        Vec x(x0, x0 + n), x_opt = x;
        int nb_iteration = 0;
        int exit_code = 0;
        int ndetail = 0;
        double f_opt = 0.0;
        auto t_start = std::chrono::steady_clock::now();
        auto elapsed = [&] { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };
        auto live_cx_sum = [&] { return dotv(cx, cx); };
        auto record = [&](int k, const IterL& it, double f_new, double acs, int ec) {
            if (!want_trace) return;
            res.trace.push_back(IterTraceL{k, W.t, it.rankA, it.rankJ2, it.dimA, it.dimJ2, it.code, it.index_del, ec,
                                           f_new, it.alpha, normv(it.p), acs, it.progress});
            res.trace_x.insert(res.trace_x.end(), x.begin(), x.end());
        };
        try {
            do_eval_point(x);
            f_opt = do_factor();
            IterL first;
            first.x = x; first.p.assign(n, 0.0); first.t = l; first.alpha = 1.0; first.lam.assign(l, 0.0);
            first.w.assign(l, 0.0); first.b_gn.assign(n, 0.0); first.d_gn.assign(n, 0.0);
            first.first = true; first.code = 1; first.alias = true;   // Iteration(x0, ..., rx, cx, ...) aliases
            init_working_set(first);
            first.t = W.t;
            gather_active();
            Vec p_gn(n, 0.0);
            evaluate_scaling();
            update_working_set(first, p_gn);
            double rx_sum = dotv(rx, rx);
            double active_cx_sum = 0.0;
            for (int i = 0; i < W.t; ++i) { double v = cx[W.active[i] - 1]; active_cx_sum += v * v; }
            first.t = W.t;
            IterL prev = copy_iter(first, rx_sum, live_cx_sum());
            int error_code = search_direction_analys(prev, first, nb_iteration, active_cx_sum, p_gn);
            Vec w;
            int Psi_error;
            double alpha = compute_steplength(first, prev, x, w, Psi_error);
            first.alpha = alpha;
            first.w = w;
            for (int j = 0; j < n; ++j) x[j] = first.x[j] + alpha * first.p[j];
            rx_sum = do_eval_point(x);
            first.restart = error_code < 0;
            double sigma_min, lam_abs_max;
            minmax_lagrangian_mult(first.lam, sigma_min, lam_abs_max);
            double delta_time = ops.agreed_elapsed(elapsed()) - opt.time_limit;
            exit_code = check_termination_criteria(first, prev, x, rx_sum, nb_iteration, error_code, delta_time,
                                                   sigma_min, lam_abs_max, Psi_error);
            if (exit_code == 0) rx_sum = do_factor();
            ++ndetail;
            record(0, first, rx_sum, active_cx_sum, exit_code);
            first.add = evaluate_violated_constraints(first.index_alpha_upp);
            gather_active();
            prev = copy_iter(first, rx_sum, live_cx_sum());
            first.x = x;
            first.alias = true;
            f_opt = rx_sum;
            ++nb_iteration;
            IterL it = copy_iter(first, rx_sum, live_cx_sum());   // it.rx is a private copy here (T1)
            it.first = false; it.add = false; it.dele = false;
            // NB: first.add is consumed through `it = first.copy()` BEFORE being reset?  No: the reference
            // resets it.add/it.del right after the copy (EF:2768-2771), so the flag of iteration 0 is dropped.
            bool took_loop = false;
            while (exit_code == 0) {
                took_loop = true;
                std::fill(p_gn.begin(), p_gn.end(), 0.0);
                evaluate_scaling();
                update_working_set(it, p_gn);
                active_cx_sum = 0.0;
                for (int i = 0; i < W.t; ++i) { double v = cx[W.active[i] - 1]; active_cx_sum += v * v; }
                it.t = W.t;
                error_code = search_direction_analys(prev, it, nb_iteration, active_cx_sum, p_gn);
                Vec xk = x;
                alpha = compute_steplength(it, prev, xk, w, Psi_error);
                it.alpha = alpha;
                it.w = w;
                for (int j = 0; j < n; ++j) x[j] = xk[j] + alpha * it.p[j];
                rx_sum = do_eval_point(x);
                it.restart = error_code < 0;
                minmax_lagrangian_mult(it.lam, sigma_min, lam_abs_max);
                delta_time = ops.agreed_elapsed(elapsed()) - opt.time_limit;
                exit_code = check_termination_criteria(it, prev, x, rx_sum, nb_iteration, error_code, delta_time,
                                                       sigma_min, lam_abs_max, Psi_error);
                if (exit_code == 0) rx_sum = do_factor();
                record(nb_iteration, it, rx_sum, active_cx_sum, exit_code);
                if (exit_code == 0) {
                    f_opt = rx_sum;
                    ++ndetail;
                    it.add = evaluate_violated_constraints(it.index_alpha_upp);
                    gather_active();
                    ++nb_iteration;
                    prev = copy_iter(it, rx_sum, live_cx_sum());
                    it.x = x;
                    it.alias = true;
                    it.dele = false;
                    it.add = false;
                } else {
                    x_opt = x;
                    f_opt = rx_sum;
                }
            }
            if (!took_loop) { ndetail = 1; /* x_opt stays x0 (SURVEY.md T5) */ }
            res.exit_code = exit_code;
            res.status = convert_exit_code(exit_code);
            res.x = x_opt;
            res.f = f_opt;
        } catch (const WouldThrow&) {
            res.exit_code = -99; res.status = -1; res.x = x; res.f = cur_rr;
        } catch (const WouldHang&) {
            res.exit_code = -98; res.status = -1; res.x = x; res.f = cur_rr;
        }
        res.iterations = ndetail;
        res.nact = W.t;
        res.active.assign(W.active.begin(), W.active.begin() + W.t);
        res.n_new_point = n_new_point;
        res.n_res_eval = n_res_eval;
        if (getenv("ENLSIP_PROF")) { host_prof().dump(); host_prof() = HostProf(); }
        return res;
    }
};

}  // namespace enl_large
