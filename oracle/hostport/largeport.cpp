// largeport.cpp -- CPU backend of enl_large::LargeOps and HostPoint for the single-index family.
//
// TEST INFRASTRUCTURE / CPU BASELINE ONLY (same role as hostport.cpp for the batched core):
//   (1) checks the large-regime ENLSIP driver (enlsip.jl_b200/csrc/enl_large_host.h) against the
//       Python oracle in the build container, which has no GPU;
//   (2) gives bench.py a compiled CPU implementation of one Gauss-Newton iteration of config 4
//       (OpenMP Householder QR of [J r]) to time as the `cpu_baseline` of the large regime.
// Never linked into libenlsip_b200.so; the product has no CPU fallback.
//
// Build: g++ -O2 -ffp-contract=off -mfma -std=c++17 -shared -fPIC -fopenmp largeport.cpp -o ../_build/liblargeport.so
#include <cstring>
#include <vector>
#define ENL_HOST_BUILD 1
#include "../../enlsip.jl_b200/csrc/enl_base.h"
#include "../../enlsip.jl_b200/csrc/enl_large_family.h"
#include "../../enlsip.jl_b200/csrc/enl_large_host.h"

using namespace enl_large;

namespace {

// collectives of the row-sharded run, supplied by the test (torch.distributed gloo) -- the CPU stand-ins for the
// ncclAllGather / ncclAllReduce calls of enl_large.cu
typedef void (*allgather_fn)(const double* send, double* recv, long long count);   // recv: world * count
typedef void (*allreduce_fn)(double* buf, int count);                              // in-place sum

struct CpuOps : LargeOps, HostPoint {
    const double* W;    // rows x n row major (this shard's rows)
    const double* y;
    long long rows = 0;  // rows held here (== m when not sharded)
    int world = 1;
    allgather_fn ag = nullptr;
    allreduce_fn ar = nullptr;
    SingleIndexConstraints sc;
    int nthreads = 1;
    std::vector<double> u, r, s, v, Jp;

    void eval_u(const double* x, std::vector<double>& out) const {
#pragma omp parallel for num_threads(nthreads) schedule(static)
        for (long long i = 0; i < rows; ++i) out[i] = dot_n(W + (size_t)i * n, x, n);
    }
    // unpivoted Householder QR (dgeqr2 order) of the column-major m x nc matrix M, in place (R in the upper triangle)
    void qr_inplace(std::vector<double>& M, long long m, int nc) const {
        for (int i = 0; i < nc && i < m; ++i) {
            double* ci = M.data() + (size_t)i * m;
            double alpha = ci[i];
            double xn = norm_n(ci + i + 1, (int)(m - i - 1));
            double tau = 0.0;
            if (xn != 0.0) {
                double beta = -copysign(lapy2(alpha, xn), alpha);
                tau = (beta - alpha) / beta;
                double sc_ = 1.0 / (alpha - beta);
                for (long long rr = i + 1; rr < m; ++rr) ci[rr] *= sc_;
                ci[i] = beta;
            }
            if (tau != 0.0) {
#pragma omp parallel for num_threads(nthreads) schedule(static)
                for (int c = i + 1; c < nc; ++c) {
                    double* cc = M.data() + (size_t)c * m;
                    double w = (cc[i] + dot_n(ci + i + 1, cc + i + 1, (int)(m - i - 1))) * tau;
                    cc[i] -= w;
                    for (long long rr = i + 1; rr < m; ++rr) cc[rr] -= w * ci[rr];
                }
            }
        }
    }
    int eval_point(const double* x, double* gradf, double* rr, double* cx, double* A) override {
        const long long m = rows;
        u.resize(m); r.resize(m); s.resize(m);
        eval_u(x, u);
        double a = 0;
#pragma omp parallel for num_threads(nthreads) schedule(static) reduction(+ : a)
        for (long long i = 0; i < m; ++i) {
            double th = enl::det_tanh(u[i]);
            r[i] = th - y[i];
            s[i] = 1.0 - th * th;
            a += r[i] * r[i];
        }
        // J'r with J = diag(s) W
        std::vector<double> g(n + 1, 0.0);
#pragma omp parallel for num_threads(nthreads) schedule(static)
        for (int j = 0; j < n; ++j) {
            double acc = 0;
            for (long long i = 0; i < m; ++i) acc += (s[i] * W[(size_t)i * n + j]) * r[i];
            g[j] = acc;
        }
        g[n] = a;
        if (world > 1) ar(g.data(), n + 1);
        for (int j = 0; j < n; ++j) gradf[j] = g[j];
        *rr = g[n];
        sc.cons(x, cx);
        sc.jac(x, A);
        return 0;
    }
    int compress(double* Jt, double* rt) override {
        const int nc = n + 1;
        long long m = rows;
        // augmented matrix [diag(s) W | r], column major for the Householder sweep
        std::vector<double> M((size_t)m * nc);
#pragma omp parallel for num_threads(nthreads) schedule(static)
        for (long long i = 0; i < m; ++i) {
            for (int j = 0; j < n; ++j) M[(size_t)j * m + i] = s[i] * W[(size_t)i * n + j];
            M[(size_t)n * m + i] = r[i];
        }
        qr_inplace(M, m, nc);
        if (world > 1) {
            // row-sharded TSQR (SURVEY.md 8e): all-gather the nc x nc factors, every rank re-factors the same stack
            std::vector<double> Rl((size_t)nc * nc, 0.0), Rall((size_t)world * nc * nc);
            for (int c = 0; c < nc; ++c)
                for (int rr = 0; rr <= c && rr < m; ++rr) Rl[(size_t)rr * nc + c] = M[(size_t)c * m + rr];
            ag(Rl.data(), Rall.data(), (long long)nc * nc);
            m = (long long)world * nc;
            M.assign((size_t)m * nc, 0.0);
            for (int g = 0; g < world; ++g)
                for (int rr = 0; rr < nc; ++rr)
                    for (int c = rr; c < nc; ++c) M[(size_t)c * m + (size_t)g * nc + rr] = Rall[((size_t)g * nc + rr) * nc + c];
            qr_inplace(M, m, nc);
        }
        const int mt = n + 1;
        for (int c = 0; c < n; ++c)
            for (int rr = 0; rr < mt; ++rr) Jt[(size_t)c * mt + rr] = (rr <= c && rr < m) ? M[(size_t)c * m + rr] : 0.0;
        for (int rr = 0; rr < mt; ++rr) rt[rr] = (rr < m) ? M[(size_t)n * m + rr] : 0.0;
        return 0;
    }
    int set_direction(const double*, const double* p, double sums[3]) override {
        const long long m = rows;
        v.resize(m); Jp.resize(m);
        eval_u(p, v);
        double a = 0, b = 0, c = 0;
#pragma omp parallel for num_threads(nthreads) schedule(static) reduction(+ : a, b, c)
        for (long long i = 0; i < m; ++i) {
            Jp[i] = s[i] * v[i];
            a += r[i] * r[i]; b += r[i] * Jp[i]; c += Jp[i] * Jp[i];
        }
        sums[0] = a; sums[1] = b; sums[2] = c;
        if (world > 1) ar(sums, 3);
        return 0;
    }
    int res_sq(double alpha, double* out) override {
        const long long m = rows;
        double a = 0;
#pragma omp parallel for num_threads(nthreads) schedule(static) reduction(+ : a)
        for (long long i = 0; i < m; ++i) {
            double ra = enl::det_tanh(__builtin_fma(alpha, v[i], u[i])) - y[i];
            a += ra * ra;
        }
        if (world > 1) ar(&a, 1);
        *out = a;
        return 0;
    }
    int ls_coeffs(double alpha, double out[4]) override {
        const long long m = rows;
        double a = 0, b = 0, c = 0, d = 0;
#pragma omp parallel for num_threads(nthreads) schedule(static) reduction(+ : a, b, c, d)
        for (long long i = 0; i < m; ++i) {
            double ra = enl::det_tanh(__builtin_fma(alpha, v[i], u[i])) - y[i];
            double v2 = ((ra - r[i]) / alpha - Jp[i]) / alpha;
            a += ra * ra; b += r[i] * v2; c += Jp[i] * v2; d += v2 * v2;
        }
        out[0] = a; out[1] = b; out[2] = c; out[3] = d;
        if (world > 1) ar(out, 4);
        return 0;
    }
    int cons(const double* x, double* cx) override { sc.cons(x, cx); return 0; }
    double agreed_elapsed(double local_elapsed) override {   // the mean over the ranks: one value for all
        if (world <= 1) return local_elapsed;
        double v = local_elapsed / world;
        ar(&v, 1);
        return v;
    }
};

}  // namespace

// Solve one single-index problem on the CPU.  trace: [trace_cap][16 + n] rows, layout of enlsip_b200.h.
// Row-sharded variant (world > 1): W / y hold `rows` of the m_global rows; `ag` / `ar` are the collectives.
extern "C" int largeport_solve_sharded(int n, long long m, long long rows, int world, allgather_fn ag, allreduce_fn ar,
                                       int nb, int ineq, const double* W, const double* y,
                                       const double* rho, const double* x_low, const double* x_upp, const double* x0,
                                       int max_iter, int scaling, double rel_tol, double x_tol, double c_tol, double* x,
                                       double* f, int* exit_code, int* status, int* iters, int* nact, int* active,
                                       double* trace, int trace_cap, int nthreads) {
    CpuOps ops;
    ops.n = n; ops.m = m; ops.rows = rows; ops.world = world; ops.ag = ag; ops.ar = ar;
    ops.W = W; ops.y = y; ops.nthreads = nthreads < 1 ? 1 : nthreads;
    ops.sc.n = n; ops.sc.nb = nb; ops.sc.ineq = ineq != 0;
    ops.sc.rho.assign(rho, rho + nb);
    ops.sc.set_bounds(x_low, x_upp);
    ops.l = ops.sc.l(); ops.q = ops.sc.q();
    LargeOptions opt;
    opt.max_iter = max_iter; opt.scaling = scaling;
    opt.eps_rel = rel_tol; opt.eps_x = x_tol; opt.eps_c = c_tol;
    HostSmall small(ops, ops.n, ops.l);
    LargeSolver S(ops, opt, small);
    LargeResult R = S.solve(x0, trace != nullptr);
    std::memcpy(x, R.x.data(), sizeof(double) * n);
    *f = R.f; *exit_code = R.exit_code; *status = R.status; *iters = R.iterations; *nact = R.nact;
    for (int i = 0; i < ops.l; ++i) active[i] = i < R.nact ? R.active[i] : 0;
    if (trace) {
        int rows = (int)R.trace.size();
        for (int k = 0; k < rows && k < trace_cap; ++k) {
            double* tr = trace + (size_t)k * (16 + n);
            const IterTraceL& t = R.trace[k];
            // same row layout as the batched engine (enl_solver.h Solver::step)
            tr[0] = t.f_new; tr[1] = t.t; tr[2] = t.rankA; tr[3] = t.rankJ2; tr[4] = t.dimA; tr[5] = t.dimJ2;
            tr[6] = t.code; tr[7] = t.alpha; tr[8] = t.p_norm; tr[9] = t.index_del; tr[10] = t.exit_code;
            tr[11] = t.active_cx_sum; tr[12] = t.progress; tr[13] = t.k; tr[14] = 0; tr[15] = 0;
            std::memcpy(tr + 16, R.trace_x.data() + (size_t)k * n, sizeof(double) * n);
        }
    }
    return 0;
}

extern "C" int largeport_solve(int n, long long m, int nb, int ineq, const double* W, const double* y,
                               const double* rho, const double* x_low, const double* x_upp, const double* x0,
                               int max_iter, int scaling, double rel_tol, double x_tol, double c_tol, double* x,
                               double* f, int* exit_code, int* status, int* iters, int* nact, int* active,
                               double* trace, int trace_cap, int nthreads) {
    return largeport_solve_sharded(n, m, m, 1, nullptr, nullptr, nb, ineq, W, y, rho, x_low, x_upp, x0, max_iter, scaling,
                                   rel_tol, x_tol, c_tol, x, f, exit_code, status, iters, nact, active, trace, trace_cap,
                                   nthreads);
}

// One Gauss-Newton iteration's dominant work on the CPU (the reference's `new_point!` + QR of J): used by
// bench.py as the large-regime cpu_baseline.  Returns seconds through *secs.
extern "C" int largeport_new_point(int n, long long m, const double* W, const double* y, const double* x, int nthreads,
                                   double* rho_out) {
    CpuOps ops;
    ops.n = n; ops.m = m; ops.rows = m; ops.W = W; ops.y = y; ops.nthreads = nthreads < 1 ? 1 : nthreads;
    ops.sc.n = n; ops.sc.nb = 0;
    std::vector<double> Jt((size_t)(n + 1) * n), rt(n + 1), cx(1), A(1), g(n);
    double rr = 0;
    ops.l = 0; ops.q = 0;
    ops.eval_point(x, g.data(), &rr, cx.data(), A.data());
    ops.compress(Jt.data(), rt.data());
    *rho_out = rt[n];
    return 0;
}

// Known-answer hook: the large regime's host `qr(., ColumnNorm())` restatement (enl_large_host.h QRP::factor):
// f [rows x cols] column major in/out, tau [min(rows, cols)], jpvt [cols] 0-based.
extern "C" void largeport_qrcp(int rows, int cols, double* f, double* tau, int* jpvt) {
    Mat M(rows, cols);
    std::memcpy(M.a.data(), f, sizeof(double) * (size_t)rows * cols);
    QRP F;
    F.factor(M);
    std::memcpy(f, F.f.a.data(), sizeof(double) * (size_t)rows * cols);
    for (int i = 0; i < F.k; ++i) tau[i] = F.tau[i];
    for (int j = 0; j < cols; ++j) jpvt[j] = F.p[j];
}

// ------------------------------------------------------------------------------------------------------------------
// CPU reference arm of the large regime (bench.py cpu_baseline "reference-algorithm" / --impl reference): ONE
// Gauss-Newton iteration's dense work done the way Enlsip.jl does it, with the LAPACK/BLAS routines Julia calls, bound at
// run time from an OpenBLAS shared library (the SciPy wheel's libscipy_openblas; Julia ships OpenBLAS_jll):
//     new_point!                      r, J = diag(1 - tanh^2) W (m x n, column major), c, A          EF:34-52
//     qr(A_active', ColumnNorm())     dgeqp3 (n x t)                                                  EF:700
//     J * F_A.Q                       dormqr('R', 'N') on the full m x n Jacobian                     EF:219
//     qr(J2, ColumnNorm())            dgeqp3 (m x (n - t))                                            EF:223
//     p1 = L11 \ (-P'c), d = Q3'(-J1 p1 - r), p2 = R22 \ d, p = Q1 [p1; p2]   dtrtrs / dgemv / dormqr  EF:133-152
// for the single-index problem at x: working set = the equalities (config 4) or the inequalities / bounds with c <= 0
// (init_working_set, EF:826-859; config 5), assumed of full rank (method code 1).  The multiplier estimates and the
// linesearch are left out, so the figure flatters the CPU slightly.  secs: {total, new_point,
// J*Q1, qr(J2), rest}.  Returns 0, or a negative code when the library / a symbol cannot be bound.
// ------------------------------------------------------------------------------------------------------------------
#include <dlfcn.h>

#include <chrono>

namespace {
struct Lapack {
    typedef void (*geqp3_t)(const int*, const int*, double*, const int*, int*, double*, double*, const int*, int*);
    typedef void (*ormqr_t)(const char*, const char*, const int*, const int*, const int*, const double*, const int*,
                            const double*, double*, const int*, double*, const int*, int*);
    typedef void (*trtrs_t)(const char*, const char*, const char*, const int*, const int*, const double*, const int*,
                            double*, const int*, int*);
    typedef void (*gemv_t)(const char*, const int*, const int*, const double*, const double*, const int*, const double*,
                           const int*, const double*, double*, const int*);
    typedef void (*setthr_t)(int);
    geqp3_t geqp3 = nullptr; ormqr_t ormqr = nullptr; trtrs_t trtrs = nullptr; gemv_t gemv = nullptr; setthr_t setthr = nullptr;
    int bind(const char* path) {
        void* h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
        if (!h) return -1;
        auto sym = [&](const char* a, const char* b) { void* p = dlsym(h, a); return p ? p : dlsym(h, b); };
        geqp3 = (geqp3_t)sym("scipy_dgeqp3_", "dgeqp3_");
        ormqr = (ormqr_t)sym("scipy_dormqr_", "dormqr_");
        trtrs = (trtrs_t)sym("scipy_dtrtrs_", "dtrtrs_");
        gemv = (gemv_t)sym("scipy_dgemv_", "dgemv_");
        setthr = (setthr_t)sym("scipy_openblas_set_num_threads", "openblas_set_num_threads");
        return (geqp3 && ormqr && trtrs && gemv) ? 0 : -2;
    }
};
double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
}  // namespace

extern "C" int largeport_ref_iteration(const char* blas_path, int n, long long m, int nb, int ineq, const double* x_low,
                                       const double* x_upp, const double* W, const double* y, const double* rho,
                                       const double* x, int nthreads, double* secs, double* p_out, int* t_out) {
    Lapack L;
    int rc = L.bind(blas_path);
    if (rc != 0) return rc;
    if (L.setthr) L.setthr(nthreads < 1 ? 1 : nthreads);
    const int mi = (int)m;
    int info = 0;
    const double t0 = now_s();
    // ---- new_point! ----
    std::vector<double> J((size_t)m * n), r(m), sv(m);
#pragma omp parallel for num_threads(nthreads) schedule(static)
    for (long long i = 0; i < m; ++i) {
        double th = enl::det_tanh(dot_n(W + (size_t)i * n, x, n));
        r[i] = th - y[i];
        sv[i] = 1.0 - th * th;
    }
#pragma omp parallel for num_threads(nthreads) schedule(static)
    for (int j = 0; j < n; ++j) {
        double* cj = J.data() + (size_t)j * m;
        for (long long i = 0; i < m; ++i) cj[i] = sv[i] * W[(size_t)i * n + j];
    }
    SingleIndexConstraints sc;
    sc.n = n; sc.nb = nb; sc.ineq = ineq != 0;
    sc.rho.assign(rho, rho + nb);
    sc.set_bounds(x_low, x_upp);
    const int l = sc.l();
    std::vector<double> call(l), Aall((size_t)l * n, 0.0);
    sc.cons(x, call.data());
    sc.jac(x, Aall.data());                                // l x n column major
    std::vector<int> act;
    for (int i = 0; i < l; ++i)
        if (i < sc.q() || call[i] <= 0.0) act.push_back(i);
    const int t = (int)act.size(), k2 = n - t;
    if (t_out) *t_out = t;
    if (t < 1 || k2 < 1) return -20;
    std::vector<double> c(t), At((size_t)n * t);
    for (int i = 0; i < t; ++i) {
        c[i] = call[act[i]];
        for (int j = 0; j < n; ++j) At[(size_t)i * n + j] = Aall[(size_t)j * l + act[i]];
    }
    const double t1 = now_s();
    // ---- qr(A', ColumnNorm()) ----
    std::vector<int> pA(t, 0), p2(k2, 0);
    std::vector<double> tauA(t), tau2(k2), wq(1);
    int lwork = -1;
    L.geqp3(&mi, &k2, J.data() + (size_t)t * m, &mi, p2.data(), tau2.data(), wq.data(), &lwork, &info);
    size_t need = (size_t)wq[0];
    L.ormqr("R", "N", &mi, &n, &t, At.data(), &n, tauA.data(), J.data(), &mi, wq.data(), &lwork, &info);
    need = std::max(need, (size_t)wq[0]);
    std::vector<double> work(std::max<size_t>(need, (size_t)8 * n + 64) + 1024);
    lwork = (int)work.size();
    L.geqp3(&n, &t, At.data(), &n, pA.data(), tauA.data(), work.data(), &lwork, &info);
    if (info != 0) return -10;
    // ---- J * Q1 ----
    L.ormqr("R", "N", &mi, &n, &t, At.data(), &n, tauA.data(), J.data(), &mi, work.data(), &lwork, &info);
    if (info != 0) return -11;
    const double t2 = now_s();
    // ---- qr(J2, ColumnNorm()) ----
    std::fill(p2.begin(), p2.end(), 0);
    L.geqp3(&mi, &k2, J.data() + (size_t)t * m, &mi, p2.data(), tau2.data(), work.data(), &lwork, &info);
    if (info != 0) return -12;
    const double t3 = now_s();
    // ---- p1 = L11 \ (-P'c) ; d = Q3'(-J1 p1 - r) ; p2 = R22 \ d[1:k2] ; p = Q1 [p1; p2[invperm]] ----
    std::vector<double> p1(t), d(m), pv(n, 0.0);
    for (int i = 0; i < t; ++i) p1[i] = -c[pA[i] - 1];
    const int one = 1;
    L.trtrs("U", "T", "N", &t, &one, At.data(), &n, p1.data(), &t, &info);
    const double neg1 = -1.0;
    for (long long i = 0; i < m; ++i) d[i] = r[i];
    L.gemv("N", &mi, &t, &neg1, J.data(), &mi, p1.data(), &one, &neg1, d.data(), &one);        // d = -J1 p1 - r
    L.ormqr("L", "T", &mi, &one, &k2, J.data() + (size_t)t * m, &mi, tau2.data(), d.data(), &mi, work.data(), &lwork, &info);
    L.trtrs("U", "N", "N", &k2, &one, J.data() + (size_t)t * m, &mi, d.data(), &mi, &info);
    for (int i = 0; i < t; ++i) pv[i] = p1[i];
    for (int j = 0; j < k2; ++j) pv[t + p2[j] - 1] = d[j];
    L.ormqr("L", "N", &n, &one, &t, At.data(), &n, tauA.data(), pv.data(), &n, work.data(), &lwork, &info);
    const double t4 = now_s();
    if (p_out) std::memcpy(p_out, pv.data(), sizeof(double) * n);
    secs[0] = t4 - t0; secs[1] = t1 - t0; secs[2] = t2 - t1; secs[3] = t3 - t2; secs[4] = t4 - t3;
    return info == 0 ? 0 : -13;
}
