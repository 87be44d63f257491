// enl_small_device.cuh -- DeviceSmall: the large regime's SmallBackend (enl_large_host.h) on the device.  Every matrix of
// the small stage (A, C.A, J~ Q1, the three pivoted QR factorisations and their compact-WY T factors, the Newton step's
// G / E / [W21 | W22] / U) lives in HBM and is worked on by the kernels of enl_small.cuh; vectors travel host <-> device
// per call (a few KB).  The m-sized world (evaluation, the factorisation of [J | r] into [J~ | r~], the Hessian) belongs
// to the DevicePoint that owns this object (LargeHandle, enl_large.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "enl_large_host.h"
#include "enl_small.cuh"

namespace enl_large {

// what DeviceSmall needs from the m-sized backend
struct DevicePoint {
    virtual ~DevicePoint() {}
    // new_point! (EF:34-52), first half, at x: J'r (n), ||r||^2 and c (l); the rows of A that depend on x go to
    // DeviceSmall::dArow.  Returns 0 or an API error.
    virtual int eval_point(const double* x, double* gradf, double* rr, double* cx) = 0;
    // [J~ | r~] of the point of the last eval_point into the device matrix DeviceSmall reads as dJc
    virtual int factor_point(bool want_host_R) = 0;
    // G (device, n x n, column major) = sum_i r_i Hess r_i - sum_{a < t} lam[a] Hess c_{active[a]} at x (EF:243-328)
    virtual int hessian(const double* x, const double* lam, const int* active, int t, double* G) = 0;
    virtual const char* last_error() const = 0;
};

struct DeviceSmall : SmallBackend {
    template <class T> using DevBuf = enl_small::DevBuf<T>;
    DevicePoint& pt;
    int device = 0, n = 0, l = 0;
    cudaStream_t st = nullptr;        // the owner's stream
    const double* dJc = nullptr;      // [J~ | r~] column major (n+1) x (n+1), written by pt.factor_point
    int tcap = 0, lv = 0;             // the working-set buffers hold tcap + 1 rows (min(l, n) + 1 at first, grown on
                                      // demand up to l); length of the scratch vectors
    DevBuf<double> dArow;             // A, row major l x n  (= column-major n x l)
    DevBuf<double> dCA, dCA2;         // C.A, row major t x n (= C.A' column major n x t); spare for row removal
    DevBuf<double> dFA, dtauA;        // factors of qr(C.A')   n x t
    DevBuf<double> dFL, dtauL;        // factors of qr(R_A')   t x min(n, t)
    DevBuf<double> dJQ1;              // J~ Q1                 (n+1) x n
    DevBuf<double> dF2, dtau2;        // factors of qr(J2)     (n+1) x (n - rankA)
    DevBuf<int> dpA, dipA, dpL, dipL, dp2, dip2, dact;
    DevBuf<double> dvec[8];           // scratch vectors
    DevBuf<double> dscal;
    // compact-WY T factors of the three factorisations (all panels; built on first use after a factorisation) and the
    // scratch of the cooperative vector kernels
    DevBuf<double> dTA, dTL, dT2, dwpart;
    bool ta_valid = false, tl_valid = false, t2_valid = false;
    enl_small::PinnedBuf<double> hst; // pinned staging, 4 * lv doubles
    enl_small::PinnedBuf<int> hsti;   // pinned staging for permutations
    enl_small::QrWork qw;             // also the scratch of the owner's QR of [J | r]
    enl_small::WyWork ww;
    int fa_rows = 0, fa_cols = 0, fa_k = 0, fl_rows = 0, fl_cols = 0, fl_k = 0, f2_rows = 0, f2_cols = 0, f2_k = 0;
    bool jq1_valid = false;
    int ca_rows = 0;
    // Newton step (midsize handles only): n x n matrices G, E = Q1' G Q1 and its scratch, the k2 x n block [W21 | W22]
    // and the Cholesky factor; the factorisation's info
    bool midsize = false;
    DevBuf<double> dG, dE, dWn, dU;
    DevBuf<int> dinfo;
    std::vector<int> hpA, hpL, hp2;   // host copies of the three permutations
    long long n_dev_qrcp = 0, n_dev_mulq = 0, n_ws_grow = 0, n_newton = 0, launches = 0;
    double ms_small = 0;              // host wall clock inside the small-stage calls (kernels + waits)

    explicit DeviceSmall(DevicePoint& p) : pt(p) {}
    ~DeviceSmall() override {
        if (small_prof_on() && !small_prof.empty())
            for (const auto& kv : small_prof)
                fprintf(stderr, "[small stage] %-24s %6lld calls %10.3f ms\n", kv.first.c_str(), kv.second.second, kv.second.first);
    }

    // the small stage's matrices and scratch (sizes from n, l); A is zeroed on `stream`
    cudaError_t alloc(int dev, int nn, int ll, bool with_newton, cudaStream_t stream, const double* jc) {
        using enl_small::dev_alloc;
        device = dev; n = nn; l = ll; midsize = with_newton; st = stream; dJc = jc;
        const size_t mt = (size_t)n + 1;
        tcap = l < n ? l : n;
        lv = (int)(mt > (size_t)l ? mt : (size_t)l) + 32;
        cudaError_t e = dev_alloc(dArow, (size_t)l * n);
        if (e == cudaSuccess) e = cudaMemsetAsync(dArow.get(), 0, sizeof(double) * (size_t)l * n, st);
        if (e == cudaSuccess) e = dev_alloc(dCA, (size_t)(tcap + 1) * n);
        if (e == cudaSuccess) e = dev_alloc(dFA, (size_t)n * (tcap + 1));
        if (e == cudaSuccess) e = dev_alloc(dtauA, tcap + 1);
        if (e == cudaSuccess) e = dev_alloc(dFL, (size_t)(tcap + 1) * (tcap + 1));
        if (e == cudaSuccess) e = dev_alloc(dtauL, tcap + 1);
        if (e == cudaSuccess) e = dev_alloc(dJQ1, mt * n);
        if (e == cudaSuccess) e = dev_alloc(dF2, mt * n);
        if (e == cudaSuccess) e = dev_alloc(dtau2, mt);
        for (DevBuf<int>* p : {&dpA, &dipA, &dpL, &dipL}) if (e == cudaSuccess) e = dev_alloc(*p, tcap + 1);
        for (DevBuf<int>* p : {&dp2, &dip2}) if (e == cudaSuccess) e = dev_alloc(*p, n + 1);
        if (e == cudaSuccess) e = dev_alloc(dact, l + 1);
        for (DevBuf<double>& p : dvec) if (e == cudaSuccess) e = dev_alloc(p, lv);
        if (e == cudaSuccess) e = dev_alloc(dscal, 8);
        if (e == cudaSuccess) e = enl_small::pinned_alloc(hst, 4 * (size_t)lv);
        if (e == cudaSuccess) e = enl_small::pinned_alloc(hsti, 2 * (size_t)lv);
        // per-column QR scratch: n + 1 columns ([J | r], J2, and qr(C.A') while t <= n + 1); ensure_ws_capacity grows it
        if (e == cudaSuccess) e = qw.alloc((int)mt);
        if (e == cudaSuccess) e = cudaMemsetAsync(qw.ticket.get(), 0, sizeof(unsigned int) * enl_small::QR_TICKET_LEN, st);
        const size_t tlen = (mt / 32 + 2) * 1024;
        for (DevBuf<double>* p : {&dTA, &dTL, &dT2}) if (e == cudaSuccess) e = dev_alloc(*p, tlen);
        if (e == cudaSuccess) e = dev_alloc(dwpart, enl_small::RW_WPART_LEN);
        if (e == cudaSuccess) e = ww.alloc(mt, mt);
        if (midsize) {
            for (DevBuf<double>* p : {&dG, &dE, &dWn, &dU}) if (e == cudaSuccess) e = dev_alloc(*p, (size_t)n * n);
            if (e == cudaSuccess) e = dev_alloc(dinfo, 1);
        }
        return e;
    }
    // Nothing bounds the working set by n: init_working_set takes every violated row, so t can reach l.  The buffers
    // sized by t are (re)allocated here, before t rows enter C.A; their contents are rebuilt by gather_active and the
    // factorisations that follow, so nothing is copied.  The small stage runs identically on every rank, so every rank
    // grows at the same call.  Starts whose working set stays within min(l, n) + 1 rows never come here.
    void ensure_ws_capacity(int t) {
        using enl_small::dev_alloc;
        if (t <= tcap + 1) return;
        // rows of C.A the new buffers hold (never fewer than alloc's min(l, n) + 1, also after a failed growth)
        const int rows = std::min(l, std::max({t, 2 * (tcap + 1), std::min(l, n) + 1}));
        sm_sync();
        // until every new buffer exists the object holds no working set: a cudaMalloc failure below throws with tcap = -1,
        // so need_ws refuses every later call and the next gather_active allocates afresh
        tcap = -1;
        for (DevBuf<double>* p : {&dCA, &dCA2, &dFA, &dtauA, &dFL, &dtauL}) p->reset();
        for (DevBuf<int>* p : {&dpA, &dipA, &dpL, &dipL}) p->reset();
        qw.drop_graphs();                 // captured QR graphs hold the old factor and scratch pointers
        sm_check(dev_alloc(dCA, (size_t)rows * n), "cudaMalloc");
        sm_check(dev_alloc(dFA, (size_t)n * rows), "cudaMalloc");
        sm_check(dev_alloc(dtauA, rows), "cudaMalloc");
        sm_check(dev_alloc(dFL, (size_t)rows * std::min(rows, n)), "cudaMalloc");   // t x min(n, t)
        sm_check(dev_alloc(dtauL, rows), "cudaMalloc");
        for (DevBuf<int>* p : {&dpA, &dipA, &dpL, &dipL}) sm_check(dev_alloc(*p, rows), "cudaMalloc");
        const int qcols = std::max(rows, n + 1);       // [J | r] and J2 need n + 1 columns whatever t is
        if (qcols > qw.cap_cols) sm_check(qw.alloc_cols(qcols), "cudaMalloc");
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

    // ENLSIP_SMALL_PROF=1: per-call breakdown of the small stage (each call is followed by a stream synchronisation, so
    // the figures include what the call left in flight), printed when the object is destroyed
    std::map<std::string, std::pair<double, long long>> small_prof;
    static bool small_prof_on() {
        static const bool v = [] { const char* e = getenv("ENLSIP_SMALL_PROF"); return e && e[0] == '1'; }();
        return v;
    }
    struct SmallScope {
        DeviceSmall* h; std::chrono::steady_clock::time_point t0; const char* name;
        explicit SmallScope(DeviceSmall* hh, const char* nm = __builtin_FUNCTION())
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
        if (cnt > 0) sm_check(cudaMemcpyAsync(hst.get() + slot_off, d, sizeof(double) * cnt, cudaMemcpyDeviceToHost, st), "D2H");
    }
    void sm_sync() {
        sm_check(cudaStreamSynchronize(st), "synchronize");
        sm_check(cudaGetLastError(), "kernel");
    }
    // T factors of a factorisation (dFA / dFL / dF2), built once per factorisation
    double* wy_t_of(const double* f, int frows, int k, const double* tau) {
        double* T = nullptr; bool* valid = nullptr;
        if (f == dFA.get()) { T = dTA.get(); valid = &ta_valid; }
        else if (f == dFL.get()) { T = dTL.get(); valid = &tl_valid; }
        else if (f == dF2.get()) { T = dT2.get(); valid = &t2_valid; }
        if (!T) return nullptr;
        if (!*valid) {
            const int rc = enl_small::wy_build_t_all(f, frows, k, tau, T, ww.part.get(), ww.part_len, st);
            if (rc < 0) return nullptr;
            launches += rc;
            *valid = true;
        }
        return T;
    }
    void k_reflect(const double* f, int frows, int k, const double* tau, double* v, int transpose) {
        launches += enl_small::reflect_vec(f, frows, k, tau, v, transpose, [&] { return wy_t_of(f, frows, k, tau); },
                                           dwpart.get(), qw.ticket.get() + 1, st);
    }
    void k_trsv_upper(const double* f, int ldf, int k, double* x) {
        launches += enl_small::trsv_upper(f, ldf, k, x, false, qw.ticket.get() + 1, st);
    }
    void k_trsv_upperT(const double* f, int ldf, int k, double* x) {
        launches += enl_small::trsv_upper(f, ldf, k, x, true, qw.ticket.get() + 1, st);
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
            enl_small::qr_finish_kernel<<<(cols + 255) / 256, 256, 0, st>>>(f, rows, cols, dperm, dvec[7].get(), diperm);
            ++launches;
            down(0, dvec[7].get(), k);
            sm_check(cudaMemcpyAsync(hsti.get(), dperm, sizeof(int) * cols, cudaMemcpyDeviceToHost, st), "D2H");
            sm_sync();
            for (int i = 0; i < k; ++i) F.diagv[i] = hst[i];
            for (int i = 0; i < cols; ++i) F.p[i] = hsti[i];
        }
        hperm = F.p;
    }

    int new_point_eval(const double* x, double* gradf, double* rr, double* cx) override {
        jq1_valid = false;
        return pt.eval_point(x, gradf, rr, cx);
    }
    int new_point_compress(double* rt, double* gradf) override {
        int rc = pt.factor_point(false);
        if (rc != 0) return rc;
        jq1_valid = false;
        SmallScope sc_(this);
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        launches += enl_small::gemv_t(dJc, mt, mt, n, rtd, dvec[0].get(), st);     // J~' r~
        down(0, rtd, mt);
        down(lv, dvec[0].get(), n);
        sm_sync();
        for (int r = 0; r < mt; ++r) rt[r] = hst[r];
        for (int j = 0; j < n; ++j) gradf[j] = hst[lv + j];
        return 0;
    }
    void gather_active(const int* active, int t) override {
        SmallScope sc_(this);
        ensure_ws_capacity(t);
        ca_rows = t;
        if (t <= 0) return;
        up_i(dact.get(), active, t);
        enl_small::gather_rows_kernel<<<t, 256, 0, st>>>(dArow.get(), n, dact.get(), dCA.get());
        ++launches;
    }
    void evaluate_scaling(int t, bool scaling, double* rown) override {
        SmallScope sc_(this);
        need_ws(t);
        if (t <= 0) return;
        enl_small::row_norm_scale_kernel<<<t, 256, 0, st>>>(dCA.get(), n, scaling ? 1 : 0, dvec[0].get());
        ++launches;
        down(0, dvec[0].get(), t);
        sm_sync();
        for (int i = 0; i < t; ++i) rown[i] = hst[i];
    }
    void rebuild_scaled_rows(const int* active, int t, const double* diag_scale) override {
        SmallScope sc_(this);
        need_ws(t);
        if (t <= 0) return;
        up_i(dact.get(), active, t);
        up(dvec[0].get(), diag_scale, t);
        enl_small::rebuild_scaled_rows_kernel<<<t, 256, 0, st>>>(dArow.get(), n, dact.get(), dvec[0].get(), dCA.get());
        ++launches;
    }
    void remove_active_row(int s0) override {
        SmallScope sc_(this);
        need_ws(ca_rows);
        const int below = ca_rows - 1 - s0;
        if (below > 0) {
            if (!dCA2) sm_check(enl_small::dev_alloc(dCA2, (size_t)(tcap + 1) * n), "cudaMalloc");
            const size_t bytes = sizeof(double) * (size_t)below * n;
            sm_check(cudaMemcpyAsync(dCA2.get(), dCA.get() + (size_t)(s0 + 1) * n, bytes, cudaMemcpyDeviceToDevice, st), "D2D");
            sm_check(cudaMemcpyAsync(dCA.get() + (size_t)s0 * n, dCA2.get(), bytes, cudaMemcpyDeviceToDevice, st), "D2D");
        }
        ca_rows -= 1;
    }
    void factor_A(int t, FactorInfo& F) override {
        SmallScope sc_(this);
        need_ws(t);
        fa_rows = n; fa_cols = t; fa_k = n < t ? n : t;
        jq1_valid = false;
        if (t > 0) {
            sm_check(cudaMemcpyAsync(dFA.get(), dCA.get(), sizeof(double) * (size_t)n * t, cudaMemcpyDeviceToDevice, st), "D2D");
            qrcp(dFA.get(), n, t, dtauA.get(), dpA.get());
            ta_valid = false;
        }
        finish_factor(dFA.get(), n, t, dpA.get(), dipA.get(), F, hpA);
    }
    void factor_L11(FactorInfo& F) override {    // qr(F_A.R', ColumnNorm()); F_A.R is min(n, t) x t
        SmallScope sc_(this);
        const int kr = fa_k, t = fa_cols;
        need_ws(t);
        fl_rows = t; fl_cols = kr; fl_k = t < kr ? t : kr;
        if (t > 0 && kr > 0) {
            const long long ne = (long long)t * kr;
            enl_small::build_rt_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(dFA.get(), n, t, kr, dFL.get());
            ++launches;
            qrcp(dFL.get(), t, kr, dtauL.get(), dpL.get());
            tl_valid = false;
        }
        finish_factor(dFL.get(), t, kr, dpL.get(), dipL.get(), F, hpL);
    }
    void ensure_jq1() {
        if (jq1_valid) return;
        const int mt = n + 1;
        sm_check(cudaMemcpyAsync(dJQ1.get(), dJc, sizeof(double) * (size_t)mt * n, cudaMemcpyDeviceToDevice, st), "D2D");
        if (fa_k > 0) {
            double* TA = wy_t_of(dFA.get(), n, fa_k, dtauA.get());   // all T factors of qr(C.A') at once; nullptr: per panel inside mulq_device
            launches += enl_small::mulq_device(dJQ1.get(), mt, n, dFA.get(), n, fa_k, dtauA.get(), ww, st, TA, false);
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
            sm_check(cudaMemcpyAsync(dF2.get(), dJQ1.get() + (size_t)rankA * mt, sizeof(double) * (size_t)mt * cols2, cudaMemcpyDeviceToDevice, st), "D2D");
            qrcp(dF2.get(), mt, cols2, dtau2.get(), dp2.get());
            t2_valid = false;
        }
        finish_factor(dF2.get(), mt, cols2, dp2.get(), dip2.get(), F, hp2);
    }
    void first_lagrange(int prankA, int t, const Vec& gradf, const Vec& Ccx, Vec& v, Vec& u, double& grad_res) override {
        SmallScope sc_(this);
        need_ws(t);
        Vec y0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < prankA; ++i) y0[i] = -Ccx[hpA[i]];
        up(dvec[0].get(), gradf.data(), n);
        up(dvec[1].get(), y0.data(), t);
        k_reflect(dFA.get(), n, fa_k, dtauA.get(), dvec[0].get(), 1);    // b = Q1' gradf
        k_copy_pad(dvec[2].get(), dvec[0].get(), prankA, t);
        k_trsv_upper(dFA.get(), n, prankA, dvec[2].get());                // v = R^-1 b[1:r]
        enl_small::norm_range_kernel<<<1, 1024, 0, st>>>(dvec[0].get(), prankA, n, dscal.get());
        ++launches;
        k_trsv_upperT(dFA.get(), n, prankA, dvec[1].get());               // u = R^-1 R^-T (-c[P])[1:r]
        k_trsv_upper(dFA.get(), n, prankA, dvec[1].get());
        down(0, dvec[2].get(), t);
        down(lv, dvec[1].get(), t);
        down(2 * lv, dscal.get(), 1);
        sm_sync();
        v.assign(hst.get(), hst.get() + t);
        u.assign(hst.get() + lv, hst.get() + lv + t);
        grad_res = (n > prankA) ? hst[2 * lv] : 0.0;
    }
    void second_lagrange(int prankA, int t, const Vec& p_gn, Vec& v) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        up(dvec[0].get(), p_gn.data(), n);
        launches += enl_small::gemv_n(dJc, mt, mt, n, dvec[0].get(), 1.0, rtd, 1.0, dvec[1].get(), st);    // s = r + J p_gn
        if (t > 0) sm_check(cudaMemsetAsync(dvec[2].get(), 0, sizeof(double) * t, st), "memset");
        launches += enl_small::gemv_t(dJQ1.get(), mt, mt, prankA, dvec[1].get(), dvec[2].get(), st);       // J1' s
        k_trsv_upper(dFA.get(), n, prankA, dvec[2].get());
        down(0, dvec[2].get(), t);
        sm_sync();
        v.assign(hst.get(), hst.get() + t);
    }
    void sub_search_direction(int t, int rankA, int dimA, int dimJ2, int code, const Vec& Ccx, Vec& p, Vec& b, Vec& d) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        double* const v[6] = {dvec[0].get(), dvec[1].get(), dvec[2].get(), dvec[3].get(), dvec[4].get(), dvec[5].get()};
        Vec b0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < t; ++i) b0[i] = -Ccx[hpA[i]];
        up(v[0], b0.data(), t);
        const double* p1;
        if (code == 1) {
            k_trsv_upperT(dFA.get(), n, t, v[0]);                      // L11 p1 = -P'c
            p1 = v[0];
        } else {
            k_reflect(dFL.get(), fl_rows, fl_k, dtauL.get(), v[0], 1);  // b = Q2'(-P'c)
            k_copy_pad(v[1], v[0], dimA, t);
            k_trsv_upper(dFL.get(), fl_rows, dimA, v[1]);               // [R11[1:dimA] \ b[1:dimA]; 0]
            if (rankA > 0) {
                enl_small::gather_pad_kernel<<<(rankA + 255) / 256, 256, 0, st>>>(v[2], v[1], dipL.get(), t, rankA);
                ++launches;
            }
            p1 = v[2];
        }
        launches += enl_small::gemv_n(dJQ1.get(), mt, mt, rankA, p1, -1.0, rtd, -1.0, v[3], st);   // -J1 p1 - r
        k_reflect(dF2.get(), mt, f2_k, dtau2.get(), v[3], 1);            // d = Q3'(...)
        const int dj = dimJ2 > 0 ? dimJ2 : 0;
        k_copy_pad(v[4], v[3], dj, dj);
        k_trsv_upper(dF2.get(), mt, dj, v[4]);
        if (rankA > 0) sm_check(cudaMemcpyAsync(v[5], p1, sizeof(double) * rankA, cudaMemcpyDeviceToDevice, st), "D2D");
        if (f2_cols > 0) {
            enl_small::gather_pad_kernel<<<(f2_cols + 255) / 256, 256, 0, st>>>(v[5] + rankA, v[4], dip2.get(), dj, f2_cols);
            ++launches;
        }
        k_reflect(dFA.get(), n, fa_k, dtauA.get(), v[5], 0);             // p = Q1 [p1; p2]
        down(0, v[5], n);
        down(lv, v[3], mt);
        if (code != 1) down(2 * lv, v[0], t);
        sm_sync();
        p.assign(hst.get(), hst.get() + n);
        d.assign(hst.get() + lv, hst.get() + lv + mt);
        if (code == 1) b.assign(b0.begin(), b0.begin() + t);
        else b.assign(hst.get() + 2 * lv, hst.get() + 2 * lv + t);
    }
    void subspace_rhs(int t, const Vec& Ccx, Vec& b) override {
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        Vec b0(t > 0 ? t : 1, 0.0);
        for (int i = 0; i < t; ++i) b0[i] = -Ccx[hpA[i]];
        up(dvec[0].get(), b0.data(), t);
        k_reflect(dFL.get(), fl_rows, fl_k, dtauL.get(), dvec[0].get(), 1);
        down(0, dvec[0].get(), t);
        sm_sync();
        b.assign(hst.get(), hst.get() + t);
    }
    void subspace_d(int rankA, int dimA, int rankJ2, const Vec& b, Vec& d) override {
        SmallScope sc_(this);
        const int mt = n + 1;
        const double* rtd = dJc + (size_t)mt * n;
        int ra = rankA > 0 ? rankA : 0;
        if (ra > 0) {
            const int da = dimA > 0 ? dimA : 0;
            up(dvec[0].get(), b.data(), (int)b.size());
            k_copy_pad(dvec[1].get(), dvec[0].get(), da, da);
            k_trsv_upper(dFL.get(), fl_rows, da, dvec[1].get());
            sm_check(cudaMemsetAsync(dvec[2].get(), 0, sizeof(double) * ra, st), "memset");
            if (da > 0) {
                enl_small::scatter_perm_kernel<<<(da + 255) / 256, 256, 0, st>>>(dvec[2].get(), dvec[1].get(), dpL.get(), da, ra);
                ++launches;
            }
        }
        launches += enl_small::gemv_n(dJQ1.get(), mt, mt, ra, dvec[2].get(), -1.0, rtd, -1.0, dvec[3].get(), st);   // -(r + J1 p1)
        if (rankJ2 > 0) k_reflect(dF2.get(), mt, f2_k, dtau2.get(), dvec[3].get(), 1);
        down(0, dvec[3].get(), mt);
        sm_sync();
        d.assign(hst.get(), hst.get() + mt);
    }
    void products(const Vec& p, int t, Vec& Jp, Vec& Ap, Vec& active_Ap) override {
        SmallScope sc_(this);
        need_ws(t);
        const int mt = n + 1;
        up(dvec[0].get(), p.data(), n);
        launches += enl_small::gemv_n(dJc, mt, mt, n, dvec[0].get(), 1.0, nullptr, 0.0, dvec[1].get(), st);
        launches += enl_small::gemv_t(dArow.get(), n, n, l, dvec[0].get(), dvec[2].get(), st);
        launches += enl_small::gemv_t(dCA.get(), n, n, t, dvec[0].get(), dvec[3].get(), st);
        down(0, dvec[1].get(), mt);
        down(lv, dvec[2].get(), l);
        down(2 * lv, dvec[3].get(), t);
        sm_sync();
        Jp.assign(hst.get(), hst.get() + mt);
        Ap.assign(hst.get() + lv, hst.get() + lv + l);
        active_Ap.assign(hst.get() + 2 * lv, hst.get() + 2 * lv + t);
    }
    double At_c_norm(int t, const Vec& Ccx) override {
        SmallScope sc_(this);
        need_ws(t);
        if (ca_rows <= 0 || t <= 0) return 0.0;
        up(dvec[0].get(), Ccx.data(), t);
        launches += enl_small::gemv_n(dCA.get(), n, n, t, dvec[0].get(), 1.0, nullptr, 0.0, dvec[1].get(), st);
        enl_small::norm_range_kernel<<<1, 1024, 0, st>>>(dvec[1].get(), 0, n, dscal.get());
        ++launches;
        down(0, dscal.get(), 1);
        sm_sync();
        return hst[0];
    }
    // EF:348-423 (the driver has checked the sizes): p1 from R_A' (t == rankA) or F_L11 (t > rankA), G at x,
    // E = (Q1' G) Q1 -- G is symmetric, so Q1' G = (G Q1)' --, permuted by F_L11.p when t > rankA, [W21 | W22] from E and
    // J~Q1 (J2'J2, J2'J1 and J2'r are invariant under the left orthogonal factor of [J | r], so the compressed problem gives
    // them), d = -W21 p1 - J2' r~, the upper Cholesky factor of (W22 + W22') / 2, two triangular solves, p = Q1 [p1; p2].
    int newton_direction(const double* x, const Vec& lam, const int* active, int t, int rankA, const Vec& Ccx, Vec& p) override {
        if (!midsize) return -1;
        SmallScope sc_(this);
        need_ws(t);
        ensure_jq1();
        const int mt = n + 1, k2 = n - rankA;
        const double* rtd = dJc + (size_t)mt * n;
        double* const v[6] = {dvec[0].get(), dvec[1].get(), dvec[2].get(), dvec[3].get(), dvec[4].get(), dvec[5].get()};
        double* p1 = v[2];                                               // rankA entries
        if (t > 0) {
            Vec b0(t);
            for (int i = 0; i < t; ++i) b0[i] = -Ccx[hpA[i]];
            up(v[0], b0.data(), t);
            if (t == rankA) {
                k_trsv_upperT(dFA.get(), n, t, v[0]);                    // R_A' p1 = -c[P]
                p1 = v[0];
            } else {
                k_reflect(dFL.get(), fl_rows, fl_k, dtauL.get(), v[0], 1);   // b = Q_L11' (-c[P])
                k_copy_pad(v[1], v[0], rankA, rankA);
                k_trsv_upper(dFL.get(), fl_rows, rankA, v[1]);          // R11 \ b[1:rankA]
                if (rankA > 0) {
                    sm_check(cudaMemsetAsync(v[2], 0, sizeof(double) * rankA, st), "memset");
                    enl_small::scatter_perm_kernel<<<(rankA + 255) / 256, 256, 0, st>>>(v[2], v[1], dpL.get(), rankA, rankA);
                    ++launches;
                }
            }
        }
        double *G = dG.get(), *E = dE.get(), *Wn = dWn.get(), *U = dU.get();
        if (pt.hessian(x, lam.data(), active, t, G) != 0) throw std::runtime_error(pt.last_error());
        if (fa_k > 0) {
            double* TA = wy_t_of(dFA.get(), n, fa_k, dtauA.get());
            launches += enl_small::mulq_device(G, n, n, dFA.get(), n, fa_k, dtauA.get(), ww, st, TA, false);   // G Q1
            dim3 grid((n + 31) / 32, (n + 31) / 32), block(32, 8);
            enl_small::transpose_kernel<<<grid, block, 0, st>>>(G, n, E);                                     // Q1' G
            ++launches;
            launches += enl_small::mulq_device(E, n, n, dFA.get(), n, fa_k, dtauA.get(), ww, st, TA, false);   // (Q1' G) Q1
            n_dev_mulq += 2;
        } else {
            sm_check(cudaMemcpyAsync(E, G, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, st), "D2D");
        }
        const long long nw = (long long)k2 * n;
        enl_small::newton_assemble_kernel<<<(unsigned)std::min<long long>((nw + 7) / 8, 148 * 16), 256, 0, st>>>(
            E, n, rankA, t > rankA ? dpL.get() : nullptr, dJQ1.get(), mt, Wn);
        const long long nu = (long long)k2 * k2;
        enl_small::newton_sym_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, st>>>(Wn, k2, rankA, U);
        launches += 2 + enl_small::gemv_t(dJQ1.get() + (size_t)rankA * mt, mt, mt, k2, rtd, v[3], st);   // J2' r~
        launches += enl_small::gemv_n(Wn, k2, k2, rankA, p1, -1.0, v[3], -1.0, v[4], st);               // d = -W21 p1 - J2' r~
        if (enl_small::potrf_upper(U, k2, k2, dinfo.get(), st) < 0) throw std::runtime_error("Newton step: reduced Hessian too large");
        ++launches;
        int info = 0;
        sm_check(cudaMemcpyAsync(hsti.get(), dinfo.get(), sizeof(int), cudaMemcpyDeviceToHost, st), "D2H");
        sm_sync();
        info = hsti[0];
        ++n_newton;
        if (info != 0) {
            p.assign(n, 0.0);
            return 1;
        }
        k_trsv_upperT(U, k2, k2, v[4]);
        k_trsv_upper(U, k2, k2, v[4]);
        if (rankA > 0) sm_check(cudaMemcpyAsync(v[5], p1, sizeof(double) * rankA, cudaMemcpyDeviceToDevice, st), "D2D");
        sm_check(cudaMemcpyAsync(v[5] + rankA, v[4], sizeof(double) * k2, cudaMemcpyDeviceToDevice, st), "D2D");
        k_reflect(dFA.get(), n, fa_k, dtauA.get(), v[5], 0);             // p = Q1 [p1; p2]
        down(0, v[5], n);
        sm_sync();
        p.assign(hst.get(), hst.get() + n);
        return 0;
    }
};

}  // namespace enl_large
