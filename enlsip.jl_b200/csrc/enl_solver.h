// enl_solver.h -- the ENLSIP iteration for one problem owned by one group of lanes.
//
// Device-side re-design of the reference hot path `enlsip` (src/enlsip_functions.jl = EF,
// EF:2638-2880) and everything it calls (EF:17-2517), for the batched regime of BASELINE.json:
// the whole solve -- forward-difference / analytic Jacobians, QRCP of the active-constraint
// Jacobian with pseudo-rank, QRCP of J*Q2, triangular solves, first/second order multiplier
// estimates, working-set update, subspace-minimisation and Newton fall-backs, penalty weights,
// Lindstrom-Wedin linesearch, termination tests -- runs inside one kernel with the state of the
// problem resident in shared memory and registers.  No intermediate ever goes to HBM.
//
// Deliberate differences from the reference's *execution* (never from its results):
//   * duplicate evaluations of the same point are deduplicated (SURVEY.md section 3.2);
//   * `J*F_A.Q` is formed once per factorisation and reused (EF:219, 526, 1249 recompute it);
//   * the always-reverted first-order deletion detour (EF:706-743, SURVEY.md T3) is skipped,
//     keeping its only surviving side effect (index_del reset, scaled-row rebuild);
//   * where Julia would throw or loop forever the solve ends with exit code -99 / -98.
// Semantic traps T1-T16 of SURVEY.md section 9 are reproduced (aliasing schedule of
// previous_iter.rx/cx, x_diff lag, min_norm_w! restart from K[4], ...).
#pragma once
#include "enl_base.h"
#include "enl_linalg.h"
#include "enl_families.h"

namespace enl {

struct Options {          // solver.jl:62-63 keyword arguments after defaulting, + EF:2646-2658
    int max_iter;         // 100
    int scaling;          // false
    int jac_mode;         // 0 analytic, 1 forward differences (cnls_model.jl:65-82)
    int second_derivatives;  // 1 (EF:2647); forced off when n+m >= 1000 (EF:2658)
    double time_limit;    // 1e3
    double eps_abs;       // 1e-10 (EF:2651; abs_tol is NOT forwarded, SURVEY.md T4)
    double eps_rel;       // rel_tol
    double eps_x;         // x_tol
    double eps_c;         // c_tol
    double eps_rank;      // sqrt(eps) (solver.jl:81)
};

constexpr int MAX_N = 32;  // largest number of parameters of a batched family (built in: <= 20; user families: <= 32)
struct Bounds {           // finite bounds in index order (cnls_model.jl:392-403)
    int nlo, nup;
    int lo_idx[MAX_N], up_idx[MAX_N];
    double lo_val[MAX_N], up_val[MAX_N];
};

constexpr int TRACE_HDR = 16;

template <class Fam, int G, int NT>
struct Layout {
    static constexpr int N = Fam::N, M = Fam::M, Q = Fam::Q, NNL = Fam::Q + Fam::NI;
    static constexpr int LMAX = NNL + Fam::MAXB;   // MAXB: bound rows the family may carry (0 or 2n)
    static constexpr int T = (LMAX < N) ? LMAX : N;
    static constexpr int PPC = NT / G;
    static constexpr int MS = (M + G - 1) / G;
    static constexpr int NS = (N > LMAX) ? N : LMAX;   // generic scratch length
    enum : int {
        oX = 0, oXPREV = oX + N, oXNEW = oXPREV + N, oCX = oXNEW + N, oCNEW = oCX + LMAX, oA = oCNEW + LMAX,
        oGRADF = oA + LMAX * N, oW = oGRADF + N, oWNEW = oW + LMAX, oK = oWNEW + LMAX, oACX = oK + 4 * LMAX,
        oAA = oACX + T, oDSC = oAA + T * N, oFA = oDSC + T, oTAUA = oFA + N * T, oFL = oTAUA + T,
        oTAUL = oFL + T * T, oR2 = oTAUL + T, oTAU2 = oR2 + N * N, oLAM = oTAU2 + N, oB = oLAM + T, oP = oB + T,
        oY = oP + N, oAP = oY + N, oAAP = oAP + LMAX, oV1C = oAAP + T, oVN1 = oV1C + LMAX, oVN2 = oVN1 + N,
        oS1 = oVN2 + N, oS2 = oS1 + NS, oS3 = oS2 + NS, oS4 = oS3 + NS, oS5 = oS4 + NS, oNW = oS5 + NS,
        oFS = oNW + 3 * N * N, nD = oFS + Fam::NSCAL
    };
    enum : int { iACT = 0, iINACT = iACT + LMAX, iPERMA = iINACT + LMAX, iPERML = iPERMA + T, iPERM2 = iPERML + T,
                 iPOS = iPERM2 + N, nI = iPOS + T };
    // r | J (n cols; J*Q1, then J1 | QR factor of J2 in place) | d | family row data
    static constexpr int DCOLS = N + 2 + Fam::NDCOLS;
    static constexpr size_t smem_bytes() {
        return (size_t)nD * PPC * 8 + (size_t)DCOLS * MS * NT * 8 + (size_t)nI * PPC * 4;
    }
};

struct IterRec {          // the scalar part of structures.jl:63-91
    int t, rankA, rankJ2, dimA, dimJ2, code, index_del, index_alpha_upp, nb_newton;
    bool restart, add, del;
    double alpha, beta, progress, predicted_reduction, grad_res, speed;
};

struct Outputs {          // per-batch output arrays (device or host memory depending on the build)
    double* x;            // [B, N]
    double* f;            // [B]
    int* exit_code;       // [B] raw EF code
    int* status;          // [B] convert_exit_code (cnls_model.jl:166-178)
    int* iters;           // [B] length(iterations_detail)
    int* nact;            // [B] |working set| at exit
    int* active;          // [B, LMAX] 1-based ids, 0 padded
    int* counters;        // [B, 2] nb_function_evaluations, nb_jacobian_evaluations (reference formula, T16)
    double* trace;        // optional [B, trace_cap, TRACE_HDR + N]
    int trace_cap;
};

template <class Fam, class Grp, int NT>
struct Solver {
    static constexpr int G = Grp::G;
    using LY = Layout<Fam, G, NT>;
    static constexpr int N = LY::N, M = LY::M, Q = LY::Q, NNL = LY::NNL, LMAX = LY::LMAX, T = LY::T, PPC = LY::PPC,
                         MS = LY::MS;
    using V = SV<PPC>;
    using VI = SI<PPC>;
    using D = DM<G, MS, NT>;

    // ---- views -------------------------------------------------------------------------
    V x, xprev, xnew, cx, cnew, A, gradf, w, wnew, K, acx, aA, dsc, FA, tauA, FL, tauL, R2, tau2, lam, b, p, y, Ap, aAp,
        v1c, vn1, vn2, s1, s2, s3, s4, s5, nw;
    VI active, inactive, permA, permL, perm2, posidx;
    D dR, dJ, dF, dD, dY;
    V fs;
    using FCtx = typename Fam::template Ctx<D, V>;
    // Nothing per-lane is stored in this object: it is one per PROBLEM and lives in shared memory, so
    // the non-inlined member functions reach it with shared loads instead of a per-thread stack copy.
    ENL_INL Grp grp() const { return Grp(); }
    ENL_INL Dist<Grp, G, MS, NT> dst() const { return Dist<Grp, G, MS, NT>(); }
    ENL_INL FCtx fctx() const { return FCtx{dY, fs}; }
    const Options& opt;
    const Bounds& bnd;

    // ---- scalar state ------------------------------------------------------------------
    int l, t, k_iter, ndetail, exit_code;
    int n_res, n_cons, n_jres, n_jcons;
    bool threw, hang;
    bool j2_factored;              // columns rankA.. of dJ hold the QR factor of J2 (else J2 itself)
    IterRec cur, prev;
    double rx_sum, active_cx_sum, f_detail, rdot_x1, cdot_x1, rdot_prev, cdot_prev;
    double jp_r, jp_jp;            // dot(Jp, rx), dot(Jp, Jp)
    double t_start;

    ENL_FN Solver(double* small, int* ints, double* distbase, int pid, const Options& o, const Bounds& bb)
        : opt(o), bnd(bb) {
#if defined(__CUDACC__)
        int s = (int)(small - enl_smem) + pid;
#else
        double* s = small + pid;
#endif
        auto mk = [&](int off) { return V{s + off * PPC}; };
        x = mk(LY::oX); xprev = mk(LY::oXPREV); xnew = mk(LY::oXNEW); cx = mk(LY::oCX); cnew = mk(LY::oCNEW);
        A = mk(LY::oA); gradf = mk(LY::oGRADF); w = mk(LY::oW); wnew = mk(LY::oWNEW); K = mk(LY::oK);
        acx = mk(LY::oACX); aA = mk(LY::oAA); dsc = mk(LY::oDSC); FA = mk(LY::oFA); tauA = mk(LY::oTAUA);
        FL = mk(LY::oFL); tauL = mk(LY::oTAUL); R2 = mk(LY::oR2); tau2 = mk(LY::oTAU2); lam = mk(LY::oLAM);
        b = mk(LY::oB); p = mk(LY::oP); y = mk(LY::oY); Ap = mk(LY::oAP); aAp = mk(LY::oAAP); v1c = mk(LY::oV1C);
        vn1 = mk(LY::oVN1); vn2 = mk(LY::oVN2); s1 = mk(LY::oS1); s2 = mk(LY::oS2); s3 = mk(LY::oS3);
        s4 = mk(LY::oS4); s5 = mk(LY::oS5); nw = mk(LY::oNW); fs = mk(LY::oFS);
#if defined(__CUDACC__)
        int ii = (int)(ints - reinterpret_cast<int*>(enl_smem)) + pid;
#else
        int* ii = ints + pid;
#endif
        auto mi = [&](int off) { return VI{ii + off * PPC}; };
        active = mi(LY::iACT); inactive = mi(LY::iINACT); permA = mi(LY::iPERMA); permL = mi(LY::iPERML);
        perm2 = mi(LY::iPERM2); posidx = mi(LY::iPOS);
#if defined(__CUDACC__)
        int grpb = (int)(distbase - enl_smem) + pid * G;
#else
        double* grpb = distbase + pid * G;
#endif
        D all{grpb};
        dR = all; dJ = all.cols(1); dF = dJ; dD = all.cols(1 + N); dY = all.cols(2 + N);
        l = NNL + bnd.nlo + bnd.nup;
    }

    // =====================================================================================
    // evaluation layer (cnls_model.jl:40-82, 381-406)
    // =====================================================================================
    ENL_FN void load_x(V src, double* xv) const {
#pragma unroll
        for (int j = 0; j < N; ++j) xv[j] = src[j];
    }

    // r(xv) -> rn[MS] (registers), c(xv) -> cout[l]
    ENL_NOINL void eval_point(const double* xv, double* rn, V cout) {
        Fam::template residuals<Grp, MS>(fctx(), grp(), xv, rn);
        double cnl[NNL > 0 ? NNL : 1];
        if (NNL > 0) Fam::template constraints<MS>(fctx(), xv, cnl);
#pragma unroll 1
        for (int i = 0; i < NNL; ++i) cout[i] = cnl[i];
#pragma unroll 1
        for (int j = 0; j < bnd.nlo; ++j) cout[NNL + j] = sub_rn(xv[bnd.lo_idx[j]], bnd.lo_val[j]);
#pragma unroll 1
        for (int j = 0; j < bnd.nup; ++j) cout[NNL + bnd.nlo + j] = sub_rn(bnd.up_val[j], xv[bnd.up_idx[j]]);
    }

    ENL_FN double sumsq_regs(const double* rn) const {
        double s = 0.0;
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) s += rn[sl] * rn[sl];
        return grp().sum(s);
    }

    // J(x) -> dJ  (x in the small state, r(x) in dR)
    const double* mat_J = nullptr;       // step_only: the Jacobian is an input ([N][M] column major), not evaluated
    ENL_NOINL void eval_res_jacobian() {
        if (mat_J) {
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                const int row = sl * G + grp().lane;
#pragma unroll
                for (int j = 0; j < N; ++j) dJ.at(sl, j) = (row < M) ? mat_J[(size_t)j * M + row] : 0.0;
            }
            j2_factored = false;
            grp().sync();
            return;
        }
        double xv[N];
        load_x(x, xv);
        double out[MS * N];
        if (opt.jac_mode == 0) {
            Fam::template jac_residuals<Grp, MS>(fctx(), grp(), xv, out);
        } else {
            double r0[MS], dl[N];
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) r0[sl] = dR.at(sl, 0);
#pragma unroll
            for (int j = 0; j < N; ++j) dl[j] = mul_rn(fmax(fabs(xv[j]), 1.0), SQRT_EPS);
            fd_res(xv, r0, dl, out);
        }
#pragma unroll
        for (int sl = 0; sl < MS; ++sl)
#pragma unroll
            for (int j = 0; j < N; ++j) dJ.at(sl, j) = out[sl * N + j];
        j2_factored = false;
        grp().sync();
    }

    template <class F2 = Fam>
    ENL_FN typename std::enable_if<F2::HAS_FAST_FD>::type fd_res(const double* xv, const double* r0, const double* dl,
                                                                 double* out) {
        F2::template fd_jac_residuals<Grp, MS>(fctx(), grp(), xv, r0, dl, out);
    }
    template <class F2 = Fam>
    ENL_FN typename std::enable_if<!F2::HAS_FAST_FD>::type fd_res(const double* xv, const double* r0, const double* dl,
                                                                  double* out) {
        double xf[N], rf[MS];
#pragma unroll
        for (int j = 0; j < N; ++j) {
#pragma unroll
            for (int i = 0; i < N; ++i) xf[i] = xv[i];
            xf[j] = add_rn(xv[j], dl[j]);
            F2::template residuals<Grp, MS>(fctx(), grp(), xf, rf);
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) out[sl * N + j] = div_z(sub_rn(rf[sl], r0[sl]), dl[j]);
        }
    }

    // A(x) (l x n, row major) -> A
    ENL_NOINL void eval_cons_jacobian() {
        double xv[N];
        load_x(x, xv);
        if (NNL > 0) {
            double An[(NNL > 0 ? NNL : 1) * N];
            if (opt.jac_mode == 0) {
                Fam::template jac_constraints<MS>(fctx(), xv, An);
            } else {
                double xf[N], cf[NNL > 0 ? NNL : 1];
#pragma unroll 1
                for (int j = 0; j < N; ++j) {
                    double dj = mul_rn(fmax(fabs(xv[j]), 1.0), SQRT_EPS);
#pragma unroll 1
                    for (int i = 0; i < N; ++i) xf[i] = xv[i];
                    xf[j] = add_rn(xv[j], dj);
                    Fam::template constraints<MS>(fctx(), xf, cf);
#pragma unroll 1
                    for (int i = 0; i < NNL; ++i) An[i * N + j] = div_z(sub_rn(cf[i], cx[i]), dj);
                }
            }
#pragma unroll 1
            for (int i = 0; i < NNL * N; ++i) A[i] = An[i];
        }
    }

    // rows of A for the bounds are constant (+-e_j, cnls_model.jl:393-403): written once per solve
    ENL_NOINL void init_bound_rows() {
#pragma unroll 1
        for (int j = 0; j < bnd.nlo; ++j)
#pragma unroll 1
            for (int c = 0; c < N; ++c) A[(NNL + j) * N + c] = (c == bnd.lo_idx[j]) ? 1.0 : 0.0;
#pragma unroll 1
        for (int j = 0; j < bnd.nup; ++j)
#pragma unroll 1
            for (int c = 0; c < N; ++c) A[(NNL + bnd.nlo + j) * N + c] = (c == bnd.up_idx[j]) ? -1.0 : 0.0;
    }

    // gradient of the objective J' r and ||r||^2 (EF:2690, 2734-2735, 2829-2830)
    ENL_NOINL void grad_and_sumsq() {
        double rr[MS];
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) rr[sl] = dR.at(sl, 0);
#pragma unroll 1
        for (int j = 0; j < N; ++j) {
            double s = 0.0;
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) s += dJ.at(sl, j) * rr[sl];
            gradf[j] = grp().sum(s);
        }
        rx_sum = sumsq_regs(rr);
    }

    // =====================================================================================
    // working set (structures.jl:209-267, EF:608-650, 826-859)
    // =====================================================================================
    ENL_FN void ws_remove(int s) {  // 1-based position in `active`
        int lt = l - t;
        int id = active[s - 1];
        int pos = lt;               // insert `id` into the sorted prefix inactive[0..lt)
#pragma unroll 1
        while (pos > 0 && inactive[pos - 1] > id) { inactive[pos] = inactive[pos - 1]; --pos; }
        inactive[pos] = id;
#pragma unroll 1
        for (int i = s; i <= t - 1; ++i) active[i - 1] = active[i];
        active[t - 1] = 0;
        t -= 1;
    }
    ENL_FN void ws_add(int s) {     // 1-based position in `inactive`
        int id = inactive[s - 1];
        int pos = t;
#pragma unroll 1
        while (pos > 0 && active[pos - 1] > id) { active[pos] = active[pos - 1]; --pos; }
        active[pos] = id;
#pragma unroll 1
        for (int i = s; i <= l - t - 1; ++i) inactive[i - 1] = inactive[i];
        inactive[l - t - 1] = 0;
        t += 1;
    }

    ENL_NOINL bool evaluate_violated_constraints(int index_alpha_upp) {
        const double delta = 0.1;
        int cap = imin(l, N);
        bool added = false;
        int swaps = 0;
        if (l > t) {
            int i = 1;
#pragma unroll 1
            while (i <= l - t) {
                int kk = inactive[i - 1];
                double ck = cx[kk - 1];
                if (ck < SQRT_EPS || (kk == index_alpha_upp && ck < delta)) {
                    if (t >= cap) {
                        int worst_k = 0;
                        double worst_val = -INFINITY;
#pragma unroll 1
                        for (int j = Q + 1; j <= t; ++j) {
                            double cj = cx[active[j - 1] - 1];
                            if (cj > worst_val) { worst_val = cj; worst_k = j; }
                        }
                        if (worst_k > 0 && worst_val > ck) {
                            // reference swap cycle (EF:621-647): provably endless beyond this cap
                            if (++swaps > 4 * l + 16) { hang = true; return added; }
                            ws_remove(worst_k);
                        } else {
                            ++i;
                            continue;
                        }
                    }
                    ws_add(i);
                    added = true;
                } else {
                    ++i;
                }
            }
        }
        return added;
    }

    // active_C.cx = cx[active], active_C.A = A[active, :]  (EF:2683-2687, 2754-2755, 2854-2855)
    ENL_NOINL void gather_active() {
#pragma unroll 1
        for (int i = 0; i < t; ++i) {
            int id = active[i] - 1;
            acx[i] = cx[id];
#pragma unroll 1
            for (int c = 0; c < N; ++c) aA[i * N + c] = A[id * N + c];
        }
    }

    // structures.jl:160-178
    ENL_NOINL void evaluate_scaling() {
#pragma unroll 1
        for (int i = 0; i < t; ++i) {
            double row = nrm2_small(aA.off(i * N), N);
            dsc[i] = row;
            if (opt.scaling) {
                if (fabs(row) < EPS) row = 1.0;
#pragma unroll 1
                for (int c = 0; c < N; ++c) aA[i * N + c] = aA[i * N + c] / row;
                acx[i] = acx[i] / row;
                dsc[i] = 1.0 / row;
            }
        }
    }

    // =====================================================================================
    // multipliers (EF:461-603)
    // =====================================================================================
    ENL_NOINL void factor_A() {
#pragma unroll 1
        for (int c = 0; c < t; ++c)
#pragma unroll 1
            for (int r = 0; r < N; ++r) FA[c * N + r] = aA[c * N + r];
        qrcp_small(FA, N, N, t, tauA, permA, vn1, vn2);
    }
    ENL_NOINL void factor_L11() {
#pragma unroll 1
        for (int c = 0; c < t; ++c)
#pragma unroll 1
            for (int r = 0; r < t; ++r) FL[c * T + r] = (c <= r) ? FA[r * N + c] : 0.0;
        qrcp_small(FL, T, t, t, tauL, permL, vn1, vn2);
    }

    ENL_NOINL void first_lagrange() {
        int pr = pseudo_rank(FA, N, t, opt.eps_rank);
#pragma unroll 1
        for (int i = 0; i < N; ++i) s1[i] = gradf[i];
        apply_qt_small(FA, N, N, t, tauA, s1);
#pragma unroll 1
        for (int i = 0; i < t; ++i) s2[i] = (i < pr) ? s1[i] : 0.0;
        if (!solve_upper_small(FA, N, pr, s2)) threw = true;
        double gr = 0.0;
#pragma unroll 1
        for (int i = pr; i < N; ++i) gr += s1[i] * s1[i];
        cur.grad_res = (N > pr) ? sqrt(gr) : 0.0;
#pragma unroll 1
        for (int j = 0; j < t; ++j) s3[j] = (j < pr) ? -acx[permA[j]] : 0.0;
        if (!solve_upperT_small(FA, N, pr, s3)) threw = true;
        if (!solve_upper_small(FA, N, pr, s3)) threw = true;
#pragma unroll 1
        for (int j = 0; j < t; ++j) lam[permA[j]] = s2[j] + s3[j];
        if (opt.scaling)
#pragma unroll 1
            for (int i = 0; i < t; ++i) lam[i] = lam[i] * dsc[i];
    }

    // uses y = Q1' p_gn and J*Q1 in dJ
    ENL_NOINL void second_lagrange() {
        int pr = pseudo_rank(FA, N, t, SQRT_EPS);
        // r + J p_gn = r + J1 p1 + J2 p2 with J2 p2 = Q3 [d(0:kq); 0]  =>  r + J p_gn = -Q3 [0; d(kq:)]
        // (J2 itself has been overwritten by its QR factor; here rankJ2 == kq == min(m, n - rankA))
        double v[MS];
        {
            const int kq = imin(M, N - cur.rankA);
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                int row = sl * G + grp().lane;
                v[sl] = (row >= kq) ? -dD.at(sl, 0) : 0.0;
            }
            dst().apply_q_regs(dF, kq, tau2, v);
        }
#pragma unroll 1
        for (int j = 0; j < t; ++j) {
            double s = 0.0;
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) s += dJ.at(sl, j) * v[sl];
            s1[j] = grp().sum(s);
        }
#pragma unroll 1
        for (int j = pr; j < t; ++j) s1[j] = 0.0;
        if (!solve_upper_small(FA, N, pr, s1)) threw = true;
#pragma unroll 1
        for (int j = 0; j < t; ++j) lam[permA[j]] = s1[j];
        if (opt.scaling)
#pragma unroll 1
            for (int i = 0; i < t; ++i) lam[i] = lam[i] * dsc[i];
    }

    ENL_NOINL int check_constraint_deletion(double grad_res) {
        double lam_max = 1.0;
        if (t > 0) {
            lam_max = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) lam_max = fmax(lam_max, fabs(lam[i]));
        }
        double sq_rel = SQRT_EPS * lam_max;
        int s = 0;
        if (t > Q) {
            double e = sq_rel;
#pragma unroll 1
            for (int i = Q + 1; i <= t; ++i) {
                double row_i = opt.scaling ? 1.0 / dsc[i - 1] : dsc[i - 1];
                double v = row_i * lam[i - 1];
                if (v <= sq_rel && v <= e) { e = v; s = i; }
            }
            if (grad_res > -e * 10.0) s = 0;
        }
        return s;
    }

    ENL_FN void minmax_lagrangian_mult(double& sigmin, double& lam_abs_max) {
        lam_abs_max = 0.0;
        sigmin = INFINITY;
        if (t > Q) {
#pragma unroll 1
            for (int i = 0; i < t; ++i) lam_abs_max = fmax(lam_abs_max, fabs(lam[i]));
#pragma unroll 1
            for (int i = Q; i < t; ++i) {
                double rows = opt.scaling ? 1.0 / dsc[i] : dsc[i];
                double li = lam[i];
                if (li * rows <= -SQRT_EPS && li < sigmin) sigmin = li;
            }
        }
    }

    // =====================================================================================
    // search directions (EF:116-234)
    // =====================================================================================
    // writes y = [p1; p2], p = Q1 y, b (t entries), dD = Q3'(-J1 p1 - r)
    ENL_NOINL void sub_search_direction(int rankA, int dimA, int dimJ2, int code) {
        const int k2 = N - rankA;
        const int kq = imin(M, k2);
        if (code == 1) {
#pragma unroll 1
            for (int j = 0; j < t; ++j) { double v = -acx[permA[j]]; b[j] = v; y[j] = v; }
            if (!solve_upperT_small(FA, N, t, y)) threw = true;
        } else {
#pragma unroll 1
            for (int j = 0; j < t; ++j) s1[j] = -acx[permA[j]];
            apply_qt_small(FL, T, t, t, tauL, s1);
#pragma unroll 1
            for (int j = 0; j < t; ++j) b[j] = s1[j];
            if (dimA > t || dimA < 0) { threw = true; dimA = imax(0, imin(dimA, t)); }
#pragma unroll 1
            for (int j = 0; j < t; ++j) s2[j] = (j < dimA) ? s1[j] : 0.0;
            if (!solve_upper_small(FL, T, dimA, s2)) threw = true;
#pragma unroll 1
            for (int j = 0; j < t; ++j) s3[permL[j]] = s2[j];
#pragma unroll 1
            for (int j = 0; j < rankA; ++j) y[j] = s3[j];
        }
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) {
            double acc = 0.0;
#pragma unroll 1
            for (int c = 0; c < rankA; ++c) acc += dJ.at(sl, c) * y[c];
            dD.at(sl, 0) = -acc - dR.at(sl, 0);
        }
        grp().sync();
        dst().apply_qt(dF, kq, tau2, dD);
        if (dimJ2 > kq || dimJ2 < 0) { threw = true; dimJ2 = imax(0, imin(dimJ2, kq)); }
#pragma unroll 1
        for (int j = 0; j < dimJ2; ++j) s2[j] = dD.row(j, 0);
        if (!solve_upper_small(R2, N, dimJ2, s2)) threw = true;
#pragma unroll 1
        for (int j = 0; j < k2; ++j) y[rankA + perm2[j]] = (j < dimJ2) ? s2[j] : 0.0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) p[j] = y[j];
        apply_q_small(FA, N, N, t, tauA, p);
    }

    ENL_NOINL void gn_search_direction(int rankA) {
        int code = (rankA == t) ? 1 : -1;
        dst().mul_q_right(dJ, N, FA, N, t, tauA);
        const int k2 = N - rankA;
        dF = dJ.cols(rankA);          // J2 is factored in place; J1 = columns [0, rankA) stays intact
        grp().sync();
        dst().qrcp(dF, M, k2, tau2, perm2, vn1, vn2, R2, N);
        j2_factored = true;
        int rankJ2 = pseudo_rank(R2, N, imin(M, k2), opt.eps_rank);
        sub_search_direction(rankA, rankA, rankJ2, code);
        cur.rankA = rankA;
        cur.rankJ2 = rankJ2;
        cur.dimA = rankA;
        cur.dimJ2 = rankJ2;
    }

    // EF:686-795
    ENL_NOINL void update_working_set() {
        factor_A();
        first_lagrange();
        int s = check_constraint_deletion(cur.grad_res);
        if (s != 0) {
            // first-order deletion: always reverted by the reference (T3); surviving side effects only
            cur.index_del = 0;
            cur.del = false;
            if (opt.scaling) {
#pragma unroll 1
                for (int i = 0; i < t; ++i) {
                    int id = active[i] - 1;
#pragma unroll 1
                    for (int c = 0; c < N; ++c) aA[i * N + c] = A[id * N + c] * dsc[i];
                }
                factor_A();
            }
        }
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            int rankA = pseudo_rank(FA, N, t, opt.eps_rank);
            factor_L11();
            gn_search_direction(rankA);
            if (pass == 0 && t == rankA && cur.rankJ2 == imin(M, N - rankA)) {
                second_lagrange();
                int s2 = check_constraint_deletion(0.0);
                if (s2 != 0) {
                    int id = active[s2 - 1];
#pragma unroll 1
                    for (int i = s2; i <= t - 1; ++i) {
                        lam[i - 1] = lam[i];
                        dsc[i - 1] = dsc[i];
                        acx[i - 1] = acx[i];
#pragma unroll 1
                        for (int c = 0; c < N; ++c) aA[(i - 1) * N + c] = aA[i * N + c];
                    }
                    ws_remove(s2);
                    cur.del = true;
                    cur.index_del = id;
                    eval_res_jacobian();   // dJ holds J*Q1: re-evaluate J(x) (deterministic)
                    factor_A();
                    continue;
                }
            }
            break;
        }
    }

    // =====================================================================================
    // subspace dimension heuristics (EF:864-1176)
    // =====================================================================================
    ENL_FN int gn_previous_step(V tau, double tau_prk, int mindim, V rho, double rho_prk, int prank) {
        const double tau_max = 2e-1, rho_min = 5e-1;
        int pm1 = prank - 1;
        if (mindim > pm1) return mindim;
        int kk = pm1;
#pragma unroll 1
        while ((tau[kk - 1] >= tau_max * tau_prk || rho[kk - 1] <= rho_min * rho_prk) && kk > mindim) --kk;
        return (kk > mindim) ? kk : imax(mindim, pm1);
    }

    ENL_NOINL int subspace_min_previous_step(V tau, V rho, int len, double rho_prk, double c1, int pseudo_rk, int pdim,
                                          double progress, double plp, double prelin_prev, double prev_alpha) {
        const double stepb = 2e-1, pgb1 = 3e-1, pgb2 = 1e-1, predb = 7e-1, rlenb = 2.0, c2 = 1e2;
        auto ok = [&](int i) { if (i < 1 || i > len) { threw = true; return false; } return true; };
        if (prev_alpha < stepb && progress <= pgb1 * plp * plp && progress <= pgb2 * prelin_prev * prelin_prev) {
            int dim = imax(1, pdim - 1);
            if (pdim > 1) {
                if (!ok(dim)) return pseudo_rk;
                if (rho[dim - 1] > c1 * rho_prk) return dim;
            }
        }
        int dim = pdim;
        bool first_cond = false;
        if (pdim < len) {
            if (!ok(dim) || !ok(dim + 1)) return pseudo_rk;
            first_cond = ((rho[dim - 1] > predb * rho_prk) && (rlenb * tau[dim - 1] < tau[dim])) || (c2 * tau[dim - 1] < tau[dim]);
        }
        if (first_cond) return dim;
        int i1 = pdim - 1;
        if (i1 <= 0) return pseudo_rk;
        int best = 0;
#pragma unroll 1
        for (int i = i1; i <= pdim; ++i) {
            if (!ok(i)) return pseudo_rk;
            if (rho[i - 1] > predb * rho_prk) { if (best == 0) best = i; }
        }
        return best == 0 ? pseudo_rk : best;
    }

    // R: column major factor (ld), yv: first rankR entries of the right-hand side
    ENL_NOINL int determine_solving_dim(int pdim, int rankR, double plp, double obj_progress, double prelin_prev, V R, int ld,
                                     V yv, double prev_alpha, bool restart) {
        const double c1 = 0.1;
        int newdim = rankR;
        int mindim = 1;
        if (rankR > 0) {
            V sd = s4, rh = s5;
            sd[0] = fabs(yv[0]);
            rh[0] = fabs(yv[0] / R[0]);
#pragma unroll 1
            for (int i = 1; i < rankR; ++i) {
                double a = yv[i], r = yv[i] / R[i * ld + i];
                rh[i] = sqrt(rh[i - 1] * rh[i - 1] + r * r);
                sd[i] = sqrt(sd[i - 1] * sd[i - 1] + a * a);
            }
            double nrm_sd = sd[rankR - 1], nrm_rh = rh[rankR - 1];
            double dsum = 0.0, psimax = 0.0;
#pragma unroll 1
            for (int i = 0; i < rankR; ++i) {
                dsum += sd[i] * sd[i];
                double psi = sqrt(dsum) * fabs(R[i * ld + i]);
                if (psi > psimax) { psimax = psi; mindim = i + 1; }
            }
            if (!restart) {
                int suggested;
                if (pdim == rankR || pdim <= 0)
                    suggested = gn_previous_step(sd, nrm_sd, mindim, rh, nrm_rh, rankR);
                else
                    suggested = subspace_min_previous_step(sd, rh, rankR, nrm_rh, c1, rankR, pdim, obj_progress, plp,
                                                           prelin_prev, prev_alpha);
                newdim = imax(mindim, suggested);
            } else {
                newdim = imax(0, imin(rankR, pdim));
            }
        }
        return newdim;
    }

    // bsub = Q2'(-c_act[P1]) in s1 on entry (t entries); returns dims; uses dD as scratch
    ENL_NOINL void choose_subspace_dimensions(int rankA, int rankJ2, bool restart, int& dimA, int& dimJ2) {
        const double alpha_low = 0.2;
        double prev_alpha = prev.alpha;
        int pdA;
        const int k2 = N - rankA;
        const int kq = imin(M, k2);
        if (rankA <= 0) {
            dimA = 0;
            pdA = 0;
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) dD.at(sl, 0) = -dR.at(sl, 0);
        } else {
            pdA = abs(prev.dimA) + t - prev.t;
            if (pdA > t) { threw = true; pdA = t; }
            double sb = 0.0, sa = 0.0;
#pragma unroll 1
            for (int j = 0; j < t; ++j) {
                sb += b[j] * b[j];
                if (j < pdA) sa += b[j] * b[j];
            }
            double nrm_b = sqrt(sb), nrm_b_asprev = sqrt(sa);
            double cprog = cdot_prev - active_cx_sum;
            dimA = determine_solving_dim(pdA, rankA, nrm_b, cprog, nrm_b_asprev, FL, T, b, prev_alpha, restart);
            if (dimA > t || rankA - dimA < 0) { threw = true; dimA = imin(dimA, rankA); }
#pragma unroll 1
            for (int j = 0; j < rankA; ++j) s2[j] = (j < dimA) ? b[j] : 0.0;
            if (!solve_upper_small(FL, T, dimA, s2)) threw = true;
#pragma unroll 1
            for (int i = 0; i < rankA; ++i) {
                double acc = 0.0;
#pragma unroll 1
                for (int j = 0; j < rankA; ++j)
                    if (permL[j] == i) acc += s2[j];
                s3[i] = acc;
            }
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                double acc = 0.0;
#pragma unroll 1
                for (int c = 0; c < rankA; ++c) acc += dJ.at(sl, c) * s3[c];
                dD.at(sl, 0) = -(dR.at(sl, 0) + acc);
            }
        }
        grp().sync();
        if (rankJ2 > 0) dst().apply_qt(dF, kq, tau2, dD);
        int pdJ = abs(prev.dimJ2) + prev.t - t;
        if (pdJ > M) { threw = true; pdJ = M; }
        double nrm_d_asprev = sqrt(dst().prefix_sq(dD, pdJ));
        double nrm_d = sqrt(dst().prefix_sq(dD, M));
        double rprog = rdot_prev - rx_sum;
        if (rankJ2 > M) { threw = true; }
#pragma unroll 1
        for (int j = 0; j < rankJ2 && j < M; ++j) s2[j] = dD.row(j, 0);
        dimJ2 = determine_solving_dim(pdJ, rankJ2, nrm_d, rprog, nrm_d_asprev, R2, N, s2, prev_alpha, restart);
        if (!restart && prev_alpha >= alpha_low) {
            dimA = imax(dimA, pdA);
            dimJ2 = imax(dimJ2, pdJ);
        }
    }

    // EF:943-1030
    ENL_NOINL int check_gn_direction(double b1nrm, double d1nrm, double d1nrm_as_km1, double dnrm, double active_c_sum,
                                  int rankA, bool restart, bool added, bool deleted, double& beta_k) {
        const double delta = 1e-1;
        const double c1 = 0.5, c2 = 0.1, c3 = 4.0, c4 = 10.0, c5 = 0.05;
        beta_k = sqrt(d1nrm * d1nrm + b1nrm * b1nrm);
        int method = 1;
        bool newton_or_restart = (prev.code == 2) || restart;
        bool first_iter = (k_iter == 0);
        bool submin_prev = prev.code == -1;
        bool add_or_del = added || deleted;
        bool conv_lower = beta_k < c1 * prev.beta;
        bool progress_not_close = (prev.progress > c2 * prev.predicted_reduction) && (dnrm <= c3 * beta_k);
        if (newton_or_restart || (!first_iter && (submin_prev || !(add_or_del || conv_lower || progress_not_close)))) {
            method = -1;
            double nonlin_k = sqrt(d1nrm * d1nrm + active_c_sum);
            double nonlin_km1 = sqrt(d1nrm_as_km1 * d1nrm_as_km1 + active_c_sum);
            bool to_reduce = false;
            if (Q < t) {
                bool any_ge = false, any_neg = false;
#pragma unroll 1
                for (int i = Q; i < t; ++i) {
                    double rows = opt.scaling ? 1.0 / dsc[i] : dsc[i];
                    if (lam[i] * rows >= -SQRT_EPS) any_ge = true;
                    if (lam[i] < 0) any_neg = true;
                }
                to_reduce = to_reduce || (any_ge && any_neg);
            }
            if (l - t > 0) {
                bool any_small = false;
#pragma unroll 1
                for (int j = 0; j < l - t; ++j)
                    if (cx[inactive[j] - 1] < delta) any_small = true;
                to_reduce = to_reduce || any_small;
            }
            bool newton_previously = (prev.code == 2) && !deleted;
            bool cond4 = active_c_sum > c2;
            bool cond5 = deleted || added || to_reduce || (t == N && t == rankA);
            double eps_ = fmax(1e-2, 10.0 * EPS);
            bool cond6 = !((l == Q) || (rankA <= t)) && !((beta_k < eps_ * dnrm) || (b1nrm < eps_ && M == N - t));
            if (newton_previously || !(cond4 || cond5 || cond6)) {
                bool cond7 = (prev.alpha < c5 && nonlin_km1 < c2 * nonlin_k) || (M == N - t);
                bool cond8 = !(dnrm <= c4 * beta_k);
                if (newton_previously || cond7 || cond8) method = 2;
            }
        }
        return method;
    }

    // =====================================================================================
    // Newton direction (EF:243-423)
    // =====================================================================================
    ENL_NOINL bool newton_search_direction(int rankA) {
        const double e1 = 6.055454452393343e-06;  // eps^(1/3)
        V Gm = nw, Em = nw.off(N * N), Wm = nw.off(2 * N * N);
        // p1 -> y[0..rankA)
        if (t == rankA) {
#pragma unroll 1
            for (int j = 0; j < t; ++j) y[j] = -acx[permA[j]];
            if (!solve_upperT_small(FA, N, t, y)) threw = true;
        } else {
#pragma unroll 1
            for (int j = 0; j < t; ++j) s1[j] = -acx[permA[j]];
            apply_qt_small(FL, T, t, t, tauL, s1);
#pragma unroll 1
            for (int j = 0; j < rankA; ++j) s2[j] = s1[j];
            if (!solve_upper_small(FL, T, rankA, s2)) threw = true;
#pragma unroll 1
            for (int i = 0; i < rankA; ++i) {
                double acc = 0.0;
#pragma unroll 1
                for (int j = 0; j < rankA; ++j)
                    if (permL[j] == i) acc += s2[j];
                y[i] = acc;
            }
        }
        if (rankA == N) { threw = true; return true; }   // EF:379-381 returns a bare vector -> TypeError
        // J2 was overwritten by its QR factor: re-evaluate J(x) (deterministic) and form J*Q1 again
        eval_res_jacobian();
        dst().mul_q_right(dJ, N, FA, N, t, tauA);
        grp().sync();
        double xv[N], xw[N], fa[MS], fb[MS];
        load_x(x, xv);
        double rr[MS];
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) rr[sl] = dR.at(sl, 0);
#pragma unroll 1
        for (int kk = 0; kk < N; ++kk)
#pragma unroll 1
            for (int j = 0; j <= kk; ++j) {
                double ek = fmax(fabs(xv[kk]), 1.0) * e1;
                double ej = fmax(fabs(xv[j]), 1.0) * e1;
                double cacc[LMAX];
                // four stencil points, order of EF:259-266 / 308-315
#pragma unroll 1
                for (int q4 = 0; q4 < 4; ++q4) {
#pragma unroll 1
                    for (int i = 0; i < N; ++i) xw[i] = xv[i];
                    double sj = (q4 == 0 || q4 == 2) ? ej : -ej;
                    double sk = (q4 < 2) ? ek : -ek;
                    xw[j] = add_rn(xw[j], sj);
                    xw[kk] = add_rn(xw[kk], sk);
                    eval_point(xw, fb, cnew);
                    n_res += 1; n_cons += 1;
                    double sgn = (q4 == 0 || q4 == 3) ? 1.0 : -1.0;
                    if (q4 == 0) {
#pragma unroll
                        for (int sl = 0; sl < MS; ++sl) fa[sl] = fb[sl];
#pragma unroll 1
                        for (int i = 0; i < l; ++i) cacc[i] = cnew[i];
                    } else {
#pragma unroll
                        for (int sl = 0; sl < MS; ++sl) fa[sl] = fa[sl] + sgn * fb[sl];
#pragma unroll 1
                        for (int i = 0; i < l; ++i) cacc[i] = cacc[i] + sgn * cnew[i];
                    }
                }
                double sr = 0.0;
#pragma unroll
                for (int sl = 0; sl < MS; ++sl) sr += fa[sl] * rr[sl];
                sr = grp().sum(sr) / (4 * ej * ek);
                double sc = 0.0;
#pragma unroll 1
                for (int i = 0; i < t; ++i) sc += cacc[active[i] - 1] * lam[i];
                sc = sc / (4.0 * ek * ej);
                Gm[j * N + kk] = sr - sc;
                Gm[kk * N + j] = sr - sc;
            }
        // E = Q1' * G * Q1
#pragma unroll 1
        for (int c = 0; c < N; ++c) apply_qt_small(FA, N, N, t, tauA, Gm.off(c * N));   // Q1' G (columns)
#pragma unroll 1
        for (int r = 0; r < N; ++r) {                                                    // (.) Q1 (rows)
#pragma unroll 1
            for (int c = 0; c < N; ++c) s1[c] = Gm[c * N + r];
            // row * Q1 = (Q1' row')'
            apply_qt_small(FA, N, N, t, tauA, s1);
#pragma unroll 1
            for (int c = 0; c < N; ++c) Em[c * N + r] = s1[c];
        }
        if (t > rankA) {
            if (t != N) { threw = true; return true; }   // E[P2,P2] is t x t, then E[rankA+1:n, .] -> BoundsError
#pragma unroll 1
            for (int c = 0; c < N; ++c)
#pragma unroll 1
                for (int r = 0; r < N; ++r) Gm[c * N + r] = Em[permL[c] * N + permL[r]];
#pragma unroll 1
            for (int i = 0; i < N * N; ++i) Em[i] = Gm[i];
        }
        const int k2 = N - rankA;
        // W22 = E22 + J2'J2 ; d = -(E21 + J2'J1) p1 - J2' r
#pragma unroll 1
        for (int a = 0; a < k2; ++a) {
#pragma unroll 1
            for (int c = 0; c < N; ++c) {
                double s = 0.0;
#pragma unroll
                for (int sl = 0; sl < MS; ++sl) s += dJ.at(sl, rankA + a) * dJ.at(sl, c);
                s1[c] = grp().sum(s);
            }
            double sjr = 0.0;
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) sjr += dJ.at(sl, rankA + a) * rr[sl];
            sjr = grp().sum(sjr);
            double dacc = 0.0;
#pragma unroll 1
            for (int c = 0; c < rankA; ++c) dacc += (Em[c * N + (rankA + a)] + s1[c]) * y[c];
            s2[a] = -dacc - sjr;
#pragma unroll 1
            for (int c2 = 0; c2 < k2; ++c2) Wm[c2 * N + a] = Em[(rankA + c2) * N + (rankA + a)] + s1[rankA + c2];
        }
        // symmetrise, Cholesky (upper, dpotrf), solve
#pragma unroll 1
        for (int a = 0; a < k2; ++a)
#pragma unroll 1
            for (int c = a; c < k2; ++c) {
                double v = (Wm[c * N + a] + Wm[a * N + c]) * 0.5;
                Gm[c * N + a] = v;   // upper part (row a, col c)
            }
#pragma unroll 1
        for (int j = 0; j < k2; ++j) {
            double ajj = Gm[j * N + j];
#pragma unroll 1
            for (int i = 0; i < j; ++i) ajj -= Gm[j * N + i] * Gm[j * N + i];
            if (!(ajj > 0.0)) {
#pragma unroll 1
                for (int i = 0; i < N; ++i) p[i] = 0.0;
#pragma unroll 1
                for (int i = 0; i < N; ++i) y[i] = 0.0;
                return true;
            }
            ajj = sqrt(ajj);
            Gm[j * N + j] = ajj;
#pragma unroll 1
            for (int c = j + 1; c < k2; ++c) {
                double v = Gm[c * N + j];
#pragma unroll 1
                for (int i = 0; i < j; ++i) v -= Gm[j * N + i] * Gm[c * N + i];
                Gm[c * N + j] = v / ajj;
            }
        }
        solve_upperT_small(Gm, N, k2, s2);
        solve_upper_small(Gm, N, k2, s2);
#pragma unroll 1
        for (int a = 0; a < k2; ++a) y[rankA + a] = s2[a];
#pragma unroll 1
        for (int j = 0; j < N; ++j) p[j] = y[j];
        apply_q_small(FA, N, N, t, tauA, p);
        return false;
    }

    // EF:1191-1291
    ENL_NOINL int search_direction_analys() {
        const int rankA = cur.rankA, rankJ2 = cur.rankJ2;
        double sb = 0.0;
#pragma unroll 1
        for (int j = 0; j < cur.dimA; ++j) sb += b[j] * b[j];
        double nrm_b1_gn = sqrt(sb);
        double nrm_d_gn = sqrt(dst().prefix_sq(dD, M));
        double nrm_d1_gn = sqrt(dst().prefix_sq(dD, cur.dimJ2));
        int pd = prev.dimJ2 + prev.t - t - 1;
        if (pd > M) { threw = true; pd = M; }
        double nrm_d1_asprev = sqrt(dst().prefix_sq(dD, pd));
        bool restart = cur.restart;
        int error_code = 0;
        double beta;
        int method = check_gn_direction(nrm_b1_gn, nrm_d1_gn, nrm_d1_asprev, nrm_d_gn, active_cx_sum, rankA, restart,
                                        cur.add, cur.del, beta);
        int dimA = rankA, dimJ2 = rankJ2;
        if (method == -1) {
#pragma unroll 1
            for (int j = 0; j < t; ++j) s1[j] = -acx[permA[j]];
            apply_qt_small(FL, T, t, t, tauL, s1);
#pragma unroll 1
            for (int j = 0; j < t; ++j) b[j] = s1[j];
            choose_subspace_dimensions(rankA, rankJ2, restart, dimA, dimJ2);
            if (!threw) sub_search_direction(rankA, dimA, dimJ2, -1);
            if (dimA == rankA && dimJ2 == rankJ2) method = 1;
        } else if (method == 2) {
            if (opt.second_derivatives) {
                bool nerr = newton_search_direction(rankA);
                dimA = -t;
                dimJ2 = t - N;
                cur.nb_newton += 1;
                if (nerr) error_code = -3;
            } else {
                error_code = -4;
            }
        }
        cur.dimA = dimA;
        cur.dimJ2 = dimJ2;
        cur.code = method;
        cur.speed = beta / prev.beta;
        cur.beta = beta;
        return error_code;
    }

    // =====================================================================================
    // merit function, penalty weights (EF:1307-1629)
    // =====================================================================================
    // psi(x + alpha p): leaves r in rn (registers) and c in cnew
    ENL_NOINL double psi(double alpha, V wv, double* rn) {
        double xv[N];
#pragma unroll
        for (int j = 0; j < N; ++j) xv[j] = add_rn(x[j], mul_rn(alpha, p[j]));
        eval_point(xv, rn, cnew);
        n_res += 1; n_cons += 1;
        double pen = 0.0;
#pragma unroll 1
        for (int i = 0; i < t; ++i) { int j = active[i] - 1; pen += wv[j] * (cnew[j] * cnew[j]); }
#pragma unroll 1
        for (int i = 0; i < l - t; ++i) {
            int j = inactive[i] - 1;
            if (cnew[j] < 0.0) pen += wv[j] * (cnew[j] * cnew[j]);
        }
        return 0.5 * (sumsq_regs(rn) + pen);
    }

    ENL_FN void assort(V wv) {
#pragma unroll 1
        for (int i = 0; i < t; ++i)
#pragma unroll 1
            for (int ii = 0; ii < 4; ++ii) {
                int kk = active[i] - 1;
                if (wv[kk] > K[ii * LMAX + kk]) {
#pragma unroll 1
                    for (int j = 3; j > ii; --j) K[j * LMAX + kk] = K[(j - 1) * LMAX + kk];
                    K[ii * LMAX + kk] = wv[kk];
                }
            }
    }

    // EF:1374-1423.  yv (nb_pos entries) and posidx are consumed.
    ENL_NOINL void min_norm_w(int ctrl, V wv, V w_old, V yv, double tau, int nb_pos) {
#pragma unroll 1
        for (int i = 0; i < l; ++i) wv[i] = w_old[i];
        if (nb_pos > 0) {
            double y_sum = 0.0;
#pragma unroll 1
            for (int i = 0; i < nb_pos; ++i) y_sum += yv[i] * yv[i];
            double y_norm = sqrt(y_sum);
            if (y_norm != 0.0)
#pragma unroll 1
                for (int i = 0; i < nb_pos; ++i) yv[i] = yv[i] / y_norm;
            double tau_new = tau, s = 0.0;
            int n_runch = nb_pos;
            bool terminated = false;
#pragma unroll 1
            while (!terminated) {
                tau_new -= s;
                double ymax = 0.0;
#pragma unroll 1
                for (int i = 0; i < nb_pos; ++i) ymax = fmax(ymax, fabs(yv[i]));
                double c = (ymax <= EPS) ? 1.0 : tau_new / y_sum;
                y_sum = 0.0;
                s = 0.0;
                int i_stop = n_runch;
                int kk = 1;
#pragma unroll 1
                while (kk <= n_runch) {
                    int i = posidx[kk - 1] - 1;
                    double buff = c * yv[kk - 1] * y_norm;
                    if (buff >= w_old[i]) {
                        wv[i] = buff;
                        y_sum += yv[kk - 1] * yv[kk - 1];
                        kk += 1;
                    } else {
                        s += w_old[i] * yv[kk - 1] * y_norm;
                        n_runch -= 1;
#pragma unroll 1
                        for (int j = kk; j <= n_runch; ++j) {
                            posidx[j - 1] = posidx[j];
                            yv[j - 1] = yv[j];
                        }
                    }
                }
                y_sum *= y_norm * y_norm;
                terminated = (n_runch <= 0) || (ctrl == 2) || (i_stop == n_runch);
            }
        }
    }

    // EF:1429-1497.  vA = Ap*nrm_Ap (t), cxs = cx*nrm_cx (l)  ->  wnew
    ENL_NOINL void euclidean_norm_weight_update(V vA, V cxs, double mu, int dimA) {
#pragma unroll 1
        for (int i = 0; i < l; ++i) wnew[i] = w[i];
        if (t != 0) {
            V w_old = K.off(3 * LMAX);
            double ztw = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) ztw += (vA[i] * vA[i]) * w_old[active[i] - 1];
            V yv = s3;
            if (ztw >= mu && dimA < t) {
                int nb_pos = 0;
                double gamma = 0.0;
#pragma unroll 1
                for (int i = 0; i < t; ++i) {
                    int kk = active[i];
                    double ye = vA[i] * (vA[i] + cxs[kk - 1]);
                    if (ye > 0) { posidx[nb_pos] = kk; yv[nb_pos] = ye; nb_pos++; }
                    else gamma -= ye * w_old[kk - 1];
                }
                min_norm_w(2, wnew, w_old, yv, gamma, nb_pos);
            } else if (ztw < mu && dimA < t) {
                int nb_pos = 0;
                double tau = mu;
#pragma unroll 1
                for (int i = 0; i < t; ++i) {
                    int kk = active[i];
                    double ee = -vA[i] * cxs[kk - 1];
                    if (ee > 0) { posidx[nb_pos] = kk; yv[nb_pos] = ee; nb_pos++; }
                    else tau -= ee * w_old[kk - 1];
                }
                min_norm_w(2, wnew, w_old, yv, tau, nb_pos);
            } else if (ztw < mu && dimA == t) {
#pragma unroll 1
                for (int i = 0; i < t; ++i) { posidx[i] = active[i]; yv[i] = vA[i] * vA[i]; }
                min_norm_w(1, wnew, w_old, yv, mu, t);
            }
            assort(wnew);
        }
    }

    // EF:1545-1629 (weight_code == 2).  jp = J p rows (registers). returns dpsi0, fills wnew
    ENL_NOINL double penalty_weight_update(const double* jp, int dimA) {
        const double delta = 0.25;
        if (dimA < 0 || dimA > t) { threw = true; dimA = imax(0, imin(dimA, t)); }
        double sAp = 0.0;
#pragma unroll 1
        for (int i = 0; i < t; ++i) sAp += aAp[i] * aAp[i];
        double nrm_Ap = sqrt(sAp);
        double nrm_cx = 0.0;
#pragma unroll 1
        for (int i = 0; i < dimA; ++i) nrm_cx = fmax(nrm_cx, fabs(cx[active[i] - 1]));
        double nrm_Jp = sqrt(jp_jp);
        double nrm_rx = sqrt(rx_sum);
        // dot(Jp/nrm_Jp, rx/nrm_rx) * nrm_Jp * nrm_rx
        double part = 0.0;
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) {
            double a = (nrm_Jp != 0) ? jp[sl] / nrm_Jp : jp[sl];
            double r = (nrm_rx != 0) ? dR.at(sl, 0) / nrm_rx : dR.at(sl, 0);
            part += a * r;
        }
        double Jp_rx = grp().sum(part) * nrm_Jp * nrm_rx;
        V Apn = s1, cxn = s2;  // normalised copies
#pragma unroll 1
        for (int i = 0; i < t; ++i) Apn[i] = (nrm_Ap != 0) ? aAp[i] / nrm_Ap : aAp[i];
#pragma unroll 1
        for (int i = 0; i < l; ++i) cxn[i] = (nrm_cx != 0) ? cx[i] / nrm_cx : cx[i];
        double AtwA = 0.0, BtwA = 0.0;
#pragma unroll 1
        for (int i = 0; i < dimA; ++i) {
            int kk = active[i] - 1;
            AtwA += w[kk] * (Apn[i] * Apn[i]);
            BtwA += w[kk] * Apn[i] * cxn[kk];
        }
        AtwA *= nrm_Ap * nrm_Ap;
        BtwA *= nrm_Ap * nrm_cx;
        double rmy = (fabs(Jp_rx + nrm_Jp * nrm_Jp) / delta) - nrm_Jp * nrm_Jp;
        // euclidean update on the re-multiplied vectors (EF:1610)
        V vA = s4, cxs = s5;
#pragma unroll 1
        for (int i = 0; i < t; ++i) vA[i] = Apn[i] * nrm_Ap;
#pragma unroll 1
        for (int i = 0; i < l; ++i) cxs[i] = cxn[i] * nrm_cx;
        euclidean_norm_weight_update(vA, cxs, rmy, dimA);
        BtwA = 0.0;
        AtwA = 0.0;
#pragma unroll 1
        for (int i = 0; i < t; ++i) {
            int kk = active[i] - 1;
            AtwA += wnew[kk] * (Apn[i] * Apn[i]);
            BtwA += wnew[kk] * Apn[i] * cxn[kk];
        }
        BtwA *= nrm_Ap * nrm_cx;
        return BtwA + Jp_rx;
    }

    // =====================================================================================
    // linesearch (EF:1635-2143)
    // =====================================================================================
    struct Quartic {   // Polynomials.jl Polynomial with trailing zeros chopped
        double c[5];
        int len;
        ENL_FN double operator()(double xx) const {
            double acc = c[len - 1];
#pragma unroll 1
            for (int i = len - 2; i >= 0; --i) acc = fma(acc, xx, c[i]);
            return acc;
        }
        ENL_FN void chop() {
#pragma unroll 1
            while (len > 1 && c[len - 1] == 0.0) --len;
        }
        ENL_FN Quartic derivative() const {
            Quartic d;
            if (len <= 1) { d.len = 1; d.c[0] = 0.0; return d; }
            d.len = len - 1;
#pragma unroll 1
            for (int i = 1; i < len; ++i) d.c[i - 1] = (double)i * c[i];
            d.chop();
            return d;
        }
    };

    ENL_FN static double minimize_quadratic(double x1, double y1, double x2, double y2, double x3, double y3) {
        double d1 = y2 - y1, d2 = y3 - y1;
        double s = (x3 - x1) * (x3 - x1) * d1 - (x2 - x1) * (x2 - x1) * d2;
        double q = 2 * ((x2 - x1) * d2 - (x3 - x1) * d1);
        return x1 - s / q;
    }

    ENL_NOINL static void minrn(double x1, double y1, double x2, double y2, double x3, double y3, double amin, double amax,
                             double p_max, double& a, double& pa) {
        double eps_ = SQRT_EPS / p_max;
        if (fabs(x1 - x2) < eps_ || fabs(x3 - x1) < eps_ || fabs(x3 - x2) < eps_) { a = 0.0; pa = 0.0; return; }
        double u = minimize_quadratic(x1, y1, x2, y2, x3, y3);
        a = (u > amax) ? amax : ((u < amin) ? amin : u);
        double t1 = (a - x1) * (a - x2) * y3 / ((x3 - x1) * (x3 - x2));
        double t2 = (a - x3) * (a - x2) * y1 / ((x1 - x3) * (x1 - x2));
        double t3 = (a - x3) * (a - x2) * y2 / ((x2 - x1) * (x2 - x3));
        pa = t1 + t2 + t3;
    }

    ENL_NOINL static double newton_raphson(double x_min, double Dm, const Quartic& ds, const Quartic& dds) {
        double alpha = x_min;
        int it = 0;
        double err = 1.0;
#pragma unroll 1
        while ((err > 1e-4 || it < 3) && it < 50) {
            double c = dds(alpha);
            if (fabs(c) < EPS) break;
            double h = -ds(alpha) / c;
            alpha += h;
            err = (2 * Dm * h * h) / fabs(c);
            it += 1;
        }
        return alpha;
    }

    ENL_NOINL void parameters_rm(double dot_v1v2, double normv2, double x_min, const Quartic& ds, const Quartic& dds,
                              double& alpha_hat, double& beta_hat) {
        double dds_best = dds(x_min);
        const double eta = 0.1;
        double d = 1.0;
        double h0 = fabs(ds(x_min) / dds_best);
        double Dm = fabs(6 * dot_v1v2 + 12 * x_min * normv2) + 24 * h0 * normv2;
        double hm = fmax(h0, 1.0);
        bool have_beta = false;
        if (dds_best * eta < 2 * Dm * hm) {
            if (ds.len < 3) { threw = true; alpha_hat = beta_hat = x_min; return; }
            double a3 = ds.c[0] / (2 * normv2), a2 = ds.c[1] / (2 * normv2), a1 = ds.c[2] / (2 * normv2);
            double bb = a2 - (a1 * a1) / 3;
            double cc = a3 - a1 * a2 / 3 + 2 * ((a1 / 3) * (a1 / 3) * (a1 / 3));
            d = (cc / 2) * (cc / 2) + (bb / 3) * (bb / 3) * (bb / 3);
            if (d < 0) {
                // two_roots (EF:1821-1837)
                double arg = fabs(cc / 2) / pow(-bb / 3, 1.5);
                if (!(arg <= 1.0)) { threw = true; alpha_hat = beta_hat = x_min; return; }
                double phi = acos(arg);
                double tt = (cc <= 0) ? 2 * sqrt(-bb / 3) : -2 * sqrt(-bb / 3);
                const double PI = 3.141592653589793;
                double b1 = tt * cos(phi / 3) - a1 / 3;
                double b2 = tt * cos((phi + 2 * PI) / 3) - a1 / 3;
                double b3 = tt * cos((phi + 4 * PI) / 3) - a1 / 3;
                double tmp;
                if (b1 > b2) { tmp = b1; b1 = b2; b2 = tmp; }
                if (b2 > b3) { tmp = b2; b2 = b3; b3 = tmp; }
                if (b1 > b2) { tmp = b1; b1 = b2; b2 = tmp; }
                if (x_min <= b2) { alpha_hat = b1; beta_hat = b3; } else { alpha_hat = b3; beta_hat = b1; }
                have_beta = true;
            } else {
                if (d != d) { threw = true; alpha_hat = beta_hat = x_min; return; }
                double sd = sqrt(d);
                alpha_hat = cbrt(-cc / 2 + sd) + cbrt(-cc / 2 - sd) - a1 / 3;
            }
        } else {
            alpha_hat = newton_raphson(x_min, Dm, ds, dds);
        }
        if (d >= 0) { beta_hat = alpha_hat; have_beta = true; }
        if (!have_beta) threw = true;
    }

    // the six dot products of v0, v1, v2 (EF:1665-1689, 1849) from r, r(alpha), cx, c(alpha)
    ENL_NOINL void minrm(const double* jp, const double* rn, double alpha_k, double x_min, double amin, double amax,
                      double& a_hat, double& s_a, double& b_hat, double& s_b) {
        double d00 = 0, d01 = 0, d02 = 0, d11 = 0, d12 = 0, d22 = 0;
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) {
            double v0 = dR.at(sl, 0), v1 = jp[sl];
            double v2 = ((rn[sl] - v0) / alpha_k - v1) / alpha_k;
            d00 += v0 * v0; d01 += v0 * v1; d02 += v0 * v2; d11 += v1 * v1; d12 += v1 * v2; d22 += v2 * v2;
        }
        d00 = grp().sum(d00); d01 = grp().sum(d01); d02 = grp().sum(d02); d11 = grp().sum(d11); d12 = grp().sum(d12); d22 = grp().sum(d22);
#pragma unroll 1
        for (int i = 0; i < l; ++i) s1[i] = 0.0;   // membership: 1 active, 0 inactive
#pragma unroll 1
        for (int i = 0; i < t; ++i) s1[active[i] - 1] = 1.0;
#pragma unroll 1
        for (int kk = 0; kk < l; ++kk) {
            const bool act = s1[kk] != 0.0;
            // inactive and satisfied at both points: v0 = v1 = v(alpha) = 0 exactly, the row adds nothing
            if (!act && cx[kk] > 0 && cnew[kk] > 0) continue;
            double sw = sqrt(wnew[kk]);
            double v0, vb;
            if (act) { v0 = sw * cx[kk]; vb = sw * cnew[kk]; }
            else { v0 = (cx[kk] > 0) ? 0.0 : sw * cx[kk]; vb = (cnew[kk] > 0) ? 0.0 : sw * cnew[kk]; }
            double v1 = v1c[kk];
            double v2 = (div_z(vb - v0, alpha_k) - v1) / alpha_k;
            d00 += v0 * v0; d01 += v0 * v1; d02 += v0 * v2; d11 += v1 * v1; d12 += v1 * v2; d22 += v2 * v2;
        }
        Quartic s;
        s.len = 5;
        s.c[0] = 0.5 * d00; s.c[1] = d01; s.c[2] = d02 + 0.5 * d11; s.c[3] = d12; s.c[4] = 0.5 * d22;
        s.chop();
        Quartic ds = s.derivative();
        Quartic dds = ds.derivative();
        parameters_rm(d12, d22, x_min, ds, dds, a_hat, b_hat);
        double a_old = a_hat;
        // bounds (EF:1785-1789); Julia min/max propagate NaN
        auto bounds = [&](double a) { if (a != a) return a; a = fmin(a, amax); a = fmax(a, amin); return a; };
        a_hat = bounds(a_hat);
        s_a = s(a_hat);
        if (a_old == b_hat) { b_hat = a_hat; s_b = s(a_hat); }
        else { b_hat = bounds(b_hat); s_b = s(b_hat); }
    }

    ENL_FN static bool check_reduction(double psi_alpha, double psi_k, double approx_k, double eta, double diff_psi) {
        if (psi_alpha - approx_k >= eta * diff_psi) return !((psi_alpha - psi_k < eta * diff_psi) && (psi_k > 0.2 * psi_alpha));
        return false;
    }

    ENL_NOINL double linesearch(const double* jp, double alpha0, double psi0, double dpsi0, double alpha_low, double alpha_upp,
                             bool& gac_error) {
        const double eta = 0.3, tau = 0.25, gamma = 0.4;
        double rn[MS];
        double amin = alpha_low, amax = alpha_upp;
        double alpha_k = fmin(alpha0, amax);
        double alpha_km1 = 0.0, psi_km1 = psi0;
        double p_max = 0.0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) p_max = fmax(p_max, fabs(p[j]));
        gac_error = false;
        // v1 constraint part (EF:1986-1998)
#pragma unroll 1
        for (int i = 0; i < l; ++i) s1[i] = 0.0;
#pragma unroll 1
        for (int i = 0; i < t; ++i) s1[active[i] - 1] = 1.0;
#pragma unroll 1
        for (int kk = 0; kk < l; ++kk) {
            if (s1[kk] == 0.0 && cx[kk] > 0) { v1c[kk] = 0.0; continue; }
            v1c[kk] = sqrt(wnew[kk]) * Ap[kk];
        }
        double psi_k = psi(alpha_k, wnew, rn);
        double diff_psi = psi0 - psi_k;
        n_res += 1; n_cons += 1;   // EF:2005-2006 duplicate evaluation (deduplicated here)
        double x_min = (diff_psi >= 0) ? alpha_k : 0.0;
        double alpha_kp1, pk, beta, pbeta;
        minrm(jp, rn, alpha_k, x_min, amin, amax, alpha_kp1, pk, beta, pbeta);
        if (threw) return alpha_k;
        if (alpha_kp1 != beta && pbeta < pk && beta <= alpha_k) { alpha_kp1 = beta; pk = pbeta; }
        double alpha_km2 = alpha_km1, psi_km2 = psi_km1;
        alpha_km1 = alpha_k; psi_km1 = psi_k;
        alpha_k = alpha_kp1;
        psi_k = psi(alpha_k, wnew, rn);
        int guard = 0;
        if ((-diff_psi <= tau * dpsi0 * alpha_km1) || (psi_km1 < gamma * psi0)) {
            diff_psi = psi0 - psi_k;
            bool likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
#pragma unroll 1
            while (likely) {
                minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, amin, amax, p_max, alpha_kp1, pk);
                alpha_km2 = alpha_km1; psi_km2 = psi_km1;
                alpha_km1 = alpha_k; psi_km1 = psi_k;
                alpha_k = alpha_kp1;
                psi_k = psi(alpha_k, wnew, rn);
                diff_psi = psi0 - psi_k;
                likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
                if (++guard > 10000) { hang = true; break; }
            }
            if ((psi_km1 - pk >= eta * diff_psi) && (psi_k < psi_km1)) { alpha_km1 = alpha_k; psi_km1 = psi_k; }
        } else {
            diff_psi = psi0 - psi_k;
            if ((-diff_psi <= tau * dpsi0 * alpha_k) || (psi_k < gamma * psi0)) {
                if (psi0 <= psi_km1) {
                    x_min = alpha_k;
                    n_res += 1; n_cons += 1;   // EF:2081-2082 (same point as the last psi)
                    minrm(jp, rn, alpha_k, x_min, amin, amax, alpha_kp1, pk, beta, pbeta);
                    if (threw) return alpha_k;
                    if (alpha_kp1 != beta && pbeta < pk && beta <= alpha_k) { alpha_kp1 = beta; pk = pbeta; }
                    alpha_km1 = 0.0;
                    psi_km1 = psi0;
                } else {
                    minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, amin, amax, p_max, alpha_kp1, pk);
                }
                alpha_km2 = alpha_km1; psi_km2 = psi_km1;
                alpha_km1 = alpha_k; psi_km1 = psi_k;
                alpha_k = alpha_kp1;
                psi_k = psi(alpha_k, wnew, rn);
                bool likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
#pragma unroll 1
                while (likely) {
                    minrn(alpha_k, psi_k, alpha_km1, psi_km1, alpha_km2, psi_km2, amin, amax, p_max, alpha_kp1, pk);
                    alpha_km2 = alpha_km1; psi_km2 = psi_km1;
                    alpha_km1 = alpha_k; psi_km1 = psi_k;
                    alpha_k = alpha_kp1;
                    psi_k = psi(alpha_k, wnew, rn);
                    likely = check_reduction(psi_km1, psi_k, pk, eta, diff_psi);
                    if (++guard > 10000) { hang = true; break; }
                }
                if ((psi_km1 - pk >= eta * diff_psi) && (psi_k < psi_km1)) { alpha_km1 = alpha_k; psi_km1 = psi_k; }
            } else {
                // goldstein_armijo_step (EF:1893-1923)
                double u = alpha_k;
                bool ex = (p_max * u < SQRT_EPS) || (u <= amin);
                double psi_u = psi(u, wnew, rn);
#pragma unroll 1
                while (!ex && (psi_u > psi0 + tau * u * dpsi0)) {
                    u *= 0.5;
                    psi_u = psi(u, wnew, rn);
                    ex = (p_max * u < SQRT_EPS) || (u <= amin);
                }
                alpha_km1 = u;
                gac_error = ex;
            }
        }
        return alpha_km1;
    }

    // EF:2149-2178
    ENL_FN double upper_bound_steplength(int index_del, int& index_alpha_upp) {
        double alpha_upper = INFINITY;
        index_alpha_upp = 0;
#pragma unroll 1
        for (int i = 0; i < l - t; ++i) {
            int j = inactive[i];
            if (j != index_del) {
                double gp = Ap[j - 1];
                double a_j = -cx[j - 1] / gp;
                if (cx[j - 1] > 0 && gp < 0 && a_j < alpha_upper) { alpha_upper = a_j; index_alpha_upp = j; }
            }
        }
        return fmin(3.0, alpha_upper);
    }

    // EF:2197-2293.  On return r(x+alpha p), c(x+alpha p) are in rfin / cnew when `have_final`.
    ENL_NOINL double compute_steplength(int& Psi_error, double* rfin, bool& have_final) {
        double jp[MS];
        if (j2_factored) {
            // J p = (J Q1) y = J1 y1 + J2 y2,  J2 = Q3 [R22 P3'; 0]  =>  J2 y2 = Q3 [R22 (P3' y2); 0]
            const int rankA = cur.rankA, k2 = N - cur.rankA, kq = imin(M, N - cur.rankA);
#pragma unroll 1
            for (int i = 0; i < kq; ++i) {
                double acc = 0.0;
#pragma unroll 1
                for (int j = i; j < k2; ++j) acc += R2[j * N + i] * y[rankA + perm2[j]];
                s1[i] = acc;
            }
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                int row = sl * G + grp().lane;
                jp[sl] = (row < kq) ? s1[row < kq ? row : 0] : 0.0;
            }
            dst().apply_q_regs(dF, kq, tau2, jp);
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                double acc = 0.0;
#pragma unroll 1
                for (int c = 0; c < rankA; ++c) acc += dJ.at(sl, c) * y[c];
                jp[sl] += acc;
            }
        } else {
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) {
                double acc = 0.0;
#pragma unroll 1
                for (int c = 0; c < N; ++c) acc += dJ.at(sl, c) * y[c];   // J p = (J Q1)(Q1' p)
                jp[sl] = acc;
            }
        }
        {
            double a = 0.0, bq = 0.0;
#pragma unroll
            for (int sl = 0; sl < MS; ++sl) { a += jp[sl] * dR.at(sl, 0); bq += jp[sl] * jp[sl]; }
            jp_r = grp().sum(a);
            jp_jp = grp().sum(bq);
        }
#pragma unroll 1
        for (int i = 0; i < NNL; ++i) {
            double acc = 0.0;
#pragma unroll 1
            for (int c = 0; c < N; ++c) acc += A[i * N + c] * p[c];
            Ap[i] = acc;
        }
        // rows of the bounds are +e_j / -e_j (cnls_model.jl:393-403): the dot product is +-p_j
#pragma unroll 1
        for (int j = 0; j < bnd.nlo; ++j) Ap[NNL + j] = p[bnd.lo_idx[j]];
#pragma unroll 1
        for (int j = 0; j < bnd.nup; ++j) Ap[NNL + bnd.nlo + j] = -p[bnd.up_idx[j]];
#pragma unroll 1
        for (int i = 0; i < t; ++i) {
            double acc = 0.0;
#pragma unroll 1
            for (int c = 0; c < N; ++c) acc += aA[i * N + c] * p[c];
            aAp[i] = opt.scaling ? acc / dsc[i] : acc;
        }
        Psi_error = 0;
        have_final = false;
        double alpha;
        if (cur.code != 2) {
            double dpsi0 = penalty_weight_update(jp, cur.dimA);
            double pen = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) { int kk = active[i] - 1; pen += wnew[kk] * (cx[kk] * cx[kk]); }
            double psi0 = 0.5 * (rx_sum + pen);
            if (dpsi0 >= 0) {
                alpha = 1.0;
                Psi_error = -1;
                cur.index_alpha_upp = 0;
            } else {
                int idx_upp;
                double alpha_upp = upper_bound_steplength(cur.index_del, idx_upp);
                double alpha_low = alpha_upp / 3000.0;
                double magfy = (cur.rankJ2 < prev.rankJ2) ? 6.0 : 3.0;
                double alpha0 = fmin(fmin(1.0, magfy * prev.alpha), alpha_upp);
                bool gac_error;
                alpha = linesearch(jp, alpha0, psi0, dpsi0, alpha_low, alpha_upp, gac_error);
                if (threw || hang) return alpha;
                if (gac_error) {
                    double psi_k = psi(alpha, wnew, rfin);
                    double psi_ma = psi(-alpha, wnew, rfin);
                    double f = (psi_k - psi0) / alpha, bk = (psi0 - psi_ma) / alpha, c = (psi_k - psi_ma) / (2 * alpha);
                    double md = fmax(fmax(fabs(f - c), fabs(f - bk)), fabs(bk - c));
                    bool inc = fabs(f - dpsi0) > md && fabs(c - dpsi0) > md;
                    Psi_error = inc ? -1 : 0;
                }
                double upp = fmin(1.0, alpha_upp);
                double atwa = 0.0;
#pragma unroll 1
                for (int i = 0; i < t; ++i) atwa += wnew[active[i] - 1] * (aAp[i] * aAp[i]);
                cur.predicted_reduction = upp * (-2.0 * jp_r - upp * jp_jp + (2.0 - upp * upp) * atwa);
                // progress: r, c at x + alpha p (EF:2274-2280); the same point as new_point! (EF:2825-2828)
                double xv[N];
#pragma unroll
                for (int j = 0; j < N; ++j) xv[j] = add_rn(x[j], mul_rn(alpha, p[j]));
                eval_point(xv, rfin, cnew);
                n_res += 1; n_cons += 1;
                have_final = true;
                double whsum = 0.0;
#pragma unroll 1
                for (int i = 0; i < t; ++i) { int kk = active[i] - 1; whsum += wnew[kk] * (cnew[kk] * cnew[kk]); }
                cur.progress = 2 * psi0 - sumsq_regs(rfin) - whsum;
                cur.index_alpha_upp = (idx_upp != 0 && fabs(alpha - alpha_upp) > 0.1) ? 0 : idx_upp;
            }
        } else {
#pragma unroll 1
            for (int i = 0; i < l; ++i) wnew[i] = w[i];
            cur.index_alpha_upp = 0;
            alpha = 1.0;
        }
        return alpha;
    }

    // =====================================================================================
    // termination (EF:2399-2517); x is still x_k, xnew = x_{k+1}; cx/gradf/rx_sum at x_{k+1}
    // =====================================================================================
    ENL_NOINL int check_termination(int error_code, bool time_up, double sigma_min, double lam_abs_max, int Psi_error) {
        int ec = 0;
        double pn = 0.0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) pn += p[j] * p[j];
        double alfnoi = EPS / (sqrt(pn) + EPS);
        bool preliminary = !(cur.restart || (cur.code == -1 && alfnoi <= 0.25));
        double xd = 0.0, xn2 = 0.0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) { double dd = xprev[j] - xnew[j]; xd += dd * dd; xn2 += xnew[j] * xnew[j]; }
        double x_diff = sqrt(xd);
        if (preliminary) {
            double ca = 0.0, gn = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) ca += acx[i] * acx[i];
#pragma unroll 1
            for (int j = 0; j < N; ++j) gn += gradf[j] * gradf[j];
            bool necessary = (!cur.del) && (sqrt(ca) < opt.eps_c) && (cur.grad_res < sqrt(opt.eps_rel) * (1 + sqrt(gn)));
            if (l - t > 0) {
                bool allpos = true;
#pragma unroll 1
                for (int i = 0; i < l - t; ++i)
                    if (!(cx[inactive[i] - 1] > 0)) allpos = false;
                necessary = necessary && allpos;
            }
            if (t > Q) {
                double factor = (t == 1) ? (1 + rx_sum) : lam_abs_max;
                necessary = necessary && (sigma_min >= opt.eps_rel * factor);
            }
            if (necessary) {
                int dj = cur.dimJ2;
                if (dj > M) { threw = true; dj = M; }
                double d1 = dst().prefix_sq(dD, dj);
                if (d1 <= rx_sum * opt.eps_rel * opt.eps_rel) ec += 10000;
                if (rx_sum <= opt.eps_abs * opt.eps_abs) ec += 2000;
                if (x_diff < opt.eps_x * sqrt(xn2)) ec += 300;
                if (alfnoi > 0.25) ec += 40;
                if (ec > 0 && l - t > 0) {
                    int feas = 1;
#pragma unroll 1
                    for (int i = 0; i < l - t; ++i)
                        if (cx[inactive[i] - 1] <= 0.0) { feas = -1; break; }
                    ec *= feas;
                }
            }
        }
        if (ec == 0) {
            double an = 0.0;
#pragma unroll 1
            for (int c = 0; c < N; ++c) {
                double acc = 0.0;
#pragma unroll 1
                for (int i = 0; i < t; ++i) acc += aA[i * N + c] * acx[i];
                an += acc * acc;
            }
            double Atcx_nrm = sqrt(an);
            double aps = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) { double wi = wnew[active[i] - 1]; aps += wi * wi; }
            if (k_iter >= opt.max_iter) ec = -2;
            else if (error_code >= -5 && error_code <= -3) ec = error_code;
            else if (cur.nb_newton > 5) ec = -9;
            else if (Psi_error == -1) ec = -6;
            else if (x_diff <= 10.0 * opt.eps_x && Atcx_nrm <= 10.0 * opt.eps_c && aps >= 1.0) ec = -10;
            else if (time_up) ec = -11;
        }
        return ec;
    }

    // =====================================================================================
    // driver (EF:2638-2880)
    // =====================================================================================
    // start a solve: x0 -> state at iteration 0
    ENL_NOINL void init(const double* x0, const FamilyData& fd, long long bidx, double now) {
        Fam::template load<Grp, MS>(fctx(), fd, bidx, grp());
#pragma unroll 1
        for (int j = 0; j < N; ++j) { double v = x0[j]; x[j] = v; xprev[j] = v; }
        l = NNL + bnd.nlo + bnd.nup;
        k_iter = 0; ndetail = 0; exit_code = 0; threw = false; hang = false;
        n_res = n_cons = n_jres = n_jcons = 0;
        t_start = now;
        double xv[N], rn[MS];
        load_x(x, xv);
        eval_point(xv, rn, cx);
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) dR.at(sl, 0) = rn[sl];
        grp().sync();
        init_bound_rows();
        eval_res_jacobian();
        eval_cons_jacobian();
        n_res += 1; n_cons += 1; n_jres += 1; n_jcons += 1;
        grad_and_sumsq();
        f_detail = rx_sum;
        // init_working_set (EF:826-859)
#pragma unroll 1
        for (int i = 0; i < 4 * LMAX; ++i) K[i] = 0.1;
#pragma unroll 1
        for (int i = 0; i < l; ++i) w[i] = fmin(fabs(cx[i]) + 0.01, 0.1);
        t = Q;
        int lmt = 0;
#pragma unroll 1
        for (int i = 0; i < LMAX; ++i) { active[i] = 0; inactive[i] = 0; }
#pragma unroll 1
        for (int i = 1; i <= Q; ++i) active[i - 1] = i;
#pragma unroll 1
        for (int i = Q + 1; i <= l; ++i) {
            if (cx[i - 1] <= 0.0) {
                active[t] = i;          // t < l <= LMAX: the whole initial working set is kept, also beyond T
                t += 1;
            } else {
                inactive[lmt++] = i;
            }
        }
        cur = IterRec{};
        cur.alpha = 1.0;
        cur.code = 1;
        // more active rows than the shared-memory factorisations hold: x = x0, f = ||r(x0)||^2, no iteration, and
        // nact / active report the whole initial working set (store)
        if (t > T) { exit_code = EXIT_CAPACITY; return; }
        cur.t = t;
        gather_active();
        prev = cur;
        rdot_x1 = cdot_x1 = 0.0;
    }

    // new_point! (EF:34-52) as an operator of its own: r, J (forward differences of cnls_model.jl:65-82 or analytic),
    // c and A at xin -- the evaluation layer without the iteration around it (enlsipb200_eval_batch)
    ENL_NOINL void eval_only(const double* xin, const FamilyData& fd, long long bidx) {
        Fam::template load<Grp, MS>(fctx(), fd, bidx, grp());
#pragma unroll 1
        for (int j = 0; j < N; ++j) x[j] = xin[j];
        l = NNL + bnd.nlo + bnd.nup;
        double xv[N], rn[MS];
        load_x(x, xv);
        eval_point(xv, rn, cx);
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) dR.at(sl, 0) = rn[sl];
        grp().sync();
        init_bound_rows();
        eval_res_jacobian();
        eval_cons_jacobian();
    }
    // r [M], J [N][M] (column major m x n, the reference's layout), c [LMAX], A [LMAX][N] (row i = gradient of c_i)
    ENL_NOINL void store_eval(double* r_out, double* J_out, double* c_out, double* A_out, long long bidx) {
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) {
            const int row = sl * G + grp().lane;
            if (row < M) {
                if (r_out) r_out[bidx * M + row] = dR.at(sl, 0);
                if (J_out)
#pragma unroll
                    for (int j = 0; j < N; ++j) J_out[(bidx * N + j) * M + row] = dJ.at(sl, j);
            }
        }
        if (grp().lane != 0) return;
        if (c_out)
#pragma unroll 1
            for (int i = 0; i < LMAX; ++i) c_out[bidx * LMAX + i] = (i < l) ? cx[i] : 0.0;
        if (A_out)
#pragma unroll 1
            for (int i = 0; i < LMAX * N; ++i) A_out[bidx * LMAX * N + i] = (i < l * N) ? A[i] : 0.0;
    }

    // One Gauss-Newton step from MATERIALISED inputs (SURVEY.md 8d, the batched step kernel): r [M], J [N][M] column
    // major, c [LMAX], A [LMAX][N] of one problem are read from global memory; the working set is the initial one of
    // init_working_set (EF:826-859); update_working_set (EF:686-795) gives the multipliers, the (possibly reduced)
    // working set and the Gauss-Newton direction -- no function evaluation anywhere.
    ENL_NOINL void step_only(const double* xin, const double* r_in, const double* J_in, const double* c_in,
                             const double* A_in) {
#pragma unroll 1
        for (int j = 0; j < N; ++j) { double v = xin[j]; x[j] = v; xprev[j] = v; }
        l = NNL + bnd.nlo + bnd.nup;
        k_iter = 0; ndetail = 0; exit_code = 0; threw = false; hang = false;
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) {
            const int row = sl * G + grp().lane;
            dR.at(sl, 0) = (row < M) ? r_in[row] : 0.0;
        }
#pragma unroll 1
        for (int i = 0; i < l; ++i) cx[i] = c_in[i];
#pragma unroll 1
        for (int i = 0; i < l * N; ++i) A[i] = A_in[i];
        mat_J = J_in;
        grp().sync();
        eval_res_jacobian();
        grad_and_sumsq();
        t = Q;
        int lmt = 0;
#pragma unroll 1
        for (int i = 0; i < LMAX; ++i) { active[i] = 0; inactive[i] = 0; }
#pragma unroll 1
        for (int i = 1; i <= Q; ++i) active[i - 1] = i;
#pragma unroll 1
        for (int i = Q + 1; i <= l; ++i) {
            if (cx[i - 1] <= 0.0) {
                active[t] = i;          // t < l <= LMAX: the whole initial working set is kept, also beyond T
                t += 1;
            } else {
                inactive[lmt++] = i;
            }
        }
        cur = IterRec{};
        cur.alpha = 1.0;
        cur.code = 1;
        if (t > T) { exit_code = EXIT_CAPACITY; return; }
        cur.t = t;
        gather_active();
        evaluate_scaling();
        update_working_set();
        if (threw) exit_code = EXIT_WOULD_THROW;
    }
    // p [N], lam [T] (in working-set order, 0 padded), active [LMAX], info = {t, rankA, rankJ2, index_del, code}.  A
    // problem that ends with an error code gets p = 0 and lam = 0: -97 returns before any direction is computed, so
    // the slot's p / lam still hold whatever problem it served before.
    ENL_NOINL void store_step(double* p_out, double* lam_out, int* active_out, int* info_out, long long bidx) {
        if (grp().lane != 0) return;
        const bool ok = exit_code == 0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) p_out[bidx * N + j] = ok ? p[j] : 0.0;
        if (lam_out)
#pragma unroll 1
            for (int i = 0; i < T; ++i) lam_out[bidx * T + i] = (ok && i < t) ? lam[i] : 0.0;
        if (active_out)
#pragma unroll 1
            for (int i = 0; i < LMAX; ++i) active_out[bidx * LMAX + i] = (i < t) ? active[i] : 0;
        if (info_out) {
            info_out[bidx * 5 + 0] = t; info_out[bidx * 5 + 1] = cur.rankA; info_out[bidx * 5 + 2] = cur.rankJ2;
            info_out[bidx * 5 + 3] = cur.index_del; info_out[bidx * 5 + 4] = exit_code;
        }
    }

    // one ENLSIP iteration; sets exit_code != 0 when the solve is over
    ENL_NOINL void step(double now, double* trace_row) {
        evaluate_scaling();
        update_working_set();
        active_cx_sum = 0.0;
#pragma unroll 1
        for (int i = 0; i < t; ++i) { double v = cx[active[i] - 1]; active_cx_sum += v * v; }
        cur.t = t;
        double cdot_now = 0.0;
#pragma unroll 1
        for (int i = 0; i < l; ++i) cdot_now += cx[i] * cx[i];
        if (k_iter == 0) {
            prev = cur;   // EF:2703
            rdot_prev = rx_sum; cdot_prev = cdot_now;
        } else if (k_iter == 2) {
            rdot_prev = rdot_x1; cdot_prev = cdot_x1;        // aliasing schedule, SURVEY.md T1
        } else {
            rdot_prev = rx_sum; cdot_prev = cdot_now;
        }
        if (k_iter == 1) { rdot_x1 = rx_sum; cdot_x1 = cdot_now; }
        int error_code = 0, Psi_error = 0;
        double alpha = 1.0;
        double rfin[MS];
        bool have_final = false;
        if (!threw) error_code = search_direction_analys();
        if (!threw) alpha = compute_steplength(Psi_error, rfin, have_final);
        if (threw || hang) { finish_abnormal(); return; }
        cur.alpha = alpha;
        double pn = 0.0;
#pragma unroll 1
        for (int j = 0; j < N; ++j) pn += p[j] * p[j];
        // x_{k+1}
        double xv[N];
#pragma unroll
        for (int j = 0; j < N; ++j) { xv[j] = add_rn(x[j], mul_rn(alpha, p[j])); xnew[j] = xv[j]; }
        // new_point! (EF:2733, 2828)
        if (!have_final) eval_point(xv, rfin, cnew);
        n_res += 1; n_cons += 1; n_jres += 1; n_jcons += 1;
        // termination needs active c / A at x_k (acx, aA) and everything else at x_{k+1}
#pragma unroll 1
        for (int i = 0; i < l; ++i) cx[i] = cnew[i];
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) dR.at(sl, 0) = rfin[sl];
        grp().sync();
#pragma unroll 1
        for (int j = 0; j < N; ++j) { s5[j] = x[j]; x[j] = xnew[j]; }   // s5 = x_k
        eval_res_jacobian();
        eval_cons_jacobian();
        grad_and_sumsq();
        cur.restart = (error_code < 0);
        double sigma_min, lam_abs_max;
        minmax_lagrangian_mult(sigma_min, lam_abs_max);
        bool time_up = (now - t_start) - opt.time_limit > 0;
        int ec = check_termination(error_code, time_up, sigma_min, lam_abs_max, Psi_error);
        if (threw) { finish_abnormal(); return; }
        if (trace_row) {
            trace_row[0] = rx_sum; trace_row[1] = t; trace_row[2] = cur.rankA; trace_row[3] = cur.rankJ2;
            trace_row[4] = cur.dimA; trace_row[5] = cur.dimJ2; trace_row[6] = cur.code; trace_row[7] = alpha;
            trace_row[8] = sqrt(pn); trace_row[9] = cur.index_del; trace_row[10] = ec; trace_row[11] = active_cx_sum;
            trace_row[12] = cur.progress; trace_row[13] = k_iter;
            double mask = 0.0;
#pragma unroll 1
            for (int i = 0; i < t; ++i) mask += ldexp(1.0, active[i] - 1);
            trace_row[14] = mask; trace_row[15] = cur.grad_res;
#pragma unroll 1
            for (int j = 0; j < N; ++j) trace_row[TRACE_HDR + j] = xnew[j];
        }
        if (ec == 0) {
            ndetail += 1;
            cur.add = evaluate_violated_constraints(cur.index_alpha_upp);
            if (hang) { finish_abnormal(); return; }
            gather_active();
            k_iter += 1;
#pragma unroll 1
            for (int i = 0; i < l; ++i) w[i] = wnew[i];   // iter.w = w ; prev = copy(iter)
            prev = cur;
            // previous_iter.x: snapshot taken before iter.x is rebound (EF:2860-2861)
            if (k_iter >= 2) for (int j = 0; j < N; ++j) xprev[j] = s5[j];
            cur.del = false;
            cur.add = false;
        } else {
            exit_code = ec;
            if (k_iter == 0) {
                // T5: the loop body never ran: x_opt = x0, ExecutionInfo() default
#pragma unroll 1
                for (int j = 0; j < N; ++j) x[j] = s5[j];
                ndetail = 1;
                n_res = n_cons = n_jres = n_jcons = 0;
            }
        }
    }

    ENL_FN void finish_abnormal() {
        exit_code = hang ? EXIT_WOULD_HANG : EXIT_WOULD_THROW;
        double rr[MS];
#pragma unroll
        for (int sl = 0; sl < MS; ++sl) rr[sl] = dR.at(sl, 0);
        rx_sum = sumsq_regs(rr);
        n_res = n_cons = n_jres = n_jcons = 0;
    }

    ENL_FN static int convert_exit_code(int code) {   // cnls_model.jl:166-178
        if (code > 0) return 1;
        if (code == -2 || code == -11) return code;
        return -1;
    }

    // lane 0 of the group writes the results of problem `bidx`
    ENL_NOINL void store(const Outputs& o, long long bidx) {
        if (grp().lane != 0) return;
#pragma unroll 1
        for (int j = 0; j < N; ++j) o.x[bidx * N + j] = x[j];
        o.f[bidx] = rx_sum;
        o.exit_code[bidx] = exit_code;
        o.status[bidx] = convert_exit_code(exit_code);
        o.iters[bidx] = ndetail;
        o.nact[bidx] = t;
        if (o.active)
#pragma unroll 1
            for (int i = 0; i < LMAX; ++i) o.active[bidx * LMAX + i] = (i < t) ? active[i] : 0;
        if (o.counters) {
            o.counters[bidx * 2 + 0] = n_res + n_cons;
            o.counters[bidx * 2 + 1] = n_jres + n_jcons;
        }
    }
};

}  // namespace enl
