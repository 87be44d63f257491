// enlsip_b200.cu -- kernels and C ABI (include/enlsip_b200.h) of the batched ENLSIP engine.
//
// One persistent kernel per solve call: every group of G lanes repeatedly takes the next problem
// from a global work counter, runs the complete ENLSIP solve (enl_solver.h) with the problem's
// state in shared memory / registers, and writes x, f, exit code, iteration count and the final
// working set.  HBM traffic is the problem data in and the solution out -- nothing else.
//
// sm_100a only.  No CPU fallback: without a CUDA device every entry point returns ENLSIPB200_ENOGPU.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <new>
#include <type_traits>
#include <string>
#include <vector>

#include <dlfcn.h>
#include <unistd.h>

#include "../../include/enlsip_b200.h"
#include "enl_solver.h"
// Run-time compiled family (enlsipb200_compile_family below): the generated prelude + the user's source are
// force-included in front of this file (-include), then the family wrapper binds them to the solver.
#if defined(ENL_USER_FAMILY)
#include "enl_user_family.h"
#endif

using namespace enl;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? ENLSIPB200_ENOGPU \
                                                                                     : ENLSIPB200_ECUDA, \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                             \
    } while (0)

struct KernelArgs {
    long long B;
    unsigned long long* counter;
    const double* x0;
    FamilyData fd;
    Options opt;
    Bounds bnd;
    Outputs out;
};

__device__ __forceinline__ double now_seconds() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return (double)t * 1e-9;
}

template <class Fam, int G, int NT>
__global__ void __launch_bounds__(NT) enlsip_solve_batch_kernel(const __grid_constant__ KernelArgs a) {
    using LY = Layout<Fam, G, NT>;
    constexpr bool SYNC_ITER = (NT > 32);
    using SolverT = Solver<Fam, DevGroup<G>, NT>;
    constexpr int SOLVER_DOUBLES = (int)((sizeof(SolverT) + 7) / 8) | 1;   // odd stride: no bank conflicts for G == 1
    const int tid = threadIdx.x;
    const int pid = tid / G;
    // CTA-shared copy of the options and bounds: reading kernel parameters through the generic pointers held
    // by the solver object costs a long-scoreboard stall per access (ncu: eval_point 50 % long_sb)
    constexpr int CFG_DOUBLES = (int)((sizeof(Options) + sizeof(Bounds) + 15) / 16) * 2;
    Options* s_opt = reinterpret_cast<Options*>(enl_smem);
    Bounds* s_bnd = reinterpret_cast<Bounds*>(reinterpret_cast<char*>(enl_smem) + sizeof(Options));
    if (tid == 0) { *s_opt = a.opt; *s_bnd = a.bnd; }
    __syncthreads();
    double* objs = enl_smem + CFG_DOUBLES;
    double* small = objs + (size_t)SOLVER_DOUBLES * LY::PPC;
    double* distb = small + (size_t)LY::nD * LY::PPC;
    int* ints = reinterpret_cast<int*>(distb + (size_t)LY::DCOLS * LY::MS * NT);
    DevGroup<G> g;
    // the per-problem solver object lives in shared memory; every lane of the group writes identical values
    SolverT& S = *new (objs + (size_t)SOLVER_DOUBLES * pid) SolverT(small, ints, distb, pid, *s_opt, *s_bnd);
    g.sync();
    const int row_w = TRACE_HDR + Fam::N;
    bool have = false, exhausted = false;
    long long b = 0;
    int row = 0;
    for (;;) {
        if (!have && !exhausted) {
            unsigned long long nb = 0;
            if (g.lane == 0) nb = atomicAdd(a.counter, 1ULL);
            if (G > 1) nb = __shfl_sync(g.mask, nb, 0, G);
            b = (long long)nb;
            if (b >= a.B) {
                exhausted = true;
            } else {
                S.init(a.x0 + b * Fam::N, a.fd, b, now_seconds());
                have = true;
                row = 0;
            }
        }
        // Multi-warp CTAs re-align their warps once per iteration: co-resident warps then run the same
        // routines at the same time and share instruction-cache lines (the kernel is fetch-bound).
        if (SYNC_ITER) {
            // (measured alternatives, all slower: re-aligning in 2 / 7 independent groups 1.26 / 0.60 M solves/s,
            //  every 2nd / 3rd pass 1.65 / 1.35 M, 1-3 extra barriers inside Solver::step 1.93-1.94 M, vs 1.96 M)
            if (!__syncthreads_or(have ? 1 : 0)) break;
        } else if (!have) {
            break;
        }
        if (have) {
            if (S.exit_code == 0) {
                double* tr = nullptr;
                if (a.out.trace && row < a.out.trace_cap && g.lane == 0)
                    tr = a.out.trace + ((size_t)b * a.out.trace_cap + row) * row_w;
                S.step(now_seconds(), tr);
                ++row;
            }
            if (S.exit_code != 0) {
                S.store(a.out, b);
                have = false;
            }
        }
    }
}

// The evaluation layer alone (new_point!, EF:34-52; jac_forward_diff, cnls_model.jl:65-82): every group takes problems
// from the work counter, evaluates r, J, c, A at the given point and writes them to HBM.
struct EvalArgs {
    long long B;
    unsigned long long* counter;
    const double* x;
    FamilyData fd;
    Options opt;
    Bounds bnd;
    double *r, *J, *c, *A;
    // step mode (enlsipb200_step_batch): r, J, c, A are INPUTS; outputs:
    int step;
    double *p, *lam;
    int *active, *info;
};
template <class Fam, int G, int NT>
__global__ void __launch_bounds__(NT) enlsip_eval_batch_kernel(const __grid_constant__ EvalArgs a) {
    using LY = Layout<Fam, G, NT>;
    using SolverT = Solver<Fam, DevGroup<G>, NT>;
    constexpr int SOLVER_DOUBLES = (int)((sizeof(SolverT) + 7) / 8) | 1;
    const int tid = threadIdx.x;
    const int pid = tid / G;
    constexpr int CFG_DOUBLES = (int)((sizeof(Options) + sizeof(Bounds) + 15) / 16) * 2;
    Options* s_opt = reinterpret_cast<Options*>(enl_smem);
    Bounds* s_bnd = reinterpret_cast<Bounds*>(reinterpret_cast<char*>(enl_smem) + sizeof(Options));
    if (tid == 0) { *s_opt = a.opt; *s_bnd = a.bnd; }
    __syncthreads();
    double* objs = enl_smem + CFG_DOUBLES;
    double* small = objs + (size_t)SOLVER_DOUBLES * LY::PPC;
    double* distb = small + (size_t)LY::nD * LY::PPC;
    int* ints = reinterpret_cast<int*>(distb + (size_t)LY::DCOLS * LY::MS * NT);
    DevGroup<G> g;
    SolverT& S = *new (objs + (size_t)SOLVER_DOUBLES * pid) SolverT(small, ints, distb, pid, *s_opt, *s_bnd);
    g.sync();
    for (;;) {
        unsigned long long nb = 0;
        if (g.lane == 0) nb = atomicAdd(a.counter, 1ULL);
        if (G > 1) nb = __shfl_sync(g.mask, nb, 0, G);
        const long long b = (long long)nb;
        if (b >= a.B) break;
        if (a.step) {
            S.step_only(a.x + b * Fam::N, a.r + b * Fam::M, a.J + b * (long long)(Fam::N * Fam::M), a.c + b * LY::LMAX,
                        a.A + b * (long long)(LY::LMAX * Fam::N));
            S.store_step(a.p, a.lam, a.active, a.info, b);
        } else {
            S.eval_only(a.x + b * Fam::N, a.fd, b);
            S.store_eval(a.r, a.J, a.c, a.A, b);
        }
        g.sync();
    }
}

__global__ void det_exp_kernel(const double* x, double* y, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) y[i] = det_exp(x[i]);
}

struct FamilyInfo { int n, m, q, ni, maxb; };

}  // namespace

struct enlsipb200_handle_s {
    int family;
    int device;
    FamilyInfo fi;
    Bounds bnd;
    int l;
    unsigned long long* counter = nullptr;
    const double* data[3] = {nullptr, nullptr, nullptr};
    long long slot_count[3] = {-1, -1, -1};      // values bound to each data slot (enlsipb200_set_data)
    double* owned[3] = {nullptr, nullptr, nullptr};
    long long owned_count[3] = {0, 0, 0};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    long long launches = 0;
    // launch geometry
    int regs = 0, smem = 0, nt = 0, ctas_per_sm = 0, grid = 0, G = 0;
    int num_sms = 0;
    // staging for host-buffer calls
    void* stage = nullptr;
    size_t stage_bytes = 0;
    // family data passed as HOST pointers is uploaded lazily: per-problem slots travel chunk by chunk inside
    // enlsipb200_solve_batch (host-buffer path), overlapped with the solves of the previous chunk
    const double* host_src[3] = {nullptr, nullptr, nullptr};
    long long host_count[3] = {0, 0, 0};
    bool host_pending[3] = {false, false, false};
    cudaStream_t copy_stream = nullptr;
    static constexpr int MAX_CHUNKS = 16;
    cudaEvent_t ev_ready[MAX_CHUNKS] = {};
};

namespace {

template <class Fam, int G, int NT>
size_t smem_total() {
    using LY = Layout<Fam, G, NT>;
    size_t sd = ((sizeof(Solver<Fam, DevGroup<G>, NT>) + 7) / 8) | 1;
    size_t cfg = ((sizeof(Options) + sizeof(Bounds) + 15) / 16) * 16;
    return LY::smem_bytes() + sd * 8 * LY::PPC + cfg;
}

template <class Fam, int G, int NT>
int configure(enlsipb200_handle h) {
    using LY = Layout<Fam, G, NT>;
    auto kern = enlsip_solve_batch_kernel<Fam, G, NT>;
    size_t smem = smem_total<Fam, G, NT>();
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, kern));
    int occ = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem));
    if (occ < 1) return fail(ENLSIPB200_ECUDA, "kernel does not fit on an SM");
    h->regs = fa.numRegs;
    h->smem = (int)smem;
    h->nt = NT;
    h->ctas_per_sm = occ;
    h->grid = occ * h->num_sms;
    h->G = G;
    return 0;
}

// first / last: this launch opens / closes the timed region of enlsipb200_last_kernel_ms (a chunked host-buffer solve
// is one region from its first to its last kernel)
template <class Fam, int G, int NT>
int launch(enlsipb200_handle h, const KernelArgs& a, cudaStream_t st, bool first = true, bool last = true) {
    using LY = Layout<Fam, G, NT>;
    long long groups_per_cta = NT / G;
    long long need = (a.B + groups_per_cta - 1) / groups_per_cta;
    int grid = (int)(need < (long long)h->grid ? need : (long long)h->grid);
    if (grid < 1) grid = 1;
    CU(cudaMemsetAsync(h->counter, 0, sizeof(unsigned long long), st));
    if (first) CU(cudaEventRecord(h->ev0, st));
    enlsip_solve_batch_kernel<Fam, G, NT><<<grid, NT, smem_total<Fam, G, NT>(), st>>>(a);
    CU(cudaGetLastError());
    if (last) CU(cudaEventRecord(h->ev1, st));
    h->timed = true;
    h->launches += 1;
    return 0;
}

// doubles per problem of a family-data slot (0 = the slot is shared by all problems of the batch)
int slot_stride(int family, int slot) {
    if (family == ENLSIPB200_FAMILY_GAUSS_PEAKS) return slot == 0 ? FamGaussPeaks::M : (slot == 1 ? 1 : 0);
#if defined(ENL_USER_FAMILY)
    if (family == ENLSIPB200_FAMILY_USER) return slot == 0 ? FamUser::STRIDE0 : (slot == 1 ? FamUser::STRIDE1 : 0);
#endif
    return 0;
}

// upload pending host slots completely: all of them (B < 0: device-buffer solves), or those that cannot travel chunk by
// chunk with a batch of B problems (slots shared by all problems, slots whose size does not match the batch)
int flush_pending(enlsipb200_handle h, cudaStream_t st, long long B) {
    for (int sl = 0; sl < 3; ++sl) {
        if (!h->host_pending[sl]) continue;
        const int sd = slot_stride(h->family, sl);
        if (B >= 0 && sd > 0 && h->host_count[sl] == B * sd) continue;
        CU(cudaMemcpyAsync(h->owned[sl], h->host_src[sl], (size_t)h->host_count[sl] * sizeof(double), cudaMemcpyHostToDevice, st));
        h->host_pending[sl] = false;
    }
    return 0;
}

template <int V>
using ic = std::integral_constant<int, V>;

// One thread per problem (families with a handful of residuals): the CTA size that fills the shared memory of an SM.
// These kernels are latency bound and gain with every resident problem (HS65: 6.6 / 7.8 / 8.4 M solves/s with 64 / 80 / 86
// problems per SM); the whole state of a problem lives in shared memory (2.6 KB for HS65).
template <class Fam>
constexpr int nt_thread_per_problem() {
    constexpr size_t cfg = ((sizeof(Options) + sizeof(Bounds) + 15) / 16) * 16;
    constexpr size_t sd = ((sizeof(Solver<Fam, DevGroup<1>, 8>) + 7) / 8) | 1;
    constexpr size_t per = Layout<Fam, 1, 8>::smem_bytes() / 8 + sd * 8;        // bytes per problem (smem_bytes is linear in NT)
    constexpr size_t budget = 225 * 1024 - cfg;
    constexpr int fit = (int)(budget / per) / 2 * 2;
    return fit > 128 ? 128 : (fit < 2 ? 1 : fit);      // (a family too large for 2 problems per SM still gets a kernel that fits)
}

// family id -> template instantiation
template <class F>
int with_family(int family, F&& f) {
#if defined(ENL_USER_FAMILY)
    // a user library holds the user's family only (compile time: one kernel instead of ten); few rows: one thread per
    // problem, otherwise one warp per problem
    if (family == ENLSIPB200_FAMILY_USER) return f(FamUser{}, ic<(FamUser::M <= 8 ? 1 : 32)>{}, ic<(FamUser::M <= 8 ? nt_thread_per_problem<FamUser>() : 32)>{});
    return fail(ENLSIPB200_EINVAL, "this library was compiled for ENLSIPB200_FAMILY_USER only");
#else
    switch (family) {
        case ENLSIPB200_FAMILY_HS65: return f(FamHS65{}, ic<1>{}, ic<nt_thread_per_problem<FamHS65>()>{});
        case ENLSIPB200_FAMILY_GAUSS_PEAKS: return f(FamGaussPeaks{}, ic<32>{}, ic<512>{});   // 16 problems per SM: all the shared memory and registers
        case ENLSIPB200_FAMILY_OSBORNE2: return f(FamOsborne2{}, ic<32>{}, ic<32>{});
        case ENLSIPB200_FAMILY_CHAINED_ROSENBROCK10: return f(FamChainedRosenbrock<10>{}, ic<32>{}, ic<32>{});
        case ENLSIPB200_FAMILY_CHAINED_WOOD20: return f(FamChainedWood<20>{}, ic<32>{}, ic<32>{});
    }
    if (family == ENLSIPB200_FAMILY_USER)
        return fail(ENLSIPB200_EINVAL, "ENLSIPB200_FAMILY_USER lives in the library written by enlsipb200_compile_family");
    return fail(ENLSIPB200_EINVAL, "unknown family id");
#endif
}

Options make_options(const enlsipb200_options* o, int n, int m) {
    enlsipb200_options d;
    enlsipb200_default_options(&d);
    if (o) d = *o;
    double abs_tol = (d.abs_tol == d.abs_tol) ? d.abs_tol : EPS;
    double rel_tol = (d.rel_tol == d.rel_tol) ? d.rel_tol : sqrt(abs_tol);
    double c_tol = (d.c_tol == d.c_tol) ? d.c_tol : rel_tol;
    double x_tol = (d.x_tol == d.x_tol) ? d.x_tol : rel_tol;
    Options r;
    r.max_iter = d.max_iter;
    r.scaling = d.scaling;
    r.jac_mode = d.jac_mode;
    r.second_derivatives = (n + m < 1000) ? 1 : 0;   // EF:2658
    r.time_limit = d.time_limit;
    r.eps_abs = 1e-10;                               // EF:2651 (abs_tol is not forwarded)
    r.eps_rel = rel_tol;
    r.eps_x = x_tol;
    r.eps_c = c_tol;
    r.eps_rank = SQRT_EPS;                           // solver.jl:81
    return r;
}

}  // namespace

extern "C" {

int enlsipb200_version(void) { return 100; }

const char* enlsipb200_last_error(void) { return g_err.c_str(); }

void enlsipb200_default_options(enlsipb200_options* o) {
    if (!o) return;
    o->max_iter = 100;
    o->scaling = 0;
    o->jac_mode = ENLSIPB200_JAC_ANALYTIC;
    o->reserved = 0;
    o->time_limit = 1e3;
    o->abs_tol = NAN;
    o->rel_tol = NAN;
    o->c_tol = NAN;
    o->x_tol = NAN;
}

int enlsipb200_create(int family, const double* x_low, const double* x_upp, int device, enlsipb200_handle* out) {
    if (!out) return fail(ENLSIPB200_EINVAL, "out is NULL");
    *out = nullptr;
    FamilyInfo fi{0, 0, 0, 0, 0};
    int known = with_family(family, [&](auto fam, auto, auto) {
        using Fm = decltype(fam);
        fi = {Fm::N, Fm::M, Fm::Q, Fm::NI, Fm::MAXB};
        return 0;
    });
    if (known != 0) return known;
    if (fi.maxb == 0 && ((x_low && [&] { for (int j = 0; j < fi.n; ++j) if (isfinite(x_low[j])) return true; return false; }()) ||
                         (x_upp && [&] { for (int j = 0; j < fi.n; ++j) if (isfinite(x_upp[j])) return true; return false; }())))
        return fail(ENLSIPB200_EINVAL, "this family is compiled without bound rows");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(ENLSIPB200_ENOGPU, "no CUDA device: the ENLSIP engine has no CPU fallback");
    if (device < 0) CU(cudaGetDevice(&device));
    if (device >= ndev) return fail(ENLSIPB200_EINVAL, "device index out of range");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(ENLSIPB200_ENOGPU, "sm_100a (B200) device required");
    auto* h = new enlsipb200_handle_s();
    h->family = family;
    h->device = device;
    h->fi = fi;
    h->num_sms = prop.multiProcessorCount;
    memset(&h->bnd, 0, sizeof(Bounds));
    for (int j = 0; j < fi.n; ++j)
        if (x_low && isfinite(x_low[j])) { h->bnd.lo_idx[h->bnd.nlo] = j; h->bnd.lo_val[h->bnd.nlo] = x_low[j]; h->bnd.nlo++; }
    for (int j = 0; j < fi.n; ++j)
        if (x_upp && isfinite(x_upp[j])) { h->bnd.up_idx[h->bnd.nup] = j; h->bnd.up_val[h->bnd.nup] = x_upp[j]; h->bnd.nup++; }
    h->l = fi.q + fi.ni + h->bnd.nlo + h->bnd.nup;
    if (h->l == 0) { delete h; return fail(ENLSIPB200_EINVAL, "There must be at least one constraint"); }  // cnls_model.jl:367
    int rc = 0;
    if (cudaMalloc(&h->counter, sizeof(unsigned long long)) != cudaSuccess) { delete h; return fail(ENLSIPB200_ENOMEM, "cudaMalloc"); }
    if (cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) { delete h; return fail(ENLSIPB200_ECUDA, "cudaEventCreate"); }
    if (family == ENLSIPB200_FAMILY_GAUSS_PEAKS) {   // the family's shared abscissa table (enl_families.h)
        double tt[128];
        for (int i = 0; i < 128; ++i) tt[i] = FamGaussPeaks::abscissa(i);
        if (cudaMemcpyToSymbol(g_gp_t, tt, sizeof(tt)) != cudaSuccess) { enlsipb200_destroy(h); return fail(ENLSIPB200_ECUDA, "cudaMemcpyToSymbol"); }
    }
    rc = with_family(family, [&](auto fam, auto g_, auto nt_) {
        return configure<decltype(fam), decltype(g_)::value, decltype(nt_)::value>(h);
    });
    if (rc != 0) { enlsipb200_destroy(h); return rc; }
    *out = h;
    return 0;
}

int enlsipb200_destroy(enlsipb200_handle h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    if (h->counter) cudaFree(h->counter);
    for (int i = 0; i < 3; ++i)
        if (h->owned[i]) cudaFree(h->owned[i]);
    if (h->stage) cudaFree(h->stage);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->copy_stream) {
        for (int c = 0; c < enlsipb200_handle_s::MAX_CHUNKS; ++c)
            if (h->ev_ready[c]) cudaEventDestroy(h->ev_ready[c]);
        cudaStreamDestroy(h->copy_stream);
    }
    delete h;
    return 0;
}

int enlsipb200_dims(enlsipb200_handle h, int* n, int* m, int* nb_eq, int* nb_constraints, int* lmax) {
    if (!h) return fail(ENLSIPB200_EINVAL, "null handle");
    if (n) *n = h->fi.n;
    if (m) *m = h->fi.m;
    if (nb_eq) *nb_eq = h->fi.q;
    if (nb_constraints) *nb_constraints = h->l;
    if (lmax) *lmax = h->fi.q + h->fi.ni + h->fi.maxb;
    return 0;
}

int enlsipb200_set_data(enlsipb200_handle h, int slot, const double* ptr, long long count, int on_device, void* stream) {
    if (!h || slot < 0 || slot > 2) return fail(ENLSIPB200_EINVAL, "bad handle/slot");
    CU(cudaSetDevice(h->device));
    h->slot_count[slot] = count;
    if (on_device) { h->data[slot] = ptr; h->host_pending[slot] = false; return 0; }
    if (h->owned_count[slot] < count) {
        if (h->owned[slot]) CU(cudaFree(h->owned[slot]));
        h->owned[slot] = nullptr;
        CU(cudaMalloc(&h->owned[slot], (size_t)count * sizeof(double)));
        h->owned_count[slot] = count;
    }
    // the copy itself is deferred to the next solve (see host_pending): the host buffer must stay valid until then
    (void)stream;
    h->host_src[slot] = ptr;
    h->host_count[slot] = count;
    h->host_pending[slot] = true;
    h->data[slot] = h->owned[slot];
    return 0;
}

int enlsipb200_solve_batch(enlsipb200_handle h, long long B, const double* x0, const enlsipb200_options* opt, double* x,
                           double* f, int* exit_code, int* status, int* iters, int* nact, int* active, int* counters,
                           double* trace, int trace_cap, int on_device, void* stream) {
    if (!h) return fail(ENLSIPB200_EINVAL, "null handle");
    if (B < 0 || !x0 || !x || !f || !exit_code || !status || !iters || !nact)
        return fail(ENLSIPB200_EINVAL, "x0, x, f, exit_code, status, iters, nact are required");
    if (B == 0) return 0;     // an empty batch is a no-op (and may come with empty data arrays)
    if ((h->family == ENLSIPB200_FAMILY_GAUSS_PEAKS || h->family == ENLSIPB200_FAMILY_OSBORNE2) && (!h->data[0] || !h->data[1]))
        return fail(ENLSIPB200_EINVAL, "this family needs data slots 0 and 1 (GAUSS_PEAKS: y, S; OSBORNE2: t, y)");
#if defined(ENL_USER_FAMILY)
    if (!FamUser::HAS_ANALYTIC && (!opt || opt->jac_mode != ENLSIPB200_JAC_FORWARD_DIFF))
        return fail(ENLSIPB200_EINVAL, "this user family was compiled without Jacobians: set jac_mode = ENLSIPB200_JAC_FORWARD_DIFF");
#endif
    for (int sl = 0; sl < 3; ++sl) {      // a per-problem data slot shorter than the batch would be read out of bounds
        const int sd = slot_stride(h->family, sl);
        if (sd > 0 && h->data[sl] && h->slot_count[sl] >= 0 && h->slot_count[sl] < B * sd)
            return fail(ENLSIPB200_EINVAL, "data slot " + std::to_string(sl) + " holds " + std::to_string(h->slot_count[sl]) +
                                               " values, the batch needs " + std::to_string(B * sd));
    }
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n = h->fi.n, lmax = h->fi.q + h->fi.ni + h->fi.maxb;
    const int row_w = TRACE_HDR + n;
    KernelArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B;
    a.counter = h->counter;
    a.fd = FamilyData{h->data[0], h->data[1], h->data[2]};
    a.opt = make_options(opt, h->fi.n, h->fi.m);
    a.bnd = h->bnd;
    a.out.trace_cap = trace ? trace_cap : 0;
    if (on_device) {
        int rcf = flush_pending(h, st, -1);
        if (rcf != 0) return rcf;
        a.x0 = x0;
        a.out.x = x; a.out.f = f; a.out.exit_code = exit_code; a.out.status = status; a.out.iters = iters;
        a.out.nact = nact; a.out.active = active; a.out.counters = counters; a.out.trace = trace;
        int rc = with_family(h->family, [&](auto fam, auto g_, auto nt_) {
            return launch<decltype(fam), decltype(g_)::value, decltype(nt_)::value>(h, a, st);
        });
        if (rc != 0) return rc;
        if (!stream) CU(cudaStreamSynchronize(st));
        return 0;
    }
    // ---- host buffers: one staging allocation [x0 | x | f | trace | ints...], the batch cut into chunks whose
    //      uploads (x0 and the pending per-problem family data) overlap the solves of the chunk before ----
    size_t nd = (size_t)B * n * 2 + (size_t)B + (trace ? (size_t)B * trace_cap * row_w : 0);
    size_t ni = (size_t)B * (4 + lmax + 2);
    size_t bytes = nd * 8 + ni * 4;
    if (h->stage_bytes < bytes) {
        if (h->stage) CU(cudaFree(h->stage));
        h->stage = nullptr;
        h->stage_bytes = 0;
        if (cudaMalloc(&h->stage, bytes) != cudaSuccess) return fail(ENLSIPB200_ENOMEM, "cudaMalloc(staging)");
        h->stage_bytes = bytes;
    }
    double* dd = (double*)h->stage;
    double* d_x0 = dd; dd += (size_t)B * n;
    double* d_x = dd; dd += (size_t)B * n;
    double* d_f = dd; dd += (size_t)B;
    double* d_tr = nullptr;
    if (trace) { d_tr = dd; dd += (size_t)B * trace_cap * row_w; }
    int* di = (int*)dd;
    int* d_ec = di; di += B;
    int* d_st = di; di += B;
    int* d_it = di; di += B;
    int* d_na = di; di += B;
    int* d_act = di; di += (size_t)B * lmax;
    int* d_cnt = di;
    if (!h->copy_stream) {
        CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int c = 0; c < enlsipb200_handle_s::MAX_CHUNKS; ++c) CU(cudaEventCreateWithFlags(&h->ev_ready[c], cudaEventDisableTiming));
    }
    int rcf = flush_pending(h, st, B);           // what cannot be chunked goes up whole, before the first kernel
    if (rcf != 0) return rcf;
    const long long min_chunk = 65536;
    int nchunk = (int)((B + min_chunk - 1) / min_chunk);
    if (nchunk > 8) nchunk = 8;
    if (nchunk < 1) nchunk = 1;
    const long long csize = (B + nchunk - 1) / nchunk;
    cudaStream_t cs = h->copy_stream;
    CU(cudaEventRecord(h->ev_ready[enlsipb200_handle_s::MAX_CHUNKS - 1], st));   // copies start after earlier work on st
    CU(cudaStreamWaitEvent(cs, h->ev_ready[enlsipb200_handle_s::MAX_CHUNKS - 1], 0));
    if (trace) CU(cudaMemsetAsync(d_tr, 0, (size_t)B * trace_cap * row_w * 8, st));
    for (int c = 0; c < nchunk; ++c) {
        const long long off = c * csize, cb = (off + csize <= B) ? csize : B - off;
        if (cb <= 0) { nchunk = c; break; }
        CU(cudaMemcpyAsync(d_x0 + off * n, x0 + off * n, (size_t)cb * n * 8, cudaMemcpyHostToDevice, cs));
        for (int sl = 0; sl < 3; ++sl) {
            const int sd = slot_stride(h->family, sl);
            if (h->host_pending[sl] && sd > 0)
                CU(cudaMemcpyAsync(h->owned[sl] + off * sd, h->host_src[sl] + off * sd, (size_t)cb * sd * 8, cudaMemcpyHostToDevice, cs));
        }
        CU(cudaEventRecord(h->ev_ready[c], cs));
    }
    for (int c = 0; c < nchunk; ++c) {
        const long long off = c * csize, cb = (off + csize <= B) ? csize : B - off;
        CU(cudaStreamWaitEvent(st, h->ev_ready[c], 0));
        KernelArgs ac = a;
        ac.B = cb;
        ac.x0 = d_x0 + off * n;
        const double* dp[3];
        for (int sl = 0; sl < 3; ++sl) {
            const int sd = slot_stride(h->family, sl);
            dp[sl] = h->data[sl] ? h->data[sl] + off * sd : nullptr;
        }
        ac.fd = FamilyData{dp[0], dp[1], dp[2]};
        ac.out.x = d_x + off * n; ac.out.f = d_f + off; ac.out.exit_code = d_ec + off; ac.out.status = d_st + off;
        ac.out.iters = d_it + off; ac.out.nact = d_na + off; ac.out.active = d_act + off * lmax; ac.out.counters = d_cnt + off * 2;
        ac.out.trace = trace ? d_tr + (size_t)off * trace_cap * row_w : nullptr;
        int rc = with_family(h->family, [&](auto fam, auto g_, auto nt_) {
            return launch<decltype(fam), decltype(g_)::value, decltype(nt_)::value>(h, ac, st, c == 0, c == nchunk - 1);
        });
        if (rc != 0) return rc;
        CU(cudaMemcpyAsync(x + off * n, ac.out.x, (size_t)cb * n * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(f + off, ac.out.f, (size_t)cb * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(exit_code + off, ac.out.exit_code, (size_t)cb * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(status + off, ac.out.status, (size_t)cb * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(iters + off, ac.out.iters, (size_t)cb * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(nact + off, ac.out.nact, (size_t)cb * 4, cudaMemcpyDeviceToHost, st));
        if (active) CU(cudaMemcpyAsync(active + off * lmax, ac.out.active, (size_t)cb * lmax * 4, cudaMemcpyDeviceToHost, st));
        if (counters) CU(cudaMemcpyAsync(counters + off * 2, ac.out.counters, (size_t)cb * 2 * 4, cudaMemcpyDeviceToHost, st));
        if (trace) CU(cudaMemcpyAsync(trace + (size_t)off * trace_cap * row_w, ac.out.trace, (size_t)cb * trace_cap * row_w * 8, cudaMemcpyDeviceToHost, st));
    }
    for (int sl = 0; sl < 3; ++sl) h->host_pending[sl] = false;
    CU(cudaStreamSynchronize(st));
    return 0;
}

static int eval_or_step(enlsipb200_handle h, long long B, const double* x, const enlsipb200_options* opt, double* r, double* J,
                        double* c, double* A, int step, double* p, double* lam, int* active, int* info, void* stream);

int enlsipb200_eval_batch(enlsipb200_handle h, long long B, const double* x, const enlsipb200_options* opt, double* r,
                          double* J, double* c, double* A, int on_device, void* stream) {
    if (!h) return fail(ENLSIPB200_EINVAL, "null handle");
    if (B < 0 || !x) return fail(ENLSIPB200_EINVAL, "x is required");
    if (B == 0) return 0;
    if (!on_device) return fail(ENLSIPB200_EINVAL, "enlsipb200_eval_batch works on device buffers (the outputs are B x m x n)");
    if ((h->family == ENLSIPB200_FAMILY_GAUSS_PEAKS || h->family == ENLSIPB200_FAMILY_OSBORNE2) && (!h->data[0] || !h->data[1]))
        return fail(ENLSIPB200_EINVAL, "this family needs data slots 0 and 1");
    return eval_or_step(h, B, x, opt, r, J, c, A, 0, nullptr, nullptr, nullptr, nullptr, stream);
}

int enlsipb200_step_batch(enlsipb200_handle h, long long B, const double* x, const double* r, const double* J, const double* c,
                          const double* A, const enlsipb200_options* opt, double* p, double* lam, int* active, int* info,
                          int on_device, void* stream) {
    if (!h) return fail(ENLSIPB200_EINVAL, "null handle");
    if (B < 0 || !x || !r || !J || !c || !A || !p) return fail(ENLSIPB200_EINVAL, "x, r, J, c, A, p are required");
    if (B == 0) return 0;
    if (!on_device) return fail(ENLSIPB200_EINVAL, "enlsipb200_step_batch works on device buffers");
    return eval_or_step(h, B, x, opt, const_cast<double*>(r), const_cast<double*>(J), const_cast<double*>(c),
                        const_cast<double*>(A), 1, p, lam, active, info, stream);
}

static int eval_or_step(enlsipb200_handle h, long long B, const double* x, const enlsipb200_options* opt, double* r, double* J,
                        double* c, double* A, int step, double* p, double* lam, int* active, int* info, void* stream) {
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    int rcf = flush_pending(h, st, -1);
    if (rcf != 0) return rcf;
    EvalArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.counter = h->counter; a.x = x;
    a.fd = FamilyData{h->data[0], h->data[1], h->data[2]};
    a.opt = make_options(opt, h->fi.n, h->fi.m);
    a.bnd = h->bnd;
    a.r = r; a.J = J; a.c = c; a.A = A;
    a.step = step; a.p = p; a.lam = lam; a.active = active; a.info = info;
    int rc = with_family(h->family, [&](auto fam, auto g_, auto nt_) {
        using Fm = decltype(fam);
        constexpr int G = decltype(g_)::value, NT = decltype(nt_)::value;
        auto kern = enlsip_eval_batch_kernel<Fm, G, NT>;
        const size_t smem = smem_total<Fm, G, NT>();
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        long long need = (B + NT / G - 1) / (NT / G);
        int grid = (int)(need < (long long)h->grid ? need : (long long)h->grid);
        CU(cudaMemsetAsync(h->counter, 0, sizeof(unsigned long long), st));
        CU(cudaEventRecord(h->ev0, st));
        kern<<<grid < 1 ? 1 : grid, NT, smem, st>>>(a);
        CU(cudaGetLastError());
        CU(cudaEventRecord(h->ev1, st));
        h->timed = true;
        h->launches += 1;
        return 0;
    });
    if (rc != 0) return rc;
    if (!stream) CU(cudaStreamSynchronize(st));
    return 0;
}

// Replaces the reference's "any closure" plugin surface (cnls_model.jl:11-62, 345-378): the user's residual /
// constraint functions arrive as CUDA C++ source and are compiled, together with the solver headers that sit next to
// this library (../csrc relative to the .so, found through dladdr), into a library with this same C ABI.
int enlsipb200_compile_family(const char* source, int n, int m, int nb_eq, int nb_ineq, int stride0, int stride1,
                              int has_jacobians, const char* out_lib_path, const char* work_dir) {
    if (!source || !out_lib_path || !work_dir) return fail(ENLSIPB200_EINVAL, "NULL argument");
    if (n < 1 || n > MAX_N) return fail(ENLSIPB200_EINVAL, "batched user families support 1 <= n <= 32 parameters (larger models: enlsipb200_large_compile_family when n + m >= 1000)");
    if (m < 1 || m > 4096) return fail(ENLSIPB200_EINVAL, "user families support 1 <= m <= 4096 residuals (larger problems: the large-Jacobian regime)");
    if (nb_eq < 0 || nb_ineq < 0 || nb_eq + nb_ineq > MAX_N) return fail(ENLSIPB200_EINVAL, "0 <= nb_eq + nb_ineq <= 32");
    if (stride0 < 0 || stride1 < 0) return fail(ENLSIPB200_EINVAL, "negative data stride");
    Dl_info info;
    if (!dladdr((void*)&enlsipb200_version, &info) || !info.dli_fname) return fail(ENLSIPB200_EINVAL, "cannot locate the library on disk");
    std::string lib = info.dli_fname;
    const size_t slash = lib.rfind('/');
    const std::string libdir = slash == std::string::npos ? "." : lib.substr(0, slash);
    const std::string csrc = libdir + "/../csrc";
    const std::string unit = csrc + "/enlsip_b200.cu";
    if (access(unit.c_str(), R_OK) != 0) return fail(ENLSIPB200_EINVAL, "solver sources not found at " + csrc);
    const std::string wd = work_dir;
    const std::string pre = wd + "/enl_user_prelude.h";
    FILE* fp = fopen(pre.c_str(), "w");
    if (!fp) return fail(ENLSIPB200_EINVAL, "cannot write " + pre);
    fprintf(fp, "// generated by enlsipb200_compile_family\n#pragma once\n#define ENL_USER_FAMILY 1\n#define ENL_USER_N %d\n"
                "#define ENL_USER_M %d\n#define ENL_USER_Q %d\n#define ENL_USER_NI %d\n#define ENL_USER_STRIDE0 %d\n"
                "#define ENL_USER_STRIDE1 %d\n#define ENL_USER_HAS_JAC %d\n#include \"%s/enl_base.h\"\nusing namespace enl;\n"
                "#line 1 \"user_family_source\"\n%s\n",
            n, m, nb_eq, nb_ineq, stride0, stride1, has_jacobians ? 1 : 0, csrc.c_str(), source);
    fclose(fp);
    const std::string log = wd + "/enl_user_build.log";
    const char* nvcc = getenv("ENLSIP_NVCC");
    std::string cmd = std::string(nvcc ? nvcc : "nvcc") +
                      " -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden -shared"
                      " -DENL_COMPACT_CODE=1 -include \"" + pre + "\" \"" + unit + "\" -o \"" + out_lib_path +
                      "\" -ldl > \"" + log + "\" 2>&1";
    const int rc = system(cmd.c_str());
    if (rc != 0) {
        std::string msg = "nvcc failed (" + cmd + "):\n";
        if (FILE* lf = fopen(log.c_str(), "r")) {
            char buf[512];
            size_t got;
            while (msg.size() < 6000 && (got = fread(buf, 1, sizeof(buf), lf)) > 0) msg.append(buf, got);
            fclose(lf);
        }
        return fail(ENLSIPB200_EINVAL, msg);
    }
    return 0;
}

// The same for the large regime (one problem, n + m >= 1000): the user's residual rows / constraints as device functions
// over a point accessor (csrc/enl_large_user.h) are compiled with csrc/enl_large.cu into a library that exports the
// enlsipb200_large_* API with family = ENLSIPB200_FAMILY_USER.
int enlsipb200_large_compile_family(const char* source, long long m, int nb_eq, int nb_ineq, int has_jacobians,
                                    const char* out_lib_path, const char* work_dir) {
    if (!source || !out_lib_path || !work_dir) return fail(ENLSIPB200_EINVAL, "NULL argument");
    if (m < 1 || nb_eq < 0 || nb_ineq < 0) return fail(ENLSIPB200_EINVAL, "bad sizes");
    Dl_info info;
    if (!dladdr((void*)&enlsipb200_version, &info) || !info.dli_fname) return fail(ENLSIPB200_EINVAL, "cannot locate the library on disk");
    std::string lib = info.dli_fname;
    const size_t slash = lib.rfind('/');
    const std::string libdir = slash == std::string::npos ? "." : lib.substr(0, slash);
    const std::string csrc = libdir + "/../csrc";
    const std::string unit = csrc + "/enl_large.cu";
    if (access(unit.c_str(), R_OK) != 0) return fail(ENLSIPB200_EINVAL, "solver sources not found at " + csrc);
    const std::string wd = work_dir;
    const std::string pre = wd + "/enl_large_user_prelude.h";
    FILE* fp = fopen(pre.c_str(), "w");
    if (!fp) return fail(ENLSIPB200_EINVAL, "cannot write " + pre);
    fprintf(fp, "// generated by enlsipb200_large_compile_family\n#pragma once\n#define ENL_LARGE_USER_FAMILY 1\n"
                "#define ENL_LUSER_M %lldLL\n#define ENL_LUSER_Q %d\n#define ENL_LUSER_NI %d\n#define ENL_LUSER_HAS_JAC %d\n"
                "#include <cuda_runtime.h>\n#include <math.h>\n#include \"%s/enl_base.h\"\n#line 1 \"user_family_source\"\n%s\n",
            m, nb_eq, nb_ineq, has_jacobians ? 1 : 0, csrc.c_str(), source);
    fclose(fp);
    const std::string log = wd + "/enl_large_user_build.log";
    const char* nvcc = getenv("ENLSIP_NVCC");
    std::string cmd = std::string(nvcc ? nvcc : "nvcc") +
                      " -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden -Xcompiler -fopenmp"
                      " -shared -include \"" + pre + "\" \"" + unit + "\" -o \"" + out_lib_path + "\" -lgomp -ldl > \"" + log + "\" 2>&1";
    const int rc = system(cmd.c_str());
    if (rc != 0) {
        std::string msg = "nvcc failed (" + cmd + "):\n";
        if (FILE* lf = fopen(log.c_str(), "r")) {
            char buf[512];
            size_t got;
            while (msg.size() < 6000 && (got = fread(buf, 1, sizeof(buf), lf)) > 0) msg.append(buf, got);
            fclose(lf);
        }
        return fail(ENLSIPB200_EINVAL, msg);
    }
    return 0;
}

int enlsipb200_last_kernel_ms(enlsipb200_handle h, float* ms) {
    if (!h || !ms) return fail(ENLSIPB200_EINVAL, "null argument");
    if (!h->timed) return fail(ENLSIPB200_EINVAL, "no solve has been launched");
    CU(cudaSetDevice(h->device));
    CU(cudaEventSynchronize(h->ev1));
    CU(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return 0;
}

int enlsipb200_kernel_info(enlsipb200_handle h, int* regs, int* smem, int* nt, int* ctas_per_sm, int* grid, int* G) {
    if (!h) return fail(ENLSIPB200_EINVAL, "null handle");
    if (regs) *regs = h->regs;
    if (smem) *smem = h->smem;
    if (nt) *nt = h->nt;
    if (ctas_per_sm) *ctas_per_sm = h->ctas_per_sm;
    if (grid) *grid = h->grid;
    if (G) *G = h->G;
    return 0;
}

long long enlsipb200_launch_count(enlsipb200_handle h) { return h ? h->launches : 0; }

int enlsipb200_det_exp(const double* x, double* y, long long n, int on_device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(ENLSIPB200_ENOGPU, "no CUDA device: the ENLSIP engine has no CPU fallback");
    if (n <= 0) return 0;
    const double* dx = x;
    double* dy = y;
    double *tx = nullptr, *ty = nullptr;
    if (!on_device) {
        CU(cudaMalloc(&tx, n * 8));
        CU(cudaMalloc(&ty, n * 8));
        CU(cudaMemcpy(tx, x, n * 8, cudaMemcpyHostToDevice));
        dx = tx; dy = ty;
    }
    det_exp_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dx, dy, n);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    if (!on_device) {
        CU(cudaMemcpy(y, ty, n * 8, cudaMemcpyDeviceToHost));
        cudaFree(tx); cudaFree(ty);
    }
    return 0;
}

}  // extern "C"
