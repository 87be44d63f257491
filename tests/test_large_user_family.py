"""User-defined problems of the large regime (enlsipb200_large_compile_family): the reference's "any closure" surface
(CnlsModel(residuals, n, m; eq_constraints, ineq_constraints, jacobian_*...), src/cnls_model.jl:345-359) for problems
with n + m >= 1000, as CUDA source over a point accessor.  GPU tests compare with the oracle; the CPU test only checks
that the sources compile for sm_100a (nvcc cross-compiles without a GPU)."""
import numpy as np
import pytest

# chained Rosenbrock (test/problems/chained_rosenbrock.jl:8-53) written as user source, analytic Jacobians
CR_SRC = r"""
namespace enl_user {
template <class X> __device__ double residual(long long i, int n, const X& x, const double*, const double*) {
    if (i < n - 1) { const double a = x[(int)i]; return __dmul_rn(10.0, __dsub_rn(__dmul_rn(a, a), x[(int)i + 1])); }
    return __dsub_rn(x[(int)(i - (n - 1))], 1.0);
}
__device__ double jac_residual(long long i, int j, int n, const double* x, const double*, const double*) {
    if (i < n - 1) return j == i ? __dmul_rn(20.0, x[j]) : (j == i + 1 ? -10.0 : 0.0);
    return j == i - (n - 1) ? 1.0 : 0.0;
}
template <class X> __device__ double constraint(int k, int, const X& x, const double*, const double*) {
    const double a = x[k], b = x[k + 1], c = x[k + 2];
    double v = __dadd_rn(__dmul_rn(3.0, __dmul_rn(__dmul_rn(b, b), b)), __dmul_rn(2.0, c));
    v = __dsub_rn(v, 5.0);
    v = __dadd_rn(v, __dmul_rn(sin(__dsub_rn(b, c)), sin(__dadd_rn(b, c))));
    v = __dadd_rn(v, __dmul_rn(4.0, b));
    v = __dsub_rn(v, __dmul_rn(a, exp(__dsub_rn(a, b))));
    return __dsub_rn(v, 3.0);
}
__device__ double jac_constraint(int k, int j, int, const double* x, const double*, const double*) {
    if (j < k || j > k + 2) return 0.0;
    const double a = x[k], b = x[k + 1], c = x[k + 2];
    const double e = exp(a - b), sm = sin(b - c), cm = cos(b - c), sp = sin(b + c), cp = cos(b + c);
    if (j == k) return -(a + 1.0) * e;
    if (j == k + 1) return 9.0 * b * b + cm * sp + sm * cp + 4.0 + a * e;
    return 2.0 - cm * sp + sm * cp;
}
}
"""

# a data-carrying problem without user Jacobians: y_i ~ x0 exp(-x1 t_i) + x2 / (1 + x3 t_i^2)  (n = 4, m points),
# one inequality (x0 + x2 <= 3), bounds on every parameter (the upper bound of x0 is active at the solution): forward
# differences throughout.  m is compiled into the library.  At m = 1200 the [J | r] QR (1200 x 5) runs in a thread-block
# cluster; at m = 50 000 it takes the unblocked column loop with reflectors too long for shared memory.
MIX_M = 1200
MIX_MS = (MIX_M, 50_000)
MIX_SRC = r"""
namespace enl_user {
template <class X> __device__ double residual(long long i, int, const X& x, const double* t, const double* y) {
    const double g = __dadd_rn(__dmul_rn(x[0], exp(__dmul_rn(-x[1], t[i]))),
                               __ddiv_rn(x[2], __dadd_rn(1.0, __dmul_rn(x[3], __dmul_rn(t[i], t[i])))));
    return __dsub_rn(y[i], g);
}
template <class X> __device__ double constraint(int, int, const X& x, const double*, const double*) {
    return __dsub_rn(3.0, __dadd_rn(x[0], x[2]));
}
}
"""


def mix_family(m=MIX_M):
    """MIX_SRC compiled for m data points (one library per m)."""
    import enlsip_jl_b200 as E
    return E.LargeUserFamily(MIX_SRC, m=m, nb_ineqcons=1, data=("t", "y"), name="mix_user" if m == MIX_M else "mix%d_user" % m)


def mix_problem(seed=3, m=MIX_M):
    """numpy restatement of MIX_SRC for the oracle (forward-difference Jacobians)."""
    from oracle import enlsip_oracle as O
    rng = np.random.default_rng(seed)
    t = np.linspace(0.0, 4.0, m)
    truth = np.array([2.0, 1.3, 0.7, 0.25])
    def model(x):
        return x[0] * np.exp(-x[1] * t) + x[2] / (1.0 + x[3] * (t * t))
    y = model(truth) + 0.01 * rng.standard_normal(m)
    lo, up = np.array([0.1, 0.1, 0.1, 0.05]), np.array([1.9, 5.0, 5.0, 5.0])
    x0 = np.minimum(truth * (1.0 + 0.2 * rng.uniform(-1, 1, 4)), up - 0.01)
    pb = O.make_problem(4, m, lambda x: y - model(x), None, ineq=lambda x: np.array([3.0 - (x[0] + x[2])]), jac_ineq=None,
                        nb_ineq=1, x_low=lo, x_upp=up, x0=x0, name="exp_plus_rational", fd=True)
    return pb, t, y, lo, up


def test_large_user_sources_compile():
    """nvcc builds both user families for sm_100a in this container (no GPU needed); the libraries export the large API."""
    import enlsip_jl_b200 as E
    for fam in (E.LargeUserFamily(CR_SRC, m=2 * (1000 - 1), nb_eqcons=998, has_jacobians=True, name="cr1000_user"),
                *(mix_family(m) for m in MIX_MS)):
        L = fam.library()
        for sym in ("enlsipb200_large_create", "enlsipb200_large_solve", "enlsipb200_large_set_data", "enlsipb200_large_stats"):
            assert hasattr(L, sym)


@pytest.mark.gpu
def test_user_chained_rosenbrock_equals_builtin():
    import enlsip_jl_b200 as E
    from oracle import problems as P
    n = 1000
    x0 = P.chained_rosenbrock(n).x0
    u = E.LargeCnlsModel(E.LargeUserFamily(CR_SRC, m=2 * (n - 1), nb_eqcons=n - 2, has_jacobians=True, name="cr1000_user"), x0)
    b = E.LargeCnlsModel("chained_rosenbrock", x0)
    E.solve(u)
    E.solve(b)
    assert np.array_equal(u.sol, b.sol) and int(u.exit_code[0]) == int(b.exit_code[0]) and float(u.obj_value[0]) == float(b.obj_value[0])
    assert int(u.iterations[0]) == int(b.iterations[0]) and np.array_equal(u.active, b.active)
    u.close(); b.close()


def check_user_data_family_vs_oracle(m):
    """n = 4, m data points (n + m >= 1000), data slots t / y, one inequality + 8 bounds, no user Jacobians (forward
    differences): status / iterations / working set as the oracle, f and x to the forward-difference noise floor."""
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O
    pb, t, y, lo, up = mix_problem(m=m)
    fam = mix_family(m)
    mod = E.LargeCnlsModel(fam, pb.x0, data={"t": t, "y": y}, x_low=lo, x_upp=up)
    assert mod.jacobian == "forward_diff" and mod.nb_constraints == 9
    E.solve(mod, trace_cap=100)
    r = O.solve(pb, wallclock=False)
    assert int(mod.status_code[0]) == r.status == 1, (mod.exit_code, mod.iterations, mod.obj_value, mod.sol, r.exit_code)
    assert sorted(int(v) for v in mod.active[0] if v > 0) == sorted(r.active)
    assert abs(int(mod.iterations[0]) - r.iterations) <= 1
    assert abs(float(mod.obj_value[0]) - r.f) <= 1e-8 * max(r.f, 1e-300)
    assert np.linalg.norm(mod.sol[0] - r.x) <= 1e-6 * np.linalg.norm(r.x)
    mod.close()


@pytest.mark.gpu
def test_user_data_family_vs_oracle():
    """m = 1200: [J | r] (1200 x 5) is factored in a thread-block cluster."""
    check_user_data_family_vs_oracle(MIX_M)


@pytest.mark.gpu
def test_tall_user_data_family_vs_oracle():
    """m = 50 000: [J | r] (50 000 x 5) is factored by the unblocked column loop, its reflectors too long for shared
    memory and read from global memory."""
    check_user_data_family_vs_oracle(MIX_MS[1])
