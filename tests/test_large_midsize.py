"""Mid-size problems (n + m < 1000) of the large regime's row families, created with ENLSIPB200_LARGE_MIDSIZE and solved
with second derivatives on, as the reference solves them at that size (second_derivatives = n + m < 1000, EF:2658):
Newton steps (method code 2, EF:348-423) with the Hessian of the Lagrangian by central differences on the device.

CPU: the flag's value in the three bindings, the create refusals (before any device is touched), the unflagged refusal
unchanged, chained Wood as large user source compiles for sm_100a, LargeCnlsModel's automatic flag and its refusals,
and why chained Wood's iteration path at n = 40 is not determined at the rounding level (oracle only).
GPU: the Cholesky hook against LAPACK dpotrf, chained Wood (user source) at n = 20 / 40 / 100, with bounds at n = 20,
and chained Rosenbrock (built in) at n = 10 / 100 against the oracle, the batched built-ins at n = 20 / 10,
determinism."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests.test_hostport import check_against_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WOOD_TOL = dict(rel_tol=1e-5, x_tol=1e-3, c_tol=1e-6)     # the reference's chained Wood test

# chained Wood (test/problems/chained_wood.jl:4-35; the batched family FamChainedWood of enl_families.h) as large user
# source: correctly rounded operations in the order numpy evaluates oracle/problems.py, so residuals, constraints and
# Jacobians are bit-identical to the oracle's.  Row = block * (n/2 - 1) + i, blocks in the order of the reference.
WOOD_SRC = r"""
namespace enl_user {
template <class X> __device__ double residual(long long row, int n, const X& x, const double*, const double*) {
    const double s = __dsqrt_rn(10.0);
    const int nb = n / 2 - 1, blk = (int)(row / nb), i = (int)(row % nb);
    const double xo = x[2 * i], xe = x[2 * i + 1], xo2 = x[2 * i + 2], xe2 = x[2 * i + 3];
    switch (blk) {
        case 0: return __dmul_rn(10.0, __dsub_rn(__dmul_rn(xo, xo), xe));
        case 1: return __dsub_rn(xo, 1.0);
        case 2: return __dmul_rn(__dmul_rn(3.0, s), __dsub_rn(__dmul_rn(xo2, xo2), xe2));
        case 3: return __dsub_rn(xo2, 1.0);
        case 4: return __dmul_rn(s, __dsub_rn(__dadd_rn(xe, xe2), 2.0));
        default: return __dmul_rn(__dsub_rn(xe, xe2), __ddiv_rn(1.0, s));
    }
}
__device__ double jac_residual(long long row, int j, int n, const double* x, const double*, const double*) {
    const double s = __dsqrt_rn(10.0);
    const int nb = n / 2 - 1, blk = (int)(row / nb), i = (int)(row % nb);
    switch (blk) {
        case 0: return j == 2 * i ? __dmul_rn(20.0, x[j]) : (j == 2 * i + 1 ? -10.0 : 0.0);
        case 1: return j == 2 * i ? 1.0 : 0.0;
        case 2: return j == 2 * i + 2 ? __dmul_rn(__dmul_rn(6.0, s), x[j]) : (j == 2 * i + 3 ? __dmul_rn(-3.0, s) : 0.0);
        case 3: return j == 2 * i + 2 ? 1.0 : 0.0;
        case 4: return (j == 2 * i + 1 || j == 2 * i + 3) ? s : 0.0;
        default: return j == 2 * i + 1 ? __ddiv_rn(1.0, s) : (j == 2 * i + 3 ? __ddiv_rn(-1.0, s) : 0.0);
    }
}
template <class X> __device__ double constraint(int kk, int, const X& x, const double*, const double*) {
    const int k = kk + 1;
    const double xk5 = x[k + 4];
    double acc = 0.0;
    for (int ii = (k - 5 > 1 ? k - 5 : 1); ii <= k + 1; ++ii) acc = __dadd_rn(acc, __dmul_rn(x[ii - 1], __dadd_rn(1.0, x[ii - 1])));
    const double v = __dmul_rn(__dadd_rn(2.0, __dmul_rn(5.0, __dmul_rn(xk5, xk5))), xk5);
    return __dadd_rn(__dadd_rn(v, 1.0), acc);
}
__device__ double jac_constraint(int kk, int j, int, const double* x, const double*, const double*) {
    const int k = kk + 1;
    if (j == k + 4) return __dadd_rn(2.0, __dmul_rn(15.0, __dmul_rn(x[j], x[j])));
    if (j >= (k - 5 > 1 ? k - 5 : 1) - 1 && j <= k) return __dadd_rn(1.0, __dmul_rn(2.0, x[j]));
    return 0.0;
}
}
"""


def wood_family(n):
    import enlsip_jl_b200 as E
    return E.LargeUserFamily(WOOD_SRC, m=6 * (n // 2 - 1), nb_eqcons=n - 7, has_jacobians=True, name="wood%d_user" % n)


def codes_of(mod):
    """method codes of the executed iterations (one trace row each)"""
    return [int(c) for c in mod.trace[0, :int(mod.iterations[0]) + 1, 6]]


def _out(mod):
    """the model's results in the layout of tests/test_hostport.py::check_against_oracle (B = 1)"""
    return dict(x=mod.sol, f=mod.obj_value, exit_code=mod.exit_code, iters=mod.iterations, active=mod.active,
                trace=mod.trace)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_flag_value_agrees_across_bindings():
    import enlsip_jl_b200 as E
    hdr = open(os.path.join(ROOT, "include", "enlsip_b200.h")).read()
    jl = open(os.path.join(ROOT, "enlsip.jl_b200", "julia", "EnlsipB200.jl")).read()
    h = int(re.search(r"#define ENLSIPB200_LARGE_MIDSIZE (0x[0-9a-fA-F]+|\d+)", hdr).group(1), 0)
    j = int(re.search(r"const LARGE_MIDSIZE = Cint\((0x[0-9a-fA-F]+|\d+)\)", jl).group(1), 0)
    assert h == j == E.capi.LARGE_MIDSIZE == 0x200
    for other in (E.capi.FAMILY_SINGLE_INDEX, E.capi.FAMILY_LARGE_CHAINED_ROSENBROCK, E.capi.FAMILY_USER,
                  E.capi.LARGE_FACTOR_TSQR):
        assert other & h == 0


def test_create_refusals_before_device():
    """Each refusal is an argument error (-1) with its own message, on a machine with or without a GPU."""
    import enlsip_jl_b200 as E
    L, M, T = E.capi.lib(), E.capi.LARGE_MIDSIZE, E.capi.LARGE_FACTOR_TSQR
    cr = E.capi.FAMILY_LARGE_CHAINED_ROSENBROCK
    h = ctypes.c_void_p()
    err = lambda: L.enlsipb200_large_last_error()
    rho = np.ones(8)
    # the single-index family has no Newton step
    assert L.enlsipb200_large_create(E.capi.FAMILY_SINGLE_INDEX | M, 32, 100, 100, 4, 0, rho.ctypes.data, None, None, -1,
                                     ctypes.byref(h)) == -1
    assert b"row families only" in err()
    # the flag never changes a large solve
    assert L.enlsipb200_large_create(cr | M, 1000, 1998, 1998, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"n + m < 1000 required" in err()
    assert L.enlsipb200_large_create(cr | M, 334, 666, 666, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1   # n + m = 1000
    assert b"n + m < 1000 required" in err()
    # no TSQR and no shards
    assert L.enlsipb200_large_create(cr | M | T, 100, 198, 198, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"do not combine" in err()
    assert L.enlsipb200_large_create(cr | M, 100, 100, 198, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"not row-sharded" in err()
    # without the flag nothing changes: n + m < 1000 stays refused with today's message
    for fam in (cr, cr | T):
        assert L.enlsipb200_large_create(fam, 100, 198, 198, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
        assert b"batched engine" in err()


def test_create_refuses_short_user_family():
    """m < n + 1: [J | r] has fewer rows than columns, so there is no tall QR to compress it; refused, not undefined.
    (A user library fixes m at compile time: chained Wood source compiled for n = 20 has m = 54 < n + 1 at n = 60.)"""
    import enlsip_jl_b200 as E
    L = wood_family(20).library()
    h = ctypes.c_void_p()
    assert L.enlsipb200_large_create(E.capi.FAMILY_USER | E.capi.LARGE_MIDSIZE, 60, 54, 54, 0, 0, None, None, None, -1,
                                     ctypes.byref(h)) == -1
    assert b"m >= n + 1" in L.enlsipb200_large_last_error()
    # the user library keeps the unflagged refusal as well
    assert L.enlsipb200_large_create(E.capi.FAMILY_USER, 20, 54, 54, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"batched engine" in L.enlsipb200_large_last_error()


def test_wood_user_source_compiles():
    """nvcc builds chained Wood as large user source for sm_100a (no GPU needed)."""
    for n in (20, 40, 100):
        L = wood_family(n).library()
        for sym in ("enlsipb200_large_create", "enlsipb200_large_solve", "enlsipb200_large_stats"):
            assert hasattr(L, sym)


def _wood40_oracle(x0):
    from oracle import enlsip_oracle as O, problems as P
    pb = P.chained_wood(40)
    pb.x0 = x0
    return O.solve(pb, wallclock=False, **WOOD_TOL)


def test_wood40_path_depends_on_one_ulp():
    """Chained Wood at n = 40 has no iteration path defined at the rounding level, in the oracle alone: moving one
    coordinate of x0 by one ulp takes 18 or 19 iterations instead of 21, to the same solution.  An engine that works on
    the compressed [J~ | r~] (its iterates agree with the oracle's to about 1e-14) cannot be held to the oracle's
    iteration count there; the converged point is determined."""
    from oracle import problems as P
    x0 = P.chained_wood(40).x0
    ref = _wood40_oracle(x0)
    assert (ref.exit_code, ref.iterations) == (10300, 21)
    for j, iters in ((1, 18), (2, 19)):
        x1 = x0.copy()
        x1[j] = np.nextafter(x1[j], np.inf)
        r = _wood40_oracle(x1)
        assert (r.exit_code, r.iterations) == (10300, iters)
        assert abs(r.f - ref.f) <= 1e-12 * ref.f
        assert np.linalg.norm(r.x - ref.x) <= 1e-12 * np.linalg.norm(ref.x)


def test_wood40_nullspace_basis_is_discontinuous():
    """Why: at the iterate where the paths part (the 12th Gauss-Newton direction), several pivot steps of
    qr(C.A', ColumnNorm()) (EF:700) reflect a column whose diagonal entry is zero up to rounding, so dlarfg's sign
    choice beta = -sign(alpha) ||x|| is decided by rounding.  A perturbation of C.A by one ulp keeps the pivot order
    but flips signs of diag(R) and turns Q1's null-space columns -- the basis of J2 = J Q1[:, rankA:] -- by O(1).  The
    subspace direction that follows (method code -1 with dimJ2 < rankJ2, EF:133-147) truncates in that basis, so its
    step, and everything after it, depends on rounding.  No Newton step is involved."""
    from scipy.linalg import lapack
    from oracle import enlsip_oracle as O, problems as P
    seen = {}
    orig_uws, orig_gn = O.update_working_set, O.gn_search_direction
    count = [0]

    def uws(W, rx, A, C, *a, **k):
        seen["CA"] = C.A.copy()
        return orig_uws(W, rx, A, C, *a, **k)

    def gn(*a, **k):
        count[0] += 1
        if count[0] == 12:
            seen["CA12"] = seen["CA"]
        return orig_gn(*a, **k)

    O.update_working_set, O.gn_search_direction = uws, gn
    try:
        O.solve(P.chained_wood(40), wallclock=False, max_iter=12, **WOOD_TOL)
    finally:
        O.update_working_set, O.gn_search_direction = orig_uws, orig_gn
    CA = seen["CA12"]
    t = CA.shape[0]

    def factor(M):
        f, jpvt, _, _, info = lapack.dgeqp3(np.asfortranarray(M.T.copy()))
        assert info == 0
        return np.sign(np.diag(f)), O.QRPivoted(M.T.copy()).Q_mul(np.eye(40))[:, t:], jpvt

    s0, N0, p0 = factor(CA)
    rng = np.random.default_rng(0)
    s1, N1, p1 = factor(CA * (1.0 + 2.3e-16 * rng.choice([-1.0, 1.0], CA.shape)))
    assert np.array_equal(p0, p1)                       # same pivots ...
    assert np.any(s0 != s1)                             # ... but reflector signs decided by rounding
    assert np.abs(N0 - N1).max() > 0.1                  # and an O(1) change of the null-space basis
    assert np.abs(CA @ N1).max() < 1e-12                # both are bases of the same null space


class _StubLib:
    """records enlsipb200_large_create's family argument and refuses, so no device is needed"""
    def __init__(self):
        self.families = []

    def enlsipb200_large_create(self, family, *args):
        self.families.append(int(family))
        return -1

    def enlsipb200_large_last_error(self):
        return b"stub"


def test_model_sets_flag_by_size(monkeypatch):
    import enlsip_jl_b200 as E
    stub = _StubLib()
    monkeypatch.setattr(E.capi, "lib", lambda: stub)
    cr, M, T = E.capi.FAMILY_LARGE_CHAINED_ROSENBROCK, E.capi.LARGE_MIDSIZE, E.capi.LARGE_FACTOR_TSQR
    for n, want in ((10, cr | M), (100, cr | M), (334, cr), (1000, cr)):     # n + m = 28, 298, 1000, 2998
        with pytest.raises(E.capi.EngineError):
            E.LargeCnlsModel("chained_rosenbrock", np.ones(n))
        assert stub.families[-1] == want, n
    with pytest.raises(E.capi.EngineError):
        E.LargeCnlsModel("chained_rosenbrock", np.ones(400), factor="tsqr")
    assert stub.families[-1] == cr | T
    # mid-size problems are neither factored by the TSQR nor sharded: refused before create
    calls = len(stub.families)
    with pytest.raises(AssertionError):
        E.LargeCnlsModel("chained_rosenbrock", np.ones(100), factor="tsqr")
    with pytest.raises(AssertionError):
        E.LargeCnlsModel("chained_rosenbrock", np.ones(100), factor="tsqr", shard=(0, 2))
    assert len(stub.families) == calls


def test_model_sets_flag_for_user_family(monkeypatch):
    import enlsip_jl_b200 as E
    stub = _StubLib()
    fam = wood_family(40)
    monkeypatch.setattr(fam, "library", lambda: stub)
    with pytest.raises(E.capi.EngineError):
        E.LargeCnlsModel(fam, np.ones(40))
    assert stub.families == [E.capi.FAMILY_USER | E.capi.LARGE_MIDSIZE]
    with pytest.raises(AssertionError):
        E.LargeCnlsModel(fam, np.ones(40), factor="tsqr")
    assert len(stub.families) == 1


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _spd(n, rng):
    B = rng.standard_normal((n, n))
    return B.T @ B + n * np.eye(n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 257, 997])
def test_dense_potrf_vs_lapack(n):
    import enlsip_jl_b200 as E
    from scipy.linalg import lapack
    rng = np.random.default_rng(n)
    A = _spd(n, rng)
    ref, info_ref = lapack.dpotrf(A, lower=0)
    a = np.asfortranarray(A.copy())
    info = ctypes.c_int(-7)
    E.capi.check(E.capi.lib().enlsipb200_dense_potrf(n, a.ctypes.data, ctypes.byref(info), -1))
    assert info.value == info_ref == 0
    print("\npotrf n=%d: %.3f ms (one CTA, CUDA events)" % (n, E.capi.lib().enlsipb200_dense_last_ms()))
    U, Ur = np.triu(a), np.triu(ref)
    assert np.linalg.norm(U - Ur) <= 1e-12 * np.linalg.norm(Ur), n
    # not positive definite: C = U' D U with D = I except D[j, j] = -1 has the negative pivot -U[j, j]^2 at step j
    for j in sorted({0, n // 2, n - 1}):
        D = np.ones(n)
        D[j] = -1.0
        C = Ur.T @ (D[:, None] * Ur)
        _, info_ref = lapack.dpotrf(C, lower=0)
        assert info_ref == j + 1
        a = np.asfortranarray(C.copy())
        E.capi.check(E.capi.lib().enlsipb200_dense_potrf(n, a.ctypes.data, ctypes.byref(info), -1))
        assert info.value == info_ref > 0, (n, j)


def _wood_oracle(n):
    """the oracle result at n = 20 / 40 (seconds), the committed fixture at n = 100 (make_midsize_fixture.py)"""
    from types import SimpleNamespace
    if n < 100:
        from oracle import enlsip_oracle as O, problems as P
        return O.solve(P.chained_wood(n), wallclock=False, **WOOD_TOL)
    g = np.load(os.path.join(ROOT, "tests", "golden", "midsize_wood%d_oracle.npz" % n))
    tr = [SimpleNamespace(t=r[0], rankA=r[1], rankJ2=r[2], dimA=r[3], dimJ2=r[4], code=r[5], index_del=r[6], exit_code=r[7],
                          x_new=None, p_norm=0.0) for r in g["trace"].tolist()]
    tr[-2].x_new = g["x_prev"]
    tr[-1].p_norm = float(g["last_p_norm"])
    return SimpleNamespace(exit_code=int(g["exit_code"]), iterations=int(g["iterations"]), active=[int(v) for v in g["active"]],
                           trace=tr, f=float(g["f"]), x=g["x"], threw=None)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [20, 40, 100])
def test_chained_wood_user_source_vs_oracle(n):
    """Chained Wood from the reference's x0 with its test's tolerances: all three direction methods, Newton steps on the
    device; n = 100 ends with -9 (more than five Newton steps) as the reference does.

    n = 20 meets the whole bar of check_against_oracle.  At n = 40 and 100 the iteration path is not determined at the
    rounding level -- the oracle itself changes it when x0 moves by one ulp (test_wood40_path_depends_on_one_ulp) -- so
    there the test checks what is determined: the exit code, the final working set and the number of Newton steps, and
    at n = 40, which converges, the solution and f to 1e-10 (the oracle's own spread over one-ulp starts is 2e-13)."""
    import enlsip_jl_b200 as E
    from oracle import problems as P
    x0 = P.chained_wood(n).x0
    mod = E.LargeCnlsModel(wood_family(n), x0)
    assert mod.midsize
    E.solve(mod, trace_cap=100, **WOOD_TOL)
    o = _wood_oracle(n)
    rows = int(mod.iterations[0]) + 1                               # one trace row per executed iteration
    if n == 20:
        check_against_oracle(_out(mod), 0, o, n, "wood%d" % n)
    else:
        assert int(mod.exit_code[0]) == o.exit_code
        assert [int(v) for v in mod.active[0] if v > 0] == o.active
        assert codes_of(mod).count(2) == [int(t.code) for t in o.trace].count(2)
        if o.exit_code > 0:      # a converged point; -9 stops wherever the sixth Newton step lands on the path taken
            assert abs(float(mod.obj_value[0]) - o.f) <= 1e-10 * abs(o.f)
            assert np.linalg.norm(mod.sol[0] - o.x) <= 1e-10 * np.linalg.norm(o.x)
    codes = [int(c) for c in mod.trace[0, :rows, 6]]
    st = mod.stats()
    print("\nchained Wood n=%d: exit %d, %d iterations, method codes %s, Newton steps %d, Hessian %.3f ms" %
          (n, int(mod.exit_code[0]), int(mod.iterations[0]), codes, st["newton_steps"], st["hessian_ms"]))
    assert 2 in codes and st["newton_steps"] == codes.count(2) and st["hessian_ms"] > 0
    if n == 100:
        assert int(mod.exit_code[0]) == -9
    if n == 20:     # the batched built-in takes the same discrete path
        b = E.CnlsModel("chained_wood20", x0[None, :])
        E.solve(b, trace_cap=100, **WOOD_TOL)
        assert (int(b.exit_code[0]), int(b.iterations[0])) == (int(mod.exit_code[0]), int(mod.iterations[0]))
        k = int(mod.iterations[0])
        cols = [1, 2, 3, 4, 5, 6, 9, 10]
        assert np.array_equal(np.asarray(b.trace)[0, :k][:, cols], mod.trace[0, :k][:, cols])
    mod.close()


@pytest.mark.gpu
def test_bounded_wood20_vs_oracle():
    """Bound rows in the Hessian: chained Wood n = 20 with x_low[18] = -1.3 and x_upp[19] = 1.9 ends with the lower
    bound (constraint 14) in the working set through four Newton steps, so the stencil evaluates (x_18 +- e) - x_low."""
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O, problems as P
    pw = P.chained_wood(20)
    lo, up = np.full(20, -np.inf), np.full(20, np.inf)
    lo[18], up[19] = -1.3, 1.9
    pb = O.make_problem(20, pw.m, pw.res, pw.jac_res, eq=pw.cons, jac_eq=pw.jac_cons, nb_eq=pw.q, x_low=lo, x_upp=up,
                        x0=pw.x0, name="wood20_bounded")
    o = O.solve(pb, wallclock=False, **WOOD_TOL)
    assert 14 in o.active and [t.code for t in o.trace].count(2) == 4
    mod = E.LargeCnlsModel(wood_family(20), pw.x0, x_low=lo, x_upp=up)
    E.solve(mod, trace_cap=100, **WOOD_TOL)
    check_against_oracle(_out(mod), 0, o, 20, "wood20 bounded")
    assert mod.stats()["newton_steps"] == 4
    mod.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,jac", [(10, "analytic"), (10, "forward_diff"), (100, "analytic"), (100, "forward_diff")])
def test_chained_rosenbrock_builtin_vs_oracle(n, jac):
    """The built-in row family at mid size: a pure Gauss-Newton solve (no code 2 in the reference's trace) through the
    mid-size path; n = 10 also against the batched chained_rosenbrock10."""
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O, problems as P
    pb = P.chained_rosenbrock(n, fd=(jac == "forward_diff"))
    mod = E.LargeCnlsModel("chained_rosenbrock", pb.x0, jacobian=jac)
    assert mod.midsize
    E.solve(mod, trace_cap=100)
    o = O.solve(pb, wallclock=False)
    check_against_oracle(_out(mod), 0, o, n, "rosenbrock%d %s" % (n, jac))
    if n == 10:
        b = E.CnlsModel("chained_rosenbrock10", pb.x0[None, :], jacobian=jac)
        E.solve(b, trace_cap=100)
        k = int(mod.iterations[0])
        assert (int(b.exit_code[0]), int(b.iterations[0])) == (int(mod.exit_code[0]), k)
        cols = [1, 2, 3, 4, 5, 6, 9, 10]
        assert np.array_equal(np.asarray(b.trace)[0, :k][:, cols], mod.trace[0, :k][:, cols])
    mod.close()


@pytest.mark.gpu
def test_midsize_deterministic():
    """Two solves with Newton steps give the same bits (fixed-order reductions in the Hessian kernel)."""
    import enlsip_jl_b200 as E
    from oracle import problems as P
    x0 = P.chained_wood(40).x0
    runs = []
    for _ in range(2):
        mod = E.LargeCnlsModel(wood_family(40), x0)
        E.solve(mod, trace_cap=100, **WOOD_TOL)
        runs.append((mod.sol.copy(), float(mod.obj_value[0]), mod.trace.copy()))
        mod.close()
    assert np.array_equal(runs[0][0].view(np.uint64), runs[1][0].view(np.uint64)) and runs[0][1] == runs[1][1]
    assert np.array_equal(runs[0][2].view(np.uint64), runs[1][2].view(np.uint64))
