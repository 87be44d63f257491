"""Row families on the TSQR path (ENLSIPB200_LARGE_FACTOR_TSQR, LargeCnlsModel(..., factor="tsqr")): [J | 0 | r] built row
major with n padded to a multiple of 32, compressed by the single-index family's tall-skinny QR, optionally row-sharded.

CPU: the flag's value in the three bindings, the create checks (before any device is touched), the shard split, and the
user sources compile for sm_100a.  GPU: the factor hook against LAPACK, chained Rosenbrock / the n = 4 data family / the
single-index model written as user source against the oracle and against the default path, determinism.  Two or more
GPUs: tools/row_tsqr_dist.py under torch.distributed.run."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.test_large_user_family import CR_SRC, MIX_MS, mix_family, mix_problem  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The single-index model of the built-in family (r_i = det_tanh(w_i . x) - y_i, csrc/enl_large_family.h) as user source:
# W [m, n] in slot 0, y in slot 1 followed by rho [nb] (the block equalities sum_{j in block k} x_j^2 - rho_k).  The dot
# product runs in a plain loop, so its bits differ from the built-in family's warp sums; the discrete decisions do not.
SI_NB = 1
SI_M = 1 << 16
SI_SRC = r"""
namespace enl_user {
__device__ __forceinline__ double si_dot(long long i, int n, const double* x, const double* W) {
    const double* w = W + i * n;
    double u = 0.0;
    for (int j = 0; j < n; ++j) u = fma(w[j], x[j], u);
    return u;
}
template <class X> __device__ double residual(long long i, int n, const X& x, const double* W, const double* y) {
    const double* w = W + i * n;
    double u = 0.0;
    for (int j = 0; j < n; ++j) u = fma(w[j], x[j], u);
    return __dsub_rn(enl::det_tanh(u), y[i]);
}
__device__ double jac_residual(long long i, int j, int n, const double* x, const double* W, const double*) {
    const double th = enl::det_tanh(si_dot(i, n, x, W));
    return __dmul_rn(__dsub_rn(1.0, __dmul_rn(th, th)), W[i * n + j]);
}
template <class X> __device__ double constraint(int k, int, const X& x, const double*, const double* y) {
    double s = 0.0;
    for (int j = 4 * k; j < 4 * k + 4; ++j) s = __dadd_rn(s, __dmul_rn(x[j], x[j]));
    return __dsub_rn(s, y[ENL_LUSER_M + k]);
}
__device__ double jac_constraint(int k, int j, int, const double* x, const double*, const double*) {
    return (j >= 4 * k && j < 4 * k + 4) ? __dmul_rn(2.0, x[j]) : 0.0;
}
}
"""


def si_family(m=SI_M):
    import enlsip_jl_b200 as E
    return E.LargeUserFamily(SI_SRC, m=m, nb_eqcons=SI_NB, has_jacobians=True, data=("W", "y"),
                             name="si_user" if m == SI_M else "si%d_user" % m)


def si_data(d):
    """data slots of SI_SRC from a synth.gen_single_index problem"""
    return {"W": d["W"], "y": np.concatenate([d["y"], d["rho"]])}


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_flag_value_agrees_across_bindings():
    import enlsip_jl_b200 as E
    hdr = open(os.path.join(ROOT, "include", "enlsip_b200.h")).read()
    jl = open(os.path.join(ROOT, "enlsip.jl_b200", "julia", "EnlsipB200.jl")).read()
    h = int(re.search(r"#define ENLSIPB200_LARGE_FACTOR_TSQR (0x[0-9a-fA-F]+|\d+)", hdr).group(1), 0)
    j = int(re.search(r"const LARGE_FACTOR_TSQR = Cint\((0x[0-9a-fA-F]+|\d+)\)", jl).group(1), 0)
    assert h == j == E.capi.LARGE_FACTOR_TSQR == 0x100
    # the flag must not collide with a family id
    for fam in (E.capi.FAMILY_SINGLE_INDEX, E.capi.FAMILY_LARGE_CHAINED_ROSENBROCK, E.capi.FAMILY_USER):
        assert fam & h == 0


def test_create_checks_before_device():
    """Refusals of enlsipb200_large_create with and without the flag: argument errors (-1) on a machine with or
    without a GPU."""
    import ctypes
    import enlsip_jl_b200 as E
    L, F = E.capi.lib(), E.capi.LARGE_FACTOR_TSQR
    cr = E.capi.FAMILY_LARGE_CHAINED_ROSENBROCK
    h = ctypes.c_void_p()
    # n + m < 1000 stays in the batched regime
    assert L.enlsipb200_large_create(cr | F, 10, 18, 18, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"batched engine" in L.enlsipb200_large_last_error()
    # more local rows than global rows
    assert L.enlsipb200_large_create(cr | F, 1000, 2000, 1998, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"m_local <= m_global" in L.enlsipb200_large_last_error()
    # m_global must be the family's m(n)
    assert L.enlsipb200_large_create(cr | F, 1000, 1000, 2000, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    # without the flag a row family is still not row-sharded, with the same error
    assert L.enlsipb200_large_create(cr, 1000, 1000, 1998, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    assert b"general families are not row-sharded" in L.enlsipb200_large_last_error()
    # the flag does not turn an unknown family into a known one
    assert L.enlsipb200_large_create(99 | F, 1000, 1998, 1998, 0, 0, None, None, None, -1, ctypes.byref(h)) == -1
    # the single-index family accepts the flag and keeps its own checks
    rho = np.ones(8)
    assert L.enlsipb200_large_create(E.capi.FAMILY_SINGLE_INDEX | F, 30, 1000, 1000, 4, 0, rho.ctypes.data, None, None, -1,
                                     ctypes.byref(h)) == -1
    assert b"multiple of 32" in L.enlsipb200_large_last_error()


def test_shard_split():
    from enlsip_jl_b200 import shard_rows
    for m in (1998, 50_000, 1 << 16, 1 << 20, 3 * 65536 + 4096, 700):
        for world in (1, 2, 3, 4, 8):
            parts = [shard_rows(m, r, world) for r in range(world)]
            assert sum(rows for _, rows in parts) == m
            assert all(rows >= 0 for _, rows in parts)
            row0 = 0
            for r, (a, rows) in enumerate(parts):
                assert a == row0
                row0 += rows
                if a + rows < m:
                    assert rows % 256 == 0                 # a shard with rows after it ends on a subtile boundary
    assert shard_rows(1 << 16, 1, 4) == (16384, 16384)
    assert shard_rows(1998, 0, 2) == (0, 768) and shard_rows(1998, 1, 2) == (768, 1230)
    assert shard_rows(700, 2, 4) == (512, 188) and shard_rows(700, 3, 4) == (700, 0)
    with pytest.raises(ValueError):
        shard_rows(1000, 2, 2)


def test_row_tsqr_user_sources_compile():
    """The single-index model as user source builds for sm_100a (no GPU needed) and exports the large API."""
    L = si_family().library()
    for sym in ("enlsipb200_large_create", "enlsipb200_large_solve", "enlsipb200_large_comm_init", "enlsipb200_large_factor"):
        assert hasattr(L, sym)


# ---------------------------------------------------------------------------------------------------------------------
# one B200
# ---------------------------------------------------------------------------------------------------------------------
def _cr_aug(x):
    n = x.size
    r = np.concatenate([10.0 * (x[:-1] ** 2 - x[1:]), x[:-1] - 1.0])      # csrc/enl_large_family.h
    J = np.zeros((2 * (n - 1), n))
    i = np.arange(n - 1)
    J[i, i] = 20.0 * x[:-1]
    J[i, i + 1] = -10.0
    J[n - 1 + i, i] = 1.0
    return np.hstack([J, r[:, None]])


def _si_aug(d, x):
    from oracle import problems as P
    th = P.det_tanh(d["W"] @ x)
    return np.hstack([(1.0 - th * th)[:, None] * d["W"], (th - d["y"])[:, None]])


def _check_factor(R, A):
    n = A.shape[1] - 1
    assert R.shape == (n + 1, n + 1)
    Rn = np.linalg.qr(A, mode="r")
    scale = np.abs(Rn).max()
    assert np.abs(np.abs(R) - np.abs(Rn)).max() <= 1e-13 * scale          # rows of R are unique up to sign
    G = A.T @ A
    assert np.abs(R.T @ R - G).max() <= 1e-13 * np.abs(G).max()
    assert np.all(np.tril(R, -1) == 0.0)
    rho, z, r = R[n, n], R[:n, n], A[:, n]
    assert rho >= 0.0
    # rho^2 = ||r||^2 - ||z||^2: the part of r outside the range of J, each unreduced entry counted once
    assert abs(rho * rho - (r @ r - z @ z)) <= 1e-12 * (r @ r)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 100, 256])
def test_row_tsqr_factor_vs_lapack_single_index_source(n):
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(SI_M, n, SI_NB, seed=60 + n)
    mod = E.LargeCnlsModel(si_family(), d["x0"], data=si_data(d), factor="tsqr")
    R, _, _ = mod.factor(d["x0"])
    assert mod.stats()["rows_pad"] == SI_M
    mod.close()
    _check_factor(R, _si_aug(d, d["x0"]))


@pytest.mark.gpu
def test_row_tsqr_factor_vs_lapack_chained_rosenbrock():
    """n = 1000 (padded to 1024), m = 1998 (padded to 2016 rows)"""
    import enlsip_jl_b200 as E
    from oracle import problems as P
    x0 = P.chained_rosenbrock(1000).x0
    x = x0 + 0.01 * np.random.default_rng(5).standard_normal(1000)
    mod = E.LargeCnlsModel("chained_rosenbrock", x0, factor="tsqr")
    R, _, _ = mod.factor(x)
    R2, _, _ = mod.factor(x)
    assert mod.stats()["rows_pad"] == 2016
    mod.close()
    assert np.array_equal(R, R2)
    _check_factor(R, _cr_aug(x))


def _solve(mod, **kw):
    import enlsip_jl_b200 as E
    E.solve(mod, trace_cap=60, **kw)
    return dict(x=mod.sol[0].copy(), f=mod.obj_value.copy(), exit_code=mod.exit_code.copy(), status=mod.status_code.copy(),
                iters=mod.iterations.copy(), nact=mod.nb_active.copy(), active=mod.active[0].copy(), trace=mod.trace[0].copy())


def _same_discrete(a, b):
    assert int(a["exit_code"][0]) == int(b["exit_code"][0]) and int(a["iters"][0]) == int(b["iters"][0])
    assert int(a["status"][0]) == int(b["status"][0]) and int(a["nact"][0]) == int(b["nact"][0])
    assert np.array_equal(np.sort(a["active"]), np.sort(b["active"]))
    k = int(a["iters"][0]) + 1
    assert np.array_equal(a["trace"][:k, 1:7], b["trace"][:k, 1:7])


@pytest.mark.gpu
@pytest.mark.parametrize("n,jac", [(1000, "analytic"), (1000, "forward_diff"), (400, "analytic"), (400, "forward_diff"),
                                   (334, "analytic"), (334, "forward_diff")])
def test_row_tsqr_chained_rosenbrock_vs_oracle(n, jac):
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O, problems as P
    from tests.test_large_host import compare_with_oracle
    pb = P.chained_rosenbrock(n, fd=(jac == "forward_diff"))
    mod = E.LargeCnlsModel("chained_rosenbrock", pb.x0, jacobian=jac, factor="tsqr")
    out = _solve(mod)
    st = mod.stats()
    assert st["rows_pad"] == (2 * (n - 1) + 31) // 32 * 32 and st["device_qrcp"] > 0
    again = _solve(mod)
    assert np.array_equal(again["x"], out["x"]) and again["f"][0] == out["f"][0]          # same bits
    mod.close()
    r = O.solve(pb, wallclock=False)
    assert int(out["status"][0]) == r.status == 1
    assert int(out["exit_code"][0]) == r.exit_code and int(out["iters"][0]) == r.iterations
    assert [int(v) for v in out["active"] if v > 0] == r.active
    if n == 1000:                                  # the reference's own run (chained_rosenbrock.jl)
        assert r.exit_code == 10300 and len(r.active) == 998
    if jac == "analytic":
        compare_with_oracle(out, r, n)
    else:
        assert abs(float(out["f"][0]) - r.f) <= 1e-8 * r.f
        assert np.linalg.norm(out["x"] - r.x) <= 1e-6 * np.linalg.norm(r.x)
    base = E.LargeCnlsModel("chained_rosenbrock", pb.x0, jacobian=jac)
    ref = _solve(base)
    assert base.stats()["rows_pad"] == 32                                                 # the default path ran
    base.close()
    _same_discrete(out, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("m", MIX_MS)
def test_row_tsqr_data_family_vs_oracle(m):
    """n = 4 (padded to 32), forward differences, one inequality + 8 bounds: the bars of
    check_user_data_family_vs_oracle."""
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O
    pb, t, y, lo, up = mix_problem(m=m)
    mod = E.LargeCnlsModel(mix_family(m), pb.x0, data={"t": t, "y": y}, x_low=lo, x_upp=up, factor="tsqr")
    E.solve(mod, trace_cap=100)
    assert mod.stats()["rows_pad"] == (m + 31) // 32 * 32
    r = O.solve(pb, wallclock=False)
    assert int(mod.status_code[0]) == r.status == 1, (mod.exit_code, mod.iterations, mod.obj_value, mod.sol, r.exit_code)
    assert sorted(int(v) for v in mod.active[0] if v > 0) == sorted(r.active)
    assert abs(int(mod.iterations[0]) - r.iterations) <= 1
    assert abs(float(mod.obj_value[0]) - r.f) <= 1e-8 * max(r.f, 1e-300)
    assert np.linalg.norm(mod.sol[0] - r.x) <= 1e-6 * np.linalg.norm(r.x)
    mod.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [256, 100])
def test_row_tsqr_single_index_source_vs_oracle(n):
    import enlsip_jl_b200 as E
    from oracle import enlsip_oracle as O, problems as P
    from tests.test_large_host import compare_with_oracle
    d = E.synth.gen_single_index(SI_M, n, SI_NB, seed=70 + n)
    mod = E.LargeCnlsModel(si_family(), d["x0"], data=si_data(d), factor="tsqr")
    assert mod.jacobian == "analytic" and mod.nb_constraints == SI_NB
    out = _solve(mod)
    assert mod.stats()["rows_pad"] == SI_M
    again = _solve(mod)
    assert np.array_equal(again["x"], out["x"]) and again["f"][0] == out["f"][0]
    mod.close()
    r = O.solve(P.single_index(d["W"], d["y"], d["rho"], d["x0"]), wallclock=False)
    compare_with_oracle(out, r, n)
    if n % 32 == 0:      # the built-in family (n a multiple of 32): same decisions
        b = E.LargeCnlsModel("single_index", d["x0"], d)
        ref = _solve(b)
        b.close()
        _same_discrete(out, ref)


@pytest.mark.gpu
def test_row_tsqr_unjoined_shard_refused():
    """A handle holding part of the rows refuses to solve or factor before comm_init has placed it."""
    import enlsip_jl_b200 as E
    from oracle import problems as P
    x0 = P.chained_rosenbrock(1000).x0
    mod = E.LargeCnlsModel("chained_rosenbrock", x0, factor="tsqr", shard=(0, 2))
    assert mod.rows == 768
    with pytest.raises(E.capi.EngineError, match="not joined"):
        mod.factor(x0)
    with pytest.raises(E.capi.EngineError, match="not joined"):
        E.solve(mod)
    with pytest.raises(E.capi.EngineError, match="one rank must hold"):
        mod.join(0, 1)
    mod.close()


# ---------------------------------------------------------------------------------------------------------------------
# two or more GPUs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_row_tsqr_sharded_matches_single_gpu():
    import torch
    ngpu = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if ngpu < 2:
        pytest.skip("needs two GPUs")
    world = 2 if ngpu < 4 else 4
    port = 29800 + (os.getpid() % 150)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "row_tsqr_dist.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "row_tsqr_dist: all checks passed" in p.stdout, p.stdout[-3000:]
