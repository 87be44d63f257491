"""Known-answer tests of the small stage's device kernels (csrc/enl_small.cuh) through the C ABI
(enlsipb200_dense_qrcp / enlsipb200_dense_mulq) against LAPACK: dgeqp3 (what `qr(M, ColumnNorm())` calls in the
reference, EF:223 / :700 / :769) and dormqr (`J * F_A.Q`, EF:219).  Sizes cover the unblocked dlaqp2 path
(min(m, n) <= 128), the blocked dlaqps path with its DMMA trailing update, panels that stop early because a column
norm has to be recomputed, and the tol3z-deciding matrices of tests/golden/qrcp_kat.npz.
Run on the B200 box:  python -m pytest tests -m gpu -x -q
"""
import ctypes

import numpy as np
import pytest
from scipy.linalg import lapack

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import enlsip_jl_b200 as E
    return E.capi.lib()


def dev_qrcp(L, A):
    vp = ctypes.c_void_p
    f = np.asfortranarray(A, dtype=float).copy(order="F")
    k = min(A.shape)
    tau = np.zeros(k); jp = np.zeros(A.shape[1], np.int32)
    rc = L.enlsipb200_dense_qrcp(A.shape[0], A.shape[1], f.ctypes.data_as(vp), tau.ctypes.data_as(vp), jp.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    return f, tau, jp


def test_qrcp_small_cases_vs_dgeqp3(L):
    from tests.test_kat import kat_cases, check_against_lapack
    for name, A in kat_cases():
        f, tau, jp = dev_qrcp(L, A)
        check_against_lapack(A, f, tau, jp, "device/" + name)


def test_qrcp_tol3z(L):
    from tests.test_kat import KAT
    for i in range(4):
        _, _, jp = dev_qrcp(L, KAT["tol3z_%d" % i])
        assert np.array_equal(jp, KAT["tol3z_%d_pivots" % i]), (i, jp)


@pytest.mark.parametrize("rows,cols,kind", [(300, 200, "random"), (257, 192, "random"), (500, 700, "random"),
                                             (700, 650, "graded"), (400, 300, "rank_deficient"),
                                             (1500, 1300, "random"), (520, 400, "near_dependent")])
def test_qrcp_blocked_vs_dgeqp3(L, rows, cols, kind):
    """min(rows, cols) > 128: dgeqp3 runs dlaqps panels of 32 for the leading min - 128 columns (trailing update here:
    mma.sync.m8n8k4.f64), then dlaqp2.  `near_dependent` makes panels stop early (a norm falls under the tol3z rule)."""
    rng = np.random.default_rng(rows * 1000 + cols)
    A = rng.standard_normal((rows, cols))
    if kind == "graded":
        A = A * np.logspace(0, -6, cols)[None, :]
    elif kind == "rank_deficient":
        A = rng.standard_normal((rows, 150)) @ rng.standard_normal((150, cols))
    elif kind == "near_dependent":
        B = rng.standard_normal((rows, 200))
        A = np.column_stack([B, B[:, :cols - 200] + 1e-5 * rng.standard_normal((rows, cols - 200))])
    f, tau, jp = dev_qrcp(L, A)
    qr, jl, tl, _, info = lapack.dgeqp3(np.asfortranarray(A))
    jl = jl - 1
    k = min(rows, cols)
    d = np.abs(np.diag(qr)[:k])
    r = int(np.sum(d > 1e-9 * d.max()))
    # a valid factorisation whatever the pivots: R'R = (A P)'(A P), non-increasing |diag| down to the numerical rank
    R = np.triu(f)[:k]
    AP = A[:, jp]
    G = AP.T @ AP
    assert np.abs(R.T @ R - G).max() <= 1e-12 * np.abs(G).max()
    assert sorted(jp.tolist()) == list(range(cols))
    # LAPACK's pivots and R (the same algorithm, different summation order inside the dot products: pivots can only
    # differ where two candidate norms agree to rounding, which these continuous random inputs do not produce)
    same = int(np.sum(jp[:r] == jl[:r]))
    assert same == r, (kind, "pivots differ from dgeqp3 at", np.nonzero(jp[:r] != jl[:r])[0][:8], jp[:8], jl[:8])
    Ro, Rlo = np.zeros_like(R), np.zeros_like(R)
    Ro[:, jp] = R
    Rlo[:, jl] = np.triu(qr)[:k]
    assert np.abs(Ro[:r] - Rlo[:r]).max() <= 1e-10 * d.max()
    assert np.abs(tau[:r] - tl[:r]).max() <= 1e-9


@pytest.mark.parametrize("mr,nq,k", [(40, 30, 7), (257, 256, 64), (300, 300, 300), (1000, 520, 129)])
def test_mulq_vs_dormqr(L, mr, nq, k):
    rng = np.random.default_rng(mr + nq + k)
    qr, tau, _, info = lapack.dgeqrf(np.asfortranarray(rng.standard_normal((nq, k))))
    M = np.asfortranarray(rng.standard_normal((mr, nq)))
    ref, _, info = lapack.dormqr("R", "N", qr, tau, M.copy(order="F"), max(1, 64 * mr))
    assert info == 0
    out = M.copy(order="F")
    vp = ctypes.c_void_p
    rc = L.enlsipb200_dense_mulq(mr, nq, k, np.asfortranarray(qr).ctypes.data_as(vp), tau.ctypes.data_as(vp), out.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    assert np.abs(out - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("frows,k", [(700, 33), (1000, 257), (4097, 520), (2000, 1999)])
@pytest.mark.parametrize("kind", [0, 1])
def test_reflect_vec_wy_vs_dormqr(L, frows, k, kind):
    """v <- Q' v / Q v by the cooperative compact-WY kernel (batched dlarft T factors) against LAPACK dormqr."""
    rng = np.random.default_rng(frows + k + kind)
    qr, tau, _, info = lapack.dgeqrf(np.asfortranarray(rng.standard_normal((frows, k))))
    v = rng.standard_normal(frows)
    ref, _, info = lapack.dormqr("L", "T" if kind == 0 else "N", qr, tau, np.asfortranarray(v.reshape(-1, 1)), max(1, 64 * frows))
    assert info == 0
    out = v.copy()
    vp = ctypes.c_void_p
    rc = L.enlsipb200_dense_vecop(kind, frows, k, np.asfortranarray(qr).ctypes.data_as(vp), tau.ctypes.data_as(vp), out.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    assert np.abs(out - ref[:, 0]).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("frows,k", [(40, 33), (300, 64), (700, 511), (3600, 3587), (5000, 4999)])
@pytest.mark.parametrize("kind", [2, 3])
def test_trsv_coop_vs_dtrtrs(L, frows, k, kind):
    """R \\ v and R' \\ v by the one-warp-per-block cooperative kernels against LAPACK dtrtrs (R well conditioned: a QR factor of
    a random matrix; the entries below the diagonal of f hold reflector data and must be ignored)."""
    rng = np.random.default_rng(frows + k + kind)
    qr, tau, _, info = lapack.dgeqrf(np.asfortranarray(rng.standard_normal((frows, k))))
    R = np.triu(qr[:k, :k])
    v = rng.standard_normal(k)
    ref, info = lapack.dtrtrs(np.asfortranarray(R), np.asfortranarray(v.reshape(-1, 1)), lower=0, trans=0 if kind == 2 else 1)
    assert info == 0
    out = v.copy()
    vp = ctypes.c_void_p
    rc = L.enlsipb200_dense_vecop(kind, frows, k, np.asfortranarray(qr).ctypes.data_as(vp), None, out.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    # forward error of a triangular solve scales with the condition number: compare residuals and a cond-scaled difference
    cond = np.linalg.cond(R)
    assert np.abs(out - ref[:, 0]).max() <= 1e-13 * cond * np.abs(ref).max()
    res = (R @ out - v) if kind == 2 else (R.T @ out - v)
    assert np.abs(res).max() <= 1e-12 * (np.abs(R).max() * np.abs(out).max() * k ** 0.5 + np.abs(v).max())


@pytest.mark.parametrize("env", [{"ENLSIP_QR_PANEL": "graph"}])
def test_qrcp_alternative_paths_vs_dgeqp3(env):
    """The graph form of the blocked QRCP stays correct: three kernels per column inside a CUDA graph (the path of
    matrices with more than 32768 rows).  The switch is read once per process, so the factorisation runs in a child
    process (tools/qrcp_time.py compares pivots, R and tau with LAPACK)."""
    import os
    import re
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "tools", "qrcp_time.py"), "700", "450", "1"], env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-1500:] + p.stderr[-1500:]
    m = re.search(r"pivots identical (\d+) / (\d+)\s+max \|R - R_lapack\| / max\|R\| = (\S+)\s+max \|tau diff\| = (\S+)", p.stdout)
    assert m, p.stdout[-1500:]
    assert m.group(1) == m.group(2) == "450" and float(m.group(3)) <= 1e-12 and float(m.group(4)) <= 1e-12
