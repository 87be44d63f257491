"""Known-answer tests of the small stage's kernels at every size where the engine switches kernels, through the hooks
enlsipb200_dense_qrcp / _qr / _vecop / _gemv, which run the engine's own dispatch (csrc/enl_small.cuh):

- QR with column pivoting vs LAPACK dgeqp3 and the plain Householder QR (the [J | r] compression of the general
  large-regime families) vs dgeqrf: thread-block clusters of 2, 4 and 8 CTAs, the unblocked dlaqp2 column loop with its
  reflector staged in shared memory or read from global memory, blocked dlaqps panels (persistent kernel up to 32768
  rows, three kernels per column in a CUDA graph above that) with the dlaqp2 tail, and wide matrices;
- Q' v, Q v vs dormqr and R \\ v, R' \\ v vs dtrtrs: one-warp, cooperative multi-CTA and one-CTA kernels;
- y = alpha A x + beta y0 and y = A' x vs sums in long double.

Where rounding order matters the bound comes from the floating-point error analysis of the same operation, so that a
skipped, doubled or misplaced term fails and a different order of the same additions does not.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.linalg import lapack

gpu = pytest.mark.gpu
EPS = np.finfo(float).eps
vp = ctypes.c_void_p
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import enlsip_jl_b200 as E
    return E.capi.lib()


# ---- the kernel selection of qrcp_device (csrc/enl_small.cuh), restated ----
QC_MAX_SMEM, QC_THREADS, QC_MAXCTAS = 200 * 1024, 512, 8
QR_NB, QR_NX = 32, 128
QP_MAXSLICES, QP_MINRW, QP_MAXRW = 64, 128, 512
VEC_STAGE_MAX = 6144          # doubles of shared memory a kernel gets without an opt-in (48 KB)


def qc_smem_bytes(rows, cols, nctas):
    ncl = -(-cols // nctas)
    return 8 * (ncl * rows + rows + 2 + 2 * ncl + QC_MAXCTAS) + 4 * (ncl + cols + 2 * QC_MAXCTAS + 2)


def qr_paths(rows, cols):
    """The kernels qrcp_device runs for a rows x cols matrix (on a B200: cooperative launch, 148 SMs)."""
    for c in (2, 4, 8):
        if qc_smem_bytes(rows, cols, c) <= QC_MAX_SMEM and -(-cols // c) <= QC_THREADS // 32:
            return {"cluster%d" % c}
    if qc_smem_bytes(rows, cols, 8) <= QC_MAX_SMEM:
        return {"cluster8"}
    minmn = min(rows, cols)
    topbmn = minmn - QR_NX if (QR_NB < minmn and QR_NX < minmn) else 0
    paths = set()
    if topbmn > 0:
        rw = max(-(-rows // QP_MAXSLICES), QP_MINRW)
        paths.add("blocked_persist" if rw <= QP_MAXRW else "blocked_graph")
    for i in range(topbmn, min(minmn, cols - 1)):          # qr_p2_apply_kernel, reflector of rows - i - 1 entries
        paths.add("p2_staged" if rows - i - 1 <= VEC_STAGE_MAX else "p2_global")
    return paths


QR_SHAPES = [(300, 20), (500, 60), (257, 192),           # clusters of 2, 4, 8 CTAs
             (12000, 5), (12800, 5),                     # the last that fits 200 KB of shared memory / the first that does not
             (6144, 64), (6146, 64), (20000, 64),        # dlaqp2 only: reflectors of 6143 / 6145 / 19999 entries
             (1000, 600), (7000, 200), (8000, 1000),     # blocked panels + a dlaqp2 tail with short / long reflectors
             (40000, 160),                               # more than 32768 rows: the panels in a CUDA graph
             (100, 3000)]                                # wide
QR_PLAIN_SHAPES = QR_SHAPES + [(50000, 5), (1998, 1001)]   # + the [J | r] of the user family at m = 50 000, chained Rosenbrock n = 1000


def test_qr_shapes_reach_every_path():
    """The shape lists exercise every kernel qrcp_device can pick; a change of the selection rule that leaves one
    unexercised fails here (update qr_paths() together with qrcp_device)."""
    want = {"cluster2", "cluster4", "cluster8", "p2_staged", "p2_global", "blocked_persist", "blocked_graph"}
    got = set().union(*(qr_paths(r, c) for r, c in QR_SHAPES))
    assert got == want, want ^ got
    assert qr_paths(12000, 5) == {"cluster8"} and qr_paths(12800, 5) == {"p2_global"}
    assert qr_paths(6144, 64) == {"p2_staged"} and "p2_global" in qr_paths(6146, 64)
    assert qr_paths(1200, 5) == {"cluster2"} and qr_paths(50000, 5) == {"p2_global"}    # the user family's [J | r]
    assert qr_paths(8000, 1000) == {"blocked_persist", "p2_global"} and qr_paths(40000, 160) == {"blocked_graph", "p2_global"}


def rand_matrix(rows, cols):
    return np.random.default_rng(rows * 7919 + cols).standard_normal((rows, cols))


def dev_qrcp(L, A):
    f = np.asfortranarray(A, dtype=float).copy(order="F")
    tau = np.zeros(min(A.shape)); jp = np.zeros(A.shape[1], np.int32)
    rc = L.enlsipb200_dense_qrcp(A.shape[0], A.shape[1], f.ctypes.data_as(vp), tau.ctypes.data_as(vp), jp.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    return f, tau, jp


def dev_qr(L, A):
    f = np.asfortranarray(A, dtype=float).copy(order="F")
    tau = np.zeros(min(A.shape))
    rc = L.enlsipb200_dense_qr(A.shape[0], A.shape[1], f.ctypes.data_as(vp), tau.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    return f, tau


def check_qrcp_vs_dgeqp3(A, f, tau, jp):
    """The pattern of test_gpu_kat.test_qrcp_blocked_vs_dgeqp3: a valid factorisation whatever the pivots, then
    LAPACK's pivots, R and tau (continuous random inputs: no two candidate norms agree to rounding)."""
    rows, cols = A.shape
    k = min(rows, cols)
    qr, jl, tl, _, info = lapack.dgeqp3(np.asfortranarray(A))
    assert info == 0
    jl = jl - 1
    assert sorted(jp.tolist()) == list(range(cols))
    R = np.triu(f)[:k]
    AP = A[:, jp]
    G = AP.T @ AP
    # R'R = (AP)'(AP): Householder QR is backward stable, error of a few eps sqrt(rows) relative to the largest entry
    assert np.abs(R.T @ R - G).max() <= 64 * EPS * np.sqrt(rows) * np.abs(G).max()
    d = np.abs(np.diag(qr)[:k])
    r = int(np.sum(d > 1e-9 * d.max()))
    assert np.array_equal(jp[:r], jl[:r]), ("pivots differ from dgeqp3 at", np.nonzero(jp[:r] != jl[:r])[0][:8])
    Ro, Rlo = np.zeros_like(R), np.zeros_like(R)
    Ro[:, jp] = R
    Rlo[:, jl] = np.triu(qr)[:k]
    assert np.abs(Ro[:r] - Rlo[:r]).max() <= 1e-10 * d.max()
    assert np.abs(tau[:r] - tl[:r]).max() <= 1e-9


def check_qr_vs_dgeqrf(A, f, tau):
    """R itself (dlarfg's sign convention is LAPACK's), the reflectors and tau against dgeqrf, to the forward error
    c kappa eps sqrt(rows) of a backward-stable QR; then Q (dorgqr of the device's reflectors): ||QR - A|| and
    ||Q'Q - I|| at a few eps sqrt(rows)."""
    rows, cols = A.shape
    k = min(rows, cols)
    qr, tl, _, info = lapack.dgeqrf(np.asfortranarray(A))
    assert info == 0
    kappa = np.linalg.cond(np.triu(qr[:k, :k]))      # = cond(A[:, :k])
    tol = 64 * EPS * np.sqrt(rows) * kappa
    colnorm = np.linalg.norm(A, axis=0)
    R, Rl = np.triu(f)[:k], np.triu(qr)[:k]
    assert (np.abs(R - Rl) <= tol * colnorm[None, :]).all(), np.max(np.abs(R - Rl) / colnorm[None, :])
    V, Vl = np.tril(f[:, :k], -1), np.tril(qr[:, :k], -1)       # |v_i| <= 1 (dlarfg scales by 1 / (alpha - beta))
    assert np.abs(V - Vl).max() <= tol, np.abs(V - Vl).max()
    assert np.abs(tau - tl).max() <= tol, np.abs(tau - tl).max()
    Q, _, info = lapack.dorgqr(np.asfortranarray(f[:, :k]), tau)
    assert info == 0
    res = np.linalg.norm(Q @ R - A, axis=0) / np.maximum(colnorm, 1e-300)
    assert res.max() <= 8 * EPS * np.sqrt(rows), res.max() / (EPS * np.sqrt(rows))
    orth = np.abs(Q.T @ Q - np.eye(k)).max()
    assert orth <= 8 * EPS * np.sqrt(rows), orth / (EPS * np.sqrt(rows))


@gpu
@pytest.mark.parametrize("rows,cols", QR_SHAPES)
def test_qrcp_dispatch_vs_dgeqp3(L, rows, cols):
    A = rand_matrix(rows, cols)
    f, tau, jp = dev_qrcp(L, A)
    check_qrcp_vs_dgeqp3(A, f, tau, jp)


@gpu
@pytest.mark.parametrize("rows,cols", QR_PLAIN_SHAPES)
def test_qr_nopivot_vs_dgeqrf(L, rows, cols):
    A = rand_matrix(rows, cols)
    f, tau = dev_qr(L, A)
    check_qr_vs_dgeqrf(A, f, tau)
    f2, tau2 = dev_qr(L, A)
    assert np.array_equal(f, f2) and np.array_equal(tau, tau2), "two runs of the same factorisation differ"


# ---- vector operations: kinds 4-7 of enlsipb200_dense_vecop run the engine's size selection ----
VEC_SIZES = [1, 31, 32, 33, 319, 320, 640, 641, 3000]      # one warp <= 640 < cooperative / one CTA; trsv cooperative from 320


def dgeqrf_factors(frows, k, zero_col=None):
    A = rand_matrix(frows, k)
    if zero_col is not None:
        A[:, zero_col] = 0.0
    qr, tau, _, info = lapack.dgeqrf(np.asfortranarray(A))
    assert info == 0
    return np.asfortranarray(qr), tau


REFLECT_CASES = ([(s, s, None) for s in VEC_SIZES] +                            # k = frows: LAPACK's last tau is 0
                 [(s, (s + 1) // 2, None) for s in VEC_SIZES if s > 1] +
                 [(s, s // 2, s // 4) for s in (33, 320, 640, 641, 3000)])      # a zero column: an interior tau = 0


@gpu
@pytest.mark.parametrize("frows,k,zero_col", REFLECT_CASES)
@pytest.mark.parametrize("kind", [4, 5])
def test_reflect_vec_dispatch_vs_dormqr(L, frows, k, zero_col, kind):
    qr, tau = dgeqrf_factors(frows, k, zero_col)
    if zero_col is not None:
        assert tau[zero_col] == 0.0
    v = np.random.default_rng(frows + k + kind).standard_normal(frows)
    ref, _, info = lapack.dormqr("L", "T" if kind == 4 else "N", qr, tau, np.asfortranarray(v.reshape(-1, 1)), max(1, 64 * frows))
    assert info == 0
    out = v.copy()
    rc = L.enlsipb200_dense_vecop(kind, frows, k, qr.ctypes.data_as(vp), tau.ctypes.data_as(vp), out.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    # k orthogonal reflections: error of order sqrt(k) eps ||v|| (||v|| is preserved)
    assert np.abs(out - ref[:, 0]).max() <= 16 * EPS * np.sqrt(k + 1) * np.linalg.norm(v), np.abs(out - ref[:, 0]).max()


TRSV_CASES = [(k, k) for k in VEC_SIZES] + [(k + 5, k) for k in VEC_SIZES]   # frows > k: leading dimension > k


def check_trsv(L, frows, k, kind):
    qr, _ = dgeqrf_factors(frows, k)
    R = np.triu(qr[:k, :k])
    v = np.random.default_rng(frows + k + kind).standard_normal(k)
    ref, info = lapack.dtrtrs(np.asfortranarray(R), np.asfortranarray(v.reshape(-1, 1)), lower=0, trans=0 if kind % 4 == 2 else 1)
    assert info == 0
    out = v.copy()
    rc = L.enlsipb200_dense_vecop(kind, frows, k, qr.ctypes.data_as(vp), None, out.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    # the bounds of test_gpu_kat.test_trsv_coop_vs_dtrtrs: forward error scaled by cond(R), residual of a backward-stable solve
    cond = np.linalg.cond(R)
    assert np.abs(out - ref[:, 0]).max() <= 1e-13 * cond * np.abs(ref).max(), (frows, k, kind)
    res = (R @ out - v) if kind % 4 == 2 else (R.T @ out - v)
    assert np.abs(res).max() <= 1e-12 * (np.abs(R).max() * np.abs(out).max() * k ** 0.5 + np.abs(v).max()), (frows, k, kind)


@gpu
@pytest.mark.parametrize("frows,k", TRSV_CASES)
@pytest.mark.parametrize("kind", [6, 7])
def test_trsv_dispatch_vs_dtrtrs(L, frows, k, kind):
    check_trsv(L, frows, k, kind)


def run_trsv_cases():
    """Child-process entry of test_trsv_single_block_kernels_vs_dtrtrs."""
    import enlsip_jl_b200 as E
    L = E.capi.lib()
    for frows, k in TRSV_CASES:
        for kind in (6, 7):
            check_trsv(L, frows, k, kind)
    print("trsv cases ok")


@gpu
def test_trsv_single_block_kernels_vs_dtrtrs():
    """With the cooperative kernels switched off (ENLSIP_TRSV_COOP_MIN, read once per process: a child process), the
    one-warp kernels solve every triangle up to 640 and the one-CTA kernels the larger ones."""
    env = dict(os.environ, ENLSIP_TRSV_COOP_MIN=str(2 ** 31 - 1))
    p = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); from tests.test_gpu_dense_dispatch import "
                        "run_trsv_cases; run_trsv_cases()" % ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "trsv cases ok" in p.stdout, p.stdout[-1500:] + p.stderr[-3000:]


# ---- gemv: gemv_n_split_kernel up to 2048 rows, gemv_n_kernel above (x staged up to 6144 columns); gemv_t ----
GEMV_ROWS = [1, 31, 2048, 2049, 9000]
GEMV_COLS = [1, 3, 4, 5, 6144, 6145, 8191]
# 9000 rows with thousands of columns (0.5 GB per matrix) add nothing: 2049 rows already run gemv_n_kernel on 9 CTAs
GEMV_SHAPES = [(r, c) for r in GEMV_ROWS for c in GEMV_COLS if r * c <= 1 << 25]
GEMV_SCALING = {"plain": (1.0, 0.0, False), "axpby": (-0.75, 2.5, True), "beta_without_y0": (1.5, 3.0, False)}


def gemv_bound_check(y, A, x, alpha, y0, beta):
    """|y - y_ref| <= 2 (n + 2) eps (|alpha| sum|A||x| + |beta y0|) entry by entry, y_ref in long double: the dot
    product bound gamma_n, plus one rounding each for the scaling by alpha, the product beta y0 and the final sum (n =
    terms of the dot product), doubled.  A skipped or doubled term is off by |A_rc x_c|, far above the bound."""
    Al, xl = A.astype(np.longdouble), x.astype(np.longdouble)
    ref = np.longdouble(alpha) * (Al @ xl)
    mag = abs(alpha) * (np.abs(Al) @ np.abs(xl))
    if y0 is not None:
        ref = ref + np.longdouble(beta) * y0.astype(np.longdouble)
        mag = mag + np.abs(np.longdouble(beta) * y0.astype(np.longdouble))
    n = A.shape[1]
    err = np.abs(y.astype(np.longdouble) - ref)
    bound = 2 * (n + 2) * np.longdouble(EPS) * mag
    bad = np.nonzero(err > bound)[0]
    assert bad.size == 0, ("entries off", bad[:8], float(err[bad[0]]), float(bound[bad[0]]))


@gpu
@pytest.mark.parametrize("rows,cols", GEMV_SHAPES)
@pytest.mark.parametrize("trans,scaling", [(0, "plain"), (0, "axpby"), (0, "beta_without_y0"), (1, "plain")])
def test_gemv_vs_longdouble(L, rows, cols, trans, scaling):
    alpha, beta, with_y0 = GEMV_SCALING[scaling]
    rng = np.random.default_rng(rows * 31 + cols + 7 * trans)
    lda = rows + 3
    Ab = np.asfortranarray(rng.standard_normal((lda, cols)))        # the rows past `rows` must not be read
    A = Ab[:rows]
    x = rng.standard_normal(rows if trans else cols)
    y0 = rng.standard_normal(rows) if with_y0 else None
    y = np.full(cols if trans else rows, np.nan)
    rc = L.enlsipb200_dense_gemv(trans, rows, cols, Ab.ctypes.data_as(vp), lda, x.ctypes.data_as(vp), alpha,
                                 y0.ctypes.data_as(vp) if y0 is not None else None, beta, y.ctypes.data_as(vp), -1)
    assert rc == 0, L.enlsipb200_large_last_error()
    if trans:
        gemv_bound_check(y, np.ascontiguousarray(A.T), x, 1.0, None, 0.0)
    else:
        gemv_bound_check(y, A, x, alpha, y0, beta)
