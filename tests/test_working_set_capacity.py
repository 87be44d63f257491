"""Working sets larger than n, against the oracle.

init_working_set (EF:826-859) puts every equality and every violated row into the working set, with no bound: a start
outside its bounds on most parameters that also violates some inequalities begins with t > n.  Only the additions of
evaluate_violated_constraints (EF:608-650) stop at min(l, n).

- Large regime: the host driver (enl_large_host.h over the CPU backend) and the device small stage (enl_large.cu, whose
  t-sized buffers are allocated for min(l, n) + 1 rows and grow on demand) against the oracle at t0 around and beyond n.
- Batched regime: the shared-memory layout holds T = min(lmax, n) active rows; a start beyond that ends at once with
  exit code -97, and what such a problem reports is pinned here (host port and device).

Every case asserts, from the oracle's own record, the working-set size it exists for.
"""
import numpy as np
import pytest

from tests.test_hostport import run
from tests.test_large_host import compare_with_oracle, run_large

N = 32


def _below_start(nb, seed, k, m=1200):
    """n = 32, bounds (0, 2): the first k parameters start at -0.5 (one violated bound row each), the others inside."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(m, N, nb, seed=seed, ineq=True)
    x0 = d["x0"].copy()
    x0[:k] = -0.5
    x0[k:] = np.clip(x0[k:], 0.05, 1.9)
    d["x0"] = x0
    return d, (0.0, 2.0)


def _issue_start():
    """x0 = -0.9 everywhere, bounds (0, 2): all 32 lower bounds and all 8 block inequalities violated."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(1200, N, 8, seed=6, ineq=True)
    d["x0"] = np.full(N, -0.9)
    return d, (0.0, 2.0)


def _scaled_start(bound, mult):
    """scaling=True starts: bounds (-bound, bound), x0 = mult * truth (most parameters beyond a bound)."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(1200, N, 8, seed=19, ineq=True)
    d["x0"] = mult * d["truth"]
    return d, (-bound, bound)


def _wide_start(m, n, nb, seed, heavy):
    """bounds (0, 2), every parameter slightly below its lower bound (n violated bound rows); the parameters of the first
    `heavy` blocks far below it, which also violates their inequality rho_k - sum x^2 >= 0: t0 = n + heavy."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(m, n, nb, seed=seed, ineq=True)
    x0 = np.full(n, -0.05)
    x0[:4 * heavy] = -1.9
    d["x0"] = x0
    return d, (0.0, 2.0)


def _oracle(d, bounds, **kw):
    from oracle import enlsip_oracle as O, problems as P
    return O.solve(P.single_index(d["W"], d["y"], d["rho"], d["x0"], ineq=True, bounds=bounds), wallclock=False, **kw)


# (label, start, initial working-set size the case exists for); n = 32, t0 = trace[0].t of the oracle
LARGE_CASES = [
    ("t0=n-1", lambda: _below_start(8, 3, 28), N - 1),
    ("t0=n", lambda: _below_start(4, 3, 30), N),
    ("t0=n+1", lambda: _below_start(4, 3, 31), N + 1),
    ("t0=n+2", lambda: _below_start(8, 6, 31), N + 2),
    ("t0=n+nb", _issue_start, N + 8),
]


@pytest.mark.parametrize("label,start,t0", LARGE_CASES, ids=[c[0] for c in LARGE_CASES])
def test_host_driver_initial_working_set_around_n(label, start, t0):
    d, bounds = start()
    r = _oracle(d, bounds)
    assert r.trace[0].t == t0 and r.iterations <= 30
    out = run_large(d, ineq=True, bounds=bounds, trace_cap=60)
    compare_with_oracle(out, r, N)


def _truth_start(nb, seed, bound, mult):
    """n = 32, unscaled: bounds (-bound, bound), x0 = mult * truth."""
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(1200, N, nb, seed=seed, ineq=True)
    d["x0"] = mult * d["truth"]
    return d, (-bound, bound)


@pytest.mark.parametrize("endless", [False, True], ids=["swaps_then_continues", "swaps_forever"])
def test_host_driver_working_set_fills_to_n_and_swaps(monkeypatch, endless):
    """t0 < n; evaluate_violated_constraints adds rows up to min(l, n) = n and then swaps at capacity.  In the first
    case each swap at capacity exchanges one row and the iteration goes on; in the second the reference swaps forever
    (its endless loop, exit -98), which the driver must reproduce."""
    from oracle import enlsip_oracle as O
    calls = []
    orig = O.evaluate_violated_constraints

    def logged(cx, W, index_alpha_upp, n):
        t_in, removed = W.t, [0]
        remove = W.remove_constraint

        def counted(s):
            removed[0] += 1
            return remove(s)
        W.remove_constraint = counted
        try:
            return orig(cx, W, index_alpha_upp, n)
        finally:
            del W.remove_constraint
            calls.append((t_in, W.t, removed[0]))
    monkeypatch.setattr(O, "evaluate_violated_constraints", logged)
    d, bounds = _below_start(8, 6, 28) if endless else _truth_start(4, 10, 0.7, 3.0)
    r = _oracle(d, bounds)
    assert r.trace[0].t < N and any(t_in < N and t_out == N for t_in, t_out, _ in calls)
    at_cap = [k for k, (t_in, _, removed) in enumerate(calls) if t_in == N and removed > 0]
    assert at_cap
    if endless:
        assert r.exit_code == -98
    else:
        assert r.exit_code != -98 and all(calls[k][2] == 1 for k in at_cap) and at_cap[0] < len(calls) - 1
    out = run_large(d, ineq=True, bounds=bounds, trace_cap=60)
    compare_with_oracle(out, r, N)


def test_host_driver_scaled_start_beyond_n():
    """scaling=True with t > n: every row of C.A has norm 1 up to an ulp, so the pivot order of qr(C.A', ColumnNorm())
    is decided by how dgeqp3's column norms round; the subspace step (method -1, dimA < rankA) depends on it."""
    d, bounds = _scaled_start(0.4, 1.5)
    r = _oracle(d, bounds, scaling=True)
    assert r.trace[0].t > N
    assert any(t.code == -1 and t.dimA < t.rankA for t in r.trace)      # the step that exposed the pivot order
    out = run_large(d, ineq=True, bounds=bounds, trace_cap=60, scaling=True)
    compare_with_oracle(out, r, N)


def _oracle_ulp_ensemble(d, bounds, seeds):
    """The oracle with the last bit of about half of the entries of every qr(C.A') input with t > n flipped at random
    (one generator per seed): solves the reference could equally give, since C.A is only defined to an ulp."""
    from oracle import enlsip_oracle as O
    n = d["x0"].size
    orig = O.QRPivoted.__init__
    for seed in seeds:
        rng = np.random.default_rng(seed)

        def perturbed(self, M):
            M = np.array(M, dtype=float, order="F")
            if M.shape[0] == n and M.shape[1] > n:
                flip = rng.random(M.shape) < 0.5
                M[flip] = np.nextafter(M[flip], np.where(rng.random(int(flip.sum())) < 0.5, np.inf, -np.inf))
            orig(self, M)
        O.QRPivoted.__init__ = perturbed
        try:
            r = _oracle(d, bounds, scaling=True)
        finally:
            O.QRPivoted.__init__ = orig
        yield seed, r


def test_host_driver_scaled_start_beyond_n_ulp_tie():
    """The second scaled start sits on ulp ties: the reference's own result changes when the last bits of C.A' change
    (dgeqp3 then picks other pivots for every one of 8 perturbations, and the solves differ by up to 64 % in f).  The
    driver must give one of those solves, to the full bars of compare_with_oracle."""
    from scipy.linalg import lapack
    d, bounds = _scaled_start(0.3, 2.0)
    r0 = _oracle(d, bounds, scaling=True)
    assert r0.trace[0].t > N + 1
    assert any(t.code == -1 and t.dimA < t.rankA for t in r0.trace)
    out = run_large(d, ineq=True, bounds=bounds, trace_cap=60, scaling=True)
    outcomes, matched = set(), None
    for seed, r in _oracle_ulp_ensemble(d, bounds, range(64)):
        outcomes.add((r.exit_code, r.iterations, round(r.f, 6)))
        try:
            compare_with_oracle(out, r, N)
        except AssertionError:
            continue
        matched = seed
        break
    assert matched is not None, outcomes
    # the tie itself: the first qr(C.A') of the unperturbed solve changes its pivot order under one-ulp perturbations
    from oracle import enlsip_oracle as O
    first = []
    orig = O.QRPivoted.__init__

    def record(self, M):
        if not first and np.shape(M)[0] == N and np.shape(M)[1] > N:
            first.append(np.array(M, dtype=float, order="F"))
        orig(self, M)
    O.QRPivoted.__init__ = record
    try:
        _oracle(d, bounds, scaling=True, max_iter=1)
    finally:
        O.QRPivoted.__init__ = orig
    M = first[0]
    p0 = lapack.dgeqp3(M.copy(order="F"))[1]
    rng = np.random.default_rng(0)
    flips = 0
    for _ in range(8):
        Mp = M.copy(order="F")
        f = rng.random(M.shape) < 0.5
        Mp[f] = np.nextafter(Mp[f], np.where(rng.random(int(f.sum())) < 0.5, np.inf, -np.inf))
        flips += not np.array_equal(lapack.dgeqp3(Mp)[1], p0)
    assert flips == 8


# ---- batched regime: exit -97 ------------------------------------------------------------------------------------
HS65_CAP = np.array([-5.0, 5.0, 6.0])      # violates constraints 1, 2, 6 and 7: t0 = 4 > T = min(7, 3)


def _hs65_capacity_facts():
    """(initial working set, f at x0) of HS65_CAP from the oracle problem; the oracle itself starts there (t0 = 4)."""
    from oracle import enlsip_oracle as O, problems as P
    pb = P.hs65(HS65_CAP.copy())
    c = np.asarray(pb.cons(HS65_CAP))                  # the inequality, then the lower and upper bound rows
    active = [i + 1 for i in range(c.size) if c[i] <= 0.0]
    o = O.solve(P.hs65(HS65_CAP.copy()), wallclock=False)
    assert o.trace[0].t == len(active) == 4 > 3 and list(o.trace[0].active) == active
    r = np.asarray(pb.res(HS65_CAP))
    return active, float(np.dot(r, r))


def check_capacity_exit(out, b, active, f0):
    assert (int(out["exit_code"][b]), int(out["status"][b]), int(out["iters"][b])) == (-97, -1, 0)
    assert np.array_equal(out["x"][b].view(np.uint64), HS65_CAP.view(np.uint64))
    assert abs(out["f"][b] - f0) <= 1e-15 * f0
    assert int(out["nact"][b]) == len(active) and list(out["active"][b][:len(active)]) == active
    assert not np.any(out["active"][b][len(active):])
    assert list(out["counters"][b]) == [2, 2]          # the one evaluation of r, c (and J, A) at x0


def test_capacity_exit_hostport_single():
    import enlsip_jl_b200 as E
    active, f0 = _hs65_capacity_facts()
    out = run(0, HS65_CAP[None, :].copy(), None, None, E.synth.HS65_LOW, E.synth.HS65_UPP, 0)
    check_capacity_exit(out, 0, active, f0)


def test_capacity_exit_hostport_between_neighbours():
    """A -97 problem between two normal ones: the neighbours give the bits they give when solved alone."""
    import enlsip_jl_b200 as E
    active, f0 = _hs65_capacity_facts()
    normal = E.synth.gen_hs65_batch(2)
    x0 = np.vstack([normal[0], HS65_CAP, normal[1]])
    out = run(0, x0, None, None, E.synth.HS65_LOW, E.synth.HS65_UPP, 0, nthreads=1)
    check_capacity_exit(out, 1, active, f0)
    for b, k in ((0, 0), (2, 1)):
        alone = run(0, normal[k:k + 1].copy(), None, None, E.synth.HS65_LOW, E.synth.HS65_UPP, 0, nthreads=1)
        assert int(alone["exit_code"][0]) > 0
        for key in ("x", "f", "exit_code", "status", "iters", "nact", "active", "counters", "trace"):
            assert np.array_equal(np.asarray(out[key][b]), np.asarray(alone[key][0])), (b, key)


# ---- the same on the device (B200) -------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def E():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import enlsip_jl_b200 as E
    E.capi.lib()
    return E


def _device_solve(E, d, bounds, n):
    lo, up = np.full(n, bounds[0]), np.full(n, bounds[1])
    mod = E.LargeCnlsModel("single_index", d["x0"], d, ineq=True, x_low=lo, x_upp=up)
    E.solve(mod, trace_cap=60)
    out = dict(x=mod.sol[0].copy(), f=np.array(mod.obj_value, copy=True), exit_code=np.array(mod.exit_code, copy=True),
               status=np.array(mod.status_code, copy=True), iters=np.array(mod.iterations, copy=True),
               nact=np.array(mod.nb_active, copy=True), active=mod.active[0].copy(), trace=mod.trace[0].copy())
    return mod, out


DEVICE_CASES = LARGE_CASES + [
    ("n=256,t0=n+16", lambda: _wide_start(3000, 256, 64, 3, 16), 256 + 16),
    ("n=512,t0=n+33", lambda: _wide_start(4096, 512, 128, 31, 33), 512 + 33),
]


@pytest.mark.gpu
@pytest.mark.parametrize("label,start,t0", DEVICE_CASES, ids=[c[0] for c in DEVICE_CASES])
def test_device_small_stage_initial_working_set_around_n(E, label, start, t0):
    """The device small stage at t0 up to n + 33: C.A (t x n), qr(C.A') (n x t, wide: t crosses a 32-column panel past
    n + 1 at n = 512) and qr(R_A') (t x n) in buffers that grow past min(l, n) + 1 rows."""
    d, bounds = start()
    n = d["x0"].size
    r = _oracle(d, bounds)
    assert r.trace[0].t == t0
    mod, out = _device_solve(E, d, bounds, n)
    st = mod.stats()
    assert st["device_qrcp"] > 0
    assert (st["ws_growths"] > 0) == (t0 > n + 1)
    compare_with_oracle(out, r, n)
    E.solve(mod, trace_cap=60)                     # a second solve on the grown buffers: the same bits
    assert np.array_equal(mod.sol[0].view(np.uint64), out["x"].view(np.uint64))
    assert np.array_equal(mod.trace[0], out["trace"]) and int(mod.iterations[0]) == int(out["iters"][0])
    assert mod.stats()["ws_growths"] == st["ws_growths"]
    mod.close()


def _slots(m):
    ki = m.kernel_info()
    return ki["threads_per_cta"] // ki["lanes_per_problem"], ki["grid"]


@pytest.mark.gpu
def test_device_capacity_exit_solve_and_step_batch(E):
    """solve_batch and step_batch with -97 problems placed first in the batch (the first problem a slot takes) and
    behind as many normal problems as there are slots (a slot that has served a normal problem before).  solve_batch
    reports what the host port reports; step_batch gives p = 0, lam = 0 and the whole initial working set; the normal
    problems give the bits they give in a batch without the -97 problems."""
    import torch
    active, f0 = _hs65_capacity_facts()
    probe = E.CnlsModel("hs65", E.synth.gen_hs65_batch(1), x_low=E.synth.HS65_LOW, x_upp=E.synth.HS65_UPP)
    ppc, grid = _slots(probe)
    probe.close()
    B = 2 * ppc * grid + 3
    x0 = E.synth.gen_hs65_batch(B)
    cap = [0, ppc * grid + 1, B - 1]
    xc = x0.copy()
    xc[cap] = HS65_CAP
    host = run(0, xc[cap], None, None, E.synth.HS65_LOW, E.synth.HS65_UPP, 0, trace_cap=1)
    for i in range(len(cap)):
        check_capacity_exit(host, i, active, f0)
    res = {}
    for name, xs in (("cap", xc), ("ref", x0)):
        m = E.CnlsModel("hs65", torch.from_numpy(xs).cuda(), x_low=E.synth.HS65_LOW, x_upp=E.synth.HS65_UPP)
        E.solve(m)
        sol = {k: getattr(m, a).cpu().numpy() for k, a in (("x", "sol"), ("f", "obj_value"), ("exit_code", "exit_code"),
                                                          ("status", "status_code"), ("iters", "iterations"),
                                                          ("nact", "nb_active"), ("active", "active"), ("counters", "counters"))}
        xd = torch.from_numpy(xs).cuda()
        st = {k: v.cpu().numpy() for k, v in E.gn_step(m, xd, E.evaluate(m, xd)).items()}
        res[name] = (sol, st)
        m.close()
    sol, st = res["cap"]
    sol_ref, st_ref = res["ref"]
    for i, b in enumerate(cap):
        check_capacity_exit(sol, b, active, f0)
        for key in ("x", "f", "nact", "active", "counters"):
            assert np.array_equal(sol[key][b], host[key][i]), (b, key)
        assert list(st["info"][b]) == [len(active), 0, 0, 0, -97], b
        assert not np.any(st["p"][b]) and not np.any(st["lam"][b]), b
        assert list(st["active"][b][:len(active)]) == active and not np.any(st["active"][b][len(active):])
    keep = np.setdiff1d(np.arange(B), cap)
    for key in sol:
        assert np.array_equal(sol[key][keep], sol_ref[key][keep]), key
    for key in st:
        assert np.array_equal(st[key][keep], st_ref[key][keep]), key
    assert np.all(st["info"][keep, 4] == 0)
