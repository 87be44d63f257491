"""Host-side mirror of the reference's model API for the LARGE-JACOBIAN regime (one problem, m >> n).

reference                                   here
---------                                   ----
CnlsModel(residuals, n, m; starting_point,  LargeCnlsModel("single_index", starting_point[n], data={"W","y","rho"},
          eq_constraints, nb_eqcons, ...)                  ineq=False, x_low, x_upp, m_global=None)
   (cnls_model.jl:345-378)                     the rows of W / y held by THIS process (a row shard when m_global > rows)
solve!(model; ...)     (solver.jl:62-91)    solve(model, ...)   (same function as the batched regime: it dispatches)
status / solution / sum_sq_residuals        same accessors (cnls_model.jl:206-221), B = 1

Row sharding over the GPUs of one box (BASELINE.json config 4): one process per GPU, each builds a model
from its own rows and calls ``model.join(rank, world)`` once (NCCL unique id broadcast through
``torch.distributed``); afterwards every rank calls ``solve`` with identical arguments and gets identical results.
Row families (chained Rosenbrock, LargeUserFamily) compress [J | r] by a plain Householder QR of the column-major matrix
unless ``factor="tsqr"``: then they take the single-index family's tall-skinny QR, and ``shard=(rank, world)`` gives this
process its slice of the rows (``shard_rows``) before ``join(rank, world)``.  Data slots stay whole on every rank.
A row family with n + m < 1000 is solved as the reference solves it at that size, with Newton steps (second derivatives
on, EF:2658; the handle is created with LARGE_MIDSIZE); such a problem is not factored by the TSQR nor sharded.
There is no CPU execution path.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import capi


def _is_torch(a):
    return type(a).__module__.startswith("torch")


# general "row families" (csrc/enl_large_family.h): name -> (family id, m(n), nb_eq(n), nb_ineq(n), data slots)
_ROW_FAMILIES = {
    "chained_rosenbrock": (capi.FAMILY_LARGE_CHAINED_ROSENBROCK, lambda n: 2 * (n - 1), lambda n: n - 2, lambda n: 0, ()),
}


SHARD_ALIGN = 256       # rows of one level-0 subtile of the TSQR tree (8 blocks of 32)


def shard_rows(m, rank, world):
    """(row0, rows) of `rank` among `world` shards of m rows: equal slices in multiples of SHARD_ALIGN, the last rank
    takes the remainder (ranks past the end of a small problem hold no rows)."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("shard must be (rank, world) with 0 <= rank < world")
    chunk = max(SHARD_ALIGN, (m // world) // SHARD_ALIGN * SHARD_ALIGN)
    row0 = min(rank * chunk, m)
    rows = m - row0 if rank == world - 1 else min(chunk, m - row0)
    return row0, rows


class LargeUserFamily:
    """A problem of the large regime defined by user CUDA source: the replacement of the reference's closure arguments
    (residuals, eq_constraints, ineq_constraints, jacobian_*; cnls_model.jl:345-359) for one problem with
    n + m >= 1000, or a smaller one (m >= n + 1) solved with Newton steps as the reference solves it.  `source` defines
    enl_user::residual / constraint as templates over a point accessor and, with has_jacobians, jac_residual /
    jac_constraint (include/enlsip_b200.h, enlsipb200_large_compile_family).  `data`: names of up to two data arrays."""

    def __init__(self, source, m, nb_eqcons=0, nb_ineqcons=0, has_jacobians=False, data=(), name="large_user"):
        self.source, self.m, self.q, self.ni = source, int(m), int(nb_eqcons), int(nb_ineqcons)
        self.has_jacobians, self.data, self.name = bool(has_jacobians), tuple(data), name
        if len(self.data) > 2:
            raise ValueError("at most two data slots")

    def library(self):
        return capi.large_compile_family(self.source, self.m, self.q, self.ni, self.has_jacobians, self.name)


class LargeCnlsModel:
    def __init__(self, family, starting_point, data=None, ineq=False, x_low=None, x_upp=None, m_global=None, device=-1,
                 jacobian="analytic", factor="householder", shard=None):
        if jacobian not in ("analytic", "forward_diff"):
            raise AssertionError("jacobian must be 'analytic' or 'forward_diff'")
        if factor not in ("householder", "tsqr"):
            raise AssertionError("factor must be 'householder' or 'tsqr'")
        if shard is not None and factor != "tsqr":
            raise AssertionError("shard=(rank, world) needs factor='tsqr'")
        self.factor_mode, self.shard = factor, shard
        self._flag = capi.LARGE_FACTOR_TSQR if factor == "tsqr" else 0
        self.jacobian = jacobian
        self.family = family
        self.B = 1
        self.starting_point = np.ascontiguousarray(starting_point, dtype=np.float64).reshape(-1)
        n = self.starting_point.size
        self._keep = {}
        self._lib = capi.lib()
        if isinstance(family, LargeUserFamily):
            self._lib = family.library()
            self.family = family.name
            if jacobian == "analytic" and not family.has_jacobians:
                self.jacobian = "forward_diff"     # no jacobian_* given: the reference differentiates for the user as well
            self._init_row_family(capi.FAMILY_USER, n, family.m, family.q, family.ni, family.data, data or {}, x_low, x_upp, device)
            return
        if family in _ROW_FAMILIES:
            fam_id, m_of, q_of, ni_of, keys = _ROW_FAMILIES[family]
            self._init_row_family(fam_id, n, int(m_of(n)), int(q_of(n)), int(ni_of(n)), keys, data or {}, x_low, x_upp, device)
            return
        if family != "single_index":
            raise AssertionError("large-regime families: %s" % (["single_index"] + sorted(_ROW_FAMILIES)))
        W, y = data["W"], data["y"]
        rho = np.ascontiguousarray(data["rho"], dtype=np.float64)
        rows = int(W.shape[0])
        if int(W.shape[1]) != n or int(y.shape[0]) != rows:
            raise ValueError("W must be [rows, n] and y [rows]")
        self.nb_parameters, self.rows = n, rows
        self.nb_residuals = int(rows if m_global is None else m_global)
        self.x_low = np.full(n, -np.inf) if x_low is None else np.ascontiguousarray(x_low, dtype=np.float64)
        self.x_upp = np.full(n, np.inf) if x_upp is None else np.ascontiguousarray(x_upp, dtype=np.float64)
        nb = rho.size
        self.nb_eqcons = 0 if ineq else nb
        self.nb_constraints = nb + int(np.isfinite(self.x_low).sum()) + int(np.isfinite(self.x_upp).sum())
        self.lmax = self.nb_constraints
        h = ctypes.c_void_p()
        capi.check_large(self._lib.enlsipb200_large_create(capi.FAMILY_SINGLE_INDEX | self._flag, n, rows, self.nb_residuals, nb,
                                                            1 if ineq else 0, rho.ctypes.data, self.x_low.ctypes.data,
                                                            self.x_upp.ctypes.data, device, ctypes.byref(h)), self._lib)
        self._h = h
        self.set_data(0, W)
        self.set_data(1, y)
        self._reset_results()

    def _init_row_family(self, fam_id, n, m, q, ni, keys, data, x_low, x_upp, device):
        """A general family: residual rows / constraints as device functions of the point (csrc/enl_large_family.h), the
        counterpart of CnlsModel(residuals, n, m; eq_constraints, nb_eqcons, ...) for an arbitrary model."""
        self.row0, self.rows = (0, m) if self.shard is None else shard_rows(m, *self.shard)
        self.nb_parameters, self.nb_residuals = n, m
        self.x_low = np.full(n, -np.inf) if x_low is None else np.ascontiguousarray(x_low, dtype=np.float64)
        self.x_upp = np.full(n, np.inf) if x_upp is None else np.ascontiguousarray(x_upp, dtype=np.float64)
        self.nb_eqcons = q
        self.nb_constraints = q + ni + int(np.isfinite(self.x_low).sum()) + int(np.isfinite(self.x_upp).sum())
        self.lmax = self.nb_constraints
        # the reference takes Newton steps below this size (second_derivatives = n + m < 1000, EF:2658)
        self.midsize = n + m < 1000
        if self.midsize and (self.factor_mode == "tsqr" or self.shard is not None):
            raise AssertionError("n + m < 1000 (Newton steps): the [J | r] of a mid-size problem is neither factored by the "
                                 "TSQR nor sharded; use factor='householder' without shard")
        flag = self._flag | (capi.LARGE_MIDSIZE if self.midsize else 0)
        h = ctypes.c_void_p()
        capi.check_large(self._lib.enlsipb200_large_create(fam_id | flag, n, self.rows, m, 0, 0, None, self.x_low.ctypes.data,
                                                            self.x_upp.ctypes.data, device, ctypes.byref(h)), self._lib)
        self._h = h
        for slot, key in enumerate(keys):
            self.set_data(slot, data[key])
        self._reset_results()

    def _reset_results(self):
        self.status_code = None
        self.sol = self.starting_point
        self.obj_value = None
        self.exit_code = None
        self.iterations = None
        self.nb_active = None
        self.active = None
        self.trace = None

    def set_data(self, slot, arr):
        """Bind family data: slot 0 = W [rows, n], slot 1 = y [rows].  CUDA torch tensors are used in place
        (zero copy); numpy arrays are copied host -> device by the library (reusing its buffer)."""
        dev = _is_torch(arr) and arr.is_cuda
        if _is_torch(arr):
            if not dev:
                raise ValueError("torch tensors must live on a CUDA device; pass numpy arrays for host buffers")
            arr = arr.contiguous()
            ptr, count = arr.data_ptr(), arr.numel()
        else:
            arr = np.ascontiguousarray(arr, dtype=np.float64)
            ptr, count = arr.ctypes.data, arr.size
        self._keep[slot] = arr if dev else None
        capi.check_large(self._lib.enlsipb200_large_set_data(self._h, slot, ctypes.c_void_p(ptr), count, 1 if dev else 0), self._lib)

    def join(self, rank, world, broadcast=None):
        """Join the row shards of `world` processes (one per GPU).  `broadcast(buf: np.uint8[128])` must
        overwrite buf on every rank with rank 0's content; default: torch.distributed.broadcast."""
        buf = np.zeros(128, dtype=np.uint8)
        if rank == 0 and world > 1:
            capi.check_large(capi.lib().enlsipb200_large_comm_id(buf.ctypes.data))
        if world > 1:
            if broadcast is None:
                import torch
                import torch.distributed as dist
                if dist.get_backend() == "nccl":
                    t = torch.from_numpy(buf).cuda()
                    dist.broadcast(t, 0)
                    buf[:] = t.cpu().numpy()
                else:
                    t = torch.from_numpy(buf)
                    dist.broadcast(t, 0)
            else:
                broadcast(buf)
        capi.check_large(self._lib.enlsipb200_large_comm_init(self._h, buf.ctypes.data, int(rank), int(world)), self._lib)

    def factor(self, x, want_R=True):
        """Measurement / test hook: one evaluation + QR of [J | r] at x.  Returns (R or None, build_ms, tsqr_ms)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = self.nb_parameters
        R = np.zeros((n + 1, n + 1)) if want_R else None
        b, t = ctypes.c_float(), ctypes.c_float()
        capi.check_large(self._lib.enlsipb200_large_factor(self._h, x.ctypes.data, None if R is None else R.ctypes.data,
                                                            ctypes.byref(b), ctypes.byref(t)), self._lib)
        return R, float(b.value), float(t.value)

    def stats(self):
        v = np.zeros(15)
        capi.check_large(self._lib.enlsipb200_large_stats(self._h, v.ctypes.data, 15), self._lib)
        keys = ("points", "build_ms", "tsqr_ms", "linesearch_ms", "solve_wall_ms", "linesearch_evals",
                "launches", "rows_pad", "device_qrcp", "device_mulq", "small_stage_ms", "factorisations", "ws_growths",
                "newton_steps", "hessian_ms")
        return dict(zip(keys, [float(a) for a in v]))

    def launch_count(self):
        return int(self.stats()["launches"])

    def close(self):
        if getattr(self, "_h", None):
            self._lib.enlsipb200_large_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def solve_large(model: LargeCnlsModel, silent=True, max_iter=100, scaling=False, time_limit=1e3, abs_tol=None,
                rel_tol=None, c_tol=None, x_tol=None, trace_cap=0):
    """solve!(model; ...) (solver.jl:62-91) for the large regime; results land in the model (B = 1 arrays)."""
    n = model.nb_parameters
    if not silent and trace_cap == 0:
        trace_cap = int(max_iter) + 1          # the iteration table of print_diagnosis needs the log
    o = capi.default_options()
    o.max_iter = int(max_iter)
    o.scaling = 1 if scaling else 0
    o.jac_mode = capi.JAC_FORWARD_DIFF if model.jacobian == "forward_diff" else capi.JAC_ANALYTIC
    o.time_limit = float(time_limit)
    nan = float("nan")
    o.abs_tol = nan if abs_tol is None else float(abs_tol)
    o.rel_tol = nan if rel_tol is None else float(rel_tol)
    o.c_tol = nan if c_tol is None else float(c_tol)
    o.x_tol = nan if x_tol is None else float(x_tol)
    x = np.zeros((1, n))
    f = np.zeros(1)
    ec, st, it, na = (np.zeros(1, dtype=np.int32) for _ in range(4))
    act = np.zeros((1, max(model.lmax, 1)), dtype=np.int32)
    tr = np.zeros((1, trace_cap, capi.TRACE_HDR + n)) if trace_cap > 0 else None
    p = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
    capi.check_large(model._lib.enlsipb200_large_solve(model._h, p(model.starting_point), ctypes.byref(o), p(x), p(f),
                                                       p(ec), p(st), p(it), p(na), p(act), p(tr), int(trace_cap)), model._lib)
    model.status_code, model.exit_code, model.sol, model.obj_value = st, ec, x, f
    model.iterations, model.nb_active, model.active, model.trace = it, na, act, tr
    if not silent:
        from .model import iteration_table, status
        print("%s problem (n=%d, m=%d, constraints=%d)" % (model.family, n, model.nb_residuals, model.nb_constraints))
        print(iteration_table(model, 0))
        print("Number of iterations...................: %4d" % int(it[0]))
        print("Square sum of residuals................: %.7e" % float(f[0]))
        print("Termination status.....................: %s (exit code %d)" % (status(model)[0], int(ec[0])))
    return None
