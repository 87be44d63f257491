"""ctypes binding of include/enlsip_b200.h (the same symbols the Julia host file binds with ccall)."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libenlsip_b200.so")
SRC = os.path.join(_HERE, "csrc", "enlsip_b200.cu")
HEADERS = [os.path.join(_HERE, "csrc", f) for f in ("enl_base.h", "enl_linalg.h", "enl_families.h", "enl_solver.h",
                                                    "enl_user_family.h")] + \
          [os.path.join(os.path.dirname(_HERE), "include", "enlsip_b200.h")]
# second translation unit: the large-Jacobian regime (TSQR + host-driven iteration)
SRC_LARGE = os.path.join(_HERE, "csrc", "enl_large.cu")
HEADERS_LARGE = [os.path.join(_HERE, "csrc", f) for f in ("enl_base.h", "enl_tsqr.cuh", "enl_small.cuh", "enl_large_host.h",
                                                          "enl_large_family.h", "enl_large_generic.cuh")] + \
                [os.path.join(os.path.dirname(_HERE), "include", "enlsip_b200.h")]
OBJ_DIR = os.path.join(_HERE, "lib", "obj")
FAMILY_SINGLE_INDEX = 16
FAMILY_LARGE_CHAINED_ROSENBROCK = 17
LARGE_FACTOR_TSQR = 0x100   # OR-ed into the family: row families factor [J | r] with the TSQR and may be row-sharded

FAMILY_HS65 = 0
FAMILY_GAUSS_PEAKS = 1
FAMILY_OSBORNE2 = 2
FAMILY_CHAINED_ROSENBROCK10 = 3
FAMILY_CHAINED_WOOD20 = 4
FAMILY_USER = 64          # run-time compiled family: lives in the library written by compile_family()
JAC_ANALYTIC = 0
JAC_FORWARD_DIFF = 1
TRACE_HDR = 16
EXIT_WOULD_THROW, EXIT_WOULD_HANG, EXIT_CAPACITY = -99, -98, -97

EXPORTS = ["enlsipb200_version", "enlsipb200_last_error", "enlsipb200_default_options", "enlsipb200_create",
           "enlsipb200_destroy", "enlsipb200_dims", "enlsipb200_set_data", "enlsipb200_solve_batch", "enlsipb200_eval_batch", "enlsipb200_step_batch",
           "enlsipb200_last_kernel_ms", "enlsipb200_kernel_info", "enlsipb200_launch_count", "enlsipb200_det_exp",
           "enlsipb200_compile_family", "enlsipb200_large_compile_family",
           "enlsipb200_large_last_error", "enlsipb200_large_create", "enlsipb200_large_destroy",
           "enlsipb200_large_set_data", "enlsipb200_large_comm_id", "enlsipb200_large_comm_init",
           "enlsipb200_large_solve", "enlsipb200_large_factor", "enlsipb200_large_stats",
           "enlsipb200_dense_qrcp", "enlsipb200_dense_qr", "enlsipb200_dense_mulq", "enlsipb200_dense_vecop",
           "enlsipb200_dense_gemv", "enlsipb200_dense_last_ms"]


class Options(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("scaling", ctypes.c_int), ("jac_mode", ctypes.c_int),
                ("reserved", ctypes.c_int), ("time_limit", ctypes.c_double), ("abs_tol", ctypes.c_double),
                ("rel_tol", ctypes.c_double), ("c_tol", ctypes.c_double), ("x_tol", ctypes.c_double)]


NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fopenmp", "-Xcompiler", "-fvisibility=hidden"]


def build(force=False, verbose=False):
    """Compile csrc/enlsip_b200.cu and csrc/enl_large.cu for sm_100a into lib/libenlsip_b200.so (in-tree).

    Each translation unit is compiled to lib/obj/*.o only when one of its sources is newer, then linked."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs, relink = [], force or not os.path.exists(LIB_PATH)
    # the batched kernel is bound by instruction fetch (DESIGN.md 5.1): its translation unit is built for small code
    # the large regime's host driver (enl_large_host.h) runs its O(n^2 k) loops on the host: AVX2 for them (every B200
    # host has it); no -mfma, so that the host arithmetic stays un-contracted like the CPU test backend's
    for src, hdrs, extra in ((SRC, HEADERS, ["-DENL_COMPACT_CODE=1"]),
                             (SRC_LARGE, HEADERS_LARGE, ["-Xcompiler", "-mavx2"])):
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        newest = max(os.path.getmtime(p) for p in [src] + hdrs)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            cmd = ["nvcc"] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            subprocess.check_call(cmd)
            relink = True
        objs.append(obj)
    if relink or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(o) for o in objs):
        subprocess.check_call(["nvcc", "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs +
                              ["-o", LIB_PATH, "-Xcompiler", "-fopenmp", "-lgomp", "-ldl"])
    return LIB_PATH


_lib = None


def _bind(L, large=True):
    """Attach the prototypes of include/enlsip_b200.h to a loaded library."""
    vp, ip, dp = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)
    ll, ci, cs = ctypes.c_longlong, ctypes.c_int, ctypes.c_char_p
    L.enlsipb200_version.restype = ctypes.c_int
    L.enlsipb200_last_error.restype = ctypes.c_char_p
    L.enlsipb200_default_options.argtypes = [ctypes.POINTER(Options)]
    L.enlsipb200_default_options.restype = None
    L.enlsipb200_create.argtypes = [ctypes.c_int, vp, vp, ctypes.c_int, ctypes.POINTER(vp)]
    L.enlsipb200_destroy.argtypes = [vp]
    L.enlsipb200_dims.argtypes = [vp, ip, ip, ip, ip, ip]
    L.enlsipb200_set_data.argtypes = [vp, ctypes.c_int, vp, ctypes.c_longlong, ctypes.c_int, vp]
    L.enlsipb200_solve_batch.argtypes = [vp, ctypes.c_longlong, vp, ctypes.POINTER(Options)] + [vp] * 9 + \
                                        [ctypes.c_int, ctypes.c_int, vp]
    L.enlsipb200_eval_batch.argtypes = [vp, ctypes.c_longlong, vp, ctypes.POINTER(Options)] + [vp] * 4 + [ctypes.c_int, vp]
    L.enlsipb200_step_batch.argtypes = [vp, ctypes.c_longlong] + [vp] * 5 + [ctypes.POINTER(Options)] + [vp] * 4 + [ctypes.c_int, vp]
    L.enlsipb200_last_kernel_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
    L.enlsipb200_kernel_info.argtypes = [vp, ip, ip, ip, ip, ip, ip]
    L.enlsipb200_launch_count.argtypes = [vp]
    L.enlsipb200_launch_count.restype = ctypes.c_longlong
    L.enlsipb200_det_exp.argtypes = [vp, vp, ctypes.c_longlong, ctypes.c_int]
    L.enlsipb200_compile_family.argtypes = [cs, ci, ci, ci, ci, ci, ci, ci, cs, cs]
    if hasattr(L, "enlsipb200_large_compile_family"):
        L.enlsipb200_large_compile_family.argtypes = [cs, ll, ci, ci, ci, cs, cs]
    if large:
        L.enlsipb200_large_last_error.restype = ctypes.c_char_p
        L.enlsipb200_large_create.argtypes = [ci, ci, ll, ll, ci, ci, vp, vp, vp, ci, ctypes.POINTER(vp)]
        L.enlsipb200_large_destroy.argtypes = [vp]
        L.enlsipb200_large_set_data.argtypes = [vp, ci, vp, ll, ci]
        L.enlsipb200_large_comm_id.argtypes = [vp]
        L.enlsipb200_large_comm_init.argtypes = [vp, vp, ci, ci]
        L.enlsipb200_large_solve.argtypes = [vp, vp, ctypes.POINTER(Options)] + [vp] * 8 + [ci]
        L.enlsipb200_large_factor.argtypes = [vp, vp, vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
        L.enlsipb200_large_stats.argtypes = [vp, vp, ci]
        L.enlsipb200_dense_qrcp.argtypes = [ci, ci, vp, vp, vp, ci]
        L.enlsipb200_dense_qr.argtypes = [ci, ci, vp, vp, ci]
        L.enlsipb200_dense_mulq.argtypes = [ci, ci, ci, vp, vp, vp, ci]
        L.enlsipb200_dense_vecop.argtypes = [ci, ci, ci, vp, vp, vp, ci]
        L.enlsipb200_dense_gemv.argtypes = [ci, ci, ci, vp, ci, vp, ctypes.c_double, vp, ctypes.c_double, vp, ci]
        L.enlsipb200_dense_last_ms.restype = ctypes.c_float
    return L


def lib():
    """Load the CUDA library.  Raises if it has not been built: no fallback of any kind."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libenlsip_b200.so is missing (%s): run __graft_entry__.build(); "
                               "the engine has no CPU fallback" % LIB_PATH)
        _lib = _bind(ctypes.CDLL(LIB_PATH))
    return _lib


USER_LIB_DIR = os.path.join(_HERE, "lib", "user")
_user_libs = {}


def compile_family(source, n, m, nb_eq=0, nb_ineq=0, stride0=0, stride1=0, has_jacobians=False, name=None):
    """enlsipb200_compile_family: compile the solver around user CUDA source (the replacement of the reference's
    closure arguments, cnls_model.jl:345-359).  Returns the loaded library, which exports the same C ABI with
    family id FAMILY_USER.  Libraries are cached in lib/user/ by a hash of (source, sizes, solver headers)."""
    import hashlib
    hsh = hashlib.sha256()
    hsh.update(repr((source, n, m, nb_eq, nb_ineq, stride0, stride1, bool(has_jacobians))).encode())
    for p in [SRC] + HEADERS:
        hsh.update(open(p, "rb").read())
    tag = (name or "family") + "_" + hsh.hexdigest()[:16]
    if tag in _user_libs:
        return _user_libs[tag]
    out = os.path.join(USER_LIB_DIR, "libenlsip_b200_%s.so" % tag)
    if not os.path.exists(out):
        # one-process-per-GPU launches build the same family concurrently: per-process work directory and library name,
        # renamed into place when complete (os.replace is atomic), so nobody loads a half-written file
        work = os.path.join(USER_LIB_DIR, "%s.%d" % (tag, os.getpid()))
        os.makedirs(work, exist_ok=True)
        tmp = os.path.join(work, "lib.so")
        try:
            rc = lib().enlsipb200_compile_family(source.encode(), n, m, nb_eq, nb_ineq, stride0, stride1,
                                                 1 if has_jacobians else 0, tmp.encode(), work.encode())
            check(rc)
            os.replace(tmp, out)
        finally:
            shutil.rmtree(work, ignore_errors=True)
    L = _bind(ctypes.CDLL(out), large=False)
    _user_libs[tag] = L
    return L


def _bind_large_only(L):
    """Prototypes of a library built by enlsipb200_large_compile_family (large-regime symbols only)."""
    vp, ll, ci = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int
    L.enlsipb200_large_last_error.restype = ctypes.c_char_p
    L.enlsipb200_large_create.argtypes = [ci, ci, ll, ll, ci, ci, vp, vp, vp, ci, ctypes.POINTER(vp)]
    L.enlsipb200_large_destroy.argtypes = [vp]
    L.enlsipb200_large_set_data.argtypes = [vp, ci, vp, ll, ci]
    L.enlsipb200_large_solve.argtypes = [vp, vp, ctypes.POINTER(Options)] + [vp] * 8 + [ci]
    L.enlsipb200_large_factor.argtypes = [vp, vp, vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    L.enlsipb200_large_stats.argtypes = [vp, vp, ci]
    return L


def large_compile_family(source, m, nb_eq=0, nb_ineq=0, has_jacobians=False, name=None):
    """enlsipb200_large_compile_family: the large-regime solver compiled around user CUDA source (row functors over a
    point accessor, csrc/enl_large_user.h).  Cached in lib/user/ by a hash of (source, sizes, solver sources); built under a
    per-process temporary name and renamed into place, so concurrent builders never load a half-written library."""
    import hashlib
    hsh = hashlib.sha256()
    hsh.update(repr((source, int(m), nb_eq, nb_ineq, bool(has_jacobians))).encode())
    for p in [SRC, SRC_LARGE] + HEADERS_LARGE + [os.path.join(_HERE, "csrc", "enl_large_user.h")]:
        hsh.update(open(p, "rb").read())
    tag = (name or "large_family") + "_" + hsh.hexdigest()[:16]
    if tag in _user_libs:
        return _user_libs[tag]
    out = os.path.join(USER_LIB_DIR, "libenlsip_b200_%s.so" % tag)
    if not os.path.exists(out):
        work = os.path.join(USER_LIB_DIR, "%s.%d" % (tag, os.getpid()))
        os.makedirs(work, exist_ok=True)
        tmp = os.path.join(work, "lib.so")
        try:
            check(lib().enlsipb200_large_compile_family(source.encode(), int(m), nb_eq, nb_ineq, 1 if has_jacobians else 0,
                                                        tmp.encode(), work.encode()))
            os.replace(tmp, out)
        finally:
            shutil.rmtree(work, ignore_errors=True)
    L = _bind_large_only(ctypes.CDLL(out))
    _user_libs[tag] = L
    return L


class EngineError(RuntimeError):
    pass


def check(rc, L=None):
    if rc != 0:
        raise EngineError("enlsip_b200 error %d: %s" % (rc, (L or lib()).enlsipb200_last_error().decode()))


def check_large(rc, L=None):
    if rc != 0:
        raise EngineError("enlsip_b200 (large regime) error %d: %s" % (rc, (L or lib()).enlsipb200_large_last_error().decode()))


def default_options() -> Options:
    o = Options()
    lib().enlsipb200_default_options(ctypes.byref(o))
    return o
