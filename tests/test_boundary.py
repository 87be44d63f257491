"""The C-ABI library loads, exports every symbol include/enlsip_b200.h declares, and refuses to compute without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

import __graft_entry__ as ge

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi():
    import enlsip_jl_b200 as E
    E.capi.build()
    return E.capi


def test_header_symbols_exported(capi):
    hdr = open(os.path.join(ROOT, "include", "enlsip_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(enlsipb200_[a-z_0-9]+)\s*\(", hdr)))
    assert declared == sorted(capi.EXPORTS)
    raw = ctypes.CDLL(capi.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert capi.lib().enlsipb200_version() >= 100


def test_default_options_match_solver_jl(capi):
    o = capi.default_options()      # solver.jl:62-63
    assert o.max_iter == 100 and o.scaling == 0 and o.time_limit == 1e3
    assert all(np.isnan(v) for v in (o.abs_tol, o.rel_tol, o.c_tol, o.x_tol))


def test_no_cpu_fallback(capi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import enlsip_jl_b200 as E
    with pytest.raises(capi.EngineError, match="no CPU fallback"):
        E.CnlsModel("hs65", np.zeros((1, 3)), x_low=E.synth.HS65_LOW, x_upp=E.synth.HS65_UPP)
    x = np.zeros(4)
    rc = capi.lib().enlsipb200_det_exp(x.ctypes.data, x.ctypes.data, 4, 0)
    assert rc == -2
    # the large-Jacobian regime fails the same way: no device, no solve
    d = E.synth.gen_single_index(1200, 32, 8, seed=1)
    with pytest.raises(capi.EngineError, match="(?i)no cuda device|cuda"):
        E.LargeCnlsModel("single_index", d["x0"], d)


def test_large_api_validation(capi):
    """Argument checks of enlsipb200_large_create happen before any device is touched."""
    import ctypes
    L = capi.lib()
    h = ctypes.c_void_p()
    rho = np.ones(8)
    assert L.enlsipb200_large_create(capi.FAMILY_SINGLE_INDEX, 30, 1000, 1000, 4, 0, rho.ctypes.data, None, None, -1, ctypes.byref(h)) != 0
    assert b"multiple of 32" in L.enlsipb200_large_last_error()
    assert L.enlsipb200_large_create(capi.FAMILY_SINGLE_INDEX, 32, 100, 100, 4, 0, rho.ctypes.data, None, None, -1, ctypes.byref(h)) != 0
    assert b"batched engine" in L.enlsipb200_large_last_error()          # n + m < 1000: Newton regime (EF:2658)
    assert L.enlsipb200_large_create(99, 32, 1000, 1000, 4, 0, rho.ctypes.data, None, None, -1, ctypes.byref(h)) != 0
    assert L.enlsipb200_large_create(capi.FAMILY_SINGLE_INDEX, 32, 2000, 1000, 4, 0, rho.ctypes.data, None, None, -1, ctypes.byref(h)) != 0
    # the single-index kernels stage x in 48 KB of shared memory: n > 6144 is refused as an argument error (-1, EINVAL)
    assert L.enlsipb200_large_create(capi.FAMILY_SINGLE_INDEX, 6176, 10000, 10000, 4, 0, rho.ctypes.data, None, None, -1, ctypes.byref(h)) == -1
    assert b"n <= 6144" in L.enlsipb200_large_last_error()


def test_product_does_not_import_oracle():
    """Only tests/, smoke() and bench.py may touch oracle/: the package never imports, includes or loads it."""
    pkg = os.path.join(ROOT, "enlsip.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            path = os.path.join(dirpath, fn)
            if fn.endswith(".py"):
                for line in open(path):
                    code = line.split("#")[0]
                    assert not re.search(r"^\s*(from|import)\s+oracle\b", code), (fn, line)
                    assert not re.search(r"[\"']oracle[\"'/]", code), (fn, line)
            elif fn.endswith((".h", ".cu", ".cuh", ".cpp")):
                for line in open(path):
                    assert not re.search(r"#\s*include.*oracle", line), (fn, line)


def test_model_api_validation():
    import enlsip_jl_b200 as E
    with pytest.raises(AssertionError):
        E.CnlsModel("no_such_family", np.zeros((1, 3)))
    assert E.dict_status_codes[1] == "found_first_order_stationary_point" and E.dict_status_codes[-11] == "time_limit_exceeded"
