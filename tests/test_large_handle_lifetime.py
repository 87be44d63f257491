"""Device memory of large-regime handles is released with them: for each path of the large regime (the single-index
family, chained Rosenbrock on both factor paths, a mid-size chained Wood with Newton steps, a solve whose working set
grows), create -> solve -> destroy three times leaves the device memory in use where the first round left it.  A handle
that refused its solve (a row shard that was never joined) is released as well.  With two GPUs, joining a handle twice
leaves the memory in use of one join (tools/handle_footprint.py --comm-twice)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the non-time fields of stats()
COUNT_KEYS = ("points", "linesearch_evals", "launches", "rows_pad", "device_qrcp", "device_mulq", "factorisations",
              "ws_growths", "newton_steps")


def _c4():
    import enlsip_jl_b200 as E
    d = E.synth.gen_single_index(65536, 256, 64, seed=4)
    return E.LargeCnlsModel("single_index", d["x0"], d), {}


def _rosenbrock(factor):
    import enlsip_jl_b200 as E
    from oracle import problems as P
    return E.LargeCnlsModel("chained_rosenbrock", P.chained_rosenbrock(1000).x0, factor=factor), {}


def _wood_midsize():
    import enlsip_jl_b200 as E
    from oracle import problems as P
    from tests.test_large_midsize import WOOD_TOL, wood_family
    return E.LargeCnlsModel(wood_family(40), P.chained_wood(40).x0), dict(WOOD_TOL)


def _ws_growth():
    """bounds (0, 2), n = 256, every parameter below its lower bound and 16 block inequalities violated: t0 = n + 16"""
    import enlsip_jl_b200 as E
    n = 256
    d = E.synth.gen_single_index(3000, n, 64, seed=3, ineq=True)
    x0 = np.full(n, -0.05)
    x0[:64] = -1.9
    return E.LargeCnlsModel("single_index", x0, d, ineq=True, x_low=np.zeros(n), x_upp=np.full(n, 2.0)), {}


CASES = {
    "c4_m65536": _c4,
    "cr1000_householder": lambda: _rosenbrock("householder"),
    "cr1000_tsqr": lambda: _rosenbrock("tsqr"),
    "wood40_midsize": _wood_midsize,
    "ws_growth": _ws_growth,
}


def _free():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_create_solve_destroy_releases_device_memory(name):
    import enlsip_jl_b200 as E
    free = []
    for _ in range(3):
        mod, kw = CASES[name]()
        E.solve(mod, **kw)
        if name == "ws_growth":
            assert mod.stats()["ws_growths"] > 0
        if name == "wood40_midsize":
            assert mod.stats()["newton_steps"] > 0
        mod.close()
        free.append(_free())
    assert free[2] == free[0], free


@pytest.mark.gpu
def test_refused_solve_releases_device_memory():
    """a row shard (m_local < m_global) whose handle was never joined refuses every solve and is released whole"""
    import enlsip_jl_b200 as E
    from oracle import problems as P
    free = []
    for _ in range(3):
        mod = E.LargeCnlsModel("chained_rosenbrock", P.chained_rosenbrock(1000).x0, factor="tsqr", shard=(0, 2))
        with pytest.raises(E.capi.EngineError, match="not joined"):
            E.solve(mod)
        mod.close()
        free.append(_free())
    assert free[2] == free[0], free


@pytest.mark.gpu
def test_comm_init_twice_keeps_device_memory():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29800 + (os.getpid() % 200)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tools", "handle_footprint.py"), "--comm-twice"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
