"""Wall clock of mid-size solves (n + m < 1000, Newton steps on: LargeCnlsModel with ENLSIPB200_LARGE_MIDSIZE) on one GPU.

Per problem: one warm-up solve, then the median of 5 solves (host clock around the blocking solve), the Newton steps and
the Hessian kernel's device time (CUDA events, from stats()) of one solve.  Problems: chained Rosenbrock n = 100 (a row of
the reference's timing table, docs/src/tutorial.md:300), chained Wood n = 100 and chained Wood at the largest even n with
n + m < 1000 (n = 250, m = 744), both from the reference's x0 with the tolerances of its chained Wood test.  The device
name and power limit are read in the same run (nvidia-smi, query only).

    python tools/midsize_time.py
"""
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import enlsip_jl_b200 as E                                        # noqa: E402
from oracle import problems as P                                  # noqa: E402
from tests.test_large_midsize import WOOD_TOL, wood_family        # noqa: E402


def device_info():
    """name and power limit of the GPU the solves run on (the current CUDA device, matched to nvidia-smi by UUID)"""
    import torch
    uuid = str(torch.cuda.get_device_properties(torch.cuda.current_device()).uuid)
    out = subprocess.run(["nvidia-smi", "--query-gpu=uuid,name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()
    for line in out:
        u, name, limit = [v.strip() for v in line.split(",")]
        if u.replace("GPU-", "") == uuid.replace("GPU-", ""):
            return "%s, %s" % (name, limit)
    raise SystemExit("the current CUDA device (%s) is not in nvidia-smi's list" % uuid)


def time_model(make, kw, reps=5):
    mod = make()
    E.solve(mod, **kw)                                             # warm-up: modules, allocations
    times = []
    for _ in range(reps):
        base = mod.stats()
        t0 = time.perf_counter()
        E.solve(mod, **kw)
        times.append(time.perf_counter() - t0)
        st = mod.stats()
    res = dict(median_s=statistics.median(times), min_s=min(times), exit_code=int(mod.exit_code[0]),
               iterations=int(mod.iterations[0]), newton_steps=int(st["newton_steps"] - base["newton_steps"]),
               hessian_ms=st["hessian_ms"] - base["hessian_ms"])
    mod.close()
    return res


def main():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("midsize_time.py measures on a GPU; none is visible")
    rows = {"device": device_info()}
    rows["chained_rosenbrock_100"] = time_model(lambda: E.LargeCnlsModel("chained_rosenbrock", P.chained_rosenbrock(100).x0), {})
    for n in (100, 250):
        rows["chained_wood_%d" % n] = time_model(lambda: E.LargeCnlsModel(wood_family(n), P.chained_wood(n).x0), WOOD_TOL)
    print(json.dumps(rows, indent=1))


if __name__ == "__main__":
    main()
