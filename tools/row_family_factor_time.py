"""Row families: the plain-Householder path (default) against the TSQR path (factor="tsqr") on one GPU.

  python tools/row_family_factor_time.py [--reps 5] [--out FILE.json]

Per shape and path: build ms and factorisation ms of the factor hook (CUDA events on the handle's stream, median of
--reps calls after one warm-up call), and the wall time of one whole solve after a warm-up solve.  Shapes: chained
Rosenbrock n = 1000 (m = 1998), the n = 4 data family of tests/test_large_user_family.py at m = 50 000 (forward
differences), and the single-index model written as user source (tests/test_large_row_tsqr.py) at m = 2^20, n = 256.
Prints one JSON line per shape and path."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import enlsip_jl_b200 as E                                                   # noqa: E402
from oracle import problems as P                                            # noqa: E402
from tests.test_large_row_tsqr import SI_NB, si_data, si_family             # noqa: E402
from tests.test_large_user_family import mix_family, mix_problem            # noqa: E402


def shapes():
    pb = P.chained_rosenbrock(1000)
    yield "chained_rosenbrock n=1000 m=1998", lambda f: E.LargeCnlsModel("chained_rosenbrock", pb.x0, factor=f), pb.x0
    m = 50_000
    mp, t, y, lo, up = mix_problem(m=m)
    fam = mix_family(m)
    yield "data family n=4 m=50000 (fd)", lambda f: E.LargeCnlsModel(fam, mp.x0, data={"t": t, "y": y}, x_low=lo, x_upp=up,
                                                                      factor=f), mp.x0
    m = 1 << 20
    d = E.synth.gen_single_index(m, 256, SI_NB, seed=90)
    sfam = si_family(m)
    yield "single-index source n=256 m=2^20", lambda f: E.LargeCnlsModel(sfam, d["x0"], data=si_data(d), factor=f), d["x0"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    rows = []
    for name, make, x0 in shapes():
        for path in ("householder", "tsqr"):
            mod = make(path)
            mod.factor(x0, want_R=False)
            b, q = [], []
            for _ in range(a.reps):
                _, bm, tm = mod.factor(x0, want_R=False)
                b.append(bm)
                q.append(tm)
            E.solve(mod)
            t0 = time.perf_counter()
            E.solve(mod)
            wall = (time.perf_counter() - t0) * 1e3
            st = mod.stats()
            row = dict(shape=name, path=path, build_ms=float(np.median(b)), factor_ms=float(np.median(q)), solve_wall_ms=wall,
                       iterations=int(mod.iterations[0]), exit_code=int(mod.exit_code[0]), f=float(mod.obj_value[0]),
                       rows_pad=int(st["rows_pad"]), gpu=torch.cuda.get_device_name(0))
            mod.close()
            print(json.dumps(row), flush=True)
            rows.append(row)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
