"""Oracle results of the mid-size Newton path (tests/test_large_midsize.py) that take too long to recompute in a test run:
chained Wood at n = 100 (m = 294) from the reference's x0 with the tolerances of the reference's chained Wood test
(rel_tol 1e-5, x_tol 1e-3, c_tol 1e-6).  The oracle's Hessian is a Python double loop: about 40 s.

    python tests/golden/make_midsize_fixture.py        ->  tests/golden/midsize_wood100_oracle.npz
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import enlsip_oracle as O, problems as P         # noqa: E402

WOOD_TOL = dict(rel_tol=1e-5, x_tol=1e-3, c_tol=1e-6)


def summarize(r):
    """the fields of an oracle Result that tests/test_hostport.py::check_against_oracle reads"""
    trace = np.array([(t.t, t.rankA, t.rankJ2, t.dimA, t.dimJ2, t.code, t.index_del, t.exit_code) for t in r.trace],
                     dtype=np.int32)
    x_prev = r.trace[-2].x_new if len(r.trace) >= 2 else np.zeros_like(r.x)
    return dict(x=r.x, f=r.f, exit_code=r.exit_code, iterations=r.iterations, active=np.array(r.active, dtype=np.int32),
                trace=trace, x_prev=x_prev, last_p_norm=r.trace[-1].p_norm)


if __name__ == "__main__":
    t0 = time.time()
    r = O.solve(P.chained_wood(100), wallclock=False, **WOOD_TOL)
    dt = time.time() - t0
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "midsize_wood100_oracle.npz"), oracle_seconds=dt,
                        **summarize(r))
    print(json.dumps({"exit_code": r.exit_code, "iterations": r.iterations, "f": r.f, "seconds": dt,
                      "codes": [t.code for t in r.trace]}))
