"""10^4-problem oracle fixtures of the batched configs (SURVEY.md section 7, step 3): C2 (HS65), C3 with analytic and with
forward-difference Jacobians.  One oracle solve per problem, all host cores (multiprocessing); ~10 min in the build
container.  The problems start at offset 10^5 of the synthetic streams (the small fixtures cover the head).

    python tests/golden/make_golden_10k.py      ->  tests/golden/{c2_hs65,c3_gp_analytic,c3_gp_fd}_10k.npz
"""
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("OMP_NUM_THREADS", "1")
import enlsip_jl_b200 as E                                   # noqa: E402
from oracle import enlsip_oracle as O, problems as P         # noqa: E402
from make_golden import pack as pack_all                     # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
B, START = 10_000, 100_000


def pack(results, n, lmax):
    """make_golden.pack without x_pen: the 10^4-problem histograms never read it, and it would take each C3 fixture over
    1 MB."""
    d = pack_all(results, n, lmax)
    del d["x_pen"]
    return d


def solve_hs65(x0):
    return O.solve(P.hs65(x0), wallclock=False)


def solve_gp(args):
    y, S, x0, fd = args
    return O.solve(P.gauss_peaks(y, S, x0, fd=fd), wallclock=False)


def main():
    t0 = time.time()
    with mp.Pool(os.cpu_count()) as pool:
        x0 = E.synth.gen_hs65_batch(B, start=START)
        res = pool.map(solve_hs65, [x0[b] for b in range(B)], chunksize=50)
        np.savez_compressed(os.path.join(HERE, "c2_hs65_10k.npz"), start=START, **pack(res, 3, 7))
        print("c2", time.time() - t0, flush=True)
        y, S, x0g, _ = E.synth.gen_gauss_peaks_batch(B, start=START)
        for fd, name in ((False, "c3_gp_analytic_10k"), (True, "c3_gp_fd_10k")):
            res = pool.map(solve_gp, [(y[b], S[b], x0g[b], fd) for b in range(B)], chunksize=25)
            np.savez_compressed(os.path.join(HERE, name + ".npz"), start=START, **pack(res, 6, 13))
            print(name, time.time() - t0, flush=True)


if __name__ == "__main__":
    main()
