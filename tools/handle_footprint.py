"""Counts and device-memory footprint of large-regime handles, one line per case: the non-time fields of stats() after one
solve, and the device memory in use (bytes below the free memory at the start of the run, cudaMemGetInfo) after create
and after solve.  The output depends on the code and the device model only, so two builds can be compared line by line.

Cases (tests/test_large_handle_lifetime.py creates, solves and destroys the same handles):
  c4_m65536          the C4 problem (single-index, n = 256, 64 equalities) at m = 65536
  cr1000_householder chained Rosenbrock n = 1000, [J | r] by the plain Householder QR
  cr1000_tsqr        chained Rosenbrock n = 1000, [J | r] by the TSQR
  wood40_midsize     chained Wood n = 40 (n + m < 1000: Newton steps)
  ws_growth          single-index n = 256 from a start whose working set grows past min(l, n) + 1 rows

    python tools/handle_footprint.py
    python -m torch.distributed.run --nproc-per-node 2 tools/handle_footprint.py --comm-twice   (two GPUs)
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import enlsip_jl_b200 as E                                        # noqa: E402
from tests.test_large_handle_lifetime import CASES, COUNT_KEYS     # noqa: E402


def used(free0):
    import torch
    return free0 - torch.cuda.mem_get_info()[0]


def footprint():
    import torch
    torch.cuda.init()
    free0 = torch.cuda.mem_get_info()[0]
    for name, make in CASES.items():
        mod, kw = make()
        after_create = used(free0)
        E.solve(mod, **kw)
        st = mod.stats()
        row = dict(case=name, exit_code=int(mod.exit_code[0]), iterations=int(mod.iterations[0]),
                   used_after_create=after_create, used_after_solve=used(free0), **{k: int(st[k]) for k in COUNT_KEYS})
        mod.close()
        print(json.dumps(row))


def comm_twice():
    """every rank joins twice; the device memory in use after the second join is what it was after the first"""
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl")
    from oracle import problems as P
    mod = E.LargeCnlsModel("chained_rosenbrock", P.chained_rosenbrock(1000).x0, factor="tsqr", shard=(rank, world), device=local)
    mod.join(rank, world)
    torch.cuda.synchronize()
    once = torch.cuda.mem_get_info()[0]
    mod.join(rank, world)
    torch.cuda.synchronize()
    twice = torch.cuda.mem_get_info()[0]
    E.solve(mod)
    mod.close()
    dist.barrier()
    print("rank %d comm_init twice: free after one join %d, after two %d" % (rank, once, twice))
    dist.destroy_process_group()
    if once != twice:
        raise SystemExit(1)


if __name__ == "__main__":
    comm_twice() if "--comm-twice" in sys.argv else footprint()
