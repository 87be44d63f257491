"""Row-sharded row families on the TSQR path (run under torch.distributed.run, one rank per GPU):
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29811 tools/row_tsqr_dist.py
Every rank also solves the whole problem alone on its GPU (factor="tsqr", one shard) and compares:
  * the single-index model as user source (m = 2^16, n = 256) and chained Rosenbrock (n = 1000), shards of
    LargeCnlsModel(shard=(rank, world)) (multiples of 256 rows) and uneven shards that cut subtiles:
    R to 1e-10 up to row signs, the same iteration count, f to 1e-10 (whether R, x and f also agree bit for bit is
    printed);
  * a wrong sum of m_local: enlsipb200_large_comm_init refuses on every rank and every process goes on to exit."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import enlsip_jl_b200 as E                                   # noqa: E402
from tests.test_large_row_tsqr import SI_M, SI_NB, si_data, si_family     # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl")


ML = sys.modules[E.LargeCnlsModel.__module__]
ALIGNED = ML.shard_rows


def uneven(m, r, w):
    """rows per rank in the proportions 3 : 5 : 7 : ... (shards that cut subtiles and 32-row blocks)"""
    p = np.arange(w) * 2 + 3
    rows = (m * p // p.sum()).astype(int)
    rows[-1] = m - rows[:-1].sum()
    return int(rows[:r].sum()), int(rows[r])


def short_by_one(m, r, w):
    row0, rows = ALIGNED(m, r, w)
    return row0, rows - (1 if r == w - 1 else 0)


def model(make, split):
    """make(shard) with LargeCnlsModel's row split replaced by `split` (None: the whole problem on this GPU)"""
    if split is None:
        return make(None)
    ML.shard_rows = split
    try:
        return make((rank, world))
    finally:
        ML.shard_rows = ALIGNED


def run(make, x0, split):
    mod = model(make, split)
    if split is not None:
        mod.join(rank, world)
    R, _, _ = mod.factor(x0)
    E.solve(mod)
    out = (R, mod.sol[0].copy(), float(mod.obj_value[0]), int(mod.iterations[0]), int(mod.exit_code[0]), mod.row0, mod.rows)
    mod.close()
    return out


def check(name, make, x0):
    one = run(make, x0, None)
    for label, split in (("aligned", ALIGNED), ("uneven", uneven)):
        got = run(make, x0, split)
        R, R1 = got[0], one[0]
        sg = np.sign(np.diag(R)) * np.sign(np.diag(R1))
        sg[sg == 0] = 1.0
        dR = np.abs(R * sg[:, None] - R1).max() / np.abs(R1).max()
        same = np.array_equal(R, R1) and np.array_equal(got[1], one[1]) and got[2] == one[2]
        print("rank %d %s %s rows [%d, %d): |R - R_1gpu| / max|R| = %.2e, iterations %d vs %d, f rel diff %.2e, "
              "bit-identical %s" % (rank, name, label, got[5], got[5] + got[6], dR, got[3], one[3],
                                    abs(got[2] - one[2]) / abs(one[2]), same), flush=True)
        assert dR <= 1e-10 and got[3] == one[3] and got[4] == one[4]
        assert abs(got[2] - one[2]) <= 1e-10 * abs(one[2])


d = E.synth.gen_single_index(SI_M, 256, SI_NB, seed=81)
fam = si_family()
check("single-index source", lambda shard: E.LargeCnlsModel(fam, d["x0"], data=si_data(d), factor="tsqr", shard=shard,
                                                             device=local), d["x0"])

from oracle import problems as P                          # noqa: E402
xcr = P.chained_rosenbrock(1000).x0
make_cr = lambda shard: E.LargeCnlsModel("chained_rosenbrock", xcr, factor="tsqr", shard=shard, device=local)  # noqa: E731
check("chained Rosenbrock n=1000", make_cr, xcr)

# one row short in all: every rank is refused by comm_init, none is left waiting in a collective
mod = model(make_cr, short_by_one)
try:
    mod.join(rank, world)
    raise SystemExit("rank %d: comm_init accepted 1997 rows of 1998" % rank)
except E.capi.EngineError as e:
    assert "row shards" in str(e), str(e)
    print("rank %d: wrong row total refused: %s" % (rank, e), flush=True)
mod.close()

dist.barrier()
if rank == 0:
    print("row_tsqr_dist: all checks passed", flush=True)
dist.destroy_process_group()
