"""One process per GPU (torchrun): b7_blr_fit_multi + b7_dngo_score_multi over a sharded grid against the one-GPU result on rank 0.
Run: python -m torch.distributed.run --nproc-per-node G --master-addr 127.0.0.1 tools/dngo_multi_check.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch.distributed as dist  # noqa: E402

import b7_oracle as o  # noqa: E402
from bot7_b200 import _lib as L  # noqa: E402
from bot7_b200 import grids, models, parallel  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
dist.init_process_group("gloo")
comm = parallel.Comm.from_env(local, world, rank)
N, d, M = 700, 6, 30011
r = np.random.default_rng(4)
Ws = [r.standard_normal((32, d)) * np.sqrt(2.0 / d), r.standard_normal((50, 32)) * np.sqrt(2.0 / 32)]
bs = [0.1 * r.standard_normal(32), 0.1 * r.standard_normal(50)]
Xo = o.sobol_points(d, N)
y = o.hartmann6(Xo)
y = (y - y.mean()) / y.std()
Z0 = o.mlp_features(Xo, Ws, bs, True)
for S in (5, 1):
    hyp = np.column_stack([np.log(0.1) + r.random(S) * np.log(100), np.log(10) + r.random(S) * np.log(100), y.mean() + 0.1 * r.random(S)])
    gs = comm.sobol_grid(d, 1 + N, M)
    blrs, info = comm.blr_fit(Z0, y, hyp)
    b, a, ao, n_, sc = comm.dngo_score(blrs, gs, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), want_scores=True)
    row = comm.grid_remove(gs, a)
    b2, a2, ao2, n2, _ = comm.dngo_score(blrs, gs, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()))
    if rank == 0:
        ctx = comm.ctxs[0]
        f = models.BLRFactors(Z0, y, hyp, ctx=ctx)
        g1 = grids.sobol({"size": N + M, "dims": d}, ctx=ctx).generate_device(first=N, count=M)
        one, am, amo, best, nn = models.dngo_score(f, g1, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), want_scores=True)
        r0, cnt = parallel.shard_range(M, world, 0)
        assert np.array_equal(info, f.info), "info differs"
        assert np.array_equal(sc.view(np.int64), one[r0:r0 + cnt].view(np.int64)), "shard scores differ"
        assert (b, a, ao, n_) == (best, am, amo, nn), ((b, a, ao, n_), (best, am, amo, nn))
        row1 = g1.remove(am)
        assert np.array_equal(row, row1.reshape(-1)), "removed rows differ"
        _, am, amo, best, nn = models.dngo_score(f, g1, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()))
        assert (b2, a2, ao2, n2) == (best, am, amo, nn)
        f.free()
        g1.free()
        print(f"S={S}: world {world}, argmax {a} then {a2} ok")
    comm.free_blr(blrs)
    for g in gs:
        g.free()
dist.barrier()
if rank == 0:
    print("dngo_multi_check ok")
comm.close()
dist.destroy_process_group()
