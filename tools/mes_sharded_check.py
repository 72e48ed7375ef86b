"""Sharded top-k with max-value entropy search on two or more ranks (one process per GPU, torch.distributed gloo for the
exchange): every rank's global top-k equals the single-GPU top-k over the whole set, bit for bit.

    python -m torch.distributed.run --nproc-per-node=2 tools/mes_sharded_check.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch.distributed as dist  # noqa: E402

import abo_b200 as abo  # noqa: E402


def main():
    dist.init_process_group("gloo")
    rank = dist.get_rank()
    ctx = abo.Context(int(os.environ.get("LOCAL_RANK", rank)))
    rng = np.random.default_rng(3)
    X = rng.random((400, 4)); y = np.sin(3 * X[:, 0]) + X.sum(1)
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.Matern52Kernel(), 0.6), 1e-4, ctx=ctx), X, y)
    Xc = rng.random((300_001, 4))
    acq = abo.MaxValueEntropySearch(11, float(y.min()), 16, 2048)
    ti, tv = abo.sharded_topk(acq, gp, Xc, 50)
    single = abo.MaxValueEntropySearch(11, float(y.min()), 16, 2048)
    _, si, sv = single.topk(gp, Xc, 50)
    assert np.array_equal(ti, si) and np.array_equal(tv, sv), (rank, ti[:5], si[:5])
    assert np.array_equal(acq._cache["ystar"], single._cache["ystar"])
    dist.barrier()
    if rank == 0:
        print("mes_sharded_check ok")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
