"""Sharded vb_init(initializer='svd') on the GPU, launched under torchrun (one rank per GPU) by
tests/test_gpu_svd_init.py: every rank holds a contiguous, nnz-balanced shard of the cells of a
golden matrix, Engine.init_svd runs collectively (sums over cells all-reduced, the Gaussian sketch
keyed by global cell index), and the gathered state must equal the one-GPU state to 1e-12."""
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from conftest import load_counts  # noqa: E402
from ccfindr_b200 import sharding  # noqa: E402
from ccfindr_b200.engine import Comm, Engine  # noqa: E402


def main():
    rank, local, world = (int(os.environ[k]) for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    uid = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        uid = torch.tensor(list(Engine.nccl_unique_id()), dtype=torch.uint8, device=dev)
    dist.broadcast(uid, 0)
    comm = Comm(world, rank, bytes(uid.cpu().tolist()), device=local)
    worst = 0.0
    for counts, r in (("pbmc", 3), ("pbmc", 5), ("c1s1", 3)):
        X = load_counts(counts)
        b = sharding.balanced_bounds(X.indptr, world)
        c0, c1 = b[rank], b[rank + 1]
        with Engine(sharding.shard_csc(X, c0, c1), device=local) as eng:
            eng.attach_comm(comm)
            eng.init_svd(r, seed=4, cell_offset=c0)
            st = eng.get_state(("lw", "lh", "ew", "eh"))
        parts = [None] * world
        dist.all_gather_object(parts, (st["lh"], st["eh"]))
        with Engine(X, device=local) as one:
            one.init_svd(r, seed=4)
            ref = one.get_state(("lw", "lh", "ew", "eh"))
        got = dict(lw=st["lw"], ew=st["ew"], lh=np.concatenate([p[0] for p in parts], axis=1),
                   eh=np.concatenate([p[1] for p in parts], axis=1))
        for k in ("lw", "lh", "ew", "eh"):
            e = float(np.max(np.abs(got[k] - ref[k])) / np.max(np.abs(ref[k])))
            assert e < 1e-12, (counts, r, k, rank, e)
            worst = max(worst, e)
    t = torch.tensor([worst], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("MGPU_SVD_OK world=%d worst_rel_err=%.3e" % (world, t.item()))
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
