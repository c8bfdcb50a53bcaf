"""Two-GPU check of candidate-restricted evaluation (run under torchrun on a box with >= 2 B200s):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29514 \
        tests/multi_gpu_evaluate_filters_check.py

Every rank builds the same model (same seeded weights) sharded over the ranks, and a single-GPU model with the same
weights.  Item-sharded ``gold_ranks`` with ``items`` / ``exclude`` must give the single-GPU ranks: rank 0 (not in the
list) at the same entries, and equal ranks outside fp32 near-ties (the sharded encoder sums its first layer's partial
products in another order, as in multi_gpu_check.py).  Once with an eligible set spread over both shards, once with
one that leaves the last shard without any eligible item, and once with exclusions only.  Prints
MULTI_GPU_EVALUATE_FILTERS_OK on rank 0."""
import os
import sys

import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "aae-recommender_b200"))


def model(V, params, rank, world, H=100, C=50):
    from aaerec_b200.aae import AdversarialAutoEncoder
    m = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=128, n_epochs=1, verbose=False, impl="auto",
                               rank=rank, world=world)
    m._build(V, C, params={k: v.clone() for k, v in params.items()})
    return m


def main():
    from aaerec_b200.synth import synth_sets
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    from oracle import aae_oracle as O
    V, n = 100000, 300
    params = O.init_params(V, 100, 50, seed=21)
    params["dec.lin3.weight"] = params["dec.lin3.weight"] * 8.0
    sharded = model(V, params, rank, world)
    single = model(V, params, 0, 1)
    X = synth_sets(n, V, 15, seed=3)
    rng = np.random.default_rng(5)
    E = sp.csr_matrix((np.ones(n * 20, np.float32), (np.repeat(np.arange(n), 20), rng.integers(0, V, n * 20))),
                      shape=(n, V))
    spread = rng.choice(V, V // 3, replace=False)
    lower = rng.choice(V // 2, 40000, replace=False)          # nothing of the upper half (the last shard) eligible
    for name, items in (("spread", spread), ("one_shard_empty", lower), ("exclusions_only", None)):
        el = np.arange(V) if items is None else np.sort(items)
        g = np.concatenate((rng.integers(0, V, n * 6), el[rng.integers(0, el.size, n * 4)]))
        Y = sp.csr_matrix((np.ones(g.size, np.float32), (np.repeat(np.arange(n), 10), g)), shape=(n, V))
        Y.data[:] = 1
        _, want = single.gold_ranks(X, Y, items=items, exclude=E)
        _, got = sharded.gold_ranks(X, Y, items=items, exclude=E)
        assert np.array_equal(got == 0, want == 0), (name, "unreturnable gold differ")
        assert (want > 0).any(), name
        same = got == want
        assert same.mean() > 0.99, (name, float(same.mean()))
        # a differing rank is a near-tie: within a few places of the single-GPU rank
        assert np.all(np.abs(got - want)[~same] <= 3), name
        ms = ["mrr@10", "map", "P@10"]
        a = sharded.evaluate_topk(X, Y, ms, items=items, exclude=E)
        b = single.evaluate_topk(X, Y, ms, items=items, exclude=E)
        assert np.allclose(np.array(a), np.array(b), atol=1e-2), (name, a, b)
    dist.barrier()
    if rank == 0:
        print("MULTI_GPU_EVALUATE_FILTERS_OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
