"""Two-GPU check of candidate-restricted ranking (run under torchrun on a box with >= 2 B200s):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \
        tests/multi_gpu_filters_check.py

Every rank builds the same model (same seeded weights) sharded over the ranks, and a single-GPU model with the same
weights.  Item-sharded and set-sharded ``predict_topk`` with ``items`` / ``exclude`` must give the single-GPU lists:
padding at the same places, no ineligible or excluded item, ids equal outside fp32 near-ties (the sharded encoder sums
its first layer's partial products in another order, as in multi_gpu_check.py) and equal scores where the ids agree.
Once with an eligible set spread over both shards, once with one that leaves the second shard without any eligible
item, and once with fewer eligible items than k.  Prints MULTI_GPU_FILTERS_OK on rank 0."""
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
    m = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=256, n_epochs=1, verbose=False, impl="auto",
                               rank=rank, world=world)
    m._build(V, C, params={k: v.clone() for k, v in params.items()})
    return m


def check(got, want, items, E, what):
    gi, gv = got
    wi, wv = want
    assert gi.shape == wi.shape, what
    assert np.array_equal(gi < 0, wi < 0), (what, "padding differs")
    assert np.all(gv[gi < 0] == -np.inf), what
    live = gi >= 0
    assert np.isin(gi[live], items).all(), (what, "an ineligible item was returned")
    rows = np.nonzero(live)[0]
    hit = E[rows, gi[live]]
    assert not np.asarray(hit.todense() if sp.issparse(hit) else hit).any(), (what, "an excluded item was returned")
    same = gi == wi
    assert same.mean() > 0.99, (what, float(same.mean()))
    np.testing.assert_allclose(gv[same & live], wv[same & live], rtol=1e-5, atol=1e-5, err_msg=what)


def main():
    from aaerec_b200.synth import synth_sets
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    from oracle import aae_oracle as O
    V, n, k = 100000, 300, 100
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
    for name, items in (("spread", spread), ("one_shard_empty", lower), ("fewer_than_k", lower[:30])):
        want = single.predict_topk(X, k, items=items, exclude=E, return_scores=True)
        if name == "fewer_than_k":
            assert (want[0][:, -1] == -1).all()
        for shard in ("items", "sets"):
            got = sharded.predict_topk(X, k, items=items, exclude=E, return_scores=True, shard=shard)
            check(got, want, items, E, "%s/%s" % (name, shard))
    dist.barrier()
    if rank == 0:
        print("MULTI_GPU_FILTERS_OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
