"""Device-timed rate of candidate-restricted evaluation (``evaluate_topk(..., items=, exclude=)``) at the MPD shape
(V = 2M items, H = 100).

    python scripts/evaluate_filters_bench.py [--rows 4096] [--batch 256] [--gold 5] [--reps 3]

``evaluate_topk`` with the metrics mrr@10, map, P@10 on ``rows`` query rows in batches of ``batch``, ``gold`` held-out
items per row, for
  * no filter;
  * eligible fractions 0.1 and 0.01, each with 50 exclusions per row.
Each leg is timed by CUDA events around whole calls (each call ends in the ranks' device-to-host copy); the rate is
query rows per second, the best of ``reps`` calls after one warm-up call.  The compact copy of the eligible rows is
built once before the warm-up and its build time is reported apart.  Prints one JSON line with the card's name and
power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "aae-recommender_b200"))


def card():
    import torch
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return torch.cuda.get_device_name(0), pl


def timed(model, X, Y, kw, batch, reps):
    import torch
    metrics = ["mrr@10", "map", "P@10"]
    res = model.evaluate_topk(X, Y, metrics, batch_size=batch, **kw)        # warm-up
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model.evaluate_topk(X, Y, metrics, batch_size=batch, **kw)
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) * 1e-3
        best = sec if best is None else min(best, sec)
    return {"rows_per_s": X.shape[0] / best, "ms_per_call": best * 1e3,
            "metrics": {m: round(v[0], 6) for m, v in zip(metrics, res)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--gold", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--V", type=int, default=2000000)
    args = ap.parse_args()
    import torch
    from aaerec_b200.aae import AdversarialAutoEncoder
    from aaerec_b200.filters import RankFilter
    from aaerec_b200.synth import synth_sets
    V, H, C, n = args.V, 100, 50, args.rows
    name, power = card()
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=args.batch, n_epochs=1, verbose=False)
    model._build(V, C)
    model.engine.Wd3.mul_(8.0)
    rng = np.random.default_rng(0)
    X = synth_sets(n, V, 50, seed=1)
    Y = sp.csr_matrix((np.ones(n * args.gold, np.float32),
                       (np.repeat(np.arange(n), args.gold), rng.integers(0, V, n * args.gold))), shape=(n, V))
    Y.data[:] = 1
    out = {"metric": "filtered evaluate_topk query rows/s", "card": name, "power_limit": power, "V": V, "H": H,
           "rows": n, "batch": args.batch, "gold_per_row": args.gold, "reps": args.reps, "legs": {}}
    out["legs"]["none"] = timed(model, X, Y, {}, args.batch, args.reps)
    for frac in (0.1, 0.01):
        items = rng.choice(V, int(frac * V), replace=False)
        # gold among the eligible items too, so that the metrics are not all zero
        Yf = Y.tolil()
        Yf[np.arange(n), items[rng.integers(0, items.size, n)]] = 1
        Yf = Yf.tocsr()
        E = sp.csr_matrix((np.ones(n * 50, np.float32), (np.repeat(np.arange(n), 50), rng.integers(0, V, n * 50))),
                          shape=(n, V))
        filt = RankFilter.build(V, n, items=items, exclude=E)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.engine._compact(filt.shard_ids(V, 0, 1))
        torch.cuda.synchronize()
        build = (time.perf_counter() - t0) * 1e3
        out["legs"]["frac_%g_excl50" % frac] = dict(timed(model, X, Yf, dict(items=items, exclude=E), args.batch,
                                                          args.reps), eligible=int(items.size), compact_build_ms=build)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
