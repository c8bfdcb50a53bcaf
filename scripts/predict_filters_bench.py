"""Device-timed rate of candidate-restricted top-k predict at the MPD shape (V = 2M items, H = 100, k = 100).

    python scripts/predict_filters_bench.py [--iters 20] [--batches 1000,16000]

Per query batch size B: sets/s of ``AAEEngine.topk`` on one device-resident batch (CUDA events around ``iters`` calls,
status word checked after the loop, as bench.py's predict leg does) for
  * no filter;
  * items = every item (the public call drops such a filter: the same path, plus the canonicalisation, timed apart);
  * eligible fractions 0.1 and 0.01, each with 50 exclusions per row (the exclusion CSR is staged per call; the compact
    copy of the eligible rows is built once, in the warm-up, and its build time is reported apart).
Prints one JSON line with the card's name and power limit, read in the same run."""
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


def timed(eng, B, k, filt, iters):
    import torch
    for _ in range(2):
        eng.topk(B, k, filt=filt)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        eng.topk(B, k, filt=filt, check=False)
    e1.record()
    torch.cuda.synchronize()
    if eng.topk_status() != 0:
        raise RuntimeError("fused top-k reported rows it could not rank exactly in the timed loop")
    sec = e0.elapsed_time(e1) * 1e-3 / iters
    return {"sets_per_s": B / sec, "ms_per_batch": sec * 1e3, "path": eng.topk_mode}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batches", default="1000,16000")
    ap.add_argument("--V", type=int, default=2000000)
    args = ap.parse_args()
    import torch
    from aaerec_b200.engine import AAEEngine
    from aaerec_b200.filters import RankFilter
    from aaerec_b200.synth import synth_sets
    V, H, C, k = args.V, 100, 50, 100
    Bs = [int(b) for b in args.batches.split(",")]
    name, power = card()
    eng = AAEEngine(V, H, C, max_batch=max(Bs))
    eng.init_uniform(3)
    eng.Wd3.mul_(8.0)
    rng = np.random.default_rng(0)
    out = {"metric": "filtered top-100 predict sets/s", "card": name, "power_limit": power, "V": V, "H": H, "k": k,
           "iters": args.iters, "legs": {}}
    for B in Bs:
        X = synth_sets(B, V, 50, seed=B)
        eng.upload_csr(X.indptr.astype(np.int32), X.indices.astype(np.int32))
        legs = out["legs"][str(B)] = {}
        legs["none"] = timed(eng, B, k, None, args.iters)
        t0 = time.perf_counter()
        every = RankFilter.build(V, B, items=np.arange(V))
        legs["items_all"] = dict(timed(eng, B, k, every, args.iters), canonicalise_ms=(time.perf_counter() - t0) * 1e3)
        for frac in (0.1, 0.01):
            items = rng.choice(V, int(frac * V), replace=False)
            E = sp.csr_matrix((np.ones(B * 50, np.float32), (np.repeat(np.arange(B), 50), rng.integers(0, V, B * 50))),
                              shape=(B, V))
            t0 = time.perf_counter()
            filt = RankFilter.build(V, B, items=items, exclude=E)
            canon = (time.perf_counter() - t0) * 1e3
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng._compact(filt.shard_ids(V, 0, 1))
            torch.cuda.synchronize()
            build = (time.perf_counter() - t0) * 1e3
            legs["frac_%g_excl50" % frac] = dict(timed(eng, B, k, filt, args.iters), eligible=int(items.size),
                                                 canonicalise_ms=canon, compact_build_ms=build)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
