"""Ranking metrics from the ranks of the held-out items (SURVEY 8(f)-2).

The reference's harness ranks the whole dense prediction matrix on the host and looks the gold items up in the
ranking (evaluation.py:70-164 ``RankingMetric`` / ``MRR`` / ``MAP`` / ``P`` on top of ``argtopk``, 202-240
``evaluate``; arithmetic in rank_metrics_with_std.py:13-40, 108-154).  Every one of those metrics is a function of
the *ranks of the gold items* alone, so the device only has to count, per gold item, the items scored above it
(``aae_rank_counts``); this module turns those ranks into the same (mean, std) pairs:

  MRR@k : 1 / (best gold rank) if that rank <= k else 0          (rank_metrics_with_std.py:13-40)
  P@k   : (# gold ranks <= k) / k                                 (evaluation.py:146-164)
  MAP@k : mean over gold ranks r_i <= k (ascending) of i / r_i    (rank_metrics_with_std.py:108-131), 0 without hits
k = None (the reference's unbounded ``mrr`` / ``map``): every gold item counts.
"""
import re

import numpy as np


def parse_metric(m):
    """'mrr@5' / 'map' / 'P@1' (the keys of evaluation.py:166-180) or a reference metric object (class MRR / MAP / P
    with a ``k`` attribute) -> (kind, k)."""
    if isinstance(m, str):
        mm = re.fullmatch(r"(mrr|map|p)(?:@(\d+))?", m.strip().lower())
        if not mm:
            raise KeyError(m)
        return mm.group(1), (int(mm.group(2)) if mm.group(2) else None)
    kind = type(m).__name__.lower()
    if kind not in ("mrr", "map", "p"):
        raise KeyError("unsupported ranking metric %r" % (m,))
    return kind, getattr(m, "k", None)


def per_row_metric(gold_indptr, ranks, kind, k, n_items):
    """Per-row values of one metric; ``ranks`` (1-based) is aligned with the gold CSR entries.  Rank 0 means "not in
    the ranked list" (a gold item a candidate filter leaves out): it sorts after every ranked gold item of its row and
    is never a hit.  ``n_items`` is the length of the ranked list (the denominator of P without k)."""
    gold_indptr = np.asarray(gold_indptr, dtype=np.int64)
    n = gold_indptr.shape[0] - 1
    ranks = np.asarray(ranks, dtype=np.int64)
    rows = np.repeat(np.arange(n), np.diff(gold_indptr))
    absent = ranks <= 0
    order = np.lexsort((np.where(absent, np.iinfo(np.int64).max, ranks), rows))
    r, rows, absent = ranks[order].astype(np.float64), rows[order], absent[order]
    pos = np.arange(r.shape[0]) - gold_indptr[rows] + 1            # i of the i-th best gold item of its row
    hit = ~absent if k is None else (~absent & (r <= k))
    out = np.zeros(n, dtype=np.float64)
    if kind == "mrr":
        first = pos == 1
        sel = first & hit
        out[rows[sel]] = 1.0 / r[sel]
    elif kind == "p":
        denom = float(n_items if k is None else k)
        if denom:                   # 0: an empty list (no eligible item), which has no hit
            np.add.at(out, rows[hit], 1.0 / denom)
    elif kind == "map":
        num = np.zeros(n, dtype=np.float64)
        cnt = np.zeros(n, dtype=np.float64)
        np.add.at(num, rows[hit], pos[hit] / r[hit])
        np.add.at(cnt, rows[hit], 1.0)
        nz = cnt > 0
        out[nz] = num[nz] / cnt[nz]
    else:
        raise KeyError(kind)
    return out


def metrics_from_ranks(gold_indptr, ranks, metrics, n_items):
    """[(mean, std)] in the order of ``metrics`` -- what evaluation.py:202-240 ``evaluate`` returns."""
    out = []
    for m in metrics:
        kind, k = parse_metric(m)
        v = per_row_metric(gold_indptr, ranks, kind, k, n_items)
        out.append((float(v.mean()), float(v.std())))
    return out
