"""Host side of candidate-restricted evaluation (``evaluate_topk(..., items=, exclude=)`` / ``gold_ranks``): the
metrics of rank-0 ("not in the list") gold items against the oracle's metric arithmetic on explicit filtered lists,
the returnable-gold mask, and the input errors."""
import types

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import aae_oracle as O
from test_predict_filters_host import rank_reference


def _old_per_row_metric(gold_indptr, ranks, kind, k, n_items):
    """per_row_metric as it was before rank 0 had a meaning: ranks >= 1 must give exactly these values."""
    gold_indptr = np.asarray(gold_indptr, dtype=np.int64)
    n = gold_indptr.shape[0] - 1
    ranks = np.asarray(ranks, dtype=np.int64)
    rows = np.repeat(np.arange(n), np.diff(gold_indptr))
    order = np.lexsort((ranks, rows))
    r, rows = ranks[order].astype(np.float64), rows[order]
    pos = np.arange(r.shape[0]) - gold_indptr[rows] + 1
    hit = np.ones(r.shape[0], dtype=bool) if k is None else (r <= k)
    out = np.zeros(n, dtype=np.float64)
    if kind == "mrr":
        sel = (pos == 1) & hit
        out[rows[sel]] = 1.0 / r[sel]
    elif kind == "p":
        np.add.at(out, rows[hit], 1.0 / float(n_items if k is None else k))
    elif kind == "map":
        num = np.zeros(n, dtype=np.float64)
        cnt = np.zeros(n, dtype=np.float64)
        np.add.at(num, rows[hit], pos[hit] / r[hit])
        np.add.at(cnt, rows[hit], 1.0)
        nz = cnt > 0
        out[nz] = num[nz] / cnt[nz]
    return out


def _case(seed, n=40, V=60, frac=0.6):
    """Scores with exact ties (a few distinct integer values), known items, an eligible set, exclusions that cover
    a known gold item, and a row whose gold are all unreturnable."""
    rng = np.random.default_rng(seed)
    Z = rng.integers(0, 6, size=(n, V)).astype(np.float32)
    X = (rng.random((n, V)) < 0.1).astype(np.float32)
    Y = (rng.random((n, V)) < 0.12).astype(np.float32)
    Y[:, 0] = 1
    X[1, 0] = 1                                      # row 1: gold item 0 is known ...
    elig = rng.random(V) < frac
    elig[0] = True
    E = (rng.random((n, V)) < 0.08).astype(np.float32)
    E[1, 0] = 1                                      # ... and excluded
    Y[2] = 0
    Y[2, 1:4] = 1
    elig[1] = False                                  # row 2: gold 1 ineligible, gold 2 and 3 excluded
    E[2, 2:4] = 1
    return Z, sp.csr_matrix(X), sp.csr_matrix(Y), np.flatnonzero(elig), sp.csr_matrix(E)


def _filtered_lists_and_ranks(Z, X, Y, items, E):
    """The k=None filtered list of every row (rank_reference), and each gold's rank: 1 + its position there, or 0."""
    ids, _ = rank_reference(Z, X, None, items=items, exclude=E, full=True)
    ranks = np.zeros(Y.nnz, dtype=np.int64)
    for r in range(Y.shape[0]):
        pos = {int(i): j for j, i in enumerate(ids[r]) if i >= 0}
        for e in range(Y.indptr[r], Y.indptr[r + 1]):
            ranks[e] = pos.get(int(Y.indices[e]), -1) + 1
    return ids, ranks


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_metrics_of_rank_zero_match_the_oracle_on_the_filtered_lists(seed):
    from aaerec_b200.ranking import metrics_from_ranks
    Z, X, Y, items, E = _case(seed)
    ids, ranks = _filtered_lists_and_ranks(Z, X, Y, items, E)
    A = items.size
    assert ranks[Y.indptr[2]:Y.indptr[3]].tolist() == [0, 0, 0]
    assert ranks[Y.indptr[1]] == 0
    Yd = Y.toarray()
    for k in (1, 3, 10, A - 1, A, A + 7, None):         # k > A: the list is shorter than k
        names = [kind if k is None else "%s@%d" % (kind, k) for kind in ("mrr", "map", "p")]
        got = metrics_from_ranks(Y.indptr, ranks, names, A)
        np.testing.assert_allclose(np.array(got), np.array(filtered_metrics(ids, Yd, A, names)), rtol=1e-12,
                                   atol=1e-15, err_msg=str(names))


def test_an_empty_list_scores_zero():
    """No eligible item: every gold has rank 0 and the list length is 0 (P without k has no hit to divide)."""
    from aaerec_b200.ranking import metrics_from_ranks
    indptr = np.array([0, 2, 2, 5])
    got = metrics_from_ranks(indptr, np.zeros(5, np.int64), ["mrr", "map", "p", "p@3", "mrr@1"], 0)
    assert got == [(0.0, 0.0)] * 5


@pytest.mark.parametrize("kind", ["mrr", "map", "p"])
@pytest.mark.parametrize("k", [None, 1, 5, 50])
def test_ranks_of_one_or_more_give_the_metrics_of_before(kind, k):
    from aaerec_b200.ranking import per_row_metric
    rng = np.random.default_rng(7)
    n, V = 200, 300
    indptr = np.concatenate(([0], np.cumsum(rng.integers(0, 9, n))))
    ranks = rng.integers(1, V + 1, indptr[-1])
    np.testing.assert_array_equal(per_row_metric(indptr, ranks, kind, k, V),
                                  _old_per_row_metric(indptr, ranks, kind, k, V))


def test_returnable_mask_is_the_dense_statement():
    from aaerec_b200.filters import RankFilter
    for seed in range(4):
        Z, X, Y, items, E = _case(seed, n=50, V=80, frac=(0.3, 0.9, 1.0, 0.0)[seed])
        n, V = Y.shape
        filt = RankFilter.build(V, n, items=items, exclude=E)
        got = filt.returnable(Y.indptr, Y.indices)
        elig = np.isin(np.arange(V), items)
        rows = np.repeat(np.arange(n), np.diff(Y.indptr))
        want = elig[Y.indices] & (E.toarray()[rows, Y.indices] == 0)
        np.testing.assert_array_equal(got, want)
        # each argument alone
        np.testing.assert_array_equal(RankFilter(filt.items, None).returnable(Y.indptr, Y.indices),
                                      elig[Y.indices])
        np.testing.assert_array_equal(RankFilter(None, filt.exclude).returnable(Y.indptr, Y.indices),
                                      E.toarray()[rows, Y.indices] == 0)


def _host_model(V):
    """An AdversarialAutoEncoder whose engine only knows V: enough to reach the argument checks, which come before
    any device work."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    m = AdversarialAutoEncoder.__new__(AdversarialAutoEncoder)
    m.engine = types.SimpleNamespace(V=V, Vloc=V, world=1)
    return m


@pytest.mark.parametrize("method", ["gold_ranks", "evaluate_topk"])
def test_bad_arguments_raise_value_error(method):
    V, n = 50, 6
    m = _host_model(V)
    X = sp.csr_matrix(np.eye(n, V, dtype=np.float32))
    Y = sp.csr_matrix(np.eye(n, V, k=1, dtype=np.float32))

    def run(Yq=Y, **kw):
        if method == "gold_ranks":
            return m.gold_ranks(X, Yq, **kw)
        return m.evaluate_topk(X, Yq, ["mrr"], **kw)
    with pytest.raises(ValueError, match="outside"):
        run(items=[0, V])
    with pytest.raises(ValueError, match="length"):
        run(items=np.ones(V + 1, dtype=bool))
    with pytest.raises(ValueError, match="1-D"):
        run(items=np.zeros((2, 2), dtype=np.int64))
    with pytest.raises(ValueError, match="shape"):
        run(exclude=sp.csr_matrix((n + 1, V)))
    with pytest.raises(ValueError, match="sparse"):
        run(exclude=np.zeros((n, V)))
    with pytest.raises(ValueError, match="gold matrix has shape"):
        run(Yq=sp.csr_matrix((n, V + 1)), items=[1, 2])
    with pytest.raises(ValueError, match="gold matrix has shape"):
        run(Yq=sp.csr_matrix((n + 1, V)))


def filtered_metrics(ids, Yd, A, metrics):
    """The oracle's metric arithmetic (_reciprocal_rank, _average_precision, precision) on explicit ranked lists:
    ``ids`` [n, w] item ids with -1 padding, ``Yd`` [n, V] dense gold, ``A`` the list length (P without k).
    [(mean, std)] per metric name."""
    rel = np.where(ids >= 0, Yd[np.arange(ids.shape[0])[:, None], np.maximum(ids, 0)], 0)
    out = []
    for name in metrics:
        kind, _, kk = name.lower().partition("@")
        k = int(kk) if kk else None
        rk = rel if k is None else rel[:, :k]
        if kind == "mrr":
            v = np.array([O._reciprocal_rank(x) for x in rk])
        elif kind == "map":
            v = np.array([O._average_precision(x) for x in rk])
        else:
            v = (rk > 0).sum(axis=1) / float(A if k is None else k)
        out.append((float(v.mean()), float(v.std())))
    return out


def test_filtered_metrics_helper_is_the_oracle_without_a_filter():
    """filtered_metrics on an unfiltered ranking == the oracle's evaluate (which ranks the dense prediction)."""
    rng = np.random.default_rng(3)
    n, V = 30, 50
    Z = rng.random((n, V))
    Yd = (rng.random((n, V)) < 0.1).astype(np.float32)
    ids = np.argsort(-Z, axis=1, kind="stable")
    metrics = ["mrr@5", "map@10", "p@3", "mrr", "map", "p"]
    got = filtered_metrics(ids, Yd, V, metrics)
    want = O.evaluate(Yd, Z, metrics)
    np.testing.assert_allclose(np.array(got), np.array(want), rtol=1e-12, atol=0)
