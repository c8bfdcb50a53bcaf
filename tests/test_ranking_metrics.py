"""Ranking metrics (SURVEY 8(f)-2): the oracle's restatement against the reference's doctest vectors and against the
reference itself, and the product's rank-based arithmetic (aaerec_b200/ranking.py) against the oracle."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from helpers import GOLDEN
from oracle import aae_oracle as O

METRICS = ["mrr@5", "mrr@10", "map@5", "map@20", "p@5", "p@20", "P@1", "mrr", "map"]


def test_metric_doctest_vectors():
    # evaluation.py:97-107 (MRR), 125-136 (MAP), 151-156 (P)
    Yt = np.array([[1, 0, 0], [0, 0, 1]])
    Yp = np.array([[0.2, 0.3, 0.1], [0.2, 0.5, 0.7]])
    assert O.relevance_in_rank_order(Yt, Yp, 2).tolist() == [[0, 1], [1, 0]]        # evaluation.py:83-87
    assert O.evaluate(Yt, Yp, ["mrr@2"])[0] == (0.75, 0.25)
    assert O.evaluate(Yt, Yp, ["map@2"])[0] == (0.75, 0.25)
    Yt = np.array([[1, 0, 1], [1, 0, 1]])
    Yp = np.array([[0.4, 0.3, 0.2], [0.4, 0.3, 0.2]])
    assert O.evaluate(Yt, Yp, ["mrr@3"])[0] == (1.0, 0.0)
    Yt = np.array([[1, 0, 1], [1, 1, 1]])
    m, s = O.evaluate(Yt, Yp, ["map@3"])[0]
    assert abs(m - 0.9166666666666666) < 1e-12 and abs(s - 0.08333333333333337) < 1e-12
    Yt = np.array([[1, 0, 1, 0], [1, 0, 1, 0]])
    Yp = np.array([[0.2, 0.3, 0.1, 0.05], [0.2, 0.5, 0.7, 0.05]])
    assert O.evaluate(Yt, Yp, ["p@2"])[0] == (0.5, 0.0)
    assert O.evaluate(Yt, Yp, ["p@4"])[0] == (0.5, 0.0)


def _random_case(seed, n=40, V=300):
    rs = np.random.RandomState(seed)
    X = (rs.rand(n, V) < 0.03).astype(np.float32)
    Y = ((rs.rand(n, V) < 0.02) & (X == 0)).astype(np.float32)
    Y[3] = 0                                              # a row without gold items
    pred = rs.rand(n, V)                                  # distinct float64 scores: no ties among unknown items
    # the reference zeroes the known items AFTER min-max scaling, so they tie with the row's lowest-scored item
    # (evaluation.py:193-197); keep that one reference-side tie out of the gold set
    Y[np.arange(n), pred.argmin(axis=1)] = 0
    return X, Y, pred


def reference_metrics(ref, case_seed=0):
    """The reference's (mean, std) of every metric on ``_random_case(case_seed)`` (evaluation.py:183-199, 202-240)."""
    X, Y, pred = _random_case(case_seed)
    masked = ref.evaluation.remove_non_missing(pred, sp.csr_matrix(X), copy=True)
    return ref.evaluation.evaluate(sp.csr_matrix(Y), masked, METRICS)


def test_oracle_metrics_match_reference():
    """Against the reference itself when its package is importable, else against what it computed on the same case,
    stored by oracle/make_golden.py in tests/golden/metrics_reference.npz."""
    from oracle import reference_loader as RL
    path = os.path.join(GOLDEN, "metrics_reference.npz")
    if RL.reference_available():
        want = reference_metrics(RL.load_reference())
    elif os.path.exists(path):
        g = np.load(path)
        assert [str(m) for m in g["metrics"]] == METRICS
        want = [tuple(row) for row in g["want"]]
    else:
        pytest.skip("neither the reference package nor its stored metrics (oracle/make_golden.py) are present")
    X, Y, pred = _random_case(0)
    got = O.evaluate(Y, O.remove_non_missing(pred, X), METRICS)
    for (a, b), (c, d) in zip(got, want):
        assert abs(a - c) < 1e-12 and abs(b - d) < 1e-12


def test_rank_based_metrics_match_oracle():
    """metrics_from_ranks on ranks computed the way aae_rank_counts defines them (count of unknown items scored
    higher; known items at the bottom) == the oracle's dense evaluate."""
    from aaerec_b200.ranking import metrics_from_ranks, parse_metric
    assert parse_metric("P@1") == ("p", 1) and parse_metric("map") == ("map", None)
    for seed in (1, 2):
        X, Y, pred = _random_case(seed)
        masked = O.remove_non_missing(pred, X)
        want = O.evaluate(Y, masked, METRICS)
        Yc = sp.csr_matrix(Y)
        z = np.where(X > 0, -np.inf, pred)                 # logits/probabilities with the known items at the bottom
        ranks = np.zeros(Yc.nnz, dtype=np.int64)
        for r in range(Yc.shape[0]):
            for p in range(Yc.indptr[r], Yc.indptr[r + 1]):
                g = Yc.indices[p]
                ranks[p] = 1 + int(np.sum(z[r] > z[r, g])) + int(np.sum((z[r] == z[r, g]) & (np.arange(z.shape[1]) < g)))
        got = metrics_from_ranks(Yc.indptr, ranks, METRICS, X.shape[1])
        for (a, b), (c, d) in zip(got, want):
            assert abs(a - c) < 1e-9 and abs(b - d) < 1e-9, (got, want)
