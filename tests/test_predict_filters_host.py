"""Host side of candidate-restricted ranking (``predict_topk(..., items=, exclude=)``): canonicalisation of the two
arguments, the input errors, the per-shard id tables, and the numpy statement of the semantics that the GPU tests
compare the kernels against."""
import numpy as np
import pytest
import scipy.sparse as sp

FLT_MAX = np.finfo(np.float32).max


def rank_reference(logits, known, k, items=None, exclude=None, mask_known=True, full=False):
    """The semantics of a filtered ranking, row by row.

    ``logits`` [n, V]; ``known`` [n, V] 0/1, dense or scipy sparse (the query sets); ``items`` eligible ids or boolean
    mask (None: all); ``exclude`` [n, V] 0/1, dense or sparse (None: none).  Ineligible items and excluded (row, item)
    pairs are never returned.  With ``mask_known`` a known item that is eligible and not excluded scores -FLT_MAX
    (below every unknown item).  Order: descending score, ties by lower item id.  Width: k (``full=False``), else A =
    number of eligible items for ``k=None`` or min(k, A).  Short rows are padded with (-1, -inf).  Returns (ids int64,
    scores float32)."""
    logits = np.asarray(logits, dtype=np.float32)
    n, V = logits.shape
    elig = np.ones(V, dtype=bool)
    if items is not None:
        items = np.asarray(items)
        elig = items.copy() if items.dtype == np.bool_ else np.isin(np.arange(V), items)
    A = int(elig.sum())
    width = (A if k is None else min(k, A)) if full else k
    ids = np.full((n, width), -1, dtype=np.int64)
    val = np.full((n, width), -np.inf, dtype=np.float32)
    known = sp.csr_matrix(known)
    ex = sp.csr_matrix((n, V)) if exclude is None else sp.csr_matrix(exclude)
    ex.eliminate_zeros()
    known.eliminate_zeros()
    for r in range(n):
        s = logits[r].copy()
        if mask_known:
            s[known.indices[known.indptr[r]:known.indptr[r + 1]]] = -FLT_MAX
        ok = elig.copy()
        ok[ex.indices[ex.indptr[r]:ex.indptr[r + 1]]] = False
        cand = np.flatnonzero(ok)
        if cand.size > width > 0:       # keep the `width` best and everything tied with the last of them
            kth = np.partition(s[cand], cand.size - width)[cand.size - width]
            cand = cand[s[cand] >= kth]
        order = cand[np.lexsort((cand, -s[cand].astype(np.float64)))][:width]
        ids[r, :order.size] = order
        val[r, :order.size] = s[order]
    return ids, val


# ---------------------------------------------------------------------------------------------- canonicalisation
def test_items_as_ids_and_as_mask_agree():
    from aaerec_b200.filters import canonical_items
    V = 10
    ids = canonical_items([7, 2, 2, 9, 0], V)
    assert ids.dtype == np.int32 and ids.tolist() == [0, 2, 7, 9]
    mask = np.zeros(V, dtype=bool)
    mask[[0, 2, 7, 9]] = True
    assert canonical_items(mask, V).tolist() == [0, 2, 7, 9]
    blocked = ~mask
    assert canonical_items(~blocked, V).tolist() == [0, 2, 7, 9]
    assert canonical_items(np.array([], dtype=np.int64), V).size == 0


def test_items_covering_every_item_is_no_restriction():
    from aaerec_b200.filters import canonical_items, RankFilter
    V = 6
    assert canonical_items(np.arange(V)[::-1], V) is None
    assert canonical_items(np.ones(V, dtype=bool), V) is None
    assert RankFilter.build(V, 3, items=np.arange(V)) is None
    assert RankFilter.build(V, 3) is None
    assert RankFilter.build(V, 3, exclude=sp.csr_matrix((3, V))) is None     # excludes nothing


def test_exclude_is_canonicalised():
    from aaerec_b200.filters import canonical_exclude
    n, V = 3, 8
    # duplicates (summed), an explicit zero (dropped), unsorted columns, COO input
    rows = np.array([0, 0, 0, 2, 2, 1])
    cols = np.array([5, 1, 5, 7, 3, 4])
    data = np.array([1, 1, 1, 1, 1, 0], dtype=np.float32)
    X = canonical_exclude(sp.coo_matrix((data, (rows, cols)), shape=(n, V)), n, V)
    assert X.indptr.tolist() == [0, 2, 2, 4]
    assert X.indices.tolist() == [1, 5, 3, 7]
    assert X.indices.dtype == np.int32 and X.indptr.dtype == np.int32
    assert np.all(X.data == 1)


def test_rows_slice_keeps_items_and_slices_exclusions():
    from aaerec_b200.filters import RankFilter
    n, V = 4, 10
    ex = sp.csr_matrix(np.eye(n, V))
    f = RankFilter.build(V, n, items=[1, 2, 3], exclude=ex)
    g = f.rows(1, 3)
    assert g.items is f.items
    assert g.exclude.shape == (2, V) and g.exclude.indices.tolist() == [1, 2]


@pytest.mark.parametrize("items, msg", [
    (np.array([0, 10]), "outside"),
    (np.array([-1, 3]), "outside"),
    (np.ones(9, dtype=bool), "length"),
    (np.ones(11, dtype=bool), "length"),
    (np.zeros((2, 5), dtype=np.int64), "1-D"),
    (np.array([0.5, 2.0]), "dtype"),
])
def test_bad_items_raise_value_error(items, msg):
    from aaerec_b200.filters import RankFilter
    with pytest.raises(ValueError, match=msg):
        RankFilter.build(10, 4, items=items)


@pytest.mark.parametrize("shape", [(3, 10), (4, 9), (5, 11)])
def test_exclude_of_wrong_shape_raises_value_error(shape):
    from aaerec_b200.filters import RankFilter
    with pytest.raises(ValueError, match="shape"):
        RankFilter.build(10, 4, exclude=sp.csr_matrix(shape))


def test_dense_exclude_raises_value_error():
    from aaerec_b200.filters import RankFilter
    with pytest.raises(ValueError, match="sparse"):
        RankFilter.build(10, 4, exclude=np.zeros((4, 10)))


# ---------------------------------------------------------------------------------------------- shard id tables
@pytest.mark.parametrize("world", [1, 2, 3])
def test_shard_tables_partition_the_eligible_set(world):
    from aaerec_b200.filters import RankFilter
    from aaerec_b200.dist import shard_range
    V = 100
    rng = np.random.default_rng(world)
    items = rng.choice(V, 30, replace=False)
    f = RankFilter.build(V, 2, items=items)
    parts = []
    for r in range(world):
        lo, hi = shard_range(V, r, world)
        ids = f.shard_ids(V, r, world)
        assert ids is not None and ids.dtype == np.int32
        assert np.all(np.diff(ids) > 0) and np.all((ids >= lo) & (ids < hi))
        parts.append(ids)
    assert np.concatenate(parts).tolist() == sorted(items.tolist())


def test_shard_tables_empty_and_full_shards():
    from aaerec_b200.filters import RankFilter
    V, world = 90, 3                  # shards [0,30) [30,60) [60,90)
    items = np.r_[np.arange(0, 30), np.arange(70, 75)]
    f = RankFilter.build(V, 1, items=items)
    assert f.shard_ids(V, 0, world) is None                   # every item of shard 0 eligible: no table
    assert f.shard_ids(V, 1, world).size == 0                 # no eligible item in shard 1
    assert f.shard_ids(V, 2, world).tolist() == list(range(70, 75))
    assert f.n_eligible(V) == 35
    # exclusions only: every shard ranks all of its items
    g = RankFilter.build(V, 1, exclude=sp.csr_matrix(([1.0], ([0], [5])), shape=(1, V)))
    assert all(g.shard_ids(V, r, world) is None for r in range(world))
    assert g.n_eligible(V) == V


# ---------------------------------------------------------------------------------------------- the semantics
def test_reference_pads_short_rows():
    logits = np.array([[0.1, 0.9, 0.5, 0.3]], dtype=np.float32)
    known = np.zeros_like(logits)
    ids, val = rank_reference(logits, known, 3, items=[1, 3])
    assert ids.tolist() == [[1, 3, -1]]
    assert val[0, :2].tolist() == [np.float32(0.9), np.float32(0.3)] and val[0, 2] == -np.inf


def test_reference_known_items():
    logits = np.array([[0.1, 0.9, 0.5, 0.3, 0.7]], dtype=np.float32)
    known = np.array([[0, 1, 0, 0, 1]])
    # item 1 known and eligible: at the bottom, still returned; item 4 known and ineligible: never returned
    ids, val = rank_reference(logits, known, 4, items=[0, 1, 2, 3])
    assert ids.tolist() == [[2, 3, 0, 1]]
    assert val[0, 3] == -FLT_MAX
    # without mask_known the known item ranks by its score
    ids, _ = rank_reference(logits, known, 4, items=[0, 1, 2, 3], mask_known=False)
    assert ids.tolist() == [[1, 2, 3, 0]]


def test_reference_exclusion_that_is_also_known():
    logits = np.array([[0.1, 0.9, 0.5, 0.3], [0.4, 0.2, 0.8, 0.6]], dtype=np.float32)
    known = np.array([[1, 0, 0, 0], [0, 0, 1, 0]])
    exclude = np.array([[1, 1, 0, 0], [0, 0, 0, 0]])     # row 0: item 0 known and excluded, item 1 excluded
    ids, val = rank_reference(logits, known, 4, exclude=exclude)
    assert ids.tolist() == [[2, 3, -1, -1], [3, 0, 1, 2]]
    assert val[1, 3] == -FLT_MAX and np.all(val[0, 2:] == -np.inf)


def test_reference_ties_go_to_lower_id_and_full_width():
    logits = np.array([[0.5, 0.5, 0.7, 0.5, 0.5]], dtype=np.float32)
    known = np.zeros_like(logits)
    ids, _ = rank_reference(logits, known, None, items=[4, 3, 1, 2], full=True)
    assert ids.tolist() == [[2, 1, 3, 4]]
    ids, _ = rank_reference(logits, known, 3, items=[4, 3, 1, 2], full=True)
    assert ids.tolist() == [[2, 1, 3]]
    ids, _ = rank_reference(logits, known, 9, items=[4, 3, 1, 2], full=True)
    assert ids.shape == (1, 4)
