"""Candidate restriction of ``predict_topk``: which items may be returned at all (``items``) and which (row, item)
pairs never (``exclude``).

``items`` is a 1-D array of item ids in [0, V) (duplicates allowed) or a boolean mask of length V; a block list is
``items=~blocked``.  ``exclude`` is a scipy sparse [n, V] matrix whose nonzero entries are never returned for their
row.  Both are canonicalised once per call on the host: the eligible set becomes a sorted, unique int32 id table,
``exclude`` a CSR with duplicates summed, zeros dropped and sorted columns.  The engines rank each item shard's
eligible rows as a compact matrix (``AAEEngine.topk(..., filt=)``), so the ranking itself never sees an ineligible
item."""
import numpy as np
import scipy.sparse as sp

from .dist import shard_range


def canonical_items(items, V):
    """Eligible items -> sorted unique int32 ids, or None when every one of the V items is eligible."""
    a = np.asarray(items)
    if a.ndim != 1:
        raise ValueError("items must be 1-D (item ids or a boolean mask of length n_items), got shape %s" % (a.shape,))
    if a.dtype == np.bool_:
        if a.shape[0] != V:
            raise ValueError("boolean items mask has length %d, expected n_items = %d" % (a.shape[0], V))
        ids = np.flatnonzero(a)
    else:
        if a.size and not np.issubdtype(a.dtype, np.integer):
            raise ValueError("items must hold integer item ids or booleans, got dtype %s" % a.dtype)
        if a.size and (int(a.min()) < 0 or int(a.max()) >= V):
            raise ValueError("items holds ids outside [0, %d)" % V)
        ids = np.unique(a)
    ids = ids.astype(np.int32)
    return None if ids.size == V else ids


def canonical_exclude(exclude, n, V):
    """Per-row exclusions -> CSR [n, V] (int32 indptr/indices, duplicates summed, zeros dropped, sorted columns), or
    None when it excludes nothing."""
    if not sp.issparse(exclude):
        raise ValueError("exclude must be a scipy sparse [n, n_items] matrix")
    if exclude.shape != (n, V):
        raise ValueError("exclude has shape %s, expected (%d, %d)" % (exclude.shape, n, V))
    X = sp.csr_matrix(exclude, copy=True)
    X.sum_duplicates()
    X.eliminate_zeros()
    X.sort_indices()
    if X.nnz == 0:
        return None
    return sp.csr_matrix((np.ones(X.nnz, np.float32), X.indices.astype(np.int32), X.indptr.astype(np.int32)),
                         shape=X.shape)


class RankFilter(object):
    """Canonical ``items`` / ``exclude`` of one ranking call (see the module docstring)."""

    def __init__(self, items, exclude):
        self.items = items          # sorted unique int32 ids, or None: every item is eligible
        self.exclude = exclude      # CSR of the rows it covers, or None: no exclusions

    @classmethod
    def build(cls, V, n, items=None, exclude=None):
        """Validate and canonicalise; None when the call is not restricted at all (the unfiltered path runs)."""
        ids = None if items is None else canonical_items(items, V)
        ex = None if exclude is None else canonical_exclude(exclude, n, V)
        if ids is None and ex is None:
            return None
        return cls(ids, ex)

    def shard_ids(self, V, rank, world):
        """Eligible global ids of item shard ``rank`` of ``world`` (int32, ascending; empty when none is), or None
        when every item of the shard is eligible."""
        lo, hi = shard_range(V, rank, world)
        if self.items is None:
            return None
        a, b = np.searchsorted(self.items, [lo, hi])
        ids = self.items[a:b]
        return None if ids.size == hi - lo else ids

    def rows(self, start, end):
        """The same filter for query rows [start, end)."""
        return RankFilter(self.items, None if self.exclude is None else self.exclude[start:end])

    def n_eligible(self, V):
        return V if self.items is None else int(self.items.size)

    def returnable(self, indptr, indices):
        """bool mask of the entries of a CSR (rows = the query rows of this filter, sorted columns) whose item may be
        returned for its row: eligible and not excluded.  The gold items of ``evaluate_topk`` that are not returnable
        are not in the ranked list."""
        indptr = np.asarray(indptr, dtype=np.int64)
        indices = np.asarray(indices, dtype=np.int64)
        ok = np.ones(indices.size, dtype=bool)
        if self.items is not None:
            pos = np.searchsorted(self.items, indices)
            ok &= pos < self.items.size
            ok[ok] = self.items[pos[ok]] == indices[ok]
        if self.exclude is not None:
            # intersection of the sorted rows of both CSRs, as ascending (row, item) keys
            V, ex = self.exclude.shape[1], self.exclude
            key = np.repeat(np.arange(indptr.size - 1, dtype=np.int64), np.diff(indptr)) * V + indices
            ekey = np.repeat(np.arange(ex.shape[0], dtype=np.int64), np.diff(ex.indptr)) * V + ex.indices
            pos = np.searchsorted(ekey, key)
            hit = pos < ekey.size
            hit[hit] = ekey[pos[hit]] == key[hit]
            ok &= ~hit
        return ok
