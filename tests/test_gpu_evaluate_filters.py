"""GPU tests of candidate-restricted evaluation (``gold_ranks`` / ``evaluate_topk(..., items=, exclude=)``): the ranks
against the positions in the list ``predict_topk(X, None, items=, exclude=)`` returns (integer equality: both score
the same compact copy with the same kernel), the metrics against the oracle's arithmetic on the oracle's logits,
``aae_rank_counts_filtered`` against an int64 count, the sibling recommenders, and the encoder exchange."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from test_evaluate_filters_host import filtered_metrics
from test_predict_filters_host import rank_reference, FLT_MAX

pytestmark = pytest.mark.gpu

METRICS = ["mrr@5", "mrr@10", "map@5", "map@20", "p@5", "p@20", "P@1", "mrr", "map", "p"]


def _sets(n, V, mean_len, seed):
    from aaerec_b200.synth import synth_sets
    return synth_sets(n, V, mean_len, seed=seed)


@functools.lru_cache(maxsize=2)
def _tied_model(V, B=64):
    """A model whose output layer repeats rows: items i + 3001 and i + 16387 have the weights and bias of item i for
    i < 3000, so exact score ties span columns and rank-count chunks."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from oracle import aae_oracle as O
    H, C = 100, 50
    params = O.init_params(V, H, C, seed=17)
    W, b = params["dec.lin3.weight"] * 8.0, params["dec.lin3.bias"].clone()
    src = torch.arange(0, 3000)
    for off in (3001, 16387):
        W[src + off] = W[src]
        b[src + off] = b[src]
    params["dec.lin3.weight"], params["dec.lin3.bias"] = W, b
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=B, n_epochs=1, verbose=False, impl="auto")
    model._build(V, C, params={k: v.clone() for k, v in params.items()})
    return model


def _gold(X, V, per_row, seed, extra=None):
    """Random gold items per row, including known ones (and the ids of ``extra`` [n] lists)."""
    rng = np.random.default_rng(seed)
    n = X.shape[0]
    rows, cols = [np.repeat(np.arange(n), per_row)], [rng.integers(0, V, n * per_row)]
    for r in range(n):
        kn = X.indices[X.indptr[r]:X.indptr[r + 1]][:2]
        rows.append(np.full(kn.size, r))
        cols.append(kn)
        if extra is not None:
            rows.append(np.full(len(extra[r]), r))
            cols.append(np.asarray(extra[r], dtype=np.int64))
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    Y = sp.csr_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(n, V))
    Y.data[:] = 1
    return Y


def _exclude(X, Y, V, n_rand, seed):
    """n_rand random exclusions per row, plus two known items and two gold items of the row."""
    rng = np.random.default_rng(seed)
    n = X.shape[0]
    rows, cols = [np.repeat(np.arange(n), n_rand)], [rng.integers(0, V, n * n_rand)]
    for r in range(n):
        c = np.concatenate((X.indices[X.indptr[r]:X.indptr[r + 1]][-2:], Y.indices[Y.indptr[r]:Y.indptr[r + 1]][:2]))
        rows.append(np.full(c.size, r))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    E = sp.csr_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(n, V))
    E.data[:] = 1
    return E


def _positions(ids, Y):
    """1 + the position of each gold entry of Y in its row of the ranked lists ``ids`` (-1 padding), 0 when absent."""
    n, V = Y.shape
    inv = np.zeros((n, V), dtype=np.int64)
    rows = np.broadcast_to(np.arange(n)[:, None], ids.shape)
    live = ids >= 0
    inv[rows[live], ids[live]] = np.broadcast_to(np.arange(ids.shape[1])[None, :] + 1, ids.shape)[live]
    grow = np.repeat(np.arange(n), np.diff(Y.indptr))
    return inv[grow, Y.indices]


CASES = ["all_but_one", "half", "one_percent", "exclusions_only", "empty"]


@pytest.mark.parametrize("V", [20000, 300000])
@pytest.mark.parametrize("case", CASES)
def test_gold_ranks_are_the_positions_in_the_filtered_full_ranking(V, case):
    model = _tied_model(V)
    n = 64 if V > 100000 else 128
    X = _sets(n, V, 12, seed=V % 97)
    rng = np.random.default_rng(11)
    items = {"all_but_one": np.delete(np.arange(V), V // 3), "half": np.sort(rng.choice(V, V // 2, replace=False)),
             "one_percent": np.sort(rng.choice(V, V // 100, replace=False)), "exclusions_only": None,
             "empty": np.zeros(0, dtype=np.int64)}[case]
    # gold among the tied items too (their twins rank next to them), and among the eligible ones
    el = np.arange(V) if items is None or items.size == 0 else items
    Y = _gold(X, V, 12, seed=3, extra=[[3001 + r, 16387 + r, r, el[r % el.size], el[(7 * r + 3) % el.size]]
                                      for r in range(n)])
    E = None if case == "empty" else _exclude(X, Y, V, 50, seed=4)
    indptr, ranks = model.gold_ranks(X, Y, batch_size=model.batch_size, items=items, exclude=E)
    np.testing.assert_array_equal(indptr, Y.indptr)
    if case == "empty":
        assert not ranks.any()
        assert all(v == (0.0, 0.0) for v in model.evaluate_topk(X, Y, METRICS, items=items))
        return
    ids = model.predict_topk(X, None, items=items, exclude=E)
    want = _positions(ids, Y)
    np.testing.assert_array_equal(ranks, want)
    assert (want == 0).any() and (want > 0).mean() > 0.05
    A = V if items is None else items.size
    got = model.evaluate_topk(X, Y, METRICS, batch_size=model.batch_size, items=items, exclude=E)
    np.testing.assert_allclose(np.array(got), np.array(filtered_metrics(ids, Y.toarray(), A, METRICS)), rtol=1e-12,
                               atol=1e-12)


def test_evaluate_topk_with_a_filter_matches_the_oracle_logits():
    """Metrics of the filtered lists stated in numpy on the oracle's logits, to 1e-6.  Gold items are drawn among
    items whose float64 logit is farther from every other item's than the fp32 rounding of the two computations (as in
    test_evaluate_topk_across_rank_count_chunks), so that both place them identically."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from oracle import aae_oracle as O
    V, H, C, n = 20000, 100, 50, 120
    params = O.init_params(V, H, C, seed=13)
    params["dec.lin3.weight"] = params["dec.lin3.weight"] * 8.0
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=50, n_epochs=1, verbose=False)
    model._build(V, C, params={k: v.clone() for k, v in params.items()})
    X = _sets(n, V, 12, seed=31)
    dense = X.toarray()
    oracle = O.OracleAAE({k: torch.as_tensor(v) for k, v in model.state_dict().items()}, n_code=C)
    Z = oracle.logits(dense).astype(np.float64)
    tol = 2e-5 * np.abs(Z).max(axis=1, keepdims=True) + 1e-6
    o = np.argsort(Z, axis=1)
    gap = np.diff(np.take_along_axis(Z, o, 1), axis=1)
    sep_sorted = np.minimum(np.c_[np.full((n, 1), np.inf), gap], np.c_[gap, np.full((n, 1), np.inf)]) > 4 * tol
    sep = np.zeros_like(sep_sorted)
    np.put_along_axis(sep, o, sep_sorted, 1)
    rs = np.random.RandomState(3)
    Yd = ((rs.rand(n, V) < 0.01) & (dense == 0) & sep).astype(np.float32)
    Y = sp.csr_matrix(Yd)
    items = np.sort(rs.choice(V, V // 4, replace=False))
    E = _exclude(X, Y, V, 50, seed=8)
    ids, _ = rank_reference(Z.astype(np.float32), X, None, items=items, exclude=E, full=True)
    want = filtered_metrics(ids, Yd, items.size, METRICS)
    got = model.evaluate_topk(X, Y, METRICS, batch_size=50, items=items, exclude=E)
    for name, (a, b), (c, d) in zip(METRICS, got, want):
        assert abs(a - c) < 1e-6 and abs(b - d) < 1e-6, (name, got, want)
    assert want[0][0] > 0


def test_unrestricting_filter_is_the_unfiltered_evaluation():
    model = _tied_model(20000)
    V = 20000
    X = _sets(100, V, 12, seed=5)
    Y = _gold(X, V, 10, seed=6)
    base = model.gold_ranks(X, Y)
    for kw in (dict(items=np.arange(V)), dict(items=np.ones(V, dtype=bool), exclude=sp.csr_matrix((100, V)))):
        got = model.gold_ranks(X, Y, **kw)
        np.testing.assert_array_equal(got[1], base[1])
        assert model.evaluate_topk(X, Y, METRICS, **kw) == model.evaluate_topk(X, Y, METRICS)


# ---- aae_rank_counts_filtered ---------------------------------------------------------------------------------------
def _csr_dev(lists):
    indptr = np.concatenate(([0], np.cumsum([len(x) for x in lists]))).astype(np.int32)
    indices = np.concatenate([np.asarray(x, dtype=np.int32) for x in lists] + [np.zeros(0, np.int32)])
    return torch.from_numpy(indptr).cuda(), torch.from_numpy(np.ascontiguousarray(indices)).cuda()


def _counts_filtered(S, Vloc, v_begin, table, known, excl, gold, zg, given):
    from aaerec_b200._native import call, ptr, AaeRankFilter
    import ctypes as C
    kp, ki = known if known is not None else (None, None)
    xp, xi = excl if excl is not None else (None, None)
    gp, gi = gold
    cnt = torch.full((gi.numel(),), -7, dtype=torch.int32, device="cuda")
    f = AaeRankFilter(ptr(table), ptr(xp), ptr(xi))
    call("aae_rank_counts_filtered", ptr(S), S.stride(0), S.shape[0], Vloc, v_begin, ptr(kp), ptr(ki), ptr(gp),
         ptr(gi), gi.numel(), ptr(zg), 1 if given else 0, ptr(cnt), None, C.byref(f))
    torch.cuda.synchronize()
    return cnt


def _reference_counts(S, T, known, excl, gold):
    """int64 statement: columns T (global ids); known ids -> -FLT_MAX, excluded ids -> -inf; for each gold g of row r
    with column c: #{columns with a higher score, or an equal one and a lower id}; NaN score and count 0 when g is not
    a column."""
    S = S.copy()
    counts, zs = [], []
    for r in range(S.shape[0]):
        s = S[r]
        s[np.isin(T, known[r])] = -FLT_MAX
        s[np.isin(T, excl[r])] = -np.inf
        for g in gold[r]:
            c = np.searchsorted(T, g)
            if c < T.size and T[c] == g:
                z = s[c]
                counts.append(int(((s > z) | ((s == z) & (T < g))).sum()))
                zs.append(z)
            else:
                counts.append(0)
                zs.append(np.nan)
    return np.array(counts, np.int64), np.array(zs, np.float32)


@pytest.mark.parametrize("layout", ["table", "no_table"])
def test_rank_counts_filtered_against_int64_count(layout):
    """A compact table with gaps over two column chunks, lds > Vloc, 0..40 gold per row (several gold groups), gold
    ids absent from the table, known and excluded ids inside and outside the table, scores in steps of 1/4 (ties
    everywhere); without a table (exclusions only) at v_begin != 0.  Then the table split into two (the two-pass
    item-shard protocol with gold_scores_given): the summed counts equal the single-table count."""
    rng = np.random.default_rng(5)
    V, B = 60000, 6
    if layout == "table":
        T = np.sort(rng.choice(V, 25000, replace=False)).astype(np.int32)
        v_begin = 0
    else:
        v_begin = 1000
        T = np.arange(v_begin, v_begin + 25000, dtype=np.int32)
    A = T.size
    S = (rng.integers(-4, 5, size=(B, A + 37)) / 4.0).astype(np.float32)
    n_gold = [0, 1, 8, 9, 20, 40]
    gold, known, excl = [], [], []
    for r in range(B):
        g_in = rng.choice(T, n_gold[r], replace=False)
        g_out = np.setdiff1d(rng.integers(0, V, 3), T)[:1] if n_gold[r] else np.zeros(0, np.int64)
        g = np.concatenate((g_in, g_out)).astype(np.int64)
        kn = np.unique(np.concatenate((rng.integers(0, V, 30), g_in[:2])))
        ex = np.setdiff1d(np.unique(np.concatenate((rng.choice(T, 40), rng.integers(0, V, 20)))), g)
        gold.append(g), known.append(kn), excl.append(ex)
    want, zwant = _reference_counts(S[:, :A], T, known, excl, gold)
    table = torch.from_numpy(T).cuda() if layout == "table" else None
    vb = 0 if layout == "table" else v_begin
    Sd = torch.from_numpy(S).cuda()
    zg = torch.empty(sum(len(g) for g in gold), dtype=torch.float32, device="cuda")
    cnt = _counts_filtered(Sd, A, vb, table, _csr_dev(known), _csr_dev(excl), _csr_dev(gold), zg, False)
    np.testing.assert_array_equal(cnt.cpu().numpy().astype(np.int64), want)
    np.testing.assert_array_equal(zg.cpu().numpy(), zwant)

    # two tables over the same columns: returnable gold only (every gold a column of one of them)
    gold_in = [g[np.isin(g, T)] for g in gold]
    want_in, _ = _reference_counts(S[:, :A], T, known, excl, gold_in)
    h = A // 2 + 123
    parts = [(0, h), (h, A)]
    gdev = _csr_dev(gold_in)
    n_in = sum(len(g) for g in gold_in)
    zsum = torch.zeros(n_in, dtype=torch.float32, device="cuda")
    shards = []
    for a, b in parts:
        Ss = torch.from_numpy(np.ascontiguousarray(S[:, a:b])).cuda()
        Ss = torch.cat((Ss, torch.zeros(B, 5, device="cuda")), 1)          # lds > Vloc
        tb = torch.from_numpy(T[a:b]).cuda() if layout == "table" else None
        z = torch.empty(n_in, dtype=torch.float32, device="cuda")
        _counts_filtered(Ss, b - a, 0 if layout == "table" else v_begin + a, tb, _csr_dev(known), _csr_dev(excl),
                         gdev, z, False)
        zsum += torch.nan_to_num(z, nan=0.0)
        shards.append((Ss, b - a, 0 if layout == "table" else v_begin + a, tb))
    total = torch.zeros(n_in, dtype=torch.int64, device="cuda")
    for Ss, n, vbs, tb in shards:
        total += _counts_filtered(Ss, n, vbs, tb, None, _csr_dev(excl), gdev, zsum, True).long()
    np.testing.assert_array_equal(total.cpu().numpy(), want_in)


def test_rank_counts_filtered_without_filter_is_rank_counts():
    """A NULL filter (both tables NULL) is aae_rank_counts."""
    rng = np.random.default_rng(9)
    B, Vloc = 3, 20000
    S = (rng.integers(-4, 5, size=(B, Vloc)) / 4.0).astype(np.float32)
    gold = [rng.choice(Vloc, 10, replace=False) for _ in range(B)]
    known = [rng.choice(Vloc, 10, replace=False) for _ in range(B)]
    T = np.arange(Vloc, dtype=np.int32)
    want, _ = _reference_counts(S, T, known, [np.zeros(0, np.int64)] * B, gold)
    zg = torch.empty(30, dtype=torch.float32, device="cuda")
    cnt = _counts_filtered(torch.from_numpy(S).cuda(), Vloc, 0, None, _csr_dev([np.sort(k) for k in known]), None,
                           _csr_dev(gold), zg, False)
    np.testing.assert_array_equal(cnt.cpu().numpy().astype(np.int64), want)


# ---- recommenders ---------------------------------------------------------------------------------------------------
class _Bags(object):
    def __init__(self, X, cond=None):
        self.X, self.cond = X, cond

    def tocsr(self):
        return self.X

    def size(self, dim=None):
        return self.X.shape[0]

    def get_attributes(self, keys):
        return [self.cond]


@pytest.mark.parametrize("kind", ["dae", "vae", "decoding"])
def test_sibling_recommenders_evaluate_their_own_rankings(kind):
    """DAE, VAE and Decoding recommenders: evaluate_topk, with and without a filter, == the metrics of their own
    predict_topk(k=None) lists (one batch of 200 rows, so that the VAE draws the same noise in both calls)."""
    V, n, D = 3000, 200, 16
    X = _sets(n, V, 10, seed=21)
    rng = np.random.default_rng(2)
    cond = rng.standard_normal((n, D)).astype(np.float32)
    bags = _Bags(X, cond)
    if kind == "dae":
        from aaerec_b200.dae import DAERecommender
        rec = DAERecommender(n_hidden=100, n_code=50, batch_size=256, n_epochs=1, verbose=False)
    elif kind == "vae":
        from aaerec_b200.vae import VAERecommender
        rec = VAERecommender(n_hidden=100, n_code=50, batch_size=256, n_epochs=1, verbose=False)
    else:
        from aaerec_b200.condition import ConditionList, PrecomputedEmbeddingCondition
        from aaerec_b200.decoding import DecodingRecommender
        rec = DecodingRecommender(ConditionList([("title", PrecomputedEmbeddingCondition(D))]), n_epochs=1,
                                  batch_size=256, n_hidden=100, verbose=False)
    rec.train(bags)
    Y = _gold(X, V, 8, seed=7)
    items = np.sort(rng.choice(V, V // 3, replace=False))
    E = _exclude(X, Y, V, 20, seed=3)
    for kw, A in ((dict(), V), (dict(items=items, exclude=E), items.size)):
        ids = rec.predict_topk(bags, None, **kw)
        got = rec.evaluate_topk(bags, Y, METRICS, **kw)
        np.testing.assert_allclose(np.array(got), np.array(filtered_metrics(ids, Y.toarray(), A, METRICS)),
                                   rtol=1e-12, atol=1e-12, err_msg=str(kw.keys()))


# ---- the encoder exchange -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("items", ["none", "all_but_one", "half", "exclusions_only", "all"])
def test_every_filtered_shard_path_runs_the_encoder_once(items, monkeypatch):
    """On item shards ``predict_h2`` is a collective (the h1pre exchange), so every rank must call it exactly once per
    batch of gold_ranks whatever its shard's eligible set: no eligible item, a compact copy, all items eligible, the
    exclusions only."""
    from aaerec_b200.engine import AAEEngine
    from aaerec_b200.filters import RankFilter
    V, B = 40000, 64
    eng = AAEEngine(V, 100, 50, max_batch=B)
    eng.init_uniform(42)
    X = _sets(B, V, 10, seed=4)
    eng.upload_csr(X.indptr.astype(np.int32), X.indices.astype(np.int32))
    Y = _gold(X, V, 6, seed=1)
    ids = {"none": np.zeros(0, np.int64), "all_but_one": np.arange(1, V), "half": np.arange(0, V, 2),
           "exclusions_only": None, "all": None}[items]
    filt = RankFilter(None, None) if items == "all" else \
        RankFilter.build(V, B, items=ids, exclude=X if items == "exclusions_only" else None)
    calls = []
    real = eng.predict_h2
    monkeypatch.setattr(eng, "predict_h2", lambda B_: calls.append(B_) or real(B_))
    r = eng.gold_ranks(B, Y.indptr.astype(np.int32), Y.indices.astype(np.int32), filt=filt)
    assert calls == [B]
    assert r.shape == (Y.nnz,)
