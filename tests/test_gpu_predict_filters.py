"""GPU tests of candidate-restricted ranking (``predict_topk(..., items=, exclude=)``): the compact candidate copy
ranked through the fused v2 / v1 and dense paths, against the numpy statement of the semantics
(``test_predict_filters_host.rank_reference``) on the CPU oracle's logits."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from test_predict_filters_host import rank_reference, FLT_MAX

pytestmark = pytest.mark.gpu


def _engine(V, H=100, C=50, B=128, seed=42):
    from aaerec_b200.engine import AAEEngine
    eng = AAEEngine(V, H, C, max_batch=B)
    eng.init_uniform(seed)
    eng.Wd3.mul_(8.0)           # spread the logits, as in test_gpu_predict_fused.py
    eng.bd3.mul_(8.0)
    return eng


def _upload(eng, X):
    eng.upload_csr(X.indptr.astype(np.int32), X.indices.astype(np.int32))


def _oracle_logits(eng, X):
    from oracle import aae_oracle as O
    sd = {k: torch.as_tensor(v) for k, v in eng.state_dict().items()}
    return O.OracleAAE(sd, n_code=eng.C).logits(X.toarray())


def _exclusions(X, elig, n_rand, seed):
    """About n_rand + 6 exclusions per row (sparse): random items, three known items of the row and three ineligible
    ones."""
    rng = np.random.default_rng(seed)
    n, V = X.shape
    inel = np.flatnonzero(~elig)
    rows, cols = [], []
    for r in range(n):
        c = [rng.choice(V, n_rand, replace=False), X.indices[X.indptr[r]:X.indptr[r + 1]][:3]]
        if inel.size:
            c.append(rng.choice(inel, min(3, inel.size), replace=False))
        c = np.concatenate(c)
        rows.append(np.full(c.size, r))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    E = sp.csr_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(n, V))
    E.data[:] = 1
    return E


def _lookup(M, r, c):
    """M[r[j], c[j]] != 0 for a scipy sparse M, as a 1-D bool array."""
    if r.size == 0:
        return np.zeros(0, dtype=bool)
    v = M[r, c]
    return np.asarray(v.todense() if sp.issparse(v) else v).ravel() != 0


def _assert_ranking(fi, fv, ref_i, Z, X, elig, E):
    """fi/fv against the reference ids outside fp32 near-ties (the rule of test_gpu_predict_fused.py, on the masked
    logits); padding exactly where the reference pads; no ineligible or excluded id."""
    assert fi.shape == ref_i.shape
    pad = ref_i < 0
    np.testing.assert_array_equal(fi < 0, pad)
    assert np.all(fv[pad] == -np.inf)
    rows = np.broadcast_to(np.arange(fi.shape[0])[:, None], fi.shape)
    live = ~pad
    assert elig[fi[live]].all(), "an ineligible item was returned"
    if E is not None:
        assert not _lookup(E, rows[live], fi[live]).any(), "an excluded item was returned"
    mism = live & (fi != ref_i)
    assert mism.mean() < 0.02

    def masked(r, i):
        z = Z[r, i].astype(np.float32)
        return np.where(_lookup(X, r, i), -FLT_MAX, z)
    a, b = masked(rows[mism], fi[mism]), masked(rows[mism], ref_i[mism])
    assert np.all(np.abs(a - b) <= 2e-5 * np.maximum(1.0, np.abs(b)))


_CASES = {}


def _case(V, B):
    """Engine, query sets and oracle logits per (V, B), shared by the parameter sets."""
    if (V, B) not in _CASES:
        from aaerec_b200.synth import synth_sets
        _CASES.clear()
        eng = _engine(V, B=B)
        X = synth_sets(B, V, 20, seed=V % 97 + B)
        _CASES[(V, B)] = (eng, X, _oracle_logits(eng, X))
    return _CASES[(V, B)]


@pytest.mark.parametrize("frac", [0.5, 0.05, 0.002])
@pytest.mark.parametrize("k", [20, 100, 500])
@pytest.mark.parametrize("V,B", [(40000, 70), (40000, 1100), (300000, 70), (300000, 1100)])
def test_filtered_topk_matches_reference(V, B, k, frac):
    from aaerec_b200.filters import RankFilter
    eng, X, Z = _case(V, B)
    _upload(eng, X)
    rng = np.random.default_rng(int(frac * 1000) + k)
    items = rng.choice(V, int(frac * V), replace=False)
    elig = np.zeros(V, dtype=bool)
    elig[items] = True
    E = _exclusions(X, elig, 14, seed=k)
    filt = RankFilter.build(V, B, items=items, exclude=E)
    fb = eng.topk_fallbacks
    fi, fv = eng.topk(B, k, filt=filt)
    fi, fv = fi.cpu().numpy(), fv.cpu().numpy()
    A = int(elig.sum())
    # every row has far more than k returnable items: the fused path must rank them without falling back
    assert eng.topk_fallbacks == fb
    assert eng.topk_mode == ("v2" if A >= 32768 else "dense")
    ref_i, _ = rank_reference(Z, X, k, items=items, exclude=E)
    _assert_ranking(fi, fv, ref_i, Z, X, elig, E)


@pytest.mark.parametrize("mode", ["v2", "dense"])
def test_unrestricted_filter_is_the_unfiltered_ranking(mode, monkeypatch):
    """items = every item (the public call drops the filter), and exclusions that cannot change the lists (each row's own
    known items, ranked last anyway; the filtered kernels with no column table) both give exactly the unfiltered
    lists."""
    from aaerec_b200.filters import RankFilter
    from aaerec_b200.synth import synth_sets
    if mode == "dense":
        monkeypatch.setenv("AAE_B200_TOPK", "dense")
    V, B, k = 60000, 200, 100
    eng = _engine(V, B=B)
    X = synth_sets(B, V, 20, seed=11)
    _upload(eng, X)
    ui, uv = (t.cpu().numpy() for t in eng.topk(B, k))
    assert eng.topk_mode == mode
    assert RankFilter.build(V, B, items=np.arange(V)) is None
    own = RankFilter.build(V, B, exclude=X)
    assert own.items is None
    fi, fv = (t.cpu().numpy() for t in eng.topk(B, k, filt=own))
    assert eng.topk_mode == mode
    np.testing.assert_array_equal(fi, ui)
    np.testing.assert_array_equal(fv, uv)


def test_dense_and_v1_return_the_lists_of_v2(monkeypatch):
    from aaerec_b200.filters import RankFilter
    V, B, k = 300000, 70, 100
    eng, X, Z = _case(V, B)
    _upload(eng, X)
    items = np.random.default_rng(3).choice(V, V // 2, replace=False)
    elig = np.zeros(V, dtype=bool)
    elig[items] = True
    E = _exclusions(X, elig, 14, seed=5)
    filt = RankFilter.build(V, B, items=items, exclude=E)
    out = {}
    for mode in ("v2", "v1", "dense"):
        monkeypatch.setenv("AAE_B200_TOPK", "" if mode == "v2" else mode)
        i, v = eng.topk(B, k, filt=filt)
        assert eng.topk_mode == mode
        out[mode] = (i.cpu().numpy(), v.cpu().numpy())
    np.testing.assert_array_equal(out["v1"][0], out["dense"][0])       # same 3xTF32 logits
    np.testing.assert_array_equal(out["v1"][1], out["dense"][1])
    (vi, vv), (di, dv) = out["v2"], out["dense"]
    np.testing.assert_allclose(vv, dv, rtol=3e-6, atol=3e-6)
    md = vi != di
    assert md.mean() < 0.01
    assert np.all(np.abs(vv[md] - dv[md]) <= 3e-6 * np.maximum(1.0, np.abs(dv[md])))


def test_candidate_set_smaller_than_k_pads_and_keeps_known_items_last():
    from aaerec_b200.filters import RankFilter
    V, B, k = 40000, 70, 50
    eng, X, Z = _case(V, B)
    _upload(eng, X)
    Xd = X.toarray()
    # 30 eligible items: 20 random ones and the first known item of each of the first 10 rows
    items = np.unique(np.r_[np.random.default_rng(1).choice(V, 20, replace=False),
                            [np.flatnonzero(Xd[r])[0] for r in range(10)]])
    fi, fv = (t.cpu().numpy() for t in eng.topk(B, k, filt=RankFilter.build(V, B, items=items)))
    assert eng.topk_mode == "dense"
    ref_i, _ = rank_reference(Z, X, k, items=items)
    elig = np.zeros(V, dtype=bool)
    elig[items] = True
    _assert_ranking(fi, fv, ref_i, Z, X, elig, None)
    for r in range(B):
        n_live = int((fi[r] >= 0).sum())
        assert n_live == items.size
        kn = Xd[r, fi[r, :n_live]] != 0
        assert np.all(fv[r, :n_live][kn] == -FLT_MAX)
        assert not np.any(kn[:-1] & ~kn[1:]), "an eligible known item ranked above an unknown one"


def _model(V, H=100, C=50, B=64, seed=42):
    from aaerec_b200.aae import AdversarialAutoEncoder
    from oracle import aae_oracle as O
    params = O.init_params(V, H, C, seed=seed)
    params["dec.lin3.weight"] = params["dec.lin3.weight"] * 8.0
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=B, n_epochs=1, verbose=False, impl="auto")
    model._build(V, C, params={k: v.clone() for k, v in params.items()})
    return model


def _model_logits(model, X):
    from oracle import aae_oracle as O
    sd = {k: torch.as_tensor(v) for k, v in model.state_dict().items()}
    return O.OracleAAE(sd, n_code=50).logits(X.toarray())


def test_full_ranking_with_items_is_a_stable_argsort_of_the_masked_logits():
    from aaerec_b200.synth import synth_sets
    V, B = 5000, 64
    model = _model(V, B=B)
    X = synth_sets(B, V, 10, seed=2)
    Xd = X.toarray()
    items = np.random.default_rng(4).choice(V, 700, replace=False)
    E = _exclusions(X, np.isin(np.arange(V), items), 14, seed=8)
    ids, val = model.predict_topk(X, None, items=items, exclude=E, return_scores=True)
    assert ids.shape == (B, 700)
    Z = _model_logits(model, X)
    ref_i, _ = rank_reference(Z, X, None, items=items, exclude=E, full=True)
    _assert_ranking(ids, val, ref_i, Z, X, np.isin(np.arange(V), items), E)
    # k beyond the selection kernels' envelope: the first min(k, A) columns of the same ranking
    ids2 = model.predict_topk(X, 5000, items=items, exclude=E)
    np.testing.assert_array_equal(ids2, ids)


def test_compact_copy_follows_training():
    """predict_topk(items=...), one partial_fit, predict_topk(items=...) == the same call on a fresh model loaded from
    the trained state_dict: the cached compact copy of the output layer is rebuilt after the weights change."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from aaerec_b200.synth import synth_sets
    V, B, k = 80000, 64, 100
    model = _model(V, B=B)
    Xq = synth_sets(200, V, 12, seed=6)
    items = np.random.default_rng(2).choice(V, V // 2, replace=False)
    model.predict_topk(Xq, k, items=items)
    assert model.engine.topk_mode == "v2"
    ver = model.engine._cmp["ver"]
    model.partial_fit(synth_sets(B, V, 12, seed=7))
    after = model.predict_topk(Xq, k, items=items)
    assert model.engine._cmp["ver"] != ver
    fresh = AdversarialAutoEncoder(n_hidden=100, n_code=50, batch_size=B, n_epochs=1, verbose=False, impl="auto")
    fresh._build(V, 50, params={kk: torch.as_tensor(v).clone() for kk, v in model.state_dict().items()})
    np.testing.assert_array_equal(fresh.predict_topk(Xq, k, items=items), after)


def test_recommender_and_vae_pass_the_filter_through():
    from aaerec_b200.aae import AAERecommender
    from aaerec_b200.vae import VAE
    from aaerec_b200.synth import synth_sets
    V, B, k = 40000, 64, 30
    X = synth_sets(B, V, 10, seed=12)
    Xd = X.toarray()
    items = np.random.default_rng(9).choice(V, 2000, replace=False)
    elig = np.isin(np.arange(V), items)
    E = _exclusions(X, elig, 14, seed=10)

    class Bags(object):
        def tocsr(self):
            return X
    rec = AAERecommender(adversarial=True, verbose=False)
    rec.model = _model(V, B=B)
    got = rec.predict_topk(Bags(), k, items=items, exclude=E)
    np.testing.assert_array_equal(got, rec.model.predict_topk(X, k, items=items, exclude=E))
    Z = _model_logits(rec.model, X)
    ref_i, _ = rank_reference(Z, X, k, items=items, exclude=E)
    _assert_ranking(got, np.where(got < 0, -np.inf, 0.0), ref_i, Z, X, elig, E)

    vae = VAE(V, V, n_hidden=100, n_code=50, batch_size=B, n_epochs=1, verbose=False)
    vae.partial_fit(X)
    vi, vv = vae.predict_topk(X, k, items=items, exclude=E, return_scores=True)
    assert vi.shape == (B, k)
    live = vi >= 0
    assert elig[vi[live]].all() and not _lookup(E, np.nonzero(live)[0], vi[live]).any()
    assert np.all(np.diff(np.where(live, vv, -np.inf), axis=1) <= 0)


def test_gather_item_rows_reports_a_bad_id_table():
    """aae_gather_item_rows copies the listed rows and counts ids outside the shard or out of order in its status
    word; the engine refuses such a table."""
    from aaerec_b200._native import call, ptr
    V, H = 1000, 100
    eng = _engine(V)
    n_bad = torch.zeros(1, dtype=torch.int32, device=eng.dev)
    Wc = torch.empty(4, H, device=eng.dev)
    bc = torch.empty(4, device=eng.dev)

    def gather(ids, v_begin=0, Vloc=V):
        t = torch.tensor(ids, dtype=torch.int32, device=eng.dev)
        call("aae_gather_item_rows", ptr(eng.Wd3), ptr(eng.bd3), H, Vloc, v_begin, ptr(t), len(ids), ptr(Wc), ptr(bc),
             ptr(n_bad), None)
        torch.cuda.synchronize()
        return int(n_bad.item())
    assert gather([3, 10, 500, 999]) == 0
    assert torch.equal(Wc, eng.Wd3[[3, 10, 500, 999]]) and torch.equal(bc, eng.bd3[[3, 10, 500, 999]])
    assert gather([3, 10, 1000, 2000]) == 2                   # outside [0, 1000)
    assert gather([10, 3, 500, 500]) == 2                     # not strictly ascending
    assert gather([3, 10, 500, 999], v_begin=5, Vloc=500) == 2
    with pytest.raises(ValueError, match="outside"):
        eng.Vloc -= 100                                       # the table below now reaches past the shard
        try:
            eng._compact(np.array([1, 950], dtype=np.int32))
        finally:
            eng.Vloc += 100


@pytest.mark.parametrize("items", ["none", "all_but_one", "half", "exclusions_only", "all"])
def test_every_filtered_shard_path_runs_the_encoder_once(items, monkeypatch):
    """On item shards ``predict_h2`` is a collective (the h1pre exchange), so every rank must call it exactly once per
    topk whatever its shard's eligible set: no eligible item, a compact copy, all items eligible (the unfiltered
    ranking), exclusions only."""
    from aaerec_b200.filters import RankFilter
    from aaerec_b200.synth import synth_sets
    V, B, k = 40000, 64, 20
    eng = _engine(V, B=B)
    X = synth_sets(B, V, 10, seed=4)
    _upload(eng, X)
    ids = {"none": np.zeros(0, np.int64), "all_but_one": np.arange(1, V), "half": np.arange(0, V, 2),
           "exclusions_only": None, "all": None}[items]
    # "all": a shard whose items are all eligible, without exclusions (another shard's items may not be)
    filt = RankFilter(None, None) if items == "all" else \
        RankFilter.build(V, B, items=ids, exclude=X if items == "exclusions_only" else None)
    calls = []
    real = eng.predict_h2
    monkeypatch.setattr(eng, "predict_h2", lambda B_: calls.append(B_) or real(B_))
    i, v = eng.topk(B, k, filt=filt)
    assert calls == [B]
    if items == "none":
        assert eng.topk_mode == "empty" and bool((i == -1).all()) and bool((v == -float("inf")).all())
