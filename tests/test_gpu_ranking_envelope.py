"""GPU tests of the ranking paths across their envelope, against a float64 reference of the same operation.

Every returned list is checked against Z = h2 . Wd3^T + bd3 computed in float64 from the engine's own h2 and weights,
with the per-item bound e = (2^-20 + (H+1) 2^-23) (|h2| . |Wd3|^T + |bd3|), which covers fp32 FMA re-scoring and
3xTF32: values within e of Z, distinct ids, descending values with ties in ascending id, and completeness (no
returnable item left out whose Z exceeds the last listed one by more than both bounds).  Covered: hidden widths of the
v2 / v1 / dense paths, the fused-plan and k boundaries, batch sizes across the cluster shapes of v2, clustered and
tied scores, the shard merges, and aae_rank_counts against an int64 count."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

FLT_MAX = float(np.finfo(np.float32).max)
V_RAGGED = 70001            # not a multiple of 128 or of 4


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _lib():
    from aaerec_b200 import _native
    return _native.load()


def _engine(V, H, B, seed=42):
    from aaerec_b200.engine import AAEEngine
    eng = AAEEngine(V, H, 50, max_batch=B)
    eng.init_uniform(seed)
    eng.Wd3.mul_(8.0)           # spread the logits, as in test_gpu_predict_fused.py
    eng.bd3.mul_(8.0)
    return eng


def _upload(eng, X):
    eng.upload_csr(X.indptr.astype(np.int32), X.indices.astype(np.int32))


def _sets(B, V, seed, mean_len=20):
    from aaerec_b200.synth import synth_sets
    return synth_sets(B, V, mean_len, seed=seed)


def _reference(h2, W, b):
    """float64 logits [B, V] and the per-item error bound e [B, V] of an fp32 / 3xTF32 evaluation."""
    H = h2.shape[1]
    h, Wd, bd = h2.double(), W.double(), b.double()
    Z = torch.addmm(bd, h, Wd.t())
    e = torch.addmm(bd.abs(), h.abs(), Wd.abs().t()).mul_(2.0 ** -20 + (H + 1) * 2.0 ** -23)
    return Z, e


def _engine_reference(eng, B):
    """Reference of the batch in the engine's device buffers: its own h2 (eval encoder) and output layer."""
    h2 = eng.predict_h2(B).clone()
    torch.cuda.synchronize()
    return _reference(h2, eng.Wd3[:eng.Vloc], eng.bd3[:eng.Vloc])


def _dense_mask(X, dev="cuda"):
    """bool [n, V] device mask of the nonzero entries of a scipy CSR matrix."""
    X = sp.csr_matrix(X)
    m = torch.zeros(X.shape, dtype=torch.bool, device=dev)
    rows = np.repeat(np.arange(X.shape[0]), np.diff(X.indptr))
    if rows.size:
        m[torch.as_tensor(rows, device=dev), torch.as_tensor(X.indices.astype(np.int64), device=dev)] = True
    return m


def _check_lists(ids, vals, Z, e, known, ret=None, what=""):
    """The contract of a ranked list against the float64 reference (see the module docstring).  ``known`` [B, V] bool:
    known items, which may only follow every returnable unknown item, with a score <= -FLT_MAX; ``ret`` [B, V] bool:
    the returnable items (eligible and not excluded; None: all).  A row with fewer returnable items than its length ends
    in (-1, -inf) padding.  Returns the number of listed unknown items."""
    ids = torch.as_tensor(np.asarray(ids) if not torch.is_tensor(ids) else ids).to(Z.device).long()
    vals = torch.as_tensor(np.asarray(vals) if not torch.is_tensor(vals) else vals).to(Z.device).double()
    B, V = Z.shape
    k = ids.shape[1]
    assert ids.shape == vals.shape == (B, k), (what, ids.shape, vals.shape)
    ret = torch.ones_like(known) if ret is None else ret
    U = ret & ~known
    KR = ret & known
    a = torch.clamp(U.sum(1), max=k)                        # unknown entries expected per row
    bk = torch.minimum(KR.sum(1), k - a)                     # then known ones
    pos = torch.arange(k, device=Z.device)[None, :]
    exp_u = pos < a[:, None]
    exp_k = (pos >= a[:, None]) & (pos < (a + bk)[:, None])
    exp_pad = ~(exp_u | exp_k)
    pad = ids < 0
    bad = (pad != exp_pad)
    assert not bad.any(), "%s: padding at the wrong place in rows %s" % (what, bad.any(1).nonzero().flatten()[:8].tolist())
    assert bool((vals[pad] == -np.inf).all()), "%s: padding without -inf" % what
    assert bool((ids < V).all()), "%s: id out of range" % what
    safe = ids.clamp(min=0)
    isU = torch.gather(U, 1, safe) & ~pad
    isK = torch.gather(KR, 1, safe) & ~pad
    bad = isU != exp_u
    assert not bad.any(), "%s: a non-returnable item listed, or a known one above an unknown one, in rows %s" % (
        what, bad.any(1).nonzero().flatten()[:8].tolist())
    assert bool((isK == exp_k).all()), "%s: a non-returnable known item listed" % what
    s, _ = torch.sort(torch.where(pad, -1 - pos.expand(B, k), ids), dim=1)
    assert bool((s[:, 1:] != s[:, :-1]).all()), "%s: an id listed twice" % what
    assert bool((vals[isK] <= -FLT_MAX).all()), "%s: a known item scored above -FLT_MAX" % what
    zi, ei = torch.gather(Z, 1, safe), torch.gather(e, 1, safe)
    err = ((vals - zi).abs() - ei)[isU]
    assert err.numel() == 0 or float(err.max()) <= 0, "%s: a value off its float64 logit by more than the bound" % what
    live = ~pad
    pair = live[:, 1:] & live[:, :-1]
    v0, v1, i0, i1 = vals[:, :-1], vals[:, 1:], ids[:, :-1], ids[:, 1:]
    order = (v0 > v1) | ((v0 == v1) & (i0 < i1))
    bad = pair & ~order
    assert not bad.any(), "%s: values increase or ties out of id order in rows %s" % (
        what, bad.any(1).nonzero().flatten()[:8].tolist())
    # completeness: an unlisted returnable unknown item may exceed the last listed unknown one only within the bounds
    rows = (a > 0).nonzero().flatten()
    if rows.numel():
        last = torch.gather(safe, 1, (a - 1).clamp(min=0)[:, None])[:, 0]
        lim = Z[torch.arange(B, device=Z.device), last] + e[torch.arange(B, device=Z.device), last]
        listed = torch.zeros(B, V, dtype=torch.int32, device=Z.device)
        listed.scatter_add_(1, safe, isU.int())
        rest = torch.where(U & (listed == 0), Z - e, torch.full_like(Z, -np.inf))
        over = rest.max(1).values > lim
        over &= a > 0
        assert not over.any(), "%s: a returnable item missing from rows %s" % (what, over.nonzero().flatten()[:8].tolist())
    return int(a.sum())


def _filter_exclusions(X, elig, n_rand, seed):
    """About n_rand + 6 exclusions per row: random items, three known items of the row and three ineligible ones."""
    rng = np.random.default_rng(seed)
    n, V = X.shape
    inel = np.flatnonzero(~elig)
    rows, cols = [], []
    for r in range(n):
        c = [rng.choice(V, n_rand, replace=False), X.indices[X.indptr[r]:X.indptr[r + 1]][:3]]
        if inel.size:
            c.append(rng.choice(inel, min(3, inel.size), replace=False))
        c = np.unique(np.concatenate(c))
        rows.append(np.full(c.size, r))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    return sp.csr_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(n, V))


def _oracle_logits(eng, X):
    from oracle import aae_oracle as O
    sd = {k: torch.as_tensor(v) for k, v in eng.state_dict().items()}
    return O.OracleAAE(sd, n_code=eng.C).logits(X.toarray())


def _pad_weights(W, b):
    from aaerec_b200._native import call, ptr
    Vloc, H = W.shape
    n = int(_lib().aae_pad_weights_floats(Vloc, H))
    assert n > 0
    wp = torch.empty(n, dtype=torch.float32, device=W.device)
    call("aae_pad_weights", ptr(W), ptr(b), Vloc, H, ptr(wp), ptr(wp[n - 64:]), None)
    return wp, wp[n - 64:]


def _csr_dev(X):
    X = sp.csr_matrix(X)
    return (torch.as_tensor(X.indptr.astype(np.int32), device="cuda"),
            torch.as_tensor(np.r_[X.indices.astype(np.int32), np.zeros(1, np.int32)], device="cuda"))


def _v2(h2, W, b, wp, wmax, X, k, v_begin=0):
    """aae_predict_topk2 called directly on (h2, one item shard): (ids, vals, n_bad)."""
    from aaerec_b200._native import call, ptr
    B, H = h2.shape
    Vloc = W.shape[0]
    need = int(_lib().aae_predict_topk2_work_bytes(B, Vloc, k, H))
    assert need > 0
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    idx = torch.empty(B, k, dtype=torch.int32, device="cuda")
    val = torch.empty(B, k, dtype=torch.float32, device="cuda")
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    ip, ii = _csr_dev(X)
    call("aae_predict_topk2", ptr(h2), B, H, ptr(W), ptr(b), ptr(wp), ptr(wmax), Vloc, v_begin, ptr(ip), ptr(ii), k,
         ptr(work), need, ptr(idx), ptr(val), ptr(n_bad), None)
    torch.cuda.synchronize()
    return idx, val, int(n_bad.item())


# ---- hidden widths ---------------------------------------------------------------------------------------------------
# (n_hidden, unfiltered path, aae_dec_out_scores impl): v2 up to 100 (n_hidden % 4 == 0), v1 for 104 and 108, the fp32
# CUDA-core scores + aae_masked_topk beyond (n_hidden % 4 != 0, or a W' row too long for the tensor-core operand tile)
WIDTHS = [(24, "v2", 1), (64, "v2", 1), (96, "v2", 1), (100, "v2", 1), (104, "v1", 1), (108, "v1", 1),
          (112, "dense", 0), (116, "dense", 0), (124, "dense", 0), (30, "dense", 0), (126, "dense", 0),
          (160, "dense", 0), (512, "dense", 0)]


@pytest.mark.parametrize("H,mode,impl", WIDTHS)
def test_ranking_at_hidden_width(H, mode, impl):
    V, B = V_RAGGED, 300
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=H)
    _upload(eng, X)
    assert eng.impl_for_scores() == impl
    Z, e = _engine_reference(eng, B)
    # the encoder / decoder head at this width (aae_predict_tail_bag) against the oracle's chain
    Zo = _oracle_logits(eng, X[:48])
    S = (e[:48] / (2.0 ** -20 + (H + 1) * 2.0 ** -23)).cpu().numpy()
    assert np.all(np.abs(Zo - Z[:48].cpu().numpy()) <= 2e-5 * S + 1e-6)
    known = _dense_mask(X)
    fb = eng.topk_fallbacks
    for k in (1, 100, 1024):
        i, v = eng.topk(B, k)
        assert eng.topk_mode == mode, (H, k, eng.topk_mode)
        _check_lists(i, v, Z, e, known, what="H=%d k=%d" % (H, k))
    # benign scores: a fused path must not have needed its dense fallback (which would hide a broken filter)
    assert eng.topk_fallbacks == fb


@pytest.mark.parametrize("H,impl", [(24, 1), (64, 1), (100, 1), (108, 1), (30, 0), (116, 0), (512, 0)])
def test_dec_out_scores_against_float64(H, impl):
    from aaerec_b200._native import call, ptr
    V, B = 9999, 257
    g = torch.Generator().manual_seed(H)
    W = ((torch.rand(V, H, generator=g) - 0.5) * 0.6).cuda()
    b = (torch.rand(V, generator=g) - 0.5).cuda()
    h2 = torch.relu(torch.randn(B, H, generator=g)).cuda()
    out = torch.full((B, V + 3), float("nan"), device="cuda")
    call("aae_dec_out_scores", ptr(h2), B, H, ptr(W), ptr(b), V, 0, ptr(out), V + 3, impl, None)
    torch.cuda.synchronize()
    Z, e = _reference(h2, W, b)
    assert bool(((out[:, :V].double() - Z).abs() <= e).all())
    assert bool(out[:, V:].isnan().all()), "wrote past Vloc"


@pytest.mark.parametrize("H", [112, 116, 124])
def test_tensor_core_scores_refuse_rows_beyond_their_operand_tile(H):
    """[Wd3 | bd3] rows longer than 112 floats do not fit the operand tile of the tensor-core scores / v1 kernel: the
    call fails with an error instead of returning scores."""
    from aaerec_b200._native import NativeError, call, ptr
    V, B = 3000, 64
    W = torch.zeros(V, H, device="cuda")
    b = torch.zeros(V, device="cuda")
    h2 = torch.zeros(B, H, device="cuda")
    out = torch.empty(B, V, device="cuda")
    with pytest.raises(NativeError, match="n_hidden"):
        call("aae_dec_out_scores", ptr(h2), B, H, ptr(W), ptr(b), V, 0, ptr(out), V, 1, None)


@pytest.mark.parametrize("frac", [0.5, 0.03, "tiny"])
@pytest.mark.parametrize("H,fused", [(24, "v2"), (108, "v1"), (116, "dense"), (30, "dense")])
def test_filtered_ranking_at_hidden_width(H, fused, frac):
    from aaerec_b200.filters import RankFilter
    V, B, k = V_RAGGED, 200, 100
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=H + 1)
    _upload(eng, X)
    rng = np.random.default_rng(H)
    if frac == "tiny":      # fewer returnable items than k: known eligible items last, then padding
        items = np.unique(np.r_[rng.choice(V, 60, replace=False),
                                np.concatenate([X.indices[X.indptr[r]:X.indptr[r + 1]][3:6] for r in range(20)])])
    else:
        items = rng.choice(V, int(frac * V), replace=False)
    elig = np.zeros(V, dtype=bool)
    elig[items] = True
    E = _filter_exclusions(X, elig, 14, seed=H)
    filt = RankFilter.build(V, B, items=items, exclude=E)
    Z, e = _engine_reference(eng, B)
    fb = eng.topk_fallbacks
    i, v = eng.topk(B, k, filt=filt)
    assert eng.topk_mode == (fused if elig.sum() >= 32768 else "dense")
    assert eng.topk_fallbacks == fb
    ret = torch.as_tensor(elig, device="cuda")[None, :] & ~_dense_mask(E)
    _check_lists(i, v, Z, e, _dense_mask(X), ret=ret, what="H=%d frac=%s" % (H, frac))


@pytest.mark.parametrize("H", [30, 100])
def test_gather_item_rows_is_exact_indexing(H):
    """aae_gather_item_rows (scalar branch for n_hidden % 4 != 0, float4 otherwise) == torch indexing, bit for bit."""
    from aaerec_b200._native import call, ptr
    Vloc, v_begin = 5003, 1000
    g = torch.Generator().manual_seed(H)
    W = torch.randn(Vloc, H, generator=g).cuda()
    b = torch.randn(Vloc, generator=g).cuda()
    ids = np.sort(np.random.default_rng(H).choice(Vloc, 1237, replace=False)) + v_begin
    t = torch.as_tensor(ids.astype(np.int32), device="cuda")
    Wc = torch.full((ids.size, H), float("nan"), device="cuda")
    bc = torch.full((ids.size,), float("nan"), device="cuda")
    n_bad = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    call("aae_gather_item_rows", ptr(W), ptr(b), H, Vloc, v_begin, ptr(t), ids.size, ptr(Wc), ptr(bc), ptr(n_bad), None)
    torch.cuda.synchronize()
    assert int(n_bad.item()) == 0
    sel = torch.as_tensor(ids - v_begin, device="cuda")
    assert torch.equal(Wc, W[sel]) and torch.equal(bc, b[sel])


# ---- plan, k and batch boundaries ------------------------------------------------------------------------------------
def _smallest(ok, lo=1, hi=1 << 22):
    assert ok(hi) and not ok(lo)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if ok(mid):
            hi = mid
        else:
            lo = mid
    return hi


def test_fused_plan_boundary():
    lib = _lib()
    B = 129
    vmin2 = _smallest(lambda n: int(lib.aae_predict_topk2_work_bytes(B, n, 100, 100)) > 0)
    vmin1 = _smallest(lambda n: int(lib.aae_predict_topk_work_bytes(B, n, 100)) > 0)
    assert vmin1 == vmin2
    for k in (1, 1024):
        assert int(lib.aae_predict_topk2_work_bytes(B, vmin2, k, 100)) > 0
        assert int(lib.aae_predict_topk2_work_bytes(B, vmin2 - 1, k, 100)) == 0
    assert int(lib.aae_predict_topk2_work_bytes(B, 10 ** 6, 1025, 100)) == 0
    assert int(lib.aae_predict_topk_work_bytes(B, 10 ** 6, 1025)) == 0
    for H, fused in ((100, "v2"), (108, "v1")):
        for V, mode in ((vmin2 - 1, "dense"), (vmin2, fused)):
            eng = _engine(V, H, B)
            X = _sets(B, V, seed=V % 97)
            _upload(eng, X)
            Z, e = _engine_reference(eng, B)
            known = _dense_mask(X)
            for k in (100, 1024):
                i, v = eng.topk(B, k)
                assert eng.topk_mode == mode, (H, V, k, eng.topk_mode)
                _check_lists(i, v, Z, e, known, what="H=%d V=%d k=%d" % (H, V, k))
            assert eng.topk_fallbacks == 0


def test_k_boundaries_of_the_selection_paths():
    V, H, B = V_RAGGED, 100, 129
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=5)
    _upload(eng, X)
    Z, e = _engine_reference(eng, B)
    known = _dense_mask(X)
    for k, mode in ((1, "v2"), (1024, "v2"), (1025, "dense"), (4096, "dense")):
        i, v = eng.topk(B, k)
        assert eng.topk_mode == mode, (k, eng.topk_mode)
        _check_lists(i, v, Z, e, known, what="k=%d" % k)
    assert eng.topk_fallbacks == 0


def test_public_topk_beyond_the_selection_envelope():
    """k = 4096 (aae_masked_topk), 4097 and k > V (the device sort of the full ranking, known items last)."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from oracle import aae_oracle as O
    V, H, C, B = 6000, 100, 50, 64
    params = O.init_params(V, H, C, seed=11)
    params["dec.lin3.weight"] = params["dec.lin3.weight"] * 8.0
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=B, n_epochs=1, verbose=False)
    model._build(V, C, params={k: v.clone() for k, v in params.items()})
    X = _sets(B, V, seed=3, mean_len=30)
    known = _dense_mask(X)
    for k in (4096, 4097, V + 5):
        ids, vals = model.predict_topk(X, k, return_scores=True)
        assert ids.shape == (B, min(k, V))
        eng = model.engine
        Z, e = _reference(eng.h2[:B].clone(), eng.Wd3, eng.bd3)
        _check_lists(ids, vals, Z, e, known, what="k=%d" % k)


def test_batch_sizes_across_cluster_shapes():
    """B = 1 ... 1100: clusters of 1 / 2 / 4 row chunks, and cluster groups whose last group is partly empty."""
    V, H = V_RAGGED, 100
    eng = _engine(V, H, 1100)
    X = _sets(1100, V, seed=8, mean_len=15)
    for B in (1, 127, 128, 129, 255, 256, 257, 300, 513, 1100):
        Xb = X[:B]
        _upload(eng, Xb)
        Z, e = _engine_reference(eng, B)
        i, v = eng.topk(B, 100)
        assert eng.topk_mode == "v2"
        _check_lists(i, v, Z, e, _dense_mask(Xb), what="B=%d" % B)
        del Z, e
    assert eng.topk_fallbacks == 0


@pytest.mark.parametrize("H", [24, 100])
def test_v2_is_independent_of_cluster_size_and_batch_split(H, monkeypatch):
    """Bit for bit: the cluster size of the filter (AAE_B200_K5_CLUSTER) and the split of the rows into batches do not
    change a v2 list (exact fp32 re-scoring of a candidate set that contains the whole top k)."""
    V, B, k = V_RAGGED, 300, 100
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=H + 2)
    _upload(eng, X)
    h2 = eng.predict_h2(B).clone()
    W, b = eng.Wd3[:V], eng.bd3[:V]
    wp, wmax = _pad_weights(W, b)
    out = {}
    for cy in (1, 2, 4, 8):
        monkeypatch.setenv("AAE_B200_K5_CLUSTER", str(cy))
        i, v, bad = _v2(h2, W, b, wp, wmax, X, k)
        assert bad == 0, cy
        out[cy] = (i.cpu().numpy(), v.cpu().numpy())
    monkeypatch.delenv("AAE_B200_K5_CLUSTER")
    for cy in (2, 4, 8):
        np.testing.assert_array_equal(out[cy][0], out[1][0])
        np.testing.assert_array_equal(out[cy][1], out[1][1])
    i, v, bad = _v2(h2, W, b, wp, wmax, X, k)
    assert bad == 0
    parts = [_v2(h2[s:s + 100].contiguous(), W, b, wp, wmax, X[s:s + 100], k) for s in (0, 100, 200)]
    assert all(p[2] == 0 for p in parts)
    np.testing.assert_array_equal(np.concatenate([p[0].cpu().numpy() for p in parts]), i.cpu().numpy())
    np.testing.assert_array_equal(np.concatenate([p[1].cpu().numpy() for p in parts]), v.cpu().numpy())
    Z, e = _reference(h2, W, b)
    _check_lists(i, v, Z, e, _dense_mask(X), what="v2 direct")


# ---- adversarial score layouts ---------------------------------------------------------------------------------------
# (first item, length, bias added): blocks of a few tiles, blocks that straddle a tile of the threshold sample (every
# 8th tile at this V), a block of more than 8192 items (more candidates than a row's list holds), every 37th tile
CLUSTERS = [(384, 300, 40.0), (10 * 1024 - 150, 3000, 40.0), (20 * 1024 - 500, 9000, 40.0),
            (20 * 1024 - 500, 9000, 3.0), ("tiles", 37, 6.0)]


@pytest.mark.parametrize("cl", CLUSTERS, ids=lambda c: "%s-%s-%g" % c)
@pytest.mark.parametrize("H,mode", [(100, "v2"), (108, "v1")])
def test_clustered_candidates_stay_exact(H, mode, cl):
    V, B = V_RAGGED, 200
    eng = _engine(V, H, B)
    lo, n, boost = cl
    if lo == "tiles":
        t = torch.arange(V, device="cuda")
        eng.bd3[:V][(t // 128) % n == 0] += boost
    else:
        eng.bd3[lo:lo + n] += boost
    eng._wp_dirty = True
    X = _sets(B, V, seed=17)
    _upload(eng, X)
    Z, e = _engine_reference(eng, B)
    known = _dense_mask(X)
    for k in (100, 1024):
        fb = eng.topk_fallbacks
        i, v = eng.topk(B, k)
        fell = eng.topk_fallbacks - fb
        assert eng.topk_mode == ("dense" if fell else mode)
        _check_lists(i, v, Z, e, known, what="cluster %s k=%d" % (cl, k))
        print("clustered candidates H=%d (%s) block=%s k=%d: fallbacks %d" % (H, mode, cl, k, fell))


def _tie_groups(V):
    """Groups of items that will get identical rows of [Wd3 | bd3]: far apart (other 128-item tiles, other CTA
    columns, both halves of a two-shard split)."""
    half = V // 2
    src = [7, 1000, 2051, 3333, 4500, 5120]
    return [np.array([s, s + 128 * 9 + 5, s + half, s + half + 128 * 40 + 1, s + 60000]) for s in src]


def _make_ties(eng, B, X, k):
    """Upload X, give each group of ``_tie_groups`` the row of its first item, its bias shifted so that the group sits
    near the k-th score of a typical row (some groups a little above, some below): returns the groups."""
    _upload(eng, X)
    Z0, _ = _engine_reference(eng, B)
    kth = Z0.topk(k, dim=1).values[:, -1]
    sd = float(Z0.std())
    groups = _tie_groups(eng.Vloc)
    for gi, g in enumerate(groups):
        s = int(g[0])
        eng.bd3[s] += float((kth - Z0[:, s]).median()) + 0.15 * (gi - 2) * sd
        rest = torch.as_tensor(g[1:], device=eng.dev)
        eng.Wd3[rest] = eng.Wd3[s].clone()
        eng.bd3[rest] = eng.bd3[s].clone()
    eng._wp_dirty = True
    return groups


def _assert_bitwise_ties(eng, B, groups):
    """The dense scores kernel of the engine's impl gives identical rows bit-identical logits."""
    from aaerec_b200._native import call, ptr
    V = eng.Vloc
    sc = torch.empty(B, V, device="cuda")
    call("aae_dec_out_scores", ptr(eng.h2), B, eng.H, ptr(eng.Wd3), ptr(eng.bd3), V, 0, ptr(sc), V,
         eng.impl_for_scores(), None)
    torch.cuda.synchronize()
    for g in groups:
        cols = sc[:, torch.as_tensor(g, device="cuda")]
        assert torch.equal(cols, cols[:, :1].expand_as(cols))


def _assert_group_prefix(ids, groups):
    """Ties at the end of a list go to the lowest ids: the members of a tie group in a row's list are its lowest ids."""
    ids = np.asarray(ids)
    hits = 0
    for r in range(ids.shape[0]):
        row = set(ids[r].tolist())
        for g in groups:
            inl = np.array([x in row for x in g])
            hits += int(inl.sum() > 0)
            assert not np.any(~inl[:-1] & inl[1:]), ("a tied item listed while a lower id of its group is not", r, g)
    return hits


@pytest.mark.parametrize("H,mode", [(100, "v2"), (108, "v1"), (100, "dense"), (30, "dense"), (116, "dense")])
def test_exact_ties_go_to_the_lower_id(H, mode, monkeypatch):
    """Where a path's arithmetic gives identical rows bit-identical logits (v2's fp32 re-scoring, the fp32 kernel; for
    the 3xTF32 paths this is asserted first), tied items come in ascending id and a tie cut by the end of the list keeps
    its lowest ids."""
    if mode == "dense" and H == 100:
        monkeypatch.setenv("AAE_B200_TOPK", "dense")          # the 3xTF32 dense scores (impl 1)
    V, B, k = V_RAGGED, 129, 100
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=23, mean_len=10)
    groups = _make_ties(eng, B, X, k)
    Z, e = _engine_reference(eng, B)
    if mode != "v2":
        _assert_bitwise_ties(eng, B, groups)
    i, v = eng.topk(B, k)
    assert eng.topk_mode == mode and eng.topk_fallbacks == 0
    _check_lists(i, v, Z, e, _dense_mask(X), what="ties H=%d %s" % (H, mode))
    assert _assert_group_prefix(i.cpu().numpy(), groups) >= B       # the groups do reach the lists

    # a tie group larger than k that straddles the k-th position: ten distinct items above it, then its lowest ids
    eng2 = _engine(V, H, B, seed=5)
    top = np.arange(300, 3300, 300)                            # 10 items
    big = np.sort(np.random.default_rng(1).choice(np.setdiff1d(np.arange(V), top), 150, replace=False))
    eng2.Wd3[torch.as_tensor(big, device="cuda")] = eng2.Wd3[int(big[0])].clone()
    eng2.bd3[torch.as_tensor(big, device="cuda")] = eng2.bd3[int(big[0])] + 200.0
    eng2.bd3[torch.as_tensor(top, device="cuda")] += 400.0
    eng2._wp_dirty = True
    _upload(eng2, X)
    Z2, e2 = _engine_reference(eng2, B)
    if mode != "v2":
        _assert_bitwise_ties(eng2, B, [big])
    known = _dense_mask(X)
    i2, v2 = eng2.topk(B, k)
    assert eng2.topk_mode == mode or (mode in ("v2", "v1") and eng2.topk_mode == "dense")
    _check_lists(i2, v2, Z2, e2, known, what="big tie group H=%d %s" % (H, mode))
    i2 = i2.cpu().numpy()
    kn = X.toarray()
    for r in range(B):
        ub = big[kn[r, big] == 0]
        ut = top[kn[r, top] == 0]
        np.testing.assert_array_equal(np.sort(i2[r, :ut.size]), ut)
        np.testing.assert_array_equal(i2[r, ut.size:], ub[:k - ut.size])


def test_two_shard_ranking_with_ties_equals_one_shard():
    """Tie groups split across two item shards (v2 on each half, v_begin = the second half's first id): the merges of
    the two lists (aae_topk_merge_seg and aae_topk_merge) give the single-shard list bit for bit."""
    from aaerec_b200._native import call, ptr
    V, H, B, k = V_RAGGED, 100, 129, 100
    eng = _engine(V, H, B)
    X = _sets(B, V, seed=29, mean_len=10)
    groups = _make_ties(eng, B, X, k)
    h2 = eng.predict_h2(B).clone()
    W, b = eng.Wd3[:V], eng.bd3[:V]
    fi, fv, bad = _v2(h2, W, b, *_pad_weights(W, b), X, k)
    assert bad == 0
    half = V // 2
    gv = torch.empty(2, B, k, device="cuda")
    gi_ = torch.empty(2, B, k, dtype=torch.int32, device="cuda")
    for r, (lo, hi) in enumerate(((0, half), (half, V))):
        Ws, bs = W[lo:hi].contiguous(), b[lo:hi].contiguous()
        i, v, bad = _v2(h2, Ws, bs, *_pad_weights(Ws, bs), X, k, v_begin=lo)
        assert bad == 0
        gv[r], gi_[r] = v, i
    oi = torch.empty(B, k, dtype=torch.int32, device="cuda")
    ov = torch.empty(B, k, device="cuda")
    call("aae_topk_merge_seg", ptr(gv), ptr(gi_), 2, B, k, k, ptr(oi), ptr(ov), None)
    torch.cuda.synchronize()
    assert torch.equal(oi, fi) and torch.equal(ov, fv)
    cv = gv.permute(1, 0, 2).reshape(B, -1).contiguous()
    ci = gi_.permute(1, 0, 2).reshape(B, -1).contiguous()
    call("aae_topk_merge", ptr(cv), ptr(ci), B, 2 * k, k, ptr(oi), ptr(ov), None)
    torch.cuda.synchronize()
    assert torch.equal(oi, fi) and torch.equal(ov, fv)
    assert _assert_group_prefix(fi.cpu().numpy(), groups) >= B


@pytest.mark.parametrize("world,kpad,k", [(2, 1024, 1024), (4, 512, 100), (8, 256, 2048), (3, 7, 5)])
def test_topk_merges_order_ties_and_padding(world, kpad, k):
    """Per-shard lists with quantised (often tied) scores and (-1, pad) entries: both merges against a numpy sort by
    (score descending, id ascending); padding never outranks a live entry."""
    from aaerec_b200._native import call, ptr
    B = 33
    rng = np.random.default_rng(world * 1000 + kpad)
    n = world * kpad
    val = (rng.integers(-40, 40, size=(world, B, kpad)) / 8.0).astype(np.float32)
    ids = np.stack([rng.permutation(3 * n)[:n].reshape(world, kpad) for _ in range(B)], 1).astype(np.int32)
    val = -np.sort(-val, axis=2)
    for r in range(world):
        for b_ in range(B):
            npad = int(rng.integers(0, kpad + 1)) if rng.random() < 0.4 else 0
            if npad:
                ids[r, b_, kpad - npad:] = -1
                val[r, b_, kpad - npad:] = -np.inf
    kk = min(k, n)
    want_i = np.full((B, kk), -1, np.int64)
    want_v = np.full((B, kk), -np.inf, np.float32)
    for b_ in range(B):
        v_, i_ = val[:, b_].ravel(), ids[:, b_].ravel()
        live = i_ >= 0
        o = np.lexsort((i_[live], -v_[live].astype(np.float64)))[:kk]
        want_i[b_, :o.size] = i_[live][o]
        want_v[b_, :o.size] = v_[live][o]
    gv, gi = torch.as_tensor(val, device="cuda"), torch.as_tensor(ids, device="cuda")
    oi = torch.empty(B, kk, dtype=torch.int32, device="cuda")
    ov = torch.empty(B, kk, device="cuda")
    padded = want_i < 0
    if n <= 2048:
        call("aae_topk_merge_seg", ptr(gv), ptr(gi), world, B, kpad, kk, ptr(oi), ptr(ov), None)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(oi.cpu().numpy(), want_i)
        np.testing.assert_array_equal(ov.cpu().numpy()[~padded], want_v[~padded])
        assert np.all(ov.cpu().numpy()[padded] == -FLT_MAX)
    if kk <= 4096:
        cv = gv.permute(1, 0, 2).reshape(B, -1).contiguous()
        ci = gi.permute(1, 0, 2).reshape(B, -1).contiguous()
        call("aae_topk_merge", ptr(cv), ptr(ci), B, n, kk, ptr(oi), ptr(ov), None)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(oi.cpu().numpy(), want_i)
        np.testing.assert_array_equal(ov.cpu().numpy(), want_v)


# ---- aae_rank_counts -------------------------------------------------------------------------------------------------
def _rank_counts(S, lds, B, Vloc, v_begin, known, gold, zg, given):
    from aaerec_b200._native import call, ptr
    kp, ki = known if known is not None else (None, None)
    gp, gi = gold
    cnt = torch.full((gi.numel() - 1,), 99, dtype=torch.int32, device="cuda")
    call("aae_rank_counts", ptr(S), lds, B, Vloc, v_begin, ptr(kp) if kp is not None else None,
         ptr(ki) if ki is not None else None, ptr(gp), ptr(gi), gi.numel() - 1, ptr(zg), 1 if given else 0, ptr(cnt),
         None)
    torch.cuda.synchronize()
    return cnt


@pytest.mark.parametrize("Vloc", [1000, 16384, 16385, 50000])
def test_rank_counts_against_int64_reference(Vloc):
    """Counts of the items ranked before each gold item (strictly higher score, or equal score and lower id), with
    known items at -FLT_MAX: rows of 0 / 1 / 8 / 9 / 40 gold items, gold items that are known, scores in steps of 1/8
    (ties everywhere), a row stride above Vloc and v_begin != 0; and the two-shard protocol of engine.gold_ranks (NaN
    gold scores from the other shard, summed, second call with the scores given, counts summed) == one shard."""
    rng = np.random.default_rng(Vloc)
    n_gold = [0, 1, 8, 9, 40, 3, 17]
    B, v_begin, lds = len(n_gold), 1234, Vloc + 37
    sc = (rng.integers(-64, 64, size=(B, Vloc)) / 8.0).astype(np.float32)
    kn_rows, gd_rows = [], []
    for r in range(B):
        kc = np.sort(rng.choice(Vloc, 30, replace=False))
        gc = rng.choice(np.setdiff1d(np.arange(Vloc), kc), n_gold[r], replace=False)
        if n_gold[r] >= 8:
            gc[:2] = kc[:2]                                    # gold items that are also known
        kn_rows.append(kc + v_begin)
        gd_rows.append(np.sort(gc) + v_begin)
    kn = sp.csr_matrix((np.ones(B * 30), np.concatenate(kn_rows), np.arange(B + 1) * 30))
    gptr = np.r_[0, np.cumsum(n_gold)].astype(np.int32)
    gidx = np.concatenate(gd_rows).astype(np.int32)
    # int64 reference
    M = sc.copy()
    for r in range(B):
        M[r, kn_rows[r] - v_begin] = -FLT_MAX
    want, zwant = [], []
    cols = np.arange(Vloc)
    for r in range(B):
        for g in gd_rows[r]:
            c = g - v_begin
            z = M[r, c]
            want.append(int(np.sum(M[r] > z, dtype=np.int64) + np.sum((M[r] == z) & (cols < c), dtype=np.int64)))
            zwant.append(z)
    want = np.array(want, dtype=np.int64)
    known = (torch.as_tensor(kn.indptr.astype(np.int32), device="cuda"),
             torch.as_tensor(kn.indices.astype(np.int32), device="cuda"))
    gold = (torch.as_tensor(gptr, device="cuda"), torch.as_tensor(np.r_[gidx, 0].astype(np.int32), device="cuda"))

    S = torch.full((B, lds), float("nan"), device="cuda")
    S[:, :Vloc] = torch.as_tensor(sc, device="cuda")
    zg = torch.empty(max(gidx.size, 1), device="cuda")
    cnt = _rank_counts(S, lds, B, Vloc, v_begin, known, gold, zg, False)
    np.testing.assert_array_equal(cnt.cpu().numpy().astype(np.int64), want)
    np.testing.assert_array_equal(zg[:gidx.size].cpu().numpy(), np.array(zwant, np.float32))

    # two item shards on one device
    split = Vloc // 2 + 3
    shards = []
    for c0, c1 in ((0, split), (split, Vloc)):
        Ss = torch.full((B, c1 - c0 + 5), float("nan"), device="cuda")
        Ss[:, :c1 - c0] = torch.as_tensor(sc[:, c0:c1], device="cuda")
        shards.append((Ss, c1 - c0, v_begin + c0))
    zsum = torch.zeros(max(gidx.size, 1), device="cuda")
    for Ss, n, vb in shards:
        z = torch.empty_like(zsum)
        _rank_counts(Ss, Ss.shape[1], B, n, vb, known, gold, z, False)
        zsum += torch.nan_to_num(z, nan=0.0)
    total = torch.zeros(gidx.size, dtype=torch.int64, device="cuda")
    for Ss, n, vb in shards:
        total += _rank_counts(Ss, Ss.shape[1], B, n, vb, None, gold, zsum, True).long()
    np.testing.assert_array_equal(total.cpu().numpy(), want)


def test_evaluate_topk_across_rank_count_chunks():
    """evaluate_topk at V > 16384 (two column chunks of aae_rank_counts, several gold groups per row) == the oracle's
    evaluate on the dense prediction.  Gold items are drawn among items whose float64 logit is farther from every other
    item's than the fp32 rounding of the two computations, so that both rankings place them identically."""
    from aaerec_b200.aae import AdversarialAutoEncoder
    from oracle import aae_oracle as O
    V, H, C, n = 20000, 100, 50, 120
    params = O.init_params(V, H, C, seed=13)
    params["dec.lin3.weight"] = params["dec.lin3.weight"] * 8.0
    model = AdversarialAutoEncoder(n_hidden=H, n_code=C, batch_size=50, n_epochs=1, verbose=False)
    model._build(V, C, params={k: v.clone() for k, v in params.items()})
    X = _sets(n, V, seed=31, mean_len=12)
    dense = X.toarray()
    oracle = O.OracleAAE({k: torch.as_tensor(v) for k, v in model.state_dict().items()}, n_code=C)
    Z = oracle.logits(dense).astype(np.float64)
    tol = 2e-5 * np.abs(Z).max(axis=1, keepdims=True) + 1e-6
    o = np.argsort(Z, axis=1)
    zs = np.take_along_axis(Z, o, 1)
    gap = np.diff(zs, axis=1)
    lo_gap = np.c_[np.full((n, 1), np.inf), gap]
    hi_gap = np.c_[gap, np.full((n, 1), np.inf)]
    sep_sorted = np.minimum(lo_gap, hi_gap) > 4 * tol
    sep = np.zeros_like(sep_sorted)
    np.put_along_axis(sep, o, sep_sorted, 1)
    rs = np.random.RandomState(3)
    Y = ((rs.rand(n, V) < 0.01) & (dense == 0) & sep).astype(np.float32)
    Y[np.arange(n), np.where(dense > 0, np.inf, Z).argmin(axis=1)] = 0   # the reference-side tie at 0 after scaling
    Y[7] = 0
    assert (Y.sum(1) > 8).mean() > 0.9                                   # several gold groups per row
    pred = 1.0 / (1.0 + np.exp(-Z))
    metrics = ["mrr@5", "mrr@10", "map@5", "map@20", "p@5", "p@20", "P@1", "mrr", "map"]
    want = O.evaluate(Y, O.remove_non_missing(pred, dense), metrics)
    got = model.evaluate_topk(X, sp.csr_matrix(Y), metrics, batch_size=50)
    for name, (a, b), (c, d) in zip(metrics, got, want):
        assert abs(a - c) < 1e-6 and abs(b - d) < 1e-6, (name, got, want)
